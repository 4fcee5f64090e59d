// PSD synthesis (simul_psd_wfm, psfrec.py:36-151).
//
//  ao_zone_kernel : the 80 x 80 AO-corrected zone per (draw, direction): GLAO LSE
//                   reconstructor (calc_mat_rec_glao_finale, :218-364, one reconstruction
//                   layer) and residual PSD = reconstruction + servo-lag + anisoplanatism
//                   + propagated noise (calc_dsp_res_glao_finale, :367-525), all terms of one
//                   frequency cell evaluated by one thread in a single pass.
//  psd_fill_kernel: the dim x dim fitting PSD (psd_fit, :616-626), one pow() per four
//                   mirror-symmetric cells, merged with the AO zone by max() (:148-149) and
//                   scaled to nm^2 (:151), written with coalesced FP64 stores.
//  var_kernel     : residual-phase variance record of every plane (fitting / noise / projection
//                   error budget, DESIGN.md 5.5) from the same AO-zone terms and fitting quadrant.
#include "psfr_internal.h"

namespace psfr {

struct cd { double x, y; };
__device__ __forceinline__ cd cmul_(cd a, cd b) { return {a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x}; }
__device__ __forceinline__ cd cexp_i(double ang) {
    double s, c;
    sincos(ang, &s, &c);
    return {c, s};
}
// numpy.sinc: sin(pi x)/(pi x), 1 at x == 0
__device__ __forceinline__ double np_sinc(double x) {
    if (x == 0.0) return 1.0;
    const double y = 3.141592653589793 * x;
    return sin(y) / y;
}

// x^(-11/6) = x^(1/6) / x^2 with x^(1/6) = sqrt(cbrt(x)): ~2 ulp (cbrt <= 1 ulp, halved by the
// correctly rounded sqrt, plus two roundings) at well under half the instructions of pow()
__device__ __forceinline__ double pow_m11_6(double x) { return sqrt(cbrt(x)) / (x * x); }

struct PsdParams {
    const double* draws;   // [ndraw][PSFR_DRAW_NPAR]
    const double* geom;    // f, f_x, f_y tables [3][80][80]
    const double* dirs;    // [2][ndir] arcsec
    const double* pos;     // [2][npos] arcsec
    double* ao;            // [nplanes][80][80] centred, reference orientation
    int ndraw, ndir;
    int ngs;               // guide stars of every draw; 0: each draw's own count (slot PSFR_DRAW_NGS)
    int npos;              // columns of pos: a draw uses the first ngs of them
};

// The residual-PSD terms of AO-zone cell `cell` (u * 80 + v, before the transpose and shift of the zone
// mapping) of plane `plane`, unscaled: returns the propagated noise err_noise and calls layer(l, err_rec_l) for
// l = 0 .. nlayers - 1 in layer order, err_rec_l = |P beta_l - corr_l|^2 Cphi_l the projection error of layer l
// (servo lag, anisoplanatism and aliasing of that layer together: they do not add up separately).
// ao_zone_kernel and var_kernel share it, so both see the same terms.
template <class Layer>
__device__ __forceinline__ double ao_cell_terms(const PsdParams& p, int cell, int plane, Layer&& layer) {
    const int draw = plane / p.ndir, dir = plane % p.ndir;
    const double* dr = p.draws + (size_t)draw * PSFR_DRAW_NPAR;
    const double f = p.geom[cell], fx = p.geom[kAO * kAO + cell], fy = p.geom[2 * kAO * kAO + cell];
    const double pi = 3.141592653589793;
    const double pitch = 8.0 / 24.0;                 // Dpup / nsspup (psfrec.py:578)
    const double fc = 1 / (2 * pitch);
    const double wfs0 = 2 * pi * f * np_sinc(pitch * fx) * np_sinc(pitch * fy);   // wfs = i * wfs0
    // cut-off masks with the reference's precedence (A & B) | C  (psfrec.py:257, 435)
    const bool cut_rec = ((f != 0) && (fabs(fx) >= fc)) || (fabs(fy) >= fc);
    const bool cut_res = ((f != 0) && (fabs(fx) > fc)) || (fabs(fy) > fc);
    const double w_rec = cut_rec ? 0.0 : wfs0;
    const double w_res = cut_res ? 0.0 : wfs0;
    const int ngs = p.ngs ? p.ngs : (int)dr[PSFR_DRAW_NGS];
    const double h_rec = 1.0, h_dm = 1.0, sig = 1.0;
    const double ti = 1 / 1000.0, td = 2.5 * 1.e-3;
    const double dT = ti + td;

    // reconstructor W_j = conj(Mr_j)/sigma / sum_k |Mr_k|^2   (LSE, :310-362)
    cd back[kMaxGS];
    double map = 0.0;
    for (int j = 0; j < ngs; ++j) {
        const double px = p.pos[j] / 60, py = p.pos[p.npos + j] / 60;   // arcmin (:536)
        const double sx = fx * px * h_rec * 60 / 206265;
        const double sy = fy * py * h_rec * 60 / 206265;
        const cd e = cexp_i(2 * pi * (sx + sy));
        const cd mr = {-w_rec * e.y, w_rec * e.x};          // i * w_rec * e
        back[j] = {mr.x * (1 / sig), -mr.y * (1 / sig)};
        map += back[j].x * mr.x - back[j].y * mr.y;          // conj(mr) * mr is exactly real
    }
    const double inv = (map != 0.0 && cell != 0) ? 1.0 / map : 0.0;

    const double bx = p.dirs[dir] / 60, by = p.dirs[p.ndir + dir] / 60;
    const double bf = bx * fx + by * fy;
    const cd pdm = cexp_i(2 * pi * h_dm * 60 / 206265 * bf);
    cd pw[kMaxGS];
    double err_noise = 0.0;
    for (int j = 0; j < ngs; ++j) {
        const cd w = {inv * back[j].x, inv * back[j].y};
        pw[j] = cmul_(pdm, w);
        err_noise += (pw[j].x * pw[j].x + pw[j].y * pw[j].y) * sig;
    }

    const int nl = (int)dr[PSFR_DRAW_NLAYERS];
    const double L0 = dr[PSFR_DRAW_L0];
    const double vk = pow_m11_6(f * f + (1 / L0) * (1 / L0));
    for (int l = 0; l < nl; ++l) {
        const double* ly = dr + PSFR_DRAW_LAYER0 + PSFR_LAYER_NPAR * l;
        const double h = ly[PSFR_LAYER_H];
        const double wx = ly[PSFR_LAYER_WX], wy = ly[PSFR_LAYER_WY];
        const double lag = np_sinc(wx * ti * fx + wy * ti * fy);
        cd acc = {0.0, 0.0};
        for (int j = 0; j < ngs; ++j) {
            const double px = p.pos[j] / 60, py = p.pos[p.npos + j] / 60;
            const double sx = fx * px * h * 60 / 206265;
            const double sy = fy * py * h * 60 / 206265;
            const cd e = cexp_i(2 * (sx + sy) * pi);
            const double a = lag * w_res;
            const cd mv = {-a * e.y, a * e.x};               // lag * i*w_res * e
            const cd t = cmul_(pw[j], mv);
            acc.x += t.x;
            acc.y += t.y;
        }
        const cd pb = cexp_i(2 * pi * (h * 60 / 206265 * bf - (wx * dT * fx + wy * dT * fy)));
        const double prx = pb.x - acc.x, pry = pb.y - acc.y;
        layer(l, (prx * prx + pry * pry) * (ly[PSFR_LAYER_CPHI] * vk));
    }
    return err_noise;
}

__global__ void ao_zone_kernel(PsdParams p) {
    const int cell = blockIdx.x * blockDim.x + threadIdx.x;
    const int plane = blockIdx.y;
    if (cell >= kAO * kAO) return;
    const int u = cell / kAO, v = cell % kAO;
    double err_rec = 0.0;
    const double err_noise = ao_cell_terms(p, cell, plane, [&](int, double t) { err_rec += t; });
    double dsp = err_rec + err_noise;
    if (cell == 0) dsp = 0.0;
    // reference: transpose (moveaxis, :613) then fftshift (:149): zone[i][j] = dsp[(j+40)%80][(i+40)%80]
    const int i = (v + kAO / 2) % kAO, j = (u + kAO / 2) % kAO;
    p.ao[((size_t)plane * kAO + i) * kAO + j] = dsp;
}

// psd_fit (psfrec.py:616-626) at quadrant cell (a, b), unscaled.  Evaluated with the smaller
// index first, so that fit(a, b) and fit(b, a) are the same bits whatever the compiler contracts
// into an FMA: psd_quad_kernel evaluates one triangle and mirrors it.
__device__ __forceinline__ double fit_cell(int a, int b, int kN, double fitc, double inv_l0sq) {
    const double L = 16.0, fc = 1 / (2 * (8.0 / 24.0));
    const int lo = min(a, b), hi = max(a, b);
    const double ua = (lo - (kN - 1) / 2.0) / L, ub = (hi - (kN - 1) / 2.0) / L;
    const double f = sqrt(ua * ua + ub * ub);
    return f >= fc ? fitc * pow_m11_6(f * f + inv_l0sq) : 0.0;
}

__global__ void psd_fill_kernel(const double* __restrict__ draws, const double* __restrict__ ao,
                                double* __restrict__ psd, int ndir, double scale2, int kN) {
    // one thread per quadrant cell (a, b), a, b in [0, N/2): fit(a,b) = fit(N-1-a, b) = ...
    const int kNH = kN / 2;
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    const int a = blockIdx.y;
    const int plane = blockIdx.z;
    if (b >= kNH) return;
    const double* dr = draws + (size_t)(plane / ndir) * PSFR_DRAW_NPAR;
    const double L0 = dr[PSFR_DRAW_L0];
    const double fit = fit_cell(a, b, kN, dr[PSFR_DRAW_FITC], (1 / L0) * (1 / L0));
    double* base = psd + (size_t)plane * kN * kN;
    const int lo = kNH - kAO / 2, hi = kNH + kAO / 2;
    const double* z = ao + (size_t)plane * kAO * kAO;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int aa = (q & 1) ? kN - 1 - a : a;
        const int bb = (q & 2) ? kN - 1 - b : b;
        double val = fit;
        if (aa >= lo && aa < hi && bb >= lo && bb < hi) val = fmax(fit, z[(aa - lo) * kAO + (bb - lo)]);
        base[(size_t)aa * kN + bb] = val * scale2;
    }
}

// one mirror quadrant of the fitting PSD, unscaled: Q[a][b], a, b < N/2 (the fit is symmetric under
// a -> N-1-a and b -> N-1-b and identical for the directions of a draw).  The fused path never
// materialises the N x N PSD: LoadEvenRowsQuad (psfr_passes.cu) applies the AO-zone max() and the
// nm^2 scale with the same operations in the same order as psd_fill_kernel, so both paths give
// bit-identical structure functions.
// The fit depends on (a, b) through ua^2 + ub^2 only: one 32 x 32 tile per unordered tile pair
// (ta <= tb) is evaluated (x^(-11/6) is what the kernel costs) and written twice, straight and
// transposed through shared memory, both coalesced.
__global__ void __launch_bounds__(256)
psd_quad_kernel(const double* __restrict__ draws, double* __restrict__ q, int kN) {
    __shared__ double tile[32][33];
    const int kNH = kN / 2, nt = kNH / 32;
    // blockIdx.x enumerates the pairs (ta, tb), ta <= tb, row by row
    int ta = 0, rest = blockIdx.x;
    while (rest >= nt - ta) {
        rest -= nt - ta;
        ++ta;
    }
    const int tb = ta + rest;
    const double* dr = draws + (size_t)blockIdx.y * PSFR_DRAW_NPAR;
    const double L0 = dr[PSFR_DRAW_L0], fitc = dr[PSFR_DRAW_FITC], inv = (1 / L0) * (1 / L0);
    double* base = q + (size_t)blockIdx.y * kNH * kNH;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
    for (int r = ty; r < 32; r += 8) {
        const int a = ta * 32 + r, b = tb * 32 + tx;
        const double v = fit_cell(a, b, kN, fitc, inv);
        tile[r][tx] = v;
        base[(size_t)a * kNH + b] = v;
    }
    if (ta == tb) return;   // uniform per block: a diagonal tile holds both of its triangles
    __syncthreads();
#pragma unroll
    for (int r = ty; r < 32; r += 8) base[(size_t)(tb * 32 + r) * kNH + ta * 32 + tx] = tile[tx][r];
}

// Residual-phase variance record of every (draw, direction) plane (DESIGN.md 5.5) from the quadrant form of the
// chunk's PSDs (d_psdq, d_ao).  One CTA per plane:
//  * the draw's fitting PSD over the whole grid, 4 x the sum of its quadrant;
//  * the 80 x 80 zone cells, each with the fit at the same full-grid cell (the value LoadEvenRowsQuad merges):
//    a cell whose AO value exceeds its fit moves that fit out of FIT and splits the AO value into NOISE and
//    PROJ = sum_l LAYER0 + l with ao_cell_terms.
// Each thread accumulates a fixed strided subset in order and the CTA adds the threads up in a fixed tree, so a
// record depends on its plane's data only: the same bits at every chunk size and through every entry point.
constexpr int kVarThreads = 256;
enum { kAccQuad = 0, kAccWonFit, kAccWonAo, kAccNoise, kAccProj, kAccLayer0, kAccN = kAccLayer0 + PSFR_MAX_LAYERS };

__global__ void __launch_bounds__(kVarThreads)
var_kernel(PsdParams p, const double* __restrict__ q, int kN, double* __restrict__ out) {
    __shared__ double acc[kAccN][kVarThreads];   // column t belongs to thread t alone until the tree sum
    const int t = threadIdx.x, plane = blockIdx.x;
    const int kNH = kN / 2, lo = kNH - kAO / 2;
    const double* qd = q + (size_t)(plane / p.ndir) * kNH * kNH;
    const double* z = p.ao + (size_t)plane * kAO * kAO;
    for (int k = 0; k < kAccN; ++k) acc[k][t] = 0.0;

    const double2* q2 = reinterpret_cast<const double2*>(qd);
    const int n2 = kNH * kNH / 2;
    double quad = 0.0;
#pragma unroll 8
    for (int i = t; i < n2; i += kVarThreads) {
        const double2 v = __ldg(q2 + i);
        quad += v.x;
        quad += v.y;
    }
    acc[kAccQuad][t] = quad;

    for (int zc = t; zc < kAO * kAO; zc += kVarThreads) {
        const int i = zc / kAO, j = zc % kAO;            // zone[i][j] sits at full-grid cell (lo + i, lo + j)
        const int a = lo + i, n = lo + j;
        const int qa = a < kNH ? a : kN - 1 - a, qn = n < kNH ? n : kN - 1 - n;
        const double fit = __ldg(qd + (size_t)qa * kNH + qn);
        const double ao = __ldg(z + zc);
        if (!(ao > fit)) continue;                       // fmax(fit, ao) is the fit: the cell counts to FIT
        // zone[i][j] = dsp[(j + 40) % 80][(i + 40) % 80] (ao_zone_kernel)
        const int cell = ((j + kAO / 2) % kAO) * kAO + (i + kAO / 2) % kAO;
        double proj = 0.0;
        const double noise = ao_cell_terms(p, cell, plane, [&](int l, double e) {
            acc[kAccLayer0 + l][t] += e;
            proj += e;
        });
        acc[kAccWonFit][t] += fit;
        acc[kAccWonAo][t] += ao;
        acc[kAccNoise][t] += noise;
        acc[kAccProj][t] += proj;
    }
    for (int s = kVarThreads / 2; s > 0; s >>= 1) {
        __syncthreads();
        if (t < s)
            for (int k = 0; k < kAccN; ++k) acc[k][t] += acc[k][t + s];
    }
    __syncthreads();
    // unscaled PSD -> nm^2 (psfrec.py:151, run_psd) and the grid step 1/L, L = 16 m: sum PSD / L^2
    const double k = 0.5 * 1000 / (2 * 3.141592653589793), L = 16.0;
    const double unit = (k * k) / (L * L);
    double* o = out + (size_t)plane * PSFR_VAR_NPAR;
    if (t < PSFR_MAX_LAYERS) o[PSFR_VAR_LAYER0 + t] = acc[kAccLayer0 + t][0] * unit;
    if (t == 0) {
        const double fit = 4.0 * acc[kAccQuad][0] - acc[kAccWonFit][0];
        o[PSFR_VAR_TOTAL] = (fit + acc[kAccWonAo][0]) * unit;
        o[PSFR_VAR_FIT] = fit * unit;
        o[PSFR_VAR_NOISE] = acc[kAccNoise][0] * unit;
        o[PSFR_VAR_PROJ] = acc[kAccProj][0] * unit;
    }
}

int run_var(Ctx* c, int ndraw, int ndir, int ngs, int npos, double* out_dev, cudaStream_t s) {
    PsdParams p{c->d_draws, c->d_geom, c->d_misc + kMiscDirs, c->d_misc + kMiscPos, c->d_ao, ndraw, ndir, ngs, npos};
    var_kernel<<<ndraw * ndir, kVarThreads, 0, s>>>(p, c->d_psdq, c->N, out_dev);
    PSFR_LAUNCH_CHECK(c);
    return PSFR_OK;
}

int run_psd(Ctx* c, int ndraw, int ndir, int ngs, int npos, cudaStream_t s, bool full) {
    const int nplanes = ndraw * ndir;
    PsdParams p{c->d_draws, c->d_geom, c->d_misc + kMiscDirs, c->d_misc + kMiscPos, c->d_ao, ndraw, ndir, ngs, npos};
    dim3 g1((kAO * kAO + 127) / 128, nplanes);
    ao_zone_kernel<<<g1, 128, 0, s>>>(p);
    PSFR_LAUNCH_CHECK(c);
    if (!full) {
        const int nt = c->NH / 32;                           // NH = 640 or 1280
        dim3 gq(nt * (nt + 1) / 2, ndraw);                   // one quadrant per DRAW, one triangle of tiles
        psd_quad_kernel<<<gq, 256, 0, s>>>(c->d_draws, c->d_psdq, c->N);
        PSFR_LAUNCH_CHECK(c);
        c->planes_loaded = 0;
        c->planes_struct = 0;
        return PSFR_OK;
    }
    const double k = 0.5 * 1000 / (2 * 3.141592653589793);
    dim3 g2((c->NH + 127) / 128, c->NH, nplanes);
    psd_fill_kernel<<<g2, 128, 0, s>>>(c->d_draws, c->d_ao, c->d_psd, ndir, k * k, c->N);
    PSFR_LAUNCH_CHECK(c);
    c->planes_loaded = nplanes;
    c->planes_struct = 0;
    return PSFR_OK;
}

}  // namespace psfr
