// Per-image tail of the path, one CTA per 40 x 40 image:
//   resample_kernel : clip >= 0, bilinear 80x80 samples -> 40x40, per-plane normalisation
//                     (psf_muse tail, psfrec.py:679-685 with interpolate :635-641)
//   (the two Moffat convolutions of convolve_final_psf live in psfr_conv.cu)
//   fit_kernel      : 5-parameter circular Moffat least squares by Levenberg-Marquardt with
//                     analytic Jacobian (fit_psf_cube -> mpdaf moffat_fit, :861-871)
//   mean / polyfit  : time mean of cubes (:1104) and polynomial smoothing (:1174-1210)
#include <algorithm>
#include <cmath>
#include <type_traits>
#include "psfr_internal.h"
#include "fast_exp.cuh"

namespace psfr {

constexpr int kImg = kPSF * kPSF;  // 1600

// deterministic block sum (blockDim.x multiple of 32, <= 1024); result valid in all threads
__device__ double block_sum(double v, double* red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
    return t;
}

// ---------------------------------------------------------------- Moffat kernels
// astropy Moffat2DKernel(gamma, alpha, x_size=41, y_size=41): amplitude (alpha-1)/(pi gamma^2),
// (1 + r^2/gamma^2)^(-alpha) at integer offsets, normalised to unit sum.
__global__ void moffat_kernels_kernel(const double* __restrict__ gam, const double* __restrict__ alp,
                                      int alp_stride, double* __restrict__ out) {
    __shared__ double red[32];
    const int k = blockIdx.x;
    const double g = gam[k], a = alp[k * alp_stride];
    const double amp = (a - 1) / (3.141592653589793 * g * g);
    double vals[7];
    double part = 0.0;
    int cnt = 0;
    for (int idx = threadIdx.x; idx < kKW * kKW; idx += blockDim.x, ++cnt) {
        const int dy = idx / kKW - kKW / 2, dx = idx % kKW - kKW / 2;
        const double rr = (double)(dx * dx + dy * dy) / (g * g);
        vals[cnt] = amp * pow(1 + rr, -a);
        part += vals[cnt];
    }
    const double tot = block_sum(part, red);
    cnt = 0;
    for (int idx = threadIdx.x; idx < kKW * kKW; idx += blockDim.x, ++cnt)
        out[(size_t)k * kKW * kKW + idx] = vals[cnt] / tot;
}

// ---------------------------------------------------------------- resample
__global__ void __launch_bounds__(256)
resample_kernel(const double* __restrict__ samp, const double* __restrict__ frac, int nlam,
                double* __restrict__ cube) {
    extern __shared__ double dyn_smem[];
    double* s = dyn_smem;               // kNS*kNS
    double* red = dyn_smem + kNS * kNS; // 32
    const int img = blockIdx.x, lam = img % nlam;
    const double* src = samp + (size_t)img * kNS * kNS;
    for (int i = threadIdx.x; i < kNS * kNS; i += blockDim.x) s[i] = fmax(src[i], 0.0);   // :680
    __syncthreads();
    const double* fr = frac + (size_t)lam * kPSF;
    double vals[7];
    double part = 0.0;
    int cnt = 0;
    for (int idx = threadIdx.x; idx < kImg; idx += blockDim.x, ++cnt) {
        const int y = idx / kPSF, x = idx % kPSF;
        const double fy = fr[y], fx = fr[x];
        const double* r0 = s + (2 * y) * kNS + 2 * x;
        const double v = (1 - fy) * ((1 - fx) * r0[0] + fx * r0[1]) +
                         fy * ((1 - fx) * r0[kNS] + fx * r0[kNS + 1]);
        vals[cnt] = v;
        part += v;
    }
    const double tot = block_sum(part, red);   // :685
    cnt = 0;
    for (int idx = threadIdx.x; idx < kImg; idx += blockDim.x, ++cnt)
        cube[(size_t)img * kImg + idx] = vals[cnt] / tot;
}

// ---------------------------------------------------------------- Moffat fit
// model f = I (1 + ((p-y0)^2 + (q-x0)^2)/a^2)^(-n), parameters x = [I, y0, x0, a, n].
// One WARP per image (4 images per CTA): the image sits in shared memory, every lane owns
// npx/32 pixels, the 21 sums of the normal equations are reduced with xor-shuffles (all lanes
// end with bit-identical sums, so the 5x5 solve and the LM control flow run redundantly and
// uniformly in every lane) - no block-level synchronisation at all.
constexpr int kFitWarps = 4;
// resident CTAs per SM the fitter is compiled for (register budget 65536 / (128 * this))
#ifndef PSFR_FIT_MINBLOCKS
#define PSFR_FIT_MINBLOCKS 4
#endif
// The two-stage fit: pixel stride and squared relative-step tolerance of the coarse stage, squared
// relative-step tolerance of the final stage = (1.49e-8)^2, the xtol at which MINPACK - the reference's
// solver behind mpdaf - stops.  Measured on the 4480 images of a config-4 chunk (tools/fit_bench.py):
// stride 4 / final 1e-9: 0.646 ms; stride 8: 0.600; final 1.49e-8: 0.610; both: 0.556 ms with FWHM / beta
// within 1.5e-8 / 4.3e-8 of the tighter solution (bar 1e-5); strides 16 and 32 need more iterations than they save.
#ifndef PSFR_FIT_COARSE_STEP
#define PSFR_FIT_COARSE_STEP 8
#endif
#ifndef PSFR_FIT_COARSE_TOL2
#define PSFR_FIT_COARSE_TOL2 1e-6
#endif
#ifndef PSFR_FIT_TOL2
#define PSFR_FIT_TOL2 2.2e-16
#endif
// Sizes of the normal equations of an NP-parameter least-squares fit: the packed upper triangle of J^T J,
// then J^T r, then the cost r.r.
template <int NP>
struct Normal {
    static constexpr int NJJ = NP * (NP + 1) / 2;
    static constexpr int NSUM = NJJ + NP + 1;
    static constexpr int COST = NSUM - 1;
};

// packed-upper index of (i, j), i <= j
template <int NP>
__device__ __forceinline__ constexpr int pk(int i, int j) { return i * NP - i * (i - 1) / 2 + (j - i); }

template <int NSUM>
__device__ __forceinline__ void warp_sum_vec(double* v) {
#pragma unroll
    for (int k = 0; k < NSUM; ++k) {
        double t = v[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
        v[k] = t;
    }
}

// 1/u for u in [1, 1e300): hardware seed + two Newton steps (no special cases to test for)
__device__ __forceinline__ double rcp_pos(double u) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(u));
    double e = fma(-u, r, 1.0);
    r = fma(r, e, r);
    e = fma(-u, r, 1.0);
    return fma(r, e, r);
}

// log(u) for u in [1, 2^60): u = 2^k m with m in [sqrt(1/2), sqrt(2)), log m = 2 atanh(s),
// s = (m - 1)/(m + 1), |s| <= 0.1716, series to s^23; k ln2 added in two words.  Branch-free and
// half as long as the library log, whose dependent chain dominated the per-pixel latency of the
// fitter (the kernel runs one image per warp in a single wave).  Max relative error 3.8e-16
// against a long-double log1p over [1 + 1e-8, 1e4] (the argument is 1 + rho^2 here).
// series coefficients 1/23 ... 1/3 and the two words of ln 2 in constant memory (see fast_exp.cuh: immediates
// cost two uniform-register moves per use)
static __constant__ double kLogPoly[11] = {1.0 / 23, 1.0 / 21, 1.0 / 19, 1.0 / 17, 1.0 / 15, 1.0 / 13,
                                           1.0 / 11, 1.0 / 9,  1.0 / 7,  1.0 / 5,  1.0 / 3};
static __constant__ double kLn2[2] = {6.93147180369123816490e-01, 1.90821492927058770002e-10};
__device__ __forceinline__ double log_ge1(double u) {
    int hi = __double2hiint(u);
    const int k = (hi - 0x3fe6a09e) >> 20;
    hi -= k << 20;
    const double m = __hiloint2double(hi, __double2loint(u));
    const double s = (m - 1.0) * rcp_pos(m + 1.0);
    const double z = s * s;
    double p = kLogPoly[0];
#pragma unroll
    for (int i = 1; i < 11; ++i) p = fma(p, z, kLogPoly[i]);
    const double kf = (double)k;
    double r = fma(s * z, 2.0 * p, kf * kLn2[1]);
    r += 2.0 * s;
    return fma(kf, kLn2[0], r);
}

// packed indices of the diagonal of J^T J
template <int NP>
struct DiagIndex {
    int v[NP];
    __device__ constexpr DiagIndex() : v() {
        for (int i = 0; i < NP; ++i) v[i] = pk<NP>(i, i);
    }
};

// one pixel's contribution J (NP entries) and residual r to the normal equations
template <int NP>
__device__ __forceinline__ void add_normal(const double* J, double r, double* sums) {
    constexpr int NJJ = Normal<NP>::NJJ;
#pragma unroll
    for (int i = 0; i < NP; ++i)
#pragma unroll
        for (int j = i; j < NP; ++j) sums[pk<NP>(i, j)] = fma(J[i], J[j], sums[pk<NP>(i, j)]);
#pragma unroll
    for (int i = 0; i < NP; ++i) sums[NJJ + i] = fma(J[i], r, sums[NJJ + i]);
    sums[NJJ + NP] = fma(r, r, sums[NJJ + NP]);
}

// the same with a pixel weight w: J^T W J, J^T W r and r^T W r.  w = 1 gives add_normal's bits (w J_i and w r are
// exact), so a unit-weight star fit reproduces the plain fit.
template <int NP>
__device__ __forceinline__ void add_normal_w(const double* J, double r, double w, double* sums) {
    constexpr int NJJ = Normal<NP>::NJJ;
#pragma unroll
    for (int i = 0; i < NP; ++i) {
        const double wj = w * J[i];
#pragma unroll
        for (int j = i; j < NP; ++j) sums[pk<NP>(i, j)] = fma(wj, J[j], sums[pk<NP>(i, j)]);
        sums[NJJ + i] = fma(wj, r, sums[NJJ + i]);
    }
    const double wr = w * r;
    sums[NJJ + NP] = fma(wr, r, sums[NJJ + NP]);
}

// The models the Levenberg-Marquardt driver below fits.  Each is built from the parameter vector x once
// per pass over the image (per-pass constants), gives one pixel's contribution to the normal equations at
// offset (dp, dq) = (row - y0, column - x0), and says which trial points it refuses.
//
// Circular Moffat f = I (1 + ((p-y0)^2 + (q-x0)^2)/a^2)^(-n), x = [I, y0, x0, a, n].
struct CircularMoffat {
    static constexpr int NP = 5;
    double I, n, ia2, ia;
    __device__ __forceinline__ explicit CircularMoffat(const double* x)
        : I(x[0]), n(x[4]), ia2(1.0 / (x[3] * x[3])), ia(1.0 / x[3]) {}
    static constexpr bool kWeighted = false;
    // model value at offset (dp, dq); J receives its NP derivatives
    __device__ __forceinline__ double eval(double dp, double dq, double* J) const {
        const double rho2 = (dp * dp + dq * dq) * ia2;
        const double uu = 1.0 + rho2;
        const double lu = log_ge1(uu);
        const double m = fast_exp(-n * lu);        // u^-n
        const double f = I * m;
        const double g = 2.0 * n * f * rcp_pos(uu);  // 2 I n u^(-n-1)
        J[0] = m;
        J[1] = g * dp * ia2;
        J[2] = g * dq * ia2;
        J[3] = g * rho2 * ia;
        J[4] = -f * lu;
        return f;
    }
    __device__ __forceinline__ void pixel(double dp, double dq, double pix, double* sums) const {
        double J[NP];
        const double f = eval(dp, dq, J);
        add_normal<NP>(J, f - pix, sums);
    }
    static __device__ __forceinline__ bool refuses(const double* xt) {
        return !(xt[3] > 0.0) || !(xt[4] > 0.0) || !isfinite(xt[0]);
    }
};

// Elliptical Moffat f = I (1 + A dp^2 + B dq^2 + C dp dq)^(-n), x = [I, y0, x0, A, B, C, n].  The quadratic
// form keeps every Jacobian column alive at a circle (A = B, C = 0), where the rotation column of the
// (a, e, rot) parameterisation vanishes.
struct EllipticalMoffat {
    static constexpr int NP = 7;
    double I, A, B, C, n;
    __device__ __forceinline__ explicit EllipticalMoffat(const double* x)
        : I(x[0]), A(x[3]), B(x[4]), C(x[5]), n(x[6]) {}
    static constexpr bool kWeighted = false;
    __device__ __forceinline__ double eval(double dp, double dq, double* J) const {
        const double pp = dp * dp, qq = dq * dq, pq = dp * dq;
        const double uu = 1.0 + fma(A, pp, fma(B, qq, C * pq));
        const double lu = log_ge1(uu);
        const double m = fast_exp(-n * lu);        // u^-n
        const double f = I * m;
        const double g = n * f * rcp_pos(uu);        // I n u^(-n-1)
        J[0] = m;
        J[1] = g * fma(2.0 * A, dp, C * dq);
        J[2] = g * fma(2.0 * B, dq, C * dp);
        J[3] = -g * pp;
        J[4] = -g * qq;
        J[5] = -g * pq;
        J[6] = -f * lu;
        return f;
    }
    __device__ __forceinline__ void pixel(double dp, double dq, double pix, double* sums) const {
        double J[NP];
        const double f = eval(dp, dq, J);
        add_normal<NP>(J, f - pix, sums);
    }
    // the form must stay positive definite (u >= 1 everywhere)
    static __device__ __forceinline__ bool refuses(const double* xt) {
        return !(xt[3] > 0.0) || !(xt[4] > 0.0) || !(4.0 * xt[3] * xt[4] - xt[5] * xt[5] > 0.0) || !(xt[6] > 0.0) ||
               !isfinite(xt[0]);
    }
};

// A star fit of model M (DESIGN.md 5.7): every pixel carries a weight w, stored in shared memory right after the image
// (npx further doubles; 0 on unused pixels, whose data were zeroed on load), and with kBack the model gains a constant
// background c, the last parameter, with the Jacobian column dc = 1.
template <class M, bool kBack>
struct StarModel {
    static constexpr int NP = M::NP + (kBack ? 1 : 0);
    static constexpr bool kWeighted = true;
    M m;
    double c;
    __device__ __forceinline__ explicit StarModel(const double* x) : m(x), c(kBack ? x[M::NP] : 0.0) {}
    __device__ __forceinline__ void pixel(double dp, double dq, double pix, double w, double* sums) const {
        double J[NP];
        const double f = m.eval(dp, dq, J);
        if constexpr (kBack) J[M::NP] = 1.0;
        add_normal_w<NP>(J, kBack ? (f + c) - pix : f - pix, w, sums);
    }
    static __device__ __forceinline__ bool refuses(const double* xt) {
        return M::refuses(xt) || (kBack && !isfinite(xt[NP - 1]));
    }
};

// accumulate normal equations at x over this lane's pixels (two independent pixel chains per
// trip so that the log / exp latencies overlap), then reduce over the warp.  STEP = 1 visits every
// pixel; STEP = 4 every fourth pixel of each lane (a quasi-uniform quarter of the image), used
// by the coarse first stage of the fit.  `env` is whatever the model needs besides x (the template fit's
// coefficient array); the Moffat models take none.
template <class M, int STEP, class... Env>
__device__ __forceinline__ void accumulate(const double* __restrict__ img, int npx, int nx, const double* x,
                                           double* sums, const Env&... env) {
#pragma unroll
    for (int k = 0; k < Normal<M::NP>::NSUM; ++k) sums[k] = 0.0;
    const double y0 = x[1], x0 = x[2];
    const M model(x, env...);
    const int lane = threadIdx.x & 31;
    int pr = lane / nx, qc = lane % nx;          // once per call; then stepped incrementally
    const int dpr = (32 * STEP) / nx, dqc = (32 * STEP) % nx;
    auto step = [&]() {
        pr += dpr;
        qc += dqc;
        if (qc >= nx) {
            qc -= nx;
            ++pr;
        }
    };
    int idx = lane;
    for (; idx + 32 * STEP < npx; idx += 64 * STEP) {
        const double dp0 = (double)pr - y0, dq0 = (double)qc - x0;
        step();
        const double dp1 = (double)pr - y0, dq1 = (double)qc - x0;
        step();
        if constexpr (M::kWeighted) {   // the weights follow the image
            model.pixel(dp0, dq0, img[idx], img[npx + idx], sums);
            model.pixel(dp1, dq1, img[idx + 32 * STEP], img[npx + idx + 32 * STEP], sums);
        } else {
            model.pixel(dp0, dq0, img[idx], sums);
            model.pixel(dp1, dq1, img[idx + 32 * STEP], sums);
        }
    }
    if (idx < npx) {
        if constexpr (M::kWeighted)
            model.pixel((double)pr - y0, (double)qc - x0, img[idx], img[npx + idx], sums);
        else
            model.pixel((double)pr - y0, (double)qc - x0, img[idx], sums);
    }
    warp_sum_vec<Normal<M::NP>::NSUM>(sums);
}

// Cholesky of A + mu diag(A) (A from the packed sums), fully unrolled in registers.
// L holds the factor with the RECIPROCAL of the diagonal on the diagonal.
template <int NP>
__device__ __forceinline__ bool cholesky(const double* s, double mu, double (&L)[NP][NP]) {
    bool ok = true;
#pragma unroll
    for (int i = 0; i < NP; ++i) {
#pragma unroll
        for (int j = 0; j <= i; ++j) {
            double t = s[pk<NP>(j, i)];
            if (i == j) t *= (1.0 + mu);
#pragma unroll
            for (int q = 0; q < j; ++q) t = fma(-L[i][q], L[j][q], t);
            if (i == j) {
                ok = ok && (t > 0.0);
                L[i][i] = rsqrt(t);
            } else {
                L[i][j] = t * L[j][j];
            }
        }
    }
    return ok;
}

// solve L L^T z = b in place
template <int NP>
__device__ __forceinline__ void chol_solve(const double (&L)[NP][NP], double* z) {
#pragma unroll
    for (int i = 0; i < NP; ++i) {
        double t = z[i];
#pragma unroll
        for (int q = 0; q < i; ++q) t = fma(-L[i][q], z[q], t);
        z[i] = t * L[i][i];
    }
#pragma unroll
    for (int i = NP - 1; i >= 0; --i) {
        double t = z[i];
#pragma unroll
        for (int q = i + 1; q < NP; ++q) t = fma(-L[q][i], z[q], t);
        z[i] = t * L[i][i];
    }
}

// Levenberg-Marquardt of model M on the pixel subset STEP from the start point x (updated in place);
// sums holds the normal equations at the final x.  tol2 = square of the relative step at which
// to stop (MINPACK, the reference's solver, stops at 1.49e-8; so does the final stage).  env as accumulate.
template <class M, int STEP, class... Env>
__device__ __forceinline__ void lm_solve(const double* __restrict__ img, int npx, int nx, double* x, double* sums,
                                         double tol2, int max_iter, int& iter, int& status, const Env&... env) {
    constexpr int kNP = M::NP, NJJ = Normal<kNP>::NJJ, kNSUM = Normal<kNP>::NSUM, COST = Normal<kNP>::COST;
    double trial[kNSUM], xt[kNP], d[kNP];
    accumulate<M, STEP>(img, npx, nx, x, sums, env...);
    double mu = 1e-3, nu = 2.0;
    status = -1;
    constexpr DiagIndex<kNP> dia;
    double L[kNP][kNP];
    for (iter = 1; iter <= max_iter; ++iter) {
        // every lane runs the identical solve on bit-identical sums
        if (!cholesky(sums, mu, L)) {
            mu *= nu;
            nu *= 2.0;
            if (mu > 1e15) break;
            continue;
        }
#pragma unroll
        for (int i = 0; i < kNP; ++i) d[i] = -sums[NJJ + i];
        chol_solve(L, d);
        double dn = 0.0, xn = 0.0, pred = 0.0;
#pragma unroll
        for (int i = 0; i < kNP; ++i) {
            xt[i] = x[i] + d[i];
            const double sc2 = sums[dia.v[i]];           // |J column|^2
            dn = fma(d[i] * d[i], sc2, dn);
            xn = fma(x[i] * x[i], sc2, xn);
            // predicted decrease of r.r : d.(mu D d - g)
            pred += d[i] * (mu * sc2 * d[i] - sums[NJJ + i]);
        }
        if (M::refuses(xt, env...)) {
            mu *= nu;
            nu *= 2.0;
            if (mu > 1e15) break;
            continue;
        }
        accumulate<M, STEP>(img, npx, nx, xt, trial, env...);
        const double actual = sums[COST] - trial[COST];
        // near the minimum the cost is flat to rounding: tolerate a noise-level increase so that
        // Gauss-Newton steps keep contracting, and stop on the (column-scaled) step size
        // MINPACK (the reference, through mpdaf -> scipy leastsq) stops at a relative step of 1.49e-8
        const bool small = dn <= tol2 * (xn + 1e-300);            // relative step <= sqrt(tol2)
        if (isfinite(trial[COST]) && actual >= -1e-13 * sums[COST]) {
            const double rho = pred > 0.0 ? actual / pred : 1.0;
#pragma unroll
            for (int i = 0; i < kNP; ++i) x[i] = xt[i];
#pragma unroll
            for (int k = 0; k < kNSUM; ++k) sums[k] = trial[k];
            const double t = 2.0 * rho - 1.0;
            mu *= fmax(1.0 / 3.0, 1.0 - t * t * t);
            if (mu < 1e-15) mu = 1e-15;
            nu = 2.0;
            if (small) {
                status = iter;
                break;
            }
        } else {
            if (dn <= 1e-18 * (xn + 1e-300)) {   // step below 1e-9 relative and no decrease: rounding floor
                status = iter;
                break;
            }
            mu *= nu;
            nu *= 2.0;
            if (mu > 1e15) break;
        }
    }
}

// ---------------------------------------------------------------- star fits (DESIGN.md 5.7)
// Load image `image` and its weights (wts NULL: every weight 1) into the warp's shared memory, img[npx] then w[npx].
// A pixel is used when w > 0; the data and weight of every other pixel are zeroed here - selected, never multiplied -
// so that whatever it holds (NaN, inf) reaches no sum.  Returns the number of used pixels; `bad` is set when the
// image has a negative or non-finite weight, or non-finite data on a used pixel.  Warp-collective and warp-uniform.
__device__ __forceinline__ int load_star_image(const double* __restrict__ imgs, const double* __restrict__ wts,
                                               int image, int npx, double* img, bool& bad) {
    const int lane = threadIdx.x & 31;
    const double* src = imgs + (size_t)image * npx;
    const double* wsrc = wts ? wts + (size_t)image * npx : nullptr;
    int used = 0;
    bool b = false;
    for (int i = lane; i < npx; i += 32) {
        const double w = wsrc ? wsrc[i] : 1.0, d = src[i];
        const bool u = w > 0.0;
        b = b || !(w >= 0.0 && isfinite(w)) || (u && !isfinite(d));
        used += u ? 1 : 0;
        img[i] = u ? d : 0.0;
        img[npx + i] = u ? w : 0.0;
    }
    used = __reduce_add_sync(0xffffffffu, used);
    bad = __any_sync(0xffffffffu, b);
    __syncwarp();
    return used;
}

// Start value c0 of the background: the mean of the used pixels on the outermost ring of the stamp (rows 0 and
// ny - 1, columns 0 and nx - 1), 0 when none of them is used.  Warp-collective; the same bits in every lane.
__device__ __forceinline__ double ring_background(const double* img, int ny, int nx) {
    const int lane = threadIdx.x & 31, npx = ny * nx, nring = 2 * nx + 2 * (ny - 2);
    double v[2] = {0.0, 0.0};
    for (int k = lane; k < nring; k += 32) {
        const int r = k - 2 * nx;
        const int i = k < nx ? k : k < 2 * nx ? (ny - 1) * nx + (k - nx) : (r / 2 + 1) * nx + (r % 2) * (nx - 1);
        if (img[npx + i] > 0.0) {
            v[0] += img[i];
            v[1] += 1.0;
        }
    }
    warp_sum_vec<2>(v);
    return v[1] > 0.0 ? v[0] / v[1] : 0.0;
}

// record of an image that fails the star fit's check: ITER = 0 and every other slot NaN
__device__ __forceinline__ void fail_record(double* o, int npar, int iter_slot) {
    for (int i = 0; i < npar; ++i) o[i] = (i == iter_slot) ? 0.0 : nan("");
}

__device__ __forceinline__ void back_record(double* b, double cont, double err_cont, int npix) {
    b[PSFR_BACK_CONT] = cont;
    b[PSFR_BACK_ERR_CONT] = err_cont;
    b[PSFR_BACK_NPIX] = (double)npix;
}

// pixel i in the start-point statistics: its data, above c0 with a background (unused pixels hold 0)
template <bool kBack>
__device__ __forceinline__ double start_value(const double* img, int npx, int i, double c0) {
    if constexpr (kBack) return img[npx + i] > 0.0 ? img[i] - c0 : 0.0;
    else return img[i];
}

// ---------------------------------------------------------------- circular Moffat fit
// One driver for every circular fit.  kW = false, kBack = false is the reconstruction's fitter (fit_kernel); kW is a
// star fit (weights after the image in shared memory, the per-image check, dof over used pixels and the side record
// `back`), kBack adds the background parameter c.
template <bool kCoarse, bool kW, bool kBack>
__device__ __forceinline__ void fit_images(const double* __restrict__ imgs, const double* __restrict__ wts, int nimg,
                                           int ny, int nx, double* __restrict__ out, double* __restrict__ back,
                                           int* __restrict__ next_image) {
    using Model = std::conditional_t<kW, StarModel<CircularMoffat, kBack>, CircularMoffat>;
    constexpr int kNP = Model::NP, kNSUM = Normal<kNP>::NSUM, COST = Normal<kNP>::COST;
    extern __shared__ double sm[];
    const int npx = ny * nx, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int img_len = kW ? 2 * npx : npx;          // npx pixels (and npx weights)
    double* img = sm + (size_t)warp * (img_len + nx);    // ... + nx column weights
    // images are handed to the warps by a global counter: the LM iteration count varies 3x
    // between images, so a static one-image-per-warp grid ends in a long tail
#pragma unroll 1
    for (;;) {
    int image = 0;
    if (lane == 0) image = atomicAdd(next_image, 1);
    image = __shfl_sync(0xffffffffu, image, 0);
    if (image >= nimg) return;                       // whole warp leaves; no block barrier is used below
    __syncwarp();
    double* colw = img + img_len;
    int npu = npx;                                   // pixels in the fit
    double c0 = 0.0;                                 // start of the background
    if constexpr (kW) {
        bool bad;
        npu = load_star_image(imgs, wts, image, npx, img, bad);
        if (bad || npu <= kNP) {
            if (lane == 0) {
                fail_record(out + (size_t)image * PSFR_FIT_NPAR, PSFR_FIT_NPAR, PSFR_FIT_ITER);
                back_record(back + (size_t)image * PSFR_BACK_NPAR, nan(""), nan(""), npu);
            }
            __syncwarp();
            continue;
        }
        if constexpr (kBack) c0 = ring_background(img, ny, nx);
    } else {
        const double* src = imgs + (size_t)image * npx;
        for (int i = lane; i < npx; i += 32) img[i] = src[i];
        __syncwarp();
    }
    // ---- start point as mpdaf: peak pixel, width from Image.moments(), n = 2; a star fit takes them over the used
    // pixels (the others hold 0) and of the data above c0
    for (int q = lane; q < nx; q += 32) {
        double t = 0.0;
        for (int p = 0; p < ny; ++p) t += p * fabs(start_value<kBack>(img, npx, p * nx + q, c0));
        colw[q] = t;
    }
    __syncwarp();
    // first maximum of colw (column of the weighted sums) and of the image (peak pixel)
    double bestw = -1.0, bestv = -1e300;
    int qb = 0, ib = 0;
    for (int q = lane; q < nx; q += 32)
        if (colw[q] > bestw) { bestw = colw[q]; qb = q; }
    for (int i = lane; i < npx; i += 32)
        if ((!kW || img[npx + i] > 0.0) && start_value<kBack>(img, npx, i, c0) > bestv) {
            bestv = start_value<kBack>(img, npx, i, c0);
            ib = i;
        }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ow = __shfl_xor_sync(0xffffffffu, bestw, o);
        const int oq = __shfl_xor_sync(0xffffffffu, qb, o);
        if (ow > bestw || (ow == bestw && oq < qb)) { bestw = ow; qb = oq; }
        const double ov = __shfl_xor_sync(0xffffffffu, bestv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, ib, o);
        if (ov > bestv || (ov == bestv && oi < ib)) { bestv = ov; ib = oi; }
    }
    double num = 0.0, den = 0.0;
    for (int p = lane; p < ny; p += 32) {
        const double v = start_value<kBack>(img, npx, p * nx + qb, c0);
        num += fabs((p - qb) * v);
        den += fabs(v);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        num += __shfl_xor_sync(0xffffffffu, num, o);
        den += __shfl_xor_sync(0xffffffffu, den, o);
    }
    double x[kNP], sums[kNSUM];
    {
        const double wp = sqrt(num / den);
        const double fwhm0 = wp * 2.0 * sqrt(2.0 * log(2.0));
        x[0] = bestv;
        x[1] = ib / nx;
        x[2] = ib % nx;
        x[3] = fwhm0 / (2.0 * sqrt(sqrt(2.0) - 1.0));
        x[4] = 2.0;
        if constexpr (kBack) x[kNP - 1] = c0;
    }
    // Stage 1: Levenberg-Marquardt on every eighth pixel down to a relative step of 1e-3 - it
    // only moves the start point (the converged minimum does not depend on it); stage 2: all
    // pixels down to MINPACK's own tolerance, 1.49e-8.  Stage 1 visits pixels lane + 256 k of each
    // lane's pair loop: on an image of at most 512 pixels that is one or two 32-pixel strips (the
    // first rows of a 16 x 16, rows 0, 1, 15 and 16 of a 17 x 17), wings that can drive the start
    // away from the core, so run_fit launches the kCoarse = false instance on such images: stage 2 from the
    // moments start directly.
    int iter = 0, status = -1, coarse_iter = 0;
    if constexpr (kCoarse) {
        lm_solve<Model, PSFR_FIT_COARSE_STEP>(img, npx, nx, x, sums, PSFR_FIT_COARSE_TOL2, 12, iter, status);
        coarse_iter = iter;
    }
    lm_solve<Model, 1>(img, npx, nx, x, sums, PSFR_FIT_TOL2, 200, iter, status);
    iter += coarse_iter;
    if (status > 0) status += coarse_iter;
    const int max_iter = 212;
    if (lane == 0) {
        double* o = out + (size_t)image * PSFR_FIT_NPAR;
        const double a = fabs(x[3]), n = x[4];
        const double kf = 2.0 * sqrt(pow(2.0, 1.0 / n) - 1.0);
        o[PSFR_FIT_PEAK] = x[0];
        o[PSFR_FIT_Y0] = x[1];
        o[PSFR_FIT_X0] = x[2];
        o[PSFR_FIT_ALPHA] = a;
        o[PSFR_FIT_N] = n;
        o[PSFR_FIT_FWHM] = a * kf;
        o[PSFR_FIT_CHISQ] = sums[COST];
        o[PSFR_FIT_ITER] = (status > 0) ? (double)status : -(double)(iter > max_iter ? max_iter : iter);
        const double dof = (double)(npu - kNP);
        double L[kNP][kNP];
        if (cholesky(sums, 0.0, L)) {
            double e[kNP];
#pragma unroll
            for (int c = 0; c < kNP; ++c) {
                double z[kNP];
#pragma unroll
                for (int i = 0; i < kNP; ++i) z[i] = (i == c) ? 1.0 : 0.0;
                chol_solve(L, z);
                e[c] = sqrt(fabs(z[c]) * fabs(sums[COST] / dof));
            }
            o[PSFR_FIT_ERR_PEAK] = e[0];
            o[PSFR_FIT_ERR_Y0] = e[1];
            o[PSFR_FIT_ERR_X0] = e[2];
            o[PSFR_FIT_ERR_ALPHA] = e[3];
            o[PSFR_FIT_ERR_N] = e[4];
            // mpdaf Image.moffat_fit (fit_n, circular): err_fwhm = err_a * n; err_flux = err_I err_n err_a^2 err_e
            // with err_e = 0 for a circular fit (restated from mpdaf 3.x; the package is not in the reference tree)
            o[PSFR_FIT_ERR_FWHM] = e[3] * n;
            o[PSFR_FIT_ERR_FLUX] = e[0] * e[4] * e[3] * e[3] * 0.0;
            if constexpr (kW)
                back_record(back + (size_t)image * PSFR_BACK_NPAR, kBack ? x[kNP - 1] : 0.0, kBack ? e[kNP - 1] : 0.0,
                            npu);
        } else {
            for (int i = PSFR_FIT_ERR_PEAK; i <= PSFR_FIT_ERR_FWHM; ++i) o[i] = nan("");
            o[PSFR_FIT_ERR_FLUX] = nan("");
            if constexpr (kW)
                back_record(back + (size_t)image * PSFR_BACK_NPAR, kBack ? x[kNP - 1] : 0.0, kBack ? nan("") : 0.0,
                            npu);
        }
        o[PSFR_FIT_FLUX] = x[0] / (n - 1.0) * (3.141592653589793 * a * a);
    }
    __syncwarp();
    }   // next image
}

template <bool kCoarse>
__global__ void __launch_bounds__(kFitWarps * 32, PSFR_FIT_MINBLOCKS)
fit_kernel(const double* __restrict__ imgs, int nimg, int ny, int nx, double* __restrict__ out,
           int* __restrict__ next_image) {
    fit_images<kCoarse, false, false>(imgs, nullptr, nimg, ny, nx, out, nullptr, next_image);
}

// circular star fit: weights [nimg][ny][nx] (NULL: all 1), back [nimg][PSFR_BACK_NPAR]
template <bool kCoarse, bool kBack>
__global__ void __launch_bounds__(kFitWarps * 32, PSFR_FIT_MINBLOCKS)
star_fit_kernel(const double* __restrict__ imgs, const double* __restrict__ wts, int nimg, int ny, int nx,
                double* __restrict__ out, double* __restrict__ back, int* __restrict__ next_image) {
    fit_images<kCoarse, true, kBack>(imgs, wts, nimg, ny, nx, out, back, next_image);
}

// ---------------------------------------------------------------- elliptical Moffat fit
// resident CTAs per SM the elliptical fitter is compiled for: 36 sums, 36 trial sums and the 7 x 7 factor
// live in registers, so it runs at half the circular fitter's occupancy
#ifndef PSFR_EFIT_MINBLOCKS
#define PSFR_EFIT_MINBLOCKS 2
#endif
constexpr int kEfitMaxIter = 200;

// g^T (J^T J)^-1 g from the Cholesky factor of J^T J
template <int NP>
__device__ __forceinline__ double inv_quad(const double (&L)[NP][NP], const double* g) {
    double z[NP];
#pragma unroll
    for (int i = 0; i < NP; ++i) z[i] = g[i];
    chol_solve<NP>(L, z);
    double t = 0.0;
#pragma unroll
    for (int i = 0; i < NP; ++i) t = fma(g[i], z[i], t);
    return t;
}

// The elliptical record of x = [I, y0, x0, A, B, C, n] (include/psfr.h, PSFR_EFIT_*).  Each derived quantity
// q gets the error sqrt(grad q^T Sigma grad q), Sigma = (J^T J)^-1 chi^2/dof, with the gradient written out.
// NT = 8: x and the sums also hold the background c (star fits, DESIGN.md 5.7); npx is the number of pixels in
// the fit.
template <int NT>
__device__ void write_efit_record(const double* x, const double* sums, int npx, int iter, int status, double* o) {
    constexpr int NP = NT, COST = Normal<NP>::COST;
    constexpr double kPi = 3.141592653589793, kDeg = 180.0 / kPi;
    const double I = x[0], A = x[3], B = x[4], C = x[5], n = x[6];
    // eigenvalues of [[A, C/2], [C/2, B]]: the major axis belongs to the smaller one
    const double hd = 0.5 * (A - B), hc = 0.5 * C, S = 0.5 * (A + B);
    const double R2 = hd * hd + hc * hc, R = sqrt(R2);
    const double lmin = S - R, lmax = S + R;
    const double amaj = 1.0 / sqrt(lmin), amin = 1.0 / sqrt(lmax);
    // major axis from +x (column) toward +y (row): B x^2 + C x y + A y^2 is smallest along
    // angle 0.5 atan2(-C, A - B)
    double pa = 0.0;
    if (R2 != 0.0) {
        pa = 0.5 * atan2(-C, A - B);
        if (pa < 0.0) pa += kPi;
        pa *= kDeg;
        if (pa >= 180.0) pa -= 180.0;
        pa = fabs(pa);       // 0, not -0, for a major axis along +x
    }
    const double kf = 2.0 * sqrt(pow(2.0, 1.0 / n) - 1.0);
    const double dkf = -2.0 * pow(2.0, 1.0 / n) * 0.6931471805599453 / (n * n * kf);   // d kf / d n
    const double q = sqrt(lmin / lmax);
    const double flux = kPi * I * amaj * amin / (n - 1.0);
    o[PSFR_EFIT_PEAK] = I;
    o[PSFR_EFIT_Y0] = x[1];
    o[PSFR_EFIT_X0] = x[2];
    o[PSFR_EFIT_A_MAJOR] = amaj;
    o[PSFR_EFIT_A_MINOR] = amin;
    o[PSFR_EFIT_PA] = pa;
    o[PSFR_EFIT_N] = n;
    o[PSFR_EFIT_FWHM_MAJOR] = amaj * kf;
    o[PSFR_EFIT_FWHM_MINOR] = amin * kf;
    o[PSFR_EFIT_AXIS_RATIO] = q;
    o[PSFR_EFIT_CHISQ] = sums[COST];
    o[PSFR_EFIT_ITER] = (status > 0) ? (double)status : -(double)(iter > kEfitMaxIter ? kEfitMaxIter : iter);
    o[PSFR_EFIT_FLUX] = flux;
    double L[NP][NP];
    if (!cholesky<NP>(sums, 0.0, L)) {
        for (int i = PSFR_EFIT_ERR_PEAK; i <= PSFR_EFIT_ERR_AXIS_RATIO; ++i) o[i] = nan("");
        o[PSFR_EFIT_ERR_FLUX] = nan("");
        if (R2 == 0.0) o[PSFR_EFIT_ERR_PA] = INFINITY;
        return;
    }
    const double s2 = fabs(sums[COST] / (double)(npx - NP));
    auto err = [&](const double* g) { return sqrt(fabs(inv_quad<NP>(L, g)) * s2); };
    // the eigenvalues are not differentiable at a circle (R = 0): there their mean (A + B)/2 stands in
    const double ca = R > 0.0 ? hd / (2.0 * R) : 0.0, cc = R > 0.0 ? hc / (2.0 * R) : 0.0;
    const double gmaj = -0.5 * amaj * amaj * amaj, gmin = -0.5 * amin * amin * amin;   // d a / d lambda
    const double g_amaj[NP] = {0, 0, 0, gmaj * (0.5 - ca), gmaj * (0.5 + ca), -gmaj * cc, 0};
    const double g_amin[NP] = {0, 0, 0, gmin * (0.5 + ca), gmin * (0.5 - ca), gmin * cc, 0};
    double g[NP];
#pragma unroll
    for (int c = 0; c < EllipticalMoffat::NP; ++c) {
        if (c == 3 || c == 4 || c == 5) continue;
#pragma unroll
        for (int i = 0; i < NP; ++i) g[i] = (i == c) ? 1.0 : 0.0;
        o[c == 6 ? PSFR_EFIT_ERR_N : PSFR_EFIT_ERR_PEAK + c] = err(g);
    }
    o[PSFR_EFIT_ERR_A_MAJOR] = err(g_amaj);
    o[PSFR_EFIT_ERR_A_MINOR] = err(g_amin);
    if (R2 == 0.0) {
        o[PSFR_EFIT_ERR_PA] = INFINITY;
    } else {
        const double k = kDeg * 0.5 / (4.0 * R2);      // d atan2(-C, A - B) / 2, in degrees
        const double g_pa[NP] = {0, 0, 0, k * C, -k * C, -k * (A - B), 0};
        o[PSFR_EFIT_ERR_PA] = err(g_pa);
    }
#pragma unroll
    for (int i = 0; i < NP; ++i) g[i] = kf * g_amaj[i];
    g[6] = amaj * dkf;
    o[PSFR_EFIT_ERR_FWHM_MAJOR] = err(g);
#pragma unroll
    for (int i = 0; i < NP; ++i) g[i] = kf * g_amin[i];
    g[6] = amin * dkf;
    o[PSFR_EFIT_ERR_FWHM_MINOR] = err(g);
#pragma unroll
    for (int i = 0; i < NP; ++i) g[i] = q * (g_amin[i] / amin - g_amaj[i] / amaj);
    o[PSFR_EFIT_ERR_AXIS_RATIO] = err(g);
    // flux = pi I / ((n - 1) sqrt(det)), det = A B - C^2 / 4
    const double det = A * B - hc * hc, fd = -flux / (2.0 * det);
    const double g_flux[NP] = {kPi * amaj * amin / (n - 1.0), 0, 0, fd * B, fd * A, -fd * hc, -flux / (n - 1.0)};
    o[PSFR_EFIT_ERR_FLUX] = err(g_flux);
}

// error of the background of an elliptical star fit: sqrt((J^T W J)^-1_cc chi^2/dof), NaN where J^T W J is singular
__device__ __forceinline__ double efit_err_back(const double* sums, int npu) {
    constexpr int NP = EllipticalMoffat::NP + 1, COST = Normal<NP>::COST;
    double L[NP][NP];
    if (!cholesky<NP>(sums, 0.0, L)) return nan("");
    double g[NP];
#pragma unroll
    for (int i = 0; i < NP; ++i) g[i] = (i == NP - 1) ? 1.0 : 0.0;
    return sqrt(fabs(inv_quad<NP>(L, g)) * fabs(sums[COST] / (double)(npu - NP)));
}

// Start point of the elliptical fit from the image alone (warp-collective): peak pixel value, the centroid and
// second moments of the pixels at or above half of it (each pixel a unit square, hence + 1/12 per axis), and the
// quadratic form whose n = 2.5 Moffat has its half maximum on the ellipse of those moments (a uniform ellipse of
// semi-axes h has variance h^2 / 4 along each).  A star fit (kW) takes the used pixels only and, with a background,
// their data above c0, the background's start; x[7] = c0.
template <bool kW, bool kBack>
__device__ __forceinline__ void moments_start(const double* __restrict__ img, int npx, int nx, double c0, double* x) {
    const int lane = threadIdx.x & 31;
    double vmax = -INFINITY;
    for (int i = lane; i < npx; i += 32)
        if (!kW || img[npx + i] > 0.0) vmax = fmax(vmax, start_value<kBack>(img, npx, i, c0));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) vmax = fmax(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
    double m[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    for (int i = lane; i < npx; i += 32) {
        if (!(start_value<kBack>(img, npx, i, c0) >= 0.5 * vmax) || (kW && !(img[npx + i] > 0.0))) continue;
        const double p = (double)(i / nx), q = (double)(i % nx);
        m[0] += 1.0;
        m[1] += p;
        m[2] += q;
        m[3] += p * p;
        m[4] += q * q;
        m[5] += p * q;
    }
    warp_sum_vec<6>(m);
    const double mp = m[1] / m[0], mq = m[2] / m[0];
    const double spp = m[3] / m[0] - mp * mp + 1.0 / 12.0, sqq = m[4] / m[0] - mq * mq + 1.0 / 12.0;
    const double spq = m[5] / m[0] - mp * mq;
    const double k = 0.25 * (pow(2.0, 0.4) - 1.0) / (spp * sqq - spq * spq);
    x[0] = vmax;
    x[1] = mp;
    x[2] = mq;
    x[3] = k * sqq;
    x[4] = k * spp;
    x[5] = -2.0 * k * spq;
    x[6] = 2.5;
    if constexpr (kBack) x[7] = c0;
}

// A solution whose minor semi-axis is under 0.05 px (largest eigenvalue of the form above 400) leaves the model
// under 401^-n of its peak on every pixel but the nearest: one pixel sets the width and any narrower one fits as
// well (a lone hot pixel), so it is no answer and is reported as not converged.
__device__ __forceinline__ bool resolved(const double* x) {
    const double hd = 0.5 * (x[3] - x[4]), hc = 0.5 * x[5];
    return 0.5 * (x[3] + x[4]) + sqrt(hd * hd + hc * hc) <= 400.0;
}

// Elliptical Moffat fit of every image, one warp per image as fit_kernel, from the image's converged
// circular record circ [nimg][PSFR_FIT_NPAR]: (I, y0, x0, 1/a^2, 1/a^2, 0, n), all pixels, down to the
// final stage's tolerance.  out [nimg][PSFR_EFIT_NPAR].  kW, kBack as fit_images: a star fit also starts c from
// the circular star fit's side record circ_back and writes its own to back (the two may be the same array).
template <bool kW, bool kBack>
__device__ __forceinline__ void efit_images(const double* __restrict__ imgs, const double* __restrict__ wts,
                                            const double* __restrict__ circ, const double* circ_back, int nimg,
                                            int ny, int nx, double* __restrict__ out, double* back,
                                            int* __restrict__ next_image) {
    using Model = std::conditional_t<kW, StarModel<EllipticalMoffat, kBack>, EllipticalMoffat>;
    constexpr int kNP = Model::NP, kNSUM = Normal<kNP>::NSUM;
    extern __shared__ double sm[];
    const int npx = ny * nx, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* img = sm + (size_t)warp * (kW ? 2 * npx : npx);
#pragma unroll 1
    for (;;) {
        int image = 0;
        if (lane == 0) image = atomicAdd(next_image, 1);
        image = __shfl_sync(0xffffffffu, image, 0);
        if (image >= nimg) return;
        __syncwarp();
        int npu = npx;
        double c0 = 0.0;
        if constexpr (kW) {
            bool bad;
            npu = load_star_image(imgs, wts, image, npx, img, bad);
            if (bad || npu <= kNP) {
                if (lane == 0) {
                    fail_record(out + (size_t)image * PSFR_EFIT_NPAR, PSFR_EFIT_NPAR, PSFR_EFIT_ITER);
                    back_record(back + (size_t)image * PSFR_BACK_NPAR, nan(""), nan(""), npu);
                }
                __syncwarp();
                continue;
            }
            if constexpr (kBack) c0 = ring_background(img, ny, nx);
        } else {
            const double* src = imgs + (size_t)image * npx;
            for (int i = lane; i < npx; i += 32) img[i] = src[i];
            __syncwarp();
        }
        const double* c = circ + (size_t)image * PSFR_FIT_NPAR;
        const double ia2 = 1.0 / (c[PSFR_FIT_ALPHA] * c[PSFR_FIT_ALPHA]);
        double x[kNP] = {c[PSFR_FIT_PEAK], c[PSFR_FIT_Y0], c[PSFR_FIT_X0], ia2, ia2, 0.0, c[PSFR_FIT_N]};
        if constexpr (kBack) x[kNP - 1] = circ_back[(size_t)image * PSFR_BACK_NPAR + PSFR_BACK_CONT];
        double sums[kNSUM];
        int iter = 0, status = -1;
        lm_solve<Model, 1>(img, npx, nx, x, sums, PSFR_FIT_TOL2, kEfitMaxIter, iter, status);
        // A circular fit that did not converge (typically collapsed onto a one-pixel spike, alpha -> 0, on a PSF
        // narrower than a pixel along one axis) is no start for the ellipse, and neither start is sure to
        // converge: then fit again from the half-maximum moments and keep the converged result of lower chi^2.
        // Both conditions are warp-uniform; images whose two fits converge keep the bits of the first.
        if (status <= 0 || !(c[PSFR_FIT_ITER] > 0.0)) {
            double x1[kNP];
#pragma unroll
            for (int i = 0; i < kNP; ++i) x1[i] = x[i];
            const double cost1 = sums[kNSUM - 1];
            const int iter1 = iter, status1 = status;
            moments_start<kW, kBack>(img, npx, nx, c0, x);
            lm_solve<Model, 1>(img, npx, nx, x, sums, PSFR_FIT_TOL2, kEfitMaxIter, iter, status);
            if (!(status > 0 && resolved(x) && (status1 <= 0 || sums[kNSUM - 1] < cost1))) {
#pragma unroll
                for (int i = 0; i < kNP; ++i) x[i] = x1[i];
                iter = iter1;
                status = status1;
                accumulate<Model, 1>(img, npx, nx, x, sums);   // the bits lm_solve left at x1
            }
        }
        if (!resolved(x)) status = -1;       // reported as not converged after iter iterations
        if (lane == 0) {
            write_efit_record<kNP>(x, sums, npu, iter, status, out + (size_t)image * PSFR_EFIT_NPAR);
            if constexpr (kW)
                back_record(back + (size_t)image * PSFR_BACK_NPAR, kBack ? x[kNP - 1] : 0.0,
                            kBack ? efit_err_back(sums, npu) : 0.0, npu);
        }
        __syncwarp();
    }
}

__global__ void __launch_bounds__(kFitWarps * 32, PSFR_EFIT_MINBLOCKS)
efit_kernel(const double* __restrict__ imgs, const double* __restrict__ circ, int nimg, int ny, int nx,
            double* __restrict__ out, int* __restrict__ next_image) {
    efit_images<false, false>(imgs, nullptr, circ, nullptr, nimg, ny, nx, out, nullptr, next_image);
}

// elliptical star fit from the circular star fit's records circ and circ_back (which back may overwrite in place)
template <bool kBack>
__global__ void __launch_bounds__(kFitWarps * 32, PSFR_EFIT_MINBLOCKS)
star_efit_kernel(const double* __restrict__ imgs, const double* __restrict__ wts, const double* __restrict__ circ,
                 const double* circ_back, int nimg, int ny, int nx, double* __restrict__ out, double* back,
                 int* __restrict__ next_image) {
    efit_images<true, kBack>(imgs, wts, circ, circ_back, nimg, ny, nx, out, back, next_image);
}

// ---------------------------------------------------------------- template fit (DESIGN.md 5.8)
// resident CTAs per SM the template fitter is compiled for; shared memory (image, weights and template per warp)
// allows two at 25 x 25 stamps and 40 x 40 templates
#ifndef PSFR_TFIT_MINBLOCKS
#define PSFR_TFIT_MINBLOCKS 2
#endif
constexpr int kTfitMaxIter = 200;   // the circular fit's final-stage cap

// Row stride of the coefficient array in shared memory: tx rounded up to an odd number of doubles, so that the
// prefilter's row pass (one lane per row, all lanes at the same column) hits 32 different 8-byte bank pairs.
__host__ __device__ constexpr int tpl_stride(int tx) { return tx | 1; }

// The warp's template: interpolating cubic B-spline coefficients [ty][tpl_stride(tx)] in shared memory, 1 / S, and
// the stamp's size (the bounds of the centre).
struct TemplateView {
    const double* coef;
    int ty, tx, ny, nx;
    double inv_s;
};

// cubic B-spline weights of the four taps floor(u) - 1 .. floor(u) + 2 at fraction t, and their derivatives in t
__device__ __forceinline__ void bspline3(double t, double* w, double* dw) {
    const double s = 1.0 - t, t2 = t * t, s2 = s * s;
    w[0] = s2 * s * (1.0 / 6.0);
    w[1] = 2.0 / 3.0 - 0.5 * t2 * (2.0 - t);
    w[2] = 2.0 / 3.0 - 0.5 * s2 * (2.0 - s);
    w[3] = t2 * t * (1.0 / 6.0);
    dw[0] = -0.5 * s2;
    dw[1] = t * (1.5 * t - 2.0);
    dw[2] = -s * (1.5 * s - 2.0);
    dw[3] = 0.5 * t2;
}

// tap index k of a line of n samples under mirror boundary conditions (d c b | a b c d | c b a); k in [-1, n + 1]
// (the taps of a point at n - 1 reach n + 1), which n >= 4 keeps inside the line
__device__ __forceinline__ int mirror_tap(int k, int n) { return k < 0 ? -k : k > n - 1 ? 2 * (n - 1) - k : k; }

// Template model m = F s(u, v) / S + c, x = [F, y0, x0(, c)], (u, v) = (row - y0 + ty/2, column - x0 + tx/2): 16 taps of
// the coefficients, no transcendental.  The weights follow the image in shared memory, as StarModel.
template <bool kBack>
struct TemplateModel {
    static constexpr int NP = kBack ? 4 : 3;
    static constexpr bool kWeighted = true;
    TemplateView v;
    double hy, hx, fs, c;   // template centre, F / S, background
    __device__ __forceinline__ TemplateModel(const double* x, const TemplateView& tv)
        : v(tv), hy((double)(tv.ty / 2)), hx((double)(tv.tx / 2)), fs(x[0] * tv.inv_s), c(kBack ? x[3] : 0.0) {}
    // s and its derivatives in u and v; all 0 outside [0, ty - 1] x [0, tx - 1]
    __device__ __forceinline__ double sample(double u, double vv, double& su, double& sv) const {
        su = sv = 0.0;
        if (!(u >= 0.0 && u <= (double)(v.ty - 1) && vv >= 0.0 && vv <= (double)(v.tx - 1))) return 0.0;
        const double fu = floor(u), fv = floor(vv);
        const int iu = (int)fu, iv = (int)fv;
        double wu[4], dwu[4], wv[4], dwv[4];
        bspline3(u - fu, wu, dwu);
        bspline3(vv - fv, wv, dwv);
        int col[4];
#pragma unroll
        for (int l = 0; l < 4; ++l) col[l] = mirror_tap(iv - 1 + l, v.tx);
        double val = 0.0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const double* row = v.coef + mirror_tap(iu - 1 + k, v.ty) * tpl_stride(v.tx);
            double rv = 0.0, rd = 0.0;
#pragma unroll
            for (int l = 0; l < 4; ++l) {
                const double cf = row[col[l]];
                rv = fma(wv[l], cf, rv);
                rd = fma(dwv[l], cf, rd);
            }
            val = fma(wu[k], rv, val);
            su = fma(dwu[k], rv, su);
            sv = fma(wu[k], rd, sv);
        }
        return val;
    }
    // model value at offset (dp, dq) = (row - y0, column - x0)
    __device__ __forceinline__ double value(double dp, double dq) const {
        double su, sv;
        return fma(fs, sample(dp + hy, dq + hx, su, sv), c);
    }
    __device__ __forceinline__ void pixel(double dp, double dq, double pix, double w, double* sums) const {
        double su, sv, J[NP];
        const double s = sample(dp + hy, dq + hx, su, sv);
        J[0] = s * v.inv_s;
        J[1] = -fs * su;
        J[2] = -fs * sv;
        if constexpr (kBack) J[3] = 1.0;
        add_normal_w<NP>(J, fma(fs, s, c) - pix, w, sums);
    }
    static __device__ __forceinline__ bool refuses(const double* xt, const TemplateView& tv) {
        bool bad = !(xt[1] >= -0.5 && xt[1] <= tv.ny - 0.5 && xt[2] >= -0.5 && xt[2] <= tv.nx - 0.5);
#pragma unroll
        for (int i = 0; i < NP; ++i) bad = bad || !isfinite(xt[i]);
        return bad;
    }
};

// scipy's spline_filter1d(order=3, mode='mirror') of one line of n samples at stride st, in place: the gain, then the
// causal recursion from its exact mirror initialisation and the anticausal one, pole z = sqrt(3) - 2
__device__ __forceinline__ void prefilter_line(double* c, int n, int st) {
    const double z = -0.26794919243112270;   // sqrt(3) - 2
    const double gain = (1.0 - z) * (1.0 - 1.0 / z);
    for (int i = 0; i < n; ++i) c[i * st] *= gain;
    const double zn1 = pow(z, (double)(n - 1));
    double c0 = c[0] + zn1 * c[(n - 1) * st], zi = z;
    for (int i = 1; i < n - 1; ++i) {
        c0 += zi * (c[i * st] + zn1 * c[(n - 1 - i) * st]);
        zi *= z;
    }
    c[0] = c0 / (1.0 - zn1 * zn1);
    for (int i = 1; i < n; ++i) c[i * st] += z * c[(i - 1) * st];
    c[(n - 1) * st] = (z * c[(n - 2) * st] + c[(n - 1) * st]) * z / (z * z - 1.0);
    for (int i = n - 2; i >= 0; --i) c[i * st] = z * (c[(i + 1) * st] - c[i * st]);
}

// Template fit of every image, one warp per image, images handed out by a global counter as fit_images.  Shared
// memory per warp: image [npx], weights [npx], template coefficients [ty][tpl_stride(tx)].  Image i (counted from
// `first`, the chunk's offset in the call) uses template (first + i) % ntpl of tpls.  out [nimg][PSFR_TFIT_NPAR];
// model [nimg][ny][nx] or NULL.
template <bool kBack>
__global__ void __launch_bounds__(kFitWarps * 32, PSFR_TFIT_MINBLOCKS)
template_fit_kernel(const double* __restrict__ imgs, const double* __restrict__ wts, int nimg, int ny, int nx,
                    const double* __restrict__ tpls, int ntpl, int ty, int tx, long long first,
                    double* __restrict__ out, double* __restrict__ model, int* __restrict__ next_image) {
    using Model = TemplateModel<kBack>;
    constexpr int kNP = Model::NP, kNSUM = Normal<kNP>::NSUM, COST = Normal<kNP>::COST;
    extern __shared__ double sm[];
    const int npx = ny * nx, ntp = ty * tx, ts = tpl_stride(tx), lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* img = sm + (size_t)warp * (2 * npx + ty * ts);
    double* coef = img + 2 * npx;
#pragma unroll 1
    for (;;) {
        int image = 0;
        if (lane == 0) image = atomicAdd(next_image, 1);
        image = __shfl_sync(0xffffffffu, image, 0);
        if (image >= nimg) return;
        __syncwarp();
        bool bad;
        const int npu = load_star_image(imgs, wts, image, npx, img, bad);
        const double* tsrc = tpls + (size_t)((first + image) % ntpl) * ntp;
        bool tb = false;
        for (int i = lane; i < ntp; i += 32) {
            const double t = tsrc[i];
            tb = tb || !isfinite(t);
            coef[(i / tx) * ts + i % tx] = t;
        }
        bad = bad || __any_sync(0xffffffffu, tb) || npu <= kNP;
        __syncwarp();
        double S = 0.0;                 // every lane, row-major: the same bits in each
        for (int r = 0; r < ty; ++r)
            for (int q = 0; q < tx; ++q) S += coef[r * ts + q];
        bad = bad || !(S > 0.0);
        double* mo = model ? model + (size_t)image * npx : nullptr;
        double x[kNP], sums[kNSUM];
        if (!bad) {
            __syncwarp();
            for (int r = lane; r < ty; r += 32) prefilter_line(coef + r * ts, tx, 1);
            __syncwarp();
            for (int q = lane; q < tx; q += 32) prefilter_line(coef + q, ty, ts);
            __syncwarp();
            const double c0 = kBack ? ring_background(img, ny, nx) : 0.0;
            // start: the used pixel of largest d - c0 (first in row-major order on a tie)
            double bestv = -INFINITY;
            int ib = npx;
            for (int i = lane; i < npx; i += 32)
                if (img[npx + i] > 0.0 && img[i] - c0 > bestv) {
                    bestv = img[i] - c0;
                    ib = i;
                }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double ov = __shfl_xor_sync(0xffffffffu, bestv, o);
                const int oi = __shfl_xor_sync(0xffffffffu, ib, o);
                if (ov > bestv || (ov == bestv && oi < ib)) { bestv = ov; ib = oi; }
            }
            x[0] = 1.0;
            x[1] = ib / nx;
            x[2] = ib % nx;
            if constexpr (kBack) x[3] = 0.0;
            // F0: closed-form linear least-squares flux at that centre
            const TemplateView tv{coef, ty, tx, ny, nx, 1.0 / S};
            {
                const Model m0(x, tv);
                double v2[2] = {0.0, 0.0};
                for (int i = lane; i < npx; i += 32) {
                    const double w = img[npx + i];
                    const double st = m0.value((double)(i / nx) - x[1], (double)(i % nx) - x[2]);   // s / S
                    v2[0] += w * st * (img[i] - c0);
                    v2[1] += w * st * st;
                }
                warp_sum_vec<2>(v2);
                bad = !(v2[1] > 0.0);
                x[0] = v2[0] / v2[1];
                if constexpr (kBack) x[3] = c0;
            }
            if (!bad) {
                int iter = 0, status = -1;
                lm_solve<Model, 1>(img, npx, nx, x, sums, PSFR_FIT_TOL2, kTfitMaxIter, iter, status, tv);
                // QFIT and the model image at the final parameters
                const Model mf(x, tv);
                double ares = 0.0;
                for (int i = lane; i < npx; i += 32) {
                    const double m = mf.value((double)(i / nx) - x[1], (double)(i % nx) - x[2]);
                    if (img[npx + i] > 0.0) ares += fabs(img[i] - m);
                    if (mo) mo[i] = m;
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) ares += __shfl_xor_sync(0xffffffffu, ares, o);
                if (lane == 0) {
                    double* o = out + (size_t)image * PSFR_TFIT_NPAR;
                    o[PSFR_TFIT_FLUX] = x[0];
                    o[PSFR_TFIT_Y0] = x[1];
                    o[PSFR_TFIT_X0] = x[2];
                    o[PSFR_TFIT_CONT] = kBack ? x[kNP - 1] : 0.0;
                    o[PSFR_TFIT_CHISQ] = sums[COST];
                    o[PSFR_TFIT_QFIT] = ares / fabs(x[0]);
                    o[PSFR_TFIT_ITER] =
                        (status > 0) ? (double)status : -(double)(iter > kTfitMaxIter ? kTfitMaxIter : iter);
                    o[PSFR_TFIT_NPIX] = (double)npu;
                    const double dof = (double)(npu - kNP);
                    double L[kNP][kNP], e[4] = {0.0, 0.0, 0.0, 0.0};
                    if (cholesky(sums, 0.0, L)) {
#pragma unroll
                        for (int k = 0; k < kNP; ++k) {
                            double z[kNP];
#pragma unroll
                            for (int i = 0; i < kNP; ++i) z[i] = (i == k) ? 1.0 : 0.0;
                            chol_solve(L, z);
                            e[k] = sqrt(fabs(z[k]) * fabs(sums[COST] / dof));
                        }
                    } else {
                        for (int k = 0; k < kNP; ++k) e[k] = nan("");
                    }
                    o[PSFR_TFIT_ERR_FLUX] = e[0];
                    o[PSFR_TFIT_ERR_Y0] = e[1];
                    o[PSFR_TFIT_ERR_X0] = e[2];
                    o[PSFR_TFIT_ERR_CONT] = e[3];
                }
            }
        }
        if (bad) {
            if (lane == 0) fail_record(out + (size_t)image * PSFR_TFIT_NPAR, PSFR_TFIT_NPAR, PSFR_TFIT_ITER);
            if (mo)
                for (int i = lane; i < npx; i += 32) mo[i] = nan("");
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------- mean of cubes
__global__ void mean_kernel(const double* __restrict__ cubes, int ncube, size_t elems,
                            double* __restrict__ out, int first, int last, int ntotal) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= elems) return;
    // straight sum in input order (np.mean over axis 0 reduces plane by plane), then / ntotal;
    // `first` / `last` let the caller stream the cubes through in slabs with identical rounding
    double t = first ? 0.0 : out[i];
    for (int k = 0; k < ncube; ++k) t += cubes[(size_t)k * elems + i];
    out[i] = last ? t / ntotal : t;
}

// Time mean of consecutive exposures (psfr_compute_groups).  One thread per element walks the draws of
// the chunk in order and keeps one unnormalised sum, started from 0.0 or from the carried sum: the
// additions and the final division are those mean_kernel makes on the same cubes, so every exposure's
// mean is bit-identical to psfr_mean_refit over its cubes wherever the chunk edges fall.
__global__ void group_mean_kernel(const double* __restrict__ cubes, size_t elems, const int* __restrict__ seg,
                                  int nseg, int carry_in, double* __restrict__ carry, double* __restrict__ out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= elems) return;
    double t = carry_in ? carry[i] : 0.0;
    int k = 0, done = 0;
    for (int g = 0; g < nseg; ++g) {
        const int end = seg[2 * g], n = seg[2 * g + 1];
        for (; k < end; ++k) t += cubes[(size_t)k * elems + i];
        if (n) {
            out[(size_t)done++ * elems + i] = t / n;
            t = 0.0;
        } else {
            carry[i] = t;      // only the last exposure of a chunk can stay open
        }
    }
}

// ---------------------------------------------------------------- polynomial smoothing
// least squares via Householder QR of the shared Vandermonde matrix (columns x^deg .. x^0,
// as np.polyfit); one thread per series applies Q^T and back-substitutes.
constexpr int kMaxLam = 256, kMaxDeg = 8;
__global__ void polyfit_kernel(const double* __restrict__ lb, int nlam, int deg, int nseries,
                               const double* __restrict__ y, double* __restrict__ coef) {
    __shared__ double V[kMaxLam * (kMaxDeg + 1)];   // column-major, overwritten by R / reflectors
    __shared__ double beta[kMaxDeg + 1], rdiag[kMaxDeg + 1];
    const int nc = deg + 1;
    for (int idx = threadIdx.x; idx < nlam * nc; idx += blockDim.x) {
        const int c = idx / nlam, r = idx % nlam;
        V[c * nlam + r] = pow(lb[r], (double)(deg - c));
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int c = 0; c < nc; ++c) {
            double nrm = 0.0;
            for (int r = c; r < nlam; ++r) nrm += V[c * nlam + r] * V[c * nlam + r];
            nrm = sqrt(nrm);
            const double alpha = V[c * nlam + c] > 0 ? -nrm : nrm;
            V[c * nlam + c] -= alpha;                    // v = x - alpha e1
            double vv = 0.0;
            for (int r = c; r < nlam; ++r) vv += V[c * nlam + r] * V[c * nlam + r];
            beta[c] = vv > 0 ? 2.0 / vv : 0.0;
            rdiag[c] = alpha;
            for (int c2 = c + 1; c2 < nc; ++c2) {
                double dot = 0.0;
                for (int r = c; r < nlam; ++r) dot += V[c * nlam + r] * V[c2 * nlam + r];
                dot *= beta[c];
                for (int r = c; r < nlam; ++r) V[c2 * nlam + r] -= dot * V[c * nlam + r];
            }
        }
    }
    __syncthreads();
    for (int sidx = threadIdx.x; sidx < nseries; sidx += blockDim.x) {
        double w[kMaxLam];
        for (int r = 0; r < nlam; ++r) w[r] = y[(size_t)sidx * nlam + r];
        for (int c = 0; c < nc; ++c) {
            double dot = 0.0;
            for (int r = c; r < nlam; ++r) dot += V[c * nlam + r] * w[r];
            dot *= beta[c];
            for (int r = c; r < nlam; ++r) w[r] -= dot * V[c * nlam + r];
        }
        double cf[kMaxDeg + 1];
        for (int c = nc - 1; c >= 0; --c) {
            double t = w[c];
            for (int c2 = c + 1; c2 < nc; ++c2) t -= V[c2 * nlam + c] * cf[c2];
            cf[c] = t / rdiag[c];
        }
        for (int c = 0; c < nc; ++c) coef[(size_t)sidx * nc + c] = cf[c];
    }
}

// ---------------------------------------------------------------- drivers
int run_build_kernels(Ctx* c, int ndraw, int nlam, const double* lambda_nm_host, bool tt, bool mu,
                      cudaStream_t s) {
    if (mu && (int)c->lam_kernels.size() == nlam &&
        std::equal(lambda_nm_host, lambda_nm_host + nlam, c->lam_kernels.begin()))
        mu = false;   // the MUSE kernels of these wavelengths and their spectra are already on the device
    std::vector<double> gb(mu ? 2 * nlam : 0);   // gamma[nlam], beta[nlam]
    for (int l = 0; mu && l < nlam; ++l) {
        // muse_intrinsic_psf (psfrec.py:1160-1168, np.polyval = Horner) and alpha = fwhm/0.2/(2 sqrt(2^(1/beta)-1)) (:923-924)
        static const double pol_beta[6] = {-0.83704697, 1.1337153, 0.0609222, -1.35581762, 1.15237178, 2.2106042};
        static const double pol_fwhm[6] = {0.60467385, -1.58905792, 1.75293264, -1.0368302, 0.21487023, 0.34851139};
        const double lb = (10 * lambda_nm_host[l] - 4750) / (9350 - 4750);
        double fw = 0.0, be = 0.0;
        for (int k = 0; k < 6; ++k) {
            fw = fw * lb + pol_fwhm[k];
            be = be * lb + pol_beta[k];
        }
        fw = fw / 0.2;
        const double g = fw / (2 * sqrt(pow(2.0, 1. / be) - 1));
        // the kernel's domain: beta <= 0 (lambda >~ 1189 nm) makes gamma NaN or 0, beta == 1 zeroes the amplitude,
        // fwhm == 0 (~303.85 nm) zeroes gamma; each would give a 0/0 kernel
        if (!(be > 0) || be == 1.0 || !moffat_width_ok(g))
            return set_error(c, PSFR_E_UNSUPPORTED,
                             "wavelength %g nm: the MUSE Moffat has beta = %g, gamma = %g px; the kernel needs beta > 0, "
                             "beta != 1 and pi gamma^2 finite and normal", lambda_nm_host[l], be, g);
        gb[l] = g;
        gb[nlam + l] = be;
    }
    if (tt) {
        // gamma = alpha_tt per draw (slot PSFR_DRAW_ALPHA_TT), Moffat power 2
        double* two = c->d_misc + kMiscTwo;   // holds the constant 2.0
        const double h2 = 2.0;
        PSFR_CUDA(c, cudaMemcpyAsync(two, &h2, sizeof(double), cudaMemcpyHostToDevice, s));
        moffat_kernels_kernel<<<ndraw, 256, 0, s>>>(c->d_misc + misc_alpha_tt(c->max_planes), two, 0, c->d_kern_tt);
        PSFR_LAUNCH_CHECK(c);
        int rc = run_kernel_spectra(c, ndraw, c->d_kern_tt, c->d_khat_tt, s);
        if (rc) return rc;
    }
    if (mu) {
        c->lam_kernels.clear();
        double* h = static_cast<double*>(c->h_pinned);
        std::copy(gb.begin(), gb.end(), h);
        double* d = c->d_misc + kMiscMuse;    // gamma[nlam], beta[nlam]
        PSFR_CUDA(c, cudaMemcpyAsync(d, h, 2 * nlam * sizeof(double), cudaMemcpyHostToDevice, s));
        PSFR_CUDA(c, cudaStreamSynchronize(s));   // pinned bounce buffer is reused by the caller
        moffat_kernels_kernel<<<nlam, 256, 0, s>>>(d, d + nlam, 1, c->d_kern_mu);
        PSFR_LAUNCH_CHECK(c);
        int rc = run_kernel_spectra(c, nlam, c->d_kern_mu, c->d_khat_mu, s);
        if (rc) return rc;
        c->lam_kernels.assign(lambda_nm_host, lambda_nm_host + nlam);
    }
    return PSFR_OK;
}

int run_resample(Ctx* c, int nimg, int nlam, double* cube_dev, cudaStream_t s) {
    const size_t smem = (size_t)(kNS * kNS + 32) * sizeof(double);
    if (int rc = ensure_dynamic_smem(c, resample_kernel, smem)) return rc;
    resample_kernel<<<nimg, 256, smem, s>>>(c->d_samp, c->d_frac, nlam, cube_dev);
    PSFR_LAUNCH_CHECK(c);
    return PSFR_OK;
}

int run_convolve(Ctx* c, int ndraw, int ndir, int nlam, const double* in_dev, double* out_dev, cudaStream_t s) {
    return run_fft_convolve(c, ndraw, ndir, nlam, in_dev, out_dev, s);
}

int run_fit(Ctx* c, int nimg, int ny, int nx, const double* img_dev, double* fit_dev, cudaStream_t s) {
    const size_t smem = (size_t)kFitWarps * (ny * nx + nx) * sizeof(double);
    if (smem > 200 * 1024) return set_error(c, PSFR_E_UNSUPPORTED, "image %dx%d too large for the fitter", ny, nx);
    // the coarse stage needs more than its two 32-pixel strips of the image (fit_kernel)
    const auto kernel = ny * nx > 2 * 32 * PSFR_FIT_COARSE_STEP ? fit_kernel<true> : fit_kernel<false>;
    if (int rc = ensure_dynamic_smem(c, kernel, smem)) return rc;
    int grid = (nimg + kFitWarps - 1) / kFitWarps;
    int per_sm = 2;                                  // persistent grid: as many CTAs as are resident at once
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kFitWarps * 32, smem) != cudaSuccess ||
        per_sm < 1) {
        cudaGetLastError();
        per_sm = 2;
    }
    const int resident = c->sm_count * per_sm;
    if (grid > resident) grid = resident;
    PSFR_CUDA(c, cudaMemsetAsync(c->d_counter + 1, 0, sizeof(int), s));
    kernel<<<grid, kFitWarps * 32, smem, s>>>(img_dev, nimg, ny, nx, fit_dev, c->d_counter + 1);
    PSFR_LAUNCH_CHECK(c);
    return PSFR_OK;
}

int run_efit(Ctx* c, int nimg, int ny, int nx, const double* img_dev, const double* circ_dev, double* efit_dev,
             cudaStream_t s) {
    const size_t smem = (size_t)kFitWarps * ny * nx * sizeof(double);
    if (smem > 200 * 1024) return set_error(c, PSFR_E_UNSUPPORTED, "image %dx%d too large for the fitter", ny, nx);
    if (int rc = ensure_dynamic_smem(c, efit_kernel, smem)) return rc;
    int grid = (nimg + kFitWarps - 1) / kFitWarps;
    int per_sm = 1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, efit_kernel, kFitWarps * 32, smem) != cudaSuccess ||
        per_sm < 1) {
        cudaGetLastError();
        per_sm = 1;
    }
    const int resident = c->sm_count * per_sm;
    if (grid > resident) grid = resident;
    PSFR_CUDA(c, cudaMemsetAsync(c->d_counter + 2, 0, sizeof(int), s));
    efit_kernel<<<grid, kFitWarps * 32, smem, s>>>(img_dev, circ_dev, nimg, ny, nx, efit_dev, c->d_counter + 2);
    PSFR_LAUNCH_CHECK(c);
    return PSFR_OK;
}

// Shared memory of the star fits (the image and its weights per warp), or 0 when a stamp is over the fitter's
// 200 KiB: the circular fit always runs, the elliptical one after it.
static size_t star_fit_smem(int ny, int nx, bool elliptical) {
    const size_t npx = (size_t)ny * nx, circ = kFitWarps * (2 * npx + nx) * sizeof(double);
    const size_t ell = kFitWarps * 2 * npx * sizeof(double);
    const size_t lim = 200 * 1024;
    return circ > lim || (elliptical && ell > lim) ? 0 : circ;
}

int check_star_fit_size(Ctx* c, int ny, int nx, bool elliptical) {
    if (!star_fit_smem(ny, nx, elliptical))
        return set_error(c, PSFR_E_UNSUPPORTED,
                         "image %dx%d too large for the star fit: its image and weights need %zu bytes of shared memory "
                         "per CTA, over 200 KiB", ny, nx,
                         (size_t)kFitWarps * (2 * (size_t)ny * nx + (elliptical ? 0 : nx)) * sizeof(double));
    return PSFR_OK;
}

// persistent grid of a fit kernel: as many CTAs as are resident at once, at most one warp per image
template <class K>
static int fit_grid(Ctx* c, K* kernel, size_t smem, int nimg, int per_sm_default) {
    int grid = (nimg + kFitWarps - 1) / kFitWarps;
    int per_sm = per_sm_default;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kFitWarps * 32, smem) != cudaSuccess ||
        per_sm < 1) {
        cudaGetLastError();
        per_sm = per_sm_default;
    }
    return std::min(grid, c->sm_count * per_sm);
}

int run_star_fit(Ctx* c, int nimg, int ny, int nx, const double* img_dev, const double* w_dev, bool fit_back,
                 double* fit_dev, double* back_dev, cudaStream_t s) {
    if (int rc = check_star_fit_size(c, ny, nx, false)) return rc;
    const size_t smem = star_fit_smem(ny, nx, false);
    const bool coarse = ny * nx > 2 * 32 * PSFR_FIT_COARSE_STEP;   // as run_fit
    const auto kernel = coarse ? (fit_back ? star_fit_kernel<true, true> : star_fit_kernel<true, false>)
                               : (fit_back ? star_fit_kernel<false, true> : star_fit_kernel<false, false>);
    if (int rc = ensure_dynamic_smem(c, kernel, smem)) return rc;
    const int grid = fit_grid(c, kernel, smem, nimg, 2);
    PSFR_CUDA(c, cudaMemsetAsync(c->d_counter + 1, 0, sizeof(int), s));
    kernel<<<grid, kFitWarps * 32, smem, s>>>(img_dev, w_dev, nimg, ny, nx, fit_dev, back_dev, c->d_counter + 1);
    PSFR_LAUNCH_CHECK(c);
    return PSFR_OK;
}

int run_star_efit(Ctx* c, int nimg, int ny, int nx, const double* img_dev, const double* w_dev, bool fit_back,
                  const double* circ_dev, const double* circ_back_dev, double* efit_dev, double* back_dev,
                  cudaStream_t s) {
    if (int rc = check_star_fit_size(c, ny, nx, true)) return rc;
    const size_t smem = (size_t)kFitWarps * 2 * ny * nx * sizeof(double);
    const auto kernel = fit_back ? star_efit_kernel<true> : star_efit_kernel<false>;
    if (int rc = ensure_dynamic_smem(c, kernel, smem)) return rc;
    const int grid = fit_grid(c, kernel, smem, nimg, 1);
    PSFR_CUDA(c, cudaMemsetAsync(c->d_counter + 2, 0, sizeof(int), s));
    kernel<<<grid, kFitWarps * 32, smem, s>>>(img_dev, w_dev, circ_dev, circ_back_dev, nimg, ny, nx, efit_dev,
                                              back_dev, c->d_counter + 2);
    PSFR_LAUNCH_CHECK(c);
    return PSFR_OK;
}

// shared memory of the template fit (image, weights and template per warp), or 0 when it is over 200 KiB
static size_t template_fit_smem(int ny, int nx, int ty, int tx) {
    const size_t b = (size_t)kFitWarps * (2 * (size_t)ny * nx + (size_t)ty * tpl_stride(tx)) * sizeof(double);
    return b > 200 * 1024 ? 0 : b;
}

int check_template_fit_size(Ctx* c, int ny, int nx, int ty, int tx) {
    if (!template_fit_smem(ny, nx, ty, tx))
        return set_error(c, PSFR_E_UNSUPPORTED,
                         "image %dx%d with a %dx%d template too large for the template fit: image, weights and "
                         "template need %zu bytes of shared memory per CTA, over 200 KiB", ny, nx, ty, tx,
                         (size_t)kFitWarps * (2 * (size_t)ny * nx + (size_t)ty * tpl_stride(tx)) * sizeof(double));
    return PSFR_OK;
}

int run_template_fit(Ctx* c, int nimg, int ny, int nx, const double* img_dev, const double* w_dev, int ntpl, int ty,
                     int tx, const double* tpl_dev, long long first, bool fit_back, double* fit_dev, double* model_dev,
                     cudaStream_t s) {
    if (int rc = check_template_fit_size(c, ny, nx, ty, tx)) return rc;
    const size_t smem = template_fit_smem(ny, nx, ty, tx);
    const auto kernel = fit_back ? template_fit_kernel<true> : template_fit_kernel<false>;
    if (int rc = ensure_dynamic_smem(c, kernel, smem)) return rc;
    const int grid = fit_grid(c, kernel, smem, nimg, 1);
    PSFR_CUDA(c, cudaMemsetAsync(c->d_counter + 4, 0, sizeof(int), s));
    kernel<<<grid, kFitWarps * 32, smem, s>>>(img_dev, w_dev, nimg, ny, nx, tpl_dev, ntpl, ty, tx, first, fit_dev,
                                              model_dev, c->d_counter + 4);
    PSFR_LAUNCH_CHECK(c);
    return PSFR_OK;
}

int run_mean(Ctx* c, int ncube, int plane_elems, const double* cubes_dev, double* out_dev, cudaStream_t s,
             bool first, bool last, int ntotal) {
    mean_kernel<<<(plane_elems + 255) / 256, 256, 0, s>>>(cubes_dev, ncube, (size_t)plane_elems, out_dev,
                                                          first ? 1 : 0, last ? 1 : 0, ntotal);
    PSFR_LAUNCH_CHECK(c);
    return PSFR_OK;
}

int run_group_mean(Ctx* c, int plane_elems, const double* cubes_dev, const int* seg_dev, int nseg,
                   bool carry_in, double* out_dev, cudaStream_t s) {
    group_mean_kernel<<<(plane_elems + 255) / 256, 256, 0, s>>>(cubes_dev, (size_t)plane_elems, seg_dev, nseg,
                                                                carry_in ? 1 : 0, c->d_carry, out_dev);
    PSFR_LAUNCH_CHECK(c);
    return PSFR_OK;
}

int run_polyfit(Ctx* c, int nseries, int nlam, int deg, const double* lb_dev, const double* y_dev,
                double* coef_dev, cudaStream_t s) {
    if (nlam > kMaxLam || deg > kMaxDeg || deg + 1 > nlam)
        return set_error(c, PSFR_E_UNSUPPORTED, "polyfit limits: nlam <= %d, deg <= %d", kMaxLam, kMaxDeg);
    polyfit_kernel<<<1, 128, 0, s>>>(lb_dev, nlam, deg, nseries, y_dev, coef_dev);
    PSFR_LAUNCH_CHECK(c);
    return PSFR_OK;
}

}  // namespace psfr
