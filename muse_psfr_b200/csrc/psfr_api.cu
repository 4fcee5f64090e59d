// C-ABI entry points of libpsfr_b200.so (see include/psfr.h for the contract).
#include <cmath>
#include <cstdarg>
#include <cstring>
#include <vector>
#include "psfr_internal.h"
#include <algorithm>
#include "warp_fft.cuh"
#include "fft_tables.h"

struct psfr_ctx : psfr::Ctx {};

namespace psfr {

static char g_create_error[512] = "";

int set_error(Ctx* c, int code, const char* fmt, ...) {
    char* dst = c ? c->err : g_create_error;
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(dst, 512, fmt, ap);
    va_end(ap);
    return code;
}

static bool is_device_ptr(const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

// copy `bytes` from src (host or device) into device memory dst
static int to_device(Ctx* c, void* dst, const void* src, size_t bytes, cudaStream_t s) {
    PSFR_CUDA(c, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, s));
    return PSFR_OK;
}
// copy device memory to dst (host or device); host destinations are complete on return
static int from_device(Ctx* c, void* dst, const void* src, size_t bytes, cudaStream_t s) {
    PSFR_CUDA(c, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, s));
    if (!is_device_ptr(dst)) PSFR_CUDA(c, cudaStreamSynchronize(s));
    return PSFR_OK;
}

template <class T>
static int dev_alloc(Ctx* c, T** p, size_t count) {
    PSFR_CUDA(c, cudaMalloc(reinterpret_cast<void**>(p), count * sizeof(T)));
    return PSFR_OK;
}

// Pass-3 records and pass-2 row masks of the group row kernel (psfr_hot2.cu) for one wavelength: thread
// pair (2q, 2q+1) gets a kept frequency k and its mirror.  A thread reads buf[base + kGS2 n3], n3 = 0..7,
// i.e. 16-byte slot (slot0 + kGS2 n3) mod 8 with slot0 = (k1 + k2) mod 8 (kGS1 = 1 mod 8): the pairs are
// dealt greedily so that the eight threads of a quarter-warp have as few equal slot0 as the frequency set
// allows (measured: 1.6 wavefronts per quarter-warp load instead of 1; reading every row from its own
// rotated start would make it exactly 1, but the extra selects made the kernel slower, DESIGN.md 3.11).
static void group_p3_table(const uint16_t* kc, int N, GroupP3* out, uint32_t* mask) {
    // rows and Horner bases belong to the 1280-point (sub-)transform: output k mod 1280
    auto k1_of = [](int k) { return (k % kNB) % kG1; };
    auto k2_of = [](int k) { return ((k % kNB) / kG1) % kG2; };
    auto slot0 = [&](int k) { return (k1_of(k) + k2_of(k)) & 7; };
    bool used[kNC] = {false};
    for (int k1 = 0; k1 < kGMaskStride; ++k1) mask[k1] = 0;
    int q = 0;
    for (int g = 0; g < kNC / 4; ++g) {          // quarter-warps of four pairs
        int cnt[8] = {0};
        for (int i = 0; i < 4; ++i, ++q) {
            int best = -1, best_cost = 1 << 30;
            for (int j = 0; j < kNC; ++j) {
                if (used[j]) continue;
                const int k = kc[j], km = (N - k) % N;
                const int a = slot0(k), b = slot0(km);
                const int cost = cnt[a] + cnt[b] + (a == b && k != km ? 1 : 0);
                if (cost < best_cost) {
                    best_cost = cost;
                    best = j;
                }
            }
            used[best] = true;
            for (int sgn = 0; sgn < 2; ++sgn) {
                const int k = sgn ? (N - kc[best]) % N : kc[best];
                ++cnt[slot0(k)];
                GroupP3& e = out[2 * q + sgn];
                e.w = unit_root(k % kNB, kNB);
                e.wc = unit_root(k, N);
                e.w32 = make_float2((float)e.w.x, (float)e.w.y);
                e.base = (uint32_t)(k1_of(k) * kGS1 + k2_of(k));
                e.col = (uint32_t)best;
                mask[k1_of(k)] |= 1u << k2_of(k);
            }
        }
    }
}

// wavelength tables: exponent scale, sampled indices, bilinear fractions (psfrec.py:663-664, 682-683)
static int set_lambda_tables(Ctx* c, int nlam, const double* lam_host, cudaStream_t s) {
    if (nlam < 1 || nlam > c->max_lambda)
        return set_error(c, PSFR_E_CAPACITY, "nlam=%d outside [1, %d]", nlam, c->max_lambda);
    if ((int)c->lam_tables.size() == nlam && std::equal(lam_host, lam_host + nlam, c->lam_tables.begin()))
        return PSFR_OK;   // the tables of these wavelengths are already on the device
    c->lam_tables.clear();
    const int kN = c->N;
    std::vector<double> cl(nlam), fr((size_t)nlam * kPSF);
    std::vector<uint16_t> kx((size_t)nlam * kNS);
    std::vector<double2> ws(c->NF == 2 ? (size_t)nlam * 2 * kNS : 0);
    for (int l = 0; l < nlam; ++l) {
        const double lb = lam_host[l];
        if (!(lb > 0)) return set_error(c, PSFR_E_ARG, "wavelength %g nm is not positive", lb);
        const double conv = 2 * 3.141592653589793 / lb;        // convnm, psfrec.py:717 (lbda*1e9 = nm)
        cl[l] = 0.5 * (conv * conv);
        const long npix = (long)(std::nearbyint(((kPSF * 0.2 * 2 * 8 * 4.85 * 1000) / lb) / 2) * 2);
        if (npix > kN)
            return set_error(c, PSFR_E_UNSUPPORTED,
                             "wavelength %g nm needs a %ld-pixel crop but dim is %d (reference: psf_muse fails)",
                             lb, npix, kN);
        if (npix < kNS)   // two distinct samples per output pixel and axis: crops of at least 80 pixels
            return set_error(c, PSFR_E_UNSUPPORTED,
                             "wavelength %g nm needs a %ld-pixel crop, fewer than the %d samples per axis this "
                             "library resamples from", lb, npix, kNS);
        const long origin = kN / 2 - npix / 2;
        for (int y = 0; y < kPSF; ++y) {
            const double pos = (double)(y * npix) / kPSF;
            const long r0 = (long)std::floor(pos);
            fr[(size_t)l * kPSF + y] = pos - (double)r0;
            kx[(size_t)l * kNS + 2 * y] = (uint16_t)((origin + r0 + kN / 2) % kN);
            kx[(size_t)l * kNS + 2 * y + 1] = (uint16_t)((origin + r0 + 1 + kN / 2) % kN);
        }
        if (c->NF == 2)
            for (int j = 0; j < kNS; ++j) {
                const long k = kx[(size_t)l * kNS + j];
                ws[((size_t)l * 2) * kNS + j] = unit_root(k, kN);
                ws[((size_t)l * 2 + 1) * kNS + j] = unit_root((kN - k) % kN, kN);
            }
    }
    if (c->NF == 2)
        PSFR_CUDA(c, cudaMemcpyAsync(c->d_wsamp, ws.data(), ws.size() * sizeof(double2), cudaMemcpyHostToDevice, s));
    // the row kernel classifies the units of a row pair by c_lambda * min(D): sorted copy + permutation
    std::vector<int> order(nlam);
    for (int l = 0; l < nlam; ++l) order[l] = l;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return cl[a] > cl[b]; });
    std::vector<double> csort(nlam);
    for (int l = 0; l < nlam; ++l) csort[l] = cl[order[l]];
    PSFR_CUDA(c, cudaMemcpyAsync(c->d_csort, csort.data(), nlam * sizeof(double), cudaMemcpyHostToDevice, s));
    PSFR_CUDA(c, cudaMemcpyAsync(c->d_lorder, order.data(), nlam * sizeof(int), cudaMemcpyHostToDevice, s));
    PSFR_CUDA(c, cudaMemcpyAsync(c->d_lam, cl.data(), nlam * sizeof(double), cudaMemcpyHostToDevice, s));
    PSFR_CUDA(c, cudaMemcpyAsync(c->d_frac, fr.data(), fr.size() * sizeof(double), cudaMemcpyHostToDevice, s));
    PSFR_CUDA(c, cudaMemcpyAsync(c->d_kidx, kx.data(), kx.size() * sizeof(uint16_t), cudaMemcpyHostToDevice, s));
    // Row-pass frequencies kept between the passes: the samples of the first 20 output pixels (k <= 0);
    // sample 1 (k = -npix/2 + 1) has weight exactly 0 (frac[0] = 0) and gives its slot to k = 0, the live
    // sample of pixel 20.  xmap: which sample index holds +k / -k of each kept frequency.
    std::vector<uint16_t> kc((size_t)nlam * kNC);
    std::vector<short2> xm((size_t)nlam * kNC);
    std::vector<ushort2> ka((size_t)nlam * kNC);
    std::vector<double2> wc(c->NF == 2 ? (size_t)nlam * 2 * kNC : 0);
    for (int l = 0; l < nlam; ++l) {
        const uint16_t* kxl = kx.data() + (size_t)l * kNS;
        bool live[kNS], covered[kNS];
        for (int y = 0; y < kPSF; ++y) {
            live[2 * y] = true;
            live[2 * y + 1] = fr[(size_t)l * kPSF + y] != 0.0;
        }
        for (int x = 0; x < kNS; ++x) covered[x] = false;
        for (int j = 0; j < kNC; ++j) {
            const int k = (j == 1) ? 0 : kxl[j], km = (kN - k) % kN;
            kc[(size_t)l * kNC + j] = (uint16_t)k;
            int xd = -1, xf = -1;
            for (int x = 0; x < kNS; ++x) {
                if (!live[x]) continue;
                if (kxl[x] == k && xd < 0) xd = x;
                if (kxl[x] == km && xf < 0) xf = x;
            }
            if (xf == xd) xf = -1;
            if (xd >= 0) covered[xd] = true;
            if (xf >= 0) covered[xf] = true;
            xm[(size_t)l * kNC + j] = make_short2((short)xd, (short)xf);
            // where the row kernel finds X[k] and X[-k] in its natural-order dump (per 1280-point sub-transform)
            ka[(size_t)l * kNC + j] = make_ushort2((unsigned short)nat_addr(k % kNB), (unsigned short)nat_addr(km % kNB));
            if (c->NF == 2) {
                wc[((size_t)l * 2) * kNC + j] = unit_root(k, kN);
                wc[((size_t)l * 2 + 1) * kNC + j] = unit_root(km, kN);
            }
        }
        for (int x = 0; x < kNS; ++x)
            if (live[x] && !covered[x])
                return set_error(c, PSFR_E_UNSUPPORTED, "wavelength %g nm: sample %d (k = %d) has no mirror among the kept "
                                 "frequencies", lam_host[l], x, (int)kxl[x]);
    }
    std::vector<GroupP3> p3;
    std::vector<uint32_t> p2m;
    if (c->d_p3) {
        p3.resize((size_t)nlam * 2 * kNC);
        p2m.resize((size_t)nlam * kGMaskStride);
        for (int l = 0; l < nlam; ++l)
            group_p3_table(kc.data() + (size_t)l * kNC, kN, p3.data() + (size_t)l * 2 * kNC, p2m.data() + (size_t)l * kGMaskStride);
        PSFR_CUDA(c, cudaMemcpyAsync(c->d_p3, p3.data(), p3.size() * sizeof(GroupP3), cudaMemcpyHostToDevice, s));
        PSFR_CUDA(c, cudaMemcpyAsync(c->d_p2mask, p2m.data(), p2m.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, s));
    }
    PSFR_CUDA(c, cudaMemcpyAsync(c->d_kcol, kc.data(), kc.size() * sizeof(uint16_t), cudaMemcpyHostToDevice, s));
    PSFR_CUDA(c, cudaMemcpyAsync(c->d_xmap, xm.data(), xm.size() * sizeof(short2), cudaMemcpyHostToDevice, s));
    PSFR_CUDA(c, cudaMemcpyAsync(c->d_kaddr, ka.data(), ka.size() * sizeof(ushort2), cudaMemcpyHostToDevice, s));
    if (c->NF == 2)
        PSFR_CUDA(c, cudaMemcpyAsync(c->d_wcol, wc.data(), wc.size() * sizeof(double2), cudaMemcpyHostToDevice, s));
    PSFR_CUDA(c, cudaStreamSynchronize(s));   // the host vectors go out of scope
    c->lam_tables.assign(lam_host, lam_host + nlam);
    return PSFR_OK;
}

// fetch a small host copy of an array that may live on either side
static int small_to_host(Ctx* c, std::vector<double>& dst, const double* src, size_t n, cudaStream_t s) {
    dst.resize(n);
    if (is_device_ptr(src)) {
        PSFR_CUDA(c, cudaMemcpyAsync(dst.data(), src, n * sizeof(double), cudaMemcpyDeviceToHost, s));
        PSFR_CUDA(c, cudaStreamSynchronize(s));
    } else {
        memcpy(dst.data(), src, n * sizeof(double));
    }
    return PSFR_OK;
}

// The tip-tilt Moffat width of every draw: alpha > 0 with pi alpha^2 a finite, normal double.  Outside, the
// kernel is 0/0: alpha = 0 (GL = 1 in tiptilt_alpha) or alpha^2 underflowing to 0 leaves its centre 0/0, pi alpha^2
// = inf its amplitude 0, and NaN (GL > 1) propagates.
static int check_alpha_tt(Ctx* c, int ndraw, const double* alpha, size_t stride) {
    for (int d = 0; d < ndraw; ++d) {
        const double a = alpha[(size_t)d * stride];
        if (!(a > 0 && moffat_width_ok(a)))
            return set_error(c, PSFR_E_ARG, "draw %d has tip-tilt alpha %g px; the kernel needs alpha > 0 with "
                             "pi alpha^2 finite and normal", d, a);
    }
    return PSFR_OK;
}

// geometry of a call: directions and guide-star positions [2][npos]; validates the whole draw list once
// (the host keeps the reference's ValueError for > 2 layers without explicit wind directions).  ngs: guide
// stars of every draw, or 0 when each draw gives its own count in slot PSFR_DRAW_NGS.  One host sync at most;
// h receives the host copy of the draw records.
static int upload_geometry(Ctx* c, int ndraw, const double* draws, int ndir, const double* dirs, int ngs,
                           int npos, const double* pos, std::vector<double>& h, cudaStream_t s) {
    if (ndraw < 1 || ndir < 1) return set_error(c, PSFR_E_ARG, "ndraw=%d ndir=%d", ndraw, ndir);
    if (ngs < 0 || ngs > kMaxGS) return set_error(c, PSFR_E_ARG, "ngs=%d outside [1,%d]", ngs, kMaxGS);
    if (npos < 1 || npos > kMaxGS) return set_error(c, PSFR_E_ARG, "npos=%d outside [1,%d]", npos, kMaxGS);
    if (ndir > kMaxDir) return set_error(c, PSFR_E_ARG, "ndir=%d exceeds %d", ndir, kMaxDir);
    if (!c->geometry_set) return set_error(c, PSFR_E_STATE, "psfr_set_geometry has not been called");
    int rc = to_device(c, c->d_misc + kMiscDirs, dirs, (size_t)2 * ndir * sizeof(double), s);
    if (rc) return rc;
    rc = to_device(c, c->d_misc + kMiscPos, pos, (size_t)2 * npos * sizeof(double), s);
    if (rc) return rc;
    rc = small_to_host(c, h, draws, (size_t)ndraw * PSFR_DRAW_NPAR, s);
    if (rc) return rc;
    for (int d = 0; d < ndraw; ++d) {
        const double nl = h[(size_t)d * PSFR_DRAW_NPAR + PSFR_DRAW_NLAYERS];
        if (!(nl >= 1.0 && nl <= (double)PSFR_MAX_LAYERS && nl == std::floor(nl)))
            return set_error(c, PSFR_E_UNSUPPORTED, "draw %d has %g layers; 1 to %d are supported", d, nl, PSFR_MAX_LAYERS);
        const double ng = h[(size_t)d * PSFR_DRAW_NPAR + PSFR_DRAW_NGS];
        if (!ngs && !(ng >= 1.0 && ng <= (double)npos && ng == std::floor(ng)))
            return set_error(c, PSFR_E_ARG, "draw %d has %g guide stars; 1 to npos = %d are supported", d, ng, npos);
    }
    return PSFR_OK;
}

// records of one chunk of draws -> d_draws, their tip-tilt alphas -> scratch; stream-ordered, no sync
static int upload_draws(Ctx* c, int ndraw, const double* draws, int ndir, cudaStream_t s) {
    if (ndraw < 1 || ndraw * ndir > c->max_planes)
        return set_error(c, PSFR_E_CAPACITY, "ndraw*ndir = %d exceeds max_planes = %d", ndraw * ndir, c->max_planes);
    PSFR_CUDA(c, cudaMemcpyAsync(c->d_draws, draws, (size_t)ndraw * PSFR_DRAW_NPAR * sizeof(double),
                                 cudaMemcpyDefault, s));
    PSFR_CUDA(c, cudaMemcpy2DAsync(c->d_misc + misc_alpha_tt(c->max_planes), sizeof(double),
                                   c->d_draws + PSFR_DRAW_ALPHA_TT, PSFR_DRAW_NPAR * sizeof(double),
                                   sizeof(double), ndraw, cudaMemcpyDeviceToDevice, s));
    return PSFR_OK;
}

// Radii and fractions of an encircled-energy call: checked on the host (either side's arrays), then radii followed
// by fractions to d_eepar, stream-ordered before the kernels that read them.
static int upload_ee_params(Ctx* c, int nrad, const double* radii, int nfrac, const double* fracs, cudaStream_t s) {
    if (nrad < 0 || nrad > PSFR_EE_MAX_RADII)
        return set_error(c, PSFR_E_ARG, "nrad=%d outside [0, %d]", nrad, PSFR_EE_MAX_RADII);
    if (nfrac < 0 || nfrac > PSFR_EE_MAX_FRACTIONS)
        return set_error(c, PSFR_E_ARG, "nfrac=%d outside [0, %d]", nfrac, PSFR_EE_MAX_FRACTIONS);
    if ((nrad && !radii) || (nfrac && !fracs)) return set_error(c, PSFR_E_ARG, "NULL radii or fractions");
    std::vector<double> r, f;
    int rc = small_to_host(c, r, radii, (size_t)nrad, s);
    if (!rc) rc = small_to_host(c, f, fracs, (size_t)nfrac, s);
    if (rc) return rc;
    for (int k = 0; k < nrad; ++k)
        if (!(std::isfinite(r[k]) && r[k] >= 0.0))
            return set_error(c, PSFR_E_ARG, "radius %d is %g: radii must be finite and >= 0", k, r[k]);
    for (int j = 0; j < nfrac; ++j)
        if (!(f[j] > 0.0 && f[j] < 1.0))
            return set_error(c, PSFR_E_ARG, "fraction %d is %g: fractions must lie in (0, 1)", j, f[j]);
    c->ee_par = r;
    c->ee_par.insert(c->ee_par.end(), f.begin(), f.end());
    if (!c->ee_par.empty())
        PSFR_CUDA(c, cudaMemcpyAsync(c->d_eepar, c->ee_par.data(), c->ee_par.size() * sizeof(double),
                                     cudaMemcpyHostToDevice, s));
    return PSFR_OK;
}

// Band weights of a call [nband][nlam] (either side): checked on the host, their ascending-k sums to `sums`, and the
// k-major zero-padded copy band_kernel reads to c->band_w, then to d_bandw (allocated on first use), stream-ordered.
static int upload_band_weights(Ctx* c, int nband, int nlam, const double* weights, BandSums& sums, cudaStream_t s) {
    if (nband < 1 || nband > PSFR_MAX_BANDS)
        return set_error(c, PSFR_E_ARG, "nband=%d outside [1, %d]", nband, PSFR_MAX_BANDS);
    if (!weights) return set_error(c, PSFR_E_ARG, "NULL band weights");
    if (nlam < 1) return set_error(c, PSFR_E_ARG, "nlam=%d", nlam);
    std::vector<double> h;
    if (int rc = small_to_host(c, h, weights, (size_t)nband * nlam, s)) return rc;
    for (int b = 0; b < PSFR_MAX_BANDS; ++b) sums.w[b] = 1.0;
    for (int b = 0; b < nband; ++b) {
        double W = 0.0;
        for (int k = 0; k < nlam; ++k) {
            const double v = h[(size_t)b * nlam + k];
            if (!(std::isfinite(v) && v >= 0.0))
                return set_error(c, PSFR_E_ARG, "band %d: weight %d is %g; weights must be finite and >= 0", b, k, v);
            W += v;
        }
        if (!(std::isfinite(W) && W > 0.0))
            return set_error(c, PSFR_E_ARG, "band %d: the weights sum to %g; the sum must be finite and > 0", b, W);
        sums.w[b] = W;
    }
    if (nlam > c->max_lambda) return set_error(c, PSFR_E_CAPACITY, "nlam=%d exceeds max_lambda=%d", nlam, c->max_lambda);
    if (!c->d_bandw) {
        int rc = dev_alloc(c, &c->d_bandw, (size_t)c->max_lambda * PSFR_MAX_BANDS);
        if (rc) return rc;
    }
    c->band_w.assign((size_t)nlam * PSFR_MAX_BANDS, 0.0);
    for (int b = 0; b < nband; ++b)
        for (int k = 0; k < nlam; ++k) c->band_w[(size_t)k * PSFR_MAX_BANDS + b] = h[(size_t)b * nlam + k];
    PSFR_CUDA(c, cudaMemcpyAsync(c->d_bandw, c->band_w.data(), c->band_w.size() * sizeof(double),
                                 cudaMemcpyHostToDevice, s));
    return PSFR_OK;
}

// the double-buffered band staging of the fused pipeline, allocated by the first call that computes bands: a context
// that never does keeps its footprint
static int alloc_band_staging(Ctx* c) {
    if (c->d_mbee[1]) return PSFR_OK;   // the last buffer allocated below
    const size_t sets = (size_t)c->max_planes * PSFR_MAX_BANDS;
    for (int i = 0; i < 2; ++i) {   // after a failed attempt, start again
        cudaFree(c->d_band[i]); cudaFree(c->d_bfit[i]); cudaFree(c->d_bee[i]);
        cudaFree(c->d_mband[i]); cudaFree(c->d_mbfit[i]); cudaFree(c->d_mbee[i]);
        c->d_band[i] = c->d_bfit[i] = c->d_bee[i] = c->d_mband[i] = c->d_mbfit[i] = c->d_mbee[i] = nullptr;
    }
    for (int i = 0; i < 2; ++i) {
        int rc = dev_alloc(c, &c->d_band[i], sets * kPSF * kPSF);
        if (!rc) rc = dev_alloc(c, &c->d_bfit[i], sets * PSFR_FIT_NPAR);
        if (!rc) rc = dev_alloc(c, &c->d_bee[i], sets * kEeMaxRecord);
        if (!rc) rc = dev_alloc(c, &c->d_mband[i], sets * kPSF * kPSF);
        if (!rc) rc = dev_alloc(c, &c->d_mbfit[i], sets * PSFR_FIT_NPAR);
        if (!rc) rc = dev_alloc(c, &c->d_mbee[i], sets * kEeMaxRecord);
        if (rc) return rc;
    }
    return PSFR_OK;
}

// Outputs of a fused call (run_batch), each NULL or an array on either side: the per-draw ones first, then those
// of the exposure means.  nrad / nfrac size the EE records, nband and sums the band images.
enum { kCube, kFit, kEfit, kEe, kStrehl, kVar, kBand, kBandFit, kBandEe,
       kMean, kMeanFit, kMeanEfit, kMeanEe, kMeanBand, kMeanBandFit, kMeanBandEe, kNumOut };
struct BatchOut {
    double* out[kNumOut] = {};
    int nrad = 0, nfrac = 0, nband = 0;
    BandSums sums;
    bool any(int first, int last) const {   // whether one of the outputs first..last is requested
        for (int i = first; i <= last; ++i)
            if (out[i]) return true;
        return false;
    }
};

constexpr int kMaxHotEvents = 512;
struct HotTimer {
    cudaEvent_t ev[2 * kMaxHotEvents];
    int n = 0;
};

}  // namespace psfr

using namespace psfr;

// the hot-kernel event pairs live outside Ctx to keep the POD simple
static HotTimer* timer_of(Ctx* c) { return reinterpret_cast<HotTimer*>(c->ev_hot0); }

static int hot_begin(Ctx* c) {
    c->hot_launches = 0;
    c->hot_psfs = 0;
    timer_of(c)->n = 0;
    return 0;
}

// The fused pipeline of psfr_compute_batch, psfr_compute_groups and psfr_compute_field, chunk by chunk of
// max_planes / ndir draws: PSD -> structure function -> pruned PSFs -> resample -> convolutions -> fit, and
// with ngroup > 0 the time mean of every exposure (draws [group_end[g-1], group_end[g])) and its fit in the
// chunk where the exposure's last draw lies.  field: every (draw, direction) plane keeps its own PSF instead
// of the draw's field mean, so a draw owns ndir x nlam images in every output (kVar: ndir records in either
// mode).  Host outputs leave through a second stream: the results of chunk i are copied out while chunk i + 1
// computes, from staging buffers that alternate between two sets.
static int run_batch(Ctx* c, int ndraw, const double* draws, int ndir, const double* dirs, int ngs, int npos,
                     const double* poslgs, int nlam, const double* lambda_nm, int ngroup, const int* group_end,
                     bool field, const BatchOut& o, cudaStream_t s) {
    PSFR_CUDA(c, cudaSetDevice(c->device));
    std::vector<double> lam;
    int rc = small_to_host(c, lam, lambda_nm, nlam > 0 ? nlam : 0, s);
    if (rc) return rc;
    rc = set_lambda_tables(c, nlam, lam.data(), s);
    if (rc) return rc;
    rc = run_build_kernels(c, 0, nlam, lam.data(), false, true, s);
    if (rc) return rc;
    std::vector<double> h;
    rc = upload_geometry(c, ndraw, draws, ndir, dirs, ngs, npos, poslgs, h, s);
    if (rc) return rc;
    rc = check_alpha_tt(c, ndraw, h.data() + PSFR_DRAW_ALPHA_TT, PSFR_DRAW_NPAR);
    if (rc) return rc;
    hot_begin(c);
    const int per_chunk = c->max_planes / ndir;
    // output planes per draw; a chunk's nd * ppd * nlam images fit every [max_planes * max_lambda]-image
    // buffer (d_samp, d_cube*, d_fit*, d_mean[b], d_mfit[b], d_carry) because nd * ndir <= max_planes
    const int ppd = field ? ndir : 1;
    const size_t img = (size_t)kPSF * kPSF, imgs = (size_t)ppd * nlam, elems = imgs * img;
    const size_t fits = imgs * PSFR_FIT_NPAR;   // fit records per draw
    const size_t efits = imgs * PSFR_EFIT_NPAR;  // elliptical records per draw
    const size_t ees = imgs * (size_t)(o.nrad + 1 + o.nfrac);   // encircled-energy values per draw
    const size_t vars = (size_t)ndir * PSFR_VAR_NPAR;           // variance values per draw
    const size_t bsets = (size_t)ppd * o.nband;                 // band images per draw and per exposure
    const size_t belems = bsets * img, bfits = bsets * PSFR_FIT_NPAR, bees = bsets * (size_t)(o.nrad + 1 + o.nfrac);
    // values per draw or exposure of each output, and the staging sets that hold it when it is not on the device
    const size_t per[kNumOut] = {elems, fits, efits, ees, imgs, vars, belems, bfits, bees,
                                 elems, fits, efits, ees, belems, bfits, bees};
    double* const stage[kNumOut][2] = {
        {c->d_cube2, c->d_cube3}, {c->d_fit, c->d_fit2}, {c->d_efit, c->d_efit2}, {c->d_ee[0], c->d_ee[1]},
        {c->d_strehl[0], c->d_strehl[1]}, {c->d_var[0], c->d_var[1]}, {c->d_band[0], c->d_band[1]},
        {c->d_bfit[0], c->d_bfit[1]}, {c->d_bee[0], c->d_bee[1]}, {c->d_mean[0], c->d_mean[1]},
        {c->d_mfit[0], c->d_mfit[1]}, {c->d_mefit[0], c->d_mefit[1]}, {c->d_mee[0], c->d_mee[1]},
        {c->d_mband[0], c->d_mband[1]}, {c->d_mbfit[0], c->d_mbfit[1]}, {c->d_mbee[0], c->d_mbee[1]}};
    bool dev[kNumOut], host_out = false;
    for (int i = 0; i < kNumOut; ++i) {
        dev[i] = o.out[i] && is_device_ptr(o.out[i]);
        host_out |= o.out[i] && !dev[i];
    }
    const bool bands = o.any(kBand, kBandEe), mbands = o.any(kMeanBand, kMeanBandEe), means = o.any(kMean, kMeanBandEe);
    int* seg_dev = reinterpret_cast<int*>(c->d_misc + misc_groups(c->max_planes));
    std::vector<int> seg;
    int g0 = 0;   // first exposure not finished in an earlier chunk
    int chunk = 0;
    for (int d0 = 0; d0 < ndraw; d0 += per_chunk, ++chunk) {
        const int nd = std::min(per_chunk, ndraw - d0);
        const int b = chunk & 1;
        // where each output of the chunk is written: the caller's array at its first draw (exposure g0 for the
        // means) when that array is on the device, staging set b otherwise
        double* dst[kNumOut];
        for (int i = 0; i < kNumOut; ++i)
            dst[i] = dev[i] ? o.out[i] + (size_t)(i < kMean ? d0 : g0) * per[i] : stage[i][b];
        rc = upload_draws(c, nd, draws + (size_t)d0 * PSFR_DRAW_NPAR, ndir, s);
        if (rc) break;
        if ((rc = run_psd(c, nd, ndir, ngs, npos, s, false))) break;
        if ((rc = run_structure_function(c, nd * ndir, s, true, ndir))) break;
        // field mode: one column pass per plane (scale 1, no sum over directions), as ndir = 1 calls would run it
        if ((rc = field ? run_pruned_psf(c, nd * ndir, 1, nlam, s) : run_pruned_psf(c, nd, ndir, nlam, s))) break;
        if ((rc = run_resample(c, nd * ppd * nlam, nlam, c->d_cube, s))) break;
        if ((rc = run_build_kernels(c, nd, nlam, lam.data(), true, false, s))) break;
        if (host_out && chunk >= 2 && cudaStreamWaitEvent(s, c->ev_copied[b], 0) != cudaSuccess) {
            rc = set_error(c, PSFR_E_CUDA, "stream wait failed: %s", cudaGetErrorString(cudaGetLastError()));
            break;
        }
        // the AO records of the chunk: d_psdq / d_ao still hold its PSDs and d_samp its raw samples, and staging
        // set b is free again
        if (o.out[kVar] && (rc = run_var(c, nd, ndir, ngs, npos, dst[kVar], s))) break;
        if (o.out[kStrehl] && (rc = run_strehl(c, nd * (int)imgs, dst[kStrehl], s))) break;
        if ((rc = run_convolve(c, nd, ppd, nlam, c->d_cube, dst[kCube], s))) break;
        // the elliptical fit starts from the circular records of the same images
        if ((o.out[kFit] || o.out[kEfit]) && (rc = run_fit(c, nd * (int)imgs, kPSF, kPSF, dst[kCube], dst[kFit], s)))
            break;
        if (o.out[kEfit] && (rc = run_efit(c, nd * (int)imgs, kPSF, kPSF, dst[kCube], dst[kFit], dst[kEfit], s))) break;
        if (o.out[kEe] &&
            (rc = run_ee(c, nd * (int)imgs, kPSF, kPSF, dst[kCube], nullptr, o.nrad, o.nfrac, dst[kEe], s)))
            break;
        // the band images of the chunk's image sets, read from the convolved planes, then their fits and EE
        if (bands &&
            (rc = run_band(c, (long long)nd * ppd, nlam, (int)img, o.nband, o.sums, dst[kCube], dst[kBand], s)))
            break;
        if (o.out[kBandFit] && (rc = run_fit(c, nd * (int)bsets, kPSF, kPSF, dst[kBand], dst[kBandFit], s))) break;
        if (o.out[kBandEe] &&
            (rc = run_ee(c, nd * (int)bsets, kPSF, kPSF, dst[kBand], nullptr, o.nrad, o.nfrac, dst[kBandEe], s)))
            break;
        // exposures g0, g0 + 1, ... that have draws in [d0, d0 + nd): all but possibly the last end here
        int ndone = 0;
        if (means) {
            seg.clear();
            for (int g = g0; g < ngroup && (g == g0 || group_end[g - 1] < d0 + nd); ++g) {
                const bool ends = group_end[g] <= d0 + nd;
                seg.push_back(std::min(group_end[g], d0 + nd) - d0);
                seg.push_back(ends ? group_end[g] - (g ? group_end[g - 1] : 0) : 0);
                ndone += ends;
            }
            const bool carry_in = (g0 ? group_end[g0 - 1] : 0) < d0;
            if (cudaMemcpyAsync(seg_dev, seg.data(), seg.size() * sizeof(int), cudaMemcpyHostToDevice, s) != cudaSuccess) {
                rc = set_error(c, PSFR_E_CUDA, "segment upload failed: %s", cudaGetErrorString(cudaGetLastError()));
                break;
            }
            if ((rc = run_group_mean(c, (int)elems, dst[kCube], seg_dev, (int)seg.size() / 2, carry_in, dst[kMean], s)))
                break;
            if ((o.out[kMeanFit] || o.out[kMeanEfit]) && ndone &&
                (rc = run_fit(c, ndone * (int)imgs, kPSF, kPSF, dst[kMean], dst[kMeanFit], s)))
                break;
            if (o.out[kMeanEfit] && ndone &&
                (rc = run_efit(c, ndone * (int)imgs, kPSF, kPSF, dst[kMean], dst[kMeanFit], dst[kMeanEfit], s)))
                break;
            if (o.out[kMeanEe] && ndone &&
                (rc = run_ee(c, ndone * (int)imgs, kPSF, kPSF, dst[kMean], nullptr, o.nrad, o.nfrac, dst[kMeanEe], s)))
                break;
            if (mbands && ndone &&
                (rc = run_band(c, (long long)ndone * ppd, nlam, (int)img, o.nband, o.sums, dst[kMean], dst[kMeanBand], s)))
                break;
            if (o.out[kMeanBandFit] && ndone &&
                (rc = run_fit(c, ndone * (int)bsets, kPSF, kPSF, dst[kMeanBand], dst[kMeanBandFit], s)))
                break;
            if (o.out[kMeanBandEe] && ndone &&
                (rc = run_ee(c, ndone * (int)bsets, kPSF, kPSF, dst[kMeanBand], nullptr, o.nrad, o.nfrac,
                             dst[kMeanBandEe], s)))
                break;
        }
        if (host_out) {
            // the host outputs of the chunk's nd draws and of the ndone exposures that end in it
            cudaError_t e = cudaEventRecord(c->ev_done[b], s);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(c->copy_stream, c->ev_done[b], 0);
            for (int i = 0; i < kNumOut && e == cudaSuccess; ++i) {
                const size_t first = i < kMean ? d0 : g0, count = i < kMean ? nd : ndone;
                if (o.out[i] && !dev[i] && count)
                    e = cudaMemcpyAsync(o.out[i] + first * per[i], dst[i], count * per[i] * sizeof(double),
                                        cudaMemcpyDefault, c->copy_stream);
            }
            if (e == cudaSuccess) e = cudaEventRecord(c->ev_copied[b], c->copy_stream);
            if (e != cudaSuccess) {
                rc = set_error(c, PSFR_E_CUDA, "result copy failed: %s", cudaGetErrorString(e));
                break;
            }
        }
        g0 += ndone;
    }
    if (host_out) {
        // host outputs are complete on return; later work on `s` must not overtake the copies
        cudaError_t e = cudaStreamSynchronize(c->copy_stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        if (e != cudaSuccess && !rc) rc = set_error(c, PSFR_E_CUDA, "compute_batch: %s", cudaGetErrorString(e));
    }
    return rc;
}

extern "C" {

int psfr_version(void) { return 108; }

const char* psfr_last_error(const psfr_ctx* ctx) { return ctx ? ctx->err : g_create_error; }

void psfr_destroy(psfr_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaFree(c->d_tw); cudaFree(c->d_pup); cudaFree(c->d_otf); cudaFree(c->d_geom); cudaFree(c->d_psd); cudaFree(c->d_psdq);
    cudaFree(c->d_bt); cudaFree(c->d_dphi); cudaFree(c->d_ybuf); cudaFree(c->d_samp); cudaFree(c->d_ao);
    cudaFree(c->d_draws); cudaFree(c->d_misc); cudaFree(c->d_lam); cudaFree(c->d_kidx); cudaFree(c->d_frac);
    cudaFree(c->d_kern_tt); cudaFree(c->d_kern_mu); cudaFree(c->d_cube); cudaFree(c->d_cube2);
    cudaFree(c->d_fit); cudaFree(c->d_poly); cudaFree(c->d_dmin); cudaFree(c->d_counter);
    cudaFree(c->d_twc); cudaFree(c->d_wsamp); cudaFree(c->d_wcol); cudaFree(c->d_kcol); cudaFree(c->d_xmap); cudaFree(c->d_khat_tt); cudaFree(c->d_khat_mu);
    cudaFree(c->d_cube3); cudaFree(c->d_fit2); cudaFree(c->d_carry); cudaFree(c->d_efit); cudaFree(c->d_efit2);
    for (int i = 0; i < 2; ++i) { cudaFree(c->d_mean[i]); cudaFree(c->d_mfit[i]); cudaFree(c->d_mefit[i]); }
    for (int i = 0; i < 2; ++i) { cudaFree(c->d_ee[i]); cudaFree(c->d_mee[i]); cudaFree(c->d_strehl[i]); cudaFree(c->d_var[i]); }
    cudaFree(c->d_eepar); cudaFree(c->d_eecen); cudaFree(c->d_bandw);
    for (int i = 0; i < 2; ++i) {
        cudaFree(c->d_band[i]); cudaFree(c->d_bfit[i]); cudaFree(c->d_bee[i]);
        cudaFree(c->d_mband[i]); cudaFree(c->d_mbfit[i]); cudaFree(c->d_mbee[i]);
    }
    cudaFree(c->d_dphi32); cudaFree(c->d_otf32); cudaFree(c->d_tw32); cudaFree(c->d_twg); cudaFree(c->d_twg32); cudaFree(c->d_p3); cudaFree(c->d_p2mask); cudaFree(c->d_csort); cudaFree(c->d_lorder); cudaFree(c->d_kaddr);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    for (int i = 0; i < 2; ++i) {
        if (c->ev_done[i]) cudaEventDestroy(c->ev_done[i]);
        if (c->ev_copied[i]) cudaEventDestroy(c->ev_copied[i]);
    }
    if (c->h_pinned) cudaFreeHost(c->h_pinned);
    HotTimer* t = timer_of(c);
    if (t) {
        for (int i = 0; i < 2 * kMaxHotEvents; ++i)
            if (t->ev[i]) cudaEventDestroy(t->ev[i]);
        delete t;
    }
    delete c;
}

int psfr_create(int device, int dim, int max_planes, int max_lambda, psfr_ctx** out) {
    if (!out) return set_error(nullptr, PSFR_E_ARG, "out is NULL");
    *out = nullptr;
    if (dim != kNB && dim != 2 * kNB)
        return set_error(nullptr, PSFR_E_UNSUPPORTED, "dim=%d: this build supports dim=%d and dim=%d only", dim, kNB,
                         2 * kNB);
    if (max_planes < 1 || max_lambda < 1 || max_lambda > kMaxLambdaCap)
        return set_error(nullptr, PSFR_E_ARG, "max_planes=%d max_lambda=%d out of range", max_planes, max_lambda);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return set_error(nullptr, PSFR_E_CUDA, "no CUDA device available (this library has no CPU fallback)");
    }
    if (device < 0 || device >= ndev) return set_error(nullptr, PSFR_E_ARG, "device %d of %d", device, ndev);
    psfr_ctx* c = new psfr_ctx();
    c->device = device;
    c->max_planes = max_planes;
    c->max_lambda = max_lambda;
    c->NF = dim / kNB;
    c->N = dim;
    c->NH = dim / 2;
    c->rows = dim / 2 + 2;
    c->pairs = c->rows / 2;
    const size_t kN = c->N, kNH = c->NH, kRows = c->rows;
#define CK(call)                         \
    do {                                 \
        int rc__ = (call);               \
        if (rc__) {                      \
            strncpy(g_create_error, c->err, 511); \
            psfr_destroy(c);             \
            return rc__;                 \
        }                                \
    } while (0)
#define CKC(call)                                                                               \
    do {                                                                                        \
        cudaError_t e__ = (call);                                                               \
        if (e__ != cudaSuccess) {                                                               \
            set_error(nullptr, PSFR_E_CUDA, "%s: %s", #call, cudaGetErrorString(e__));          \
            psfr_destroy(c);                                                                    \
            return PSFR_E_CUDA;                                                                 \
        }                                                                                       \
    } while (0)
    CKC(cudaSetDevice(device));
    cudaDeviceProp prop;
    CKC(cudaGetDeviceProperties(&prop, device));
    c->sm_count = prop.multiProcessorCount;
    if (prop.major != 10) {   // the library holds an sm_100a cubin and no PTX
        set_error(nullptr, PSFR_E_UNSUPPORTED, "device %d has compute capability %d.%d; this library is built for sm_100a (B200) only",
                  device, prop.major, prop.minor);
        psfr_destroy(c);
        return PSFR_E_UNSUPPORTED;
    }
    const size_t P = max_planes, LM = max_lambda;
    CK(dev_alloc(c, &c->d_tw, (size_t)FftGeom<kR3>::TW1 + FftGeom<kR3>::TW2));
    CK(dev_alloc(c, &c->d_twc, (size_t)kNB));
    CK(dev_alloc(c, &c->d_wsamp, LM * 2 * kNS));
    CK(dev_alloc(c, &c->d_wcol, LM * 2 * kNC));
    CK(dev_alloc(c, &c->d_kcol, LM * kNC));
    CK(dev_alloc(c, &c->d_xmap, LM * kNC));
    CK(dev_alloc(c, &c->d_pup, (size_t)kNH * kNH));
    CK(dev_alloc(c, &c->d_otf, (size_t)kRows * kN));
    CK(dev_alloc(c, &c->d_geom, (size_t)3 * kAO * kAO));
    CK(dev_alloc(c, &c->d_psd, P * kN * kN));
    CK(dev_alloc(c, &c->d_psdq, P * kNH * kNH));
    CK(dev_alloc(c, &c->d_bt, P * kN * kRows));
    CK(dev_alloc(c, &c->d_dphi, P * kRows * kN));
    CK(dev_alloc(c, &c->d_dmin, P * kRows));
    if (c->NF == 1) {
        CK(dev_alloc(c, &c->d_dphi32, P * kRows * kN));
        CK(dev_alloc(c, &c->d_otf32, (size_t)kRows * kN));
        CK(dev_alloc(c, &c->d_tw32, (size_t)FftGeom<kR3>::TW1 + FftGeom<kR3>::TW2));
        CK(dev_alloc(c, &c->d_twg32, (size_t)kGroupTw));
    }
    CK(dev_alloc(c, &c->d_twg, (size_t)kGroupTw));
    CK(dev_alloc(c, &c->d_p3, LM * 2 * kNC));
    CK(dev_alloc(c, &c->d_p2mask, LM * kGMaskStride));
    CK(dev_alloc(c, &c->d_counter, (size_t)16));
    CK(dev_alloc(c, &c->d_ybuf, P * LM * kNC * kRows));
    CK(dev_alloc(c, &c->d_samp, P * LM * kNS * kNS));
    // samples with bilinear weight 0 are never written: keep them finite (0 * stale value must be 0)
    CKC(cudaMemset(c->d_samp, 0, P * LM * kNS * kNS * sizeof(double)));
    CK(dev_alloc(c, &c->d_ao, P * kAO * kAO));
    CK(dev_alloc(c, &c->d_draws, P * PSFR_DRAW_NPAR));
    CK(dev_alloc(c, &c->d_misc, (size_t)misc_size(max_planes)));
    CK(dev_alloc(c, &c->d_lam, LM));
    CK(dev_alloc(c, &c->d_csort, LM));
    CK(dev_alloc(c, &c->d_lorder, LM));
    CK(dev_alloc(c, &c->d_kidx, LM * kNS));
    CK(dev_alloc(c, &c->d_kaddr, LM * kNC));
    CK(dev_alloc(c, &c->d_frac, LM * kPSF));
    CK(dev_alloc(c, &c->d_kern_tt, P * kKW * kKW));
    CK(dev_alloc(c, &c->d_kern_mu, LM * kKW * kKW));
    CK(dev_alloc(c, &c->d_khat_tt, P * 80 * 41));
    CK(dev_alloc(c, &c->d_khat_mu, LM * 80 * 41));
    CK(dev_alloc(c, &c->d_cube, P * LM * kPSF * kPSF));
    CK(dev_alloc(c, &c->d_cube2, P * LM * kPSF * kPSF));
    CK(dev_alloc(c, &c->d_fit, P * LM * PSFR_FIT_NPAR));
    CK(dev_alloc(c, &c->d_cube3, P * LM * kPSF * kPSF));
    CK(dev_alloc(c, &c->d_fit2, P * LM * PSFR_FIT_NPAR));
    CK(dev_alloc(c, &c->d_carry, P * LM * kPSF * kPSF));
    CK(dev_alloc(c, &c->d_efit, P * LM * PSFR_EFIT_NPAR));
    CK(dev_alloc(c, &c->d_efit2, P * LM * PSFR_EFIT_NPAR));
    for (int i = 0; i < 2; ++i) {
        CK(dev_alloc(c, &c->d_mean[i], P * LM * kPSF * kPSF));
        CK(dev_alloc(c, &c->d_mfit[i], P * LM * PSFR_FIT_NPAR));
        CK(dev_alloc(c, &c->d_mefit[i], P * LM * PSFR_EFIT_NPAR));
        CK(dev_alloc(c, &c->d_ee[i], P * LM * kEeMaxRecord));
        CK(dev_alloc(c, &c->d_mee[i], P * LM * kEeMaxRecord));
        CK(dev_alloc(c, &c->d_strehl[i], P * LM));
        CK(dev_alloc(c, &c->d_var[i], P * PSFR_VAR_NPAR));
    }
    CK(dev_alloc(c, &c->d_eepar, (size_t)PSFR_EE_MAX_RADII + PSFR_EE_MAX_FRACTIONS));
    CK(dev_alloc(c, &c->d_eecen, P * LM * 2));
    CKC(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
        CKC(cudaEventCreateWithFlags(&c->ev_done[i], cudaEventDisableTiming));
        CKC(cudaEventCreateWithFlags(&c->ev_copied[i], cudaEventDisableTiming));
    }
    CK(dev_alloc(c, &c->d_poly, (size_t)65536));
    c->h_pinned_bytes = 1 << 20;
    CKC(cudaMallocHost(&c->h_pinned, c->h_pinned_bytes));
    HotTimer* t = new HotTimer();
    for (int i = 0; i < 2 * kMaxHotEvents; ++i) t->ev[i] = nullptr;
    c->ev_hot0 = reinterpret_cast<cudaEvent_t>(t);   // owned by the context from here on (psfr_destroy frees it)
    for (int i = 0; i < 2 * kMaxHotEvents; ++i) CKC(cudaEventCreate(&t->ev[i]));
    std::vector<double2> tw1, tw2;
    build_twiddles<kR3>(tw1, tw2);
    CKC(cudaMemcpy(c->d_tw, tw1.data(), tw1.size() * sizeof(double2), cudaMemcpyHostToDevice));
    CKC(cudaMemcpy(c->d_tw + tw1.size(), tw2.data(), tw2.size() * sizeof(double2), cudaMemcpyHostToDevice));
    if (c->d_tw32) {
        std::vector<float2> tw32(tw1.size() + tw2.size());
        for (size_t i = 0; i < tw1.size(); ++i) tw32[i] = make_float2((float)tw1[i].x, (float)tw1[i].y);
        for (size_t i = 0; i < tw2.size(); ++i) tw32[tw1.size() + i] = make_float2((float)tw2[i].x, (float)tw2[i].y);
        CKC(cudaMemcpy(c->d_tw32, tw32.data(), tw32.size() * sizeof(float2), cudaMemcpyHostToDevice));
    }
    if (c->d_twg) {
        std::vector<double2> twg(kGroupTw);
        std::vector<float2> twg32(kGroupTw);
        for (int n2 = 0; n2 < kG2; ++n2)
            for (int k1 = 1; k1 < kG1; ++k1) {
                const double2 w = unit_root((long long)n2 * k1, 160);
                twg[n2 * (kG1 - 1) + k1 - 1] = w;
                twg32[n2 * (kG1 - 1) + k1 - 1] = make_float2((float)w.x, (float)w.y);
            }
        CKC(cudaMemcpy(c->d_twg, twg.data(), twg.size() * sizeof(double2), cudaMemcpyHostToDevice));
        if (c->d_twg32)
            CKC(cudaMemcpy(c->d_twg32, twg32.data(), twg32.size() * sizeof(float2), cudaMemcpyHostToDevice));
    }
    {
        std::vector<double2> twc(kNB);
        for (int k = 0; k < kNB; ++k) twc[k] = unit_root(k, c->N);
        CKC(cudaMemcpy(c->d_twc, twc.data(), twc.size() * sizeof(double2), cudaMemcpyHostToDevice));
    }
    CK(run_build_otf(c, 0));
    CK(run_otf_sum(c, 0));
    CKC(cudaDeviceSynchronize());
#undef CK
#undef CKC
    *out = c;
    return PSFR_OK;
}

int psfr_set_geometry(psfr_ctx* c, const double* f, const double* fx, const double* fy) {
    if (!c || !f || !fx || !fy) return set_error(c, PSFR_E_ARG, "NULL argument");
    PSFR_CUDA(c, cudaSetDevice(c->device));
    const size_t n = (size_t)kAO * kAO * sizeof(double);
    PSFR_CUDA(c, cudaMemcpy(c->d_geom, f, n, cudaMemcpyDefault));
    PSFR_CUDA(c, cudaMemcpy(c->d_geom + kAO * kAO, fx, n, cudaMemcpyDefault));
    PSFR_CUDA(c, cudaMemcpy(c->d_geom + 2 * kAO * kAO, fy, n, cudaMemcpyDefault));
    c->geometry_set = true;
    return PSFR_OK;
}

int psfr_psd(psfr_ctx* c, int ndraw, const double* draws, int ndir, const double* dirs, int ngs,
             const double* poslgs, double* out_psd, void* stream) {
    if (!c || !draws || !dirs || !poslgs) return set_error(c, PSFR_E_ARG, "NULL argument");
    if (ngs < 1) return set_error(c, PSFR_E_ARG, "ngs=%d outside [1,%d]", ngs, kMaxGS);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    PSFR_CUDA(c, cudaSetDevice(c->device));
    std::vector<double> h;   // psfr_psd never reads the tip-tilt alpha: records with any value in it pass
    int rc = upload_geometry(c, ndraw, draws, ndir, dirs, ngs, ngs, poslgs, h, s);
    if (rc) return rc;
    if ((rc = upload_draws(c, ndraw, draws, ndir, s))) return rc;
    rc = run_psd(c, ndraw, ndir, ngs, ngs, s);
    if (rc) return rc;
    if (out_psd) return from_device(c, out_psd, c->d_psd, (size_t)ndraw * ndir * c->N * c->N * sizeof(double), s);
    return PSFR_OK;
}

int psfr_load_psd(psfr_ctx* c, int nplanes, const double* psd, void* stream) {
    if (!c || !psd) return set_error(c, PSFR_E_ARG, "NULL argument");
    if (nplanes < 1 || nplanes > c->max_planes)
        return set_error(c, PSFR_E_CAPACITY, "nplanes=%d exceeds max_planes=%d", nplanes, c->max_planes);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    PSFR_CUDA(c, cudaSetDevice(c->device));
    int rc = to_device(c, c->d_psd, psd, (size_t)nplanes * c->N * c->N * sizeof(double), s);
    if (rc) return rc;
    c->planes_loaded = nplanes;
    c->planes_struct = 0;
    return PSFR_OK;
}

int psfr_structure_function(psfr_ctx* c, int nplanes, void* stream) {
    if (!c) return set_error(c, PSFR_E_ARG, "NULL context");
    if (nplanes < 1 || nplanes > c->planes_loaded)
        return set_error(c, PSFR_E_STATE, "nplanes=%d but %d PSD planes are loaded", nplanes, c->planes_loaded);
    PSFR_CUDA(c, cudaSetDevice(c->device));
    return run_structure_function(c, nplanes, static_cast<cudaStream_t>(stream));
}

int psfr_psd_to_psf(psfr_ctx* c, int plane, double lambda_m, double* out_psf, void* stream) {
    if (!c || !out_psf) return set_error(c, PSFR_E_ARG, "NULL argument");
    if (plane < 0 || plane >= c->planes_struct)
        return set_error(c, PSFR_E_STATE, "plane %d has no structure function (call psfr_structure_function)", plane);
    if (!(lambda_m > 0)) return set_error(c, PSFR_E_ARG, "lambda must be positive");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    PSFR_CUDA(c, cudaSetDevice(c->device));
    const double conv = 2 * 3.141592653589793 / (lambda_m * 1e9);
    // the PSD workspace of the LAST plane slot is not needed any more once D exists; write the
    // PSF into the transposed-buffer-free psd slot of this plane and copy it out
    double* dst = is_device_ptr(out_psf) ? out_psf : c->d_psd + (size_t)plane * c->N * c->N;
    int rc = run_full_psf(c, plane, 0.5 * (conv * conv), dst, s);
    if (rc) return rc;
    if (dst != out_psf) {
        rc = from_device(c, out_psf, dst, (size_t)c->N * c->N * sizeof(double), s);
        if (rc) return rc;
        c->planes_loaded = 0;   // the PSD of that slot was overwritten
    }
    return PSFR_OK;
}

int psfr_psf_cube(psfr_ctx* c, int ndraw, int ndir, int nlam, const double* lambda_nm, double* out_cube,
                  void* stream) {
    if (!c || !lambda_nm || !out_cube) return set_error(c, PSFR_E_ARG, "NULL argument");
    if (ndraw < 1 || ndir < 1 || ndraw * ndir > c->planes_struct)
        return set_error(c, PSFR_E_STATE, "ndraw*ndir=%d but %d structure-function planes exist", ndraw * ndir,
                         c->planes_struct);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    PSFR_CUDA(c, cudaSetDevice(c->device));
    std::vector<double> lam;
    int rc = small_to_host(c, lam, lambda_nm, nlam > 0 ? nlam : 0, s);
    if (rc) return rc;
    rc = set_lambda_tables(c, nlam, lam.data(), s);
    if (rc) return rc;
    hot_begin(c);
    rc = run_pruned_psf(c, ndraw, ndir, nlam, s);
    if (rc) return rc;
    double* dst = is_device_ptr(out_cube) ? out_cube : c->d_cube;
    rc = run_resample(c, ndraw * nlam, nlam, dst, s);
    if (rc) return rc;
    if (dst != out_cube) return from_device(c, out_cube, dst, (size_t)ndraw * nlam * kPSF * kPSF * sizeof(double), s);
    return PSFR_OK;
}

int psfr_convolve(psfr_ctx* c, int ndraw, int nlam, const double* lambda_nm, const double* alpha_tt,
                  const double* cube, double* out_cube, void* stream) {
    if (!c || !lambda_nm || !alpha_tt || !cube || !out_cube) return set_error(c, PSFR_E_ARG, "NULL argument");
    if (ndraw < 1 || ndraw > c->max_planes || nlam < 1 || nlam > c->max_lambda)
        return set_error(c, PSFR_E_CAPACITY, "ndraw=%d nlam=%d exceed the context capacity", ndraw, nlam);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    PSFR_CUDA(c, cudaSetDevice(c->device));
    std::vector<double> lam, att;
    int rc = small_to_host(c, lam, lambda_nm, nlam, s);
    if (!rc) rc = small_to_host(c, att, alpha_tt, ndraw, s);
    if (rc) return rc;
    for (int l = 0; l < nlam; ++l)
        if (!(std::isfinite(lam[l]) && lam[l] > 0))
            return set_error(c, PSFR_E_ARG, "wavelength %g nm is not finite and positive", lam[l]);
    if ((rc = check_alpha_tt(c, ndraw, att.data(), 1))) return rc;
    rc = to_device(c, c->d_misc + misc_alpha_tt(c->max_planes), alpha_tt, ndraw * sizeof(double), s);
    if (rc) return rc;
    rc = run_build_kernels(c, ndraw, nlam, lam.data(), true, true, s);
    if (rc) return rc;
    const size_t bytes = (size_t)ndraw * nlam * kPSF * kPSF * sizeof(double);
    const double* src = cube;
    if (!is_device_ptr(cube)) {
        rc = to_device(c, c->d_cube, cube, bytes, s);
        if (rc) return rc;
        src = c->d_cube;
    }
    double* dst = is_device_ptr(out_cube) ? out_cube : c->d_cube2;
    rc = run_convolve(c, ndraw, 1, nlam, src, dst, s);
    if (rc) return rc;
    if (dst != out_cube) return from_device(c, out_cube, dst, bytes, s);
    return PSFR_OK;
}

int psfr_moffat_fit(psfr_ctx* c, int nimg, int ny, int nx, const double* imgs, double* params, void* stream) {
    if (!c || !imgs || !params) return set_error(c, PSFR_E_ARG, "NULL argument");
    if (nimg < 1 || ny < 3 || nx < 3) return set_error(c, PSFR_E_ARG, "nimg=%d ny=%d nx=%d", nimg, ny, nx);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    PSFR_CUDA(c, cudaSetDevice(c->device));
    const size_t cap = (size_t)c->max_planes * c->max_lambda;
    const size_t per = (size_t)ny * nx;
    const bool in_dev = is_device_ptr(imgs), out_dev = is_device_ptr(params);
    // chunk through the staging buffers when the caller's arrays live on the host
    const size_t chunk_imgs = std::min(cap, (cap * kPSF * kPSF) / per);
    if (chunk_imgs < 1) return set_error(c, PSFR_E_CAPACITY, "image %dx%d does not fit the staging buffer", ny, nx);
    for (size_t i0 = 0; i0 < (size_t)nimg; i0 += chunk_imgs) {
        const int n = (int)std::min(chunk_imgs, (size_t)nimg - i0);
        const double* src = imgs + i0 * per;
        if (!in_dev) {
            int rc = to_device(c, c->d_cube, src, (size_t)n * per * sizeof(double), s);
            if (rc) return rc;
            src = c->d_cube;
        }
        double* dst = out_dev ? params + i0 * PSFR_FIT_NPAR : c->d_fit;
        int rc = run_fit(c, n, ny, nx, src, dst, s);
        if (rc) return rc;
        if (!out_dev) {
            rc = from_device(c, params + i0 * PSFR_FIT_NPAR, dst, (size_t)n * PSFR_FIT_NPAR * sizeof(double), s);
            if (rc) return rc;
        }
    }
    return PSFR_OK;
}

int psfr_moffat_fit_elliptical(psfr_ctx* c, int nimg, int ny, int nx, const double* imgs, double* params,
                               void* stream) {
    if (!c || !imgs || !params) return set_error(c, PSFR_E_ARG, "NULL argument");
    if (nimg < 1 || ny < 3 || nx < 3) return set_error(c, PSFR_E_ARG, "nimg=%d ny=%d nx=%d", nimg, ny, nx);
    if ((long long)ny * nx <= 7)
        return set_error(c, PSFR_E_ARG, "image %dx%d: the elliptical fit needs more than 7 pixels", ny, nx);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    PSFR_CUDA(c, cudaSetDevice(c->device));
    const size_t cap = (size_t)c->max_planes * c->max_lambda;
    const size_t per = (size_t)ny * nx;
    const bool in_dev = is_device_ptr(imgs), out_dev = is_device_ptr(params);
    // the circular records go to d_fit and, for host outputs, the elliptical ones to d_efit: both hold cap records
    const size_t chunk_imgs = std::min(cap, (cap * kPSF * kPSF) / per);
    if (chunk_imgs < 1) return set_error(c, PSFR_E_CAPACITY, "image %dx%d does not fit the staging buffer", ny, nx);
    for (size_t i0 = 0; i0 < (size_t)nimg; i0 += chunk_imgs) {
        const int n = (int)std::min(chunk_imgs, (size_t)nimg - i0);
        const double* src = imgs + i0 * per;
        if (!in_dev) {
            int rc = to_device(c, c->d_cube, src, (size_t)n * per * sizeof(double), s);
            if (rc) return rc;
            src = c->d_cube;
        }
        double* dst = out_dev ? params + i0 * PSFR_EFIT_NPAR : c->d_efit;
        int rc = run_fit(c, n, ny, nx, src, c->d_fit, s);
        if (rc) return rc;
        rc = run_efit(c, n, ny, nx, src, c->d_fit, dst, s);
        if (rc) return rc;
        if (!out_dev) {
            rc = from_device(c, params + i0 * PSFR_EFIT_NPAR, dst, (size_t)n * PSFR_EFIT_NPAR * sizeof(double), s);
            if (rc) return rc;
        }
    }
    return PSFR_OK;
}

int psfr_moffat_fit_weighted(psfr_ctx* c, int nimg, int ny, int nx, const double* imgs, const double* weights,
                             int fit_back, int elliptical, double* params, double* back, void* stream) {
    if (!c || !imgs || !params) return set_error(c, PSFR_E_ARG, "NULL argument");
    if (nimg < 1 || ny < 3 || nx < 3) return set_error(c, PSFR_E_ARG, "nimg=%d ny=%d nx=%d", nimg, ny, nx);
    if (int rc = check_star_fit_size(c, ny, nx, elliptical != 0)) return rc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    PSFR_CUDA(c, cudaSetDevice(c->device));
    const size_t cap = (size_t)c->max_planes * c->max_lambda;
    const size_t per = (size_t)ny * nx;
    const int npar = elliptical ? PSFR_EFIT_NPAR : PSFR_FIT_NPAR;
    const bool in_dev = is_device_ptr(imgs), w_dev = !weights || is_device_ptr(weights);
    const bool out_dev = is_device_ptr(params), back_dev = back && is_device_ptr(back);
    // host images and weights go through d_cube and d_cube2, host records through d_fit (circular) or d_efit
    // (elliptical; d_fit then holds the circular start records), and the side records through d_fit2 unless the
    // caller's are on the device: each holds cap images' worth
    const size_t chunk_imgs = std::min(cap, (cap * kPSF * kPSF) / per);
    if (chunk_imgs < 1) return set_error(c, PSFR_E_CAPACITY, "image %dx%d does not fit the staging buffer", ny, nx);
    for (size_t i0 = 0; i0 < (size_t)nimg; i0 += chunk_imgs) {
        const int n = (int)std::min(chunk_imgs, (size_t)nimg - i0);
        const size_t bytes = (size_t)n * per * sizeof(double);
        const double* src = imgs + i0 * per;
        const double* w = weights ? weights + i0 * per : nullptr;
        int rc;
        if (!in_dev) {
            if ((rc = to_device(c, c->d_cube, src, bytes, s))) return rc;
            src = c->d_cube;
        }
        if (!w_dev) {
            if ((rc = to_device(c, c->d_cube2, w, bytes, s))) return rc;
            w = c->d_cube2;
        }
        double* dst = out_dev ? params + i0 * npar : (elliptical ? c->d_efit : c->d_fit);
        double* bdst = back_dev ? back + i0 * PSFR_BACK_NPAR : c->d_fit2;
        if (elliptical) {
            if ((rc = run_star_fit(c, n, ny, nx, src, w, fit_back != 0, c->d_fit, bdst, s))) return rc;
            rc = run_star_efit(c, n, ny, nx, src, w, fit_back != 0, c->d_fit, bdst, dst, bdst, s);
        } else {
            rc = run_star_fit(c, n, ny, nx, src, w, fit_back != 0, dst, bdst, s);
        }
        if (rc) return rc;
        if (!out_dev && (rc = from_device(c, params + i0 * npar, dst, (size_t)n * npar * sizeof(double), s))) return rc;
        if (back && !back_dev &&
            (rc = from_device(c, back + i0 * PSFR_BACK_NPAR, bdst, (size_t)n * PSFR_BACK_NPAR * sizeof(double), s)))
            return rc;
    }
    return PSFR_OK;
}

int psfr_template_fit(psfr_ctx* c, int nimg, int ny, int nx, const double* imgs, const double* weights, int ntpl,
                      int ty, int tx, const double* tpls, int fit_back, double* params, double* model, void* stream) {
    if (!c || !imgs || !tpls || !params) return set_error(c, PSFR_E_ARG, "NULL argument");
    if (nimg < 1 || ny < 3 || nx < 3 || ntpl < 1 || nimg % ntpl != 0 || ty < 4 || tx < 4)
        return set_error(c, PSFR_E_ARG, "nimg=%d ny=%d nx=%d ntpl=%d ty=%d tx=%d (nimg must be a multiple of ntpl)",
                         nimg, ny, nx, ntpl, ty, tx);
    if (int rc = check_template_fit_size(c, ny, nx, ty, tx)) return rc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    PSFR_CUDA(c, cudaSetDevice(c->device));
    const size_t cap = (size_t)c->max_planes * c->max_lambda * kPSF * kPSF;   // doubles per staging buffer
    const size_t per = (size_t)ny * nx, tpl_len = (size_t)ntpl * ty * tx;
    const bool in_dev = is_device_ptr(imgs), w_dev = !weights || is_device_ptr(weights);
    const bool t_dev = is_device_ptr(tpls), out_dev = is_device_ptr(params), m_dev = model && is_device_ptr(model);
    // host stamps, weights and models go through d_cube, d_cube2 and d_cube3, host records through d_fit, and host
    // templates, which every chunk reads whole, through d_mean[0]; when no stamp-sized array is on the host, one
    // launch fits every image
    const bool all_dev = in_dev && w_dev && out_dev && (!model || m_dev);
    const size_t chunk_imgs = all_dev ? (size_t)nimg : std::min((size_t)c->max_planes * c->max_lambda, cap / per);
    if (chunk_imgs < 1) return set_error(c, PSFR_E_CAPACITY, "image %dx%d does not fit the staging buffer", ny, nx);
    if (!t_dev && tpl_len > cap)
        return set_error(c, PSFR_E_CAPACITY, "%d host templates of %dx%d do not fit the staging buffer (%zu doubles)",
                         ntpl, ty, tx, cap);
    int rc;
    const double* tpl = tpls;
    if (!t_dev) {
        if ((rc = to_device(c, c->d_mean[0], tpls, tpl_len * sizeof(double), s))) return rc;
        tpl = c->d_mean[0];
    }
    for (size_t i0 = 0; i0 < (size_t)nimg; i0 += chunk_imgs) {
        const int n = (int)std::min(chunk_imgs, (size_t)nimg - i0);
        const size_t bytes = (size_t)n * per * sizeof(double);
        const double* src = imgs + i0 * per;
        const double* w = weights ? weights + i0 * per : nullptr;
        if (!in_dev) {
            if ((rc = to_device(c, c->d_cube, src, bytes, s))) return rc;
            src = c->d_cube;
        }
        if (!w_dev) {
            if ((rc = to_device(c, c->d_cube2, w, bytes, s))) return rc;
            w = c->d_cube2;
        }
        double* dst = out_dev ? params + i0 * PSFR_TFIT_NPAR : c->d_fit;
        double* mdst = !model ? nullptr : m_dev ? model + i0 * per : c->d_cube3;
        if ((rc = run_template_fit(c, n, ny, nx, src, w, ntpl, ty, tx, tpl, (long long)i0, fit_back != 0, dst, mdst,
                                   s)))
            return rc;
        if (!out_dev &&
            (rc = from_device(c, params + i0 * PSFR_TFIT_NPAR, dst, (size_t)n * PSFR_TFIT_NPAR * sizeof(double), s)))
            return rc;
        if (model && !m_dev && (rc = from_device(c, model + i0 * per, mdst, bytes, s))) return rc;
    }
    return PSFR_OK;
}

int psfr_encircled_energy(psfr_ctx* c, int nimg, int ny, int nx, const double* imgs, const double* centres, int nrad,
                          const double* radii_px, int nfrac, const double* fracs, double* out, void* stream) {
    if (!c || !imgs || !out) return set_error(c, PSFR_E_ARG, "NULL argument");
    if (nimg < 1 || ny < 3 || nx < 3) return set_error(c, PSFR_E_ARG, "nimg=%d ny=%d nx=%d", nimg, ny, nx);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    PSFR_CUDA(c, cudaSetDevice(c->device));
    int rc = upload_ee_params(c, nrad, radii_px, nfrac, fracs, s);
    if (rc) return rc;
    if (centres) {
        std::vector<double> h;
        if ((rc = small_to_host(c, h, centres, (size_t)nimg * 2, s))) return rc;
        for (size_t i = 0; i < h.size(); ++i)
            if (!std::isfinite(h[i]))
                return set_error(c, PSFR_E_ARG, "centre of image %zu is not finite", i / 2);
    }
    const size_t cap = (size_t)c->max_planes * c->max_lambda;
    const size_t per = (size_t)ny * nx, rec = (size_t)nrad + 1 + nfrac;
    const bool in_dev = is_device_ptr(imgs), out_dev = is_device_ptr(out);
    const bool cen_dev = centres && is_device_ptr(centres);
    // host images, centres and records go through d_cube, d_eecen and d_ee[0]: each holds cap images' worth
    const size_t chunk_imgs = std::min(cap, (cap * kPSF * kPSF) / per);
    if (chunk_imgs < 1) return set_error(c, PSFR_E_CAPACITY, "image %dx%d does not fit the staging buffer", ny, nx);
    for (size_t i0 = 0; i0 < (size_t)nimg; i0 += chunk_imgs) {
        const int n = (int)std::min(chunk_imgs, (size_t)nimg - i0);
        const double* src = imgs + i0 * per;
        if (!in_dev) {
            if ((rc = to_device(c, c->d_cube, src, (size_t)n * per * sizeof(double), s))) return rc;
            src = c->d_cube;
        }
        const double* cen = centres ? centres + 2 * i0 : nullptr;
        if (centres && !cen_dev) {
            if ((rc = to_device(c, c->d_eecen, cen, (size_t)n * 2 * sizeof(double), s))) return rc;
            cen = c->d_eecen;
        }
        double* dst = out_dev ? out + i0 * rec : c->d_ee[0];
        if ((rc = run_ee(c, n, ny, nx, src, cen, nrad, nfrac, dst, s))) return rc;
        if (!out_dev && (rc = from_device(c, out + i0 * rec, dst, (size_t)n * rec * sizeof(double), s))) return rc;
    }
    return PSFR_OK;
}

int psfr_compute_batch(psfr_ctx* c, int ndraw, const double* draws, int ndir, const double* dirs, int ngs,
                       const double* poslgs, int nlam, const double* lambda_nm, double* out_cube,
                       double* out_fit, void* stream) {
    if (!c || !draws || !dirs || !poslgs || !lambda_nm) return set_error(c, PSFR_E_ARG, "NULL argument");
    if (ndraw < 1 || ndir < 1 || ndir > c->max_planes)
        return set_error(c, PSFR_E_CAPACITY, "ndraw=%d ndir=%d max_planes=%d", ndraw, ndir, c->max_planes);
    if (ngs < 1) return set_error(c, PSFR_E_ARG, "ngs=%d outside [1,%d]", ngs, kMaxGS);
    BatchOut o;
    o.out[kCube] = out_cube;
    o.out[kFit] = out_fit;
    return run_batch(c, ndraw, draws, ndir, dirs, ngs, ngs, poslgs, nlam, lambda_nm, 0, nullptr, false, o,
                     static_cast<cudaStream_t>(stream));
}

// the arguments of psfr_compute_groups and psfr_compute_field that run_batch does not check itself
static int check_groups(Ctx* c, int ndraw, const double* draws, const double* poslgs, int ndir, const double* dirs,
                        const double* lambda_nm, int ngroup, const int* group_end, const BatchOut& o) {
    if (!c || !draws || !dirs || !poslgs || !lambda_nm || (ngroup > 0 && !group_end))
        return set_error(c, PSFR_E_ARG, "NULL argument");
    if (ndraw < 1 || ndir < 1 || ndir > c->max_planes)
        return set_error(c, PSFR_E_CAPACITY, "ndraw=%d ndir=%d max_planes=%d", ndraw, ndir, c->max_planes);
    if (ngroup < 0) return set_error(c, PSFR_E_ARG, "ngroup=%d", ngroup);
    if (ngroup == 0 && o.any(kMean, kMeanBandEe))
        return set_error(c, PSFR_E_ARG, "exposure means need at least one exposure (ngroup=0)");
    for (int g = 0; g < ngroup; ++g)
        if (group_end[g] <= (g ? group_end[g - 1] : 0))
            return set_error(c, PSFR_E_ARG, "group_end[%d]=%d does not close a non-empty exposure", g, group_end[g]);
    if (ngroup > 0 && group_end[ngroup - 1] != ndraw)
        return set_error(c, PSFR_E_ARG, "group_end ends at %d, not at ndraw=%d", group_end[ngroup - 1], ndraw);
    return PSFR_OK;
}

int psfr_compute_groups(psfr_ctx* c, int ndraw, const double* draws, int npos, const double* poslgs, int ndir,
                        const double* dirs, int nlam, const double* lambda_nm, int ngroup, const int* group_end,
                        double* out_cube, double* out_fit, double* out_mean, double* out_mean_fit, void* stream) {
    BatchOut o;
    o.out[kCube] = out_cube;
    o.out[kFit] = out_fit;
    o.out[kMean] = out_mean;
    o.out[kMeanFit] = out_mean_fit;
    if (int rc = check_groups(c, ndraw, draws, poslgs, ndir, dirs, lambda_nm, ngroup, group_end, o)) return rc;
    return run_batch(c, ndraw, draws, ndir, dirs, 0, npos, poslgs, nlam, lambda_nm, ngroup, group_end, false, o,
                     static_cast<cudaStream_t>(stream));
}

int psfr_compute_field(psfr_ctx* c, int ndraw, const double* draws, int npos, const double* poslgs, int ndir,
                       const double* dirs, int nlam, const double* lambda_nm, int ngroup, const int* group_end,
                       double* out_cube, double* out_fit, double* out_mean, double* out_mean_fit, void* stream) {
    BatchOut o;
    o.out[kCube] = out_cube;
    o.out[kFit] = out_fit;
    o.out[kMean] = out_mean;
    o.out[kMeanFit] = out_mean_fit;
    if (int rc = check_groups(c, ndraw, draws, poslgs, ndir, dirs, lambda_nm, ngroup, group_end, o)) return rc;
    return run_batch(c, ndraw, draws, ndir, dirs, 0, npos, poslgs, nlam, lambda_nm, ngroup, group_end, true, o,
                     static_cast<cudaStream_t>(stream));
}

int psfr_compute_field_shapes(psfr_ctx* c, int ndraw, const double* draws, int npos, const double* poslgs, int ndir,
                              const double* dirs, int nlam, const double* lambda_nm, int ngroup, const int* group_end,
                              double* out_cube, double* out_fit, double* out_mean, double* out_mean_fit,
                              double* out_efit, double* out_mean_efit, void* stream) {
    BatchOut o;
    o.out[kCube] = out_cube;
    o.out[kFit] = out_fit;
    o.out[kEfit] = out_efit;
    o.out[kMean] = out_mean;
    o.out[kMeanFit] = out_mean_fit;
    o.out[kMeanEfit] = out_mean_efit;
    if (int rc = check_groups(c, ndraw, draws, poslgs, ndir, dirs, lambda_nm, ngroup, group_end, o)) return rc;
    return run_batch(c, ndraw, draws, ndir, dirs, 0, npos, poslgs, nlam, lambda_nm, ngroup, group_end, true, o,
                     static_cast<cudaStream_t>(stream));
}

int psfr_compute_energy(psfr_ctx* c, int field, int ndraw, const double* draws, int npos, const double* poslgs,
                        int ndir, const double* dirs, int nlam, const double* lambda_nm, int ngroup, const int* group_end,
                        int nrad, const double* radii_px, int nfrac, const double* fracs, double* out_cube,
                        double* out_fit, double* out_mean, double* out_mean_fit, double* out_efit,
                        double* out_mean_efit, double* out_ee, double* out_mean_ee, void* stream) {
    BatchOut o;
    o.out[kCube] = out_cube;
    o.out[kFit] = out_fit;
    o.out[kEfit] = out_efit;
    o.out[kEe] = out_ee;
    o.out[kMean] = out_mean;
    o.out[kMeanFit] = out_mean_fit;
    o.out[kMeanEfit] = out_mean_efit;
    o.out[kMeanEe] = out_mean_ee;
    o.nrad = nrad;
    o.nfrac = nfrac;
    if (int rc = check_groups(c, ndraw, draws, poslgs, ndir, dirs, lambda_nm, ngroup, group_end, o)) return rc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    PSFR_CUDA(c, cudaSetDevice(c->device));
    if (int rc = upload_ee_params(c, nrad, radii_px, nfrac, fracs, s)) return rc;
    return run_batch(c, ndraw, draws, ndir, dirs, 0, npos, poslgs, nlam, lambda_nm, ngroup, group_end, field != 0, o, s);
}

int psfr_compute_ao(psfr_ctx* c, int field, int ndraw, const double* draws, int npos, const double* poslgs, int ndir,
                    const double* dirs, int nlam, const double* lambda_nm, int ngroup, const int* group_end, int nrad,
                    const double* radii_px, int nfrac, const double* fracs, double* out_cube, double* out_fit,
                    double* out_mean, double* out_mean_fit, double* out_efit, double* out_mean_efit, double* out_ee,
                    double* out_mean_ee, double* out_strehl, double* out_var, void* stream) {
    BatchOut o;
    o.out[kCube] = out_cube;
    o.out[kFit] = out_fit;
    o.out[kEfit] = out_efit;
    o.out[kEe] = out_ee;
    o.out[kStrehl] = out_strehl;
    o.out[kVar] = out_var;
    o.out[kMean] = out_mean;
    o.out[kMeanFit] = out_mean_fit;
    o.out[kMeanEfit] = out_mean_efit;
    o.out[kMeanEe] = out_mean_ee;
    o.nrad = nrad;
    o.nfrac = nfrac;
    if (int rc = check_groups(c, ndraw, draws, poslgs, ndir, dirs, lambda_nm, ngroup, group_end, o)) return rc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    PSFR_CUDA(c, cudaSetDevice(c->device));
    if (int rc = upload_ee_params(c, nrad, radii_px, nfrac, fracs, s)) return rc;
    return run_batch(c, ndraw, draws, ndir, dirs, 0, npos, poslgs, nlam, lambda_nm, ngroup, group_end, field != 0, o, s);
}

int psfr_compute_bands(psfr_ctx* c, int field, int ndraw, const double* draws, int npos, const double* poslgs,
                       int ndir, const double* dirs, int nlam, const double* lambda_nm, int ngroup, const int* group_end,
                       int nrad, const double* radii_px, int nfrac, const double* fracs, double* out_cube,
                       double* out_fit, double* out_mean, double* out_mean_fit, double* out_efit, double* out_mean_efit,
                       double* out_ee, double* out_mean_ee, double* out_strehl, double* out_var, int nband,
                       const double* weights, double* out_band, double* out_band_fit, double* out_band_ee,
                       double* out_mean_band, double* out_mean_band_fit, double* out_mean_band_ee, void* stream) {
    BatchOut o;
    o.out[kCube] = out_cube;
    o.out[kFit] = out_fit;
    o.out[kEfit] = out_efit;
    o.out[kEe] = out_ee;
    o.out[kStrehl] = out_strehl;
    o.out[kVar] = out_var;
    o.out[kBand] = out_band;
    o.out[kBandFit] = out_band_fit;
    o.out[kBandEe] = out_band_ee;
    o.out[kMean] = out_mean;
    o.out[kMeanFit] = out_mean_fit;
    o.out[kMeanEfit] = out_mean_efit;
    o.out[kMeanEe] = out_mean_ee;
    o.out[kMeanBand] = out_mean_band;
    o.out[kMeanBandFit] = out_mean_band_fit;
    o.out[kMeanBandEe] = out_mean_band_ee;
    o.nrad = nrad;
    o.nfrac = nfrac;
    if (int rc = check_groups(c, ndraw, draws, poslgs, ndir, dirs, lambda_nm, ngroup, group_end, o)) return rc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    PSFR_CUDA(c, cudaSetDevice(c->device));
    const bool band_out = o.any(kBand, kBandEe) || o.any(kMeanBand, kMeanBandEe);
    if (band_out || nband != 0) {
        if (int rc = upload_band_weights(c, nband, nlam, weights, o.sums, s)) return rc;
        o.nband = nband;
    }
    if (band_out)
        if (int rc = alloc_band_staging(c)) return rc;
    if (int rc = upload_ee_params(c, nrad, radii_px, nfrac, fracs, s)) return rc;
    return run_batch(c, ndraw, draws, ndir, dirs, 0, npos, poslgs, nlam, lambda_nm, ngroup, group_end, field != 0, o, s);
}

int psfr_band_psf(psfr_ctx* c, int ncube, int nlam, int ny, int nx, const double* cubes, int nband,
                  const double* weights, double* out, void* stream) {
    if (!c || !cubes || !out) return set_error(c, PSFR_E_ARG, "NULL argument");
    if (ncube < 1 || nlam < 1 || ny < 1 || nx < 1)
        return set_error(c, PSFR_E_ARG, "ncube=%d nlam=%d ny=%d nx=%d", ncube, nlam, ny, nx);
    if ((long long)ny * nx > 0x7fffffff) return set_error(c, PSFR_E_ARG, "image %dx%d is too large", ny, nx);
    if (nlam > c->max_lambda) return set_error(c, PSFR_E_CAPACITY, "nlam=%d exceeds max_lambda=%d", nlam, c->max_lambda);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    PSFR_CUDA(c, cudaSetDevice(c->device));
    BandSums sums;
    int rc = upload_band_weights(c, nband, nlam, weights, sums, s);
    if (rc) return rc;
    const size_t per = (size_t)ny * nx, in_set = (size_t)nlam * per, out_set = (size_t)nband * per;
    const bool in_dev = is_device_ptr(cubes), out_dev = is_device_ptr(out);
    // host arrays go through d_cube (inputs) and d_cube2 (outputs), each of cap doubles
    const size_t cap = (size_t)c->max_planes * c->max_lambda * kPSF * kPSF;
    const size_t chunk = (in_dev && out_dev) ? (size_t)ncube : cap / std::max(in_set, out_set);
    if (chunk < 1) return set_error(c, PSFR_E_CAPACITY, "image set %dx%dx%d does not fit the staging buffer", nlam, ny, nx);
    for (size_t i0 = 0; i0 < (size_t)ncube; i0 += chunk) {
        const size_t n = std::min(chunk, (size_t)ncube - i0);
        const double* src = cubes + i0 * in_set;
        if (!in_dev) {
            if ((rc = to_device(c, c->d_cube, src, n * in_set * sizeof(double), s))) return rc;
            src = c->d_cube;
        }
        double* dst = out_dev ? out + i0 * out_set : c->d_cube2;
        if ((rc = run_band(c, (long long)n, nlam, (int)per, nband, sums, src, dst, s))) return rc;
        if (!out_dev && (rc = from_device(c, out + i0 * out_set, dst, n * out_set * sizeof(double), s))) return rc;
    }
    return PSFR_OK;
}

int psfr_mean_refit(psfr_ctx* c, int ncube, int nlam, const double* cubes, double* out_mean, double* out_fit,
                    void* stream) {
    if (!c || !cubes) return set_error(c, PSFR_E_ARG, "NULL argument");
    if (ncube < 1 || nlam < 1 || nlam > c->max_lambda) return set_error(c, PSFR_E_ARG, "ncube=%d nlam=%d", ncube, nlam);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    PSFR_CUDA(c, cudaSetDevice(c->device));
    const size_t elems = (size_t)nlam * kPSF * kPSF;
    const size_t cap = (size_t)c->max_planes * c->max_lambda * kPSF * kPSF;
    double* mean = c->d_cube2;
    int rc = PSFR_OK;
    if (is_device_ptr(cubes)) {
        rc = run_mean(c, ncube, (int)elems, cubes, mean, s, true, true, ncube);
        if (rc) return rc;
    } else {
        // host cubes stream through the staging buffer in slabs; the running sum keeps the
        // input order, so the result does not depend on the slab size
        const int slab = (int)std::max<size_t>(1, cap / elems);
        if (elems > cap) return set_error(c, PSFR_E_CAPACITY, "nlam=%d exceeds the staging capacity", nlam);
        for (int k0 = 0; k0 < ncube; k0 += slab) {
            const int n = std::min(slab, ncube - k0);
            rc = to_device(c, c->d_cube, cubes + (size_t)k0 * elems, (size_t)n * elems * sizeof(double), s);
            if (rc) return rc;
            rc = run_mean(c, n, (int)elems, c->d_cube, mean, s, k0 == 0, k0 + n == ncube, ncube);
            if (rc) return rc;
            if (k0 + n < ncube) PSFR_CUDA(c, cudaStreamSynchronize(s));   // pageable source may be reused
        }
    }
    if (out_fit) {
        double* fit = is_device_ptr(out_fit) ? out_fit : c->d_fit;
        rc = run_fit(c, nlam, kPSF, kPSF, mean, fit, s);
        if (rc) return rc;
        if (fit != out_fit) {
            rc = from_device(c, out_fit, fit, (size_t)nlam * PSFR_FIT_NPAR * sizeof(double), s);
            if (rc) return rc;
        }
    }
    if (out_mean) return from_device(c, out_mean, mean, elems * sizeof(double), s);
    return PSFR_OK;
}

int psfr_polyfit(psfr_ctx* c, int nseries, int nlam, const double* lambda_nm, int deg, const double* y,
                 double* coef, void* stream) {
    if (!c || !lambda_nm || !y || !coef) return set_error(c, PSFR_E_ARG, "NULL argument");
    if (nseries < 1 || nlam < 2 || deg < 0) return set_error(c, PSFR_E_ARG, "nseries=%d nlam=%d deg=%d", nseries, nlam, deg);
    if ((size_t)nseries * (nlam + deg + 1) + nlam > 65536)
        return set_error(c, PSFR_E_CAPACITY, "polyfit batch too large");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    PSFR_CUDA(c, cudaSetDevice(c->device));
    std::vector<double> lam;
    int rc = small_to_host(c, lam, lambda_nm, nlam, s);
    if (rc) return rc;
    for (auto& v : lam) v = (v - 475) / (935 - 475) - 0.5;        // _norm_lbda, psfrec.py:1213-1215
    double* d_lb = c->d_poly;
    double* d_y = d_lb + nlam;
    double* d_c = d_y + (size_t)nseries * nlam;
    PSFR_CUDA(c, cudaMemcpyAsync(d_lb, lam.data(), nlam * sizeof(double), cudaMemcpyHostToDevice, s));
    PSFR_CUDA(c, cudaStreamSynchronize(s));
    rc = to_device(c, d_y, y, (size_t)nseries * nlam * sizeof(double), s);
    if (rc) return rc;
    rc = run_polyfit(c, nseries, nlam, deg, d_lb, d_y, d_c, s);
    if (rc) return rc;
    return from_device(c, coef, d_c, (size_t)nseries * (deg + 1) * sizeof(double), s);
}

int psfr_get_otf(psfr_ctx* c, double* out) {
    if (!c || !out) return set_error(c, PSFR_E_ARG, "NULL argument");
    PSFR_CUDA(c, cudaSetDevice(c->device));
    return from_device(c, out, c->d_otf, (size_t)c->rows * c->N * sizeof(double), 0);
}

int psfr_get_structure_function(psfr_ctx* c, int plane, double* out) {
    if (!c || !out) return set_error(c, PSFR_E_ARG, "NULL argument");
    if (plane < 0 || plane >= c->planes_struct) return set_error(c, PSFR_E_STATE, "plane %d not available", plane);
    PSFR_CUDA(c, cudaSetDevice(c->device));
    return from_device(c, out, c->d_dphi + (size_t)plane * c->rows * c->N, (size_t)c->rows * c->N * sizeof(double), 0);
}

int psfr_debug_exp(psfr_ctx* c, int n, const double* x, double* y) {
    if (!c || !x || !y) return set_error(c, PSFR_E_ARG, "NULL argument");
    if (n < 1 || (size_t)n > (size_t)c->max_planes * c->max_lambda * kPSF * kPSF)
        return set_error(c, PSFR_E_CAPACITY, "n=%d exceeds the staging buffer", n);
    PSFR_CUDA(c, cudaSetDevice(c->device));
    int rc = to_device(c, c->d_cube, x, (size_t)n * sizeof(double), 0);
    if (rc) return rc;
    if ((rc = run_debug_exp(c, c->d_cube, c->d_cube2, n, 0))) return rc;
    return from_device(c, y, c->d_cube2, (size_t)n * sizeof(double), 0);
}

int psfr_set_option(psfr_ctx* c, int key, double value) {
    if (!c) return set_error(c, PSFR_E_ARG, "NULL context");
    switch (key) {
        case PSFR_OPT_EXP_CUT:
            if (!(value > 0)) return set_error(c, PSFR_E_ARG, "exp cut must be positive (got %g)", value);
            c->exp_cut = value;
            return PSFR_OK;
        case PSFR_OPT_EXP_GRADE:
            if (!(value > 0)) return set_error(c, PSFR_E_ARG, "exp grade must be positive (got %g)", value);
            c->exp_grade = value;
            return PSFR_OK;
        case PSFR_OPT_ROW_KERNEL:
            if (value != 1.0 && value != 2.0) return set_error(c, PSFR_E_ARG, "row kernel must be 1 or 2 (got %g)", value);
            c->row_kernel = (int)value;
            return PSFR_OK;
        case PSFR_OPT_F32_ROWS:
            if (!(value > 0)) return set_error(c, PSFR_E_ARG, "f32 row threshold must be positive (got %g)", value);
            c->f32_rows = value;
            return PSFR_OK;
        default:
            return set_error(c, PSFR_E_ARG, "unknown option %d", key);
    }
}

long long psfr_kernel_launches(const psfr_ctx* c) { return c ? c->launches : 0; }

int psfr_get_info(const psfr_ctx* c, int key, double* out) {
    if (!c || !out) return PSFR_E_ARG;
    switch (key) {
        case PSFR_INFO_Y_COLS: *out = kNC; return PSFR_OK;
        case PSFR_INFO_EXP_CUT: *out = c->exp_cut; return PSFR_OK;
        case PSFR_INFO_EXP_GRADE: *out = c->exp_grade; return PSFR_OK;
        case PSFR_INFO_F32_ROWS: *out = c->f32_rows; return PSFR_OK;
        case PSFR_INFO_ROW_KERNEL: *out = c->row_kernel; return PSFR_OK;
        case PSFR_INFO_MAX_PLANES: *out = c->max_planes; return PSFR_OK;
        case PSFR_INFO_MAX_LAMBDA: *out = c->max_lambda; return PSFR_OK;
        case PSFR_INFO_DIM: *out = c->N; return PSFR_OK;
        default: return PSFR_E_ARG;
    }
}

int psfr_last_hot_timing(psfr_ctx* c, double* ms, int* launches, long long* psfs) {
    if (!c) return set_error(c, PSFR_E_ARG, "NULL context");
    PSFR_CUDA(c, cudaSetDevice(c->device));
    HotTimer* t = timer_of(c);
    double total = 0.0;
    for (int i = 0; i < t->n; ++i) {
        PSFR_CUDA(c, cudaEventSynchronize(t->ev[2 * i + 1]));
        float e = 0.f;
        PSFR_CUDA(c, cudaEventElapsedTime(&e, t->ev[2 * i], t->ev[2 * i + 1]));
        total += e;
    }
    if (ms) *ms = total;
    if (launches) *launches = c->hot_launches;
    if (psfs) *psfs = c->hot_psfs;
    return PSFR_OK;
}

}  // extern "C"

// hook used by psfr_hot.cu to bracket the row kernel with events
namespace psfr {
int hot_event(Ctx* c, int which, cudaStream_t s) {
    HotTimer* t = reinterpret_cast<HotTimer*>(c->ev_hot0);
    if (!t) return PSFR_OK;
    if (which == 0) {
        if (t->n >= kMaxHotEvents) return PSFR_OK;
        PSFR_CUDA(c, cudaEventRecord(t->ev[2 * t->n], s));
    } else {
        if (t->n >= kMaxHotEvents) return PSFR_OK;
        PSFR_CUDA(c, cudaEventRecord(t->ev[2 * t->n + 1], s));
        t->n++;
    }
    return PSFR_OK;
}
}  // namespace psfr
