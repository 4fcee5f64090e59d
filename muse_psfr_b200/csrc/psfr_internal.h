// Internal declarations shared by the translation units of libpsfr_b200.so.
#pragma once
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cuda_runtime.h>
#include <vector>
#include "../../include/psfr.h"

namespace psfr {

constexpr int kR3 = 20;                 // the warp transform has length 64*R3 = 1280
constexpr int kNB = 64 * kR3;           // base line length 1280
// Grid sizes: N = NF * 1280 with NF = 1 (dim 1280, compute_psf) or NF = 2 (dim 2560, BASELINE
// config 5).  A length-N line is NF interleaved 1280-point warp transforms plus one radix-NF
// combine (decimation in time).
template <int NF>
struct Dim {
    static_assert(NF == 1 || NF == 2, "dim must be 1280 or 2560");
    static constexpr int N = NF * kNB;
    static constexpr int NH = N / 2;
    static constexpr int Rows = NH + 2;      // half-plane rows 0..N/2 plus one zero pad row
    static constexpr int Pairs = Rows / 2;   // row pairs
};
// Group row kernel (psfr_hot2.cu).  A transform of 1280 points is split as kG1 x kG2 x 8 and belongs to
// a group of kGThreads = 8 kG2 threads; kGGroups groups share a CTA.  Two geometries are compiled in:
//   PSFR_G_GEOM 1 (default): 10 x 16 x 8, four groups of 128 threads (16 warps; passes of 128 / 80 / 80 threads)
//   PSFR_G_GEOM 0          :  8 x 20 x 8, three groups of 160 threads (15 warps; 160 / 64 / 80)
// Index maps: n = n1*kGThreads + n2*8 + n3,  k = k1 + kG1*k2 + 160*k3.
// Tables: pass-1 twiddles w_160^(n2 k1) [kG2][kG1 - 1], and per wavelength
//  * the record of the pruned third pass for thread t: output k (a kept frequency or its mirror), as the
//    Horner base w = w_1280^k in FP64 and FP32, the offset of its row k1*kGS1 + k2 in the transform buffer and
//    the kept frequency (column of Y) the pair (t, t xor 1) = (X[k], X[-k]) belongs to;
//  * the rows (k1, k2) pass 3 reads, as one kG2-bit mask per k1: pass 2 stores only those.
#ifndef PSFR_G_GEOM
#define PSFR_G_GEOM 1
#endif
#if PSFR_G_GEOM == 0
constexpr int kG1 = 8, kG2 = 20, kGGroups = 3;
#else
constexpr int kG1 = 10, kG2 = 16, kGGroups = 4;
#endif
constexpr int kGThreads = 8 * kG2;       // threads per group = inputs per pass-1 butterfly stride
constexpr int kGS2 = kG2 + 1;            // stride of n3 in a transform buffer (odd)
constexpr int kGS1 = 8 * kGS2 + 1;       // stride of k1
constexpr int kGroupTw = kG2 * (kG1 - 1);
constexpr int kGMaskStride = 16;         // uint32 masks per wavelength (kG1 used)
static_assert(kG1 * kG2 * 8 == kNB && kG1 <= kGMaskStride, "group geometry");
struct alignas(16) GroupP3 {
    double2 w;       // w_1280^(k mod 1280): Horner base of the 1280-point (sub-)transform
    double2 wc;      // w_N^k: combine twiddle of the two interleaved sub-transforms (dim 2560)
    float2 w32;
    uint32_t base;
    uint32_t col;
};
static_assert(sizeof(GroupP3) == 48, "GroupP3 is loaded as three 16-byte words");
constexpr int kAO = PSFR_AO_DIM;        // 80
constexpr int kPSF = PSFR_PSF_DIM;      // 40
constexpr int kNS = 2 * kPSF;           // 80 sampled rows / columns per PSF
// The sampled frequencies with a non-zero bilinear weight are closed under negation (up to the single
// sample -npix/2), and the PSF is point-symmetric: P[-ky][-kx] = P[ky][kx].  The row pass therefore
// keeps only the kNC = 40 frequencies k <= 0 (set_lambda_tables) and the column pass fills the
// mirrored samples from its outputs at -ky.
constexpr int kNC = kPSF;
constexpr int kKW = 41;                 // Moffat kernel width
constexpr int kMaxGS = 4;
constexpr int kMaxDir = 256;            // field directions per draw
constexpr int kMaxLambdaCap = 4096;
constexpr int kEeMaxRecord = PSFR_EE_MAX_RADII + 1 + PSFR_EE_MAX_FRACTIONS;   // doubles per EE record, at most

// layout of the small scratch array d_misc (doubles)
constexpr int kMiscDirs = 0;            // [2][ndir]
constexpr int kMiscPos = 1024;          // [2][ngs]
constexpr int kMiscTwo = 2048;          // the constant 2.0
constexpr int kMiscMuse = 4096;         // gamma[nlam], beta[nlam] of the MUSE kernels
constexpr int kMiscCentre = 16384;      // [max_planes] structure-function centres
inline int misc_alpha_tt(int max_planes) { return kMiscCentre + max_planes; }   // [max_planes]
// int [2 * max_planes] exposure segments of one chunk (psfr_compute_groups, run_group_mean)
inline int misc_groups(int max_planes) { return kMiscCentre + 2 * max_planes + 64; }
inline int misc_size(int max_planes) { return misc_groups(max_planes) + max_planes + 64; }

struct Ctx {
    int device = 0;
    int NF = 1;                  // N / 1280
    int N = kNB;                 // PSD grid size (dim)
    int NH = kNB / 2;            // N / 2
    int rows = kNB / 2 + 2;      // half-plane rows incl. the zero pad row
    int pairs = kNB / 4 + 1;     // row pairs
    int max_planes = 0;
    int max_lambda = 0;
    int sm_count = 148;
    long long launches = 0;
    bool geometry_set = false;
    int planes_loaded = 0;       // planes whose PSD sits in d_psd
    int planes_struct = 0;       // planes whose structure function sits in d_dphi
    double pup_sum = 0;
    double otf_sum = 0;          // sum of the telescope OTF over the full N x N grid (run_otf_sum): Strehl denominator

    double2* d_tw = nullptr;     // twiddles: TW1 then TW2
    double2* d_twc = nullptr;    // [1280] combine twiddles exp(+2 pi i k / N) (NF = 2)
    double* d_pup = nullptr;     // [N/2][N/2] pupil as doubles
    double* d_otf = nullptr;     // [rows][N] telescope OTF half-plane (centred, pad row zero)
    double* d_geom = nullptr;    // f, f_x, f_y: 3 x 80 x 80
    double* d_psd = nullptr;     // [max_planes][N][N]
    double* d_psdq = nullptr;    // [max_planes][N/2][N/2] fitting PSD, one mirror quadrant, unscaled (fused path)
    double2* d_bt = nullptr;     // [max_planes][N][rows] transposed row-pass output (full mode)
    double* d_dphi = nullptr;    // [max_planes][rows][N] structure function (transposed half-plane)
    double* d_dmin = nullptr;    // [max_planes][rows] smallest structure-function value of each row
    float* d_dphi32 = nullptr;   // [max_planes][rows][N] single-precision copy of d_dphi (dim 1280: block grading + FP32 row pairs)
    float* d_otf32 = nullptr;    // [rows][N] single-precision copy of d_otf
    float2* d_tw32 = nullptr;    // twiddles of d_tw rounded to single precision
    double2* d_twg = nullptr;    // [kGroupTw] pass-1 twiddles of the group row kernel
    float2* d_twg32 = nullptr;   // the same in single precision
    GroupP3* d_p3 = nullptr;     // [max_lambda][2 kNC] pass-3 records of the group row kernel
    uint32_t* d_p2mask = nullptr; // [max_lambda][8] rows (k1, k2) that pass 3 reads
    double* d_csort = nullptr;   // [max_lambda] c_lambda in descending order (unit classes of the row kernel)
    int* d_lorder = nullptr;     // [max_lambda] wavelength index of sorted position i
    int* d_counter = nullptr;    // work counter of the persistent stage-B row kernel
    double exp_cut = 45.0;       // OTF entries below exp(-exp_cut) are flushed to zero (PSFR_OPT_EXP_CUT)
    double exp_grade = 20.0;     // blocks entirely below exp(-exp_grade) use the single-precision exp (PSFR_OPT_EXP_GRADE)
    double f32_rows = 25.0;      // row pairs entirely below exp(-f32_rows) run in single precision (PSFR_OPT_F32_ROWS)
    int row_kernel = 2;          // 2 group_rows_kernel (psfr_hot2.cu), 1 hot_rows_kernel (PSFR_OPT_ROW_KERNEL)
    double2* d_ybuf = nullptr;   // [max_planes*max_lambda][kNC][rows] pruned row-pass output
    double2* d_wsamp = nullptr;  // [max_lambda][2][kNS] combine twiddles of the sampled outputs / mirrors (NF = 2)
    double2* d_wcol = nullptr;   // [max_lambda][2][kNC] the same for the kept row-pass frequencies (NF = 2)
    uint16_t* d_kcol = nullptr;  // [max_lambda][kNC] row-pass frequencies kept in d_ybuf
    short2* d_xmap = nullptr;    // [max_lambda][kNC] sample index whose frequency is +kcol / -kcol (-1: none)
    double* d_samp = nullptr;    // [max_draws*max_lambda][kNS][kNS] PSF samples
    double* d_ao = nullptr;      // [max_planes][80][80] AO-zone PSD (centred, reference orientation)
    double* d_draws = nullptr;   // [max_planes][PSFR_DRAW_NPAR]
    double* d_misc = nullptr;    // small: dirs, poslgs, lambda tables ...
    double* d_lam = nullptr;     // [max_lambda] c_lambda = 0.5 (2 pi/lambda_nm)^2
    uint16_t* d_kidx = nullptr;  // [max_lambda][kNS] sampled output indices (shifted by N/2)
    ushort2* d_kaddr = nullptr;  // [max_lambda][kNC] dump addresses nat_addr(k mod 1280), nat_addr(-k mod 1280) of d_kcol
    double* d_frac = nullptr;    // [max_lambda][kPSF] bilinear fractions
    double* d_kern_tt = nullptr; // [max_planes][41][41] normalised tip-tilt kernels
    double* d_kern_mu = nullptr; // [max_lambda][41][41] normalised MUSE kernels
    double2* d_khat_tt = nullptr; // [max_planes][80][41] half spectra of the tip-tilt kernels
    double2* d_khat_mu = nullptr; // [max_lambda][80][41] half spectra of the MUSE kernels
    double* d_cube = nullptr;    // [max_planes*max_lambda][40][40] staging for cubes
    double* d_cube2 = nullptr;   // second staging buffer
    double* d_cube3 = nullptr;   // third staging buffer (double-buffered device -> host copies)
    double* d_fit = nullptr;     // [max_planes*max_lambda][PSFR_FIT_NPAR]
    double* d_fit2 = nullptr;    // second fit buffer (double-buffered device -> host copies)
    double* d_carry = nullptr;   // [max_planes*max_lambda][40][40] unnormalised sum of the exposure open at a chunk
                                 // edge: [ndir][nlam][40][40] in psfr_compute_field, and ndir <= max_planes
    double* d_mean[2] = {nullptr, nullptr};  // [max_planes*max_lambda][40][40] exposure means finished in a chunk
    double* d_mfit[2] = {nullptr, nullptr};  // [max_planes*max_lambda][PSFR_FIT_NPAR] their fits
    double* d_efit = nullptr;    // [max_planes*max_lambda][PSFR_EFIT_NPAR] elliptical records (double-buffered
    double* d_efit2 = nullptr;   // with d_efit2 as d_fit / d_fit2)
    double* d_mefit[2] = {nullptr, nullptr};  // [max_planes*max_lambda][PSFR_EFIT_NPAR] elliptical fits of the means
    double* d_ee[2] = {nullptr, nullptr};     // [max_planes*max_lambda][kEeMaxRecord] encircled-energy records
    double* d_mee[2] = {nullptr, nullptr};    // the same for the exposure means (double-buffered as d_mean)
    double* d_eepar = nullptr;   // [PSFR_EE_MAX_RADII + PSFR_EE_MAX_FRACTIONS] radii then fractions of the call
    double* d_eecen = nullptr;   // [max_planes*max_lambda][2] staging for host centres (psfr_encircled_energy)
    std::vector<double> ee_par;  // host copy of d_eepar's contents (outlives the asynchronous upload)
    double* d_strehl[2] = {nullptr, nullptr}; // [max_planes*max_lambda] Strehl ratios (double-buffered as d_ee)
    double* d_var[2] = {nullptr, nullptr};    // [max_planes][PSFR_VAR_NPAR] variance records (double-buffered)
    // band images (DESIGN.md 5.6), allocated by the first call that needs them (alloc_band_staging): weights
    // [max_lambda][PSFR_MAX_BANDS] k-major, and per staging set b images [max_planes * PSFR_MAX_BANDS][40][40], fit and
    // EE records of the per-draw bands and of the exposure means' bands
    double* d_bandw = nullptr;
    std::vector<double> band_w;  // host copy of d_bandw's contents (outlives the asynchronous upload)
    double* d_band[2] = {nullptr, nullptr};
    double* d_bfit[2] = {nullptr, nullptr};
    double* d_bee[2] = {nullptr, nullptr};
    double* d_mband[2] = {nullptr, nullptr};
    double* d_mbfit[2] = {nullptr, nullptr};
    double* d_mbee[2] = {nullptr, nullptr};
    cudaStream_t copy_stream = nullptr;      // device -> host copies of finished chunks
    cudaEvent_t ev_done[2] = {nullptr, nullptr};    // chunk results ready (compute stream)
    cudaEvent_t ev_copied[2] = {nullptr, nullptr};  // chunk results copied out (copy stream)
    double* d_poly = nullptr;    // polynomial fit scratch
    void* h_pinned = nullptr;    // pinned bounce buffer
    size_t h_pinned_bytes = 0;

    cudaEvent_t ev_hot0 = nullptr;
    int hot_launches = 0;
    long long hot_psfs = 0;

    // kernels whose dynamic shared-memory limit has been raised on THIS device (the attribute is
    // per device, so a process-wide flag would break a second context on another GPU)
    const void* smem_funcs[64] = {nullptr};
    size_t smem_bytes[64] = {0};
    int n_smem_funcs = 0;

    // wavelengths whose tables (set_lambda_tables) / MUSE kernels (run_build_kernels) currently sit on the
    // device: a call with the same wavelengths skips the rebuild and its host synchronisation
    std::vector<double> lam_tables, lam_kernels;

    char err[512] = {0};
};

int set_error(Ctx* c, int code, const char* fmt, ...);

// Raise cudaFuncAttributeMaxDynamicSharedMemorySize of `func` to at least `bytes`, never lower it.  The attribute
// belongs to the function on the device, shared by every context of the process, so lowering it would break a
// context that cached a larger value.
template <class F>
inline cudaError_t raise_dynamic_smem(F* func, size_t bytes) {
    cudaFuncAttributes a;
    cudaError_t e = cudaFuncGetAttributes(&a, func);
    if (e != cudaSuccess || (size_t)a.maxDynamicSharedSizeBytes >= bytes) return e;
    return cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

// raise_dynamic_smem once per context and size: the attribute only grows, so a cached size stays valid
template <class F>
inline int ensure_dynamic_smem(Ctx* c, F* func, size_t bytes) {
    const void* key = reinterpret_cast<const void*>(func);
    for (int i = 0; i < c->n_smem_funcs; ++i)
        if (c->smem_funcs[i] == key) {
            if (c->smem_bytes[i] >= bytes) return PSFR_OK;
            cudaError_t e = raise_dynamic_smem(func, bytes);
            if (e != cudaSuccess) return set_error(c, PSFR_E_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
            c->smem_bytes[i] = bytes;
            return PSFR_OK;
        }
    if (bytes > 48 * 1024) {
        cudaError_t e = raise_dynamic_smem(func, bytes);
        if (e != cudaSuccess) return set_error(c, PSFR_E_CUDA, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    }
    if (c->n_smem_funcs < 64) {
        c->smem_funcs[c->n_smem_funcs] = key;
        c->smem_bytes[c->n_smem_funcs++] = bytes > 48 * 1024 ? bytes : 48 * 1024;
    }
    return PSFR_OK;
}

#define PSFR_CUDA(ctx, call)                                                             \
    do {                                                                                 \
        cudaError_t e__ = (call);                                                        \
        if (e__ != cudaSuccess)                                                          \
            return psfr::set_error((ctx), PSFR_E_CUDA, "%s failed at %s:%d: %s", #call,  \
                                   __FILE__, __LINE__, cudaGetErrorString(e__));         \
    } while (0)

#define PSFR_LAUNCH_CHECK(ctx)                                                           \
    do {                                                                                 \
        (ctx)->launches++;                                                               \
        cudaError_t e__ = cudaGetLastError();                                            \
        if (e__ != cudaSuccess)                                                          \
            return psfr::set_error((ctx), PSFR_E_CUDA, "kernel launch failed at %s:%d: %s", \
                                   __FILE__, __LINE__, cudaGetErrorString(e__));         \
    } while (0)

// ---- psfr_passes.cu: generic row/column FFT passes ----------------------------------
// stage A (PSD -> D_unit) on planes [0, nplanes) of the workspace; from_quadrant: the PSD is the
// quadrant form (d_psdq + d_ao) written by run_psd(..., full = false) instead of d_psd
int run_structure_function(Ctx* c, int nplanes, cudaStream_t s, bool from_quadrant = false, int ndir = 1);
// full-grid stage B: plane `plane`, exponent scale clam -> d_psd-sized output in `out_dev`
int run_full_psf(Ctx* c, int plane, double clam, double* out_dev, cudaStream_t s);
// context init: pupil + telescope OTF
int run_build_otf(Ctx* c, cudaStream_t s);
// test hook: y = fast_exp(x) elementwise
int run_debug_exp(Ctx* c, const double* x_dev, double* y_dev, int n, cudaStream_t s);

// ---- psfr_hot.cu: pruned stage B ----------------------------------------------------
// row pass with fused exp(-c D) * OTF for nplanes x nlam, then pruned column pass summing
// the ndir planes of each draw into d_samp [ndraw*nlam][80][80]
int run_pruned_psf(Ctx* c, int ndraw, int ndir, int nlam, cudaStream_t s);
// psfr_hot2.cu: the row pass by groups of threads (one transform per 128-thread group, data in shared memory)
int run_group_rows(Ctx* c, int nplanes, int nlam, cudaStream_t s);

// ---- psfr_psd.cu ---------------------------------------------------------------------
// uses d_draws, d_misc.  full: write the N x N PSD of every plane into d_psd (simul_psd_wfm);
// otherwise only the AO zones (d_ao) and one mirror quadrant of the fitting PSD (d_psdq)
// ngs: guide stars of every draw, or 0 for each draw's own count (slot PSFR_DRAW_NGS); the positions
// are the first ngs columns of the [2][npos] table at d_misc + kMiscPos
int run_psd(Ctx* c, int ndraw, int ndir, int ngs, int npos, cudaStream_t s, bool full = true);

// residual-phase variance record [ndraw * ndir][PSFR_VAR_NPAR] of the planes whose quadrant-form PSD run_psd(...,
// full = false) left in d_psdq / d_ao (same draws, directions and guide stars)
int run_var(Ctx* c, int ndraw, int ndir, int ngs, int npos, double* out_dev, cudaStream_t s);

// ---- psfr_ao.cu ----------------------------------------------------------------------
// context init, after run_build_otf: c->otf_sum = sum of the telescope OTF over the full grid (one sync)
int run_otf_sum(Ctx* c, cudaStream_t s);
// Strehl ratio of the nimg PSFs run_pruned_psf left in d_samp (raw samples, before clip and normalisation)
int run_strehl(Ctx* c, int nimg, double* out_dev, cudaStream_t s);

// ---- psfr_band.cu --------------------------------------------------------------------
// W_b = sum_k w[b][k] in ascending k of every band; unused slots hold 1
struct BandSums {
    double w[PSFR_MAX_BANDS];
};
// band images out [nset][nband][npix] of the image sets in [nset][nlam][npix]: (sum_k fma(w[b][k], in[k], .)) / W_b in
// ascending k, with the weights c->d_bandw [nlam][PSFR_MAX_BANDS] holds
int run_band(Ctx* c, long long nset, int nlam, int npix, int nband, const BandSums& sums, const double* in_dev,
             double* out_dev, cudaStream_t s);

// ---- psfr_plane.cu -------------------------------------------------------------------
// moffat_kernels_kernel divides by pi * gamma^2, evaluated as (pi * gamma) * gamma: the kernel is finite for
// every gamma that leaves that product a finite, normal double (|gamma| in about [8.5e-155, 7.5e153])
inline bool moffat_width_ok(double gamma) { return std::isnormal(3.141592653589793 * gamma * gamma); }
int run_build_kernels(Ctx* c, int ndraw, int nlam, const double* lambda_nm_host, bool tt, bool mu,
                      cudaStream_t s);
// samples -> 40x40 resampled + normalised cube (psf_muse tail)
int run_resample(Ctx* c, int nimg, int nlam, double* cube_dev, cudaStream_t s);
// psfr_conv.cu: spectra of nk 41x41 kernels, and the two FFT convolutions of every image
int run_kernel_spectra(Ctx* c, int nk, const double* kern_dev, double2* khat_dev, cudaStream_t s);
int run_fft_convolve(Ctx* c, int ndraw, int ndir, int nlam, const double* in_dev, double* out_dev, cudaStream_t s);
// two Moffat convolutions; img index = (draw*ndir + k)*nlam + lam, one tip-tilt kernel per draw (ndir = 1
// unless every field position of a draw keeps its own image, psfr_compute_field)
int run_convolve(Ctx* c, int ndraw, int ndir, int nlam, const double* in_dev, double* out_dev, cudaStream_t s);
int run_fit(Ctx* c, int nimg, int ny, int nx, const double* img_dev, double* fit_dev, cudaStream_t s);
// elliptical fit of every image from its circular record circ_dev [nimg][PSFR_FIT_NPAR]
int run_efit(Ctx* c, int nimg, int ny, int nx, const double* img_dev, const double* circ_dev, double* efit_dev,
             cudaStream_t s);
// star fits (DESIGN.md 5.7): weights w_dev may be NULL (all 1); back_dev [nimg][PSFR_BACK_NPAR]; the elliptical one
// starts from run_star_fit's records circ_dev / circ_back_dev (back_dev may be circ_back_dev)
int check_star_fit_size(Ctx* c, int ny, int nx, bool elliptical);
int run_star_fit(Ctx* c, int nimg, int ny, int nx, const double* img_dev, const double* w_dev, bool fit_back,
                 double* fit_dev, double* back_dev, cudaStream_t s);
int run_star_efit(Ctx* c, int nimg, int ny, int nx, const double* img_dev, const double* w_dev, bool fit_back,
                  const double* circ_dev, const double* circ_back_dev, double* efit_dev, double* back_dev,
                  cudaStream_t s);
// template fit (DESIGN.md 5.8): tpl_dev [ntpl][ty][tx]; image i of the call uses template (first + i) % ntpl;
// model_dev [nimg][ny][nx] or NULL
int check_template_fit_size(Ctx* c, int ny, int nx, int ty, int tx);
int run_template_fit(Ctx* c, int nimg, int ny, int nx, const double* img_dev, const double* w_dev, int ntpl, int ty,
                     int tx, const double* tpl_dev, long long first, bool fit_back, double* fit_dev, double* model_dev,
                     cudaStream_t s);
// psfr_energy.cu: encircled-energy record [nimg][nrad + 1 + nfrac] of every image, radii and fractions from
// d_eepar, centres_dev [nimg][2] (row, column) or nullptr for (ny / 2, nx / 2)
int run_ee(Ctx* c, int nimg, int ny, int nx, const double* img_dev, const double* centres_dev, int nrad, int nfrac,
           double* out_dev, cudaStream_t s);
// out = (running sum of the cubes) ; first: start from zero, last: divide by ntotal
int run_mean(Ctx* c, int ncube, int plane_elems, const double* cubes_dev, double* out_dev,
             cudaStream_t s, bool first, bool last, int ntotal);
// segmented time mean of the cubes of a chunk, exposure by exposure: seg[2k] is the end (chunk-local
// draw index) of the k-th of nseg exposures that touch the chunk, seg[2k + 1] its draw count when it ends in
// this chunk and 0 when it stays open.  carry_in: the first exposure continues the sum left in d_carry.
// Finished means go to out_dev one after another; the open sum goes back to d_carry.
int run_group_mean(Ctx* c, int plane_elems, const double* cubes_dev, const int* seg_dev, int nseg,
                   bool carry_in, double* out_dev, cudaStream_t s);
int run_polyfit(Ctx* c, int nseries, int nlam, int deg, const double* lb_dev, const double* y_dev,
                double* coef_dev, cudaStream_t s);

}  // namespace psfr
