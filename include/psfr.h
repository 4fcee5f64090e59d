/* psfr.h - C ABI of the B200-native PSF-reconstruction hot path (libpsfr_b200.so).
 *
 * The reference (musevlt/muse-psfr) has no FFI: the path sits behind plain Python
 * functions in muse_psfr/psfrec.py.  Each entry point below cites the reference
 * function it replaces; the Python host (muse_psfr_b200/psfrec.py) binds them with
 * ctypes and keeps the reference's signatures.  INTEGRATION.md shows the stub a
 * maintainer of the reference would add.
 *
 * Conventions
 *  - every function returns 0 on success, a negative PSFR_E_* code on failure and
 *    never throws; psfr_last_error() gives the message of the last failure;
 *  - all arrays are C-contiguous FP64 unless stated; every data pointer may be a HOST
 *    pointer (pageable or pinned) or a DEVICE pointer on the context's GPU - the
 *    library detects which and stages copies on the given stream;
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); all
 *    work is stream-ordered, host outputs are complete when the call returns,
 *    device outputs when the stream reaches that point;
 *  - one context per GPU, not thread-safe; the context owns twiddles, the telescope
 *    OTF, geometry tables and all workspaces;
 *  - there is no CPU fallback: without a CUDA device psfr_create fails.
 */
#ifndef PSFR_H
#define PSFR_H

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define PSFR_API __attribute__((visibility("default")))
#else
#define PSFR_API
#endif

typedef struct psfr_ctx psfr_ctx;

enum {
    PSFR_OK = 0,
    PSFR_E_CUDA = -1,      /* CUDA runtime error (message in psfr_last_error) */
    PSFR_E_ARG = -2,       /* invalid argument */
    PSFR_E_UNSUPPORTED = -3, /* e.g. dim other than 1280 / 2560, more than PSFR_MAX_LAYERS layers */
    PSFR_E_CAPACITY = -4,  /* batch larger than the context was created for */
    PSFR_E_STATE = -5      /* call order (e.g. geometry not set) */
};

/* Size of the AO-corrected zone (Dimpup*2, psfrec.py:103,138) and of the final PSF. */
#define PSFR_AO_DIM 80
#define PSFR_PSF_DIM 40

/* Per-draw parameter record (array of doubles, one row per draw).
 * Filled by the host exactly as simul_psd_wfm / convolve_final_psf derive them. */
#define PSFR_MAX_LAYERS 8    /* the reference works for 1 or 2 layers only (wind directions are a hard-coded
                              * 2-vector, psfrec.py:66,594); more need explicit wind directions from the host */
enum {
    PSFR_DRAW_R0 = 0,        /* r0 at 0.5 um on the line of sight (seeing2r01, psfrec.py:108,183-187; holds the zenith angle) */
    PSFR_DRAW_L0 = 1,        /* outer scale [m] */
    PSFR_DRAW_FITC = 2,      /* cst r0^(-5/3) of the fitting PSD (psfrec.py:622-625) */
    PSFR_DRAW_ALPHA_TT = 3,  /* Moffat alpha of the tip-tilt kernel [px] (psfrec.py:881-905) */
    PSFR_DRAW_NLAYERS = 4,   /* 1 .. PSFR_MAX_LAYERS */
    PSFR_DRAW_NGS = 5,       /* guide stars of the draw (psfr_compute_groups only; 3 in the reference's three lasers mode) */
    PSFR_DRAW_LAYER0 = 8,    /* layer l occupies PSFR_DRAW_LAYER0 + PSFR_LAYER_NPAR * l + PSFR_LAYER_* */
    PSFR_DRAW_NPAR = 40
};
enum {
    PSFR_LAYER_CPHI = 0,     /* 0.0229 (Cn2_l^(-3/5) r0)^(-5/3) (psfrec.py:569-571) */
    PSFR_LAYER_H = 1,        /* altitude [m] */
    PSFR_LAYER_WX = 2,       /* wind vector [m/s] (psfrec.py:61,66,594) */
    PSFR_LAYER_WY = 3,
    PSFR_LAYER_NPAR = 4
};

/* Per-image fit record written by the Moffat fitter (mpdaf Image.moffat_fit columns,
 * psfrec.py:861-871; fwhm still in pixels).  The err_* entries are sqrt(|diag((J^T J)^-1)| chi^2/dof), the
 * estimate scipy.optimize.leastsq's cov_x gives mpdaf. */
enum {
    PSFR_FIT_PEAK = 0,   /* I */
    PSFR_FIT_Y0 = 1,     /* centre, first (row) axis */
    PSFR_FIT_X0 = 2,     /* centre, second (column) axis */
    PSFR_FIT_ALPHA = 3,  /* a */
    PSFR_FIT_N = 4,      /* beta */
    PSFR_FIT_FWHM = 5,   /* 2 a sqrt(2^(1/n)-1) [px] */
    PSFR_FIT_CHISQ = 6,
    PSFR_FIT_ITER = 7,   /* LM iterations used; negative = not converged */
    PSFR_FIT_ERR_PEAK = 8, PSFR_FIT_ERR_Y0 = 9, PSFR_FIT_ERR_X0 = 10,
    PSFR_FIT_ERR_ALPHA = 11, PSFR_FIT_ERR_N = 12,
    PSFR_FIT_ERR_FWHM = 13,  /* mpdaf's expression: err_a * n [px] */
    PSFR_FIT_FLUX = 14,      /* pi a^2 I / (n - 1) */
    PSFR_FIT_ERR_FLUX = 15,  /* mpdaf's expression err_I err_n err_a^2 err_e with err_e = 0 (circular fit) */
    PSFR_FIT_NPAR = 16
};

/* Per-image record of the elliptical Moffat fit, f = I (1 + A dp^2 + B dq^2 + C dp dq)^(-n) with dp = p - y0
 * (row) and dq = q - x0 (column), fitted over theta = (I, y0, x0, A, B, C, n) from the image's circular record.
 * The reference has no elliptical fit (it calls mpdaf's moffat_fit with circular=True): these columns are
 * this library's own and their parity with mpdaf's elliptical fit is unpinned.  Widths and FWHM in pixels.
 * Every err_* entry is sqrt(grad g^T Sigma grad g) of its quantity g, Sigma = (J^T J)^-1 chi^2/dof over theta,
 * dof = npx - 7 (the delta method; not mpdaf's err_fwhm = err_a * n). */
enum {
    PSFR_EFIT_PEAK = 0, PSFR_EFIT_Y0 = 1, PSFR_EFIT_X0 = 2,   /* as the circular record */
    PSFR_EFIT_A_MAJOR = 3,   /* 1/sqrt(lambda_min) of [[A, C/2], [C/2, B]] */
    PSFR_EFIT_A_MINOR = 4,   /* 1/sqrt(lambda_max) */
    PSFR_EFIT_PA = 5,        /* major axis [deg] in [0, 180), from +x (column) toward +y (row); 0 at a circle */
    PSFR_EFIT_N = 6,         /* beta */
    PSFR_EFIT_FWHM_MAJOR = 7, PSFR_EFIT_FWHM_MINOR = 8,   /* a 2 sqrt(2^(1/n) - 1) */
    PSFR_EFIT_AXIS_RATIO = 9,   /* minor / major, in (0, 1] */
    PSFR_EFIT_CHISQ = 10,
    PSFR_EFIT_ITER = 11,     /* LM iterations of the elliptical stage; negative = not converged */
    PSFR_EFIT_ERR_PEAK = 12, PSFR_EFIT_ERR_Y0 = 13, PSFR_EFIT_ERR_X0 = 14,
    PSFR_EFIT_ERR_A_MAJOR = 15, PSFR_EFIT_ERR_A_MINOR = 16,
    PSFR_EFIT_ERR_PA = 17,   /* [deg]; +inf at an exact circle */
    PSFR_EFIT_ERR_N = 18, PSFR_EFIT_ERR_FWHM_MAJOR = 19, PSFR_EFIT_ERR_FWHM_MINOR = 20,
    PSFR_EFIT_ERR_AXIS_RATIO = 21,
    PSFR_EFIT_FLUX = 22,     /* pi I a_major a_minor / (n - 1) */
    PSFR_EFIT_ERR_FLUX = 23,
    PSFR_EFIT_NPAR = 24
};

/* Moffat fits of observed star images (DESIGN.md section 5.7, psfr_moffat_fit_weighted).  The fit minimises
 * sum_i w_i (f(p_i, q_i; theta) + c - d_i)^2 over the used pixels, f the circular or elliptical Moffat of the records
 * above and c a constant background when it is requested (otherwise c = 0, not fitted).
 *  - A pixel is used when w_i > 0.  A pixel with w_i = 0 takes part in no sum, the start point included, whatever its
 *    data value (NaN and +-inf included).
 *  - An image fails when it has a weight that is negative or not finite, a used pixel whose data is not finite, or
 *    npix_used <= NP (NP = 5 circular, 7 elliptical, plus 1 with a background).  A failed image gets ITER = 0 and NaN
 *    in every other slot of its record and in CONT / ERR_CONT; the other images of the call are unaffected.
 *  - Errors as the records above with chi^2 = sum w r^2 and dof = npix_used - NP: sqrt(diag((J^T W J)^-1) chi^2/dof),
 *    the delta method over the same Sigma for the elliptical record.  With w = 1 / variance, chi^2/dof ~ 1.
 *  - Start point: with every weight 1 and no background, the start of psfr_moffat_fit bit for bit.  Otherwise the
 *    peak and column moments are taken over the used pixels only; with a background, c0 = the mean of the used
 *    pixels on the outermost ring of the stamp (rows 0 and ny - 1, columns 0 and nx - 1; 0 when none is used), and
 *    the moments are taken of d - c0.  The elliptical fit starts from the image's own circular star-fit record
 *    with its c, as psfr_moffat_fit_elliptical.
 *  - FIT / EFIT records as above: PEAK and FLUX are above the background.  Side record [nimg][PSFR_BACK_NPAR]: */
enum {
    PSFR_BACK_CONT = 0,      /* c (0 without a background) */
    PSFR_BACK_ERR_CONT = 1,  /* its error (0 without a background) */
    PSFR_BACK_NPIX = 2,      /* used pixels */
    PSFR_BACK_NPAR = 3
};
/* Shared memory of the star fits: the image and its weights, 4 images per CTA.  The circular fit needs
 * 4 (2 ny nx + nx) doubles, the elliptical one also 4 * 2 ny nx doubles, each at most 200 KiB; otherwise
 * PSFR_E_UNSUPPORTED.  The largest accepted square stamp is 56 x 56 (57 x 57 is refused). */

/* Template fits of star images (DESIGN.md section 5.8, psfr_template_fit): each stamp d [ny][nx] with weights w is
 * fitted as F * T(shifted) + c, T the reconstructed PSF tpl [ty][tx] of the same wavelength.
 *  - s(u, v) is the interpolating cubic B-spline of tpl with mirror boundary conditions, exactly
 *    scipy.ndimage.map_coordinates(tpl, [[u], [v]], order=3, mode='mirror'); outside [0, ty - 1] x [0, tx - 1] s and
 *    its derivatives are 0.
 *  - Pixel (p, q) has the model m = F * s(p - y0 + ty/2, q - x0 + tx/2) / S + c (integer halves), S the sum of tpl's
 *    pixels in FP64 in row-major order: F is the flux of the template's whole footprint.  c is fitted only with a
 *    background, otherwise 0.  Parameters x = [F, y0, x0(, c)], NP = 3 or 4.
 *  - Used pixels, objective and errors as the star fits above: minimise sum w r^2 over the pixels with w > 0, errors
 *    sqrt(diag((J^T W J)^-1) chi^2/dof), dof = npix_used - NP.
 *  - Start point: c0 = the ring background of the star fits (0 without a background); (y0, x0) = the used pixel with
 *    the largest d - c0 (lowest row-major index on a tie); F0 = sum w s~ (d - c0) / sum w s~^2 at that centre,
 *    s~ = s / S.  Levenberg-Marquardt over every pixel to the relative step 1.49e-8, at most 200 iterations
 *    (ITER < 0: not converged); a trial point with a non-finite parameter or a centre outside
 *    [-0.5, ny - 0.5] x [-0.5, nx - 0.5] is refused.
 *  - An image fails for the star fits' causes (NP as above), for a template with a non-finite pixel or S <= 0, and when
 *    no used pixel overlaps the template (sum w s~^2 = 0 at the start): ITER = 0 and NaN in every other slot of its
 *    record and of its model image; the other images of the call are unaffected.
 *  Record [nimg][PSFR_TFIT_NPAR]: */
enum {
    PSFR_TFIT_FLUX = 0,      /* F */
    PSFR_TFIT_Y0 = 1,        /* centre row [px] */
    PSFR_TFIT_X0 = 2,        /* centre column [px] */
    PSFR_TFIT_CONT = 3,      /* c (0 without a background) */
    PSFR_TFIT_CHISQ = 4,     /* sum w r^2 */
    PSFR_TFIT_QFIT = 5,      /* sum_used |r| / |F|: the template's misfit, independent of the weights */
    PSFR_TFIT_ITER = 6,      /* LM iterations (< 0: not converged, 0: failed) */
    PSFR_TFIT_NPIX = 7,      /* used pixels */
    PSFR_TFIT_ERR_FLUX = 8,
    PSFR_TFIT_ERR_Y0 = 9,
    PSFR_TFIT_ERR_X0 = 10,
    PSFR_TFIT_ERR_CONT = 11, /* 0 without a background */
    PSFR_TFIT_NPAR = 12
};
/* Shared memory of the template fit: the image, its weights and the template's B-spline coefficients, 4 images per
 * CTA: 4 (2 ny nx + ty tx') doubles with tx' = tx rounded up to odd (a row stride free of bank conflicts), at most
 * 200 KiB; otherwise PSFR_E_UNSUPPORTED.  With a 40 x 40 template the largest accepted square stamp is 48 x 48
 * (49 x 49 is refused). */

/* Encircled energy (DESIGN.md section 5.4).  Pixel (p, q) is the unit square [p - 1/2, p + 1/2] x [q - 1/2, q + 1/2]
 * with its value spread uniformly over it; EE(r) = sum img[p][q] * area(pixel AND disc(centre, r)), the exact
 * overlap area in FP64, over the pixels of the image only (a circle that leaves the image is clipped by its edge),
 * in the image's own units (no renormalisation).  A record of nrad + 1 + nfrac doubles per image: */
#define PSFR_EE_MAX_RADII 64
#define PSFR_EE_MAX_FRACTIONS 16
/*  [0, nrad)              EE(radii[k])
 *  [nrad]                 TOTAL = sum img, summed in the order of the EE sums (EE == TOTAL bit for bit once the
 *                         circle contains every pixel)
 *  [nrad + 1 + j]         r_q [px] for q = fracs[j], to a bracket of 1e-10 px; NaN when TOTAL <= 0 (or NaN).
 *                         Without negative pixels, the smallest r >= 0 with EE(r) >= q TOTAL; with them, an r
 *                         where EE crosses q TOTAL from below: EE(r) >= q TOTAL > EE(r') for an r' less than
 *                         1e-10 px below r
 * Radii must be finite and >= 0, fractions in (0, 1), centres finite; otherwise PSFR_E_ARG, nothing written. */

/* AO summaries of every PSF (DESIGN.md section 5.5).  N = dim, L = 16 m (the PSD grid step is 1/L), OTF_tel the
 * telescope OTF on the N x N grid and D_lambda = (2 pi / lambda_nm)^2 D_unit the structure function at lambda.
 *
 * Strehl ratio S(lambda) = sum_f OTF_tel(f) exp(-D_lambda(f) / 2) / sum_f OTF_tel(f) over the full N x N grid: the
 * centre ratio psf[N/2][N/2] / psf_diff[N/2][N/2] of the reference's psd_to_psf, the first PSF from the PSD and
 * the second from a PSD of zeros (both unit-sum).  In field-mean mode (ndir > 1 without field) it is the mean of
 * the per-direction values, the origin value of the field-mean PSF.  It is the AO Strehl, before the tip-tilt and
 * MUSE-intrinsic kernels: those act on the 0.2" grid, which does not resolve the diffraction core, and a
 * "delivered" Strehl after them is not computed.
 *
 * Residual-phase variance record of every (draw, direction) plane, nm^2, independent of lambda (multiply by
 * (2 pi / lambda_nm)^2 for rad^2 at lambda).  TOTAL = sum over the plane's merged N x N PSD / L^2 (psfrec.py:148-151,
 * the bg[0,0] of psfrec.py:718).  Each cell counts to exactly one source: outside the 80 x 80 AO zone to FIT; inside
 * it, where the merged value max(fit, ao) is the fit (fit >= ao), to FIT; otherwise its ao value splits into NOISE
 * (err_noise) and PROJ = sum_l err_rec_l, each err_rec_l also in LAYER0 + l (unused layer slots 0).  PROJ is the
 * reference's |P beta_l - corr_l|^2 Cphi_l: servo lag, anisoplanatism and aliasing do not add up separately in
 * that formula, so it is not split further.  TOTAL = FIT + NOISE + PROJ up to rounding. */
enum {
    PSFR_VAR_TOTAL = 0,
    PSFR_VAR_FIT = 1,
    PSFR_VAR_NOISE = 2,
    PSFR_VAR_PROJ = 3,
    PSFR_VAR_LAYER0 = 4,     /* LAYER0 + l, l < PSFR_MAX_LAYERS */
    PSFR_VAR_NPAR = 12
};

/* Band images (DESIGN.md section 5.6): throughput-weighted sums of the wavelength planes of an image set, the PSF of a
 * white-light, narrow-band or filter image.  A call carries 1 <= nband <= PSFR_MAX_BANDS bands with weights
 * w [nband][nlam], finite and >= 0, and every band sum W_b = sum_k w[b][k] (added in ascending k) finite and > 0;
 * otherwise PSFR_E_ARG before any launch, nothing written.  The band image of a set of planes C[k] is
 *   B[b][pix] = acc / W_b,  acc = fma(w[b][k], C[k][pix], acc) in ascending k from acc = 0, in FP64,
 * with no clip and no renormalisation: B keeps the flux scale of the planes.  One-hot weights give plane k bit for
 * bit, and scaling a band's weights by a power of two leaves its bits unchanged.  The reference has no band PSF:
 * parity with it is unpinned. */
#define PSFR_MAX_BANDS 16

/* Context ------------------------------------------------------------------------- */

/* dim: PSD grid size (1280; the reference hard-codes it in compute_psf, psfrec.py:955).
 * max_planes: largest number of (draw x direction) planes processed at once;
 * max_lambda: largest number of wavelengths per call.  Builds twiddles, the pupil
 * (pupil_mask, psfrec.py:190-203,656) and the telescope OTF (psfrec.py:784-790) on the GPU. */
PSFR_API int psfr_create(int device, int dim, int max_planes, int max_lambda, psfr_ctx** out);
PSFR_API void psfr_destroy(psfr_ctx* ctx);
PSFR_API const char* psfr_last_error(const psfr_ctx* ctx);   /* ctx may be NULL: last create error */
PSFR_API int psfr_version(void);

/* AO-zone frequency tables f, f_x = f cos(arg f), f_y = f sin(arg f) on the 80x80 grid,
 * formed by the host exactly as psfrec.py:548-554,241-242 (the cutoff masks depend on
 * their 1-ulp rounding). */
PSFR_API int psfr_set_geometry(psfr_ctx* ctx, const double* f, const double* f_x, const double* f_y);

/* Stages (each mirrors one reference function) -------------------------------------- */

/* simul_psd_wfm (psfrec.py:36-151) incl. dsp4muse / calc_mat_rec_glao_finale /
 * calc_dsp_res_glao_finale / psd_fit.  Planes are ordered draw-major: plane = draw*ndir+dir.
 * dirs[2*ndir]: field directions [arcsec] (direction_perf); poslgs[2*ngs]: LGS positions
 * [arcsec], x then y.  The PSD stays in the context workspace; if out_psd != NULL it is
 * also copied there ([ndraw*ndir][dim][dim], nm^2). */
PSFR_API int psfr_psd(psfr_ctx* ctx, int ndraw, const double* draws, int ndir, const double* dirs,
             int ngs, const double* poslgs, double* out_psd, void* stream);

/* Load user PSDs into the workspace instead (psf_muse / psd_to_psf called on an array). */
PSFR_API int psfr_load_psd(psfr_ctx* ctx, int nplanes, const double* psd, void* stream);

/* PSD -> wavelength-free structure function D_unit on the workspace planes
 * (psfrec.py:717-722 with the (2 pi/lambda)^2 factor left out). */
PSFR_API int psfr_structure_function(psfr_ctx* ctx, int nplanes, void* stream);

/* psd_to_psf (psfrec.py:689-807, live branch): full dim x dim PSF of workspace plane
 * `plane` at wavelength lambda_m [m], normalised to unit sum.  Parity mode. */
PSFR_API int psfr_psd_to_psf(psfr_ctx* ctx, int plane, double lambda_m, double* out_psf, void* stream);

/* psf_muse (psfrec.py:644-686): 40x40 PSFs at 0.2"/px for ndraw draws x nlam wavelengths,
 * averaging the ndir planes of each draw; pruned transform (only the 80x80 samples the
 * bilinear resampling reads).  out_cube: [ndraw][nlam][40][40]. */
PSFR_API int psfr_psf_cube(psfr_ctx* ctx, int ndraw, int ndir, int nlam, const double* lambda_nm,
                  double* out_cube, void* stream);

/* convolve_final_psf (psfrec.py:874-930): tip-tilt Moffat (beta=2, alpha_tt[draw] in px)
 * then MUSE intrinsic Moffat (muse_intrinsic_psf, psfrec.py:1144-1171) per wavelength.
 * cube [ndraw][nlam][40][40] in -> out (may alias).
 * Domain of the kernels (outside, the kernel would be 0/0; nothing is launched or written):
 *   alpha_tt[d] > 0 with pi alpha_tt^2 a finite, normal double (alpha_tt in about [8.5e-155, 7.5e153]), else
 *   PSFR_E_ARG (tiptilt_alpha is 0 at GL = 1 and NaN at GL > 1); the same holds for the PSFR_DRAW_ALPHA_TT slot
 *   in every batch call that convolves;
 *   lambda finite and > 0, else PSFR_E_ARG;
 *   MUSE beta(lambda) > 0 and != 1 and pi gamma^2 finite and normal, else PSFR_E_UNSUPPORTED: beta crosses 0 at
 *   lambda ~ 1188.99 nm, so the convolutions (and every batch call) stop there; beta = 1 at ~ 1132.77 nm and
 *   fwhm = 0 at ~ 303.85 nm are isolated points. */
PSFR_API int psfr_convolve(psfr_ctx* ctx, int ndraw, int nlam, const double* lambda_nm,
                  const double* alpha_tt, const double* cube, double* out_cube, void* stream);

/* fit_psf_cube (psfrec.py:861-871 -> mpdaf Image.moffat_fit, circular, no background):
 * batched Levenberg-Marquardt, one CTA per image.  imgs [nimg][ny][nx], params
 * [nimg][PSFR_FIT_NPAR]. */
PSFR_API int psfr_moffat_fit(psfr_ctx* ctx, int nimg, int ny, int nx, const double* imgs,
                    double* params, void* stream);

/* Elliptical Moffat fit of every image (PSFR_EFIT_* record): the circular fit of psfr_moffat_fit, then a
 * 7-parameter Levenberg-Marquardt from its converged record, one warp per image.  Images, sizes, host / device
 * handling and refusals as psfr_moffat_fit, and ny*nx must exceed 7.  params [nimg][PSFR_EFIT_NPAR]. */
PSFR_API int psfr_moffat_fit_elliptical(psfr_ctx* ctx, int nimg, int ny, int nx, const double* imgs,
                                        double* params, void* stream);

/* Moffat fit of star images with per-pixel weights and an optional constant background (DESIGN.md section 5.7; the
 * definitions are above PSFR_BACK_CONT).  imgs and weights [nimg][ny][nx]; weights NULL means every weight is 1.
 * fit_back != 0 fits the background; elliptical != 0 writes PSFR_EFIT_* records to params [nimg][PSFR_EFIT_NPAR],
 * otherwise PSFR_FIT_* records to params [nimg][PSFR_FIT_NPAR].  back [nimg][PSFR_BACK_NPAR] may be NULL.  Host or
 * device arrays in any mix; host arrays are chunked through the staging buffers as psfr_moffat_fit (images and
 * weights each take one, at the same chunk size), and an image that does not fit them is PSFR_E_CAPACITY.  NULL imgs
 * or params, nimg < 1 or a side under 3 are PSFR_E_ARG, a stamp over the shared-memory limit above
 * PSFR_E_UNSUPPORTED: all before any launch, nothing written.  With weights NULL and fit_back = 0 the records are
 * those of psfr_moffat_fit / psfr_moffat_fit_elliptical bit for bit, and back holds (0, 0, ny nx). */
PSFR_API int psfr_moffat_fit_weighted(psfr_ctx* ctx, int nimg, int ny, int nx, const double* imgs,
                                      const double* weights, int fit_back, int elliptical, double* params,
                                      double* back, void* stream);

/* Template fit of star images (DESIGN.md section 5.8; the definitions are above PSFR_TFIT_FLUX).  imgs and weights
 * [nimg][ny][nx]; weights NULL means every weight is 1.  tpls [ntpl][ty][tx]: image i is fitted with template
 * i % ntpl, so stamps stacked star-major share one template cube.  fit_back != 0 fits the background.  params
 * [nimg][PSFR_TFIT_NPAR]; model [nimg][ny][nx] (may be NULL) receives the model m at the final parameters on every
 * pixel, used or not.  Host or device arrays in any mix; host stamps, weights, records and models are chunked through
 * the staging buffers as psfr_moffat_fit_weighted, and host templates are uploaded once per call (PSFR_E_CAPACITY when
 * they exceed the staging buffer, max_planes * max_lambda * 1600 doubles).  When imgs, weights, params and model are
 * all device arrays (or NULL), one launch fits every image, whatever the context's capacity.  NULL imgs, tpls or params, nimg < 1, ny or nx < 3, ntpl < 1, nimg % ntpl != 0 and
 * ty or tx < 4 are PSFR_E_ARG, a stamp and template over the shared-memory limit above PSFR_E_UNSUPPORTED: all before
 * any launch, nothing written. */
PSFR_API int psfr_template_fit(psfr_ctx* ctx, int nimg, int ny, int nx, const double* imgs, const double* weights,
                               int ntpl, int ty, int tx, const double* tpls, int fit_back, double* params,
                               double* model, void* stream);

/* compute_psf (psfrec.py:933-978) for a batch of draws, fused on the device:
 * PSD -> structure function -> pruned PSFs -> resample -> convolutions -> fit.
 * out_cube [ndraw][nlam][40][40] and out_fit [ndraw][nlam][PSFR_FIT_NPAR]; either may be NULL.
 * Every draw uses all ngs stars of poslgs [2][ngs]; the PSFR_DRAW_NGS slot is ignored. */
PSFR_API int psfr_compute_batch(psfr_ctx* ctx, int ndraw, const double* draws, int ndir, const double* dirs,
                       int ngs, const double* poslgs, int nlam, const double* lambda_nm,
                       double* out_cube, double* out_fit, void* stream);

/* compute_psf_from_sparta (psfrec.py:981-1113) for many exposures at once.  draws
 * [ndraw][PSFR_DRAW_NPAR], exposure by exposure; draw d uses the first draws[d][PSFR_DRAW_NGS]
 * (1..npos) stars of poslgs [2][npos] (npos <= 4; the reference's three-laser asterism is the first
 * three of its four-laser one, so one table serves both modes).  Exposure g owns draws [group_end[g-1],
 * group_end[g]) (host array, strictly increasing, last = ndraw; ngroup may be 0).
 * out_cube / out_fit as psfr_compute_batch - a draw gives the same bits through either entry point;
 * out_mean [ngroup][nlam][40][40] and out_mean_fit [ngroup][nlam][PSFR_FIT_NPAR] as psfr_mean_refit per
 * exposure, bit for bit, formed on the device while the exposure's draws are resident: each mean is
 * summed in draw order and, at a chunk edge, carried on as one unnormalised sum.  Every output may be
 * NULL; the mean outputs need ngroup > 0.  All arguments are checked before any output is written. */
PSFR_API int psfr_compute_groups(psfr_ctx* ctx, int ndraw, const double* draws, int npos, const double* poslgs,
                        int ndir, const double* dirs, int nlam, const double* lambda_nm, int ngroup, const int* group_end,
                        double* out_cube, double* out_fit, double* out_mean, double* out_mean_fit, void* stream);

/* psfr_compute_groups without the field average: the PSF of every draw at every one of the ndir
 * positions of dirs [2][ndir] (arcsec, ndir <= 256 and <= max_planes).  The PSF at position k of draw d
 * is the reference's psf_muse of that direction's PSD alone, convolved with draw d's kernels and fitted:
 * bit for bit what psfr_compute_batch / psfr_compute_groups give for draw d with dirs = position k only.
 * Arguments and checks as psfr_compute_groups; the outputs gain a position axis:
 * out_cube [ndraw][ndir][nlam][40][40], out_fit [ndraw][ndir][nlam][PSFR_FIT_NPAR],
 * out_mean [ngroup][ndir][nlam][40][40] and out_mean_fit [ngroup][ndir][nlam][PSFR_FIT_NPAR], where
 * out_mean[g][k] and its fit are psfr_mean_refit of exposure g's cubes at position k, bit for bit. */
PSFR_API int psfr_compute_field(psfr_ctx* ctx, int ndraw, const double* draws, int npos, const double* poslgs,
                       int ndir, const double* dirs, int nlam, const double* lambda_nm, int ngroup, const int* group_end,
                       double* out_cube, double* out_fit, double* out_mean, double* out_mean_fit, void* stream);

/* psfr_compute_field plus the elliptical fit of every image it fits: out_efit [ndraw][ndir][nlam][PSFR_EFIT_NPAR]
 * of the per-draw cubes and out_mean_efit [ngroup][ndir][nlam][PSFR_EFIT_NPAR] of the exposure means, each
 * bit for bit psfr_moffat_fit_elliptical of the images in out_cube / out_mean.  The elliptical fit runs in the
 * chunk of its images, right after their circular fit.  Every output may be NULL; the other outputs are those
 * of psfr_compute_field, bit for bit. */
PSFR_API int psfr_compute_field_shapes(psfr_ctx* ctx, int ndraw, const double* draws, int npos, const double* poslgs,
                       int ndir, const double* dirs, int nlam, const double* lambda_nm, int ngroup, const int* group_end,
                       double* out_cube, double* out_fit, double* out_mean, double* out_mean_fit,
                       double* out_efit, double* out_mean_efit, void* stream);

/* Encircled-energy record of every image.  centres [nimg][2] = (y0, x0) in pixels (row, column; pixel centres at
 * integers), or NULL for (ny / 2, nx / 2) - pixel (20, 20) of a 40 x 40 PSF, its point of symmetry.  radii_px
 * [nrad] (0 <= nrad <= PSFR_EE_MAX_RADII), fracs [nfrac] (0 <= nfrac <= PSFR_EE_MAX_FRACTIONS); out
 * [nimg][nrad + 1 + nfrac].  Image sizes, host / device handling and refusals as psfr_moffat_fit. */
PSFR_API int psfr_encircled_energy(psfr_ctx* ctx, int nimg, int ny, int nx, const double* imgs, const double* centres,
                                   int nrad, const double* radii_px, int nfrac, const double* fracs, double* out,
                                   void* stream);

/* The fused pipeline with the encircled energy of every image it returns.  field = 0: psfr_compute_groups (the
 * field mean of the ndir directions of every draw), field != 0: psfr_compute_field (one PSF per direction);
 * arguments and checks as those entry points.  out_efit / out_mean_efit as psfr_compute_field_shapes, in either
 * mode.  out_ee [ndraw][P][nlam][nrad + 1 + nfrac] and out_mean_ee [ngroup][P][nlam][nrad + 1 + nfrac] (P = ndir
 * with field, 1 without) are psfr_encircled_energy of the images in out_cube / out_mean about their default
 * centre, bit for bit; each runs in the chunk of its images, right after their fits.  Every output may be NULL;
 * the other outputs are those of psfr_compute_groups / psfr_compute_field_shapes, bit for bit. */
PSFR_API int psfr_compute_energy(psfr_ctx* ctx, int field, int ndraw, const double* draws, int npos,
                       const double* poslgs, int ndir, const double* dirs, int nlam, const double* lambda_nm,
                       int ngroup, const int* group_end, int nrad, const double* radii_px, int nfrac,
                       const double* fracs, double* out_cube, double* out_fit, double* out_mean, double* out_mean_fit,
                       double* out_efit, double* out_mean_efit, double* out_ee, double* out_mean_ee, void* stream);

/* psfr_compute_energy plus the AO summaries of every draw (PSFR_VAR_* above): out_strehl [ndraw][P][nlam] (P = ndir
 * with field, 1 without), the Strehl ratio of each PSF the pipeline forms, and out_var [ndraw][ndir][PSFR_VAR_NPAR],
 * the variance record of each (draw, direction) plane in either mode.  Both are computed in the chunk of their draws
 * and depend on a draw's data only (the same bits at every chunk size and through either mode for the variance).
 * Exposure means of them are not formed: they are a few doubles per draw.  Every output may be NULL, and a NULL
 * output launches nothing; the other outputs are those of psfr_compute_energy, bit for bit. */
PSFR_API int psfr_compute_ao(psfr_ctx* ctx, int field, int ndraw, const double* draws, int npos,
                       const double* poslgs, int ndir, const double* dirs, int nlam, const double* lambda_nm,
                       int ngroup, const int* group_end, int nrad, const double* radii_px, int nfrac,
                       const double* fracs, double* out_cube, double* out_fit, double* out_mean, double* out_mean_fit,
                       double* out_efit, double* out_mean_efit, double* out_ee, double* out_mean_ee,
                       double* out_strehl, double* out_var, void* stream);

/* Band images (PSFR_MAX_BANDS above) of ncube image sets cubes [ncube][nlam][ny][nx] -> out [ncube][nband][ny][nx],
 * weights [nband][nlam].  Host or device pointers; host arrays go through the staging buffers in chunks.  nlam must
 * not exceed max_lambda (PSFR_E_CAPACITY). */
PSFR_API int psfr_band_psf(psfr_ctx* ctx, int ncube, int nlam, int ny, int nx, const double* cubes, int nband,
                           const double* weights, double* out, void* stream);

/* psfr_compute_ao plus the band images of every image set it forms (P = ndir with field, 1 without):
 * out_band [ndraw][P][nband][40][40], the bands of the planes in out_cube; out_band_fit [ndraw][P][nband][PSFR_FIT_NPAR]
 * and out_band_ee [ndraw][P][nband][nrad + 1 + nfrac], psfr_moffat_fit and psfr_encircled_energy (default centre) of
 * those band images, bit for bit; out_mean_band, out_mean_band_fit and out_mean_band_ee [ngroup][P][nband]... the same
 * for the exposure means, bit for bit psfr_band_psf of out_mean (not the mean of the per-draw bands).  The bands of a
 * chunk run after its convolutions, those of the means after the exposure's mean is formed.  Every output may be NULL,
 * and a NULL output launches nothing; with nband = 0 and every band output NULL the call is psfr_compute_ao (weights
 * may then be NULL).  The other outputs are those of psfr_compute_ao, bit for bit. */
PSFR_API int psfr_compute_bands(psfr_ctx* ctx, int field, int ndraw, const double* draws, int npos,
                       const double* poslgs, int ndir, const double* dirs, int nlam, const double* lambda_nm,
                       int ngroup, const int* group_end, int nrad, const double* radii_px, int nfrac,
                       const double* fracs, double* out_cube, double* out_fit, double* out_mean, double* out_mean_fit,
                       double* out_efit, double* out_mean_efit, double* out_ee, double* out_mean_ee,
                       double* out_strehl, double* out_var, int nband, const double* weights, double* out_band,
                       double* out_band_fit, double* out_band_ee, double* out_mean_band, double* out_mean_band_fit,
                       double* out_mean_band_ee, void* stream);

/* Time-mean of ncube cubes + refit (psfrec.py:1104-1105). cubes [ncube][nlam][40][40]. */
PSFR_API int psfr_mean_refit(psfr_ctx* ctx, int ncube, int nlam, const double* cubes,
                    double* out_mean, double* out_fit, void* stream);

/* fit_psf_with_polynom (psfrec.py:1174-1210): least-squares polynomials of degree `deg`
 * in the normalised wavelength for nseries series of nlam values each (one shared design
 * matrix).  y [nseries][nlam] -> coef [nseries][deg+1], highest power first (np.polyfit). */
PSFR_API int psfr_polyfit(psfr_ctx* ctx, int nseries, int nlam, const double* lambda_nm, int deg,
                 const double* y, double* coef, void* stream);

/* Options.  PSFR_OPT_EXP_CUT (default 45): in the pruned stage-B row pass (psfr_psf_cube,
 * psfr_compute_batch) entries of exp(-Dphi/2) smaller than exp(-cut) are flushed to zero and
 * row pairs that are below the cut everywhere are not transformed.  The OTF peak is 1, so the
 * default drops terms below 2.9e-20 of it - four orders of magnitude under the FP64 rounding of a
 * single kept term; beyond the cut radius exp(-Dphi/2) falls off faster than exponentially, so even
 * a coherent sum of everything dropped stays below ~1e-15 of the OTF peak, against a PSF peak of
 * 15 (2 arcsec seeing) to several 1000.  tools/parity_sweep.py holds the default against the oracle
 * over the BASELINE configs and the corners of the config-4 sweep (profiles/).  A value >= 745 (exp
 * underflows) disables the cut; psfr_psd_to_psf (full-grid parity mode) never applies it (nor the
 * grades below).
 *
 * Graded precision of the same pass (the OTF peak is exactly 1, so an entry's size bounds
 * what an error in it can do to the result):
 * PSFR_OPT_EXP_GRADE (default 20): a segment of 2 x 32 OTF entries whose every live entry is
 * below exp(-grade) = 2.1e-9 evaluates exp on the special-function unit in single precision
 * (relative error ~4e-6, i.e. < 1e-14 of the peak per entry); other blocks use the FP64 exp.
 * PSFR_OPT_F32_ROWS (default 25, dim 1280 only; dim 2560 runs every unit in FP64): a row pair whose every entry is below
 * exp(-thr) = 1.4e-11 is evaluated AND transformed in single precision; all other rows and
 * the whole column pass are FP64.
 * Measured against the all-FP64 evaluation (tools/diag_grade.py, seven seeing/L0 cases x five
 * wavelengths): largest difference 1.5e-14 of the PSF peak, 1.1e-11 pointwise on pixels above
 * 1e-6 of the peak - the all-FP64 kernel and numpy differ by 1e-10 there.  A threshold >= the
 * cut disables the respective grade (e.g. 1e30). */
enum { PSFR_OPT_EXP_CUT = 1, PSFR_OPT_EXP_GRADE = 2, PSFR_OPT_F32_ROWS = 3,
       /* row kernel of the pruned stage B: 2 (default) one 128-thread group per row transform, data in
        * shared memory, pruned third pass (csrc/psfr_hot2.cu); 1 one warp per transform, data in
        * registers (csrc/psfr_hot.cu) */
       PSFR_OPT_ROW_KERNEL = 4 };
PSFR_API int psfr_set_option(psfr_ctx* ctx, int key, double value);

/* Introspection used by tests and the bench --------------------------------------- */
/* numeric properties of a context: option values, capacities, and the number of sampled row-pass
 * frequencies kept per PSF in the hand-off buffer between the two passes of the pruned stage B */
enum { PSFR_INFO_Y_COLS = 1, PSFR_INFO_EXP_CUT = 2, PSFR_INFO_EXP_GRADE = 3, PSFR_INFO_F32_ROWS = 4,
       PSFR_INFO_ROW_KERNEL = 5, PSFR_INFO_MAX_PLANES = 6, PSFR_INFO_MAX_LAMBDA = 7, PSFR_INFO_DIM = 8 };
PSFR_API int psfr_get_info(const psfr_ctx* ctx, int key, double* out);
PSFR_API int psfr_get_otf(psfr_ctx* ctx, double* out);            /* [dim/2+2][dim] half-plane telescope OTF */
PSFR_API int psfr_get_structure_function(psfr_ctx* ctx, int plane, double* out); /* [dim/2+2][dim], transposed half-plane */
/* test hook: y[i] = the device exp() used for exp(-Dphi/2) (csrc/fast_exp.cuh), x[i] <= 0 */
PSFR_API int psfr_debug_exp(psfr_ctx* ctx, int n, const double* x, double* y);
PSFR_API long long psfr_kernel_launches(const psfr_ctx* ctx);     /* kernels launched by this context so far */
/* device-side duration [ms] of the stage-B row kernel in the last psfr_psf_cube /
 * psfr_compute_batch / psfr_compute_groups call (CUDA events on the launching stream), and its launch count */
PSFR_API int psfr_last_hot_timing(psfr_ctx* ctx, double* ms, int* launches, long long* psfs);

#ifdef __cplusplus
}
#endif
#endif /* PSFR_H */
