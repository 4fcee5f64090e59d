"""ctypes binding of libpsfr_b200.so (C ABI in include/psfr.h).

The product path has no CPU fallback: if the shared library is missing, cannot be
loaded, or no CUDA device is present, every entry point raises ``PsfrError``.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libpsfr_b200.so')
if os.environ.get('PSFR_LIB_TAG'):      # tuning experiments only: a variant built by build.py with the same tag
    LIB_PATH = LIB_PATH.replace('.so', '_%s.so' % os.environ['PSFR_LIB_TAG'])

# record layouts (keep in sync with include/psfr.h)
DRAW_R0, DRAW_L0, DRAW_FITC, DRAW_ALPHA_TT, DRAW_NLAYERS, DRAW_NGS = 0, 1, 2, 3, 4, 5
DRAW_LAYER0, DRAW_NPAR = 8, 40
LAYER_CPHI, LAYER_H, LAYER_WX, LAYER_WY, LAYER_NPAR = 0, 1, 2, 3, 4
MAX_LAYERS = 8


def layer_slot(layer, field):
    """Index of ``field`` (LAYER_*) of turbulence layer ``layer`` in a draw record."""
    return DRAW_LAYER0 + LAYER_NPAR * layer + field

FIT_PEAK, FIT_Y0, FIT_X0, FIT_ALPHA, FIT_N, FIT_FWHM, FIT_CHISQ, FIT_ITER = range(8)
FIT_ERR_PEAK, FIT_ERR_Y0, FIT_ERR_X0, FIT_ERR_ALPHA, FIT_ERR_N, FIT_ERR_FWHM, FIT_FLUX, FIT_ERR_FLUX = range(8, 16)
FIT_NPAR = 16
# elliptical record (PSFR_EFIT_*): widths and FWHM in pixels, PA in degrees
(EFIT_PEAK, EFIT_Y0, EFIT_X0, EFIT_A_MAJOR, EFIT_A_MINOR, EFIT_PA, EFIT_N, EFIT_FWHM_MAJOR, EFIT_FWHM_MINOR,
 EFIT_AXIS_RATIO, EFIT_CHISQ, EFIT_ITER) = range(12)
(EFIT_ERR_PEAK, EFIT_ERR_Y0, EFIT_ERR_X0, EFIT_ERR_A_MAJOR, EFIT_ERR_A_MINOR, EFIT_ERR_PA, EFIT_ERR_N,
 EFIT_ERR_FWHM_MAJOR, EFIT_ERR_FWHM_MINOR, EFIT_ERR_AXIS_RATIO, EFIT_FLUX, EFIT_ERR_FLUX) = range(12, 24)
EFIT_NPAR = 24
# side record of the star fits (PSFR_BACK_*): background, its error, used pixels
BACK_CONT, BACK_ERR_CONT, BACK_NPIX = range(3)
BACK_NPAR = 3
# template-fit record (PSFR_TFIT_*): flux, centre [px], background, chi^2, QFIT, iterations, used pixels, errors
(TFIT_FLUX, TFIT_Y0, TFIT_X0, TFIT_CONT, TFIT_CHISQ, TFIT_QFIT, TFIT_ITER, TFIT_NPIX, TFIT_ERR_FLUX, TFIT_ERR_Y0,
 TFIT_ERR_X0, TFIT_ERR_CONT) = range(12)
TFIT_NPAR = 12
# encircled-energy record (include/psfr.h): EE at nrad radii, TOTAL, then the radius at each of nfrac fractions
EE_MAX_RADII = 64
EE_MAX_FRACTIONS = 16


def ee_slots(nrad, nfrac):
    """(EE slice, TOTAL index, radius-at-fraction slice, record length) of an encircled-energy record."""
    nrad, nfrac = int(nrad), int(nfrac)
    return slice(0, nrad), nrad, slice(nrad + 1, nrad + 1 + nfrac), nrad + 1 + nfrac

# residual-phase variance record of a (draw, direction) plane (PSFR_VAR_*), nm^2
VAR_TOTAL, VAR_FIT, VAR_NOISE, VAR_PROJ, VAR_LAYER0 = 0, 1, 2, 3, 4
VAR_NPAR = 12
# band images (PSFR_MAX_BANDS): at most this many filter-weighted wavelength sums per call
MAX_BANDS = 16

AO_DIM = 80
PSF_DIM = 40

E_CUDA, E_ARG, E_UNSUPPORTED, E_CAPACITY, E_STATE = -1, -2, -3, -4, -5
OPT_EXP_CUT = 1
OPT_EXP_GRADE = 2
OPT_F32_ROWS = 3
OPT_ROW_KERNEL = 4
INFO_KEYS = {'y_cols': 1, 'exp_cut': 2, 'exp_grade': 3, 'f32_rows': 4, 'row_kernel': 5, 'max_planes': 6,
             'max_lambda': 7, 'dim': 8}


class PsfrError(RuntimeError):
    """Failure reported by the CUDA library (or the library itself is unavailable)."""

    def __init__(self, code, msg):
        super().__init__('psfr error %d: %s' % (code, msg))
        self.code = code


_lib = None
_P = ctypes.c_void_p
_I = ctypes.c_int
_D = ctypes.c_double

_SIGNATURES = {
    'psfr_create': (_I, [_I, _I, _I, _I, ctypes.POINTER(_P)]),
    'psfr_destroy': (None, [_P]),
    'psfr_last_error': (ctypes.c_char_p, [_P]),
    'psfr_version': (_I, []),
    'psfr_set_geometry': (_I, [_P, _P, _P, _P]),
    'psfr_psd': (_I, [_P, _I, _P, _I, _P, _I, _P, _P, _P]),
    'psfr_load_psd': (_I, [_P, _I, _P, _P]),
    'psfr_structure_function': (_I, [_P, _I, _P]),
    'psfr_psd_to_psf': (_I, [_P, _I, _D, _P, _P]),
    'psfr_psf_cube': (_I, [_P, _I, _I, _I, _P, _P, _P]),
    'psfr_convolve': (_I, [_P, _I, _I, _P, _P, _P, _P, _P]),
    'psfr_moffat_fit': (_I, [_P, _I, _I, _I, _P, _P, _P]),
    'psfr_moffat_fit_elliptical': (_I, [_P, _I, _I, _I, _P, _P, _P]),
    'psfr_moffat_fit_weighted': (_I, [_P, _I, _I, _I, _P, _P, _I, _I, _P, _P, _P]),
    'psfr_template_fit': (_I, [_P, _I, _I, _I, _P, _P, _I, _I, _I, _P, _I, _P, _P, _P]),
    'psfr_compute_batch': (_I, [_P, _I, _P, _I, _P, _I, _P, _I, _P, _P, _P, _P]),
    'psfr_compute_groups': (_I, [_P, _I, _P, _I, _P, _I, _P, _I, _P, _I, _P, _P, _P, _P, _P, _P]),
    'psfr_compute_field': (_I, [_P, _I, _P, _I, _P, _I, _P, _I, _P, _I, _P, _P, _P, _P, _P, _P]),
    'psfr_compute_field_shapes': (_I, [_P, _I, _P, _I, _P, _I, _P, _I, _P, _I, _P, _P, _P, _P, _P, _P, _P, _P]),
    'psfr_encircled_energy': (_I, [_P, _I, _I, _I, _P, _P, _I, _P, _I, _P, _P, _P]),
    'psfr_compute_energy': (_I, [_P, _I, _I, _P, _I, _P, _I, _P, _I, _P, _I, _P, _I, _P, _I, _P,
                                 _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    'psfr_compute_ao': (_I, [_P, _I, _I, _P, _I, _P, _I, _P, _I, _P, _I, _P, _I, _P, _I, _P,
                             _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    'psfr_band_psf': (_I, [_P, _I, _I, _I, _I, _P, _I, _P, _P, _P]),
    'psfr_compute_bands': (_I, [_P, _I, _I, _P, _I, _P, _I, _P, _I, _P, _I, _P, _I, _P, _I, _P,
                                _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _P, _P, _P, _P, _P, _P, _P, _P]),
    'psfr_mean_refit': (_I, [_P, _I, _I, _P, _P, _P, _P]),
    'psfr_polyfit': (_I, [_P, _I, _I, _P, _I, _P, _P, _P]),
    'psfr_set_option': (_I, [_P, _I, _D]),
    'psfr_get_otf': (_I, [_P, _P]),
    'psfr_get_structure_function': (_I, [_P, _I, _P]),
    'psfr_debug_exp': (_I, [_P, _I, _P, _P]),
    'psfr_kernel_launches': (ctypes.c_longlong, [_P]),
    'psfr_get_info': (_I, [_P, _I, ctypes.POINTER(_D)]),
    'psfr_last_hot_timing': (_I, [_P, ctypes.POINTER(_D), ctypes.POINTER(_I), ctypes.POINTER(ctypes.c_longlong)]),
}


def exported_symbols():
    """Names every build of the library must export (checked by the CPU tests)."""
    return sorted(_SIGNATURES)


def load():
    """Load the shared library (once).  Raises PsfrError when it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PsfrError(E_STATE, 'libpsfr_b200.so is not built (run `python -m muse_psfr_b200.build`); '
                                 'there is no CPU fallback')
    try:
        lib = ctypes.CDLL(LIB_PATH)
    except OSError as exc:  # pragma: no cover - depends on the host
        raise PsfrError(E_STATE, 'cannot load %s: %s' % (LIB_PATH, exc))
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def ptr(a):
    """Raw address of a numpy array, a torch tensor (device or host), an int, or None."""
    if a is None:
        return None
    if isinstance(a, int):
        return a
    if isinstance(a, np.ndarray):
        if not a.flags['C_CONTIGUOUS']:
            raise ValueError('array must be C-contiguous')
        return a.ctypes.data
    if hasattr(a, 'data_ptr'):  # torch tensor used purely as a buffer carrier
        if not a.is_contiguous():
            raise ValueError('tensor must be contiguous')
        return a.data_ptr()
    raise TypeError('unsupported buffer type %r' % type(a))


def f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def group_end_ptr(group_end):
    """(ngroup, address) of the exposure table of psfr_compute_groups after checking what the C ABI takes
    on trust: a 1-D, C-contiguous int32 numpy array in host memory (the library checks its values), or None."""
    if group_end is None:
        return 0, None
    if not isinstance(group_end, np.ndarray) or group_end.dtype != np.int32 or group_end.ndim != 1:
        raise ValueError('group_end must be a 1-D int32 numpy array (host memory)')
    if not group_end.flags['C_CONTIGUOUS']:
        raise ValueError('group_end must be C-contiguous')
    return int(group_end.size), (group_end.ctypes.data if group_end.size else None)


def band_weights_array(weights, nlam):
    """Band weights as a C-contiguous float64 array [nband, nlam] (one band from a 1-D array, [0, nlam] from None);
    the library checks their values."""
    if weights is None:
        return np.empty((0, int(nlam)))
    w = np.array(weights, dtype=np.float64, ndmin=2, order='C')
    if w.ndim != 2 or w.shape[1] != int(nlam):
        raise ValueError('band weights must be [nband, %d] (got shape %s)' % (int(nlam), w.shape))
    return w


def checked_ptr(a, count, device, name, writable=False):
    """Address of a caller-supplied FP64 buffer after checking what the C ABI takes on trust:
    dtype float64, C-contiguous, at least ``count`` elements, and - for a torch tensor - host
    memory or the context's own GPU.  ``None`` passes through (optional outputs)."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        if a.dtype != np.float64:
            raise ValueError('%s must be float64 (got %s)' % (name, a.dtype))
        if not a.flags['C_CONTIGUOUS']:
            raise ValueError('%s must be C-contiguous' % name)
        if writable and not a.flags['WRITEABLE']:
            raise ValueError('%s is read-only' % name)
        if a.size < count:
            raise ValueError('%s holds %d elements, %d are needed' % (name, a.size, count))
        return a.ctypes.data
    if hasattr(a, 'data_ptr'):      # torch tensor used purely as a buffer carrier
        if 'float64' not in str(a.dtype):
            raise ValueError('%s must be float64 (got %s)' % (name, a.dtype))
        if not a.is_contiguous():
            raise ValueError('%s must be contiguous' % name)
        if a.numel() < count:
            raise ValueError('%s holds %d elements, %d are needed' % (name, a.numel(), count))
        dev = a.device
        if dev.type == 'cuda':
            if dev.index is not None and dev.index != device:
                raise ValueError('%s lives on cuda:%d but the context runs on cuda:%d' % (name, dev.index, device))
        elif dev.type != 'cpu':
            raise ValueError('%s lives on unsupported device %s' % (name, dev))
        return a.data_ptr()
    raise TypeError('%s: unsupported buffer type %r (numpy array or torch tensor expected)' % (name, type(a)))


class Context:
    """One psfr_ctx: twiddles, telescope OTF and workspaces on one GPU.

    The Python object outlives capacity changes: ``ensure`` rebuilds the native context in place
    (geometry and options are re-applied), so a caller holding a Context never ends up with a
    dead handle because somebody else asked for more planes."""

    def __init__(self, device=0, dim=1280, max_planes=16, max_lambda=35):
        self._lib = load()
        self._h = None
        self._geom = None
        self._opts = {}
        self.device = int(device)
        self.dim = int(dim)
        self._create(int(max_planes), int(max_lambda))

    def _create(self, max_planes, max_lambda):
        handle = _P()
        rc = self._lib.psfr_create(self.device, self.dim, max_planes, max_lambda, ctypes.byref(handle))
        if rc != 0:
            raise PsfrError(rc, self._lib.psfr_last_error(None).decode())
        self._h = handle
        self.max_planes = max_planes
        self.max_lambda = max_lambda
        if self._geom is not None:
            self.set_geometry(*self._geom)
        for key, value in self._opts.items():
            self._check(self._lib.psfr_set_option(self._h, key, value))

    def ensure(self, max_planes=None, max_lambda=None):
        """Grow the workspaces (never shrink) so that they hold max_planes x max_lambda."""
        planes = max(self.max_planes, int(max_planes or 0))
        lam = max(self.max_lambda, int(max_lambda or 0))
        if planes != self.max_planes or lam != self.max_lambda or not self._h:
            self.close()
            self._create(planes, lam)
        return self

    def close(self):
        if getattr(self, '_h', None):
            self._lib.psfr_destroy(self._h)
            self._h = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise PsfrError(rc, self._lib.psfr_last_error(self._h).decode())

    def _handle(self):
        if not self._h:
            raise PsfrError(E_STATE, 'the context has been closed')
        return self._h

    def _buf(self, a, count, name, writable=False):
        return checked_ptr(a, int(count), self.device, name, writable)

    # thin wrappers -------------------------------------------------------------------
    def set_geometry(self, f, f_x, f_y):
        f, f_x, f_y = f64(f), f64(f_x), f64(f_y)
        n = AO_DIM * AO_DIM
        self._check(self._lib.psfr_set_geometry(self._handle(), self._buf(f, n, 'f'), self._buf(f_x, n, 'f_x'),
                                                self._buf(f_y, n, 'f_y')))
        self._geom = (f, f_x, f_y)

    def psd(self, draws, dirs, poslgs, out=None, stream=None):
        draws, dirs, poslgs = f64(draws), f64(dirs), f64(poslgs)
        nd, ndir = draws.shape[0], dirs.shape[1]
        self._check(self._lib.psfr_psd(self._handle(), nd, ptr(draws), ndir, ptr(dirs), poslgs.shape[1], ptr(poslgs),
                                       self._buf(out, nd * ndir * self.dim * self.dim, 'out', True), stream))

    def load_psd(self, psd, nplanes, stream=None):
        self._check(self._lib.psfr_load_psd(self._handle(), int(nplanes),
                                            self._buf(psd, int(nplanes) * self.dim * self.dim, 'psd'), stream))

    def structure_function(self, nplanes, stream=None):
        self._check(self._lib.psfr_structure_function(self._handle(), int(nplanes), stream))

    def psd_to_psf(self, plane, lambda_m, out, stream=None):
        self._check(self._lib.psfr_psd_to_psf(self._handle(), int(plane), float(lambda_m),
                                              self._buf(out, self.dim * self.dim, 'out', True), stream))

    def psf_cube(self, ndraw, ndir, lambda_nm, out, stream=None):
        lam = f64(lambda_nm)
        self._check(self._lib.psfr_psf_cube(self._handle(), int(ndraw), int(ndir), lam.size, ptr(lam),
                                            self._buf(out, int(ndraw) * lam.size * PSF_DIM * PSF_DIM, 'out', True), stream))

    def convolve(self, ndraw, lambda_nm, alpha_tt, cube, out, stream=None):
        lam, att = f64(lambda_nm), f64(alpha_tt)
        n = int(ndraw) * lam.size * PSF_DIM * PSF_DIM
        if att.size < int(ndraw):
            raise ValueError('alpha_tt holds %d values for %d draws' % (att.size, ndraw))
        self._check(self._lib.psfr_convolve(self._handle(), int(ndraw), lam.size, ptr(lam), ptr(att),
                                            self._buf(cube, n, 'cube'), self._buf(out, n, 'out', True), stream))

    def moffat_fit(self, nimg, ny, nx, imgs, params, stream=None):
        nimg, ny, nx = int(nimg), int(ny), int(nx)
        self._check(self._lib.psfr_moffat_fit(self._handle(), nimg, ny, nx, self._buf(imgs, nimg * ny * nx, 'imgs'),
                                              self._buf(params, nimg * FIT_NPAR, 'params', True), stream))

    def moffat_fit_elliptical(self, nimg, ny, nx, imgs, params, stream=None):
        """psfr_moffat_fit_elliptical: ``params`` [nimg, EFIT_NPAR]."""
        nimg, ny, nx = int(nimg), int(ny), int(nx)
        self._check(self._lib.psfr_moffat_fit_elliptical(
            self._handle(), nimg, ny, nx, self._buf(imgs, nimg * ny * nx, 'imgs'),
            self._buf(params, nimg * EFIT_NPAR, 'params', True), stream))

    def moffat_fit_weighted(self, nimg, ny, nx, imgs, weights, params, back=None, fit_back=False, elliptical=False,
                            stream=None):
        """psfr_moffat_fit_weighted: ``weights`` [nimg, ny, nx] or None (every weight 1); ``params`` [nimg, FIT_NPAR]
        or, with ``elliptical``, [nimg, EFIT_NPAR]; ``back`` [nimg, BACK_NPAR] or None."""
        nimg, ny, nx = int(nimg), int(ny), int(nx)
        npar = EFIT_NPAR if elliptical else FIT_NPAR
        self._check(self._lib.psfr_moffat_fit_weighted(
            self._handle(), nimg, ny, nx, self._buf(imgs, nimg * ny * nx, 'imgs'),
            self._buf(weights, nimg * ny * nx, 'weights'), int(bool(fit_back)), int(bool(elliptical)),
            self._buf(params, nimg * npar, 'params', True), self._buf(back, nimg * BACK_NPAR, 'back', True), stream))

    def template_fit(self, nimg, ny, nx, imgs, weights, tpls, params, model=None, fit_back=False, stream=None):
        """psfr_template_fit: ``weights`` [nimg, ny, nx] or None (every weight 1); ``tpls`` [ntpl, ty, tx] with nimg a
        multiple of ntpl (image i uses template i % ntpl); ``params`` [nimg, TFIT_NPAR]; ``model`` [nimg, ny, nx] or
        None."""
        nimg, ny, nx = int(nimg), int(ny), int(nx)
        ntpl, ty, tx = (int(v) for v in tpls.shape)
        self._check(self._lib.psfr_template_fit(
            self._handle(), nimg, ny, nx, self._buf(imgs, nimg * ny * nx, 'imgs'),
            self._buf(weights, nimg * ny * nx, 'weights'), ntpl, ty, tx, self._buf(tpls, ntpl * ty * tx, 'tpls'),
            int(bool(fit_back)), self._buf(params, nimg * TFIT_NPAR, 'params', True),
            self._buf(model, nimg * ny * nx, 'model', True), stream))

    def encircled_energy(self, nimg, ny, nx, imgs, radii_px, fracs, out, centres=None, stream=None):
        """psfr_encircled_energy: ``out`` [nimg, len(radii_px) + 1 + len(fracs)]; ``centres`` [nimg, 2] (y0, x0)
        in pixels or None for (ny // 2, nx // 2)."""
        nimg, ny, nx = int(nimg), int(ny), int(nx)
        rad, fr = f64(radii_px).ravel(), f64(fracs).ravel()
        rec = ee_slots(rad.size, fr.size)[3]
        self._check(self._lib.psfr_encircled_energy(
            self._handle(), nimg, ny, nx, self._buf(imgs, nimg * ny * nx, 'imgs'),
            self._buf(centres, 2 * nimg, 'centres'), rad.size, ptr(rad) if rad.size else None, fr.size,
            ptr(fr) if fr.size else None, self._buf(out, nimg * rec, 'out', True), stream))

    def compute_energy(self, field, draws, dirs, poslgs, lambda_nm, radii_px, fracs, group_end=None, out_cube=None,
                       out_fit=None, out_mean=None, out_mean_fit=None, out_efit=None, out_mean_efit=None, out_ee=None,
                       out_mean_ee=None, stream=None):
        """psfr_compute_energy: ``compute_groups`` (``field`` false) or ``compute_field`` (``field`` true) with the
        encircled-energy records of every returned image, ``out_ee`` [ndraw, P, nl, rec] and ``out_mean_ee``
        [ngroup, P, nl, rec] (P = npos with ``field``, 1 without; rec = len(radii_px) + 1 + len(fracs)), and the
        elliptical fits ``out_efit`` / ``out_mean_efit`` of ``compute_field``."""
        rad, fr = f64(radii_px).ravel(), f64(fracs).ravel()
        self._groups(self._lib.psfr_compute_energy, bool(field), draws, dirs, poslgs, lambda_nm, group_end, out_cube,
                     out_fit, out_mean, out_mean_fit, stream, shapes=(out_efit, out_mean_efit),
                     energy=(rad, fr, out_ee, out_mean_ee))

    def compute_ao(self, field, draws, dirs, poslgs, lambda_nm, radii_px=(), fracs=(), group_end=None,
                   out_cube=None, out_fit=None, out_mean=None, out_mean_fit=None, out_efit=None, out_mean_efit=None,
                   out_ee=None, out_mean_ee=None, out_strehl=None, out_var=None, stream=None):
        """psfr_compute_ao: ``compute_energy`` plus the Strehl ratio of every PSF it forms, ``out_strehl`` [ndraw, P,
        nl] (P = npos with ``field``, 1 without), and the variance record of every (draw, direction) plane,
        ``out_var`` [ndraw, ndir, VAR_NPAR] in nm^2 (``VAR_*``)."""
        rad, fr = f64(radii_px).ravel(), f64(fracs).ravel()
        self._groups(self._lib.psfr_compute_ao, bool(field), draws, dirs, poslgs, lambda_nm, group_end, out_cube,
                     out_fit, out_mean, out_mean_fit, stream, shapes=(out_efit, out_mean_efit),
                     energy=(rad, fr, out_ee, out_mean_ee), ao=(out_strehl, out_var))

    def compute_bands(self, field, draws, dirs, poslgs, lambda_nm, weights, radii_px=(), fracs=(), group_end=None,
                      out_cube=None, out_fit=None, out_mean=None, out_mean_fit=None, out_efit=None, out_mean_efit=None,
                      out_ee=None, out_mean_ee=None, out_strehl=None, out_var=None, out_band=None, out_band_fit=None,
                      out_band_ee=None, out_mean_band=None, out_mean_band_fit=None, out_mean_band_ee=None,
                      stream=None):
        """psfr_compute_bands: ``compute_ao`` plus the band images of every image set it forms for the weights
        [nband, nl] (or None: no bands), ``out_band`` [ndraw, P, nband, 40, 40], ``out_band_fit`` [ndraw, P, nband,
        FIT_NPAR], ``out_band_ee`` [ndraw, P, nband, rec], and the same of the exposure means, ``out_mean_band*``
        [ngroup, P, nband, ...] (P = npos with ``field``, 1 without)."""
        rad, fr = f64(radii_px).ravel(), f64(fracs).ravel()
        self._groups(self._lib.psfr_compute_bands, bool(field), draws, dirs, poslgs, lambda_nm, group_end, out_cube,
                     out_fit, out_mean, out_mean_fit, stream, shapes=(out_efit, out_mean_efit),
                     energy=(rad, fr, out_ee, out_mean_ee), ao=(out_strehl, out_var),
                     bands=(weights, out_band, out_band_fit, out_band_ee, out_mean_band, out_mean_band_fit,
                            out_mean_band_ee))

    def band_psf(self, ncube, nlam, ny, nx, cubes, weights, out, stream=None):
        """psfr_band_psf: band images ``out`` [ncube, nband, ny, nx] of ``cubes`` [ncube, nlam, ny, nx] for the
        weights [nband, nlam]."""
        ncube, nlam, ny, nx = int(ncube), int(nlam), int(ny), int(nx)
        w = band_weights_array(weights, nlam)
        self._check(self._lib.psfr_band_psf(self._handle(), ncube, nlam, ny, nx,
                                            self._buf(cubes, ncube * nlam * ny * nx, 'cubes'), w.shape[0],
                                            ptr(w) if w.size else None,
                                            self._buf(out, ncube * w.shape[0] * ny * nx, 'out', True), stream))

    def compute_batch(self, draws, dirs, poslgs, lambda_nm, out_cube=None, out_fit=None, stream=None):
        if not hasattr(draws, 'data_ptr'):      # numpy / sequence; torch tensors pass through as buffers
            draws = f64(draws)
        if len(draws.shape) != 2 or draws.shape[1] != DRAW_NPAR:
            raise ValueError('draws must be [ndraw, %d]' % DRAW_NPAR)
        dirs, poslgs, lam = f64(dirs), f64(poslgs), f64(lambda_nm)
        nd = int(draws.shape[0])
        self._check(self._lib.psfr_compute_batch(
            self._handle(), nd, self._buf(draws, nd * DRAW_NPAR, 'draws'), dirs.shape[1], ptr(dirs),
            poslgs.shape[1], ptr(poslgs), lam.size, ptr(lam),
            self._buf(out_cube, nd * lam.size * PSF_DIM * PSF_DIM, 'out_cube', True),
            self._buf(out_fit, nd * lam.size * FIT_NPAR, 'out_fit', True), stream))

    def compute_groups(self, draws, dirs, poslgs, lambda_nm, group_end=None, out_cube=None, out_fit=None,
                       out_mean=None, out_mean_fit=None, stream=None):
        """psfr_compute_groups: ``draws`` [ndraw, DRAW_NPAR] with each draw's guide-star count in slot
        DRAW_NGS (first stars of ``poslgs`` [2, npos]), exposures closed at the draw indices of
        ``group_end`` (int32); per-draw outputs as ``compute_batch``, per-exposure ``out_mean``
        [ngroup, nl, 40, 40] and ``out_mean_fit`` [ngroup, nl, FIT_NPAR]."""
        self._groups(self._lib.psfr_compute_groups, False, draws, dirs, poslgs, lambda_nm, group_end, out_cube,
                     out_fit, out_mean, out_mean_fit, stream)

    def compute_field(self, draws, dirs, poslgs, lambda_nm, group_end=None, out_cube=None, out_fit=None,
                      out_mean=None, out_mean_fit=None, stream=None, out_efit=None, out_mean_efit=None):
        """psfr_compute_field: ``compute_groups`` with one PSF per field position of ``dirs`` [2, npos]
        instead of their average.  Outputs ``out_cube`` [ndraw, npos, nl, 40, 40], ``out_fit`` [ndraw, npos,
        nl, FIT_NPAR], ``out_mean`` [ngroup, npos, nl, 40, 40], ``out_mean_fit`` [ngroup, npos, nl, FIT_NPAR].
        ``out_efit`` [ndraw, npos, nl, EFIT_NPAR] and ``out_mean_efit`` [ngroup, npos, nl, EFIT_NPAR], the
        elliptical fits of the same images, bind psfr_compute_field_shapes instead."""
        if out_efit is None and out_mean_efit is None:
            self._groups(self._lib.psfr_compute_field, True, draws, dirs, poslgs, lambda_nm, group_end, out_cube,
                         out_fit, out_mean, out_mean_fit, stream)
        else:
            self._groups(self._lib.psfr_compute_field_shapes, True, draws, dirs, poslgs, lambda_nm, group_end,
                         out_cube, out_fit, out_mean, out_mean_fit, stream, shapes=(out_efit, out_mean_efit))

    def _groups(self, fn, field, draws, dirs, poslgs, lambda_nm, group_end, out_cube, out_fit, out_mean,
                out_mean_fit, stream, shapes=None, energy=None, ao=None, bands=None):
        if not hasattr(draws, 'data_ptr'):
            draws = f64(draws)
        if len(draws.shape) != 2 or draws.shape[1] != DRAW_NPAR:
            raise ValueError('draws must be [ndraw, %d]' % DRAW_NPAR)
        dirs, poslgs, lam = f64(dirs), f64(poslgs), f64(lambda_nm)
        nd = int(draws.shape[0])
        ng, gp = group_end_ptr(group_end)
        nimg = lam.size * (dirs.shape[1] if field else 1)      # images per draw and per exposure
        img = nimg * PSF_DIM * PSF_DIM
        args = [self._handle(), nd, self._buf(draws, nd * DRAW_NPAR, 'draws'), poslgs.shape[1], ptr(poslgs),
                dirs.shape[1], ptr(dirs), lam.size, ptr(lam), ng, gp]
        if energy is not None:
            rad, fr = energy[0], energy[1]
            args = args[:1] + [int(field)] + args[1:] + [rad.size, ptr(rad) if rad.size else None, fr.size,
                                                         ptr(fr) if fr.size else None]
        args += [self._buf(out_cube, nd * img, 'out_cube', True),
                 self._buf(out_fit, nd * nimg * FIT_NPAR, 'out_fit', True),
                 self._buf(out_mean, ng * img, 'out_mean', True),
                 self._buf(out_mean_fit, ng * nimg * FIT_NPAR, 'out_mean_fit', True)]
        if shapes is not None:
            args += [self._buf(shapes[0], nd * nimg * EFIT_NPAR, 'out_efit', True),
                     self._buf(shapes[1], ng * nimg * EFIT_NPAR, 'out_mean_efit', True)]
        if energy is not None:
            rec = ee_slots(energy[0].size, energy[1].size)[3]
            args += [self._buf(energy[2], nd * nimg * rec, 'out_ee', True),
                     self._buf(energy[3], ng * nimg * rec, 'out_mean_ee', True)]
        if ao is not None:
            args += [self._buf(ao[0], nd * nimg, 'out_strehl', True),
                     self._buf(ao[1], nd * dirs.shape[1] * VAR_NPAR, 'out_var', True)]
        if bands is not None:
            w = band_weights_array(bands[0], lam.size)
            sets = w.shape[0] * (dirs.shape[1] if field else 1)     # band images per draw and per exposure
            rec = ee_slots(energy[0].size, energy[1].size)[3]
            args += [w.shape[0], ptr(w) if w.size else None]
            img1 = PSF_DIM * PSF_DIM
            for name, a, n, per in (('out_band', bands[1], nd, img1), ('out_band_fit', bands[2], nd, FIT_NPAR),
                                    ('out_band_ee', bands[3], nd, rec), ('out_mean_band', bands[4], ng, img1),
                                    ('out_mean_band_fit', bands[5], ng, FIT_NPAR),
                                    ('out_mean_band_ee', bands[6], ng, rec)):
                args.append(self._buf(a, n * sets * per, name, True))
        self._check(fn(*args, stream))

    def mean_refit(self, ncube, nlam, cubes, out_mean=None, out_fit=None, stream=None):
        ncube, nlam = int(ncube), int(nlam)
        img = PSF_DIM * PSF_DIM
        self._check(self._lib.psfr_mean_refit(self._handle(), ncube, nlam, self._buf(cubes, ncube * nlam * img, 'cubes'),
                                              self._buf(out_mean, nlam * img, 'out_mean', True),
                                              self._buf(out_fit, nlam * FIT_NPAR, 'out_fit', True), stream))

    def polyfit(self, lambda_nm, deg, y, stream=None):
        lam, y = f64(lambda_nm), f64(np.atleast_2d(y))
        if y.shape[1] != lam.size:
            raise ValueError('y must hold one value per wavelength')
        coef = np.empty((y.shape[0], deg + 1))
        self._check(self._lib.psfr_polyfit(self._handle(), y.shape[0], lam.size, ptr(lam), int(deg), ptr(y), ptr(coef), stream))
        return coef

    def set_option(self, key, value):
        self._check(self._lib.psfr_set_option(self._handle(), int(key), float(value)))
        self._opts[int(key)] = float(value)

    def get_otf(self):
        out = np.empty((self.dim // 2 + 2, self.dim))
        self._check(self._lib.psfr_get_otf(self._handle(), ptr(out)))
        return out

    def get_structure_function(self, plane):
        out = np.empty((self.dim // 2 + 2, self.dim))
        self._check(self._lib.psfr_get_structure_function(self._handle(), int(plane), ptr(out)))
        return out

    def debug_exp(self, x):
        x = f64(x)
        y = np.empty_like(x)
        self._check(self._lib.psfr_debug_exp(self._handle(), x.size, ptr(x), ptr(y)))
        return y

    def info(self):
        """Numeric properties of the native context (psfr_get_info) as a dict."""
        out = {}
        for name, key in INFO_KEYS.items():
            v = _D()
            self._check(self._lib.psfr_get_info(self._handle(), key, ctypes.byref(v)))
            out[name] = v.value
        return out

    def kernel_launches(self):
        return int(self._lib.psfr_kernel_launches(self._handle()))

    def last_hot_timing(self):
        ms, n, psfs = _D(), _I(), ctypes.c_longlong()
        self._check(self._lib.psfr_last_hot_timing(self._handle(), ctypes.byref(ms), ctypes.byref(n), ctypes.byref(psfs)))
        return ms.value, n.value, psfs.value
