"""Host-side mirror of the reference's ``muse_psfr/psfrec.py`` for the PSF-reconstruction
hot path: same function names, argument meaning and error behaviour, computed by the
sm_100a CUDA library behind the C ABI of ``include/psfr.h``.

Only scalar bookkeeping happens here (per-draw constants such as r0, the 80x80
frequency tables whose 1-ulp rounding the reference's cut-off masks depend on, result
packaging).  Every array-sized computation runs on the GPU; there is no CPU fallback.
"""
import logging
import os
from math import gamma

import numpy as np

from . import _fits, _lib
from ._lib import PsfrError

__all__ = ['compute_psf_from_sparta', 'compute_psf_from_sparta_batch', 'compute_psf', 'compute_psf_batch',
           'reconstruct_psf', 'create_sparta_table', 'fit_psf_with_polynom', 'simul_psd_wfm', 'psd_to_psf', 'psf_muse',
           'convolve_final_psf', 'fit_psf_cube', 'fit_psf_template', 'compute_psf_field', 'encircled_energy',
           'band_weights', 'band_psf',
           'muse_intrinsic_psf', 'direction_perf', 'seeing2r01', 'pupil_mask', 'select_sparta_rows', 'FitTable',
           'PsfrError', 'MIN_L0', 'MAX_L0']

logger = logging.getLogger('muse_psfr.psfrec')   # the reference's logger name (tests assert on it)

MIN_L0 = 8    # psfrec.py:30-31
MAX_L0 = 30

_HERE = os.path.dirname(os.path.abspath(__file__))
_WIND_DIR = np.array([0.628163, -0.326497])      # psfrec.py:66
_DIM = 1280                                      # psfrec.py:955 (compute_psf's fixed grid)
_DIMS = (1280, 2560)                             # grids the CUDA library is built for
_MAX_POSITIONS = 256                             # directions per draw the library takes (kMaxDir)
_PIXSCALE = 0.2                                  # arcsec per pixel of the 40 x 40 PSFs (psfrec.py:901)
_CONTEXTS = {}
_DEFAULT_DEVICE = [None]


# --------------------------------------------------------------------------- contexts
def set_device(device):
    """Select the GPU used by the module-level functions (default: LOCAL_RANK or 0)."""
    _DEFAULT_DEVICE[0] = int(device)


def _device():
    if _DEFAULT_DEVICE[0] is None:
        _DEFAULT_DEVICE[0] = int(os.environ.get('LOCAL_RANK', '0'))
    return _DEFAULT_DEVICE[0]


def _check_dim(dim):
    if int(dim) not in _DIMS:
        raise NotImplementedError('this build supports dim in %s only (got %r)' % (_DIMS, dim))
    return int(dim)


def get_context(max_planes=None, max_lambda=None, device=None, dim=_DIM):
    """Context cache: one context per (device, dim).  ``max_planes`` / ``max_lambda`` are minimum
    capacities - ``None`` means "whatever exists" - and a cached context only ever grows, in place
    (``Context.ensure``): objects handed out earlier stay valid."""
    device = _device() if device is None else int(device)
    dim = _check_dim(dim)
    ctx = _CONTEXTS.get((device, dim))
    if ctx is None:
        ctx = _lib.Context(device=device, dim=dim, max_planes=max_planes or (16 if dim == _DIM else 4),
                           max_lambda=max(35, max_lambda or 0))
        ctx.set_geometry(*ao_frequency_tables())
        _CONTEXTS[(device, dim)] = ctx
    else:
        ctx.ensure(max_planes, max_lambda)
    return ctx


def release_contexts():
    for ctx in _CONTEXTS.values():
        ctx.close()
    _CONTEXTS.clear()


# --------------------------------------------------------------------------- scalar helpers
def seeing2r01(seeing, lbda, zenith):
    """seeing @ 0.5 microns, lambda in microns (psfrec.py:183-187)."""
    r00p5 = 0.976 * 0.5 / seeing / 4.85
    return r00p5 * (lbda * 2) ** (6 / 5) * np.cos(np.deg2rad(zenith)) ** (3 / 5)


def direction_perf(npts, field_size=60, plot=False, lgs=None, ngs=None, ax=None):
    """Grid of directions where the PSF is estimated (psfrec.py:154-180).  The plotting
    branch of the reference (matplotlib) is outside the hot path and not provided."""
    if plot:
        raise NotImplementedError('plotting is outside the B200 hot path')
    x, y = (np.mgrid[:npts, :npts] - npts // 2) * field_size / 2
    return np.array([x, y]).reshape(2, -1)


def pupil_mask(radius, width, oc=0, inverse=False):
    """Annular pupil (psfrec.py:190-203); host helper kept for API parity - the library
    builds its own pupil and telescope OTF on the device."""
    center = (width - 1) / 2
    x, y = np.ogrid[:int(width), :int(width)]
    rho = np.hypot(x - center, y - center) / radius
    mask = (rho < 1) & (rho >= oc)
    return (~mask if inverse else mask).astype(int)


def ao_frequency_tables(dimall=80, step=8. / 40):
    """f, f_x, f_y of the AO zone, formed exactly as psfrec.py:548-554 and 241-242."""
    fx = np.fft.fftfreq(int(dimall), step)[:, np.newaxis]
    fy = fx.T
    f = np.sqrt(fx ** 2 + fy ** 2)
    with np.errstate(all='ignore'):
        arg_f = fy / fx
    arg_f[0, 0] = 0
    arg_f = np.arctan(arg_f)
    return f, f * np.cos(arg_f), f * np.sin(arg_f)


def _lgs_positions(three_lgs_mode):
    if three_lgs_mode:
        poslgs = np.array([[1, 1], [-1, -1], [-1, 1]], dtype=float).T
    else:
        poslgs = np.array([[1, 1], [-1, -1], [-1, 1], [1, -1]], dtype=float).T
    return poslgs * 63.          # psfrec.py:83-93


_COEFF = [None]


def _coeff_hl(L0):
    """coeffHL(L0) from the reference's coeffL0 calibration table (psfrec.py:895-897)."""
    if _COEFF[0] is None:
        tab = np.loadtxt(os.path.join(_HERE, 'data', 'coeffL0.txt'), dtype=np.float32)
        _COEFF[0] = (np.arange(1, tab.size + 1, dtype=np.float32), tab)
    return np.interp(L0, *_COEFF[0])


def tiptilt_alpha(seeing, GL, L0):
    """Moffat alpha [px] of the residual tip-tilt kernel, beta = 2 (psfrec.py:879-905)."""
    beta_tt = 2
    seeingHL = seeing * (1 - GL) ** (3. / 5.)
    r0HL = 0.976 * 0.5 / seeingHL / 4.85
    coeffHL = _coeff_hl(L0)
    pixscale = 0.2
    fwhmTTopt = (np.sqrt(coeffHL * 0.97 * 6.88 * (.5 * 1.e-6 / (2. * np.pi)) ** 2 *
                         8 ** (-1 / 3.) * r0HL ** (-5 / 3.)) / (4.85 * 1.e-6) * 2.35 / pixscale)
    return fwhmTTopt / (2 * np.sqrt(2 ** (1. / beta_tt) - 1))


def _wind_vectors(h_arr, wind_dir):
    """Wind vector per layer [2, nl]: 12.5 m/s (12 for integer altitudes, as ``np.full_like(h, 12.5)``
    does in the reference, psfrec.py:60-61) along the reference's two hard-coded directions
    (psfrec.py:66) or along ``wind_dir`` [rad] - required beyond two layers, where the reference
    itself fails (ValueError from broadcasting at psfrec.py:594)."""
    nl = h_arr.shape[-1]
    if wind_dir is None:
        if nl > 2:
            raise ValueError('operands could not be broadcast together: the reference has wind directions for '
                             '2 layers only; pass wind_dir= (one angle [rad] per layer) for more')
        arg_v = _WIND_DIR[:nl]
    else:
        arg_v = np.asarray(wind_dir, dtype=float)
        if arg_v.shape != (nl,):
            raise ValueError('wind_dir must hold one angle [rad] per layer')
    vent = np.full_like(h_arr, 12.5)
    return np.stack([vent * np.cos(arg_v), vent * np.sin(arg_v)])


def draw_record(Cn2, h, seeing, L0, zenith=0., alpha_tt=1.0, wind_dir=None):
    """Per-draw constants of simul_psd_wfm / dsp4muse / psd_fit, evaluated with the
    reference's own scalar expressions (psfrec.py:57-66, 108, 569-571, 594, 622-625)."""
    Cn2 = np.array(Cn2, dtype=float)
    Cn2 = Cn2 / Cn2.sum()
    h_arr = np.array(h)
    if h_arr.ndim != 1 or h_arr.size != Cn2.size:
        raise ValueError('Cn2 and h must be 1-D sequences of the same length')
    if h_arr.size > _lib.MAX_LAYERS:
        raise ValueError('at most %d turbulence layers are supported' % _lib.MAX_LAYERS)
    wind = _wind_vectors(h_arr, wind_dir)
    r0ref = seeing2r01(seeing, 0.5, zenith)
    rec = np.zeros(_lib.DRAW_NPAR)
    rec[_lib.DRAW_R0] = r0ref
    rec[_lib.DRAW_L0] = L0
    cst = ((gamma(11 / 6) ** 2 / (2 * np.pi ** (11 / 3))) * (24 * gamma(6 / 5) / 5) ** (5 / 6))
    rec[_lib.DRAW_FITC] = cst * r0ref ** (-5 / 3)
    for l in range(h_arr.size):
        rec[_lib.layer_slot(l, _lib.LAYER_CPHI)] = 0.0229 * (Cn2[l] ** (-3 / 5) * r0ref) ** (-5 / 3)
        rec[_lib.layer_slot(l, _lib.LAYER_H)] = float(h_arr[l])
        rec[_lib.layer_slot(l, _lib.LAYER_WX)] = wind[0, l]
        rec[_lib.layer_slot(l, _lib.LAYER_WY)] = wind[1, l]
    rec[_lib.DRAW_ALPHA_TT] = alpha_tt
    rec[_lib.DRAW_NLAYERS] = h_arr.size
    return rec


def draw_records(seeing, GL, L0, h=(100, 10000), zenith=0., Cn2=None, wind_dir=None):
    """Vectorised ``draw_record``.  Default profile: compute_psf's two layers Cn2 = [GL, 1 - GL]
    (psfrec.py:953); ``Cn2`` ([nl] or [ndraw, nl]) replaces it.  ``h`` is one altitude per layer or an
    array [ndraw, nl].  Same expressions as the scalar version evaluated with numpy's array kernels,
    which may differ from libm's scalar pow() by a few ulp (measured <= 3 ulp on the pow chains)."""
    seeing, GL, L0 = (np.atleast_1d(np.asarray(v, dtype=float)) for v in (seeing, GL, L0))
    nd = seeing.size
    h_arr = np.array(h)
    cn2 = np.stack([GL, 1 - GL], axis=1) if Cn2 is None else np.broadcast_to(np.asarray(Cn2, dtype=float),
                                                                               (nd, np.shape(Cn2)[-1]))
    nl = cn2.shape[1]
    if h_arr.shape[-1] != nl or h_arr.ndim > 2:
        raise ValueError('operands could not be broadcast together: h must hold %d layer altitudes' % nl)
    if nl > _lib.MAX_LAYERS:
        raise ValueError('at most %d turbulence layers are supported' % _lib.MAX_LAYERS)
    wx, wy = _wind_vectors(h_arr, wind_dir)
    cn2 = cn2 / cn2.sum(axis=1)[:, None]
    r0ref = seeing2r01(seeing, 0.5, zenith)
    cst = ((gamma(11 / 6) ** 2 / (2 * np.pi ** (11 / 3))) * (24 * gamma(6 / 5) / 5) ** (5 / 6))
    recs = np.zeros((nd, _lib.DRAW_NPAR))
    recs[:, _lib.DRAW_R0] = r0ref
    recs[:, _lib.DRAW_L0] = L0
    recs[:, _lib.DRAW_FITC] = cst * r0ref ** (-5 / 3)
    for l in range(nl):
        recs[:, _lib.layer_slot(l, _lib.LAYER_CPHI)] = 0.0229 * (cn2[:, l] ** (-3 / 5) * r0ref) ** (-5 / 3)
        recs[:, _lib.layer_slot(l, _lib.LAYER_H)] = h_arr[..., l]
        recs[:, _lib.layer_slot(l, _lib.LAYER_WX)] = wx[..., l]
        recs[:, _lib.layer_slot(l, _lib.LAYER_WY)] = wy[..., l]
    recs[:, _lib.DRAW_ALPHA_TT] = tiptilt_alpha(seeing, GL, L0)
    recs[:, _lib.DRAW_NLAYERS] = nl
    return recs


# --------------------------------------------------------------------------- result table
class FitTable:
    """Column store with the columns of the reference's ``fit_psf_cube`` table
    (psfrec.py:866-870).  ``to_astropy()`` converts when astropy is installed."""

    def __init__(self, columns, meta=None):
        self._cols = dict(columns)
        self.meta = dict(meta or {})

    @property
    def colnames(self):
        return list(self._cols)

    def __len__(self):
        return len(next(iter(self._cols.values())))

    def __getitem__(self, key):
        if isinstance(key, str):
            return self._cols[key]
        if isinstance(key, (int, np.integer)):
            return {k: v[key] for k, v in self._cols.items()}
        return FitTable({k: v[key] for k, v in self._cols.items()}, self.meta)

    def __setitem__(self, key, value):
        n = len(self) if self._cols else None
        arr = np.asarray(value)
        self._cols[key] = np.full(n, value) if arr.ndim == 0 and n is not None else arr

    def to_astropy(self):
        from astropy.table import Table
        return Table(self._cols, meta=self.meta)

    @staticmethod
    def vstack(tables):
        names = tables[0].colnames
        return FitTable({k: np.concatenate([np.atleast_1d(t[k]) for t in tables]) for k in names},
                        tables[0].meta)


def _table_from_fit(lbda, fit, pixscale=0.2):
    """Columns of the reference's fit table (psfrec.py:866-870: mpdaf Moffat2D attributes minus
    ima / rot / cont / err_rot / err_cont, fwhm and err_fwhm x 0.2) plus ``converged``, an extension:
    0 where the Levenberg-Marquardt iteration ran out of steps (PSFR_FIT_ITER < 0); such rows are
    also reported by a warning on the module logger."""
    fwhm = fit[:, _lib.FIT_FWHM] * pixscale
    efw = fit[:, _lib.FIT_ERR_FWHM] * pixscale
    converged = fit[:, _lib.FIT_ITER] > 0
    if not converged.all():
        bad = np.flatnonzero(~converged)
        logger.warning('Moffat fit did not converge for %d of %d images (first at index %d)',
                       bad.size, len(fit), bad[0])
    return FitTable({
        'lbda': np.asarray(lbda, dtype=float),
        'center': fit[:, [_lib.FIT_Y0, _lib.FIT_X0]].copy(),
        'flux': fit[:, _lib.FIT_FLUX].copy(),
        'fwhm': np.stack([fwhm, fwhm], axis=1),
        'n': fit[:, _lib.FIT_N].copy(),
        'peak': fit[:, _lib.FIT_PEAK].copy(),
        'err_center': fit[:, [_lib.FIT_ERR_Y0, _lib.FIT_ERR_X0]].copy(),
        'err_flux': fit[:, _lib.FIT_ERR_FLUX].copy(),
        'err_fwhm': np.stack([efw, efw], axis=1),
        'err_n': fit[:, _lib.FIT_ERR_N].copy(),
        'err_peak': fit[:, _lib.FIT_ERR_PEAK].copy(),
        'converged': converged.astype(np.int64),
    })


def _shape_table_from_fit(lbda, efit, pixscale=0.2):
    """Columns of the elliptical fit (``fit_psf_cube(circular=False)``) for records [n, EFIT_NPAR]: ``fwhm`` and
    ``err_fwhm`` hold (major, minor) in arcsec in the reference's two-element columns, ``pa`` and ``err_pa``
    are in degrees (major axis from +x toward +y), ``center`` in pixels.  The reference has no elliptical
    fit: these columns are this package's own (DESIGN.md section 5.3).  ``converged`` as ``_table_from_fit``."""
    converged = efit[:, _lib.EFIT_ITER] > 0
    if not converged.all():
        bad = np.flatnonzero(~converged)
        logger.warning('elliptical Moffat fit did not converge for %d of %d images (first at index %d)',
                       bad.size, len(efit), bad[0])
    return FitTable({
        'lbda': np.asarray(lbda, dtype=float),
        'center': efit[:, [_lib.EFIT_Y0, _lib.EFIT_X0]].copy(),
        'fwhm': efit[:, [_lib.EFIT_FWHM_MAJOR, _lib.EFIT_FWHM_MINOR]] * pixscale,
        'axis_ratio': efit[:, _lib.EFIT_AXIS_RATIO].copy(),
        'pa': efit[:, _lib.EFIT_PA].copy(),
        'n': efit[:, _lib.EFIT_N].copy(),
        'peak': efit[:, _lib.EFIT_PEAK].copy(),
        'flux': efit[:, _lib.EFIT_FLUX].copy(),
        'err_center': efit[:, [_lib.EFIT_ERR_Y0, _lib.EFIT_ERR_X0]].copy(),
        'err_fwhm': efit[:, [_lib.EFIT_ERR_FWHM_MAJOR, _lib.EFIT_ERR_FWHM_MINOR]] * pixscale,
        'err_axis_ratio': efit[:, _lib.EFIT_ERR_AXIS_RATIO].copy(),
        'err_pa': efit[:, _lib.EFIT_ERR_PA].copy(),
        'err_n': efit[:, _lib.EFIT_ERR_N].copy(),
        'err_peak': efit[:, _lib.EFIT_ERR_PEAK].copy(),
        'err_flux': efit[:, _lib.EFIT_ERR_FLUX].copy(),
        'converged': converged.astype(np.int64),
    })


def _ee_params(radii, fractions, pixscale=_PIXSCALE):
    """Radii [arcsec] and fractions of an encircled-energy request, checked, as (radii [px], fractions)."""
    rad = np.array(radii, dtype=float, ndmin=1)
    frac = np.array(fractions, dtype=float, ndmin=1)
    if rad.ndim != 1 or frac.ndim != 1:
        raise ValueError('radii and fractions must be 1-D sequences')
    if rad.size > _lib.EE_MAX_RADII or frac.size > _lib.EE_MAX_FRACTIONS:
        raise ValueError('at most %d radii and %d fractions (got %d and %d)'
                         % (_lib.EE_MAX_RADII, _lib.EE_MAX_FRACTIONS, rad.size, frac.size))
    if not np.all(np.isfinite(rad)) or np.any(rad < 0):
        raise ValueError('radii must be finite and >= 0 (got %s)' % rad.tolist())
    if not np.all((frac > 0) & (frac < 1)):
        raise ValueError('fractions must lie in (0, 1) (got %s)' % frac.tolist())
    if not (np.isfinite(pixscale) and pixscale > 0):
        raise ValueError('pixscale must be positive')
    return np.ascontiguousarray(rad / pixscale), np.ascontiguousarray(frac)


def _ee_table(lbda, ee, radii, fractions, pixscale=_PIXSCALE):
    """Columns of the encircled-energy table for records [n, nrad + 1 + nfrac] (``_lib.ee_slots``): ``ee``
    [n, nrad] (flux inside each radius, in the images' units), ``ee_total`` (the sum of each image), ``r_ee``
    [n, nfrac] in arcsec.  ``radii`` [arcsec] and ``fractions`` go to the meta."""
    radii = np.array(radii, dtype=float, ndmin=1)
    fractions = np.array(fractions, dtype=float, ndmin=1)
    sl_ee, i_tot, sl_r, rec = _lib.ee_slots(radii.size, fractions.size)
    ee = np.asarray(ee).reshape(-1, rec)
    return FitTable({
        'lbda': np.asarray(lbda, dtype=float),
        'ee': ee[:, sl_ee].copy(),
        'ee_total': ee[:, i_tot].copy(),
        'r_ee': ee[:, sl_r] * pixscale,
    }, meta={'radii': radii, 'fractions': fractions})


def _ao_table(lbda, strehl, var):
    """Columns of the AO summary table (DESIGN.md section 5.5): ``strehl`` [n] (the AO Strehl ratio at each
    wavelength) and, from the variance records ``var`` [n, VAR_NPAR] or one record [VAR_NPAR] for every row, the
    residual-phase variance ``var_total`` = ``var_fit`` + ``var_noise`` + ``var_proj`` in nm^2 (independent of the
    wavelength; multiply by (2 pi / lbda_nm)^2 for rad^2)."""
    lbda = np.asarray(lbda, dtype=float)
    var = np.broadcast_to(np.asarray(var, dtype=float), (lbda.size, _lib.VAR_NPAR))
    return FitTable({
        'lbda': lbda,
        'strehl': np.asarray(strehl, dtype=float).reshape(lbda.size).copy(),
        'var_total': var[:, _lib.VAR_TOTAL].copy(),
        'var_fit': var[:, _lib.VAR_FIT].copy(),
        'var_noise': var[:, _lib.VAR_NOISE].copy(),
        'var_proj': var[:, _lib.VAR_PROJ].copy(),
    })


def band_weights(lbda, band_lbda, throughput):
    """Weights [nl] of one band on the wavelength grid ``lbda`` [nm] (DESIGN.md section 5.6): the trapezoid-rule
    quadrature of the throughput curve ``T = np.interp(lbda, band_lbda, throughput, left=0, right=0)`` on that grid,
    ``w_k = T(lbda_k) * delta_k`` with ``delta_k`` half the distance between the neighbours of k (of its one neighbour
    at either end; 1 for a single wavelength).  ``sum(w)`` is the trapezoid integral of T over the grid.

    A top-hat is ``band_lbda=[lo, hi], throughput=[1, 1]``; stack several calls for several bands.  The weights are
    those of a photon-flat source: an SED and photon-counting factors (such as lambda) are the caller's, folded into
    ``throughput``.  Raises ValueError for a grid (``lbda`` or ``band_lbda``) that is not strictly increasing, a
    negative or non-finite throughput, and a band that puts no weight on the grid."""
    lam = np.array(lbda, dtype=float, ndmin=1)
    bl = np.array(band_lbda, dtype=float, ndmin=1)
    tp = np.array(throughput, dtype=float, ndmin=1)
    for name, x in (('lbda', lam), ('band_lbda', bl)):
        if x.ndim != 1 or x.size == 0 or not np.all(np.isfinite(x)) or np.any(np.diff(x) <= 0):
            raise ValueError('%s must be a finite, strictly increasing 1-D grid' % name)
    if tp.shape != bl.shape:
        raise ValueError('throughput must hold one value per band_lbda (got %d for %d)' % (tp.size, bl.size))
    if not np.all(np.isfinite(tp)) or np.any(tp < 0):
        raise ValueError('throughput must be finite and >= 0')
    delta = np.ones(1)
    if lam.size > 1:
        delta = np.empty(lam.size)
        delta[0], delta[-1] = (lam[1] - lam[0]) / 2, (lam[-1] - lam[-2]) / 2
        delta[1:-1] = (lam[2:] - lam[:-2]) / 2
    w = np.interp(lam, bl, tp, left=0, right=0) * delta
    if not w.sum() > 0:
        raise ValueError('the band [%g, %g] nm puts no weight on the grid [%g, %g] nm' % (bl[0], bl[-1], lam[0], lam[-1]))
    return w


def _band_params(bands, nl):
    """Band weights of a request, [nband, nl] or [nl] for one band, checked as the library checks them (DESIGN.md
    section 5.6): 1 to MAX_BANDS bands, weights finite and >= 0, each band's sum in ascending order finite and > 0.
    Returns a C-contiguous float64 array [nband, nl]."""
    w = np.array(bands, dtype=float, ndmin=2)
    if w.ndim != 2 or w.shape[1] != nl:
        raise ValueError('bands must be [nband, %d] or [%d] (got shape %s)' % (nl, nl, w.shape))
    if not 1 <= w.shape[0] <= _lib.MAX_BANDS:
        raise ValueError('bands must hold 1 to %d bands (got %d)' % (_lib.MAX_BANDS, w.shape[0]))
    if not np.all(np.isfinite(w)) or np.any(w < 0):
        raise ValueError('band weights must be finite and >= 0')
    total = _band_sums(w)
    if not np.all(np.isfinite(total) & (total > 0)):
        raise ValueError('every band\'s weights must sum to a finite value > 0 (sums %s)' % total.tolist())
    return np.ascontiguousarray(w)


def _band_sums(w):
    """W_b = sum_k w[b][k], added in ascending k (the order of the library's sums)."""
    return np.cumsum(w, axis=1)[:, -1] if w.shape[1] else np.zeros(len(w))


def _band_lbda_eff(lbda, w):
    """Effective wavelength of every band [nband]: sum_k w[b][k] lbda[k] / W_b, summed in ascending k."""
    return _band_sums(w * np.asarray(lbda, dtype=float)) / _band_sums(w)


def _band_columns(lbda, w, fit, ee=None, radii=(), fractions=()):
    """Columns of a band table for the band fit records [n, nband, FIT_NPAR] (flattened; n = 1 or the positions):
    the ``_fit_columns`` with ``lbda`` the band's effective wavelength, ``band`` (index), ``weights`` [nl] per row,
    and the ``_ee_columns`` of the band EE records [n, nband, rec] when given."""
    lbda_eff = _band_lbda_eff(lbda, w)
    cols = _fit_columns(lbda_eff, fit)
    reps = len(cols['lbda']) // len(w)
    cols['band'] = np.tile(np.arange(len(w), dtype=np.int64), reps)
    cols['weights'] = np.tile(w, (reps, 1))
    if ee is not None:
        cols.update(_ee_columns(lbda_eff, ee, radii, fractions))
    return cols


def band_psf(psfcube, weights):
    """Band images of a cube [nl, ny, nx] -> [nband, ny, nx], or of cubes [n, nl, ny, nx] -> [n, nband, ny, nx], on
    the device (DESIGN.md section 5.6): ``B[b] = sum_k w[b][k] C[k] / W_b`` with the FP64 sum in ascending k, for
    ``weights`` [nband, nl] or [nl] (``band_weights``).  The band image keeps the flux scale of the planes.  Invalid
    weights raise ValueError before any device call."""
    data = getattr(psfcube, 'data', psfcube)
    data = np.ascontiguousarray(np.ma.getdata(data), dtype=np.float64)
    if data.ndim not in (3, 4):
        raise ValueError('psfcube must be [nl, ny, nx] or [n, nl, ny, nx]')
    cubes = data if data.ndim == 4 else data[None]
    n, nl, ny, nx = cubes.shape
    w = _band_params(weights, nl)
    out = np.empty((n, w.shape[0], ny, nx))
    if out.size:
        get_context(max_lambda=nl).band_psf(n, nl, ny, nx, cubes, w, out)
    return out if data.ndim == 4 else out[0]


# --------------------------------------------------------------------------- reference API
def simul_psd_wfm(Cn2, h, seeing, L0, zenith=0., plot=False, npsflin=1, dim=1280,
                  three_lgs_mode=False, verbose=True, wind_dir=None):
    """Residual-phase PSD per field direction, [npsflin**2, dim, dim] in nm^2
    (psfrec.py:36-151), synthesised on the GPU.  Extension: up to 8 layers when ``wind_dir`` gives
    one wind direction [rad] per layer (without it more than 2 layers raise ValueError, as the
    reference does)."""
    dim = _check_dim(dim)
    if three_lgs_mode and verbose:
        logger.info('Using three lasers mode')
    rec = draw_record(Cn2, h, seeing, L0, zenith, wind_dir=wind_dir)
    dirs = direction_perf(npsflin)
    ctx = get_context(max_planes=max(16 if dim == _DIM else 4, dirs.shape[1]), dim=dim)
    out = np.empty((dirs.shape[1], dim, dim))
    ctx.psd(rec[None], dirs, _lgs_positions(three_lgs_mode), out=out)
    return out


def _standard_pupil_ok(pup, dim):
    return pup is None or (np.shape(pup) == (dim // 2, dim // 2))


def psd_to_psf(psd, pup, D, lbda, phase_static=None, samp=None, FoV=None, return_all=False):
    """PSF from a residual-phase PSD (psfrec.py:689-807).  Only the branch the reference
    itself exercises is provided (SURVEY F6): MUSE pupil of dim/2 pixels, D = 8 m,
    samp = 2, FoV equal to the numerical field, no static phase."""
    psd = np.ascontiguousarray(psd, dtype=np.float64)
    dim = psd.shape[0]
    if psd.ndim != 2 or dim not in _DIMS or psd.shape[1] != dim:
        raise NotImplementedError('psd must be a square array of size %s' % (_DIMS,))
    if phase_static is not None or return_all:
        raise NotImplementedError('static phase / return_all are not on the hot path')
    if samp is not None and samp != 2:
        raise NotImplementedError("FIXME: use gridddata or spline ?")   # the reference fails here too (:640)
    if D != 8 or not _standard_pupil_ok(pup, dim):
        raise NotImplementedError('only the MUSE pupil (D=8, dim/2 pixels, oc=0.14) is supported')
    if pup is not None and not np.array_equal(np.asarray(pup) != 0, pupil_mask(dim / 4, dim / 2, oc=0.14) != 0):
        raise NotImplementedError('only the MUSE pupil (D=8, dim/2 pixels, oc=0.14) is supported')
    FoVnum = (lbda / (2 * D)) * dim / (4.85 * 1.e-6)
    if FoV is not None and not np.allclose(FoV, FoVnum):
        raise NotImplementedError("FIXME: use gridddata or spline ?")
    ctx = get_context(dim=dim)
    ctx.load_psd(psd, 1)
    ctx.structure_function(1)
    out = np.empty((dim, dim))
    ctx.psd_to_psf(0, lbda, out)
    return out


def psf_muse(psd, lambdamuse):
    """40x40 PSFs at 0.2 arcsec/pixel for each wavelength [nm] (psfrec.py:644-686)."""
    psd = np.ascontiguousarray(psd, dtype=np.float64)
    lam = np.atleast_1d(np.asarray(lambdamuse, dtype=float))
    if psd.ndim == 2:
        psd = psd[None]
    dim = psd.shape[1] if psd.ndim == 3 else 0
    if psd.ndim != 3 or dim not in _DIMS or psd.shape[2] != dim:
        raise NotImplementedError('psd must be [ndir, dim, dim] with dim in %s' % (_DIMS,))
    ndir = psd.shape[0]
    ctx = get_context(max_planes=max(16 if dim == _DIM else 4, ndir), max_lambda=max(35, lam.size), dim=dim)
    ctx.load_psd(psd, ndir)
    ctx.structure_function(ndir)
    out = np.empty((lam.size, _lib.PSF_DIM, _lib.PSF_DIM))
    try:
        ctx.psf_cube(1, ndir, lam, out)
    except PsfrError as exc:
        if exc.code == _lib.E_UNSUPPORTED:
            raise ValueError(str(exc))      # the reference raises ValueError from interpn / crop here
        raise
    return out


def muse_intrinsic_psf(lbda):
    """MUSE PSF polynomial approximation (psfrec.py:1144-1171): fwhm, beta, fwhm_std, beta_std."""
    pol_beta = [-0.83704697, 1.1337153, 0.0609222, -1.35581762, 1.15237178, 2.2106042]
    pol_fwhm = [0.60467385, -1.58905792, 1.75293264, -1.0368302, 0.21487023, 0.34851139]
    pol_beta_std = [0.18187424, -0.17841793, 0.30962616]
    pol_fwhm_std = [0.00707504, -0.0303464, 0.04596354]
    lb = (10 * np.asarray(lbda, dtype=float) - 4750) / (9350 - 4750)
    return (np.polyval(pol_fwhm, lb), np.polyval(pol_beta, lb),
            np.polyval(pol_fwhm_std, lb), np.polyval(pol_beta_std, lb))


def convolve_final_psf(lbda, seeing, GL, L0, psf):
    """Convolve with the tip-tilt and MUSE Moffat kernels (psfrec.py:874-930)."""
    lam = np.atleast_1d(np.asarray(lbda, dtype=float))
    psf = np.ascontiguousarray(psf, dtype=np.float64)
    if psf.shape != (lam.size, _lib.PSF_DIM, _lib.PSF_DIM):
        raise NotImplementedError('psf must be [nl, 40, 40]')
    ctx = get_context(max_lambda=max(35, lam.size))
    out = np.empty_like(psf)
    ctx.convolve(1, lam, [tiptilt_alpha(seeing, GL, L0)], psf, out)
    return out


def fit_psf_cube(lbda, psfcube, circular=True, var=None, mask=None, fit_back=False):
    """Fit a Moffat PSF on each wavelength plane (psfrec.py:861-871).  ``psfcube`` is an
    array [nl, ny, nx] (or anything with a ``.data`` array, like an mpdaf Cube).

    ``circular=False`` (mpdaf's keyword; the reference passes True) fits an elliptical Moffat instead and
    returns the columns of ``_shape_table_from_fit``: ``fwhm`` = (major, minor), ``axis_ratio``, ``pa`` [deg]
    and their errors.

    Star images (DESIGN.md section 5.7): ``var`` (the cube's variance), ``mask`` (True = bad pixel) and
    ``fit_back`` (fit a constant background) turn the fit into a weighted one.  ``var`` and ``mask`` have the
    cube's shape or [ny, nx] for every plane.  The weights are 1 / ``var`` (1 without ``var``) and 0 where ``mask``
    is true, where a masked input is masked, or where the data or the variance is not finite (NaN marks bad
    pixels in MUSE cubes).  The table then also holds ``cont`` (the background, 0 without ``fit_back``),
    ``err_cont`` and ``npix`` (the pixels used); ``peak`` and ``flux`` are above the background.  ``var <= 0`` on a
    pixel that would be used, and shapes that do not match, raise ValueError before any device call.  With all
    three keywords at their defaults the fit is the reference's unweighted one, unchanged."""
    if var is None and mask is None and not fit_back:
        data = getattr(psfcube, 'data', psfcube)
        data = np.ascontiguousarray(np.ma.getdata(data), dtype=np.float64)
        lam = np.atleast_1d(np.asarray(lbda, dtype=float))
        nimg, ny, nx = data.shape
        if not circular:
            efit = np.empty((nimg, _lib.EFIT_NPAR))
            if nimg:
                get_context().moffat_fit_elliptical(nimg, ny, nx, data, efit)
            return _shape_table_from_fit(lam, efit)
        ctx = get_context()
        fit = np.empty((nimg, _lib.FIT_NPAR))
        ctx.moffat_fit(nimg, ny, nx, data, fit)
        return _table_from_fit(lam, fit)
    lam = np.atleast_1d(np.asarray(lbda, dtype=float))
    data, weights = _star_weights(psfcube, var, mask)
    nimg, ny, nx = data.shape
    npar = _lib.FIT_NPAR if circular else _lib.EFIT_NPAR
    rec = np.empty((nimg, npar))
    back = np.empty((nimg, _lib.BACK_NPAR))
    if nimg:
        get_context().moffat_fit_weighted(nimg, ny, nx, data, weights, rec, back, fit_back=fit_back,
                                          elliptical=not circular)
    tab = _table_from_fit(lam, rec) if circular else _shape_table_from_fit(lam, rec)
    tab['cont'] = back[:, _lib.BACK_CONT].copy()
    tab['err_cont'] = back[:, _lib.BACK_ERR_CONT].copy()
    tab['npix'] = back[:, _lib.BACK_NPIX].astype(np.int64)
    return tab


def _star_weights(psfcube, var, mask):
    """(data, weights) of a star fit, both C-contiguous float64 [nl, ny, nx]; see ``fit_psf_cube``.  Unused pixels
    (weight 0) keep whatever data they hold: the library never reads them into a sum."""
    raw = psfcube if np.ma.isMaskedArray(psfcube) else getattr(psfcube, 'data', psfcube)   # an mpdaf Cube's .data
    data = np.array(np.ma.getdata(raw), dtype=np.float64, order='C')
    if data.ndim != 3:
        raise ValueError('psfcube must be [nl, ny, nx] (got shape %s)' % (data.shape,))
    shape = data.shape

    def planes(a, name):
        a = np.asarray(a)
        if a.shape == shape[1:]:
            a = np.broadcast_to(a, shape)
        if a.shape != shape:
            raise ValueError('%s must have the cube\'s shape %s or %s (got %s)' % (name, shape, shape[1:], a.shape))
        return a

    bad = ~np.isfinite(data)
    inmask = np.ma.getmask(raw)
    if inmask is not np.ma.nomask:
        bad |= planes(inmask, 'the mask of psfcube').astype(bool)
    if mask is not None:
        bad |= planes(np.ma.filled(mask, True) if np.ma.isMaskedArray(mask) else mask, 'mask').astype(bool)
    if var is None:
        weights = np.where(bad, 0.0, 1.0)
    else:
        v = planes(np.ma.filled(var, np.nan) if np.ma.isMaskedArray(var) else var, 'var').astype(np.float64)
        bad |= ~np.isfinite(v)
        if np.any(v[~bad] <= 0):
            i = np.argwhere((v <= 0) & ~bad)[0]
            raise ValueError('var must be > 0 on every used pixel (var[%d, %d, %d] = %g)'
                             % (i[0], i[1], i[2], v[tuple(i)]))
        weights = np.zeros(shape)
        np.divide(1.0, v, out=weights, where=~bad)
    return data, np.ascontiguousarray(weights)


def fit_psf_template(lbda, psfcube, template, var=None, mask=None, fit_back=False, return_model=False):
    """Fit each star stamp with a reconstructed PSF as the model (DESIGN.md section 5.8): plane i of ``psfcube``
    [n, ny, nx] (an array, a masked array or anything with a ``.data`` array) is fitted as F * T(shifted) + c, T =
    ``template[i % ntpl]`` interpolated by a cubic B-spline (``scipy.ndimage.map_coordinates(order=3,
    mode='mirror')``) and shifted so that its pixel (ty // 2, tx // 2) lands on the fitted centre.  ``template`` is
    [ntpl, ty, tx] with ``n % ntpl == 0`` (ten stars stacked star-major share one template cube) or [ty, tx].

    ``var``, ``mask`` and ``fit_back`` build the weights and the background as ``fit_psf_cube``.  The table has one
    row per stamp: ``lbda``, ``center`` (y, x) [px] and ``err_center``, ``flux`` (the flux of the template's whole
    footprint, template normalised to unit sum) and ``err_flux``, ``cont`` and ``err_cont`` (0 without
    ``fit_back``), ``chisq`` (sum w r^2; ``chisq / (npix - NP)`` ~ 1 when the template describes the star, NP = 3, or
    4 with ``fit_back``), ``qfit`` (sum |r| / |flux| over the used pixels), ``npix`` and ``converged``.  With
    ``return_model`` the call returns ``(table, model)``, model [n, ny, nx] the fitted image on every pixel (NaN for
    a failed stamp); the residual image is ``psfcube - model``.  Shape mismatches, ``var <= 0`` on a used pixel and a
    template that is not finite or does not sum to > 0 raise ValueError before any device call."""
    lam = np.atleast_1d(np.asarray(lbda, dtype=float))
    data, weights = _star_weights(psfcube, var, mask)
    nimg, ny, nx = data.shape
    tpl = np.array(template, dtype=np.float64, order='C')
    if tpl.ndim == 2:
        tpl = tpl[None]
    if tpl.ndim != 3 or tpl.shape[0] < 1 or nimg % tpl.shape[0]:
        raise ValueError('template must be [ty, tx] or [ntpl, ty, tx] with ntpl dividing the %d stamps (got shape %s)'
                         % (nimg, np.shape(template)))
    if lam.size != nimg:
        raise ValueError('lbda holds %d wavelengths for %d stamps' % (lam.size, nimg))
    if not np.all(np.isfinite(tpl)):
        raise ValueError('template has non-finite pixels (first at %s)' % (tuple(np.argwhere(~np.isfinite(tpl))[0]),))
    sums = tpl.reshape(tpl.shape[0], -1).sum(axis=1)
    if np.any(sums <= 0):
        raise ValueError('template %d sums to %g; every template must sum to > 0' % (np.argmax(sums <= 0),
                                                                                      sums[sums <= 0][0]))
    rec = np.empty((nimg, _lib.TFIT_NPAR))
    model = np.empty((nimg, ny, nx)) if return_model else None
    if nimg:
        # the host templates are staged whole on the device: grow the context until they fit its staging buffer
        # (max_planes * max_lambda 40 x 40 planes)
        ctx = get_context()
        ctx = get_context(max_lambda=-(-tpl.size // (ctx.max_planes * _lib.PSF_DIM * _lib.PSF_DIM)))
        ctx.template_fit(nimg, ny, nx, data, weights, tpl, rec, model, fit_back=fit_back)
    converged = rec[:, _lib.TFIT_ITER] > 0
    if not converged.all():
        bad = np.flatnonzero(~converged)
        logger.warning('template fit did not converge for %d of %d images (first at index %d)',
                       bad.size, nimg, bad[0])
    tab = FitTable({
        'lbda': lam,
        'center': rec[:, [_lib.TFIT_Y0, _lib.TFIT_X0]].copy(),
        'err_center': rec[:, [_lib.TFIT_ERR_Y0, _lib.TFIT_ERR_X0]].copy(),
        'flux': rec[:, _lib.TFIT_FLUX].copy(),
        'err_flux': rec[:, _lib.TFIT_ERR_FLUX].copy(),
        'cont': rec[:, _lib.TFIT_CONT].copy(),
        'err_cont': rec[:, _lib.TFIT_ERR_CONT].copy(),
        'chisq': rec[:, _lib.TFIT_CHISQ].copy(),
        'qfit': rec[:, _lib.TFIT_QFIT].copy(),
        'npix': np.nan_to_num(rec[:, _lib.TFIT_NPIX]).astype(np.int64),
        'converged': converged.astype(np.int64),
    })
    return (tab, model) if return_model else tab


def encircled_energy(lbda, psfcube, radii, fractions=(0.5, 0.8), center=None, pixscale=_PIXSCALE):
    """Encircled energy of each plane of ``psfcube`` [nl, ny, nx] on the device (DESIGN.md section 5.4).

    Pixel (p, q) is the unit square about (p, q) with its value spread uniformly over it, and EE(r) is the sum
    of every pixel times the exact area of its overlap with the disc of radius r: no supersampling, no
    renormalisation (the flux inside the aperture in the cube's own units).  ``radii`` and the returned radii are
    in arcsec at ``pixscale`` arcsec per pixel.  ``center`` is (y0, x0) in pixels (row, column; pixel centres at
    integers) for every plane or [nl, 2] per plane; the default (ny // 2, nx // 2) is pixel (20, 20) of a 40 x 40
    PSF of this package, its point of symmetry.  The image stops 19.5 px beyond that centre on its high side, so a
    larger circle is clipped by the edge.

    Returns a ``FitTable`` with ``lbda``, ``ee`` [nl, nrad], ``ee_total`` (the sum of the plane) and ``r_ee`` [nl,
    nfrac], the smallest radius holding each fraction of ``ee_total`` (NaN where ``ee_total`` <= 0); its meta
    holds the radii and fractions.  Invalid radii, fractions or centres raise ValueError before any device call."""
    data = getattr(psfcube, 'data', psfcube)
    data = np.ascontiguousarray(np.ma.getdata(data), dtype=np.float64)
    if data.ndim != 3:
        raise ValueError('psfcube must be [nl, ny, nx]')
    lam = np.atleast_1d(np.asarray(lbda, dtype=float))
    nimg, ny, nx = data.shape
    rad_px, frac = _ee_params(radii, fractions, pixscale)
    cen = None
    if center is not None:
        cen = np.array(center, dtype=float)
        if cen.shape == (2,):
            cen = np.tile(cen, (nimg, 1))
        if cen.shape != (nimg, 2):
            raise ValueError('center must be (y0, x0) or [nl, 2] (got shape %s)' % (cen.shape,))
        if not np.all(np.isfinite(cen)):
            raise ValueError('center must be finite')
        cen = np.ascontiguousarray(cen)
    ee = np.empty((nimg, _lib.ee_slots(rad_px.size, frac.size)[3]))
    if nimg:
        get_context().encircled_energy(nimg, ny, nx, data, rad_px, frac, ee, centres=cen)
    return _ee_table(lam, ee, rad_px * pixscale, frac, pixscale)


def compute_psf(lbda, seeing, GL, L0, npsflin=1, h=(100, 10000), three_lgs_mode=False, verbose=True,
                dim=_DIM, zenith=0., Cn2=None, wind_dir=None):
    """Reconstruct a PSF from seeing, GL and L0 (psfrec.py:933-978): returns (table, psf).
    Extensions of this backend (the reference hard-codes them, psfrec.py:953-955): ``dim`` (1280 or
    2560), ``zenith`` [deg], and a turbulence profile ``Cn2`` / ``h`` / ``wind_dir`` of up to 8 layers
    in place of [GL, 1 - GL] (GL still sets the tip-tilt kernel, psfrec.py:881)."""
    if verbose:
        logger.info('Compute PSF with seeing=%.2f GL=%.2f L0=%.2f', seeing, GL, L0)
        if three_lgs_mode:
            logger.info('Using three lasers mode')
    lam = np.atleast_1d(np.asarray(lbda, dtype=float))
    fit, cube = compute_psf_batch(lam, [seeing], [GL], [L0], npsflin=npsflin, h=h,
                                  three_lgs_mode=three_lgs_mode, dim=dim, zenith=zenith, Cn2=Cn2,
                                  wind_dir=wind_dir)
    res = _table_from_fit(lam, fit[0])
    res.meta.update({'SEEING': seeing, 'GL': GL, 'L0': L0})
    res['SEEING'] = seeing
    res['GL'] = GL
    res['L0'] = L0
    return res, cube[0]


reconstruct_psf = compute_psf   # pre-1.0 name used by BASELINE.json's north_star (CHANGELOG:6)


def _batch_records(seeing, GL, L0, h, zenith, Cn2, wind_dir):
    """Draw records of one ``compute_psf_batch`` call: the scalar ``draw_record`` (bit-identical to the
    reference's own scalars) up to 64 draws, the vectorised ``draw_records`` above.  The two can differ
    by a few ulp, so a caller that splits draws into subsets builds the records subset by subset."""
    nd = seeing.size
    if nd <= 64:
        h_arr = np.array(h)
        prof = None if Cn2 is None else np.asarray(Cn2, dtype=float)
        return np.stack([draw_record([GL[i], 1 - GL[i]] if prof is None else (prof[i] if prof.ndim == 2 else prof),
                                     h_arr[i] if h_arr.ndim == 2 else h_arr, seeing[i], L0[i], zenith,
                                     alpha_tt=tiptilt_alpha(seeing[i], GL[i], L0[i]), wind_dir=wind_dir)
                         for i in range(nd)])
    return draw_records(seeing, GL, L0, h, zenith=zenith, Cn2=Cn2, wind_dir=wind_dir)


def _mode_records(three, seeing, GL, L0, h=(100, 10000), zenith=0., Cn2=None, wind_dir=None):
    """Records of draws with one three-lasers flag each, built per mode as two ``compute_psf_batch`` calls
    would build them, with the guide-star count (3 or 4) in slot DRAW_NGS."""
    recs = np.empty((seeing.size, _lib.DRAW_NPAR))
    h_arr = np.array(h)
    prof = None if Cn2 is None else np.asarray(Cn2, dtype=float)
    for mode in (False, True):
        sel = np.flatnonzero(three == mode)
        if sel.size:
            recs[sel] = _batch_records(seeing[sel], GL[sel], L0[sel], h_arr[sel] if h_arr.ndim == 2 else h, zenith,
                                       prof[sel] if prof is not None and prof.ndim == 2 else Cn2, wind_dir)
    recs[:, _lib.DRAW_NGS] = np.where(three, 3, 4)
    return recs


def _mode_flags(three_lgs_mode, nd):
    """One three-lasers flag per draw from one flag or a sequence of nd flags."""
    three = np.asarray(three_lgs_mode, dtype=bool)
    if three.ndim == 0:
        return np.full(nd, bool(three))
    if three.shape != (nd,):
        raise ValueError('three_lgs_mode must be one flag or one flag per draw (got shape %s for %d draws)'
                         % (three.shape, nd))
    return three


def _field_positions(positions):
    """Field positions [2, npos] in arcsec (x row, then y row) as a C-contiguous float64 array, checked."""
    pos = np.array(positions, dtype=float, ndmin=2)
    if pos.ndim != 2 or pos.shape[0] != 2:
        raise ValueError('positions must be [2, npos] (x row, then y row, arcsec); got shape %s' % (pos.shape,))
    if not 1 <= pos.shape[1] <= _MAX_POSITIONS:
        raise ValueError('positions must hold 1 to %d field positions (got %d)' % (_MAX_POSITIONS, pos.shape[1]))
    if not np.all(np.isfinite(pos)):
        raise ValueError('positions must be finite')
    return np.ascontiguousarray(pos)


def _planes_context(nd, ndir, nlam, max_planes, device, dim):
    if max_planes is None:
        max_planes = 128 if dim == _DIM else 16      # planes per chunk of the fused pipeline (~8 GB of workspace)
    return get_context(max_planes=max(ndir, min(max_planes, nd * ndir)), max_lambda=max(35, nlam), device=device,
                       dim=dim)


def _band_outputs(bands, nl, lead, ee_rec):
    """(band_fit, band_cube[, band_ee]) buffers [*lead, nband, ...] of a ``bands=`` request (checked by
    ``_band_params``; ValueError before any device call), or () without one."""
    if bands is None:
        return ()
    nb = _band_params(bands, nl).shape[0]
    out = (np.empty(lead + (nb, _lib.FIT_NPAR)), np.empty(lead + (nb, _lib.PSF_DIM, _lib.PSF_DIM)))
    return out + ((np.empty(lead + (nb, ee_rec)),) if ee_rec is not None else ())


def _fused(ctx, field, recs, dirs, lam, group_end=None, ee=None, bands=None, stream=None, **outs):
    """One pass of the fused pipeline (``Context.compute_bands``) over draws that each carry their guide-star count:
    ``ee`` (radii [px], fractions) or None, ``bands`` weights [nband, nl] or None, and the outputs ``outs`` (keywords
    of ``compute_bands``).  PSFR_E_UNSUPPORTED (a wavelength or draw outside the library's range) raises ValueError."""
    rad, frac = ((), ()) if ee is None else ee
    try:
        ctx.compute_bands(field, recs, dirs, _lgs_positions(False), lam, bands, rad, frac, group_end, stream=stream,
                          **outs)
    except PsfrError as exc:
        if exc.code == _lib.E_UNSUPPORTED:
            raise ValueError(str(exc))
        raise


def compute_psf_batch(lbda, seeing, GL, L0, npsflin=1, h=(100, 10000), three_lgs_mode=False,
                      out_cube=None, out_fit=None, want_cube=True, device=None, max_planes=None, stream=None,
                      dim=_DIM, zenith=0., Cn2=None, wind_dir=None, ee_radii=None, ee_fractions=(0.5, 0.8),
                      ao_budget=False, bands=None):
    """Batched ``compute_psf``: one fused device pipeline for many (seeing, GL, L0[, h]) draws.

    ``h`` is one (h0, h1) pair or an array [ndraw, 2].  ``three_lgs_mode`` is one flag for all draws or
    one per draw; each draw gives the same bits as in a call of its own mode.  Returns (fit [ndraw, nl,
    FIT_NPAR], cube [ndraw, nl, 40, 40]); ``out_cube`` / ``out_fit`` may be preallocated numpy arrays or
    torch tensors (host-pinned or device) used as plain buffers.

    ``ee_radii`` [arcsec] adds the encircled energy of every returned PSF about its centre pixel (20, 20),
    computed on the device right after its fit (``encircled_energy``): the result gains a third entry, the raw
    records [ndraw, nl, nrad + 1 + nfrac] in pixels (``_lib.ee_slots``; ``_ee_table`` turns them into the
    columns of ``encircled_energy``), for the fractions ``ee_fractions``.  With ``want_cube=False`` no cube leaves
    the device.  fit and cube are those of a call without ``ee_radii``, bit for bit.

    ``ao_budget=True`` appends (strehl [ndraw, nl], var [ndraw, npsflin**2, VAR_NPAR]) after the other results:
    the AO Strehl ratio of every PSF and the residual-phase variance record (nm^2, ``_lib.VAR_*``) of every
    (draw, direction) plane, computed on the device in the same pass (DESIGN.md section 5.5; ``_ao_table`` turns
    them into columns).  Every other result is that of a call without it, bit for bit.

    ``bands`` (weights [nband, nl] or [nl], ``band_weights``) appends (band_fit [ndraw, nband, FIT_NPAR], band_cube
    [ndraw, nband, 40, 40]) after every other result, and band_ee [ndraw, nband, nrad + 1 + nfrac] when ``ee_radii``
    is given: the band image of every draw, ``sum_k w[b][k] cube[k] / W_b``, its Moffat fit and encircled energy,
    formed on the device from the convolved planes (DESIGN.md section 5.6).  band_cube is returned with
    ``want_cube=False`` too.  Every other result is that of a call without ``bands``, bit for bit; invalid weights
    raise ValueError before any device call."""
    lam = np.atleast_1d(np.asarray(lbda, dtype=float))
    seeing, GL, L0 = (np.atleast_1d(np.asarray(v, dtype=float)) for v in (seeing, GL, L0))
    nd = seeing.size
    if GL.size != nd or L0.size != nd:
        raise ValueError('seeing, GL and L0 must have one entry per draw (got %d, %d, %d)' % (nd, GL.size, L0.size))
    per_draw = np.ndim(three_lgs_mode) > 0
    if per_draw:
        three = _mode_flags(three_lgs_mode, nd)
    energy = ee_radii is not None
    if energy:
        rad_px, frac = _ee_params(ee_radii, ee_fractions)
        ee = np.empty((nd, lam.size, _lib.ee_slots(rad_px.size, frac.size)[3]))
    ndir = npsflin * npsflin
    ao = (np.empty((nd, lam.size)), np.empty((nd, ndir, _lib.VAR_NPAR))) if ao_budget else ()
    band = _band_outputs(bands, lam.size, (nd,), ee.shape[-1] if energy else None)
    extra = ((ee,) if energy else ()) + ao + band
    if nd == 0 or lam.size == 0:
        # nothing to compute: empty results of the right shape, written through nothing
        return (np.empty((nd, lam.size, _lib.FIT_NPAR)),
                np.empty((nd, lam.size, _lib.PSF_DIM, _lib.PSF_DIM)) if want_cube else None) + extra
    if per_draw:
        recs = _mode_records(three, seeing, GL, L0, h, zenith, Cn2, wind_dir)
    else:
        recs = _batch_records(seeing, GL, L0, h, zenith, Cn2, wind_dir)
        if energy or ao_budget or band:      # the groups path takes each draw's guide-star count from its record
            recs[:, _lib.DRAW_NGS] = 3 if three_lgs_mode else 4
    dirs = direction_perf(npsflin)
    dim = _check_dim(dim)
    ctx = _planes_context(nd, dirs.shape[1], lam.size, max_planes, device, dim)
    if out_fit is None:
        out_fit = np.empty((nd, lam.size, _lib.FIT_NPAR))
    if out_cube is None and want_cube:
        out_cube = np.empty((nd, lam.size, _lib.PSF_DIM, _lib.PSF_DIM))
    if per_draw or energy or ao_budget or band:
        # each draw's own guide-star count: the three-laser asterism is the first three stars of the four-laser one
        _fused(ctx, False, recs, dirs, lam, ee=(rad_px, frac) if energy else None,
               bands=_band_params(bands, lam.size) if band else None, stream=stream, out_cube=out_cube,
               out_fit=out_fit, out_ee=ee if energy else None, out_strehl=ao[0] if ao else None,
               out_var=ao[1] if ao else None, out_band=band[1] if band else None,
               out_band_fit=band[0] if band else None, out_band_ee=band[2] if band and energy else None)
        return (out_fit, out_cube) + extra
    try:
        ctx.compute_batch(recs, dirs, _lgs_positions(three_lgs_mode), lam, out_cube=out_cube, out_fit=out_fit,
                          stream=stream)
    except PsfrError as exc:
        if exc.code == _lib.E_UNSUPPORTED:
            raise ValueError(str(exc))
        raise
    return out_fit, out_cube


def compute_psf_field(lbda, seeing, GL, L0, positions=None, npsflin=3, field_size=60, h=(100, 10000),
                      three_lgs_mode=False, out_cube=None, out_fit=None, want_cube=True, device=None, max_planes=None,
                      stream=None, dim=_DIM, zenith=0., Cn2=None, wind_dir=None, elliptical=False, ee_radii=None,
                      ee_fractions=(0.5, 0.8), ao_budget=False, bands=None):
    """Field-resolved ``compute_psf_batch``: the PSF of every draw at every field position instead of
    their average.

    ``positions`` is [2, npos] in arcsec (x row, then y row, the convention of ``direction_perf``), at most
    256 positions; the default is ``direction_perf(npsflin, field_size)``.  The PSF at position k of a draw
    is the reference's ``psf_muse`` of that direction's PSD alone, then ``convolve_final_psf`` and the
    Moffat fit: bit for bit what ``compute_psf_batch`` gives for that draw with the single direction k
    (so ``positions=[[0], [0]]`` reproduces ``compute_psf_batch(npsflin=1)``).  It is not the field mean
    ``compute_psf_batch(npsflin=n)`` returns, and the field mean is not the average of these PSFs (each
    is normalised on its own).  Other arguments as ``compute_psf_batch``.  Returns (fit [ndraw, npos, nl,
    FIT_NPAR], cube [ndraw, npos, nl, 40, 40]).

    ``elliptical=True`` also fits an elliptical Moffat to every PSF on the device, right after its circular fit
    and from it, and returns (fit, cube, efit) with efit [ndraw, npos, nl, EFIT_NPAR] (``_lib.EFIT_*``); fit and
    cube are those of a call without it, bit for bit.

    ``ee_radii`` [arcsec] appends the encircled-energy records [ndraw, npos, nl, nrad + 1 + nfrac] of every PSF, in
    pixels, as ``compute_psf_batch(ee_radii=...)`` does, after ``efit`` where present.

    ``ao_budget=True`` appends (strehl [ndraw, npos, nl], var [ndraw, npos, VAR_NPAR]) last, as
    ``compute_psf_batch(ao_budget=True)`` does: the Strehl ratio of each position's PSF and the variance record of
    each (draw, position) plane.

    ``bands`` appends (band_fit [ndraw, npos, nband, FIT_NPAR], band_cube [ndraw, npos, nband, 40, 40]) and, with
    ``ee_radii``, band_ee [ndraw, npos, nband, nrad + 1 + nfrac] after everything else, as ``compute_psf_batch(bands=...)``
    does, for the PSF of each position."""
    pos = _field_positions(direction_perf(npsflin, field_size) if positions is None else positions)
    npos = pos.shape[1]
    lam = np.atleast_1d(np.asarray(lbda, dtype=float))
    seeing, GL, L0 = (np.atleast_1d(np.asarray(v, dtype=float)) for v in (seeing, GL, L0))
    nd = seeing.size
    if GL.size != nd or L0.size != nd:
        raise ValueError('seeing, GL and L0 must have one entry per draw (got %d, %d, %d)' % (nd, GL.size, L0.size))
    three = _mode_flags(three_lgs_mode, nd)
    efit = np.empty((nd, npos, lam.size, _lib.EFIT_NPAR)) if elliptical else None
    energy = ee_radii is not None
    if energy:
        rad_px, frac = _ee_params(ee_radii, ee_fractions)
        ee = np.empty((nd, npos, lam.size, _lib.ee_slots(rad_px.size, frac.size)[3]))
    ao = (np.empty((nd, npos, lam.size)), np.empty((nd, npos, _lib.VAR_NPAR))) if ao_budget else ()
    band = _band_outputs(bands, lam.size, (nd, npos), ee.shape[-1] if energy else None)
    extra = ((efit,) if elliptical else ()) + ((ee,) if energy else ()) + ao + band
    if nd == 0 or lam.size == 0:
        return (np.empty((nd, npos, lam.size, _lib.FIT_NPAR)),
                np.empty((nd, npos, lam.size, _lib.PSF_DIM, _lib.PSF_DIM)) if want_cube else None) + extra
    # the records compute_psf_batch builds in either laser mode; the three-laser asterism is the first three
    # stars of the four-laser one
    recs = _mode_records(three, seeing, GL, L0, h, zenith, Cn2, wind_dir)
    dim = _check_dim(dim)
    ctx = _planes_context(nd, npos, lam.size, max_planes, device, dim)
    if out_fit is None:
        out_fit = np.empty((nd, npos, lam.size, _lib.FIT_NPAR))
    if out_cube is None and want_cube:
        out_cube = np.empty((nd, npos, lam.size, _lib.PSF_DIM, _lib.PSF_DIM))
    _fused(ctx, True, recs, pos, lam, ee=(rad_px, frac) if energy else None,
           bands=_band_params(bands, lam.size) if band else None, stream=stream, out_cube=out_cube, out_fit=out_fit,
           out_efit=efit, out_ee=ee if energy else None, out_strehl=ao[0] if ao else None,
           out_var=ao[1] if ao else None, out_band=band[1] if band else None, out_band_fit=band[0] if band else None,
           out_band_ee=band[2] if band and energy else None)
    return (out_fit, out_cube) + extra


def _norm_lbda(lbda, lb1, lb2):
    return (lbda - lb1) / (lb2 - lb1) - 0.5


def fit_psf_with_polynom(lbda, fwhm, beta, deg=(5, 5), output=0):
    """Fit MUSE PSF fwhm and beta with polynomials in the normalised wavelength
    (psfrec.py:1174-1210); least squares solved on the device (Householder QR)."""
    lbda = np.asarray(lbda, dtype=float)
    ctx = get_context()
    if deg[0] == deg[1]:
        coef = ctx.polyfit(lbda, deg[0], np.stack([np.asarray(fwhm, float), np.asarray(beta, float)]))
        fwhm_pol, beta_pol = coef[0], coef[1]
    else:
        fwhm_pol = ctx.polyfit(lbda, deg[0], np.asarray(fwhm, float))[0]
        beta_pol = ctx.polyfit(lbda, deg[1], np.asarray(beta, float))[0]
    res = dict(fwhm_pol=fwhm_pol, beta_pol=beta_pol, lbda=lbda, lbda_lim=(475, 935))
    if output > 0:
        lbda_fit = np.linspace(475, 935, 50)
        lbf = _norm_lbda(lbda_fit, 475, 935)
        res['lbda_fit'] = lbda_fit
        res['fwhm_fit'] = np.polyval(fwhm_pol, lbf)
        res['beta_fit'] = np.polyval(beta_pol, lbf)
    return res


# --------------------------------------------------------------------------- SPARTA shell
def select_sparta_rows(values, mean_of_lgs=True, verbose=False):
    """Row rejection and laser averaging of ``compute_psf_from_sparta`` (psfrec.py:1041-1076).

    ``values``: [nrows, 4, 3] = (SEEING, TUR_GND, L0) of the 4 lasers.  Returns a list of
    (seeing, GL, L0, three_lgs_mode, row_idx, lgs_idx) and logs the reference's messages."""
    values = np.asarray(values, dtype=float)
    nrows = len(values)
    jobs = []
    for irow, v in enumerate(values, start=1):
        # GL > 0 and MIN_L0 < L0 < MAX_L0: "apparently the 4th value is often crap" (psfrec.py:1047-1051)
        ok = (v[:, 1] > 0) & (v[:, 2] < MAX_L0) & (v[:, 2] > MIN_L0)
        nb_gs = int(ok.sum())
        three_lgs_mode = nb_gs < 4
        if nb_gs == 0:
            if verbose:
                logger.info('%d/%d : No valid values, skipping this row', irow, nrows)
                logger.debug('Values: %s', v.tolist())
            continue
        elif nb_gs < 4:
            if verbose:
                logger.info('%d/%d : Using only %d values out of 4 after outliers '
                            'rejection', irow, nrows, nb_gs)
        if mean_of_lgs:
            seeing, GL, L0 = v[ok].mean(axis=0)
            jobs.append((seeing, GL, L0, three_lgs_mode, irow, -1))
        else:
            for i in np.where(ok)[0]:
                jobs.append((v[i, 0], v[i, 1], v[i, 2], three_lgs_mode, irow, i + 1))
    return jobs


def _fit_columns(lam, fit):
    """Columns of the reference's fit table for fit records [n, nl, FIT_NPAR] (flattened)."""
    nl = lam.size
    fit = np.asarray(fit).reshape(-1, _lib.FIT_NPAR)
    tab = _table_from_fit(np.tile(lam, len(fit) // nl), fit)
    return {k: tab[k] for k in tab.colnames}


def _shape_columns(lam, efit):
    """Columns of the elliptical fit table for records [n, nl, EFIT_NPAR] (flattened)."""
    nl = lam.size
    efit = np.asarray(efit).reshape(-1, _lib.EFIT_NPAR)
    tab = _shape_table_from_fit(np.tile(lam, len(efit) // nl), efit)
    return {k: tab[k] for k in tab.colnames}


def _ee_columns(lam, ee, radii, fractions):
    """Columns of the encircled-energy table for records [n, nl, nrad + 1 + nfrac] (flattened)."""
    ee = np.asarray(ee).reshape(-1, _lib.ee_slots(len(radii), len(fractions))[3])
    tab = _ee_table(np.tile(lam, len(ee) // lam.size), ee, radii, fractions)
    return {k: tab[k] for k in tab.colnames}


def _draw_mean(x):
    """Mean of ``x`` over its first axis, summed in order (the mean of an exposure's draws, in draw order)."""
    x = np.asarray(x, dtype=float)
    acc = np.zeros(x.shape[1:])
    for row in x:
        acc = acc + row
    return acc / len(x)


def _ee_cards(meta, radii, fractions):
    """``meta`` plus one card per radius [arcsec] (EERADk) and per fraction (EEFRACk), k from 1."""
    cards = dict(meta)
    cards.update({'EERAD%d' % (k + 1): float(r) for k, r in enumerate(radii)})
    cards.update({'EEFRAC%d' % (j + 1): float(f) for j, f in enumerate(fractions)})
    return cards


def compute_psf_from_sparta(filename, extname='SPARTA_ATM_DATA', npsflin=1, lmin=490, lmax=930, nl=35,
                            lbda=None, h=(100, 10000), n_jobs=-1, plot=False, mean_of_lgs=True,
                            verbose=True, device=None, field_positions=None, elliptical=False, ee_radii=None,
                            ee_fractions=(0.5, 0.8), ao_budget=False, bands=None):
    """Reconstruct a PSF from SPARTA data (psfrec.py:981-1120).

    ``filename``: path of a FITS file, a binary file object, or an HDUList (this package's or
    astropy's) holding the SPARTA table.  Every valid row (or laser) becomes one draw of a single
    batched GPU call (the reference fans them out over joblib processes, psfrec.py:1082-1083;
    ``n_jobs`` is accepted and only reported).  Returns an HDUList [PRIMARY, <extname>, FIT_ROWS,
    FIT_MEAN, PSF_MEAN] - an ``astropy.io.fits.HDUList`` when astropy is installed, otherwise
    the equivalent object of ``muse_psfr_b200._fits`` - or None when no row is valid.  With
    ``field_positions`` [2, npos] (arcsec), FIT_FIELD and PSF_FIELD follow, with ``elliptical=True``
    SHAPE_MEAN (and SHAPE_FIELD), with ``ee_radii`` EE_MEAN (and EE_FIELD), with ``ao_budget=True`` AO_MEAN
    (and AO_FIELD), and with ``bands`` BAND_MEAN and PSF_BAND (and BAND_FIELD, PSF_BAND_FIELD): see
    ``compute_psf_from_sparta_batch``."""
    if plot:
        raise NotImplementedError('plotting is outside the B200 hot path')
    return compute_psf_from_sparta_batch([filename], extname=extname, npsflin=npsflin, lmin=lmin, lmax=lmax, nl=nl,
                                         lbda=lbda, h=h, n_jobs=n_jobs, mean_of_lgs=mean_of_lgs, verbose=verbose,
                                         device=device, field_positions=field_positions, elliptical=elliptical,
                                         ee_radii=ee_radii, ee_fractions=ee_fractions, ao_budget=ao_budget,
                                         bands=bands)[0]


def compute_psf_from_sparta_batch(sources, extname='SPARTA_ATM_DATA', npsflin=1, lmin=490, lmax=930, nl=35,
                                  lbda=None, h=(100, 10000), n_jobs=-1, mean_of_lgs=True, verbose=True,
                                  device=None, max_planes=None, field_positions=None, elliptical=False,
                                  ee_radii=None, ee_fractions=(0.5, 0.8), ao_budget=False, bands=None):
    """``compute_psf_from_sparta`` for many exposures in one device pass: returns one entry per source,
    the HDUList ``compute_psf_from_sparta(source, ...)`` returns, bit for bit, or None for a table
    without a valid row.

    The valid rows of every table, in three- and four-laser mode alike, form one batch; each
    exposure's time-mean PSF and its refit are formed on the device while its draws are resident, and
    only the fit records and the means come back to the host.  Each table logs the messages of a
    single-table call, in the same order.  ``max_planes`` caps the (draw x direction) planes per
    chunk of the pipeline, as in ``compute_psf_batch``.

    ``field_positions`` [2, npos] (arcsec, x row then y row, as ``direction_perf``) adds the exposure's
    time-mean PSF at each of those positions, from one more device pass over the same draws
    (``compute_psf_field``): FIT_FIELD, the columns of FIT_MEAN plus ``x`` and ``y`` [arcsec], one row per
    (position, wavelength), position-major, with the cards of FIT_MEAN; and PSF_FIELD, an image [npos,
    nl, 40, 40].  The first five HDUs are those of a call without ``field_positions``, bit for bit.

    ``elliptical=True`` appends SHAPE_MEAN, the elliptical fit table (``fit_psf_cube(circular=False)``
    columns) of PSF_MEAN with the cards of FIT_MEAN, and with ``field_positions`` SHAPE_FIELD, the same
    columns plus ``x`` and ``y`` for the PSFs of PSF_FIELD, position-major.  Every HDU before them is that of
    a call without ``elliptical``, bit for bit.

    ``ee_radii`` [arcsec] appends EE_MEAN, the ``encircled_energy`` table of PSF_MEAN (radii ``ee_radii``, fractions
    ``ee_fractions``) with the cards of FIT_MEAN plus EERADk / EEFRACk, and with ``field_positions`` EE_FIELD, the
    same columns plus ``x`` and ``y`` for the PSFs of PSF_FIELD, position-major.  Both are computed on the device
    in the passes that form the means, and follow the SHAPE_* HDUs; every HDU before them is that of a call
    without ``ee_radii``, bit for bit.

    ``ao_budget=True`` appends AO_MEAN, one row per wavelength with the ``_ao_table`` columns and the cards of
    FIT_MEAN: the Strehl ratio and the residual-phase variance budget (nm^2) of the exposure, each the mean over
    its draws in draw order (for the variance, over the directions of each draw too), from the Strehl ratios and
    variance records the mean pass computes on the device.  With ``field_positions`` AO_FIELD follows, the same
    columns plus ``x`` and ``y`` per (position, wavelength), position-major, from the field pass.  Every HDU before
    them is that of a call without ``ao_budget``, bit for bit.

    ``bands`` (weights [nband, nl] or [nl] on ``lbda``, ``band_weights``) appends BAND_MEAN and PSF_BAND after every
    other HDU.  PSF_BAND is an image [nband, 40, 40], the band images of PSF_MEAN (DESIGN.md section 5.6), formed on
    the device in the mean pass; it is the band of the exposure's mean cube, not the mean of its draws' bands.
    BAND_MEAN holds one row per band: the columns of FIT_MEAN for the Moffat fit of the band image, with ``lbda`` the
    band's effective wavelength sum_k w_k lbda_k / sum_k w_k, a ``band`` index, the band's ``weights`` [nl], and the
    ``encircled_energy`` columns when ``ee_radii`` is given; the cards of FIT_MEAN (plus EERADk / EEFRACk with
    ``ee_radii``).  With ``field_positions`` BAND_FIELD (the same columns plus ``x`` and ``y``, one row per (position,
    band), position-major) and PSF_BAND_FIELD [npos, nband, 40, 40] follow, from the field pass.  Every HDU before
    them is that of a call without ``bands``, bit for bit; invalid weights raise ValueError before any device call."""
    if lbda is None:
        lbda = np.linspace(lmin, lmax, nl)
    lbda = np.atleast_1d(np.asarray(lbda, dtype=float))
    pos = None if field_positions is None else _field_positions(field_positions)
    w_band = None if bands is None else _band_params(bands, lbda.size)
    energy = ee_radii is not None
    if energy:
        rad_px, frac = _ee_params(ee_radii, ee_fractions)
        ee_rec = _lib.ee_slots(rad_px.size, frac.size)[3]
        ee_rad = rad_px * _PIXSCALE
    files, recs = [], []
    for source in sources:
        hdul = _fits.from_any(source, only={extname.upper()})
        sparta = hdul[extname]
        tbl = sparta.data
        nrows = len(tbl)
        if verbose:
            logger.info('Processing SPARTA table with %d values, njobs=%d ...', nrows, 1 if nrows == 1 else n_jobs)
        values = np.array([[[row['LGS%d_%s' % (k, col)] for col in ('SEEING', 'TUR_GND', 'L0')]
                            for k in range(1, 5)] for row in tbl], dtype=float).reshape(nrows, 4, 3)
        jobs = select_sparta_rows(values, mean_of_lgs=mean_of_lgs, verbose=verbose)
        if len(jobs) == 0:
            logger.warning('No valid values')
            files.append(None)
            continue
        seeing, GL, L0, three, row_idx, lgs_idx = (np.array(c) for c in zip(*jobs))
        if verbose:
            for j in range(len(jobs)):      # the messages compute_psf / simul_psd_wfm log per draw
                logger.info('Compute PSF with seeing=%.2f GL=%.2f L0=%.2f', seeing[j], GL[j], L0[j])
                if three[j]:
                    logger.info('Using three lasers mode')
        recs.append(_mode_records(three, seeing, GL, L0, h))
        files.append((sparta, seeing, GL, L0, lgs_idx))
    if not recs:
        return [None] * len(files)

    draws = np.concatenate(recs)
    group_end = np.cumsum([len(r) for r in recs]).astype(np.int32)
    nd, ng, nlam = len(draws), len(recs), lbda.size
    fit = np.empty((nd, nlam, _lib.FIT_NPAR))
    psftot = np.empty((ng, nlam, _lib.PSF_DIM, _lib.PSF_DIM))
    fit_mean = np.empty((ng, nlam, _lib.FIT_NPAR))
    dirs = direction_perf(npsflin)
    ctx = _planes_context(nd, dirs.shape[1], nlam, max_planes, device, _DIM)
    ee_par = (rad_px, frac) if energy else None
    ee_mean = np.empty((ng, nlam, ee_rec)) if energy else None
    if ao_budget:
        strehl = np.empty((nd, nlam))
        var = np.empty((nd, dirs.shape[1], _lib.VAR_NPAR))
    band_mean = _band_outputs(w_band, nlam, (ng,), ee_rec if energy else None)
    _fused(ctx, False, draws, dirs, lbda, group_end, ee=ee_par, bands=w_band, out_fit=fit, out_mean=psftot,
           out_mean_fit=fit_mean, out_mean_ee=ee_mean, out_strehl=strehl if ao_budget else None,
           out_var=var if ao_budget else None, out_mean_band=band_mean[1] if band_mean else None,
           out_mean_band_fit=band_mean[0] if band_mean else None,
           out_mean_band_ee=band_mean[2] if band_mean and energy else None)
    if pos is not None:
        npos = pos.shape[1]
        psf_field = np.empty((ng, npos, nlam, _lib.PSF_DIM, _lib.PSF_DIM))
        fit_field = np.empty((ng, npos, nlam, _lib.FIT_NPAR))
        ctx = _planes_context(nd, npos, nlam, max_planes, device, _DIM)
        shape_field = np.empty((ng, npos, nlam, _lib.EFIT_NPAR)) if elliptical else None
        ee_field = np.empty((ng, npos, nlam, ee_rec)) if energy else None
        if ao_budget:
            strehl_field = np.empty((nd, npos, nlam))
            var_field = np.empty((nd, npos, _lib.VAR_NPAR))
        band_field = _band_outputs(w_band, nlam, (ng, npos), ee_rec if energy else None)
        _fused(ctx, True, draws, pos, lbda, group_end, ee=ee_par, bands=w_band, out_mean=psf_field,
               out_mean_fit=fit_field, out_mean_efit=shape_field, out_mean_ee=ee_field,
               out_strehl=strehl_field if ao_budget else None, out_var=var_field if ao_budget else None,
               out_mean_band=band_field[1] if band_field else None,
               out_mean_band_fit=band_field[0] if band_field else None,
               out_mean_band_ee=band_field[2] if band_field and energy else None)
    if elliptical:      # the time means are on the host already: one standalone fit of all of them
        shape_mean = np.empty((ng, nlam, _lib.EFIT_NPAR))
        ctx.moffat_fit_elliptical(ng * nlam, _lib.PSF_DIM, _lib.PSF_DIM, psftot, shape_mean)

    results, g = [], 0
    for entry in files:
        if entry is None:
            results.append(None)
            continue
        sparta, seeing, GL, L0, lgs_idx = entry
        nj = seeing.size
        d0 = int(group_end[g]) - nj
        out = _fits.HDUList([_fits.PrimaryHDU(), sparta.copy()])
        # fit values of all rows in one table (psfrec.py:1086-1101)
        cols = _fit_columns(lbda, fit[d0:d0 + nj])
        cols['SEEING'] = np.repeat(seeing, nlam)
        cols['GL'] = np.repeat(GL, nlam)
        cols['L0'] = np.repeat(L0, nlam)
        cols['row_idx'] = np.repeat(np.arange(1, nj + 1, dtype=np.int64), nlam)
        cols['lgs_idx'] = np.repeat(lgs_idx.astype(np.int64), nlam)
        out.append(_fits.table_to_hdu(cols, name='FIT_ROWS'))
        # mean PSF over the draws, refit, median seeing / GL / L0 (psfrec.py:1104-1113)
        med = np.median(np.stack([seeing, GL, L0], axis=1), axis=0)
        meta = {'SEEING': float(med[0]), 'GL': float(med[1]), 'L0': float(med[2])}
        out.append(_fits.table_to_hdu(_fit_columns(lbda, fit_mean[g][None]), meta=meta, name='FIT_MEAN'))
        out.append(_fits.ImageHDU(data=psftot[g], name='PSF_MEAN'))
        if pos is not None:
            cols = _fit_columns(lbda, fit_field[g])
            cols['x'] = np.repeat(pos[0], nlam)
            cols['y'] = np.repeat(pos[1], nlam)
            out.append(_fits.table_to_hdu(cols, meta=meta, name='FIT_FIELD'))
            out.append(_fits.ImageHDU(data=psf_field[g], name='PSF_FIELD'))
        if elliptical:
            out.append(_fits.table_to_hdu(_shape_columns(lbda, shape_mean[g]), meta=meta, name='SHAPE_MEAN'))
            if pos is not None:
                cols = _shape_columns(lbda, shape_field[g])
                cols['x'] = np.repeat(pos[0], nlam)
                cols['y'] = np.repeat(pos[1], nlam)
                out.append(_fits.table_to_hdu(cols, meta=meta, name='SHAPE_FIELD'))
        if energy:
            cards = _ee_cards(meta, ee_rad, frac)
            out.append(_fits.table_to_hdu(_ee_columns(lbda, ee_mean[g], ee_rad, frac), meta=cards, name='EE_MEAN'))
            if pos is not None:
                cols = _ee_columns(lbda, ee_field[g], ee_rad, frac)
                cols['x'] = np.repeat(pos[0], nlam)
                cols['y'] = np.repeat(pos[1], nlam)
                out.append(_fits.table_to_hdu(cols, meta=cards, name='EE_FIELD'))
        if ao_budget:
            tab = _ao_table(lbda, _draw_mean(strehl[d0:d0 + nj]),
                            _draw_mean(var[d0:d0 + nj].reshape(-1, _lib.VAR_NPAR)))
            out.append(_fits.table_to_hdu({k: tab[k] for k in tab.colnames}, meta=meta, name='AO_MEAN'))
            if pos is not None:
                s_f, v_f = _draw_mean(strehl_field[d0:d0 + nj]), _draw_mean(var_field[d0:d0 + nj])
                tab = FitTable.vstack([_ao_table(lbda, s_f[k], v_f[k]) for k in range(npos)])
                cols = {k: tab[k] for k in tab.colnames}
                cols['x'] = np.repeat(pos[0], nlam)
                cols['y'] = np.repeat(pos[1], nlam)
                out.append(_fits.table_to_hdu(cols, meta=meta, name='AO_FIELD'))
        if w_band is not None:
            cards = _ee_cards(meta, ee_rad, frac) if energy else meta
            ee_args = (band_mean[2][g], ee_rad, frac) if energy else ()
            out.append(_fits.table_to_hdu(_band_columns(lbda, w_band, band_mean[0][g], *ee_args), meta=cards,
                                          name='BAND_MEAN'))
            out.append(_fits.ImageHDU(data=band_mean[1][g], name='PSF_BAND'))
            if pos is not None:
                ee_args = (band_field[2][g], ee_rad, frac) if energy else ()
                cols = _band_columns(lbda, w_band, band_field[0][g], *ee_args)
                cols['x'] = np.repeat(pos[0], len(w_band))
                cols['y'] = np.repeat(pos[1], len(w_band))
                out.append(_fits.table_to_hdu(cols, meta=cards, name='BAND_FIELD'))
                out.append(_fits.ImageHDU(data=band_field[1][g], name='PSF_BAND_FIELD'))
        try:
            results.append(_fits.to_astropy(out))
        except ImportError:
            results.append(out)
        g += 1
    return results


def create_sparta_table(nlines=1, seeing=1, L0=25, GL=0.7, bad_l0=False, outfile=None):
    """Helper function to create a SPARTA table with the given seeing, L0, and GL values
    (psfrec.py:1123-1141).  Returns the table HDU; ``outfile`` may be a path or a file object."""
    cols = {}
    for k in range(1, 5):
        for col, v in (('SEEING', seeing), ('TUR_GND', GL), ('L0', L0)):
            cols['LGS%d_%s' % (k, col)] = np.full(nlines, float(v))
    if bad_l0:
        cols['LGS4_L0'] = np.full(nlines, 150.0)
    hdu = _fits.table_to_hdu(cols, name='SPARTA_ATM_DATA')
    if outfile is not None:
        hdu.writeto(outfile, overwrite=True)
    return hdu
