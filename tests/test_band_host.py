"""CPU tests of the band images (DESIGN.md section 5.6): PSFR_MAX_BANDS and the psfr_band_psf / psfr_compute_bands
bindings against include/psfr.h, the quadrature of ``band_weights``, the effective wavelength, the BAND_* table columns
and cards through a FITS round trip, empty-batch shapes, and refusals of bad ``bands=`` before any device call."""
import io
import os
import re

import numpy as np
import pytest

import band_oracle as bo
from muse_psfr_b200 import _fits, _lib, psfrec

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LBDA = np.linspace(490, 930, 35)


def header():
    with open(os.path.join(ROOT, 'include', 'psfr.h')) as fh:
        return fh.read()


def declaration(name):
    decl = re.search(r'PSFR_API int %s\(([^;]*)\);' % name, header()).group(1)
    return [' '.join(a.split()) for a in decl.split(',')]


def test_max_bands_matches_header():
    assert int(re.search(r'#define PSFR_MAX_BANDS (\d+)', header()).group(1)) == _lib.MAX_BANDS == 16


def test_band_psf_binding_matches_declaration():
    args = declaration('psfr_band_psf')
    res, sig = _lib._SIGNATURES['psfr_band_psf']
    assert len(sig) == len(args) == 10
    assert sig == [_lib._I if re.match(r'int \w+$', a) else _lib._P for a in args]
    assert 'psfr_band_psf' in _lib.exported_symbols()


def test_compute_bands_binding_matches_declaration():
    args = declaration('psfr_compute_bands')
    res, sig = _lib._SIGNATURES['psfr_compute_bands']
    assert len(sig) == len(args) == 35
    assert sig == [_lib._I if re.match(r'int \w+$', a) else _lib._P for a in args]
    # psfr_compute_ao's arguments, then nband, weights, the six band outputs and the stream
    ao = _lib._SIGNATURES['psfr_compute_ao'][1]
    assert sig[:len(ao) - 1] == ao[:-1]
    assert args[len(ao) - 1:] == ['int nband', 'const double* weights', 'double* out_band', 'double* out_band_fit',
                                  'double* out_band_ee', 'double* out_mean_band', 'double* out_mean_band_fit',
                                  'double* out_mean_band_ee', 'void* stream']
    assert 'psfr_compute_bands' in _lib.exported_symbols()


# ---------------------------------------------------------------- band_weights
GRIDS = {'uniform': LBDA, 'non_uniform': np.cumsum(np.random.default_rng(4).uniform(2.0, 25.0, 30)) + 470.0}
CURVES = [([480.0, 930.0], [1.0, 1.0]), ([550.0, 600.0, 700.0, 750.0], [0.0, 0.9, 0.7, 0.0]),
          ([400.0, 640.0, 1000.0], [0.2, 1.0, 0.4])]


@pytest.mark.parametrize('grid', list(GRIDS))
@pytest.mark.parametrize('curve', range(len(CURVES)))
def test_weights_sum_to_the_trapezoid_integral(grid, curve):
    lam = GRIDS[grid]
    bl, tp = CURVES[curve]
    w = psfrec.band_weights(lam, bl, tp)
    T = np.interp(lam, bl, tp, left=0, right=0)
    assert w.shape == lam.shape and np.all(w >= 0)
    assert abs(w.sum() - bo.trapezoid(T, lam)) <= 1e-12 * bo.trapezoid(T, lam)
    # w_k = T_k delta_k with delta_k half the span of k's neighbours
    delta = np.gradient(lam) * np.r_[0.5, np.ones(lam.size - 2), 0.5]
    assert np.allclose(w, T * delta, rtol=1e-14, atol=0)


@pytest.mark.parametrize('grid', list(GRIDS))
def test_constant_throughput_integrates_to_the_grid_span(grid):
    lam = GRIDS[grid]
    w = psfrec.band_weights(lam, [lam[0] - 50, lam[-1] + 50], [0.5, 0.5])
    assert abs(2 * w.sum() - (lam[-1] - lam[0])) <= 1e-12
    w = psfrec.band_weights(lam, [lam[0], lam[-1]], [1.0, 1.0])
    assert abs(w.sum() - (lam[-1] - lam[0])) <= 1e-12


def test_single_wavelength_has_unit_width():
    assert np.array_equal(psfrec.band_weights([700.0], [600.0, 800.0], [0.3, 0.7]), [0.5])
    assert np.array_equal(psfrec.band_weights(700.0, [700.0], [0.25]), [0.25])


def test_bands_partly_off_the_grid():
    w = psfrec.band_weights(LBDA, [900.0, 1100.0], [1.0, 1.0])
    assert np.all(w[LBDA < 900] == 0) and np.all(w[LBDA >= 900] > 0)
    w = psfrec.band_weights(LBDA, [300.0, 495.0], [1.0, 1.0])
    assert np.array_equal(np.flatnonzero(w), [0]) and w[0] == (LBDA[1] - LBDA[0]) / 2


@pytest.mark.parametrize('args, match', [
    ((LBDA, [100.0, 400.0], [1.0, 1.0]), 'no weight'),
    ((LBDA, [940.0, 1000.0], [1.0, 1.0]), 'no weight'),
    ((LBDA, [500.0, 600.0], [0.0, 0.0]), 'no weight'),
    ((LBDA[::-1], [500.0, 600.0], [1.0, 1.0]), 'lbda'),
    ((np.r_[LBDA[:3], LBDA[2:]], [500.0, 600.0], [1.0, 1.0]), 'lbda'),
    ((LBDA, [600.0, 500.0], [1.0, 1.0]), 'band_lbda'),
    ((LBDA, [500.0, np.nan], [1.0, 1.0]), 'band_lbda'),
    (([], [500.0, 600.0], [1.0, 1.0]), 'lbda'),
    ((LBDA, [500.0, 600.0], [1.0, -0.1]), 'throughput'),
    ((LBDA, [500.0, 600.0], [1.0, np.inf]), 'throughput'),
    ((LBDA, [500.0, 600.0], [np.nan, 1.0]), 'throughput'),
    ((LBDA, [500.0, 600.0, 700.0], [1.0, 1.0]), 'throughput'),
])
def test_band_weights_refusals(args, match):
    with pytest.raises(ValueError, match=match):
        psfrec.band_weights(*args)


def test_effective_wavelength():
    w = np.stack([psfrec.band_weights(LBDA, [480.0, 940.0], [1.0, 1.0]), np.eye(35)[7],
                  psfrec.band_weights(LBDA, [600.0, 700.0], [0.2, 1.0])])
    eff = psfrec._band_lbda_eff(LBDA, w)
    assert abs(eff[0] - 710.0) < 1e-12 and eff[1] == LBDA[7] and 650 < eff[2] < 700
    assert np.allclose(eff, bo.lbda_eff(LBDA, w), rtol=1e-15, atol=0)
    # a power-of-two scale of the weights leaves the effective wavelength unchanged
    assert np.array_equal(psfrec._band_lbda_eff(LBDA, w * 2.0 ** 30), eff)


# ---------------------------------------------------------------- tables and shapes
def test_band_tables_through_fits():
    rng = np.random.default_rng(6)
    nb, npos, radii, fracs = 3, 2, np.array([0.4, 1.0]), np.array([0.5])
    w = np.stack([psfrec.band_weights(LBDA, bl, tp) for bl, tp in CURVES])
    fit = rng.random((1, nb, _lib.FIT_NPAR))
    fit[..., _lib.FIT_ITER] = 5
    ee = rng.random((1, nb, 4))
    meta = {'SEEING': 0.8, 'GL': 0.7, 'L0': 20.0}
    cols = psfrec._band_columns(LBDA, w, fit, ee, radii, fracs)
    assert list(cols) == ['lbda', 'center', 'flux', 'fwhm', 'n', 'peak', 'err_center', 'err_flux', 'err_fwhm',
                          'err_n', 'err_peak', 'converged', 'band', 'weights', 'ee', 'ee_total', 'r_ee']
    fit_f, ee_f = rng.random((npos, nb, _lib.FIT_NPAR)), rng.random((npos, nb, 4))
    fcols = psfrec._band_columns(LBDA, w, fit_f, ee_f, radii, fracs)
    fcols['x'] = np.repeat([0.0, 12.0], nb)
    fcols['y'] = np.repeat([0.0, -3.0], nb)
    cards = psfrec._ee_cards(meta, radii, fracs)
    hdul = _fits.HDUList([_fits.PrimaryHDU(), _fits.table_to_hdu(cols, meta=cards, name='BAND_MEAN'),
                          _fits.table_to_hdu(fcols, meta=cards, name='BAND_FIELD'),
                          _fits.table_to_hdu(psfrec._band_columns(LBDA, w, fit), meta=meta, name='PLAIN')])
    buf = io.BytesIO()
    hdul.writeto(buf)
    back = _fits.open(buf.getvalue())
    m = back['BAND_MEAN']
    assert np.array_equal(m.data['lbda'], psfrec._band_lbda_eff(LBDA, w))
    assert np.array_equal(m.data['band'], [0, 1, 2]) and np.array_equal(m.data['weights'], w)
    assert np.array_equal(m.data['fwhm'][:, 0], fit[0, :, _lib.FIT_FWHM] * 0.2)
    assert np.array_equal(m.data['ee_total'], ee[0, :, 2]) and np.array_equal(np.ravel(m.data['r_ee']), ee[0, :, 3] * 0.2)
    assert m.header['SEEING'] == 0.8 and m.header['L0'] == 20.0 and m.header['EERAD2'] == 1.0
    f = back['BAND_FIELD']
    assert np.array_equal(f.data['band'], [0, 1, 2, 0, 1, 2]) and np.array_equal(f.data['x'], [0, 0, 0, 12, 12, 12])
    assert np.array_equal(f.data['weights'], np.tile(w, (2, 1)))
    assert np.array_equal(f.data['n'], fit_f[..., _lib.FIT_N].ravel())
    assert np.array_equal(f.data['lbda'], np.tile(psfrec._band_lbda_eff(LBDA, w), 2))
    assert 'ee' not in back['PLAIN'].data.dtype.names and back['PLAIN'].header['GL'] == 0.7


def test_empty_batches_keep_the_shapes():
    lam = LBDA[:4]
    e = np.empty(0)
    w = np.ones((3, 4))
    fit, cube, bfit, bcube = psfrec.compute_psf_batch(lam, e, e, e, npsflin=3, bands=w, want_cube=False)
    assert cube is None and bfit.shape == (0, 3, _lib.FIT_NPAR) and bcube.shape == (0, 3, 40, 40)
    out = psfrec.compute_psf_batch(lam, e, e, e, bands=w[0], ee_radii=[0.5, 1.0], ao_budget=True)
    assert [o.shape for o in out[2:]] == [(0, 4, 5), (0, 4), (0, 1, _lib.VAR_NPAR), (0, 1, _lib.FIT_NPAR),
                                          (0, 1, 40, 40), (0, 1, 5)]
    pos = np.array([[0.0, 10.0], [0.0, -5.0]])
    out = psfrec.compute_psf_field(lam, e, e, e, positions=pos, elliptical=True, bands=w, ee_radii=[0.5])
    assert [o.shape for o in out[2:]] == [(0, 2, 4, _lib.EFIT_NPAR), (0, 2, 4, 4), (0, 2, 3, _lib.FIT_NPAR),
                                          (0, 2, 3, 40, 40), (0, 2, 3, 4)]


BAD_BANDS = [np.ones(34), np.ones((2, 36)), np.ones((17, 35)), np.ones((0, 35)), np.full(35, np.nan),
             np.r_[np.ones(34), -1.0], np.r_[np.ones(34), np.inf], np.zeros(35), np.full((2, 35), 1e308),
             np.ones((2, 2, 35))]


@pytest.mark.parametrize('bad', range(len(BAD_BANDS)))
def test_bad_bands_refused_before_any_device_call(bad, monkeypatch):
    def no_device(*a, **k):
        pytest.fail('a device context was requested')
    monkeypatch.setattr(psfrec, 'get_context', no_device)
    monkeypatch.setattr(psfrec, '_planes_context', no_device)
    w = BAD_BANDS[bad]
    with pytest.raises(ValueError):
        psfrec.compute_psf_batch(LBDA, [1.0], [0.7], [25.0], bands=w)
    with pytest.raises(ValueError):
        psfrec.compute_psf_batch(LBDA, [], [], [], bands=w)
    with pytest.raises(ValueError):
        psfrec.compute_psf_field(LBDA, [1.0], [0.7], [25.0], bands=w, ee_radii=[0.5])
    with pytest.raises(ValueError):
        psfrec.compute_psf_from_sparta(psfrec.create_sparta_table(nlines=2), bands=w)
    with pytest.raises(ValueError):
        psfrec.band_psf(np.ones((35, 40, 40)), w)


def test_restatement_identities():
    rng = np.random.default_rng(2)
    cube = rng.random((5, 6, 7))
    assert np.array_equal(bo.band_images(cube, np.eye(5)[3]), cube[3:4])
    w = rng.random((2, 5))
    ref = np.einsum('bk,kyx->byx', w, cube) / w.sum(axis=1)[:, None, None]
    assert np.allclose(bo.band_images(cube, w), ref, rtol=1e-14, atol=0)
    assert bo.band_sets(np.stack([cube, 2 * cube]), w).shape == (2, 2, 6, 7)
