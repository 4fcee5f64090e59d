"""CPU checks of the star fits (psfr_moffat_fit_weighted, fit_psf_cube(var=, mask=, fit_back=)): the header's
record layout, the argument refusals made before any device call, the table layout, that the default
fit_psf_cube keeps its unweighted path, and the scipy restatement in star_fit_oracle against exact images and
finite differences."""
import os
import re

import numpy as np
import pytest

import efit_oracle as eo
import star_fit_oracle as so
from muse_psfr_b200 import _lib, psfrec

HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'include', 'psfr.h')


def test_back_record_matches_header():
    header = open(HEADER).read()
    for name in ('CONT', 'ERR_CONT', 'NPIX', 'NPAR'):
        m = re.search(r'PSFR_BACK_%s = (\d+)' % name, header)
        assert m and int(m.group(1)) == getattr(_lib, 'BACK_' + name)
    assert (so.CONT, so.ERR_CONT, so.NPIX, so.BACK_NPAR) == (0, 1, 2, 3)
    assert so.FIT_NPAR == _lib.FIT_NPAR and so.ITER == _lib.FIT_ITER and so.FLUX == _lib.FIT_FLUX
    assert 'psfr_moffat_fit_weighted' in _lib.exported_symbols()
    assert re.search(r'PSFR_API int psfr_moffat_fit_weighted\(', header)


class _NoDevice:
    """Stands in for the context: any device call fails the test."""

    def __getattr__(self, name):
        raise AssertionError('device call %s made' % name)


@pytest.fixture
def no_device(monkeypatch):
    monkeypatch.setattr(psfrec, 'get_context', lambda *a, **k: _NoDevice())


def _cube(nl=2, ny=9, nx=11):
    return np.ones((nl, ny, nx))


@pytest.mark.parametrize('kw', [
    dict(var=np.ones((2, 9, 10))),                 # wrong plane shape
    dict(var=np.ones((3, 9, 11))),                 # wrong plane count
    dict(mask=np.zeros((9, 10), bool)),
    dict(mask=np.zeros((1, 9, 11), bool)),
])
def test_shape_mismatch_refused(no_device, kw):
    with pytest.raises(ValueError):
        psfrec.fit_psf_cube([500., 600.], _cube(), **kw)


def test_nonpositive_variance_on_used_pixel_refused(no_device):
    var = np.ones((2, 9, 11))
    var[1, 4, 5] = 0.0
    with pytest.raises(ValueError, match=r'var\[1, 4, 5\]'):
        psfrec.fit_psf_cube([500., 600.], _cube(), var=var)
    var[1, 4, 5] = -2.0
    with pytest.raises(ValueError):
        psfrec.fit_psf_cube([500., 600.], _cube(), var=var[1], fit_back=True)


def test_nonpositive_variance_on_unused_pixel_accepted():
    """var <= 0 where the pixel is masked or not finite is not refused: such pixels get weight 0."""
    data = _cube()
    var = np.ones((2, 9, 11))
    var[0, 1, 1], var[1, 2, 2], var[0, 3, 3] = 0.0, -1.0, 0.0
    mask = np.zeros((9, 11), bool)
    mask[1, 1] = True
    data[1, 2, 2] = np.nan
    cube = np.ma.array(data, mask=np.zeros(data.shape, bool))
    cube.mask[0, 3, 3] = True
    d, w = psfrec._star_weights(cube, var, mask)
    assert w[0, 1, 1] == 0 and w[1, 2, 2] == 0 and w[0, 3, 3] == 0 and w[1, 1, 1] == 0
    assert np.count_nonzero(w == 0) == 4 and np.all(w[w > 0] == 1.0)
    assert np.isnan(d[1, 2, 2])          # the data are passed as they are; the library never reads them


def test_weights_are_inverse_variance():
    var = np.full((2, 9, 11), 4.0)
    var[:, 0, 0] = np.inf
    var[1, 3, 4] = np.nan
    _, w = psfrec._star_weights(_cube(), var, None)
    assert w.flags['C_CONTIGUOUS'] and w.dtype == np.float64
    assert w[0, 0, 0] == 0 and w[1, 3, 4] == 0 and np.all(w[w > 0] == 0.25)


@pytest.mark.parametrize('circular', [True, False])
def test_empty_cube_table(no_device, circular):
    tab = psfrec.fit_psf_cube(np.zeros(0), np.zeros((0, 9, 11)), circular=circular, fit_back=True)
    assert len(tab) == 0
    for col in ('cont', 'err_cont', 'npix', 'fwhm', 'n', 'converged'):
        assert col in tab.colnames
    assert tab['fwhm'].shape == (0, 2) and tab['npix'].dtype == np.int64


class _Recorder:
    def __init__(self, fill):
        self.calls, self.fill = [], fill

    def moffat_fit(self, nimg, ny, nx, imgs, params):
        self.calls.append('moffat_fit')
        params[:] = self.fill(params.shape[1])

    def moffat_fit_elliptical(self, nimg, ny, nx, imgs, params):
        self.calls.append('moffat_fit_elliptical')
        params[:] = self.fill(params.shape[1])

    def moffat_fit_weighted(self, nimg, ny, nx, imgs, weights, params, back=None, fit_back=False, elliptical=False):
        self.calls.append(('moffat_fit_weighted', weights is None, fit_back, elliptical))
        params[:] = self.fill(params.shape[1])
        back[:] = [0.5, 0.25, 42]


def _fill(npar):
    r = np.arange(npar, dtype=float) + 1.0
    r[_lib.FIT_ITER if npar == _lib.FIT_NPAR else _lib.EFIT_ITER] = 3
    return r


@pytest.mark.parametrize('circular', [True, False])
def test_default_path_unchanged(monkeypatch, circular):
    rec = _Recorder(_fill)
    monkeypatch.setattr(psfrec, 'get_context', lambda *a, **k: rec)
    tab = psfrec.fit_psf_cube([500., 600.], _cube(), circular=circular)
    assert rec.calls == ['moffat_fit' if circular else 'moffat_fit_elliptical']
    assert 'cont' not in tab.colnames


@pytest.mark.parametrize('circular', [True, False])
def test_star_table_columns_and_units(monkeypatch, circular):
    rec = _Recorder(_fill)
    monkeypatch.setattr(psfrec, 'get_context', lambda *a, **k: rec)
    tab = psfrec.fit_psf_cube([500., 600.], _cube(), circular=circular, var=np.full((9, 11), 2.0), fit_back=True)
    assert rec.calls == [('moffat_fit_weighted', False, True, not circular)]
    base = psfrec._table_from_fit if circular else psfrec._shape_table_from_fit
    ref = base(np.array([500., 600.]), np.tile(_fill(_lib.FIT_NPAR if circular else _lib.EFIT_NPAR), (2, 1)))
    assert tab.colnames == ref.colnames + ['cont', 'err_cont', 'npix']
    for c in ref.colnames:
        np.testing.assert_array_equal(tab[c], ref[c])        # fwhm in arcsec, centre in pixels, as today
    np.testing.assert_array_equal(tab['cont'], [0.5, 0.5])
    np.testing.assert_array_equal(tab['err_cont'], [0.25, 0.25])
    np.testing.assert_array_equal(tab['npix'], [42, 42])
    rec.calls.clear()
    psfrec.fit_psf_cube([500., 600.], _cube(), circular=circular, mask=np.zeros((9, 11), bool))
    assert rec.calls == [('moffat_fit_weighted', False, False, not circular)]


# ---- oracle self-checks

CIRC = np.array([3.0, 6.3, 7.8, 2.2, 2.6])
ELL = eo.theta_of(3.0, 6.3, 7.8, 2.8, 1.9, 35.0, 2.6)


@pytest.mark.parametrize('elliptical', [False, True])
@pytest.mark.parametrize('c', [0.0, 0.4, -0.3])
def test_oracle_recovers_exact_images(elliptical, c):
    rng = np.random.default_rng(7)
    truth = np.concatenate([ELL if elliptical else CIRC, [c]])
    img = so.render((13, 15), truth, elliptical, True)
    w = rng.uniform(0.2, 3.0, img.shape)
    w[rng.random(img.shape) < 0.2] = 0.0
    img[w == 0] = np.nan                              # unused pixels are never read
    start = truth * (1 + 1e-3 * np.where(np.arange(truth.size) % 2, 1, -1))
    start[-1] = c + 0.01
    rec, back, theta = so.star_fit(img, w, start, elliptical, True)
    scale = so.param_scale(truth, elliptical, peak=truth[0])
    assert np.all(np.abs(theta - truth) / scale < 1e-9)
    assert back[so.NPIX] == np.count_nonzero(w > 0)
    assert abs(back[so.CONT] - c) < 1e-9 * truth[0]


@pytest.mark.parametrize('elliptical', [False, True])
def test_oracle_jacobian_matches_finite_differences(elliptical):
    theta = np.concatenate([ELL if elliptical else CIRC, [0.3]])
    p, q = (a.ravel().astype(float) for a in np.indices((11, 12)))
    J = so.star_jacobian(theta, p, q, elliptical, True)
    for k in range(theta.size):
        h = 1e-6 * max(abs(theta[k]), 1e-2)
        tp, tm = theta.copy(), theta.copy()
        tp[k] += h
        tm[k] -= h
        fd = (so.star_model(tp, p, q, elliptical, True) - so.star_model(tm, p, q, elliptical, True)) / (2 * h)
        np.testing.assert_allclose(J[:, k], fd, rtol=1e-6, atol=1e-8 * np.abs(fd).max())


def test_oracle_unit_weights_reduce_to_unweighted_record():
    """With unit weights and no background the record is the unweighted one of efit_oracle / psfr_oracle."""
    img = so.render((13, 15), ELL, True, False)
    rng = np.random.default_rng(3)
    img = img + rng.normal(0, 1e-3, img.shape)
    rec, back, theta = so.star_fit(img, np.ones(img.shape), ELL, True, False)
    ref, th = eo.moffat_fit_elliptical(img, start=ELL)
    np.testing.assert_allclose(theta, th, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(rec, ref, rtol=1e-6)
    assert list(back) == [0.0, 0.0, img.size]
