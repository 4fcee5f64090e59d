"""CPU checks of the template fit (psfr_template_fit, fit_psf_template): the header's record layout against the _lib
constants, the exported symbol and its signature, the argument refusals made before any device call, the table
layout, and the scipy restatement in template_fit_oracle against scipy's own interpolation, finite differences and
exact images."""
import os
import re

import numpy as np
import pytest

import template_fit_oracle as to
from muse_psfr_b200 import _lib, psfrec

HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'include', 'psfr.h')
NAMES = ('FLUX', 'Y0', 'X0', 'CONT', 'CHISQ', 'QFIT', 'ITER', 'NPIX', 'ERR_FLUX', 'ERR_Y0', 'ERR_X0', 'ERR_CONT',
         'NPAR')


def test_record_matches_header():
    header = open(HEADER).read()
    for name in NAMES:
        m = re.search(r'PSFR_TFIT_%s = (\d+)' % name, header)
        assert m and int(m.group(1)) == getattr(_lib, 'TFIT_' + name)
        assert getattr(to, 'TFIT_NPAR' if name == 'NPAR' else name) == getattr(_lib, 'TFIT_' + name)


def test_symbol_and_signature():
    header = open(HEADER).read()
    m = re.search(r'PSFR_API int psfr_template_fit\(([^)]*)\)', header)
    assert m and 'psfr_template_fit' in _lib.exported_symbols()
    args = [a.strip() for a in m.group(1).split(',')]
    kinds = [_lib._P if '*' in a else _lib._I for a in args]
    res, sig = _lib._SIGNATURES['psfr_template_fit']
    assert res is _lib._I and sig == kinds and len(args) == 14


class _NoDevice:
    """Stands in for the context: any device call fails the test."""

    def __getattr__(self, name):
        raise AssertionError('device call %s made' % name)


@pytest.fixture
def no_device(monkeypatch):
    monkeypatch.setattr(psfrec, 'get_context', lambda *a, **k: _NoDevice())


def _stamps(n=4, ny=9, nx=11):
    return np.ones((n, ny, nx))


def _tpl(ntpl=2, ty=8, tx=8):
    return np.ones((ntpl, ty, tx))


def _nonfinite_tpl():
    t = _tpl()
    t[1, 3, 4] = np.nan
    return t


def _zero_sum_tpl():
    t = _tpl()
    t[0] -= 1.0
    return t


@pytest.mark.parametrize('args, kw', [
    ((_stamps(), _tpl(3)), {}),                                    # ntpl does not divide n
    ((_stamps(), np.ones(8)), {}),                                 # template not 2-d or 3-d
    ((_stamps(), np.ones((1, 1, 8, 8))), {}),
    ((_stamps(), _tpl()), dict(var=np.ones((4, 9, 10)))),          # wrong plane shape
    ((_stamps(), _tpl()), dict(var=np.ones((3, 9, 11)))),          # wrong plane count
    ((_stamps(), _tpl()), dict(mask=np.zeros((9, 10), bool))),
    ((np.ones((9, 11)), _tpl(1)), {}),                             # stamps not 3-d
    ((_stamps(), _nonfinite_tpl()), {}),
    ((_stamps(), _tpl(1) * -1.0), {}),                             # sums to < 0
    ((_stamps(), _zero_sum_tpl()), {}),                            # sums to 0
])
def test_refusals_before_device_call(no_device, args, kw):
    with pytest.raises(ValueError):
        psfrec.fit_psf_template(np.arange(args[0].shape[0] if args[0].ndim == 3 else 1) + 500.0, *args, **kw)


def test_wavelength_count_refused(no_device):
    with pytest.raises(ValueError):
        psfrec.fit_psf_template([500.0, 600.0], _stamps(), _tpl())


def test_nonpositive_variance_on_used_pixel_refused(no_device):
    var = np.ones((4, 9, 11))
    var[2, 4, 5] = 0.0
    with pytest.raises(ValueError, match=r'var\[2, 4, 5\]'):
        psfrec.fit_psf_template(np.arange(4.0), _stamps(), _tpl(), var=var)


class _Recorder:
    max_planes = 16

    def __init__(self):
        self.calls = []

    def template_fit(self, nimg, ny, nx, imgs, weights, tpls, params, model=None, fit_back=False):
        self.calls.append((nimg, ny, nx, tpls.shape, weights.shape, fit_back, model is not None))
        params[:] = np.arange(_lib.TFIT_NPAR, dtype=float) + 1.0
        params[:, _lib.TFIT_ITER] = np.resize([3, -200, 0, 5], nimg)
        if model is not None:
            model[:] = 7.0


def test_table_columns(monkeypatch, caplog):
    rec = _Recorder()
    monkeypatch.setattr(psfrec, 'get_context', lambda *a, **k: rec)
    tab, model = psfrec.fit_psf_template(np.arange(4.0) + 500, _stamps(), _tpl()[0], fit_back=True,
                                         return_model=True)
    assert rec.calls == [(4, 9, 11, (1, 8, 8), (4, 9, 11), True, True)]
    assert tab.colnames == ['lbda', 'center', 'err_center', 'flux', 'err_flux', 'cont', 'err_cont', 'chisq', 'qfit',
                            'npix', 'converged']
    r = np.arange(_lib.TFIT_NPAR, dtype=float) + 1.0
    np.testing.assert_array_equal(tab['center'][0], r[[_lib.TFIT_Y0, _lib.TFIT_X0]])
    np.testing.assert_array_equal(tab['err_center'][0], r[[_lib.TFIT_ERR_Y0, _lib.TFIT_ERR_X0]])
    for col, slot in (('flux', 'FLUX'), ('err_flux', 'ERR_FLUX'), ('cont', 'CONT'), ('err_cont', 'ERR_CONT'),
                      ('chisq', 'CHISQ'), ('qfit', 'QFIT')):
        assert tab[col][0] == r[getattr(_lib, 'TFIT_' + slot)]
    assert tab['npix'].dtype == np.int64 and tab['npix'][0] == r[_lib.TFIT_NPIX]
    np.testing.assert_array_equal(tab['converged'], [1, 0, 0, 1])
    assert 'did not converge for 2 of 4' in caplog.text
    assert model.shape == (4, 9, 11) and np.all(model == 7.0)
    assert isinstance(psfrec.fit_psf_template(np.arange(4.0), _stamps(), _tpl()), psfrec.FitTable)


def test_empty_input_table(no_device):
    tab = psfrec.fit_psf_template(np.zeros(0), np.zeros((0, 9, 11)), _tpl(1))
    assert len(tab) == 0 and 'qfit' in tab.colnames


# ---- oracle self-checks

def _psf(shape=(40, 40), c=(20.3, 19.6), a=2.5, n=2.7):
    p, q = np.indices(shape, dtype=float)
    return (1 + ((p - c[0]) ** 2 + (q - c[1]) ** 2) / a ** 2) ** (-n)


@pytest.mark.parametrize('shape', [(40, 40), (41, 37), (6, 5)])
def test_oracle_reproduces_samples_at_integer_points(shape):
    tpl = np.random.default_rng(2).random(shape)
    p, q = np.indices(shape, dtype=float)
    s, _, _ = to.sample_grad(to.coefficients(tpl), p.ravel(), q.ravel())
    np.testing.assert_allclose(s, tpl.ravel(), rtol=0, atol=1e-14)
    np.testing.assert_allclose(to.sample(tpl, p.ravel(), q.ravel()), tpl.ravel(), rtol=0, atol=1e-14)


def test_oracle_taps_match_map_coordinates():
    tpl = np.random.default_rng(3).random((17, 13))
    rng = np.random.default_rng(4)
    u, v = rng.uniform(-1, 17, 500), rng.uniform(-1, 13, 500)
    s, _, _ = to.sample_grad(to.coefficients(tpl), u, v)
    np.testing.assert_allclose(s, to.sample(tpl, u, v), rtol=0, atol=1e-14)
    assert np.all(s[(u < 0) | (u > 16) | (v < 0) | (v > 12)] == 0)


@pytest.mark.parametrize('shape', [(40, 40), (41, 37), (4, 7)])
def test_kernel_recursion_matches_spline_filter(shape):
    tpl = np.random.default_rng(5).random(shape)
    np.testing.assert_allclose(to.prefilter(tpl), to.coefficients(tpl), rtol=0, atol=1e-13)


@pytest.mark.parametrize('fit_back', [False, True])
def test_oracle_jacobian_matches_finite_differences(fit_back):
    tpl = _psf()
    coef, S = to.coefficients(tpl), tpl.sum()
    theta = np.array([150.0, 11.3, 12.7] + ([0.4] if fit_back else []))
    p, q = (a.ravel().astype(float) for a in np.indices((25, 25)))
    J = to.jacobian(theta, coef, S, p, q, fit_back)
    for k in range(theta.size):
        h = 1e-6 * max(abs(theta[k]), 1.0)
        tp, tm = theta.copy(), theta.copy()
        tp[k] += h
        tm[k] -= h
        fd = (to.model(tp, tpl, (25, 25), fit_back) - to.model(tm, tpl, (25, 25), fit_back)).ravel() / (2 * h)
        np.testing.assert_allclose(J[:, k], fd, rtol=1e-6, atol=1e-7 * np.abs(fd).max())


@pytest.mark.parametrize('fit_back', [False, True])
def test_oracle_recovers_noiseless_shifted_template(fit_back):
    tpl = _psf()
    truth = np.array([250.0, 12.37, 11.71] + ([0.8] if fit_back else []))
    img = to.model(truth, tpl, (25, 25), fit_back)
    rng = np.random.default_rng(6)
    w = rng.uniform(0.5, 2.0, img.shape)
    w[rng.random(img.shape) < 0.05] = 0.0
    img[w == 0] = np.nan
    rec, theta = to.template_fit(img, w, tpl, fit_back)
    np.testing.assert_allclose(theta, truth, rtol=1e-10, atol=1e-10)
    assert rec[to.CHISQ] < 1e-18 and rec[to.NPIX] == np.count_nonzero(w > 0)


def test_context_sized_for_host_templates(monkeypatch):
    """The host templates are staged whole: the context is asked for max_planes x max_lambda >= ntpl 40 x 40 planes
    (3681 templates with the default 16 planes: 231 wavelengths)."""
    rec, asked = _Recorder(), []

    def get_context(*a, **k):
        asked.append(k.get('max_lambda'))
        return rec

    monkeypatch.setattr(psfrec, 'get_context', get_context)
    psfrec.fit_psf_template(np.arange(3681.0), np.ones((3681, 5, 5)), np.ones((3681, 40, 40)))
    assert asked[-1] == 231 and 16 * 231 >= 3681 and 16 * 230 < 3681
    assert rec.calls[0][3] == (3681, 40, 40)
