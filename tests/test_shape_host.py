"""CPU tests of the elliptical fit's Python surface and of its CPU reference (tests/efit_oracle.py): argument
checks and empty inputs that need no device, the table layout, and the reference's own known answers."""
import numpy as np
import pytest
from numpy.testing import assert_allclose

import efit_oracle as eo
from muse_psfr_b200 import _lib, psfrec

LBDA = np.array([500., 700.])


def test_record_layout_matches_header():
    assert _lib.EFIT_NPAR == eo.NPAR == 24
    header = open(__file__.replace('tests/test_shape_host.py', 'include/psfr.h')).read()
    for name in ('PEAK', 'Y0', 'X0', 'A_MAJOR', 'A_MINOR', 'PA', 'N', 'FWHM_MAJOR', 'FWHM_MINOR', 'AXIS_RATIO',
                 'CHISQ', 'ITER', 'ERR_PEAK', 'ERR_Y0', 'ERR_X0', 'ERR_A_MAJOR', 'ERR_A_MINOR', 'ERR_PA', 'ERR_N',
                 'ERR_FWHM_MAJOR', 'ERR_FWHM_MINOR', 'ERR_AXIS_RATIO', 'FLUX', 'ERR_FLUX'):
        slot = getattr(_lib, 'EFIT_' + name)
        assert slot == getattr(eo, name), name
        assert 'PSFR_EFIT_%s = %d' % (name, slot) in header, name
    assert 'psfr_moffat_fit_elliptical' in _lib.exported_symbols()
    assert 'psfr_compute_field_shapes' in _lib.exported_symbols()


def test_compute_psf_field_elliptical_empty():
    fit, cube, efit = psfrec.compute_psf_field(LBDA, [], [], [], positions=[[0., 10.], [0., 5.]], elliptical=True)
    assert fit.shape == (0, 2, 2, 16) and cube.shape == (0, 2, 2, 40, 40) and efit.shape == (0, 2, 2, 24)
    fit, cube, efit = psfrec.compute_psf_field([], [1.0], [0.7], [25.], want_cube=False, elliptical=True)
    assert fit.shape == (1, 9, 0, 16) and cube is None and efit.shape == (1, 9, 0, 24)
    out = psfrec.compute_psf_field(LBDA, [], [], [])
    assert len(out) == 2


def test_compute_psf_field_elliptical_checks_arguments():
    with pytest.raises(ValueError, match=r'\[2, npos\]'):
        psfrec.compute_psf_field(LBDA, [1.0], [0.7], [25.], positions=np.zeros(2), elliptical=True)
    with pytest.raises(ValueError, match='one entry per draw'):
        psfrec.compute_psf_field(LBDA, [1.0, 0.9], [0.7], [25., 20.], elliptical=True)
    with pytest.raises(ValueError, match='finite'):
        psfrec.compute_psf_from_sparta(psfrec.create_sparta_table(nlines=2), field_positions=[[0.], [np.nan]],
                                       elliptical=True)


def test_empty_elliptical_table_layout_and_units():
    tab = psfrec.fit_psf_cube([], np.empty((0, 40, 40)), circular=False)
    assert tab.colnames == ['lbda', 'center', 'fwhm', 'axis_ratio', 'pa', 'n', 'peak', 'flux', 'err_center',
                            'err_fwhm', 'err_axis_ratio', 'err_pa', 'err_n', 'err_peak', 'err_flux', 'converged']
    assert len(tab) == 0 and tab['fwhm'].shape == (0, 2)
    rec = np.arange(2 * 24, dtype=float).reshape(2, 24) + 1
    rec[1, _lib.EFIT_ITER] = -200
    tab = psfrec._shape_table_from_fit(LBDA, rec)
    assert_allclose(tab['fwhm'], rec[:, [_lib.EFIT_FWHM_MAJOR, _lib.EFIT_FWHM_MINOR]] * 0.2)
    assert_allclose(tab['err_fwhm'], rec[:, [_lib.EFIT_ERR_FWHM_MAJOR, _lib.EFIT_ERR_FWHM_MINOR]] * 0.2)
    assert np.array_equal(tab['pa'], rec[:, _lib.EFIT_PA])          # degrees, no pixel scale
    assert np.array_equal(tab['center'], rec[:, [_lib.EFIT_Y0, _lib.EFIT_X0]])
    assert np.array_equal(tab['converged'], [1, 0])


@pytest.mark.parametrize('q', [1.0, 0.999, 0.98, 0.7])
@pytest.mark.parametrize('pa', [0., 30., 45., 90., 135., 179.9])
def test_oracle_known_answers(q, pa):
    n = {0.7: 1.5, 0.98: 2.5}.get(q, 4.0)
    truth = (1.9, 19.3, 20.6, 3.0, 3.0 * q, pa, n)
    rec, _ = eo.moffat_fit_elliptical(eo.render((40, 40), *truth))
    assert_allclose(rec[[eo.PEAK, eo.Y0, eo.X0, eo.A_MAJOR, eo.A_MINOR, eo.N, eo.AXIS_RATIO]],
                    [1.9, 19.3, 20.6, 3.0, 3.0 * q, n, q], rtol=1e-8)
    if q < 1:
        d = (rec[eo.PA] - pa + 90) % 180 - 90
        assert abs(np.deg2rad(d)) <= 1e-6 / (1 - q)
    assert 0 <= rec[eo.PA] < 180


def test_oracle_exact_circle_record():
    """At A = B, C = 0 the orientation is undefined: PA = 0 and its error +inf."""
    jtj = np.eye(7)
    rec = eo.record(np.array([1.0, 20., 20., 0.25, 0.25, 0.0, 2.5]), jtj, 1e-10, 100)
    assert rec[eo.PA] == 0 and rec[eo.ERR_PA] == np.inf and rec[eo.AXIS_RATIO] == 1.0
    assert np.isfinite(rec[eo.ERR_A_MAJOR]) and np.isfinite(rec[eo.ERR_AXIS_RATIO])


def test_oracle_delta_method_matches_finite_differences():
    """The analytic gradients of the derived quantities against central differences of record()."""
    theta = np.array([1.3, 19.1, 20.4, 0.13, 0.11, -0.02, 2.7])
    rng = np.random.default_rng(1)
    M = rng.normal(size=(7, 7))
    jtj = M @ M.T + 7 * np.eye(7)
    base = eo.record(theta, jtj, 1.0, 1)
    sigma = np.linalg.inv(jtj)
    h = 1e-6
    for slot, err in ((eo.A_MAJOR, eo.ERR_A_MAJOR), (eo.A_MINOR, eo.ERR_A_MINOR), (eo.PA, eo.ERR_PA),
                      (eo.FWHM_MAJOR, eo.ERR_FWHM_MAJOR), (eo.FWHM_MINOR, eo.ERR_FWHM_MINOR),
                      (eo.AXIS_RATIO, eo.ERR_AXIS_RATIO), (eo.FLUX, eo.ERR_FLUX)):
        g = np.empty(7)
        for i in range(7):
            d = np.zeros(7)
            d[i] = h * max(1.0, abs(theta[i]))
            g[i] = (eo.record(theta + d, jtj, 1.0, 1)[slot] - eo.record(theta - d, jtj, 1.0, 1)[slot]) / (2 * d[i])
        assert_allclose(base[err], np.sqrt(g @ sigma @ g), rtol=1e-6, err_msg=str(slot))


def test_oracle_delta_method_matches_finite_differences_long_double():
    """The same gradients through record_ld: the long-double record's errors against central differences of its
    own derived columns, with J^T J, chi^2 and dof over a noisy render."""
    truth = (1.3, 19.1, 20.4, 3.1, 2.2, 37.0, 2.7)
    img = eo.render_noisy((40, 40), truth, 1e-2, 3)
    theta = eo.theta_of(*truth)
    base = eo.record_ld(theta, img)
    p, q = (a.ravel().astype(float) for a in np.indices(img.shape))
    J = eo.jacobian(theta, p, q)
    r = eo.model(theta, p, q) - img.ravel()
    sigma = np.linalg.inv(J.T @ J) * (r @ r) / (img.size - 7)
    h = 1e-6
    for slot, err in ((eo.PEAK, eo.ERR_PEAK), (eo.Y0, eo.ERR_Y0), (eo.X0, eo.ERR_X0), (eo.N, eo.ERR_N),
                      (eo.A_MAJOR, eo.ERR_A_MAJOR), (eo.A_MINOR, eo.ERR_A_MINOR), (eo.PA, eo.ERR_PA),
                      (eo.FWHM_MAJOR, eo.ERR_FWHM_MAJOR), (eo.FWHM_MINOR, eo.ERR_FWHM_MINOR),
                      (eo.AXIS_RATIO, eo.ERR_AXIS_RATIO), (eo.FLUX, eo.ERR_FLUX)):
        g = np.empty(7)
        for i in range(7):
            d = np.zeros(7)
            d[i] = h * max(1.0, abs(theta[i]))
            up, dn = eo.record(theta + d, np.eye(7), 1.0, 1), eo.record(theta - d, np.eye(7), 1.0, 1)
            g[i] = (up[slot] - dn[slot]) / (2 * d[i])
        assert_allclose(base[err], np.sqrt(g @ sigma @ g), rtol=1e-6, err_msg=str(slot))


@pytest.mark.parametrize('seed', range(8))
def test_record_ld_matches_record_in_fp64(seed):
    """record_ld on random theta and a noisy image against record() fed the same J^T J, chi^2 and dof in FP64."""
    rng = np.random.default_rng(seed)
    shape = (int(rng.integers(8, 41)), int(rng.integers(8, 41)))
    amaj = rng.uniform(1.0, min(shape) / 4)
    truth = (rng.uniform(0.5, 3), (shape[0] - 1) / 2 + rng.uniform(-1, 1), (shape[1] - 1) / 2 + rng.uniform(-1, 1),
             amaj, amaj * rng.uniform(0.2, 0.99), rng.uniform(0, 180), rng.uniform(1.3, 6))
    img = eo.render_noisy(shape, truth, 10 ** rng.uniform(-4, -1), seed)
    theta = eo.theta_of(*truth) * (1 + 1e-4 * rng.normal(size=7))
    p, q = (a.ravel().astype(float) for a in np.indices(shape))
    J = eo.jacobian(theta, p, q)
    r = eo.model(theta, p, q) - img.ravel()
    ref = eo.record(theta, J.T @ J, r @ r, img.size - 7)
    got = eo.record_ld(theta, img)
    assert_allclose(got, ref, rtol=1e-12, atol=0)


@pytest.mark.parametrize('pa', [0.0, 1e-7, 30.0, 90.0 - 1e-6, 90.0, 135.0, 180.0 - 1e-7])
def test_theta_of_record_round_trips(pa):
    theta = eo.theta_of(1.7, 12.3, 15.8, 4.0, 2.5, pa, 2.2)
    rec = eo.record(theta, np.eye(7), 1.0, 1)
    back = eo.theta_of_record(rec)
    assert_allclose(back, theta, rtol=0, atol=1e-13 * np.abs(theta).max())
    assert_allclose(eo.record(back, np.eye(7), 1.0, 1), rec, rtol=1e-12)


@pytest.mark.parametrize('truth,shape', [
    ((1.0, 8.0, 8.0, 300.0, 270.0, 20.0, 1.05), (17, 17)),    # flat to 1e-3 over the image: I, a and n trade off
    ((1.0, 8.3, 7.7, 0.7, 0.14, 20.0, 10.0), (17, 17)),       # the whole PSF inside one pixel
])
def test_well_posed_refuses_ill_posed_images(truth, shape):
    with pytest.raises(AssertionError):
        eo.well_posed(eo.render(shape, *truth), truth)


@pytest.mark.parametrize('shape', [(40, 40), (17, 17)])
def test_grid_removals_are_exactly_the_ill_posed_cases(shape):
    """Every case the GPU grid keeps passes the guard; every case it removes fails it; every axis value is kept at
    least once."""
    kept, removed = eo.grid(shape)
    for i, t in kept:
        eo.well_posed(eo.render(shape, *t), t)
    for i, t in removed:
        with pytest.raises(AssertionError):
            eo.well_posed(eo.render(shape, *t), t)
    truths = [t for _, t in kept]
    assert {t[3] for t in truths} == set(eo.GRID_A_MAJOR)
    assert {round(t[4] / t[3], 6) for t in truths} == set(eo.GRID_Q)
    assert {t[6] for t in truths} == set(eo.GRID_N)
    assert {t[5] for t in truths} == set(eo.GRID_PA)

