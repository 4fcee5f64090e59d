"""CPU tests: the oracle (oracle/psfr_oracle.py) against the fixtures generated from
the reference's own code (tests/golden/ref_*.npz, made by oracle/make_goldens.py) and
against the reference's 2-decimal known answers (test_psfrec.py)."""
import numpy as np
import pytest
from numpy.testing import assert_allclose

import psfr_oracle as orc

LBDA35 = np.linspace(490, 930, 35)


def reduce_check(a, g, name, rtol):
    n = a.shape[-1]
    c = n // 2
    assert_allclose(a[c - 48:c + 48, c - 48:c + 48], g[name + '_centre'], rtol=rtol, atol=0)
    assert_allclose(a[::16, ::16], g[name + '_lattice'], rtol=rtol, atol=0)
    assert_allclose(a[[0, 1, c - 1, c, c + 1, n - 1], :], g[name + '_rows'], rtol=rtol, atol=0)
    assert_allclose(a.sum(), g[name + '_sum'], rtol=1e-13)
    assert_allclose(a.max(), g[name + '_max'], rtol=rtol)


@pytest.fixture(scope='module')
def psd1():
    return orc.simul_psd_wfm([0.7, 0.3], (100, 10000), 1.0, 25., npsflin=1, dim=1280)


def test_psd_config1(psd1, golden):
    g = golden('ref_config1')
    reduce_check(psd1[0], g, 'psd', 1e-13)
    assert_allclose(psd1[0, 600:680, 600:680], g['psd_aozone'], rtol=1e-13)
    # survey probe numbers (SURVEY 8c)
    assert_allclose(psd1.sum(), 197983124.22863141, rtol=1e-12)
    assert psd1[0, 640, 640] == 0
    assert_allclose(psd1[0, 600, 600], 67.99229083018449, rtol=1e-12)
    assert psd1[0, 640, 641] == psd1[0].max() == 11264666.183809344


def test_psd_to_psf_config1(psd1, golden):
    g = golden('ref_config1')
    pup = orc.pupil_mask(320, 640, 0.14)
    assert pup.sum() == 315376
    for lb in (490., 930.):
        psf = orc.psd_to_psf(psd1[0], pup, 8, lb * 1e-9)
        reduce_check(psf, g, 'psf%d' % lb, 1e-12)


def test_psf_muse_subset(psd1, golden):
    g = golden('ref_config1')
    idx = [0, 17, 34]
    cube = orc.psf_muse(psd1[0], LBDA35[idx])
    assert_allclose(cube, g['psf_muse'][idx], rtol=1e-12, atol=1e-18)
    assert_allclose(cube[0].max(), 0.06878001975345309, rtol=1e-12)
    assert_allclose(cube[2].max(), 0.1438347394519584, rtol=1e-12)


def test_structure_function_scaling(psd1):
    # SURVEY F5: Dphi(lbda) = (2 pi / lbda)^2 * Dphi_unit, OTF_tel is a constant
    pup = orc.pupil_mask(320, 640, 0.14)
    du = orc.structure_function_unit(psd1[0])
    otf = np.exp(-0.5 * (2 * np.pi / 710.) ** 2 * du) * orc.telescope_otf(pup, 1280)
    psf = np.real(np.fft.fftshift(np.fft.ifft2(np.fft.fftshift(otf))))
    psf /= psf.sum()
    assert_allclose(psf, orc.psd_to_psf(psd1[0], pup, 8, 710e-9), rtol=0, atol=1e-13 * psf.max())


def test_ao_zone_config3_and_sample(golden):
    g = golden('ref_config3')
    f, _, _, _ = orc.ao_frequency_tables()
    r0 = orc.seeing2r01(1.0, 0.5, 0.)
    ao = orc.dsp4muse([0.7, 0.3], np.array([100., 10000.]), 25., r0, orc.lgs_positions(True),
                      orc.direction_perf(3), vent=orc.wind_speed_for((100, 10000)))
    fit = orc.psd_fit(1280, 16, r0, 25., 1.5)[600:680, 600:680]
    zone = np.maximum(fit, np.fft.fftshift(ao, axes=(1, 2))) * (500 / (2 * np.pi)) ** 2
    assert_allclose(zone, g['psd_aozone'], rtol=1e-13)
    g4 = golden('ref_config4_sample')
    for k, i in enumerate(g4['pick']):
        p = orc.simul_psd_wfm([g4['GL'][i], 1 - g4['GL'][i]], (g4['h0'][i], g4['h1'][i]),
                              g4['seeing'][i], g4['L0'][i])
        assert_allclose(p[0, 600:680, 600:680], g4['psd_aozone'][k], rtol=1e-13)


def test_wind_dtype_quirk():
    assert orc.wind_speed_for((100, 10000))[0] == 12.0
    assert orc.wind_speed_for((100., 10000.))[0] == 12.5


def test_intrinsic_and_polyfit(golden):
    g = golden('ref_config1')
    fw, be = orc.muse_intrinsic_psf(LBDA35)
    assert_allclose(fw, g['intrinsic_fwhm'], rtol=1e-15)
    assert_allclose(be, g['intrinsic_beta'], rtol=1e-15)
    go = golden('oracle_config1')
    pol = orc.fit_psf_with_polynom(LBDA35, go['fwhm'], go['n'], output=1)
    assert_allclose(pol['fwhm_pol'], go['ref_fwhm_pol'], rtol=1e-12)
    assert_allclose(pol['beta_pol'], go['ref_beta_pol'], rtol=1e-12)
    assert_allclose(pol['fwhm_fit'], go['ref_fwhm_fit'], rtol=1e-12)


def test_known_answers_reference_tests(golden):
    """test_psfrec.py:121-128,162-170: (1, 0.7, 25) at 500/700/900 nm."""
    g = golden('ref_config1')
    lb = np.array([500., 700., 900.])
    psd = orc.simul_psd_wfm([0.7, 0.3], (100, 10000), 1.0, 25.)
    res, psf = orc.compute_psf(lb, 1.0, 0.7, 25.)
    assert ['%.2f' % v for v in res['fwhm']] == ['0.85', '0.73', '0.62']
    assert ['%.2f' % v for v in res['n']] == ['2.73', '2.55', '2.23']
    assert_allclose(res['center'], 20, atol=1e-3)
    assert_allclose(res['fwhm'], [0.8472, 0.7300, 0.6211], atol=1e-4)   # SURVEY 8c probe
    assert_allclose(res['n'], [2.7337, 2.5471, 2.2289], atol=1e-4)


def test_oracle_fit_goldens(golden):
    """Restated third-party pieces are stable against their committed outputs and
    reproduce the survey's probe values (config 1 final fit, pixels)."""
    g, go = golden('ref_config1'), golden('oracle_config1')
    idx = [0, 17, 34]
    conv = orc.convolve_final_psf(LBDA35[idx], 1.0, 0.7, 25., g['psf_muse'][idx])
    assert_allclose(conv, go['conv'][idx], rtol=1e-12, atol=1e-18)
    fit = orc.fit_psf_cube(LBDA35[idx], conv)
    assert_allclose(fit['fwhm'], go['fwhm'][idx], rtol=1e-7)
    assert_allclose(fit['n'], go['n'][idx], rtol=1e-7)
    assert_allclose(fit['fwhm'] / 0.2, [4.259131082, 3.617918095, 3.074829769], rtol=2e-7)
    assert_allclose(fit['n'], [2.734382913, 2.532256124, 2.191668971], rtol=2e-7)
    # test_psfrec.py:36-44 polynomial pins
    lb9 = np.linspace(500, 900, 9)
    assert abs(go['fwhm_pol'][0]) < 10  # sanity only; pins below use the 9-point grid


def test_kernel_is_normalised():
    k = orc.moffat2d_kernel(3.3, 2.0)
    assert k.shape == (41, 41)
    assert_allclose(k.sum(), 1.0, rtol=1e-14)
    assert k[20, 20] == k.max()


def test_sparta_row_selection():
    v = np.tile(np.array([1.0, 0.7, 25.0]), (2, 4, 1))
    v[0, 3, 2] = 150          # bad L0 on laser 4 -> three-LGS mode
    v[1, :, 2] = 1000         # whole row invalid
    jobs = orc.select_sparta_rows(v)
    assert len(jobs) == 1 and jobs[0][3] is True and jobs[0][4] == 1 and jobs[0][5] == -1
    jobs = orc.select_sparta_rows(v, mean_of_lgs=False)
    assert [j[5] for j in jobs] == [1, 2, 3]
