"""CPU tests of the AO summaries (DESIGN.md section 5.5): the PSFR_VAR_* layout and the psfr_compute_ao binding
against include/psfr.h, the table and mean helpers of the Python surface, the empty-batch shapes, and the
identities of the numpy restatement in tests/ao_oracle.py."""
import os
import re

import numpy as np
import pytest

import ao_oracle as ao
from muse_psfr_b200 import _lib, psfrec

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header():
    with open(os.path.join(ROOT, 'include', 'psfr.h')) as fh:
        return fh.read()


def test_var_record_layout_matches_header():
    values = dict((k, int(v)) for k, v in re.findall(r'PSFR_VAR_([A-Z0-9]+)\s*=\s*(\d+)', header()))
    assert values == {'TOTAL': _lib.VAR_TOTAL, 'FIT': _lib.VAR_FIT, 'NOISE': _lib.VAR_NOISE, 'PROJ': _lib.VAR_PROJ,
                      'LAYER0': _lib.VAR_LAYER0, 'NPAR': _lib.VAR_NPAR}
    assert _lib.VAR_LAYER0 + _lib.MAX_LAYERS == _lib.VAR_NPAR == ao.VAR_NPAR


def test_compute_ao_binding_matches_declaration():
    decl = re.search(r'PSFR_API int psfr_compute_ao\(([^;]*)\);', header()).group(1)
    args = [a.strip() for a in decl.split(',')]
    res, sig = _lib._SIGNATURES['psfr_compute_ao']
    assert len(sig) == len(args) == 27
    kinds = [_lib._I if re.match(r'int \w+$', a) else _lib._P for a in args]
    assert sig == kinds
    # psfr_compute_energy's arguments, then out_strehl and out_var, then the stream
    energy = _lib._SIGNATURES['psfr_compute_energy'][1]
    assert sig[:-3] == energy[:-1] and args[-3:] == ['double* out_strehl', 'double* out_var', 'void* stream']
    assert 'psfr_compute_ao' in _lib.exported_symbols()


def test_ao_table_columns_and_broadcast():
    lbda = np.array([490.0, 700.0, 930.0])
    strehl = np.array([0.1, 0.3, 0.5])
    rec = np.arange(_lib.VAR_NPAR, dtype=float) + 1
    tab = psfrec._ao_table(lbda, strehl, rec)
    assert tab.colnames == ['lbda', 'strehl', 'var_total', 'var_fit', 'var_noise', 'var_proj']
    assert np.array_equal(tab['strehl'], strehl)
    for name, slot in (('var_total', 0), ('var_fit', 1), ('var_noise', 2), ('var_proj', 3)):
        assert np.array_equal(tab[name], np.full(3, rec[slot])), name
    recs = np.stack([rec, 2 * rec, 3 * rec])
    tab = psfrec._ao_table(lbda, strehl, recs)
    assert np.array_equal(tab['var_noise'], recs[:, _lib.VAR_NOISE])
    assert len(psfrec._ao_table(np.empty(0), np.empty(0), np.empty((0, _lib.VAR_NPAR)))) == 0


def test_draw_mean_sums_in_draw_order():
    x = np.array([[1e16, 1.0], [1.0, 2.0], [-1e16, 3.0], [1.0, 4.0]])
    # in order: ((1e16 + 1) - 1e16) + 1 = 1 (the first 1 is absorbed), a pairwise sum would give 2
    assert np.array_equal(psfrec._draw_mean(x), np.array([1.0 / 4, 10.0 / 4]))
    y = np.random.default_rng(1).random((7, 3, 5))
    acc = y[0].copy()
    for row in y[1:]:
        acc = acc + row
    assert np.array_equal(psfrec._draw_mean(y), acc / 7)


def test_empty_batches_keep_the_shapes():
    lam = np.array([500.0, 700.0])
    e = np.empty(0)
    fit, cube, strehl, var = psfrec.compute_psf_batch(lam, e, e, e, npsflin=3, ao_budget=True)
    assert fit.shape == (0, 2, _lib.FIT_NPAR) and cube.shape == (0, 2, 40, 40)
    assert strehl.shape == (0, 2) and var.shape == (0, 9, _lib.VAR_NPAR)
    fit, cube, ee, strehl, var = psfrec.compute_psf_batch(e, [1.0], [0.7], [25.0], ee_radii=[0.5], ao_budget=True)
    assert ee.shape == (1, 0, 4) and strehl.shape == (1, 0) and var.shape == (1, 1, _lib.VAR_NPAR)
    pos = np.array([[0.0, 10.0], [0.0, -5.0]])
    out = psfrec.compute_psf_field(lam, e, e, e, positions=pos, elliptical=True, ao_budget=True)
    assert [o.shape for o in out[2:]] == [(0, 2, 2, _lib.EFIT_NPAR), (0, 2, 2), (0, 2, _lib.VAR_NPAR)]


@pytest.mark.parametrize('case', [
    dict(Cn2=[0.7, 0.3], h=(100, 10000), seeing=1.0, L0=25.0),
    dict(Cn2=[0.5, 0.5], h=(300.0, 8000.0), seeing=0.6, L0=12.0, zenith=30.0, npsflin=2, three_lgs_mode=True),
])
def test_restatement_identities(case):
    """TOTAL = FIT + NOISE + PROJ and PROJ = sum of LAYER to 1e-13; TOTAL = sum(simul_psd_wfm) / L^2 to 1e-12."""
    rec = ao.variance_record(**case)
    assert np.all(rec[:, :4] > 0)
    for r in rec:
        assert abs(r[1] + r[2] + r[3] - r[0]) <= 1e-13 * r[0]
        assert abs(r[4:].sum() - r[3]) <= 1e-13 * r[3]
        assert np.all(r[4 + len(case['Cn2']):] == 0)
    assert np.allclose(rec[:, 0], ao.psd_total(**case), rtol=1e-12, atol=0)


def assert_identities(rec, nl):
    for r in rec:
        assert abs(r[1] + r[2] + r[3] - r[0]) <= 1e-13 * r[0]
        assert abs(r[4:].sum() - r[3]) <= 1e-13 * r[3]
        assert np.all(r[4 + nl:] == 0)


def test_restatement_dim2560():
    """At dim 2560 the zone sits at the same frequencies as at 1280: NOISE, PROJ and the layers are the same,
    FIT and TOTAL gain the fitting PSD of the wider grid (0.3 % of FIT for config 1)."""
    case = dict(Cn2=[0.7, 0.3], h=(100, 10000), seeing=1.0, L0=25.0, npsflin=2)
    big, small = ao.variance_record(dim=2560, **case), ao.variance_record(**case)
    assert_identities(big, 2)
    assert np.allclose(big[:, 0], ao.psd_total(dim=2560, **case), rtol=1e-12, atol=0)
    assert np.allclose(big[:, 2:], small[:, 2:], rtol=1e-13, atol=0)
    assert np.all(big[:, 1] / small[:, 1] - 1 > 2e-3)
    assert ao.zone_margin(dim=2560, **case) > 1e-12


def test_restatement_with_dirs():
    """dirs = direction_perf(n) is npsflin = n bit for bit, and every direction's record is that of a call with
    that direction alone, far outside the laser asterism too."""
    case = dict(Cn2=[0.6, 0.4], h=(300.0, 9000.0), seeing=1.3, L0=18.0, zenith=15.0, three_lgs_mode=True)
    assert np.array_equal(ao.variance_record(dirs=psfrec.direction_perf(3), **case),
                          ao.variance_record(npsflin=3, **case))
    pos = np.array([[0., -30., 12.5, 120., -120., 300.], [0., 30., -7.3, 60., 60., 0.]])
    rec = ao.variance_record(dirs=pos, **case)
    assert_identities(rec, 2)
    for k in range(pos.shape[1]):
        assert np.array_equal(rec[k], ao.variance_record(dirs=pos[:, k:k + 1], **case)[0])
    assert ao.zone_margin(dirs=pos, **case) > 1e-12


def test_restatement_zero_weight_layer():
    """A layer of weight 0 has the slot 0 exactly, and the record is that of the profile without the layer."""
    kw = dict(seeing=0.8, L0=30.0, zenith=45.0)
    rec = ao.variance_record([0.5, 0.0, 0.3, 0.2], (50.0, 2000.0, 6000.0, 14000.0), wind_dir=[0.3, 1.1, -2.0, 2.6],
                             dirs=[[0.0, 40.0], [0.0, -20.0]], **kw)
    assert_identities(rec, 4)
    assert np.all(rec[:, 5] == 0) and np.all(rec[:, [4, 6, 7]] > 0)
    ref = ao.variance_record([0.5, 0.3, 0.2], (50.0, 6000.0, 14000.0), wind_dir=[0.3, -2.0, 2.6],
                             dirs=[[0.0, 40.0], [0.0, -20.0]], **kw)
    assert np.array_equal(rec[:, :4], ref[:, :4])
    assert np.array_equal(rec[:, [4, 6, 7]], ref[:, 4:7])
