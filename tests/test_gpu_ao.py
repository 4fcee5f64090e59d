"""GPU tests of the AO summaries (DESIGN.md section 5.5): the Strehl ratio and the residual-phase variance record of
``psfr_compute_ao``, their Python surface (``compute_psf_batch`` / ``compute_psf_field(ao_budget=True)``) and the
AO_MEAN / AO_FIELD HDUs of the SPARTA shell.

The Strehl ratio against the full-grid centre ratio of psfr_psd_to_psf and of the numpy oracle, the variance record
against the restatement of tests/ao_oracle.py, the records against themselves across chunk sizes, entry points and
host / device outputs, and every other output against psfr_compute_energy bit for bit."""
import numpy as np
import pytest
from numpy.testing import assert_allclose

import ao_oracle as ao
from test_gpu_field import GRID3, GROUPS3, LBDA6, POS7, group_inputs, own_context
from test_gpu_sparta_batch import config2_table, seeded_table

pytestmark = pytest.mark.gpu

LAM3 = np.array([490.0, 700.0, 930.0])
# config 1 and the corners of the seeing / L0 envelope
DRAWS = [(1.0, 0.7, 25.0), (0.4, 0.7, 9.0), (0.4, 0.7, 29.0), (2.0, 0.7, 9.0), (2.0, 0.7, 29.0)]


@pytest.fixture(scope='module')
def psfrec():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    from muse_psfr_b200 import psfrec as mod
    mod.set_device(0)
    mod.release_contexts()
    yield mod
    mod.release_contexts()


def draw_records(psfrec, draws=DRAWS):
    seeing, GL, L0 = (np.array(c) for c in zip(*draws))
    return psfrec._mode_records(np.zeros(len(draws), bool), seeing, GL, L0)


def ao_outputs(nd, P, ndir, nl):
    from muse_psfr_b200 import _lib
    return dict(out_strehl=np.full((nd, P, nl), np.nan), out_var=np.full((nd, ndir, _lib.VAR_NPAR), np.nan))


def launches(ctx, fn, *args, **kw):
    n0 = ctx.kernel_launches()
    fn(*args, **kw)
    return ctx.kernel_launches() - n0


# ---------------------------------------------------------------- 1. Strehl against the full grid
def full_grid_strehl(ctx, recs, lgs, lam, dim):
    """psf[N/2][N/2] / psf_diff[N/2][N/2] of psfr_psd_to_psf: the PSD of each draw from psfr_psd, the diffraction
    PSF from psfr_load_psd of zeros, all in one workspace."""
    nd = len(recs)
    psd = np.zeros((nd + 1, dim, dim))
    ctx.psd(recs, np.zeros((2, 1)), lgs, out=psd[:nd])
    ctx.load_psd(psd, nd + 1)
    ctx.structure_function(nd + 1)
    out = np.empty((dim, dim))
    centre = np.empty((nd + 1, lam.size))
    for p in range(nd + 1):
        for k, lb in enumerate(lam):
            ctx.psd_to_psf(p, lb * 1e-9, out)
            centre[p, k] = out[dim // 2, dim // 2]
    return centre[:nd] / centre[nd], psd[:nd]


OPTION_SETS = {'default': {}, 'all_fp64': {'OPT_EXP_GRADE': 1e30, 'OPT_F32_ROWS': 1e30},
               'no_cut': {'OPT_EXP_CUT': 1000.0}}


@pytest.mark.parametrize('dim', [1280, 2560])
@pytest.mark.parametrize('options', list(OPTION_SETS))
def test_strehl_against_full_grid(psfrec, dim, options):
    from muse_psfr_b200 import _lib
    recs = draw_records(psfrec)
    lgs = psfrec._lgs_positions(False)
    ctx = own_context(psfrec, len(recs) + 1, dim)
    try:
        base = ao_outputs(len(recs), 1, 1, LAM3.size)
        ctx.compute_ao(False, recs, np.zeros((2, 1)), lgs, LAM3, **base)
        for key, value in OPTION_SETS[options].items():
            ctx.set_option(getattr(_lib, key), value)
        out = ao_outputs(len(recs), 1, 1, LAM3.size)
        ctx.compute_ao(False, recs, np.zeros((2, 1)), lgs, LAM3, **out)
        s = out['out_strehl'][:, 0]
        # the cut and the single-precision grades move the sum by less than 1e-14 of sum OTF_tel
        assert np.max(np.abs(s - base['out_strehl'][:, 0])) < 1e-14
        ref, psd = full_grid_strehl(ctx, recs, lgs, LAM3, dim)
        assert_allclose(s, ref, rtol=1e-9, atol=0)
        assert np.all((s > 0) & (s <= 1))
        if dim == 1280 and options == 'default':      # two cases against the numpy oracle
            for i, k in ((0, 1), (3, 2)):
                assert_allclose(s[i, k], ao.strehl(psd[i], LAM3[k] * 1e-9), rtol=1e-9, atol=0)
    finally:
        ctx.close()


def test_strehl_field_mean_and_single_position(psfrec):
    seeing, GL, L0 = [0.8, 1.3], [0.6, 0.8], [15.0, 22.0]
    _, _, s_mean, v_mean = psfrec.compute_psf_batch(LBDA6, seeing, GL, L0, npsflin=3, want_cube=False,
                                                    ao_budget=True)
    _, _, s_pos, v_pos = psfrec.compute_psf_field(LBDA6, seeing, GL, L0, positions=GRID3, want_cube=False,
                                                  ao_budget=True)
    assert_allclose(s_mean, s_pos.mean(axis=1), rtol=1e-12, atol=0)
    assert np.array_equal(v_mean, v_pos)          # the same (draw, direction) planes
    _, _, s1, v1 = psfrec.compute_psf_batch(LBDA6, seeing, GL, L0, want_cube=False, ao_budget=True)
    _, _, s1f, v1f = psfrec.compute_psf_field(LBDA6, seeing, GL, L0, positions=[[0.0], [0.0]], want_cube=False,
                                              ao_budget=True)
    assert np.array_equal(s1, s1f[:, 0]) and np.array_equal(v1, v1f)


def test_strehl_physics_on_a_seeded_sweep(psfrec):
    rng = np.random.default_rng(11)
    seeing = np.sort(rng.uniform(0.4, 2.0, 12))
    lam = np.linspace(490, 930, 35)
    _, _, s, _ = psfrec.compute_psf_batch(lam, seeing, np.full(12, 0.7), np.full(12, 20.0), want_cube=False,
                                          ao_budget=True)
    assert np.all((s > 0) & (s <= 1))
    assert np.all(np.diff(s, axis=1) > 0)          # rises with the wavelength
    assert np.all(np.diff(s, axis=0) < 0)          # falls with the seeing


# ---------------------------------------------------------------- 2. variance against the restatement
VAR_CASES = [
    dict(Cn2=[1.0], h=(4000.0,), wind_dir=[0.4], seeing=0.9, L0=20.0),
    dict(Cn2=[0.7, 0.3], h=(100, 10000), seeing=1.1, L0=25.0, three_lgs_mode=True),
    dict(Cn2=[0.3, 0.15, 0.1, 0.1, 0.1, 0.1, 0.05, 0.1], h=(30.0, 200.0, 800.0, 2000.0, 4500.0, 8000.0, 12000.0,
                                                             16000.0),
         wind_dir=[0.1, 0.9, -0.4, 2.0, 3.0, -2.5, 1.3, 0.0], seeing=0.7, L0=15.0, npsflin=3, zenith=30.0),
    dict(Cn2=[0.6, 0.4], h=(300.0, 9000.0), seeing=1.6, L0=12.0, npsflin=2, zenith=45.0, three_lgs_mode=True),
]


@pytest.mark.parametrize('case', range(len(VAR_CASES)))
def test_variance_against_restatement(psfrec, case):
    c = dict(VAR_CASES[case])
    npsflin, three, zenith = c.pop('npsflin', 1), c.pop('three_lgs_mode', False), c.pop('zenith', 0.0)
    Cn2, h, wind_dir = c['Cn2'], c['h'], c.get('wind_dir')
    _, _, s, var = psfrec.compute_psf_batch(LAM3, [c['seeing']], [0.7], [c['L0']], npsflin=npsflin, h=h,
                                            three_lgs_mode=three, want_cube=False, zenith=zenith, Cn2=Cn2,
                                            wind_dir=wind_dir, ao_budget=True)
    ref = ao.variance_record(Cn2, h, c['seeing'], c['L0'], zenith, npsflin, three, wind_dir)
    assert var.shape == (1, npsflin ** 2, ao.VAR_NPAR)
    assert_allclose(var[0], ref, rtol=1e-10, atol=0)
    assert_allclose(var[0, :, 0], ao.psd_total(Cn2, h, c['seeing'], c['L0'], zenith, npsflin, three, wind_dir),
                    rtol=1e-10, atol=0)
    for r in var[0]:
        assert abs(r[1] + r[2] + r[3] - r[0]) <= 1e-13 * r[0]
        assert abs(r[4:].sum() - r[3]) <= 1e-13 * r[3]
        assert np.all(r[4 + len(Cn2):] == 0)


def test_variance_total_is_the_psd_sum(psfrec):
    """TOTAL is the sum of psfr_psd's N x N PSD over L^2 = 256 m^2."""
    recs = draw_records(psfrec)[:2]
    ctx = own_context(psfrec, 2)
    try:
        out = ao_outputs(2, 1, 1, 1)
        ctx.compute_ao(False, recs, np.zeros((2, 1)), psfrec._lgs_positions(False), LAM3[:1], **out)
        psd = np.empty((2, 1280, 1280))
        ctx.psd(recs, np.zeros((2, 1)), psfrec._lgs_positions(False), out=psd)
        assert_allclose(out['out_var'][:, 0, 0], psd.sum(axis=(1, 2)) / 256, rtol=1e-12, atol=0)
    finally:
        ctx.close()


# ---------------------------------------------------------------- 3. bits and plumbing
def full_outputs(nd, P, ndir, nl, ng, rec):
    from muse_psfr_b200 import _lib
    out = dict(out_cube=np.full((nd, P, nl, 40, 40), np.nan), out_fit=np.full((nd, P, nl, _lib.FIT_NPAR), np.nan),
               out_mean=np.full((ng, P, nl, 40, 40), np.nan), out_mean_fit=np.full((ng, P, nl, _lib.FIT_NPAR), np.nan),
               out_efit=np.full((nd, P, nl, _lib.EFIT_NPAR), np.nan),
               out_mean_efit=np.full((ng, P, nl, _lib.EFIT_NPAR), np.nan),
               out_ee=np.full((nd, P, nl, rec), np.nan), out_mean_ee=np.full((ng, P, nl, rec), np.nan))
    out.update(ao_outputs(nd, P, ndir, nl))
    return out


RAD, FR = np.array([1.0, 3.5]), np.array([0.5])


@pytest.mark.parametrize('field', [False, True])
def test_records_across_chunks_entry_points_and_outputs(psfrec, field):
    import torch
    recs, lgs = group_inputs(psfrec)
    npos = 3
    pos = np.ascontiguousarray(POS7[:, [1, 5, 6]] if field else GRID3[:, [0, 4, 8]])
    P = npos if field else 1
    nl, nd, ng = LBDA6.size, len(recs), len(GROUPS3)
    first = None
    for max_planes in (3, 8, 128):
        ctx = own_context(psfrec, max_planes)
        try:
            out = full_outputs(nd, P, npos, nl, ng, 4)
            ctx.compute_groups(recs, pos, lgs, LBDA6, GROUPS3, out_fit=out['out_fit'])   # MUSE kernels built once
            n_ao = launches(ctx, ctx.compute_ao, field, recs, pos, lgs, LBDA6, RAD, FR, GROUPS3, **out)
            plain = {k: np.full(v.shape, np.nan) for k, v in out.items() if k not in ('out_strehl', 'out_var')}
            n_energy = launches(ctx, ctx.compute_energy, field, recs, pos, lgs, LBDA6, RAD, FR, GROUPS3, **plain)
            for k, v in plain.items():
                assert np.array_equal(out[k], v), (max_planes, k)
            # NULL AO outputs launch nothing new; each adds one launch per chunk
            same = {k: np.full(v.shape, np.nan) for k, v in plain.items()}
            assert launches(ctx, ctx.compute_ao, field, recs, pos, lgs, LBDA6, RAD, FR, GROUPS3, **same) == n_energy
            chunks = -(-nd // (max_planes // npos))
            assert n_ao == n_energy + 2 * chunks, max_planes
            only = ao_outputs(nd, P, npos, nl)
            ctx.compute_ao(field, recs, pos, lgs, LBDA6, group_end=GROUPS3, out_var=only['out_var'])
            ctx.compute_ao(field, recs, pos, lgs, LBDA6, group_end=GROUPS3, out_strehl=only['out_strehl'])
            dev = {k: torch.full(v.shape, float('nan'), dtype=torch.float64, device='cuda') for k, v in only.items()}
            ctx.compute_ao(field, recs, pos, lgs, LBDA6, group_end=GROUPS3, **dev)
            torch.cuda.synchronize()
            for k in only:
                assert np.array_equal(only[k], out[k]), (max_planes, k)
                assert np.array_equal(dev[k].cpu().numpy(), out[k]), (max_planes, k)
            mixed = dict(out_strehl=dev['out_strehl'].zero_(), out_var=np.full(out['out_var'].shape, np.nan))
            ctx.compute_ao(field, recs, pos, lgs, LBDA6, group_end=GROUPS3, out_fit=out['out_fit'], **mixed)
            torch.cuda.synchronize()
            assert np.array_equal(mixed['out_strehl'].cpu().numpy(), out['out_strehl'])
            assert np.array_equal(mixed['out_var'], out['out_var'])
        finally:
            ctx.close()
        got = (out['out_strehl'], out['out_var'])
        if first is None:
            first = got
        else:
            assert all(np.array_equal(a, b) for a, b in zip(got, first)), max_planes
    # the variance of a plane does not depend on the mode, nor the Strehl ratio of a one-position field
    ctx = own_context(psfrec, 8)
    try:
        other = ao_outputs(nd, npos if not field else 1, npos, nl)
        ctx.compute_ao(not field, recs, pos, lgs, LBDA6, group_end=GROUPS3, **other)
        assert np.array_equal(other['out_var'], first[1])
        one = ao_outputs(nd, 1, 1, nl)
        ctx.compute_ao(True, recs, np.ascontiguousarray(pos[:, :1]), lgs, LBDA6, **one)
        two = ao_outputs(nd, 1, 1, nl)
        ctx.compute_ao(False, recs, np.ascontiguousarray(pos[:, :1]), lgs, LBDA6, **two)
        assert np.array_equal(one['out_strehl'], two['out_strehl']) and np.array_equal(one['out_var'], two['out_var'])
        if field:
            assert np.array_equal(one['out_strehl'][:, 0], first[0][:, 0])
    finally:
        ctx.close()


def test_python_results_unchanged_by_ao_budget(psfrec):
    seeing, GL, L0 = [0.9, 1.4, 0.6], [0.7, 0.5, 0.8], [25.0, 14.0, 20.0]
    for three in (False, [False, True, False]):
        ref = psfrec.compute_psf_batch(LBDA6, seeing, GL, L0, npsflin=2, three_lgs_mode=three, ee_radii=[0.3])
        got = psfrec.compute_psf_batch(LBDA6, seeing, GL, L0, npsflin=2, three_lgs_mode=three, ee_radii=[0.3],
                                       ao_budget=True)
        assert len(got) == 5 and all(np.array_equal(a, b) for a, b in zip(got[:3], ref))
        plain = psfrec.compute_psf_batch(LBDA6, seeing, GL, L0, npsflin=2, three_lgs_mode=three)
        got = psfrec.compute_psf_batch(LBDA6, seeing, GL, L0, npsflin=2, three_lgs_mode=three, ao_budget=True)
        assert all(np.array_equal(a, b) for a, b in zip(got[:2], plain))
    ref = psfrec.compute_psf_field(LBDA6, seeing, GL, L0, positions=POS7, elliptical=True)
    got = psfrec.compute_psf_field(LBDA6, seeing, GL, L0, positions=POS7, elliptical=True, ao_budget=True)
    assert len(got) == 5 and all(np.array_equal(a, b) for a, b in zip(got[:3], ref))
    assert got[3].shape == (3, 7, LBDA6.size) and got[4].shape == (3, 7, ao.VAR_NPAR)


def test_refusals_match_compute_energy(psfrec):
    from muse_psfr_b200 import _lib
    recs, lgs = group_inputs(psfrec)
    ctx = own_context(psfrec, 8)
    try:
        bad = [dict(group_end=np.array([4, 3, 11], dtype=np.int32)),
               dict(group_end=np.array([4, 5, 10], dtype=np.int32)),
               dict(group_end=None, out_mean=np.empty((1, 1, LBDA6.size, 40, 40))),
               dict(group_end=GROUPS3, fracs=[1.5]),
               dict(group_end=GROUPS3, radii=[-1.0])]
        for kw in bad:
            kw = dict(kw)
            rad, fr = kw.pop('radii', RAD), kw.pop('fracs', FR)
            codes = []
            for fn in (ctx.compute_energy, ctx.compute_ao):
                out = ao_outputs(len(recs), 1, 3, LBDA6.size) if fn == ctx.compute_ao else {}
                with pytest.raises(_lib.PsfrError) as exc:
                    fn(False, recs, GRID3[:, :3].copy(), lgs, LBDA6, rad, fr, **kw, **out)
                codes.append(exc.value.code)
                assert all(np.all(np.isnan(v)) for v in out.values())
            assert codes[0] == codes[1] != 0, kw
    finally:
        ctx.close()


# ---------------------------------------------------------------- 4. SPARTA shell
def test_sparta_ao_hdus(psfrec):
    from muse_psfr_b200 import _lib
    tables = [config2_table(), seeded_table(7, 5, bad4=(1,))]
    lbda = LBDA6
    pos = np.array([[0.0, 20.0], [0.0, -10.0]])
    ref = psfrec.compute_psf_from_sparta_batch(tables, lbda=lbda, npsflin=2, field_positions=pos, ee_radii=[0.4],
                                               elliptical=True, verbose=False)
    got = psfrec.compute_psf_from_sparta_batch(tables, lbda=lbda, npsflin=2, field_positions=pos, ee_radii=[0.4],
                                               elliptical=True, verbose=False, ao_budget=True)
    ctx = own_context(psfrec, 128)
    try:
        for t, (g, r) in enumerate(zip(got, ref)):
            names = [h.name for h in r]
            assert [h.name for h in g] == names + ['AO_MEAN', 'AO_FIELD']
            for key in ('SEEING', 'GL', 'L0'):
                assert g['FIT_MEAN'].header[key] == r['FIT_MEAN'].header[key], key
            for name in names[2:]:
                a, b = g[name].data, r[name].data
                if a.dtype.names:
                    assert all(np.array_equal(a[c], b[c], equal_nan=True) for c in b.dtype.names), name
                else:
                    assert np.array_equal(a, b), name
            # the per-draw records of the same draws, averaged on the host in draw order
            vals = np.array([[[row['LGS%d_%s' % (k, c)] for c in ('SEEING', 'TUR_GND', 'L0')] for k in range(1, 5)]
                             for row in tables[t].data], dtype=float)
            seeing, GL, L0, three, _, _ = (np.array(c) for c in zip(*psfrec.select_sparta_rows(vals)))
            recs = psfrec._mode_records(three, seeing, GL, L0)
            dirs = psfrec.direction_perf(2)
            out = ao_outputs(len(recs), 1, 4, lbda.size)
            ctx.compute_ao(False, recs, dirs, psfrec._lgs_positions(False), lbda, **out)
            fld = ao_outputs(len(recs), 2, 2, lbda.size)
            ctx.compute_ao(True, recs, pos, psfrec._lgs_positions(False), lbda, **fld)
            m = g['AO_MEAN']
            assert np.array_equal(m.data['strehl'], psfrec._draw_mean(out['out_strehl'][:, 0]))
            vm = psfrec._draw_mean(out['out_var'].reshape(-1, _lib.VAR_NPAR))
            for col, slot in (('var_total', 0), ('var_fit', 1), ('var_noise', 2), ('var_proj', 3)):
                assert np.all(m.data[col] == vm[slot]), col
            assert m.header['SEEING'] == g['FIT_MEAN'].header['SEEING']
            f = g['AO_FIELD']
            sf, vf = psfrec._draw_mean(fld['out_strehl']), psfrec._draw_mean(fld['out_var'])
            assert np.array_equal(f.data['strehl'], sf.ravel())
            assert np.array_equal(f.data['var_noise'], np.repeat(vf[:, _lib.VAR_NOISE], lbda.size))
            assert np.array_equal(f.data['x'], np.repeat(pos[0], lbda.size))
    finally:
        ctx.close()
    bad = seeded_table(3, 2, invalid=(0, 1))
    assert psfrec.compute_psf_from_sparta(bad, lbda=lbda, verbose=False, ao_budget=True) is None
