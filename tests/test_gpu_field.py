"""GPU tests of the field-resolved reconstruction: ``psfr_compute_field``, ``Context.compute_field``,
``compute_psf_field`` and the FIT_FIELD / PSF_FIELD extensions of the SPARTA shell.

The PSF at field position k of draw d is the reference's ``psf_muse`` of that direction's PSD alone, then
``convolve_final_psf`` and the Moffat fit.  The library gives it bit for bit as a one-direction
``compute_batch`` of draw d at position k, so every per-position output is compared with such calls by
``np.array_equal``, and a few with the oracle to the tolerances of tests/test_gpu_parity.py.  The field
mean of ``compute_psf_batch(npsflin=n)`` is a different quantity and is not compared with these PSFs.
"""
import io

import numpy as np
import pytest
from numpy.testing import assert_allclose

import psfr_oracle as orc
from test_gpu_envelope import FIT_RTOL, assert_image_close
from test_gpu_sparta_batch import assert_same_result, config2_table, seeded_table

pytestmark = pytest.mark.gpu

LBDA6 = np.linspace(490, 930, 35)[::6]
# (0, 0), the four corners of the 3 x 3 grid, two positions off the grid
POS7 = np.array([[0., -30., 30., -30., 30., 12.5, 45.],
                 [0., -30., -30., 30., 30., -7.3, 0.]])
GRID3 = np.array([[-30., -30., -30., 0., 0., 0., 30., 30., 30.],
                  [-30., 0., 30., -30., 0., 30., -30., 0., 30.]])     # direction_perf(3)


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


def draws5():
    """5 draws, draws 1 and 3 in three-lasers mode, one (h0, h1) pair per draw."""
    rng = np.random.default_rng(5)
    seeing, GL, L0 = rng.uniform(0.5, 1.8, 5), rng.uniform(0.35, 0.9, 5), rng.uniform(10, 28, 5)
    three = np.array([False, True, False, True, False])
    h = np.stack([rng.uniform(50, 500, 5), rng.uniform(5000, 15000, 5)], axis=1)
    return seeing, GL, L0, three, h


def one_direction_reference(ctx, psfrec, recs, three, pos, lam):
    """compute_batch of each draw at each position alone (its own laser table, dirs = [2, 1])."""
    from muse_psfr_b200 import _lib
    nd, npos, nl = len(recs), pos.shape[1], lam.size
    cube, fit = np.empty((nd, npos, nl, 40, 40)), np.empty((nd, npos, nl, _lib.FIT_NPAR))
    for d in range(nd):
        for k in range(npos):
            ctx.compute_batch(recs[[d]], np.ascontiguousarray(pos[:, [k]]), psfrec._lgs_positions(bool(three[d])),
                              lam, out_cube=cube[d, k], out_fit=fit[d, k])
    return cube, fit


def own_context(psfrec, max_planes, dim=1280):
    from muse_psfr_b200 import _lib
    ctx = _lib.Context(device=0, dim=dim, max_planes=max_planes, max_lambda=35)
    ctx.set_geometry(*psfrec.ao_frequency_tables())
    return ctx


# ---------------------------------------------------------------- 1. every position = its own one-direction call
@pytest.fixture(scope='module')
def reference7(psfrec):
    seeing, GL, L0, three, h = draws5()
    recs = psfrec._mode_records(three, seeing, GL, L0, h)
    ctx = own_context(psfrec, 16)
    try:
        return one_direction_reference(ctx, psfrec, recs, three, POS7, LBDA6)
    finally:
        ctx.close()


@pytest.mark.parametrize('max_planes', [7, 10, 128])
def test_each_position_matches_one_direction_call(psfrec, reference7, max_planes):
    """7 positions: at 7 planes one draw per chunk, at 10 one draw per chunk with 3 planes unused, at 128
    all 5 draws in one chunk."""
    seeing, GL, L0, three, h = draws5()
    psfrec.release_contexts()
    fit, cube = psfrec.compute_psf_field(LBDA6, seeing, GL, L0, positions=POS7, h=h, three_lgs_mode=three,
                                         max_planes=max_planes)
    assert psfrec.get_context().info()['max_planes'] == min(max_planes, 35)
    assert cube.shape == (5, 7, LBDA6.size, 40, 40) and fit.shape == (5, 7, LBDA6.size, 16)
    ref_cube, ref_fit = reference7
    for d in range(5):
        for k in range(7):
            assert np.array_equal(cube[d, k], ref_cube[d, k]), (d, k)
            assert np.array_equal(fit[d, k], ref_fit[d, k]), (d, k)
    # the positions differ from each other: a field pass that averaged or repeated planes would not pass
    assert not np.array_equal(cube[:, 0], cube[:, 6])
    psfrec.release_contexts()


# ---------------------------------------------------------------- 2. on axis = compute_psf_batch(npsflin=1)
@pytest.mark.parametrize('mode', ['four', 'three', 'per_draw'])
def test_on_axis_equals_compute_psf_batch(psfrec, mode):
    seeing, GL, L0, three, _ = draws5()
    flag = {'four': False, 'three': True, 'per_draw': three}[mode]
    fit_b, cube_b = psfrec.compute_psf_batch(LBDA6, seeing, GL, L0, npsflin=1, three_lgs_mode=flag)
    fit, cube = psfrec.compute_psf_field(LBDA6, seeing, GL, L0, positions=[[0], [0]], three_lgs_mode=flag)
    assert cube.shape == (5, 1, LBDA6.size, 40, 40)
    assert np.array_equal(cube[:, 0], cube_b) and np.array_equal(fit[:, 0], fit_b)
    # the default positions are the 3 x 3 grid of direction_perf
    fit9, _ = psfrec.compute_psf_field(LBDA6, seeing[:1], GL[:1], L0[:1], three_lgs_mode=flag if mode != 'per_draw'
                                       else three[:1], want_cube=False)
    assert fit9.shape == (1, 9, LBDA6.size, 16)
    assert np.array_equal(fit9[0, 4], fit[0, 0])          # position 4 of the grid is (0, 0)


# ---------------------------------------------------------------- 3. oracle parity
def oracle_field(lam, seeing, GL, L0, three, pos, dim=1280, h=(100, 10000)):
    """The reference's pipeline for one draw, one PSD per field position (simul_psd_wfm with
    dir_arcsec = pos, psf_muse of one plane, convolve_final_psf, Moffat fit)."""
    Cn2 = np.array([GL, 1 - GL])
    Cn2 = Cn2 / Cn2.sum()
    r0ref = orc.seeing2r01(seeing, orc.LAMBDA_REF_UM, 0.)
    fc = 1 / (2 * (orc.D_PUP / orc.N_ACT))
    ao = orc.dsp4muse(Cn2, np.array(h, dtype=float), L0, r0ref, orc.lgs_positions(three), pos,
                      vent=orc.wind_speed_for(h))
    fit = orc.psd_fit(dim, 2 * orc.D_PUP, r0ref, L0, fc)
    sl = slice(dim // 2 - orc.DIM_PUP, dim // 2 + orc.DIM_PUP)
    out = []
    for k in range(pos.shape[1]):
        psd = fit.copy()
        psd[sl, sl] = np.maximum(fit[sl, sl], np.fft.fftshift(ao[k]))
        psd *= (orc.LAMBDA_REF_UM * 1000 / (2 * np.pi)) ** 2
        psf = orc.convolve_final_psf(lam, seeing, GL, L0, orc.psf_muse(psd, lam))
        out.append((orc.fit_psf_cube(lam, psf), psf))
    return out


def assert_matches_oracle(fit, cube, ref):
    from muse_psfr_b200 import _lib
    for k, (rfit, rpsf) in enumerate(ref):
        for j in range(rpsf.shape[0]):
            assert_image_close(cube[k, j], rpsf[j])
        assert_allclose(fit[k, :, _lib.FIT_FWHM] * 0.2, rfit['fwhm'], rtol=FIT_RTOL)
        assert_allclose(fit[k, :, _lib.FIT_N], rfit['n'], rtol=FIT_RTOL)


def test_oracle_parity_off_axis(psfrec):
    pos = np.array([[12.5, -30., 45.], [-7.3, 30., 0.]])
    lam = np.array([490., 710., 930.])
    seeing, GL, L0, three = np.array([0.8, 1.3]), np.array([0.7, 0.45]), np.array([22., 14.]), np.array([False, True])
    fit, cube = psfrec.compute_psf_field(lam, seeing, GL, L0, positions=pos, three_lgs_mode=three)
    for d in range(2):
        assert_matches_oracle(fit[d], cube[d], oracle_field(lam, seeing[d], GL[d], L0[d], three[d], pos))


def test_oracle_parity_dim2560(psfrec):
    pos = np.array([[12.5, -30.], [-7.3, 30.]])
    lam = np.array([600.])
    fit, cube = psfrec.compute_psf_field(lam, [1.1], [0.6], [18.], positions=pos, dim=2560)
    assert_matches_oracle(fit[0], cube[0], oracle_field(lam, 1.1, 0.6, 18., False, pos, dim=2560))
    psfrec.release_contexts()


# ---------------------------------------------------------------- 4. per-position exposure means
GROUPS3 = np.array([4, 5, 11], dtype=np.int32)       # exposures of 4, 1 and 6 draws


def group_inputs(psfrec):
    rng = np.random.default_rng(3)
    n = int(GROUPS3[-1])
    seeing, GL, L0 = rng.uniform(0.5, 1.8, n), rng.uniform(0.35, 0.9, n), rng.uniform(10, 28, n)
    three = rng.random(n) < 0.4
    return psfrec._mode_records(three, seeing, GL, L0), psfrec._lgs_positions(False)


def field_outputs(recs, npos, nl, ngroup):
    from muse_psfr_b200 import _lib
    nd = len(recs)
    return dict(out_cube=np.full((nd, npos, nl, 40, 40), np.nan), out_fit=np.full((nd, npos, nl, _lib.FIT_NPAR), np.nan),
                out_mean=np.full((ngroup, npos, nl, 40, 40), np.nan),
                out_mean_fit=np.full((ngroup, npos, nl, _lib.FIT_NPAR), np.nan))


@pytest.mark.parametrize('npos', [2, 3])
def test_position_means_match_mean_refit(psfrec, npos):
    """At 3 planes per chunk every draw is a chunk of its own; at 8, chunks of 4 (npos 2) or 2 (npos 3)
    draws, so the exposures of 4 and 6 draws span chunk edges; at 128 everything is one chunk."""
    recs, lgs = group_inputs(psfrec)
    pos = np.ascontiguousarray(POS7[:, [1, 5, 6][:npos]])
    nl = LBDA6.size
    first = None
    for max_planes in (3, 8, 128):
        ctx = own_context(psfrec, max_planes)
        try:
            out = field_outputs(recs, npos, nl, len(GROUPS3))
            ctx.compute_field(recs, pos, lgs, LBDA6, GROUPS3, **out)
            for g, (a, b) in enumerate(zip(np.r_[0, GROUPS3[:-1]], GROUPS3)):
                for k in range(npos):
                    mean, mfit = np.empty((nl, 40, 40)), np.empty((nl, 16))
                    ctx.mean_refit(int(b - a), nl, np.ascontiguousarray(out['out_cube'][a:b, k]), mean, mfit)
                    assert np.array_equal(out['out_mean'][g, k], mean), (max_planes, g, k)
                    assert np.array_equal(out['out_mean_fit'][g, k], mfit), (max_planes, g, k)
        finally:
            ctx.close()
        if first is None:
            first = out
        for name in out:      # the chunking changes no bit of any output
            assert np.array_equal(out[name], first[name]), (max_planes, name)


# ---------------------------------------------------------------- 5. output buffers
def test_device_outputs_and_partial_calls(psfrec):
    import torch
    recs, lgs = group_inputs(psfrec)
    pos = np.ascontiguousarray(POS7[:, :3])
    nl = LBDA6.size
    ctx = own_context(psfrec, 8)
    try:
        full = field_outputs(recs, 3, nl, len(GROUPS3))
        ctx.compute_field(recs, pos, lgs, LBDA6, GROUPS3, **full)
        dev = {n: torch.full(a.shape, np.nan, dtype=torch.float64, device='cuda') for n, a in full.items()}
        ctx.compute_field(recs, pos, lgs, LBDA6, GROUPS3, **dev)
        torch.cuda.synchronize()
        for n, a in full.items():
            assert np.array_equal(dev[n].cpu().numpy(), a), n
        for keep in (('out_cube',), ('out_fit',), ('out_mean', 'out_mean_fit'), ('out_mean',), ('out_mean_fit',)):
            part = {n: np.full(full[n].shape, np.nan) for n in keep}
            ctx.compute_field(recs, pos, lgs, LBDA6, GROUPS3, **part)
            for n in keep:
                assert np.array_equal(part[n], full[n]), (keep, n)
        # mixed: device cube, host means
        mixed = {'out_cube': torch.full(full['out_cube'].shape, np.nan, dtype=torch.float64, device='cuda'),
                 'out_mean_fit': np.full(full['out_mean_fit'].shape, np.nan)}
        ctx.compute_field(recs, pos, lgs, LBDA6, GROUPS3, **mixed)
        torch.cuda.synchronize()
        assert np.array_equal(mixed['out_cube'].cpu().numpy(), full['out_cube'])
        assert np.array_equal(mixed['out_mean_fit'], full['out_mean_fit'])
        # the per-exposure path is unchanged after a field call on the same context
        cube, mean = np.empty((len(recs), nl, 40, 40)), np.empty((3, nl, 40, 40))
        ctx.compute_groups(recs, pos, lgs, LBDA6, GROUPS3, out_cube=cube, out_mean=mean)
        ref = np.empty_like(cube)
        ctx.compute_groups(recs, pos, lgs, LBDA6, None, out_cube=ref)
        assert np.array_equal(cube, ref)
    finally:
        ctx.close()


# ---------------------------------------------------------------- 6. refusals of the C ABI
def test_compute_field_refusals(psfrec):
    from muse_psfr_b200 import _lib
    recs, lgs = group_inputs(psfrec)
    pos = np.ascontiguousarray(POS7[:, :3])
    nl = LBDA6.size
    SENT = 12345.0
    ctx = own_context(psfrec, 8)
    outs = {n: np.full(a.shape, SENT) for n, a in field_outputs(recs, 3, nl, len(GROUPS3)).items()}

    def untouched():
        for n, a in outs.items():
            assert np.all(a == SENT), n

    def refused(code, group_end=GROUPS3, dirs=pos, **kw):
        with pytest.raises(_lib.PsfrError) as exc:
            ctx.compute_field(recs, dirs, lgs, LBDA6, group_end, **{**outs, **kw})
        assert exc.value.code == code, str(exc.value)
        untouched()
    def raw(ndir, dirs):
        """The C entry point itself, past the binding's buffer-size checks."""
        rc = ctx._lib.psfr_compute_field(ctx._handle(), len(recs), _lib.ptr(recs), 4,
                                         _lib.ptr(np.ascontiguousarray(lgs)), ndir, dirs, nl,
                                         _lib.ptr(np.ascontiguousarray(LBDA6)), 3, GROUPS3.ctypes.data,
                                         *[_lib.ptr(outs[n]) for n in ('out_cube', 'out_fit', 'out_mean',
                                                                      'out_mean_fit')], None)
        untouched()
        return rc
    try:
        assert raw(3, None) == _lib.E_ARG
        assert raw(9, _lib.ptr(GRID3)) == _lib.E_CAPACITY           # 9 positions > 8 planes per chunk
        for ge in ([4, 4, 11], [5, 4, 11], [4, 5, 10], [4, 5, 12]):
            refused(_lib.E_ARG, group_end=np.array(ge, dtype=np.int32))
        refused(_lib.E_ARG, group_end=None)                         # means without exposures
        refused(_lib.E_ARG, group_end=None, out_mean=None)
        # the context still works
        ctx.compute_field(recs, pos, lgs, LBDA6, GROUPS3, out_fit=outs['out_fit'])
        assert np.all(outs['out_fit'][..., _lib.FIT_ITER] > 0)
    finally:
        ctx.close()


# ---------------------------------------------------------------- 7. the SPARTA shell
def field_restatement(psfrec, tbl, lbda, positions):
    """FIT_FIELD columns and PSF_FIELD of one table: compute_psf_field over its valid rows, then
    mean_refit per position."""
    from muse_psfr_b200 import _lib
    data = tbl.data
    values = np.array([[[row['LGS%d_%s' % (k, c)] for c in ('SEEING', 'TUR_GND', 'L0')] for k in range(1, 5)]
                       for row in data], dtype=float).reshape(len(data), 4, 3)
    jobs = psfrec.select_sparta_rows(values)
    seeing, GL, L0, three = (np.array(c) for c in list(zip(*jobs))[:4])
    _, cube = psfrec.compute_psf_field(lbda, seeing, GL, L0, positions=positions, three_lgs_mode=three)
    npos, nl = positions.shape[1], lbda.size
    ctx = psfrec.get_context()
    psf = np.empty((npos, nl, 40, 40))
    fit = np.empty((npos, nl, _lib.FIT_NPAR))
    for k in range(npos):
        ctx.mean_refit(len(seeing), nl, np.ascontiguousarray(cube[:, k]), psf[k], fit[k])
    cols = psfrec._fit_columns(lbda, fit)
    cols['x'] = np.repeat(positions[0], nl)
    cols['y'] = np.repeat(positions[1], nl)
    return cols, psf


def assert_field_hdus(hdul, cols, psf, mean_header):
    tab = hdul['FIT_FIELD'].data
    assert list(tab.dtype.names) == list(cols)
    for name, ref in cols.items():
        assert np.array_equal(tab[name], ref, equal_nan=np.asarray(ref).dtype.kind == 'f'), name
    assert np.array_equal(hdul['PSF_FIELD'].data, psf)
    for key in ('SEEING', 'GL', 'L0'):
        assert hdul['FIT_FIELD'].header[key] == mean_header[key], key


def test_sparta_field_positions(psfrec):
    from muse_psfr_b200 import _fits
    tbl, empty = config2_table(), seeded_table(3, 4, invalid=range(4))
    plain = psfrec.compute_psf_from_sparta_batch([tbl, empty], lbda=LBDA6, verbose=False)
    none = psfrec.compute_psf_from_sparta_batch([tbl, empty], lbda=LBDA6, verbose=False, field_positions=None)
    assert_same_result(none[0], plain[0])
    assert none[1] is None
    assert [h.name for h in none[0]] == ['PRIMARY', 'SPARTA_ATM_DATA', 'FIT_ROWS', 'FIT_MEAN', 'PSF_MEAN']
    got = psfrec.compute_psf_from_sparta_batch([tbl, empty], lbda=LBDA6, verbose=False, field_positions=GRID3)
    assert got[1] is None
    got = got[0]
    assert [h.name for h in got] == ['PRIMARY', 'SPARTA_ATM_DATA', 'FIT_ROWS', 'FIT_MEAN', 'PSF_MEAN', 'FIT_FIELD',
                                     'PSF_FIELD']
    assert_same_result(_fits.HDUList(list(got)[:5]), plain[0])
    cols, psf = field_restatement(psfrec, tbl, LBDA6, GRID3)
    assert psf.shape == (9, LBDA6.size, 40, 40)
    assert_field_hdus(got, cols, psf, got['FIT_MEAN'].header)
    buf = io.BytesIO()
    got.writeto(buf)
    back = _fits.open(buf.getvalue())
    assert_field_hdus(back, cols, psf, got['FIT_MEAN'].header)
    # the single-table call passes the positions on
    one = psfrec.compute_psf_from_sparta(tbl, lbda=LBDA6, verbose=False, field_positions=GRID3)
    assert_field_hdus(one, cols, psf, got['FIT_MEAN'].header)
