"""GPU tests of the band images (DESIGN.md section 5.6): ``psfr_compute_bands`` and ``psfr_band_psf``, their Python
surface (``bands=`` on ``compute_psf_batch`` / ``compute_psf_field``, ``band_psf``) and the BAND_MEAN / PSF_BAND
(/ _FIELD) HDUs of the SPARTA shell.

Known answers (one-hot weights give the planes, power-of-two scales leave the bits), the numpy restatement of
tests/band_oracle.py, the band fits and EE against the standalone entry points, the bits across chunk sizes, entry
points and host / device outputs, every other output against psfr_compute_ao bit for bit, and the refusals."""
import numpy as np
import pytest

import band_oracle as bo
from test_gpu_field import GRID3, GROUPS3, LBDA6, POS7, group_inputs, own_context
from test_gpu_sparta_batch import config2_table, seeded_table

pytestmark = pytest.mark.gpu

RAD, FR = np.array([1.0, 3.5]), np.array([0.5, 0.8])
REC = RAD.size + 1 + FR.size


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


def launches(ctx, fn, *args, **kw):
    n0 = ctx.kernel_launches()
    fn(*args, **kw)
    return ctx.kernel_launches() - n0


def random_weights(rng, nband, nl):
    """Non-negative weights with a few exact zeros, every band with a positive sum."""
    w = rng.random((nband, nl)) * (rng.random((nband, nl)) > 0.2)
    w[:, rng.integers(nl)] += 0.5
    return w


def plain_outputs(nd, P, ndir, nl, ng, rec=REC):
    from muse_psfr_b200 import _lib
    nan = lambda *shape: np.full(shape, np.nan)   # noqa: E731
    return dict(out_cube=nan(nd, P, nl, 40, 40), out_fit=nan(nd, P, nl, _lib.FIT_NPAR), out_mean=nan(ng, P, nl, 40, 40),
                out_mean_fit=nan(ng, P, nl, _lib.FIT_NPAR), out_efit=nan(nd, P, nl, _lib.EFIT_NPAR),
                out_mean_efit=nan(ng, P, nl, _lib.EFIT_NPAR), out_ee=nan(nd, P, nl, rec),
                out_mean_ee=nan(ng, P, nl, rec), out_strehl=nan(nd, P, nl), out_var=nan(nd, ndir, _lib.VAR_NPAR))


def band_outputs(nd, P, nb, ng, rec=REC, dev=False):
    from muse_psfr_b200 import _lib
    if dev:
        import torch
        nan = lambda *shape: torch.full(shape, float('nan'), dtype=torch.float64, device='cuda')   # noqa: E731
    else:
        nan = lambda *shape: np.full(shape, np.nan)   # noqa: E731
    return dict(out_band=nan(nd, P, nb, 40, 40), out_band_fit=nan(nd, P, nb, _lib.FIT_NPAR),
                out_band_ee=nan(nd, P, nb, rec), out_mean_band=nan(ng, P, nb, 40, 40),
                out_mean_band_fit=nan(ng, P, nb, _lib.FIT_NPAR), out_mean_band_ee=nan(ng, P, nb, rec))


def host(out):
    import torch
    torch.cuda.synchronize()
    return {k: (v.cpu().numpy() if hasattr(v, 'cpu') else v) for k, v in out.items()}


def field_args(field):
    pos = np.ascontiguousarray(POS7[:, [0, 5, 6]] if field else GRID3[:, [0, 4, 8]])
    return pos, (pos.shape[1] if field else 1)


# ---------------------------------------------------------------- 1. known answers
@pytest.mark.parametrize('field', [False, True])
def test_one_hot_weights_give_the_planes(psfrec, field):
    recs, lgs = group_inputs(psfrec)
    pos, P = field_args(field)
    nd, nl, ng = len(recs), LBDA6.size, len(GROUPS3)
    ctx = own_context(psfrec, 8)
    try:
        out = plain_outputs(nd, P, pos.shape[1], nl, ng)
        band = band_outputs(nd, P, nl, ng)
        ctx.compute_bands(field, recs, pos, lgs, LBDA6, np.eye(nl), RAD, FR, GROUPS3, **out, **band)
        for k in range(nl):
            assert np.array_equal(band['out_band'][:, :, k], out['out_cube'][:, :, k]), k
            assert np.array_equal(band['out_band_fit'][:, :, k], out['out_fit'][:, :, k]), k
            assert np.array_equal(band['out_band_ee'][:, :, k], out['out_ee'][:, :, k]), k
            assert np.array_equal(band['out_mean_band'][:, :, k], out['out_mean'][:, :, k]), k
            assert np.array_equal(band['out_mean_band_fit'][:, :, k], out['out_mean_fit'][:, :, k]), k
            assert np.array_equal(band['out_mean_band_ee'][:, :, k], out['out_mean_ee'][:, :, k]), k
        # one band picking plane 4 only (a power of two divides out exactly), the others a mix
        w = np.zeros((3, nl))
        w[0, 4] = 4.0
        w[1:] = 1.0
        one = band_outputs(nd, P, 3, ng)
        ctx.compute_bands(field, recs, pos, lgs, LBDA6, w, RAD, FR, GROUPS3, **one)
        assert np.array_equal(one['out_band'][:, :, 0], out['out_cube'][:, :, 4])
        assert np.array_equal(one['out_mean_band_fit'][:, :, 0], out['out_mean_fit'][:, :, 4])
    finally:
        ctx.close()


def test_power_of_two_scaling_keeps_the_bits(psfrec):
    recs, lgs = group_inputs(psfrec)
    nd, nl, ng = len(recs), LBDA6.size, len(GROUPS3)
    w = random_weights(np.random.default_rng(8), 3, nl)
    ctx = own_context(psfrec, 16)
    try:
        first = None
        for e in (-40, -7, 0, 13, 40):
            band = band_outputs(nd, 1, 3, ng)
            ctx.compute_bands(False, recs, GRID3[:, :2].copy(), lgs, LBDA6, w * 2.0 ** e, RAD, FR, GROUPS3, **band)
            got = {k: v.view(np.int64) for k, v in band.items()}
            if first is None:
                first = got
            else:
                assert all(np.array_equal(got[k], first[k]) for k in got), e
    finally:
        ctx.close()


def test_equal_weights_give_the_plane_mean(psfrec):
    lam = np.linspace(490, 930, 35)
    fit, cube, bfit, bcube = psfrec.compute_psf_batch(lam, [0.7, 1.5], [0.7, 0.4], [25.0, 12.0], bands=np.ones(35))
    for d in range(2):
        ref = bo.band_images(cube[d], np.ones(35))[0]
        assert np.max(np.abs(bcube[d, 0] - ref)) <= 1e-13 * ref.max()
        assert np.max(np.abs(bcube[d, 0] - cube[d].mean(axis=0))) <= 1e-13 * ref.max()


# ---------------------------------------------------------------- 2. against the restatement
def assert_bands_close(bands, cubes, w):
    ref = bo.band_sets(cubes, w)
    assert bands.shape == ref.shape
    peak = np.abs(ref).max(axis=(-2, -1), keepdims=True)
    assert np.all(np.abs(bands - ref) <= 1e-13 * peak)


ORACLE_CASES = [
    dict(mode='batch', nband=3, nl=35),
    dict(mode='batch', nband=1, nl=1, three=True),
    dict(mode='batch', nband=16, nl=100, npsflin=3, three=[False, True]),
    dict(mode='field', nband=16, nl=35),
    dict(mode='field', nband=3, nl=100, three=[True, False]),
    dict(mode='field', nband=1, nl=35, three=True),
    dict(mode='batch', nband=3, nl=35, dim=2560),
]


@pytest.mark.parametrize('case', range(len(ORACLE_CASES)))
def test_against_restatement(psfrec, case):
    c = ORACLE_CASES[case]
    rng = np.random.default_rng(100 + case)
    lam = np.array([700.0]) if c['nl'] == 1 else np.linspace(490, 930, c['nl'])
    w = random_weights(rng, c['nband'], c['nl'])
    seeing, GL, L0 = [0.6, 1.4], [0.75, 0.5], [18.0, 27.0]
    kw = dict(three_lgs_mode=c.get('three', False), dim=c.get('dim', 1280), bands=w, ee_radii=[0.3])
    if c['mode'] == 'batch':
        fit, cube, ee, bfit, bcube, bee = psfrec.compute_psf_batch(lam, seeing, GL, L0, npsflin=c.get('npsflin', 1),
                                                                   **kw)
        assert bcube.shape == (2, c['nband'], 40, 40)
    else:
        fit, cube, ee, bfit, bcube, bee = psfrec.compute_psf_field(lam, seeing, GL, L0, positions=POS7[:, :3], **kw)
        assert bcube.shape == (2, 3, c['nband'], 40, 40)
    assert_bands_close(bcube, cube, w)
    assert np.all(np.isfinite(bfit)) and np.all(np.isfinite(bee))


# ---------------------------------------------------------------- 3. self-consistency
@pytest.mark.parametrize('field', [False, True])
def test_band_fit_ee_and_means_against_standalone(psfrec, field):
    recs, lgs = group_inputs(psfrec)
    pos, P = field_args(field)
    nd, nl, ng = len(recs), LBDA6.size, len(GROUPS3)
    w = random_weights(np.random.default_rng(9), 4, nl)
    ctx = own_context(psfrec, 8)
    try:
        out = plain_outputs(nd, P, pos.shape[1], nl, ng)
        band = band_outputs(nd, P, 4, ng)
        ctx.compute_bands(field, recs, pos, lgs, LBDA6, w, RAD, FR, GROUPS3, **out, **band)
        for img, fit, ee in (('out_band', 'out_band_fit', 'out_band_ee'),
                             ('out_mean_band', 'out_mean_band_fit', 'out_mean_band_ee')):
            n = band[img].size // 1600
            f, e = np.empty_like(band[fit]), np.empty_like(band[ee])
            ctx.moffat_fit(n, 40, 40, band[img], f)
            ctx.encircled_energy(n, 40, 40, band[img], RAD, FR, e)
            assert np.array_equal(f, band[fit]) and np.array_equal(e, band[ee]), img
        mb = np.empty_like(band['out_mean_band'])
        ctx.band_psf(ng * P, nl, 40, 40, out['out_mean'], w, mb)
        assert np.array_equal(mb, band['out_mean_band'])
        db = np.empty_like(band['out_band'])
        ctx.band_psf(nd * P, nl, 40, 40, out['out_cube'], w, db)
        assert np.array_equal(db, band['out_band'])
        assert_bands_close(band['out_band'], out['out_cube'], w)
        assert_bands_close(band['out_mean_band'], out['out_mean'], w)
    finally:
        ctx.close()


@pytest.mark.parametrize('shape', [(40, 40), (13, 29), (1, 1), (48, 50)])
def test_standalone_band_psf_host_and_device(psfrec, shape):
    import torch
    rng = np.random.default_rng(sum(shape))
    ny, nx = shape
    n, nl = 21, 35
    cubes = rng.normal(size=(n, nl, ny, nx))
    w = random_weights(rng, 5, nl)
    ctx = own_context(psfrec, 2)    # staging of 2 x 35 planes of 40 x 40: host arrays go through in chunks
    try:
        got = np.full((n, 5, ny, nx), np.nan)
        ctx.band_psf(n, nl, ny, nx, cubes, w, got)
        dev_in = torch.from_numpy(cubes).cuda()
        dev_out = torch.full((n, 5, ny, nx), float('nan'), dtype=torch.float64, device='cuda')
        ctx.band_psf(n, nl, ny, nx, dev_in, w, dev_out)
        mixed = np.full((n, 5, ny, nx), np.nan)
        ctx.band_psf(n, nl, ny, nx, dev_in, w, mixed)
        dev_out2 = torch.full((n, 5, ny, nx), float('nan'), dtype=torch.float64, device='cuda')
        ctx.band_psf(n, nl, ny, nx, cubes, w, dev_out2)
        torch.cuda.synchronize()
        for other in (dev_out.cpu().numpy(), mixed, dev_out2.cpu().numpy()):
            assert np.array_equal(other, got)
        assert_bands_close(got, cubes, w)
    finally:
        ctx.close()
    # the Python surface: one cube or a stack of cubes
    one = psfrec.band_psf(cubes[3], w)
    assert one.shape == (5, ny, nx) and np.array_equal(one, got[3])
    assert np.array_equal(psfrec.band_psf(cubes[:4], w[1]), got[:4, 1:2])


# ---------------------------------------------------------------- 4. invariance and nothing else moves
@pytest.mark.parametrize('field', [False, True])
def test_bits_across_chunks_and_outputs(psfrec, field):
    recs, lgs = group_inputs(psfrec)
    pos, P = field_args(field)
    nd, nl, ng = len(recs), LBDA6.size, len(GROUPS3)
    w = random_weights(np.random.default_rng(10), 3, nl)
    first = None
    for max_planes in (3, 8, 128):       # 1, 2 and 11 draws per chunk with 3 positions: exposures straddle edges
        ctx = own_context(psfrec, max_planes)
        try:
            out = plain_outputs(nd, P, pos.shape[1], nl, ng)
            ctx.compute_groups(recs, pos, lgs, LBDA6, GROUPS3, out_fit=np.empty((nd, nl, 16)))  # kernels built once
            n_ao = launches(ctx, ctx.compute_ao, field, recs, pos, lgs, LBDA6, RAD, FR, GROUPS3, **out)
            same = {k: np.full(v.shape, np.nan) for k, v in out.items()}
            # nband = 0 and no band output: psfr_compute_ao, launch for launch
            assert launches(ctx, ctx.compute_bands, field, recs, pos, lgs, LBDA6, None, RAD, FR, GROUPS3,
                            **same) == n_ao
            assert all(np.array_equal(same[k], out[k], equal_nan=True) for k in out)
            both = {k: np.full(v.shape, np.nan) for k, v in out.items()}
            band = band_outputs(nd, P, 3, ng)
            assert launches(ctx, ctx.compute_bands, field, recs, pos, lgs, LBDA6, w, RAD, FR, GROUPS3, **both,
                            **band) > n_ao
            for k in out:      # every other output keeps its bits
                assert np.array_equal(both[k], out[k], equal_nan=True), (max_planes, k)
            dev = band_outputs(nd, P, 3, ng, dev=True)
            ctx.compute_bands(field, recs, pos, lgs, LBDA6, w, RAD, FR, GROUPS3, **dev)
            dev = host(dev)
            # each band output alone, and a host / device mix
            alone = {}
            for k in band:
                one = band_outputs(nd, P, 3, ng)[k]
                ctx.compute_bands(field, recs, pos, lgs, LBDA6, w, RAD, FR, GROUPS3, **{k: one})
                alone[k] = one
            mix = band_outputs(nd, P, 3, ng)
            mix.update({k: v for k, v in band_outputs(nd, P, 3, ng, dev=True).items() if 'fit' in k})
            ctx.compute_bands(field, recs, pos, lgs, LBDA6, w, RAD, FR, GROUPS3, out_cube=out['out_cube'], **mix)
            mix = host(mix)
        finally:
            ctx.close()
        for k in band:
            assert not np.any(np.isnan(band[k])), k
            for other in (dev, alone, mix):
                assert np.array_equal(other[k], band[k]), (max_planes, k)
        if first is None:
            first = band
        else:
            assert all(np.array_equal(band[k], first[k]) for k in band), max_planes


def test_python_results_unchanged_and_field_on_axis(psfrec):
    seeing, GL, L0 = [0.9, 1.4, 0.6], [0.7, 0.5, 0.8], [25.0, 14.0, 20.0]
    w = random_weights(np.random.default_rng(12), 2, LBDA6.size)
    for three in (False, True, [False, True, False]):
        ref = psfrec.compute_psf_batch(LBDA6, seeing, GL, L0, npsflin=2, three_lgs_mode=three, ee_radii=[0.3],
                                       ao_budget=True)
        got = psfrec.compute_psf_batch(LBDA6, seeing, GL, L0, npsflin=2, three_lgs_mode=three, ee_radii=[0.3],
                                       ao_budget=True, bands=w)
        assert len(got) == len(ref) + 3 and all(np.array_equal(a, b) for a, b in zip(got, ref))
        plain = psfrec.compute_psf_batch(LBDA6, seeing, GL, L0, three_lgs_mode=three)
        got = psfrec.compute_psf_batch(LBDA6, seeing, GL, L0, three_lgs_mode=three, bands=w, want_cube=False)
        assert np.array_equal(got[0], plain[0]) and got[1] is None and len(got) == 4
        assert got[3].shape == (3, 2, 40, 40)
        field = psfrec.compute_psf_field(LBDA6, seeing, GL, L0, positions=[[0.0], [0.0]], three_lgs_mode=three,
                                         bands=w)
        assert all(np.array_equal(a[:, 0], b) for a, b in zip(field, (plain[0], plain[1], got[2], got[3])))
    ref = psfrec.compute_psf_field(LBDA6, seeing, GL, L0, positions=POS7, elliptical=True, ee_radii=[0.5])
    got = psfrec.compute_psf_field(LBDA6, seeing, GL, L0, positions=POS7, elliptical=True, ee_radii=[0.5], bands=w)
    assert len(got) == 7 and all(np.array_equal(a, b) for a, b in zip(got, ref))
    assert got[4].shape == (3, 7, 2, 16) and got[6].shape == (3, 7, 2, 4)


# ---------------------------------------------------------------- 5. refusals
class _NullWeights:
    """The library with the weights argument of psfr_compute_bands replaced by NULL."""

    def __init__(self, lib):
        self._l = lib

    def __getattr__(self, name):
        fn = getattr(self._l, name)
        if name != 'psfr_compute_bands':
            return fn

        def call(*args):
            args = list(args)
            args[27] = None
            return fn(*args)
        return call


def test_refusals_leave_the_outputs_untouched(psfrec):
    from muse_psfr_b200 import _lib
    recs, lgs = group_inputs(psfrec)
    pos, P = field_args(True)
    nd, nl, ng = len(recs), LBDA6.size, len(GROUPS3)
    ok = np.ones((2, nl))
    bad = {'too_many': np.ones((17, nl)), 'none': None, 'negative': np.where(np.eye(2, nl) > 0, -1.0, 1.0),
           'nan': np.where(np.eye(2, nl) > 0, np.nan, 1.0), 'inf': np.where(np.eye(2, nl) > 0, np.inf, 1.0),
           'zero_sum': np.stack([np.ones(nl), np.zeros(nl)]), 'inf_sum': np.full((2, nl), 1e308),
           'null_weights': ok}
    ctx = own_context(psfrec, 8)
    n0 = ctx.kernel_launches()
    try:
        for name, w in bad.items():
            out = plain_outputs(nd, P, pos.shape[1], nl, ng)
            nb = 17 if name == 'too_many' else 2
            band = band_outputs(nd, P, nb, ng)
            lib = ctx._lib
            if name == 'null_weights':
                ctx._lib = _NullWeights(lib)
            try:
                with pytest.raises(_lib.PsfrError) as exc:
                    ctx.compute_bands(True, recs, pos, lgs, LBDA6, w, RAD, FR, GROUPS3, **out, **band)
            finally:
                ctx._lib = lib
            assert exc.value.code == _lib.E_ARG, name
            assert all(np.all(np.isnan(v)) for v in list(out.values()) + list(band.values())), name
            if name not in ('none', 'null_weights'):
                img = np.full((3, nb, 40, 40), np.nan)
                with pytest.raises(_lib.PsfrError) as exc:
                    ctx.band_psf(3, nl, 40, 40, np.ones((3, nl, 40, 40)), w, img)
                assert exc.value.code == _lib.E_ARG and np.all(np.isnan(img)), name
        assert ctx.kernel_launches() == n0
        # weights with nband = 0 while a band output is set, and more wavelengths than the context holds
        with pytest.raises(_lib.PsfrError) as exc:
            ctx.compute_bands(True, recs, pos, lgs, LBDA6, None, group_end=GROUPS3,
                              out_band=np.empty((nd, P, 1, 40, 40)))
        assert exc.value.code == _lib.E_ARG
        with pytest.raises(_lib.PsfrError) as exc:
            ctx.band_psf(1, 36, 40, 40, np.ones((1, 36, 40, 40)), np.ones(36), np.empty((1, 1, 40, 40)))
        assert exc.value.code == _lib.E_CAPACITY
        assert ctx.kernel_launches() == n0
    finally:
        ctx.close()


# ---------------------------------------------------------------- 6. SPARTA shell
def test_sparta_band_hdus(psfrec):
    from muse_psfr_b200 import _lib
    tables = [config2_table(), seeded_table(7, 5, bad4=(1,))]
    lbda = LBDA6
    pos = np.array([[0.0, 20.0], [0.0, -10.0]])
    w = np.stack([psfrec.band_weights(lbda, [480.0, 930.0], [1.0, 1.0]),
                  psfrec.band_weights(lbda, [600.0, 700.0, 800.0], [0.2, 1.0, 0.3])])
    kw = dict(lbda=lbda, npsflin=2, field_positions=pos, ee_radii=[0.4], elliptical=True, ao_budget=True,
              verbose=False)
    ref = psfrec.compute_psf_from_sparta_batch(tables, **kw)
    got = psfrec.compute_psf_from_sparta_batch(tables, bands=w, **kw)
    ctx = own_context(psfrec, 16)
    try:
        for g, r in zip(got, ref):
            names = [h.name for h in r]
            assert [h.name for h in g] == names + ['BAND_MEAN', 'PSF_BAND', 'BAND_FIELD', 'PSF_BAND_FIELD']
            for name in names[2:]:
                a, b = g[name].data, r[name].data
                if a.dtype.names:
                    assert all(np.array_equal(a[c], b[c], equal_nan=True) for c in b.dtype.names), name
                else:
                    assert np.array_equal(a, b), name
            for img, src, table in (('PSF_BAND', 'PSF_MEAN', 'BAND_MEAN'),
                                    ('PSF_BAND_FIELD', 'PSF_FIELD', 'BAND_FIELD')):
                cubes = np.ascontiguousarray(g[src].data, dtype=np.float64).reshape(-1, lbda.size, 40, 40)
                n = len(cubes)
                mb = np.empty((n, 2, 40, 40))
                ctx.band_psf(n, lbda.size, 40, 40, cubes, w, mb)
                band = np.asarray(g[img].data, dtype=np.float64)
                assert band.shape == ((2, 40, 40) if n == 1 else (n, 2, 40, 40))
                assert np.array_equal(band.reshape(mb.shape), mb), img
                assert_bands_close(mb, cubes, w)
                fit = np.empty((2 * n, _lib.FIT_NPAR))
                ctx.moffat_fit(2 * n, 40, 40, mb, fit)
                t = g[table].data
                assert np.array_equal(t['fwhm'][:, 0], fit[:, _lib.FIT_FWHM] * 0.2)
                assert np.array_equal(t['n'], fit[:, _lib.FIT_N])
                assert np.array_equal(t['lbda'], np.tile(psfrec._band_lbda_eff(lbda, w), n))
                assert np.array_equal(t['band'], np.tile([0, 1], n)) and np.array_equal(t['weights'], np.tile(w, (n, 1)))
                ee = np.empty((2 * n, 4))
                ctx.encircled_energy(2 * n, 40, 40, mb, [0.4 / 0.2], [0.5, 0.8], ee)
                assert np.array_equal(t['ee_total'], ee[:, 1])
                assert g[table].header['SEEING'] == g['FIT_MEAN'].header['SEEING']
            assert np.array_equal(g['BAND_FIELD'].data['x'], np.repeat(pos[0], 2))
    finally:
        ctx.close()
    bad = seeded_table(3, 2, invalid=(0, 1))
    assert psfrec.compute_psf_from_sparta(bad, lbda=lbda, verbose=False, bands=w) is None
