"""GPU tests of the AO summaries (DESIGN.md section 5.5) across their whole input envelope.

The Strehl ratio of ``psfr_compute_ao`` against the full-grid centre ratio psf[N/2][N/2] / psf_diff[N/2][N/2] of
psfr_psd + psfr_structure_function + psfr_psd_to_psf (and, in a few cases, the numpy oracle): every wavelength
limit and crop class at both grid sizes, wavelength tables of 64, 65 and 300 entries, every option set, field
positions far outside the laser asterism, 256 positions, field means, both laser modes and the corners of the
seeing / L0 envelope.  The variance record against the restatement of tests/ao_oracle.py slot by slot: dim 2560,
field positions, mixed laser modes in one call, per-draw profiles of 1 to 8 layers with zero-weight layers, and
chunk boundaries.  Every record also satisfies the identities of DESIGN.md 5.5, and its TOTAL is the sum of the
full-grid PSD."""
import numpy as np
import pytest
from numpy.testing import assert_allclose

import ao_oracle as ao
from test_gpu_ao import ao_outputs
from test_gpu_envelope import BAD_SEEING
from test_gpu_field import LBDA6, POS7

pytestmark = pytest.mark.gpu

orc = ao.orc
LGS4 = orc.lgs_positions(False)        # the three-laser asterism is its first three stars
FAR3 = np.array([[120., -120., 300.], [60., 60., 0.]])                 # far outside the 63" asterism
POS10 = np.ascontiguousarray(np.concatenate([POS7, FAR3], axis=1))
STREHL_RTOL = 1e-9
# The underflow cut and the single-precision grades move the device sum by less than 1e-14 of sum OTF_tel
# (DESIGN.md 5.5), an absolute error of 1e-14 on S whatever its size; above S = 1e-5 the relative 1e-9 is the
# larger bound, below it (the Strehl ratios under 1e-6 of the worst seeing at the shortest wavelengths) the
# absolute one.
STREHL_ATOL = 1e-14
VAR_RTOL = 1e-10
MARGIN = 1e-12
# config 1, the cut / precision-grade draw of test_gpu_envelope.py and the corners of seeing 0.3..3.0" x L0 5..100 m:
# (seeing, GL, L0, three lasers)
DRAWS = [(1.0, 0.7, 25.0, False), (BAD_SEEING[2], BAD_SEEING[0][0], BAD_SEEING[3], False),
         (0.3, 0.7, 5.0, True), (0.3, 0.5, 100.0, False), (3.0, 0.7, 5.0, False), (3.0, 0.4, 100.0, True)]


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


@pytest.fixture(scope='module')
def contexts(psfrec):
    """contexts(max_planes, dim, max_lambda): contexts of this file, made once each and closed at its end."""
    from muse_psfr_b200 import _lib
    made = {}

    def get(max_planes, dim=1280, max_lambda=35):
        key = (max_planes, dim, max_lambda)
        if key not in made:
            made[key] = _lib.Context(device=0, dim=dim, max_planes=max_planes, max_lambda=max_lambda)
            made[key].set_geometry(*psfrec.ao_frequency_tables())
        return made[key]
    yield get
    for ctx in made.values():
        ctx.close()


def records(psfrec, draws):
    seeing, GL, L0, three = (np.array(c) for c in zip(*draws))
    return psfrec._mode_records(three.astype(bool), seeing, GL, L0), three.astype(bool)


def centre_ratios(ctx, recs, three, dirs, lam):
    """psf[N/2][N/2] / psf_diff[N/2][N/2] of psfr_psd_to_psf, [ndraw, ndir, nl]: the PSD of every (draw,
    direction) from psfr_psd with the draw's own laser asterism, the diffraction PSF from a PSD of zeros, all
    in one workspace; and the PSDs [ndraw, ndir, N, N]."""
    dirs = np.ascontiguousarray(dirs, dtype=float)
    nd, ndir, dim = len(recs), dirs.shape[1], ctx.dim
    n = nd * ndir
    psd = np.zeros((n + 1, dim, dim))
    for d in range(nd):
        ctx.psd(recs[d:d + 1], dirs, orc.lgs_positions(three[d]), out=psd[d * ndir:(d + 1) * ndir])
    ctx.load_psd(psd, n + 1)
    ctx.structure_function(n + 1)
    out = np.empty((dim, dim))
    centre = np.empty((n + 1, len(lam)))
    for p in range(n + 1):
        for k, lb in enumerate(lam):
            ctx.psd_to_psf(p, lb * 1e-9, out)
            centre[p, k] = out[dim // 2, dim // 2]
    return (centre[:n] / centre[n]).reshape(nd, ndir, len(lam)), psd[:n].reshape(nd, ndir, dim, dim)


def assert_strehl(got, ref):
    got, ref = np.asarray(got), np.asarray(ref)
    assert np.all((got > 0) & (got <= 1))
    err = np.abs(got - ref)
    bound = STREHL_RTOL * ref + STREHL_ATOL
    assert np.all(err <= bound), 'worst error %.3g of the bound' % (err / bound).max()


def strehl_run(ctx, recs, dirs, lam, field=False):
    nd, ndir = len(recs), dirs.shape[1]
    out = ao_outputs(nd, ndir if field else 1, ndir, len(lam))
    ctx.compute_ao(field, recs, np.ascontiguousarray(dirs, dtype=float), LGS4, np.asarray(lam, dtype=float),
                   **out)
    return out['out_strehl'], out['out_var']


# ---------------------------------------------------------------- 1. Strehl against the full grid
# dim 1280: the shortest wavelength (crop 1280 = N; the boundary is 620800 / 1281), 490 nm, the crops that are
# multiples of 40 (1200, 1000, 800, 640: every bilinear fraction is 0), 1100 nm and the longest wavelength the
# convolutions accept (MUSE beta crosses 0 near 1188.99 nm)
LAM1280 = np.array([484.63, 490.0, 517.33, 620.8, 776.0, 970.0, 1100.0, 1188.9])
# dim 2560: crop 2560 = N, 250 nm, the 1280 limit, 930 nm and the longest (303.85 nm is refused: no mirror)
LAM2560 = np.array([242.42, 250.0, 484.63, 930.0, 1188.9])


def test_crop_classes_of_the_wavelengths():
    assert list(orc.npixc_of(LAM1280)[[0, 2, 3, 4, 5]]) == [1280, 1200, 1000, 800, 640]
    assert orc.npixc_of(620800 / 1281 - 1e-9)[0] == 1282
    assert orc.npixc_of(LAM2560)[0] == 2560


@pytest.mark.parametrize('dim', [1280, 2560])
def test_strehl_wavelength_limits(psfrec, contexts, dim):
    draws = DRAWS if dim == 1280 else [DRAWS[0], DRAWS[1], DRAWS[5]]
    lam = LAM1280 if dim == 1280 else LAM2560
    recs, three = records(psfrec, draws)
    ctx = contexts(16, dim)
    s, _ = strehl_run(ctx, recs, np.zeros((2, 1)), lam)
    ref, psd = centre_ratios(ctx, recs, three, np.zeros((2, 1)), lam)
    assert_strehl(s[:, 0], ref[:, 0])
    assert np.all(np.diff(s[:, 0], axis=1) > 0)          # rises with the wavelength
    if dim == 1280:                                     # the numpy oracle at both ends of the range
        for i, k in ((0, 0), (1, 7), (4, 0), (5, 4)):
            assert_strehl(s[i, 0, k], ao.strehl(psd[i, 0], lam[k] * 1e-9))


@pytest.mark.parametrize('nlam', [64, 65, 300])
def test_strehl_wavelength_tables(psfrec, contexts, nlam):
    """Per-wavelength tables staged in shared memory (64), one past (65) and 300 wavelengths, with duplicates:
    equal wavelengths give equal bits, the whole table rises with the wavelength, and every draw agrees with the
    full grid at a sampled subset of the wavelengths that includes both ends and duplicated entries."""
    rng = np.random.default_rng(nlam)
    lam = rng.uniform(484.63, 1188.9, nlam)
    lam[:4] = [484.63, 1188.9, 620.8, 970.0]
    dup = rng.choice(np.arange(4, nlam), nlam // 8, replace=False)
    lam[dup] = lam[rng.integers(0, 4, dup.size)]
    recs, three = records(psfrec, [DRAWS[0], DRAWS[1], DRAWS[2]])
    ctx = contexts(8, 1280, 300)
    s, _ = strehl_run(ctx, recs, np.zeros((2, 1)), lam)
    s = s[:, 0]
    for k in range(nlam):
        same = np.flatnonzero(lam == lam[k])
        assert all(np.array_equal(s[:, k], s[:, j]) for j in same), k
    order = np.argsort(lam, kind='stable')
    assert np.all(np.diff(s[:, order], axis=1) >= 0)
    pick = np.unique(np.concatenate([[0, 1, 2, 3, nlam - 1], dup[:2], rng.choice(nlam, 5, replace=False)]))
    ref, _ = centre_ratios(ctx, recs, three, np.zeros((2, 1)), lam[pick])
    assert_strehl(s[:, pick], ref[:, 0])


OPTION_SETS = {'default': {}, 'all_fp64': {'OPT_EXP_GRADE': 1e30, 'OPT_F32_ROWS': 1e30},
               'no_cut': {'OPT_EXP_CUT': 1000.0}, 'row_kernel_1': {'OPT_ROW_KERNEL': 1.0}}


@pytest.mark.parametrize('options', list(OPTION_SETS))
def test_strehl_option_sets(psfrec, contexts, options):
    """The bad-seeing draw (the cut and both precision grades occur) and the worst corner, at the crop limits:
    every option set within 1e-14 of sum OTF_tel of the default and within the bound of the full grid."""
    from muse_psfr_b200 import _lib
    lam = LAM1280[[0, 3, 5, 7]]
    recs, three = records(psfrec, [DRAWS[1], DRAWS[0], DRAWS[4]])
    base, _ = strehl_run(contexts(16), recs, np.zeros((2, 1)), lam)
    ctx = _lib.Context(device=0, max_planes=8, max_lambda=35)
    try:
        ctx.set_geometry(*psfrec.ao_frequency_tables())
        for key, value in OPTION_SETS[options].items():
            ctx.set_option(getattr(_lib, key), value)
        s, _ = strehl_run(ctx, recs, np.zeros((2, 1)), lam)
        assert np.max(np.abs(s - base)) < 1e-14
        ref, _ = centre_ratios(ctx, recs, three, np.zeros((2, 1)), lam)
        assert_strehl(s[:, 0], ref[:, 0])
    finally:
        ctx.close()


def test_strehl_field_positions(psfrec, contexts):
    """Field mode at every position of POS7 and three far outside the asterism, a three- and a four-laser draw:
    each position against the full-grid ratio of its own one-direction PSD."""
    lam = LAM1280[[0, 4, 7]]
    recs, three = records(psfrec, [DRAWS[5], DRAWS[0]])
    ctx = contexts(32)
    s, _ = strehl_run(ctx, recs, POS10, lam, field=True)
    ref, _ = centre_ratios(ctx, recs, three, POS10, lam)
    assert_strehl(s, ref)


def test_strehl_256_positions(psfrec, contexts):
    """256 positions in one field-mode call: a seeded subset against the full grid, and the same bits as a call
    with that subset alone."""
    rng = np.random.default_rng(256)
    pos = np.ascontiguousarray(rng.uniform(-150, 150, (2, 256)))
    lam = np.array([490.0, 776.0, 1100.0])
    recs, three = records(psfrec, [DRAWS[2]])
    ctx = contexts(256)
    s, _ = strehl_run(ctx, recs, pos, lam, field=True)
    pick = np.concatenate([[0, 255], rng.choice(np.arange(1, 255), 6, replace=False)])
    ref, _ = centre_ratios(ctx, recs, three, pos[:, pick], lam)
    assert_strehl(s[:, pick], ref)
    alone, _ = strehl_run(ctx, recs, pos[:, pick], lam, field=True)
    assert np.array_equal(alone, s[:, pick])


@pytest.mark.parametrize('npsflin', [2, 3, 5])
def test_strehl_field_mean(psfrec, contexts, npsflin):
    """Field-mean mode: the Strehl ratio of the mean PSF is the mean of the per-direction full-grid ratios."""
    lam = LAM1280[[0, 5, 7]]
    recs, three = records(psfrec, [DRAWS[0], DRAWS[2]])
    dirs = psfrec.direction_perf(npsflin)
    ctx = contexts(64)
    s, _ = strehl_run(ctx, recs, dirs, lam)
    ref, _ = centre_ratios(ctx, recs, three, dirs, lam)
    assert_strehl(s[:, 0], ref.mean(axis=1))


# ---------------------------------------------------------------- 2. variance against the restatement
def check_records(var, refs, nls):
    """var [nd, ndir, VAR_NPAR] against the restatement refs per draw, slot by slot, and the identities of every
    record: TOTAL = FIT + NOISE + PROJ, PROJ = sum LAYER, the slots past the draw's layers exactly 0."""
    for d, (ref, nl) in enumerate(zip(refs, nls)):
        assert_allclose(var[d], ref, rtol=VAR_RTOL, atol=0, err_msg='draw %d' % d)
        for r in var[d]:
            assert abs(r[1] + r[2] + r[3] - r[0]) <= 1e-13 * r[0]
            assert abs(r[4:].sum() - r[3]) <= 1e-13 * r[3]
            assert np.all(r[4 + nl:] == 0)


def restated(draws, dim=1280, dirs=None, npsflin=1, **kw):
    """The restatement and its zone margin for each (seeing, GL, L0, three) draw of the two-layer profile."""
    refs = []
    for seeing, GL, L0, three in draws:
        args = dict(Cn2=[GL, 1 - GL], h=(100, 10000), seeing=seeing, L0=L0, npsflin=npsflin, three_lgs_mode=three,
                    dim=dim, dirs=dirs, **kw)
        assert ao.zone_margin(**args) > MARGIN
        refs.append(ao.variance_record(**args))
    return refs


@pytest.mark.parametrize('field', [False, True])
def test_variance_dim2560(psfrec, contexts, field):
    """dim 2560: the 1280 x 1280 fitting quadrant of each draw at its own offset, the zone at lo = N/2 - 40."""
    draws = [DRAWS[0], DRAWS[1], DRAWS[5]]
    dirs = POS10[:, [0, 5, 9]] if field else psfrec.direction_perf(2)
    recs, _ = records(psfrec, draws)
    _, var = strehl_run(contexts(16, 2560), recs, dirs, [700.0], field=field)
    check_records(var, restated(draws, 2560, dirs), [2] * len(draws))


def test_variance_total_is_the_psd_sum_off_axis(psfrec, contexts):
    """TOTAL is the sum of psfr_psd's full N x N PSD over L^2 = 256 m^2 at dim 2560 and off axis at both sizes."""
    for dim, draws, dirs in ((2560, [DRAWS[1], DRAWS[2]], FAR3[:, [0, 2]]), (1280, [DRAWS[5]], POS10[:, 5:])):
        recs, three = records(psfrec, draws)
        ctx = contexts(16, dim)
        _, var = strehl_run(ctx, recs, dirs, [700.0], field=True)
        for d in range(len(recs)):
            psd = np.empty((dirs.shape[1], dim, dim))
            ctx.psd(recs[d:d + 1], np.ascontiguousarray(dirs), orc.lgs_positions(three[d]), out=psd)
            assert_allclose(var[d, :, 0], psd.sum(axis=(1, 2)) / 256, rtol=1e-12, atol=0)


def test_variance_field_positions(psfrec, contexts):
    """POS7 and the far positions through compute_psf_field(ao_budget=True) and the raw compute_ao(True, ...),
    one three- and one four-laser draw, each against the restatement at its own positions."""
    draws = [DRAWS[5], DRAWS[0], DRAWS[1]]
    seeing, GL, L0, three = (np.array(c) for c in zip(*draws))
    out = psfrec.compute_psf_field(LBDA6[:2], seeing, GL, L0, positions=POS10, three_lgs_mode=three.astype(bool),
                                   want_cube=False, ao_budget=True)
    recs, _ = records(psfrec, draws)
    _, raw = strehl_run(contexts(32), recs, POS10, LBDA6[:2], field=True)
    assert np.array_equal(out[-1], raw)
    check_records(raw, restated(draws, dirs=POS10), [2] * len(draws))


def test_variance_256_positions(psfrec, contexts):
    rng = np.random.default_rng(2560)
    pos = np.ascontiguousarray(rng.uniform(-150, 150, (2, 256)))
    draws = [DRAWS[3]]
    recs, _ = records(psfrec, draws)
    _, var = strehl_run(contexts(256), recs, pos, [700.0], field=True)
    check_records(var, restated(draws, dirs=pos), [2])


def test_variance_mixed_laser_modes(psfrec, contexts):
    """A seeded batch of three- and four-laser draws in one call (per-draw guide-star count) through
    compute_psf_batch(three_lgs_mode=[...]) and compute_ao with exposures: each draw against the restatement of
    its own mode, both paths the same bits."""
    rng = np.random.default_rng(17)
    nd = 9
    seeing, GL, L0 = rng.uniform(0.3, 3.0, nd), rng.uniform(0.3, 0.9, nd), rng.uniform(5, 100, nd)
    three = rng.random(nd) < 0.5
    assert 0 < three.sum() < nd
    _, _, _, var = psfrec.compute_psf_batch(LBDA6[:2], seeing, GL, L0, npsflin=2, three_lgs_mode=three,
                                            want_cube=False, ao_budget=True)
    recs = psfrec._mode_records(three, seeing, GL, L0)
    out = ao_outputs(nd, 1, 4, 2)
    contexts(16).compute_ao(False, recs, psfrec.direction_perf(2), LGS4, LBDA6[:2],
                            group_end=np.array([2, 3, 7, 9], dtype=np.int32), out_var=out['out_var'])
    assert np.array_equal(out['out_var'], var)
    check_records(var, restated(list(zip(seeing, GL, L0, three)), npsflin=2), [2] * nd)


# per-draw profiles: (zenith, integer altitudes, seeing and L0 of the draws); the layer count is the case index + 1
PROFILES = [(0.0, True, [0.3, 3.0], [5.0, 100.0]), (15.0, False, [3.0, 0.3], [100.0, 5.0]),
            (45.0, True, [0.3, 1.2], [100.0, 30.0]), (60.0, False, [3.0, 0.7], [5.0, 20.0]),
            (0.0, False, [0.9, 3.0], [12.0, 100.0]), (15.0, True, [0.3, 2.0], [5.0, 60.0]),
            (45.0, False, [1.5, 0.3], [100.0, 8.0]), (60.0, True, [3.0, 0.5], [40.0, 5.0])]


@pytest.mark.parametrize('nl', range(1, 9))
def test_variance_per_draw_profiles(psfrec, nl):
    """h and Cn2 of shape [ndraw, nl], arbitrary wind directions, zenith 0 to 60 degrees, integer altitudes (12 m/s
    wind, the reference's np.full_like) and float ones (12.5 m/s); from 2 layers on, the second draw has a
    zero-weight layer whose slot must be exactly 0."""
    zenith, integer, seeing, L0 = PROFILES[nl - 1]
    rng = np.random.default_rng(100 + nl)
    nd = len(seeing)
    h = np.sort(rng.uniform(20, 18000, (nd, nl)), axis=1)
    h = np.round(h).astype(int) if integer else h
    Cn2 = rng.uniform(0.05, 1.0, (nd, nl))
    if nl > 1:
        Cn2[1, nl // 2] = 0.0
    wind_dir = rng.uniform(-np.pi, np.pi, nl)
    GL = np.full(nd, 0.6)
    with np.errstate(divide='ignore'):
        _, _, _, var = psfrec.compute_psf_batch(LBDA6[:2], seeing, GL, L0, npsflin=2, h=h, Cn2=Cn2, wind_dir=wind_dir,
                                                zenith=zenith, want_cube=False, ao_budget=True)
    refs = []
    for d in range(nd):
        args = dict(Cn2=Cn2[d], h=h[d], seeing=seeing[d], L0=L0[d], zenith=zenith, npsflin=2, wind_dir=wind_dir)
        assert ao.zone_margin(**args) > MARGIN
        refs.append(ao.variance_record(**args))
    check_records(var, refs, [nl] * nd)
    if nl > 1:
        assert np.all(var[1, :, 4 + nl // 2] == 0) and np.all(np.delete(var[:, :, 4:4 + nl], nl // 2, axis=2)[1] > 0)


@pytest.mark.parametrize('ndir', [3, 7])
def test_variance_chunk_boundaries(psfrec, contexts, ndir):
    """11 draws at ndir positions with max_planes = ndir (one draw per chunk), 2 ndir + 1 (two draws per chunk,
    one plane unused, a partial last chunk) and 256 (not a multiple of ndir, one chunk): the same bits at every
    size, and the restatement."""
    rng = np.random.default_rng(ndir)
    nd = 11
    draws = list(zip(rng.uniform(0.3, 3.0, nd), rng.uniform(0.3, 0.9, nd), rng.uniform(5, 100, nd),
                     rng.random(nd) < 0.5))
    dirs = POS10[:, rng.choice(10, ndir, replace=False)]
    recs, _ = records(psfrec, draws)
    lam = LBDA6[:2]
    first = None
    for max_planes in (ndir, 2 * ndir + 1, 256):
        got = strehl_run(contexts(max_planes), recs, dirs, lam, field=True)
        if first is None:
            first = got
        else:
            assert all(np.array_equal(a, b) for a, b in zip(got, first)), max_planes
    check_records(first[1], restated(draws, dirs=dirs), [2] * nd)
