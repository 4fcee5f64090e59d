"""GPU tests of the elliptical Moffat fit (``psfr_moffat_fit_elliptical``, ``efit_kernel`` / ``write_efit_record``)
across its whole input envelope.

Every comparison has a concrete reference: the known truth of a noise-free render (each case first passes
``efit_oracle.well_posed``, so that a failure points at the kernel and not at an ill-posed image), scipy leastsq
started from the GPU's own solution (the solution is stationary), and ``efit_oracle.record_ld``, the whole record
recomputed in long double from the GPU's own parameters.  Covered: image shapes from 3 x 3 to the shared-memory
limits 79 x 80 and 3 x 1600 (small images are where the coarse first stage of the circular fit, the start point of
the elliptical one, sees only part of the image), a seeded grid of widths, axis ratios, n, position angles and
centres, noisy images, degenerate inputs, refusals, staging of host images in chunks, and the fused pipeline at its
edges bit for bit against the standalone call."""
import logging

import numpy as np
import pytest
from numpy.testing import assert_allclose

import efit_oracle as eo
from test_gpu_ao_envelope import DRAWS, records
from test_gpu_field import LBDA6
from test_gpu_shape import assert_matches_reference, efit_of, pa_diff_rad

pytestmark = pytest.mark.gpu

SENT = 12345.0
KNOWN_RTOL = 1e-8           # every parameter slot of an exact render against the truth (as test_known_answers)
STAT_RTOL = 1e-7            # FWHM_MAJOR, FWHM_MINOR, AXIS_RATIO and N moved by the CPU refit at most this much
STAT_CHI2 = 1e-12           # ... and chi^2 lowered by at most this much, relative
LD_RTOL = 1e-9              # every slot against record_ld at the GPU's own parameters


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
    """contexts(max_planes, max_lambda, dim): contexts of this file, made once each and closed at its end."""
    from muse_psfr_b200 import _lib
    made = {}

    def get(max_planes=16, max_lambda=35, dim=1280):
        key = (max_planes, max_lambda, dim)
        if key not in made:
            made[key] = _lib.Context(device=0, dim=dim, max_planes=max_planes, max_lambda=max_lambda)
            made[key].set_geometry(*psfrec.ao_frequency_tables())
        return made[key]
    yield get
    for ctx in made.values():
        ctx.close()


def fit_of(ctx, imgs):
    from muse_psfr_b200 import _lib
    imgs = np.ascontiguousarray(imgs, dtype=float)
    n, ny, nx = imgs.shape
    out = np.full((n, _lib.FIT_NPAR), np.nan)
    ctx.moffat_fit(n, ny, nx, imgs, out)
    return out


def assert_known_answer(r, truth, what):
    """Record r of an exact render of truth (render() arguments)."""
    I, y0, x0, amaj, amin, pa, n = truth
    q = amin / amaj
    assert r[eo.ITER] > 0, what
    for slot, ref in ((eo.PEAK, I), (eo.Y0, y0), (eo.X0, x0), (eo.A_MAJOR, amaj), (eo.A_MINOR, amin), (eo.N, n),
                      (eo.AXIS_RATIO, q)):
        assert_allclose(r[slot], ref, rtol=KNOWN_RTOL, err_msg='%s slot %d' % (what, slot))
    assert 0 <= r[eo.PA] < 180 and not np.signbit(r[eo.PA]), (what, r[eo.PA])
    assert pa_diff_rad(r[eo.PA], pa) <= 1e-6 / (1 - q), (what, r[eo.PA], pa)
    kf = 2 * np.sqrt(2 ** (1 / n) - 1)
    assert_allclose(r[[eo.FWHM_MAJOR, eo.FWHM_MINOR]], [amaj * kf, amin * kf], rtol=KNOWN_RTOL, err_msg=what)
    assert_allclose(r[eo.FLUX], np.pi * I * amaj * amin / (n - 1), rtol=KNOWN_RTOL, err_msg=what)


def assert_stationary(img, r, what):
    """The CPU fit started from the GPU's solution moves it by at most STAT_RTOL and lowers chi^2 by at most
    STAT_CHI2."""
    with np.errstate(all='ignore'):
        ref, _ = eo.moffat_fit_elliptical(img, start=eo.theta_of_record(r))
    for slot in (eo.FWHM_MAJOR, eo.FWHM_MINOR, eo.AXIS_RATIO, eo.N):
        assert abs(ref[slot] - r[slot]) <= STAT_RTOL * abs(r[slot]), (what, slot, ref[slot], r[slot])
    assert ref[eo.CHISQ] >= r[eo.CHISQ] * (1 - STAT_CHI2), (what, ref[eo.CHISQ], r[eo.CHISQ])


def assert_matches_record_ld(img, r, what):
    """Every slot but ITER against the long-double record at the GPU's own parameters; PA as a distance modulo
    180 degrees, and PA / ERR_PA only where 1 - q >= 1e-3 (assert_matches_reference)."""
    ref = eo.record_ld(eo.theta_of_record(r), img)
    skip = {eo.ITER, eo.PA}
    if 1 - r[eo.AXIS_RATIO] < 1e-3:
        skip.add(eo.ERR_PA)
    else:
        assert pa_diff_rad(r[eo.PA], ref[eo.PA]) <= LD_RTOL * np.pi, (what, r[eo.PA], ref[eo.PA])
    for slot in sorted(set(range(eo.NPAR)) - skip):
        assert_allclose(r[slot], ref[slot], rtol=LD_RTOL, atol=0, err_msg='%s slot %d' % (what, slot))


# ---------------------------------------------------------------- 1. image shapes
SQUARE = [(3, 3), (5, 5), (8, 8), (12, 12), (16, 16), (17, 17), (20, 20), (22, 22), (33, 33), (64, 64)]
NONSQUARE = [(13, 29), (29, 13), (3, 40), (40, 3)]
LIMITS = [(79, 80), (80, 79), (3, 1600), (1600, 3)]


def shape_truths(shape):
    """A centred render and two 1.5 px from an edge (the centre 1.5 px inside the first row, and inside the last
    column), semi-major axis a fifth of the short side between 0.8 and 3 px, q = 0.7 at 30 degrees."""
    ny, nx = shape
    a = float(np.clip(min(shape) / 5, 0.8, 3.0))
    cy, cx = (ny - 1) / 2 + 0.23, (nx - 1) / 2 - 0.17
    return [(1.7, cy, cx, a, 0.7 * a, 30.0, 2.5), (1.3, 1.5, cx, a, 0.7 * a, 30.0, 2.5),
            (2.1, cy, nx - 2.5, a, 0.7 * a, 30.0, 2.5)]


# Cases the kernel still gets wrong, kept as strict expected failures: each must keep failing until the kernel
# is fixed, then move to the passing set.  Every image passes efit_oracle.well_posed, so the failure is the
# kernel's.  Two fixes already moved cases out of this list: the circular fit skips its coarse stage on images of
# at most 512 pixels (17 x 17 grid cases 4, 36 and 68 went wrong from a start fitted to wings), and the elliptical
# fit restarts from the half-maximum moments when its circular start or its first attempt did not converge (40 x 40
# grid cases 26, 35 and 65, 17 x 17 cases 12, 26, 28, 48, 51 and 75, and noisy cases 2, 5, 8 and 23).  What remains:
# - the 3-pixel strips and the 3 x 3 / 5 x 5 renders 1.5 px from an edge (a_major 0.8 or 1 px): the circular fit
#   collapses onto a one-pixel spike and both elliptical attempts stop short of the truth or at the iteration limit;
# - 40 x 40 case 22 and 17 x 17 cases 14 and 20: minor semi-axis 0.14 or 0.3 px;
# - 17 x 17 cases 33 and 67: minor semi-axis 0.3 px, n = 4, 200 iterations from either start;
# - 40 x 40 cases 51 and 71 and 17 x 17 case 24: n = 10 with a_major <= 1.5 px, stopped 1e-8 to 1e-5 from the
#   truth by the 1.49e-8 relative-step rule.
# {shape: case indices of shape_truths / efit_oracle.grid / noisy_cases}
START_FAILS_SHAPES = {(3, 3): (1, 2), (5, 5): (2,), (3, 40): (0, 1, 2), (40, 3): (0, 2), (3, 1600): (0, 1, 2),
                      (1600, 3): (0, 2)}
START_FAILS_GRID = {(40, 40): (22, 51, 71), (17, 17): (14, 20, 24, 33, 67)}
START_FAILS_NOISY = ()
START_REASON = 'known kernel failure on a PSF narrower than about a pixel (see START_FAILS_SHAPES)'


def cases_with_known_failures(keys, fails):
    return [pytest.param(*k, marks=pytest.mark.xfail(strict=True, reason=START_REASON)) if k in fails
            else pytest.param(*k) for k in keys]


SHAPE_KEYS = [(shape, i) for shape in SQUARE + NONSQUARE + LIMITS for i in range(3)]


@pytest.mark.parametrize('shape,case', cases_with_known_failures(
    SHAPE_KEYS, {(s, i) for s, ii in START_FAILS_SHAPES.items() for i in ii}),
    ids=['%dx%d-%d' % (s + (i,)) for s, i in SHAPE_KEYS])
def test_shapes_known_answers(psfrec, contexts, shape, case):
    from muse_psfr_b200 import _lib
    ctx = contexts()
    t = shape_truths(shape)[case]
    img = eo.render(shape, *t)
    eo.well_posed(img, t)
    # the circular record the elliptical fit starts from converged on the same image
    assert fit_of(ctx, img[None])[0, _lib.FIT_ITER] > 0
    assert_known_answer(efit_of(ctx, img[None])[0], t, '%s case %d' % (shape, case))
    # and the circular fit recovers a circular render of the same shape
    circ = (t[0], t[1], t[2], t[3], t[3], 0.0, t[6])
    f = fit_of(ctx, eo.render(shape, *circ)[None])[0]
    kf = 2 * np.sqrt(2 ** (1 / t[6]) - 1)
    assert f[_lib.FIT_ITER] > 0, (shape, circ)
    assert_allclose(f[[_lib.FIT_FWHM, _lib.FIT_N]], [t[3] * kf, t[6]], rtol=KNOWN_RTOL, err_msg=str((shape, circ)))


# ---------------------------------------------------------------- 2. parameter grid
GRID_KEYS = [(shape, i) for shape in [(40, 40), (17, 17)] for i, _ in eo.grid(shape)[0]]


@pytest.mark.parametrize('shape', [(40, 40), (17, 17)], ids=lambda s: '%dx%d' % s)
def test_parameter_grid(psfrec, contexts, shape):
    """The seeded grid of efit_oracle.grid (every a_major, q, n, PA and centre class), minus the cases listed in
    efit_oracle.GRID_REMOVED with their reason and the known failures of START_FAILS_GRID; every record, those
    included, has 0 <= PA < 180 and a clear sign bit."""
    kept, _ = eo.grid(shape)
    imgs = np.stack([eo.render(shape, *t) for _, t in kept])
    rec = efit_of(contexts(), imgs)
    assert np.all((rec[:, eo.PA] >= 0) & (rec[:, eo.PA] < 180) & ~np.signbit(rec[:, eo.PA]))
    failed = []
    for img, r, (i, t) in zip(imgs, rec, kept):
        if i not in START_FAILS_GRID.get(shape, ()):
            eo.well_posed(img, t)
            try:
                assert_known_answer(r, t, '%s grid case %d' % (shape, i))
            except AssertionError as e:
                failed.append((i, str(e).splitlines()[0]))
    if failed:
        pytest.fail('grid cases failing: %s' % ' '.join(str(i) for i, _ in failed))


@pytest.mark.parametrize('shape,case', [k for k in GRID_KEYS if k[1] in START_FAILS_GRID.get(k[0], ())],
                         ids=lambda v: '%dx%d' % v if isinstance(v, tuple) else str(v))
@pytest.mark.xfail(strict=True, reason=START_REASON)
def test_parameter_grid_known_failures(psfrec, contexts, shape, case):
    t = dict(eo.grid(shape)[0])[case]
    img = eo.render(shape, *t)
    eo.well_posed(img, t)
    assert_known_answer(efit_of(contexts(), img[None])[0], t, '%s grid case %d' % (shape, case))


# ---------------------------------------------------------------- 3. noisy images
NOISY_SHAPES = [(8, 8), (17, 17), (40, 40), (79, 80)]
NOISY_QPA = [(0.95, 20.0), (0.6, 110.0), (0.3, 165.0)]


def noisy_cases():
    cases = []
    for shape in NOISY_SHAPES:
        a = float(np.clip(min(shape) / 6, 1.2, 4.0))
        for level in (1e-3, 1e-2):
            for j, (q, pa) in enumerate(NOISY_QPA):
                truth = (1.0, (shape[0] - 1) / 2 + 0.21, (shape[1] - 1) / 2 - 0.37, a, q * a, pa, 2.2 + 0.4 * j)
                cases.append((shape, level, truth, eo.render_noisy(shape, truth, level, len(cases))))
    return cases


NOISY = noisy_cases()


def test_noisy_images_go_negative():
    assert any(np.any(c[3] < 0) for c in NOISY)


@pytest.mark.parametrize('case', cases_with_known_failures([(k,) for k in range(len(NOISY))],
                                                           {(k,) for k in START_FAILS_NOISY}),
                         ids=['%dx%d-%g-%d' % (c[0] + (c[1], k)) for k, c in enumerate(NOISY)])
def test_noisy_images(psfrec, contexts, case):
    shape, level, truth, img = NOISY[case]
    r = efit_of(contexts(), img[None])[0]
    what = '%s noise %g case %d' % (shape, level, case)
    assert r[eo.ITER] > 0, what
    assert_stationary(img, r, what)
    assert_matches_record_ld(img, r, what)


# ---------------------------------------------------------------- 4. degenerate inputs
def degenerate_images():
    shape = (17, 17)
    hot = np.zeros(shape)
    hot[8, 9] = 1.0
    plateau = eo.render(shape, 1.0, 8.0, 8.5, 2.0, 1.5, 0.0, 2.5)
    plateau[8, 8] = plateau[8, 9] = plateau.max() * 1.01
    nan = eo.render(shape, 1.0, 8.2, 7.9, 2.5, 1.8, 40.0, 2.5)
    nan[3, 11] = np.nan
    return {'zero': np.zeros(shape), 'constant': np.full(shape, 0.7), 'nan': nan, 'hot': hot, 'plateau': plateau}


def test_degenerate_inputs(psfrec, contexts, caplog):
    from muse_psfr_b200 import _lib
    imgs = degenerate_images()
    rec = efit_of(contexts(), np.stack(list(imgs.values())))
    derived = [eo.A_MAJOR, eo.A_MINOR, eo.FWHM_MAJOR, eo.FWHM_MINOR, eo.AXIS_RATIO, eo.FLUX]
    for (name, img), r in zip(imgs.items(), rec):
        converged = r[_lib.EFIT_ITER] > 0
        if name in ('zero', 'constant', 'nan'):
            assert not converged or not np.all(np.isfinite(r[derived])), (name, r)
        elif converged:
            assert_stationary(img, r, name)
        with caplog.at_level(logging.WARNING, logger='muse_psfr_b200'):
            caplog.clear()
            tab = psfrec.fit_psf_cube([700.0], img[None], circular=False)
        assert tab['converged'][0] == int(converged), name
        assert any('did not converge' in m for m in caplog.messages) == (not converged), name


# ---------------------------------------------------------------- 5. refusals and staging
@pytest.mark.parametrize('shape', [(80, 80), (81, 79), (3, 1601)], ids=lambda s: '%dx%d' % s)
def test_refuses_images_over_the_shared_memory_limit(psfrec, contexts, shape):
    from muse_psfr_b200 import _lib
    ctx = contexts()
    img = np.ones((2,) + shape)
    rec = np.full((2, 24), SENT)
    fn = ctx._lib.psfr_moffat_fit_elliptical
    assert fn(ctx._handle(), 2, shape[0], shape[1], _lib.ptr(img), _lib.ptr(rec), None) == _lib.E_UNSUPPORTED
    assert np.all(rec == SENT)


def test_refuses_an_image_over_the_staging_buffer(psfrec, contexts):
    from muse_psfr_b200 import _lib
    ctx = contexts(1, 1)
    img = np.ones((1, 41, 40))
    rec = np.full((1, 24), SENT)
    fn = ctx._lib.psfr_moffat_fit_elliptical
    assert fn(ctx._handle(), 1, 41, 40, _lib.ptr(img), _lib.ptr(rec), None) == _lib.E_CAPACITY
    assert np.all(rec == SENT)
    # 40 x 40 fits the same context
    ok = efit_of(ctx, eo.render((40, 40), 1.0, 20.2, 19.6, 3.0, 2.0, 30.0, 2.5)[None])
    assert ok[0, eo.ITER] > 0


# (shape, images): on a 1 plane x 35 wavelength context 79 x 80 images go 8 per chunk, 3 x 1600 11 and 8 x 8 35
STAGING = [((79, 80), 19), ((3, 1600), 25), ((8, 8), 75)]


@pytest.mark.parametrize('shape,nimg', STAGING, ids=lambda v: '%dx%d' % v if isinstance(v, tuple) else str(v))
def test_staging_chunks(psfrec, contexts, shape, nimg):
    import torch
    ctx = contexts(1, 35)
    rng = np.random.default_rng(nimg)
    a = float(np.clip(min(shape) / 5, 0.8, 3.0))
    imgs = np.stack([eo.render_noisy(shape, ((1.0 + 0.1 * k, (shape[0] - 1) / 2 + rng.uniform(-0.5, 0.5),
                                               (shape[1] - 1) / 2 + rng.uniform(-0.5, 0.5), a, a * rng.uniform(0.4, 1),
                                               rng.uniform(0, 180), rng.uniform(1.5, 4))), 1e-3, k)
                     for k in range(nimg)])
    host = efit_of(ctx, imgs)
    assert np.sum(host[:, eo.ITER] > 0) > nimg // 2
    one = np.concatenate([efit_of(ctx, imgs[k:k + 1]) for k in range(nimg)])
    assert np.array_equal(host, one, equal_nan=True)
    d_img = torch.from_numpy(imgs).cuda()
    outs = {}
    for name, src, dst in (('device', d_img, 'cuda'), ('host in, device out', imgs, 'cuda'),
                           ('device in, host out', d_img, 'cpu')):
        out = torch.full((nimg, 24), np.nan, dtype=torch.float64, device=dst)
        ctx.moffat_fit_elliptical(nimg, shape[0], shape[1], src, out)
        torch.cuda.synchronize()
        outs[name] = out.cpu().numpy()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    out = torch.full((nimg, 24), np.nan, dtype=torch.float64, device='cuda')
    with torch.cuda.stream(side):
        ctx.moffat_fit_elliptical(nimg, shape[0], shape[1], d_img, out, stream=side.cuda_stream)
    side.synchronize()
    outs['side stream'] = out.cpu().numpy()
    for name, o in outs.items():
        assert np.array_equal(o, host, equal_nan=True), name


# ---------------------------------------------------------------- 6. the fused path at its edges
def fused_outputs(nd, P, nl, ng):
    from muse_psfr_b200 import _lib
    return dict(out_cube=np.full((nd, P, nl, 40, 40), np.nan), out_mean=np.full((ng, P, nl, 40, 40), np.nan),
                out_efit=np.full((nd, P, nl, _lib.EFIT_NPAR), np.nan),
                out_mean_efit=np.full((ng, P, nl, _lib.EFIT_NPAR), np.nan))


def fused_case(psfrec, case):
    """(records, dirs, lam, group_end, dim, max_planes) of each edge of the fused path.  A field call needs one plane
    per direction, so 256 positions run at 256 planes (one draw per chunk) and 512 (both draws in one)."""
    if case == 'dim2560':
        recs, _ = records(psfrec, [DRAWS[0], DRAWS[5]])
        return recs, np.array([[0.0, 12.5], [0.0, -7.3]]), np.array([490.0, 930.0]), [1, 2], 2560, (3, 8, 128)
    if case == 'pos256':
        rng = np.random.default_rng(256)
        recs, _ = records(psfrec, [DRAWS[2], DRAWS[3]])
        return recs, rng.uniform(-150, 150, (2, 256)), np.array([700.0]), [2], 1280, (256, 512)
    if case == 'mixed_lasers':
        rng = np.random.default_rng(17)
        nd = 6
        three = np.array([True, False, False, True, True, False])
        recs = psfrec._mode_records(three, rng.uniform(0.3, 3.0, nd), rng.uniform(0.3, 0.9, nd),
                                    rng.uniform(5, 100, nd))
        return recs, np.array([[0.0, -30.0, 45.0], [0.0, 30.0, 0.0]]), LBDA6[:3], [2, 5, 6], 1280, (3, 8, 128)
    nl = {'layers1': 1, 'layers8': 8}[case]
    rng = np.random.default_rng(100 + nl)
    h = np.sort(rng.uniform(20, 18000, (2, nl)), axis=1)
    Cn2 = rng.uniform(0.05, 1.0, (2, nl))
    recs = psfrec._mode_records(np.array([False, True]), np.array([0.6, 1.4]), np.full(2, 0.6),
                                np.array([20.0, 60.0]), h=h, Cn2=Cn2, wind_dir=rng.uniform(-np.pi, np.pi, nl))
    return recs, np.array([[0.0, 30.0], [0.0, -30.0]]), LBDA6[[0, 5]], [1, 2], 1280, (3, 8, 128)


@pytest.mark.parametrize('case', ['dim2560', 'pos256', 'mixed_lasers', 'layers1', 'layers8'])
def test_fused_equals_standalone(psfrec, case):
    """psfr_compute_field_shapes and psfr_compute_ao (field and field-mean modes) with per-draw laser counts from
    the records: out_efit and out_mean_efit are psfr_moffat_fit_elliptical of out_cube and out_mean bit for bit at
    every max_planes, every max_planes gives the same bits, and a seeded sample of 32 images per mode matches the
    CPU reference."""
    from muse_psfr_b200 import _lib
    recs, dirs, lam, ge, dim, planes = fused_case(psfrec, case)
    dirs = np.ascontiguousarray(dirs)
    group_end = np.array(ge, dtype=np.int32)
    nd, ndir, nl, ng = len(recs), dirs.shape[1], len(lam), len(ge)
    lgs = psfrec._lgs_positions(False)
    first = {}
    for max_planes in planes:
        ctx = _lib.Context(device=0, dim=dim, max_planes=max_planes, max_lambda=35)
        try:
            ctx.set_geometry(*psfrec.ao_frequency_tables())
            for field in (True, False):
                outs = fused_outputs(nd, ndir if field else 1, nl, ng)
                if field and max_planes == planes[0]:
                    ctx.compute_field(recs, dirs, lgs, lam, group_end, **outs)
                else:
                    ctx.compute_ao(field, recs, dirs, lgs, lam, group_end=group_end, **outs)
                assert np.array_equal(outs['out_efit'].reshape(-1, 24),
                                      efit_of(ctx, outs['out_cube'].reshape(-1, 40, 40))), (field, max_planes)
                assert np.array_equal(outs['out_mean_efit'].reshape(-1, 24),
                                      efit_of(ctx, outs['out_mean'].reshape(-1, 40, 40))), (field, max_planes)
                ref = first.setdefault(field, outs)
                for k in outs:
                    assert np.array_equal(outs[k], ref[k]), (field, max_planes, k)
        finally:
            ctx.close()
    rng = np.random.default_rng(len(case))
    for field, outs in first.items():
        imgs = np.concatenate([outs['out_cube'].reshape(-1, 40, 40), outs['out_mean'].reshape(-1, 40, 40)])
        rec = np.concatenate([outs['out_efit'].reshape(-1, 24), outs['out_mean_efit'].reshape(-1, 24)])
        assert np.all(rec[:, eo.ITER] > 0)
        pick = rng.choice(len(imgs), min(32, len(imgs)), replace=False)
        ref = np.stack([eo.moffat_fit_elliptical(imgs[k])[0] for k in pick])
        assert_matches_reference(rec[pick], ref)
