"""GPU tests of ``psfr_encircled_energy`` across the inputs it accepts, against the long-double restatement
tests/ee_oracle.py and closed forms: every image shape from 3 x 3 to the shared-memory limit (5120 pixels), the
staging of host arrays in chunks at sizes other than 40 x 40, centres on half-integers, on the border and far
outside the image, radii from 1e-300 to 1e300 in any order, fractions next to 0 and 1 and on a plateau of EE,
images with negative pixels, two contexts of different image sizes in one process, and a side stream.

Bounds as in tests/test_gpu_energy.py: EE and TOTAL to 1e-14 times the image's absolute sum, radii at fractions
to 1e-9 px.  For an image with negative pixels the oracle's brentq finds one root of several, so there r_q is
checked to be a crossing of the oracle's EE instead."""
import itertools

import numpy as np
import pytest
from numpy.testing import assert_allclose

import ee_oracle as eo

pytestmark = pytest.mark.gpu

FRACS = np.array([0.2, 0.5, 0.8, 0.9])
SHAPES = [(3, 3), (3, 40), (40, 3), (5, 7), (8, 8), (31, 31), (32, 32), (33, 33), (41, 41), (30, 50), (50, 30),
          (63, 65)]
PIXSCALE = 0.2


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
def ctx(psfrec):
    return psfrec.get_context()


def ee_of(ctx, imgs, radii, fracs, centres=None):
    imgs = np.ascontiguousarray(imgs, dtype=float)
    n, ny, nx = imgs.shape
    radii, fracs = np.asarray(radii, dtype=float), np.asarray(fracs, dtype=float)
    out = np.full((n, radii.size + 1 + fracs.size), np.nan)
    ctx.encircled_energy(n, ny, nx, imgs, radii, fracs, out,
                         centres=None if centres is None else np.ascontiguousarray(centres, dtype=float))
    return out


def rmax_of(ny, nx, y0, x0):
    """Distance from (y0, x0) to the farthest pixel corner."""
    return np.hypot(max(y0 + 0.5, ny - 0.5 - y0), max(x0 + 0.5, nx - 0.5 - x0))


def assert_parity(imgs, recs, radii, fracs, centres=None):
    nrad = len(radii)
    for i, img in enumerate(imgs):
        c = None if centres is None else tuple(centres[i])
        ref = eo.record(img, radii, fracs, c)
        scale = float(np.sum(np.abs(img)))
        assert np.max(np.abs(recs[i, :nrad + 1] - ref[:nrad + 1])) <= 1e-14 * scale, (i, c)
        assert np.max(np.abs(recs[i, nrad + 1:] - ref[nrad + 1:]), initial=0.0) <= 1e-9, (i, c)


def assert_crossings(img, rec, radii, fracs, centre=None):
    """Every r_q is a radius where the oracle's EE crosses q TOTAL from below."""
    scale = float(np.sum(np.abs(img)))
    total = rec[len(radii)]
    for q, r in zip(fracs, rec[len(radii) + 1:]):
        target = q * total
        assert float(eo.ee(img, r, centre)) >= target - 1e-14 * scale, (q, r)
        assert float(eo.ee(img, r - 2e-10, centre)) < target + 1e-14 * scale, (q, r)


# ---------------------------------------------------------------- 1. image shapes
@pytest.mark.parametrize('shape', SHAPES, ids=['%dx%d' % s for s in SHAPES])
def test_image_shapes(psfrec, ctx, shape):
    ny, nx = shape
    cy, cx = ny // 2, nx // 2
    inner = min(cy + 0.5, ny - 0.5 - cy, cx + 0.5, nx - 0.5 - cx)      # largest disc about the centre inside
    rmax = rmax_of(ny, nx, cy, cx)
    radii = np.array([0.0, 0.25, 0.5, 0.7 * inner, inner, 0.5 * (inner + rmax), np.nextafter(rmax, 0), rmax + 1.0])
    rng = np.random.default_rng(100 * ny + nx)
    lit = np.zeros((ny, nx))
    lp, lq = int(rng.integers(0, ny)), int(rng.integers(0, nx))
    lit[lp, lq] = 1.5
    imgs = np.stack([np.ones((ny, nx)), lit, rng.random((ny, nx)), rng.random((ny, nx)) ** 4])
    rec = ee_of(ctx, imgs, radii, FRACS)
    nrad = len(radii)
    # uniform image: pi r^2 while the disc is inside, every pixel beyond the farthest corner
    assert rec[0, 0] == 0.0
    assert_allclose(rec[0, 1:5], np.pi * radii[1:5] ** 2, rtol=1e-13)
    assert rec[0, nrad] == ny * nx
    assert np.all(rec[:, nrad - 1] == rec[:, nrad])
    # one lit pixel: its overlap with the disc
    area = np.array([float(eo.pixel_area(lp - cy, lq - cx, r)) for r in radii])
    assert_allclose(rec[1, :nrad], 1.5 * area, rtol=1e-14, atol=1e-15)
    assert_parity(imgs, rec, radii, FRACS)
    # the default centre is (ny // 2, nx // 2), also on odd sizes
    assert np.array_equal(ee_of(ctx, imgs, radii, FRACS, np.tile([float(cy), float(cx)], (len(imgs), 1))), rec)

    # the Python surface: radii and r_ee in arcsec, centre per plane
    lbda = np.linspace(500., 900., len(imgs))
    radii_as = radii[:-2] * PIXSCALE
    rad_px = psfrec._ee_params(radii_as, FRACS)[0]
    centres = np.stack([cy + np.array([0.0, 0.3, -0.5, 1.25]), cx - np.array([0.0, 0.2, 0.5, 0.75])], axis=1)
    for center, cen in ((None, None), (centres, centres)):
        tab = psfrec.encircled_energy(lbda, imgs, radii_as, FRACS, center=center)
        ref = ee_of(ctx, imgs, rad_px, FRACS, cen)
        assert np.array_equal(tab['ee'], ref[:, :len(rad_px)]) and np.array_equal(tab['ee_total'], ref[:, len(rad_px)])
        assert np.array_equal(tab['r_ee'], ref[:, len(rad_px) + 1:] * PIXSCALE)
        assert np.array_equal(tab['lbda'], lbda)
        assert_allclose(tab.meta['radii'], radii_as, rtol=1e-15)
        assert_allclose(tab['r_ee'] / PIXSCALE, [[eo.r_at(img, q, None if cen is None else tuple(cen[i]))
                                                  for q in FRACS] for i, img in enumerate(imgs)], atol=1e-9)


# ---------------------------------------------------------------- 2. the shared-memory budget
@pytest.mark.parametrize('shape', [(64, 80), (80, 64)])
def test_largest_images(ctx, shape):
    """4 warps x 5120 pixels x (8 + 2) bytes = 200 KiB: the largest image the kernel takes."""
    ny, nx = shape
    rng = np.random.default_rng(ny)
    imgs = rng.random((3, ny, nx))
    centres = np.array([[ny // 2, nx // 2], [10.3, nx - 9.2], [ny - 1.0, 0.0]])
    radii = np.array([0.0, 1.5, 7.3, 20.0, 31.5, 45.0, 60.0, 110.0])      # 110 > hypot(80.5, 64.5) = 103.2
    rec = ee_of(ctx, imgs, radii, FRACS, centres)
    assert_parity(imgs, rec, radii, FRACS, centres)
    assert np.all(rec[:, 7] == rec[:, 8])


@pytest.mark.parametrize('shape', [(3, 1707), (71, 73)])
def test_too_large_images_refused(ctx, shape):
    import torch
    from muse_psfr_b200 import _lib
    ny, nx = shape
    imgs = np.ones((2, ny, nx))
    for out in (np.full((2, 4), 12345.0), torch.full((2, 4), 12345.0, dtype=torch.float64, device='cuda')):
        with pytest.raises(_lib.PsfrError, match='too large for the encircled-energy kernel') as exc:
            ctx.encircled_energy(2, ny, nx, imgs, np.array([1.0, 2.0]), np.array([0.5]), out)
        assert exc.value.code == _lib.E_UNSUPPORTED
        torch.cuda.synchronize()
        assert np.all(np.asarray(out.cpu() if hasattr(out, 'cpu') else out) == 12345.0)
    assert_allclose(ee_of(ctx, np.ones((1, 40, 40)), [2.0], [])[0, 0], 4 * np.pi, rtol=1e-14)


# ---------------------------------------------------------------- 3. staging in chunks
@pytest.mark.parametrize('shape', [(64, 64), (40, 40), (33, 50)])
def test_staging_across_chunks(psfrec, shape):
    """A context of 1 x 35 planes stages cap * 1600 / (ny * nx) host images at a time (13 of 64 x 64, 35 of
    40 x 40, 33 of 33 x 50).  Every mix of host and device images, centres and records gives the bits of one
    device-resident call on a context that holds all the images at once, and so do calls of one chunk each."""
    import torch
    from muse_psfr_b200 import _lib
    ny, nx = shape
    n = 200
    rng = np.random.default_rng(ny * nx)
    imgs = rng.random((n, ny, nx))
    cen = np.ascontiguousarray(np.stack([rng.uniform(-2, ny + 1, n), rng.uniform(-2, nx + 1, n)], axis=1))
    radii, fracs = np.array([0.7, 3.0, 9.5, 17.25, 30.0]), np.array([0.3, 0.5, 0.75])
    rec = len(radii) + 1 + len(fracs)
    big = _lib.Context(device=0, max_planes=16, max_lambda=35)
    small = _lib.Context(device=0, max_planes=1, max_lambda=35)
    try:
        chunk = min(35, 35 * 1600 // (ny * nx))
        assert chunk == {(64, 64): 13, (40, 40): 35, (33, 50): 33}[shape] and n > 5 * chunk
        assert 16 * 35 * 1600 // (ny * nx) >= n
        d_img, d_cen = torch.from_numpy(imgs).cuda(), torch.from_numpy(cen).cuda()
        ref = torch.full((n, rec), np.nan, dtype=torch.float64, device='cuda')
        big.encircled_energy(n, ny, nx, d_img, radii, fracs, ref, centres=d_cen)
        torch.cuda.synchronize()
        ref = ref.cpu().numpy()
        assert not np.isnan(ref).any()
        for img_dev, cen_dev, out_dev in itertools.product((False, True), repeat=3):
            out = (torch.full((n, rec), np.nan, dtype=torch.float64, device='cuda') if out_dev
                   else np.full((n, rec), np.nan))
            small.encircled_energy(n, ny, nx, d_img if img_dev else imgs, radii, fracs, out,
                                   centres=d_cen if cen_dev else cen)
            if out_dev:
                torch.cuda.synchronize()
                out = out.cpu().numpy()
            assert np.array_equal(out, ref), (img_dev, cen_dev, out_dev)
        parts = [ee_of(small, imgs[k:k + chunk], radii, fracs, cen[k:k + chunk]) for k in range(0, n, chunk)]
        assert np.array_equal(np.concatenate(parts), ref)
        edge = [0, chunk - 1, chunk, n - 1]
        assert_parity(imgs[edge], ref[edge], radii, fracs, cen[edge])
    finally:
        big.close()
        small.close()


def test_image_beyond_the_staging_buffer_refused(psfrec):
    from muse_psfr_b200 import _lib
    tiny = _lib.Context(device=0, max_planes=1, max_lambda=1)
    try:
        out = np.full((1, 3), 7.0)
        with pytest.raises(_lib.PsfrError) as exc:
            tiny.encircled_energy(1, 41, 41, np.ones((1, 41, 41)), np.array([1.0]), np.array([0.5]), out)
        assert exc.value.code == _lib.E_CAPACITY and np.all(out == 7.0)
        rec = ee_of(tiny, np.ones((3, 40, 40)), [1.0], [0.5])         # 40 x 40 fits, one image per chunk
        assert_allclose(rec[:, 0], np.pi, rtol=1e-14) and np.all(rec[:, 1] == 1600.0)
    finally:
        tiny.close()


# ---------------------------------------------------------------- 4. centres
def test_centres(ctx):
    ny, nx = 33, 50
    up, down = np.inf, -np.inf
    centres = np.array([
        (17.3, 22.65), (4.71, 41.09),                                        # off-grid
        (16.5, 24.5), (16.5, 25.0), (3.0, 40.5),                             # half-integers: pixel edges on the axes
        (0.5 + 1e-15, 0.5 - 1e-15), (np.nextafter(16.5, up), np.nextafter(24.5, down)),   # just off them
        (0.0, 0.0), (-0.5, 25.0), (32.5, 49.5), (32.0, 10.0), (16.0, -0.5), (16.0, 49.0),  # on the border
        (-5.0, 25.0), (ny + 4.0, 25.0), (16.0, -5.0), (16.0, nx + 4.0),     # 5 px outside
        (-1000.0, 25.0), (ny + 999.0, 25.0), (16.0, -1000.0), (16.0, nx + 999.0)])        # 1000 px outside
    radii = np.array([0.0, 0.5, 2.0, 5.5, 13.0, 30.0, 1000.0, 1012.5, 1030.0, 1060.0])
    rng = np.random.default_rng(31)
    imgs = rng.random((len(centres), ny, nx))
    rec = ee_of(ctx, imgs, radii, FRACS, centres)
    assert_parity(imgs, rec, radii, FRACS, centres)
    # a uniform image about a half-integer centre: pi r^2 while the disc is inside
    uni = ee_of(ctx, np.ones((3, ny, nx)), [0.5, 3.0, 7.25, 12.0], [], [[16.5, 24.5], [16.5, 25.0], [16.0, 24.5]])
    assert_allclose(uni[:, :4], np.tile(np.pi * np.array([0.5, 3.0, 7.25, 12.0]) ** 2, (3, 1)), rtol=1e-13)


FAR = [(1e8, 20.0), (-1e8, 20.0), (20.0, 3e9)]


def test_far_centres(ctx):
    """Centres 1e8 and 3e9 px away: the row window is empty for radii short of the image, not a wrapped int range.
    Exact answers only (the oracle's long double is not reliable at r ~ 1e8): EE = 0 short of the image, EE ==
    TOTAL beyond the farthest corner, r_q between the nearest pixel edge and the farthest corner."""
    import torch
    rng = np.random.default_rng(41)
    imgs = rng.random((len(FAR), 40, 40))
    for img, (y0, x0) in zip(imgs, FAR):
        near = max(abs(y0 - 19.5) - 20.0, abs(x0 - 19.5) - 20.0)         # distance to the nearest pixel edge
        far = rmax_of(40, 40, y0, x0)
        short = [0.0, 1.0, 1e3, near * (1 - 1e-9)]
        beyond = [far * (1 + 1e-9), 2 * far, 1e300]
        rec = ee_of(ctx, img[None], short + beyond, FRACS, np.array([[y0, x0]]))[0]
        total = rec[len(short) + len(beyond)]
        assert np.all(rec[:len(short)] == 0.0), (y0, x0)
        assert np.all(rec[len(short):len(short) + len(beyond)] == total), (y0, x0)
        assert total == ee_of(ctx, img[None], [], [])[0, 0]
        rq = rec[-len(FRACS):]
        assert np.all((rq >= near) & (rq <= far)), (y0, x0, rq)
    # timing guard: a few ms per far image (one B200: 3.7 ms, against 0.95 ms about its own centre; at r ~ 1e8
    # adjacent doubles lie further apart than the 1e-10 px tolerance, so each r_q takes the solve's 200 steps),
    # not the seconds of millions of warp trips over a window that wraps around
    d_img = torch.from_numpy(imgs[:1]).cuda()
    radii = np.array([1.0, 1e3, 2e8, 3e8])
    out = torch.empty((1, len(radii) + 1 + len(FRACS)), dtype=torch.float64, device='cuda')

    def timed(centre):
        cen = torch.tensor([centre], dtype=torch.float64, device='cuda')
        ctx.encircled_energy(1, 40, 40, d_img, radii, FRACS, out, centres=cen)        # warm-up
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        ctx.encircled_energy(1, 40, 40, d_img, radii, FRACS, out, centres=cen)
        t1.record()
        t1.synchronize()
        return t0.elapsed_time(t1)
    assert timed(list(FAR[0])) < 50.0                                   # ms
    assert timed(list(FAR[1])) < 50.0


# ---------------------------------------------------------------- 5. radii
def test_record_layout_at_the_limits(ctx):
    """64 radii and 16 fractions: EE slots equal a call with the radii alone, TOTAL sits at slot 64, r_q at 65..80."""
    rng = np.random.default_rng(51)
    imgs = rng.random((3, 40, 40)) ** 3
    radii = np.sort(rng.uniform(0, 32, 64))
    fracs = np.linspace(0.03, 0.97, 16)
    rec = ee_of(ctx, imgs, radii, fracs)
    assert rec.shape == (3, 81)
    alone = ee_of(ctx, imgs, radii, [])
    assert np.array_equal(rec[:, :65], alone)
    assert np.array_equal(rec[:, 64], ee_of(ctx, imgs, [], [])[:, 0])
    assert_parity(imgs, rec, radii, fracs)
    assert np.max(np.abs(rec[:, 65:] - ee_of(ctx, imgs, [], fracs)[:, 1:])) <= 1e-10


def test_tangent_and_corner_radii_off_grid(ctx):
    y0, x0 = 17.3, 22.65
    tangent = [abs(k + s - y0) for k in (14, 17, 18, 25) for s in (-0.5, 0.5)] + \
              [abs(m + s - x0) for m in (16, 22, 23, 30) for s in (-0.5, 0.5)]
    corner = [np.hypot(k - y0, m - x0) for k in (16.5, 17.5, 19.5, 24.5) for m in (18.5, 22.5, 23.5, 29.5)]
    radii = np.array(sorted(tangent + corner))
    assert radii.size <= 64 and radii.max() < 16.85          # 16.85: the largest disc inside the image
    rng = np.random.default_rng(52)
    imgs = np.stack([np.ones((40, 40)), rng.random((40, 40))])
    cen = np.array([[y0, x0]] * 2)
    rec = ee_of(ctx, imgs, radii, FRACS, cen)
    assert_allclose(rec[0, :radii.size], np.pi * radii ** 2, rtol=1e-13)
    assert_parity(imgs, rec, radii, FRACS, cen)


def test_extreme_radii(ctx):
    """1e-300, 1e300 and the neighbours of the farthest-corner distance: above it EE == TOTAL bit for bit."""
    rng = np.random.default_rng(53)
    imgs = rng.random((2, 40, 40))
    rmax = rmax_of(40, 40, 20, 20)
    radii = np.array([1e-300, np.nextafter(rmax, 0), rmax, np.nextafter(rmax, np.inf), 1e300])
    rec = ee_of(ctx, imgs, radii, FRACS)
    assert np.all(rec[:, 0] == 0.0)
    assert np.all(rec[:, 3] == rec[:, 5]) and np.all(rec[:, 4] == rec[:, 5])
    # the oracle's arcsin form loses the area at r ~ 1e20 and beyond: parity up to the corner's neighbours
    assert_parity(imgs, np.delete(rec, 4, axis=1), radii[:4], FRACS)
    cen = np.array([[17.3, 22.65]] * 2)
    rmax = rmax_of(40, 40, 17.3, 22.65)
    radii = np.array([1e-300, np.nextafter(rmax, 0), rmax, np.nextafter(rmax, np.inf), 1e300])
    rec = ee_of(ctx, imgs, radii, FRACS, cen)
    assert np.all(rec[:, 4] == rec[:, 5])
    assert_parity(imgs, np.delete(rec, 4, axis=1), radii[:4], FRACS, cen)


def test_unsorted_and_duplicated_radii(ctx):
    """Permuting the radii permutes the EE slots bit for bit and leaves every r_q's bits, on positive images and
    on images with negative pixels."""
    rng = np.random.default_rng(54)
    imgs = np.stack([rng.random((40, 40)), rng.random((40, 40)) ** 6, rng.normal(0.3, 1.0, (40, 40))])
    radii = np.array([5.0, 1.0, 12.5, 5.0, 0.0, 30.0, 1.0, 7.7, 2.2, 12.5, 3.3])
    fracs = np.array([0.1, 0.5, 0.8, 0.95])
    base = ee_of(ctx, imgs, radii, fracs)
    for p in [np.arange(radii.size)[::-1]] + [rng.permutation(radii.size) for _ in range(5)]:
        rec = ee_of(ctx, imgs, radii[p], fracs)
        assert np.array_equal(rec[:, :radii.size], base[:, p])
        assert np.array_equal(rec[:, radii.size:], base[:, radii.size:])
    assert np.all(base[:, 0] == base[:, 3]) and np.all(base[:, 1] == base[:, 6])


def test_fraction_radius_without_tabulated_radii(ctx):
    rng = np.random.default_rng(55)
    imgs = np.stack([rng.random((40, 40)), rng.random((40, 40)) ** 4, np.ones((40, 40))])
    radii = np.linspace(0.4, 27.0, 20)
    with_r = ee_of(ctx, imgs, radii, FRACS)[:, radii.size + 1:]
    without = ee_of(ctx, imgs, [], FRACS)[:, 1:]
    assert np.max(np.abs(with_r - without)) <= 1e-10


# ---------------------------------------------------------------- 6. fractions
def square_ee(r, a):
    """EE of the uniform square [-a, a]^2 (unit pixels) about its centre, for a <= r <= a sqrt(2), in mpmath."""
    import mpmath as mp
    xa = mp.sqrt(r * r - a * a)
    return 4 * (a * xa + r * r * (mp.asin(a / r) - mp.asin(xa / r)) / 2)


def test_fractions_next_to_zero_and_one(ctx):
    """q = 1e-12 and 1 - 1e-12 on a uniform 3 x 3 image about its centre: r = sqrt(q 9 / pi) inside the centre
    pixel, and near the corners r where the square minus its four corner caps holds q 9."""
    import mpmath as mp
    mp.mp.dps = 40
    fracs = np.array([1e-12, 1 - 1e-12])
    rec = ee_of(ctx, np.ones((1, 3, 3)), [], fracs)[0]
    assert rec[0] == 9.0
    assert abs(rec[1] - np.sqrt(fracs[0] * 9.0 / np.pi)) <= 1e-9
    target = mp.mpf(float(fracs[1] * 9.0))              # q TOTAL as the kernel forms it
    a, lo, hi = mp.mpf(1.5), mp.mpf(1.5), mp.sqrt(2) * mp.mpf(1.5)
    for _ in range(140):
        mid = (lo + hi) / 2
        lo, hi = (mid, hi) if square_ee(mid, a) < target else (lo, mid)
    assert abs(rec[2] - float(hi)) <= 1e-9
    assert_parity(np.ones((1, 3, 3)), rec[None], [], fracs)
    # 40 x 40: near 1 the single farthest corner is cut off, and 1e-13 of rounding in EE moves r by 2e-9 px there
    big = ee_of(ctx, np.ones((1, 40, 40)), [1.0, 10.0], fracs[:1])[0]
    assert abs(big[3] - np.sqrt(1e-12 * 1600.0 / np.pi)) <= 1e-9
    assert_parity(np.ones((1, 40, 40)), big[None], [1.0, 10.0], fracs[:1])


def test_target_equal_to_a_tabulated_ee(ctx):
    """Two lit pixels of 1, q = 0.5: EE = 1 = q TOTAL exactly at r = 5, and on all of [sqrt(1/2), 9.5].  r_q is
    the left end sqrt(1/2), where the first pixel is covered, not the tabulated 5.  EE meets the plateau with a
    quadratic contact at the pixel's corners, so FP64 reaches it up to 1e-8 px early."""
    img = np.zeros((1, 40, 40))
    img[0, 20, 20] = img[0, 20, 30] = 1.0
    for radii in ([5.0], [5.0, 12.0], [12.0, 0.3, 5.0], []):
        rec = ee_of(ctx, img, radii, [0.5])[0]
        if radii:
            assert rec[radii.index(5.0)] == 1.0
        r = rec[-1]
        assert np.sqrt(0.5) - 1e-8 <= r <= np.sqrt(0.5) + 1e-10, (radii, r)
        assert_crossings(img[0], rec, radii, [0.5])


def test_target_on_a_plateau(ctx):
    """Eight pixels of 1/8 about (20, 20), zero pixels out to d = 6.4, eight more of 1/8 beyond: EE is flat at 1 =
    TOTAL / 2 from hypot(1.5, 1.5) (the corners of the inner block) to 6.36 (the nearest corner of the outer
    ones).  r_50 is the plateau's left end whatever radii are tabulated on it."""
    img = np.zeros((40, 40))
    img[19:22, 19:22] = 0.125
    img[20, 20] = 0.0
    for p, q in ((13, 20), (27, 20), (20, 13), (20, 27), (15, 15), (25, 25), (15, 25), (25, 15)):
        img[p, q] = 0.125
    left = np.hypot(1.5, 1.5)
    for radii in ([1.0, 4.0, 6.0, 10.0], [10.0, 6.0, 4.0, 1.0], [3.0], [2.5, 2.2, 6.3], []):
        rec = ee_of(ctx, img[None], radii, [0.5])[0]
        assert rec[len(radii)] == 2.0
        assert all(e == 1.0 for r, e in zip(radii, rec) if left <= r <= 6.3)
        assert left - 1e-7 <= rec[-1] <= left + 1e-10, (radii, rec[-1])
        assert_crossings(img, rec, radii, [0.5])


# ---------------------------------------------------------------- 7. negative pixels
def worked_example():
    """1.0 at (20, 20), -0.8 spread over the ring 4.5 < d < 5.5 and +0.8 over 9.5 < d < 10.5: EE rises to 1 by
    r = sqrt(1/2), falls to 0.2 across the first ring and comes back to 1 across the second."""
    img = np.zeros((40, 40))
    img[20, 20] = 1.0
    p, q = np.mgrid[:40, :40]
    d = np.hypot(p - 20, q - 20)
    inner, outer = (d > 4.5) & (d < 5.5), (d > 9.5) & (d < 10.5)
    img[inner] = -0.8 / inner.sum()
    img[outer] = 0.8 / outer.sum()
    return img


def test_negative_pixels_worked_example(ctx):
    """With radii [2, 7] (EE 1.0 and 0.2) the solve starts from [0, 2], where EE crosses 0.5 once, at
    sqrt(0.5 / pi) = 0.3989: r_50 is that smallest crossing, not the tabulated 2."""
    from scipy.optimize import brentq
    img = worked_example()
    first = brentq(lambda r: float(eo.ee(img, r) - eo.LD(0.5) * np.sum(np.asarray(img, dtype=eo.LD))), 0.0, 0.7,
                   xtol=1e-14, rtol=1e-15)
    assert abs(first - np.sqrt(0.5 / np.pi)) < 1e-12
    for radii in ([2.0, 7.0], [7.0, 2.0], [7.0, 2.0, 7.0, 0.2], [2.0, 7.0, 12.0]):
        rec = ee_of(ctx, img[None], radii, [0.5])[0]
        assert abs(rec[-1] - first) <= 1e-9, (radii, rec[-1])
        assert_crossings(img, rec, radii, [0.5])
    rec = ee_of(ctx, img[None], [], FRACS)[0]            # [0, farthest corner]: one of the crossings
    assert_crossings(img, rec, [], FRACS)


def test_negative_pixels_random(ctx):
    rng = np.random.default_rng(71)
    imgs = np.stack([rng.normal(0.3, 1.0, (40, 40)), rng.normal(0.1, 1.0, (40, 40)), rng.random((40, 40)) - 0.45])
    fracs = np.array([0.05, 0.2, 0.5, 0.8, 0.95])
    radii = np.array([9.0, 2.0, 14.5, 2.0, 0.0, 21.0, 5.5, 30.0, 3.7])
    cen = np.array([[20.0, 20.0], [17.3, 22.65], [25.5, 10.0]])
    rec = ee_of(ctx, imgs, radii, fracs, cen)
    for i, img in enumerate(imgs):
        assert rec[i, radii.size] > 0
        ref = eo.record(img, radii, [], tuple(cen[i]))
        assert np.max(np.abs(rec[i, :radii.size + 1] - ref)) <= 1e-14 * np.sum(np.abs(img))
        assert_crossings(img, rec[i], radii, fracs, tuple(cen[i]))
        bare = ee_of(ctx, img[None], [], fracs, cen[i:i + 1])[0]
        assert_crossings(img, bare, [], fracs, tuple(cen[i]))


def test_nonpositive_totals(ctx):
    rng = np.random.default_rng(72)
    zero = np.zeros((40, 40))
    zero[10, 10], zero[30, 25] = 1.0, -1.0
    imgs = np.stack([-rng.random((40, 40)), zero, np.zeros((40, 40))])
    radii = np.array([0.0, 3.0, 15.0, 40.0])
    rec = ee_of(ctx, imgs, radii, FRACS)
    assert np.all(np.isnan(rec[:, radii.size + 1:]))
    assert rec[1, radii.size] == 0.0 and rec[2, radii.size] == 0.0
    for i, img in enumerate(imgs):
        ref = eo.record(img, radii, [])
        assert np.max(np.abs(rec[i, :radii.size + 1] - ref)) <= 1e-14 * max(np.sum(np.abs(img)), 1.0)


# ---------------------------------------------------------------- 8. contexts and streams
def test_contexts_with_different_image_sizes(psfrec):
    """The dynamic shared-memory limit of a kernel is one setting of the process, not of a context: a context that
    first sees small images must not lower it under another context that has already raised it for large ones.
    Context a raises ee_kernel's limit for 64 x 80 images and fit_kernel's for 64 x 64, b then runs 40 x 40
    images, and a runs sizes between the two."""
    from muse_psfr_b200 import _lib
    a = _lib.Context(device=0, max_planes=1, max_lambda=35)
    b = _lib.Context(device=0, max_planes=1, max_lambda=35)
    try:
        rng = np.random.default_rng(91)
        ee_of(a, rng.random((2, 64, 80)), [3.0], [0.5])
        fit = np.empty((2, _lib.FIT_NPAR))
        a.moffat_fit(2, 64, 64, rng.random((2, 64, 64)), fit)
        ee_of(b, rng.random((2, 40, 40)), [3.0], [0.5])
        b.moffat_fit(2, 40, 40, rng.random((2, 40, 40)), fit)
        imgs = rng.random((3, 33, 50))
        assert np.array_equal(ee_of(a, imgs, [3.0, 9.0], FRACS), ee_of(b, imgs, [3.0, 9.0], FRACS))
        p, q = np.mgrid[:41, :41]
        moffat = np.stack([(1 + ((p - 20.3) ** 2 + (q - 19.6) ** 2) / w ** 2) ** -2.5 for w in (3.0, 4.0)])
        fa, fb = np.empty((2, _lib.FIT_NPAR)), np.empty((2, _lib.FIT_NPAR))
        a.moffat_fit(2, 41, 41, moffat, fa)
        b.moffat_fit(2, 41, 41, moffat, fb)
        assert np.array_equal(fa, fb)
    finally:
        a.close()
        b.close()



def test_side_stream(ctx):
    import torch
    rng = np.random.default_rng(81)
    imgs = torch.from_numpy(rng.random((300, 33, 50))).cuda()
    cen = torch.from_numpy(np.stack([rng.uniform(0, 33, 300), rng.uniform(0, 50, 300)], axis=1)).cuda()
    radii, fracs = np.array([0.5, 4.0, 11.0, 25.0]), np.array([0.5, 0.8])
    ref = torch.full((300, 7), np.nan, dtype=torch.float64, device='cuda')
    ctx.encircled_energy(300, 33, 50, imgs, radii, fracs, ref, centres=cen)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        out = torch.full((300, 7), np.nan, dtype=torch.float64, device='cuda')
        ctx.encircled_energy(300, 33, 50, imgs, radii, fracs, out, centres=cen, stream=side.cuda_stream)
    side.synchronize()
    assert torch.equal(out, ref)
