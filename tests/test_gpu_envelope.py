"""GPU tests at the edges of the kernels' envelope: the ends of the crop-width range, the size of the
per-wavelength tables staged in shared memory, the underflow cut at dim 2560, batches of many draws
times many directions across chunk boundaries, stage A beyond plane 0, and the staging paths of the
small kernels (fit, mean + refit, convolve, polynomial fit).

Conventions of tests/test_gpu_parity.py: PSF images agree with the oracle to relative 1e-9
(``assert_image_close``), two paths of this library to 1e-13 of the peak, fits to ``FIT_RTOL``, and
runs that must not depend on batching are compared bit for bit.
"""
import numpy as np
import pytest
from numpy.testing import assert_allclose

import psfr_oracle as orc

pytestmark = pytest.mark.gpu

LBDA35 = np.linspace(490, 930, 35)
PSF_RTOL = 1e-9      # PSF images to relative 1e-9
FIT_RTOL = 1e-5      # FWHM / beta to relative 1e-5
CROP = 40 * 0.2 * 2 * 8 * 4.85 * 1000       # npix = CROP / lambda_nm, rounded to even (psfrec.py:663-664)
BAD_SEEING = ([0.36, 0.64], (100, 10000), 1.68, 19.9)     # cut, both precision grades and dead row pairs occur


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
def psd1():
    return orc.simul_psd_wfm([0.7, 0.3], (100, 10000), 1.0, 25.)[0]


@pytest.fixture(scope='module')
def bad1():
    return orc.simul_psd_wfm(*BAD_SEEING)[0]


@pytest.fixture(scope='module')
def psd5(psfrec):
    return psfrec.simul_psd_wfm([0.7, 0.3], (100, 10000), 1.0, 25., dim=2560, verbose=False)[0]


@pytest.fixture(scope='module')
def bad5(psfrec):
    return psfrec.simul_psd_wfm(*BAD_SEEING, dim=2560, verbose=False)[0]


def rel_to_peak(got, ref):
    return np.abs(np.asarray(got) - np.asarray(ref)).max() / np.abs(ref).max()


def assert_image_close(got, ref, rtol=PSF_RTOL, floor=1e-6):
    """Relative 1e-9: every pixel above `floor` (1e-6) of the peak agrees to rtol pointwise, and
    the whole image agrees to rtol of the peak."""
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape
    assert np.isfinite(got).all()
    assert rel_to_peak(got, ref) < rtol
    sig = np.abs(ref) > floor * np.abs(ref).max()
    assert_allclose(got[sig], ref[sig], rtol=rtol, atol=0)


FP64_OPTS = 'fp64'


def resolve(opts):
    from muse_psfr_b200 import _lib
    if isinstance(opts, str) and opts == FP64_OPTS:
        return {_lib.OPT_EXP_GRADE: 1e30, _lib.OPT_F32_ROWS: 1e30}
    return dict(opts or {})


def run_with(ctx, opts, fn):
    """fn() with context options set (PSFR_OPT_* -> value), restored afterwards.  FP64_OPTS turns
    both single-precision grades off."""
    from muse_psfr_b200 import _lib
    opts = resolve(opts)
    names = {_lib.OPT_EXP_CUT: 'exp_cut', _lib.OPT_EXP_GRADE: 'exp_grade', _lib.OPT_F32_ROWS: 'f32_rows',
             _lib.OPT_ROW_KERNEL: 'row_kernel'}
    saved = ctx.info()
    try:
        for k, v in opts.items():
            ctx.set_option(k, v)
        return fn()
    finally:
        for k in opts:
            ctx.set_option(k, saved[names[k]])


def both_row_kernels(psfrec, psd, lam, dim=1280, opts=None):
    """psf_muse with row kernel 2 (default) and row kernel 1."""
    from muse_psfr_b200 import _lib
    ctx = psfrec.get_context(dim=dim)
    opts = resolve(opts)
    got2 = run_with(ctx, opts, lambda: psfrec.psf_muse(psd, lam))
    got1 = run_with(ctx, {**opts, _lib.OPT_ROW_KERNEL: 1}, lambda: psfrec.psf_muse(psd, lam))
    assert ctx.info()['row_kernel'] == 2
    return got2, got1


def exponent_at(ctx, lam_nm, rows):
    """c_lambda * min over each structure-function row of plane 0: the exponent of the row's largest
    OTF entry relative to the peak (the row kernel's classification)."""
    d = ctx.get_structure_function(0)
    return 0.5 * (2 * np.pi / lam_nm) ** 2 * d[:rows].min(axis=1)


# ---------------------------------------------------------------- 1. crop width limits
CROPS = {1280: [1280, 82, 126, 310, 80], 2560: [2560, 126, 80]}


@pytest.mark.parametrize('dim', [1280, 2560])
def test_crop_width_limits(psfrec, psd1, psd5, dim):
    """npix == dim (the crop is the whole grid, sample indices wrap modulo N), npix == 80 (every
    bilinear fraction is 0, every second sample is dead) and small odd-ratio crops between them."""
    psd = psd1 if dim == 1280 else psd5
    lam = CROP / np.array(CROPS[dim], dtype=float)
    assert list(orc.npixc_of(lam)) == CROPS[dim]
    got2, got1 = both_row_kernels(psfrec, psd, lam, dim)
    assert rel_to_peak(got1, got2) < 1e-13
    ref = orc.psf_muse(psd, lam)
    for k in range(lam.size):
        assert_image_close(got2[k], ref[k])
        assert_image_close(got1[k], ref[k])


def test_full_grid_crop_bad_seeing(psfrec, bad1):
    lam = np.array([485.0])
    assert orc.npixc_of(lam)[0] == 1280
    got2, got1 = both_row_kernels(psfrec, bad1, lam)
    assert rel_to_peak(got1, got2) < 1e-13
    ref = orc.psf_muse(bad1, lam)
    assert_image_close(got2[0], ref[0])
    assert_image_close(got1[0], ref[0])


def test_crop_width_refusals(psfrec, psd1, psd5):
    """Beyond the grid (the oracle is no reference there: its crop slice degenerates and broadcasts)
    and below 80 pixels (2 samples per output pixel) the library refuses the wavelength."""
    assert orc.npixc_of(484.5)[0] == 1282 and orc.npixc_of(242.4)[0] == 2562 and orc.npixc_of(7960.)[0] == 78
    with pytest.raises(ValueError, match='1282-pixel crop but dim is 1280'):
        psfrec.psf_muse(psd1, np.array([600., 484.5]))
    with pytest.raises(ValueError, match='2562-pixel crop but dim is 2560'):
        psfrec.psf_muse(psd5, np.array([242.4]))
    for psd in (psd1, psd5):
        with pytest.raises(ValueError, match='78-pixel crop, fewer than the 80 samples per axis'):
            psfrec.psf_muse(psd, np.array([7960.]))
    # the context is still usable after a refusal
    assert np.isfinite(psfrec.psf_muse(psd1, np.array([7760.]))).all()


# ---------------------------------------------------------------- 2. wavelength tables and precision classes
@pytest.mark.parametrize('nlam', [64, 65, 300])
def test_wavelength_table_sizes(psfrec, bad1, nlam):
    """Per-wavelength scalars are staged in shared memory for nlam <= 64 and read from global memory
    above: on the bad-seeing PSD (cut, FP32 rows and the FP32 exp all occur) every size must agree
    with one-wavelength calls, with the all-FP64 options, between the row kernels and with the oracle."""
    rng = np.random.default_rng(nlam)
    lam = rng.permutation(np.linspace(488., 1050., nlam))
    ctx = psfrec.get_context(max_lambda=nlam)
    got2, got1 = both_row_kernels(psfrec, bad1, lam)
    assert got2.shape == (nlam, 40, 40) and np.isfinite(got2).all()
    assert rel_to_peak(got1, got2) < 1e-13
    fp2, fp1 = both_row_kernels(psfrec, bad1, lam, opts=FP64_OPTS)
    assert rel_to_peak(fp2, got2) < 1e-13
    assert rel_to_peak(fp1, got2) < 1e-13
    # the single-precision class really ran at the shortest wavelength: some row lies entirely between
    # the FP32 threshold (e^-25) and the cut (e^-45), and some row entirely below the cut
    x = exponent_at(ctx, lam.min(), 641)
    assert ((x >= 25) & (x <= 45)).any() and (x > 45).any()
    picks = sorted({0, 1, nlam // 3, nlam // 2, nlam - 1, int(np.argmin(lam)), int(np.argmax(lam))})
    for k in picks:
        one2, one1 = both_row_kernels(psfrec, bad1, lam[[k]])
        assert rel_to_peak(got2[k], one2[0]) < 1e-13
        assert rel_to_peak(got1[k], one1[0]) < 1e-13
    sel = [int(np.argmin(lam)), nlam // 2]
    ref = orc.psf_muse(bad1, lam[sel])
    for i, k in enumerate(sel):
        assert_image_close(got2[k], ref[i])
        assert_image_close(got1[k], ref[i])


@pytest.mark.parametrize('filler', [0, 62])
def test_duplicated_wavelengths(psfrec, bad1, filler):
    """Equal wavelengths sort next to each other; in the single-precision class two of them run as
    the two halves of one packed transform.  Duplicates must give bit-identical planes, with the
    tables staged (8 wavelengths) and not staged (70)."""
    dup = np.array([490., 490., 490., 640., 700., 640., 930., 930.])
    lam = np.concatenate([dup, np.linspace(500., 920., filler)])
    groups = ([0, 1, 2], [3, 5], [6, 7])
    ctx = psfrec.get_context(max_lambda=lam.size)
    got2, got1 = both_row_kernels(psfrec, bad1, lam)
    x = exponent_at(ctx, 490., 641)
    assert ((x >= 25) & (x <= 45)).any()
    for got in (got2, got1):
        for g in groups:
            for k in g[1:]:
                assert np.array_equal(got[k], got[g[0]]), (g, k)
    assert rel_to_peak(got1, got2) < 1e-13
    uniq2, uniq1 = both_row_kernels(psfrec, bad1, np.array([490., 640., 700., 930.]))
    assert rel_to_peak(got2[[0, 3, 4, 6]], uniq2) < 1e-13
    assert rel_to_peak(got1[[0, 3, 4, 6]], uniq1) < 1e-13
    ref = orc.psf_muse(bad1, np.array([490.]))
    assert_image_close(got2[1], ref[0])


# ---------------------------------------------------------------- 3. underflow cut at dim 2560
def test_underflow_cut_dim2560(psfrec, bad5):
    """dim 2560 (group row kernel on two 1280-point sub-transforms): the cut at e^-45 against the cut
    disabled, both against the oracle, and the two row kernels against each other."""
    from muse_psfr_b200 import _lib
    lam = np.array([490., 640., 930.])
    ctx = psfrec.get_context(dim=2560)
    assert ctx.info()['exp_cut'] == 45.0
    full = run_with(ctx, {_lib.OPT_EXP_CUT: 1000.0}, lambda: psfrec.psf_muse(bad5, lam))
    cut2, cut1 = both_row_kernels(psfrec, bad5, lam, dim=2560)
    # whole row pairs lie below the cut at 490 nm: the skip really ran
    x = exponent_at(ctx, 490., 1281)
    assert (np.minimum(x[0:1280:2], x[1:1281:2]) > 45).any()
    assert ctx.info()['exp_cut'] == 45.0
    assert rel_to_peak(cut2, full) < 1e-13
    assert rel_to_peak(cut1, cut2) < 1e-13
    ref = orc.psf_muse(bad5, lam)
    for k in range(lam.size):
        assert_image_close(cut2[k], ref[k])
        assert_image_close(full[k], ref[k])


# ---------------------------------------------------------------- 4. many draws x many directions
DRAWS7 = (np.array([0.5, 0.8, 1.1, 1.4, 1.7, 2.0, 0.65]), np.array([0.9, 0.35, 0.6, 0.75, 0.45, 0.8, 0.5]),
          np.array([10., 27., 15., 22., 12., 18., 28.]))


def fresh_batch_context(psfrec, max_planes, dim=1280):
    """Contexts are cached and only grow: start from a fresh one whose capacity sets the chunking."""
    psfrec.release_contexts()
    return psfrec.get_context(max_planes=max_planes, dim=dim)


@pytest.mark.parametrize('three', [True, False])
def test_many_draws_many_directions(psfrec, three):
    """7 draws x 9 directions with max_planes = 20: 2 draws (18 planes) per chunk, a partial last
    chunk, host outputs.  The column kernel averages plane draw * ndir + d: every draw must equal its
    own one-draw call bit for bit, and two draws the oracle."""
    from muse_psfr_b200 import _lib
    s, g, l0 = DRAWS7
    lam = LBDA35[::6]
    ctx = fresh_batch_context(psfrec, 20)
    fit, cube = psfrec.compute_psf_batch(lam, s, g, l0, npsflin=3, three_lgs_mode=three, max_planes=20)
    assert ctx.info()['max_planes'] == 20
    assert np.isfinite(cube).all() and np.all(fit[:, :, _lib.FIT_ITER] > 0)
    for i in range(s.size):
        f1, c1 = psfrec.compute_psf_batch(lam, s[[i]], g[[i]], l0[[i]], npsflin=3, three_lgs_mode=three,
                                          max_planes=20)
        assert np.array_equal(cube[i], c1[0]), i
        assert np.array_equal(fit[i], f1[0]), i
    assert ctx.info()['max_planes'] == 20
    i = 1 if three else 6             # second draw of the first chunk / the draw of the partial last chunk
    sel = [0, lam.size - 1]
    ref, ref_cube = orc.compute_psf(lam[sel], s[i], g[i], l0[i], npsflin=3, three_lgs_mode=three)
    for j, k in enumerate(sel):
        assert_image_close(cube[i, k], ref_cube[j])
    assert_allclose(fit[i, sel, _lib.FIT_FWHM] * 0.2, ref['fwhm'], rtol=FIT_RTOL)
    assert_allclose(fit[i, sel, _lib.FIT_N], ref['n'], rtol=FIT_RTOL)
    psfrec.release_contexts()


def test_many_draws_many_directions_dim2560(psfrec):
    """dim 2560, 2 x 2 directions, max_planes = 10 (2 draws per chunk, 10 % 4 != 0), 5 draws."""
    s, g, l0 = (v[:5] for v in DRAWS7)
    lam = np.array([500., 700., 900.])
    ctx = fresh_batch_context(psfrec, 10, dim=2560)
    fit, cube = psfrec.compute_psf_batch(lam, s, g, l0, npsflin=2, max_planes=10, dim=2560)
    assert ctx.info()['max_planes'] == 10
    assert np.isfinite(cube).all()
    for i in range(s.size):
        f1, c1 = psfrec.compute_psf_batch(lam, s[[i]], g[[i]], l0[[i]], npsflin=2, max_planes=10, dim=2560)
        assert np.array_equal(cube[i], c1[0]), i
        assert np.array_equal(fit[i], f1[0]), i
    psfrec.release_contexts()


def test_mixed_device_and_host_outputs(psfrec):
    """One output on the device and the other on the host, over 4 chunks: the host output leaves
    through the copy stream from alternating staging buffers while the device output is written in
    place.  Both must be bit-identical to the all-host call."""
    import torch
    from muse_psfr_b200 import _lib
    s, g, l0 = DRAWS7
    lam = LBDA35[::6]
    fresh_batch_context(psfrec, 20)
    kw = dict(npsflin=3, max_planes=20)
    fit_h, cube_h = psfrec.compute_psf_batch(lam, s, g, l0, **kw)
    shape_c, shape_f = cube_h.shape, fit_h.shape
    d_cube = torch.full(shape_c, np.nan, dtype=torch.float64, device='cuda')
    h_fit = np.full(shape_f, np.nan)
    psfrec.compute_psf_batch(lam, s, g, l0, out_cube=d_cube, out_fit=h_fit, **kw)
    torch.cuda.synchronize()
    assert np.array_equal(d_cube.cpu().numpy(), cube_h)
    assert np.array_equal(h_fit, fit_h)
    h_cube = np.full(shape_c, np.nan)
    d_fit = torch.full(shape_f, np.nan, dtype=torch.float64, device='cuda')
    psfrec.compute_psf_batch(lam, s, g, l0, out_cube=h_cube, out_fit=d_fit, **kw)
    torch.cuda.synchronize()
    assert np.array_equal(h_cube, cube_h)
    assert np.array_equal(d_fit.cpu().numpy(), fit_h)
    assert psfrec.get_context().info()['max_planes'] == 20
    assert np.all(fit_h[:, :, _lib.FIT_ITER] > 0)
    psfrec.release_contexts()


# ---------------------------------------------------------------- 5. stage A beyond plane 0
@pytest.mark.parametrize('dim', [1280, 2560])
def test_structure_function_every_plane(psfrec, dim):
    """Three distinct PSDs in one call: the structure function of every plane, and the full-grid PSF
    of plane 2, against the oracle."""
    psd = np.ascontiguousarray(np.stack([
        psfrec.simul_psd_wfm([0.7, 0.3], (100, 10000), 1.0, 25., dim=dim, verbose=False)[0],
        psfrec.simul_psd_wfm(*BAD_SEEING, dim=dim, verbose=False)[0],
        psfrec.simul_psd_wfm([0.5, 0.5], (250, 12000), 0.6, 11., dim=dim, verbose=False)[0]]))
    h = dim // 2
    ctx = psfrec.get_context(dim=dim)
    ctx.load_psd(psd, 3)
    ctx.structure_function(3)
    for p in range(3):
        d = ctx.get_structure_function(p)
        ref = orc.structure_function_unit(psd[p])
        assert rel_to_peak(d[:h + 1], ref.T[:h + 1]) < 1e-13, p
        assert d[h, h] == 0.0 and np.all(d[h + 1] == 0), p
    lb = 640e-9
    out = np.empty((dim, dim))
    ctx.psd_to_psf(2, lb, out)
    ref = orc.psd_to_psf(psd[2], orc.pupil_mask(dim // 4, dim // 2, 0.14), 8, lb)
    assert rel_to_peak(out, ref) < 1e-13
    # at 2560 the two FP64 transforms differ by ~1e-15 of the peak: pointwise bar from 1e-5 of the peak
    assert_image_close(out, ref, floor=1e-6 if dim == 1280 else 1e-5)
    assert_allclose(out.sum(), 1.0, rtol=1e-12)


# ---------------------------------------------------------------- 6. staging paths of the small kernels
def moffat_images(rng, n, ny, nx, noise=0.0):
    """n Moffat images of random parameters [peak, y0, x0, alpha, n] near the image centre."""
    p, q = np.mgrid[:ny, :nx].astype(float)
    scale = min(ny, nx) / 40.
    truth = np.stack([rng.uniform(0.02, 0.2, n), (ny - 1) / 2 + rng.uniform(-1, 1, n) * scale,
                      (nx - 1) / 2 + rng.uniform(-1, 1, n) * scale, rng.uniform(2.0, 4.0, n) * max(scale, 0.5),
                      rng.uniform(1.6, 3.5, n)], axis=1)
    imgs = np.stack([orc.moffat_model(v, p, q) for v in truth])
    if noise:
        imgs += noise * truth[:, :1, None] * rng.standard_normal(imgs.shape)
    return np.ascontiguousarray(imgs), truth


def assert_fit_matches_truth(fit, truth, rtol=1e-8):
    from muse_psfr_b200 import _lib
    assert np.all(fit[:, _lib.FIT_ITER] > 0)
    assert_allclose(fit[:, _lib.FIT_PEAK], truth[:, 0], rtol=rtol)
    assert_allclose(fit[:, _lib.FIT_Y0], truth[:, 1], rtol=rtol)
    assert_allclose(fit[:, _lib.FIT_X0], truth[:, 2], rtol=rtol)
    assert_allclose(fit[:, _lib.FIT_N], truth[:, 4], rtol=rtol)
    fwhm = truth[:, 3] * 2 * np.sqrt(2 ** (1 / truth[:, 4]) - 1)
    assert_allclose(fit[:, _lib.FIT_FWHM], fwhm, rtol=rtol)


@pytest.fixture
def own_context(psfrec):
    """A context of default capacity (16 planes x 35 wavelengths: 560 staged 40 x 40 images)."""
    from muse_psfr_b200 import _lib
    ctx = _lib.Context(device=0, max_planes=16, max_lambda=35)
    yield ctx
    ctx.close()


def test_fit_more_images_than_one_chunk(own_context):
    """1300 host images go through the 560-image staging buffer in three chunks: the result must be
    bit-identical to fitting the same images in slices of one chunk each, and right."""
    from muse_psfr_b200 import _lib
    ctx = own_context
    rng = np.random.default_rng(5)
    n = 1300
    clean, truth = moffat_images(rng, n, 40, 40)
    noisy, _ = moffat_images(np.random.default_rng(5), n, 40, 40, noise=1e-3)
    imgs = np.ascontiguousarray(np.where((np.arange(n) % 2 == 0)[:, None, None], clean, noisy))
    fit = np.full((n, _lib.FIT_NPAR), np.nan)
    ctx.moffat_fit(n, 40, 40, imgs, fit)
    sliced = np.full_like(fit, np.nan)
    for i0 in range(0, n, 500):
        m = min(500, n - i0)
        out = np.empty((m, _lib.FIT_NPAR))
        ctx.moffat_fit(m, 40, 40, np.ascontiguousarray(imgs[i0:i0 + m]), out)
        sliced[i0:i0 + m] = out
    assert np.array_equal(fit, sliced)
    assert_fit_matches_truth(fit[0::2], truth[0::2])
    for k in (1, 601, 1299):          # noisy images of each chunk against mpdaf's fit (the oracle)
        ref = orc.moffat_fit(imgs[k])
        assert_allclose(fit[k, _lib.FIT_FWHM], ref['fwhm'], rtol=FIT_RTOL)
        assert_allclose(fit[k, _lib.FIT_N], ref['n'], rtol=FIT_RTOL)
        assert_allclose(fit[k, [_lib.FIT_Y0, _lib.FIT_X0]], ref['center'], atol=1e-5)


@pytest.mark.parametrize('size,n', [(8, 40), (33, 300), (64, 450)])
def test_fit_image_sizes(own_context, size, n):
    """Square images other than 40 x 40; 450 images of 64 x 64 take three chunks (218 per chunk)."""
    from muse_psfr_b200 import _lib
    imgs, truth = moffat_images(np.random.default_rng(size), n, size, size)
    fit = np.full((n, _lib.FIT_NPAR), np.nan)
    own_context.moffat_fit(n, size, size, imgs, fit)
    assert_fit_matches_truth(fit, truth)


def test_fit_image_over_shared_memory_budget(own_context):
    from muse_psfr_b200 import _lib
    imgs, _ = moffat_images(np.random.default_rng(1), 2, 81, 81)
    fit = np.full((2, _lib.FIT_NPAR), np.nan)
    with pytest.raises(_lib.PsfrError, match='too large for the fitter'):
        own_context.moffat_fit(2, 81, 81, imgs, fit)
    assert np.isnan(fit).all()


def test_mean_refit_slabs(psfrec, golden):
    """max_planes = 1, max_lambda = 35: each host cube is its own slab.  Five slabs must give the
    mean and fit of the device-input path bit for bit."""
    import torch
    from muse_psfr_b200 import _lib
    conv = golden('oracle_config1')['conv']
    cubes = np.ascontiguousarray(np.stack([conv, conv[::-1], 0.5 * conv, np.roll(conv, 3, axis=2), 2.0 * conv[::-1]]))
    ctx = _lib.Context(device=0, max_planes=1, max_lambda=35)
    try:
        mean_h, fit_h = np.empty((35, 40, 40)), np.empty((35, _lib.FIT_NPAR))
        ctx.mean_refit(5, 35, cubes, mean_h, fit_h)
        mean_d, fit_d = np.empty((35, 40, 40)), np.empty((35, _lib.FIT_NPAR))
        ctx.mean_refit(5, 35, torch.from_numpy(cubes).cuda(), mean_d, fit_d)
    finally:
        ctx.close()
    assert np.array_equal(mean_h, mean_d)
    assert np.array_equal(fit_h, fit_d)
    assert_allclose(mean_h, np.mean(cubes, axis=0), rtol=1e-15)
    ref = orc.fit_psf_cube(LBDA35[[0, 34]], np.mean(cubes, axis=0)[[0, 34]])
    assert_allclose(fit_h[[0, 34], _lib.FIT_FWHM] * 0.2, ref['fwhm'], rtol=FIT_RTOL)
    assert_allclose(fit_h[[0, 34], _lib.FIT_N], ref['n'], rtol=FIT_RTOL)


def test_convolve_many_draws_and_aliasing(psfrec, golden):
    """Three draws whose tip-tilt alpha spans the config-4 range (seeing 0.4-2, GL 0.3-0.95, L0 9-29),
    against the oracle per draw; with device buffers, output written over the input."""
    import torch
    g = golden('ref_config1')['psf_muse']
    sel = [0, 17, 34]
    lam = LBDA35[sel]
    draws = [(0.4, 0.95, 9.), (1.0, 0.7, 25.), (2.0, 0.3, 29.)]
    att = np.array([psfrec.tiptilt_alpha(*d) for d in draws])
    assert att.min() < 0.05 and att.max() > 1.5
    cube = np.ascontiguousarray(np.stack([g[sel], g[sel][::-1], np.roll(g[sel], 2, axis=1)]))
    ctx = psfrec.get_context()
    out = np.empty_like(cube)
    ctx.convolve(3, lam, att, cube, out)
    for k, d in enumerate(draws):
        ref = orc.convolve_final_psf(lam, *d, cube[k])
        for i in range(lam.size):
            assert_image_close(out[k, i], ref[i])
    buf = torch.from_numpy(cube).cuda()
    ctx.convolve(3, lam, att, buf, buf)
    torch.cuda.synchronize()
    assert np.array_equal(buf.cpu().numpy(), out)


def polyfit_tolerance(x, y, deg):
    """Norm-wise forward error bound of a backward-stable least-squares solver (Householder QR, as
    np.polyfit's SVD): eps (kappa + kappa^2 |r| / (|V| |c|)), kappa the condition number of the
    Vandermonde matrix, with a factor 64 for the different rounding of the two solvers."""
    V = np.vander(x, deg + 1)
    kappa = np.linalg.cond(V)
    c = np.linalg.lstsq(V, y.T, rcond=None)[0].T
    r = np.linalg.norm(y - c @ V.T, axis=1)
    return 64 * np.finfo(float).eps * (kappa + kappa ** 2 * r / (np.linalg.norm(V, 2) * np.linalg.norm(c, axis=1)))


@pytest.mark.parametrize('nlam,nseries', [(100, 300), (256, 240)])
def test_polyfit_sizes_and_degrees(psfrec, nlam, nseries):
    """Up to the kernel's limits (256 wavelengths, degree 8): the device QR against np.polyfit, to
    a bound derived from the conditioning of the Vandermonde matrix (kappa ~ 8e4 at degree 8)."""
    rng = np.random.default_rng(nlam)
    lam = np.linspace(490, 930, nlam)
    x = orc.norm_lbda(lam)
    y = np.concatenate([0.9 - 0.3 * (x + 0.5) ** 1.3 + 1e-3 * rng.standard_normal((nseries // 2, nlam)),
                        2.5 + 0.5 * np.cos(3 * x) + 1e-2 * rng.standard_normal((nseries - nseries // 2, nlam))])
    ctx = psfrec.get_context()
    for deg in range(9):
        got = ctx.polyfit(lam, deg, y)
        assert got.shape == (nseries, deg + 1) and np.isfinite(got).all()
        ref = np.stack([np.polyfit(x, s, deg) for s in y])
        err = np.linalg.norm(got - ref, axis=1) / np.linalg.norm(ref, axis=1)
        tol = polyfit_tolerance(x, y, deg)
        assert (err < tol).all(), (deg, err.max(), tol.min())


def test_polyfit_limits(psfrec):
    """Inputs past the kernel's limits are refused with an error, never answered wrongly."""
    from muse_psfr_b200 import _lib
    ctx = psfrec.get_context()
    rng = np.random.default_rng(3)
    lam257 = np.linspace(490, 930, 257)
    with pytest.raises(_lib.PsfrError, match='polyfit limits'):
        ctx.polyfit(lam257, 3, rng.standard_normal((2, 257)))
    with pytest.raises(_lib.PsfrError, match='polyfit limits'):
        ctx.polyfit(LBDA35, 9, rng.standard_normal((2, 35)))
    lam5 = np.linspace(490, 930, 5)
    with pytest.raises(_lib.PsfrError, match='polyfit limits'):
        ctx.polyfit(lam5, 5, rng.standard_normal((2, 5)))
    # degree nlam - 1 is the square system: interpolation
    y5 = rng.standard_normal((2, 5))
    c5 = np.stack([np.polyfit(orc.norm_lbda(lam5), s, 4) for s in y5])
    assert np.linalg.norm(ctx.polyfit(lam5, 4, y5) - c5) / np.linalg.norm(c5) < 1e-12
    # scratch of 65536 doubles: nseries * (nlam + deg + 1) + nlam; 1597 series of 35 values at degree 5 fit
    y = 2.5 + 0.01 * rng.standard_normal((1598, 35))
    with pytest.raises(_lib.PsfrError, match='too large'):
        ctx.polyfit(LBDA35, 5, y[:1598])
    got = ctx.polyfit(LBDA35, 5, y[:1597])
    x = orc.norm_lbda(LBDA35)
    ref = np.stack([np.polyfit(x, s, 5) for s in y[[0, 800, 1596]]])
    assert_allclose(got[[0, 800, 1596]], ref, rtol=1e-9, atol=1e-9 * np.abs(ref).max())
