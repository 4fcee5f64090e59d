"""GPU tests of the star fits (``psfr_moffat_fit_weighted``, ``fit_psf_cube(var=, mask=, fit_back=)``, DESIGN.md
section 5.7): known answers of exact images with weights, masks and a background; masked pixels that are inert
whatever they hold; the reduction to the reconstruction's fitter bit for bit; the scale of the weights; the scipy
restatement of tests/star_fit_oracle.py on noisy stamps; the calibration of the reported errors; per-image failures;
the shared-memory and staging envelope; and the intended workflow on a reconstructed PSF made into a star."""
import numpy as np
import pytest
from numpy.testing import assert_allclose

import efit_oracle as eo
import star_fit_oracle as so

pytestmark = pytest.mark.gpu

SENT = 12345.0


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


def star_fit(ctx, imgs, w, fit_back, elliptical):
    from muse_psfr_b200 import _lib
    imgs = np.ascontiguousarray(imgs, dtype=float)
    n, ny, nx = imgs.shape
    rec = np.full((n, _lib.EFIT_NPAR if elliptical else _lib.FIT_NPAR), SENT)
    back = np.full((n, _lib.BACK_NPAR), SENT)
    ctx.moffat_fit_weighted(n, ny, nx, imgs, None if w is None else np.ascontiguousarray(w, dtype=float), rec, back,
                            fit_back=fit_back, elliptical=elliptical)
    return rec, back


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def assert_bits(a, b):
    np.testing.assert_array_equal(bits(a), bits(b))


def iter_slot(elliptical):
    return eo.ITER if elliptical else so.ITER


# ---------------------------------------------------------------- 1. known answers
def truth_of(elliptical, shape, centre, c):
    if elliptical:
        th = eo.theta_of(2.0, centre[0], centre[1], 3.0, 2.0, 30.0, 2.5)
    else:
        th = np.array([2.0, centre[0], centre[1], 2.6, 2.8])
    return np.concatenate([th, [c]])


def known_cases():
    cases = []
    for elliptical in (False, True):
        for shape, centre in (((25, 25), (12.3, 11.6)), ((21, 31), (9.7, 16.2)), ((17, 23), (2.0, 11.4)),
                              ((23, 19), (11.2, 2.3))):
            for c in (0.3, -0.2, 0.0):
                cases.append((elliptical, shape, centre, c))
    return cases


def masked_weights(shape, peak_rc, seed, frac):
    rng = np.random.default_rng(seed)
    w = rng.uniform(0.3, 3.0, shape)
    w[rng.random(shape) < frac] = 0.0
    w[peak_rc] = 0.0                     # the peak pixel
    w[-1, :] = 0.0                       # a whole edge row
    return w


@pytest.mark.parametrize('case', known_cases(), ids=lambda c: '%s-%dx%d-%.1f,%.1f-c%g' % (
    'ell' if c[0] else 'circ', c[1][0], c[1][1], c[2][0], c[2][1], c[3]))
def test_known_answers(ctx, case):
    elliptical, shape, centre, c = case
    truth = truth_of(elliptical, shape, centre, c)
    for seed, frac in ((1, 0.1), (2, 0.25)):
        img = so.render(shape, truth, elliptical, True)
        w = masked_weights(shape, (int(round(centre[0])), int(round(centre[1]))), seed, frac)
        img[w == 0] = np.nan
        for fit_back in ((True, False) if c == 0.0 else (True,)):
            rec, back = star_fit(ctx, img[None], w[None], fit_back, elliptical)
            rec, back = rec[0], back[0]
            assert rec[iter_slot(elliptical)] > 0, rec
            got = so.theta_of_records(rec, back, elliptical, fit_back)
            want = truth if fit_back else truth[:-1]
            scale = so.param_scale(want, elliptical, peak=truth[0])
            dev = np.abs(got - want) / scale
            assert np.all(dev < 1e-8), (dev, got, want)
            assert back[so.NPIX] == np.count_nonzero(w > 0)
            if not fit_back:
                assert back[so.CONT] == 0 and back[so.ERR_CONT] == 0


# ---------------------------------------------------------------- 2. masks are inert
@pytest.mark.parametrize('elliptical', [False, True])
def test_masked_pixels_are_inert(psfrec, ctx, elliptical):
    rng = np.random.default_rng(5)
    truth = truth_of(elliptical, (25, 25), (12.4, 11.7), 0.1)
    imgs = np.stack([so.render((25, 25), truth, elliptical, True) + rng.normal(0, 0.01, (25, 25)) for _ in range(6)])
    w = np.full(imgs.shape, 1e4)
    w[rng.random(imgs.shape) < 0.2] = 0.0
    ref = None
    for fill in (np.nan, np.inf, -np.inf, 0.0, 1e300):
        x = imgs.copy()
        x[w == 0] = fill
        got = star_fit(ctx, x, w, True, elliptical)
        if ref is None:
            ref = got
        assert_bits(got[0], ref[0])
        assert_bits(got[1], ref[1])
    # mask=True through fit_psf_cube gives the records of weight 0 through the entry point
    var = 1.0 / np.where(w > 0, w, 1.0)
    tab = psfrec.fit_psf_cube(np.arange(6.), imgs, circular=not elliptical, var=var, mask=w == 0, fit_back=True)
    col = 'fwhm'
    ref_tab = psfrec.fit_psf_cube(np.arange(6.), np.where(w > 0, imgs, np.nan), circular=not elliptical, var=var,
                                  fit_back=True)
    for k in ref_tab.colnames:
        assert_bits(np.asarray(tab[k], dtype=float), np.asarray(ref_tab[k], dtype=float))
    assert tab[col].shape == (6, 2)


# ---------------------------------------------------------------- 3. reduces to today's fitter
@pytest.fixture(scope='module')
def config4(psfrec):
    from muse_psfr_b200 import _lib
    nd, nl = 16, 35
    lam = np.linspace(490, 930, nl)
    rng = np.random.default_rng(20261020)
    seeing, GL, L0 = rng.uniform(0.5, 1.8, nd), rng.uniform(0.35, 0.9, nd), rng.uniform(10, 28, nd)
    fit, cube = psfrec.compute_psf_batch(lam, seeing, GL, L0)
    return cube.reshape(-1, 40, 40), fit.reshape(-1, _lib.FIT_NPAR)


def test_unit_weights_reduce_to_plain_fit(ctx, config4):
    from muse_psfr_b200 import _lib
    imgs, _ = config4
    n = imgs.shape[0]
    fit = np.full((n, _lib.FIT_NPAR), SENT)
    ctx.moffat_fit(n, 40, 40, np.ascontiguousarray(imgs), fit)
    rec, back = star_fit(ctx, imgs, None, False, False)
    assert_bits(rec, fit)
    rec1, back1 = star_fit(ctx, imgs, np.ones(imgs.shape), False, False)
    assert_bits(rec1, fit)
    assert_bits(back, np.tile([0.0, 0.0, 1600.0], (n, 1)))
    assert_bits(back1, back)
    efit = np.full((n, _lib.EFIT_NPAR), SENT)
    ctx.moffat_fit_elliptical(n, 40, 40, np.ascontiguousarray(imgs), efit)
    erec, eback = star_fit(ctx, imgs, None, False, True)
    assert_bits(erec, efit)
    assert_bits(eback, back)


# ---------------------------------------------------------------- 4. weight scale
@pytest.mark.parametrize('elliptical', [False, True])
def test_weight_scale(ctx, elliptical):
    rng = np.random.default_rng(11)
    truth = truth_of(elliptical, (25, 25), (12.2, 12.9), 0.05)
    imgs = np.stack([so.render((25, 25), truth, elliptical, True) + rng.normal(0, 0.02, (25, 25)) for _ in range(8)])
    w = rng.uniform(100, 5000, imgs.shape)
    w[rng.random(imgs.shape) < 0.1] = 0
    ref = star_fit(ctx, imgs, w, True, elliptical)
    x4 = star_fit(ctx, imgs, w * 4, True, elliptical)
    # every sum scales by exactly 4, and neither the step, the acceptance test nor the errors depend on the scale;
    # CHISQ itself is sum w r^2, 4 times larger
    chisq = eo.CHISQ if elliptical else so.CHISQ
    assert_bits(x4[0][:, chisq], 4 * ref[0][:, chisq])
    x4[0][:, chisq] = ref[0][:, chisq]
    assert_bits(x4[0], ref[0])
    assert_bits(x4[1], ref[1])
    x37 = star_fit(ctx, imgs, w * 3.7, True, elliptical)
    for r, b, r0, b0 in zip(*x37, *ref):
        th, th0 = so.theta_of_records(r, b, elliptical, True), so.theta_of_records(r0, b0, elliptical, True)
        assert np.all(np.abs(th - th0) / so.param_scale(th0, elliptical) < 1e-9)
        err = [s for s in range(eo.ERR_PEAK, eo.ERR_FLUX + 1) if s != eo.FLUX] if elliptical else \
            [so.ERR_PEAK, so.ERR_Y0, so.ERR_X0, so.ERR_ALPHA, so.ERR_N, so.ERR_FWHM]
        assert_allclose(r[err], r0[err], rtol=1e-8)
        assert_allclose(b[so.ERR_CONT], b0[so.ERR_CONT], rtol=1e-8)


# ---------------------------------------------------------------- 5. against the oracle
def noisy_star(shape, truth, elliptical, seed, rn=0.01, gain=2e3, mask=0.05):
    """(image, inverse-variance weights) of a star with sigma^2 = rn^2 + model / gain, masks and NaN there."""
    rng = np.random.default_rng(seed)
    model = so.render(shape, truth, elliptical, True)
    var = rn ** 2 + np.abs(model) / gain
    img = model + rng.normal(size=shape) * np.sqrt(var)
    w = 1 / var
    w[rng.random(shape) < mask] = 0
    img[w == 0] = np.nan
    return img, w


ORACLE_CASES = [(ell, fb, seed) for ell in (False, True) for fb in (True, False) for seed in range(3)]


@pytest.mark.parametrize('case', ORACLE_CASES, ids=lambda c: '%s-%s-%d' % ('ell' if c[0] else 'circ',
                                                                             'back' if c[1] else 'noback', c[2]))
def test_against_oracle(ctx, case):
    elliptical, fit_back, seed = case
    shape = ((25, 25), (23, 29), (31, 27))[seed]
    truth = truth_of(elliptical, shape, (shape[0] / 2 - 0.4 + 0.3 * seed, shape[1] / 2 + 0.2), 0.04 * (seed - 1))
    img, w = noisy_star(shape, truth, elliptical, 100 + seed)
    if not fit_back:
        img = img - truth[-1]
    rec, back = star_fit(ctx, img[None], w[None], fit_back, elliptical)
    rec, back = rec[0], back[0]
    assert rec[iter_slot(elliptical)] > 0
    start = truth if fit_back else truth[:-1]
    orec, oback, oth = so.star_fit(img, w, start, elliptical, fit_back)
    got = so.theta_of_records(rec, back, elliptical, fit_back)
    scale = so.param_scale(oth, elliptical, peak=truth[0])
    dev = np.abs(got - oth) / scale
    if not np.all(dev < 1e-7):
        # which one is off the stationary point: the gradient of chi^2 at each, scaled
        p, q, d, wu = so.used_pixels(img, w)
        for name, th in (('gpu', got), ('oracle', oth)):
            J = so.star_jacobian(th, p, q, elliptical, fit_back)
            r = so.star_model(th, p, q, elliptical, fit_back) - d
            g = (J * wu[:, None]).T @ r * scale
            print(name, 'scaled gradient', g)
    assert np.all(dev < 1e-7), dev
    if elliptical:
        err = [s for s in range(eo.ERR_PEAK, eo.ERR_FLUX + 1) if s not in (eo.FLUX,)]
        err = [s for s in err if np.isfinite(orec[s])]
    else:
        err = [so.ERR_PEAK, so.ERR_Y0, so.ERR_X0, so.ERR_ALPHA, so.ERR_N, so.ERR_FWHM]
    assert_allclose(rec[err], orec[err], rtol=1e-6)
    assert_allclose(back[[so.CONT, so.ERR_CONT]], oback[[so.CONT, so.ERR_CONT]], rtol=1e-6, atol=1e-9 * truth[0])
    assert back[so.NPIX] == oback[so.NPIX]
    assert_allclose(rec[eo.CHISQ if elliptical else so.CHISQ], orec[eo.CHISQ if elliptical else so.CHISQ], rtol=1e-9)


# ---------------------------------------------------------------- 6. error calibration
def test_error_calibration(ctx):
    shape, nreal = (25, 25), 2000
    truth = np.array([1.0, 12.3, 11.8, 2.5, 2.5, 0.05])
    model = so.render(shape, truth, False, True)
    # peak S/N ~ 50: sigma^2 = r^2 + model / g with sigma = 0.02 at the peak
    var = 0.01 ** 2 + model / (truth[0] + truth[-1]) * 3e-4
    rng = np.random.default_rng(2026)
    imgs = model[None] + rng.normal(size=(nreal,) + shape) * np.sqrt(var)[None]
    rec, back = star_fit(ctx, imgs, np.broadcast_to(1 / var, imgs.shape), True, False)
    assert np.all(rec[:, so.ITER] > 0)
    # ERR_FWHM is mpdaf's err_a * n, not an error of the FWHM: the width is checked through a, whose scatter sets
    # the FWHM's (FWHM = a kf(n))
    n, a = rec[:, so.N], rec[:, so.ALPHA]
    kf = 2 * np.sqrt(2 ** (1 / n) - 1)
    checks = {'n': (rec[:, so.N], rec[:, so.ERR_N]), 'y0': (rec[:, so.Y0], rec[:, so.ERR_Y0]),
              'x0': (rec[:, so.X0], rec[:, so.ERR_X0]), 'a': (a, rec[:, so.ERR_ALPHA]),
              'c': (back[:, so.CONT], back[:, so.ERR_CONT])}
    for name, (val, err) in checks.items():
        ratio = val.std(ddof=1) / err.mean()
        assert abs(ratio - 1) < 0.1, (name, ratio)
    assert_allclose(rec[:, so.FWHM], kf * a, rtol=1e-14)
    chi2 = rec[:, so.CHISQ] / (back[:, so.NPIX] - 6)
    assert abs(chi2.mean() - 1) < 0.05, chi2.mean()


# ---------------------------------------------------------------- 7. per-image failures
@pytest.mark.parametrize('elliptical', [False, True])
def test_per_image_failures(ctx, elliptical):
    rng = np.random.default_rng(9)
    truth = truth_of(elliptical, (21, 21), (10.3, 9.8), 0.1)
    good = [so.render((21, 21), truth, elliptical, True) + rng.normal(0, 0.01, (21, 21)) for _ in range(2)]
    wgood = [rng.uniform(1e3, 1e4, (21, 21)) for _ in range(2)]
    npar = 8 if elliptical else 6
    bad_imgs, bad_w = [], []
    bad_imgs.append(good[0].copy()); bad_w.append(np.zeros((21, 21)))             # all masked
    w = np.zeros((21, 21)); w.flat[rng.choice(441, npar, replace=False)] = 1.0
    bad_imgs.append(good[0].copy()); bad_w.append(w)                             # npix_used = NP
    x = good[0].copy(); x[10, 10] = np.nan
    bad_imgs.append(x); bad_w.append(wgood[0].copy())                            # NaN on a used pixel
    w = wgood[0].copy(); w[3, 4] = -1.0
    bad_imgs.append(good[0].copy()); bad_w.append(w)                             # a negative weight
    w = wgood[0].copy(); w[5, 5] = np.inf
    bad_imgs.append(good[0].copy()); bad_w.append(w)                             # an infinite weight
    imgs = np.stack([good[0]] + bad_imgs + [good[1]])
    ws = np.stack([wgood[0]] + bad_w + [wgood[1]])
    rec, back = star_fit(ctx, imgs, ws, True, elliptical)
    ref, rback = star_fit(ctx, np.stack(good), np.stack(wgood), True, elliptical)
    assert_bits(rec[[0, -1]], ref)
    assert_bits(back[[0, -1]], rback)
    it = iter_slot(elliptical)
    for k in range(1, 1 + len(bad_imgs)):
        assert rec[k, it] == 0
        assert np.all(np.isnan(np.delete(rec[k], it)))
        assert np.all(np.isnan(back[k, :2]))
    assert back[1, so.NPIX] == 0 and back[2, so.NPIX] == npar


# ---------------------------------------------------------------- 8. envelope
@pytest.mark.parametrize('elliptical', [False, True])
def test_shared_memory_limit(ctx, elliptical):
    from muse_psfr_b200 import _lib
    truth = truth_of(elliptical, (56, 56), (27.6, 28.2), 0.1)
    img = so.render((56, 56), truth, elliptical, True)
    rec, back = star_fit(ctx, img[None], np.ones((1, 56, 56)), True, elliptical)
    assert rec[0, iter_slot(elliptical)] > 0
    got = so.theta_of_records(rec[0], back[0], elliptical, True)
    assert np.all(np.abs(got - truth) / so.param_scale(truth, elliptical) < 1e-8)
    big = np.ones((2, 57, 57))
    out = np.full((2, _lib.EFIT_NPAR if elliptical else _lib.FIT_NPAR), SENT)
    bk = np.full((2, 3), SENT)
    with pytest.raises(_lib.PsfrError) as e:
        ctx.moffat_fit_weighted(2, 57, 57, big, big, out, bk, fit_back=True, elliptical=elliptical)
    assert e.value.code == _lib.E_UNSUPPORTED and 'shared memory' in str(e.value)
    assert np.all(out == SENT) and np.all(bk == SENT)


def test_refusals_before_launch(ctx):
    from muse_psfr_b200 import _lib
    out, bk = np.full((1, 16), SENT), np.full((1, 3), SENT)
    lib, h = ctx._lib, ctx._handle()
    img = np.ones((1, 9, 9))
    assert lib.psfr_moffat_fit_weighted(h, 1, 9, 9, None, None, 1, 0, out.ctypes.data, bk.ctypes.data, None) == \
        _lib.E_ARG
    assert lib.psfr_moffat_fit_weighted(h, 1, 9, 9, img.ctypes.data, None, 1, 0, None, bk.ctypes.data, None) == \
        _lib.E_ARG
    assert lib.psfr_moffat_fit_weighted(h, 1, 2, 9, img.ctypes.data, None, 1, 0, out.ctypes.data, bk.ctypes.data,
                                        None) == _lib.E_ARG
    assert lib.psfr_moffat_fit_weighted(h, 0, 9, 9, img.ctypes.data, None, 1, 0, out.ctypes.data, bk.ctypes.data,
                                        None) == _lib.E_ARG
    assert np.all(out == SENT) and np.all(bk == SENT)


@pytest.mark.parametrize('elliptical', [False, True])
def test_host_device_and_chunks(psfrec, ctx, elliptical):
    import torch
    from muse_psfr_b200 import _lib
    rng = np.random.default_rng(21)
    truth = truth_of(elliptical, (25, 25), (12.1, 12.6), 0.1)
    n = 11
    imgs, ws = zip(*(noisy_star((25, 25), truth, elliptical, 300 + k) for k in range(n)))
    imgs, ws = np.ascontiguousarray(imgs), np.ascontiguousarray(ws)
    ref = star_fit(ctx, imgs, ws, True, elliptical)
    npar = ref[0].shape[1]
    d_img, d_w = torch.from_numpy(imgs).cuda(), torch.from_numpy(ws).cuda()
    for img_a, w_a, dev_out in ((d_img, d_w, True), (imgs, d_w, False), (d_img, ws, True), (d_img, ws, False)):
        out = torch.full((n, npar), SENT, dtype=torch.float64, device='cuda' if dev_out else 'cpu')
        bk = torch.full((n, 3), SENT, dtype=torch.float64, device='cuda' if dev_out else 'cpu')
        ctx.moffat_fit_weighted(n, 25, 25, img_a, w_a, out, bk, fit_back=True, elliptical=elliptical)
        torch.cuda.synchronize()
        assert_bits(out.cpu().numpy(), ref[0])
        assert_bits(bk.cpu().numpy(), ref[1])
    # no back output
    out = np.full((n, npar), SENT)
    ctx.moffat_fit_weighted(n, 25, 25, imgs, ws, out, None, fit_back=True, elliptical=elliptical)
    assert_bits(out, ref[0])
    # host arrays chunked through small staging buffers: chunks of 1, 3 and 7 images
    for lam in (1, 3, 7):
        small = _lib.Context(device=0, max_planes=1, max_lambda=lam)
        try:
            got = star_fit(small, imgs, ws, True, elliptical)
            assert_bits(got[0], ref[0])
            assert_bits(got[1], ref[1])
            big = np.ones((1, 41, 41))              # 1681 pixels: more than one 40 x 40 image of staging
            o, b = np.full((1, npar), SENT), np.full((1, 3), SENT)
            if lam == 1:
                with pytest.raises(_lib.PsfrError) as e:
                    small.moffat_fit_weighted(1, 41, 41, big, big, o, b, fit_back=True, elliptical=elliptical)
                assert e.value.code == _lib.E_CAPACITY
                assert np.all(o == SENT) and np.all(b == SENT)
        finally:
            small.close()


# ---------------------------------------------------------------- 9. the workflow
def test_workflow_reconstructed_star(psfrec):
    lam = np.linspace(500, 900, 8)
    _, cube = psfrec.compute_psf_batch(lam, [0.9], [0.6], [22.])
    psf = cube[0]
    star = 5e4 * psf / psf.sum(axis=(1, 2), keepdims=True) + 3.0      # flux 5e4 e-, sky residual 3 e-
    var = 4.0 + star / 1.5
    rng = np.random.default_rng(77)
    noisy = star + rng.normal(size=star.shape) * np.sqrt(var)
    mask = rng.random(star.shape) < 0.02
    clean = psfrec.fit_psf_cube(lam, star, var=var, mask=mask, fit_back=True)
    got = psfrec.fit_psf_cube(lam, noisy, var=var, mask=mask, fit_back=True)
    assert np.all(got['converged'] == 1) and np.all(clean['converged'] == 1)
    for col in ('fwhm', 'n'):
        d = np.abs(np.asarray(got[col]) - np.asarray(clean[col]))
        assert np.all(d <= 4 * np.asarray(got['err_' + col])), (col, d, got['err_' + col])
    assert np.all(np.abs(got['cont'] - clean['cont']) <= 4 * got['err_cont'])
    assert np.all(got['npix'] == 1600 - mask.reshape(8, -1).sum(axis=1))
