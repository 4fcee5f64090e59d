"""GPU tests of the template fit (``psfr_template_fit``, ``fit_psf_template``, DESIGN.md section 5.8): known answers
of exact shifted templates; masked pixels that are inert whatever they hold and the scale of the weights; template
broadcast and host, device, mixed and chunked inputs; the scipy restatement of tests/template_fit_oracle.py on noisy
stamps; the calibration of the reported errors; per-image failures; the shared-memory and argument envelope; and the
workflow on a reconstructed PSF made into a star."""
import numpy as np
import pytest
from numpy.testing import assert_allclose

import template_fit_oracle as to

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


def tfit(ctx, imgs, w, tpls, fit_back, model=False):
    from muse_psfr_b200 import _lib
    imgs = np.ascontiguousarray(imgs, dtype=float)
    tpls = np.ascontiguousarray(tpls, dtype=float)
    if tpls.ndim == 2:
        tpls = tpls[None]
    n, ny, nx = imgs.shape
    rec = np.full((n, _lib.TFIT_NPAR), SENT)
    mo = np.full((n, ny, nx), SENT) if model else None
    ctx.template_fit(n, ny, nx, imgs, None if w is None else np.ascontiguousarray(w, dtype=float), tpls, rec, mo,
                     fit_back=fit_back)
    return (rec, mo) if model else rec


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def assert_bits(a, b):
    np.testing.assert_array_equal(bits(a), bits(b))


def psf_template(shape=(40, 40), centre=None, a=2.4, n=2.6, halo=0.03):
    """A smooth PSF-like template: a Moffat core and a wide Moffat halo, centred near (ty // 2, tx // 2)."""
    ty, tx = shape
    cy, cx = centre if centre is not None else (ty // 2 + 0.2, tx // 2 - 0.3)
    p, q = np.indices(shape, dtype=float)
    r2 = (p - cy) ** 2 + (q - cx) ** 2
    return (1 + r2 / a ** 2) ** (-n) + halo * (1 + r2 / (3 * a) ** 2) ** (-1.6)


def theta_of(rec, fit_back):
    return rec[[to.FLUX, to.Y0, to.X0] + ([to.CONT] if fit_back else [])]


# ---------------------------------------------------------------- 1. known answers
KNOWN = [((25, 25), (40, 40), (12.3, 11.6)), ((21, 31), (40, 40), (10.4, 17.2)), ((17, 23), (40, 40), (2.4, 20.3)),
         ((25, 25), (41, 37), (12.7, 12.1)), ((21, 31), (41, 37), (9.6, 13.8)), ((17, 23), (41, 37), (14.3, 1.7))]


@pytest.mark.parametrize('fit_back', [False, True])
@pytest.mark.parametrize('case', KNOWN, ids=lambda c: '%dx%d-tpl%dx%d' % (c[0] + c[1]))
def test_known_answers(ctx, case, fit_back):
    shape, tshape, (y0, x0) = case
    tpl = psf_template(tshape)
    truth = np.array([850.0, y0, x0] + ([0.6] if fit_back else []))
    img = to.model(truth, tpl, shape, fit_back)
    rng = np.random.default_rng(sum(shape) + tshape[1])
    w = rng.uniform(0.5, 4.0, shape)
    rec, mo = tfit(ctx, img[None], w[None], tpl, fit_back, model=True)
    r = rec[0]
    assert r[to.ITER] > 0 and r[to.NPIX] == img.size
    got = theta_of(r, fit_back)
    assert abs(got[0] / truth[0] - 1) < 1e-9
    assert np.all(np.abs(got[1:3] - truth[1:3]) < 1e-9)
    if fit_back:
        assert abs(got[3] - truth[3]) < 1e-9 * truth[0] / tpl.sum() * tpl.max()
    else:
        assert r[to.CONT] == 0 and r[to.ERR_CONT] == 0
    # The model output is m at the fitted parameters, to 1e-12 of the peak.  Against the stamp itself the bound is
    # 2e-12, not 1e-12: the fit stops at MINPACK's relative step of 1.49e-8, which leaves the parameters ~1e-12 from
    # the truth.  Measured on a B200: 1.34e-12 of the peak for the 21 x 31 stamp with the 41 x 37 template and no
    # background (a 3e-12 px centre offset), 1.0e-12 with a background; under 1e-12 in the ten other cases.
    assert np.abs(mo[0] - to.model(got, tpl, shape, fit_back)).max() < 1e-12 * img.max()
    assert np.abs(mo[0] - img).max() < 2e-12 * img.max()
    assert r[to.CHISQ] < 1e-20 * (w * img * img).sum()
    assert r[to.QFIT] < 1e-9


# ---------------------------------------------------------------- 2. masked pixels and the weight scale
def noisy_stamps(shape, tpl, truth, fit_back, n, seed, mask=0.05, rn=2.0, gain=1.0):
    """(stamps, inverse-variance weights) around the exact image of truth: sigma^2 = rn^2 + model / gain, masked
    pixels weight 0 and NaN."""
    rng = np.random.default_rng(seed)
    model = to.model(truth, tpl, shape, fit_back)
    var = rn ** 2 + np.abs(model) / gain
    imgs = model[None] + rng.normal(size=(n,) + shape) * np.sqrt(var)[None]
    w = np.broadcast_to(1 / var, imgs.shape).copy()
    w[rng.random(imgs.shape) < mask] = 0.0
    imgs[w == 0] = np.nan
    return imgs, w


@pytest.mark.parametrize('fit_back', [False, True])
def test_masked_pixels_and_weight_scale(ctx, fit_back):
    tpl = psf_template()
    truth = np.array([5e3, 12.2, 12.8] + ([4.0] if fit_back else []))
    imgs, w = noisy_stamps((25, 25), tpl, truth, fit_back, 8, 11, mask=0.1)
    ref = tfit(ctx, imgs, w, tpl, fit_back)
    assert np.all(ref[:, to.ITER] > 0)
    for fill in (np.inf, -np.inf, 0.0, 1e300):
        x = imgs.copy()
        x[w == 0] = fill
        assert_bits(tfit(ctx, x, w, tpl, fit_back), ref)
    # every sum scales by exactly 4: the parameters, QFIT, the errors and the iterations keep their bits
    x4 = tfit(ctx, imgs, 4 * w, tpl, fit_back)
    assert_bits(x4[:, to.CHISQ], 4 * ref[:, to.CHISQ])
    x4[:, to.CHISQ] = ref[:, to.CHISQ]
    assert_bits(x4, ref)


# ---------------------------------------------------------------- 3. broadcast, pointer kinds, chunks
def test_broadcast_pointer_kinds_and_chunks(psfrec, ctx):
    import torch
    from muse_psfr_b200 import _lib
    nt, reps = 3, 4
    tpls = np.stack([psf_template(a=2.0 + 0.3 * k) for k in range(nt)])
    imgs, ws = [], []
    for r in range(reps):
        for k in range(nt):
            i, wi = noisy_stamps((25, 25), tpls[k], np.array([4e3, 12.1 + 0.1 * r, 12.4, 3.0]), True, 1, 10 * r + k)
            imgs.append(i[0])
            ws.append(wi[0])
    imgs, ws = np.ascontiguousarray(imgs), np.ascontiguousarray(ws)
    n = imgs.shape[0]
    ref, mref = tfit(ctx, imgs, ws, np.tile(tpls, (reps, 1, 1)), True, model=True)
    assert np.all(ref[:, to.ITER] > 0)
    got, mgot = tfit(ctx, imgs, ws, tpls, True, model=True)
    assert_bits(got, ref)
    assert_bits(mgot, mref)
    d_img, d_w, d_t = (torch.from_numpy(a).cuda() for a in (imgs, ws, tpls))
    for img_a, w_a, t_a, dev_out in ((d_img, d_w, d_t, True), (imgs, d_w, d_t, False), (d_img, ws, tpls, True),
                                     (imgs, ws, d_t, False), (d_img, d_w, tpls, False)):
        dev = 'cuda' if dev_out else 'cpu'
        out = torch.full((n, _lib.TFIT_NPAR), SENT, dtype=torch.float64, device=dev)
        mo = torch.full((n, 25, 25), SENT, dtype=torch.float64, device='cpu' if dev_out else 'cuda')
        ctx.template_fit(n, 25, 25, img_a, w_a, t_a, out, mo, fit_back=True)
        torch.cuda.synchronize()
        assert_bits(out.cpu().numpy(), ref)
        assert_bits(mo.cpu().numpy(), mref)
    # no model output
    assert_bits(tfit(ctx, imgs, ws, tpls, True), ref)
    # host arrays chunked through small staging buffers: chunks of 1, 3 and 7 stamps; with one, the three host
    # templates do not fit and device templates are used
    for lam in (1, 3, 7):
        small = _lib.Context(device=0, max_planes=1, max_lambda=lam)
        try:
            # every stamp-sized array on the device: one launch, whatever the staging capacity
            d_out = torch.full((n, _lib.TFIT_NPAR), SENT, dtype=torch.float64, device='cuda')
            d_mo = torch.full((n, 25, 25), SENT, dtype=torch.float64, device='cuda')
            before = small.kernel_launches()
            small.template_fit(n, 25, 25, d_img, d_w, d_t, d_out, d_mo, fit_back=True)
            torch.cuda.synchronize()
            assert small.kernel_launches() - before == 1
            assert_bits(d_out.cpu().numpy(), ref)
            assert_bits(d_mo.cpu().numpy(), mref)
            if lam >= nt:
                before = small.kernel_launches()
                g, m = tfit(small, imgs, ws, tpls, True, model=True)
                assert small.kernel_launches() - before == -(-n // lam)
                assert_bits(g, ref)
                assert_bits(m, mref)
            else:      # the host templates do not fit the staging buffer
                o = np.full((n, _lib.TFIT_NPAR), SENT)
                with pytest.raises(_lib.PsfrError) as e:
                    small.template_fit(n, 25, 25, imgs, ws, tpls, o, None, fit_back=True)
                assert e.value.code == _lib.E_CAPACITY and np.all(o == SENT)
                g = np.full((n, _lib.TFIT_NPAR), SENT)
                small.template_fit(n, 25, 25, imgs, ws, d_t, g, None, fit_back=True)
                assert_bits(g, ref)
        finally:
            small.close()


# ---------------------------------------------------------------- 4. against the oracle
@pytest.mark.parametrize('fit_back', [False, True])
@pytest.mark.parametrize('seed', range(3))
def test_against_oracle(ctx, fit_back, seed):
    tpl = psf_template((41, 37))
    truth = np.array([2e4, 11.7 + 0.3 * seed, 12.4 - 0.2 * seed] + ([5.0] if fit_back else []))
    imgs, w = noisy_stamps((25, 25), tpl, truth, fit_back, 1, 40 + seed)
    rec = tfit(ctx, imgs, w, tpl, fit_back)[0]
    orec, oth = to.template_fit(imgs[0], w[0], tpl, fit_back)
    assert rec[to.ITER] > 0
    err = rec[[to.ERR_FLUX, to.ERR_Y0, to.ERR_X0] + ([to.ERR_CONT] if fit_back else [])]
    assert np.all(np.abs(theta_of(rec, fit_back) - oth) < 1e-3 * err)
    errs = [to.ERR_FLUX, to.ERR_Y0, to.ERR_X0, to.ERR_CONT]
    assert_allclose(rec[errs], orec[errs], rtol=1e-5)
    # chi^2 is stationary at the minimum, QFIT is not: it moves to first order with the parameters' 1e-3 sigma
    assert_allclose(rec[to.CHISQ], orec[to.CHISQ], rtol=1e-9)
    assert_allclose(rec[to.QFIT], orec[to.QFIT], rtol=1e-6)
    assert rec[to.NPIX] == orec[to.NPIX]


# ---------------------------------------------------------------- 5. error calibration
def test_error_calibration(ctx):
    nreal = 2000
    tpl = psf_template()
    truth = np.array([3e3, 12.3, 11.8, 5.0])
    imgs, w = noisy_stamps((25, 25), tpl, truth, True, nreal, 2026, mask=0.0)
    rec = tfit(ctx, imgs, w, tpl, True)
    assert np.all(rec[:, to.ITER] > 0)
    for val, err in ((to.FLUX, to.ERR_FLUX), (to.Y0, to.ERR_Y0), (to.X0, to.ERR_X0), (to.CONT, to.ERR_CONT)):
        ratio = rec[:, val].std(ddof=1) / np.median(rec[:, err])
        assert abs(ratio - 1) < 0.1, (val, ratio)
    chi2 = rec[:, to.CHISQ] / (rec[:, to.NPIX] - 4)
    assert abs(chi2.mean() - 1) < 0.05, chi2.mean()


# ---------------------------------------------------------------- 6. per-image failures
@pytest.mark.parametrize('fit_back', [False, True])
def test_per_image_failures(ctx, fit_back):
    rng = np.random.default_rng(9)
    tpl = psf_template()
    npar = 4 if fit_back else 3
    truth = np.array([4e3, 10.3, 9.8] + ([2.0] if fit_back else []))
    good, wgood = noisy_stamps((21, 21), tpl, truth, fit_back, 2, 5, mask=0.0)
    cases = []                                                                   # (image, weights, template)
    cases.append((good[0], np.zeros((21, 21)), tpl))                             # all masked
    w = np.zeros((21, 21))
    w.flat[rng.choice(441, npar, replace=False)] = 1.0
    cases.append((good[0], w, tpl))                                              # npix_used = NP
    x = good[0].copy()
    x[10, 10] = np.nan
    cases.append((x, wgood[0], tpl))                                             # NaN on a used pixel
    w = wgood[0].copy()
    w[3, 4] = -1.0
    cases.append((good[0], w, tpl))                                              # a negative weight
    w = wgood[0].copy()
    w[5, 5] = np.inf
    cases.append((good[0], w, tpl))                                              # an infinite weight
    t = tpl.copy()
    t[7, 30] = np.nan
    cases.append((good[0], wgood[0], t))                                         # a non-finite template pixel
    cases.append((good[0], wgood[0], -tpl))                                      # S < 0
    t = np.zeros_like(tpl)
    t[5, 5], t[6, 6] = 1.0, -1.0
    cases.append((good[0], wgood[0], t))                                         # S = 0
    imgs = np.stack([good[0]] + [c[0] for c in cases] + [good[1]])
    ws = np.stack([wgood[0]] + [c[1] for c in cases] + [wgood[1]])
    tpls = np.stack([tpl] + [c[2] for c in cases] + [tpl])
    rec, mo = tfit(ctx, imgs, ws, tpls, fit_back, model=True)
    ref, mref = tfit(ctx, good, wgood, tpl, fit_back, model=True)
    assert_bits(rec[[0, -1]], ref)
    assert_bits(mo[[0, -1]], mref)
    for k in range(1, 1 + len(cases)):
        assert rec[k, to.ITER] == 0
        assert np.all(np.isnan(np.delete(rec[k], to.ITER)))
        assert np.all(np.isnan(mo[k]))


@pytest.mark.parametrize('fit_back', [False, True])
def test_no_overlap_failure(ctx, fit_back):
    """A template whose B-spline is exactly 0 on every used pixel (its only non-zero pixel is 35 rows and columns
    away, and the recursion's z^70 underflows): the start denominator sum w s~^2 is 0."""
    tpl = psf_template((70, 70), centre=(35.2, 34.7))
    far = np.zeros((70, 70))
    far[0, 0] = 1e-300
    p, q = np.indices((5, 5))           # every pixel of a 3 x 3 stamp from any start centre in it
    assert np.all(to.sample_grad(to.prefilter(far), p.ravel() + 33.0, q.ravel() + 33.0)[0] == 0)
    truth = np.array([50.0, 1.1, 0.9] + ([0.5] if fit_back else []))
    good = np.stack([to.model(truth, tpl, (3, 3), fit_back)] * 2)
    imgs = np.stack([good[0], good[0], good[1]])
    rec = tfit(ctx, imgs, None, np.stack([tpl, far, tpl]), fit_back)
    ref = tfit(ctx, good, None, tpl, fit_back)
    assert_bits(rec[[0, -1]], ref)
    assert np.all(ref[:, to.ITER] > 0)
    assert rec[1, to.ITER] == 0 and np.all(np.isnan(np.delete(rec[1], to.ITER)))


# ---------------------------------------------------------------- 7. envelope
def test_shared_memory_limit(ctx):
    from muse_psfr_b200 import _lib
    tpl = psf_template()
    truth = np.array([900.0, 23.6, 24.2, 0.3])
    img = to.model(truth, tpl, (48, 48), True)
    rec = tfit(ctx, img[None], np.ones((1, 48, 48)), tpl, True)[0]
    assert rec[to.ITER] > 0
    assert np.all(np.abs(theta_of(rec, True)[1:3] - truth[1:3]) < 1e-9)
    big = np.ones((2, 49, 49))
    out, mo = np.full((2, _lib.TFIT_NPAR), SENT), np.full((2, 49, 49), SENT)
    with pytest.raises(_lib.PsfrError) as e:
        ctx.template_fit(2, 49, 49, big, big, tpl[None], out, mo, fit_back=True)
    assert e.value.code == _lib.E_UNSUPPORTED and 'shared memory' in str(e.value)
    assert np.all(out == SENT) and np.all(mo == SENT)


def test_refusals_before_launch(ctx):
    from muse_psfr_b200 import _lib
    lib, h = ctx._lib, ctx._handle()
    img, tpl = np.ones((4, 9, 9)), np.ones((2, 8, 8))
    out, mo = np.full((4, _lib.TFIT_NPAR), SENT), np.full((4, 9, 9), SENT)
    I, T, O, M = img.ctypes.data, tpl.ctypes.data, out.ctypes.data, mo.ctypes.data
    calls = [
        (4, 9, 9, None, None, 2, 8, 8, T, 1, O, M),       # NULL imgs
        (4, 9, 9, I, None, 2, 8, 8, None, 1, O, M),       # NULL tpls
        (4, 9, 9, I, None, 2, 8, 8, T, 1, None, M),       # NULL params
        (0, 9, 9, I, None, 2, 8, 8, T, 1, O, M),          # nimg < 1
        (4, 2, 9, I, None, 2, 8, 8, T, 1, O, M),          # ny < 3
        (4, 9, 2, I, None, 2, 8, 8, T, 1, O, M),          # nx < 3
        (4, 9, 9, I, None, 0, 8, 8, T, 1, O, M),          # ntpl < 1
        (4, 9, 9, I, None, 3, 8, 8, T, 1, O, M),          # nimg % ntpl != 0
        (4, 9, 9, I, None, 2, 3, 8, T, 1, O, M),          # ty < 4
        (4, 9, 9, I, None, 2, 8, 3, T, 1, O, M),          # tx < 4
    ]
    for args in calls:
        assert lib.psfr_template_fit(h, *args, None) == _lib.E_ARG, args
    assert np.all(out == SENT) and np.all(mo == SENT)


# ---------------------------------------------------------------- 8. the workflow
def test_workflow_reconstructed_star(psfrec):
    lam = np.linspace(500, 900, 8)
    _, cube = psfrec.compute_psf_batch(lam, [0.9], [0.6], [22.])
    _, other = psfrec.compute_psf_batch(lam, [1.4], [0.6], [22.])         # a different seeing
    psf, wrong = cube[0], other[0]
    truth_flux, sky = 5e4, 3.0
    star = np.stack([to.model(np.array([truth_flux, 12.3, 11.6, sky]), psf[k], (25, 25), True) for k in range(8)])
    var = 4.0 + star / 1.5
    rng = np.random.default_rng(77)
    noisy = star + rng.normal(size=star.shape) * np.sqrt(var)
    mask = rng.random(star.shape) < 0.02
    tab, model = psfrec.fit_psf_template(lam, noisy, psf, var=var, mask=mask, fit_back=True, return_model=True)
    assert np.all(tab['converged'] == 1)
    assert np.all(np.abs(tab['flux'] - truth_flux) <= 4 * tab['err_flux'])
    assert np.all(np.abs(tab['cont'] - sky) <= 4 * tab['err_cont'])
    assert np.all(np.abs(tab['center'] - [12.3, 11.6]) <= 4 * tab['err_center'])
    assert np.all(tab['npix'] == 625 - mask.reshape(8, -1).sum(axis=1))
    dof = tab['npix'] - 4
    red = tab['chisq'] / dof
    assert np.all(np.abs(red - 1) < 5 * np.sqrt(2 / dof)), red
    resid = (noisy - model)[~mask]
    assert abs(resid.mean()) < 0.1 * np.sqrt(var).mean()
    bad = psfrec.fit_psf_template(lam, noisy, wrong, var=var, mask=mask, fit_back=True)
    assert np.all(bad['chisq'] / dof > 2 * red)
    assert np.all(bad['qfit'] > 1.5 * tab['qfit'])


# ---------------------------------------------------------------- 9. a full template cube in a fresh context
def test_full_template_cube_fresh_context(psfrec):
    """One [3681, 40, 40] host template cube (a MUSE cube's wavelengths) through fit_psf_template in a new process's
    default context, whose staging buffer holds 16 x 35 = 560 templates: the call sizes the context for them.  Kept
    last in the file: it releases the module's contexts."""
    import torch
    from muse_psfr_b200 import _lib
    nt = 3681
    rng = np.random.default_rng(3681)
    widths = np.linspace(2.8, 1.9, nt)
    tpls = np.stack([psf_template(a=a) for a in widths])
    truth = np.array([3e3, 5.4, 5.7, 1.0])
    var = 4.0 + np.abs(to.model(truth, tpls[nt // 2], (11, 11), True)) / 2
    stamps = np.stack([to.model(truth, tpls[k], (11, 11), True) for k in range(nt)])
    stamps += rng.normal(size=stamps.shape) * np.sqrt(var)
    psfrec.release_contexts()
    tab = psfrec.fit_psf_template(np.linspace(490, 930, nt), stamps, tpls, var=var, fit_back=True)
    ctx = psfrec.get_context()
    assert ctx.max_planes * ctx.max_lambda >= nt
    assert np.all(tab['converged'] == 1) and np.all(tab['npix'] == 121)
    # the same records as device templates give
    w = np.broadcast_to(1 / var, stamps.shape).copy()
    ref = np.full((nt, _lib.TFIT_NPAR), SENT)
    ctx.template_fit(nt, 11, 11, stamps, w, torch.from_numpy(tpls).cuda(), ref, None, fit_back=True)
    assert_bits(tab['flux'], ref[:, to.FLUX])
    assert_bits(tab['center'], ref[:, [to.Y0, to.X0]])
    assert_bits(tab['chisq'], ref[:, to.CHISQ])
