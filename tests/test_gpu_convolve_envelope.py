"""GPU tests of the two Moffat convolutions (fft_convolve_kernel, csrc/psfr_conv.cu) across their whole input
envelope, against the long-double restatement of tests/conv_oracle.py.

The stage is pure FP64 and linear, so it is held to 1e-14 * sum|img| * max(K) per pixel (``conv_oracle.bar``),
K the largest kernel value of the pair: about 1e5 times tighter than the 1e-9-of-the-peak bar of the parity
tests, and still some 1e8 times below a misplaced wing value.  Each test prints its worst error as a fraction of
that bar.  The inputs break the point symmetry every pipeline PSF has: impulses at every pixel, signed, one-sided
and Nyquist images.  Identities that hold exactly (power-of-two scaling, in-place, per-image independence, the
per-image kernel indexing and the MUSE-kernel cache) are compared bit for bit, and inputs outside the kernels'
domain are refused with every output left as it was."""
import numpy as np
import pytest

import conv_oracle as co

pytestmark = pytest.mark.gpu

ALPHA_LO, ALPHA_HI = 0.043927131328125577, 1.5988674591100165   # tiptilt_alpha(0.4, 0.95, 9), (2.0, 0.3, 29)
LAM6 = np.linspace(490, 930, 35)[::6]
N = 40


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


def new_context(psfrec, max_planes=N, max_lambda=N):
    from muse_psfr_b200 import _lib
    ctx = _lib.Context(device=0, dim=1280, max_planes=max_planes, max_lambda=max_lambda)
    ctx.set_geometry(*psfrec.ao_frequency_tables())
    return ctx


@pytest.fixture(scope='module')
def ctx(psfrec):
    c = new_context(psfrec)
    yield c
    c.close()


def convolve(ctx, lam, alpha, cube):
    cube = np.ascontiguousarray(cube, dtype=np.float64)
    out = np.full_like(cube, np.nan)
    ctx.convolve(cube.shape[0], np.asarray(lam, dtype=float), np.asarray(alpha, dtype=float), cube, out)
    return out


def report(name, ratio):
    print('\n%s: worst error / bar = %.3e' % (name, ratio))
    assert ratio < 1, name


def test_tiptilt_alphas_are_the_config4_extremes(psfrec):
    assert psfrec.tiptilt_alpha(0.4, 0.95, 9.0) == ALPHA_LO and psfrec.tiptilt_alpha(2.0, 0.3, 29.0) == ALPHA_HI


# ---------------------------------------------------------------- 1. the whole linear operator, pixel by pixel
@pytest.mark.parametrize('lam', [465.0, 490.0, 700.0, 930.0, 1100.0, 1130.0, 1150.0, 1180.0, 250.0])
def test_impulse_response_matrix(ctx, lam):
    """40 draws x 40 copies of one wavelength = the 1600 unit impulses: image (d, l) is the impulse at pixel (d, l).
    With alpha_tt = 1e-9 the tip-tilt kernel is a delta to ~1e-36, so the answer is the shifted, cropped MUSE
    kernel: the stage's full 1600 x 1600 matrix, with no arithmetic in the reference."""
    cube = np.eye(N * N).reshape(N, N, N, N)
    out = convolve(ctx, [lam] * N, [1e-9] * N, cube)
    K = co.muse_kernel(lam)
    ref = co.same_matrix(K).reshape(N, N, N, N)
    err = np.abs(out - ref).max()
    report('impulse matrix %g nm' % lam, err / co.bar(cube[0, 0], K))
    assert np.isfinite(out).all()


def edge_and_interior(seed=11, ninterior=100):
    edge = [(i, j) for i in range(N) for j in range(N) if i in (0, N - 1) or j in (0, N - 1)]
    inner = [(i, j) for i in range(1, N - 1) for j in range(1, N - 1)]
    rng = np.random.default_rng(seed)
    pick = rng.choice(len(inner), ninterior, replace=False)
    return edge + [inner[k] for k in sorted(pick)]


@pytest.mark.parametrize('alpha,lams,interior', [(ALPHA_LO, (490.0, 930.0), 100), (ALPHA_HI, (490.0, 930.0), 100),
                                                 (1e3, (700.0,), 0)])
def test_impulses_through_both_passes(ctx, alpha, lams, interior):
    """The 156 edge pixels and seeded interior impulses through a real tip-tilt kernel, then the MUSE kernel.
    The first pass of an impulse is exact (the shifted, cropped tip-tilt kernel); the second is summed in long
    double.  alpha_tt = 1e3 is nearly flat over the 41 x 41 kernel."""
    pix = edge_and_interior(ninterior=interior)
    assert len(pix) == 156 + interior
    ktt = co.tiptilt_kernel(alpha)
    step1 = np.stack([co.shifted_kernel(ktt, i, j) for i, j in pix])
    worst = 0.0
    for lam in lams:
        kmu = co.muse_kernel(lam)
        ref = co.convolve_same(step1, kmu)
        for c0 in range(0, len(pix), N):
            chunk = pix[c0:c0 + N]
            cube = np.zeros((len(chunk), 1, N, N))
            for k, (i, j) in enumerate(chunk):
                cube[k, 0, i, j] = 1
            out = convolve(ctx, [lam], [alpha] * len(chunk), cube)
            worst = max(worst, np.abs(out[:, 0] - ref[c0:c0 + N]).max() / co.bar(cube[0], ktt, kmu))
    report('impulses alpha_tt %g' % alpha, worst)


# ---------------------------------------------------------------- 2. asymmetric and signed inputs
def asymmetric_images():
    rng = np.random.default_rng(23)
    imgs = [rng.standard_normal((N, N)) * s for s in (1.0, 1e-3, 37.0, 2.0)]      # seeded random signed
    for cy, cx in ((0, 0), (0, N - 7), (N - 7, 0), (N - 7, N - 7)):                  # all energy in one corner
        img = np.zeros((N, N))
        img[cy:cy + 7, cx:cx + 7] = rng.uniform(0, 1, (7, 7))
        imgs.append(img)
    row, col = np.zeros((N, N)), np.zeros((N, N))
    row[3] = rng.uniform(-1, 1, N)
    col[:, 36] = rng.uniform(-1, 1, N)
    y, x = np.indices((N, N))
    imgs += [row, col, (-1.0) ** (y + x), (-1.0) ** y, (-1.0) ** x]                # checkerboards: Nyquist bins
    return np.stack(imgs)


@pytest.mark.parametrize('alpha', [ALPHA_LO, ALPHA_HI, 1e3])
def test_asymmetric_and_signed_inputs(ctx, alpha):
    imgs = asymmetric_images()
    lams = [490.0, 930.0]
    cube = np.ascontiguousarray(np.repeat(imgs[:, None], len(lams), axis=1))
    out = convolve(ctx, lams, [alpha] * len(imgs), cube)
    ktt = co.tiptilt_kernel(alpha)
    worst = 0.0
    for li, lam in enumerate(lams):
        kmu = co.muse_kernel(lam)
        ref = co.two_pass(imgs, alpha, lam, kernels=(ktt, kmu))
        for k in range(len(imgs)):
            worst = max(worst, np.abs(out[k, li] - ref[k]).max() / co.bar(imgs[k], ktt, kmu))
    report('asymmetric inputs alpha_tt %g' % alpha, worst)


# ---------------------------------------------------------------- 3. exact identities
def signed_cube(nd, nl, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal((nd, nl, N, N)) * rng.uniform(0.1, 10, (nd, nl, 1, 1))


def test_power_of_two_scaling_is_exact(ctx):
    """Every rounding of the transform commutes with a scaling by 2^+-400 (no overflow or underflow on the way)."""
    cube = signed_cube(5, 3, 31)
    lam, alpha = [490.0, 700.0, 930.0], [ALPHA_LO, 0.3, 0.9, ALPHA_HI, 1e3]
    out = convolve(ctx, lam, alpha, cube)
    for e in (400, -400):
        s = np.ldexp(1.0, e)
        assert np.array_equal(convolve(ctx, lam, alpha, cube * s), out * s), e


def test_in_place_and_device_paths_equal_the_host_path(ctx):
    import torch
    cube = signed_cube(6, 4, 37)
    lam, alpha = [490.0, 610.0, 800.0, 1150.0], [0.05, 0.2, 0.7, 1.1, ALPHA_HI, 40.0]
    out = convolve(ctx, lam, alpha, cube)
    buf = torch.from_numpy(cube).cuda()
    dst = torch.full_like(buf, float('nan'))
    ctx.convolve(6, np.array(lam), np.array(alpha), buf, dst)
    ctx.convolve(6, np.array(lam), np.array(alpha), buf, buf)
    torch.cuda.synchronize()
    assert np.array_equal(dst.cpu().numpy(), out) and np.array_equal(buf.cpu().numpy(), out)


def test_nan_stays_in_its_image(ctx):
    cube = signed_cube(4, 3, 41)
    lam, alpha = [490.0, 700.0, 930.0], [0.05, 0.5, 1.5, 3.0]
    out = convolve(ctx, lam, alpha, cube)
    cube[2, 1, 5, 33] = np.nan
    got = convolve(ctx, lam, alpha, cube)
    assert np.isnan(got[2, 1]).all()
    keep = np.ones((4, 3), bool)
    keep[2, 1] = False
    assert np.array_equal(got[keep], out[keep])


# ---------------------------------------------------------------- 4. kernel indexing at capacity
def test_every_image_at_capacity_uses_its_own_kernels(ctx):
    """max_planes x max_lambda images, a distinct alpha_tt per draw and a distinct wavelength per slot: each image
    equals a one-image call with its own (alpha, lambda), bit for bit."""
    alpha = np.geomspace(0.03, 30.0, N)
    lam = np.linspace(465.0, 1180.0, N)
    cube = np.abs(signed_cube(N, N, 43))
    out = convolve(ctx, lam, alpha, cube)
    one = np.empty((1, 1, N, N))
    for d in range(N):
        for k in range(N):
            ctx.convolve(1, lam[[k]], alpha[[d]], np.ascontiguousarray(cube[d, k][None, None]), one)
            assert np.array_equal(one[0, 0], out[d, k]), (d, k)


def test_field_chunk_indexes_tiptilt_per_draw(psfrec):
    """One compute_field chunk (a draw owns ndir x nlam images): four draws of the same turbulence with distinct
    alpha_tt, each position against compute_batch of that draw alone, bit for bit."""
    from muse_psfr_b200 import _lib
    nd, lam = 4, LAM6[:5]
    pos = np.array([[0.0, -30.0, 12.5], [0.0, 30.0, -7.3]])
    recs = psfrec._mode_records(np.zeros(nd, bool), np.full(nd, 1.0), np.full(nd, 0.7), np.full(nd, 25.0))
    recs[:, _lib.DRAW_ALPHA_TT] = [0.05, 0.4, 1.2, 3.0]
    lgs = psfrec._lgs_positions(False)
    ctx = new_context(psfrec, max_planes=nd * pos.shape[1])
    try:
        cube = np.full((nd, pos.shape[1], lam.size, N, N), np.nan)
        ctx.compute_field(recs, pos, lgs, lam, out_cube=cube)
        for d in range(nd):
            for k in range(pos.shape[1]):
                ref = np.full((1, lam.size, N, N), np.nan)
                ctx.compute_batch(recs[[d]], np.ascontiguousarray(pos[:, [k]]), lgs, lam, out_cube=ref)
                assert np.array_equal(cube[d, k], ref[0]), (d, k)
    finally:
        ctx.close()
    for d in range(1, nd):
        assert not np.array_equal(cube[d], cube[0])


# ---------------------------------------------------------------- 5. the MUSE-kernel cache
def test_muse_kernel_cache(psfrec):
    """One context through wavelength sets A, B (A with one value changed), a permutation of A, a compute_batch on A
    and A again: each result equals a fresh context's, bit for bit; so does A after a refused call."""
    from muse_psfr_b200 import _lib
    A = LAM6.copy()
    B = A.copy()
    B[3] = 712.5
    P = A[[4, 0, 5, 2, 1, 3]]
    cube, alpha = signed_cube(2, A.size, 47), [0.3, ALPHA_HI]
    recs = psfrec._mode_records(np.zeros(2, bool), np.array([0.8, 1.3]), np.array([0.7, 0.5]), np.array([22.0, 14.0]))
    dirs, lgs = np.zeros((2, 1)), psfrec._lgs_positions(False)

    def batch(c, lam):
        out = np.full((2, len(lam), N, N), np.nan)
        c.compute_batch(recs, dirs, lgs, np.asarray(lam), out_cube=out)
        return out

    def fresh(fn, lam):
        c = new_context(psfrec, max_planes=4)
        try:
            return fn(c, lam)
        finally:
            c.close()

    conv = lambda c, lam: convolve(c, lam, alpha, cube)   # noqa: E731
    ctx = new_context(psfrec, max_planes=4)
    try:
        steps = [(conv, A), (conv, B), (conv, P), (batch, A), (conv, A)]
        for n, (fn, lam) in enumerate(steps):
            assert np.array_equal(fn(ctx, lam), fresh(fn, lam)), n
        ref_a, ref_batch = conv(ctx, A), batch(ctx, A)
        bad = A.copy()
        bad[2] = 1200.0
        for fn in (conv, batch):
            with pytest.raises(_lib.PsfrError) as exc:
                fn(ctx, bad)
            assert exc.value.code == _lib.E_UNSUPPORTED
            assert np.array_equal(conv(ctx, A), ref_a) and np.array_equal(batch(ctx, A), ref_batch)
    finally:
        ctx.close()


# ---------------------------------------------------------------- 6. refusals
BAD_LAMBDA = [1189.0, 1200.0, 2002.0, 7760.0]
BAD_ALPHA = [0.0, -1.0, np.nan, np.inf, 1e-170, 1e160, 1e154, 8e-155]


def nan_outputs(shape_host):
    import torch
    return np.full(shape_host, np.nan), torch.full(shape_host, float('nan'), dtype=torch.float64, device='cuda')


def test_convolve_refuses_outside_the_domain(ctx):
    import torch
    from muse_psfr_b200 import _lib
    cube = signed_cube(2, 3, 53)
    cases = [([490.0, lb, 930.0], [0.5, 1.0], _lib.E_UNSUPPORTED) for lb in BAD_LAMBDA]
    cases += [([490.0, lb, 930.0], [0.5, 1.0], _lib.E_ARG) for lb in (0.0, -500.0, np.nan, np.inf)]
    cases += [([490.0, 700.0, 930.0], [0.5, a], _lib.E_ARG) for a in BAD_ALPHA]
    dev_in = torch.from_numpy(cube).cuda()
    for lam, alpha, code in cases:
        host, dev = nan_outputs(cube.shape)
        for src, dst in ((cube, host), (dev_in, dev), (cube, dev), (dev_in, host)):
            with pytest.raises(_lib.PsfrError) as exc:
                ctx.convolve(2, np.array(lam), np.array(alpha), src, dst)
            assert exc.value.code == code, (lam, alpha)
        torch.cuda.synchronize()
        assert np.isnan(host).all() and torch.isnan(dev).all(), (lam, alpha)
    # the edges of the domain are accepted: pi alpha^2 just normal or just finite, lambda just below the beta root
    out = convolve(ctx, [490.0, 1188.9, 930.0], [9e-155, 7.5e153], cube)
    assert np.isfinite(out).all()


def test_python_batch_and_field_refuse(psfrec):
    """compute_psf_batch / compute_psf_field past the beta root, or with GL = 1 (alpha_tt = 0) or GL > 1 (NaN),
    raise and leave the caller's outputs untouched."""
    from muse_psfr_b200 import _lib
    cases = [(dict(lbda=[490.0, lb]), ValueError) for lb in BAD_LAMBDA]
    cases += [(dict(GL=[0.7, g]), _lib.PsfrError) for g in (1.0, 1.2)]
    for kw, err in cases:
        args = dict(lbda=[490.0, 930.0], seeing=[1.0, 0.8], GL=[0.7, 0.5], L0=[25.0, 20.0])
        args.update(kw)
        nl = len(args['lbda'])
        cube, fit = np.full((2, nl, N, N), np.nan), np.full((2, nl, _lib.FIT_NPAR), np.nan)
        with pytest.raises(err) as exc, np.errstate(all='ignore'):
            psfrec.compute_psf_batch(**args, out_cube=cube, out_fit=fit)
        if err is _lib.PsfrError:
            assert exc.value.code == _lib.E_ARG
        assert np.isnan(cube).all() and np.isnan(fit).all(), kw
        pos = np.array([[0.0, 12.5], [0.0, -7.3]])
        cube, fit = np.full((2, 2, nl, N, N), np.nan), np.full((2, 2, nl, _lib.FIT_NPAR), np.nan)
        with pytest.raises(err), np.errstate(all='ignore'):
            psfrec.compute_psf_field(**args, positions=pos, out_cube=cube, out_fit=fit)
        assert np.isnan(cube).all() and np.isnan(fit).all(), kw


def test_energy_and_ao_refuse(psfrec):
    """psfr_compute_energy / psfr_compute_ao in both modes, with NaN-filled host and device outputs."""
    import torch
    from muse_psfr_b200 import _lib
    recs = psfrec._mode_records(np.zeros(3, bool), np.array([1.0, 0.6, 1.5]), np.array([0.7, 0.5, 0.8]),
                                np.array([25.0, 12.0, 18.0]))
    pos, lgs, ge = np.array([[0.0, 12.5], [0.0, -7.3]]), psfrec._lgs_positions(False), np.array([1, 3], np.int32)
    rad, fr = np.array([1.0, 3.5]), np.array([0.5])
    cases = [(recs, [490.0, lb], _lib.E_UNSUPPORTED) for lb in BAD_LAMBDA]
    for a in BAD_ALPHA:
        r = recs.copy()
        r[1, _lib.DRAW_ALPHA_TT] = a
        cases.append((r, [490.0, 930.0], _lib.E_ARG))
    ctx = new_context(psfrec, max_planes=4)
    try:
        for field in (False, True):
            P = pos.shape[1] if field else 1
            for r, lam, code in cases:
                nl = len(lam)
                shapes = dict(out_cube=(3, P, nl, N, N), out_fit=(3, P, nl, _lib.FIT_NPAR),
                              out_mean=(2, P, nl, N, N), out_mean_fit=(2, P, nl, _lib.FIT_NPAR),
                              out_ee=(3, P, nl, 4), out_mean_ee=(2, P, nl, 4))
                ao = dict(out_strehl=(3, P, nl), out_var=(3, pos.shape[1], _lib.VAR_NPAR))
                for fn, extra in ((ctx.compute_energy, {}), (ctx.compute_ao, ao)):
                    for side in (0, 1):
                        out = {k: nan_outputs(s)[side] for k, s in dict(shapes, **extra).items()}
                        with pytest.raises(_lib.PsfrError) as exc:
                            fn(field, r, pos, lgs, np.array(lam), rad, fr, ge, **out)
                        assert exc.value.code == code, (field, lam, fn)
                        torch.cuda.synchronize()
                        for k, v in out.items():
                            assert bool(np.isnan(v).all() if side == 0 else torch.isnan(v).all()), (k, lam)
        # psfr_psd never reads alpha_tt and keeps accepting such records
        psd = np.empty((1, 1280, 1280))
        ctx.psd(cases[-1][0][1:2], np.zeros((2, 1)), lgs, out=psd)
        assert np.isfinite(psd).all()
    finally:
        ctx.close()


def test_psf_muse_keeps_its_range(psfrec):
    """psf_muse has no convolution: 7760 nm, past the beta root, still works."""
    psd = psfrec.simul_psd_wfm([0.7, 0.3], (100, 10000), 1.0, 25., verbose=False)[0]
    out = psfrec.psf_muse(psd, [7760.0])
    assert np.isfinite(out).all() and abs(out.sum() - 1) < 1e-12
