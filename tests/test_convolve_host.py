"""CPU tests of the convolution stage's yardsticks and input rules (DESIGN.md section 5, fft_convolve_kernel):
the long-double restatement of tests/conv_oracle.py against the numpy oracle, its MUSE parameters against
np.polyval, the domain of the two Moffat kernels, and the argument checks of Context.convolve that run before
the library is called."""
import numpy as np
import pytest
from scipy.optimize import brentq

import conv_oracle as co
import psfr_oracle as orc
from muse_psfr_b200 import _lib, psfrec

LBDA35 = np.linspace(490, 930, 35)
DRAWS = [(1.0, 0.7, 25.0), (0.4, 0.95, 9.0), (2.0, 0.3, 29.0)]


def signed_images(n, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal((n, 40, 40)) * rng.uniform(0.1, 10, (n, 1, 1))


@pytest.mark.parametrize('draw', DRAWS)
def test_restatement_equals_oracle(golden, draw):
    """two_pass against oracle.convolve_final_psf (scipy fftconvolve) to 1e-15 of the input's L1 norm, on golden
    PSFs and on random signed images."""
    sel = [0, 17, 34]
    lam = LBDA35[sel]
    imgs = np.concatenate([golden('ref_config1')['psf_muse'][sel], signed_images(3, 7)])
    lam6 = np.concatenate([lam, lam])
    ref = np.concatenate([orc.convolve_final_psf(lam, *draw, imgs[:3]), orc.convolve_final_psf(lam, *draw, imgs[3:])])
    alpha = orc.tiptilt_alpha(*draw)
    for k in range(6):
        got = co.two_pass(imgs[k], alpha, lam6[k])
        assert got.dtype == np.longdouble
        assert np.abs(got - ref[k]).max() <= 1e-15 * np.abs(imgs[k]).sum(), k


def test_kernels_are_the_oracle_kernels():
    for lam in (465.0, 700.0, 1130.0, 1180.0, 250.0):
        fwhm, beta = orc.muse_intrinsic_psf(lam)
        gamma = (fwhm / 0.2) / (2 * np.sqrt(2 ** (1. / beta) - 1))
        K = co.muse_kernel(lam)
        assert abs(K.sum() - 1) < 1e-18 and K.min() > 0
        assert np.abs(K - orc.moffat2d_kernel(gamma, beta)).max() <= 1e-15 * K.max(), lam
    for alpha in (1e-9, 0.0439, 1.6, 1e3):
        K = co.tiptilt_kernel(alpha)
        assert np.abs(K - orc.moffat2d_kernel(alpha, 2)).max() <= 1e-15 * K.max(), alpha
    assert co.tiptilt_kernel(1e-9)[20, 20] == 1          # a delta to ~1e-36
    flat = co.tiptilt_kernel(1e3)
    assert flat.max() / flat.min() < 1.002


def test_same_sum_of_an_impulse_is_the_shifted_kernel():
    K = co.muse_kernel(700.0)
    for i, j in [(0, 0), (0, 39), (39, 0), (39, 39), (20, 20), (3, 31), (37, 20)]:
        img = np.zeros((40, 40))
        img[i, j] = 1
        ref = co.shifted_kernel(K, i, j)
        assert np.array_equal(co.convolve_same(img, K), ref)
        assert ref[i, j] == K[20, 20]
        if (i, j) == (20, 20):
            assert np.array_equal(ref, K[:40, :40])
    # the crop: the impulse at the corner keeps 21 x 21 of the kernel's 41 x 41 values
    assert np.count_nonzero(co.shifted_kernel(K, 0, 0)) == 21 * 21


def test_muse_params_match_polyval():
    lam = np.concatenate([np.linspace(240, 7760, 997), [250.0, 303.85, 465.0, 1132.77, 1188.99, 1189.0]])
    fwhm, beta = orc.muse_intrinsic_psf(lam)
    for k, lb in enumerate(lam):
        gamma, be = co.muse_params(lb)
        assert be == beta[k], lb
        with np.errstate(all='ignore'):
            g = (fwhm[k] / 0.2) / (2 * np.sqrt(2 ** (1. / beta[k]) - 1))
        assert gamma == g or (np.isnan(gamma) and np.isnan(g)), lb


def test_domain_roots():
    """beta = 0 at ~1188.99 nm, beta = 1 at ~1132.77 nm, fwhm = 0 at ~303.85 nm."""
    beta0 = brentq(lambda x: co.muse_params(x)[1], 1100, 1300, xtol=1e-9)
    beta1 = brentq(lambda x: co.muse_params(x)[1] - 1, 1100, 1150, xtol=1e-9)
    fwhm0 = brentq(lambda x: orc.muse_intrinsic_psf(x)[0], 250, 400, xtol=1e-9)
    assert round(beta0, 2) == 1188.99 and round(beta1, 2) == 1132.77 and round(fwhm0, 2) == 303.85
    # inside (0, 1) the kernel is finite and positive; past the root gamma is NaN or 0
    assert 0 < co.muse_params(1150.0)[1] < 1 and 0 < co.muse_params(1180.0)[1] < 1
    assert np.isnan(co.muse_params(1200.0)[0]) and co.muse_params(1188.99)[0] == 0


@pytest.mark.parametrize('lam', [1189.0, 1200.0, 2002.0, 7760.0, 1188.99])
def test_muse_domain_refuses(lam):
    assert not co.muse_in_domain(lam)


@pytest.mark.parametrize('lam', [250.0, 465.0, 490.0, 700.0, 930.0, 1100.0, 1130.0, 1150.0, 1180.0, 1188.9])
def test_muse_domain_accepts(lam):
    assert co.muse_in_domain(lam)
    K = co.muse_kernel(lam)
    assert np.isfinite(K).all() and K.min() > 0


def test_muse_domain_isolated_points():
    """The rule's other two exclusions, at the doubles closest to the roots."""
    assert not co.width_ok(0.0) and not co.width_ok(1e-170) and not co.width_ok(1e160)
    # pi gamma^2 overflows before gamma^2 does, and is normal a little below the normal gamma^2
    assert not co.width_ok(1e154) and co.width_ok(7.5e153) and not co.width_ok(8e-155) and co.width_ok(9e-155)
    beta1 = brentq(lambda x: co.muse_params(x)[1] - 1, 1100, 1150, xtol=1e-13)
    near = [beta1 + k * np.spacing(beta1) for k in range(-64, 65)]
    hit = [x for x in near if co.muse_params(x)[1] == 1]
    for x in hit:
        assert not co.muse_in_domain(x)
    assert all(co.muse_in_domain(x) for x in near if x not in hit)


@pytest.mark.parametrize('alpha', [0.0, -1.0, np.nan, np.inf, -np.inf, 1e-170, 1e160, 1e154, 8e-155])
def test_alpha_tt_domain_refuses(alpha):
    assert not co.alpha_tt_in_domain(alpha)


@pytest.mark.parametrize('alpha', [1e-9, 9e-155, 1e-150, 0.0439, 1.6, 1e3, 1e150, 7.5e153])
def test_alpha_tt_domain_accepts(alpha):
    assert co.alpha_tt_in_domain(alpha)


def test_tiptilt_alpha_at_the_ground_layer_limit():
    """GL = 1 gives alpha 0 and GL > 1 NaN: both outside the domain, so the batch paths refuse them."""
    with np.errstate(all='ignore'):
        assert psfrec.tiptilt_alpha(np.array([1.0]), np.array([1.0]), np.array([25.0]))[0] == 0
        assert np.isnan(psfrec.tiptilt_alpha(np.array([1.0]), np.array([1.2]), np.array([25.0]))[0])
    assert co.alpha_tt_in_domain(psfrec.tiptilt_alpha(1.0, 0.999, 25.0))


class _StubLib:
    """Records psfr_convolve calls instead of reaching a device."""

    def __init__(self):
        self.calls = []

    def psfr_convolve(self, *args):
        self.calls.append(args)
        return 0


def stub_context():
    ctx = _lib.Context.__new__(_lib.Context)
    ctx._lib, ctx._h, ctx.device, ctx._geom, ctx._opts = _StubLib(), 1, 0, None, {}
    return ctx


def test_context_convolve_checks_arguments_before_the_call():
    ctx = stub_context()
    lam = np.array([490.0, 700.0])
    cube = np.zeros((3, 2, 40, 40))
    out = np.empty_like(cube)
    bad = [dict(alpha_tt=[1.0, 1.0]),                               # 2 alphas for 3 draws
           dict(cube=cube.astype(np.float32)),
           dict(cube=cube[:, :1].copy()),                           # too few elements
           dict(cube=np.zeros((3, 2, 40, 80))[..., ::2]),          # not contiguous
           dict(out=out[:2]),
           dict(out=np.frombuffer(np.zeros(cube.size).tobytes()))]   # read-only
    for kw in bad:
        args = dict(ndraw=3, lambda_nm=lam, alpha_tt=[1.0, 1.0, 1.0], cube=cube, out=out)
        args.update(kw)
        with pytest.raises(ValueError):
            ctx.convolve(**args)
    assert ctx._lib.calls == []
    ctx.convolve(3, lam, [1.0, 2.0, 3.0], cube, out)
    (call,) = ctx._lib.calls
    assert call[1:3] == (3, 2) and call[-1] is None
    ctx._h = None
    with pytest.raises(_lib.PsfrError) as exc:
        ctx.convolve(3, lam, [1.0, 2.0, 3.0], cube, out)
    assert exc.value.code == _lib.E_STATE


def test_convolve_final_psf_checks_the_shape_first():
    with pytest.raises(NotImplementedError):
        psfrec.convolve_final_psf([490.0, 700.0], 1.0, 0.7, 25.0, np.zeros((3, 40, 40)))
