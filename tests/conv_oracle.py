"""Long-double restatement of the two Moffat convolutions of psfr_convolve (csrc/psfr_conv.cu,
convolve_final_psf psfrec.py:874-930): the kernels and the direct 'same' sums, with no transform.

``muse_params`` evaluates the MUSE polynomials in double exactly as the host code of run_build_kernels does,
so the kernels start from the same (gamma, beta); everything after that is np.longdouble."""
import math

import numpy as np

LD = np.longdouble
KW = 41                 # kernel width
PSF = 40                # image width
C = PSF // 2            # 'same' keeps rows / columns C .. C + PSF - 1 of the full 80 x 80 convolution
POL_BETA = (-0.83704697, 1.1337153, 0.0609222, -1.35581762, 1.15237178, 2.2106042)
POL_FWHM = (0.60467385, -1.58905792, 1.75293264, -1.0368302, 0.21487023, 0.34851139)
TINY = np.finfo(np.float64).tiny


def muse_params(lam):
    """(gamma [px], beta) of the MUSE Moffat at ``lam`` nm: Horner in double, then
    gamma = fwhm / 0.2 / (2 sqrt(2^(1/beta) - 1)) (psfrec.py:923-924, :1160-1168)."""
    lb = (10 * np.float64(lam) - 4750) / np.float64(9350 - 4750)
    fw, be = np.float64(0.0), np.float64(0.0)
    for pf, pb in zip(POL_FWHM, POL_BETA):
        fw = fw * lb + pf
        be = be * lb + pb
    fw, be = float(fw / 0.2), float(be)
    # libm's pow and sqrt as the host calls them (the vectorised np.power can differ by an ulp), with C's
    # results where Python raises
    x = 1.0 / be if be != 0 else math.copysign(math.inf, be)
    try:
        p = math.pow(2.0, x)
    except OverflowError:
        p = math.inf
    s = math.sqrt(p - 1) if p >= 1 else math.nan
    return np.float64(fw / (2 * s)), np.float64(be)


def width_ok(gamma):
    """(pi gamma) gamma is a finite, normal double: the amplitude of moffat_kernels_kernel divides by it."""
    p = math.pi * float(gamma) * float(gamma)
    return bool(math.isfinite(p) and p >= TINY)


def muse_in_domain(lam):
    """The rule of run_build_kernels: beta > 0, beta != 1 and pi gamma^2 finite and normal."""
    gamma, beta = muse_params(lam)
    return bool(beta > 0 and beta != 1 and width_ok(gamma))


def alpha_tt_in_domain(alpha):
    """The rule of psfr_convolve and the batch paths for the tip-tilt width: alpha > 0, pi alpha^2 finite and
    normal."""
    return bool(float(alpha) > 0 and width_ok(alpha))


def moffat_kernel(gamma, beta):
    """41 x 41 Moffat kernel in long double, the formula of oracle.moffat2d_kernel: amplitude
    (beta - 1) / (pi gamma^2) times (1 + r^2 / gamma^2)^(-beta), normalised to unit sum."""
    r = np.arange(KW, dtype=LD) - KW // 2
    g2 = LD(gamma) * LD(gamma)
    b = LD(beta)
    rr = (r[:, None] ** 2 + r[None, :] ** 2) / g2
    k = (b - 1) / (LD(np.pi) * g2) * (1 + rr) ** (-b)
    return k / k.sum()


def tiptilt_kernel(alpha):
    return moffat_kernel(alpha, 2)


def muse_kernel(lam):
    return moffat_kernel(*muse_params(lam))


def same_matrix(K):
    """The 'same' convolution with K as a [PSF^2, PSF^2] matrix: M[(i, j), (y, x)] = K[C + y - i][C + x - j]
    where that index lies inside the kernel, else 0."""
    pad = np.zeros((3 * PSF, 3 * PSF), dtype=LD)
    pad[PSF:PSF + KW, PSF:PSF + KW] = K          # pad[PSF + t] = K[t]
    win = np.lib.stride_tricks.sliding_window_view(pad, (PSF, PSF))
    # the image pixel (i, j) reads the window that starts at (PSF + C - i, PSF + C - j)
    lo = PSF + C - (PSF - 1)
    M = win[lo:lo + PSF, lo:lo + PSF][::-1, ::-1]
    return np.ascontiguousarray(M).reshape(PSF * PSF, PSF * PSF)


def convolve_same(img, K):
    """Direct long-double 'same' convolution of images [..., 40, 40] with the 41 x 41 kernel K."""
    img = np.asarray(img)
    flat = img.reshape(-1, PSF * PSF).astype(LD)
    return (flat @ same_matrix(K)).reshape(img.shape)


def two_pass(img, alpha_tt, lam, kernels=None):
    """Tip-tilt then MUSE convolution of images [..., 40, 40], each cropped to 'same' like the reference.
    ``kernels`` = (K_tt, K_mu) skips building them."""
    ktt, kmu = kernels if kernels is not None else (tiptilt_kernel(alpha_tt), muse_kernel(lam))
    return convolve_same(convolve_same(img, ktt), kmu)


def shifted_kernel(K, i, j):
    """'same' response to the unit impulse at (i, j): K[C + y - i][C + x - j], zero outside the kernel."""
    out = np.zeros((PSF, PSF), dtype=LD)
    y0, y1 = max(0, i - C), min(PSF, i - C + KW)
    x0, x1 = max(0, j - C), min(PSF, j - C + KW)
    out[y0:y1, x0:x1] = K[C + y0 - i:C + y1 - i, C + x0 - j:C + x1 - j]
    return out


def bar(img, *kernels):
    """Per-pixel bound of the FP64 stage: 1e-14 * sum|img| * the largest kernel value."""
    return 1e-14 * float(np.abs(np.asarray(img, dtype=np.float64)).sum()) * max(float(k.max()) for k in kernels)
