"""CPU reference of the elliptical Moffat fit (psfr_moffat_fit_elliptical): scipy.optimize.leastsq over
theta = (I, y0, x0, A, B, C, n) of f = I (1 + A dp^2 + B dq^2 + C dp dq)^(-n), dp = p - y0 (row), dq = q - x0
(column), started from the oracle's circular solution, and the derived quantities with their delta-method
errors, laid out as the library's PSFR_EFIT_* record.  Also renders exact elliptical Moffat images.

The reference has no elliptical fit; this module restates the library's definitions (DESIGN.md section 5.3)
independently of its CUDA implementation."""
import numpy as np
from scipy.optimize import leastsq

import psfr_oracle as orc

NPAR = 24
(PEAK, Y0, X0, A_MAJOR, A_MINOR, PA, N, FWHM_MAJOR, FWHM_MINOR, AXIS_RATIO, CHISQ, ITER,
 ERR_PEAK, ERR_Y0, ERR_X0, ERR_A_MAJOR, ERR_A_MINOR, ERR_PA, ERR_N, ERR_FWHM_MAJOR, ERR_FWHM_MINOR,
 ERR_AXIS_RATIO, FLUX, ERR_FLUX) = range(NPAR)


def quad_form(a_major, a_minor, pa_deg):
    """(A, B, C) of an ellipse with semi-axes a_major, a_minor [px] whose major axis makes pa_deg with +x
    (column), counted toward +y (row)."""
    t = np.deg2rad(pa_deg)
    c, s = np.cos(t), np.sin(t)
    iM, im = 1 / a_major ** 2, 1 / a_minor ** 2
    return s * s * iM + c * c * im, c * c * iM + s * s * im, 2 * c * s * (iM - im)


def model(theta, p, q):
    I, y0, x0, A, B, C, n = theta
    dp, dq = p - y0, q - x0
    return I * (1 + A * dp * dp + B * dq * dq + C * dp * dq) ** (-n)


def render(shape, I, y0, x0, a_major, a_minor, pa_deg, n):
    """Exact elliptical Moffat image [ny, nx]."""
    p, q = np.indices(shape, dtype=float)
    return model((I, y0, x0) + tuple(quad_form(a_major, a_minor, pa_deg)) + (n,), p, q)


def jacobian(theta, p, q):
    I, y0, x0, A, B, C, n = theta
    dp, dq = p - y0, q - x0
    u = 1 + A * dp * dp + B * dq * dq + C * dp * dq
    m = u ** (-n)
    f = I * m
    g = n * f / u
    return np.stack([m, g * (2 * A * dp + C * dq), g * (2 * B * dq + C * dp), -g * dp * dp, -g * dq * dq,
                     -g * dp * dq, -f * np.log(u)], axis=1)


def record(theta, jtj, chisq, dof):
    """The PSFR_EFIT_* record of a solution theta (ITER is left at 0)."""
    I, y0, x0, A, B, C, n = theta
    hd, hc, S = (A - B) / 2, C / 2, (A + B) / 2
    R2 = hd * hd + hc * hc
    R = np.sqrt(R2)
    lmin, lmax = S - R, S + R
    amaj, amin = 1 / np.sqrt(lmin), 1 / np.sqrt(lmax)
    pa = 0.0
    if R2 != 0:
        pa = np.degrees(0.5 * np.arctan2(-C, A - B) % np.pi) % 180.0
    kf = 2 * np.sqrt(2 ** (1 / n) - 1)
    dkf = -2 * 2 ** (1 / n) * np.log(2) / (n * n * kf)
    q = np.sqrt(lmin / lmax)
    flux = np.pi * I * amaj * amin / (n - 1)
    o = np.zeros(NPAR)
    o[[PEAK, Y0, X0, A_MAJOR, A_MINOR, PA, N, FWHM_MAJOR, FWHM_MINOR, AXIS_RATIO, CHISQ, FLUX]] = \
        [I, y0, x0, amaj, amin, pa, n, amaj * kf, amin * kf, q, chisq, flux]
    sigma = np.linalg.inv(jtj) * abs(chisq / dof)

    def err(g):
        g = np.asarray(g, dtype=float)
        return np.sqrt(abs(g @ sigma @ g))
    e = np.eye(7)
    ca, cc = (hd / (2 * R), hc / (2 * R)) if R > 0 else (0.0, 0.0)
    gmaj, gmin = -0.5 * amaj ** 3, -0.5 * amin ** 3
    g_amaj = np.array([0, 0, 0, gmaj * (0.5 - ca), gmaj * (0.5 + ca), -gmaj * cc, 0])
    g_amin = np.array([0, 0, 0, gmin * (0.5 + ca), gmin * (0.5 - ca), gmin * cc, 0])
    o[ERR_PEAK], o[ERR_Y0], o[ERR_X0], o[ERR_N] = err(e[0]), err(e[1]), err(e[2]), err(e[6])
    o[ERR_A_MAJOR], o[ERR_A_MINOR] = err(g_amaj), err(g_amin)
    if R2 == 0:
        o[ERR_PA] = np.inf
    else:
        k = np.degrees(0.5 / (4 * R2))
        o[ERR_PA] = err([0, 0, 0, k * C, -k * C, -k * (A - B), 0])
    o[ERR_FWHM_MAJOR] = err(kf * g_amaj + amaj * dkf * e[6])
    o[ERR_FWHM_MINOR] = err(kf * g_amin + amin * dkf * e[6])
    o[ERR_AXIS_RATIO] = err(q * (g_amin / amin - g_amaj / amaj))
    det = A * B - hc * hc
    fd = -flux / (2 * det)
    o[ERR_FLUX] = err([np.pi * amaj * amin / (n - 1), 0, 0, fd * B, fd * A, -fd * hc, -flux / (n - 1)])
    return o


def moffat_fit_elliptical(img, start=None):
    """Least-squares elliptical Moffat fit of one image from the oracle's circular solution (or ``start``,
    theta); returns (record [NPAR], theta)."""
    img = np.asarray(img, dtype=float)
    p, q = np.indices(img.shape, dtype=float)
    p, q, data = p.ravel(), q.ravel(), img.ravel()
    if start is None:
        v = orc.moffat_fit(img)['v']
        start = np.array([v[0], v[1], v[2], 1 / v[3] ** 2, 1 / v[3] ** 2, 0.0, v[4]])
    theta = leastsq(lambda t: model(t, p, q) - data, np.array(start, dtype=float),
                         Dfun=lambda t: jacobian(t, p, q), xtol=1e-15, ftol=1e-15, gtol=0.0, maxfev=10000)[0]
    r = model(theta, p, q) - data
    J = jacobian(theta, p, q)
    return record(theta, J.T @ J, float(r @ r), data.size - 7), theta
