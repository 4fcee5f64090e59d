"""CPU reference of the elliptical Moffat fit (psfr_moffat_fit_elliptical): scipy.optimize.leastsq over
theta = (I, y0, x0, A, B, C, n) of f = I (1 + A dp^2 + B dq^2 + C dp dq)^(-n), dp = p - y0 (row), dq = q - x0
(column), started from the oracle's circular solution, and the derived quantities with their delta-method
errors, laid out as the library's PSFR_EFIT_* record.  Also renders exact and noisy elliptical Moffat images,
recomputes a record in long double from given parameters (``record_ld``), and guards known-answer images against
ill-posed fits (``well_posed``).

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


def record(theta, jtj, chisq, dof, inv=np.linalg.inv):
    """The PSFR_EFIT_* record of a solution theta (ITER is left at 0).  The arithmetic follows the dtype of theta
    and jtj; ``inv`` inverts jtj in that dtype."""
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
    sigma = inv(jtj) * abs(chisq / dof)

    def err(g):
        g = np.asarray(g, dtype=sigma.dtype)
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


def render_noisy(shape, truth, sigma, seed):
    """``render(shape, *truth)`` plus seeded Gaussian noise of standard deviation ``sigma`` (pixels may go
    negative)."""
    rng = np.random.default_rng(seed)
    return render(shape, *truth) + rng.normal(0.0, sigma, shape)


def theta_of(I, y0, x0, a_major, a_minor, pa_deg, n):
    """theta = (I, y0, x0, A, B, C, n) of render() arguments."""
    return np.array((I, y0, x0) + tuple(quad_form(a_major, a_minor, pa_deg)) + (n,), dtype=float)


def theta_of_record(rec):
    """theta = (I, y0, x0, A, B, C, n) of a record's peak, centre, semi-axes, PA and n."""
    return theta_of(*(rec[s] for s in (PEAK, Y0, X0, A_MAJOR, A_MINOR, PA, N)))


LD = np.longdouble


def inv_ld(M):
    """Inverse of a small matrix in long double (Gauss-Jordan with partial pivoting; numpy.linalg has no long
    double)."""
    n = M.shape[0]
    a = np.concatenate([np.array(M, dtype=LD), np.eye(n, dtype=LD)], axis=1)
    for c in range(n):
        r = c + int(np.argmax(np.abs(a[c:, c])))
        a[[c, r]] = a[[r, c]]
        a[c] /= a[c, c]
        for i in range(n):
            if i != c:
                a[i] -= a[i, c] * a[c]
    return a[:, n:]


def record_ld(theta, img):
    """The PSFR_EFIT_* record at theta, recomputed in long double: J^T J, chi^2 and dof = npx - 7 over every pixel of
    img, every derived column and every delta-method error (ITER is left at 0)."""
    img = np.asarray(img, dtype=float)
    p, q = (a.ravel().astype(LD) for a in np.indices(img.shape))
    data = img.ravel().astype(LD)
    th = np.asarray(theta, dtype=float).astype(LD)
    J = jacobian(th, p, q)
    r = model(th, p, q) - data
    return record(th, J.T @ J, r @ r, data.size - 7, inv=inv_ld)


def param_scale(theta):
    """Per-parameter scale of theta: |I|, one pixel for the centre, (A + B)/2 for the quadratic form, n."""
    S = 0.5 * (theta[3] + theta[4])
    return np.array([abs(theta[0]), 1.0, 1.0, S, S, S, theta[6]])


# the guard of every known-answer case: the CPU fit must come back from a 1e-3 relative perturbation to within
# WELL_POSED_RTOL of the truth, and the column-scaled J^T J at the truth must have a condition number below
# WELL_POSED_COND.  A solution accurate to 1e-8 from normal equations whose entries carry 1e-16 relative rounding
# needs a scaled condition number well below 1e16; 1e12 keeps four orders of margin.
WELL_POSED_RTOL = 1e-10
WELL_POSED_COND = 1e12


def well_posed(img, truth):
    """Assert that the exact render img of ``truth`` (render() arguments) is a well-posed elliptical fit; return
    the scaled condition number of J^T J at the truth."""
    img = np.asarray(img, dtype=float)
    theta = theta_of(*truth)
    p, q = (a.ravel().astype(float) for a in np.indices(img.shape))
    J = jacobian(theta, p, q)
    jtj = J.T @ J
    d = 1 / np.sqrt(np.diag(jtj))
    cond = np.linalg.cond(jtj * d[:, None] * d[None, :])
    assert cond < WELL_POSED_COND, 'cond(J^T J) = %.3g' % cond
    scale = param_scale(theta)
    start = theta + 1e-3 * scale * np.array([1, -1, 1, 1, -1, 0.5, -1])
    try:
        with np.errstate(all='ignore'):
            _, got = moffat_fit_elliptical(img, start=start)
    except np.linalg.LinAlgError as e:
        raise AssertionError('the fit from the perturbed truth fails: %s' % e)
    dev = np.abs(got - theta) / scale
    assert np.all(np.isfinite(dev)), 'the fit from the perturbed truth is not finite'
    assert np.all(dev <= WELL_POSED_RTOL), 'the fit stops %.3g (relative) from the truth' % dev.max()
    return cond


# ---- the seeded parameter grid of the GPU envelope tests (tests/test_gpu_shape_envelope.py)
GRID_A_MAJOR = (0.7, 1.5, 3.0, 8.0, 15.0)
GRID_Q = (0.999, 0.9, 0.5, 0.2)
GRID_N = (1.05, 1.5, 2.5, 4.0, 10.0)
GRID_PA = (0.0, 1e-7, 45.0, 90.0 - 1e-6, 90.0, 90.0 + 1e-6, 135.0, 180.0 - 1e-7)
# centre offsets from (ny // 2, nx // 2): a pixel centre, a pixel corner, an arbitrary sub-pixel position
GRID_CENTRE = ((0.0, 0.0), (0.5, -0.5), (0.3137, -0.2718))
GRID_CASES = 80
# Cases of grid() that fail well_posed, removed from the GPU comparison.  Every one has n = 10 and a minor
# semi-axis of at most 0.7 px off a pixel centre: the core sits inside one pixel, the intensity, width and n columns
# of J are nearly parallel, and the scaled cond(J^T J) is 6e13 to 6e16, above WELL_POSED_COND.
GRID_REMOVED = {(40, 40): (4, 6, 13, 38, 49, 68), (17, 17): (6, 40)}


def grid(shape):
    """The seeded subset of GRID_A_MAJOR x GRID_Q x GRID_N x GRID_PA x GRID_CENTRE for images of ``shape``:
    GRID_CASES render() argument tuples, each axis cycled through seeded permutations so that every value of every
    axis occurs at least GRID_CASES // 8 times.  Returns (kept, removed) lists of (index, truth)."""
    rng = np.random.default_rng(shape[0])
    axes = (GRID_A_MAJOR, GRID_Q, GRID_N, GRID_PA, GRID_CENTRE)
    cols = [np.concatenate([rng.permutation(len(a)) for _ in range(GRID_CASES // len(a) + 1)])[:GRID_CASES]
            for a in axes]
    kept, removed = [], []
    for i in range(GRID_CASES):
        a, q, n, pa, (dy, dx) = (ax[c[i]] for ax, c in zip(axes, cols))
        truth = (1.0 + 0.01 * i, shape[0] // 2 + dy, shape[1] // 2 + dx, a, a * q, pa, n)
        (removed if i in GRID_REMOVED[tuple(shape)] else kept).append((i, truth))
    return kept, removed
