"""CPU reference of the template fit (psfr_template_fit, DESIGN.md section 5.8): a star stamp d [ny, nx] with weights
w is fitted as m = F s(p - y0 + ty//2, q - x0 + tx//2) / S + c, s the interpolating cubic B-spline of the template
with mirror boundary conditions (scipy.ndimage.map_coordinates(order=3, mode='mirror')), 0 outside the template,
and S the template's sum.  The minimum is found by scipy.optimize.least_squares(method='lm') on sqrt(w) r over the
used pixels (w > 0) with an analytic Jacobian from the restated B-spline taps on spline_filter coefficients, started
from the library's start point.  Records are laid out as PSFR_TFIT_*.

This restates the library's definitions independently of its CUDA implementation."""
import numpy as np
from scipy import ndimage
from scipy.optimize import least_squares

TFIT_NPAR = 12
(FLUX, Y0, X0, CONT, CHISQ, QFIT, ITER, NPIX, ERR_FLUX, ERR_Y0, ERR_X0, ERR_CONT) = range(TFIT_NPAR)


def coefficients(tpl):
    """B-spline coefficients of the template: spline_filter(order=3, mode='mirror')."""
    return ndimage.spline_filter(np.asarray(tpl, dtype=float), order=3, mode='mirror')


def prefilter(tpl):
    """The same coefficients by the recursion the kernel runs (gain, causal recursion from scipy's exact mirror
    initialisation, anticausal recursion; pole sqrt(3) - 2), rows then columns."""
    z = np.sqrt(3.0) - 2.0

    def line(c):
        n = c.size
        c = c * ((1 - z) * (1 - 1 / z))
        zn1 = z ** (n - 1)
        c0 = c[0] + zn1 * c[n - 1]
        zi = z
        for i in range(1, n - 1):
            c0 += zi * (c[i] + zn1 * c[n - 1 - i])
            zi *= z
        c[0] = c0 / (1 - zn1 * zn1)
        for i in range(1, n):
            c[i] += z * c[i - 1]
        c[n - 1] = (z * c[n - 2] + c[n - 1]) * z / (z * z - 1)
        for i in range(n - 2, -1, -1):
            c[i] = z * (c[i + 1] - c[i])
        return c

    c = np.array(tpl, dtype=float)
    c = np.stack([line(r) for r in c])
    return np.stack([line(col) for col in c.T], axis=1)


def sample(tpl, u, v):
    """s(u, v) by map_coordinates(order=3, mode='mirror'), 0 outside [0, ty - 1] x [0, tx - 1]."""
    u, v = np.atleast_1d(np.asarray(u, dtype=float)), np.atleast_1d(np.asarray(v, dtype=float))
    ty, tx = np.shape(tpl)
    out = ndimage.map_coordinates(np.asarray(tpl, dtype=float), [u, v], order=3, mode='mirror')
    inside = (u >= 0) & (u <= ty - 1) & (v >= 0) & (v <= tx - 1)
    return np.where(inside, out, 0.0)


def _weights(t):
    s = 1 - t
    w = np.stack([s ** 3 / 6, 2 / 3 - 0.5 * t * t * (2 - t), 2 / 3 - 0.5 * s * s * (2 - s), t ** 3 / 6])
    dw = np.stack([-0.5 * s * s, t * (1.5 * t - 2), -s * (1.5 * s - 2), 0.5 * t * t])
    return w, dw


def _mirror(k, n):
    return np.where(k < 0, -k, np.where(k > n - 1, 2 * (n - 1) - k, k))


def sample_grad(coef, u, v):
    """(s, ds/du, ds/dv) from the 4 x 4 taps of the coefficients, 0 outside the template."""
    u, v = np.atleast_1d(np.asarray(u, dtype=float)), np.atleast_1d(np.asarray(v, dtype=float))
    ty, tx = coef.shape
    inside = (u >= 0) & (u <= ty - 1) & (v >= 0) & (v <= tx - 1)
    uc, vc = np.where(inside, u, 0.0), np.where(inside, v, 0.0)
    iu, iv = np.floor(uc).astype(int), np.floor(vc).astype(int)
    wu, dwu = _weights(uc - iu)
    wv, dwv = _weights(vc - iv)
    s = np.zeros(u.shape)
    su, sv = np.zeros(u.shape), np.zeros(u.shape)
    for k in range(4):
        r = _mirror(iu - 1 + k, ty)
        for l in range(4):
            c = coef[r, _mirror(iv - 1 + l, tx)]
            s += wu[k] * wv[l] * c
            su += dwu[k] * wv[l] * c
            sv += wu[k] * dwv[l] * c
    z = np.where(inside, 1.0, 0.0)
    return s * z, su * z, sv * z


def _grid(shape):
    p, q = np.indices(shape, dtype=float)
    return p.ravel(), q.ravel()


def model(theta, tpl, shape, fit_back=False):
    """Exact image [ny, nx] of theta = (F, y0, x0[, c]) by map_coordinates."""
    ty, tx = np.shape(tpl)
    p, q = _grid(shape)
    S = float(np.sum(tpl))
    m = theta[0] * sample(tpl, p - theta[1] + ty // 2, q - theta[2] + tx // 2) / S
    return (m + (theta[3] if fit_back else 0.0)).reshape(shape)


def jacobian(theta, coef, S, p, q, fit_back):
    """d m / d (F, y0, x0[, c]) at the pixels (p, q), from the restated taps."""
    ty, tx = coef.shape
    s, su, sv = sample_grad(coef, p - theta[1] + ty // 2, q - theta[2] + tx // 2)
    cols = [s / S, -theta[0] / S * su, -theta[0] / S * sv]
    if fit_back:
        cols.append(np.ones_like(s))
    return np.stack(cols, axis=1)


def start(img, w, tpl, fit_back):
    """The library's start point: ring background, brightest used pixel above it, closed-form flux."""
    img, w = np.asarray(img, dtype=float), np.asarray(w, dtype=float)
    ny, nx = img.shape
    used = w > 0
    ring = np.zeros(img.shape, bool)
    ring[0, :] = ring[-1, :] = ring[:, 0] = ring[:, -1] = True
    c0 = 0.0
    if fit_back and np.any(ring & used):
        c0 = img[ring & used].mean()
    vals = np.where(used, img - c0, -np.inf).ravel()
    ib = int(np.argmax(vals))
    y0, x0 = ib // nx, ib % nx
    st = model((1.0, y0, x0), tpl, img.shape)
    d = np.where(used, img - c0, 0.0)
    F0 = np.sum(w * st * d) / np.sum(w * st * st)
    return np.array([F0, y0, x0] + ([c0] if fit_back else []), dtype=float)


def record(theta, img, w, tpl, fit_back):
    """PSFR_TFIT_* record of theta (ITER left at 0)."""
    img, w = np.asarray(img, dtype=float), np.asarray(w, dtype=float)
    p, q = _grid(img.shape)
    u = (w > 0).ravel()
    wu = w.ravel()[u]
    coef = coefficients(tpl)
    S = float(np.sum(tpl))
    r = model(theta, tpl, img.shape, fit_back).ravel()[u] - img.ravel()[u]
    J = jacobian(theta, coef, S, p[u], q[u], fit_back)
    chisq = float(wu @ (r * r))
    dof = u.sum() - theta.size
    e = np.sqrt(np.abs(np.diag(np.linalg.inv((J * wu[:, None]).T @ J))) * abs(chisq / dof))
    o = np.zeros(TFIT_NPAR)
    o[[FLUX, Y0, X0]] = theta[:3]
    o[CONT] = theta[3] if fit_back else 0.0
    o[CHISQ] = chisq
    o[QFIT] = np.abs(r).sum() / abs(theta[0])
    o[NPIX] = u.sum()
    o[[ERR_FLUX, ERR_Y0, ERR_X0]] = e[:3]
    o[ERR_CONT] = e[3] if fit_back else 0.0
    return o


def template_fit(img, w, tpl, fit_back=False, x0=None):
    """Weighted least-squares fit of one stamp from the library's start point (or x0); returns (record, theta)."""
    img, w = np.asarray(img, dtype=float), np.asarray(w, dtype=float)
    p, q = _grid(img.shape)
    u = (w > 0).ravel()
    sw, d = np.sqrt(w.ravel()[u]), img.ravel()[u]
    coef = coefficients(tpl)
    S = float(np.sum(tpl))
    ty, tx = np.shape(tpl)
    pu, qu = p[u], q[u]

    def resid(t):
        s, _, _ = sample_grad(coef, pu - t[1] + ty // 2, qu - t[2] + tx // 2)
        return sw * (t[0] * s / S + (t[3] if fit_back else 0.0) - d)

    th0 = start(img, w, tpl, fit_back) if x0 is None else np.asarray(x0, dtype=float)
    res = least_squares(resid, th0, jac=lambda t: sw[:, None] * jacobian(t, coef, S, pu, qu, fit_back),
                        method='lm', xtol=1e-15, ftol=1e-15, gtol=1e-15, max_nfev=20000)
    return record(res.x, img, w, tpl, fit_back), res.x
