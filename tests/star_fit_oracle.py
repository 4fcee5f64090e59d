"""CPU reference of the star fits (psfr_moffat_fit_weighted, DESIGN.md section 5.7): scipy.optimize.leastsq on
sqrt(w) (f + c - d) over the used pixels (w > 0), with an analytic Jacobian and xtol = ftol = 1e-15, f the circular
Moffat of psfr_oracle or the elliptical one of efit_oracle and c an optional constant background.  Results are laid
out as the library's records: PSFR_FIT_* or PSFR_EFIT_*, and the side record (CONT, ERR_CONT, NPIX).

This restates the library's definitions independently of its CUDA implementation; the start point is the caller's
(a well-posed fit reaches the same minimum from any nearby start)."""
import numpy as np
from scipy.optimize import leastsq

import efit_oracle as eo
import psfr_oracle as orc

FIT_NPAR = 16
(PEAK, Y0, X0, ALPHA, N, FWHM, CHISQ, ITER, ERR_PEAK, ERR_Y0, ERR_X0, ERR_ALPHA, ERR_N, ERR_FWHM, FLUX,
 ERR_FLUX) = range(FIT_NPAR)
BACK_NPAR = 3
CONT, ERR_CONT, NPIX = range(BACK_NPAR)


def circ_model(v, p, q):
    return orc.moffat_model(v, p, q)


def circ_jacobian(v, p, q):
    """d f / d (I, y0, x0, a, n) of the circular Moffat, one row per pixel."""
    I, y0, x0, a, n = v
    dp, dq = p - y0, q - x0
    rho2 = (dp * dp + dq * dq) / (a * a)
    u = 1 + rho2
    m = u ** (-n)
    f = I * m
    g = 2 * n * f / u
    return np.stack([m, g * dp / (a * a), g * dq / (a * a), g * rho2 / a, -f * np.log(u)], axis=1)


def model_and_jacobian(elliptical):
    return (eo.model, eo.jacobian) if elliptical else (circ_model, circ_jacobian)


def star_model(theta, p, q, elliptical, fit_back):
    """f + c at the pixels (p, q) for theta = (model parameters[, c])."""
    f, _ = model_and_jacobian(elliptical)
    k = 7 if elliptical else 5
    return f(theta[:k], p, q) + (theta[k] if fit_back else 0.0)


def star_jacobian(theta, p, q, elliptical, fit_back):
    _, jac = model_and_jacobian(elliptical)
    k = 7 if elliptical else 5
    J = jac(theta[:k], p, q)
    return np.concatenate([J, np.ones((J.shape[0], 1))], axis=1) if fit_back else J


def render(shape, theta, elliptical, fit_back):
    """Exact image [ny, nx] of theta (circular (I, y0, x0, a, n) or elliptical efit_oracle theta, then c)."""
    p, q = np.indices(shape, dtype=float)
    return star_model(np.asarray(theta, dtype=float), p.ravel(), q.ravel(), elliptical, fit_back).reshape(shape)


def used_pixels(img, w):
    w = np.asarray(w, dtype=float)
    p, q = np.indices(img.shape, dtype=float)
    u = (w > 0).ravel()
    return p.ravel()[u], q.ravel()[u], np.asarray(img, dtype=float).ravel()[u], w.ravel()[u]


def normal(theta, img, w, elliptical, fit_back):
    """(J^T W J, chi^2 = sum w r^2, dof) over the used pixels at theta."""
    p, q, d, wu = used_pixels(img, w)
    J = star_jacobian(theta, p, q, elliptical, fit_back)
    r = star_model(theta, p, q, elliptical, fit_back) - d
    return (J * wu[:, None]).T @ J, float(wu @ (r * r)), d.size - theta.size


def circ_record(theta, jtj, chisq, dof):
    """PSFR_FIT_* record (ITER left at 0) of theta = (I, y0, x0, a, n[, c]); errors from the full covariance."""
    I, y0, x0, a, n = theta[:5]
    a = abs(a)
    kf = 2 * np.sqrt(2 ** (1 / n) - 1)
    e = np.sqrt(np.abs(np.diag(np.linalg.inv(jtj))) * abs(chisq / dof))
    o = np.zeros(FIT_NPAR)
    o[[PEAK, Y0, X0, ALPHA, N, FWHM, CHISQ]] = [I, y0, x0, a, n, a * kf, chisq]
    o[[ERR_PEAK, ERR_Y0, ERR_X0, ERR_ALPHA, ERR_N]] = e[:5]
    o[ERR_FWHM] = e[3] * n
    o[FLUX] = I / (n - 1) * (np.pi * a * a)
    o[ERR_FLUX] = 0.0
    return o, e


def star_record(theta, img, w, elliptical, fit_back):
    """(record, side record) of theta on img with weights w."""
    theta = np.asarray(theta, dtype=float)
    jtj, chisq, dof = normal(theta, img, w, elliptical, fit_back)
    npix = int(np.count_nonzero(np.asarray(w) > 0))
    if elliptical:
        rec = eo.record(theta[:7], jtj, chisq, dof, inv=lambda M: np.linalg.inv(M)[:7, :7])
        e = np.sqrt(np.abs(np.diag(np.linalg.inv(jtj))) * abs(chisq / dof))
    else:
        rec, e = circ_record(theta, jtj, chisq, dof)
    back = np.array([theta[-1], e[-1], npix]) if fit_back else np.array([0.0, 0.0, npix])
    return rec, back


def star_fit(img, w, start, elliptical=False, fit_back=False):
    """Weighted least-squares fit of one image from ``start`` (theta, with c last when fit_back); returns
    (record, side record, theta)."""
    p, q, d, wu = used_pixels(img, w)
    sw = np.sqrt(wu)
    theta = leastsq(lambda t: sw * (star_model(t, p, q, elliptical, fit_back) - d), np.array(start, dtype=float),
                    Dfun=lambda t: sw[:, None] * star_jacobian(t, p, q, elliptical, fit_back),
                    xtol=1e-15, ftol=1e-15, gtol=0.0, maxfev=10000)[0]
    rec, back = star_record(theta, img, w, elliptical, fit_back)
    return rec, back, theta


def theta_of_records(rec, back, elliptical, fit_back):
    """theta of a library record pair (the inverse of star_record's parameter columns)."""
    if elliptical:
        th = list(eo.theta_of_record(rec))
    else:
        th = [rec[PEAK], rec[Y0], rec[X0], rec[ALPHA], rec[N]]
    return np.array(th + ([back[CONT]] if fit_back else []), dtype=float)


def param_scale(theta, elliptical, peak=None):
    """Per-parameter scale: efit_oracle.param_scale for the model (|I|, 1 px, the form's mean, n; a for the circular
    width), and the peak for c."""
    if elliptical:
        s = list(eo.param_scale(theta[:7]))
    else:
        s = [abs(theta[0]), 1.0, 1.0, abs(theta[3]), theta[4]]
    if theta.size > len(s):
        s.append(abs(theta[0]) if peak is None else peak)
    return np.array(s)
