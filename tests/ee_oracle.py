"""CPU restatement of the encircled energy (psfr_encircled_energy, DESIGN.md section 5.4) in numpy / scipy.

Pixel (p, q) is the unit square about (p, q), its value spread uniformly over it.  The overlap of a pixel with
the disc is formed here by inclusion-exclusion of the signed quadrant area G(x, y) = area(disc ∩ [0, x] x [0, y])
with its arcsin antiderivative, in numpy's extended precision (long double): a different formula from the
library's (csrc/ee_geometry.h, which folds the pixel into one quadrant and adds a trapezoid and a segment), whose
cancellation the extra precision absorbs.  The radius at a fraction is scipy's brentq on that EE."""
import numpy as np
from scipy.optimize import brentq

LD = np.longdouble


def _quadrant(x, y, r):
    """Signed area of the disc of radius r about the origin inside [0, x] x [0, y] (odd in x and in y)."""
    sx, sy = np.sign(x), np.sign(y)
    x, y = np.minimum(np.abs(x), r), np.minimum(np.abs(y), r)
    r2 = r * r

    def chord(X):    # sqrt(r^2 - X^2) as sqrt((r - X)(r + X)): no cancellation where X is within an ulp of r
        return np.sqrt(np.maximum((r - X) * (r + X), 0))

    def prim(X):     # integral of sqrt(r^2 - X^2) from 0 to X; arcsin(X / r) as atan2, exact near X = r too
        s = chord(X)
        return (X * s + r2 * np.arctan2(X, s)) / 2

    xa = np.minimum(chord(y), x)      # the arc is above Y = y for X < xa
    return sx * sy * (xa * y + prim(x) - prim(xa))


def pixel_area(dy, dx, r):
    """Overlap of the unit pixel centred at (dy, dx) from the disc's centre with the disc of radius r (arrays
    broadcast), as long double."""
    dy, dx, r = (np.asarray(v, dtype=LD) for v in (dy, dx, r))
    if np.all(r == 0):
        return np.zeros(np.broadcast(dy, dx, r).shape, dtype=LD)
    h = LD(0.5)
    return (_quadrant(dx + h, dy + h, r) - _quadrant(dx - h, dy + h, r) - _quadrant(dx + h, dy - h, r)
            + _quadrant(dx - h, dy - h, r))


def default_centre(img):
    ny, nx = np.shape(img)
    return ny // 2, nx // 2


def _offsets(img, centre):
    ny, nx = np.shape(img)
    y0, x0 = default_centre(img) if centre is None else centre
    p, q = np.mgrid[:ny, :nx]
    return p - LD(y0), q - LD(x0)


def ee(img, r, centre=None):
    """EE(r) of one image about ``centre`` = (y0, x0) px (default (ny // 2, nx // 2)), as long double."""
    dy, dx = _offsets(img, centre)
    if r <= 0:
        return LD(0)
    return np.sum(np.asarray(img, dtype=LD) * pixel_area(dy, dx, LD(r)))


def r_at(img, frac, centre=None, total=None):
    """Smallest r with EE(r) >= frac * TOTAL [px] by brentq (EE is increasing for a positive image), NaN for
    TOTAL <= 0."""
    total = np.sum(np.asarray(img, dtype=LD)) if total is None else LD(total)
    if not total > 0:
        return np.nan
    dy, dx = _offsets(img, centre)
    rmax = float(np.sqrt(np.max((np.abs(dy) + 0.5) ** 2 + (np.abs(dx) + 0.5) ** 2)))
    target = LD(frac) * total
    return brentq(lambda r: float(ee(img, r, centre) - target), 0.0, rmax, xtol=1e-13, rtol=1e-15, maxiter=200)


def record(img, radii, fracs, centre=None):
    """The library's record: EE at each radius, TOTAL, radius at each fraction [px] (float64)."""
    total = np.sum(np.asarray(img, dtype=LD))
    out = [float(ee(img, r, centre)) for r in radii] + [float(total)]
    return np.array(out + [r_at(img, f, centre, total) for f in fracs])
