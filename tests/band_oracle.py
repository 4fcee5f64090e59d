"""Numpy restatement of the band images of DESIGN.md section 5.6, independent of the library: every pixel of a band
image is the correctly rounded sum (math.fsum) of the products w[b][k] * C[k][pix] over the wavelengths, over the
correctly rounded sum of the band's weights.  The library sums in ascending k with fused multiply-adds, so the two
agree to rounding, not bit for bit."""
import math

import numpy as np


def band_images(cube, weights):
    """Band images [nband, ny, nx] of one image set ``cube`` [nl, ny, nx] for ``weights`` [nband, nl]."""
    cube = np.asarray(cube, dtype=float)
    w = np.array(weights, dtype=float, ndmin=2)
    nl, ny, nx = cube.shape
    flat = cube.reshape(nl, -1)
    out = np.empty((w.shape[0], ny * nx))
    for b, wb in enumerate(w):
        total = math.fsum(wb)
        prod = wb[:, None] * flat
        for p in range(ny * nx):
            out[b, p] = math.fsum(prod[:, p]) / total
    return out.reshape(w.shape[0], ny, nx)


def band_sets(cubes, weights):
    """Band images [..., nband, ny, nx] of image sets [..., nl, ny, nx]."""
    cubes = np.asarray(cubes, dtype=float)
    lead = cubes.shape[:-3]
    flat = cubes.reshape((-1,) + cubes.shape[-3:])
    out = np.stack([band_images(c, weights) for c in flat])
    return out.reshape(lead + out.shape[1:])


def lbda_eff(lbda, weights):
    """Effective wavelength sum_k w[b][k] lbda[k] / sum_k w[b][k] of every band, correctly rounded sums."""
    w = np.array(weights, dtype=float, ndmin=2)
    lbda = np.asarray(lbda, dtype=float)
    return np.array([math.fsum(wb * lbda) / math.fsum(wb) for wb in w])


def trapezoid(y, x):
    """Trapezoid rule of samples y on the grid x."""
    y, x = np.asarray(y, dtype=float), np.asarray(x, dtype=float)
    return float(np.sum((y[1:] + y[:-1]) * np.diff(x)) / 2)
