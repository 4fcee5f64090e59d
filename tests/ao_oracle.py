"""Numpy restatement of the AO summaries (DESIGN.md section 5.5) from the oracle's pieces.

``variance_record`` splits the oracle's ``glao_residual_psd`` into the projection error of each layer and the
propagated noise, merges the AO zone with ``psd_fit`` by the reference's max() and attributes every cell of the
dim x dim grid to one source.  ``strehl`` is the centre ratio of the oracle's ``psd_to_psf`` with and without the
PSD.  Both follow oracle/psfr_oracle.py step for step; only the split and the sums are new."""
import os
import sys

import numpy as np
from numpy.fft import fftshift

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'oracle'))
import psfr_oracle as orc  # noqa: E402

VAR_NPAR, MAX_LAYERS = 12, 8
L = 2 * orc.D_PUP                                   # 16 m: the PSD grid step is 1 / L
NM2 = (orc.LAMBDA_REF_UM * 1000 / (2 * np.pi)) ** 2   # unscaled PSD -> nm^2 (psfrec.py:151)


def ao_terms(Cn2, h, seeing, L0, zenith=0., npsflin=1, three_lgs_mode=False, wind_dir=None, dirs=None):
    """(err_rec [ndir, nl, 80, 80], err_noise [ndir, 80, 80], r0 at 500 nm) of ``orc.simul_psd_wfm``:
    the terms of ``glao_residual_psd`` per direction, in the zone's final orientation (transposed, centred),
    unscaled.  err_rec[:, l] is |P beta_l - corr_l|^2 Cphi_l of layer l; err_rec.sum(1) + err_noise is the zone."""
    Cn2 = np.array(Cn2, dtype=float)
    Cn2 = Cn2 / Cn2.sum()
    vent = orc.wind_speed_for(h)
    h = np.atleast_1d(np.array(h, dtype=float))
    pos = orc.lgs_positions(three_lgs_mode) / 60
    dirs = (orc.direction_perf(npsflin) if dirs is None else np.asarray(dirs, dtype=float)) / 60
    r0ref = orc.seeing2r01(seeing, orc.LAMBDA_REF_UM, zenith)
    f, _, f_x, f_y = orc.ao_frequency_tables()
    if wind_dir is None:
        wind_dir = orc.WIND_DIR[:h.size]
    wind_dir = np.asarray(wind_dir, dtype=float)
    with np.errstate(divide='ignore'):         # a zero-weight layer: 0^(-3/5) = inf, its PSD exactly 0
        layer_psd = (0.0229 * (Cn2[:, None, None] ** (-3 / 5) * r0ref) ** (-5 / 3) *
                     (f ** 2 + (1 / L0) ** 2) ** (-11 / 6))
    ngs = pos.shape[1]
    pitch = orc.D_PUP / orc.N_ACT
    sig2 = np.repeat(orc.NOISE_LGS2, ngs)
    ti = 1 / np.repeat(orc.F_SAMP, ngs)
    td = orc.DELAY_MS * 1e-3
    wind = np.stack([vent * np.cos(wind_dir), vent * np.sin(wind_dir)])
    W = orc.glao_reconstructor(f, f_x, f_y, pitch, pos, sig2, orc.ALT_DM)
    wfs = orc._wfs_transfer(f, f_x, f_y, pitch, strict=True)
    dT = ti.max() + td
    nd = dirs.shape[1]
    rec = np.zeros((nd, h.size) + f.shape)
    noise = np.zeros((nd,) + f.shape)
    for b in range(nd):                         # glao_residual_psd with the layer terms kept apart
        bx, by = dirs[:, b]
        pw = np.exp(2j * np.pi * 1.0 * 60 / 206265 * (bx * f_x + by * f_y))[None] * W
        for l in range(h.size):
            acc = np.zeros(f.shape, dtype=complex)
            for j in range(ngs):
                sx = f_x * pos[0, j] * h[l] * 60 / 206265
                sy = f_y * pos[1, j] * h[l] * 60 / 206265
                lag = np.sinc(wind[0, l] * ti[j] * f_x + wind[1, l] * ti[j] * f_y)
                acc += pw[j] * (lag * wfs * np.exp(2j * (sx + sy) * np.pi))
            p_beta = np.exp(2j * np.pi * (h[l] * 60 / 206265 * (bx * f_x + by * f_y) -
                                          (wind[0, l] * dT * f_x + wind[1, l] * dT * f_y)))
            proj = p_beta - acc
            rec[b, l] = (proj * layer_psd[l] * proj.conj()).real
        rec[b, :, 0, 0] = 0
        noise[b] = (pw * sig2[:, None, None] * pw.conj()).sum(axis=0).real
        noise[b, 0, 0] = 0
    # the reference's moveaxis (:613) and fftshift (:149)
    rec = fftshift(np.moveaxis(rec, -1, -2), axes=(-2, -1))
    noise = fftshift(np.moveaxis(noise, -1, -2), axes=(-2, -1))
    return rec, noise, r0ref


def _zone(Cn2, h, seeing, L0, zenith, npsflin, three_lgs_mode, wind_dir, dim, dirs):
    """The terms of ``ao_terms``, the fitting PSD on the 80 x 80 zone and the sum of the fitting PSD over the
    whole dim x dim grid."""
    rec, noise, r0ref = ao_terms(Cn2, h, seeing, L0, zenith, npsflin, three_lgs_mode, wind_dir, dirs)
    fit = orc.psd_fit(dim, L, r0ref, L0, 1 / (2 * (orc.D_PUP / orc.N_ACT)))
    sl = slice(dim // 2 - orc.DIM_PUP, dim // 2 + orc.DIM_PUP)
    return rec, noise, fit[sl, sl], fit.sum()


def variance_record(Cn2, h, seeing, L0, zenith=0., npsflin=1, three_lgs_mode=False, wind_dir=None, dim=1280,
                    dirs=None):
    """PSFR_VAR_* records [ndir, VAR_NPAR] in nm^2 by the attribution rule of DESIGN.md 5.5.  ``dirs`` [2, ndir]
    (arcsec) replaces the directions of ``direction_perf(npsflin)``."""
    rec, noise, fz, fit_total = _zone(Cn2, h, seeing, L0, zenith, npsflin, three_lgs_mode, wind_dir, dim, dirs)
    out = np.zeros((rec.shape[0], VAR_NPAR))
    unit = NM2 / L ** 2
    for b in range(rec.shape[0]):
        ao = rec[b].sum(axis=0) + noise[b]
        won = ao > fz
        out[b, 1] = fit_total - fz[won].sum()
        out[b, 2] = noise[b][won].sum()
        out[b, 4:4 + rec.shape[1]] = rec[b][:, won].sum(axis=1)
        out[b, 3] = out[b, 4:4 + rec.shape[1]].sum()
        out[b, 0] = out[b, 1] + ao[won].sum()
    return out * unit


def zone_margin(Cn2, h, seeing, L0, zenith=0., npsflin=1, three_lgs_mode=False, wind_dir=None, dim=1280,
                dirs=None):
    """Smallest |ao - fit| / fit over the zone cells of every direction where the fit is positive.

    A cell whose AO value and fit agree to within rounding can fall on different sides of ``ao > fit`` here and
    on the device, which moves its fit, noise and projection terms between the slots of the record: a comparison
    with the record is only meaningful when this margin is well above the rounding of either side.  Where the fit
    is 0 (inside the correction radius) any positive AO value wins on both sides, and the centre cell is 0 on
    both."""
    rec, noise, fz, _ = _zone(Cn2, h, seeing, L0, zenith, npsflin, three_lgs_mode, wind_dir, dim, dirs)
    ao = rec.sum(axis=1) + noise
    live = fz > 0
    return float((np.abs(ao[:, live] - fz[live]) / fz[live]).min())


def psd_total(Cn2, h, seeing, L0, zenith=0., npsflin=1, three_lgs_mode=False, wind_dir=None, dim=1280):
    """sum(simul_psd_wfm) / L^2 per direction, nm^2 (the bg[0, 0] of psfrec.py:718)."""
    psd = orc.simul_psd_wfm(Cn2, h, seeing, L0, zenith, npsflin, dim, three_lgs_mode, wind_dir)
    return psd.sum(axis=(1, 2)) / L ** 2


def strehl(psd, lbda_m):
    """psf[N/2][N/2] / psf_diff[N/2][N/2] of the oracle's psd_to_psf for one N x N PSD."""
    dim = psd.shape[0]
    pup = orc.pupil_mask(dim / 4, dim / 2, oc=0.14)
    c = dim // 2
    return orc.psd_to_psf(psd, pup, orc.D_PUP, lbda_m)[c, c] / orc.psd_to_psf(np.zeros_like(psd), pup, orc.D_PUP,
                                                                               lbda_m)[c, c]
