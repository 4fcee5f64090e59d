"""Timing of the encircled-energy stage on one GPU.

    python tools/energy_bench.py [--steps 10] [--out profiles/energy_bench.json]

(a) The 4480 convolved images of one config-4 chunk (128 seeded draws x 35 wavelengths, from
    ``compute_psf_batch``), device-resident: ``psfr_encircled_energy`` (ee_kernel) at 20 radii and 2 fractions
    next to ``psfr_moffat_fit`` (fit_kernel) on the same images, device outputs, CUDA events around each call.
(b) ``compute_psf_batch`` on config 4 (512 seeded draws x 35 wavelengths, npsflin 1, four lasers; host
    outputs): without ``ee_radii``, with it, and with it and ``want_cube=False``.
(c) ``compute_psf_field`` at 128 draws x the 3 x 3 grid x 35 wavelengths, host outputs, without and with
    ``ee_radii``.
Every arm is warmed up at the size it times and the arms alternate call by call; the fit and cube of the arms
must be the same bits.  The card's name and power limit are read in the same run and written beside the numbers.
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'tools')]

from field_bench import timed_arms  # noqa: E402
from shape_bench import event_arms  # noqa: E402
from sparta_batch_bench import card, summary  # noqa: E402

RADII_ARCSEC = np.linspace(0.1, 3.9, 20)       # 0.5 to 19.5 px
FRACTIONS = (0.5, 0.8)


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'energy_bench.json'))
    args = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: this tool measures the GPU and has no CPU mode')
    from muse_psfr_b200 import _lib, psfrec
    psfrec.set_device(0)
    res = {'card': card(), 'nlam': 35, 'radii_arcsec': RADII_ARCSEC.tolist(), 'fractions': list(FRACTIONS)}
    nd, nl = 128, 35
    lam = np.linspace(490, 930, nl)
    rng = np.random.default_rng(20261021)
    seeing, GL, L0 = rng.uniform(0.5, 1.8, 4 * nd), rng.uniform(0.35, 0.9, 4 * nd), rng.uniform(10, 28, 4 * nd)
    rad_px, frac = psfrec._ee_params(RADII_ARCSEC, FRACTIONS)
    rec_len = _lib.ee_slots(rad_px.size, frac.size)[3]

    # (a) one config-4 chunk of convolved images, on the device
    nimg = nd * nl
    imgs = torch.empty((nimg, 40, 40), dtype=torch.float64, device='cuda')
    psfrec.compute_psf_batch(lam, seeing[:nd], GL[:nd], L0[:nd], out_cube=imgs, out_fit=np.empty((nd, nl, 16)))
    fit = torch.empty((nimg, _lib.FIT_NPAR), dtype=torch.float64, device='cuda')
    ee = torch.empty((nimg, rec_len), dtype=torch.float64, device='cuda')
    ctx = psfrec.get_context()
    stream = torch.cuda.current_stream().cuda_stream or None
    arms = {'fit_kernel': lambda: ctx.moffat_fit(nimg, 40, 40, imgs, fit, stream=stream),
            'ee_kernel': lambda: ctx.encircled_energy(nimg, 40, 40, imgs, rad_px, frac, ee, stream=stream)}
    for fn in arms.values():
        fn()
    torch.cuda.synchronize()
    t = event_arms(arms, max(args.steps, 20))
    e = ee.cpu().numpy()
    res['a_one_chunk'] = {
        'images': nimg, **{name: summary(ms, nimg) for name, ms in t.items()},
        'ee_over_fit_median': float(np.median(t['ee_kernel']) / np.median(t['fit_kernel'])),
        'r50_px_min_max': [float(e[:, rad_px.size + 1].min()), float(e[:, rad_px.size + 1].max())],
        'total_min_max': [float(e[:, rad_px.size].min()), float(e[:, rad_px.size].max())]}

    # (b) compute_psf_batch on config 4 (512 draws, four 128-draw chunks), host outputs
    nb = 4 * nd
    out = {k: (np.empty((nb, nl, _lib.FIT_NPAR)), np.empty((nb, nl, 40, 40))) for k in ('plain', 'ee')}
    ee_b = {k: np.empty((nb, nl, rec_len)) for k in ('ee', 'nocube')}
    fit_nocube = np.empty((nb, nl, _lib.FIT_NPAR))

    def plain():
        psfrec.compute_psf_batch(lam, seeing, GL, L0, out_fit=out['plain'][0], out_cube=out['plain'][1])

    def with_ee():
        ee_b['ee'][...] = psfrec.compute_psf_batch(lam, seeing, GL, L0, out_fit=out['ee'][0], out_cube=out['ee'][1],
                                                   ee_radii=RADII_ARCSEC, ee_fractions=FRACTIONS)[2]

    def no_cube():
        ee_b['nocube'][...] = psfrec.compute_psf_batch(lam, seeing, GL, L0, out_fit=fit_nocube, want_cube=False,
                                                       ee_radii=RADII_ARCSEC, ee_fractions=FRACTIONS)[2]

    arms = {'compute_psf_batch': plain, 'compute_psf_batch_ee': with_ee, 'compute_psf_batch_ee_no_cube': no_cube}
    for fn in arms.values():
        fn()
    t = timed_arms(arms, args.steps)
    work = nb * nl
    res['b_batch_config4'] = {
        'draws': nb, 'images': work, **{name: summary(ms, work) for name, ms in t.items()},
        'ee_over_plain_median': float(np.median(t['compute_psf_batch_ee']) / np.median(t['compute_psf_batch'])),
        'fit_and_cube_identical': bool(np.array_equal(out['plain'][0], out['ee'][0]) and
                                       np.array_equal(out['plain'][1], out['ee'][1]) and
                                       np.array_equal(out['plain'][0], fit_nocube)),
        'ee_identical_without_cube': bool(np.array_equal(ee_b['ee'], ee_b['nocube']))}

    # (c) compute_psf_field, 128 draws x 3 x 3 x 35, host outputs
    pos = psfrec.direction_perf(3)
    npos = pos.shape[1]
    s, g, l0 = seeing[:nd], GL[:nd], L0[:nd]
    outf = {k: (np.empty((nd, npos, nl, _lib.FIT_NPAR)), np.empty((nd, npos, nl, 40, 40))) for k in ('plain', 'ee')}

    def field_plain():
        psfrec.compute_psf_field(lam, s, g, l0, positions=pos, out_fit=outf['plain'][0], out_cube=outf['plain'][1])

    def field_ee():
        psfrec.compute_psf_field(lam, s, g, l0, positions=pos, out_fit=outf['ee'][0], out_cube=outf['ee'][1],
                                 ee_radii=RADII_ARCSEC, ee_fractions=FRACTIONS)

    arms = {'compute_psf_field': field_plain, 'compute_psf_field_ee': field_ee}
    for fn in arms.values():
        fn()
    t = timed_arms(arms, args.steps)
    work = nd * npos * nl
    res['c_field_grid3x3'] = {
        'draws': nd, 'positions': npos, 'images': work, **{name: summary(ms, work) for name, ms in t.items()},
        'ee_over_plain_median': float(np.median(t['compute_psf_field_ee']) / np.median(t['compute_psf_field'])),
        'fit_and_cube_identical': bool(np.array_equal(outf['plain'][0], outf['ee'][0]) and
                                       np.array_equal(outf['plain'][1], outf['ee'][1]))}
    res['method'] = ('(a) CUDA events around each call on the current stream, device-resident images and records, '
                     'one warm-up call per arm, medians; the images (4480 x 12.8 kB = 57 MB) fit in L2. (b), (c) host '
                     'wall clock around each call ended by torch.cuda.synchronize(), preallocated host outputs, one '
                     'warm-up call per arm; the arms alternate call by call; psf_per_s counts images')
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
