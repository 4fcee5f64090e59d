"""Timing of the elliptical Moffat fit on one GPU.

    python tools/shape_bench.py [--steps 10] [--out profiles/shape_bench.json]

(a) The 4480 convolved images of one config-4 chunk (128 seeded draws x 35 wavelengths, from
    ``compute_psf_batch``), device-resident: ``psfr_moffat_fit`` (fit_kernel) against
    ``psfr_moffat_fit_elliptical`` (fit_kernel + efit_kernel), device outputs, CUDA events around each call.
(b) ``compute_psf_field`` at 128 draws x the 3 x 3 grid x 35 wavelengths, host outputs, without and with
    ``elliptical=True``; the fit and cube of both arms must be the same bits.
Every arm is warmed up at the size it times and the arms alternate call by call.  The card's name and power
limit are read in the same run and written beside the numbers.
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'tools')]

from field_bench import timed_arms  # noqa: E402
from sparta_batch_bench import card, summary  # noqa: E402


def event_arms(arms, steps):
    """Alternating device times (ms per call, CUDA events on the current stream) of every callable in ``arms``."""
    import torch
    acc = {name: [] for name in arms}
    for _ in range(steps):
        for name, fn in arms.items():
            start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            start.record()
            fn()
            end.record()
            end.synchronize()
            acc[name].append(start.elapsed_time(end))
    return {name: np.array(v) for name, v in acc.items()}


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'shape_bench.json'))
    args = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: this tool measures the GPU and has no CPU mode')
    from muse_psfr_b200 import _lib, psfrec
    psfrec.set_device(0)
    res = {'card': card(), 'nlam': 35}
    nd, nl = 128, 35
    lam = np.linspace(490, 930, nl)
    rng = np.random.default_rng(20261020)
    seeing, GL, L0 = rng.uniform(0.5, 1.8, nd), rng.uniform(0.35, 0.9, nd), rng.uniform(10, 28, nd)

    # (a) one config-4 chunk of convolved images, on the device
    nimg = nd * nl
    imgs = torch.empty((nimg, 40, 40), dtype=torch.float64, device='cuda')
    psfrec.compute_psf_batch(lam, seeing, GL, L0, out_cube=imgs, out_fit=np.empty((nd, nl, _lib.FIT_NPAR)))
    fit = torch.empty((nimg, _lib.FIT_NPAR), dtype=torch.float64, device='cuda')
    efit = torch.empty((nimg, _lib.EFIT_NPAR), dtype=torch.float64, device='cuda')
    ctx = psfrec.get_context()
    stream = torch.cuda.current_stream().cuda_stream or None
    arms = {'fit_kernel': lambda: ctx.moffat_fit(nimg, 40, 40, imgs, fit, stream=stream),
            'fit_kernel_plus_efit_kernel': lambda: ctx.moffat_fit_elliptical(nimg, 40, 40, imgs, efit, stream=stream)}
    for fn in arms.values():
        fn()
    torch.cuda.synchronize()
    t = event_arms(arms, max(args.steps, 20))
    e = efit.cpu().numpy()
    f = fit.cpu().numpy()
    res['a_fit_one_chunk'] = {
        'images': nimg, **{name: summary(ms, nimg) for name, ms in t.items()},
        'efit_kernel_ms_median': float(np.median(t['fit_kernel_plus_efit_kernel']) - np.median(t['fit_kernel'])),
        'elliptical_over_circular_median': float(np.median(t['fit_kernel_plus_efit_kernel']) /
                                                 np.median(t['fit_kernel'])),
        'elliptical_converged': int((e[:, _lib.EFIT_ITER] > 0).sum()),
        'elliptical_iterations_median': float(np.median(np.abs(e[:, _lib.EFIT_ITER]))),
        'axis_ratio_min_max': [float(e[:, _lib.EFIT_AXIS_RATIO].min()), float(e[:, _lib.EFIT_AXIS_RATIO].max())],
        'chisq_elliptical_le_circular': bool(np.all(e[:, _lib.EFIT_CHISQ] <= f[:, _lib.FIT_CHISQ] * (1 + 1e-12)))}

    # (b) compute_psf_field, 128 draws x 3 x 3 x 35, host outputs
    pos = psfrec.direction_perf(3)
    npos = pos.shape[1]
    out = {k: (np.empty((nd, npos, nl, _lib.FIT_NPAR)), np.empty((nd, npos, nl, 40, 40))) for k in ('plain', 'shapes')}
    shapes = np.empty((nd, npos, nl, _lib.EFIT_NPAR))

    def plain():
        psfrec.compute_psf_field(lam, seeing, GL, L0, positions=pos, out_fit=out['plain'][0], out_cube=out['plain'][1])

    def with_shapes():
        _, _, s = psfrec.compute_psf_field(lam, seeing, GL, L0, positions=pos, out_fit=out['shapes'][0],
                                           out_cube=out['shapes'][1], elliptical=True)
        shapes[...] = s

    arms = {'compute_psf_field': plain, 'compute_psf_field_elliptical': with_shapes}
    for fn in arms.values():
        fn()
    t = timed_arms(arms, args.steps)
    work = nd * npos * nl
    res['b_field_grid3x3'] = {
        'draws': nd, 'positions': npos, 'images': work, **{name: summary(ms, work) for name, ms in t.items()},
        'elliptical_over_plain_median': float(np.median(t['compute_psf_field_elliptical']) /
                                              np.median(t['compute_psf_field'])),
        'fit_and_cube_identical': bool(np.array_equal(out['plain'][0], out['shapes'][0]) and
                                       np.array_equal(out['plain'][1], out['shapes'][1]))}
    res['method'] = ('(a) CUDA events around each call on the current stream, device-resident images and records, '
                     'one warm-up call per arm, medians; the images (4480 x 12.8 kB = 57 MB) fit in L2. (b) host wall '
                     'clock around each call ended by torch.cuda.synchronize(), preallocated host outputs, one warm-up '
                     'call per arm; the arms alternate call by call; psf_per_s counts images')
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
