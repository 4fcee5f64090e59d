"""Timing of the band images (DESIGN.md section 5.6) on one GPU.

    python tools/band_bench.py [--steps 10] [--out profiles/band_bench.json]

(a) One config-4 chunk (128 seeded draws x 35 wavelengths, npsflin 1, 3 bands) through ``psfr_compute_bands`` with
    device-resident outputs: the device time of ``band_kernel`` per chunk from ``torch.profiler`` (CUDA activities, a
    profiled phase of its own), next to every other kernel of the chunk; and CUDA events around the
    chunk with and without the band outputs, the arms alternating.
(b) ``compute_psf_batch`` on config 4 (512 seeded draws x 35 wavelengths, host outputs) without ``bands`` and with 3
    bands (a white-light top-hat 480-930 nm and two synthetic filter curves), the arms alternating call by call,
    profiler off; the fit and cube of the arms must be the same bits.  The card's name and power limit are read in the
    same run and written beside the numbers.
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


def kernel_times(prof, calls):
    """Device microseconds and launches per chunk of every kernel and copy of the profiled calls."""
    out = {}
    for e in prof.key_averages():
        total = getattr(e, 'device_time_total', None)
        if total is None:
            total = e.cuda_time_total
        if total > 0:
            out[e.key] = {'us_per_chunk': total / calls, 'launches_per_chunk': e.count / calls}
    return out


def filters(psfrec, lam):
    """Weights [3, nl]: a white-light top-hat 480-930 nm and two synthetic filter curves (a smooth 80 nm wide
    bump about 606 nm with a sloped top, and a trapezoid 760-880 nm)."""
    x = np.linspace(520, 700, 19)
    bump = np.exp(-0.5 * ((x - 606) / 40.0) ** 4) * (1 + 0.002 * (x - 606))
    return np.stack([psfrec.band_weights(lam, [480.0, 930.0], [1.0, 1.0]),
                     psfrec.band_weights(lam, x, bump),
                     psfrec.band_weights(lam, [740.0, 760.0, 880.0, 900.0], [0.0, 0.9, 0.85, 0.0])])


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'band_bench.json'))
    args = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: this tool measures the GPU and has no CPU mode')
    from muse_psfr_b200 import _lib, psfrec
    psfrec.set_device(0)
    res = {'card': card(), 'nlam': 35, 'nband': 3}
    nd, nl = 128, 35
    lam = np.linspace(490, 930, nl)
    w = filters(psfrec, lam)
    res['lbda_eff_nm'] = psfrec._band_lbda_eff(lam, w).tolist()
    rng = np.random.default_rng(20261022)
    seeing, GL, L0 = rng.uniform(0.5, 1.8, 4 * nd), rng.uniform(0.35, 0.9, 4 * nd), rng.uniform(10, 28, 4 * nd)

    # (a) one config-4 chunk, device outputs
    recs = psfrec._batch_records(seeing[:nd], GL[:nd], L0[:nd], (100, 10000), 0., None, None)
    recs[:, _lib.DRAW_NGS] = 4
    dirs, lgs = psfrec.direction_perf(1), psfrec._lgs_positions(False)
    ctx = psfrec._planes_context(nd, 1, nl, None, None, 1280)
    dev = lambda *shape: torch.empty(shape, dtype=torch.float64, device='cuda')   # noqa: E731
    fit, band, bfit = dev(nd, 1, nl, _lib.FIT_NPAR), dev(nd, 1, 3, 40, 40), dev(nd, 1, 3, _lib.FIT_NPAR)
    stream = torch.cuda.current_stream().cuda_stream or None
    arms = {'chunk': lambda: ctx.compute_bands(False, recs, dirs, lgs, lam, None, out_fit=fit, stream=stream),
            'chunk_bands': lambda: ctx.compute_bands(False, recs, dirs, lgs, lam, w, out_fit=fit, out_band=band,
                                                     out_band_fit=bfit, stream=stream)}
    for fn in arms.values():
        fn()
    torch.cuda.synchronize()
    t = event_arms(arms, max(args.steps, 10))
    calls = 5
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            arms['chunk_bands']()
        torch.cuda.synchronize()
    bytes_read = nd * nl * 40 * 40 * 8
    kt = kernel_times(prof, calls)
    band_us = sum(v['us_per_chunk'] for k, v in kt.items() if 'band_kernel' in k)
    res['a_one_chunk'] = {
        'draws': nd, 'images': nd * nl, **{name: summary(ms, nd * nl) for name, ms in t.items()},
        'bands_over_plain_median': float(np.median(t['chunk_bands']) / np.median(t['chunk'])),
        'kernels': kt, 'band_kernel_bytes_read': bytes_read,
        'band_kernel_read_GB_per_s': bytes_read / (band_us * 1e-6) / 1e9 if band_us else None}

    # (b) compute_psf_batch on config 4 (512 draws, four 128-draw chunks), host outputs
    nb = 4 * nd
    out = {k: (np.empty((nb, nl, _lib.FIT_NPAR)), np.empty((nb, nl, 40, 40))) for k in ('plain', 'bands')}

    def plain():
        psfrec.compute_psf_batch(lam, seeing, GL, L0, out_fit=out['plain'][0], out_cube=out['plain'][1])

    def with_bands():
        psfrec.compute_psf_batch(lam, seeing, GL, L0, out_fit=out['bands'][0], out_cube=out['bands'][1], bands=w)

    arms = {'compute_psf_batch': plain, 'compute_psf_batch_bands': with_bands}
    for fn in arms.values():
        fn()
    t = timed_arms(arms, args.steps)
    work = nb * nl
    identical = bool(np.array_equal(out['plain'][0], out['bands'][0]) and
                     np.array_equal(out['plain'][1], out['bands'][1]))
    res['b_batch_config4'] = {
        'draws': nb, 'images': work, **{name: summary(ms, work) for name, ms in t.items()},
        'bands_over_plain_median': float(np.median(t['compute_psf_batch_bands']) / np.median(t['compute_psf_batch'])),
        'fit_and_cube_identical': identical}
    res['method'] = ('(a) CUDA events around each call on the current stream, device-resident outputs, one warm-up '
                     'call per arm, arms alternating, medians; kernel times from torch.profiler (CUDA activities) '
                     'over 5 further calls, a separate phase; bytes read by band_kernel from the shapes (each '
                     'convolved plane once). (b) host wall clock around each call ended by torch.cuda.synchronize(), '
                     'preallocated host outputs, one warm-up call per arm, arms alternating call by call, profiler '
                     'off; psf_per_s counts monochromatic images')
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')
    assert identical, 'bands changed the fit or the cube'


if __name__ == '__main__':
    main()
