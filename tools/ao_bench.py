"""Timing of the AO summaries (Strehl ratio and variance record) on one GPU.

    python tools/ao_bench.py [--steps 10] [--out profiles/ao_bench.json]

(a) One config-4 chunk (128 seeded draws x 35 wavelengths, npsflin 1) through ``psfr_compute_ao`` with
    device-resident outputs: the device time of ``var_kernel`` and ``strehl_kernel`` per launch from
    ``torch.profiler`` (CUDA activities, a profiled phase of its own), next to ``ao_zone_kernel`` and the whole
    chunk; and CUDA events around the chunk with and without the two AO outputs, the arms alternating.
(b) ``compute_psf_batch`` on config 4 (512 seeded draws x 35 wavelengths, host outputs) without and with
    ``ao_budget``, the arms alternating call by call, profiler off; the fit and cube of the arms must be the same
    bits.  The card's name and power limit are read in the same run and written beside the numbers.
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

KERNELS = ('var_kernel', 'strehl_kernel', 'ao_zone_kernel')


def kernel_times(prof, calls):
    """Device microseconds per chunk and launches per chunk of every kernel in KERNELS, from a profiler run."""
    out = {}
    for e in prof.key_averages():
        for name in KERNELS:
            if name in e.key:
                total = getattr(e, 'device_time_total', None)
                if total is None:
                    total = e.cuda_time_total
                out[name] = {'us_per_chunk': total / calls, 'launches_per_chunk': e.count / calls}
    return out


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'ao_bench.json'))
    args = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: this tool measures the GPU and has no CPU mode')
    from muse_psfr_b200 import _lib, psfrec
    psfrec.set_device(0)
    res = {'card': card(), 'nlam': 35}
    nd, nl = 128, 35
    lam = np.linspace(490, 930, nl)
    rng = np.random.default_rng(20261021)
    seeing, GL, L0 = rng.uniform(0.5, 1.8, 4 * nd), rng.uniform(0.35, 0.9, 4 * nd), rng.uniform(10, 28, 4 * nd)

    # (a) one config-4 chunk, device outputs
    recs = psfrec._batch_records(seeing[:nd], GL[:nd], L0[:nd], (100, 10000), 0., None, None)
    recs[:, _lib.DRAW_NGS] = 4
    dirs, lgs = psfrec.direction_perf(1), psfrec._lgs_positions(False)
    ctx = psfrec._planes_context(nd, 1, nl, None, None, 1280)
    dev = lambda *shape: torch.empty(shape, dtype=torch.float64, device='cuda')   # noqa: E731
    fit, strehl, var = dev(nd, 1, nl, _lib.FIT_NPAR), dev(nd, 1, nl), dev(nd, 1, _lib.VAR_NPAR)
    stream = torch.cuda.current_stream().cuda_stream or None
    arms = {'chunk': lambda: ctx.compute_ao(False, recs, dirs, lgs, lam, out_fit=fit, stream=stream),
            'chunk_ao': lambda: ctx.compute_ao(False, recs, dirs, lgs, lam, out_fit=fit, out_strehl=strehl,
                                               out_var=var, stream=stream)}
    for fn in arms.values():
        fn()
    torch.cuda.synchronize()
    t = event_arms(arms, max(args.steps, 10))
    calls = 5
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            arms['chunk_ao']()
        torch.cuda.synchronize()
    res['a_one_chunk'] = {
        'draws': nd, 'images': nd * nl, **{name: summary(ms, nd * nl) for name, ms in t.items()},
        'ao_over_plain_median': float(np.median(t['chunk_ao']) / np.median(t['chunk'])),
        'kernels': kernel_times(prof, calls),
        'strehl_min_max': [float(strehl.min()), float(strehl.max())],
        'var_total_nm2_min_max': [float(var[..., _lib.VAR_TOTAL].min()), float(var[..., _lib.VAR_TOTAL].max())]}

    # (b) compute_psf_batch on config 4 (512 draws, four 128-draw chunks), host outputs
    nb = 4 * nd
    out = {k: (np.empty((nb, nl, _lib.FIT_NPAR)), np.empty((nb, nl, 40, 40))) for k in ('plain', 'ao')}

    def plain():
        psfrec.compute_psf_batch(lam, seeing, GL, L0, out_fit=out['plain'][0], out_cube=out['plain'][1])

    def with_ao():
        psfrec.compute_psf_batch(lam, seeing, GL, L0, out_fit=out['ao'][0], out_cube=out['ao'][1], ao_budget=True)

    arms = {'compute_psf_batch': plain, 'compute_psf_batch_ao': with_ao}
    for fn in arms.values():
        fn()
    t = timed_arms(arms, args.steps)
    work = nb * nl
    identical = bool(np.array_equal(out['plain'][0], out['ao'][0]) and np.array_equal(out['plain'][1], out['ao'][1]))
    res['b_batch_config4'] = {
        'draws': nb, 'images': work, **{name: summary(ms, work) for name, ms in t.items()},
        'ao_over_plain_median': float(np.median(t['compute_psf_batch_ao']) / np.median(t['compute_psf_batch'])),
        'fit_and_cube_identical': identical}
    res['method'] = ('(a) CUDA events around each call on the current stream, device-resident outputs, one warm-up '
                     'call per arm, arms alternating, medians; kernel times from torch.profiler (CUDA activities) '
                     'over 5 further calls, a separate phase. (b) host wall clock around each call ended by '
                     'torch.cuda.synchronize(), preallocated host outputs, one warm-up call per arm, arms alternating '
                     'call by call, profiler off; psf_per_s counts images')
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')
    assert identical, 'ao_budget changed the fit or the cube'


if __name__ == '__main__':
    main()
