"""Timing of the field-resolved reconstruction on one GPU.

    python tools/field_bench.py [--draws 128] [--steps 10] [--out result.json]

(a) ``--draws`` seeded draws x the 3 x 3 grid of ``direction_perf(3)`` x 35 wavelengths, three arms:
    ``compute_psf_batch(npsflin=3)`` (the field mean), ``compute_psf_field(npsflin=3)`` (one PSF per
    position), and a loop of 9 one-direction ``compute_batch`` calls (one per position), which is what a
    caller had to run for per-position PSFs before ``compute_psf_field``.  The field arm and the loop must
    give the same bits; the field mean is a different quantity and is not compared.
(b) BASELINE config 2 (30 rows x 35 wavelengths): ``compute_psf_from_sparta`` without and with
    ``field_positions`` on the 3 x 3 grid; the first five HDUs must be the same bits.
Every arm writes into preallocated host arrays, is warmed up at the size it times, and each timed call
ends in a device synchronise; the arms alternate call by call.  The card's name and power limit are read
in the same run and written beside the numbers.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'tests'), os.path.join(ROOT, 'tools')]

from bench import sparta_rows  # noqa: E402
from sparta_batch_bench import card, summary  # noqa: E402
from test_gpu_sparta_batch import assert_same_result, table_of  # noqa: E402


def timed_arms(arms, steps):
    """Alternating timings (ms per call) of every callable in ``arms``, each ended by a device synchronise."""
    import torch
    acc = {name: [] for name in arms}
    for _ in range(steps):
        for name, fn in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            acc[name].append((time.perf_counter() - t0) * 1e3)
    return {name: np.array(v) for name, v in acc.items()}


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument('--draws', type=int, default=128)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--out', default=None)
    args = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: this tool measures the GPU and has no CPU mode')
    from muse_psfr_b200 import _lib, psfrec
    psfrec.set_device(0)
    res = {'card': card(), 'nlam': 35}

    # (a) draws x 3 x 3 positions x 35 wavelengths
    nd, nl = args.draws, 35
    lam = np.linspace(490, 930, nl)
    rng = np.random.default_rng(20261020)
    seeing, GL, L0 = rng.uniform(0.5, 1.8, nd), rng.uniform(0.35, 0.9, nd), rng.uniform(10, 28, nd)
    pos = psfrec.direction_perf(3)
    npos = pos.shape[1]
    mean_fit, mean_cube = np.empty((nd, nl, _lib.FIT_NPAR)), np.empty((nd, nl, 40, 40))
    field_fit, field_cube = np.empty((nd, npos, nl, _lib.FIT_NPAR)), np.empty((nd, npos, nl, 40, 40))
    loop_fit, loop_cube = np.empty((npos, nd, nl, _lib.FIT_NPAR)), np.empty((npos, nd, nl, 40, 40))
    recs = psfrec._batch_records(seeing, GL, L0, (100, 10000), 0., None, None)
    lgs = psfrec._lgs_positions(False)

    def averaged():
        psfrec.compute_psf_batch(lam, seeing, GL, L0, npsflin=3, out_cube=mean_cube, out_fit=mean_fit)

    def field():
        psfrec.compute_psf_field(lam, seeing, GL, L0, npsflin=3, out_cube=field_cube, out_fit=field_fit)

    def loop():
        ctx = psfrec._planes_context(nd, 1, nl, None, None, 1280)
        for k in range(npos):
            ctx.compute_batch(recs, np.ascontiguousarray(pos[:, [k]]), lgs, lam, out_cube=loop_cube[k],
                              out_fit=loop_fit[k])

    arms = {'compute_psf_batch_npsflin3': averaged, 'compute_psf_field_npsflin3': field, 'loop_9_one_direction': loop}
    for fn in arms.values():          # warm-up at the timed size; the cached context reaches its final capacity
        fn()
    t = timed_arms(arms, args.steps)
    work = nd * npos * nl             # (plane x wavelength) PSFs the row pass computes in every arm
    res['a_grid3x3'] = {
        'draws': nd, 'positions': npos, 'plane_lambda': work,
        **{name: summary(ms, work) for name, ms in t.items()},
        'field_over_mean_median': float(np.median(t['compute_psf_field_npsflin3']) /
                                        np.median(t['compute_psf_batch_npsflin3'])),
        'loop_over_field_median': float(np.median(t['loop_9_one_direction']) /
                                        np.median(t['compute_psf_field_npsflin3'])),
        'field_equals_loop': bool(np.array_equal(field_cube, loop_cube.transpose(1, 0, 2, 3, 4)) and
                                  np.array_equal(field_fit, loop_fit.transpose(1, 0, 2, 3)))}

    # (b) config 2 with and without the field pass
    tbl = table_of(sparta_rows(30))
    out = {}

    def plain():
        out['plain'] = psfrec.compute_psf_from_sparta(tbl, verbose=False)

    def with_field():
        out['field'] = psfrec.compute_psf_from_sparta(tbl, verbose=False, field_positions=pos)

    arms = {'compute_psf_from_sparta': plain, 'with_field_positions_3x3': with_field}
    for fn in arms.values():
        fn()
    t = timed_arms(arms, args.steps)
    try:
        from muse_psfr_b200 import _fits
        assert_same_result(_fits.HDUList(list(out['field'])[:5]), out['plain'])
        same = True
    except AssertionError:
        same = False
    res['b_config2'] = {'draws': 30, 'positions': npos, 'psfs_mean': 30 * nl, 'plane_lambda_field': 30 * npos * nl,
                        'compute_psf_from_sparta': summary(t['compute_psf_from_sparta'], 30 * nl),
                        'with_field_positions_3x3': summary(t['with_field_positions_3x3'], 30 * nl),
                        'first_five_hdus_identical': same}
    res['method'] = ('host wall clock around each call, ended by torch.cuda.synchronize(); the arms alternate call by '
                     'call; one warm-up call of each arm at the timed size first; preallocated host outputs in (a); '
                     'medians over the timed calls; psf_per_s counts (plane x wavelength) PSFs in (a) and the rows x '
                     'wavelengths of the table in (b)')
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
