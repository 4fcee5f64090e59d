"""Timing of the template fit (psfr_template_fit, DESIGN.md section 5.8) on one GPU.

    python tools/template_fit_bench.py [--steps 20] [--cpu-sample 200] [--out profiles/template_fit_bench.json]

(a) 36 810 seeded 25 x 25 star stamps (ten stars x 3681 planes): the reconstructed PSF of each plane (one seeded
    draw, ``compute_psf_batch`` over 3681 wavelengths from 490 to 930 nm, 40 x 40) shifted to the star's sub-pixel
    centre by the oracle's interpolation (map_coordinates, order 3, mirror), scaled to the star's flux, plus a
    background, Gaussian noise from sigma^2 = 4 + model / 2 and 2 % of the pixels masked (NaN data, weight 0).
    Device-resident stamps, weights, templates and records: the template fit without and with a background
    (templates broadcast, ntpl = 3681) against ``psfr_moffat_fit_weighted`` (circular) without and with a background
    on the same stamps.
(b) The scipy restatement (tests/template_fit_oracle.py, one process pinned to one core) on a subsample of (a).
CUDA events around each call on the current stream, one warm-up call per arm, arms alternating call by call.  The
card's name and power limit are read in the same run and written beside the numbers.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'tools'), os.path.join(ROOT, 'tests'), os.path.join(ROOT, 'oracle')]

from shape_bench import event_arms  # noqa: E402
from sparta_batch_bench import card, summary  # noqa: E402


def templates(psfrec, nplane=3681, chunk=35):
    """Reconstructed PSFs [nplane, 40, 40] of one seeded draw (seeing 0.9", GL 0.7, L0 20 m)."""
    lam = np.linspace(490.0, 930.0, nplane)
    out = np.empty((nplane, 40, 40))
    for l0 in range(0, nplane, chunk):
        _, cube = psfrec.compute_psf_batch(lam[l0:l0 + chunk], [0.9], [0.7], [20.0])
        out[l0:l0 + chunk] = cube[0]
    return lam, out


def star_stamps(tpl, nstar=10, size=25, seed=20261022):
    """Stars made of the templates: (data, weights, truth [n, 4] = (F, y0, x0, c)), star-major."""
    import template_fit_oracle as to
    rng = np.random.default_rng(seed)
    nplane = tpl.shape[0]
    F = rng.uniform(2e3, 5e4, nstar)
    y0, x0 = rng.uniform(10.0, 14.0, nstar), rng.uniform(10.0, 14.0, nstar)
    c = rng.uniform(-2.0, 5.0, nstar)
    model = np.empty((nstar * nplane, size, size))
    for s in range(nstar):
        for k in range(nplane):
            model[s * nplane + k] = to.model((F[s], y0[s], x0[s], c[s]), tpl[k], (size, size), True)
    var = 4.0 + np.abs(model) / 2.0
    data = model + rng.normal(size=model.shape) * np.sqrt(var)
    w = 1 / var
    bad = rng.random(model.shape) < 0.02
    data[bad] = np.nan
    w[bad] = 0.0
    truth = np.stack([np.repeat(v, nplane) for v in (F, y0, x0, c)], axis=1)
    return np.ascontiguousarray(data), np.ascontiguousarray(w), truth


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--cpu-sample', type=int, default=200)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'template_fit_bench.json'))
    args = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: this tool measures the GPU and has no CPU mode')
    from muse_psfr_b200 import _lib, psfrec
    psfrec.set_device(0)
    res = {'card': card()}
    stream = torch.cuda.current_stream().cuda_stream or None
    dev = dict(dtype=torch.float64, device='cuda')
    # the config-4 context (128 planes x 35 wavelengths): psfr_moffat_fit_weighted chunks device arrays by its
    # capacity, 4480 stamps per launch as in tools/star_fit_bench.py; the template fit takes device arrays in one launch
    ctx = psfrec.get_context(max_planes=128)

    # (a) 36 810 star stamps
    lam, tpl = templates(psfrec)
    data, w, truth = star_stamps(tpl)
    n, ny, nx = data.shape
    d_data, d_w, d_tpl = (torch.from_numpy(a).cuda() for a in (data, w, tpl))
    tfit = {fb: torch.empty((n, _lib.TFIT_NPAR), **dev) for fb in (False, True)}
    mfit = {fb: torch.empty((n, _lib.FIT_NPAR), **dev) for fb in (False, True)}
    mback = torch.empty((n, _lib.BACK_NPAR), **dev)
    arms = {}
    for fb, tag in ((False, ''), (True, '_background')):
        arms['template' + tag] = (lambda fb=fb: ctx.template_fit(n, ny, nx, d_data, d_w, d_tpl, tfit[fb], None,
                                                                 fit_back=fb, stream=stream))
        arms['moffat_circular' + tag] = (lambda fb=fb: ctx.moffat_fit_weighted(n, ny, nx, d_data, d_w, mfit[fb], mback,
                                                                               fit_back=fb, stream=stream))
    launches = {}
    for name, fn in arms.items():
        before = ctx.kernel_launches()
        fn()
        launches[name] = ctx.kernel_launches() - before
    torch.cuda.synchronize()
    t = event_arms(arms, args.steps)
    rec = {fb: tfit[fb].cpu().numpy() for fb in (False, True)}
    rb = rec[True]
    ok = rb[:, _lib.TFIT_ITER] > 0
    res['a_star_stamps_25x25'] = {
        'stamps': n, 'templates': int(tpl.shape[0]), 'masked_fraction': float((w == 0).mean()),
        'context_capacity': ctx.max_planes * ctx.max_lambda, 'launches_per_call': launches,
        **{k: summary(ms, n) for k, ms in t.items()},
        'template_over_moffat_median': float(np.median(t['template']) / np.median(t['moffat_circular'])),
        'template_background_over_moffat_background_median': float(
            np.median(t['template_background']) / np.median(t['moffat_circular_background'])),
        'template_converged': int((rec[False][:, _lib.TFIT_ITER] > 0).sum()),
        'template_background_converged': int(ok.sum()),
        'moffat_converged': int((mfit[False].cpu().numpy()[:, _lib.FIT_ITER] > 0).sum()),
        'moffat_background_converged': int((mfit[True].cpu().numpy()[:, _lib.FIT_ITER] > 0).sum()),
        'template_background_iterations_median': float(np.median(rb[ok, _lib.TFIT_ITER])),
        'template_background_chi2_per_dof_median': float(np.median(
            rb[ok, _lib.TFIT_CHISQ] / (rb[ok, _lib.TFIT_NPIX] - 4))),
        'template_background_flux_pull_std': float(np.std(
            (rb[ok, _lib.TFIT_FLUX] - truth[ok, 0]) / rb[ok, _lib.TFIT_ERR_FLUX])),
        'template_background_y0_pull_std': float(np.std(
            (rb[ok, _lib.TFIT_Y0] - truth[ok, 1]) / rb[ok, _lib.TFIT_ERR_Y0]))}

    # (b) scipy restatement, one core
    import template_fit_oracle as to
    if hasattr(os, 'sched_setaffinity'):
        os.sched_setaffinity(0, {sorted(os.sched_getaffinity(0))[0]})
    idx = np.random.default_rng(1).choice(n, args.cpu_sample, replace=False)
    t0 = time.perf_counter()
    worst = 0.0
    for i in idx:
        orec, _ = to.template_fit(data[i], w[i], tpl[i % tpl.shape[0]], True)
        if ok[i]:
            d = np.abs(orec[[to.FLUX, to.Y0, to.X0, to.CONT]] - rb[i, [to.FLUX, to.Y0, to.X0, to.CONT]])
            worst = max(worst, float(np.max(d / rb[i, [to.ERR_FLUX, to.ERR_Y0, to.ERR_X0, to.ERR_CONT]])))
    cpu = (time.perf_counter() - t0) / idx.size
    res['b_scipy_restatement'] = {
        'stamps': int(idx.size), 'ms_per_stamp': cpu * 1e3, 'cores': 1, 'cpu_count': os.cpu_count(),
        'projected_s_for_a': cpu * n,
        'gpu_speedup_background': float(cpu * 1e3 / (np.median(t['template_background']) / n)),
        'max_abs_difference_over_error': worst}
    res['method'] = ('CUDA events around each call on the current stream, device-resident stamps, weights, templates '
                     'and records, one warm-up call per arm, medians over --steps alternating calls; psf_per_s counts '
                     'stamps. (b) scipy least_squares(method=lm) with analytic Jacobian from the library start, one '
                     'core, host wall clock; max_abs_difference_over_error compares it with the GPU records')
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
