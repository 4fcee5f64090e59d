"""Timing of the star fits (psfr_moffat_fit_weighted, DESIGN.md section 5.7) on one GPU.

    python tools/star_fit_bench.py [--steps 20] [--cpu-sample 200] [--out profiles/star_fit_bench.json]

(a) The 4480 convolved images of one config-4 chunk (128 seeded draws x 35 wavelengths, 40 x 40, from
    ``compute_psf_batch``), device-resident: ``psfr_moffat_fit`` against the weighted fit with unit weights, with
    variance weights, and with variance weights and a background, circular and elliptical.  The variance is
    sigma^2 = r^2 + model / g with r = 1e-3 and g = 1e4 of the peak-normalised images (no noise is added).
(b) 36 810 seeded 25 x 25 star stamps (ten stars x 3681 planes) with a background, Gaussian noise from the same
    variance model and 2 % of the pixels masked (NaN data, weight 0): the weighted circular and elliptical fits with
    a background, device-resident.
(c) The scipy restatement (tests/star_fit_oracle.py, one process, one core) on a subsample of (b).
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


def star_stamps(nstar=10, nplane=3681, size=25, seed=20261022):
    """Seeded circular Moffat stars with a background, noise and masked pixels: (data, weights, truth [n, 6])."""
    rng = np.random.default_rng(seed)
    n = nstar * nplane
    lam = np.linspace(0.0, 1.0, nplane)
    I = np.repeat(rng.uniform(50.0, 500.0, nstar), nplane)
    y0 = np.repeat(rng.uniform(10.0, 14.0, nstar), nplane)
    x0 = np.repeat(rng.uniform(10.0, 14.0, nstar), nplane)
    fw = np.tile(4.2 - 1.2 * lam, nstar)                  # FWHM [px] falling with wavelength
    beta = np.tile(2.8 - 0.6 * lam, nstar)
    a = fw / (2 * np.sqrt(2 ** (1 / beta) - 1))
    c = np.repeat(rng.uniform(-2.0, 5.0, nstar), nplane)
    p, q = np.indices((size, size), dtype=float)
    rho2 = ((p[None] - y0[:, None, None]) ** 2 + (q[None] - x0[:, None, None]) ** 2) / (a[:, None, None] ** 2)
    model = I[:, None, None] * (1 + rho2) ** (-beta[:, None, None]) + c[:, None, None]
    var = 4.0 + np.abs(model) / 2.0                        # read noise 2, gain 2
    data = model + rng.normal(size=model.shape) * np.sqrt(var)
    w = 1 / var
    bad = rng.random(model.shape) < 0.02
    data[bad] = np.nan
    w[bad] = 0.0
    return (np.ascontiguousarray(data), np.ascontiguousarray(w),
            np.stack([I, y0, x0, a, beta, c], axis=1))


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--cpu-sample', type=int, default=200)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'star_fit_bench.json'))
    args = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: this tool measures the GPU and has no CPU mode')
    from muse_psfr_b200 import _lib, psfrec
    psfrec.set_device(0)
    res = {'card': card()}
    stream = torch.cuda.current_stream().cuda_stream or None
    dev = dict(dtype=torch.float64, device='cuda')

    # (a) one config-4 chunk
    nd, nl = 128, 35
    lam = np.linspace(490, 930, nl)
    rng = np.random.default_rng(20261020)
    seeing, GL, L0 = rng.uniform(0.5, 1.8, nd), rng.uniform(0.35, 0.9, nd), rng.uniform(10, 28, nd)
    nimg = nd * nl
    imgs = torch.empty((nimg, 40, 40), **dev)
    psfrec.compute_psf_batch(lam, seeing, GL, L0, out_cube=imgs, out_fit=np.empty((nd, nl, _lib.FIT_NPAR)))
    peak = imgs.amax(dim=(1, 2), keepdim=True)
    wvar = 1.0 / ((1e-3 * peak) ** 2 + imgs.clamp(min=0) * peak / 1e4)
    ctx = psfrec.get_context()
    out = {k: torch.empty((nimg, _lib.FIT_NPAR if k == 'c' else _lib.EFIT_NPAR), **dev) for k in 'ce'}
    back = torch.empty((nimg, _lib.BACK_NPAR), **dev)
    arms = {}
    for shape, ell in (('circular', False), ('elliptical', True)):
        o = out['e' if ell else 'c']
        plain = ctx.moffat_fit_elliptical if ell else ctx.moffat_fit
        arms[shape + '_plain'] = lambda plain=plain, o=o: plain(nimg, 40, 40, imgs, o, stream=stream)
        for name, w, fb in (('unit_weights', None, False), ('variance_weights', wvar, False),
                            ('variance_weights_background', wvar, True)):
            arms['%s_%s' % (shape, name)] = (lambda w=w, fb=fb, ell=ell, o=o: ctx.moffat_fit_weighted(
                nimg, 40, 40, imgs, w, o, back, fit_back=fb, elliptical=ell, stream=stream))
    for fn in arms.values():
        fn()
    torch.cuda.synchronize()
    t = event_arms(arms, args.steps)
    res['a_config4_chunk_40x40'] = {'images': nimg, **{name: summary(ms, nimg) for name, ms in t.items()}}
    for shape in ('circular', 'elliptical'):
        base = np.median(t[shape + '_plain'])
        res['a_config4_chunk_40x40'][shape + '_over_plain_median'] = {
            k[len(shape) + 1:]: float(np.median(v) / base) for k, v in t.items() if k.startswith(shape + '_')}

    # (b) 36 810 star stamps
    data, w, truth = star_stamps()
    n, ny, nx = data.shape
    d_data, d_w = torch.from_numpy(data).cuda(), torch.from_numpy(w).cuda()
    recs = {'circular': torch.empty((n, _lib.FIT_NPAR), **dev), 'elliptical': torch.empty((n, _lib.EFIT_NPAR), **dev)}
    backs = {k: torch.empty((n, _lib.BACK_NPAR), **dev) for k in recs}
    arms = {k: (lambda k=k: ctx.moffat_fit_weighted(n, ny, nx, d_data, d_w, recs[k], backs[k], fit_back=True,
                                                    elliptical=k == 'elliptical', stream=stream)) for k in recs}
    for fn in arms.values():
        fn()
    torch.cuda.synchronize()
    t = event_arms(arms, args.steps)
    circ = recs['circular'].cpu().numpy()
    ell = recs['elliptical'].cpu().numpy()
    res['b_star_stamps_25x25'] = {
        'stamps': n, 'masked_fraction': float((w == 0).mean()),
        **{k + '_background': summary(ms, n) for k, ms in t.items()},
        'circular_converged': int((circ[:, _lib.FIT_ITER] > 0).sum()),
        'elliptical_converged': int((ell[:, _lib.EFIT_ITER] > 0).sum()),
        'circular_beta_minus_truth_median': float(np.median(circ[:, _lib.FIT_N] - truth[:, 4])),
        'circular_chi2_per_dof_median': float(np.median(
            circ[:, _lib.FIT_CHISQ] / (backs['circular'].cpu().numpy()[:, _lib.BACK_NPIX] - 6)))}

    # (c) scipy restatement, one core
    import star_fit_oracle as so
    idx = np.random.default_rng(1).choice(n, args.cpu_sample, replace=False)
    t0 = time.perf_counter()
    for i in idx:
        img, wi = data[i], w[i]
        ring = np.concatenate([img[0], img[-1], img[1:-1, 0], img[1:-1, -1]])
        wring = np.concatenate([wi[0], wi[-1], wi[1:-1, 0], wi[1:-1, -1]])
        c0 = ring[wring > 0].mean()
        pk = np.unravel_index(np.nanargmax(np.where(wi > 0, img, -np.inf)), img.shape)
        so.star_fit(img, wi, [img[pk] - c0, pk[0], pk[1], 2.0, 2.5, c0], False, True)
    cpu = (time.perf_counter() - t0) / idx.size
    res['c_scipy_restatement'] = {
        'stamps': int(idx.size), 'ms_per_stamp': cpu * 1e3, 'cores': 1, 'cpu_count': os.cpu_count(),
        'projected_s_for_b': cpu * n,
        'gpu_speedup_circular': float(cpu * 1e3 / (np.median(t['circular']) / n))}
    res['method'] = ('CUDA events around each call on the current stream, device-resident images, weights and '
                     'records, one warm-up call per arm, medians over --steps alternating calls; psf_per_s counts '
                     'images. (a) 4480 x 12.8 kB images and their weights fit in L2. (c) scipy leastsq with analytic '
                     'Jacobian, xtol = ftol = 1e-15, one core, host wall clock')
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
