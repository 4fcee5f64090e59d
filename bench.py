"""Benchmark of the PSF-reconstruction hot path (BASELINE.json metric: PSFs/sec at dim 1280,
PSD -> PSF -> Moffat fit).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config 1|2|3|4|5]
                    [--scaling strong|weak] [--draws D] [--dump-outputs DIR]

Workload (config.workload): BASELINE.json configs[3] - the sweep of 4096 random (seeing, GL, L0,
Cn2 profile) draws x 35 wavelengths (`--draws` changes the count).  One step = the whole path for
every draw: PSD synthesis, structure function, 35 pruned OTF -> PSF transforms, resample, the two
Moffat convolutions and the Moffat fit.  On N > 1 GPUs the sweep is SHARDED over the ranks (strong
scaling, as BASELINE.json states the config) through muse_psfr_b200.sharding.compute_psf_sharded and
the fit records are gathered to rank 0 over NCCL inside the timed region; `--scaling weak` gives every
rank its own sweep instead (rank r: seed 12345 + r).  `--config` times another BASELINE config on one
GPU (1, 2, 3: latency of one call; 5: dim 2560 x 100 wavelengths).

One JSON line on rank 0; DESIGN.md section 6 says how each field is obtained.  `--dump-outputs DIR`
writes what the timed config-4 path returned in its last timed step as .npy files (see dump_outputs), so
that two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True      # no __pycache__: the benchmark writes nothing into the tree it runs from,
os.environ['PYTHONDONTWRITEBYTECODE'] = '1'     # nor do the joblib workers of the CPU arm
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
NLAM = int(os.environ.get('PSFR_BENCH_NLAM', '35'))   # 35 = BASELINE config; env override for tuning only
LBDA = np.linspace(490, 930, NLAM)
METRIC = 'PSFs/sec (dim 1280, PSD->PSF->Moffat fit)'
FP64_PEAK_TFLOPS = 36.4      # tools/fp64_peak.cu on this pool's B200 (DFMA, 148 SMs)
HOT_METRICS = os.path.join(ROOT, 'profiles', 'hot_kernel_metrics.json')   # written by tools/ncu_summary.py --json


def canonical_bytes(dim, nlam):
    """SURVEY 8(d): canonical algorithmic bytes per PSF (two-pass real-input 2-D FFT, FP64, no pruning /
    symmetry / L2 credit): stage B 32 N^2, stage A 40 N^2 / nlam."""
    return 32.0 * dim * dim, 32.0 * dim * dim + 40.0 * dim * dim / nlam


def draws_for(seed, nd):
    rng = np.random.default_rng(seed)
    seeing = rng.uniform(0.4, 2.0, nd)
    GL = rng.uniform(0.3, 0.95, nd)
    L0 = rng.uniform(9, 29, nd)
    h = np.stack([rng.uniform(50, 500, nd), rng.uniform(5000, 15000, nd)], axis=1)
    return seeing, GL, L0, h


def sparta_rows(n=30):
    """SURVEY 8(d) config 2: 30 jittered rows, rows 3 / 11 / 27 with a bad fourth laser."""
    rng = np.random.default_rng(20261018)
    seeing = np.clip(rng.lognormal(np.log(0.8), 0.25, n), 0.4, 2.0)
    GL = np.clip(rng.normal(0.7, 0.1, n), 0.3, 0.95)
    L0 = np.clip(rng.normal(18, 5, n), 9, 29)
    vals = np.stack([seeing, GL, L0], axis=1)[:, None, :] * (1 + 0.03 * rng.standard_normal((n, 4, 3)))
    for r in (3, 11, 27):
        if r < n:
            vals[r, 3, 2] = 150.0
    return vals


def workload_config(args):
    """`config` of the JSON line: the same dict in both arms (the reference arm times a bounded sample
    of it and says so in cpu_baseline.sample)."""
    if args.config == 4:
        return {'workload': 'configs[3]: sweep of %d random (seeing, GL, L0, Cn2 profile) draws x %d wavelengths '
                            '490-930 nm, dim 1280, npsflin 1, 4 LGS' % (args.draws, NLAM),
                'draws': args.draws, 'wavelengths': NLAM, 'dim': 1280,
                'l2': '256 MB buffer rewritten before every step (inside the timed region); per-chunk working set '
                      '~8 GB >> 126 MB L2'}
    names = {1: 'configs[0]: compute_psf single field (1.0", GL 0.7, L0 25 m), dim 1280, 35 wavelengths',
             2: 'configs[1]: compute_psf_from_sparta, 30 time slices x 35 wavelengths, time-averaged PSF + Moffat fit',
             3: 'configs[2]: npsflin=3 field grid, three-LGS mode, 35 wavelengths',
             5: 'configs[4]: dim 2560, 100 wavelengths (1.0", GL 0.7, L0 25 m); batch = %d such draws' % args.draws5}
    return {'workload': names[args.config], 'dim': 2560 if args.config == 5 else 1280,
            'l2': '256 MB buffer rewritten before every step (inside the timed region)'}


def measured_peak():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            return float(json.load(f)['hbm_gbs']), 'MEASURED_PEAKS.json hbm_gbs'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index, interval=0.2):
        super().__init__(daemon=True)
        self.index = index
        self.interval = interval
        self.rows = []
        self.stop_flag = threading.Event()

    def run(self):
        q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q,
                                      '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=5)
                if out.returncode == 0 and out.stdout.strip():
                    self.rows.append([c.strip() for c in out.stdout.strip().split(',')])
            except Exception:
                pass
            self.stop_flag.wait(self.interval)

    def summary(self):
        if not self.rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace('.', '').isdigit())
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for k, n in enumerate(names) if any(r[3 + k].lower() == 'active' for r in self.rows if len(r) > 3 + k)]
        return {'sm_mhz': sm[len(sm) // 2] if sm else None,
                'sm_max_mhz': float(self.rows[0][1]) if self.rows[0][1].replace('.', '').isdigit() else None,
                'power_w_max': max(float(r[2]) for r in self.rows if r[2].replace('.', '').isdigit()) if self.rows else None,
                'samples': len(self.rows), 'reasons': reasons}


# ------------------------------------------------------------------------------- CPU arm
def _cpu_draw(args):
    """One draw through the CPU oracle (the reference's algorithm), single-threaded numpy."""
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import psfr_oracle as orc
    seeing, GL, L0, h, lbda, kw = args
    orc.compute_psf(lbda, seeing, GL, L0, h=tuple(h), **kw)
    return len(lbda) * kw.get('npsflin', 1) ** 2


def cpu_sample(cfg, cores, ndraw=None):
    """Bounded sample of workload `cfg` for the CPU arm: a list of per-draw jobs and its description."""
    kw = {}
    if cfg == 4:
        ndraw = ndraw or cores
        seeing, GL, L0, h = draws_for(12345, ndraw)
        lbda = LBDA
        what = '%d draws of the config-4 sweep (seed 12345) x %d wavelengths' % (ndraw, lbda.size)
    elif cfg == 5:
        ndraw = ndraw or max(1, cores // 2)
        nl = 4
        seeing, GL, L0 = np.full(ndraw, 1.0), np.full(ndraw, 0.7), np.full(ndraw, 25.0)
        h = np.tile(np.array([100, 10000]), (ndraw, 1))
        lbda = np.linspace(490, 930, 100)[:: 100 // nl][:nl]
        kw = {'dim': 2560}
        what = '%d draws at dim 2560 x %d of the 100 wavelengths' % (ndraw, nl)
    elif cfg == 3:
        ndraw = 1
        seeing, GL, L0, h = np.array([1.0]), np.array([0.7]), np.array([25.0]), np.array([[100, 10000]])
        lbda = LBDA[::9]
        kw = {'npsflin': 3, 'three_lgs_mode': True}
        what = 'the 9-direction draw at %d of the 35 wavelengths (one core: a single draw does not fan out)' % lbda.size
    else:
        ndraw = ndraw or cores
        vals = sparta_rows(30)[:ndraw, :3].mean(axis=1) if cfg == 2 else np.tile([1.0, 0.7, 25.0], (ndraw, 1))
        seeing, GL, L0 = vals[:, 0], vals[:, 1], vals[:, 2]
        h = np.tile(np.array([100, 10000]), (len(vals), 1))
        lbda = LBDA
        what = '%d rows x %d wavelengths' % (len(vals), lbda.size)
    jobs = [(seeing[i], GL[i], L0[i], h[i], lbda, kw) for i in range(len(seeing))]
    return jobs, what


def cpu_throughput(jobs, cores):
    """PSFs/s of the oracle driven like the reference (joblib over draws, psfrec.py:1082)."""
    from joblib import Parallel, delayed
    with Parallel(n_jobs=cores) as par:
        par(delayed(time.sleep)(0.01) for _ in range(cores))     # start the workers outside the timing
        t0 = time.time()
        done = par(delayed(_cpu_draw)(j) for j in jobs)
        dt = time.time() - t0
    return sum(done) / dt, dt


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    # bounded sample: one full draw per core and step (~10 s); --draws caps it (config 4)
    ndraw = min(args.draws, cores) if args.config == 4 else None
    jobs, what = cpu_sample(args.config, cores, ndraw)
    times, vals = [], []
    for step in range(args.warmup + args.steps):
        v, dt = cpu_throughput(jobs, cores)
        if step >= args.warmup:
            vals.append(v)
            times.append(dt)
    value = float(np.mean(vals))
    sample = ('%s per step, one joblib worker per host core; numpy oracle port of psfrec.py (the reference itself '
              'needs astropy/mpdaf, absent here)' % what)
    line = {'impl': 'reference', 'metric': METRIC, 'value': value,
            'unit': 'PSF/s', 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': float(np.mean(times) * 1e3), 'higher_is_better': True,
            'scaling': args.scaling if args.gpus > 1 else 'weak',
            'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': workload_config(args),
            'cpu_baseline': {'value': value, 'unit': 'PSF/s', 'cores': cores, 'kind': 'port', 'sample': sample},
            'e2e': {'value': value, 'unit': 'PSF/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    emit(line)


# ------------------------------------------------------------------------------- GPU arm
class Gpu:
    """Process-group / device plumbing shared by the GPU legs."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get('RANK', '0'))
        self.world = int(os.environ.get('WORLD_SIZE', '1'))
        self.local = int(os.environ.get('LOCAL_RANK', '0'))
        if self.world > 1:
            # keep stdout to the one JSON line: NCCL prints its version banner there at VERSION level
            if os.environ.get('NCCL_DEBUG', '').upper() in ('', 'VERSION'):
                os.environ['NCCL_DEBUG'] = 'WARN'
            dist.init_process_group('nccl', device_id=torch.device('cuda', self.local))
        torch.cuda.set_device(self.local)
        self.dev = torch.device('cuda', self.local)
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)     # > 126 MB L2
        self.stream = torch.cuda.current_stream().cuda_stream

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, fn, steps, warmup, after_step=None):
        """ms for `steps` calls of fn (CUDA events on the current stream, L2 flush before every call,
        barrier + synchronize on both sides), max over ranks."""
        torch = self.torch
        for _ in range(warmup):
            self.flush.zero_()
            fn()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            self.flush.zero_()
            fn()
            if after_step:
                after_step()
        e1.record()
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1))

    def timed_wall(self, fn, steps, warmup):
        """seconds of wall clock for `steps` calls (end-to-end legs: host buffers, copies inside)."""
        for _ in range(warmup):
            fn()
        self.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        self.barrier()
        return self.max_over_ranks(time.perf_counter() - t0)

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def apply_options(ctx, args, _lib):
    # tuning knobs (None = the library defaults, which is what the reported line uses)
    for key, val in ((_lib.OPT_EXP_GRADE, args.grade), (_lib.OPT_F32_ROWS, args.f32_rows),
                     (_lib.OPT_EXP_CUT, args.exp_cut), (_lib.OPT_ROW_KERNEL, args.row_kernel)):
        if val is not None:
            ctx.set_option(key, val)


def hot_metrics():
    """ncu figures of the dominant kernel that cannot be measured live (written from an ncu --set full
    capture by tools/ncu_summary.py --json; the file names its capture)."""
    try:
        with open(HOT_METRICS) as f:
            return json.load(f)
    except Exception:
        return {}


def roofline_block(value_per_gpu, dim, nlam, hot_ms, hot_n, hot_psfs, own_bytes_launch, own_bytes_step, ms_step, psfs_step):
    """Roofline of the dominant kernel (the stage-B row kernel).  `achieved` = the bytes the kernel has
    to move in ITS formulation (D and its FP32 copy in, the pruned row-pass output out: own_bytes) over
    the live launch duration; `canonical_*` = the same with SURVEY 8(d)'s full-grid bytes, which the
    pruned, wavelength-batched kernel never moves (so that figure exceeds 1 and is not a bandwidth)."""
    peak, peak_src = measured_peak()
    stage_b, per_psf = canonical_bytes(dim, nlam)
    m = hot_metrics()
    if not hot_n:
        return {'bound': m.get('bound', 'hbm'), 'achieved': None, 'peak': peak, 'unit': 'GB/s', 'frac': None, 'traffic': None}
    avg_ms = hot_ms / hot_n
    per_launch = hot_psfs / hot_n
    achieved = own_bytes_launch / (avg_ms * 1e-3) / 1e9
    canonical = stage_b * per_launch / (avg_ms * 1e-3) / 1e9
    return {
        'bound': m.get('bound', 'hbm'),
        'kernel': 'stage-B row kernel (exp(-c D) * OTF + pruned 1280-point FFT per row pair and wavelength)',
        'achieved': achieved, 'peak': peak, 'peak_source': peak_src, 'unit': 'GB/s', 'frac': achieved / peak,
        'traffic': m.get('dram_bytes_per_launch'),
        'dram_frac': achieved / peak,
        'own_bytes_per_launch': own_bytes_launch, 'own_bytes_per_psf': own_bytes_launch / per_launch,
        'psfs_per_launch': per_launch, 'avg_launch_ms': avg_ms,
        'pipeline_dram_frac': own_bytes_step / (ms_step * 1e-3) / 1e9 / peak,
        'pipeline_own_bytes_per_psf': own_bytes_step / psfs_step,
        'smem_frac': m.get('smem_wavefront_frac'), 'fp64_frac': m.get('fp64_pipe_frac'),
        'issue_frac': m.get('issue_frac'), 'fp64_peak_tflops': FP64_PEAK_TFLOPS,
        'ncu_source': m.get('source'),
        'canonical_frac': canonical / peak, 'canonical_bytes_per_psf': stage_b,
        'canonical_pipeline_frac': value_per_gpu * per_psf / 1e9 / peak,
        'note': 'frac = bytes the kernel moves in its own (pruned, wavelength-batched, Hermitian) formulation / live '
                'kernel time / HBM peak: the kernel is NOT HBM-bound (bound = what ncu shows; smem_frac, fp64_frac, '
                'issue_frac from the named ncu capture).  canonical_frac uses SURVEY 8(d)\'s full-grid bytes, which '
                'the kernel never moves - it measures the restructuring, not bandwidth.'}


def own_bytes(ctx_info, nplanes, ndraw, nlam, dim):
    """Bytes one chunk has to move in this implementation's formulation (the traffic ncu should see).
    Row kernel: D (FP64 + FP32 copy at dim 1280) of every plane and the telescope OTF once in, Y out.
    Whole chunk: + stage A (quadrant PSD, transposed hand-off twice, D out) + column pass (Y in, samples
    out) + cubes / fits."""
    rows = dim // 2 + 2
    ycols = ctx_info['y_cols']
    d_in = nplanes * rows * dim * (12 if dim == 1280 else 8) + rows * dim * (12 if dim == 1280 else 8)
    y = nplanes * nlam * ycols * rows * 16
    hot = d_in + y
    stage_a = ndraw * (dim // 2) ** 2 * 8 * 2 + nplanes * (dim * rows * 16 * 2 + rows * dim * (12 if dim == 1280 else 8))
    tail = y + ndraw * nlam * (80 * 80 * 8 * 2 + 1600 * 8 * 4 + 128)
    return hot, hot + stage_a + tail


DUMP_FIT_BYTES = 24 << 20       # the two budgets keep a dump under 64 MB whatever --draws is
DUMP_CUBE_BYTES = 36 << 20


def dump_outputs(out_dir, cube, fit, first_draw):
    """Write what one compute_batch call returned, as float64 .npy files in out_dir:
        fit.npy              [n, wavelengths, FIT_NPAR] fit records (psfr.h PSFR_FIT_*)
        fit_draws.npy        [n] sweep index of each draw in fit.npy
        psf_cube.npy         [m, wavelengths, 40, 40] PSF cubes
        psf_cube_draws.npy   [m] sweep index of each draw in psf_cube.npy
    Every draw goes in where its records fit the budget; beyond that a fixed, seeded sample of draws
    (in sweep order).  `first_draw` is the sweep index of the buffers' first draw (the rank's block)."""
    import torch
    nd = cube.shape[0]
    order = np.random.default_rng(0).permutation(nd)
    os.makedirs(out_dir, exist_ok=True)
    for name, buf, budget in (('fit', fit, DUMP_FIT_BYTES), ('psf_cube', cube, DUMP_CUBE_BYTES)):
        per_draw = (buf[0].numel() + 1) * 8
        pick = np.sort(order[:min(nd, budget // per_draw)])
        rows = buf.index_select(0, torch.as_tensor(pick, device=buf.device))
        np.save(os.path.join(out_dir, name + '.npy'), rows.cpu().numpy())
        np.save(os.path.join(out_dir, name + '_draws.npy'), (first_draw + pick).astype(np.float64))


def run_gpu(args):
    from muse_psfr_b200 import _lib, psfrec, sharding
    g = Gpu()
    torch = g.torch
    psfrec.set_device(g.local)
    nlam = LBDA.size
    strong = g.world > 1 and args.scaling == 'strong'
    total = args.draws
    if strong:
        (a, b), _ = sharding.block_of(total, nlam, g.world, g.rank)
        seeing, GL, L0, h = draws_for(12345, total)
        loc = slice(a, b)
    else:
        seeing, GL, L0, h = draws_for(12345 + g.rank, total)
        loc = slice(0, total)
    nd = loc.stop - loc.start
    ctx = psfrec.get_context(max_planes=args.max_planes, max_lambda=nlam, device=g.local)
    apply_options(ctx, args, _lib)
    info = ctx.info()

    # ---- device-resident leg: inputs (draw records, tables) and outputs live in HBM
    recs = psfrec.draw_records(seeing[loc], GL[loc], L0[loc], h[loc])
    d_recs = torch.from_numpy(recs).to(g.dev)
    dirs = psfrec.direction_perf(1)
    pos = psfrec._lgs_positions(False)
    d_cube = torch.empty((nd, nlam, 40, 40), dtype=torch.float64, device=g.dev)
    d_fit = torch.empty((nd, nlam, _lib.FIT_NPAR), dtype=torch.float64, device=g.dev)
    hot = {'ms': 0.0, 'n': 0, 'psfs': 0}

    gather_ev = []
    h_fit_all = torch.empty((total, nlam, _lib.FIT_NPAR), dtype=torch.float64, pin_memory=True) if strong and g.rank == 0 else None

    def step_device():
        ctx.compute_batch(d_recs, dirs, pos, LBDA, out_cube=d_cube, out_fit=d_fit, stream=g.stream)
        if strong:
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            ev[0].record()
            sharding.gather_grid(d_fit, total, nlam, host_out=h_fit_all)   # NCCL gather of the fit records + D2H on rank 0
            ev[1].record()
            gather_ev.append(ev)

    def collect_hot():
        ms, n, psfs = ctx.last_hot_timing()     # CUDA events around every launch of the row kernel
        hot['ms'] += ms
        hot['n'] += n
        hot['psfs'] += psfs

    sampler = ClockSampler(g.local)
    launches0 = None

    def first_timed():
        nonlocal launches0
        launches0 = ctx.kernel_launches()

    for _ in range(args.warmup):
        g.flush.zero_()
        step_device()
    g.barrier()
    if g.rank == 0:
        sampler.start()
    first_timed()
    ms_total = g.timed(step_device, args.steps, 0, after_step=collect_hot)
    launches = ctx.kernel_launches() - launches0
    gather_ms = float(np.mean([a.elapsed_time(b) for a, b in gather_ev[-args.steps:]])) if gather_ev else None
    if args.dump_outputs and g.rank == 0:      # before the legs below reuse d_cube / d_fit
        dump_outputs(args.dump_outputs, d_cube, d_fit, loc.start)

    # ---- the same leg with both precision grades off (everything FP64): 3 steps, same draws
    ms_fp64 = None
    if not args.no_fp64_leg and args.grade is None and args.f32_rows is None:
        ctx.set_option(_lib.OPT_EXP_GRADE, 1e30)
        ctx.set_option(_lib.OPT_F32_ROWS, 1e30)
        ms_fp64 = g.timed(step_device, 3, 1)
        ctx.set_option(_lib.OPT_EXP_GRADE, info['exp_grade'])
        ctx.set_option(_lib.OPT_F32_ROWS, info['f32_rows'])

    # ---- end-to-end leg: the public Python API with HOST buffers (pinned outputs)
    h_cube = torch.empty((nd, nlam, 40, 40), dtype=torch.float64, pin_memory=True)
    h_fit = torch.empty((nd, nlam, _lib.FIT_NPAR), dtype=torch.float64, pin_memory=True)
    gathered = {}

    def step_e2e():
        if strong:
            # every rank: parameters on the host -> its block on its GPU -> its cube block into pinned host
            # memory; the fit records go device -> rank 0 over NCCL and from there to the host
            fit_all, _, _ = sharding.compute_psf_sharded(LBDA, seeing, GL, L0, h=h, out_cube=h_cube, want_sum=False, fit_host=h_fit_all,
                                                         device=g.local, max_planes=args.max_planes, stream=g.stream)
            gathered['fit'] = fit_all
        else:
            psfrec.compute_psf_batch(LBDA, seeing, GL, L0, h=h, out_cube=h_cube, out_fit=h_fit,
                                     device=g.local, max_planes=args.max_planes, stream=g.stream)

    t_e2e = g.timed_wall(step_e2e, args.steps, max(1, args.warmup // 2))

    # ---- weak-scaling companion (N > 1, strong run): every rank its own full sweep, no gather
    weak = None
    if strong and not args.no_weak_leg:
        sw, gw, lw, hw = draws_for(12345 + g.rank, total)
        d_recs_w = torch.from_numpy(psfrec.draw_records(sw, gw, lw, hw)).to(g.dev)
        d_cube_w = torch.empty((total, nlam, 40, 40), dtype=torch.float64, device=g.dev)
        d_fit_w = torch.empty((total, nlam, _lib.FIT_NPAR), dtype=torch.float64, device=g.dev)
        ms_w = g.timed(lambda: ctx.compute_batch(d_recs_w, dirs, pos, LBDA, out_cube=d_cube_w, out_fit=d_fit_w,
                                                 stream=g.stream), 2, 1)
        weak = {'value': g.world * total * nlam * 2 / (ms_w * 1e-3), 'unit': 'PSF/s', 'ms_per_step': ms_w / 2,
                'draws_per_gpu': total, 'steps': 2}
    if g.rank == 0:
        sampler.stop_flag.set()
        sampler.join(timeout=2)

    # sanity on the result of the last step (loss-like read-back): fitted FWHM must be finite
    fit_last = gathered['fit'] if strong and g.rank == 0 else (h_fit.numpy() if not strong else None)
    finite = bool(np.isfinite(fit_last[:, :, _lib.FIT_FWHM]).all()) if fit_last is not None else None
    nonconv = int((fit_last[:, :, _lib.FIT_ITER] < 0).sum()) if fit_last is not None else None
    fit_iter = float(np.abs(fit_last[:, :, _lib.FIT_ITER]).mean()) if fit_last is not None else None

    if g.rank != 0:
        g.close()
        return
    job_psfs = (total if strong else g.world * total) * nlam
    value = job_psfs * args.steps / (ms_total * 1e-3)
    e2e = job_psfs * args.steps / t_e2e
    chunk_planes = min(args.max_planes, nd)
    hot_launch, _ = own_bytes(info, chunk_planes, chunk_planes, nlam, 1280)
    _, step_bytes = own_bytes(info, nd, nd, nlam, 1280)
    cfg = workload_config(args)      # identical in both arms; what this run did beyond it goes to `run`
    run = {'chunk_planes': args.max_planes, 'draws_per_gpu': nd,
           'sharding': ('strong: the %d draws are split over %d GPUs, fit records gathered to rank 0 (NCCL) '
                        'inside the timed region' % (total, g.world)) if strong else
                       ('single GPU' if g.world == 1 else 'weak: every rank runs its own %d-draw sweep' % total),
           'exp_cut': 'OTF entries below exp(-%g) of the peak are flushed to zero (DESIGN.md 3.7)' % info['exp_cut'],
           'graded_precision': 'row pairs entirely below exp(-%g) of the OTF peak are evaluated and transformed '
                               'in FP32, blocks entirely below exp(-%g) use the FP32 exp; everything else FP64 '
                               '(psfr.h PSFR_OPT_F32_ROWS / PSFR_OPT_EXP_GRADE; value_allfp64 = both off)'
                               % (info['f32_rows'], info['exp_grade'])}
    line = {
        'metric': METRIC, 'value': value, 'unit': 'PSF/s',
        'n_gpus': g.world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_total / args.steps,
        'higher_is_better': True, 'scaling': 'strong' if strong else 'weak', 'vs_baseline': None, 'dtype': 'f64',
        'data': 'synthetic', 'config': cfg, 'run': run,
        'e2e': {'value': e2e, 'unit': 'PSF/s',
                'h2d_bytes_per_step': int(recs.nbytes + dirs.nbytes + pos.nbytes + LBDA.nbytes),
                'd2h_bytes_per_step': int(h_cube.numel() * 8 + (total if strong else nd) * nlam * _lib.FIT_NPAR * 8),
                'api': 'sharding.compute_psf_sharded' if strong else 'psfrec.compute_psf_batch'},
        'gpu_launches': int(launches),
        'results_finite': finite, 'fits_not_converged': nonconv, 'fit_iterations_mean': fit_iter,
        'roofline': roofline_block(value / g.world, 1280, nlam, hot['ms'], hot['n'], hot['psfs'], hot_launch,
                                   step_bytes, ms_total / args.steps, nd * nlam),
        'clocks': sampler.summary(),
    }
    if ms_fp64 is not None:
        line['value_allfp64'] = job_psfs * 3 / (ms_fp64 * 1e-3)
    if weak:
        line['weak_scaling'] = weak
    if gather_ms is not None:
        line['collective'] = {'op': 'gather of the fit records [draws, 35, 16] f64 to rank 0 (NCCL) + device -> host copy',
                              'ms_per_step_rank0': gather_ms, 'share_of_step': gather_ms / (ms_total / args.steps),
                              'bytes': int(total * nlam * _lib.FIT_NPAR * 8)}
    if g.world == 1 and not args.no_cpu:
        cores = os.cpu_count() or 1
        jobs, what = cpu_sample(4, cores)
        v, dt = cpu_throughput(jobs, cores)
        line['cpu_baseline'] = {'value': v, 'unit': 'PSF/s', 'cores': cores, 'kind': 'port',
                                'sample': '%s, joblib over draws (one worker per core), numpy oracle port of '
                                          'psfrec.py (%.1f s)' % (what, dt)}
    if g.world == 1 and not args.no_configs:
        line['other_configs'] = other_configs(g, args, psfrec, _lib)
    emit(line)
    g.close()


# ------------------------------------------------------------------------------- other BASELINE configs
def time_config(g, args, psfrec, _lib, cfg, steps=3, warmup=2):
    """Latency / throughput of one BASELINE config on one GPU through the public API (host buffers)."""
    torch = g.torch
    out = {}
    if cfg == 1:
        fn = lambda: psfrec.compute_psf(LBDA, 1.0, 0.7, 25.0, verbose=False)      # noqa: E731
        psfs = NLAM
    elif cfg == 3:
        fn = lambda: psfrec.compute_psf(LBDA, 1.0, 0.7, 25.0, npsflin=3, three_lgs_mode=True, verbose=False)   # noqa: E731
        psfs = 9 * NLAM
    elif cfg == 2:
        vals = sparta_rows(30)
        jobs = psfrec.select_sparta_rows(vals)
        s_, g_, l_, three = (np.array(c) for c in list(zip(*jobs))[:4])

        def fn():
            cubes = np.empty((len(jobs), NLAM, 40, 40))
            for mode in (False, True):
                sel = np.where(three == mode)[0]
                if sel.size:
                    _, c = psfrec.compute_psf_batch(LBDA, s_[sel], g_[sel], l_[sel], three_lgs_mode=bool(mode))
                    cubes[sel] = c
            mean, fit = np.empty((NLAM, 40, 40)), np.empty((NLAM, _lib.FIT_NPAR))
            psfrec.get_context().mean_refit(len(jobs), NLAM, cubes, mean, fit)
        psfs = len(jobs) * NLAM
        out['rows'] = len(jobs)
    else:
        lam5 = np.linspace(490, 930, 100)
        ctx5 = psfrec.get_context(max_planes=16, max_lambda=100, dim=2560)
        apply_options(ctx5, argparse.Namespace(grade=None, f32_rows=None, exp_cut=args.exp_cut, row_kernel=None), _lib)
        fn = lambda: psfrec.compute_psf(lam5, 1.0, 0.7, 25.0, verbose=False, dim=2560)   # noqa: E731
        psfs = 100
    if os.environ.get('PSFR_BENCH_BATCH_ONLY') and cfg == 5:
        warmup = steps = 1          # profiling runs: go straight to the batch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        g.flush.zero_()
        fn()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / steps
    out.update({'latency_ms': dt * 1e3, 'psfs': psfs, 'psf_per_s': psfs / dt})
    if cfg == 5:
        # batch at dim 2560: device-resident, `draws5` copies of the config-5 draw x 100 wavelengths
        nd = args.draws5
        recs = np.tile(psfrec.draw_record([0.7, 0.3], (100, 10000), 1.0, 25.0, 0.,
                                          alpha_tt=psfrec.tiptilt_alpha(1.0, 0.7, 25.0)), (nd, 1))
        d_recs = torch.from_numpy(recs).to(g.dev)
        d_fit = torch.empty((nd, 100, _lib.FIT_NPAR), dtype=torch.float64, device=g.dev)
        d_cube = torch.empty((nd, 100, 40, 40), dtype=torch.float64, device=g.dev)
        dirs, pos = psfrec.direction_perf(1), psfrec._lgs_positions(False)
        hot = {'ms': 0.0, 'n': 0, 'psfs': 0}

        def batch():
            ctx5.compute_batch(d_recs, dirs, pos, lam5, out_cube=d_cube, out_fit=d_fit, stream=g.stream)

        def collect():
            ms, n, p = ctx5.last_hot_timing()
            hot['ms'] += ms
            hot['n'] += n
            hot['psfs'] += p
        ms = g.timed(batch, steps, 1, after_step=collect)
        val = nd * 100 * steps / (ms * 1e-3)
        info = ctx5.info()
        chunk = min(16, nd)
        hot_launch, _ = own_bytes(info, chunk, chunk, 100, 2560)
        _, step_bytes = own_bytes(info, nd, nd, 100, 2560)
        out['batch'] = {'draws': nd, 'value': val, 'unit': 'PSF/s', 'ms_per_step': ms / steps,
                        'roofline': roofline_block(val, 2560, 100, hot['ms'], hot['n'], hot['psfs'], hot_launch,
                                                   step_bytes, ms / steps, nd * 100)}
        out['batch']['roofline'].update({'smem_frac': None, 'fp64_frac': None, 'issue_frac': None, 'traffic': None,
                                         'ncu_source': 'profiles/ (dim-2560 captures, see profiles/README.md)'})
    return out


def other_configs(g, args, psfrec, _lib):
    res = {}
    for cfg in (1, 2, 3, 5):
        try:
            res['config%d' % cfg] = time_config(g, args, psfrec, _lib, cfg)
        except Exception as exc:     # a failure here must not lose the headline line
            res['config%d' % cfg] = {'error': repr(exc)}
    return res


def run_config(args):
    """--config 1|2|3|5: one BASELINE config on one GPU, as its own JSON line."""
    from muse_psfr_b200 import _lib, psfrec
    g = Gpu()
    if g.rank != 0:
        g.close()
        return
    psfrec.set_device(g.local)
    sampler = ClockSampler(g.local, interval=1.0)   # a millisecond-scale call: nvidia-smi queries stall the driver
    sampler.start()
    res = time_config(g, args, psfrec, _lib, args.config, steps=args.steps, warmup=args.warmup)
    sampler.stop_flag.set()
    sampler.join(timeout=2)
    ctx = psfrec.get_context(dim=2560 if args.config == 5 else 1280)
    head = res.get('batch', res)
    line = {'metric': METRIC if args.config != 5 else 'PSFs/sec (dim 2560, PSD->PSF->Moffat fit)',
            'value': head.get('value', res['psf_per_s']), 'unit': 'PSF/s', 'n_gpus': 1, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': head.get('ms_per_step', res['latency_ms']), 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic', 'config': workload_config(args),
            'e2e': {'value': res['psf_per_s'], 'unit': 'PSF/s', 'latency_ms': res['latency_ms'],
                    'h2d_bytes_per_step': int(_lib.DRAW_NPAR * 8 + 8 * (100 if args.config == 5 else NLAM)),
                    'd2h_bytes_per_step': int(res['psfs'] * (1600 + _lib.FIT_NPAR) * 8),
                    'api': 'psfrec.compute_psf (one call, host buffers)'},
            'gpu_launches': ctx.kernel_launches(), 'clocks': sampler.summary(), 'detail': res}
    if 'batch' in res:
        line['roofline'] = res['batch']['roofline']
    if not args.no_cpu:
        cores = os.cpu_count() or 1
        jobs, what = cpu_sample(args.config, cores)
        v, dt = cpu_throughput(jobs, cores if args.config != 3 else 1)
        line['cpu_baseline'] = {'value': v, 'unit': 'PSF/s', 'cores': cores if args.config != 3 else 1, 'kind': 'port',
                                'sample': '%s, numpy oracle port of psfrec.py (%.1f s)' % (what, dt)}
    emit(line)
    g.close()


_JSON_FD = [1]


def own_stdout():
    """Keep stdout to the ONE JSON line: file descriptor 1 is pointed at stderr for the whole run (NCCL and
    other native libraries print banners straight to fd 1) and the line goes to the saved descriptor."""
    sys.stdout.flush()
    _JSON_FD[0] = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    os.write(_JSON_FD[0], (json.dumps(line) + '\n').encode())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--draws', type=int, default=4096, help='draws of the config-4 sweep (total when sharded, per GPU with --scaling weak)')
    ap.add_argument('--draws5', type=int, default=64, help='draws of the dim-2560 batch (--config 5 / other_configs)')
    ap.add_argument('--config', type=int, default=4, choices=[1, 2, 3, 4, 5], help='BASELINE config (1-based); 4 = the headline sweep')
    ap.add_argument('--scaling', default='strong', choices=['strong', 'weak'], help='N > 1: shard the sweep (default) or replicate it')
    ap.add_argument('--max-planes', type=int, default=128, dest='max_planes', help='planes per chunk (the library default)')
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--no-configs', action='store_true', help='skip the other_configs leg')
    ap.add_argument('--no-fp64-leg', action='store_true', dest='no_fp64_leg', help='skip value_allfp64')
    ap.add_argument('--no-weak-leg', action='store_true', dest='no_weak_leg', help='skip weak_scaling (N > 1)')
    ap.add_argument('--grade', type=float, default=None, help='PSFR_OPT_EXP_GRADE override (tuning)')
    ap.add_argument('--f32-rows', type=float, default=None, dest='f32_rows', help='PSFR_OPT_F32_ROWS override (tuning)')
    ap.add_argument('--row-kernel', type=int, default=None, dest='row_kernel', help='PSFR_OPT_ROW_KERNEL override (tuning)')
    ap.add_argument('--exp-cut', type=float, default=None, dest='exp_cut', help='PSFR_OPT_EXP_CUT override (tuning)')
    ap.add_argument('--dump-outputs', default=None, dest='dump_outputs', metavar='DIR',
                    help='write the fit records and PSF cubes of the last timed step to DIR/*.npy (config 4; on N GPUs '
                         'rank 0\'s draws)')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if args.dump_outputs and (args.impl != 'b200' or args.config != 4):
        ap.error('--dump-outputs dumps the config-4 sweep of the b200 implementation')
    own_stdout()
    if args.impl == 'reference':
        run_reference(args)
    elif args.config != 4:
        run_config(args)
    else:
        run_gpu(args)


if __name__ == '__main__':
    main()
