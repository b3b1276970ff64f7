#!/usr/bin/env python
"""bench.py — LM iterations/s of the bundle-adjustment hot path on B200 (BASELINE.json metric).

A "step" is one Levenberg-Marquardt iteration (levenberg_marquardt.m:117-206): residual + Jacobian +
normal-equation assembly, damped Schur reduction onto the camera system, sparse tile Cholesky of the
reduced system (FP64 DMMA), back-substitution, |Jp| statistics and the trial-point residual.  Accepted
trial points are taken, so successive steps walk the real LM path.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

N = 1: BASELINE config 4 (1000 cameras x 200k points x 2M observations, shared Brown IO, depend datum).
N > 1 (torchrun, one rank per GPU): BASELINE config 5 cut to N/8 of its cameras and points - 1250 cameras, 500k
points and 5M observations PER RANK, so that N = 8 runs config 5 itself (10k cameras x 4M points x 40M
observations) and N = 2 / 4 the same block density at 2500 / 5000 cameras.  The reduced camera system and its
collectives grow with N; every rank generates only its own points.  `value` counts 2M-observation equivalents,
i.e. it aggregates over ranks (weak scaling).  --nimg / --nop-per-rank select other shapes.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

C4 = dict(nImg=1000, nOP=200000, rays=10)
C5_PER_RANK = dict(nImg=1250, nOP=500000)          # config 5 / 8: N = 8 is config 5 itself
UNIT = 'LM iterations/s (2M-observation equivalents)'
# algorithmic HBM bytes per observation (DESIGN.md §4; SURVEY §8d): what the kernel has to move at least
ALG_BYTES = {
    'cam_side': 64.0,                       # uv 16 + 1/sigma 16 + indices 8 + point gather 24
    'point_side': 64.0 + 144.0 + 41.6,      # reads as above; writes W_o 144 B/obs + point record 416 B/point
    'resid': 64.0,
    'jp': 64.0 + 24.0,
    'schur': 144.0 + 41.6,                  # W_o + point records read once
    'backsub': 144.0 + 41.6 + 2.4,          # W_o + records read, 24 B/point written
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200')
    ap.add_argument('--nimg', type=int, default=0, help='cameras in total (default: 1000 at N = 1, 1250 per rank at N > 1)')
    ap.add_argument('--nop', '--nop-per-rank', dest='nop', type=int, default=0,
                    help='object points per rank (default: 200k at N = 1, 500k at N > 1)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--ref-budget', type=float, default=420.0, help='wall seconds for the reference arm')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed step returned as DIR/<name>.npy: the step p (float64; at N > 1 '
                         'p_rank<r>.npy per rank) and its statistics f, jp2, rjp, f_new, singular')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of the GPU path; the reference arm has none')
    return args


DUMP_BYTES = 64_000_000


def dump_outputs(d, p, st, rank, world):
    """The outputs of the last timed step, for comparing two builds on the same seeded scene.  A step vector larger
    than this rank's share of DUMP_BYTES (less 4 kB for file headers and the statistics) is cut to a fixed, seeded
    sample of its entries (same sample every run)."""
    os.makedirs(d, exist_ok=True)
    p = np.asarray(p, dtype=np.float64)
    keep = (DUMP_BYTES // world - 4096) // 8
    if len(p) > keep:
        p = p[np.sort(np.random.default_rng(rank).choice(len(p), keep, replace=False))]
    np.save(os.path.join(d, 'p.npy' if world == 1 else 'p_rank%d.npy' % rank), p)
    if rank == 0:
        for k in ('f', 'jp2', 'rjp', 'f_new', 'singular'):
            np.save(os.path.join(d, k + '.npy'), np.array([st[k]], dtype=np.float64))


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md): one
    long-running `nvidia-smi -lms 10` whose lines are collected by this thread.  The timed region of the
    device-resident arm is only tens of milliseconds long, so the samples that count are those taken from the
    start of its warm-up steps to the end of the end-to-end arm - the device runs the same iteration throughout."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.proc = index, [], False, None
        self.t_mark = None

    def run(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '10'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                line = line.strip()
                if line:
                    self.rows.append((time.perf_counter(), [c.strip() for c in line.split(',')]))
        except Exception:
            pass

    def mark(self):
        """Only samples taken after this call count (start of the timed region)."""
        self.t_mark = time.perf_counter()

    def stop(self):
        self.stop_flag = True
        if self.proc is not None:
            try:
                self.proc.kill()
            except Exception:
                pass

    def summary(self):
        rows = [r for t, r in self.rows if self.t_mark is None or t >= self.t_mark]
        sm = [float(r[0]) for r in rows if r and r[0].replace('.', '').isdigit()]
        mx = [float(r[1]) for r in rows if len(r) > 1 and r[1].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({names[k] for r in rows if len(r) >= 7 for k in range(4)
                          if r[3 + k].lower().startswith('active')})
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': reasons, 'samples': len(rows)}


# ------------------------------------------------------------------------------------------------
# reference CPU path
# ------------------------------------------------------------------------------------------------
CPU_DESC = ("oracle port of levenberg_marquardt.m:76-82,117-206 on the host cores: sparse Jacobian as multi_res.m "
            "builds it (SciPy CSC), J'J by sparse product, (J'J+lambda I)\\(-J'r) as MATLAB's CHOLMOD would order it "
            "(3x3 point blocks first, dense LAPACK Cholesky of the camera front: oracle.lsa.solve_spd_pointfirst), "
            "trial residual; the sparse products run on one thread (SciPy), the dense factorisation on all `cores` "
            "(LAPACK); no MATLAB/Octave exists in this image")


def host_threads():
    """All host cores for the LAPACK part of the CPU arm.  torchrun exports OMP_NUM_THREADS=1 to its workers,
    which would silently make the reference arm at N > 1 single-threaded; the limit is lifted here and the
    thread count actually in effect is what the JSON line reports as `cores`."""
    want = os.cpu_count() or 1
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        threadpool_limits(limits=want)
        got = [p.get('num_threads', 1) for p in threadpool_info() if p.get('user_api') == 'blas']
        return max(got) if got else 1
    except Exception:
        return int(os.environ.get('OMP_NUM_THREADS', want))


def cpu_lm_iterations(s, max_iters, budget_s, phases=None):
    """LM iterations of the reference CPU algorithm on scene `s` until `max_iters` or the wall budget.
    Returns (iterations done, seconds); `phases` (a dict) receives the seconds spent per stage."""
    import scipy.sparse as sp
    from oracle import lsa
    from oracle.cameramodel import brown_euler_cam4
    from oracle.dbatstruct import buildweightmatrix, serialize
    x = serialize(s)
    R = np.sqrt(buildweightmatrix(s))
    n = len(x)
    nC = n - len(s.bundle.serial.OP.dest)
    I = sp.identity(n, format='csc')
    done = 0
    ph = phases if phases is not None else {}
    clk = [time.perf_counter()]

    def lap(name):
        t = time.perf_counter()
        ph[name] = ph.get(name, 0.0) + t - clk[0]
        clk[0] = t

    t0 = clk[0]
    while done < max_iters:
        f, J = brown_euler_cam4(x, s, True)
        lap('residual_jacobian')
        r = R * f
        Jw = (sp.diags(R) @ J).tocsc()
        N = (Jw.T @ Jw).tocsc()
        g = Jw.T @ r
        lap('normal_equations')
        lam = 1e-10 * N.diagonal().sum() / n if done == 0 else 0.0          # levenberg_marquardt.m:88-106,181
        p = lsa.solve_spd_pointfirst(N + lam * I, -g, nC)
        lap('solve')
        Jp = Jw @ p                                                          # :162
        fNew = brown_euler_cam4(x + p, s, False)[0]
        if np.sum((R * fNew) ** 2) < r @ r:
            x = x + p
        lap('trial_residual')
        done += 1
        if time.perf_counter() - t0 > budget_s:
            break
    return done, time.perf_counter() - t0


def workload_name(nImg, nOP, nObs, n, nRed):
    return ('BASELINE config 4: synthetic %d cameras x %d points x %d observations, shared IO + Brown '
            'self-calibration (model 3), LM iteration; n=%d unknowns, reduced order %d' % (nImg, nOP, nObs, n, nRed))


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU algorithm on THE SAME scene as the GPU arm at N=1 (config 4
    itself, no scaled-down sample).  One LM iteration costs tens of seconds on the host, so the arm runs as many
    of the K requested iterations as fit a wall budget (at least one) and reports how many it timed."""
    if rank != 0:
        return
    from dbat_b200.synth import make_scene
    nImg = args.nimg or C4['nImg']
    args.nop = args.nop or C4['nOP']
    s, _ = make_scene(nImg, args.nop, rays=C4['rays'], cache_dir=os.environ.get('DBAT_SCENE_CACHE', '/tmp'))
    nobs = len(s.IP.img)
    n = s.bundle.serial.n
    import scipy.linalg  # noqa: F401  (loads the BLAS whose thread limit host_threads() lifts)
    cores = host_threads()
    ph = {}
    done, dt = cpu_lm_iterations(s, max(1, args.steps), args.ref_budget, ph)
    its = done / dt
    value = its * nobs / 2.0e6
    line = {
        'impl': 'reference', 'metric': 'lm_iterations_per_s', 'value': value, 'unit': UNIT, 'n_gpus': 0,
        'steps': done, 'steps_requested': args.steps, 'warmup': 0, 'ms_per_step': 1e3 / its,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': workload_name(nImg, args.nop, nobs, n, n - 3 * args.nop),
                   'same_config': world == 1,
                   'note': 'full config, %d of %d requested iterations inside the %.0f s budget' % (done, args.steps, args.ref_budget)
                           + ('' if world == 1 else '; the GPU arm at %d ranks runs BASELINE config 5 cut to %d/8 (%.1fx the '
                              'observations of this block, which is config 4): the CPU figure is per 2M-observation equivalent '
                              'of config 4, which flatters the CPU (its cost per observation grows with the block)'
                              % (world, world, 2.5 * world))},
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                         'sample': '%d full LM iterations on the config itself; %s' % (done, CPU_DESC),
                         'seconds_per_iteration': {k: v / done for k, v in ph.items()}},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0, 'seconds': dt,
    }
    print(json.dumps(line), flush=True)


def fp64_peak_tflops():
    """cuBLAS DGEMM yardstick for the FP64 tensor pipe (MEASURED_PEAKS.json has no FP64 figure): best of 3
    runs of an 8192^3 torch.matmul, the method fixed since round 1 so that fractions stay comparable."""
    import torch
    n = 8192
    a = torch.randn(n, n, dtype=torch.float64, device='cuda')
    b = torch.randn(n, n, dtype=torch.float64, device='cuda')
    torch.matmul(a, b)
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    torch.cuda.empty_cache()
    return 2.0 * n ** 3 / (best * 1e-3) / 1e12


def main():
    args = parse()
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if args.impl == 'reference':
        run_reference(args, rank, world)
        return
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    if world > 1:
        dist.barrier()
    import dbat_b200
    from dbat_b200.parallel import ShardedProblem
    from dbat_b200.synth import make_scene, make_scene_shard

    # nvidia-smi needs about a second before its first line: start it before the scene is generated
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    per = C4 if world == 1 else C5_PER_RANK
    args.nop = args.nop or per['nOP']
    nImg = args.nimg or per['nImg'] * world
    nOP = args.nop * world
    if world > 1:
        # every rank generates its own share of the points; the cameras are the same everywhere
        s, _ = make_scene_shard(nImg, nOP, rank, world, rays=C4['rays'])
        P = ShardedProblem(s, rank, world, local=True)
        nObsLocal = len(s.IP.img)
        t = torch.tensor([nObsLocal], dtype=torch.float64, device='cuda')
        dist.all_reduce(t)
        nObsGlobal = int(t.item())
    else:
        s, _ = make_scene(nImg, nOP, rays=C4['rays'], cache_dir=os.environ.get('DBAT_SCENE_CACHE', '/tmp'))
        P = dbat_b200.Problem(s)
        nObsLocal = nObsGlobal = len(s.IP.img)
    x0 = dbat_b200.serialize(s)
    n = P.n
    nRed = n - 3 * s.OP.val.shape[1]
    nGlobal = nRed + 3 * nOP
    info = P.reduced_info()

    # pinned host buffers for the end-to-end leg
    xh = torch.empty(n, dtype=torch.float64).pin_memory()
    ph = torch.empty(n, dtype=torch.float64).pin_memory()
    xh.numpy()[:] = x0
    lam = 0.0

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(k, resident):
        """k LM iterations; returns (wall seconds, device ms list, launches)."""
        dev_ms, launches = [], 0
        sync()
        t0 = time.perf_counter()
        for _ in range(k):
            if resident:
                _, st = P.normal_step(None, lam, trial=True, accept=True, want_p=False)
            else:
                _, st = P.normal_step(xh.numpy(), lam, trial=True, accept=False, p_out=ph.numpy())
            dev_ms.append(st['device_ms'])
            launches += st['launches']
        sync()
        return time.perf_counter() - t0, dev_ms, launches

    # device-resident arm
    P.normal_step(x0, lam, trial=True, accept=False, want_p=False)       # upload x0
    sampler.mark()
    timed(args.warmup, True)
    P.normal_step(x0, lam, trial=True, accept=False, want_p=False)       # restart the path at x0
    wall, dev_ms, launches = timed(args.steps, True)
    phases = P.phase_times() if hasattr(P, 'phase_times') else {}
    # end-to-end arm (host x in, host p out every step)
    timed(min(args.warmup, 3), False)
    wall_e2e, dev_ms_e2e, _ = timed(args.steps, False)
    sampler.stop()
    if args.dump_outputs:
        # The timed device-resident path once more from x0, its last step handed back to the host.  The default path is
        # bit-reproducible, so these are the timed steps' outputs; taking them here leaves the timed steps untouched.
        P.normal_step(x0, lam, trial=True, accept=False, want_p=False)   # restart the path at x0
        for i in range(args.steps):
            p, st = P.normal_step(None, lam, trial=True, accept=True, want_p=i == args.steps - 1)
        dump_outputs(args.dump_outputs, p, st, rank, world)

    t = torch.tensor([wall, wall_e2e, float(np.sum(dev_ms))], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    wall, wall_e2e, dev_total = [float(v) for v in t.cpu()]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    equiv = nObsGlobal / 2.0e6
    its = args.steps / (dev_total * 1e-3)
    value = its * equiv
    e2e_value = args.steps / wall_e2e * equiv
    if world == 1:
        wl = workload_name(nImg, nOP, nObsGlobal, n, nRed)
    else:
        c5 = (nImg, nOP) == (10000, 4000000)
        wl = ('%s: synthetic %d cameras x %d points x %d observations (%d points and %d observations per rank, '
              'every rank sees all cameras), shared IO + Brown self-calibration (model 3), LM iteration; n=%d '
              'unknowns, reduced order %d'
              % ('BASELINE config 5' if c5 else 'BASELINE config 5 cut to %d/8 of its cameras and points (config 5 itself: 10000 x 4M x 40M at 8 ranks)' % world,
                 nImg, nOP, nObsGlobal, args.nop, nObsLocal, nGlobal, nRed))
    sbytes = info['nSlotsS'] * 4096 * 8
    line = {
        'metric': 'lm_iterations_per_s', 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': dev_total / args.steps, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': wl,
                   'l2': 'inputs (>600 MB of observation, cross-block and reduced-system arrays per rank) exceed the 126 MB L2',
                   'timing': 'CUDA events on the library stream around each step (max over ranks); wall '
                             'clock %.3f ms/step' % (1e3 * wall / args.steps),
                   'parallelism': ('single GPU' if world == 1 else
                                   'points sharded over %d ranks (every rank generates and uploads only its own points); per '
                                   'evaluation one ncclAllReduce of the per-image Grams; per solve the factorisation of the '
                                   'reduced system is distributed by elimination subtree: ncclReduce of the %d tiles of S '
                                   '(%.1f MB) to their owners, ncclAllReduce of the separator tiles, of the rhs and of the '
                                   'solution; the separators above the cut are factored on every rank'
                                   % (world, info['nSlotsS'], sbytes / 1e6)),
                   'reduced_system': {k: info[k] for k in ('nT', 'nSlots', 'nSlotsS', 'nTasks', 'nTerms', 'depth', 'order_mode', 'nSeg')}},
        'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': 8 * n * world, 'd2h_bytes_per_step': (8 * n + 64) * world,
                'ms_per_step_wall': 1e3 * wall_e2e / args.steps,
                # rank 0's CUDA-event time of the same steps: upload of x + the iteration (the download of the step
                # runs on the second stream beside the trial residual and is not inside this figure)
                'ms_per_step_device_rank0': float(np.mean(dev_ms_e2e))},
        'gpu_launches': int(launches),
        'clocks': sampler.summary(),
        'phases_ms_last_step': {k: v[0] for k, v in phases.items()},
    }
    # rooflines: every kernel family of the step against its bound; the dominant one is the headline entry
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        hbm_peak, peak_src = float(peaks['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    except Exception:
        hbm_peak, peak_src = 6650.0, 'fallback (B200_PROFILING.md)'
    try:
        traffic = json.load(open(os.path.join(ROOT, 'profiles', 'r2_dram_traffic.json')))
    except Exception:
        traffic = {}
    ph_ms = {k: v[0] for k, v in phases.items() if k != 'total'}
    fp64 = fp64_peak_tflops()
    roofs = {}
    if ph_ms.get('cholesky', 0) > 0:
        ach = info['flops'] / (ph_ms['cholesky'] * 1e-3) / 1e12
        roofs['cholesky'] = {'bound': 'tensor', 'achieved': ach, 'peak': fp64, 'unit': 'TFLOP/s', 'frac': ach / fp64,
                             'traffic': traffic.get('k_tchol_factor') if world == 1 else None,
                             'kernel': 'k_tchol_factor (sparse tile Cholesky, DMMA; %.2f useful GFLOP per factorisation: '
                                       '%d tile products + %d triangular solves + %d 64x64 factorisations; the dense '
                                       'factorisation of the same system would be %.1f GFLOP)'
                                       % (info['flops'] / 1e9, info['nTerms'], info['nSlots'] - info['nT'], info['nT'], nRed ** 3 / 3e9),
                             'peak_source': 'cuBLAS DGEMM 8192^3 measured in this run (FP64; MEASURED_PEAKS.json holds no FP64 figure)',
                             'limit': 'dependency chain of %d tile columns, not the tensor pipe' % info['depth']}
    for phn, (b, kern) in {'eval_jac_assembly': (ALG_BYTES['cam_side'] + ALG_BYTES['point_side'], 'k_cam_side+k_point_side'),
                           'trial_residual': (ALG_BYTES['resid'], 'k_resid'),
                           'jp_stats': (ALG_BYTES['jp'], 'k_jp'),
                           'build_schur': (ALG_BYTES['schur'], 'k_schur_win+k_schur_reduce')}.items():
        if ph_ms.get(phn, 0) > 0:
            g = b * nObsLocal / (ph_ms[phn] * 1e-3) / 1e9
            roofs[phn] = {'bound': 'hbm', 'achieved': g, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': g / hbm_peak,
                          'traffic': traffic.get(kern) if world == 1 else None, 'kernel': kern, 'bytes_per_obs': b,
                          'ms': ph_ms[phn], 'peak_source': peak_src}
    dom = max(ph_ms, key=ph_ms.get) if ph_ms else 'cholesky'
    line['dominant_phase'] = dom
    line['roofline'] = roofs.get(dom, roofs.get('cholesky'))
    line['rooflines'] = roofs
    if world == 1 and not args.no_cpu_baseline:
        import scipy.linalg  # noqa: F401
        cores = host_threads()
        ph = {}
        done, dt = cpu_lm_iterations(s, 1, 1.0, ph)
        line['cpu_baseline'] = {'value': done / dt * nObsGlobal / 2.0e6, 'unit': UNIT, 'cores': cores,
                                'kind': 'port', 'sample': '%d full LM iteration(s) on the config itself (%.1f s); %s' % (done, dt, CPU_DESC),
                                'seconds_per_iteration': {k: v / done for k, v in ph.items()}}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
