#!/usr/bin/env python
"""Benchmark of the VCGPCM ELBO + gradient hot path (BASELINE.json's metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU algorithm (oracle port)

One "step" = one full-regime evaluation (ELBO + gradient w.r.t. every variable, Psi statistics rebuilt
and differentiated) on the synthetic scaling-sweep series with N = 1e5 observations and nh = nx = 200
inducing points (SURVEY.md §8d).  With several ranks the N observations are sharded (strong scaling:
total work fixed); every rank ends each step with the same ELBO and gradient.

Timing: every step is timed on the device with CUDA events on the library's stream (returned by
cgpcm_last_timing), L2 is flushed between steps, the per-step maximum over ranks is summed.  `e2e` times the
same step through the C-ABI with HOST buffers (pinned) by wall clock, including the upload of the
observations and the variables and the download of ELBO / terms / gradient.
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

from tests.workload import NAMED_SHAPES, named_workload, sweep_workload  # noqa: E402

METRIC = 'VCGPCM ELBO+grad evals/sec (N=1e5, M=200)'
UNIT = 'evals/s'
FP64_PEAK_FALLBACK_TFLOPS = 37.16     # tools/fp64_peaks.cu on this pool's B200 (profiles/fp64_peaks_r01.json)


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed summary of
    the latest `ncu --set full` capture of the bench command (profiles/traffic.json, written by tools/ncu_summary.py)."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'traffic.json')) as f:
            return json.load(f)
    except (OSError, ValueError):
        return None


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5,
                    help='timed steps of the headline evaluation (and of every shape with --mode restarts); the side '
                         'measurements reported beside the headline (other_window_settings, frozen_regime) time the '
                         'fixed number of steps each reports as its "steps"')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--n', type=int, default=100000)
    ap.add_argument('--m', type=int, default=200)
    ap.add_argument('--cull', type=float, default=746.0,
                    help='headline (746): nothing is approximated -- the only Psi elements / GEMM tiles skipped are '
                         'those that are exactly 0.0 in IEEE double (their Gaussian envelope exp(E), E < -745.2, '
                         'underflows); 0 = every tile multiplied, 80 = envelope < exp(-80) dropped; both reported beside')
    ap.add_argument('--chunk', type=int, default=0, help='0 = the library default: chosen per evaluation by the planner')
    ap.add_argument('--cpu-sample', type=int, default=300,
                    help='observations in the CPU baseline sample of our arm (oracle port).  Its cost is linear in N '
                         'already here: 20.8 s at 300 observations (69 ms each), 239 s at 3000 (80 ms each) on 8 '
                         'threads at M = 200 -- the M^3 algebra is 0.3 s')
    ap.add_argument('--ref-sample', type=int, default=96,
                    help='observations per step of the reference arm (the reference\'s own code, oracle/_ref: it '
                         'materialises N x nx x nx tensors and keeps them for autodiff)')
    ap.add_argument('--mode', default='sharded', choices=['sharded', 'restarts'],
                    help='sharded: one evaluation, observations sharded over the GPUs (the headline); restarts: '
                         'independent restarts / hyper-parameter batches, one replica per GPU, no communication')
    ap.add_argument('--shape', default='sweep', help='restarts mode: sweep | toy | ou | hrir | crude | all')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed step returned -- elbo, terms (7), grad (every variable) -- as '
                         'DIR/<name>.npy in float64; the inputs are seeded, so two builds can be compared output for output')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'ours' or args.mode != 'sharded'):
        ap.error('--dump-outputs needs --impl ours --mode sharded')
    return args


def dump_outputs(out_dir, budget=64 << 20, **arrays):
    """Writes every array as out_dir/<name>.npy in float64, at most `budget` bytes in all: above it the largest array
    is replaced by a fixed, seeded sample of its entries (in index order), the same for every run at that shape."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    big = max(arrays, key=lambda k: arrays[k].size)
    room = (budget - 8 * sum(a.size for k, a in arrays.items() if k != big)) // 8
    if arrays[big].size > room:
        keep = np.sort(np.random.default_rng(0).choice(arrays[big].size, room, replace=False))
        arrays[big] = arrays[big].ravel()[keep]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


# ----------------------------------------------------------------------------- clocks
class ClockSampler(object):
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            f = [x.strip() for x in r.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
                power.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(nm)
        # "under load": samples in the upper half of the observed power range
        if sm:
            thr = min(power) + .5 * (max(power) - min(power))
            load = [s for s, p in zip(sm, power) if p >= thr] or sm
            return {'sm_mhz': float(np.median(load)), 'sm_max_mhz': float(max(mx)), 'reasons': sorted(reasons),
                    'power_w_max': float(max(power)), 'samples': len(sm)}
        return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples']}


# ----------------------------------------------------------------------------- CPU baselines
def host_threads():
    """All the host threads the CPU arms may use: set explicitly, also under torchrun (which exports
    OMP_NUM_THREADS=1 to every rank)."""
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        pass
    return max(1, n)


def cpu_port_eval(wl, sample, steps=1, warmup=0):
    """Times the CPU oracle PORT (oracle/model.py: numpy / torch-CPU restatement of the reference's algorithm with
    closed-form Psi statistics, chunk-free) on the first `sample` observations of the workload with every host thread.
    The cost of the path is linear in N (measured at M = 200 on 8 threads: 69 ms per observation at 300 observations,
    80 ms at 3000; the M^3 algebra is a fixed 0.3 s); evals/s at N is stated with the extrapolation factor N / sample."""
    import torch
    from oracle import model as om
    threads = host_threads()
    torch.set_num_threads(threads)
    sl = slice(0, sample)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        om.elbo_and_grad(wl['params'], wl['t'][sl], wl['y'][sl], wl['th'], wl['tx'], wl['reg'])
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    per_eval_s = float(np.mean(times)) * wl['n'] / sample
    return {'value': 1.0 / per_eval_s, 'unit': UNIT, 'cores': threads, 'kind': 'port',
            'sample': 'oracle port (numpy/torch-CPU FP64 restatement of the reference, closed-form Psi statistics) on the '
                      'first %d of %d observations, nh=nx=%d, full regime, %d torch threads; %.2f s per sample '
                      'evaluation, extrapolated x%.1f to N' % (sample, wl['n'], wl['nh'], threads,
                                                              float(np.mean(times)), wl['n'] / sample),
            'seconds_per_sample_eval': float(np.mean(times)), 'extrapolation_factor': wl['n'] / sample}


def cpu_reference_eval(wl, sample, steps=1, warmup=1):
    """Times the REFERENCE'S OWN CODE (oracle/_ref: py3-patched copies of /root/reference/src on the TensorFlow stand-in
    oracle/tfshim, torch-CPU FP64 underneath; built by oracle/build_ref.py) through its own API --
    VCGPCM.from_recipe, mod.elbo(), tf.gradients -- on the first `sample` observations, in a process of its own.
    The reference materialises N x nx x nx and N x nh x nx tensors and keeps every intermediate for autodiff, so the
    sample is what fits; its cost is linear in N."""
    from oracle import ref
    threads = host_threads()
    sl = slice(0, sample)
    t, m = wl['t'], wl['nh']
    r = ref.call(threads=threads, timeout=3000, t=t[sl], y=wl['y'][sl], nx=m, nh=m, tau_w=.1, tau_f=.025, causal=True,
                 causal_id=False, reg=wl['reg'], params=wl['params'], tx_range=np.array([t.min(), t.max()]),
                 time=max(1, steps) + warmup, want_mats=False)
    if not (np.array_equal(r['th'], wl['th']) and np.array_equal(r['tx'], wl['tx'])):
        raise RuntimeError('reference recipe does not reproduce the workload\'s inducing inputs')
    secs = np.asarray(r['seconds'])[warmup:]
    per_eval_s = float(np.mean(secs)) * wl['n'] / sample
    return {'value': 1.0 / per_eval_s, 'unit': UNIT, 'cores': threads, 'kind': 'reference',
            'sample': "the reference's own code (oracle/_ref = /root/reference/src, py3-patched, on a torch-CPU TensorFlow "
                      'stand-in) on the first %d of %d observations, nh=nx=%d, full regime: sess.run([elbo, '
                      'tf.gradients]) %.2f s per sample evaluation with %d threads (graph construction excluded), '
                      'extrapolated x%.1f to N' % (sample, wl['n'], m, float(np.mean(secs)), threads, wl['n'] / sample),
            'seconds_per_sample_eval': float(np.mean(secs)), 'extrapolation_factor': wl['n'] / sample,
            'elbo_of_sample': float(r['elbo'])}


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    wl = sweep_workload(args.n, args.m)
    from oracle import ref
    if ref.available():
        cb = cpu_reference_eval(wl, args.ref_sample, steps=max(1, args.steps), warmup=min(args.warmup, 1))
        port = None
        try:
            port = cpu_port_eval(wl, args.cpu_sample)
        except Exception as exc:            # the port beside it is informative only
            port = {'error': repr(exc)}
    else:
        cb = cpu_port_eval(wl, args.cpu_sample, steps=max(1, args.steps), warmup=min(args.warmup, 1))
        port = None
    line = {'impl': 'reference', 'metric': METRIC, 'value': cb['value'], 'unit': UNIT, 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 / cb['value'], 'higher_is_better': True,
            'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': {'workload': 'scaling sweep N=%d, nh=nx=%d, causal VCGPCM, full regime' % (args.n, args.m),
                       'n': args.n, 'nh': args.m, 'nx': args.m,
                       'extrapolation_factor': cb['extrapolation_factor']},
            'cpu_baseline': cb,
            'e2e': {'value': cb['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'note': 'CPU arm on %d host threads, kind = %s; each step evaluates a bounded sample of the observations '
                    'and the rate is scaled to N (cost linear in N)' % (cb['cores'], cb['kind'])}
    if port is not None:
        line['cpu_baseline_port'] = port
    print(json.dumps(line))


# ----------------------------------------------------------------------------- our arm
def fp64_peak():
    """Measured FP64 tensor (DMMA) peak: live from tools/fp64_peaks if present, else the committed number."""
    exe = os.path.join(ROOT, 'tools', 'fp64_peaks')
    if os.path.exists(exe):
        try:
            out = subprocess.run([exe], capture_output=True, text=True, timeout=120).stdout.strip().splitlines()[-1]
            d = json.loads(out)
            return float(d['dmma_m8n8k4_tflops']), 'measured live by tools/fp64_peaks (DMMA m8n8k4 burst)', d
        except Exception:
            pass
    return FP64_PEAK_FALLBACK_TFLOPS, 'tools/fp64_peaks on this pool (profiles/fp64_peaks_r01.json)', None


def run_ours(args):
    import torch
    import cgpcm_b200
    from cgpcm_b200.cgpcm import shard_bounds, window_costs, window_radius

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit('launch with torch.distributed.run --nproc-per-node %d' % args.gpus)
    dist = None
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))

    wl = sweep_workload(args.n, args.m)
    # shards of equal estimated cost (observations near the ends of the series have narrower windows)
    cost = window_costs(wl['t'], wl['tx'], args.m, window_radius(*wl['hyp'], args.cull)) if world > 1 else None
    lo, hi = shard_bounds(args.n, rank, world, cost)
    eng = cgpcm_b200.Engine(args.m, args.m, causal=True, device=local_rank)
    if world > 1:
        box = [cgpcm_b200.Engine.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        eng.comm_init(box[0], rank, world)
    eng.set_option('chunk', args.chunk)
    eng.set_option('cull', args.cull)
    # pinned host buffers for the e2e leg
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    t_h, y_h = pin(wl['t'][lo:hi]), pin(wl['y'][lo:hi])
    th_h, tx_h, p_h = pin(wl['th']), pin(wl['tx']), pin(wl['params'])
    g_h = torch.empty(p_h.shape[0], dtype=torch.float64).pin_memory()
    eng.set_data(t_h, y_h, th_h, tx_h)
    flush = torch.empty(512 * 1024 * 1024 // 8, dtype=torch.float64, device='cuda')   # 512 MB > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        return eng.elbo_grad(p_h, mode=cgpcm_b200.MODE_FULL, grad_mask=cgpcm_b200.GRAD_ALL, reg=wl['reg'],
                             out_grad=g_h)

    for _ in range(args.warmup):
        step()
    # Shards of equal MEASURED time: the per-observation model is refined with the device time of every rank's sweeps
    # (two rounds, during warm-up; cgpcm_b200.rebalance_costs) -- the end shards' narrow, rounded windows run the GEMM
    # kernels less efficiently than the model says.  The partition is fixed before the timed region starts.
    balance = None
    if world > 1:
        from cgpcm_b200.cgpcm import rebalance_costs
        balance = []
        for _ in range(2):
            step()
            tm = eng.last_timing()
            mine = torch.tensor([tm['own_sweeps_ms']], dtype=torch.float64, device='cuda')
            every = [torch.zeros_like(mine) for _ in range(world)]
            dist.all_gather(every, mine)
            times = np.array([float(v.item()) for v in every])
            balance.append(float(times.max() / times.mean()))
            bounds = [shard_bounds(args.n, r, world, cost) for r in range(world)]
            cost = rebalance_costs(cost, bounds, times)
            lo, hi = shard_bounds(args.n, rank, world, cost)
            t_h, y_h = pin(wl['t'][lo:hi]), pin(wl['y'][lo:hi])
            eng.set_data(t_h, y_h, th_h, tx_h)
            step()
    # ---- timed region: K steps, device time per step from CUDA events on the library's stream
    eng.set_option('profile', 1)
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    wall0 = time.perf_counter()
    dev_ms, gemm_ms, gemm_flops, gemm_launches, launches, axx_ms, gemm_flops_exec = [], 0.0, 0.0, 0, 0, 0.0, 0.0
    gen_ms = 0.0
    last = None
    for _ in range(args.steps):
        flush.zero_()                      # L2 flush between timed iterations (not inside the event bracket)
        torch.cuda.synchronize()
        last = step()
        tm = eng.last_timing()
        dev_ms.append(tm['total_ms'])
        gemm_ms += tm['gemm_ms']
        gemm_flops += tm['gemm_flops']
        gemm_flops_exec += tm['gemm_flops_executed']
        gemm_launches += tm['gemm_launches']
        launches += tm['launches']
        axx_ms += tm['axx_ms']
        gen_ms += tm['ahx_gen_ms']
    barrier()
    wall = time.perf_counter() - wall0
    _np = lambda x: x.numpy().copy() if hasattr(x, 'numpy') else np.array(x)
    last = (last[0], _np(last[1]), _np(last[2]))               # the gradient buffer g_h is reused by later steps
    clocks = sampler.stop()
    eng.set_option('profile', 0)
    if args.dump_outputs and rank == 0:       # every rank holds the same all-reduced result
        dump_outputs(args.dump_outputs, elbo=last[0], terms=last[1], grad=last[2])
    dev = torch.tensor(dev_ms, dtype=torch.float64, device='cuda')
    if dist is not None:
        dist.all_reduce(dev, op=dist.ReduceOp.MAX)
    total_ms = float(dev.sum().item())
    value = args.steps / (total_ms * 1e-3)

    # ---- e2e: the same step through the C-ABI with host buffers, wall clock, uploads/downloads included
    barrier()
    e0 = time.perf_counter()
    for _ in range(args.steps):
        eng.set_data(t_h, y_h, th_h, tx_h)
        step()
    barrier()
    e2e_s = time.perf_counter() - e0
    e2e_t = torch.tensor([e2e_s], dtype=torch.float64, device='cuda')
    if dist is not None:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_value = args.steps / float(e2e_t.item())
    npar = p_h.shape[0]
    h2d = 8 * (2 * (hi - lo) + 2 * args.m + npar)
    d2h = 8 * (npar + 8 + (hi - lo) + 2 * args.m)    # gradient, ELBO + terms; set_data reads t, th, tx back for planning

    # ---- the other window settings beside the headline: every tile multiplied (0), exact-zero windows (746),
    # envelope < exp(-80) dropped (80, the library default)
    other = []
    eng.set_option('profile', 1)
    for alt in (0.0, 746.0, 80.0):
        if alt == args.cull:
            continue
        eng.set_option('cull', alt)
        for _ in range(2):
            step()
        ms, g_ms, g_fl = [], 0.0, 0.0
        for _ in range(max(2, min(args.steps, 5))):
            flush.zero_()
            torch.cuda.synchronize()
            alt_out = step()
            alt_tm = eng.last_timing()
            ms.append(alt_tm['total_ms'])
            g_ms += alt_tm['gemm_ms']
            g_fl += alt_tm['gemm_flops']
        alt_dev = torch.tensor(ms, dtype=torch.float64, device='cuda')
        if dist is not None:
            dist.all_reduce(alt_dev, op=dist.ReduceOp.MAX)
        other.append({'cull': alt, 'value': len(ms) / (float(alt_dev.sum().item()) * 1e-3), 'unit': UNIT, 'steps': len(ms),
                      'gemm_flops_per_step': alt_tm['gemm_flops'],
                      'gemm_tflops': g_fl / (g_ms * 1e-3) / 1e12 if g_ms > 0 else None,
                      'elbo_rel_diff_vs_headline': abs(alt_out[0] - last[0]) / abs(last[0]),
                      'grad_rel_diff_vs_headline': float(np.abs(_np(alt_out[2]) - last[2]).max() / np.abs(last[2]).max())})
    eng.set_option('profile', 0)
    eng.set_option('cull', args.cull)

    # ---- frozen ("precomputed") regime, reported beside (SURVEY.md §8d)
    eng.precompute(*wl['hyp'], reg=wl['reg'])
    fms = []
    for i in range(4):
        # the unit SURVEY.md 8d names for the precomputed regime: gradient w.r.t. log s2, log s2_f, mu_u, var_u
        eng.elbo_grad(p_h, mode=cgpcm_b200.MODE_FROZEN, reg=wl['reg'], out_grad=g_h,
                      grad_mask=cgpcm_b200.GRAD_S2 | cgpcm_b200.GRAD_S2F | cgpcm_b200.GRAD_MU_U | cgpcm_b200.GRAD_VAR_U)
        if i >= 1:
            fms.append(eng.last_timing()['total_ms'])
    fdev = torch.tensor(fms, dtype=torch.float64, device='cuda')
    if dist is not None:
        dist.all_reduce(fdev, op=dist.ReduceOp.MAX)
    frozen_value = len(fms) / (float(fdev.sum().item()) * 1e-3)

    # ---- the widened rows (SURVEY.md 8f ranks 1-3) on the same frozen statistics: device time per unit of work
    rng = np.random.default_rng(1)
    nh = args.m
    eng.fpi(p_h.numpy(), 1, reg=wl['reg'])
    eng.fpi(p_h.numpy(), 2, reg=wl['reg'])
    fpi_ms = eng.last_timing()['total_ms'] / 2.5          # 2 rounds + the convert half round
    smp = wl['params'][5:5 + nh] + .01 * rng.standard_normal(nh)
    eng.elbo_smf(p_h.numpy(), smp, mode=cgpcm_b200.MODE_FROZEN, reg=wl['reg'])
    eng.elbo_smf(p_h.numpy(), smp, mode=cgpcm_b200.MODE_FROZEN, reg=wl['reg'])
    smf_ms = eng.last_timing()['total_ms']
    t_star = np.linspace(wl['t'][0], wl['t'][-1], 2048)
    samples = wl['params'][5:5 + nh] + .01 * rng.standard_normal((8, nh))
    eng.predict_f(p_h.numpy(), t_star, samples, reg=wl['reg'])
    eng.predict_f(p_h.numpy(), t_star, samples, reg=wl['reg'])
    pred_ms = eng.last_timing()['total_ms']
    rows = torch.tensor([fpi_ms, smf_ms, pred_ms], dtype=torch.float64, device='cuda')
    if dist is not None:
        dist.all_reduce(rows, op=dist.ReduceOp.MAX)
    fpi_ms, smf_ms, pred_ms = [float(v) for v in rows.cpu()]

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    # the sharded result against the unsharded one, same inputs, same process: rank 0 evaluates the whole series on a
    # second handle without a communicator (outside every timed region)
    elbo_vs_n1 = grad_vs_n1 = None
    if world > 1:
        # (the sharded handle stays open: closing it here would destroy this rank's NCCL communicator while the other
        # ranks have already left, and ncclCommDestroy waits for them)
        del flush
        torch.cuda.empty_cache()
        eng1 = cgpcm_b200.Engine(args.m, args.m, causal=True, device=local_rank)
        eng1.set_option('chunk', args.chunk)
        eng1.set_option('cull', args.cull)
        eng1.set_data(wl['t'], wl['y'], wl['th'], wl['tx'])
        e1, _, g1 = eng1.elbo_grad(wl['params'], reg=wl['reg'])
        elbo_vs_n1 = abs(last[0] - e1) / max(abs(e1), float(np.abs(last[1]).max()))
        grad_vs_n1 = float(np.abs(last[2] - g1).max() / np.abs(g1).max())
        eng1.close()
    peak, peak_src, peak_raw = fp64_peak()
    headline_shape = args.n == 100000 and args.m == 200 and args.chunk <= 0 and args.cull == 746.0 and world == 1
    psi_flops = (ncu_traffic() or {}).get('fp64_scalar_flops_executed_per_step') if headline_shape else None
    achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    n, m = args.n, args.m
    line = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': total_ms / args.steps, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None,
        'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': 'scaling sweep N=%d observations, nh=nx=%d, causal VCGPCM, full regime (Psi rebuilt '
                               'and differentiated), grad w.r.t. all %d variables' % (n, m, npar),
                   'n': n, 'nh': m, 'nx': m, 'cull': args.cull,
                   'chunk': args.chunk if args.chunk > 0 else 'planner (512 / 1024 / 2048 x nx columns per chunk by its cost model)',
                   'windows': {746.0: 'exact: only Psi elements / GEMM tiles that are exactly 0.0 in IEEE double '
                                      '(exp underflow of the Gaussian envelope) are skipped; same sums as the '
                                      'all-tiles evaluation in another order (other_window_settings[cull=0] holds '
                                      'the measured difference)',
                               0.0: 'every Psi tile and GEMM tile evaluated',
                               80.0: 'envelope < exp(-80) dropped'}.get(args.cull, 'envelope < exp(-cull) dropped'),
                   'l2': 'flushed between timed steps (512 MB write); every chunk streams 3 x >= %.0f MB of operands '
                         '(> 126 MB L2) and the sweep stores hold 2 x %.1f GB' % (8e-6 * m * max(args.chunk, 512) * m,
                                                                                   8e-9 * m * (hi - lo) * m),
                   'parallelism': 'observations sharded over %d GPU(s), one packed ncclAllReduce per sweep' % world,
                   'shard_balance_max_over_mean_before_each_round': balance},
        'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h),
                'how': 'wall clock of set_data(host t, y, th, tx) + cgpcm_elbo_grad(host params) -> host gradient'},
        'gpu_launches': int(launches),
        'clocks': clocks,
        'roofline': {'bound': 'tensor',
                     'kernel': 'FP64 DMMA (mma.sync m8n8k4.f64) contraction kernels: dgemm_sl_kernel (4 per chunk, '
                               'dominant), dgemm_sym_kernel (3 per chunk), dgemm_dmma_kernel (M x M algebra)',
                     'achieved': achieved, 'peak': peak, 'unit': 'TFLOP/s', 'frac': achieved / peak if peak else None,
                     'traffic': ((ncu_traffic() or {}).get('dgemm_sl_kernel_T1_bytes_per_launch')
                                 if (args.n == 100000 and args.m == 200 and args.chunk <= 0 and args.cull == 746.0
                                     and world == 1) else None),
                     'traffic_note': (ncu_traffic() or {}).get('note'),
                     'peak_source': peak_src,
                     'launches_per_step': gemm_launches / args.steps,
                     'flops_per_step': gemm_flops / args.steps,
                     'avg_launch_ms': gemm_ms / max(1, gemm_launches),
                     'share_of_step': gemm_ms / total_ms if total_ms else None,
                     # algorithmic GEMM flops of the step over the WHOLE step time (Psi kernels, M x M algebra,
                     # collectives and launch gaps included) against the same peak, per GPU
                     'whole_step_frac': (gemm_flops / (total_ms * 1e-3) / 1e12 / peak) if (total_ms and peak) else None,
                     # every FP64 instruction of the step on the pipe DMMA and DFMA share: the DMMA flops the launches
                     # executed (counted live) + the scalar FP64 flops of the Psi kernels (DFMA = 2, DMUL / DADD = 1;
                     # ncu instruction counts of one step at this shape, profiles/traffic.json), over the step time
                     'fp64_pipe_frac_whole_step': ((gemm_flops_exec / args.steps + psi_flops) / (total_ms / args.steps * 1e-3)
                                                   / 1e12 / peak) if (total_ms and peak and psi_flops is not None) else None,
                     'fp64_scalar_flops_per_step_ncu': psi_flops,
                     'dram_bytes_per_step_ncu': (ncu_traffic() or {}).get('dram_bytes_per_step') if psi_flops is not None else None,
                     'flops_executed_per_step': gemm_flops_exec / args.steps,
                     'note': 'MEASURED_PEAKS.json has no FP64 figure; peak = FP64 tensor (DMMA) rate measured by '
                             'tools/fp64_peaks.cu; flops are algorithmic: 2 K M N per launch, K M (M + 1) for the '
                             'symmetric M x M results (only the lower triangle is needed); launch durations from '
                             'CUDA events around every run of consecutive GEMM launches on the library stream'},
        'breakdown_ms_per_step': {'axx_kernel': axx_ms / args.steps, 'ahx_gen_kernels': gen_ms / args.steps,
                                  'gemm_kernels': gemm_ms / args.steps},
        # BASELINE.json's second figure: logical bytes of the Psi statistics the reference materialises
        # (8 (N nx^2 + N nh nx), SURVEY.md 8d) over the time of the kernels that construct (and reduce) them
        'psi_stat': {'value': 8e-9 * n * m * (m + m) / (1e-3 * (axx_ms + gen_ms) / args.steps)
                     if (axx_ms + gen_ms) > 0 else None,
                     'unit': 'GB/s (logical Psi-statistic bytes of the whole job / Axx + Ahx kernel time of rank 0)',
                     'logical_bytes_per_eval': 8.0 * n * m * (m + m),
                     'note': 'the statistics are never materialised: Axx is reduced in registers, Ahx is written once '
                             '(8 N nh nx bytes) for the contractions'},
        'elbo': last[0],
        'elbo_rel_diff_vs_n1': elbo_vs_n1, 'grad_rel_diff_vs_n1': grad_vs_n1,
        'other_window_settings': other,
        'frozen_regime': {'value': frozen_value, 'unit': UNIT, 'steps': len(fms),
                          'note': 'Psi sums frozen by precompute(); gradient w.r.t. log s2, log s2_f, mu_u, var_u'},
        'next_rows': {'fpi_ms_per_round': fpi_ms, 'elbo_smf_ms_per_sample': smf_ms,
                      'predict_f_ms': pred_ms, 'predict_f_shape': '2048 test inputs x 8 filter samples',
                      'note': 'SURVEY.md 8f ranks 1-3 (fpi, SMF bound / sampler target, predict_f) on the frozen '
                              'statistics at the same cull setting; device time, max over ranks'},
        'wall_s_timed_region': wall,
    }
    if not args.no_cpu_baseline and world == 1:           # the CPU leg runs beside the 1-GPU line only
        line['cpu_baseline'] = cpu_port_eval(wl, args.cpu_sample)
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


# ----------------------------------------------------------------------------- independent restarts (replicas)
def run_restarts(args):
    """`--mode restarts`: independent restarts / hyper-parameter batches, one replica (handle) per GPU and no
    communication (BASELINE.json north_star; the reference's unit is one controller.py process per resample index,
    src/experiment_toy.sh:7-11).  Every replica evaluates its own parameter vector (a different seed per task) at the
    requested shape(s); the aggregate evaluations/s is the sum over GPUs (weak scaling).  Under torchrun every rank is
    one replica; in a single process with --gpus N the replicas are driven by cgpcm_b200.batch.run, one host thread
    per GPU."""
    import torch
    import cgpcm_b200
    from cgpcm_b200 import batch

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    shapes = (['sweep'] + list(NAMED_SHAPES)) if args.shape == 'all' else [args.shape]
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))

    def workload(shape, seed):
        wl = sweep_workload(args.n, args.m, seed=seed) if shape == 'sweep' else named_workload(shape, seed=seed)
        return wl

    def replica(shape, seed, device, steps, warmup):
        """One restart: its own handle, data and variables; returns (device ms per step list, elbo)."""
        wl = workload(shape, seed)
        eng = cgpcm_b200.Engine(wl['nh'], wl['nx'], causal=True, device=device)
        eng.set_option('cull', args.cull)
        eng.set_data(wl['t'], wl['y'], wl['th'], wl['tx'])
        out = None
        for _ in range(warmup):
            out = eng.elbo_grad(wl['params'], reg=wl['reg'])
        ms, launches = [], 0
        for _ in range(steps):
            out = eng.elbo_grad(wl['params'], reg=wl['reg'])
            tm = eng.last_timing()
            ms.append(tm['total_ms'])
            launches += tm['launches']
        eng.close()
        return ms, out[0], launches

    res = {}
    sampler = ClockSampler(local_rank)
    sampler.start()
    for shape in shapes:
        steps = args.steps
        if world > 1:
            torch.cuda.synchronize()
            dist.barrier()
            w0 = time.perf_counter()
            ms, elbo, launches = replica(shape, rank, local_rank, steps, args.warmup)
            torch.cuda.synchronize()
            wall = time.perf_counter() - w0
            tt = torch.tensor([sum(ms), wall, float(launches)], dtype=torch.float64, device='cuda')
            mx = tt.clone()
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            sm = tt.clone()
            dist.all_reduce(sm, op=dist.ReduceOp.SUM)
            dev_s, n_rep, launches = float(mx[0]) * 1e-3, world, int(sm[2])
        else:
            devices = list(range(args.gpus))
            tasks = [(lambda sess, k=k: replica(shape, k, sess.device, steps, args.warmup)) for k in range(args.gpus)]
            outs = batch.run(tasks, devices=devices)
            dev_s = max(sum(o[0]) for o in outs) * 1e-3
            n_rep, launches = len(outs), sum(o[2] for o in outs)
            elbo = outs[0][1]
        res[shape] = {'value': n_rep * steps / dev_s, 'unit': UNIT, 'replicas': n_rep, 'steps_per_replica': steps,
                      'ms_per_step_per_replica': dev_s * 1e3 / steps, 'gpu_launches': launches, 'elbo_replica0': elbo}
    clocks = sampler.stop()
    if rank == 0:
        head = res[shapes[0]]
        n_gpus = world if world > 1 else args.gpus
        line = {'metric': 'VCGPCM ELBO+grad evals/sec, independent restarts (one replica per GPU, no communication)',
                'value': head['value'], 'unit': UNIT, 'n_gpus': n_gpus, 'steps': args.steps, 'warmup': args.warmup,
                'ms_per_step': head['ms_per_step_per_replica'], 'higher_is_better': True, 'scaling': 'weak',
                'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic', 'mode': 'restarts',
                'config': {'workload': 'independent restarts at shape %s (N=%d, M=%d for the sweep), full regime, one '
                                       'replica per GPU, a different seed per replica' % (shapes[0], args.n, args.m),
                           'cull': args.cull,
                           'driver': 'torchrun ranks' if world > 1 else 'cgpcm_b200.batch.run, one host thread per GPU'},
                'gpu_launches': head['gpu_launches'], 'clocks': clocks, 'shapes': res}
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == 'reference':
        run_reference(args)
    elif args.mode == 'restarts':
        run_restarts(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
