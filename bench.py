#!/usr/bin/env python
"""Benchmark of the hot path: MU iterations/s (FRO and KL, k=32, 65536 x 65536 fp32) on N B200s.

    python bench.py --gpus N --steps K --warmup W            # this implementation
    python bench.py --impl reference --steps K --warmup W     # the CPU path of the reference's algorithm
    python bench.py --steps K --warmup W --dump-outputs DIR   # also writes W and H after the last timed step, .npy

A "step" is one MU iteration = the body of the reference's fit loop (pyDNMF.py:151-172):
``update()`` + the every-10th-iteration clamp.  For each norm W warm-up steps run untimed, then
exactly K steps are timed between barrier + synchronize, with CUDA events on the launching stream;
the maximum over ranks is taken.  ``value`` = total timed iterations / total time over both norms
(the per-norm numbers are in ``by_norm``).  The data shard is far larger than L2 (A = 16 GiB per
pass), so no extra L2 flush is needed between steps.

Workload (BASELINE.json configs[1]): synthetic i.i.d. uniform(0,1) fp32 matrix, 65536 x 65536, k=32,
grid N x 1 (row shards; the matrix is fixed as N grows => strong scaling), prune off, rand init.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'MU iters/s (FRO & KL, k=32, 65536^2 fp32)'


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=30)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', default='cfg2', choices=['cfg2', 'cfg3', 'cfg4'],
                    help='BASELINE.json configuration: cfg2 (default, the headline metric), cfg3 (k=64 on a 2-D grid), cfg4 (HALS/BCD)')
    ap.add_argument('--m', type=int, default=None)
    ap.add_argument('--n', type=int, default=None)
    ap.add_argument('--k', type=int, default=None)
    ap.add_argument('--shard-side', type=int, default=None, help='cfg3: side of the square shard per GPU (default 65536); same as --m, but a name torchrun does not mistake for one of its own options')
    ap.add_argument('--no-verify', action='store_true', help='skip the distributed-vs-one-GPU check of the first step')
    ap.add_argument('--norms', default='fro,kl')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--cpu-sample', type=int, default=32768, help='side of the bounded sample of the in-line cpu_baseline leg')
    ap.add_argument('--force-generic', action='store_true', help='disable the tcgen05 path (A/B runs)')
    ap.add_argument('--no-graph', action='store_true', help='launch every step eagerly instead of replaying a CUDA graph')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write the factors W and H of every leg as DIR/<leg>_<W|H>.npy')
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.shard_side is not None:
        a.m = a.shard_side
    a.m_given, a.n_given, a.k_given = a.m is not None, a.n is not None, a.k is not None
    a.m = a.m if a.m_given else 65536
    a.n = a.n if a.n_given else 65536
    a.k = a.k if a.k_given else 32
    return a


# ------------------------------------------------------------------------------------------------
# CPU baseline: the oracle port (numpy restatement of the reference's loop) on the host cores
# ------------------------------------------------------------------------------------------------
class _RowGridView:
    """What oracle.nmf_oracle reads of a grid, for ONE forked rank of a C x 1 row grid: per-rank lists have one entry
    (p = 1) but the 1-D update takes its reducing branches (p_r = C), as a rank of `mpirun -n C` does."""

    def __init__(self, cores):
        self.p, self.p_r, self.p_c = 1, cores, 1
        self.world, self.row, self.col = [[0]], [[0]], [[0]]
        self.coords = [(0, 0)]


class _ShmAllreduce:
    """SUM all-reduce between the forked ranks through shared memory: every rank writes its operand, rank r reduces
    chunk r over the ranks in rank order, every rank reads the result (reduce-scatter + all-gather, what an MPI
    all-reduce of this size does).  Stands in for the reference's comm.allreduce (dist_nmf.py:681, :707, :799)."""

    def __init__(self, ctx, cores, max_elems):
        import ctypes
        self.cores, self.max_elems = cores, max_elems
        self.slots = ctx.RawArray(ctypes.c_float, cores * max_elems)
        self.result = ctx.RawArray(ctypes.c_float, max_elems)
        self.barrier = ctx.Barrier(cores)

    def bind(self, rank):
        self.rank = rank
        self._slots = np.frombuffer(self.slots, dtype=np.float32).reshape(self.cores, self.max_elems)
        self._result = np.frombuffer(self.result, dtype=np.float32)

    def __call__(self, vals, groups):
        x = np.ascontiguousarray(vals[0], dtype=np.float32)
        n = x.size
        self._slots[self.rank, :n] = x.ravel()
        self.barrier.wait()
        per = -(-n // self.cores)
        lo, hi = min(n, self.rank * per), min(n, (self.rank + 1) * per)
        if hi > lo:
            acc = self._slots[0, lo:hi].copy()
            for q in range(1, self.cores):
                acc += self._slots[q, lo:hi]
            self._result[lo:hi] = acc
        self.barrier.wait()
        out = self._result[:n].reshape(x.shape).astype(vals[0].dtype, copy=True)
        self.barrier.wait()
        return [out]


def _cpu_rank_work(q, red, rank, cores, shard_rows, n, k, norms, steps, warmup, seed, probe=False):
    """One forked rank of a C x 1 row grid: the oracle's update on its own row shard, single BLAS thread (the
    reference forces OMP_NUM_THREADS=1 per MPI rank, main.py:3), all-reducing W^T W / W^T A with the other ranks."""
    try:
        from threadpoolctl import threadpool_limits
        limiter = threadpool_limits(1)
    except Exception:
        limiter = None
    from oracle import nmf_oracle as O
    red.bind(rank)
    O.allreduce = red                       # cross-process instead of the in-process virtual-rank reduction
    rng = np.random.default_rng(seed + rank)
    A = rng.random((shard_rows, n), dtype=np.float32)
    rs = np.random.RandomState(7)
    H0 = rs.rand(k, n).astype(np.float32)   # replicated: identical on every rank
    res = {}
    for norm in norms:
        st = O._State()
        st.grid, st.k, st.norm, st.method, st.W_update = _RowGridView(cores), k, norm, 'mu', True
        st.A, st.dt, st.eps, st.topo = [A], A.dtype, np.finfo(np.float32).eps, '1d'
        st.W = [np.random.RandomState(11 + rank).rand(shard_rows, k).astype(np.float32)]
        st.H = [H0.copy()]
        for i in range(warmup):
            O.update(st, 1)
        red.barrier.wait()
        t0 = time.perf_counter()
        for i in range(steps):
            O.update(st, 1)
            if i % 10 == 0:
                st.H = [np.maximum(h, st.eps) for h in st.H]
                st.W = [np.maximum(w, st.eps) for w in st.W]
        red.barrier.wait()
        res[norm] = time.perf_counter() - t0
        if probe:                           # tests/test_host_logic.py: the factors this rank ends with
            res[norm + '_factors'] = (rank, st.W[0], st.H[0])
    q.put(res)
    del limiter


def _cpu_sample_side(args, want_full):
    """Largest square-equivalent sample the host can hold: the KL path of the reference materialises W@H and
    A/(W@H+eps) (two A-sized temporaries, dist_nmf.py:806) next to A and the generator's scratch."""
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        avail = 32 << 30
    m, n = args.m, args.n
    if not want_full:
        m, n = min(m, args.cpu_sample), min(n, args.cpu_sample)
    while m * n * 4 * 5 + (8 << 30) > avail and m > 1024:
        m //= 2
        n //= 2
    return m, n


def cpu_probe(m, n, k, norm, steps, cores):
    """Factors after `steps` iterations of the forked-rank CPU arm (test hook: the shared-memory all-reduce must
    reproduce the oracle's own virtual-rank result)."""
    import multiprocessing as mp
    ctx = mp.get_context('fork')
    q = ctx.Queue()
    red = _ShmAllreduce(ctx, cores, max(k * n, k * k))
    shard = m // cores
    procs = [ctx.Process(target=_cpu_rank_work, args=(q, red, r, cores, shard, n, k, [norm], steps, 0, 1234, True))
             for r in range(cores)]
    for p in procs:
        p.start()
    out = [q.get()[norm + '_factors'] for _ in procs]
    for p in procs:
        p.join()
    return sorted(out, key=lambda t: t[0])


def cpu_baseline(args, steps, warmup, full=False):
    """Times oracle.nmf_oracle (kind "port") the way the reference runs on a CPU: C = host cores forked ranks of a
    C x 1 row grid (mpirun -n C), one BLAS thread each, every rank updating its own row shard and all-reducing the
    k x k / k x n partials with the others through shared memory.  Time = slowest rank.  With `full` the workload
    is the benchmark's own matrix when the host's memory holds it; otherwise a bounded sample whose iterations/s
    are scaled by the element ratio (the loop is O(m n k)) -- `sample` says which."""
    import multiprocessing as mp
    m, n = _cpu_sample_side(args, full)
    if getattr(args, 'ref_rows', None):
        m = min(m, int(args.ref_rows))          # a row slab of the full-width matrix (time budget of the reference arm)
    k = args.k
    cores = os.cpu_count() or 1
    shard = max(1, m // cores)
    m_used = shard * cores
    scale = (m_used * n) / float(args.m * args.n)
    norms = args.norms.split(',')
    ctx = mp.get_context('fork')
    q = ctx.Queue()
    red = _ShmAllreduce(ctx, cores, max(k * n, k * k))
    procs = [ctx.Process(target=_cpu_rank_work, args=(q, red, r, cores, shard, n, k, norms, steps, warmup, 1234))
             for r in range(cores)]
    for p in procs:
        p.start()
    results = [q.get() for _ in procs]
    for p in procs:
        p.join()
    out = {}
    tot_t = 0.0
    for norm in norms:
        dt = max(r[norm] for r in results)
        out[norm] = steps / dt * scale
        tot_t += dt
    tot_it = steps * len(norms)
    exact = abs(scale - 1.0) < 1e-9
    return dict(value=tot_it / tot_t * scale, unit='iters/s', cores=int(cores), kind='port',
                sample=('oracle/nmf_oracle.py (numpy %s + OpenBLAS, 1 BLAS thread per rank) as %d forked ranks of a %dx1 grid '
                        'on %s %dx%d k=%d fp32 (%d rows per rank), shared-memory all-reduce of W^T W and W^T A between the '
                        'ranks, %d warm-up + %d timed iterations per norm, slowest rank%s'
                        % (np.__version__, cores, cores, 'the full workload' if exact else 'a sample', m_used, n, k, shard,
                           warmup, steps, '' if exact else '; iterations/s scaled by the element ratio %.5f to %dx%d'
                           % (scale, args.m, args.n))),
                by_norm=out, measured_s=tot_t, scale=scale)


def workload_config(args, world=None):
    """`config` of both arms (the reference arm runs on this arm's configuration)."""
    return {'workload': 'synthetic %dx%d fp32 non-negative, KL and FRO MU k=%d (BASELINE.json configs[1]); row grid Nx1, '
                        'one row shard per GPU' % (args.m, args.n, args.k), 'norms': args.norms}


def _bounded_rows_for_budget(args, steps, warmup, budget_s):
    """Rows of the matrix the reference arm can afford within `budget_s` seconds for `steps + warmup` iterations per norm:
    a one-iteration calibration on a thin slab (512 rows per rank, full width) gives the host's seconds per element, the
    loop is O(m n k).  Returns None when the full workload fits the budget."""
    cores = os.cpu_count() or 1
    m_full, _ = _cpu_sample_side(args, True)
    m_cal = min(m_full, cores * 512)
    probe = argparse.Namespace(**vars(args))
    probe.m, probe.cpu_sample = m_cal, m_cal
    cal = cpu_baseline(probe, steps=1, warmup=1, full=True)
    # cal['measured_s'] = one timed iteration per norm on m_cal rows
    predicted = cal['measured_s'] * (float(m_full) / m_cal) * (steps + warmup)
    if predicted <= budget_s:
        return None
    rows = int(m_full * budget_s / predicted) // cores * cores
    return max(rows, cores * 256)


def run_reference_arm(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    t0 = time.perf_counter()
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    # the whole run must end within a few minutes whatever --steps / --warmup ask for: full workload when the host
    # affords it (16 cores: ~10 s per FRO + KL iteration pair at 65536^2), else a bounded row slab of it, scaled
    rows = _bounded_rows_for_budget(args, steps, warmup, float(os.environ.get('DNMF_REF_BUDGET_S', '200')))
    if rows is not None:
        args = argparse.Namespace(**vars(args))
        args.ref_rows = rows
    cb = cpu_baseline(args, steps, warmup, full=True)
    wall = time.perf_counter() - t0
    steps_total = args.steps * len(args.norms.split(','))
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': cb['value'], 'unit': 'iters/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup,
        # measured time per step of what actually ran (equals 1000 / value when the full workload ran)
        'ms_per_step': 1000.0 * cb['measured_s'] / steps_total,
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args),
        'cpu_baseline': {kk: cb[kk] for kk in ('value', 'unit', 'cores', 'kind', 'sample')},
        'e2e': {'value': cb['value'], 'unit': 'iters/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0, 'by_norm': cb['by_norm'], 'wall_s': wall,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# clocks sampling (nvidia-smi during the timed region)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons of one GPU while the timed region runs.  Polls NVML every few milliseconds from a
    thread (an 8-GPU timed region lasts ~30 ms, shorter than nvidia-smi's sampling period); falls back to
    `nvidia-smi -lms 100` when the NVML binding is missing."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
    NAMES = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']

    def __init__(self, index):
        self.rows = []          # (t, sm_mhz, sm_max_mhz, [reason names])
        self.proc = None
        self._stop = False
        self.source = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates all GPUs of the box; CUDA_VISIBLE_DEVICES may remap the index torch sees
            vis = os.environ.get('CUDA_VISIBLE_DEVICES')
            phys = index
            if vis:
                ent = vis.split(',')[index].strip()
                phys = int(ent) if ent.isdigit() else index
            h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            bits = [(getattr(pynvml, 'nvmlClocksEventReasonHwSlowdown', 0x8), 'hw_slowdown'),
                    (getattr(pynvml, 'nvmlClocksEventReasonHwThermalSlowdown', 0x40), 'hw_thermal_slowdown'),
                    (getattr(pynvml, 'nvmlClocksEventReasonSwThermalSlowdown', 0x20), 'sw_thermal_slowdown'),
                    (getattr(pynvml, 'nvmlClocksEventReasonSwPowerCap', 0x4), 'sw_power_cap')]
            reasons_fn = getattr(pynvml, 'nvmlDeviceGetCurrentClocksEventReasons', None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons

            def poll():
                while not self._stop:
                    try:
                        sm = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                        r = int(reasons_fn(h))
                        self.rows.append((time.perf_counter(), sm, mx, [nm for bit, nm in bits if r & bit]))
                    except Exception:
                        pass
                    time.sleep(0.004)
            self.th = threading.Thread(target=poll, daemon=True)
            self.th.start()
            self.source = 'nvml'
            return
        except Exception:
            pass
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '--query-gpu=' + self.Q, '--format=csv,noheader,nounits',
                                          '-lms', '100', '-i', str(index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._pump, daemon=True)
            self.th.start()
            self.source = 'nvidia-smi'
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.strip().split(',')]
            if len(f) < 7:
                continue
            try:
                self.rows.append((time.perf_counter(), float(f[0]), float(f[1]),
                                  [nm for nm, v in zip(self.NAMES, f[3:7]) if v.lower().startswith('active')]))
            except ValueError:
                continue

    def stop(self):
        self._stop = True
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                pass

    def summary(self, windows):
        sm, mx, reasons = [], [], set()
        for t, s_, m_, rs in self.rows:
            if not any(a <= t <= b for a, b in windows):
                continue
            sm.append(s_)
            mx.append(m_)
            reasons.update(rs)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0, 'source': self.source}
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(max(mx)), 'reasons': sorted(reasons),
                'samples': len(sm), 'source': self.source}


# ------------------------------------------------------------------------------------------------
# this implementation
# ------------------------------------------------------------------------------------------------
# BASELINE.json configs measured by this file (cfg1 / cfg5, the tiny-matrix ones, live in tools/bench_configs.py)
CONFIGS = {
    'cfg2': dict(legs=[('fro', 'mu'), ('kl', 'mu')], k=32, scaling='strong', metric=METRIC),
    'cfg3': dict(legs=[('fro', 'mu')], k=64, scaling='weak',
                 metric='MU iters/s (FRO, k=64, 65536^2 fp32 per GPU; 262144x131072 on the 4x2 grid of 8 B200)'),
    'cfg4': dict(legs=[('fro', 'hals'), ('fro', 'bcd')], k=16, scaling='strong',
                 metric='HALS & BCD iters/s (FRO, k=16, 131072x65536 fp32)'),
}
CFG3_GRIDS = {1: (1, 1), 2: (2, 1), 4: (2, 2), 8: (4, 2)}
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays, limit):
    """Writes every array of `arrays` (name -> numpy array) as out_dir/<name>.npy.  When together they exceed `limit`
    bytes, each keeps the same seeded sample of its longest axis on every run, so two builds stay comparable."""
    os.makedirs(out_dir, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > limit:
            ax = int(np.argmax(a.shape))
            keep = max(1, a.shape[ax] * limit // total)
            idx = np.sort(np.random.default_rng(0).choice(a.shape[ax], keep, replace=False))
            a = np.take(a, idx, axis=ax)
        np.save(os.path.join(out_dir, name + '.npy'), a)


def resolve_config(args, world):
    """(m, n, k, p_r, p_c) of the run.  cfg2 / cfg4: the matrix is fixed, row grid N x 1 (strong scaling).  cfg3: every
    GPU holds a 65536 x 65536 shard of a (65536 p_r) x (65536 p_c) matrix; 8 GPUs = BASELINE's 262144 x 131072 on 4 x 2."""
    c = CONFIGS[args.config]
    if args.config == 'cfg3':
        p_r, p_c = CFG3_GRIDS[world]
        side = args.m if args.m_given else 65536
        return side * p_r, side * p_c, (args.k if args.k_given else c['k']), p_r, p_c
    if args.config == 'cfg4':
        m = args.m if args.m_given else 131072
        n = args.n if args.n_given else 65536
        return m, n, (args.k if args.k_given else c['k']), world, 1
    return args.m, args.n, args.k, world, 1


def run_ours(args):
    import torch
    import torch.distributed as dist
    from pydnmfk_b200 import _lib as L
    from pydnmfk_b200 import device as D
    from pydnmfk_b200.dist_comm import MPI, MPI_comm
    from pydnmfk_b200.dist_nmf import nmf_algorithms_1D, nmf_algorithms_2D
    from pydnmfk_b200.graphs import StepGraphs, graphs_enabled
    from pydnmfk_b200.pyDNMF import PyNMF
    from pydnmfk_b200.utils import parse, determine_block_params, data_operations

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('DNMF_BENCH_DEVICE', os.environ.get('LOCAL_RANK', '0')))   # (override: several ranks on one GPU, gloo, script checks)
    cfg = CONFIGS[args.config]
    legs = [l for l in cfg['legs'] if args.config != 'cfg2' or l[0] in args.norms.split(',')]
    # CPU baseline first (forks workers; done before this process creates a CUDA context)
    cb = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and args.config == 'cfg2':
        cb = cpu_baseline(args, steps=3, warmup=1)
        cb = {kk: cb[kk] for kk in ('value', 'unit', 'cores', 'kind', 'sample', 'by_norm')}
    assert torch.cuda.is_available(), 'bench.py needs a GPU (no CPU fallback)'
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if args.force_generic:
        L.set_force_generic(True)
    comm = MPI.COMM_WORLD          # initialises NCCL from the torchrun environment when world > 1
    assert comm.size == world
    m, n, k, p_r, p_c = resolve_config(args, world)
    comms = MPI_comm(comm, p_r, p_c)
    two_d = p_r != 1 and p_c != 1
    blk = determine_block_params(rank, (p_r, p_c), (m, n))
    (r0, c0), (r1, c1) = blk.determine_block_index_range_asymm()
    m_i, n_j = r1 - r0 + 1, c1 - c0 + 1
    eps = float(np.finfo(np.float32).eps)

    def make_params(norm, method, itr):
        p = parse()
        p.comm1, p.comm, p.row_comm, p.col_comm = comm, comms, comms.cart_1d_row(), comms.cart_1d_column()
        p.p_r, p.p_c, p.k, p.m, p.n, p.itr, p.init, p.verbose = p_r, p_c, k, m, n, itr, 'rand', False
        p.norm, p.method, p.prune, p.W_update, p.eps = norm, method, False, True, np.finfo(np.float32).eps
        p.rank, p.topo = rank, ('2d' if two_d else '1d')
        return p

    # synthetic shard, generated on the device (Philox seed 1234 + rank), strictly positive
    g = torch.Generator(device=dev)
    g.manual_seed(1234 + rank)
    A = torch.rand((m_i, n_j), generator=g, device=dev, dtype=torch.float32)
    dims = data_operations(A, make_params('fro', 'mu', 1)).params
    w_rows, h_cols = (dims.m_loc, dims.n_loc) if two_d else (m_i, n_j)
    g.manual_seed(7 + (rank if two_d else 0))
    W0 = torch.rand((w_rows, k), generator=g, device=dev, dtype=torch.float32)
    g.manual_seed(7 + (rank if two_d else 0))
    H0 = torch.rand((k, h_cols), generator=g, device=dev, dtype=torch.float32)
    if not two_d and world > 1:
        g.manual_seed(99 + rank)              # row shards of W differ per rank; H is the replicated factor
        W0 = torch.rand((w_rows, k), generator=g, device=dev, dtype=torch.float32)
    ops = D.default_ops()
    Alg = nmf_algorithms_2D if two_d else nmf_algorithms_1D

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        if world > 1:
            t = torch.tensor([x], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return float(x)

    # ---- correctness of the distributed step before anything is timed -----------------------------------------
    # (1) one iteration per leg on the grid vs the same iteration on ONE GPU holding the whole matrix (rank 0
    #     regenerates every shard from its seed), when the whole matrix fits next to the shard;
    # (2) replicated factors must be identical on every rank.
    verify = {}
    total_bytes = float(m) * n * 4
    if world > 1 and not args.no_verify:
        for norm, method in legs:
            if method == 'bcd':
                continue                      # BCD scales the factors by a global norm first; covered by tests/
            W, H = W0.clone(), H0.clone()
            alg = Alg(A, W, H, params=make_params(norm, method, 1))
            alg.update()
            torch.cuda.synchronize()
            rec = {}
            if not two_d:
                ref = H.clone()
                dist.broadcast(ref, src=0)
                rec['replica_max_abs_diff'] = allmax(float((H - ref).abs().max().item()))
                if total_bytes <= 24 * 2 ** 30:
                    Wall = [torch.empty_like(W0) for _ in range(world)]
                    dist.all_gather(Wall, W)
                    W0all = [torch.empty_like(W0) for _ in range(world)]
                    dist.all_gather(W0all, W0)
                    if rank == 0:
                        shards = []
                        for q in range(world):
                            gq = torch.Generator(device=dev)
                            gq.manual_seed(1234 + q)
                            bq = determine_block_params(q, (p_r, p_c), (m, n)).determine_block_index_range_asymm()
                            shards.append(torch.rand((bq[1][0] - bq[0][0] + 1, n), generator=gq, device=dev, dtype=torch.float32))
                        Afull = torch.cat(shards)
                        del shards
                        Wf, Hf = torch.cat(W0all), H0.clone()
                        solo = MPI_comm(type(comm)([rank], None), 1, 1)
                        ps = make_params(norm, method, 1)
                        ps.comm1, ps.comm, ps.row_comm, ps.col_comm = solo.comm, solo, solo.cart_1d_row(), solo.cart_1d_column()
                        ps.p_r, ps.p_c = 1, 1
                        nmf_algorithms_1D(Afull, Wf, Hf, params=ps).update()
                        torch.cuda.synchronize()
                        dW = float((torch.cat(Wall) - Wf).norm() / Wf.norm())
                        dH = float((H - Hf).norm() / Hf.norm())
                        rec['vs_one_gpu'] = {'relW': dW, 'relH': dH}
                        del Afull, Wf, Hf
                        assert dW < 1e-5 and dH < 1e-5, 'distributed step differs from the 1-GPU step: %r' % rec
                    del Wall, W0all
                    torch.cuda.empty_cache()
                assert rec['replica_max_abs_diff'] <= 1e-6, 'H replicas differ across ranks: %r' % rec
            if two_d:
                # 2-D grids (the whole matrix does not fit one GPU at cfg3): the squared error of the updated factors two
                # independent ways -- (1) the direct residual over the resident shards (all-gathers of W and H + one pass),
                # (2) the trace identity ||A||^2 - 2 <W, A H^T> + <W^T W, H H^T> through the update's own distributed
                # contraction (all-gather -> pass -> reduce-scatter) and Grams.  A wrong shard order or collective shows
                # up as a mismatch; the two share no kernel on the A side.
                try:
                    res = alg._residual_global(W, H)                 # [||A - W H||^2, ||A||^2], all-reduced
                    AH = alg._AH(H)                                  # rows of this rank's W shard
                    tt = ops.trace_terms(W, AH, alg._gram_W(W), alg._gram_H(H))
                    tt[:, 1] /= float(world)                         # the Gram term is global on every rank already
                    tt = comm.allreduce_(tt)
                    torch.cuda.synchronize()
                    direct, a2 = float(res[0].item()), float(res[1].item())
                    trace = a2 - 2.0 * float(tt[0, 0].item()) + float(tt[0, 1].item())
                    rec['residual_direct_vs_trace_identity'] = {'direct': direct, 'trace': trace,
                                                                'rel_diff': abs(direct - trace) / max(direct, 1e-300)}
                    assert abs(direct - trace) <= 1e-3 * direct, '2-D step: direct residual and trace identity disagree: %r' % rec
                except AssertionError:
                    raise
                except Exception as ex:          # the check must never take the benchmark down
                    rec['residual_direct_vs_trace_identity'] = {'error': repr(ex)}
            verify['%s-%s' % (norm, method)] = rec
            del alg
            sync_all()

    sampler = ClockSampler(local) if rank == 0 else None
    windows = []
    by_leg, pass_stats, outputs = {}, {}, {}
    launches = 0
    tot_ms, tot_it = 0.0, 0
    paths = {}
    for norm, method in legs:
        leg = '%s-%s' % (norm, method) if args.config != 'cfg2' else norm
        p = make_params(norm, method, args.steps)
        W, H = W0.clone(), H0.clone()
        alg = Alg(A, W, H, params=p)

        def clamp():
            ops.clamp_min(H, eps)
            ops.clamp_min(W, eps)

        can_graph = graphs_enabled(comm, 'mu') and not args.no_graph
        if method == 'bcd':
            alg.bcd_begin()                        # initWandH once; a step = one iteration of dist_nmf.py:996-1047
            eager_step, with_clamp = alg.bcd_step, False
        else:
            eager_step, with_clamp = alg.update, True
        sg = StepGraphs(eager_step, clamp if with_clamp else (lambda: None)) if can_graph else None

        def step(i):
            # the product's own loop body (PyNMF.fit): CUDA-graph replay of update() [+ clamp every 10th iteration]
            if sg is not None:
                sg.clamped() if (with_clamp and i % 10 == 0) else sg.plain()
            else:
                eager_step()
                if with_clamp and i % 10 == 0:
                    clamp()

        L.launch_count(reset=True)
        L.pass_count(True, reset=True)
        L.pass_count(False, reset=True)
        eager_step()                       # eager step: sizes the workspace, counts the launches of one step
        if with_clamp:
            clamp()
        launches_per_step = L.launch_count()
        passes_per_step = L.pass_count(True) + L.pass_count(False)
        paths[leg] = 'tcgen05' if (L.pass_count(True) > 0 and L.pass_count(False) == 0) else (
            'generic' if L.pass_count(True) == 0 else 'mixed')
        for i in range(args.warmup):
            step(i)
        sync_all()
        ops.timers = {} if sg is None else None
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_a = time.perf_counter()
        e0.record()
        for i in range(args.steps):
            step(i)
        e1.record()
        sync_all()
        t_b = time.perf_counter()
        windows.append((t_a, t_b))
        ms = allmax(e0.elapsed_time(e1))
        if args.dump_outputs:
            # the factors after the last timed step (the eager roofline replica below steps them further)
            sfx = '_rank%d' % rank if world > 1 else ''
            outputs[leg + '_W' + sfx] = alg._W().cpu().numpy()
            outputs[leg + '_H' + sfx] = alg._H().cpu().numpy()
        launches += launches_per_step * args.steps     # same launches per replayed step as in the eager one
        if sg is not None:
            # per-kernel CUDA events cannot be placed inside a replayed graph: time the same steps once more, eagerly,
            # with an event pair around every A-streaming pass (not part of `value`)
            ops.timers = {}
            for i in range(min(args.steps, 10)):
                eager_step()
                if with_clamp and i % 10 == 0:
                    clamp()
            sync_all()
        pass_stats[leg] = ops.timer_summary()
        ops.timers = None
        by_leg[leg] = {'iters_per_s': args.steps / (ms / 1000.0), 'ms_per_step': ms / args.steps,
                       'a_passes_per_step': int(passes_per_step)}
        tot_ms += ms
        tot_it += args.steps
        assert torch.isfinite(W).all() and torch.isfinite(H).all()
        if not two_d and world > 1 and p_c == 1:
            ref = H.clone()
            dist.broadcast(ref, src=0)
            d = allmax(float((H - ref).abs().max().item()))
            by_leg[leg]['replica_max_abs_diff_after_timed_steps'] = d
            assert d <= 1e-5, 'H replicas drifted apart across ranks (%g)' % d
        if getattr(alg, '_px', None) is not None:
            alg._px.check()
            by_leg[leg]['h_half_step'] = 'peer-memory exchange (dnmf_xchg_update_h)'
        del alg, sg, step, clamp, eager_step      # captured graphs (with their NCCL nodes) must die before the process group does
        gc.collect()
        torch.cuda.synchronize()

    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs, DUMP_LIMIT_BYTES // world)
    value = tot_it / (tot_ms / 1000.0)

    # ---- roofline of the dominant kernel (A-streaming pass), measured live with CUDA events ----
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    peak = float(peaks.get('hbm_gbs', 6650.0))
    peak_src = 'MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)' if 'hbm_gbs' in peaks else 'fallback 6650 GB/s'
    pass_bytes = float(m_i) * n_j * 4.0
    per_kernel = {}
    dom = None
    for leg, st in pass_stats.items():
        for opn, (cnt, mean_ms) in st.items():
            gbs = pass_bytes / (mean_ms * 1e-3) / 1e9
            per_kernel['%s:%s' % (leg, opn)] = {'launches': cnt, 'mean_ms': mean_ms, 'GBps': gbs, 'frac': gbs / peak}
            if dom is None or cnt * mean_ms > dom[1]:
                dom = ('%s:%s' % (leg, opn), cnt * mean_ms, gbs)
    # DRAM traffic of the dominant kernel from the committed ncu --set full capture (same shard shape only)
    traffic = None
    try:
        cap = json.load(open(os.path.join(ROOT, 'profiles', 'ncu_traffic.json')))
        if dom and (cap['m_loc'], cap['n'], cap['k']) == (m_i, n_j, k) and dom[0] in cap['kernels']:
            traffic = cap['kernels'][dom[0]]['dram_bytes_per_launch']
    except Exception:
        pass
    # tensor-pipe side of the same kernel: 3 tf32 terms per product (fp32-accurate split), 2 GEMMs per pass for KL.
    # Peak = half the measured bf16 throughput (kind::tf32 runs at half the bf16 rate); nominal dense tf32 = 1125 TF/s.
    tensor = None
    if dom:
        kp = 16 if k <= 16 else (32 if k <= 32 else 64)
        gemms = 2 if dom[0].split(':')[-1].startswith('kl') or dom[0].endswith('ah_res') else 1
        flops = 2.0 * float(m_i) * n_j * kp * 3 * gemms
        t_ms = per_kernel[dom[0]]['mean_ms']
        tf32_peak = float(peaks.get('bf16_tflops_sustained', 1380.0)) / 2.0
        ach = flops / (t_ms * 1e-3) / 1e12
        tensor = {'tf32_flops_per_launch': flops, 'achieved_tflops': ach, 'peak_tflops': tf32_peak,
                  'peak_source': 'MEASURED_PEAKS.json bf16_tflops_sustained / 2' if 'bf16_tflops_sustained' in peaks else 'fallback 690 TF/s',
                  'frac': ach / tf32_peak, 'frac_of_nominal_1125': ach / 1125.0}
    roofline = {'bound': 'hbm', 'achieved': dom[2] if dom else None, 'peak': peak, 'unit': 'GB/s', 'tensor': tensor,
                'frac': (dom[2] / peak) if dom else None, 'traffic': traffic,
                'traffic_source': 'profiles/ncu_traffic.json (dram__bytes_read.sum + dram__bytes_write.sum per launch)' if traffic else None, 'kernel': dom[0] if dom else None,
                'peak_source': peak_src, 'algorithmic_bytes_per_launch': pass_bytes, 'per_kernel': per_kernel,
                'iteration_frac_of_A_streaming_roofline': {
                    nm: (2.0 * pass_bytes / (v['ms_per_step'] * 1e-3) / 1e9) / peak for nm, v in by_leg.items()}}

    # ---- end to end through the public API with HOST buffers (PyNMF(A_host).fit()) ----------------
    e2e = None
    if not args.no_e2e:
        try:
            host = torch.empty((m_i, n_j), dtype=torch.float32, pin_memory=True)
            host.copy_(A)
            torch.cuda.synchronize()
            A_host = host.numpy()
            del A
            torch.cuda.empty_cache()
            e_t, e_it, h2d, d2h = 0.0, 0, 0, 0
            for norm, method in legs:
                # one untimed short fit through the same call first: communicator / peer-exchange set-up, kernel
                # attributes, the tf32 calibration probe and the first graph capture are one-off costs of the process,
                # not of a fit (tools/e2e_phases.py: 1.4 s + 1.0 s on the first two fits of a 2-GPU job, then 0.35 s per fit)
                pw = make_params(norm, method, 4)
                np.random.seed(7 + rank)
                PyNMF(A_host, params=pw).fit()
                p = make_params(norm, method, args.steps)
                np.random.seed(7 + rank)
                sync_all()
                t0 = time.perf_counter()
                Wn, Hn, err = PyNMF(A_host, params=p).fit()
                torch.cuda.synchronize()
                dt = allmax(time.perf_counter() - t0)
                e_t += dt
                e_it += args.steps
                h2d += A_host.nbytes + (w_rows * k + k * h_cols) * 4
                d2h += Wn.nbytes + Hn.nbytes + 8
                assert np.isfinite(float(err))
            e2e = {'value': e_it / e_t, 'unit': 'iters/s', 'h2d_bytes_per_step': h2d * world / e_it,
                   'd2h_bytes_per_step': d2h * world / e_it,
                   'note': 'PyNMF(A_host, params).fit() with itr=%d per leg: pinned host shard -> HBM copy, rand init on '
                           'host, %d iterations, normalise + relative error, factors and error back to host; bytes are '
                           'the whole-fit transfers divided by the iterations; one untimed 4-iteration fit per leg runs first (one-off process set-up)' % (args.steps, args.steps)}
        except Exception as ex:  # pinned host memory may be unavailable on a small host
            e2e = {'value': None, 'unit': 'iters/s', 'h2d_bytes_per_step': None, 'd2h_bytes_per_step': None,
                   'note': 'e2e leg failed: %r' % (ex,)}

    clocks = None
    if sampler is not None:
        sampler.stop()
        clocks = sampler.summary(windows)

    if rank == 0:
        config = workload_config(args) if args.config == 'cfg2' else {
            'workload': 'synthetic %dx%d fp32 non-negative, %s, k=%d (BASELINE.json %s)' % (
                m, n, ' and '.join('%s-%s' % (a.upper(), b.upper()) for a, b in legs), k, args.config)}
        config.update({'grid': '%dx%d' % (p_r, p_c), 'shard': '%dx%d per GPU' % (m_i, n_j),
                       'l2': 'inputs larger than L2 (one A pass streams %.1f GiB per GPU)' % (pass_bytes / 2 ** 30),
                       'math_mode': 'fp32-accurate', 'paths': paths,
                       'launch': 'cuda-graph replay of the step (as PyNMF.fit does)' if not args.no_graph else 'eager',
                       'roofline_timing': 'CUDA events around each A-streaming pass, eager replica of the timed steps' if not args.no_graph else 'CUDA events around each A-streaming pass inside the timed steps'})
        line = {
            'metric': cfg['metric'], 'value': value, 'unit': 'iters/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': tot_ms / tot_it, 'higher_is_better': True, 'scaling': cfg['scaling'],
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': config,
            ('by_norm' if args.config == 'cfg2' else 'by_leg'): by_leg, 'roofline': roofline, 'cpu_baseline': cb, 'e2e': e2e,
            'gpu_launches': int(launches), 'clocks': clocks, 'verify': verify or None,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        # Leave without tearing NCCL down: destroy_process_group() can block for minutes once collectives have been
        # captured into CUDA graphs, and the JSON line is already out.  Every rank exits 0 right after a final barrier.
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def main():
    args = parse_args()
    if args.impl == 'reference':
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
