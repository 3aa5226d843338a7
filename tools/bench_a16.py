#!/usr/bin/env python
"""16-bit storage of the data shard (params.a_storage) against fp32, on one GPU, in one process.

    python tools/bench_a16.py [--m 65536 --n 65536 --k 32] [--reps 20] [--steps 20] [--itr 50] [--out FILE.json]

Shape: bench.py's cfg2 (65536 x 65536 uniform(0,1) data, k = 32).  The three legs -- fp32, fp16, bf16 storage -- run
alternately, every measurement with CUDA events:
  - per pass (A H^T, W^T A, and the fused KL contractions): mean over --reps launches after one warm-up launch, with
    the achieved rate m n b / t (b = 4 or 2 bytes per element read) over a device-to-device copy bandwidth measured in
    the same process (2 x bytes / t of an 8 GiB cudaMemcpyAsync);
  - per replayed iteration of FRO-MU, HALS, KL-MU and BCD: the update step of PyNMF's loop on the device-resident
    shard, run once eagerly, captured as a CUDA graph (graphs.StepGraphs, as PyNMF.fit replays it) and replayed --steps
    times between two events; two alternating rounds of the three legs, the faster round kept;
  - end to end: PyNMF(numpy fp32 A, a_storage).fit() for FRO-MU from host memory (rounding and upload included),
    host clock around work that ends in a device synchronise;
  - the output difference of the 16-bit fits from the fp32 fit of the rounded matrix (relative Frobenius of W and H,
    relative difference of recon_err), next to a yardstick of how sensitive the fit is to rounding-level differences:
    the same fp32 fit on the tcgen05 kernels vs on the generic CUDA-core kernels.
The card's name and power limit are read in the same process and stored with the numbers.  A 16 GiB shard is far larger
than L2, so no cache flush is needed between passes.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

LEGS = ['float32', 'float16', 'bfloat16']
TD = {'float32': torch.float32, 'float16': torch.float16, 'bfloat16': torch.bfloat16}


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i',
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(), nvidia_smi=q.stdout.strip())


def ev_time(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def copy_bw():
    src = torch.empty(8 << 30, dtype=torch.uint8, device='cuda')
    dst = torch.empty_like(src)
    ms = ev_time(lambda: dst.copy_(src), 5)
    del src, dst
    torch.cuda.empty_cache()
    return 2.0 * (8 << 30) / (ms * 1e-3)


def params(k, itr, norm, method, a_storage):
    from pydnmfk_b200.dist_comm import MPI, MPI_comm
    from pydnmfk_b200.utils import parse
    MPI._reset()
    comms = MPI_comm(MPI.COMM_WORLD, 1, 1)
    p = parse()
    p.size, p.rank, p.comm1, p.comm, p.p_r, p.p_c = 1, 0, comms.comm, comms, 1, 1
    p.row_comm, p.col_comm = comms.cart_1d_row(), comms.cart_1d_column()
    p.k, p.itr, p.init, p.verbose, p.norm, p.method, p.prune = k, itr, 'rand', False, norm, method, False
    p.a_storage = a_storage
    return p


def fit(A, k, itr, norm, method, a_storage, seed=7):
    from pydnmfk_b200.pyDNMF import PyNMF
    np.random.seed(seed)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    nmf = PyNMF(A, params=params(k, itr, norm, method, a_storage))
    W, H, err = nmf.fit()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, W, H, float(err)


def step_ms(A, k, norm, method, a_storage, steps):
    """CUDA-event time of one replayed update step (the body of PyNMF's loop without the every-10th clamp; for BCD the
    iteration of FRO_BCD_update) on PyNMF's device-resident shard and factors."""
    from pydnmfk_b200.dist_nmf import nmf_algorithms_1D
    from pydnmfk_b200.graphs import StepGraphs
    from pydnmfk_b200.pyDNMF import PyNMF
    np.random.seed(7)
    nmf = PyNMF(A, params=params(k, steps, norm, method, a_storage))
    W, H = nmf._get_factors()
    alg = nmf_algorithms_1D(nmf.A_ij, W, H, params=nmf.params)
    if method == 'bcd':
        alg.bcd_begin()
        step = alg.bcd_step
    else:
        step = alg.update
    step()                                   # eager: kernel attributes, workspaces
    sg = StepGraphs(step, lambda: None)
    sg.plain()                               # capture + first replay
    ms = ev_time(sg.plain, steps)
    del sg, alg, nmf
    torch.cuda.empty_cache()
    return ms


def rel(x, y):
    x = x.double() if isinstance(x, torch.Tensor) else torch.from_numpy(np.asarray(x, np.float64))
    y = y.double() if isinstance(y, torch.Tensor) else torch.from_numpy(np.asarray(y, np.float64))
    return float(torch.linalg.norm(x.cpu() - y.cpu()) / torch.linalg.norm(y.cpu()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--m', type=int, default=65536)
    ap.add_argument('--n', type=int, default=65536)
    ap.add_argument('--k', type=int, default=32)
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--steps', type=int, default=20, help='replays of the captured step per timing')
    ap.add_argument('--itr', type=int, default=50, help='iterations of the fits whose outputs are compared')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    from pydnmfk_b200 import _lib as L
    from pydnmfk_b200 import device as D
    m, n, k = a.m, a.n, a.k
    it2 = a.itr
    res = dict(tool='tools/bench_a16.py', shape=[m, n, k], card=card(), copy_bw_Bps=copy_bw())
    ops = D.default_ops()
    torch.manual_seed(0)
    A32 = torch.rand((m, n), device='cuda')
    A = {'float32': A32, 'float16': A32.to(torch.float16), 'bfloat16': A32.to(torch.bfloat16)}
    H = torch.rand((k, n), device='cuda') + 0.1
    W = torch.rand((m, k), device='cuda') + 0.1
    eps = float(np.finfo(np.float32).eps)

    # ---- passes ----
    passes = {leg: {} for leg in LEGS}
    ops_list = [('ah', lambda X: ops.ah(X, H)), ('wta', lambda X: ops.wta(X, W, transposed_out=True)),
                ('kl_uht', lambda X: ops.kl_uht(X, W, H, eps)), ('kl_wtu', lambda X: ops.kl_wtu(X, W, H, eps, True))]
    for rnd in range(2):                         # two alternating rounds of the three legs
        for leg in LEGS:
            for name, f in ops_list:
                ms = ev_time(lambda: f(A[leg]), a.reps)
                path = L.last_path()
                passes[leg].setdefault(name, []).append(dict(ms=ms, path=path))
    for leg in LEGS:
        b = 4 if leg == 'float32' else 2
        for name in list(passes[leg]):
            runs = passes[leg][name]
            ms = min(r['ms'] for r in runs)
            passes[leg][name] = dict(ms_rounds=[r['ms'] for r in runs], ms=ms, tcgen05=runs[-1]['path'] == 1,
                                     bytes_per_s=m * n * b / (ms * 1e-3),
                                     share_of_copy_bw=m * n * b / (ms * 1e-3) / res['copy_bw_Bps'])
    for name, _ in ops_list:
        passes.setdefault('speedup_vs_float32', {})[name] = {
            leg: passes['float32'][name]['ms'] / passes[leg][name]['ms'] for leg in LEGS[1:]}
    res['passes'] = passes

    # ---- replayed iterations (CUDA events) ----
    methods = (('fro', 'mu'), ('fro', 'hals'), ('kl', 'mu'), ('fro', 'bcd'))
    iters = {}
    for norm, method in methods:
        key = '%s-%s' % (norm, method)
        runs = {leg: [] for leg in LEGS}
        for rnd in range(2):                     # two alternating rounds of the three legs
            for leg in LEGS:
                runs[leg].append(step_ms(A32, k, norm, method, None if leg == 'float32' else leg, a.steps))
        iters[key] = {leg: dict(ms_per_iter=min(runs[leg]), ms_rounds=runs[leg]) for leg in LEGS}
        for leg in LEGS[1:]:
            iters[key][leg]['speedup_vs_float32'] = iters[key]['float32']['ms_per_iter'] / iters[key][leg]['ms_per_iter']
    res['iterations'] = iters
    res['iterations_note'] = ('CUDA events around %d replays of the captured update step after an eager step and the '
                              'capture; 16-bit legs round the fp32 shard on the device at set-up' % a.steps)

    # ---- output difference from the fp32 fit of the rounded matrix ----
    diffs = {}
    for norm, method in methods:
        key = '%s-%s' % (norm, method)
        _, W32, H32, e32 = fit(A32, k, it2, norm, method, None)
        L.set_force_generic(True)
        _, Wg, Hg, eg = fit(A32, k, it2, norm, method, None)
        L.set_force_generic(False)
        diffs[key] = dict(yardstick_fp32_tcgen05_vs_generic=dict(rel_W=rel(W32, Wg), rel_H=rel(H32, Hg),
                                                                 rel_err=abs(e32 - eg) / eg))
        for leg in LEGS[1:]:
            _, W2, H2, e2 = fit(A32, k, it2, norm, method, leg)
            Ar = A[leg].to(torch.float32)                     # the rounded matrix, as fp32
            _, Wr, Hr, er = fit(Ar, k, it2, norm, method, None)
            del Ar
            torch.cuda.empty_cache()
            diffs[key][leg] = dict(rel_W=rel(W2, Wr), rel_H=rel(H2, Hr), rel_err=abs(e2 - er) / er)
    res['output_diff_vs_fp32_fit_of_rounded'] = diffs
    res['output_diff_note'] = '%d-iteration fits, same seed' % it2

    # ---- end to end from host memory ----
    if not a.no_e2e:
        Ah = A32.cpu().numpy()
        del A, A32
        torch.cuda.empty_cache()
        e2e = {}
        for leg in LEGS:
            st = None if leg == 'float32' else leg
            e2e[leg] = dict(seconds=fit(Ah, k, it2, 'fro', 'mu', st)[0], itr=it2)
        res['e2e_host_fro_mu'] = e2e
    line = json.dumps(res, indent=1)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
