"""Sparse data shards on one GPU: per-pass times, FRO-MU / KL-MU iteration times under CUDA-graph replay, compulsory and
gathered byte rates, and the dense fp32 iteration on the densified 65536^2 matrices, run in the same process in
alternating rounds.  Writes one JSON document (``--out``, default stdout).

    python tools/bench_sparse.py --out profiles/r05_bench_sparse.json

Shapes: 65536^2 at 0.1 / 1 / 5 % density with a uniform pattern, and a 1M x 128K matrix whose row and column degrees
follow a Zipf law (P(index i) ~ 1 / (i + 1)), about 1e8 non-zeros before duplicates are summed.  Ranks k = 32 and 64.
Times come from CUDA events over ``--reps`` launches after ``--warmup`` launches of the same shape.
Compulsory bytes of a pass: the walked compressed matrix once (pointers, indices, values), the factors it reads and the
output it writes; gathered bytes: nnz * k * sizeof(T), the factor rows the non-zeros fetch (mostly from L2).
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
sys.path.insert(0, ROOT)

from pydnmfk_b200 import device as D                    # noqa: E402
from pydnmfk_b200.sparse import SparseShard             # noqa: E402


def gpu_context():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[:1])


def uniform_shard(n, density, seed):
    g = torch.Generator(device='cuda').manual_seed(seed)
    nnz = int(n * n * density)
    ij = torch.randint(0, n, (2, nnz), device='cuda', generator=g)
    v = torch.rand(nnz, device='cuda', generator=g) + 0.01
    S = SparseShard.from_any(torch.sparse_coo_tensor(ij, v, (n, n)).coalesce().to_sparse_csr())
    return S


def zipf_shard(m, n, nnz, seed):
    g = torch.Generator(device='cuda').manual_seed(seed)
    # inverse CDF of the log-uniform law: P(i) ~ 1 / (i + 1) on [0, size)
    r = (torch.exp(torch.rand(nnz, device='cuda', generator=g, dtype=torch.float64) * np.log(m + 1)) - 1).long().clamp_(0, m - 1)
    c = (torch.exp(torch.rand(nnz, device='cuda', generator=g, dtype=torch.float64) * np.log(n + 1)) - 1).long().clamp_(0, n - 1)
    v = torch.rand(nnz, device='cuda', generator=g) + 0.01
    return SparseShard.from_any(torch.sparse_coo_tensor(torch.stack([r, c]), v, (m, n)).coalesce().to_sparse_csr())


def time_ms(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def pass_times(ops, S, k, reps, warmup):
    m, n = S.shape
    g = torch.Generator(device='cuda').manual_seed(1)
    W = torch.rand((m, k), device='cuda', generator=g)
    H = torch.rand((k, n), device='cuda', generator=g)
    eps = float(np.finfo(np.float32).eps)
    es, nnz = 4, S.nnz
    walk_rows = 8 * (m + 1) + nnz * (4 + es)
    walk_cols = 8 * (n + 1) + nnz * (4 + es)
    passes = {
        'ah': (lambda: ops.ah(S, H), walk_rows + n * k * es + m * k * es),
        'wta': (lambda: ops.wta(S, W, transposed_out=True), walk_cols + m * k * es + n * k * es),
        'kl_uht': (lambda: ops.kl_uht(S, W, H, eps), walk_rows + (n + 2 * m) * k * es),
        'kl_wtu': (lambda: ops.kl_wtu(S, W, H, eps, transposed_out=True), walk_cols + (m + 2 * n) * k * es),
        'ah_residual': (lambda: ops.ah_residual(S, W, H), walk_rows + (n + 2 * m) * k * es),
    }
    out = {}
    for name, (fn, comp) in passes.items():
        ms = time_ms(fn, reps, warmup)
        gath = nnz * k * es
        out[name] = dict(ms=round(ms, 4), compulsory_GB=round(comp / 1e9, 4), compulsory_GBps=round(comp / ms / 1e6, 1),
                         gathered_GB=round(gath / 1e9, 4), gathered_GBps=round(gath / ms / 1e6, 1))
    return out


class Iteration:
    """One FRO-MU or KL-MU step of the 1 x 1 grid on A (sparse shard or dense tensor), captured as a CUDA graph."""

    def __init__(self, A, k, norm):
        from pydnmfk_b200.dist_comm import MPI, MPI_comm
        from pydnmfk_b200.dist_nmf import nmf_algorithms_1D
        from pydnmfk_b200.graphs import StepGraphs
        from pydnmfk_b200.utils import parse
        MPI._reset()
        comm = MPI.COMM_WORLD
        MPI_comm(comm, 1, 1)
        m, n = A.shape
        g = torch.Generator(device='cuda').manual_seed(2)
        W = torch.rand((m, k), device='cuda', generator=g)
        H = torch.rand((k, n), device='cuda', generator=g)
        p = parse()
        p.m, p.n, p.p_r, p.p_c, p.k, p.comm1, p.norm, p.method = m, n, 1, 1, k, comm, norm, 'mu'
        p.eps, p.W_update, p.itr = np.finfo(np.float32).eps, True, 1000
        self.alg = nmf_algorithms_1D(A, W, H, params=p)
        self.alg.update()                          # eager first step: workspace sized, attributes set
        torch.cuda.synchronize()
        self.sg = StepGraphs(self.alg.update, lambda: None)
        self.sg.plain()

    def __call__(self):
        self.sg.plain()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--rounds', type=int, default=2, help='alternating sparse / dense rounds of the iteration timing')
    ap.add_argument('--quick', action='store_true', help='small shapes only (a rehearsal of the script)')
    a = ap.parse_args()
    assert torch.cuda.is_available(), 'bench_sparse needs a GPU'
    torch.cuda.set_device(0)
    ops = D.default_ops()
    doc = dict(context=gpu_context(), reps=a.reps, warmup=a.warmup, rounds=a.rounds, dtype='float32', results=[])
    n = 4096 if a.quick else 65536
    shapes = [('uniform', n, n, d) for d in (0.001, 0.01, 0.05)]
    shapes.append(('zipf', 1 << 14 if a.quick else 1 << 20, 1 << 11 if a.quick else 1 << 17, 10 ** 6 if a.quick else 10 ** 8))
    for kind, m, nc, param in shapes:
        t0 = time.time()
        S = uniform_shard(m, param, 7) if kind == 'uniform' else zipf_shard(m, nc, param, 7)
        torch.cuda.synchronize()
        rc, cc = S.nnz_counts()
        shape_doc = dict(kind=kind, m=m, n=nc, nnz=S.nnz, density=S.nnz / (m * nc), shard_GB=round(S.nbytes() / 1e9, 3),
                         max_row_share=float(rc.max().item()) / max(S.nnz, 1),
                         max_col_share=float(cc.max().item()) / max(S.nnz, 1), build_s=round(time.time() - t0, 1))
        dense = S.to_dense() if kind == 'uniform' and param == 0.01 else None
        for k in (32, 64):
            entry = dict(shape_doc, k=k, passes=pass_times(ops, S, k, a.reps, a.warmup), iteration_ms={})
            for norm in ('fro', 'kl'):
                arms = {'sparse': Iteration(S, k, norm)}
                if dense is not None:
                    arms['dense_fp32'] = Iteration(dense, k, norm)
                times = {name: [] for name in arms}
                for _ in range(a.rounds):
                    for name, it in arms.items():
                        times[name].append(time_ms(it, a.reps, a.warmup))
                entry['iteration_ms'][norm] = {name: dict(min=round(min(v), 4), all=[round(x, 4) for x in v])
                                               for name, v in times.items()}
                del arms
            doc['results'].append(entry)
            print(json.dumps(entry), flush=True)
        del S, dense
        torch.cuda.empty_cache()
    text = json.dumps(doc, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(text + '\n')
    else:
        print(text)


if __name__ == '__main__':
    main()
