"""A/B timing of the A-streaming tcgen05 kernels of two or more builds of the library (one GPU, ONE process):

    python tools/kl_lab.py --variants default,parent [--m 65536 --n 65536 --k 32] [--rounds 6]

Every variant is a library file loaded side by side with ctypes: "default" = pydnmfk_b200/libdnmf.so, any other name =
pydnmfk_b200/libdnmf_<name>.so (for example the build of another commit, copied there).  The (variant, op) combinations
are timed in a reshuffled order for `--rounds` rounds, each paired with a reference launch issued right before it (see
below); the report is the median ratio to the reference plus the median and minimum time per combination.  Every
variant is also checked against float64 numpy on a 2048 x 1536 shard."""
import argparse
import ctypes as C
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--variants', default='default')
    ap.add_argument('--ops', default='ah,wta,kl_uht,kl_wtu')
    ap.add_argument('--m', type=int, default=65536)
    ap.add_argument('--n', type=int, default=65536)
    ap.add_argument('--k', type=int, default=32)
    ap.add_argument('--rounds', type=int, default=6)
    ap.add_argument('--sustained', type=int, default=0, help='also time blocks of N back-to-back (op, op, ...) sequences per variant: the power-capped steady state of the product loop')
    a = ap.parse_args()
    import numpy as np
    import torch
    from pydnmfk_b200 import _lib as L
    k = a.k
    eps = float(np.finfo(np.float32).eps)
    libs = {}
    for v in a.variants.split(','):
        path = L.LIB_PATH if v == 'default' else os.path.join(ROOT, 'pydnmfk_b200', 'libdnmf_%s.so' % v)
        lib = C.CDLL(path)
        for name, (res, args) in L.SIGNATURES.items():
            if hasattr(lib, name):
                fn = getattr(lib, name)
                fn.restype, fn.argtypes = res, args
        libs[v] = lib
    st = torch.cuda.current_stream().cuda_stream

    def run(lib, op, A, W, H, out, ws, wsb):
        m, n = A.shape
        if op == 'ah':
            rc = lib.dnmf_ah(A.data_ptr(), n, H.data_ptr(), n, out.data_ptr(), k, m, n, k, 0, 0, ws.data_ptr(), wsb, st)
        elif op == 'wta':
            rc = lib.dnmf_wta(A.data_ptr(), n, W.data_ptr(), k, out.data_ptr(), n, m, n, k, 0, 0, 0, ws.data_ptr(), wsb, st)
        elif op == 'kl_uht':
            rc = lib.dnmf_kl_uht(A.data_ptr(), n, W.data_ptr(), k, H.data_ptr(), n, out.data_ptr(), k, m, n, k, eps, 0, 0,
                                 ws.data_ptr(), wsb, st)
        else:
            rc = lib.dnmf_kl_wtu(A.data_ptr(), n, W.data_ptr(), k, H.data_ptr(), n, out.data_ptr(), n, m, n, k, eps, 0, 0, 0,
                                 ws.data_ptr(), wsb, st)
        assert rc == 0, (op, rc, lib.dnmf_last_error())

    def outs(m, n):
        return {'ah': torch.empty((m, k), device='cuda'), 'kl_uht': torch.empty((m, k), device='cuda'),
                'wta': torch.empty((k, n), device='cuda'), 'kl_wtu': torch.empty((k, n), device='cuda')}

    def workspace(lib, m, n):
        nb = max(lib.dnmf_workspace_bytes(op, m, n, k, 0) for op in range(4))
        return torch.empty(nb, dtype=torch.uint8, device='cuda'), nb

    # accuracy of every variant on a small shard
    rs = np.random.RandomState(1)
    m0, n0 = 2048, 1536
    A0, W0, H0 = rs.rand(m0, n0).astype(np.float32), rs.rand(m0, k).astype(np.float32), rs.rand(k, n0).astype(np.float32)
    f = np.float64
    U = A0.astype(f) / (W0.astype(f) @ H0.astype(f) + eps)
    ref = {'kl_uht': U @ H0.astype(f).T, 'kl_wtu': W0.astype(f).T @ U, 'ah': A0.astype(f) @ H0.astype(f).T,
           'wta': W0.astype(f).T @ A0.astype(f)}
    dA, dW, dH = (torch.from_numpy(x).cuda() for x in (A0, W0, H0))
    names = a.ops.split(',')
    for v, lib in libs.items():
        lib.dnmf_set_tc_min_elems(1)
        o = outs(m0, n0)
        ws, wsb = workspace(lib, m0, n0)
        for nm in names:
            run(lib, nm, dA, dW, dH, o[nm], ws, wsb)
        torch.cuda.synchronize()
        acc = {nm: float(np.linalg.norm(o[nm].cpu().numpy() - ref[nm]) / np.linalg.norm(ref[nm])) for nm in names}
        print(json.dumps({'variant': v, 'accuracy_vs_fp64': acc, 'tc_passes': int(lib.dnmf_pass_count(1, 0)) if hasattr(lib, 'dnmf_pass_count') else None}), flush=True)
    del dA, dW, dH
    A = torch.rand((a.m, a.n), device='cuda')
    H = torch.rand((k, a.n), device='cuda')
    W = torch.rand((a.m, k), device='cuda')
    o = outs(a.m, a.n)
    gb = a.m * a.n * 4 / 1e9
    wss = {v: workspace(lib, a.m, a.n) for v, lib in libs.items()}
    first = a.variants.split(',')[0]
    combos = [(v, nm) for v in libs for nm in names]
    # Every measurement is PAIRED with a reference launch (the first variant's FRO pass `ah`) issued right
    # before it on the same stream with no host synchronisation in between: the whole round is one back-to-back queue
    # (sustained clocks, like the product's loop), the order of the combinations is reshuffled every round, and the
    # report is the median of the per-pair ratio t / t_ref next to the absolute times -- box drift cancels in the ratio.
    import random
    rng = random.Random(1)
    times = {c: [] for c in combos}
    ratios = {c: [] for c in combos}
    ref_times = []
    for rnd in range(a.rounds + 1):
        order = combos[:]
        rng.shuffle(order)
        evs = []
        for (v, nm) in order:
            lib = libs[v]
            e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            e0.record()
            run(libs[first], 'ah', A, W, H, o['ah'], *wss[first])
            e1.record()
            run(lib, nm, A, W, H, o[nm], *wss[v])
            e2.record()
            evs.append(((v, nm), e0, e1, e2))
        torch.cuda.synchronize()
        if rnd > 0:                          # round 0 = warm-up (attributes, calibration)
            for c, e0, e1, e2 in evs:
                tr, t = e0.elapsed_time(e1), e1.elapsed_time(e2)
                ref_times.append(tr)
                times[c].append(t)
                ratios[c].append(t / tr)
    print(json.dumps({'reference': first + ':ah', 'median_ms': statistics.median(ref_times), 'min_ms': min(ref_times),
                      'max_ms': max(ref_times)}), flush=True)
    for v in libs:
        rec = {'variant': v}
        for nm in names:
            t = times[(v, nm)]
            rec[nm] = {'median_ms': statistics.median(t), 'min_ms': min(t), 'ratio_to_ref_median': statistics.median(ratios[(v, nm)]),
                       'GBps_median': gb / statistics.median(t) * 1e3}
        print(json.dumps(rec), flush=True)

    if a.sustained:
        # Sustained blocks: `--sustained` back-to-back repetitions of the op list per variant with no host sync (what a
        # CUDA-graph replayed fit does to the power budget), variants in a reshuffled order every round.
        blocks = {v: [] for v in libs}
        for rnd in range(a.rounds + 1):
            order = list(libs)
            rng.shuffle(order)
            for v in order:
                lib = libs[v]
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(a.sustained):
                    for nm in names:
                        run(lib, nm, A, W, H, o[nm], *wss[v])
                e1.record()
                torch.cuda.synchronize()
                if rnd > 0:
                    blocks[v].append(e0.elapsed_time(e1) / (a.sustained * len(names)))
        for v in libs:
            print(json.dumps({'variant': v, 'sustained_ms_per_pass_median': statistics.median(blocks[v]),
                              'min': min(blocks[v]), 'max': max(blocks[v]), 'ops': names, 'reps': a.sustained}), flush=True)


if __name__ == '__main__':
    main()
