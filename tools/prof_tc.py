"""Tiny driver for ncu captures of the A-streaming passes (one GPU, short):
    ncu --set full --clock-control none --import-source on -k regex:tc_pass_kernel -s 4 -c 2 -o gpurun_out/prof \
        python tools/prof_tc.py --m 32768 --n 32768 --k 32
Launch order: calibration (k=16 probe, 1-2 launches), then `--reps` x (ah, wta[, kl_uht, kl_wtu])."""
import argparse
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pydnmfk_b200 import device as D  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument('--m', type=int, default=32768)
ap.add_argument('--n', type=int, default=32768)
ap.add_argument('--k', type=int, default=32)
ap.add_argument('--reps', type=int, default=3)
ap.add_argument('--kl', action='store_true')
a = ap.parse_args()
ops = D.default_ops()


def copy_peak():
    """STREAM-style copy on this box (what MEASURED_PEAKS.json's hbm_gbs is): read + write bytes / time, best of 5."""
    x = torch.empty(1 << 30, dtype=torch.bfloat16, device='cuda')
    y = torch.empty_like(x)
    best = 1e9
    for _ in range(6):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); y.copy_(x); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return 2 * x.numel() * 2 / best / 1e6


print('copy peak on this box: %.0f GB/s' % copy_peak(), flush=True)
A = torch.rand((a.m, a.n), device='cuda')
H = torch.rand((a.k, a.n), device='cuda')
W = torch.rand((a.m, a.k), device='cuda')
for _ in range(a.reps):
    e = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
    e[0].record(); ops.ah(A, H); e[1].record(); ops.wta(A, W); e[2].record()
    if a.kl:
        ops.kl_uht(A, W, H, 1.2e-7); e[3].record(); ops.kl_wtu(A, W, H, 1.2e-7); e[4].record()
    torch.cuda.synchronize()
    gb = a.m * a.n * 4 / 1e9
    msg = 'ah %.3f ms (%.0f GB/s)  wta %.3f ms (%.0f GB/s)' % (e[0].elapsed_time(e[1]), gb / e[0].elapsed_time(e[1]) * 1e3,
                                                                e[1].elapsed_time(e[2]), gb / e[1].elapsed_time(e[2]) * 1e3)
    if a.kl:
        msg += '  kl_uht %.3f ms  kl_wtu %.3f ms' % (e[2].elapsed_time(e[3]), e[3].elapsed_time(e[4]))
    print(msg, flush=True)
