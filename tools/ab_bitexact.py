"""Two builds of libdnmf.so must give BIT-IDENTICAL results when they differ only in scheduling (loop structure, ring
depths, wait flavour): run the four A-streaming contractions of both on a list of shapes (ragged edges, odd tile counts,
one x-block with a deep split-K, k = 10 / 16 / 32 / 48 / 64) and compare the outputs bit for bit (one GPU, one process).

    cp <other build>/libdnmf.so pydnmfk_b200/libdnmf_other.so
    python tools/ab_bitexact.py other           # libdnmf.so against libdnmf_other.so

Exit code 0 = identical everywhere and every call took the tcgen05 path in both libraries."""
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = [(2048, 1536), (4096, 1024), (1000, 2052), (8192, 8192), (128, 40000), (40000, 128), (2048, 1184), (1184, 2048),
          (3333, 4444), (16384, 4096)]
KS = [10, 16, 32, 48, 64]


def main():
    import numpy as np
    import torch
    from pydnmfk_b200 import _lib as L
    variant = sys.argv[1]
    libs = {}
    for v, path in (('default', L.LIB_PATH), (variant, os.path.join(ROOT, 'pydnmfk_b200', 'libdnmf_%s.so' % variant))):
        lib = C.CDLL(path)
        for name, (res, args) in L.SIGNATURES.items():
            if hasattr(lib, name):
                fn = getattr(lib, name)
                fn.restype, fn.argtypes = res, args
        lib.dnmf_set_tc_min_elems(1)
        libs[v] = lib
    st = torch.cuda.current_stream().cuda_stream
    eps = float(np.finfo(np.float32).eps)
    bad, n_cmp = [], 0
    g = torch.Generator(device='cuda').manual_seed(7)
    for (m, n) in SHAPES:
        A = torch.rand((m, n), device='cuda', generator=g)
        for k in KS:
            W = torch.rand((m, k), device='cuda', generator=g)
            H = torch.rand((k, n), device='cuda', generator=g)
            res = {}
            for v, lib in libs.items():
                nb = max(lib.dnmf_workspace_bytes(op, m, n, k, 0) for op in range(4))
                ws = torch.empty(nb, dtype=torch.uint8, device='cuda')
                o = {'ah': torch.zeros((m, k), device='cuda'), 'kl_uht': torch.zeros((m, k), device='cuda'),
                     'wta': torch.zeros((k, n), device='cuda'), 'kl_wtu': torch.zeros((k, n), device='cuda')}
                before = int(lib.dnmf_pass_count(1, 0))
                rcs = [lib.dnmf_ah(A.data_ptr(), n, H.data_ptr(), n, o['ah'].data_ptr(), k, m, n, k, 0, 0, ws.data_ptr(), nb, st),
                       lib.dnmf_wta(A.data_ptr(), n, W.data_ptr(), k, o['wta'].data_ptr(), n, m, n, k, 0, 0, 0, ws.data_ptr(), nb, st),
                       lib.dnmf_kl_uht(A.data_ptr(), n, W.data_ptr(), k, H.data_ptr(), n, o['kl_uht'].data_ptr(), k, m, n, k, eps,
                                       0, 0, ws.data_ptr(), nb, st),
                       lib.dnmf_kl_wtu(A.data_ptr(), n, W.data_ptr(), k, H.data_ptr(), n, o['kl_wtu'].data_ptr(), n, m, n, k, eps,
                                       0, 0, 0, ws.data_ptr(), nb, st)]
                torch.cuda.synchronize()
                assert all(rc == 0 for rc in rcs), (v, m, n, k, rcs)
                res[v] = (o, int(lib.dnmf_pass_count(1, 0)) - before)
            (o0, p0), (o1, p1) = res['default'], res[variant]
            for nm in o0:
                n_cmp += 1
                if not torch.equal(o0[nm], o1[nm]) or not bool(torch.isfinite(o0[nm]).all()):
                    bad.append((m, n, k, nm, float((o0[nm] - o1[nm]).abs().max())))
            if p0 != 4 or p1 != 4:
                bad.append((m, n, k, 'tcgen05 passes', p0, p1))
        del A
    print(json.dumps({'variant': variant, 'comparisons': n_cmp, 'mismatches': bad[:20], 'n_bad': len(bad)}), flush=True)
    sys.exit(1 if bad else 0)


if __name__ == '__main__':
    main()
