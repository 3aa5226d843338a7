"""Two builds of libdnmf.so must give BIT-IDENTICAL results when they differ only in scheduling (loop structure, ring
depths, wait flavour) or in host code: run the A-streaming contractions of both on a list of shapes (ragged edges, odd
tile counts, one x-block with a deep split-K, k = 10 / 16 / 32 / 48 / 64) and compare the outputs bit for bit (one GPU,
one process).  Covered per shape and k:
  - dnmf_ah / dnmf_wta / dnmf_kl_uht / dnmf_kl_wtu on an fp32 A, the WTA forms with transposed_out = 0 and 1;
  - dnmf_ah / dnmf_wta on a 16-bit A (DNMF_A_F16, DNMF_A_BF16; lda padded to a multiple of 8);
  - the _p forms, each followed by its _p update, compared on the updated factor;
  - dnmf_ah_residual: V and both norms;
and for every call the return code, the kernels it launched (dnmf_launch_count) and the tcgen05 passes it issued.

    cp <other build>/libdnmf.so pydnmfk_b200/libdnmf_other.so
    python tools/ab_bitexact.py other           # libdnmf.so against libdnmf_other.so

Exit code 0 = identical everywhere, and every call issued its passes on the tcgen05 path in both libraries."""
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = [(2048, 1536), (4096, 1024), (1000, 2052), (8192, 8192), (128, 40000), (40000, 128), (2048, 1184), (1184, 2048),
          (3333, 4444), (16384, 4096)]
KS = [10, 16, 32, 48, 64]
F32, A_F16, A_BF16 = 0, 3, 4
OP_AH_RESIDUAL = 8


def run_calls(lib, A, A16, W, H, G, xk, m, n, k, ws, nb, st):
    """Every call of one library on one shape: name -> (return code, launches, tcgen05 passes, output tensors)."""
    import numpy as np
    import torch
    eps = float(np.finfo(np.float32).eps)
    p = lambda t: t.data_ptr()
    res = {}

    def call(name, fn, outs):
        l0, t0 = int(lib.dnmf_launch_count(0)), int(lib.dnmf_pass_count(1, 0))
        rc = fn()
        torch.cuda.synchronize()
        res[name] = (rc, int(lib.dnmf_launch_count(0)) - l0, int(lib.dnmf_pass_count(1, 0)) - t0, outs)

    z = lambda *s: torch.zeros(s, device='cuda')
    wsp = p(ws)
    # plain forms on an fp32 A
    V, Y0, Y1 = z(m, k), z(k, n), z(n, k)
    call('ah', lambda: lib.dnmf_ah(p(A), n, p(H), n, p(V), k, m, n, k, F32, 0, wsp, nb, st), [V])
    call('wta', lambda: lib.dnmf_wta(p(A), n, p(W), k, p(Y0), n, m, n, k, 0, F32, 0, wsp, nb, st), [Y0])
    call('wta_t', lambda: lib.dnmf_wta(p(A), n, p(W), k, p(Y1), k, m, n, k, 1, F32, 0, wsp, nb, st), [Y1])
    V, Y0, Y1 = z(m, k), z(k, n), z(n, k)
    call('kl_uht', lambda: lib.dnmf_kl_uht(p(A), n, p(W), k, p(H), n, p(V), k, m, n, k, eps, F32, 0, wsp, nb, st), [V])
    call('kl_wtu', lambda: lib.dnmf_kl_wtu(p(A), n, p(W), k, p(H), n, p(Y0), n, m, n, k, eps, 0, F32, 0, wsp, nb, st), [Y0])
    call('kl_wtu_t', lambda: lib.dnmf_kl_wtu(p(A), n, p(W), k, p(H), n, p(Y1), k, m, n, k, eps, 1, F32, 0, wsp, nb, st),
         [Y1])
    # plain forms on a 16-bit A
    for dt, (A2, lda2) in A16.items():
        V, Y0, Y1 = z(m, k), z(k, n), z(n, k)
        call('ah/%d' % dt, lambda: lib.dnmf_ah(p(A2), lda2, p(H), n, p(V), k, m, n, k, dt, 0, wsp, nb, st), [V])
        call('wta/%d' % dt, lambda: lib.dnmf_wta(p(A2), lda2, p(W), k, p(Y0), n, m, n, k, 0, dt, 0, wsp, nb, st), [Y0])
        call('wta_t/%d' % dt, lambda: lib.dnmf_wta(p(A2), lda2, p(W), k, p(Y1), k, m, n, k, 1, dt, 0, wsp, nb, st), [Y1])
    # _p forms, each followed by the update that sums the splits itself
    v4 = (C.c_int64 * 4)()
    vp = C.addressof(v4)
    for dt, (A2, lda2) in [(F32, (A, n))] + list(A16.items()):
        W1, H1 = W.clone(), H.clone()
        call('ah_p/%d' % dt, lambda: lib.dnmf_ah_p(p(A2), lda2, p(H), n, m, n, k, dt, 0, wsp, nb, vp, st)
             or lib.dnmf_mu_update_w_p(p(W1), k, vp, p(G), m, k, eps, F32, st), [W1])
        call('wta_p/%d' % dt, lambda: lib.dnmf_wta_p(p(A2), lda2, p(W), k, m, n, k, dt, 0, wsp, nb, vp, st)
             or lib.dnmf_mu_update_h_p(p(H1), n, vp, p(G), k, n, eps, 0, F32, st), [H1])
    W1, H1 = W.clone(), H.clone()
    call('kl_uht_p', lambda: lib.dnmf_kl_uht_p(p(A), n, p(W), k, p(H), n, m, n, k, eps, F32, 0, wsp, nb, vp, st)
         or lib.dnmf_kl_update_w_p(p(W1), k, vp, p(xk), m, k, eps, F32, st), [W1])
    call('kl_wtu_p', lambda: lib.dnmf_kl_wtu_p(p(A), n, p(W), k, p(H), n, m, n, k, eps, F32, 0, wsp, nb, vp, st)
         or lib.dnmf_kl_update_h_p(p(H1), n, vp, p(xk), k, n, eps, 0, F32, st), [H1])
    # A H^T with the residual and ||A||^2 in the same pass (the fused pass for k <= 32)
    V, nrm = z(m, k), torch.zeros(2, dtype=torch.float64, device='cuda')
    call('ah_residual', lambda: lib.dnmf_ah_residual(p(A), n, p(W), k, p(H), n, p(V), k, m, n, k, p(nrm), F32, wsp, nb,
                                                     st), [V, nrm])
    return res


def main():
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
    bad, n_cmp, n_calls = [], 0, 0
    g = torch.Generator(device='cuda').manual_seed(7)
    for (m, n) in SHAPES:
        A = torch.rand((m, n), device='cuda', generator=g)
        lda16 = (n + 7) // 8 * 8          # 16-byte rows: what the kind::f16 kernels need
        A16 = {}
        for dt, ty in ((A_F16, torch.float16), (A_BF16, torch.bfloat16)):
            A2 = torch.zeros((m, lda16), dtype=ty, device='cuda')
            A2[:, :n] = A.to(ty)
            A16[dt] = (A2, lda16)
        for k in KS:
            W = torch.rand((m, k), device='cuda', generator=g)
            H = torch.rand((k, n), device='cuda', generator=g)
            G = H @ H.T
            xk = torch.rand(k, device='cuda', generator=g) + 0.5
            res = {}
            for v, lib in libs.items():
                nb = max(lib.dnmf_workspace_bytes(op, m, n, k, dt)
                         for op in (0, 1, 2, 3, OP_AH_RESIDUAL) for dt in (F32, A_F16, A_BF16))
                ws = torch.empty(nb, dtype=torch.uint8, device='cuda')
                res[v] = run_calls(lib, A, A16, W, H, G, xk, m, n, k, ws, nb, st)
                del ws
            r0, r1 = res['default'], res[variant]
            for nm in r0:
                n_calls += 1
                (rc0, l0, t0, o0), (rc1, l1, t1, o1) = r0[nm], r1[nm]
                if rc0 != 0 or rc1 != 0:
                    bad.append((m, n, k, nm, 'return code', rc0, rc1))
                    continue
                if (l0, t0) != (l1, t1):
                    bad.append((m, n, k, nm, 'launches / tcgen05 passes', l0, l1, t0, t1))
                if t0 == 0:
                    bad.append((m, n, k, nm, 'no tcgen05 pass'))
                for a, b in zip(o0, o1):
                    n_cmp += 1
                    if not torch.equal(a, b) or not bool(torch.isfinite(a).all()):
                        bad.append((m, n, k, nm, float((a.double() - b.double()).abs().max())))
        del A, A16
    print(json.dumps({'variant': variant, 'calls': n_calls, 'comparisons': n_cmp, 'mismatches': bad[:20],
                      'n_bad': len(bad)}), flush=True)
    sys.exit(1 if bad else 0)


if __name__ == '__main__':
    main()
