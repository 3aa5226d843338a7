"""The tcgen05 / TMA / TMEM path of the A-streaming contractions (fp32, k <= 64; kernels for 16 / 32 / 64, zero-padded).

Checked three ways: bit-exact on small-integer data (every product and partial sum is exact in tf32/fp32, so
any descriptor / swizzle / layout mistake shows up as a hard mismatch), against float64 numpy on random data
(the 3-term tf32 split must deliver fp32-level accuracy), and against the generic CUDA-core kernels.
"""
import json
import os

import numpy as np
import pytest
import torch

from tests import common as T

pytestmark = pytest.mark.gpu

SHAPES = [(128, 32, 16), (128, 64, 32), (256, 96, 64), (1000, 1000, 32), (515, 2052, 32), (2048, 2048, 32),
          (4100, 300, 64), (3000, 5000, 16), (1024, 8192, 32), (8192, 1024, 32), (129, 4100, 64),
          # factor widths between the instantiated 16 / 32 / 64 ride along zero-padded
          (1000, 1000, 4), (2048, 2048, 10), (515, 2052, 20), (4100, 300, 48), (3000, 5000, 1), (640, 640, 33)]


@pytest.fixture(scope='module')
def ops():
    from pydnmfk_b200 import _lib as L
    from pydnmfk_b200 import device as D
    L.set_force_generic(False)
    L.set_tc_min_elems(1)
    yield D.default_ops()
    L.set_tc_min_elems(1 << 20)


def _dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _diag(tag, got, ref):
    bad = np.argwhere(got != ref)
    rec = dict(tag=tag, shape=list(got.shape), n_bad=int(bad.shape[0]),
               first_bad=[[int(i), int(j), float(got[i, j]), float(ref[i, j])] for i, j in bad[:12]])
    d = os.environ.get('DNMF_TEST_LOG_DIR')          # kept as a JSON line in $DNMF_TEST_LOG_DIR/tc_diag.jsonl if set
    if d:
        os.makedirs(d, exist_ok=True)
        with open(os.path.join(d, 'tc_diag.jsonl'), 'a') as f:
            f.write(json.dumps(rec) + '\n')
    return rec


def test_tensor_path_is_taken(ops):
    from pydnmfk_b200 import _lib as L
    A = torch.rand((1024, 1024), device='cuda')
    H = torch.rand((32, 1024), device='cuda')
    ops.ah(A, H)
    torch.cuda.synchronize()
    assert L.last_path() == 1, 'tcgen05 path not active (calibration failed or device is not sm_100)'
    ops.wta(A, torch.rand((1024, 32), device='cuda'))
    torch.cuda.synchronize()
    assert L.last_path() == 1


@pytest.mark.parametrize('m,n,k', SHAPES)
def test_exact_on_integer_data(ops, m, n, k):
    rs = np.random.RandomState(m + n + k)
    A = rs.randint(0, 8, size=(m, n)).astype(np.float32)
    H = rs.randint(0, 4, size=(k, n)).astype(np.float32)
    W = rs.randint(0, 4, size=(m, k)).astype(np.float32)
    V = ops.ah(_dev(A), _dev(H)).cpu().numpy()
    Vr = (A.astype(np.int64) @ H.astype(np.int64).T).astype(np.float32)
    assert np.array_equal(V, Vr), _diag('ah %dx%dx%d' % (m, n, k), V, Vr)
    Y = ops.wta(_dev(A), _dev(W)).cpu().numpy()
    Yr = (W.astype(np.int64).T @ A.astype(np.int64)).astype(np.float32)
    assert np.array_equal(Y, Yr), _diag('wta %dx%dx%d' % (m, n, k), Y, Yr)
    Yt = ops.wta(_dev(A), _dev(W), transposed_out=True).cpu().numpy()
    assert np.array_equal(Yt, Yr.T)


@pytest.mark.parametrize('m,n,k', SHAPES)
def test_fp32_accuracy_of_the_split(ops, m, n, k):
    from pydnmfk_b200 import _lib as L
    rs = np.random.RandomState(7)
    A, H, W = rs.rand(m, n).astype(np.float32), rs.rand(k, n).astype(np.float32), rs.rand(m, k).astype(np.float32)
    f = np.float64
    V = ops.ah(_dev(A), _dev(H)).cpu().numpy()
    assert L.last_path() == 1
    Y = ops.wta(_dev(A), _dev(W)).cpu().numpy()
    eV, eY = T.rel_fro(V, A.astype(f) @ H.astype(f).T), T.rel_fro(Y, W.astype(f).T @ A.astype(f))
    L.set_force_generic(True)
    Vg = ops.ah(_dev(A), _dev(H)).cpu().numpy()
    Yg = ops.wta(_dev(A), _dev(W)).cpu().numpy()
    L.set_force_generic(False)
    gV, gY = T.rel_fro(Vg, A.astype(f) @ H.astype(f).T), T.rel_fro(Yg, W.astype(f).T @ A.astype(f))
    _diag('acc %dx%dx%d tc(V %.2e Y %.2e) generic(V %.2e Y %.2e)' % (m, n, k, eV, eY, gV, gY), V[:1, :1], V[:1, :1])
    # fp32-accurate: within a small factor of the plain-fp32 kernels, far below single-pass tf32 (~3e-4)
    assert eV <= 2e-6 and eY <= 2e-6, (eV, eY, gV, gY)


def test_strided_window_and_wide_values(ops):
    """lda > n (TMA global stride), values spanning many binades."""
    rs = np.random.RandomState(11)
    big = (rs.rand(700, 1200) * 2.0 ** rs.randint(-8, 8, size=(700, 1200))).astype(np.float32)
    Ad = torch.from_numpy(big).cuda()[100:612, 64:1088]        # 512 x 1024 window, ld = 1200, 16-byte aligned
    A = big[100:612, 64:1088]
    H, W = rs.rand(32, 1024).astype(np.float32), rs.rand(512, 32).astype(np.float32)
    f = np.float64
    assert T.rel_fro(ops.ah(Ad, _dev(H)).cpu().numpy(), A.astype(f) @ H.astype(f).T) <= 2e-6
    assert T.rel_fro(ops.wta(Ad, _dev(W)).cpu().numpy(), W.astype(f).T @ A.astype(f)) <= 2e-6


def test_deterministic(ops):
    A, H = torch.rand((4096, 4096), device='cuda'), torch.rand((32, 4096), device='cuda')
    W = torch.rand((4096, 32), device='cuda')
    assert torch.equal(ops.ah(A, H), ops.ah(A, H)) and torch.equal(ops.wta(A, W), ops.wta(A, W))


KL_SHAPES = [(128, 32, 32), (256, 96, 32), (1000, 1000, 32), (515, 2052, 32), (2048, 2048, 32), (4100, 300, 32),
             (1024, 8192, 32), (8192, 1024, 32),
             # k < 32 rides along zero-padded
             (1000, 1000, 4), (2048, 2048, 10), (515, 2052, 20), (4100, 300, 1), (1024, 8192, 31),
             # 32 < k <= 64: the 64-wide build of the kernel (dnmf_tc_kl64.cu)
             (128, 64, 64), (256, 96, 64), (1000, 1000, 64), (515, 2052, 48), (2048, 2048, 64), (4100, 300, 33),
             (1024, 8192, 64), (8192, 1024, 40)]


@pytest.mark.parametrize('m,n,k', KL_SHAPES)
def test_kl_tensor_path(ops, m, n, k):
    """Fused KL contractions on the tcgen05 path (k <= 64; kernels built for 32 and 64 factor columns): S = W H recomputed on the tensor cores, U = A / (S + eps)
    in the splitter warps, second MMA; compared with float64 numpy and with the generic fused kernels."""
    from pydnmfk_b200 import _lib as L
    rs = np.random.RandomState(3)
    A = rs.rand(m, n).astype(np.float32)
    A[rs.rand(m, n) < 0.2] = 0                       # exact zeros must stay exact zeros in U
    H, W = (rs.rand(k, n) + 0.05).astype(np.float32), (rs.rand(m, k) + 0.05).astype(np.float32)
    eps = float(np.finfo(np.float32).eps)
    f = np.float64
    U = A.astype(f) / (W.astype(f) @ H.astype(f) + eps)
    V = ops.kl_uht(_dev(A), _dev(W), _dev(H), eps).cpu().numpy()
    assert L.last_path() == 1, 'tcgen05 KL path not taken'
    Y = ops.kl_wtu(_dev(A), _dev(W), _dev(H), eps).cpu().numpy()
    Yt = ops.kl_wtu(_dev(A), _dev(W), _dev(H), eps, transposed_out=True).cpu().numpy()
    eV, eY = T.rel_fro(V, U @ H.astype(f).T), T.rel_fro(Y, W.astype(f).T @ U)
    L.set_force_generic(True)
    Vg = ops.kl_uht(_dev(A), _dev(W), _dev(H), eps).cpu().numpy()
    Yg = ops.kl_wtu(_dev(A), _dev(W), _dev(H), eps).cpu().numpy()
    L.set_force_generic(False)
    gV, gY = T.rel_fro(Vg, U @ H.astype(f).T), T.rel_fro(Yg, W.astype(f).T @ U)
    _diag('kl %dx%dx%d tc(V %.2e Y %.2e) generic(V %.2e Y %.2e)' % (m, n, k, eV, eY, gV, gY), V[:1, :1], V[:1, :1])
    assert np.isfinite(V).all() and np.isfinite(Y).all()
    assert eV <= 3e-6 and eY <= 3e-6, (eV, eY, gV, gY)
    assert np.array_equal(Yt, Y.T)


def test_kl_deterministic(ops):
    A, H = torch.rand((4096, 4096), device='cuda'), torch.rand((32, 4096), device='cuda') + 0.1
    W = torch.rand((4096, 32), device='cuda') + 0.1
    assert torch.equal(ops.kl_uht(A, W, H, 1e-7), ops.kl_uht(A, W, H, 1e-7))
    assert torch.equal(ops.kl_wtu(A, W, H, 1e-7), ops.kl_wtu(A, W, H, 1e-7))


@pytest.mark.parametrize('m,n,k', [(2048, 1536, 32), (4096, 1024, 16), (515, 2052, 10), (1000, 1000, 32)])
def test_ah_residual_fused_pass(ops, m, n, k):
    """dnmf_ah_residual: V = A H^T together with ||A - W H||^2 and ||A||^2 in one tcgen05 pass (tc_kl_kernel<3>), against
    float64 numpy and against the two separate passes."""
    from pydnmfk_b200 import _lib as L
    rs = np.random.RandomState(m + n + k)
    A, W, H = rs.rand(m, n).astype(np.float32), rs.rand(m, k).astype(np.float32), rs.rand(k, n).astype(np.float32)
    L.pass_count(True, reset=True)
    L.pass_count(False, reset=True)
    V, res = ops.ah_residual(_dev(A), _dev(W), _dev(H))
    torch.cuda.synchronize()
    assert L.pass_count(True) == 1 and L.pass_count(False) == 0, 'fused pass did not take the tcgen05 kernel'
    f = np.float64
    Vr = A.astype(f) @ H.astype(f).T
    rr = np.linalg.norm(A.astype(f) - W.astype(f) @ H.astype(f)) ** 2
    ar = np.linalg.norm(A.astype(f)) ** 2
    assert T.rel_fro(V.cpu().numpy(), Vr) < 2e-6
    got = res.cpu().numpy()
    assert abs(got[0] - rr) <= 2e-6 * rr and abs(got[1] - ar) <= 1e-6 * ar, (got, rr, ar)
    sep = ops.residual_sqnorm(_dev(A), _dev(W), _dev(H)).cpu().numpy()
    assert abs(got[0] - sep[0]) <= 2e-6 * rr and abs(got[1] - sep[1]) <= 1e-6 * ar


def test_residual_on_the_tensor_pipeline(ops):
    """tc_kl_kernel<2> (dnmf_set_tc_residual(1)) against the CUDA-core residual kernel and float64 numpy."""
    from pydnmfk_b200 import _lib as L
    rs = np.random.RandomState(5)
    m, n, k = 2048, 2048, 32
    A, W, H = rs.rand(m, n).astype(np.float32), rs.rand(m, k).astype(np.float32), rs.rand(k, n).astype(np.float32)
    ref = ops.residual_sqnorm(_dev(A), _dev(W), _dev(H)).cpu().numpy()
    L.call('dnmf_set_tc_residual', 1)
    try:
        got = ops.residual_sqnorm(_dev(A), _dev(W), _dev(H)).cpu().numpy()
    finally:
        L.call('dnmf_set_tc_residual', 0)
    f = np.float64
    rr = np.linalg.norm(A.astype(f) - W.astype(f) @ H.astype(f)) ** 2
    assert abs(got[0] - rr) <= 2e-6 * rr and abs(got[0] - ref[0]) <= 2e-6 * rr and abs(got[1] - ref[1]) <= 1e-6 * ref[1]


@pytest.mark.parametrize('m,n,k', [(2048, 2048, 32), (1000, 1000, 32), (515, 2052, 20), (4100, 300, 64), (8192, 1024, 10),
                                   (1024, 8192, 32)])
def test_fused_epilogue_is_bit_identical(ops, m, n, k):
    """dnmf_*_p + dnmf_*_update_*_p (the update sums the pass's split partials itself) must give exactly the factors of
    pass -> reduce_partials -> update, for the FRO and (k <= 32) KL half-steps."""
    rs = np.random.RandomState(7)
    A, W, H = (_dev(rs.rand(*s).astype(np.float32)) for s in ((m, n), (m, k), (k, n)))
    eps = 1.1920929e-07
    G_h = ops.gram(H, trans=True)
    G_w = ops.gram(W, trans=False)
    # FRO W
    W1 = W.clone(); ops.mu_update_w(W1, ops.ah(A, H), G_h, eps)
    view = ops.ah_p(A, H); assert view is not None and view[2] >= 1
    W2 = W.clone(); ops.mu_update_w_p(W2, view, G_h, eps)
    assert torch.equal(W1, W2)
    # FRO H
    H1 = H.clone(); ops.mu_update_h(H1, ops.wta(A, W, transposed_out=True), G_w, eps, y_transposed=True)
    view = ops.wta_p(A, W); assert view is not None
    H2 = H.clone(); ops.mu_update_h_p(H2, view, G_w, eps)
    assert torch.equal(H1, H2)
    H3 = H.clone(); ops.mu_update_h(H3, ops.wta(A, W), G_w, eps)          # and the non-transposed plain form
    assert torch.equal(H1, H3)
    x2, x1 = ops.rowsum(H), ops.colsum(W)
    W1 = W.clone(); ops.kl_update_w(W1, ops.kl_uht(A, W, H, eps), x2, eps)
    view = ops.kl_uht_p(A, W, H, eps); assert view is not None
    W2 = W.clone(); ops.kl_update_w_p(W2, view, x2, eps)
    assert torch.equal(W1, W2)
    H1 = H.clone(); ops.kl_update_h(H1, ops.kl_wtu(A, W, H, eps, transposed_out=True), x1, eps, y_transposed=True)
    view = ops.kl_wtu_p(A, W, H, eps); assert view is not None
    H2 = H.clone(); ops.kl_update_h_p(H2, view, x1, eps)
    assert torch.equal(H1, H2)


def test_fused_epilogue_falls_back(ops):
    """fp64 and forced-generic calls are not served by the _p passes."""
    from pydnmfk_b200 import _lib as L
    A = torch.rand((512, 512), device='cuda', dtype=torch.float64)
    H = torch.rand((8, 512), device='cuda', dtype=torch.float64)
    assert ops.ah_p(A, H) is None
    L.set_force_generic(True)
    try:
        assert ops.ah_p(A.float(), H.float()) is None
    finally:
        L.set_force_generic(False)
