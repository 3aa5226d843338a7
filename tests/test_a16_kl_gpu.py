"""The fused KL contractions (and BCD's fused A H^T + residual pass) on a data shard stored in 16 bits (fp16 / bf16).

The 16-bit build of tc_kl_kernel widens each element of A to fp32 exactly where the splitters read the tile, and runs
the fp32 kernel from there on (same tiles, split plan and summation order).  So every 16-bit pass must be BIT-IDENTICAL
to the fp32 pass on the widened matrix A16.float() -- a far stronger check than a tolerance, and one that any swizzle,
box or slot-size mistake fails.  Also covered: the deferred (_p) forms, dnmf_ah_residual, the fallback of shards the
tensor path cannot read, and KL-MU / BCD fits end to end.
"""
import numpy as np
import pytest
import torch

from tests import common as T
from tests.test_a16_gpu import FMTS, SCHEDULE_SHAPES, TD, dev, dev16, rnd
from tests.test_tc_gpu import KL_SHAPES

pytestmark = pytest.mark.gpu

EPS = float(np.finfo(np.float32).eps)


@pytest.fixture
def ops():
    from pydnmfk_b200 import _lib as L
    from pydnmfk_b200 import device as D
    L.set_force_generic(False)
    L.set_tc_min_elems(1)
    yield D.default_ops()
    L.set_force_generic(False)
    L.set_tc_min_elems(1 << 20)


def shard_pair(m, n, fmt, seed, zeros=0.2):
    """(A16, A32): an m x n window of a 16-bit shard whose leading dimension is n rounded up to a multiple of 8 (16-byte
    rows, so the tensor path serves any n), and the same window of the widened shard.  Uniform data with exact zeros."""
    g = torch.Generator(device='cuda').manual_seed(seed)
    ld = -(-n // 8) * 8
    A = torch.rand((m, ld), generator=g, device='cuda')
    A[torch.rand((m, ld), generator=g, device='cuda') < zeros] = 0
    big16 = A.to(TD[fmt])
    return big16[:, :n], big16.float()[:, :n]


def factors(m, n, k, seed):
    g = torch.Generator(device='cuda').manual_seed(seed)
    return (torch.rand((m, k), generator=g, device='cuda') + 0.05,
            torch.rand((k, n), generator=g, device='cuda') + 0.05)


def kl_calls(ops, A, W, H):
    """kl_uht, kl_wtu and kl_wtu(transposed_out); each asserted to run on the tcgen05 path"""
    from pydnmfk_b200 import _lib as L
    out = []
    for f in (lambda: ops.kl_uht(A, W, H, EPS), lambda: ops.kl_wtu(A, W, H, EPS),
              lambda: ops.kl_wtu(A, W, H, EPS, transposed_out=True)):
        out.append(f())
        assert L.last_path() == 1, 'tcgen05 KL path not taken for %s' % A.dtype
    return out


@pytest.mark.parametrize('fmt', FMTS)
@pytest.mark.parametrize('m,n,k', KL_SHAPES + SCHEDULE_SHAPES)
def test_bit_identical_to_fp32_kernel(ops, fmt, m, n, k):
    A16, A32 = shard_pair(m, n, fmt, m + n + k)
    W, H = factors(m, n, k, k)
    got, ref = kl_calls(ops, A16, W, H), kl_calls(ops, A32, W, H)
    for name, g, r in zip(('kl_uht', 'kl_wtu', 'kl_wtu^T'), got, ref):
        assert torch.isfinite(r).all()
        assert torch.equal(g, r), '%s %s %dx%dx%d: %d elements differ' % (name, fmt, m, n, k, int((g != r).sum()))


@pytest.mark.parametrize('fmt', FMTS)
@pytest.mark.parametrize('k', [32, 48])
def test_deferred_forms(ops, fmt, k):
    """kl_uht_p / kl_wtu_p serve a 16-bit A with a split-K partial view; the _p updates equal pass + update bit for bit."""
    m, n = 8192, 4096
    A16, _ = shard_pair(m, n, fmt, 5)
    W, H = factors(m, n, k, 6)
    x2, x1 = ops.rowsum(H), ops.colsum(W)
    W1, W2 = W.clone(), W.clone()
    ops.kl_update_w(W1, ops.kl_uht(A16, W, H, EPS), x2, EPS)
    view = ops.kl_uht_p(A16, W, H, EPS)
    assert view is not None and view[2] > 1, 'expected a split-K partial view'
    ops.kl_update_w_p(W2, view, x2, EPS)
    assert torch.equal(W1, W2)
    H1, H2 = H.clone(), H.clone()
    ops.kl_update_h(H1, ops.kl_wtu(A16, W, H, EPS, transposed_out=True), x1, EPS, y_transposed=True)
    view = ops.kl_wtu_p(A16, W, H, EPS)
    assert view is not None and view[2] > 1, 'expected a split-K partial view'
    ops.kl_update_h_p(H2, view, x1, EPS)
    assert torch.equal(H1, H2)


@pytest.mark.parametrize('fmt', FMTS)
@pytest.mark.parametrize('m,n,k', [(2048, 1536, 32), (4096, 1024, 16), (515, 2052, 10), (1000, 1000, 32)])
def test_ah_residual_fused_pass(ops, fmt, m, n, k):
    """dnmf_ah_residual on a 16-bit A: one tcgen05 pass (the 16-bit tc_kl_kernel<3>), V and both norms bit-identical to
    the fp32 call on the widened matrix."""
    from pydnmfk_b200 import _lib as L
    A16, A32 = shard_pair(m, n, fmt, m + k, zeros=0.05)
    W, H = factors(m, n, k, n)
    L.pass_count(True, reset=True)
    L.pass_count(False, reset=True)
    V, res = ops.ah_residual(A16, W, H)
    torch.cuda.synchronize()
    assert L.pass_count(True) == 1 and L.pass_count(False) == 0, 'fused pass did not take the tcgen05 kernel'
    V32, res32 = ops.ah_residual(A32, W, H)
    assert torch.equal(V, V32)
    assert torch.equal(res, res32), (res.cpu().numpy(), res32.cpu().numpy())


@pytest.mark.parametrize('fmt', FMTS)
def test_unreadable_shards_fall_back(ops, fmt):
    """A shard whose rows are not 16-byte multiples (lda % 8 != 0), or whose base is not 16-byte aligned, streams
    through the generic 16-bit kernels, and the deferred forms decline it."""
    from pydnmfk_b200 import _lib as L
    m, n, k = 1024, 1030, 20
    rs = np.random.RandomState(9)
    A = rnd(rs.rand(m, n + 1), fmt)
    A[rs.rand(m, n + 1) < 0.1] = 0
    Wn, Hn = (rs.rand(m, k) + 0.05).astype(np.float32), (rs.rand(k, n) + 0.05).astype(np.float32)
    W, H = dev(Wn), dev(Hn)
    f = np.float64
    big = dev16(A, fmt)
    for A16, A64 in ((big[:, :n].contiguous(), A[:, :n].astype(f)),     # lda = 1030
                     (big[:, 1:], A[:, 1:].astype(f))):                   # base 2 bytes past an aligned one
        assert A16.shape == (m, n)
        U = A64 / (Wn.astype(f) @ Hn.astype(f) + EPS)
        V = ops.kl_uht(A16, W, H, EPS)
        assert L.last_path() == 0
        Y = ops.kl_wtu(A16, W, H, EPS)
        assert L.last_path() == 0
        assert T.rel_fro(V.cpu().numpy(), U @ Hn.astype(f).T) <= 1e-5
        assert T.rel_fro(Y.cpu().numpy(), Wn.astype(f).T @ U) <= 1e-5
        assert ops.kl_uht_p(A16, W, H, EPS) is None and ops.kl_wtu_p(A16, W, H, EPS) is None


# ---- end to end ---------------------------------------------------------------------------------------------------
def fit_pair(fmt, norm, method, k, itr, seed=4, m=1024, n=1024):
    """PyNMF(A, a_storage=fmt).fit() and PyNMF(round_fmt(A)).fit() from the same random init on a 1 x 1 grid, both
    through the per-kernel path (resident_fit=False) with the library's default routing"""
    from pydnmfk_b200 import _lib as L
    from pydnmfk_b200.dist_comm import MPI, MPI_comm
    from pydnmfk_b200.pyDNMF import PyNMF
    from pydnmfk_b200.utils import parse
    L.set_force_generic(False)
    L.set_tc_min_elems(1 << 20)
    A = (np.random.RandomState(seed).rand(m, n) * 8).astype(np.float32)
    out = {}
    for arm, data, storage in (('a16', A, fmt), ('f32', rnd(A, fmt), None)):
        MPI._reset()
        comms = MPI_comm(MPI.COMM_WORLD, 1, 1)
        p = parse()
        p.size, p.rank, p.comm1, p.comm, p.p_r, p.p_c = 1, 0, comms.comm, comms, 1, 1
        p.row_comm, p.col_comm = comms.cart_1d_row(), comms.cart_1d_column()
        p.m, p.n, p.k, p.itr, p.init, p.verbose = m, n, k, itr, 'rand', False
        p.norm, p.method, p.prune, p.W_update = norm, method, False, True
        p.a_storage, p.resident_fit = storage, False
        np.random.seed(seed + 1)
        L.pass_count(True, reset=True)
        L.pass_count(False, reset=True)
        W, H, err = PyNMF(data, params=p).fit()
        out[arm] = dict(W=np.asarray(W), H=np.asarray(H), err=float(err), tc=int(L.pass_count(True)),
                        generic=int(L.pass_count(False)))
    return out['a16'], out['f32']


@pytest.mark.parametrize('fmt', FMTS)
@pytest.mark.parametrize('k', [16, 48])
def test_kl_mu_fit_is_bit_identical(fmt, k):
    a, b = fit_pair(fmt, 'kl', 'mu', k, itr=30)
    assert a['tc'] > 0 and a['generic'] == 0, '%d passes on the generic kernels' % a['generic']
    assert np.array_equal(a['W'], b['W']) and np.array_equal(a['H'], b['H']), \
        'W %.3g H %.3g' % (T.rel_fro(a['W'], b['W']), T.rel_fro(a['H'], b['H']))
    assert abs(a['err'] - b['err']) <= T.TOL_ERR['float32'] * abs(b['err']), (a['err'], b['err'])


@pytest.mark.parametrize('fmt', FMTS)
def test_bcd_fit(fmt):
    """BCD's A H^T + residual pass runs on the 16-bit KL kernel and its W^T A pass on kind::f16 (not bit-exact)."""
    a, b = fit_pair(fmt, 'fro', 'bcd', 16, itr=30)
    assert a['tc'] > 0 and a['generic'] == 0, '%d passes on the generic kernels' % a['generic']
    dW, dH = T.rel_fro(a['W'], b['W']), T.rel_fro(a['H'], b['H'])
    assert dW <= 1e-4 and dH <= 1e-4, (dW, dH)
    assert abs(a['err'] - b['err']) <= 1e-4 * abs(b['err']), (a['err'], b['err'])
