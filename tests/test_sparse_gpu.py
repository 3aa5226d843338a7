"""Sparse data shards on the device: the six sparse passes against float64 numpy, residual accuracy near convergence,
parity of sparse fits with the unmodified reference's goldens, and a fit at a size users run.

Kernel tolerances are those of tests/test_kernels_gpu.py (2e-5 relative Frobenius in fp32, 1e-12 in fp64); small-integer
data and factors must match exactly, which pins the indexing and the chunk boundaries (512 non-zeros per chunk)."""
import numpy as np
import pytest

from tests import common as T
from tests import mp_util, sparse_workers

pytestmark = pytest.mark.gpu

TOL = {np.float32: 2e-5, np.float64: 1e-12}
KS = (1, 3, 4, 16, 31, 32, 33, 64)


def _sparse(m, n, density, rs, dt, integer=False, empty=True):
    import scipy.sparse as sp
    A = sp.random(m, n, density=density, format='csr', random_state=rs, dtype=np.float64)
    if integer:
        A.data = np.ceil(A.data * 3)
    A = A.toarray()
    if empty and m > 4 and n > 4:
        A[rs.permutation(m)[:max(1, m // 10)], :] = 0           # empty rows and columns
        A[:, rs.permutation(n)[:max(1, n // 10)]] = 0
    return A.astype(dt)


def _skewed(m, n, rs, dt):
    """Row 7 and column 11 each hold >= 30 % of the non-zeros."""
    A = _sparse(m, n, 4000.0 / (m * n), rs, np.float64, empty=False)
    A[7, :] = rs.rand(n) + 0.1
    A[:, 11] = rs.rand(m) + 0.1
    nnz = np.count_nonzero(A)
    assert np.count_nonzero(A[7]) >= 0.3 * nnz and np.count_nonzero(A[:, 11]) >= 0.3 * nnz
    return A.astype(dt)


SHAPES = [('1xn', lambda rs, dt: _sparse(1, 3000, 0.5, rs, dt, empty=False)),
          ('mx1', lambda rs, dt: _sparse(3000, 1, 0.5, rs, dt, empty=False)),
          ('ragged', lambda rs, dt: _sparse(517, 389, 0.08, rs, dt)),
          ('wide', lambda rs, dt: _sparse(300, 4100, 0.05, rs, dt)),
          ('skewed', lambda rs, dt: _skewed(6000, 5000, rs, dt))]


def _passes(ops, S, W, H, eps):
    """The six sparse passes (outputs as host float64-comparable arrays)."""
    out = {}
    out['ah'] = ops.ah(S, H)
    out['wta'] = ops.wta(S, W)
    out['wta_t'] = ops.wta(S, W, transposed_out=True)
    out['kl_uht'] = ops.kl_uht(S, W, H, eps)
    out['kl_wtu'] = ops.kl_wtu(S, W, H, eps)
    out['kl_wtu_t'] = ops.kl_wtu(S, W, H, eps, transposed_out=True)
    out['res'] = ops.residual_sqnorm(S, W, H)
    V, r = ops.ah_residual(S, W, H)
    out['ahr_v'], out['ahr'] = V, r
    return {k: v.cpu().numpy() for k, v in out.items()}


def _expected(A, W, H, eps):
    A64, W64, H64 = (x.astype(np.float64) for x in (A, W, H))
    WH = W64 @ H64
    U = np.where(A64 != 0, A64 / (WH + eps), 0.0)
    res = np.array([((A64 - WH) ** 2).sum(), (A64 ** 2).sum()])
    return dict(ah=A64 @ H64.T, wta=W64.T @ A64, wta_t=(W64.T @ A64).T, kl_uht=U @ H64.T, kl_wtu=W64.T @ U,
                kl_wtu_t=(W64.T @ U).T, res=res, ahr_v=A64 @ H64.T, ahr=res)


@pytest.mark.parametrize('dt', [np.float32, np.float64], ids=['fp32', 'fp64'])
@pytest.mark.parametrize('k', KS)
def test_sparse_passes_match_numpy(k, dt):
    import torch
    from pydnmfk_b200 import device as D
    from pydnmfk_b200.sparse import SparseShard
    import scipy.sparse as sp
    ops = D.default_ops()
    eps = float(np.finfo(dt).eps)
    for name, make in SHAPES:
        rs = np.random.RandomState(k * 7 + len(name))
        A = make(rs, dt)
        m, n = A.shape
        W, H = rs.rand(m, k).astype(dt), rs.rand(k, n).astype(dt)
        S = SparseShard.from_any(sp.csr_matrix(A))
        assert S.nnz == np.count_nonzero(A)
        got = _passes(ops, S, torch.from_numpy(W).cuda(), torch.from_numpy(H).cuda(), eps)
        want = _expected(A, W, H, eps)
        for key, g in got.items():
            assert g.shape == want[key].shape, (name, key)
            tol = TOL[dt] if key not in ('res', 'ahr') else 1e-12
            assert T.rel_fro(g, want[key]) <= tol, (name, key, T.rel_fro(g, want[key]))
        again = _passes(ops, S, torch.from_numpy(W).cuda(), torch.from_numpy(H).cuda(), eps)
        for key in got:
            assert np.array_equal(got[key], again[key]), ('not bit-identical on a second call', name, key)


@pytest.mark.parametrize('dt', [np.float32, np.float64], ids=['fp32', 'fp64'])
@pytest.mark.parametrize('k', KS)
def test_sparse_passes_exact_on_small_integers(k, dt):
    """Small-integer data and factors: every product and partial sum is exact, so A H^T, W^T A and the residual must
    equal numpy bit for bit -- a wrong index, a lost or doubled chunk partial would show."""
    import torch
    from pydnmfk_b200 import device as D
    from pydnmfk_b200.sparse import SparseShard
    import scipy.sparse as sp
    ops = D.default_ops()
    for name, make in SHAPES[:4] + [('skewed_int', None)]:
        rs = np.random.RandomState(100 + k)
        if make is None:
            A = np.ceil(_skewed(6000, 5000, rs, np.float64) * 2).astype(dt)
        else:
            A = np.ceil(make(rs, np.float64) * 3).astype(dt)
        m, n = A.shape
        W, H = rs.randint(0, 3, (m, k)).astype(dt), rs.randint(0, 3, (k, n)).astype(dt)
        S = SparseShard.from_any(sp.csr_matrix(A))
        Wd, Hd = torch.from_numpy(W).cuda(), torch.from_numpy(H).cuda()
        A64, W64, H64 = (x.astype(np.float64) for x in (A, W, H))
        assert np.array_equal(ops.ah(S, Hd).cpu().numpy(), A64 @ H64.T), name
        assert np.array_equal(ops.wta(S, Wd).cpu().numpy(), W64.T @ A64), name
        assert np.array_equal(ops.wta(S, Wd, transposed_out=True).cpu().numpy(), (W64.T @ A64).T), name
        res = ops.residual_sqnorm(S, Wd, Hd).cpu().numpy()
        assert res[0] == ((A64 - W64 @ H64) ** 2).sum() and res[1] == (A64 ** 2).sum(), name


def test_sparse_residual_accurate_near_convergence():
    """||A - W H||^2 ~ 1e-6 ||A||^2 from factors near an exact masked low-rank matrix (block-sparse W0 H0): the
    sparse residual forms s in float64 and <W^T W, H H^T> from float64 Grams, so the difference of the two large terms
    keeps the small residual to 1e-6 relative."""
    import torch
    from pydnmfk_b200 import device as D
    from pydnmfk_b200.sparse import SparseShard
    import scipy.sparse as sp
    ops = D.default_ops()
    rs = np.random.RandomState(11)
    m, n, k = 3000, 2200, 12
    W0 = np.zeros((m, k))
    W0[np.arange(m), rs.randint(0, k, m)] = rs.rand(m) + 0.5
    H0 = np.zeros((k, n))
    H0[rs.randint(0, k, n), np.arange(n)] = rs.rand(n) + 0.5
    A = W0 @ H0
    W = (W0 * (1 + 1e-3 * rs.randn(m, k))).astype(np.float32)
    H = (H0 * (1 + 1e-3 * rs.randn(k, n))).astype(np.float32)
    A = A.astype(np.float32)
    A64, W64, H64 = A.astype(np.float64), W.astype(np.float64), H.astype(np.float64)
    ref = ((A64 - W64 @ H64) ** 2).sum()
    a2 = (A64 ** 2).sum()
    assert 1e-8 < ref / a2 < 1e-5
    S = SparseShard.from_any(sp.csr_matrix(A))
    got = ops.residual_sqnorm(S, torch.from_numpy(W).cuda(), torch.from_numpy(H).cuda()).cpu().numpy()
    assert abs(got[0] - ref) <= 1e-6 * ref and abs(got[1] - a2) <= 1e-12 * a2
    _, got2 = ops.ah_residual(S, torch.from_numpy(W).cuda(), torch.from_numpy(H).cuda())
    assert np.allclose(got2.cpu().numpy(), got, rtol=1e-12, atol=0)


# ---- parity with the unmodified reference's goldens ---------------------------------------------------------------
def _parity_sets():
    from tests.test_parity_gpu import SINGLE, MULTI_PICK
    return SINGLE, MULTI_PICK


SINGLE, MULTI_PICK = _parity_sets()


@pytest.mark.parametrize('case', SINGLE, ids=[c['name'] for c in SINGLE])
def test_sparse_single_rank_matches_reference(case):
    from tests.test_parity_gpu import _compare
    from pydnmfk_b200.dist_comm import MPI
    MPI._reset()
    _compare(case, [sparse_workers.sparse_fit_worker(0, 1, case)])


_multi_cache = {}


@pytest.mark.parametrize('case', MULTI_PICK, ids=[c['name'] for c in MULTI_PICK])
def test_sparse_multi_rank_matches_reference(case):
    from tests.test_parity_gpu import _compare
    world = case['grid'][0] * case['grid'][1]
    if world not in _multi_cache:
        batch = [c for c in MULTI_PICK if c['grid'][0] * c['grid'][1] == world]
        _multi_cache[world] = mp_util.run(world, sparse_workers.sparse_fit_many_worker, (batch,), backend='gloo',
                                          timeout=1800)
    res = []
    for r in range(world):
        if case['name'] not in _multi_cache[world][r]:
            pytest.fail('case did not run (an earlier case of this batch failed on rank %d)' % r)
        tag, val = _multi_cache[world][r][case['name']]
        if tag == 'err':
            pytest.fail('rank %d raised:\n%s' % (r, val))
        res.append(val)
    _compare(case, res)


@pytest.mark.parametrize('name', ['u64x48k4_1x1_fro_mu_i10_32', 'u64x48k4_1x1_kl_mu_i10_64', 'zeros40x36k3_1x1_kl_mu_prune',
                                  'u2048k32_1x1_fro_mu_i100', 'u2048k32_1x1_kl_mu_i100'])
def test_torch_cuda_csr_input_matches_scipy_input(name):
    """A CUDA torch CSR shard fits bit-identically to the same shard given as scipy.sparse, and comes back as tensors."""
    from oracle import cases as C
    from pydnmfk_b200.dist_comm import MPI
    case = C.CASES_BY_NAME[name]
    MPI._reset()
    a = sparse_workers.sparse_fit_worker(0, 1, case, 'scipy')
    MPI._reset()
    b = sparse_workers.sparse_fit_worker(0, 1, case, 'torch')
    assert a['out_type'] == 'ndarray' and b['out_type'] == 'Tensor'
    assert np.array_equal(a['W'], b['W']) and np.array_equal(a['H'], b['H']) and a['err'] == b['err']


# ---- a size users run --------------------------------------------------------------------------------------------
def _big_fit(A, norm, itr, graph, seed=3):
    from pydnmfk_b200.dist_comm import MPI, MPI_comm
    from pydnmfk_b200.pyDNMF import PyNMF
    from pydnmfk_b200.utils import parse
    MPI._reset()
    comm = MPI.COMM_WORLD
    comms = MPI_comm(comm, 1, 1)
    p = parse()
    p.comm1, p.comm, p.row_comm, p.col_comm = comm, comms, comms.cart_1d_row(), comms.cart_1d_column()
    p.p_r, p.p_c, p.k, p.itr, p.init, p.verbose = 1, 1, 32, itr, 'rand', False
    p.norm, p.method, p.prune, p.cuda_graph = norm, 'mu', False, graph
    np.random.seed(seed)
    W, H, err = PyNMF(A, params=p).fit()
    return W.cpu().numpy(), H.cpu().numpy(), float(err)


def test_sparse_fit_at_user_size_matches_dense_fit():
    """65536^2 at 0.5 % density, k = 32, 20 iterations of FRO-MU and KL-MU: within 1e-4 of the dense fp32 fit of the
    densified matrix, bit-identical between two sparse fits and between graph replay on and off."""
    import torch
    from pydnmfk_b200.sparse import SparseShard
    n, nnz = 65536, int(65536 * 65536 * 0.005)
    g = torch.Generator(device='cuda').manual_seed(5)
    ij = torch.randint(0, n, (2, nnz), device='cuda', generator=g)
    v = torch.rand(nnz, device='cuda', generator=g) + 0.01
    coo = torch.sparse_coo_tensor(ij, v, (n, n)).coalesce()
    S = SparseShard.from_any(coo.to_sparse_csr())
    del coo, ij, v
    for norm in ('fro', 'kl'):
        W1, H1, e1 = _big_fit(S, norm, 20, True)
        W2, H2, e2 = _big_fit(S, norm, 20, True)
        W3, H3, e3 = _big_fit(S, norm, 20, False)
        assert np.array_equal(W1, W2) and np.array_equal(H1, H2) and e1 == e2, norm
        assert np.array_equal(W1, W3) and np.array_equal(H1, H3) and e1 == e3, norm
        dense = S.to_dense()
        Wd, Hd, ed = _big_fit(dense, norm, 20, True)
        del dense
        torch.cuda.empty_cache()
        assert T.rel_fro(W1, Wd) <= 1e-4 and T.rel_fro(H1, Hd) <= 1e-4, (norm, T.rel_fro(W1, Wd), T.rel_fro(H1, Hd))
        assert abs(e1 - ed) <= 1e-5 * ed, (norm, e1, ed)
