"""16-bit storage of the data shard (params.a_storage; DNMF_A_F16 / DNMF_A_BF16) on the GPU.

- tcgen05 kind::f16 contractions (dnmf_tc16.cu): bit-exact on small-integer data (any descriptor, swizzle or layout
  mistake is a hard mismatch), fp32-accurate on random data against float64 products of the rounded matrix, on the
  multi-unit, multi-split schedule that production shapes run, deterministic, and the deferred-reduction (_p) forms
  equal to the plain ones bit for bit;
- the generic CUDA-core kernels on a 16-bit A against float64 references of the rounded matrix;
- end to end: PyNMF(A, a_storage=s).fit() equals the float32 fit of round_s(A) on 1x1, 2x1 and 2x2 grids.
"""
import numpy as np
import pytest
import torch

from tests import common as T
from tests import mp_util

pytestmark = pytest.mark.gpu

FMTS = ['float16', 'bfloat16']
TD = {'float16': torch.float16, 'bfloat16': torch.bfloat16}

# the shape list of the fp32 tcgen05 tests (ragged edges, k between the 16 / 32 / 64 builds), plus shapes whose plan has
# more units than SMs and more than one K split
SHAPES = [(128, 32, 16), (128, 64, 32), (256, 96, 64), (1000, 1000, 32), (515, 2052, 32), (2048, 2048, 32),
          (4100, 300, 64), (3000, 5000, 16), (1024, 8192, 32), (8192, 1024, 32), (129, 4100, 64),
          (1000, 1000, 4), (2048, 2048, 10), (515, 2052, 20), (4100, 300, 48), (3000, 5000, 1), (640, 640, 33)]
SCHEDULE_SHAPES = [(4096, 24576, 32), (12288, 12288, 48)]


def rnd(A, fmt):
    """round_s: nearest-even rounding of float32 data into the storage format, back as float32 (numpy)."""
    if fmt == 'float16':
        return np.asarray(A, np.float32).astype(np.float16).astype(np.float32)
    return torch.from_numpy(np.ascontiguousarray(A, np.float32)).to(torch.bfloat16).to(torch.float32).numpy()


def dev16(A, fmt):
    return torch.from_numpy(np.ascontiguousarray(A, np.float32)).cuda().to(TD[fmt])


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def tc_path(lda):
    """the kind::f16 kernel serves 16-byte rows (lda % 8 == 0); other shards stream through the generic kernels"""
    return 1 if lda % 8 == 0 else 0


@pytest.fixture
def ops():
    from pydnmfk_b200 import _lib as L
    from pydnmfk_b200 import device as D
    L.set_force_generic(False)
    L.set_tc_min_elems(1)
    yield D.default_ops()
    L.set_force_generic(False)
    L.set_tc_min_elems(1 << 20)


@pytest.mark.parametrize('fmt', FMTS)
@pytest.mark.parametrize('m,n,k', SHAPES + SCHEDULE_SHAPES)
def test_exact_on_integer_data(ops, fmt, m, n, k):
    from pydnmfk_b200 import _lib as L
    rs = np.random.RandomState(m + n + k)
    A = rs.randint(0, 4, size=(m, n)).astype(np.float32)       # every sum < 2^24: exact in fp32 in any order
    H = rs.randint(0, 4, size=(k, n)).astype(np.float32)
    W = rs.randint(0, 4, size=(m, k)).astype(np.float32)
    Ad = dev16(A, fmt)
    f = np.float64
    V = ops.ah(Ad, dev(H))
    assert L.last_path() == tc_path(n), 'kind::f16 path taken iff lda % 8 == 0'
    Vr = (A.astype(f) @ H.astype(f).T).astype(np.float32)
    assert V.dtype == torch.float32 and np.array_equal(V.cpu().numpy(), Vr), 'ah %s %dx%dx%d' % (fmt, m, n, k)
    Yr = (W.astype(f).T @ A.astype(f)).astype(np.float32)
    Y = ops.wta(Ad, dev(W))
    assert L.last_path() == tc_path(n)
    assert np.array_equal(Y.cpu().numpy(), Yr), 'wta %s %dx%dx%d' % (fmt, m, n, k)
    Yt = ops.wta(Ad, dev(W), transposed_out=True)
    assert np.array_equal(Yt.cpu().numpy(), Yr.T), 'wta^T %s %dx%dx%d' % (fmt, m, n, k)


@pytest.mark.parametrize('fmt', FMTS)
def test_schedule_shapes_are_multi_unit_and_split(ops, fmt):
    """Both passes of the SCHEDULE_SHAPES run more (128-wide, K-split) units than the device has SMs, with more than
    one K split (read from the partial view the library returns): every CTA loops over several units and the split
    partials are summed afterwards."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    for m, n, k in SCHEDULE_SHAPES:
        Ad = torch.zeros((m, n), dtype=TD[fmt], device='cuda')
        H, W = torch.zeros((k, n), device='cuda'), torch.zeros((m, k), device='cuda')
        for x_len, view in ((m, ops.ah_p(Ad, H)), (n, ops.wta_p(Ad, W))):
            assert view is not None, 'kind::f16 path not taken'
            splits = int(view[2])
            assert splits > 1 and -(-x_len // 128) * splits > sms, (m, n, x_len, splits)


def _wide_h(rs, k, n):
    """factor rows spanning many binades, entries down to 1e-7 (the clamp eps is 1.2e-7); row 0 is a dying component,
    every entry in [1e-7, 1e-6]: without the per-row fp16 scale it would fall into fp16's subnormal range"""
    H = np.exp(rs.uniform(np.log(1e-7), np.log(30.0), size=(k, n))).astype(np.float32)
    H[:, ::7] = 1e-7
    H[0] = np.exp(rs.uniform(np.log(1e-7), np.log(1e-6), size=n)).astype(np.float32)
    return H


@pytest.mark.parametrize('fmt', FMTS)
@pytest.mark.parametrize('m,n,k', SHAPES + SCHEDULE_SHAPES[:1])
def test_fp32_accuracy(ops, fmt, m, n, k):
    from pydnmfk_b200 import _lib as L
    rs = np.random.RandomState(7)
    A = rnd(rs.rand(m, n) * 4, fmt)
    H, W = _wide_h(rs, k, n), _wide_h(rs, k, m).T.copy()
    Ad = dev16(A, fmt)
    f = np.float64
    V = ops.ah(Ad, dev(H)).cpu().numpy()
    assert L.last_path() == tc_path(n)
    Y = ops.wta(Ad, dev(W)).cpu().numpy()
    Vr, Yr = A.astype(f) @ H.astype(f).T, W.astype(f).T @ A.astype(f)
    eV, eY = T.rel_fro(V, Vr), T.rel_fro(Y, Yr)
    assert eV <= 2e-6 and eY <= 2e-6, (fmt, eV, eY)
    # the dying component on its own (its share of the Frobenius norm is ~1e-7)
    e0V, e0Y = T.rel_fro(V[:, 0], Vr[:, 0]), T.rel_fro(Y[0], Yr[0])
    assert e0V <= 2e-6 and e0Y <= 2e-6, (fmt, e0V, e0Y)


@pytest.mark.parametrize('fmt', FMTS)
def test_strided_window(ops, fmt):
    """lda > n: a 512 x 1024 window of a 700 x 1208 shard (the TMA global stride)."""
    from pydnmfk_b200 import _lib as L
    rs = np.random.RandomState(11)
    big = rnd(rs.rand(700, 1208) * 2.0 ** rs.randint(-8, 8, size=(700, 1208)), fmt)
    Ad = dev16(big, fmt)[100:612, 64:1088]
    A = big[100:612, 64:1088].astype(np.float64)
    H, W = _wide_h(rs, 32, 1024), rs.rand(512, 32).astype(np.float32)
    V = ops.ah(Ad, dev(H)).cpu().numpy()
    assert L.last_path() == 1
    assert T.rel_fro(V, A @ H.astype(np.float64).T) <= 2e-6
    Y = ops.wta(Ad, dev(W)).cpu().numpy()
    assert L.last_path() == 1
    assert T.rel_fro(Y, W.astype(np.float64).T @ A) <= 2e-6


@pytest.mark.parametrize('fmt', FMTS)
def test_deterministic_and_deferred_forms(ops, fmt):
    """Repeated calls are bit-identical; the _p passes + fused-epilogue updates equal pass + update bit for bit."""
    rs = np.random.RandomState(5)
    m, n, k = 8192, 4096, 32
    Ad = dev16(rs.rand(m, n), fmt)
    H, W = dev(rs.rand(k, n).astype(np.float32) + 0.1), dev(rs.rand(m, k).astype(np.float32) + 0.1)
    assert torch.equal(ops.ah(Ad, H), ops.ah(Ad, H))
    assert torch.equal(ops.wta(Ad, W, transposed_out=True), ops.wta(Ad, W, transposed_out=True))
    eps = float(np.finfo(np.float32).eps)
    HHT, WTW = ops.gram(H, trans=True), ops.gram(W, trans=False)
    W1, W2 = W.clone(), W.clone()
    ops.mu_update_w(W1, ops.ah(Ad, H), HHT, eps)
    view = ops.ah_p(Ad, H)
    assert view is not None and view[2] > 1, 'expected a split-K partial view'
    ops.mu_update_w_p(W2, view, HHT, eps)
    assert torch.equal(W1, W2)
    H1, H2 = H.clone(), H.clone()
    ops.mu_update_h(H1, ops.wta(Ad, W, transposed_out=True), WTW, eps, y_transposed=True)
    view = ops.wta_p(Ad, W)
    assert view is not None
    ops.mu_update_h_p(H2, view, WTW, eps)
    assert torch.equal(H1, H2)


# ---- generic CUDA-core kernels on a 16-bit A ------------------------------------------------------------------------
GEN_SHAPES = [(300, 517, 5), (1000, 1000, 32), (257, 1030, 64), (64, 64, 1)]


@pytest.fixture
def generic():
    from pydnmfk_b200 import _lib as L
    L.set_force_generic(True)
    yield
    L.set_force_generic(False)


@pytest.mark.parametrize('fmt', FMTS)
@pytest.mark.parametrize('m,n,k', GEN_SHAPES)
def test_generic_kernels(ops, generic, fmt, m, n, k):
    from pydnmfk_b200 import _lib as L
    rs = np.random.RandomState(m * k + 1)
    A = rnd(rs.rand(m, n), fmt)
    A[rs.rand(m, n) < 0.1] = 0
    A[3] = 0
    A[:, 5] = 0
    H, W = (rs.rand(k, n) + 0.05).astype(np.float32), (rs.rand(m, k) + 0.05).astype(np.float32)
    Ad = dev16(A, fmt)
    f = np.float64
    A64, H64, W64 = A.astype(f), H.astype(f), W.astype(f)
    assert T.rel_fro(ops.ah(Ad, dev(H)).cpu().numpy(), A64 @ H64.T) <= 1e-6
    assert L.last_path() == 0
    assert T.rel_fro(ops.wta(Ad, dev(W)).cpu().numpy(), W64.T @ A64) <= 1e-6
    assert T.rel_fro(ops.wta(Ad, dev(W), transposed_out=True).cpu().numpy(), (W64.T @ A64).T) <= 1e-6
    eps = float(np.finfo(np.float32).eps)
    U = A64 / (W64 @ H64 + eps)
    assert T.rel_fro(ops.kl_uht(Ad, dev(W), dev(H), eps).cpu().numpy(), U @ H64.T) <= 1e-5
    assert T.rel_fro(ops.kl_wtu(Ad, dev(W), dev(H), eps).cpu().numpy(), W64.T @ U) <= 1e-5
    R = A64 - W64 @ H64
    res = ops.residual_sqnorm(Ad, dev(W), dev(H)).cpu().numpy()
    assert abs(res[0] - (R * R).sum()) <= 1e-5 * (R * R).sum() and abs(res[1] - (A64 * A64).sum()) <= 1e-9 * (A64 * A64).sum()
    num, den = (t.cpu().numpy() for t in ops.column_err(Ad, dev(W), dev(H)))
    assert np.allclose(num, (R * R).sum(0), rtol=1e-5) and np.allclose(den, (A64 * A64).sum(0), rtol=1e-9, atol=0)
    assert abs(float(ops.sqnorm(Ad).item()) - (A64 * A64).sum()) <= 1e-9 * (A64 * A64).sum()
    rows, cols = ops.nnz_counts(Ad)
    assert np.array_equal(rows.cpu().numpy(), (A != 0).sum(1)) and np.array_equal(cols.cpu().numpy(), (A != 0).sum(0))
    ri = torch.from_numpy(np.flatnonzero((A != 0).sum(1))).cuda()
    ci = torch.from_numpy(np.flatnonzero((A != 0).sum(0))).cuda()
    C = ops.compact(Ad, ri, ci)
    assert C.dtype == TD[fmt] and torch.equal(C, Ad[ri][:, ci])


def test_underflow_counts_as_zero(ops):
    """An entry that rounds to 0 in float16 is a zero for pruning."""
    A = np.ones((64, 64), np.float32)
    A[:, 7] = 1e-9
    rows, cols = ops.nnz_counts(dev16(A, 'float16'))
    assert int(cols[7]) == 0 and int(rows[0]) == 63
    rows, cols = ops.nnz_counts(dev16(A, 'bfloat16'))
    assert int(cols[7]) == 64


# ---- end to end ---------------------------------------------------------------------------------------------------
def _data(spec):
    rs = np.random.RandomState(spec['seed'])
    m, n = spec['m'], spec['n']
    A = (rs.rand(m, n) * 8).astype(np.float32)
    if spec.get('prune'):
        A[[1, 17, m - 2]] = 0
        A[:, [0, 9, n - 1]] = 0
    return A


def pair_worker(rank, world, spec):
    """PyNMF(A, a_storage=s).fit() and PyNMF(round_s(A)).fit() on this rank's shard, from the same random init."""
    from pydnmfk_b200 import _lib as L
    from pydnmfk_b200.dist_comm import MPI, MPI_comm
    from pydnmfk_b200.utils import parse, determine_block_params
    from pydnmfk_b200.pyDNMF import PyNMF
    torch.cuda.set_device(0)
    L.set_force_generic(False)
    L.set_tc_min_elems(1 << 20)                           # the library's default routing, whatever ran before
    p_r, p_c = spec['grid']
    A = _data(spec)
    blk = determine_block_params(rank, (p_r, p_c), A.shape).determine_block_index_range_asymm()
    A_ij = np.ascontiguousarray(A[blk[0][0]:blk[1][0] + 1, blk[0][1]:blk[1][1] + 1])
    out = {}
    for arm, data, storage in (('a16', A_ij, spec['fmt']), ('f32', rnd(A_ij, spec['fmt']), None)):
        comms = MPI_comm(MPI.COMM_WORLD, p_r, p_c)          # (a 2-D fit frees its communicators at the end)
        args = parse()
        args.size, args.rank, args.comm1, args.comm, args.p_r, args.p_c = world, rank, comms.comm, comms, p_r, p_c
        args.row_comm, args.col_comm = comms.cart_1d_row(), comms.cart_1d_column()
        args.m, args.n, args.k = spec['m'], spec['n'], spec['k']
        args.itr, args.init, args.verbose = spec['itr'], 'rand', False
        args.norm, args.method, args.prune, args.W_update = spec['norm'], spec['method'], spec.get('prune', False), True
        args.a_storage = storage
        np.random.seed(spec['seed'] + 1)
        L.pass_count(True, reset=True)
        L.pass_count(False, reset=True)
        W, H, err = PyNMF(data, params=args).fit()
        out[arm] = dict(W=np.asarray(W), H=np.asarray(H), err=float(err), err_dtype=str(np.asarray(err).dtype),
                        tc=int(L.pass_count(True)), generic=int(L.pass_count(False)))
    return out


def _check(spec, res):
    tf, te = T.TOL_FACTOR['float32'], T.TOL_ERR['float32']
    if spec['method'] == 'bcd':
        tf, te = 1e-4, 1e-4                                   # as test_parity_gpu._tol for fp32 BCD
    for r, o in enumerate(res):
        a, b = o['a16'], o['f32']
        assert a['W'].dtype == b['W'].dtype and a['H'].dtype == b['H'].dtype
        assert a['W'].dtype == (np.float64 if spec.get('prune') else np.float32)
        assert a['err_dtype'] == 'float32'
        dW, dH = T.rel_fro(a['W'], b['W']), T.rel_fro(a['H'], b['H'])
        assert dW <= tf and dH <= tf, '%s rank %d: W %.3g H %.3g' % (spec, r, dW, dH)
        assert abs(a['err'] - b['err']) <= te * abs(b['err']), '%s rank %d: err %.9g vs %.9g' % (spec, r, a['err'], b['err'])
        if spec.get('expect_tc'):
            assert a['tc'] > 0 and a['generic'] == 0, '%s: %d passes on the generic kernels' % (spec, a['generic'])


ALGS = [('fro', 'mu', 100), ('kl', 'mu', 100), ('fro', 'hals', 50), ('fro', 'bcd', 50)]
E2E = []
for _fmt in FMTS:
    for _norm, _method, _itr in ALGS:
        E2E.append(dict(fmt=_fmt, norm=_norm, method=_method, itr=_itr, grid=(1, 1), m=300, n=260, k=8, seed=1,
                        prune=(_method == 'mu')))
        E2E.append(dict(fmt=_fmt, norm=_norm, method=_method, itr=_itr, grid=(2, 1), m=300, n=260, k=8, seed=2))
        E2E.append(dict(fmt=_fmt, norm=_norm, method=_method, itr=_itr, grid=(2, 2), m=300, n=260, k=8, seed=3,
                        prune=(_norm == 'fro' and _method == 'mu')))
    # a shard of 2^20 elements: the FRO passes run on the kind::f16 kernel
    for _method in ('mu', 'hals'):
        E2E.append(dict(fmt=_fmt, norm='fro', method=_method, itr=30, grid=(1, 1), m=1024, n=1024, k=16, seed=4,
                        expect_tc=True))


def _id(s):
    return '%s-%s-%s-%dx%d%s%s' % (s['fmt'], s['norm'], s['method'], s['grid'][0], s['grid'][1],
                                   '-prune' if s.get('prune') else '', '-tc' if s.get('expect_tc') else '')


@pytest.mark.parametrize('spec', E2E, ids=[_id(s) for s in E2E])
def test_fit_equals_float32_fit_of_rounded_matrix(spec):
    world = spec['grid'][0] * spec['grid'][1]
    if world == 1:
        from pydnmfk_b200.dist_comm import MPI
        MPI._reset()
        res = [pair_worker(0, 1, spec)]
    else:
        res = mp_util.run(world, pair_worker, (spec,), backend='gloo', timeout=900)
    _check(spec, res)


# ---- inputs and rejections ------------------------------------------------------------------------------------------
def _params(**kw):
    from pydnmfk_b200.dist_comm import MPI, MPI_comm
    from pydnmfk_b200.utils import parse
    MPI._reset()
    comms = MPI_comm(MPI.COMM_WORLD, 1, 1)
    p = parse()
    p.size, p.rank, p.comm1, p.comm, p.p_r, p.p_c = 1, 0, comms.comm, comms, 1, 1
    p.row_comm, p.col_comm = comms.cart_1d_row(), comms.cart_1d_column()
    p.k, p.itr, p.init, p.verbose, p.norm, p.method, p.prune = 4, 10, 'rand', False, 'fro', 'mu', False
    for key, val in kw.items():
        setattr(p, key, val)
    return p


@pytest.mark.parametrize('fmt', FMTS)
def test_cuda_inputs(fmt):
    from pydnmfk_b200.pyDNMF import PyNMF
    A = torch.rand((64, 48), device='cuda')
    A16 = A.to(TD[fmt])
    nmf = PyNMF(A16, params=_params(a_storage=fmt))
    assert nmf.A_ij.data_ptr() == A16.data_ptr(), 'a matching 16-bit CUDA tensor is used without a copy'
    nmf = PyNMF(A, params=_params(a_storage=fmt))
    assert nmf.A_ij.dtype == TD[fmt] and torch.equal(nmf.A_ij, A16)
    W, H, err = nmf.fit()
    assert W.dtype == torch.float32 and H.dtype == torch.float32
    other = 'bfloat16' if fmt == 'float16' else 'float16'
    with pytest.raises(ValueError, match='a_storage'):
        PyNMF(A16, params=_params(a_storage=other))


def test_rejections():
    from pydnmfk_b200.pyDNMF import PyNMF
    from pydnmfk_b200.pyDNMFk import PyNMFk
    A = np.random.rand(64, 48).astype(np.float32)
    A[5, 7] = 70000.0                                        # beyond float16's 65504
    with pytest.raises(ValueError, match='float16'):
        PyNMF(A, params=_params(a_storage='float16'))
    PyNMF(A, params=_params(a_storage='bfloat16'))           # in range for bfloat16
    with pytest.raises(ValueError, match='nnsvd'):
        PyNMF(A, params=_params(a_storage='bfloat16', init='nnsvd'))
    with pytest.raises(ValueError, match='a_storage'):
        PyNMF(A.astype(np.float64), params=_params(a_storage='float16'))
    with pytest.raises(ValueError, match='a_storage'):
        PyNMFk(A, params=_params(a_storage='float16'))
    from pydnmfk_b200.pyDNMFk import sample
    for dt in (torch.float16, torch.bfloat16):
        with pytest.raises(ValueError, match='a_storage'):
            sample(torch.from_numpy(A).cuda().to(dt), 0.03, 'uniform')
    with pytest.raises(TypeError):                           # no knob: today's behaviour for float16 data
        PyNMF(A.astype(np.float16), params=_params())
