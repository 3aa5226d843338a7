"""Parity of the CUDA product (PyNMF.fit through the C-ABI) with the reference.

Every case is replayed from the same seeded random init on the same input and compared with
(1) the golden vectors produced by the unmodified reference (tests/golden/nmf_cases.npz) and
(2) the numpy oracle.  Multi-rank grids run one process per rank on cuda:0 over gloo.

Tolerances (BASELINE.json north_star): W, H within 1e-4 relative Frobenius in fp32 (1e-10 in fp64),
reconstruction error within 1e-5 relative (1e-10 fp64); masks / index maps bit-exact.
BCD is compared at a looser factor tolerance: its accept/restore branch is a discrete decision and the
reference's BCD silently runs in float64 under numpy >= 2 (SURVEY 7.3, A12).
"""
import numpy as np
import pytest

from oracle import cases as C
from tests import common as T
from tests import mp_util, workers

pytestmark = pytest.mark.gpu


def _tol(case):
    tf, te = T.TOL_FACTOR[case['dtype']], T.TOL_ERR[case['dtype']]
    if case['method'] == 'bcd' and case['dtype'] == 'float32':
        # fp32 device path vs a reference that numpy >= 2 silently runs in float64 (SURVEY A12); measured 7e-7
        tf, te = 1e-4, 1e-4
    if case['data'] == 'lowrank':
        # exact rank-k data converges to err ~ 1e-9: the factors are then determined only up to the
        # conditioning of the problem; the reference's own test only asserts err < 1e-3
        tf = max(tf, 1e-6)
    return tf, te


def _log(rec):
    """Per-case differences, appended to $DNMF_TEST_LOG_DIR/parity_diffs.jsonl when that variable is set."""
    import json
    import os
    d = os.environ.get('DNMF_TEST_LOG_DIR')
    if not d:
        return
    try:
        os.makedirs(d, exist_ok=True)
        with open(os.path.join(d, 'parity_diffs.jsonl'), 'a') as f:
            f.write(json.dumps(rec) + '\n')
    except OSError:
        pass


def _compare(case, res):
    gold = T.golden_case(case['name'])
    tf, te = _tol(case)
    for r, o in enumerate(res):
        g = gold[r]
        _log(dict(case=case['name'], rank=r, relW=T.rel_fro(o['W'], g['W']), relH=T.rel_fro(o['H'], g['H']),
                  err=o['err'], err_ref=float(g['err']), tol_factor=tf, tol_err=te,
                  tc_passes=o.get('tc_passes'), generic_passes=o.get('generic_passes')))
        assert o['geom'] == [int(v) for v in g['geom'][:8]], 'shard geometry differs on rank %d' % r
        assert o['W'].shape == g['W'].shape and o['H'].shape == g['H'].shape
        if case['method'] != 'bcd':
            # (the reference's BCD returns float64 only because numpy >= 2 promotes it by accident, SURVEY A12;
            #  the device path keeps the data dtype)
            assert o['W'].dtype == g['W'].dtype and o['H'].dtype == g['H'].dtype, 'output dtype (float64 after unprune)'
        if case['prune']:
            for key in ('row_zero_idx_x', 'col_zero_idx_x', 'row_zero_idx_w', 'col_zero_idx_h'):
                assert np.array_equal(o[key], g[key]), key
        dW, dH = T.rel_fro(o['W'], g['W']), T.rel_fro(o['H'], g['H'])
        assert dW <= tf and dH <= tf, '%s rank %d: rel diff W %.3g H %.3g (tol %.1g)' % (case['name'], r, dW, dH, tf)
        ge = float(g['err'])
        # (absolute slack: on exact low-rank data the error converges towards 0 and only its magnitude is meaningful)
        slack = 1e-6 if case['dtype'] == 'float32' else 1e-9
        assert abs(o['err'] - ge) <= te * abs(ge) + (slack if case['data'] == 'lowrank' else 0.0), \
            '%s rank %d: err %.9g vs %.9g' % (case['name'], r, o['err'], ge)


def _run(case, force_generic=False, resident=True):
    world = case['grid'][0] * case['grid'][1]
    if world == 1:
        from pydnmfk_b200.dist_comm import MPI
        MPI._reset()
        return [workers.fit_worker(0, 1, case, force_generic, resident)]
    return mp_util.run(world, workers.fit_worker, (case, force_generic, resident), backend='gloo', timeout=900)


SINGLE = [c for c in C.CASES if c['grid'] == (1, 1)]
MULTI = [c for c in C.CASES if c['grid'] != (1, 1)]
# a representative multi-rank subset keeps the GPU suite to a few minutes (process spawn dominates)
MULTI_PICK = [c for c in MULTI if c['itr'] in (10, 300) or c['prune'] or c['given_factors'] or c['expect_tc']
              or (c['method'] == 'bcd' and c['itr'] == 100) or c['data'] == 'swim']
MULTI_PICK = [c for c in MULTI_PICK if not (c['name'].startswith('u64x48k4') and c['dtype'] == 'float64' and c['grid'] in ((1, 2), (4, 2)))]


@pytest.mark.parametrize('case', SINGLE, ids=[c['name'] for c in SINGLE])
def test_single_rank_matches_reference(case):
    """Per-kernel path (CUDA-graph replay of the update step)."""
    _compare(case, _run(case, resident=False))


SINGLE_MU = [c for c in SINGLE if c['method'] == 'mu']


@pytest.mark.parametrize('case', SINGLE_MU, ids=[c['name'] for c in SINGLE_MU])
def test_single_rank_resident_fit_matches_reference(case):
    """Whole-fit on-chip kernel (dnmf_mu_fit_resident) for shards that fit in one SM's shared memory; larger ones fall
    through to the per-kernel path."""
    _compare(case, _run(case, resident=True))


_multi_cache = {}


def _multi_results(case):
    """All picked cases of one world size run in a single spawn (results cached for the module)."""
    world = case['grid'][0] * case['grid'][1]
    if world not in _multi_cache:
        batch = [c for c in MULTI_PICK if c['grid'][0] * c['grid'][1] == world]
        per_rank = mp_util.run(world, workers.fit_many_worker, (batch,), backend='gloo', timeout=1800)
        _multi_cache[world] = per_rank
    per_rank = _multi_cache[world]
    res = []
    for r in range(world):
        if case['name'] not in per_rank[r]:
            pytest.fail('case did not run (an earlier case of this batch failed on rank %d)' % r)
        tag, val = per_rank[r][case['name']]
        if tag == 'err':
            pytest.fail('rank %d raised:\n%s' % (r, val))
        res.append(val)
    return res


@pytest.mark.parametrize('case', MULTI_PICK, ids=[c['name'] for c in MULTI_PICK])
def test_multi_rank_matches_reference(case):
    _compare(case, _multi_results(case))


@pytest.mark.parametrize('name', ['u2048k32_1x1_fro_mu_i100', 'u2048k32_1x1_kl_mu_i100', 'u2048k64_1x1_fro_mu_i10',
                                  'u2048k10_1x1_kl_mu_i10', 'u2048k64_1x1_kl_mu_i10'])
def test_generic_and_tensor_core_paths_agree_with_reference(name):
    """Both device code paths (tcgen05 and generic CUDA-core) are held to the same reference tolerance on shards
    large enough for the tcgen05 kernels; fit_worker asserts which kernels each arm actually ran."""
    case = C.CASES_BY_NAME[name]
    gen = _run(case, force_generic=True)
    assert gen[0]['tc_passes'] == 0 and gen[0]['generic_passes'] > 0
    _compare(case, gen)
    tc = _run(case, force_generic=False)
    assert tc[0]['generic_passes'] == 0 and tc[0]['tc_passes'] > 0
    _compare(case, tc)


def test_matches_oracle_live():
    """Same comparison against the numpy oracle run now (not only the stored vectors)."""
    for name in ('u64x48k4_1x1_fro_mu_i10_32', 'u64x48k4_1x1_kl_mu_i10_64', 'zeros40x36k3_1x1_kl_mu_prune'):
        case = C.CASES_BY_NAME[name]
        res = _run(case)
        out = T.run_oracle(case)
        tf, te = _tol(case)
        assert T.rel_fro(res[0]['W'], out[0][0]) <= tf and T.rel_fro(res[0]['H'], out[0][1]) <= tf
        assert abs(res[0]['err'] - float(out[0][2])) <= te * abs(float(out[0][2]))


def test_update_objects_accept_numpy_like_the_reference():
    """nmf_algorithms_1D(A, W, H, params).update() with host arrays (the reference's call shape)."""
    from pydnmfk_b200.dist_comm import MPI, MPI_comm
    from pydnmfk_b200.dist_nmf import nmf_algorithms_1D
    from pydnmfk_b200.utils import parse
    MPI._reset()
    comm = MPI.COMM_WORLD
    comms = MPI_comm(comm, 1, 1)
    rs = np.random.RandomState(3)
    A, W, H = rs.rand(50, 40).astype(np.float32), rs.rand(50, 3).astype(np.float32), rs.rand(3, 40).astype(np.float32)
    p = parse()
    p.m, p.n, p.p_r, p.p_c, p.k, p.comm1, p.norm, p.method = 50, 40, 1, 1, 3, comm, 'fro', 'mu'
    p.eps, p.W_update, p.itr = np.finfo(np.float32).eps, True, 1
    W1, H1 = nmf_algorithms_1D(A, W.copy(), H.copy(), params=p).update()
    f = np.float64
    Wr = W.astype(f) * ((A.astype(f) @ H.astype(f).T) / (W.astype(f) @ (H.astype(f) @ H.astype(f).T) + p.eps))
    Hr = H.astype(f) * ((Wr.T @ A.astype(f)) / ((H.astype(f).T @ (Wr.T @ Wr)) + p.eps).T)
    assert T.rel_fro(W1, Wr) < 1e-5 and T.rel_fro(H1, Hr) < 1e-5
    for bad in (('fro', 'xx', 'Not a valid method: Choose (mu/hals/bcd)'), ('kl', 'hals', 'Not a valid method: Choose (mu)'),
                ('l1', 'mu', 'Not a valid norm: Choose (fro/kl)')):
        p.norm, p.method = bad[0], bad[1]
        with pytest.raises(Exception) as e:
            nmf_algorithms_1D(A, W.copy(), H.copy(), params=p).update()
        assert str(e.value) == bad[2]


def test_public_helpers_accept_any_operands_like_the_reference():
    """global_mm / global_gram / sum_along_axis of nmf_algorithms_1D (dist_nmf.py:662-711, :775-801) with operands that
    are NOT the resident shard (the reference's helpers are plain ``A @ B``): chunked skinny contractions."""
    from pydnmfk_b200.dist_comm import MPI, MPI_comm
    from pydnmfk_b200.dist_nmf import nmf_algorithms_1D
    from pydnmfk_b200.utils import parse
    MPI._reset()
    comm = MPI.COMM_WORLD
    MPI_comm(comm, 1, 1)
    rs = np.random.RandomState(4)
    A, W, H = rs.rand(60, 45).astype(np.float32), rs.rand(60, 5).astype(np.float32), rs.rand(5, 45).astype(np.float32)
    p = parse()
    p.m, p.n, p.p_r, p.p_c, p.k, p.comm1, p.norm, p.method = 60, 45, 1, 1, 5, comm, 'fro', 'mu'
    p.eps, p.W_update, p.itr = np.finfo(np.float32).eps, True, 1
    alg = nmf_algorithms_1D(A, W, H, params=p)
    f = np.float64

    def host(t):
        return t.cpu().numpy() if hasattr(t, 'cpu') else np.asarray(t)

    X, Y = rs.rand(33, 70).astype(np.float32), rs.rand(70, 150).astype(np.float32)      # 150 > 64 output columns: chunked
    assert T.rel_fro(host(alg.global_mm(X, Y, 1)), X.astype(f) @ Y.astype(f)) < 2e-6
    assert T.rel_fro(host(alg.global_mm(A, H.T, 1)), A.astype(f) @ H.astype(f).T) < 2e-6          # the update's own calls
    assert T.rel_fro(host(alg.global_mm(W.T, A, 1)), W.astype(f).T @ A.astype(f)) < 2e-6
    wide = rs.rand(45, 100).astype(np.float32)                                                   # resident shard x wide matrix
    assert T.rel_fro(host(alg.global_mm(A, wide, 1)), A.astype(f) @ wide.astype(f)) < 2e-6
    assert T.rel_fro(host(alg.global_gram(W, 1)), W.astype(f).T @ W.astype(f)) < 2e-6
    assert T.rel_fro(host(alg.sum_along_axis(H, 1, axis=1)), H.astype(f).sum(1)) < 2e-6


def test_ensemble_spread_over_ranks_equals_sequential():
    """NMFk perturbation ensemble (pyDNMFk.py:226-238): spreading the perturbations over ranks gives exactly the
    sequential stacking; the W-fixed regression fit (pyDNMFk.py:245-248) leaves W untouched up to normalisation."""
    from oracle import nmf_oracle as O
    seq = mp_util.run(1, workers.ensemble_worker, (False,), backend='gloo', timeout=600)[0]
    par = mp_util.run(2, workers.ensemble_worker, (True,), backend='gloo', timeout=600)
    for r in range(2):
        assert np.array_equal(par[r]['Wall'], seq['Wall']) and np.array_equal(par[r]['Hall'], seq['Hall'])
        assert par[r]['errs'] == seq['errs']
    assert seq['Wall'].shape == (96, 3, 6) and seq['Hall'].shape == (3, 21, 6)
    # oracle replay of perturbation 2 (seed 2000): noise, then init from the same stream (SURVEY A8)
    rs = np.random.RandomState(5)
    A = (rs.rand(96, 21) * 100).astype(np.float32)
    rng = np.random.RandomState(2000)
    X = O.perturb(A, 0.015, 'uniform', rng)
    ref = O.fit([X], 1, 1, 3, 'kl', 'mu', 30, rngs=[rng], prune=True)[0]
    # (Hall is the reference's vstack + C-order reshape, pyDNMFk.py:236-237: perturbation p is rows [p k, (p+1) k) of
    #  the (P k, n) stack, not the slice [:, :, p])
    H2 = seq['Hall'].reshape(6 * 3, 21)[2 * 3:3 * 3]
    assert T.rel_fro(seq['Wall'][:, :, 2], ref[0]) <= 1e-4 and T.rel_fro(H2, ref[1]) <= 1e-4
    assert abs(seq['errs'][2] - float(ref[2])) <= 1e-5 * float(ref[2])
    assert np.isfinite(seq['col_err']).all() and seq['col_err'].shape == (21,)


@pytest.mark.parametrize('name', ['u2048k32_2x1_fro_mu_i10', 'u2048k32_1x2_fro_mu_i10', 'u2048k32_2x2_fro_mu_i10',
                                  'u4096x1024k32_1x1_fro_mu_i10', 'u64x48k4_4x2_fro_mu_i10_32'])
def test_trace_identity_monitor_matches_direct_residual(name):
    """params.err_monitor (dnmf_trace_terms): entry j-1 of the per-iteration history is the relative error after j
    iterations, i.e. what a fit cut at j iterations returns from its direct residual pass; the monitored fit itself still
    matches the reference golden."""
    case = C.CASES_BY_NAME[name]
    world = case['grid'][0] * case['grid'][1]
    checkpoints = [1, 4, 9]
    res = mp_util.run(world, workers.monitor_worker, (case, checkpoints), backend='gloo', timeout=900) if world > 1 \
        else [workers.monitor_worker(0, 1, case, checkpoints)]
    _compare(case, [r['full'] for r in res])
    for r in res:
        hist = r['full']['err_history']
        assert hist is not None and len(hist) == case['itr'] - 1
        for j in checkpoints:
            # fp32 factors, float64 accumulation; err ~ 0.3-0.5 on these random matrices, no cancellation
            assert abs(hist[j - 1] - r['err_at_%d' % j]) <= 2e-5 * r['err_at_%d' % j], (j, hist[j - 1], r['err_at_%d' % j])
