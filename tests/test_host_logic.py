"""Host-side logic that needs no GPU: shard index maps, argument helpers, error messages."""
import os

import numpy as np
import pytest

from oracle import nmf_oracle as O
from tests import common as T


def test_determine_block_params_known_answers():
    from pydnmfk_b200.utils import determine_block_params
    # the reference's own known-answer test (tests/test_dist_file_split.py:26-30)
    d0 = determine_block_params(0, (2, 1), (96, 21))
    d1 = determine_block_params(1, (2, 1), (96, 21))
    assert d0.determine_block_index_range_asymm() == ([0, 0], [47, 20])
    assert d0.determine_block_shape_asymm() == [48, 21]
    assert d1.determine_block_index_range_asymm() == ([48, 0], [95, 20])
    assert d1.determine_block_shape_asymm() == [48, 21]
    aux = T.golden('aux_cases.npz')
    n = 0
    for key, val in aux.items():
        if not key.startswith('blocks/'):
            continue
        shape = tuple(int(v) for v in key.split('/')[1].split('x'))
        grid = tuple(int(v) for v in key.split('/')[2].split('x'))
        for r in range(grid[0] * grid[1]):
            d = determine_block_params(r, grid, shape)
            s, e = d.determine_block_index_range_asymm()
            assert list(s) + list(e) + d.determine_block_shape_asymm() == [int(v) for v in val[r]]
            n += 1
    assert n > 30


def test_block_params_match_oracle_on_random_shapes():
    from pydnmfk_b200.utils import determine_block_params
    rs = np.random.RandomState(0)
    for _ in range(200):
        grid = (int(rs.randint(1, 7)), int(rs.randint(1, 7)))
        shape = (int(rs.randint(grid[0], 500)), int(rs.randint(grid[1], 500)))
        for r in range(grid[0] * grid[1]):
            d = determine_block_params(r, grid, shape)
            s, e = d.determine_block_index_range_asymm()
            so, eo = O.block_range(r, grid, shape)
            assert (list(s), list(e)) == (so, eo)


def test_arg_helpers():
    from pydnmfk_b200.utils import parse, var_init, str2bool
    p = parse()
    assert var_init(p, 'norm', 'kl') == 'kl' and p.norm == 'kl'
    p.norm = 'fro'
    assert var_init(p, 'norm', 'kl') == 'fro'
    assert str2bool('Yes') is True and str2bool('0') is False and str2bool(True) is True
    with pytest.raises(NameError, match='Boolean value expected.'):
        str2bool('maybe')


def test_single_process_comm_is_a_noop_world():
    from pydnmfk_b200.dist_comm import MPI, MPI_comm
    comm = MPI.COMM_WORLD
    assert comm.size == 1 and comm.rank == 0 and comm.Get_rank() == 0 and comm.Get_size() == 1
    comms = MPI_comm(comm, 1, 1)
    assert comms.coord2d == [0, 0]
    row, col = comms.cart_1d_row(), comms.cart_1d_column()
    assert row.size == 1 and col.size == 1
    assert comm.allreduce(5) == 5
    x = np.arange(4.0)
    assert np.array_equal(comm.allreduce(x), x)
    assert comm.allgather('a') == ['a']
    assert comm.bcast({'k': 1}, root=0) == {'k': 1}
    comm.barrier()
    comms.Free()


def test_data_operations_dims_single_rank():
    from pydnmfk_b200.dist_comm import MPI, MPI_comm
    from pydnmfk_b200.utils import parse, data_operations
    comm = MPI.COMM_WORLD
    comms = MPI_comm(comm, 1, 1)
    p = parse()
    p.comm1, p.row_comm, p.col_comm, p.p_r, p.p_c, p.topo, p.k = comm, comms.cart_1d_row(), comms.cart_1d_column(), 1, 1, '1d', 3
    A = np.zeros((26, 14), dtype=np.float32)
    data_operations(A, p)
    assert (p.m, p.n, p.m_loc, p.n_loc, p.W_start, p.W_end, p.H_start, p.H_end) == (26, 14, 26, 14, 0, 26, 0, 14)


def test_reference_import_surface():
    """`from pyDNMFk.pyDNMF import *` style imports of the reference's tests resolve to this package and export the names
    those tests use (tests/test_dist_nmf_1d.py:8-9,29,35 of the reference)."""
    ns = {}
    exec('from pyDNMFk.pyDNMF import *\nfrom pyDNMFk.dist_comm import *\nimport pyDNMFk.config as config', ns)
    for name in ('PyNMF', 'np', 'MPI', 'MPI_comm', 'parse', 'determine_block_params', 'data_read', 'nmf_algorithms_1D',
                 'nmf_algorithms_2D', 'var_init', 'data_operations'):
        assert name in ns, name
    ns['config'].init(0)
    import pydnmfk_b200.pyDNMF as real
    assert ns['PyNMF'] is real.PyNMF


def test_cli_flag_surface():
    import main as cli
    import argparse
    p = cli.parser_pyNMFk(cli.parser_pyNMF(argparse.ArgumentParser()))
    a = p.parse_args(['--p_r', '2', '--p_c', '1'])
    assert (a.k, a.itr, a.norm, a.method, a.prune, a.precision, a.init) == (4, 5000, 'kl', 'mu', False, 'float32', 'rand')
    assert (a.perturbations, a.noise_var, a.start_k, a.end_k, a.step_k, a.sill_thr, a.sampling) == (20, 0.015, 1, 10, 1, 0.6, 'uniform')


def test_rank_selection_matches_reference():
    """pvalueAnalysis on fabricated per-k results written through the product's own results store."""
    import tempfile
    from oracle import nmfk_cases as K
    with np.load(os.path.join(K.GOLDEN, 'nmfk_cases.npz')) as z:
        gold = {k: z[k] for k in z.files}
    from pydnmfk_b200.data_io import write_results
    from pydnmfk_b200.pyDNMFk import PyNMFk
    from pydnmfk_b200.utils import parse
    for name, sc in K.pvalue_scenarios().items():
        with tempfile.TemporaryDirectory() as tmp:
            p = parse()
            p.start_k, p.end_k, p.results_path = sc['start_k'], sc['end_k'], tmp + '/'
            for i, k in enumerate(range(sc['start_k'], sc['end_k'] + 1, sc['step_k'])):
                os.makedirs('%s/%d' % (tmp, k))
                write_results('%s/%d/' % (tmp, k), {'L_err': sc['L_err'][i],
                                                     'clusterSilhouetteCoefficients': np.array([sc['sil_min'][i], 1.0])})
            obj = object.__new__(PyNMFk)
            obj.params, obj.step_k, obj.sill_thr = p, sc['step_k'], sc['sill_thr']
            nopt, pv = obj.pvalueAnalysis()
        assert nopt == int(gold['pvalue/%s/0/nopt' % name])
        assert np.allclose(pv, gold['pvalue/%s/0/pvalue' % name], rtol=1e-12, atol=0)


def test_data_io_formats(tmp_path):
    """Shard input formats (data_io.py:12-105) and the per-k results / factor files (data_io.py:139-261), host only."""
    import scipy.io
    from pydnmfk_b200.data_io import data_read, data_write, read_factors, read_results, write_results
    from pydnmfk_b200.utils import parse

    class _Comm:
        def __init__(self, rank):
            self.rank = rank

        def barrier(self):
            pass

    rs = np.random.RandomState(0)
    X = rs.rand(26, 14)
    d = str(tmp_path) + '/'
    np.save(d + 'X.npy', X)
    np.savetxt(d + 'X.csv', X, delimiter=',')
    scipy.io.savemat(d + 'X.mat', {'X': X})
    for rank in range(4):
        s, e = O.block_range(rank, (2, 2), X.shape)
        np.save(d + 'A_%d.npy' % rank, X[s[0]:e[0] + 1, s[1]:e[1] + 1])
    from pydnmfk_b200.data_io import split_files_save
    split_files_save(X, (2, 2), d + 'split/').save_data_to_file()
    for rank in range(4):
        assert np.array_equal(np.load(d + 'split/A_%d.npy' % rank), np.load(d + 'A_%d.npy' % rank))
    for ftype, fname in (('npy', 'X'), ('csv', 'X'), ('mat', 'X'), ('folder', 'A_')):
        for rank in range(4):
            p = parse()
            p.fpath, p.fname, p.ftype, p.p_r, p.p_c, p.comm1, p.precision = d, fname, ftype, 2, 2, _Comm(rank), 'float32'
            got = data_read(p).read()
            s, e = O.block_range(rank, (2, 2), X.shape)
            assert got.dtype == np.float32 and got.flags.c_contiguous
            assert np.allclose(got, X[s[0]:e[0] + 1, s[1]:e[1] + 1].astype(np.float32), rtol=1e-6), (ftype, rank)
    # regression factors of a 2 x 2 grid: W blocks stack by rank, H blocks are ordered (j, i) (SURVEY A2)
    W = rs.rand(26, 3)
    H = rs.rand(3, 14)
    for rank in range(4):
        i, j = divmod(rank, 2)
        p = parse()
        p.p_r, p.p_c, p.comm1, p.results_paths, p.ftype = 2, 2, _Comm(rank), d + 'res/', 'npy'
        (r0, _), (r1, _) = O.block_range(rank, (4, 1), (26, 3))           # W rows: rank order
        hb = j * 2 + i                                                  # H columns: (j, i) order
        (_, c0), (_, c1) = O.block_range(hb, (1, 4), (3, 14))
        data_write(p).save_factors([W[r0:r1 + 1], H[:, c0:c1 + 1]], reg=True)
    Wr, Hr = read_factors(d + 'res/', (2, 2)).load_factors()
    assert np.array_equal(Wr, W) and np.array_equal(Hr, H)
    # 1-D grids: the replicated factor is written once without a rank suffix (data_io.py:184-192)
    for grid, once, per_rank in (((2, 1), 'H_reg_factors/H.npy', 'W_reg_factors/W_%d.npy'),
                                 ((1, 2), 'W_reg_factors/W.npy', 'H_reg_factors/H_%d.npy')):
        out = d + 'res_%dx%d/' % grid
        for rank in range(2):
            p = parse()
            p.p_r, p.p_c, p.comm1, p.results_paths, p.ftype = grid[0], grid[1], _Comm(rank), out, 'npy'
            data_write(p).save_factors([W[:3] + rank, H[:, :4] + rank], reg=True)
        import os as _os
        found = sorted(_os.path.join(dp, f)[len(out):] for dp, _, fs in _os.walk(out) for f in fs)
        assert found == sorted([once, per_rank % 0, per_rank % 1]), found
        assert np.array_equal(np.load(out + once), (H[:, :4] if once.startswith('H') else W[:3]))      # rank 0's copy
    stats = {'clusterSilhouetteCoefficients': np.array([0.9, 0.8]), 'avgSilhouetteCoefficients': 0.85, 'L_err': rs.rand(14),
             'L_errDist': 0.1, 'avgErr': 0.2, 'recon_err': [0.2, 0.21], 'AIC': -3.0}
    p = parse()
    p.p_r, p.p_c, p.comm1, p.results_paths, p.ftype = 1, 1, _Comm(0), d + 'res/', 'npy'
    data_write(p).save_cluster_results(stats)
    back = read_results(d + 'res/')
    assert set(back) == {'clusterSilhouetteCoefficients', 'avgSilhouetteCoefficients', 'L_err', 'L_errDist', 'avgErr', 'ErrTol', 'AIC'}
    assert np.array_equal(back['L_err'], stats['L_err']) and np.array_equal(back['ErrTol'], np.array(stats['recon_err']))
    write_results(d + 'res/', {'L_err': np.arange(3.0)})
    assert np.array_equal(read_results(d + 'res/')['L_err'], np.arange(3.0))


def test_runner_front_end(monkeypatch, tmp_path):
    """pyDNMFk_Runner (runner.py:12-191): defaults, argument checks, and that the runner object is the params bag handed
    to data_read / PyNMF / PyNMFk with the grid, k range and communicators set."""
    from pyDNMFk.runner import pyDNMFk_Runner
    import pydnmfk_b200.runner as R
    r = pyDNMFk_Runner()
    assert (r.init, r.itr, r.norm, r.method, r.prune, r.precision, r.perturbations, r.noise_var, r.sill_thr, r.sampling,
            r.process) == ('rand', 5000, 'kl', 'mu', False, 'float32', 20, 0.015, 0.6, 'uniform', 'pyDNMF')
    assert pyDNMFk_Runner('nnsvd', 10).itr == 10
    with pytest.raises(ValueError):
        pyDNMFk_Runner(process='nmf')
    with pytest.raises(TypeError):
        pyDNMFk_Runner(iterations=3)
    with pytest.raises(ValueError):
        r.run(grid=[1, 1, 1])
    seen = {}

    class FakeRead:
        def __init__(self, params):
            seen['read'] = (params.fpath, params.fname, params.ftype, params.p_r, params.p_c, params.precision)

        def read(self):
            return np.ones((4, 3), dtype=np.float32)

    class FakeNMF:
        def __init__(self, A, factors=None, params=None):
            seen['nmf'] = (A.shape, params.k, params.itr, params.grid, params.comm1.size, params.row_comm.size)

        def fit(self):
            return 'W', 'H', 0.25

    class FakeNMFk(FakeNMF):
        def __init__(self, A, factors=None, params=None):
            seen['nmfk'] = (params.start_k, params.end_k, params.step_k, params.perturbations, params.sill_thr)

        def fit(self):
            return 3

    monkeypatch.setattr(R, 'data_read', FakeRead)
    monkeypatch.setattr(R, 'PyNMF', FakeNMF)
    monkeypatch.setattr(R, 'PyNMFk', FakeNMFk)
    out = pyDNMFk_Runner(itr=7).run(grid=[1, 1], fpath='d/', fname='x', ftype='npy', results_path=str(tmp_path) + '/', k=5)
    assert out == {'W': 'W', 'H': 'H', 'err': 0.25}
    assert seen['read'] == ('d/', 'x', 'npy', 1, 1, 'float32') and seen['nmf'] == ((4, 3), 5, 7, [1, 1], 1, 1)
    out = pyDNMFk_Runner(process='pyDNMFk', perturbations=4, timing_stats=False).run(grid=[1, 1], k_range=[2, 6], step_k=2)
    assert out == {'nopt': 3} and seen['nmfk'] == (2, 6, 2, 4, 0.6)


def test_transform_H_index_orders_shards_by_block_column():
    from pydnmfk_b200.utils import transform_H_index
    assert transform_H_index((2, 2)).rankidx2blkidx() == [0, 2, 1, 3]            # same as the reference on square grids
    assert transform_H_index((4, 2)).rankidx2blkidx() == [0, 2, 4, 6, 1, 3, 5, 7]
    assert transform_H_index((2, 3)).rankidx2blkidx() == [0, 3, 1, 4, 2, 5]
    # cross-check with the oracle's shard geometry: concatenating the H shards in this order restores the columns
    for p_r, p_c in ((2, 3), (4, 2), (3, 3)):
        n = 37
        cols = {}
        for r in range(p_r * p_c):
            i, j = divmod(r, p_c)
            (_, c0), (_, c1) = O.block_range(r, (p_r, p_c), (5, n))               # block column j of A
            width = c1 - c0 + 1
            s = i * (width // p_r) + min(i, width % p_r)
            e = (i + 1) * (width // p_r) + min(i + 1, width % p_r)
            cols[r] = list(range(c0 + s, c0 + e))                                # sub-block i of block column j
        order = transform_H_index((p_r, p_c)).rankidx2blkidx()
        assert sum((cols[r] for r in order), []) == list(range(n))


def test_bench_cpu_arm_allreduce_matches_oracle():
    """bench.py's CPU arm runs one forked process per rank and all-reduces through shared memory; its factors must be
    the oracle's own virtual-rank result for the same shards (float32 summation order aside)."""
    import bench
    from oracle import nmf_oracle as O
    m, n, k, cores, steps = 96, 64, 4, 3, 3
    for norm in ('fro', 'kl'):
        got = bench.cpu_probe(m, n, k, norm, steps, cores)
        shard = m // cores
        st = O._State()
        st.grid, st.k, st.norm, st.method, st.W_update = O.VGrid(cores, 1), k, norm, 'mu', True
        st.A = [np.random.default_rng(1234 + r).random((shard, n), dtype=np.float32) for r in range(cores)]
        st.dt, st.eps, st.topo = np.dtype(np.float32), np.finfo(np.float32).eps, '1d'
        st.W = [np.random.RandomState(11 + r).rand(shard, k).astype(np.float32) for r in range(cores)]
        H0 = np.random.RandomState(7).rand(k, n).astype(np.float32)
        st.H = [H0.copy() for _ in range(cores)]
        for i in range(steps):
            O.update(st, 1)
            if i % 10 == 0:
                st.H = [np.maximum(h, st.eps) for h in st.H]
                st.W = [np.maximum(w, st.eps) for w in st.W]
        for r, W, H in got:
            assert np.allclose(W, st.W[r], rtol=2e-5, atol=1e-7) and np.allclose(H, st.H[r], rtol=2e-5, atol=1e-7)


def test_bench_dump_outputs_sample_is_fixed_and_within_the_limit(tmp_path):
    """bench.py --dump-outputs: arrays under the limit are written whole; above it every array keeps the same seeded
    sample of its longest axis on every run, and the files together stay within the limit."""
    import bench
    rs = np.random.RandomState(0)
    arrays = {'fro_W': rs.rand(1000, 8).astype(np.float32), 'fro_H': rs.rand(8, 1000).astype(np.float32)}
    bench.dump_outputs(str(tmp_path / 'whole'), arrays, 1 << 20)
    for name, a in arrays.items():
        assert np.array_equal(np.load(tmp_path / 'whole' / (name + '.npy')), a)
    limit = 16000
    for run in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / run), arrays, limit)
    sizes = 0
    for name, a in arrays.items():
        x, y = np.load(tmp_path / 'a' / (name + '.npy')), np.load(tmp_path / 'b' / (name + '.npy'))
        assert np.array_equal(x, y) and x.dtype == np.float32 and 0 < x.size < a.size
        sizes += x.nbytes
    assert sizes <= limit
    W = np.load(tmp_path / 'a' / 'fro_W.npy')
    assert all(any(np.array_equal(row, r) for r in arrays['fro_W']) for row in W[:5])
