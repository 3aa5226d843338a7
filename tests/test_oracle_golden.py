"""Pin the numpy oracle (oracle/nmf_oracle.py) to the reference's own outputs.

tests/golden/nmf_cases.npz was produced by oracle/gen_golden.py running the UNMODIFIED reference
(PyNMF.fit under a fork-based mpi4py stand-in).  The oracle must reproduce those factors, shard
geometries and prune masks.
"""
import numpy as np
import pytest

from oracle import cases as C
from oracle import nmf_oracle as O
from tests import common as T

FAST = [c for c in C.CASES if not (c['m'] >= 512 and c['itr'] >= 100)]
SLOW = [c for c in C.CASES if c not in FAST]


def _check(case, out):
    gold = T.golden_case(case['name'])
    assert len(gold) == len(out)
    dt = case['dtype']
    tol = 1e-5 if dt == 'float32' else 1e-11   # same numpy/BLAS => normally identical; slack for BLAS threading
    for r, (W, H, err) in enumerate(out):
        g = gold[r]
        assert W.shape == g['W'].shape and H.shape == g['H'].shape
        assert W.dtype == g['W'].dtype and H.dtype == g['H'].dtype
        assert T.rel_fro(W, g['W']) <= tol, (case['name'], r, 'W')
        assert T.rel_fro(H, g['H']) <= tol, (case['name'], r, 'H')
        assert abs(float(err) - float(g['err'])) <= tol * abs(float(g['err'])) + 1e-12


@pytest.mark.parametrize('case', FAST, ids=[c['name'] for c in FAST])
def test_oracle_matches_reference_golden(case):
    _check(case, T.run_oracle(case))


@pytest.mark.parametrize('case', SLOW, ids=[c['name'] for c in SLOW])
def test_oracle_matches_reference_golden_long(case):
    _check(case, T.run_oracle(case))


def test_golden_covers_every_case():
    g = T.golden()
    for c in C.CASES:
        P = c['grid'][0] * c['grid'][1]
        for r in range(P):
            assert '%s/%d/W' % (c['name'], r) in g, c['name']


@pytest.mark.parametrize('case', [c for c in C.CASES if c['prune']], ids=lambda c: c['name'])
def test_oracle_masks_and_geometry_bit_exact(case):
    """Shard index maps and prune masks are integer work: exact equality (north_star)."""
    A, blocks, rngs, factors = T.oracle_inputs(case)
    grid = O.VGrid(*case['grid'])
    sh = O.compute_dims(blocks, grid, case['k'])
    masks = O.zero_idx_prune(blocks, grid, sh)
    gold = T.golden_case(case['name'])
    for r in range(grid.p):
        geom = gold[r]['geom']
        assert [sh.m[r], sh.n[r], sh.m_loc[r], sh.n_loc[r], sh.W_start[r], sh.W_end[r], sh.H_start[r],
                sh.H_end[r]] == [int(v) for v in geom[:8]]
        for key, mk in zip(('row_zero_idx_x', 'col_zero_idx_x', 'row_zero_idx_w', 'col_zero_idx_h'), masks):
            assert np.array_equal(mk[r], gold[r][key]), (case['name'], r, key)


def test_geometry_all_cases():
    for case in C.CASES:
        A, blocks, rngs, factors = T.oracle_inputs(case)
        grid = O.VGrid(*case['grid'])
        sh = O.compute_dims(blocks, grid, case['k'])
        gold = T.golden_case(case['name'])
        for r in range(grid.p):
            geom = [int(v) for v in gold[r]['geom']]
            assert [sh.m[r], sh.n[r], sh.m_loc[r], sh.n_loc[r], sh.W_start[r], sh.W_end[r], sh.H_start[r],
                    sh.H_end[r]] == geom[:8], case['name']
            s, e = O.block_range(r, case['grid'], (case['m'], case['n']))
            assert [s[0], e[0], s[1], e[1]] == geom[8:12]


def test_block_known_answers():
    """tests/test_dist_file_split.py:26-30 of the reference + generated known answers."""
    assert O.block_range(0, (2, 1), (96, 21)) == ([0, 0], [47, 20])
    assert O.block_range(1, (2, 1), (96, 21)) == ([48, 0], [95, 20])
    assert O.block_shape(1, (2, 1), (96, 21)) == [48, 21]
    aux = T.golden('aux_cases.npz')
    for key, val in aux.items():
        if not key.startswith('blocks/'):
            continue
        shp, grd = key.split('/')[1:]
        shape = tuple(int(v) for v in shp.split('x'))
        grid = tuple(int(v) for v in grd.split('x'))
        for r in range(grid[0] * grid[1]):
            s, e = O.block_range(r, grid, shape)
            assert s + e + O.block_shape(r, grid, shape) == [int(v) for v in val[r]]


def test_perturb_matches_reference_sample():
    aux = T.golden('aux_cases.npz')
    X = (np.arange(12 * 7, dtype=np.float32).reshape(12, 7) % 17) + 1
    for method, seed in (('uniform', 0), ('uniform', 1000), ('poisson', 3000)):
        rs = np.random.RandomState(seed)
        Y = O.perturb(X, 0.015, method, rs)
        assert np.array_equal(Y, aux['sample/%s/%d/Y' % (method, seed)])
        assert np.array_equal(rs.rand(3), aux['sample/%s/%d/nxt' % (method, seed)])


def test_oracle_vs_live_reference():
    """Two cases at a tighter tolerance against the output of the reference's own PyNMF.fit (oracle.gen_golden._ref_fit,
    stored in tests/golden/nmf_cases.npz)."""
    for name in ('u64x48k4_2x1_fro_mu_i10_32', 'ragged26x14k3_2x2_kl_mu'):
        case = C.CASES_BY_NAME[name]
        P = case['grid'][0] * case['grid'][1]
        ref = T.golden_case(name)
        out = T.run_oracle(case)
        for r in range(P):
            assert T.rel_fro(out[r][0], ref[r]['W']) <= 1e-6
            assert T.rel_fro(out[r][1], ref[r]['H']) <= 1e-6
