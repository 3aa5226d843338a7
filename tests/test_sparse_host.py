"""Sparse data shards without a GPU: canonical form of scipy and torch input, what a sparse A_ij rejects, and argument
checks of the sparse C-ABI entry points."""
import numpy as np
import pytest
import torch


def _messy_coo():
    """Unsorted indices, a duplicate pair summing to 9, a duplicate pair cancelling to 0 and an explicit zero."""
    import scipy.sparse as sp
    r = np.array([2, 0, 0, 1, 2, 2, 0, 3, 3, 1])
    c = np.array([1, 3, 0, 2, 1, 0, 3, 4, 4, 0])
    v = np.array([1.0, 2.0, 0.0, 4.0, 5.0, 6.0, 7.0, 1.5, -1.5, 3.0], dtype=np.float32)
    return sp.coo_matrix((v, (r, c)), shape=(5, 6)), r, c, v


def _expected_arrays(dense):
    m, n = dense.shape
    rows, cols = np.nonzero(dense)
    row_ptr = np.concatenate([[0], np.cumsum(np.count_nonzero(dense, axis=1))])
    ct, rt = np.nonzero(dense.T)
    col_ptr = np.concatenate([[0], np.cumsum(np.count_nonzero(dense, axis=0))])
    return row_ptr, cols, dense[rows, cols], col_ptr, rt, dense[rt, ct]


def test_canonical_form_is_the_same_from_scipy_and_torch():
    from pydnmfk_b200.sparse import canonical_arrays
    A, r, c, v = _messy_coo()
    dense = A.toarray()
    want = _expected_arrays(dense)
    inputs = [A, A.tocsr(), A.tocsc(), torch.sparse_coo_tensor(np.stack([r, c]), v, (5, 6)).to_sparse_csr()]
    # an unsorted CSR with a duplicate and a stored zero, built directly
    crow = torch.tensor([0, 3, 4, 7, 9, 9])
    col = torch.tensor([3, 0, 3, 2, 1, 0, 1, 4, 4])
    val = torch.tensor([2.0, 0.0, 7.0, 4.0, 1.0, 6.0, 5.0, 1.5, -1.5])
    d2 = np.zeros((5, 6), np.float32)
    for i in range(5):
        for e in range(int(crow[i]), int(crow[i + 1])):
            d2[i, int(col[e])] += float(val[e])
    inputs.append(torch.sparse_csr_tensor(crow, col, val, (5, 6)))
    for i, X in enumerate(inputs):
        shape, arrays = canonical_arrays(X)
        exp = want if i < len(inputs) - 1 else _expected_arrays(d2)
        assert shape == (5, 6)
        for got, e in zip(arrays, exp):
            assert np.array_equal(got.numpy().astype(np.float64), np.asarray(e, dtype=np.float64)), i
        assert arrays[2].dtype == torch.float32 and 0 not in arrays[2].numpy() and 0 not in arrays[5].numpy()


def test_integer_values_raise_the_dense_type_error():
    import scipy.sparse as sp
    from pydnmfk_b200.sparse import canonical_arrays
    with pytest.raises(TypeError, match='float32/float64'):
        canonical_arrays(sp.csr_matrix(np.eye(3, dtype=np.int64)))
    with pytest.raises(TypeError, match='float32/float64'):
        canonical_arrays(torch.eye(3, dtype=torch.int32).to_sparse_csr())


def _params(**kw):
    from pydnmfk_b200.utils import parse
    p = parse()
    p.init, p.k, p.p_r, p.p_c, p.verbose = 'rand', 2, 1, 1, False
    for key, val in kw.items():
        setattr(p, key, val)
    return p


def test_sparse_rejections_raise_value_error_before_the_device():
    import scipy.sparse as sp
    from pydnmfk_b200.pyDNMF import PyNMF
    from pydnmfk_b200.pyDNMFk import PyNMFk
    A = sp.random(20, 10, density=0.3, format='csr', random_state=0, dtype=np.float32)
    with pytest.raises(ValueError, match='nnsvd'):
        PyNMF(A, params=_params(init='nnsvd'))
    with pytest.raises(ValueError, match='a_storage'):
        PyNMF(A, params=_params(a_storage='bfloat16'))
    with pytest.raises(ValueError, match='PyNMFk'):
        PyNMFk(A, params=_params())
    with pytest.raises(ValueError, match='PyNMFk'):
        PyNMFk(torch.from_numpy(A.toarray()).to_sparse_csr(), params=_params())
    nmf = PyNMF.__new__(PyNMF)
    nmf._sparse = True
    with pytest.raises(ValueError, match='column_err'):
        nmf.column_err()


def test_sparse_entry_points_reject_bad_arguments_without_a_device():
    from pydnmfk_b200 import _lib as L
    one = 1
    # (row_ptr, col_idx, val, H, ldh, V, ldv, m, n, nnz, k, dtype, ws, ws_bytes, stream)
    with pytest.raises(L.DnmfError) as e:
        L.call('dnmf_sp_ah', one, one, one, one, 8, one, 80, 8, 8, 10, L.MAX_K + 1, L.F32, None, 0, None)
    assert e.value.status == -2 and 'DNMF_MAX_K' in str(e.value)
    with pytest.raises(L.DnmfError) as e:
        L.call('dnmf_sp_ah', None, None, None, None, 8, None, 8, 8, 8, 10, 4, L.F32, None, 0, None)
    assert e.value.status == -1
    with pytest.raises(L.DnmfError) as e:
        L.call('dnmf_sp_wta', one, one, one, one, 8, one, 8, 8, 8, 10, 4, 0, 7, None, 0, None)   # bad dtype
    assert e.value.status == -1
    with pytest.raises(L.DnmfError) as e:
        L.call('dnmf_sp_kl_uht', one, one, one, one, 4, one, 8, one, 4, -1, 8, 10, 4, 1e-7, L.F32, None, 0, None)
    assert e.value.status == -1
    with pytest.raises(L.DnmfError) as e:
        L.call('dnmf_sp_kl_wtu', one, one, one, None, 4, one, 8, one, 8, 8, 8, 10, 4, 1e-7, 1, L.F64, None, 0, None)
    assert e.value.status == -1
    with pytest.raises(L.DnmfError) as e:
        L.call('dnmf_sp_residual_sqnorm', one, one, one, one, 4, one, 8, 8, 8, 10, L.MAX_K + 1, one, L.F64, None, 0, None)
    assert e.value.status == -2
    with pytest.raises(L.DnmfError) as e:
        L.call('dnmf_sp_ah_residual', one, one, one, one, 4, one, 8, None, 4, 8, 8, 10, 4, one, L.F32, None, 0, None)
    assert e.value.status == -1
    with pytest.raises(L.DnmfError) as e:    # workspace missing: refused before any launch
        L.call('dnmf_sp_ah', one, one, one, one, 8, one, 8, 8, 8, 10, 4, L.F32, None, 0, None)
    assert e.value.status == -3
    with pytest.raises(L.DnmfError):
        L.sp_workspace_bytes(8, 8, 10, 4, 7)
    with pytest.raises(L.DnmfError):
        L.sp_workspace_bytes(1 << 31, 8, 10, 4, L.F32)
    # the shard, the padded factors and the chunk partials: grows with nnz, a pure function of the shape
    a = L.sp_workspace_bytes(65536, 65536, 43 * 10 ** 6, 32, L.F32)
    assert a == L.sp_workspace_bytes(65536, 65536, 43 * 10 ** 6, 32, L.F32)
    assert a > L.sp_workspace_bytes(65536, 65536, 10 ** 6, 32, L.F32) > 0
