"""``SparseShard``: a sparse data shard held on the device in compressed rows and compressed columns.

PyNMF accepts a ``scipy.sparse`` matrix or array, or a ``torch`` sparse CSR tensor (host or device), as ``A_ij``; it is
converted once into a ``SparseShard`` and every pass over A runs on the sparse kernels of ``csrc/dnmf_sparse.cu``.

Device format (include/dnmf.h, "sparse shards"):
  * CSR: ``row_ptr`` int64[m+1], ``col_idx`` int32[nnz], ``val`` [nnz];
  * CSC: ``col_ptr`` int64[n+1], ``row_idx`` int32[nnz], ``val_t`` [nnz].
``W^T A`` walks the CSC, so it needs no float atomics: the shard costs ``2 nnz (sizeof(val) + 4) + 8 (m + n + 2)`` bytes.

Canonical form: indices sorted within every row and column, duplicates summed, explicitly stored zeros removed.  The
summation order of every kernel is then a function of the matrix alone, the row / column non-zero counts (the prune
masks) are pointer differences equal to the dense path's ``(A != 0)`` counts, and no product, KL quotient or residual
changes.  Conversion is plumbing (scipy on the host, torch layout ops for torch input); scipy is imported only when a
scipy matrix is given.
"""
import numpy as np
import torch

_INT32_LIMIT = 1 << 31


def is_sparse_input(A):
    """True for the inputs ``SparseShard.from_any`` converts: a SparseShard, a scipy.sparse matrix / array, or a torch
    sparse CSR tensor."""
    if isinstance(A, SparseShard):
        return True
    if isinstance(A, torch.Tensor):
        return A.layout == torch.sparse_csr
    mod = type(A).__module__ or ''
    return mod.startswith('scipy.sparse')


def _value_dtype(dtype):
    from .device import torch_dtype
    if isinstance(dtype, torch.dtype):
        if dtype in (torch.float32, torch.float64):
            return dtype
        dtype = str(dtype).replace('torch.', '')
    return torch_dtype(dtype)       # the dense path's TypeError for anything but float32 / float64


def canonical_arrays(A):
    """``(shape, (row_ptr, col_idx, val, col_ptr, row_idx, val_t))`` of the canonical CSR and CSC of a scipy.sparse
    matrix / array or a torch sparse CSR tensor, as torch tensors on the input's device (the host for scipy input).
    Values keep the input dtype, which must be float32 or float64 (TypeError otherwise, as on the dense path)."""
    if isinstance(A, torch.Tensor):
        if A.layout != torch.sparse_csr:
            raise TypeError('torch input must be a sparse CSR tensor (layout torch.sparse_csr), got %s' % A.layout)
        _value_dtype(A.dtype)
        m, n = A.shape
        _check_shape(m, n)
        coo = A.to_sparse_coo()
        # (torch flags the COO of any CSR tensor as coalesced; a fresh tensor makes coalesce() sort and sum duplicates)
        coo = torch.sparse_coo_tensor(coo.indices(), coo.values(), (m, n)).coalesce()
        keep = coo.values() != 0
        ij, v = coo.indices()[:, keep], coo.values()[keep]
        csr = torch.sparse_coo_tensor(ij, v, (m, n)).coalesce().to_sparse_csr()
        csc = torch.sparse_coo_tensor(ij, v, (m, n)).coalesce().to_sparse_csc()
        return (m, n), (csr.crow_indices(), csr.col_indices(), csr.values(),
                        csc.ccol_indices(), csc.row_indices(), csc.values())
    import scipy.sparse as sp
    _value_dtype(A.dtype)
    m, n = A.shape
    _check_shape(m, n)
    csr = sp.csr_matrix(A, copy=True)
    csr.sum_duplicates()               # sorts the indices of every row and sums duplicates
    csr.eliminate_zeros()
    csc = csr.tocsc()
    csc.sum_duplicates()
    return (m, n), tuple(torch.from_numpy(np.ascontiguousarray(x))
                         for x in (csr.indptr, csr.indices, csr.data, csc.indptr, csc.indices, csc.data))


def _check_shape(m, n):
    if m >= _INT32_LIMIT or n >= _INT32_LIMIT:
        raise ValueError('a sparse shard must have fewer than 2^31 rows and columns, got %d x %d' % (m, n))


class SparseShard:
    """One rank's sparse shard on the device (CSR + CSC, canonical).  ``shape``, ``dtype`` (torch.float32 /
    torch.float64) and ``device`` mirror a dense tensor's attributes."""

    def __init__(self, shape, row_ptr, col_idx, val, col_ptr, row_idx, val_t):
        self.shape = (int(shape[0]), int(shape[1]))
        self.row_ptr, self.col_idx, self.val = row_ptr, col_idx, val
        self.col_ptr, self.row_idx, self.val_t = col_ptr, row_idx, val_t
        self.dtype = val.dtype
        self.device = val.device

    @property
    def nnz(self):
        return int(self.val.numel())

    def nbytes(self):
        """Device bytes of the shard: 2 nnz (sizeof(val) + 4) + 8 (m + n + 2)."""
        return sum(t.numel() * t.element_size() for t in (self.row_ptr, self.col_idx, self.val, self.col_ptr,
                                                           self.row_idx, self.val_t))

    # ---- construction --------------------------------------------------------------------------------------------
    @classmethod
    def from_any(cls, A, device=None):
        """A SparseShard on ``device`` (default: the current CUDA device) from any input ``is_sparse_input`` accepts."""
        if isinstance(A, SparseShard):
            return A
        from .device import require_cuda
        require_cuda()
        if device is None:
            device = torch.device('cuda', torch.cuda.current_device())
        shape, arrays = canonical_arrays(A)

        def t(x, dtype):
            return x.to(device=device, dtype=dtype).contiguous()
        dt = arrays[2].dtype
        it = (torch.int64, torch.int32, dt) * 2
        return cls(shape, *(t(x, d) for x, d in zip(arrays, it)))

    # ---- shard ops -------------------------------------------------------------------------------------------------
    def nnz_counts(self):
        """Non-zeros per row and per column (int64 device tensors): pointer differences."""
        return self.row_ptr[1:] - self.row_ptr[:-1], self.col_ptr[1:] - self.col_ptr[:-1]

    def compact(self, keep_rows, keep_cols):
        """The shard restricted to the kept rows and columns (int64 index tensors on the device, increasing).  The
        dropped rows and columns must be empty: compaction renumbers indices and changes no value."""
        m, n = self.shape
        rc, cc = self.nnz_counts()
        kept = int(rc[keep_rows].sum().item()) if keep_rows.numel() else 0
        kept_c = int(cc[keep_cols].sum().item()) if keep_cols.numel() else 0
        if kept != self.nnz or kept_c != self.nnz:
            raise ValueError('sparse prune would drop non-zeros: only empty rows and columns can be removed')

        def renumber(keep, size):
            new = torch.full((size,), -1, dtype=torch.int32, device=self.device)
            new[keep] = torch.arange(keep.numel(), dtype=torch.int32, device=self.device)
            return new

        def ptr_of(ptr, keep, total):
            return torch.cat([ptr[keep], ptr[total:total + 1]]).contiguous()

        row_map, col_map = renumber(keep_rows, m), renumber(keep_cols, n)
        return SparseShard((keep_rows.numel(), keep_cols.numel()),
                           ptr_of(self.row_ptr, keep_rows, m), col_map[self.col_idx.long()].contiguous(), self.val,
                           ptr_of(self.col_ptr, keep_cols, n), row_map[self.row_idx.long()].contiguous(), self.val_t)

    def to_dense(self):
        """Dense copy on the device (tests and small diagnostics only)."""
        m, n = self.shape
        return torch.sparse_csr_tensor(self.row_ptr, self.col_idx.long(), self.val, (m, n)).to_dense()
