"""``PyNMF``: the NMF driver (init -> prune -> iterate -> normalise -> relative error -> unprune).

Drop-in for ``pyDNMFk/pyDNMF.py`` (:55-239): same constructor, same ``params`` protocol and side
effects, same ``fit() -> (W, H, recon_err)``; the data shard and the factors live in HBM for the
whole fit and every arithmetic step is a libdnmf kernel (no CPU fallback).

Differences that do not change results: one persistent update object instead of a new
``nmf_algorithms_*`` per iteration (SURVEY A17); the relative error is computed by a fused
residual kernel with float64 accumulation instead of materialising ``A - W @ H`` (the reference's
fp32 ``sdot`` norm loses accuracy beyond ~2^22 elements per rank, SURVEY section 7.3).
"""
import numpy as np
import torch

from .data_io import *      # noqa: F401,F403  (star-import chain kept like the reference)
from .dist_nmf import *     # noqa: F401,F403
from .utils import *        # noqa: F401,F403
from . import device as D
from .dist_nmf import nmf_algorithms_1D, nmf_algorithms_2D
from .utils import data_operations, determine_block_params, var_init, comm_timing
from .dist_comm import MPI
from .graphs import StepGraphs, graphs_enabled
from .sparse import SparseShard, is_sparse_input


_A_STORAGE = {'float16': torch.float16, 'bfloat16': torch.bfloat16}


def a_storage_dtype(a_storage, A):
    """The torch dtype the data shard ``A`` is stored in on the device for ``params.a_storage``, or None (``a_storage`` None:
    the data dtype, nothing changes).  With 'float16' / 'bfloat16' only the shard is held in 16 bits -- the fit is the
    float32 fit of the rounded matrix -- so the data must be float32, or a CUDA tensor already in that 16-bit format.
    Raises ValueError otherwise.  Needs no device."""
    if a_storage is None:
        return None
    if a_storage not in _A_STORAGE:
        raise ValueError("params.a_storage must be None, 'float16' or 'bfloat16', not %r" % (a_storage,))
    want = _A_STORAGE[a_storage]
    if isinstance(A, torch.Tensor):
        if A.dtype == torch.float32 or (A.dtype == want and A.is_cuda):
            return want
        got = str(A.dtype).replace('torch.', '') + ('' if A.is_cuda else ' (host tensor)')
    else:
        got = str(np.asarray(A).dtype)
        if got == 'float32':
            return want
    raise ValueError('params.a_storage=%r needs float32 data (or a CUDA tensor already in %s), got %s'
                     % (a_storage, a_storage, got))


def draw_rand_factors(topo, p_c, rank, a_shape, factor_shape, k, dt):
    """Host draws of the 'rand' initialisation in the reference's exact order (pyDNMF.py:110-129):
    2-D: W_ij = rand(m_loc, k) then H_ij = rand(k, n_loc) on every rank; 1-D row grid: W_i on every
    rank, then the replicated H on rank 0 only; 1-D column grid mirrored.  Returns (W, H) with None
    for a replicated factor this rank must receive by broadcast."""
    if topo == '2d':
        W = np.random.rand(factor_shape[0], k).astype(dt)
        H = np.random.rand(k, factor_shape[1]).astype(dt)
    elif p_c == 1:
        W = np.random.rand(a_shape[0], k).astype(dt)
        H = np.random.rand(k, a_shape[1]).astype(dt) if rank == 0 else None
    else:
        H = np.random.rand(k, a_shape[1]).astype(dt)
        W = np.random.rand(a_shape[0], k).astype(dt) if rank == 0 else None
    return W, H


def _check_sparse_params(params):
    """What a sparse A_ij does not support; raised before anything reaches the device."""
    if getattr(params, 'a_storage', None) is not None:
        raise ValueError('params.a_storage does not apply to a sparse A_ij (its values are stored as float32 / float64)')
    if getattr(params, 'init', None) == 'nnsvd':
        raise ValueError("init='nnsvd' is not supported for a sparse A_ij (DistSVD deflates a dense copy of A); use "
                         "init='rand' or given factors")


class PyNMF():
    r"""Distributed NMF decomposition of the matrix whose local shard is ``A_ij``.

    Parameters (identical to the reference, pyDNMF.py:9-52): ``A_ij`` local shard (numpy array or
    CUDA tensor), ``factors`` optional ``[W, H]`` shards, ``params`` attribute bag with ``init,
    comm1, comm, k, p_r, p_c (or grid), row_comm, col_comm, verbose`` and optional ``itr, norm,
    method, prune, W_update``, ``a_storage``.

    ``A_ij`` may also be sparse: a ``scipy.sparse`` matrix / array (results come back as numpy arrays) or a ``torch``
    sparse CSR tensor (results come back as tensors).  The shard is then held on the device as CSR + CSC
    (``sparse.SparseShard``) and every pass reads only its non-zeros; FRO-MU, KL-MU, HALS and BCD, pruning, given
    factors, ``err_monitor`` and CUDA-graph replay work as for dense data.  ``init='nnsvd'``, ``a_storage`` and
    ``column_err`` raise ValueError for sparse data.

    ``params.a_storage`` = 'float16' / 'bfloat16' holds only the data shard in 16 bits on the device (half the memory and
    half the bytes each pass streams); W, H, every update and every reduction stay float32.  The fit is then the float32
    fit of the rounded matrix (round to nearest even): ``recon_err`` is relative to the rounded matrix, prune masks come
    from it (an entry that underflows to 0 is a zero), W and H come back as float32 (float64 after un-pruning).  Float32
    data only; 'float16' raises ValueError when an entry overflows (|a| > 65504); ``init='nnsvd'`` is not supported.
    """

    @comm_timing()
    def __init__(self, A_ij, factors=None, save_factors=False, params=None):
        self.params = params
        self._sparse = is_sparse_input(A_ij)
        if self._sparse:
            _check_sparse_params(params)
        self._numpy_in = not isinstance(A_ij, (torch.Tensor, SparseShard))
        self._a_dtype = a_storage_dtype(getattr(params, 'a_storage', None), A_ij)
        if self._a_dtype is not None:
            self._np_dtype = np.dtype(np.float32)                   # factors, eps and recon_err stay float32
        else:
            self._np_dtype = np.dtype(A_ij.dtype) if self._numpy_in else np.dtype(str(A_ij.dtype).replace('torch.', ''))
        self.m_loc, self.n_loc = A_ij.shape
        self.init = self.params.init if self.params.init else 'rand'
        if self._a_dtype is not None and self.init == 'nnsvd':
            raise ValueError("params.a_storage does not support init='nnsvd' (DistSVD deflates a copy of A in the data "
                             "dtype); use init='rand' or given factors")
        if "grid" in vars(self.params) and self.params.grid:
            self.p_r, self.p_c, self.k = self.params.grid[0], self.params.grid[1], self.params.k
        else:
            self.p_r, self.p_c, self.k = self.params.p_r, self.params.p_c, self.params.k
        self.comm1 = self.params.comm1
        self.cart_1d_row, self.cart_1d_column, self.comm = self.params.row_comm, self.params.col_comm, self.params.comm
        self.verbose = self.params.verbose if self.params.verbose else False
        self.rank = self.comm1.rank
        self.eps = np.finfo(self._np_dtype).eps                     # pyDNMF.py:68
        self.params.eps = self.eps
        self.norm = var_init(self.params, 'norm', default='kl')
        self.method = var_init(self.params, 'method', default='mu')
        self.prune = var_init(self.params, 'prune', default=True)
        self.save_factors = save_factors
        self.params.itr = var_init(self.params, 'itr', default=5000)
        self.itr = self.params.itr
        self.W_start, self.W_end = 0, 0
        self.H_start, self.H_end = 0, 0
        try:
            self.W_update = self.params.W_update
        except AttributeError:
            self.params.W_update = True
        self.p = self.p_r * self.p_c
        self.topo = '2d' if (self.p_r != 1 and self.p_c != 1) else '1d'
        self.params.topo = self.topo
        self.ops = D.default_ops()
        self._tdtype = D.torch_dtype(self._np_dtype)
        # the shard goes to HBM once and stays there.  From page-locked host memory the copy runs asynchronously while
        # the host draws the initial factors (the RNG replay below is ~0.1 s at 65536 x 32); the constructor waits for it
        # before returning, so the caller's buffer is never read after this call
        if self._sparse:
            self.A_ij = SparseShard.from_any(A_ij)
        elif self._a_dtype is not None:
            self.A_ij = D.to_device_a16(A_ij, self._a_dtype)
        else:
            self.A_ij = D.to_device(A_ij, self._tdtype, non_blocking=True)
        self.data_op = data_operations(self.A_ij, self.params)
        self.params = self.data_op.params
        if factors is not None:
            W0 = D.to_device(factors[0], self._tdtype)               # .astype(A.dtype), pyDNMF.py:90-96
            H0 = D.to_device(factors[1], self._tdtype)
            W0, H0 = W0.clone(), H0.clone()
        else:
            W0, H0 = self.init_factors()
        self._set_factors(W0, H0)
        if self.prune:
            W, H = self._get_factors()
            self.A_ij, W, H = self.data_op.prune_all(W, H)
            self._set_factors(W, H)
        if self._numpy_in:
            torch.cuda.current_stream().synchronize()

    def _set_factors(self, W, H):
        if self.topo == '2d':
            self.W_ij, self.H_ij = W, H
        else:
            self.W_i, self.H_j = W, H

    def _get_factors(self):
        return (self.W_ij, self.H_ij) if self.topo == '2d' else (self.W_i, self.H_j)

    @comm_timing()
    def init_factors(self):
        """rand / nnsvd initialisation.  Draws come from this process's global legacy numpy stream in
        the reference's order (pyDNMF.py:107-135; SURVEY section 8a P3) so a seeded run reproduces
        the reference's starting point bit for bit."""
        dt = self._np_dtype
        if self.init == 'rand':
            W, H = draw_rand_factors(self.topo, self.p_c, self.rank, (self.m_loc, self.n_loc),
                                     (self.params.m_loc, self.params.n_loc), self.k, dt)
            if self.topo == '1d':
                if self.p_c == 1:
                    H = self._bcast_factor(H, (self.k, self.n_loc))
                else:
                    W = self._bcast_factor(W, (self.m_loc, self.k))
            return D.to_device(W, self._tdtype), D.to_device(H, self._tdtype)
        elif self.init == 'nnsvd':
            if self.topo == '1d':
                # pyDNMF.py:131-134.  The reference keeps DistSVD's float64 factors (numpy then promotes the whole fit
                # to float64 even for float32 data); the device path casts them to the data dtype like every other
                # initialisation, parity is asserted at the fp32 tolerance.
                from .dist_svd import DistSVD
                W, H = DistSVD(self.params, self.A_ij).nnsvd(flag=1, verbose=0)
                return W.to(self._tdtype).contiguous(), H.to(self._tdtype).contiguous()
            raise Exception('NNSVD init only available for 1D topology, please try with 1d topo.')
        raise Exception('unknown init: %s' % self.init)

    def _bcast_factor(self, X, shape):
        """Rank 0's replicated factor to everyone (pyDNMF.py:121,129)."""
        if self.comm1.size == 1:
            return X
        t = D.to_device(X if X is not None else np.empty(shape, dtype=self._np_dtype), self._tdtype)
        return self.comm1.bcast_(t, root=0)

    def _resident_ok(self):
        """Whole-fit on-chip path (dnmf_mu_fit_resident): single-process grid, MU, shard + factors fit in one SM."""
        W, H = self._get_factors()
        # (the on-chip kernel reads A in the factor dtype: a 16-bit shard takes the per-kernel path)
        return (self._a_dtype is None and not self._sparse and self.comm1.size == 1 and self.method.lower() == 'mu'
                and self.norm.lower() in ('fro', 'kl')
                and var_init(self.params, 'resident_fit', True) and self.itr >= 1 and W.shape[0] > 0 and H.shape[1] > 0
                and self.ops.resident_fit_fits(W.shape[0], H.shape[1], self.k, self.norm, self._tdtype))

    def _run_loop(self):
        """The ``itr`` update steps of pyDNMF.py:151-172 (update + every-10th clamp) on the resident factors."""
        W, H = self._get_factors()
        if self._resident_ok():
            self.ops.mu_fit_resident([self.A_ij], [W], [H], self.norm, self.params.W_update, 0, self.itr, self.eps)
            return
        Alg = nmf_algorithms_2D if self.topo == '2d' else nmf_algorithms_1D
        alg = Alg(self.A_ij, W, H, params=self.params)
        self._alg = alg

        def clamp():                                                    # pyDNMF.py:155-157 / :170-172
            self.ops.clamp_min(H, self.eps)
            self.ops.clamp_min(W, self.eps)

        # iteration 0 runs eagerly; the rest replay a captured CUDA graph of the same launches (see graphs.py)
        use_graph = (self.itr >= 4 and var_init(self.params, 'cuda_graph', True)
                     and graphs_enabled(self.comm1, self.method))
        sg = StepGraphs(alg.update, clamp) if use_graph else None
        for i in range(self.itr):
            if self.method.lower() == 'bcd':
                i = self.itr - 1                                        # pyDNMF.py:152
            if sg is not None and i >= 1:
                if i % 10 == 0:
                    sg.clamped()
                else:
                    sg.plain()
            else:
                alg.update()
                if i % 10 == 0:
                    clamp()
            if i == self.itr - 1:
                break
        sg = None                              # drop the captured graphs (and their NCCL nodes) with the loop
        if getattr(alg, '_px', None) is not None:
            alg._px.check()                    # a peer that died mid-exchange must not go unnoticed

    def _finish(self):
        """What the reference does on the last iteration (pyDNMF.py:158-166,173-181): normalise, relative error,
        optional save, un-prune; returns ``(W, H, recon_err)``."""
        W, H = self._get_factors()
        W, H = self.normalize_features(W, H)
        self._set_factors(W, H)
        if self.topo == '2d' and not hasattr(self, '_alg'):
            self._alg = nmf_algorithms_2D(self.A_ij, W, H, params=self.params)
        self.relative_err()
        if getattr(self.params, 'err_monitor', False) and getattr(self, '_alg', None) is not None:
            # opt-in: relative error after every iteration from the trace identity (no extra pass over A)
            self.err_history = self._alg.monitor_history()
        if self.verbose == True:  # noqa: E712
            if self.rank == 0:
                print('relative error is:', self.recon_err)
        if self.save_factors:
            data_write(self.params).save_factors([W.cpu().numpy(), H.cpu().numpy()])  # noqa: F405
        if self.topo == '2d':
            self.comm.Free()
        if self.prune:
            W, H = self.data_op.unprune_factors(W, H)
        return self._to_host(W), self._to_host(H), self.recon_err

    @comm_timing()
    def fit(self):
        r"""Run ``itr`` update steps; returns ``(W, H, recon_err)`` as host arrays (W, H in the data
        dtype, or float64 after un-pruning -- utils.py:195,198) and a numpy scalar."""
        if self.itr < 1:
            return None
        self._run_loop()
        return self._finish()

    def _to_host(self, t):
        return t.cpu().numpy() if self._numpy_in else t

    @comm_timing()
    def normalize_features(self, Wall, Hall):
        """W /= colsum(W) + eps ; H *= colsum(W)  (pyDNMF.py:185-194; SURVEY A4)."""
        s = self.ops.colsum(Wall)
        if self.topo == '2d' or self.p_r != 1:
            s = self.comm1.allreduce_(s)
        self.ops.normalize(Wall, Hall, s, self.eps)
        return Wall, Hall

    @comm_timing()
    def cart_2d_collect_factors(self):
        """H_ij -> H_j over the row communicator, W_ij -> W_i over the column one (pyDNMF.py:197-202)."""
        self.H_j = self._alg._gather_H(self.H_ij)
        self.W_i = self._alg._gather_W(self.W_ij)

    @comm_timing()
    def relative_err(self):
        """||A - W H||_F / ||A||_F over the whole grid (pyDNMF.py:205-218), one fused pass over A."""
        if self.topo == '2d':
            self.cart_2d_collect_factors()
        sq = self.ops.residual_sqnorm(self.A_ij, self.W_i, self.H_j)
        sq = self.comm1.allreduce_(sq).cpu().numpy()
        self.glob_norm_err = np.sqrt(sq[0])
        self.glob_norm_A = np.sqrt(sq[1])
        self.recon_err = self._np_dtype.type(self.glob_norm_err / self.glob_norm_A)

    @comm_timing()
    def dist_norm(self, X, proc=-1, norm='fro', axis=None):
        """Distributed Frobenius norm (pyDNMF.py:212-218)."""
        sq = self.ops.sqnorm(D.to_device(X, self._tdtype))
        if proc != 1:
            sq = self.comm1.allreduce_(sq)
        return np.sqrt(sq.item())

    @comm_timing()
    def column_err(self):
        """Per-column relative L2 error over the global column range (pyDNMF.py:221-239)."""
        if self._sparse:
            raise ValueError('column_err is not available for a sparse A_ij')
        dtr_blk = determine_block_params(self.comm1, (self.p_r, self.p_c), (self.params.m, self.params.n))
        dtr_blk_idx = dtr_blk.determine_block_index_range_asymm()
        num, den = self.ops.column_err(self.A_ij, self.W_i, self.H_j)
        n_here = num.shape[0]
        col_num = torch.zeros(self.params.n, dtype=torch.float64, device=num.device)
        col_den = torch.zeros(self.params.n, dtype=torch.float64, device=num.device)
        lo = dtr_blk_idx[0][1]
        col_num[lo:lo + n_here] = num
        col_den[lo:lo + n_here] = den
        col_num = self.comm1.allreduce_(col_num)
        col_den = self.comm1.allreduce_(col_den)
        return np.sqrt((col_num / col_den).cpu().numpy())
