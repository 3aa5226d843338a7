"""One NMF update step on a 1-D or 2-D processor grid -- device-resident.

Mirrors the public surface of ``pyDNMFk/dist_nmf.py`` (``nmf_algorithms_2D`` :7-579,
``nmf_algorithms_1D`` :582-1047): same class names, constructor, ``update()`` dispatch and
error messages, same helper names (``global_gram``, ``global_mm``, ``AH_glob``, ``ATW_glob``,
``gather_W_H``, ``UHT_glob``, ``WTU_glob``, ``sum_axis`` / ``sum_along_axis``, ``glob_UX``,
``Fro_MU_update[_W/_H]``, ``KL_MU_update[_W/_H]``, ``FRO_HALS_update[_W/_H]``,
``FRO_BCD_update``, ``globalSqNorm``, ``initWandH``).

What differs is *where* the arithmetic runs: every numpy expression of the reference is one
hand-written sm_100a kernel behind ``libdnmf.so`` (see ``device.DeviceOps``), the shard ``A_ij``
and both factors stay in HBM for the whole fit, the KL path never materialises ``W @ H``,
and MPI collectives become NCCL collectives on communicators owned by the library
(``dist_comm``), or -- for the H half-step of row grids -- one exchange over NVLink peer memory
(``peer.PeerExchange``).  On the tcgen05 path a MU half-step is two launches: the A-streaming
pass and an update kernel that sums the pass's split-K partials itself (``DeviceOps.*_p``).  The
redundant gathers of the reference's 2-D KL/HALS paths (SURVEY A10) are dropped; results are
unaffected.

Inputs may be numpy arrays (uploaded once per object, results downloaded by ``update()``) or
CUDA tensors (updated in place, returned as tensors) -- ``PyNMF.fit`` uses the latter.
"""
import numpy as np
import torch

from . import device as D
from . import peer
from .utils import norm, comm_timing, parse, var_init  # noqa: F401  (re-exported like the reference)
from .dist_comm import MPI  # noqa: F401


def _sqrt_host(t):
    return float(np.sqrt(t.item()))


class _AlgBase:
    """State shared by the 1-D and 2-D variants."""

    def _setup(self, A_ij, W, H, params):
        self.params = params
        self.m, self.n, self.p_r, self.p_c, self.k = params.m, params.n, params.p_r, params.p_c, params.k
        self.comm1 = params.comm1
        self.comm = params.comm1
        self.norm = params.norm
        self.method = params.method
        self.eps = params.eps
        self.p = self.p_r * self.p_c
        self.W_update = params.W_update
        self.rank = self.comm1.rank
        self.ops = D.default_ops()
        self._A_orig = A_ij
        self._numpy_io = not isinstance(A_ij, torch.Tensor)
        self._np_dtype = A_ij.dtype if self._numpy_io else None
        A = D.to_device(A_ij)
        # factor dtype: the data dtype, or float32 when the shard is stored in 16 bits (PyNMF's params.a_storage)
        self.fdtype = D.out_dtype(A.dtype)
        return A, D.to_device(W, self.fdtype), D.to_device(H, self.fdtype)

    def _out(self, W, H):
        if self._numpy_io:
            torch.cuda.current_stream().synchronize()
            return W.cpu().numpy(), H.cpu().numpy()
        return W, H

    def _dispatch(self):
        if self.norm.upper() == 'FRO':
            if self.method.upper() == 'MU':
                self.Fro_MU_update(self.W_update)
            elif self.method.upper() == 'HALS':
                self.FRO_HALS_update(self.W_update)
            elif self.method.upper() == 'BCD':
                self.FRO_BCD_update(self.W_update, itr=self.params.itr)
            else:
                raise Exception('Not a valid method: Choose (mu/hals/bcd)')
        elif self.norm.upper() == 'KL':
            if self.method.upper() == 'MU':
                self.KL_MU_update(self.W_update)
            else:
                raise Exception('Not a valid method: Choose (mu)')
        else:
            raise Exception('Not a valid norm: Choose (fro/kl)')

    # ---- per-iteration error monitor (trace identity) ---------------------------------------------------
    # ||A - W H||^2 = ||A||^2 - 2 <W, A H^T> + <W^T W, H H^T>.  At the top of a FRO-MU W half-step H H^T and A H^T of the
    # current H are at hand and W^T W of the current W was formed by the preceding H half-step: the error of the state the
    # previous iteration left costs two factor-sized inner products (dnmf_trace_terms), no pass over A.  Samples are
    # appended to a device history through a device-side counter, so CUDA-graph replays of the step keep recording.
    def _monitor_setup(self):
        self._mon = None
        if not getattr(self.params, 'err_monitor', False) or self.norm.upper() != 'FRO' or self.method.upper() != 'MU':
            return
        slots = int(getattr(self.params, 'itr', 1)) + 1
        dev = self.A_ij.device
        m = type('Monitor', (), {})()
        m.hist = torch.zeros((slots, 2), dtype=torch.float64, device=dev)
        m.counter = torch.zeros(1, dtype=torch.int64, device=dev)
        m.wtw = torch.zeros((self.k, self.k), dtype=self.fdtype, device=dev)   # persistent: captured graphs keep its address
        m.have_wtw = False
        m.anorm2 = self._sqnorm_dev(self.A_ij)            # global ||A||^2, float64 device scalar
        m.w_sharded = (self.p > 1) and not (self.p_r == 1)   # <W, A H^T> is a sum over the ranks that own W rows
        self._mon = m
        self.params.err_monitor_state = m

    def _monitor_sample(self, W, AH, HHT):
        m = self._mon
        if m is None or not m.have_wtw or self.W_update != True:  # noqa: E712  (no W^T W of the current W yet)
            return
        # every rank appends ITS pair (graph-replay safe); on grids that shard W the histories are summed once at the end
        self.ops.trace_terms(W, AH, m.wtw, HHT, out=m.hist, slot_counter=m.counter)

    def _monitor_keep(self, W_TW):
        if self._mon is not None:
            self._mon.wtw.copy_(W_TW)
            self._mon.have_wtw = True

    def monitor_history(self):
        """Relative errors ||A - W H||_F / ||A||_F recorded so far (numpy float64): entry i is the state at the top of
        iteration i + 1, i.e. the result of iteration i."""
        m = getattr(self, '_mon', None)
        if m is None:
            return None
        n = min(int(m.counter.item()), m.hist.shape[0])
        hist = m.hist
        if m.w_sharded:
            # <W, A H^T> is a sum over the ranks that own W rows; <W^T W, H H^T> is global on every rank already
            hist = self.comm1.allreduce_(m.hist.clone())
            hist[:, 1] /= float(self.comm1.size)
        h = hist[:n].cpu().numpy()
        a2 = float(m.anorm2.item())
        return np.sqrt(np.maximum(a2 - 2.0 * h[:, 0] + h[:, 1], 0.0) / a2)

    # ---- BCD shared by both grids (dist_nmf.py:503-579, :971-1047) ---------------------------------
    # The Lipschitz bounds, objective, momentum weights and the accept / restore decision live in a float64 device
    # vector (csrc/dnmf_bcd.cu): one iteration is a fixed sequence of launches with no host round trip, replayed as a
    # CUDA graph.  H_old H_old^T and A H_old^T of the restore branch are the copies kept when H_old was accepted.
    def bcd_begin(self):
        """initWandH (dist_nmf.py:482-501 / :951-969): scale the factors, form H H^T and A H^T, obj_old = ||A||^2 / 2."""
        ops = self.ops
        W, H = self._W(), self._H()
        Xnorm = self._sqnorm_dev(self.A_ij)
        nW = float(self._sqnorm_dev(W, 'w').item())
        nH = float(self._sqnorm_dev(H, 'h').item())
        scale = np.sqrt(np.sqrt(float(Xnorm.item())))
        b = self._bcd = type('BcdState', (), {})()
        b.W_old, b.H_old = torch.empty_like(W), torch.empty_like(H)
        ops.axpby(b.W_old, W, W, scale / np.sqrt(nW), 0.0)
        ops.axpby(b.H_old, H, H, scale / np.sqrt(nH), 0.0)
        b.Wm, b.Hm = b.W_old.clone(), b.H_old.clone()
        b.HHT = self._gram_H(b.H_old)
        b.AHT = self._AH(b.H_old)
        b.HHT_kept, b.AHT_kept = b.HHT.clone(), b.AHT.clone()
        b.state = torch.zeros(16, dtype=torch.float64, device=W.device)
        ops.bcd_state(0, b.state, Xnorm)
        self.params.rw = 1

    def bcd_step(self):
        """One iteration of dist_nmf.py:996-1047 on the device-resident state."""
        ops, b = self.ops, self._bcd
        W, H = self._W(), self._H()
        ops.bcd_state(1, b.state, ops.sqnorm(b.HHT))
        ops.bcd_pg_w_dev(W, b.Wm, b.AHT, b.HHT, b.state, 0)
        ops.div_cols(W, self._colsum_W(W, force=False))
        WTW = self._gram_W(W)
        ops.bcd_state(2, b.state, ops.sqnorm(WTW))
        WTA, yT = self._WTA(W)
        ops.bcd_pg_h_dev(H, b.Hm, WTA, WTW, b.state, 2, y_transposed=yT)
        HHT = self._gram_H(H)
        AHT, res = self._AH_and_residual(W, H)
        b.HHT.copy_(HHT)
        b.AHT.copy_(AHT)
        ops.bcd_state(3, b.state, res)
        ops.bcd_advance(W, b.Wm, b.W_old, b.state, 0)
        ops.bcd_advance(H, b.Hm, b.H_old, b.state, 1)
        ops.bcd_keep(b.HHT, b.HHT_kept, b.state)
        ops.bcd_keep(b.AHT, b.AHT_kept, b.state)

    def _AH_and_residual(self, W, H):
        """A H^T and the global ||A - W H||^2 (float64 device scalar in element 0)."""
        return self._AH(H), self._residual_global(W, H)

    def _bcd_loop(self, itr):
        from .graphs import StepGraphs, graphs_enabled
        self.bcd_begin()
        use_graph = itr >= 4 and graphs_enabled(self.comm1, 'mu') and getattr(self.params, 'cuda_graph', True)
        sg = None
        for i in range(itr):
            if use_graph and i >= 1:
                if sg is None:
                    sg = StepGraphs(self.bcd_step, lambda: None)
                sg.plain()
            else:
                self.bcd_step()
        sg = None


class nmf_algorithms_2D(_AlgBase):
    """Distributed NMF step on a 2-D p_r x p_c grid (dist_nmf.py:7-579).

    Per rank: ``A_ij`` (m/p_r x n/p_c), ``W_ij`` (m/p x k), ``H_ij`` (k x n/p)."""

    @comm_timing()
    def __init__(self, A_ij, W_ij, H_ij, params=None):
        self.A_ij, self.W_ij, self.H_ij = self._setup(A_ij, W_ij, H_ij, params)
        self.cartesian1d_row, self.cartesian1d_column = params.row_comm, params.col_comm
        self.comm = params.comm
        self.local_W_m = self.W_ij.shape[0]
        self.local_H_n = self.H_ij.shape[1]
        # shard sizes of every member (ragged grids / pruned shards): exchanged once, integers
        self._w_sizes = [int(s) for s in self.cartesian1d_column.allgather(int(self.local_W_m))]
        self._h_sizes = [int(s) for s in self.cartesian1d_row.allgather(int(self.local_H_n))]
        self.W_i = None
        self.H_j = None
        self._monitor_setup()

    def _W(self):
        return self.W_ij

    def _H(self):
        return self.H_ij

    def update(self):
        """One update of W_ij and H_ij (dist_nmf.py:66-92)."""
        self._dispatch()
        return self._out(self.W_ij, self.H_ij)

    # ---- distributed building blocks -------------------------------------------------------
    @comm_timing()
    def global_gram(self, A):
        """A^T A summed over all ranks (dist_nmf.py:94-116); ``A`` is W_ij or H_ij.T."""
        A = D.to_device_view(A, self.fdtype)
        G = self.ops.gram(A, trans=False) if A.is_contiguous() else self.ops.gram(A.t().contiguous(), trans=True)
        return self.comm1.allreduce_(G)

    def _gram_W(self, W):
        return self.comm1.allreduce_(self.ops.gram(W, trans=False))

    def _gram_H(self, H):
        return self.comm1.allreduce_(self.ops.gram(H, trans=True))

    @comm_timing()
    def gather_W_H(self, gW=True, gH=True):
        """H_ij -> H_j over the row communicator, W_ij -> W_i over the column communicator
        (dist_nmf.py:267-291)."""
        if gH:
            self.H_j = self._gather_H(self.H_ij)
        if gW:
            self.W_i = self._gather_W(self.W_ij)

    def _gather_H(self, H_ij):
        # gather the transposed shards (n_loc x k): concatenation along rows == hstack of H shards
        Ht = self.cartesian1d_row.allgather_cat(H_ij.t().contiguous(), self._h_sizes)
        return Ht.t().contiguous()

    def _gather_W(self, W_ij):
        return self.cartesian1d_column.allgather_cat(W_ij, self._w_sizes)

    def _AH(self, H_ij):
        H_j = self._gather_H(H_ij)
        V = self.ops.ah(self.A_ij, H_j)
        return self.cartesian1d_column.reduce_scatter_rows(V, self._w_sizes)

    def _WTA(self, W_ij):
        W_i = self._gather_W(W_ij)
        Yt = self.ops.wta(self.A_ij, W_i, transposed_out=True)
        return self.cartesian1d_row.reduce_scatter_rows(Yt, self._h_sizes), True

    @comm_timing()
    def AH_glob(self, H_ij=None):
        """A H^T: allgather(row comm) -> skinny GEMM -> reduce-scatter(column comm) (dist_nmf.py:174-205)."""
        return self._AH(self.H_ij if H_ij is None else D.to_device(H_ij, self.fdtype))

    @comm_timing()
    def ATW_glob(self):
        """W^T A as a k x n/p view: allgather(column comm) -> skinny GEMM emitted directly in the
        transposed reduce-scatter layout -> reduce-scatter(row comm) (dist_nmf.py:144-172)."""
        Yt, _ = self._WTA(self.W_ij)
        return Yt.t()

    @comm_timing()
    def UHT_glob(self):
        """(A / (W_i H_j + eps)) H_j^T, fused, then reduce-scatter (dist_nmf.py:320-343)."""
        V = self.ops.kl_uht(self.A_ij, self.W_i, self.H_j, self.eps)
        return self.cartesian1d_column.reduce_scatter_rows(V, self._w_sizes)

    @comm_timing()
    def WTU_glob(self):
        """W_i^T (A / (W_i H_j + eps)), fused, then reduce-scatter (dist_nmf.py:293-318)."""
        Yt = self.ops.kl_wtu(self.A_ij, self.W_i, self.H_j, self.eps, transposed_out=True)
        return self.cartesian1d_row.reduce_scatter_rows(Yt, self._h_sizes).t()

    @comm_timing()
    def sum_axis(self, dat, axis):
        """dat.sum(axis) all-reduced over the world (dist_nmf.py:345-349)."""
        s = self.ops.colsum(dat) if axis == 0 else self.ops.rowsum(dat)
        return self.comm1.allreduce_(s)

    # ---- FRO / MU -----------------------------------------------------------------------------
    def Fro_MU_update_H(self):
        """dist_nmf.py:207-225."""
        W_TW = self._gram_W(self.W_ij)
        self._monitor_keep(W_TW)
        Yt, _ = self._WTA(self.W_ij)
        self.ops.mu_update_h(self.H_ij, Yt, W_TW, self.eps, y_transposed=True)

    def Fro_MU_update_W(self):
        """dist_nmf.py:227-245."""
        HH_T = self._gram_H(self.H_ij)
        AH = self._AH(self.H_ij)
        self._monitor_sample(self.W_ij, AH, HH_T)
        self.ops.mu_update_w(self.W_ij, AH, HH_T, self.eps)

    def Fro_MU_update(self, W_update=True):
        """dist_nmf.py:247-263: W first, then H with the new W."""
        if W_update == True:  # noqa: E712 (same test as the reference)
            self.Fro_MU_update_W()
        self.Fro_MU_update_H()

    # ---- KL / MU ------------------------------------------------------------------------------
    def KL_MU_update_W(self):
        """dist_nmf.py:351-369."""
        x2 = self.sum_axis(self.H_ij, axis=1)
        self.gather_W_H()
        sk = self.UHT_glob()
        self.ops.kl_update_w(self.W_ij, sk, x2, self.eps)

    def KL_MU_update_H(self):
        """dist_nmf.py:371-389."""
        x1 = self.sum_axis(self.W_ij, axis=0)
        self.gather_W_H()
        Yt = self.ops.kl_wtu(self.A_ij, self.W_i, self.H_j, self.eps, transposed_out=True)
        Yt = self.cartesian1d_row.reduce_scatter_rows(Yt, self._h_sizes)
        self.ops.kl_update_h(self.H_ij, Yt, x1, self.eps, y_transposed=True)

    def KL_MU_update(self, W_update=True):
        """dist_nmf.py:391-407."""
        if W_update == True:  # noqa: E712
            self.KL_MU_update_W()
        self.KL_MU_update_H()

    # ---- FRO / HALS -----------------------------------------------------------------------------
    def FRO_HALS_update_W(self):
        """dist_nmf.py:411-432: Gauss-Seidel over columns, global column norm after each."""
        HHT = self._gram_H(self.H_ij)
        AH = self._AH(self.H_ij)
        for kk in range(self.k):
            sq = self.ops.hals_w_col(self.W_ij, AH, HHT, kk, self.eps)
            if self.p_r != 1:
                sq = self.comm1.allreduce_(sq)
            self.ops.div_col(self.W_ij, kk, sq)

    def FRO_HALS_update_H(self):
        """dist_nmf.py:434-452."""
        WTW = self._gram_W(self.W_ij)
        Yt, _ = self._WTA(self.W_ij)
        self.ops.hals_h(self.H_ij, Yt, WTW, self.eps, y_transposed=True)

    def FRO_HALS_update(self, W_update=True):
        """dist_nmf.py:454-470."""
        if W_update == True:  # noqa: E712
            self.FRO_HALS_update_W()
        self.FRO_HALS_update_H()

    # ---- FRO / BCD ------------------------------------------------------------------------------
    def _sqnorm_global(self, X, which=None):
        return float(self.comm1.allreduce_(self.ops.sqnorm(X)).item())

    @comm_timing()
    def globalSqNorm(self, comm, X):
        """Global squared Frobenius norm (dist_nmf.py:474-480)."""
        return self._sqnorm_global(D.to_device(X, self.fdtype))

    def _colsum_W(self, W, force):
        return self.comm1.allreduce_(self.ops.colsum(W))

    def _residual_global(self, W, H):
        W_i, H_j = self._gather_W(W), self._gather_H(H)
        return self.comm1.allreduce_(self.ops.residual_sqnorm(self.A_ij, W_i, H_j))

    def _sqnorm_dev(self, X, which=None):
        return self.comm1.allreduce_(self.ops.sqnorm(X))

    def _AH_and_residual(self, W, H):
        W_i, H_j = self._gather_W(W), self._gather_H(H)
        V, res = self.ops.ah_residual(self.A_ij, W_i, H_j)
        return self.cartesian1d_column.reduce_scatter_rows(V, self._w_sizes), self.comm1.allreduce_(res)

    def initWandH(self):
        """dist_nmf.py:482-501: scaled factors, H H^T, A H^T and obj_old, left on the device (see bcd_begin)."""
        self.bcd_begin()

    def FRO_BCD_update(self, W_update=True, itr=1000):
        """dist_nmf.py:503-579 (its own ``itr`` loop; ignores W_update, SURVEY A11)."""
        self._bcd_loop(itr)


class nmf_algorithms_1D(_AlgBase):
    """Distributed NMF step on a 1-D grid (dist_nmf.py:582-1047).

    Row grid (p_c = 1): ``A_ij`` is an m/p_r x n block, ``W_i`` its m/p_r x k rows, ``H_j``
    (k x n) is replicated.  Column grid (p_r = 1) is the mirror image."""

    def __init__(self, A_ij, W_i, H_j, params=None):
        self.A_ij, self.W_i, self.H_j = self._setup(A_ij, W_i, H_j, params)
        self.local_W_m = self.W_i.shape[0]
        self.local_H_n = self.H_j.shape[1]
        # row grid: the H half-step runs as one exchange over peer memory instead of two all-reduces (peer.py)
        self._px = None
        if self.p_c == 1 and self.p_r > 1 and self.comm1.size == self.p_r and self.H_j.stride(1) == 1:
            self._px = peer.get(self.comm1, self.H_j.shape[1], self.k, self.H_j.dtype)
        self._monitor_setup()
        if self._mon is not None:
            self._px = None          # the monitor needs the global W^T W, which the peer exchange never materialises

    def _W(self):
        return self.W_i

    def _H(self):
        return self.H_j

    def update(self):
        """One update of W_i and H_j (dist_nmf.py:634-660)."""
        self._dispatch()
        return self._out(self.W_i, self.H_j)

    # ---- distributed building blocks -------------------------------------------------------
    @comm_timing()
    def global_gram(self, A, p=1):
        """A^T A, all-reduced iff p != 1 (dist_nmf.py:662-685)."""
        A = D.to_device_view(A, self.fdtype)
        G = self.ops.gram(A, trans=False) if A.is_contiguous() else self.ops.gram(A.t().contiguous(), trans=True)
        return self.comm1.allreduce_(G) if p != 1 else G

    @comm_timing()
    def global_mm(self, A, B, p=-1):
        """``A @ B`` all-reduced iff ``p != 1`` (dist_nmf.py:687-711).  The two A-streaming products of the update loop,
        ``global_mm(A_ij, H_j.T, p_c)`` and ``global_mm(W_i.T, A_ij, p_r)``, run as one pass over the resident shard; any
        other pair of matrices goes through the same skinny contraction in column chunks of the factor width the kernels
        support (the left operand is streamed once per chunk)."""
        dt = self.fdtype
        if A is self.A_ij or A is self._A_orig:
            Bt = D.to_device_view(B, dt).t().contiguous()
            if Bt.shape[0] <= D.L.MAX_K:
                out = self.ops.ah(self.A_ij, Bt)
            else:
                out = self._mm_chunked(self.A_ij, D.to_device_view(B, dt))
        elif (B is self.A_ij or B is self._A_orig) and D.to_device_view(A, dt).shape[0] <= D.L.MAX_K:
            out = self.ops.wta(self.A_ij, D.to_device_view(A, dt).t().contiguous())
        else:
            out = self._mm_chunked(D.to_device_view(A, dt).contiguous(), D.to_device_view(B, dt))
        return self.comm1.allreduce_(out) if p != 1 else out

    def _mm_chunked(self, A, B):
        """A [r x c] @ B [c x s] for any s: out[:, j0:j1] = A (B[:, j0:j1]^T)^T in chunks of <= MAX_K columns."""
        r, s_cols = A.shape[0], B.shape[1]
        out = self.ops.empty((r, s_cols), D.out_dtype(A.dtype))
        step = D.L.MAX_K
        for j0 in range(0, s_cols, step):
            j1 = min(s_cols, j0 + step)
            out[:, j0:j1] = self.ops.ah(A, B[:, j0:j1].t().contiguous())
        return out

    def _gram_W(self, W):
        G = self.ops.gram(W, trans=False)
        return self.comm1.allreduce_(G) if self.p_r != 1 else G

    def _gram_H(self, H):
        G = self.ops.gram(H, trans=True)
        return self.comm1.allreduce_(G) if self.p_c != 1 else G

    def _AH(self, H):
        V = self.ops.ah(self.A_ij, H)
        return self.comm1.allreduce_(V) if self.p_c != 1 else V

    def _WTA(self, W):
        Y = self.ops.wta(self.A_ij, W)
        return (self.comm1.allreduce_(Y) if self.p_r != 1 else Y), False

    # ---- FRO / MU -----------------------------------------------------------------------------
    @comm_timing()
    def Fro_MU_update_W(self):
        """dist_nmf.py:715-732."""
        HH_T = self._gram_H(self.H_j)
        if self.p_c == 1 and self._mon is None:
            # pass + ONE epilogue launch: the update sums the pass's split partials itself (dnmf_ah_p / dnmf_mu_update_w_p)
            view = self.ops.ah_p(self.A_ij, self.H_j)
            if view is not None:
                self.ops.mu_update_w_p(self.W_i, view, HH_T, self.eps)
                return
        AH = self._AH(self.H_j)
        self._monitor_sample(self.W_i, AH, HH_T)
        self.ops.mu_update_w(self.W_i, AH, HH_T, self.eps)

    @comm_timing()
    def Fro_MU_update_H(self):
        """dist_nmf.py:735-751."""
        if self._px is not None:
            G = self.ops.gram(self.W_i, trans=False)                      # this rank's W_i^T W_i
            view = self.ops.wta_p(self.A_ij, self.W_i)
            if view is not None:                                          # the push kernel sums the split partials itself
                self._px.update_h_p(0, self.H_j, view, G, self.eps)
                return
            Yt = self.ops.wta(self.A_ij, self.W_i, transposed_out=True)   # this rank's (W_i^T A_i)^T
            self._px.update_h(0, self.H_j, Yt, G, self.eps)
            return
        W_TW = self._gram_W(self.W_i)
        self._monitor_keep(W_TW)
        if self.p_r == 1 and self._mon is None:
            view = self.ops.wta_p(self.A_ij, self.W_i)
            if view is not None:
                self.ops.mu_update_h_p(self.H_j, view, W_TW, self.eps)
                return
        AtW, _ = self._WTA(self.W_i)
        self.ops.mu_update_h(self.H_j, AtW, W_TW, self.eps)

    @comm_timing()
    def Fro_MU_update(self, W_update=True):
        """dist_nmf.py:754-771."""
        if W_update == True:  # noqa: E712
            self.Fro_MU_update_W()
        self.Fro_MU_update_H()

    # ---- KL / MU ------------------------------------------------------------------------------
    @comm_timing()
    def sum_along_axis(self, X, p=1, axis=0):
        """dist_nmf.py:775-801."""
        X = D.to_device(X, self.fdtype)
        s = self.ops.colsum(X) if axis == 0 else self.ops.rowsum(X)
        return self.comm1.allreduce_(s) if p != 1 else s

    @comm_timing()
    def glob_UX(self, axis):
        """Fused ``A / (W H + eps)`` contraction (dist_nmf.py:803-811); no m x n temporaries."""
        if axis == 1:
            UX = self.ops.kl_wtu(self.A_ij, self.W_i, self.H_j, self.eps)
            return self.comm1.allreduce_(UX) if self.p_r != 1 else UX
        elif axis == 0:
            UX = self.ops.kl_uht(self.A_ij, self.W_i, self.H_j, self.eps)
            return self.comm1.allreduce_(UX) if self.p_c != 1 else UX

    def KL_MU_update_W(self):
        """dist_nmf.py:813-830."""
        x2 = self.sum_along_axis(self.H_j, p=self.p_c, axis=1)
        if self.p_c == 1:
            view = self.ops.kl_uht_p(self.A_ij, self.W_i, self.H_j, self.eps)
            if view is not None:
                self.ops.kl_update_w_p(self.W_i, view, x2, self.eps)
                return
        sk = self.glob_UX(axis=0)
        self.ops.kl_update_w(self.W_i, sk, x2, self.eps)

    def KL_MU_update_H(self):
        """dist_nmf.py:832-849."""
        if self._px is not None:
            x = self.ops.colsum(self.W_i)                                  # this rank's column sums of W_i
            view = self.ops.kl_wtu_p(self.A_ij, self.W_i, self.H_j, self.eps)
            if view is not None:
                self._px.update_h_p(3, self.H_j, view, x, self.eps)
                return
            Yt = self.ops.kl_wtu(self.A_ij, self.W_i, self.H_j, self.eps, transposed_out=True)
            self._px.update_h(3, self.H_j, Yt, x, self.eps)
            return
        x2 = self.sum_along_axis(self.W_i, p=self.p_r, axis=0)
        if self.p_r == 1:
            view = self.ops.kl_wtu_p(self.A_ij, self.W_i, self.H_j, self.eps)
            if view is not None:
                self.ops.kl_update_h_p(self.H_j, view, x2, self.eps)
                return
        sk = self.glob_UX(axis=1)
        self.ops.kl_update_h(self.H_j, sk, x2, self.eps)

    def KL_MU_update(self, W_update=True):
        """dist_nmf.py:851-869."""
        if W_update == True:  # noqa: E712
            self.KL_MU_update_W()
        self.KL_MU_update_H()

    # ---- FRO / HALS -----------------------------------------------------------------------------
    def FRO_HALS_update_W(self):
        """dist_nmf.py:873-893."""
        HHT = self._gram_H(self.H_j)
        AH = self._AH(self.H_j)
        if self.p_r == 1 or self._px is not None:
            # one cooperative launch for the whole sweep; on a row grid the k column norms cross the ranks through
            # peer memory inside the kernel instead of k all-reduces
            self.ops.hals_w_sweep(self.W_i, AH, HHT, self.eps, peer=self._px if self.p_r != 1 else None)
            return
        for kk in range(self.k):
            sq = self.ops.hals_w_col(self.W_i, AH, HHT, kk, self.eps)
            if self.p_r != 1:
                sq = self.comm1.allreduce_(sq)
            self.ops.div_col(self.W_i, kk, sq)

    def FRO_HALS_update_H(self):
        """dist_nmf.py:895-913."""
        if self._px is not None:
            G = self.ops.gram(self.W_i, trans=False)
            view = self.ops.wta_p(self.A_ij, self.W_i)
            if view is not None:
                self._px.update_h_p(2, self.H_j, view, G, self.eps)
                return
            Yt = self.ops.wta(self.A_ij, self.W_i, transposed_out=True)
            self._px.update_h(2, self.H_j, Yt, G, self.eps)
            return
        WTW = self._gram_W(self.W_i)
        AtW, _ = self._WTA(self.W_i)
        self.ops.hals_h(self.H_j, AtW, WTW, self.eps)

    def FRO_HALS_update(self, W_update=True):
        """dist_nmf.py:916-934."""
        if W_update == True:  # noqa: E712
            self.FRO_HALS_update_W()
        self.FRO_HALS_update_H()

    # ---- FRO / BCD ------------------------------------------------------------------------------
    def _sqnorm_global(self, X, which=None):
        sq = self.ops.sqnorm(X)
        p = {None: -1, 'w': self.p_r, 'h': self.p_c}[which]
        if p != 1:
            sq = self.comm1.allreduce_(sq)
        return float(sq.item())

    @comm_timing()
    def globalSqNorm(self, X, p=-1):
        """dist_nmf.py:939-949."""
        sq = self.ops.sqnorm(D.to_device(X, self.fdtype))
        if p != 1:
            sq = self.comm1.allreduce_(sq)
        return float(sq.item())

    def _colsum_W(self, W, force):
        s = self.ops.colsum(W)
        return self.comm1.allreduce_(s) if self.p_r != 1 else s

    def _residual_global(self, W, H):
        return self.comm1.allreduce_(self.ops.residual_sqnorm(self.A_ij, W, H))

    def _sqnorm_dev(self, X, which=None):
        sq = self.ops.sqnorm(X)
        p = {None: -1, 'w': self.p_r, 'h': self.p_c}[which]
        return self.comm1.allreduce_(sq) if p != 1 else sq

    def _AH_and_residual(self, W, H):
        V, res = self.ops.ah_residual(self.A_ij, W, H)
        return (self.comm1.allreduce_(V) if self.p_c != 1 else V), self.comm1.allreduce_(res)

    def initWandH(self):
        """dist_nmf.py:951-969: scaled factors, H H^T, A H^T and obj_old, left on the device (see bcd_begin)."""
        self.bcd_begin()

    def FRO_BCD_update(self, W_update=True, itr=1000):
        """dist_nmf.py:971-1047."""
        self._bcd_loop(itr)
