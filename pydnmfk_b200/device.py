"""Device-side operator layer: torch CUDA tensors in, libdnmf kernels underneath.

PyTorch is used only to own device memory and streams (and, in dist_comm, for
the process groups).  Every numeric operation of the update loop is one of the
hand-written kernels behind the C-ABI (include/dnmf.h); there is no CPU or
eager-PyTorch fallback -- calling this layer without a CUDA device raises.
"""
import ctypes as C
import os

import numpy as np
import torch

from . import _lib as L

_DT = {torch.float32: L.F32, torch.float64: L.F64}
# dtype codes of the entry points that read the data shard A, which may also be stored in 16 bits
_DT_A = {**_DT, torch.float16: L.A_F16, torch.bfloat16: L.A_BF16}
_A16 = (torch.float16, torch.bfloat16)


def out_dtype(a_dtype):
    """dtype of the factors and of every result computed from a shard stored as ``a_dtype`` (float32 for 16-bit A)."""
    return torch.float32 if a_dtype in _A16 else a_dtype


def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError('pydnmfk_b200 needs a CUDA device (sm_100a); it has no CPU fallback')


def fused_epilogue_enabled():
    """DNMF_FUSED_EPILOGUE=0 keeps pass, split reduction and update as separate launches (A/B runs)."""
    return os.environ.get('DNMF_FUSED_EPILOGUE', '1') != '0'


def to_device(x, dtype=None, device=None, non_blocking=False):
    """numpy / torch (host or device) -> contiguous CUDA tensor.  ``non_blocking``: a page-locked host source is copied
    asynchronously on the current stream (the caller synchronises before the host buffer may change)."""
    require_cuda()
    if device is None:
        device = torch.device('cuda', torch.cuda.current_device())
    if isinstance(x, torch.Tensor):
        t = x
    else:
        a = np.asarray(x)
        if not a.flags.c_contiguous:
            a = np.ascontiguousarray(a)
        if not a.flags.writeable:
            a = a.copy()
        t = torch.from_numpy(a)
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    t = t.to(device, non_blocking=bool(non_blocking) and (not t.is_cuda) and t.is_pinned())
    return t.contiguous()


def to_device_view(x, dtype=None):
    """Like to_device but keeps the strides of a (possibly transposed) device tensor / numpy view."""
    require_cuda()
    if isinstance(x, torch.Tensor):
        t = x if x.is_cuda else x.cuda()
    else:
        a = np.asarray(x)
        t = torch.from_numpy(a.copy() if not a.flags.writeable else a).cuda()
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    return t


def to_device_a16(x, dtype):
    """The data shard rounded to nearest even into ``dtype`` (torch.float16 / torch.bfloat16) as a contiguous CUDA tensor.
    Host data is rounded on the host by torch's CPU cast (multi-threaded; the same nearest-even result as numpy's
    ``astype(np.float16)``), so only 2 bytes per element cross the bus; a CUDA float32 tensor is rounded on the device; a CUDA tensor already in ``dtype`` is used as it
    is.  Raises ValueError when an entry overflows to inf (|a| > 65504 in float16)."""
    require_cuda()
    if isinstance(x, torch.Tensor) and x.is_cuda:
        t = x.to(dtype).contiguous()
    else:
        h = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x))
        h = h.contiguous().to(dtype)
        t = h.to(torch.device('cuda', torch.cuda.current_device()))
    if t.numel() > 0:
        lo, hi = torch.aminmax(t)
        if bool(torch.isinf(lo) | torch.isinf(hi)):
            raise ValueError('params.a_storage=%r: the data has entries beyond the %s range (largest finite magnitude %g)'
                             % (str(dtype).replace('torch.', ''), dtype, torch.finfo(dtype).max))
    return t


def torch_dtype(np_dtype):
    np_dtype = np.dtype(np_dtype)
    if np_dtype == np.float32:
        return torch.float32
    if np_dtype == np.float64:
        return torch.float64
    raise TypeError('precision %s is not supported on the device path (float32/float64 only)' % np_dtype)


def _ld(t):
    """Leading dimension of a row-major 2-D tensor (elements)."""
    assert t.dim() == 2 and (t.shape[1] <= 1 or t.stride(1) == 1), 'row-major matrix expected'
    return t.stride(0) if t.shape[0] > 1 else max(t.shape[1], 1)


class DeviceOps:
    """Kernel launcher bound to one device; owns the scratch workspace."""

    def __init__(self, device=None, math_mode=L.MATH_ACCURATE):
        require_cuda()
        self.device = device if device is not None else torch.device('cuda', torch.cuda.current_device())
        self.math_mode = math_mode
        self._ws = None
        self._ws_bytes = 0
        self.timers = None      # set to {} to bracket the A-streaming passes with CUDA events (bench.py)

    def _t0(self, name):
        if self.timers is None:
            return None
        ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        ev[0].record(torch.cuda.current_stream(self.device))
        self.timers.setdefault(name, []).append(ev)
        return ev

    def _t1(self, ev):
        if ev is not None:
            ev[1].record(torch.cuda.current_stream(self.device))

    def timer_summary(self):
        """{op: (launches, mean ms)} from the recorded events (call after a synchronize)."""
        out = {}
        for name, evs in (self.timers or {}).items():
            ms = [a.elapsed_time(b) for a, b in evs]
            out[name] = (len(ms), sum(ms) / max(len(ms), 1))
        return out

    # ---- plumbing -------------------------------------------------------------------------
    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def workspace(self, nbytes):
        if nbytes > self._ws_bytes:
            self._ws = torch.empty(int(nbytes), dtype=torch.uint8, device=self.device)
            self._ws_bytes = int(nbytes)
        return self._ws.data_ptr() if self._ws is not None else 0

    def _ws_for(self, op, m, n, k, dt):
        nb = L.workspace_bytes(op, m, n, k, dt)
        return self.workspace(nb), max(nb, self._ws_bytes)

    def empty(self, shape, dtype):
        return torch.empty(shape, dtype=dtype, device=self.device)

    # ---- A-streaming contractions -----------------------------------------------------------
    def ah(self, A, H, out=None):
        """V = A @ H.T   (dist_nmf.py:198, :730)"""
        m, n = A.shape
        k = H.shape[0]
        dt = _DT_A[A.dtype]
        V = out if out is not None else self.empty((m, k), out_dtype(A.dtype))
        ws, wsb = self._ws_for(L.OP_AH, m, n, k, dt)
        ev = self._t0('ah')
        L.call('dnmf_ah', A.data_ptr(), _ld(A), H.data_ptr(), _ld(H), V.data_ptr(), _ld(V), m, n, k, dt,
               self.math_mode, ws, wsb, self._stream())
        self._t1(ev)
        return V

    def wta(self, A, W, transposed_out=False, out=None):
        """Y = W.T @ A (k x n), or Y.T (n x k) when transposed_out   (dist_nmf.py:166, :749)"""
        m, n = A.shape
        k = W.shape[1]
        dt = _DT_A[A.dtype]
        Y = out if out is not None else self.empty((n, k) if transposed_out else (k, n), out_dtype(A.dtype))
        ws, wsb = self._ws_for(L.OP_WTA, m, n, k, dt)
        ev = self._t0('wta')
        L.call('dnmf_wta', A.data_ptr(), _ld(A), W.data_ptr(), _ld(W), Y.data_ptr(), _ld(Y), m, n, k,
               1 if transposed_out else 0, dt, self.math_mode, ws, wsb, self._stream())
        self._t1(ev)
        return Y

    def kl_uht(self, A, W, H, eps, out=None):
        """V = (A / (W @ H + eps)) @ H.T without materialising W @ H   (dist_nmf.py:338-339, :806,:810)"""
        m, n = A.shape
        k = H.shape[0]
        dt = _DT_A[A.dtype]
        V = out if out is not None else self.empty((m, k), out_dtype(A.dtype))
        ws, wsb = self._ws_for(L.OP_KL_UHT, m, n, k, dt)
        ev = self._t0('kl_uht')
        L.call('dnmf_kl_uht', A.data_ptr(), _ld(A), W.data_ptr(), _ld(W), H.data_ptr(), _ld(H), V.data_ptr(),
               _ld(V), m, n, k, float(eps), dt, self.math_mode, ws, wsb, self._stream())
        self._t1(ev)
        return V

    def kl_wtu(self, A, W, H, eps, transposed_out=False, out=None):
        """Y = W.T @ (A / (W @ H + eps))   (dist_nmf.py:312-313, :806,:808)"""
        m, n = A.shape
        k = H.shape[0]
        dt = _DT_A[A.dtype]
        Y = out if out is not None else self.empty((n, k) if transposed_out else (k, n), out_dtype(A.dtype))
        ws, wsb = self._ws_for(L.OP_KL_WTU, m, n, k, dt)
        ev = self._t0('kl_wtu')
        L.call('dnmf_kl_wtu', A.data_ptr(), _ld(A), W.data_ptr(), _ld(W), H.data_ptr(), _ld(H), Y.data_ptr(),
               _ld(Y), m, n, k, float(eps), 1 if transposed_out else 0, dt, self.math_mode, ws, wsb,
               self._stream())
        self._t1(ev)
        return Y

    # ---- pass with the split reduction deferred to the consumer (include/dnmf.h: dnmf_*_p) ---------------------------
    def _pass_partials(self, name, timer, op, A, k, *args):
        """Run a `_p` pass; returns the int64[4] view (host array kept alive by the caller) or None when the call is
        not served by the tcgen05 path (the caller then uses the plain op)."""
        if not fused_epilogue_enabled() or out_dtype(A.dtype) != torch.float32:
            return None
        m, n = A.shape
        dt = _DT_A[A.dtype]
        ws, wsb = self._ws_for(op, m, n, k, dt)
        view = (C.c_int64 * 4)()
        ev = self._t0(timer)
        rc = getattr(L.raw(), name)(*args, dt, self.math_mode, ws, wsb, view, self._stream())
        if rc == L.E_UNSUPPORTED:
            if ev is not None:
                self.timers[timer].pop()
            return None
        if rc != 0:
            raise L.DnmfError(name, rc, L.raw().dnmf_last_error().decode())
        self._t1(ev)
        return view

    def ah_p(self, A, H):
        m, n = A.shape
        k = H.shape[0]
        return self._pass_partials('dnmf_ah_p', 'ah', L.OP_AH, A, k, A.data_ptr(), _ld(A), H.data_ptr(), _ld(H), m, n, k)

    def wta_p(self, A, W):
        m, n = A.shape
        k = W.shape[1]
        return self._pass_partials('dnmf_wta_p', 'wta', L.OP_WTA, A, k, A.data_ptr(), _ld(A), W.data_ptr(), _ld(W), m, n, k)

    def kl_uht_p(self, A, W, H, eps):
        m, n = A.shape
        k = W.shape[1]
        return self._pass_partials('dnmf_kl_uht_p', 'kl_uht', L.OP_KL_UHT, A, k, A.data_ptr(), _ld(A), W.data_ptr(), _ld(W),
                                   H.data_ptr(), _ld(H), m, n, k, float(eps))

    def kl_wtu_p(self, A, W, H, eps):
        m, n = A.shape
        k = W.shape[1]
        return self._pass_partials('dnmf_kl_wtu_p', 'kl_wtu', L.OP_KL_WTU, A, k, A.data_ptr(), _ld(A), W.data_ptr(), _ld(W),
                                   H.data_ptr(), _ld(H), m, n, k, float(eps))

    def mu_update_w_p(self, W, view, G, eps):
        m, k = W.shape
        L.call('dnmf_mu_update_w_p', W.data_ptr(), _ld(W), view, G.data_ptr(), m, k, float(eps), _DT[W.dtype], self._stream())

    def mu_update_h_p(self, H, view, G, eps, clamp=False):
        k, n = H.shape
        L.call('dnmf_mu_update_h_p', H.data_ptr(), _ld(H), view, G.data_ptr(), k, n, float(eps), 1 if clamp else 0,
               _DT[H.dtype], self._stream())

    def kl_update_w_p(self, W, view, x, eps):
        m, k = W.shape
        L.call('dnmf_kl_update_w_p', W.data_ptr(), _ld(W), view, x.data_ptr(), m, k, float(eps), _DT[W.dtype], self._stream())

    def kl_update_h_p(self, H, view, x, eps, clamp=False):
        k, n = H.shape
        L.call('dnmf_kl_update_h_p', H.data_ptr(), _ld(H), view, x.data_ptr(), k, n, float(eps), 1 if clamp else 0,
               _DT[H.dtype], self._stream())

    def gram(self, X, trans):
        """trans=False: X.T @ X for X [rows x k];  trans=True: X @ X.T for X [k x rows]."""
        if trans:
            k, rows = X.shape
        else:
            rows, k = X.shape
        dt = _DT[X.dtype]
        G = self.empty((k, k), X.dtype)
        ws, wsb = self._ws_for(L.OP_GRAM, rows, 0, k, dt)
        L.call('dnmf_gram', X.data_ptr(), _ld(X), rows, k, 1 if trans else 0, G.data_ptr(), dt, ws, wsb,
               self._stream())
        return G

    # ---- updates ----------------------------------------------------------------------------
    @staticmethod
    def _ystrides(Y, transposed):
        # element (kk, c) of the k x n quantity; Y may be stored as its transpose (n x k)
        return (1, _ld(Y)) if transposed else (_ld(Y), 1)

    def mu_update_w(self, W, V, G, eps):
        m, k = W.shape
        L.call('dnmf_mu_update_w', W.data_ptr(), _ld(W), V.data_ptr(), _ld(V), G.data_ptr(), m, k, float(eps),
               _DT[W.dtype], self._stream())

    def mu_update_h(self, H, Y, G, eps, y_transposed=False, clamp=False):
        k, n = H.shape
        sk, sc = self._ystrides(Y, y_transposed)
        L.call('dnmf_mu_update_h', H.data_ptr(), _ld(H), Y.data_ptr(), sk, sc, G.data_ptr(), k, n, float(eps),
               1 if clamp else 0, _DT[H.dtype], self._stream())

    def kl_update_w(self, W, V, x, eps):
        m, k = W.shape
        L.call('dnmf_kl_update_w', W.data_ptr(), _ld(W), V.data_ptr(), _ld(V), x.data_ptr(), m, k, float(eps),
               _DT[W.dtype], self._stream())

    def kl_update_h(self, H, Y, x, eps, y_transposed=False, clamp=False):
        k, n = H.shape
        sk, sc = self._ystrides(Y, y_transposed)
        L.call('dnmf_kl_update_h', H.data_ptr(), _ld(H), Y.data_ptr(), sk, sc, x.data_ptr(), k, n, float(eps),
               1 if clamp else 0, _DT[H.dtype], self._stream())

    def clamp_min(self, X, lo):
        r, c = X.shape
        L.call('dnmf_clamp_min', X.data_ptr(), _ld(X), r, c, float(lo), _DT[X.dtype], self._stream())

    # ---- small reductions ---------------------------------------------------------------------
    def colsum(self, X):
        r, c = X.shape
        out = self.empty((c,), X.dtype)
        ws, wsb = self._ws_for(L.OP_SUMS, r, c, c, _DT[X.dtype])
        L.call('dnmf_colsum', X.data_ptr(), _ld(X), r, c, out.data_ptr(), _DT[X.dtype], ws, wsb, self._stream())
        return out

    def rowsum(self, X):
        r, c = X.shape
        out = self.empty((r,), X.dtype)
        ws, wsb = self._ws_for(L.OP_SUMS, r, c, r, _DT[X.dtype])
        L.call('dnmf_rowsum', X.data_ptr(), _ld(X), r, c, out.data_ptr(), _DT[X.dtype], ws, wsb, self._stream())
        return out

    def sqnorm(self, X):
        """sum(X**2) as a float64 device scalar (shape [1])."""
        r, c = X.shape
        out = self.empty((1,), torch.float64)
        ws, wsb = self._ws_for(L.OP_SUMS, r, c, min(c, L.MAX_K), _DT[out_dtype(X.dtype)])
        L.call('dnmf_sqnorm', X.data_ptr(), _ld(X), r, c, out.data_ptr(), _DT_A[X.dtype], ws, wsb, self._stream())
        return out

    def normalize(self, W, H, s, eps):
        m, k = W.shape
        n = H.shape[1]
        L.call('dnmf_normalize', W.data_ptr(), _ld(W), m, H.data_ptr(), _ld(H), n, k, s.data_ptr(), float(eps),
               _DT[W.dtype], self._stream())

    def trace_terms(self, W, V, G1, G2, out=None, slot_counter=None):
        """[<W, V>, <G1, G2>] as float64 (include/dnmf.h: dnmf_trace_terms).  With ``out`` [slots, 2] and an int64
        ``slot_counter`` device tensor the pair is appended at the counter's position (graph-replay safe)."""
        m, k = W.shape
        dt = _DT[W.dtype]
        if out is None:
            out = self.empty((1, 2), torch.float64)
        wsb = int(L.call('dnmf_trace_terms_workspace_bytes'))
        ws = self.workspace(wsb)
        L.call('dnmf_trace_terms', W.data_ptr(), _ld(W), V.data_ptr(), _ld(V), m, G1.data_ptr(), G2.data_ptr(), k,
               out.data_ptr(), slot_counter.data_ptr() if slot_counter is not None else None, out.shape[0], dt,
               ws, wsb, self._stream())
        return out

    def residual_sqnorm(self, A, W, H):
        """[||A - W H||_F^2, ||A||_F^2] as a float64 device tensor of shape [2]."""
        m, n = A.shape
        k = W.shape[1]
        dt = _DT_A[A.dtype]
        out = self.empty((2,), torch.float64)
        ws, wsb = self._ws_for(L.OP_RESIDUAL, m, n, k, dt)
        L.call('dnmf_residual_sqnorm', A.data_ptr(), _ld(A), W.data_ptr(), _ld(W), H.data_ptr(), _ld(H), m, n, k,
               out.data_ptr(), dt, ws, wsb, self._stream())
        return out

    def ah_residual(self, A, W, H):
        """(A @ H.T, [||A - W H||_F^2, ||A||_F^2]) in one pass over A (dist_nmf.py:1023-1024)."""
        m, n = A.shape
        k = W.shape[1]
        dt = _DT_A[A.dtype]
        V = self.empty((m, k), out_dtype(A.dtype))
        out = self.empty((2,), torch.float64)
        ws, wsb = self._ws_for(L.OP_AH_RESIDUAL, m, n, k, dt)
        ev = self._t0('ah_res')
        L.call('dnmf_ah_residual', A.data_ptr(), _ld(A), W.data_ptr(), _ld(W), H.data_ptr(), _ld(H), V.data_ptr(), _ld(V),
               m, n, k, out.data_ptr(), dt, ws, wsb, self._stream())
        self._t1(ev)
        return V, out

    def column_err(self, A, W, H):
        m, n = A.shape
        k = W.shape[1]
        num = self.empty((n,), torch.float64)
        den = self.empty((n,), torch.float64)
        L.call('dnmf_column_err', A.data_ptr(), _ld(A), W.data_ptr(), _ld(W), H.data_ptr(), _ld(H), m, n, k,
               num.data_ptr(), den.data_ptr(), _DT_A[A.dtype], self._stream())
        return num, den

    # ---- HALS / BCD ---------------------------------------------------------------------------
    def hals_w_col(self, W, V, G, kk, eps):
        m, k = W.shape
        sq = self.empty((1,), torch.float64)
        ws, wsb = self._ws_for(L.OP_SUMS, m, k, k, _DT[W.dtype])
        L.call('dnmf_hals_w_col', W.data_ptr(), _ld(W), V.data_ptr(), _ld(V), G.data_ptr(), m, k, kk, float(eps),
               sq.data_ptr(), _DT[W.dtype], ws, wsb, self._stream())
        return sq

    def hals_w_sweep(self, W, V, G, eps, peer=None):
        """All k column updates of the HALS W sweep (+ their global norms) in one cooperative launch; `peer` = the
        PeerExchange of a row grid (column norms summed over the ranks through peer memory) or None (one rank)."""
        m, k = W.shape
        need = k * 1024 * 8 + 256
        if getattr(self, '_hals_scratch', None) is None or self._hals_scratch.numel() < need:
            self._hals_scratch = torch.zeros(need, dtype=torch.uint8, device=self.device)
        sc = self._hals_scratch
        if peer is None:
            bases, P, me, xn = None, 1, 0, 0
        else:
            bases, P, me, xn = peer._bases, peer.P, peer.me, peer.n
        L.call('dnmf_hals_w_sweep', W.data_ptr(), _ld(W), V.data_ptr(), _ld(V), G.data_ptr(), m, k, float(eps), bases, P, me,
               xn, sc.data_ptr(), sc.numel(), _DT[W.dtype], self._stream())

    def div_col(self, W, kk, ss_sq):
        L.call('dnmf_div_col', W.data_ptr(), _ld(W), W.shape[0], kk, ss_sq.data_ptr(), _DT[W.dtype], self._stream())

    def hals_h(self, H, Y, G, eps, y_transposed=False):
        k, n = H.shape
        sk, sc = self._ystrides(Y, y_transposed)
        L.call('dnmf_hals_h', H.data_ptr(), _ld(H), Y.data_ptr(), sk, sc, G.data_ptr(), k, n, float(eps),
               _DT[H.dtype], self._stream())

    def bcd_pg_w(self, W, Wm, V, G, Lip):
        m, k = W.shape
        L.call('dnmf_bcd_pg_w', W.data_ptr(), _ld(W), Wm.data_ptr(), _ld(Wm), V.data_ptr(), _ld(V), G.data_ptr(),
               m, k, float(Lip), _DT[W.dtype], self._stream())

    def bcd_pg_h(self, H, Hm, Y, G, Lip, y_transposed=False):
        k, n = H.shape
        sk, sc = self._ystrides(Y, y_transposed)
        L.call('dnmf_bcd_pg_h', H.data_ptr(), _ld(H), Hm.data_ptr(), _ld(Hm), Y.data_ptr(), sk, sc, G.data_ptr(),
               k, n, float(Lip), _DT[H.dtype], self._stream())

    # BCD with device-resident scalars (dnmf_bcd.cu): `state` is a 16-element float64 device vector
    def bcd_pg_w_dev(self, W, Wm, V, G, state, idx):
        m, k = W.shape
        L.call('dnmf_bcd_pg_w_dev', W.data_ptr(), _ld(W), Wm.data_ptr(), _ld(Wm), V.data_ptr(), _ld(V), G.data_ptr(),
               m, k, state.data_ptr() + 8 * idx, _DT[W.dtype], self._stream())

    def bcd_pg_h_dev(self, H, Hm, Y, G, state, idx, y_transposed=False):
        k, n = H.shape
        sk, sc = self._ystrides(Y, y_transposed)
        L.call('dnmf_bcd_pg_h_dev', H.data_ptr(), _ld(H), Hm.data_ptr(), _ld(Hm), Y.data_ptr(), sk, sc, G.data_ptr(),
               k, n, state.data_ptr() + 8 * idx, _DT[H.dtype], self._stream())

    def bcd_state(self, phase, state, scalar_in):
        assert state.dtype == torch.float64 and scalar_in.dtype == torch.float64
        L.call('dnmf_bcd_state', int(phase), state.data_ptr(), scalar_in.data_ptr(), self._stream())

    def bcd_advance(self, X, Xm, X_old, state, which):
        assert X.is_contiguous() and Xm.is_contiguous() and X_old.is_contiguous()
        L.call('dnmf_bcd_advance', X.data_ptr(), Xm.data_ptr(), X_old.data_ptr(), X.numel(), state.data_ptr(), int(which),
               _DT[X.dtype], self._stream())

    def bcd_keep(self, cur, kept, state):
        assert cur.is_contiguous() and kept.is_contiguous()
        L.call('dnmf_bcd_keep', cur.data_ptr(), kept.data_ptr(), cur.numel(), state.data_ptr(), _DT[cur.dtype],
               self._stream())

    def div_cols(self, W, s):
        m, k = W.shape
        L.call('dnmf_div_cols', W.data_ptr(), _ld(W), m, k, s.data_ptr(), _DT[W.dtype], self._stream())

    def axpby(self, out, x, y, a, b):
        assert out.is_contiguous() and x.is_contiguous() and y.is_contiguous()
        L.call('dnmf_axpby', out.data_ptr(), x.data_ptr(), y.data_ptr(), float(a), float(b), out.numel(),
               _DT[out.dtype], self._stream())

    # ---- shard ops ------------------------------------------------------------------------------
    def nnz_counts(self, A):
        m, n = A.shape
        rows = self.empty((m,), torch.int64)
        cols = self.empty((n,), torch.int64)
        L.call('dnmf_nnz_counts', A.data_ptr(), _ld(A), m, n, rows.data_ptr(), cols.data_ptr(), _DT_A[A.dtype],
               self._stream())
        return rows, cols

    def compact(self, A, row_idx, col_idx):
        mr, nc = row_idx.numel(), col_idx.numel()
        out = self.empty((mr, nc), A.dtype)
        L.call('dnmf_compact', A.data_ptr(), _ld(A), row_idx.data_ptr(), mr, col_idx.data_ptr(), nc, out.data_ptr(),
               max(nc, 1), _DT_A[A.dtype], self._stream())
        return out

    def scatter_rows(self, X, row_idx, total_rows):
        out = torch.zeros((total_rows, X.shape[1]), dtype=torch.float64, device=self.device)
        L.call('dnmf_scatter_rows', X.data_ptr(), _ld(X), row_idx.data_ptr(), X.shape[0], X.shape[1],
               out.data_ptr(), max(X.shape[1], 1), _DT[X.dtype], self._stream())
        return out

    def scatter_cols(self, X, col_idx, total_cols):
        out = torch.zeros((X.shape[0], total_cols), dtype=torch.float64, device=self.device)
        L.call('dnmf_scatter_cols', X.data_ptr(), _ld(X), col_idx.data_ptr(), X.shape[1], X.shape[0],
               out.data_ptr(), max(total_cols, 1), _DT[X.dtype], self._stream())
        return out

    def perturb_uniform(self, A, U, noise_var):
        X = torch.empty_like(A)
        assert A.is_contiguous() and U.is_contiguous()
        L.call('dnmf_perturb_uniform', A.data_ptr(), U.data_ptr(), X.data_ptr(), A.numel(), float(noise_var),
               _DT[A.dtype], self._stream())
        return X

    # ---- NMFk-level rows: clustering / silhouettes (dist_clustering.py) -------------------------------
    def colsum_wide(self, X, squares=False):
        """Column sums (or sums of squares) of a matrix with any number of columns (the m x kP view of W_all)."""
        r, c = X.shape
        out = self.empty((c,), X.dtype)
        nb = L.call('dnmf_colsum_workspace_bytes', r, c)
        ws = self.workspace(nb)
        L.call('dnmf_colsumsq' if squares else 'dnmf_colsum', X.data_ptr(), _ld(X), r, c, out.data_ptr(), _DT[X.dtype],
               ws, max(nb, self._ws_bytes), self._stream())
        return out

    def scale_groups(self, X, s, s_strides, mode, eps=0.0):
        """In place X[i0,i1,i2] op= f(s[...]); X contiguous 3-D (2-D inputs are viewed as [1, d0, d1])."""
        assert X.is_contiguous() and s.is_contiguous() and s.dtype == X.dtype
        d = list(X.shape)
        while len(d) < 3:
            d.insert(0, 1)
            s_strides = (0,) + tuple(s_strides)
        L.call('dnmf_scale_groups', X.data_ptr(), d[0], d[1], d[2], s.data_ptr(), int(s_strides[0]), int(s_strides[1]),
               int(s_strides[2]), int(mode), float(eps), _DT[X.dtype], self._stream())
        return X

    def greedy_lsa(self, Dm, k, P):
        """order[p, r] = feature of perturbation p assigned to centroid r (int32 [P, k])."""
        assert Dm.shape == (k, k * P)
        order = self.empty((P, k), torch.int32)
        L.call('dnmf_greedy_lsa', Dm.data_ptr(), _ld(Dm), k, P, order.data_ptr(), _DT[Dm.dtype], self._stream())
        return order

    def permute_groups(self, X, order, axis, sequential=False):
        """out[.., r, .., p] = X[.., order[p, r], .., p] for a contiguous [d0, d1, P] tensor; ``sequential`` gives the
        result of the in-place row-by-row assignment ``for r: X[r] = X[order[p, r]]`` instead (see include/dnmf.h)."""
        assert X.is_contiguous() and X.dim() == 3 and order.is_contiguous() and order.dtype == torch.int32
        out = torch.empty_like(X)
        L.call('dnmf_permute_groups', X.data_ptr(), out.data_ptr(), X.shape[0], X.shape[1], X.shape[2], int(axis),
               order.data_ptr(), 1 if sequential else 0, _DT[X.dtype], self._stream())
        return out

    def median_last(self, X, want_mad=False):
        """np.median(X, axis=-1) (and the median absolute deviation around it) of a contiguous tensor."""
        assert X.is_contiguous()
        P = X.shape[-1]
        rows = X.numel() // max(P, 1)
        med = self.empty(tuple(X.shape[:-1]), X.dtype)
        mad = self.empty(tuple(X.shape[:-1]), X.dtype) if want_mad else None
        L.call('dnmf_median_last', X.data_ptr(), rows, P, med.data_ptr(), mad.data_ptr() if want_mad else 0,
               _DT[X.dtype], self._stream())
        return (med, mad) if want_mad else med

    def silhouettes(self, G, k, P):
        assert G.shape == (k * P, k * P)
        out = self.empty((k, P), torch.float64)
        L.call('dnmf_silhouettes', G.data_ptr(), _ld(G), k, P, out.data_ptr(), _DT[G.dtype], self._stream())
        return out

    # ---- NMFk-level rows: nnsvd initialisation (dist_svd.py) -------------------------------------------
    def rank1_sub(self, M, u, v, sigma):
        assert u.dtype == v.dtype == sigma.dtype == torch.float64
        L.call('dnmf_rank1_sub', M.data_ptr(), _ld(M), M.shape[0], M.shape[1], u.data_ptr(), v.data_ptr(),
               sigma.data_ptr(), _DT[M.dtype], self._stream())
        return M

    def matvec_f64(self, A, x, trans=False):
        """A @ x or A.T @ x with float64 vectors and accumulation (A keeps its dtype in memory)."""
        assert x.dtype == torch.float64 and x.is_contiguous()
        r, c = A.shape
        y = self.empty((c if trans else r,), torch.float64)
        nb = L.call('dnmf_matvec_workspace_bytes', r, c, 1 if trans else 0)
        ws = self.workspace(nb)
        L.call('dnmf_matvec_f64', A.data_ptr(), _ld(A), r, c, x.data_ptr(), y.data_ptr(), 1 if trans else 0,
               _DT[A.dtype], ws, max(nb, self._ws_bytes), self._stream())
        return y

    def power_normalize(self, y, v_last, r_out):
        v = torch.empty_like(y)
        L.call('dnmf_power_normalize', y.data_ptr(), v_last.data_ptr(), v.data_ptr(), r_out.data_ptr(), y.numel(),
               self._stream())
        return v

    def power_iterate(self, B, v0, thr, max_iter=1000000):
        """The whole power iteration on B [d x d] (d <= 512) in one launch, until |<v, v_prev>| > thr; returns the unit
        vector.  ``thr`` is the caller's ``1. - eps`` scalar: when it is a numpy float32 the comparison runs in float32, as
        numpy's own ``python_float > np.float32`` does (the reference's stopping rule for fp32 data)."""
        d = B.shape[0]
        assert B.shape == (d, d) and v0.dtype == torch.float64 and v0.numel() == d
        v = v0.clone()
        scratch = self.empty((2 * d,), torch.float64)
        cmp32 = 1 if isinstance(thr, np.float32) else 0
        L.call('dnmf_power_iterate', B.data_ptr(), _ld(B), d, v.data_ptr(), float(thr), cmp32, int(max_iter),
               scratch.data_ptr(), None, _DT[B.dtype], self._stream())
        return v

    def div_store(self, src, sq, dst_col):
        """dst_col (a strided column view) = src / sqrt(sq)."""
        L.call('dnmf_div_store', src.data_ptr(), sq.data_ptr(), dst_col.data_ptr(), src.numel(),
               dst_col.stride(0) if dst_col.numel() > 1 else 1, self._stream())

    def posneg_colsumsq(self, X):
        r, k = X.shape
        out = self.empty((2, k), torch.float64)
        L.call('dnmf_posneg_colsumsq', X.data_ptr(), _ld(X), r, k, out.data_ptr(), self._stream())
        return out

    def nnsvd_pick(self, X, coef, pos, transpose_out=False):
        r, k = X.shape
        out = self.empty((k, r) if transpose_out else (r, k), torch.float64)
        L.call('dnmf_nnsvd_pick', X.data_ptr(), _ld(X), r, k, coef.data_ptr(), pos.data_ptr(), out.data_ptr(),
               max(r, 1) if transpose_out else k, 1 if transpose_out else 0, self._stream())
        return out

    def gram_wide(self, X, chunk=L.MAX_K):
        """X.T @ X for a tall matrix with any number of columns (the (kP)^2 cosine Gram, the nnsvd d x d Gram):
        column chunks of X act as the skinny factor of the A-streaming W^T A contraction."""
        m, c = X.shape
        G = self.empty((c, c), X.dtype)
        for c0 in range(0, c, chunk):
            c1 = min(c0 + chunk, c)
            self.wta(X, X[:, c0:c1], out=G[c0:c1])
        return G

    def outer_gram_wide(self, X, Y, chunk=L.MAX_K):
        """X @ Y.T for wide matrices with few rows (m x m): row chunks of Y act as the skinny factor of A H^T."""
        m = X.shape[0]
        r = Y.shape[0]
        G = self.empty((m, r), X.dtype)
        for r0 in range(0, r, chunk):
            r1 = min(r0 + chunk, r)
            self.ah(X, Y[r0:r1], out=G[:, r0:r1])
        return G

    # ---- whole-fit on-chip MU (tiny shards; the batch is the NMFk perturbation ensemble) ---------------------
    @staticmethod
    def resident_fit_fits(m, n, k, norm, dtype):
        """True when one (m x n, k) MU fit fits in an SM's shared memory (dnmf_mu_fit_resident)."""
        if norm.lower() not in ('fro', 'kl') or dtype not in _DT:
            return False
        return L.call('dnmf_mu_fit_resident_smem_bytes', int(m), int(n), int(k), 1 if norm.lower() == 'kl' else 0, _DT[dtype]) > 0

    @staticmethod
    def resident_fit_ctas(m, n, k, norm, dtype):
        """CTAs per fit the on-chip path uses for this shape: 1, a cluster size 2..16, or 0 when it does not apply."""
        if norm.lower() not in ('fro', 'kl') or dtype not in _DT:
            return 0
        return L.call('dnmf_mu_fit_resident_cluster_size', int(m), int(n), int(k), 1 if norm.lower() == 'kl' else 0, _DT[dtype])

    def mu_fit_resident(self, As, Ws, Hs, norm, w_update, it_begin, it_end, eps):
        """Iterations [it_begin, it_end) of the MU loop (+ every-10th clamp) for len(As) independent fits in one launch;
        W and H are updated in place."""
        m, n = As[0].shape
        k = Ws[0].shape[1]
        for A, W, H in zip(As, Ws, Hs):
            assert A.shape == (m, n) and W.shape == (m, k) and H.shape == (k, n) and A.dtype == W.dtype == H.dtype
            assert W.is_contiguous() and H.is_contiguous() and _ld(A) == _ld(As[0])
        ptrs = torch.tensor([[t.data_ptr() for t in grp] for grp in (As, Ws, Hs)], dtype=torch.int64).to(self.device)
        L.call('dnmf_mu_fit_resident', ptrs[0].data_ptr(), _ld(As[0]), ptrs[1].data_ptr(), ptrs[2].data_ptr(), len(As),
               m, n, k, 1 if norm.lower() == 'kl' else 0, 1 if w_update else 0, int(it_begin), int(it_end), float(eps),
               _DT[As[0].dtype], self._stream())
        self._keep = ptrs          # the pointer table must outlive the asynchronous launch


_default_ops = {}


def default_ops():
    require_cuda()
    dev = torch.cuda.current_device()
    if dev not in _default_ops:
        _default_ops[dev] = DeviceOps(torch.device('cuda', dev))
    return _default_ops[dev]
