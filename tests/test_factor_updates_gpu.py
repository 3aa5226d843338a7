"""The factor-side kernels of an iteration, against float64 references at every padded width and operand layout.

The A-streaming passes have unit tests at production schedules; the kernels that update the factors mostly had only the
end-to-end goldens (k in {2, 4, 16}, m <= 2048), which never give the HALS sweep several rows per thread, never reach
BCD's restore branch on purpose and never run a padded width of 32 or 64 with a transposed or windowed operand.
K_ALL below covers every padded width KP in {4, 8, 16, 32, 64}, exactly filled and padded.

Sections:
1. HALS W sweep (dnmf_hals_w_sweep, one rank): one cooperative launch that walks the k columns behind a grid barrier and
   applies each column's scaling lazily.  Rows from 1 to shapes where every thread owns at least 3 and 4 rows (derived
   from the device's SM count and the sweep's grid cap; the grid the launch ran is read back), strided operands with NaN padding, a column clamped everywhere,
   back-to-back launches on one scratch (the barrier word must be reset), m = 0, and agreement with the per-column
   path (hals_w_col + div_col).
2. Device-resident BCD (dnmf_bcd.cu): the 16-double state vector launch by launch against a float64 transcription of
   the reference's scalar logic, including the `obj == obj_old` tie; bcd_advance / bcd_keep on both branches; the
   _dev projected-gradient steps bit-identical to the host-scalar ones; whole fp64 iterations whose accept / restore
   sequence must equal a host transcription (checked bit for bit against oracle.nmf_oracle.fro_bcd_update on the CPU);
   graph replay bit-identical to eager steps.
3. The update kernels (MU, KL, HALS H, BCD, normalize, div_cols, clamp_min) at every width, at the row-block and
   128-column-block edges, with Y as k x n, as its transpose and as windows (both read paths of col_update_kernel),
   factor windows with NaN padding, and an exact small-integer check of the BCD and HALS steps.  G, L and V / Y are
   built as an iteration meets them, and each BCD / HALS case asserts that most of its reference is above the clamp.
4. The _p updates on synthetic split-K partial views: bit-identical to the plain update of the splits' sum in split
   order, the contract of sum_splits.
5. The generic A-streaming passes at padded widths 20, 33, 48 and 63, and an unaligned odd-lda window.

References are float64 (numpy on the host, or torch on the device).  Each case prints its measured error beside its
bound; run with -rP to see them, the HALS sweep's grid and rows per thread and the BCD accept / restore sequence.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from tests import common as T

K_ALL = [1, 3, 5, 8, 13, 16, 20, 31, 32, 33, 48, 63, 64]
DTS = [torch.float32, torch.float64]
DT_IDS = ['f32', 'f64']
TOL = {torch.float32: 2e-5, torch.float64: 1e-12}       # test_kernels_gpu.py: test_updates
F64 = torch.float64


def sweep_bound(dt, k):
    """HALS W sweep: relative error of the worst column after the whole sweep.  The error grows with k (column kk
    depends on the kk columns before it); measured on a B200 it is at most 2.9e-7 k (fp32) and 5.8e-16 k (fp64) over
    all shapes here, so the bound is 1.5e-6 k and 3e-15 k: at least 5x the measured error at every k, and below the
    50 x TOL that test_updates allows the per-column path (1e-3 fp32, 5e-11 fp64)."""
    return (1.5e-6 if dt == torch.float32 else 3e-15) * k


@pytest.fixture(scope='module')
def ops():
    from pydnmfk_b200 import device as D
    return D.default_ops()


def _gen(seed):
    return torch.Generator(device='cuda').manual_seed(seed)


def urand(shape, dt, seed, lo=0.0):
    return (torch.rand(shape, generator=_gen(seed), device='cuda', dtype=F64) + lo).to(dt)


def irand(shape, dt, seed, hi=4):
    """integers in [0, hi): every sum and product below stays exact"""
    return torch.randint(0, hi, shape, generator=_gen(seed), device='cuda').to(dt)


def eps_of(dt):
    return float(torch.finfo(dt).eps)


def esize(dt):
    return torch.empty((), dtype=dt).element_size()


def kp_of(k):
    """padded_k (csrc/common.cuh)"""
    return 4 if k <= 4 else 8 if k <= 8 else 16 if k <= 16 else 32 if k <= 32 else 64


def row_block(dt, k):
    """RowUpdCfg<T, KP>::RB (csrc/generic_small.cuh): rows per block of row_update_kernel"""
    raw = 8192 // (kp_of(k) * esize(dt))
    return 64 if raw > 64 else 16 if raw < 16 else raw


def col_stages(dt, k):
    """col_update_kernel's kStage: Y read with ysk == 1 is staged through shared memory when this holds"""
    kp = kp_of(k)
    return esize(dt) * ((kp + 1) * 128 + kp * kp) <= 46 * 1024


def window(rows, cols, pad, dt, src=None):
    """(buffer, view): a rows x cols view of a rows x (cols + pad) buffer whose padding columns hold NaN"""
    buf = torch.full((rows, cols + pad), float('nan'), dtype=dt, device='cuda')
    view = buf[:, :cols]
    if src is not None:
        view.copy_(src)
    return buf, view


def pad_bits(buf, cols):
    ity = torch.int32 if buf.dtype == torch.float32 else torch.int64
    return buf[:, cols:].contiguous().view(ity).clone()


def col_err(X, R):
    """relative 2-norm error of the worst column"""
    X, R = X.to(F64), R.to(F64)
    return float(((X - R).norm(dim=0) / R.norm(dim=0).clamp_min(1e-300)).max())


def rel(X, R):
    return T.rel_fro(np.asarray(X.cpu() if torch.is_tensor(X) else X, dtype=np.float64),
                     np.asarray(R.cpu() if torch.is_tensor(R) else R, dtype=np.float64))


class Worst:
    """worst error per kernel over a test's cases, printed beside its bound"""

    def __init__(self, tag):
        self.tag, self.err, self.bound = tag, {}, {}

    def add(self, name, err, bound, case):
        assert err <= bound, '%s %s %s: error %.3e > bound %.1e' % (self.tag, name, case, err, bound)
        if err >= self.err.get(name, -1.0):
            self.err[name] = err
        self.bound[name] = bound

    def report(self):
        for name in sorted(self.err):
            print('%-28s %-16s worst %.3e  bound %.1e' % (name, self.tag, self.err[name], self.bound[name]))


# ======================================================================================================================
# 1. HALS W sweep
# ======================================================================================================================
def device_sms():
    from pydnmfk_b200 import _lib as L
    sms, ma, mi = C.c_int(), C.c_int(), C.c_int()
    assert L.raw().dnmf_device_info(C.byref(sms), C.byref(ma), C.byref(mi)) == 0
    return sms.value


def sweep_cap():
    """the sweep's grid cap before occupancy, min(2 * SMs, 1024) (dnmf_hals_w_sweep).  The launch also caps the grid at
    the CTAs that fit on the device at once, which is lower for the register-heavy builds (fp64 at KP = 64 fits one CTA
    per SM), so this is an upper bound on the grid and rows per thread derived from it are a lower bound."""
    return min(2 * device_sms(), 1024)


def sweep_launched_grid(own, k):
    """the grid the last sweep on `own` (a DeviceOps whose sweep scratch was fresh, i.e. zero) actually ran: CTA b of
    column kk leaves its block sum, > 0 because every entry is >= eps, in partials[kk * grid + b] (the scratch after the
    256-byte barrier header), so k * grid of them are non-zero"""
    torch.cuda.synchronize()
    part = own._hals_scratch[256:].view(F64)[:k * 1024]
    nz = int((part != 0).sum().item())
    assert nz % k == 0 and bool((part[:nz] > 0).all()), 'unexpected partials layout (%d non-zero for k=%d)' % (nz, k)
    return nz // k


def sweep_rows(tag):
    cap = sweep_cap()
    return {'tall3': 2 * cap * 256 + 17, 'tall4': 3 * cap * 256 + 5}.get(tag, tag)


def hals_inputs(m, k, dt, seed):
    """W, V = A H^T, G = H H^T as an iteration meets them: A is a rank-k product with unit-norm columns in W0 plus 1 %
    noise and W is W0 perturbed by 5 %, so most t of the sweep are positive and of the size of the final column."""
    g = _gen(seed)
    n = 2 * k + 8
    W0 = torch.rand((m, k), generator=g, device='cuda', dtype=F64) + 0.1
    W0 /= W0.norm(dim=0)
    H = torch.rand((k, n), generator=g, device='cuda', dtype=F64) + 0.1
    A = W0 @ H
    A += 0.01 * A.mean() * torch.rand((m, n), generator=g, device='cuda', dtype=F64)
    W = W0 * (1 + 0.05 * torch.rand((m, k), generator=g, device='cuda', dtype=F64))
    return W.to(dt), (A @ H.T).to(dt), (H @ H.T).to(dt)


def hals_w_ref(W, V, G, eps):
    """the W half of oracle.nmf_oracle.fro_hals_update for one rank, in float64 on the device"""
    W, V, G = W.to(F64).clone(), V.to(F64), G.to(F64)
    for kk in range(W.shape[1]):
        t = W[:, kk] * G[kk, kk] + V[:, kk] - W @ G[:, kk]
        W[:, kk] = t.clamp_min(eps)
        ss = W[:, kk].norm()
        W[:, kk] /= torch.where(ss > 0, ss, torch.ones_like(ss))
    return W


@pytest.mark.gpu
@pytest.mark.parametrize('k', K_ALL)
@pytest.mark.parametrize('dt', DTS, ids=DT_IDS)
def test_hals_sweep_rows(ops, dt, k):
    """m from one row to shapes where every thread owns at least 3 and 4 rows: 2 cap 256 + 17 and 3 cap 256 + 5 rows
    with cap = min(2 SMs, 1024).  For those two the grid the launch ran is read back from its scratch and printed."""
    from pydnmfk_b200 import device as D
    eps, worst = eps_of(dt), Worst('%s k=%d' % (DT_IDS[DTS.index(dt)], k))
    for tag in [1, 255, 256, 257, 2048, 65536, 'tall3', 'tall4']:
        m = sweep_rows(tag)
        W, V, G = hals_inputs(m, k, dt, 100 + k)
        R = hals_w_ref(W, V, G, eps)
        if isinstance(tag, str):
            own = D.DeviceOps()
            own.hals_w_sweep(W, V, G, eps)
            grid = sweep_launched_grid(own, k)
            rpt = -(-m // (grid * 256))
            assert 1 <= grid <= sweep_cap() and rpt >= int(tag[-1]) and rpt > 1, (m, grid, rpt)
            print('sweep %s k=%d m=%d: grid %d CTAs (cap before occupancy %d), %d rows per thread'
                  % (DT_IDS[DTS.index(dt)], k, m, grid, sweep_cap(), rpt))
        else:
            ops.hals_w_sweep(W, V, G, eps)
        worst.add('hals_w_sweep', col_err(W, R), sweep_bound(dt, k), 'm=%d' % m)
    worst.report()


@pytest.mark.gpu
@pytest.mark.parametrize('k', K_ALL)
@pytest.mark.parametrize('dt', DTS, ids=DT_IDS)
def test_hals_sweep_strided(ops, dt, k):
    """W and V are windows (ld = k + 3) with NaN padding: no NaN may leak in, no padding element may change"""
    eps, worst = eps_of(dt), Worst('%s k=%d' % (DT_IDS[DTS.index(dt)], k))
    for m in (257, sweep_rows('tall3')):
        W0, V0, G = hals_inputs(m, k, dt, 200 + k)
        Wb, W = window(m, k, 3, dt, W0)
        Vb, V = window(m, k, 3, dt, V0)
        wpad, vpad = pad_bits(Wb, k), pad_bits(Vb, k)
        ops.hals_w_sweep(W, V, G, eps)
        assert not torch.isnan(W).any(), 'NaN from the padding reached W (m=%d)' % m
        assert torch.equal(pad_bits(Wb, k), wpad) and torch.equal(pad_bits(Vb, k), vpad), 'padding changed (m=%d)' % m
        worst.add('hals_w_sweep ld=k+3', col_err(W, hals_w_ref(W0, V0, G, eps)), sweep_bound(dt, k), 'm=%d' % m)
    worst.report()


@pytest.mark.gpu
@pytest.mark.parametrize('k', [3, 16, 33, 64])
@pytest.mark.parametrize('dt', DTS, ids=DT_IDS)
def test_hals_sweep_clamped_column(ops, dt, k):
    """V[:, kk] very negative: column kk clamps to eps in every row and comes out as eps / ||eps 1|| exactly (the
    squares sum exactly in float64); the columns after it still match the reference"""
    eps, kk = eps_of(dt), k // 2
    npdt = np.float32 if dt == torch.float32 else np.float64
    for m in (257, sweep_rows('tall3')):
        W, V, G = hals_inputs(m, k, dt, 300 + k)
        V[:, kk] = -1e3
        R = hals_w_ref(W, V, G, eps)
        ops.hals_w_sweep(W, V, G, eps)
        want = npdt(eps) / npdt(np.sqrt(m * eps * eps))
        col = W[:, kk].cpu().numpy()
        assert np.all(col == want), 'clamped column: %d rows differ from %r (m=%d)' % (np.sum(col != want), want, m)
        err = col_err(W[:, kk + 1:], R[:, kk + 1:]) if kk + 1 < k else 0.0
        print('m=%d k=%d: clamped column %d exact; columns after it %.3e (bound %.1e)' % (m, k, kk, err, sweep_bound(dt, k)))
        assert err <= sweep_bound(dt, k)


@pytest.mark.gpu
@pytest.mark.parametrize('dt', DTS, ids=DT_IDS)
def test_hals_sweep_back_to_back(dt):
    """two sweeps on one scratch equal the reference applied twice, the barrier word reads 0 after each launch, and
    a sweep with another k on the same scratch is right (the last CTA out resets the barrier)"""
    from pydnmfk_b200 import device as D
    own = D.DeviceOps()
    eps, m = eps_of(dt), 3 * 256 * 40 + 11

    def gbar():
        torch.cuda.synchronize()
        return int(own._hals_scratch[:4].view(torch.int32).item())

    W, V, G = hals_inputs(m, 20, dt, 400)
    R = hals_w_ref(hals_w_ref(W, V, G, eps), V, G, eps)
    own.hals_w_sweep(W, V, G, eps)
    assert gbar() == 0
    scratch = own._hals_scratch.data_ptr()
    own.hals_w_sweep(W, V, G, eps)
    assert gbar() == 0
    err2 = col_err(W, R)
    W5, V5, G5 = hals_inputs(m, 5, dt, 401)
    R5 = hals_w_ref(W5, V5, G5, eps)
    own.hals_w_sweep(W5, V5, G5, eps)
    assert own._hals_scratch.data_ptr() == scratch, 'the k = 5 sweep must reuse the k = 20 scratch'
    assert gbar() == 0
    err5 = col_err(W5, R5)
    print('two k=20 sweeps %.3e (bound %.1e), then k=5 %.3e (bound %.1e)' % (err2, sweep_bound(dt, 20), err5, sweep_bound(dt, 5)))
    assert err2 <= sweep_bound(dt, 20) and err5 <= sweep_bound(dt, 5)


@pytest.mark.gpu
@pytest.mark.parametrize('dt', DTS, ids=DT_IDS)
def test_hals_sweep_no_rows(ops, dt):
    """m = 0 returns without a launch.  Called through the C-ABI with real pointers: torch gives an empty tensor a
    null data pointer, which every entry point rejects."""
    from pydnmfk_b200 import _lib as L
    k = 5
    buf = torch.zeros((4, 8), dtype=dt, device='cuda')
    G = torch.ones((k, k), dtype=dt, device='cuda')
    scratch = torch.zeros(k * 1024 * 8 + 256, dtype=torch.uint8, device='cuda')
    before = L.launch_count()
    L.call('dnmf_hals_w_sweep', buf.data_ptr(), 8, buf.data_ptr(), 8, G.data_ptr(), 0, k, eps_of(dt), None, 1, 0, 0,
           scratch.data_ptr(), scratch.numel(), L.F32 if dt == torch.float32 else L.F64, ops._stream())
    assert L.launch_count() == before
    assert torch.equal(buf, torch.zeros_like(buf))


@pytest.mark.gpu
@pytest.mark.parametrize('k', K_ALL)
@pytest.mark.parametrize('dt', DTS, ids=DT_IDS)
def test_hals_sweep_matches_column_path(ops, dt, k):
    """hals_w_col + div_col (row grids without the peer exchange) agree with the sweep within the sweep's bound.  They
    are not bit-identical: the sweep adds its per-CTA partials in CTA order, the column path its 256-row block
    partials in a block tree, so the float64 column norms are summed in a different order (in fp64 the factors differ
    in the last bits; in fp32 the norm's rounding to float usually hides it)."""
    eps, worst = eps_of(dt), Worst('%s k=%d' % (DT_IDS[DTS.index(dt)], k))
    for m in (257, 65536, sweep_rows('tall3')):
        W, V, G = hals_inputs(m, k, dt, 500 + k)
        Wc = W.clone()
        ops.hals_w_sweep(W, V, G, eps)
        for kk in range(k):
            ops.div_col(Wc, kk, ops.hals_w_col(Wc, V, G, kk, eps))
        worst.add('sweep vs hals_w_col', col_err(W, Wc), sweep_bound(dt, k), 'm=%d' % m)
    worst.report()


# ======================================================================================================================
# 2. Device-resident BCD
# ======================================================================================================================
def bcd_state_ref(phase, s, x):
    """float64 transcription of the scalar logic of oracle.nmf_oracle.fro_bcd_update, on the layout of dnmf_bcd.cu:
    [0] L_W [1] previous L_W [2] L_H [3] previous L_H [4] obj_old [5] t_old [6] accept [7] ww [8] wh [9] obj [10] rw
    [11] restores so far"""
    s = [float(v) for v in s]
    if phase == 0:
        return [1.0, 1.0, 1.0, 1.0, 0.5 * x, 1.0, 1.0, 0.0, 0.0, 0.0, 1.0, 0.0] + s[12:]
    if phase == 1:
        s[1], s[0] = s[0], float(np.sqrt(x))
    elif phase == 2:
        s[3], s[2] = s[2], float(np.sqrt(x))
    else:
        obj, t_old = 0.5 * x, s[5]
        t = (1 + np.sqrt(1 + 4 * t_old ** 2)) / 2
        s[9] = obj
        if obj >= s[4]:
            s[6], s[11] = 0.0, s[11] + 1
        else:
            w = (t_old - 1) / t
            s[6] = 1.0
            s[7] = float(np.min([w, s[10] * np.sqrt(s[1] / s[0])]))
            s[8] = float(min([w, s[10] * np.sqrt(s[3] / s[2])]))
            s[5], s[4] = float(t), obj
    return s


@pytest.mark.gpu
def test_bcd_state_machine(ops):
    """Every launch of dnmf_bcd_state against the transcription applied to the state before it.  The objectives give
    accept, accept, restore, restore, accept, then obj == obj_old exactly (restore: the test is >=), then accept."""
    Xn = 1000.0
    rounds = [  # (||H H^T||^2, ||W^T W||^2, ||A - W H||^2, accept)
        (4.0, 9.0, 800.0, True),
        (40000.0, 4.0, 600.0, True),          # L_W grows 100x: ww = rw sqrt(L_old / L) < w
        (2.25, 7.0, 700.0, False),
        (1234.5678, 0.3, 601.0, False),
        (3.0, 5.0, 500.0, True),
        (17.0, 11.0, 500.0, False),           # the tie
        (2.0, 3.0, 499.5, True),
    ]
    state = torch.zeros(16, dtype=F64, device='cuda')
    state[12:] = torch.tensor([7.0, 8.0, 9.0, 10.0])          # untouched slots
    script = [(0, Xn)] + [(ph, x) for a, b, c, _ in rounds for ph, x in ((1, a), (2, b), (3, c))]
    exact = [0, 1, 2, 3, 4, 6, 9, 10, 11]
    seq = []
    for phase, x in script:
        before = state.cpu().numpy().copy()
        ops.bcd_state(phase, state, torch.tensor([x], dtype=F64, device='cuda'))
        got = state.cpu().numpy()
        want = np.array(bcd_state_ref(phase, before, x))
        for i in exact + [12, 13, 14, 15]:
            assert got[i] == want[i], 'phase %d: state[%d] = %r, want %r' % (phase, i, got[i], want[i])
        for i in (5, 7, 8):           # t, ww, wh: nvcc may contract 1 + 4 t_old^2 into an FMA
            assert abs(got[i] - want[i]) <= 2 * np.spacing(abs(want[i])), \
                'phase %d: state[%d] = %r, want %r (%.1f ulp)' % (phase, i, got[i], want[i], abs(got[i] - want[i]) / np.spacing(abs(want[i])))
        if phase == 3:
            seq.append(bool(got[6]))
            if not got[6]:
                assert got[5] == before[5] and got[4] == before[4], 'a restore moved t_old or obj_old'
    print('accept / restore:', ''.join('a' if a else 'R' for a in seq))
    assert seq == [r[3] for r in rounds]
    assert state[11].item() == sum(not r[3] for r in rounds)


COUNTS = [1, 255, 257, 1000, 70001]


@pytest.mark.gpu
@pytest.mark.parametrize('count', COUNTS)
@pytest.mark.parametrize('dt', DTS, ids=DT_IDS)
def test_bcd_advance_and_keep(ops, dt, count):
    """bcd_advance: accept gives X + w (X - X_old) within a few ulp (w = state[7] for W, state[8] for H) and
    X_old = X; restore gives Xm = X_old bit for bit and leaves X_old alone.  bcd_keep: both branches bit-exact."""
    X, X_old, junk = urand(count, dt, 1), urand(count, dt, 2), urand(count, dt, 3)
    state = torch.zeros(16, dtype=F64, device='cuda')
    state[7], state[8] = 0.37, 0.81
    ueps = eps_of(dt)
    worst = 0.0
    for which, w in ((0, 0.37), (1, 0.81)):
        state[6] = 1.0
        Xm, Xo = junk.clone(), X_old.clone()
        ops.bcd_advance(X, Xm, Xo, state, which)
        x, xo = X.to(F64), X_old.to(F64)
        err = ((Xm.to(F64) - (x + w * (x - xo))).abs() / ((1 + w) * x.abs() + w * xo.abs())).max().item() / ueps
        worst = max(worst, err)
        assert err <= 4, 'accept, which=%d: %.2f ulp' % (which, err)
        assert torch.equal(Xo, X), 'accept must copy X into X_old'
        state[6] = 0.0
        Xm, Xo = junk.clone(), X_old.clone()
        ops.bcd_advance(X, Xm, Xo, state, which)
        assert torch.equal(Xm, X_old) and torch.equal(Xo, X_old), 'restore: Xm = X_old, X_old untouched'
    print('bcd_advance %s n=%d: accept within %.2f ulp (bound 4)' % (dt, count, worst))
    for acc in (1.0, 0.0):
        state[6] = acc
        cur, kept = X.clone(), X_old.clone()
        ops.bcd_keep(cur, kept, state)
        if acc:
            assert torch.equal(kept, X) and torch.equal(cur, X)
        else:
            assert torch.equal(cur, X_old) and torch.equal(kept, X_old)


@pytest.mark.gpu
@pytest.mark.parametrize('dt', DTS, ids=DT_IDS)
def test_bcd_pg_dev_reads_its_slot(ops, dt):
    """bcd_pg_w_dev / bcd_pg_h_dev bit-identical to bcd_pg_w / bcd_pg_h given the same L on the host; L_W (state[0])
    and L_H (state[2]) differ, and so does every other slot, so reading the wrong one fails"""
    state = torch.arange(16, dtype=F64, device='cuda') + 100.0
    state[0], state[2] = 3.7, 5.3
    for k in K_ALL:
        m, n = 257, 129
        Wm, V, G = urand((m, k), dt, 10), urand((m, k), dt, 11), urand((k, k), dt, 12)
        Hm, Y = urand((k, n), dt, 13), urand((k, n), dt, 14)
        a, b = torch.zeros_like(Wm), torch.zeros_like(Wm)
        ops.bcd_pg_w(a, Wm, V, G, 3.7)
        ops.bcd_pg_w_dev(b, Wm, V, G, state, 0)
        assert torch.equal(a, b), 'bcd_pg_w_dev k=%d' % k
        for yT in (False, True):
            Yarg = Y.T.contiguous() if yT else Y
            a, b = torch.zeros_like(Hm), torch.zeros_like(Hm)
            ops.bcd_pg_h(a, Hm, Yarg, G, 5.3, y_transposed=yT)
            ops.bcd_pg_h_dev(b, Hm, Yarg, G, state, 2, y_transposed=yT)
            assert torch.equal(a, b), 'bcd_pg_h_dev k=%d y_transposed=%s' % (k, yT)


# ---- whole iterations ---------------------------------------------------------------------------------------------
BCD_CASE = dict(m=80, n=60, k=3, noise=0.01, seed=1, itr=60)   # 2 restores, each followed by accepts


def bcd_case_inputs(m, n, k, noise, seed, **_):
    """a rank-k product plus noise: BCD's extrapolation overshoots now and then, so the fit restores"""
    rs = np.random.RandomState(seed)
    A = rs.rand(m, k) @ rs.rand(k, n) + noise * rs.rand(m, n)
    return A, rs.rand(m, k), rs.rand(k, n)


def bcd_transcript(A, W, H, itr):
    """The 1-D single-rank loop of oracle.nmf_oracle.fro_bcd_update in float64 with the same numpy expressions, so it
    reproduces the oracle bit for bit; it also returns the accept / restore decisions and |obj - obj_old| / obj."""
    def sq(x):
        nx = np.linalg.norm(x)
        return nx * nx
    Xnorm, nW, nH = sq(A), sq(W), sq(H)
    W_old = W / np.sqrt(nW) * np.sqrt(np.sqrt(Xnorm))
    H_old = H / np.sqrt(nH) * np.sqrt(np.sqrt(Xnorm))
    Wm, Hm = W_old.copy(), H_old.copy()
    HHT, AHT = np.matmul(H_old, H_old.T), np.matmul(A, H_old.T)
    obj_old, t_old, rw, LW, LH = 0.5 * Xnorm, 1, 1, 1, 1
    accepts, margins = [], []
    for _ in range(itr):
        LW_old, LW = LW, np.linalg.norm(HHT)
        W = np.maximum(0, Wm - (Wm @ HHT - AHT) / LW)
        W = W / np.sum(W, 0, keepdims=True)
        WTW = np.matmul(W.T, W)
        LH_old, LH = LH, np.linalg.norm(WTW)
        H = np.maximum(0, Hm - (WTW @ Hm - np.matmul(W.T, A)) / LH)
        HHT, AHT = np.matmul(H, H.T), np.matmul(A, H.T)
        obj = 0.5 * sq(A - W @ H)
        t = (1 + np.sqrt(1 + 4 * t_old ** 2)) / 2
        margins.append(abs(obj - obj_old) / obj)
        accepts.append(not obj >= obj_old)
        if obj >= obj_old:
            Wm, Hm = W_old.copy(), H_old.copy()
            HHT, AHT = np.matmul(H_old, H_old.T), np.matmul(A, H_old.T)
        else:
            w = (t_old - 1) / t
            ww = np.min([w, rw * np.sqrt(LW_old / LW)])
            wh = min([w, rw * np.sqrt(LH_old / LH)])
            Wm, Hm = W + ww * (W - W_old), H + wh * (H - H_old)
            W_old, H_old = W.copy(), H.copy()
            t_old, obj_old = t, obj
    return W, H, accepts, margins


def _check_bcd_sequence(accepts, margins):
    restores = [i for i, a in enumerate(accepts) if not a]
    assert len(restores) >= 2 and all(i + 1 < len(accepts) and accepts[i + 1] for i in restores), \
        'the case must restore at least twice, each time followed by an accept'
    assert min(margins) > 1e-8, 'a decision within 1e-8 of a tie (%.1e)' % min(margins)


def test_bcd_transcript_matches_oracle():
    """host only: the transcription reproduces oracle.nmf_oracle.fro_bcd_update bit for bit on the chosen case, and the
    case has the restores the GPU test relies on, with a clear margin at every decision"""
    from oracle import nmf_oracle as O
    A, W0, H0 = bcd_case_inputs(**BCD_CASE)
    W, H, accepts, margins = bcd_transcript(A, W0, H0, BCD_CASE['itr'])
    st = O._State()
    st.grid, st.topo, st.k, st.dt = O.VGrid(1, 1), '1d', BCD_CASE['k'], A.dtype
    st.A, st.W, st.H = [A], [W0.copy()], [H0.copy()]
    O.fro_bcd_update(st, BCD_CASE['itr'])
    assert np.array_equal(st.W[0], W) and np.array_equal(st.H[0], H)
    _check_bcd_sequence(accepts, margins)
    print('accept / restore:', ''.join('a' if a else 'R' for a in accepts), ' smallest margin %.1e' % min(margins))


def _bcd_alg(A, W0, H0, k, itr, dtype):
    from pydnmfk_b200.dist_comm import MPI, MPI_comm
    from pydnmfk_b200.dist_nmf import nmf_algorithms_1D
    from pydnmfk_b200.utils import parse
    MPI._reset()
    comm = MPI.COMM_WORLD
    comms = MPI_comm(comm, 1, 1)
    p = parse()
    p.m, p.n, p.p_r, p.p_c, p.k, p.comm1, p.norm, p.method = A.shape[0], A.shape[1], 1, 1, k, comm, 'fro', 'bcd'
    p.row_comm, p.col_comm = comms.cart_1d_row(), comms.cart_1d_column()
    p.eps, p.W_update, p.itr = np.finfo(dtype).eps, True, itr
    dev = lambda x: torch.from_numpy(np.ascontiguousarray(x, dtype=dtype)).cuda()     # noqa: E731
    return nmf_algorithms_1D(dev(A), dev(W0), dev(H0), params=p)


@pytest.mark.gpu
def test_bcd_iterations_follow_host_decisions():
    """fp64, one rank: after every bcd_step the accept flag and the restore counter equal the host sequence, and the
    factors match the oracle at the end"""
    A, W0, H0 = bcd_case_inputs(**BCD_CASE)
    itr, k = BCD_CASE['itr'], BCD_CASE['k']
    Wr, Hr, accepts, margins = bcd_transcript(A, W0, H0, itr)
    _check_bcd_sequence(accepts, margins)
    alg = _bcd_alg(A, W0, H0, k, itr, np.float64)
    alg.bcd_begin()
    got = []
    for i in range(itr):
        alg.bcd_step()
        s = alg._bcd.state.cpu().numpy()
        got.append(bool(s[6]))
        assert s[6] == (1.0 if accepts[i] else 0.0) and s[11] == sum(not a for a in accepts[:i + 1]), \
            'step %d: device %s, host %s' % (i, ''.join('a' if a else 'R' for a in got), ''.join('a' if a else 'R' for a in accepts[:i + 1]))
    dW, dH = rel(alg.W_i, Wr), rel(alg.H_j, Hr)
    print('accept / restore:', ''.join('a' if a else 'R' for a in got), ' W %.2e H %.2e (bound %.0e)' % (dW, dH, T.TOL_FACTOR['float64']))
    assert dW <= T.TOL_FACTOR['float64'] and dH <= T.TOL_FACTOR['float64']


@pytest.mark.gpu
def test_bcd_graph_replay_equals_eager(monkeypatch):
    """fp32: _bcd_loop (step 0 eager, then CUDA-graph replays) is bit-identical to the same number of eager steps,
    state vector included.  Graph capture is switched on through the environment switch the fit reads."""
    from pydnmfk_b200.dist_comm import MPI
    from pydnmfk_b200.graphs import graphs_enabled
    rs = np.random.RandomState(7)
    m, n, k, itr = 1024, 1100, 16, 12
    A = (rs.rand(m, k) @ rs.rand(k, n) + 0.05 * rs.rand(m, n)).astype(np.float32)
    W0, H0 = rs.rand(m, k).astype(np.float32), rs.rand(k, n).astype(np.float32)
    monkeypatch.delenv('DNMF_NO_GRAPH', raising=False)
    g = _bcd_alg(A, W0, H0, k, itr, np.float32)
    assert graphs_enabled(MPI.COMM_WORLD, 'mu') and getattr(g.params, 'cuda_graph', True)
    g._bcd_loop(itr)
    e = _bcd_alg(A, W0, H0, k, itr, np.float32)
    e.bcd_begin()
    for _ in range(itr):
        e.bcd_step()
    torch.cuda.synchronize()
    print('state after %d steps: accept %d, restores %d' % (itr, g._bcd.state[6].item(), g._bcd.state[11].item()))
    assert torch.equal(g.W_i, e.W_i) and torch.equal(g.H_j, e.H_j)
    assert torch.equal(g._bcd.state, e._bcd.state)


# ======================================================================================================================
# 3. Update kernels at every padded width and operand layout
# ======================================================================================================================
# The operands are built the way an iteration meets them.  With G ~ U(0, 1) and L a constant, G H grows like k / 4 and
# the BCD and HALS steps clamp almost every output to 0 or eps once k > 20: a comparison of zeros with zeros that any
# kernel writing zeros, or reading at a wrong index, passes.  So G is the Gram matrix of a factor with unit-norm columns
# (what HALS and BCD see after their column normalisation), L = ||G||_F (BCD's Lipschitz bound), and V / Y are
# consistent with a factor near the current one; every BCD and HALS case asserts that most of its reference is live.
LIVE_SHARE = 0.25          # least share of reference entries above the clamp, per case of >= LIVE_MIN entries
LIVE_MIN = 100


def iter_gram(k, dt, seed):
    """(G, L): G = X^T X for an X with unit-norm, fairly distinct columns (cubed uniforms), so G_kk = 1 and the
    off-diagonal is below 1; L = ||G||_F rounded to dt, so the kernel's (T) L is the reference's L"""
    X = torch.rand((2 * k + 8, k), generator=_gen(seed), device='cuda', dtype=F64) ** 3 + 0.01
    X /= X.norm(dim=0)
    G = (X.T @ X).to(dt)
    return G, float(torch.linalg.norm(G.to(F64)).to(dt))


def near(F, seed):
    """F perturbed by up to +-25 % per entry, in float64: the factor a right-hand side V = F G or Y = G F comes from"""
    return F.to(F64) * (1 + 0.5 * (urand(F.shape, F64, seed) - 0.5))


def pow2_at_least(P):
    """a power of two >= every entry of P: dividing by it is exact, and X - (X G - V) / L stays mostly positive"""
    return float(2.0 ** np.ceil(np.log2(max(float(P.max()), 1.0))))


def assert_live(ref, floor, name, case):
    """the check must not be a comparison of clamped values: most reference entries lie above the clamp"""
    share = float((ref > floor).double().mean())
    if ref.numel() >= LIVE_MIN:
        assert share > LIVE_SHARE, '%s %s: only %.1f %% of the reference above the clamp' % (name, case, 100 * share)
    return share


@pytest.mark.gpu
@pytest.mark.parametrize('k', K_ALL)
@pytest.mark.parametrize('dt', DTS, ids=DT_IDS)
def test_row_side_updates(ops, dt, k):
    """mu_update_w, kl_update_w, bcd_pg_w, div_cols, normalize, clamp_min on W windows (ld = k + 3, NaN padding) at the
    row-block edges of row_update_kernel"""
    eps, tol = eps_of(dt), TOL[dt]
    rb = row_block(dt, k)
    worst = Worst('%s k=%d' % (DT_IDS[DTS.index(dt)], k))
    G, L = iter_gram(k, dt, 20)
    x = urand(k, dt, 21, 0.5)
    G64, x64 = G.to(F64), x.to(F64)
    live = []
    for m in sorted({1, rb - 1, rb, rb + 1, 10000}):
        case = 'm=%d (RB %d)' % (m, rb)
        W0 = urand((m, k), dt, 22 + m)
        V0 = (near(W0, 23 + m) @ G64).to(dt)
        W64, V64 = W0.to(F64), V0.to(F64)
        Vb, V = window(m, k, 5, dt, V0)
        vpad = pad_bits(Vb, k)

        def run(name, fn, ref, bound, src=W0, exact=False):
            Wb, W = window(m, k, 3, dt, src)
            wpad = pad_bits(Wb, k)
            fn(W)
            assert torch.equal(pad_bits(Wb, k), wpad), '%s %s: padding changed' % (name, case)
            if exact:
                assert torch.equal(W.to(F64), ref), '%s %s: not exact' % (name, case)
                worst.add(name, 0.0, 0.0, case)
            else:
                worst.add(name, rel(W, ref), bound, case)

        run('mu_update_w', lambda W: ops.mu_update_w(W, V, G, eps), W64 * (V64 / (W64 @ G64 + eps)), tol)
        run('kl_update_w', lambda W: ops.kl_update_w(W, V, x, eps), W64 * (V64 / (x64[None, :] + eps)), tol)
        Wmb, Wm = window(m, k, 3, dt, W0)
        ref = torch.clamp_min(W64 - (W64 @ G64 - V64) / L, 0)
        live.append(assert_live(ref, 0.0, 'bcd_pg_w', case))
        run('bcd_pg_w', lambda W: ops.bcd_pg_w(W, Wm, V, G, L), ref, 10 * tol, src=torch.zeros_like(W0))
        run('div_cols', lambda W: ops.div_cols(W, x), W64 / x64[None, :], tol)
        Z0 = (urand((m, k), dt, 24 + m) - 0.5).to(dt)
        run('clamp_min', lambda W: ops.clamp_min(W, eps), torch.clamp_min(Z0.to(F64), eps), 0.0, src=Z0, exact=True)
        # normalize: W /= s + eps and H (k x n, a window with ldh > n) *= s
        H0 = urand((k, m), dt, 25 + m)
        Hb, H = window(k, m, 7, dt, H0)
        hpad = pad_bits(Hb, m)
        run('normalize (W)', lambda W: ops.normalize(W, H, x, eps), W64 / (x64[None, :] + eps), tol)
        assert torch.equal(pad_bits(Hb, m), hpad), 'normalize %s: H padding changed' % case
        worst.add('normalize (H)', rel(H, H0.to(F64) * x64[:, None]), tol, case)
        # small integers and L a power of two >= every entry of Wm G: the projected-gradient step is exact
        Wi, Vi, Gi = irand((m, k), dt, 26 + m), irand((m, k), dt, 27 + m, 16), irand((k, k), dt, 28)
        WGi = Wi.to(F64) @ Gi.to(F64)
        Li = pow2_at_least(WGi)
        ref = torch.clamp_min(Wi.to(F64) - (WGi - Vi.to(F64)) / Li, 0)
        live.append(assert_live(ref, 0.0, 'bcd_pg_w integer', case))
        Wib, Wiw = window(m, k, 3, dt, Wi)
        run('bcd_pg_w integer', lambda W: ops.bcd_pg_w(W, Wiw, Vi, Gi, Li), ref, 0.0, src=torch.zeros_like(Wi), exact=True)
        assert torch.equal(pad_bits(Vb, k), vpad), 'V padding changed (%s)' % case
        assert not torch.isnan(Wm).any() and not torch.isnan(Wiw).any()
    print('bcd_pg_w reference entries above the clamp: %s' % ' '.join('%.0f%%' % (100 * v) for v in live))
    worst.report()


Y_LAYOUTS = ['k x n', 'n x k', 'k x n window', 'n x k window']


def y_operand(Y0, layout):
    """Y (k x n) as the kernels may receive it; returns (tensor, y_transposed, buffer or None, padded width)"""
    k, n = Y0.shape
    if layout == 'k x n':
        return Y0.contiguous(), False, None, 0
    if layout == 'n x k':
        return Y0.T.contiguous(), True, None, 0
    if layout == 'k x n window':
        b, v = window(k, n, 5, Y0.dtype, Y0)
        return v, False, b, n
    b, v = window(n, k, 3, Y0.dtype, Y0.T)
    return v, True, b, k


def hals_h_ref(H, Y, G, eps):
    H = H.clone()
    for kk in range(H.shape[0]):
        H[kk, :] = torch.clamp_min(H[kk, :] + Y[kk, :] - G[kk, :] @ H, eps)
    return H


@pytest.mark.gpu
@pytest.mark.parametrize('k', K_ALL)
@pytest.mark.parametrize('dt', DTS, ids=DT_IDS)
def test_col_side_updates(ops, dt, k):
    """mu_update_h and kl_update_h (with and without clamp), hals_h and bcd_pg_h on H windows (ldh = n + 7, NaN
    padding) at the 128-column block edges, with Y as k x n, as its transpose and as windows of both: the staged and
    the strided read of col_update_kernel"""
    from pydnmfk_b200.device import DeviceOps
    eps, tol = eps_of(dt), TOL[dt]
    worst = Worst('%s k=%d' % (DT_IDS[DTS.index(dt)], k))
    G, L = iter_gram(k, dt, 30)
    x = urand(k, dt, 31, 0.5)
    G64, x64 = G.to(F64), x.to(F64)
    paths, live = set(), {}
    for n in (1, 127, 128, 129, 4097):
        case = 'n=%d' % n
        H0 = urand((k, n), dt, 32 + n)
        Y0 = (G64 @ near(H0, 33 + n)).to(dt)
        H64, Y64 = H0.to(F64), Y0.to(F64)
        mu = H64 * (Y64 / (G64.T @ H64 + eps))
        kl = H64 * (Y64 / (x64[:, None] + eps))
        hals_ref = hals_h_ref(H64, Y64, G64, eps)
        bcd_ref = torch.clamp_min(H64 - (G64 @ H64 - Y64) / L, 0)
        # small integers, L a power of two >= every entry of G Hm: the BCD step is exact
        Hi, Yi, Gi = irand((k, n), dt, 34 + n), irand((k, n), dt, 35 + n, 16), irand((k, k), dt, 36)
        Hi64, Yi64, Gi64 = Hi.to(F64), Yi.to(F64), Gi.to(F64)
        Li = pow2_at_least(Gi64 @ Hi64)
        bcd_int_ref = torch.clamp_min(Hi64 - (Gi64 @ Hi64 - Yi64) / Li, 0)
        # HALS with eps = 0 on integers: G upper triangular with unit diagonal and Y = G H + E, E in {-1, 0, 1}, so the
        # exact result is max(H + E, 0); a kernel that reads G or Y at a wrong index differs (the order of the
        # Gauss-Seidel sweep is checked by the float case, whose G is full)
        Gt64 = torch.triu(Gi64, 1) + torch.eye(k, dtype=F64, device='cuda')
        Yt = (Gt64 @ Hi64 + irand((k, n), F64, 37 + n, 3) - 1).to(dt)
        hals_int_ref = hals_h_ref(Hi64, Yt.to(F64), Gt64, 0.0)
        assert torch.equal(hals_int_ref, torch.clamp_min(Hi64 + Yt.to(F64) - Gt64 @ Hi64, 0))
        Gt = Gt64.to(dt)
        for name, ref, floor in (('hals_h', hals_ref, eps), ('bcd_pg_h', bcd_ref, 0.0),
                                 ('bcd_pg_h integer', bcd_int_ref, 0.0), ('hals_h integer', hals_int_ref, 0.0)):
            live.setdefault(name, []).append(assert_live(ref, floor, name, case))
        for layout in Y_LAYOUTS:
            Y, yT, Yb, yw = y_operand(Y0, layout)
            Yint, Yhint = y_operand(Yi, layout)[0], y_operand(Yt, layout)[0]
            sk, _ = DeviceOps._ystrides(Y, yT)
            path = 'staged' if col_stages(dt, k) and sk == 1 else 'strided'
            if n > 1 and k > 1:
                assert path == ('staged' if yT and col_stages(dt, k) else 'strided')
            paths.add(path)
            ypad = pad_bits(Yb, yw) if Yb is not None else None
            case = 'n=%d Y %s (%s)' % (n, layout, path)

            def run(name, fn, ref, bound, src=H0, exact=False):
                Hb, H = window(k, n, 7, dt, src)
                hpad = pad_bits(Hb, n)
                fn(H)
                assert torch.equal(pad_bits(Hb, n), hpad), '%s %s: padding changed' % (name, case)
                if exact:
                    assert torch.equal(H.to(F64), ref), '%s %s: not exact' % (name, case)
                    worst.add(name, 0.0, 0.0, case)
                else:
                    worst.add(name, rel(H, ref), bound, case)

            for clamp in (False, True):
                cname = ' clamp' if clamp else ''
                run('mu_update_h' + cname, lambda H: ops.mu_update_h(H, Y, G, eps, y_transposed=yT, clamp=clamp),
                    mu.clamp_min(eps) if clamp else mu, tol)
                run('kl_update_h' + cname, lambda H: ops.kl_update_h(H, Y, x, eps, y_transposed=yT, clamp=clamp),
                    kl.clamp_min(eps) if clamp else kl, tol)
            run('hals_h', lambda H: ops.hals_h(H, Y, G, eps, y_transposed=yT), hals_ref, 50 * tol)
            Hmb, Hm = window(k, n, 7, dt, H0)
            run('bcd_pg_h', lambda H: ops.bcd_pg_h(H, Hm, Y, G, L, y_transposed=yT), bcd_ref, 10 * tol,
                src=torch.zeros_like(H0))
            Himb, Him = window(k, n, 7, dt, Hi)
            run('bcd_pg_h integer', lambda H: ops.bcd_pg_h(H, Him, Yint, Gi, Li, y_transposed=yT), bcd_int_ref, 0.0,
                src=torch.zeros_like(Hi), exact=True)
            run('hals_h integer', lambda H: ops.hals_h(H, Yhint, Gt, 0.0, y_transposed=yT), hals_int_ref, 0.0, src=Hi,
                exact=True)
            if Yb is not None:
                assert torch.equal(pad_bits(Yb, yw), ypad), 'Y padding changed (%s)' % case
    assert paths == ({'staged', 'strided'} if col_stages(dt, k) else {'strided'}), paths
    print('col_update_kernel read paths at KP=%d: %s' % (kp_of(k), ', '.join(sorted(paths))))
    for name in sorted(live):
        print('%s reference entries above the clamp: %s' % (name, ' '.join('%.0f%%' % (100 * v) for v in live[name])))
    worst.report()


# ======================================================================================================================
# 4. _p updates on synthetic partial views (fp32)
# ======================================================================================================================
def partial_view(rows, k, ldp, splits, seed):
    """`splits` partial buffers [rows][ldp], 37 elements of NaN between them and NaN in columns k..ldp-1; returns the
    int64[4] view, the buffer (kept alive by the caller) and the fp32 sum of the splits in split order"""
    sstride = rows * ldp + 37
    buf = torch.full((splits * sstride,), float('nan'), device='cuda')
    parts = []
    for s in range(splits):
        p = urand((rows, k), torch.float32, seed + s, 0.05)
        buf[s * sstride:s * sstride + rows * ldp].view(rows, ldp)[:, :k] = p
        parts.append(p)
    acc = parts[0].clone()
    for p in parts[1:]:
        acc = acc + p
    return (C.c_int64 * 4)(buf.data_ptr(), ldp, splits, sstride), buf, acc


@pytest.mark.gpu
@pytest.mark.parametrize('k', K_ALL)
def test_p_updates_on_partial_views(ops, k):
    """each _p update is bit-identical to the plain update of the fp32 sum of the splits, added in split order; W layout
    [row][ldp], H layout [column][ldp]"""
    dt, eps = torch.float32, eps_of(torch.float32)
    G, x = urand((k, k), dt, 40), urand(k, dt, 41, 0.5)
    rb, cases = row_block(dt, k), 0
    for splits in (1, 2, 3, 7):
        for ldp in sorted({k, kp_of(k)}):
            for m in (1, rb + 1, 1000):
                view, buf, Vs = partial_view(m, k, ldp, splits, 50 + 10 * splits + m)
                W0 = urand((m, k), dt, 42 + m)
                for name, fp, fplain in (('mu_update_w', ops.mu_update_w_p, ops.mu_update_w),
                                         ('kl_update_w', ops.kl_update_w_p, ops.kl_update_w)):
                    other = G if name.startswith('mu') else x
                    a, b = W0.clone(), W0.clone()
                    fp(a, view, other, eps)
                    fplain(b, Vs, other, eps)
                    assert torch.equal(a, b), '%s_p splits=%d ldp=%d m=%d' % (name, splits, ldp, m)
                    cases += 1
                del buf
            for n in (1, 63, 64, 65, 127, 128, 129, 1000):
                view, buf, Ys = partial_view(n, k, ldp, splits, 60 + 10 * splits + n)     # Ys: n x k
                H0 = urand((k, n), dt, 43 + n)
                for clamp in (False, True):
                    for name, fp, fplain, other in (('mu_update_h', ops.mu_update_h_p, ops.mu_update_h, G),
                                                    ('kl_update_h', ops.kl_update_h_p, ops.kl_update_h, x)):
                        a, b = H0.clone(), H0.clone()
                        fp(a, view, other, eps, clamp=clamp)
                        fplain(b, Ys, other, eps, y_transposed=True, clamp=clamp)
                        assert torch.equal(a, b), '%s_p splits=%d ldp=%d n=%d clamp=%s' % (name, splits, ldp, n, clamp)
                        cases += 1
                del buf
    print('k=%d: %d _p cases bit-identical (splits 1/2/3/7, ldp %s)' % (k, cases, sorted({k, kp_of(k)})))


# ======================================================================================================================
# 5. Generic A-streaming passes at padded widths
# ======================================================================================================================
@pytest.fixture
def generic_ops(ops):
    from pydnmfk_b200 import _lib as L
    L.set_force_generic(True)
    yield ops
    L.set_force_generic(False)


def _check_passes(ops, A, A64, k, dt, seed, tag):
    from pydnmfk_b200 import _lib as L
    m, n = A.shape
    H, W = urand((k, n), dt, seed, 0.05), urand((m, k), dt, seed + 1, 0.05)
    H64, W64 = H.to(F64), W.to(F64)
    eps, tol = eps_of(dt), TOL[dt]
    U = A64 / (W64 @ H64 + eps)
    worst = Worst(tag)
    worst.add('ah', rel(ops.ah(A, H), A64 @ H64.T), tol, '')
    worst.add('wta', rel(ops.wta(A, W), W64.T @ A64), tol, '')
    worst.add('wta transposed_out', rel(ops.wta(A, W, transposed_out=True), A64.T @ W64), tol, '')
    worst.add('kl_uht', rel(ops.kl_uht(A, W, H, eps), U @ H64.T), tol, '')
    worst.add('kl_wtu', rel(ops.kl_wtu(A, W, H, eps), W64.T @ U), tol, '')
    worst.add('kl_wtu transposed_out', rel(ops.kl_wtu(A, W, H, eps, transposed_out=True), U.T @ W64), tol, '')
    assert L.last_path() == 0, 'the generic kernels were expected'
    worst.report()


@pytest.mark.gpu
@pytest.mark.parametrize('m,n,k', [(1000, 700, 20), (333, 1025, 48), (2000, 130, 63), (130, 2000, 33)])
@pytest.mark.parametrize('dt', DTS, ids=DT_IDS)
def test_generic_passes_padded_widths(generic_ops, dt, m, n, k):
    A = urand((m, n), dt, 70)
    _check_passes(generic_ops, A, A.to(F64), k, dt, 71, '%s %dx%d k=%d' % (DT_IDS[DTS.index(dt)], m, n, k))


@pytest.mark.gpu
@pytest.mark.parametrize('dt', DTS, ids=DT_IDS)
def test_generic_passes_unaligned_window(generic_ops, dt):
    """A is a 517 x 1023 window at offset (3, 2) of a buffer with odd lda = 1031: no load is 16-byte aligned"""
    big = urand((530, 1031), dt, 72)
    A = big[3:520, 2:1025]
    assert A.stride(0) == 1031 and A.data_ptr() % 16 != 0
    _check_passes(generic_ops, A, A.to(F64), 48, dt, 73, '%s window k=48' % DT_IDS[DTS.index(dt)])
