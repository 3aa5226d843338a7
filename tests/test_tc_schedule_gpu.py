"""The tcgen05 contractions on the multi-unit schedules that production shapes run.

Every tcgen05 kernel is persistent: tc_plan cuts a pass into units (a 128-wide x block times a K split) and CTA b runs
units b, b + grid, b + 2 grid, ...  Ring slots and phases, the running tile counter that deals tiles to the splitter
groups, the accumulator rotation, the B-slot release of tile t - NT, the KL kernel's S-pair ring and per-unit reload of
the x-side factor, and the drain's per-unit partial all carry over from one unit to the next.  The shapes of
test_tc_gpu.py give every CTA one unit, so none of that is exercised there.  Here real shapes go through the library's
own planner and reach: several units per CTA, odd tile counts per unit (lone-tile S pairs), every residue of the
running tile counter at later units (mod 2: the FRO splitter groups, mod 3: the KL ones), ragged x tails, a last split
shorter than the others, and the production schedule (65536^2: 1024 units, 7 per CTA, 1024 tiles per unit).

The schedule of each case is derived from the partial view the library returns and the device's SM count, and the
property a case exists for is asserted, so a planner change that loses it fails the case instead of silently testing
something easier.  Checks:
- the split partials of the _p forms, unit by unit: exact on small-integer data (FRO), within the suite's fp32 bounds
  on uniform data (FRO and KL, next to the generic kernels' error on the same inputs); a failure lists every bad unit
  with its CTA, ordinal on that CTA, tile-counter residues and tile count;
- the fused A H^T + residual pass (MODE 3 of the KL kernel) bit-exact on integer data: V and both norms;
- the plain outputs (global and worst-row error, transposed form bit-equal), the deferred-reduction updates bit-equal
  to pass + update, and determinism at production size;
- the kind::f16 kernel on units of 1, 3 and 7 tiles, exact on integer data.
References are float64 products on the device, in row slabs.  Run with -rP to see each case's schedule and errors.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

EPS = float(np.finfo(np.float32).eps)
BM = 128                     # x-block width of every tcgen05 kernel
SLAB_BYTES = 1 << 30         # float64 bytes of one row slab of a reference
FRO_BOUND, KL_BOUND = 2e-6, 3e-6     # relative Frobenius error of a unit's partial (the bounds of test_tc_gpu.py)
ROW_BOUND = 1e-5             # worst row of V / column of Y; one stale 32-wide tile moves a row of a 65536-long
                             # reduction by ~5e-4, of a 3000-long one by ~1e-2
PROD = 65536                 # the production shard: 65536^2 fp32 (BASELINE cfg1, the cfg2 shard)


@pytest.fixture(scope='module')
def ops():
    from pydnmfk_b200 import _lib as L
    from pydnmfk_b200 import device as D
    L.set_force_generic(False)
    L.set_tc_min_elems(1)
    yield D.default_ops()
    L.set_force_generic(False)
    L.set_tc_min_elems(1 << 20)


def _gen(seed):
    return torch.Generator(device='cuda').manual_seed(seed)


def int_data(shape, seed, dtype=torch.float32):
    """entries in {0, 1, 2, 3}: every product and every sum below stays an exact fp32 integer"""
    return torch.randint(0, 4, shape, generator=_gen(seed), device='cuda', dtype=torch.float32).to(dtype)


def uniform_data(shape, seed, zeros=0.0, out=None):
    """uniform [0, 1), a fraction `zeros` of them exact zeros (KL: a zero of A must stay a zero of U); filled in row
    slabs so that a 16 GiB matrix needs no second matrix-sized temporary"""
    g = _gen(seed)
    A = out if out is not None else torch.empty(shape, device='cuda')
    step = max(1, SLAB_BYTES // (8 * A.shape[1]))
    for i in range(0, A.shape[0], step):
        s = A[i:i + step]
        s.uniform_(generator=g)
        if zeros:
            s[torch.rand(s.shape, generator=g, device='cuda') < zeros] = 0
    return A


def factors(m, n, k, seed, integer):
    """W (m x k), H (k x n): integers in [0, 3], or uniform + 0.05 (S = W H stays away from 0, as test_kl_tensor_path)"""
    if integer:
        return int_data((m, k), seed), int_data((k, n), seed + 1)
    g = _gen(seed)
    return (torch.rand((m, k), generator=g, device='cuda') + 0.05,
            torch.rand((k, n), generator=g, device='cuda') + 0.05)


# ---- the schedule, derived from the library's partial view ------------------------------------------------------------
PROPS = {
    'units>=2': lambda s: s.per_cta >= 2,
    'units>=3': lambda s: s.per_cta >= 3,
    'odd T': lambda s: any(u['T'] % 2 for u in s.units),
    'tile0%2': lambda s: {u['tile0'] % 2 for u in s.units if u['ord'] >= 1} == {0, 1},
    'tile0%3': lambda s: {u['tile0'] % 3 for u in s.units if u['ord'] >= 1} == {0, 1, 2},
    'x tail': lambda s: s.x_len % BM != 0,
    'short split': lambda s: s.splits > 1 and s.units[-1]['T'] < s.per,
}


class Schedule:
    """tc_plan's units as the kernels walk them: unit u = (x block u % x_blocks, split u // x_blocks) runs on CTA
    u % grid as that CTA's (u // grid)-th unit, after tile0 tiles of its earlier units."""

    def __init__(self, x_len, r_len, splits, bk):
        self.x_len, self.r_len, self.splits, self.bk = x_len, r_len, int(splits), bk
        self.sms = torch.cuda.get_device_properties(0).multi_processor_count
        self.x_blocks = -(-x_len // BM)
        self.kt_total = -(-r_len // bk)
        self.per = -(-self.kt_total // self.splits)
        assert -(-self.kt_total // self.per) == self.splits, 'partial view inconsistent with tc_plan'
        n_units = self.x_blocks * self.splits
        self.grid = min(n_units, self.sms)
        done = [0] * self.grid
        self.units = []
        for u in range(n_units):
            xb, sp = u % self.x_blocks, u // self.x_blocks
            T = min(self.kt_total, (sp + 1) * self.per) - sp * self.per
            cta = u % self.grid
            self.units.append(dict(xb=xb, sp=sp, cta=cta, ord=u // self.grid, tile0=done[cta], T=T))
            done[cta] += T
        self.per_cta = max(u['ord'] for u in self.units) + 1

    def r_range(self, sp):
        """reduced indices [lo, hi) of split sp"""
        return sp * self.per * self.bk, min(self.r_len, (sp + 1) * self.per * self.bk)

    def require(self, props):
        missing = [p for p in props if not PROPS[p](self)]
        assert not missing, 'schedule lost %s: %s' % (missing, self)
        return self

    def __str__(self):
        return ('x %d (%d blocks, tail %d) x r %d: %d splits of %d tiles (last %d), %d units on %d CTAs, up to %d per CTA'
                % (self.x_len, self.x_blocks, self.x_len % BM, self.r_len, self.splits, self.per, self.units[-1]['T'],
                   len(self.units), self.grid, self.per_cta))

    def report(self, bad):
        """bad: bool per (split, x block); every bad unit as (xb, split, CTA, ordinal, tile0 % 2, tile0 % 3, T), and
        the count of bad units per ordinal"""
        lines, per_ord, tot_ord = [], {}, {}
        for u in self.units:
            tot_ord[u['ord']] = tot_ord.get(u['ord'], 0) + 1
            if bad[u['sp'], u['xb']]:
                per_ord[u['ord']] = per_ord.get(u['ord'], 0) + 1
                lines.append('(xb %d, split %d, cta %d, ord %d, tile0%%2 %d, tile0%%3 %d, T %d)'
                             % (u['xb'], u['sp'], u['cta'], u['ord'], u['tile0'] % 2, u['tile0'] % 3, u['T']))
        counts = ', '.join('ord %d: %d/%d' % (o, per_ord.get(o, 0), tot_ord[o]) for o in sorted(tot_ord))
        return '%s\n%d bad units; per ordinal %s\n%s' % (self, len(lines), counts, '\n'.join(lines))


def partials(ops, view, x_len):
    """P[split][x][ldp] of a _p call, copied out of the ops workspace before the next call reuses it"""
    P, ldp, splits, stride = (int(v) for v in view)
    assert stride == x_len * ldp
    base = ops._ws.data_ptr()
    nbytes = splits * stride * 4
    assert base <= P and P + nbytes <= base + ops._ws.numel(), 'partials outside the ops workspace'
    return ops._ws[P - base:P - base + nbytes].view(torch.float32).view(splits, x_len, ldp).clone(), splits


# ---- float64 references, per split -------------------------------------------------------------------------------------
def _rows(n):
    return max(1, SLAB_BYTES // (8 * n))


def ref_partials(op, A, W, H, sched):
    """R[split][x][k] in float64: the split's reduced range of the product, for
    ah: A H^T (x = rows), wta: (W^T A)^T (x = columns), kl_uht: U H^T, kl_wtu: (W^T U)^T with U = A / (W H + eps)"""
    m, n = A.shape
    k = H.shape[0] if H is not None else W.shape[1]
    f = torch.float64
    R = torch.zeros((sched.splits, sched.x_len, k), dtype=f, device='cuda')
    H64 = H.to(f) if H is not None else None
    if op in ('ah', 'kl_uht'):
        for i in range(0, m, _rows(n)):
            X = A[i:i + _rows(n)].to(f)
            if op == 'kl_uht':
                X = X / (W[i:i + _rows(n)].to(f) @ H64 + EPS)
            for sp in range(sched.splits):
                lo, hi = sched.r_range(sp)
                R[sp, i:i + X.shape[0]] = X[:, lo:hi] @ H64[:, lo:hi].T
            del X
    else:
        for sp in range(sched.splits):
            lo, hi = sched.r_range(sp)
            for i in range(lo, hi, _rows(n)):
                j = min(hi, i + _rows(n))
                X = A[i:j].to(f)
                W64 = W[i:j].to(f)
                if op == 'kl_wtu':
                    X = X / (W64 @ H64 + EPS)
                R[sp] += (W64.T @ X).T
                del X
    return R


def unit_sq(D):
    """sum of squares of D[split][x][:] per (split, 128-wide x block)"""
    s = torch.nn.functional.pad((D * D).sum(2), (0, -D.shape[1] % BM))
    return s.view(D.shape[0], -1, BM).sum(2)


def rel_rows(got, ref):
    """global relative Frobenius error and the worst per-row one (rows = the x index)"""
    got, ref = got.to(torch.float64), ref.to(torch.float64)
    d = got - ref
    rn = (ref * ref).sum(1)
    rows = torch.sqrt((d * d).sum(1) / torch.where(rn > 0, rn, torch.ones_like(rn)))
    return float(torch.linalg.norm(d) / torch.linalg.norm(ref)), float(rows.max())


# ---- the calls ----------------------------------------------------------------------------------------------------------
def x_len_of(op, A):
    return A.shape[0] if op in ('ah', 'kl_uht', 'res') else A.shape[1]


def r_len_of(op, A):
    return A.shape[1] if op in ('ah', 'kl_uht', 'res') else A.shape[0]


def call_p(ops, op, A, W, H):
    return {'ah': lambda: ops.ah_p(A, H), 'wta': lambda: ops.wta_p(A, W),
            'kl_uht': lambda: ops.kl_uht_p(A, W, H, EPS), 'kl_wtu': lambda: ops.kl_wtu_p(A, W, H, EPS)}[op]()


def call_plain(ops, op, A, W, H, transposed_out=False):
    """x-major result (V, Y^T); transposed_out: Y^T written by the kernel instead of Y transposed here"""
    if op == 'ah':
        return ops.ah(A, H)
    if op == 'kl_uht':
        return ops.kl_uht(A, W, H, EPS)
    if op == 'wta':
        return ops.wta(A, W, transposed_out=True) if transposed_out else ops.wta(A, W).T
    return ops.kl_wtu(A, W, H, EPS, transposed_out=True) if transposed_out else ops.kl_wtu(A, W, H, EPS).T


def run_p(ops, op, A, W, H, bk, props):
    from pydnmfk_b200 import _lib as L
    view = call_p(ops, op, A, W, H)
    assert view is not None and L.last_path() == 1, '%s not served by the tcgen05 path' % op
    P, splits = partials(ops, view, x_len_of(op, A))
    sched = Schedule(x_len_of(op, A), r_len_of(op, A), splits, bk).require(props)
    return P, sched


def check_exact_partials(ops, op, A, W, H, bk, props):
    """each unit's block of the split partials equals its float64 reference exactly; padded columns are 0"""
    k = H.shape[0] if op == 'ah' else W.shape[1]
    P, sched = run_p(ops, op, A, W, H, bk, props)
    R = ref_partials(op, A, W, H, sched)
    assert float(R.abs().max()) < 2 ** 24, 'reference not exact in fp32'
    got = P[:, :, :k].to(torch.float64)
    bad = unit_sq(got - R).cpu().numpy() > 0
    assert torch.equal(got, R) and not bad.any(), '%s %s partials differ:\n%s' % (op, tuple(A.shape), sched.report(bad))
    assert torch.equal(P[:, :, k:], torch.zeros_like(P[:, :, k:])), 'padded columns of the partials are not 0'
    print('%s %s k %d exact: %s' % (op, tuple(A.shape), k, sched))
    return sched


def check_accuracy(ops, op, A, W, H, bound, props, plain=True):
    """per-unit relative error of the split partials <= bound (every unit, reported per ordinal), then the plain
    outputs against the summed reference; the generic kernels' error on the same inputs is printed beside both"""
    from pydnmfk_b200 import _lib as L
    k = H.shape[0]
    P, sched = run_p(ops, op, A, W, H, 32, props)
    R = ref_partials(op, A, W, H, sched)
    e2 = unit_sq(P[:, :, :k].to(torch.float64) - R)
    r2 = unit_sq(R)
    err = torch.sqrt(e2 / torch.where(r2 > 0, r2, torch.ones_like(r2))).cpu().numpy()
    assert torch.equal(P[:, :, k:], torch.zeros_like(P[:, :, k:])), 'padded columns of the partials are not 0'
    Rf = R.sum(0)
    del R, P
    L.set_force_generic(True)
    try:
        G = call_plain(ops, op, A, W, H)
        assert L.last_path() == 0
        g_glob, g_row = rel_rows(G, Rf)
        g_units = rel_units(G, Rf)
    finally:
        L.set_force_generic(False)
    del G
    per_ord = {}
    for u in sched.units:
        per_ord.setdefault(u['ord'], []).append(err[u['sp'], u['xb']])
    spread = ', '.join('ord %d: mean %.2e max %.2e' % (o, np.mean(v), np.max(v)) for o, v in sorted(per_ord.items()))
    msg = ('%s %s k %d: %s\n  per-unit error max %.2e (bound %.0e; generic kernel per x block max %.2e), %s'
           % (op, tuple(A.shape), k, sched, err.max(), bound, g_units, spread))
    assert err.max() <= bound, '%s\n%s' % (msg, sched.report(err > bound))
    if plain:
        out = call_plain(ops, op, A, W, H)
        assert L.last_path() == 1
        glob, row = rel_rows(out, Rf)
        msg += ('\n  plain: global %.2e (bound %.0e, generic %.2e), worst row %.2e (bound %.0e, generic %.2e)'
                % (glob, bound, g_glob, row, ROW_BOUND, g_row))
        assert glob <= bound and row <= ROW_BOUND, msg
        if op in ('wta', 'kl_wtu'):
            assert torch.equal(call_plain(ops, op, A, W, H, transposed_out=True), out), 'transposed_out differs'
    print(msg)
    return sched


def rel_units(G, Rf):
    """worst relative error of the generic result over the 128-wide x blocks (for comparison with the units)"""
    s_d, s_r = unit_sq((G.to(torch.float64) - Rf).unsqueeze(0)), unit_sq(Rf.unsqueeze(0))
    return float(torch.sqrt(s_d / torch.where(s_r > 0, s_r, torch.ones_like(s_r))).max())


def check_residual_exact(ops, A, W, H, props):
    """MODE 3 on integer data: S = W H is exact, so is every per-tile fp32 sum of (a - s)^2 and a^2 and their float64
    sum; V and both norms must equal the float64 ones exactly"""
    from pydnmfk_b200 import _lib as L
    m, n = A.shape
    view = ops.kl_uht_p(A, W, H, EPS)          # MODE 3 runs tc_plan(m, n, 32) like UHT with k <= 32
    assert view is not None
    sched = Schedule(m, n, int(view[2]), 32).require(props)
    L.pass_count(True, reset=True)
    L.pass_count(False, reset=True)
    V, res = ops.ah_residual(A, W, H)
    torch.cuda.synchronize()
    assert L.pass_count(True) == 1 and L.pass_count(False) == 0, 'fused pass did not take the tcgen05 kernel'
    f = torch.float64
    H64 = H.to(f)
    Vr = torch.empty((m, H.shape[0]), dtype=f, device='cuda')
    rr = ar = 0.0
    for i in range(0, m, _rows(n)):
        X = A[i:i + _rows(n)].to(f)
        Vr[i:i + X.shape[0]] = X @ H64.T
        rr += float(((X - W[i:i + X.shape[0]].to(f) @ H64) ** 2).sum())
        ar += float((X * X).sum())
        del X
    assert rr < 2 ** 53 and float(Vr.max()) < 2 ** 24
    Vd = V.to(f)
    bad_rows = ((Vd - Vr) != 0).any(1)
    if bad_rows.any():
        # V is summed over the splits: a bad row marks its x block in every split
        bad = torch.nn.functional.pad(bad_rows, (0, -m % BM)).view(1, sched.x_blocks, BM).any(2)
        bad = bad.expand(sched.splits, -1).cpu().numpy()
        pytest.fail('ah_residual %s: V differs\n%s' % (tuple(A.shape), sched.report(bad)))
    got = res.cpu().numpy()
    assert got[0] == rr and got[1] == ar, 'norms (%r, %r) != float64 (%r, %r); %s' % (got[0], got[1], rr, ar, sched)
    print('ah_residual %s k %d exact: %s' % (tuple(A.shape), H.shape[0], sched))
    return sched


# ---- cases ------------------------------------------------------------------------------------------------------------
# AH / UHT / MODE 3 run on A = m x n (x = rows); WTA / WTU on the transposed shapes (x = columns).  n % 4 == 0 everywhere
# (fp32 shards need lda % 4 == 0).  Property sets verified against tc_plan at 148 SMs; asserted on the device.
TALL = ['units>=3', 'odd T', 'tile0%2', 'tile0%3', 'x tail']
# 75853 x {20, 148, 196}: 593 units, up to 5 per CTA, T = 1 / 5 / 7, x tail 77 (76 for the transposes of 75852 columns)
# 132557 x 20: 1036 units, 7 on every CTA, T = 1 (a lone-tile S pair per unit on every CTA)
FRO_CASES = []
for _k in (10, 32, 48):
    FRO_CASES += [('ah', 75853, 20, _k, TALL), ('ah', 75853, 148, _k, TALL), ('ah', 75853, 196, _k, TALL),
                  ('wta', 20, 75852, _k, TALL), ('wta', 196, 75852, _k, TALL)]
FRO_CASES += [
    # 20000 x 3000: 157 x blocks (tail 32); 5 splits of 19 tiles, last 18 (padded k 16), 6 per CTA
    ('ah', 20000, 3000, 10, ['units>=3', 'odd T', 'short split', 'tile0%2', 'tile0%3', 'x tail']),
    # 4 splits of 24, last 22 (k 32); 3 splits of 32, last 30 (k 64)
    ('ah', 20000, 3000, 32, ['units>=3', 'short split', 'x tail']),
    ('ah', 20000, 3000, 48, ['units>=3', 'short split', 'tile0%3', 'x tail']),
    ('wta', 3000, 20000, 32, ['units>=3', 'short split', 'x tail']),
    # 4096 x 24576, WTA: 192 x blocks, 3 splits of 43, last 42, 4 per CTA
    ('wta', 4096, 24576, 32, ['units>=3', 'odd T', 'short split', 'tile0%2', 'tile0%3']),
    # 37000 x 5000: one split of T = 157, 2 per CTA, x tail 8
    ('ah', 37000, 5000, 32, ['units>=2', 'odd T', 'x tail']),
]
MULTI_SPLIT = (['units>=3', 'short split', 'x tail'], ['units>=3', 'short split', 'tile0%3', 'x tail'])
KL_CASES = []
for _k in (20, 32, 33, 64):
    KL_CASES += [('kl_uht', 75853, 20, _k, TALL), ('kl_uht', 75853, 148, _k, TALL), ('kl_uht', 75853, 196, _k, TALL),
                 ('kl_wtu', 20, 75852, _k, TALL), ('kl_wtu', 196, 75852, _k, TALL),
                 # 4 splits of 24, last 22 (KK 32); 3 splits of 32, last 30 (KK 64, every tile0 residue mod 3)
                 ('kl_uht', 20000, 3000, _k, MULTI_SPLIT[_k > 32]), ('kl_wtu', 3000, 20000, _k, MULTI_SPLIT[_k > 32])]
KL_CASES += [('kl_uht', 132557, 20, 32, TALL), ('kl_wtu', 20, 132556, 32, TALL),
             ('kl_uht', 132557, 20, 64, TALL), ('kl_wtu', 20, 132556, 64, TALL)]
RES_CASES = [(m, n, k, p) for k in (16, 32) for m, n, p in
             [(75853, 20, TALL), (75853, 148, TALL), (75853, 196, TALL), (132557, 20, TALL),
              (20000, 3000, MULTI_SPLIT[0])]]


def _id(c):
    return '%s-%dx%d-k%d' % c[:4]


@pytest.mark.parametrize('case', FRO_CASES, ids=[_id(c) for c in FRO_CASES])
def test_fro_partials_exact(ops, case):
    op, m, n, k, props = case
    A = int_data((m, n), m + n + k)
    W, H = factors(m, n, k, k, integer=True)
    check_exact_partials(ops, op, A, W, H, 32, props)


@pytest.mark.parametrize('case', FRO_CASES, ids=[_id(c) for c in FRO_CASES])
def test_fro_partials_accuracy(ops, case):
    op, m, n, k, props = case
    A = uniform_data((m, n), m + n + k)
    W, H = factors(m, n, k, k, integer=False)
    check_accuracy(ops, op, A, W, H, FRO_BOUND, props)


@pytest.mark.parametrize('case', KL_CASES, ids=[_id(c) for c in KL_CASES])
def test_kl_partials_accuracy(ops, case):
    op, m, n, k, props = case
    A = uniform_data((m, n), m + n + k, zeros=0.2)
    W, H = factors(m, n, k, k, integer=False)
    check_accuracy(ops, op, A, W, H, KL_BOUND, props)


@pytest.mark.parametrize('case', RES_CASES, ids=['res-%dx%d-k%d' % c[:3] for c in RES_CASES])
def test_ah_residual_exact(ops, case):
    m, n, k, props = case
    A = int_data((m, n), m + n + k)
    W, H = factors(m, n, k, k, integer=True)
    check_residual_exact(ops, A, W, H, props)


@pytest.mark.parametrize('m,n,k', [(75853, 148, 32), (75853, 20, 20), (20000, 3000, 32), (20000, 3000, 48)])
def test_deferred_updates_bit_identical(ops, m, n, k):
    """_p pass + _p update (the update sums the split partials itself) == pass + update, on several units per CTA"""
    A = uniform_data((m, n), 7, zeros=0.2)
    W, H = factors(m, n, k, 8, integer=False)
    G_h, G_w = ops.gram(H, trans=True), ops.gram(W, trans=False)
    W1 = W.clone(); ops.mu_update_w(W1, ops.ah(A, H), G_h, EPS)
    W2 = W.clone(); ops.mu_update_w_p(W2, ops.ah_p(A, H), G_h, EPS)
    assert torch.equal(W1, W2), 'FRO W'
    H1 = H.clone(); ops.mu_update_h(H1, ops.wta(A, W, transposed_out=True), G_w, EPS, y_transposed=True)
    H2 = H.clone(); ops.mu_update_h_p(H2, ops.wta_p(A, W), G_w, EPS)
    assert torch.equal(H1, H2), 'FRO H'
    x2, x1 = ops.rowsum(H), ops.colsum(W)
    W1 = W.clone(); ops.kl_update_w(W1, ops.kl_uht(A, W, H, EPS), x2, EPS)
    W2 = W.clone(); ops.kl_update_w_p(W2, ops.kl_uht_p(A, W, H, EPS), x2, EPS)
    assert torch.equal(W1, W2), 'KL W'
    H1 = H.clone(); ops.kl_update_h(H1, ops.kl_wtu(A, W, H, EPS, transposed_out=True), x1, EPS, y_transposed=True)
    H2 = H.clone(); ops.kl_update_h_p(H2, ops.kl_wtu_p(A, W, H, EPS), x1, EPS)
    assert torch.equal(H1, H2), 'KL H'


# ---- kind::f16 (dnmf_tc16.cu) on units of 1, 3 and 7 tiles of 64 ---------------------------------------------------------
A16_CASES = [('ah', 75853, 40, 10), ('ah', 75853, 136, 32), ('ah', 75853, 392, 48),
             ('wta', 40, 75856, 10), ('wta', 392, 75856, 48)]


@pytest.mark.parametrize('fmt', ['float16', 'bfloat16'])
@pytest.mark.parametrize('case', A16_CASES, ids=['%s-%dx%d-k%d' % c for c in A16_CASES])
def test_a16_partials_exact(ops, fmt, case):
    op, m, n, k = case
    A = int_data((m, n), m + n + k, dtype=getattr(torch, fmt))
    W, H = factors(m, n, k, k, integer=True)
    check_exact_partials(ops, op, A, W, H, 64, ['units>=3', 'odd T', 'tile0%2', 'x tail'])


# ---- production: 65536^2, 1024 units, 7 per CTA, 1024 tiles per unit ----------------------------------------------------
PROD_PROPS = ['units>=3']


@pytest.fixture(scope='module')
def prod():
    """one 65536^2 fp32 matrix (16 GiB) for every production test, refilled in place: integer data for the exact
    checks, uniform data with 20 % zeros for the accuracy checks"""
    state = {}

    def get(kind):
        if state.get('kind') != kind:
            if 'A' not in state:
                state['A'] = torch.empty((PROD, PROD), device='cuda')
            A = state['A']
            if kind == 'int':
                step = _rows(PROD)
                g = _gen(1)
                for i in range(0, PROD, step):
                    A[i:i + step].random_(0, 4, generator=g)
            else:
                uniform_data(A.shape, 2, zeros=0.2, out=A)
            state['kind'] = kind
        return state['A']
    yield get
    state.clear()
    torch.cuda.empty_cache()


def _prod_schedule_check(sched):
    assert sched.per_cta == 7 and sched.per == 1024 and all(u['T'] == 1024 for u in sched.units), sched


@pytest.mark.parametrize('op', ['ah', 'wta'])
def test_production_fro_partials_exact(ops, prod, op):
    A = prod('int')
    W, H = factors(PROD, PROD, 32, 3, integer=True)
    _prod_schedule_check(check_exact_partials(ops, op, A, W, H, 32, PROD_PROPS + ['tile0%3']))


@pytest.mark.parametrize('k', [16, 32])
def test_production_ah_residual_exact(ops, prod, k):
    A = prod('int')
    W, H = factors(PROD, PROD, k, 4, integer=True)
    _prod_schedule_check(check_residual_exact(ops, A, W, H, PROD_PROPS + ['tile0%3']))


@pytest.mark.parametrize('op,k', [('ah', 32), ('wta', 32), ('kl_uht', 32), ('kl_wtu', 32), ('kl_uht', 64),
                                  ('kl_wtu', 64)])
def test_production_partials_accuracy(ops, prod, op, k):
    A = prod('uniform')
    W, H = factors(PROD, PROD, k, 5, integer=False)
    _prod_schedule_check(check_accuracy(ops, op, A, W, H, KL_BOUND if op.startswith('kl') else FRO_BOUND,
                                        PROD_PROPS + ['tile0%3']))


def test_production_deterministic(ops, prod):
    A = prod('uniform')
    W, H = factors(PROD, PROD, 32, 6, integer=False)
    for name, f in (('ah', lambda: ops.ah(A, H)), ('wta', lambda: ops.wta(A, W, transposed_out=True)),
                    ('kl_uht', lambda: ops.kl_uht(A, W, H, EPS)), ('kl_wtu', lambda: ops.kl_wtu(A, W, H, EPS)),
                    ('ah_residual', lambda: torch.cat([t.flatten().double() for t in ops.ah_residual(A, W, H)]))):
        assert torch.equal(f(), f()), '%s is not deterministic' % name
