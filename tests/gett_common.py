"""Checks of the contraction kernel (be_gett) and the trace closure (be_dot), shared by the host-simulation and GPU suites.

peps_test_gett / peps_test_dot run one call of each with caller-given offset tables, hints, tails and operands (host
buffers uploaded whole), and return the whole C buffer and, for be_gett, the kernel variant its dispatch chose. The
reference is float64 numpy built from the same tables. A kernel passes when every element obeys

    |C - ref| <= (2K + 4) u (|alpha| (|A||B|)_mn + |beta| |C0_mn|),     u = 2^-53,

with the product of absolute values taken over the gathered operands: a single wrong or missing product breaks it, which a
max-norm tolerance does not notice. Operand entries the tables do not address hold NaN, so a read outside the operand shows
up too; C entries they do not address hold a sentinel that must survive bit for bit, and with beta = 0 the addressed
entries of C start as NaN (beta = 0 must not read C).

Variants that differ only in how operands reach shared memory (16- or 8-byte copies, storage layout) or in skipping exact
zeros (structural-zero hints, zero tails) must agree exactly; so must two identical calls. "Exactly" compares values:
+0 and -0 are equal (a tile skipped as a zero tail writes +0 where the computed tile writes alpha * +0)."""
import ctypes as C
import math
import threading

import numpy as np

from peps_b200 import _lib

U = 2.0 ** -53
SENTINEL = -1234.5678
KERNEL_SMALL, KERNEL_LARGE = 1, 2
ALPHA_BETA = [(1.0, 0.0), (-1.0, 1.0), (1.0, 1.0), (0.5, -2.0)]
# worst |C - ref| / bound seen per kernel variant (reported by the GPU suite)
WORST = {}


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double)) if a is not None else None


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32)) if a is not None else None


def _i32(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.int32)


def is_gpu(lib):
    return lib.peps_backend_name() == b"cuda-sm_100a"


# ---- operands -------------------------------------------------------------------------------------------------------
class Op:
    """One walker-batched operand: walker w starts at data[off + w * ws (+ gidx[w * gws] * gs)]."""

    def __init__(self, data, off=0, ws=0, gidx=None, gws=0, gs=0):
        self.data = np.ascontiguousarray(data, dtype=np.float64)
        self.off, self.ws, self.gs, self.gws = int(off), int(ws), int(gs), int(gws)
        self.gidx = _i32(gidx)

    def bases(self, W):
        b = self.off + self.ws * np.arange(W, dtype=np.int64)
        if self.gidx is not None:
            b = b + self.gidx[np.arange(W) * self.gws].astype(np.int64) * self.gs
        return b

    def struct(self):
        g = self.gidx
        return _lib.PepsTestOperand(_dp(self.data), self.data.size, self.off, self.ws, _ip(g), 0 if g is None else g.size,
                                    self.gws, self.gs)

    def aligned(self):
        """The backend's 16-byte test of the base (the device buffer itself is 256-byte aligned)."""
        return self.off % 2 == 0 and self.ws % 2 == 0 and (self.gidx is None or self.gs % 2 == 0)


def store(X, s_fast, off=0, pad=0, ws_pad=0, fill=np.nan):
    """X [W][R][S] stored with S (s_fast) or R the unit-stride index, leading dimension (that index's size + pad), walker
    stride (slab + ws_pad), walker 0 at element `off`. Returns (Op, table of R, table of S); other entries hold `fill`."""
    W, R, S = X.shape
    if s_fast:
        ld = S + pad
        tr, ts, slab = np.arange(R) * ld, np.arange(S), R * ld
    else:
        ld = R + pad
        tr, ts, slab = np.arange(R), np.arange(S) * ld, S * ld
    ws = slab + ws_pad
    data = np.full(off + W * ws + 1, fill)
    for w in range(W):
        data[off + w * ws + tr[:, None] + ts[None, :]] = X[w]
    return Op(data, off, ws), _i32(tr), _i32(ts)


def gathered(slices, cfg, site, s_fast, off=0, pad=0, slice_pad=0):
    """Physical-slice gather as Engine::site_ref forms it: slices [P][R][S] laid out one after the other (slice size gs =
    slab + slice_pad) from element `off`; walker w reads slice cfg[w][site] (gidx = cfg + site, gws = nsites)."""
    P, R, S = slices.shape
    op, tr, ts = store(slices, s_fast, off, pad, slice_pad)
    nsites = cfg.shape[1]
    return Op(op.data, off, 0, cfg.ravel()[site:], nsites, op.ws), tr, ts


# ---- one contraction call -------------------------------------------------------------------------------------------
class Call:
    def __init__(self, M, N, K, am, ak, bk, bn, cm, cn, a_kfast, b_nfast, A, B, Cop, W, alpha=1.0, beta=0.0, klo_m=None,
                 klo_n=None, m_cnt=None, m_scale=0, n_cnt=None, n_scale=0):
        self.M, self.N, self.K, self.W = M, N, K, W
        self.am, self.ak, self.bk, self.bn, self.cm, self.cn = map(_i32, (am, ak, bk, bn, cm, cn))
        self.a_kfast, self.b_nfast = int(a_kfast), int(b_nfast)
        self.A, self.B, self.C = A, B, Cop
        self.alpha, self.beta = float(alpha), float(beta)
        self.klo_m, self.klo_n, self.m_cnt, self.n_cnt = map(_i32, (klo_m, klo_n, m_cnt, n_cnt))
        self.m_scale, self.n_scale = int(m_scale), int(n_scale)

    def but(self, **kw):
        c = Call.__new__(Call)
        c.__dict__.update(self.__dict__)
        for k, v in kw.items():
            setattr(c, k, _i32(v) if k in ("klo_m", "klo_n", "m_cnt", "n_cnt") else v)
        return c

    def with_scalars(self, alpha, beta, rng):
        """The same call with (alpha, beta) and a C0 to match: NaN at the addressed entries when beta = 0."""
        return self.but(alpha=float(alpha), beta=float(beta), C=c_initial(self.C, self.cm, self.cn, self.W, beta, rng))

    def logical(self, w):
        a, b, c = self.A.bases(self.W)[w], self.B.bases(self.W)[w], self.C.bases(self.W)[w]
        Aw = self.A.data[a + self.am[:, None].astype(np.int64) + self.ak[None, :]]
        Bw = self.B.data[b + self.bk[:, None].astype(np.int64) + self.bn[None, :]]
        ci = c + self.cm[:, None].astype(np.int64) + self.cn[None, :]
        return Aw, Bw, ci


def c_initial(cop, cm, cn, W, beta, rng):
    """Copy of the C operand with the addressed entries NaN (beta = 0) or random (beta != 0); the rest keeps its sentinel."""
    data = cop.data.copy()
    for b in cop.bases(W):
        idx = b + np.asarray(cm, np.int64)[:, None] + np.asarray(cn, np.int64)[None, :]
        data[idx] = np.nan if beta == 0.0 else rng.standard_normal(idx.shape)
    return Op(data, cop.off, cop.ws, cop.gidx, cop.gws, cop.gs)


def pairs_ok(fast, other):
    """Planner::pairs_ok: pairs (2i, 2i+1) along the fast table adjacent and even, every offset of the other table even."""
    fast, other = np.asarray(fast), np.asarray(other)
    if fast.size < 2 or fast.size % 2:
        return 0
    return int(bool(np.all(fast[0::2] % 2 == 0) and np.all(fast[1::2] == fast[0::2] + 1) and np.all(other % 2 == 0)))


def expected_variant(call, kernel, tile_m, tile_n):
    """The report peps_test_gett must give for a call that targets this kernel and tile."""
    akf, bkf = call.a_kfast, 1 - call.b_nfast
    if kernel != KERNEL_LARGE:
        return (kernel, tile_m, tile_n, akf, bkf, 0, 0, 0)
    av = pairs_ok(call.ak, call.am) if akf else pairs_ok(call.am, call.ak)
    bv = pairs_ok(call.bk, call.bn) if bkf else pairs_ok(call.bn, call.bk)
    cv = pairs_ok(call.cn, call.cm)
    return (kernel, tile_m, tile_n, akf, bkf, int(av and call.A.aligned()), int(bv and call.B.aligned()),
            int(cv and call.C.aligned()))


def run(lib, call, target=None):
    """One peps_test_gett call: (C buffer, variant report). target = (kernel, tile_m, tile_n): the report must match it
    exactly, with the 16-byte-copy bits the tables and alignments allow. The report is the dispatch decision of be_gett
    (gett_dispatch.h), a host function, so the host simulation gives the same report as the GPU backend."""
    out = np.empty_like(call.C.data)
    var = np.zeros(8, np.int32)
    a, b, c = call.A.struct(), call.B.struct(), call.C.struct()
    rc = lib.peps_test_gett(0, call.W, call.M, call.N, call.K, _ip(call.am), _ip(call.ak), _ip(call.bk), _ip(call.bn),
                            _ip(call.cm), _ip(call.cn), call.a_kfast, call.b_nfast, _ip(call.klo_m), _ip(call.klo_n),
                            _ip(call.m_cnt), call.m_scale, _ip(call.n_cnt), call.n_scale, call.alpha, call.beta, C.byref(a),
                            C.byref(b), C.byref(c), _dp(out), _ip(var))
    assert rc == 0, lib.peps_last_error(None)
    var = tuple(int(v) for v in var)
    if target is not None:
        assert var == expected_variant(call, *target), (var, expected_variant(call, *target))
    return out, var


def check(call, out, var=None):
    """Element-wise bound against the float64 reference, sentinel entries untouched; returns the worst error / bound."""
    cdata = call.C.data
    addressed = np.zeros(cdata.size, bool)
    worst = 0.0
    for w in range(call.W):
        Aw, Bw, ci = call.logical(w)
        assert np.all(np.isfinite(Aw)) and np.all(np.isfinite(Bw)), "test input addresses a NaN filler"
        ref = call.alpha * (Aw @ Bw)
        size = abs(call.alpha) * (np.abs(Aw) @ np.abs(Bw))
        if call.beta != 0.0:
            ref = ref + call.beta * cdata[ci]
            size = size + abs(call.beta) * np.abs(cdata[ci])
        bound = (2 * call.K + 4) * U * size
        got = out[ci]
        assert np.all(np.isfinite(got)), f"walker {w}: non-finite output (beta = {call.beta})"
        err = np.abs(got - ref)
        bad = err > bound
        if bad.any():
            m, n = np.argwhere(bad)[0]
            raise AssertionError(f"walker {w} ({m}, {n}): |C - ref| = {err[m, n]:.3e} > bound {bound[m, n]:.3e} "
                                 f"(C = {got[m, n]!r}, ref = {ref[m, n]!r}); {int(bad.sum())} elements out of bound")
        nz = bound > 0
        if nz.any():
            worst = max(worst, float((err[nz] / bound[nz]).max()))
        addressed[ci.ravel()] = True
    untouched = ~addressed
    assert np.array_equal(out[untouched].view(np.int64), cdata[untouched].view(np.int64)), "an unaddressed C entry changed"
    if var is not None:
        WORST[var] = max(WORST.get(var, 0.0), worst)
    return worst


def same(x, y, what):
    assert np.all(np.isfinite(x)) and np.all(np.isfinite(y)), what
    diff = np.argwhere(x != y)
    assert diff.size == 0, f"{what}: {diff.size} entries differ, first at {diff[0]}: {x[diff[0]]} vs {y[diff[0]]}"


def run_checked(lib, call, target=None):
    out, var = run(lib, call, target)
    check(call, out, var if is_gpu(lib) else None)
    return out, var


# ---- dense cases ----------------------------------------------------------------------------------------------------
def dense_call(rng, W, M, N, K, a_kfast=True, b_nfast=True, offs=(0, 0, 0), pads=(0, 0, 0), ws_pads=(0, 0, 0), A=None,
               B=None, alpha=1.0, beta=0.0, c_pad=2):
    """C[w] = A[w] B[w] with A [W][M][K] stored K-fast or M-fast, B [W][K][N] stored N-fast or K-fast and C [W][M][N] with a
    padded leading dimension (N + c_pad; the padding holds the sentinel)."""
    A = rng.standard_normal((W, M, K)) if A is None else A
    B = rng.standard_normal((W, K, N)) if B is None else B
    if a_kfast:
        Aop, am, ak = store(A, True, offs[0], pads[0], ws_pads[0])
    else:
        Aop, am, ak = store(A, False, offs[0], pads[0], ws_pads[0])
    Bop, bk, bn = store(B, b_nfast, offs[1], pads[1], ws_pads[1])
    Cop, cm, cn = store(np.zeros((W, M, N)), True, offs[2], pads[2] + c_pad, ws_pads[2], fill=SENTINEL)
    call = Call(M, N, K, am, ak, bk, bn, cm, cn, a_kfast, b_nfast, Aop, Bop, Cop, W)
    return call.with_scalars(alpha, beta, rng)


LAYOUTS = [(True, True), (True, False), (False, True), (False, False)]     # (A K-fast, B N-fast)


def case_reference(lib, rng, W, M, N, K, a_kfast, b_nfast, alpha, beta, target=None, **kw):
    call = dense_call(rng, W, M, N, K, a_kfast, b_nfast, alpha=alpha, beta=beta, **kw)
    return run_checked(lib, call, target)


def case_layouts(lib, rng, W, M, N, K, kernel, tile_m, tile_n, alpha=-1.0, beta=1.0):
    """The same logical A and B in all four storage layouts: every run passes the reference and all four agree exactly."""
    A, B = rng.standard_normal((W, M, K)), rng.standard_normal((W, K, N))
    outs = []
    c0 = None
    for akf, bnf in LAYOUTS:
        call = dense_call(rng, W, M, N, K, akf, bnf, A=A, B=B, alpha=alpha, beta=beta)
        if c0 is None:
            c0 = call.C
        call = call.but(C=c0)
        out, _ = run_checked(lib, call, (kernel, tile_m, tile_n))
        outs.append(out)
    for o, lay in zip(outs[1:], LAYOUTS[1:]):
        same(o, outs[0], f"layout {lay} vs {LAYOUTS[0]}")


def case_copy_paths(lib, rng, W, M, N, K, a_kfast, b_nfast, kernel, tile_m, tile_n):
    """16-byte against 8-byte copies: the aligned operands and copies of them at an odd element offset (one operand at a
    time, then all three) give the same C. The aligned run must take every 16-byte path its layout allows."""
    base = dense_call(rng, W, M, N, K, a_kfast, b_nfast, alpha=1.0, beta=1.0)
    out0, var0 = run_checked(lib, base, (kernel, tile_m, tile_n))
    if kernel == KERNEL_LARGE and M % 2 == 0 and N % 2 == 0 and K % 2 == 0:
        assert var0[5:] == (1, 1, 1), var0
    for moved in ("A", "B", "C", "ABC"):
        call = base
        for name in moved:
            op = getattr(call, name)
            data = np.concatenate([[np.nan if name != "C" else SENTINEL], op.data])
            call = call.but(**{name: Op(data, op.off + 1, op.ws, op.gidx, op.gws, op.gs)})
        out, var = run_checked(lib, call, (kernel, tile_m, tile_n))
        if kernel == KERNEL_LARGE:
            for i, name in enumerate("ABC"):
                assert var[5 + i] == (0 if name in moved else var0[5 + i]), (moved, var)
        off = 1 if "C" in moved else 0
        same(out[off:], out0, f"odd offset of {moved}")


def klo_truth(rng, n, K, kind):
    """First possibly non-zero K index per row (column)."""
    if kind == "offset":           # every tile starts at K step 5 (a multiple of neither ring depth)
        return np.minimum(K, 80 + rng.integers(0, 24, n))
    if kind == "per_row":          # changes inside every tile
        return np.minimum(K, 100 + (np.arange(n) * 13) % 150)
    return np.minimum(K, rng.integers(0, K + 1, n))


def zero_below(A, klo_m=None, klo_n=None):
    """A [W][M][K] with A(m, k) = 0 for k < klo_m[m], or B [W][K][N] with B(k, n) = 0 for k < klo_n[n]."""
    A = A.copy()
    if klo_m is not None:
        A[:, np.arange(A.shape[2])[None, :] < np.asarray(klo_m)[:, None]] = 0.0
    if klo_n is not None:
        A[:, np.arange(A.shape[1])[:, None] < np.asarray(klo_n)[None, :]] = 0.0
    return A


def case_hints(lib, rng, W, M, N, K, a_kfast, b_nfast, kind, target=None, alpha=-1.0, beta=1.0, tile_m=64):
    """Structural-zero hints: the hinted call passes the reference and equals the call without hints.
    kind: offset (both sides, K loops start at step 5), per_row (klo_m changes inside every tile), skip (the second row tile
    is all zero, so its K loop is skipped whole and C = beta C0), m_only / n_only (one side), weak (valid hints below the
    true zero structure)."""
    km = klo_truth(rng, M, K, "per_row" if kind == "per_row" else "offset" if kind in ("offset", "skip") else "random")
    kn = klo_truth(rng, N, K, "offset" if kind in ("offset", "skip") else "random")
    if kind == "skip":
        km[tile_m:2 * tile_m] = K
    A = zero_below(rng.standard_normal((W, M, K)), klo_m=km)
    B = zero_below(rng.standard_normal((W, K, N)), klo_n=kn)
    call = dense_call(rng, W, M, N, K, a_kfast, b_nfast, A=A, B=B, alpha=alpha, beta=beta)
    hm, hn = km, kn
    if kind == "m_only":
        hn = None
    elif kind == "n_only":
        hm = None
    elif kind == "weak":
        hm = np.maximum(0, km - rng.integers(0, 40, M))
        hn = np.maximum(0, kn - rng.integers(0, 40, N))
    plain, _ = run_checked(lib, call, target)
    hinted, _ = run_checked(lib, call.but(klo_m=hm, klo_n=hn), target)
    same(hinted, plain, f"hints ({kind}) on vs off")
    if kind == "skip":
        rows = call.cm[tile_m:2 * tile_m, None].astype(np.int64) + call.cn[None, :]
        for w, b in enumerate(call.C.bases(W)):
            c0 = call.C.data[b + rows]
            want = beta * c0 if beta != 0.0 else np.zeros_like(c0)
            assert np.array_equal(hinted[b + rows], want), "a skipped tile must hold beta * C0"


def tail_counts(W, n, scale):
    """Per-walker counts: 0, full, past the end, and partial ones whose limit falls inside a tile."""
    full = -(-n // scale)
    base = [0, full, full + 3, max(1, (n // 2) // scale), max(1, 37 // scale), max(1, (n - 5) // scale)]
    return np.array([base[w % len(base)] for w in range(W)], np.int32)


def case_tails(lib, rng, W, M, N, K, a_kfast, b_nfast, side, scale, alpha, beta, target=None):
    """Per-walker zero tails on the M side (rows of A) or the N side (columns of B): the call with tails passes the
    reference and equals the call without them."""
    A, B = rng.standard_normal((W, M, K)), rng.standard_normal((W, K, N))
    cnt = tail_counts(W, M if side == "m" else N, scale)
    for w in range(W):
        if side == "m":
            A[w, cnt[w] * scale:, :] = 0.0
        else:
            B[w, :, cnt[w] * scale:] = 0.0
    call = dense_call(rng, W, M, N, K, a_kfast, b_nfast, A=A, B=B, alpha=alpha, beta=beta)
    plain, _ = run_checked(lib, call, target)
    kw = dict(m_cnt=cnt, m_scale=scale) if side == "m" else dict(n_cnt=cnt, n_scale=scale)
    tails, _ = run_checked(lib, call.but(**kw), target)
    same(tails, plain, f"zero tails ({side}) on vs off")


def case_gather(lib, rng, W, M, N, K, which, gs_pad, b_nfast=True, a_kfast=False, target=None, alpha=1.0, beta=0.0,
                site=2, nsites=5, phys=3, site_off=0):
    """One operand gathered from per-site slices as Engine::site_ref reads the TPS: gws = nsites, gs = slab + gs_pad
    (odd or even), several walkers reading the same slice."""
    cfg = rng.integers(0, phys, (W, nsites)).astype(np.int32)
    cfg[: min(W, 3), site] = 1                           # at least three walkers read one slice
    if which == "B":
        slices = rng.standard_normal((phys, K, N))
        Bop, bk, bn = gathered(slices, cfg, site, b_nfast, site_off, 0, gs_pad)
        A = rng.standard_normal((W, M, K))
        Aop, am, ak = store(A, a_kfast)
    else:
        slices = rng.standard_normal((phys, M, K))
        Aop, am, ak = gathered(slices, cfg, site, a_kfast, site_off, 0, gs_pad)
        B = rng.standard_normal((W, K, N))
        Bop, bk, bn = store(B, b_nfast)
    Cop, cm, cn = store(np.zeros((W, M, N)), True, 0, 2, fill=SENTINEL)
    call = Call(M, N, K, am, ak, bk, bn, cm, cn, a_kfast, b_nfast, Aop, Bop, Cop, W).with_scalars(alpha, beta, rng)
    out, var = run_checked(lib, call, target)
    return call, out, var


def case_determinism(lib, rng, W, M, N, K, a_kfast, b_nfast, target=None):
    call = dense_call(rng, W, M, N, K, a_kfast, b_nfast, alpha=-1.0, beta=1.0)
    o1, _ = run_checked(lib, call, target)
    o2, _ = run(lib, call, target)
    same(o1, o2, "two identical calls")


# ---- the three hinted chain contractions of Engine::absorb_svd ------------------------------------------------------
def plan(spec, da, db):
    """Planner::get: offset tables and fast-index flags of a row-major einsum (M and N labels in output order, K labels in
    A order)."""
    lhs, lc = spec.split("->")
    la, lb = lhs.split(",")
    dim, sa, sb = {}, {}, {}
    for labels, d, st in ((la, da, sa), (lb, db, sb)):
        acc = 1
        for i in range(len(labels) - 1, -1, -1):
            dim[labels[i]] = d[i]
            st[labels[i]] = acc
            acc *= d[i]
    sc, acc = {}, 1
    for c in reversed(lc):
        sc[c] = acc
        acc *= dim[c]
    ml = "".join(c for c in lc if c in sa and c not in sb)
    nl = "".join(c for c in lc if c in sb and c not in sa)
    kl = "".join(c for c in la if c in sb)

    def table(labels, st):
        t = np.zeros(1, np.int64)
        for c in labels:
            t = (t[:, None] + np.arange(dim[c]) * st[c]).ravel()
        return t.astype(np.int32)

    def fast(labels, st):
        cands = [c for c in labels if dim[c] > 1]
        return min(cands, key=lambda c: st[c]) if cands else None

    fa, fb = fast(la, sa), fast(lb, sb)
    return dict(am=table(ml, sa), ak=table(kl, sa), bk=table(kl, sb), bn=table(nl, sb), cm=table(ml, sc), cn=table(nl, sc),
                a_kfast=int(fa is not None and fa in kl), b_nfast=int(not (fb is not None and fb in kl)), outn=acc)


def site_labels(post):
    """Engine::site_labels(post, 'e', 'p', 'f', 'o')."""
    s = ["?"] * 4
    s[(post + 3) % 4], s[post], s[(post + 1) % 4], s[(post + 2) % 4] = "e", "p", "f", "o"
    return "".join(s)


def r_hint_table(which, k, e, a, p, b):
    """Engine::r_hints: first possibly non-zero K index per row / column of the three chain contractions."""
    if which == 0:
        kk, ee = np.meshgrid(np.arange(k), np.arange(e), indexing="ij")
        return np.minimum(a, np.maximum(0, kk - ee * a)).ravel()
    if which == 1:
        kk = np.repeat(np.arange(k), b)
        return np.minimum(e * p, p * (kk // a))
    return np.minimum(e * a, np.arange(k))


def r_factor(rng, W, rk, e, a, rc):
    """R factor r[k][e][a] of the chain: upper trapezoidal (zero for e * a + a' < k) and zero from row rc[w] on."""
    r = rng.standard_normal((W, rk, e * a))
    r[:, np.arange(e * a)[None, :] < np.arange(rk)[:, None]] = 0.0
    for w in range(W):
        r[w, rc[w]:] = 0.0
    return r.reshape(W, rk, e, a)


def chain_counts(W, rk):
    base = [rk, 0, rk // 2 + 3, 1, rk - 5, rk // 3]
    return np.array([base[w % len(base)] for w in range(W)], np.int32)


def headline_call(rng, which, W, D, chi, post=0):
    """The hinted contractions of absorb_svd at boundary bond chi and PEPS bond D, with r of rk = chi D rows, hints as
    Engine::r_hints builds them and per-walker tails as absorb_svd sets them:
      kepb: apb,kea->kepb (hint on N, tail on N with scale D)
      kofb: kepb,<site>->kofb (hint on M, tail on M with scale chi; the site tensor gathered from per-site slices)
      koj:  kea,eaoj->koj (hint on M, tail on M with scale 1)."""
    rk = chi * D
    rc = chain_counts(W, rk)
    if which == "kepb":
        mps = rng.standard_normal((W, chi, D, chi))
        r = r_factor(rng, W, rk, D, chi, rc)
        pl = plan("apb,kea->kepb", mps.shape[1:], r.shape[1:])
        A, B = mps.reshape(W, -1), r.reshape(W, -1)
        hints = dict(klo_n=r_hint_table(0, rk, D, chi, D, chi), n_cnt=rc, n_scale=D)
        Aop, Bop = Op(A.ravel(), 0, A.shape[1]), Op(B.ravel(), 0, B.shape[1])
    elif which == "kofb":
        tmp = rng.standard_normal((W, rk, D, D, chi))
        tmp[:, np.arange(D)[None, :] < (np.arange(rk) // chi)[:, None]] = 0.0
        for w in range(W):
            tmp[w, rc[w]:] = 0.0
        sl = site_labels(post)
        phys, nsites, site = 2, 7, 3
        slices = rng.standard_normal((phys, D ** 4))
        pl = plan("kepb," + sl + "->kofb", tmp.shape[1:], (D, D, D, D))
        cfg = rng.integers(0, phys, (W, nsites)).astype(np.int32)
        Aop = Op(tmp.reshape(-1), 0, tmp[0].size)
        Bop = Op(slices.ravel(), 0, 0, cfg.ravel()[site:], nsites, D ** 4)
        hints = dict(klo_m=r_hint_table(1, rk, D, chi, D, chi), m_cnt=rc, m_scale=chi)
    else:
        r = r_factor(rng, W, rk, D, chi, rc)
        X = rng.standard_normal((W, D, chi, D, chi))
        pl = plan("kea,eaoj->koj", r.shape[1:], X.shape[1:])
        Aop, Bop = Op(r.ravel(), 0, r[0].size), Op(X.ravel(), 0, X[0].size)
        hints = dict(klo_m=r_hint_table(2, rk, D, chi, 0, 0), m_cnt=rc, m_scale=1)
    Cop = Op(np.zeros(W * pl["outn"]), 0, pl["outn"])
    call = Call(len(pl["am"]), len(pl["bn"]), len(pl["ak"]), pl["am"], pl["ak"], pl["bk"], pl["bn"], pl["cm"], pl["cn"],
                pl["a_kfast"], pl["b_nfast"], Aop, Bop, Cop, W)
    return call.with_scalars(1.0, 0.0, rng), hints


def case_headline(lib, rng, which, W, D, chi, post=0, target=None):
    """The hinted call (hints and tails as absorb_svd passes them) passes the reference and equals the call without
    hints and the call without tails."""
    call, hints = headline_call(rng, which, W, D, chi, post)
    full = call.but(**hints)
    out, var = run_checked(lib, full, target)
    no_hint = {k: (None if k.startswith("klo") else v) for k, v in hints.items()}
    no_tail = {k: (None if k.endswith("cnt") else v) for k, v in hints.items()}
    same(run(lib, call.but(**no_hint), target)[0], out, f"{which}: hints on vs off")
    same(run(lib, call.but(**no_tail), target)[0], out, f"{which}: tails on vs off")
    return var


# ---- trace closure --------------------------------------------------------------------------------------------------
DOT_DIMS = {8192: (8, 16, 64), 131072: (64, 32, 64), 262144: (64, 8, 8, 64)}


def reversed_legs(dims):
    """Engine::reverse_dot tables: a in row-major order, b with the reversed leg order of a."""
    dims = list(dims)
    ak = np.arange(int(np.prod(dims)))
    idx = np.unravel_index(ak, dims)
    bstride = np.cumprod([1] + dims[:-1])
    bk = sum(i * s for i, s in zip(idx, bstride))
    return ak.astype(np.int32), bk.astype(np.int32)


def dot_operands(rng, W, K, gather=False, ws=None):
    """Operand pair of a trace: walker strides `ws` (the default: disjoint slabs) or, with gather, A read from per-site
    slices through a configuration table."""
    ws = K if ws is None else ws
    if gather:
        phys, nsites, site = 3, 4, 1
        cfg = rng.integers(0, phys, (W, nsites)).astype(np.int32)
        A = Op(rng.standard_normal(phys * (K + 1) + 1), 1, 0, cfg.ravel()[site:], nsites, K + 1)
    else:
        A = Op(rng.standard_normal(3 + (W - 1) * ws + K), 3, ws)
    B = Op(rng.standard_normal(5 + (W - 1) * ws + K), 5, ws)
    return A, B


def run_dot(lib, W, K, ak, bk, A, B):
    out = np.empty(W)
    a, b = A.struct(), B.struct()
    assert lib.peps_test_dot(0, W, K, _ip(ak), _ip(bk), C.byref(a), C.byref(b), _dp(out)) == 0, lib.peps_last_error(None)
    return out


def check_dot(W, K, ak, bk, A, B, out):
    ba, bb = A.bases(W), B.bases(W)
    worst = 0.0
    for w in range(W):
        a, b = A.data[ba[w] + ak.astype(np.int64)], B.data[bb[w] + bk.astype(np.int64)]
        ref = float(np.dot(a, b))
        bound = (2 * K + 4) * U * float(np.dot(np.abs(a), np.abs(b)))
        err = abs(out[w] - ref)
        assert math.isfinite(out[w]) and err <= bound, f"walker {w}: |out - ref| = {err:.3e} > {bound:.3e} (K = {K})"
        worst = max(worst, err / bound if bound > 0 else 0.0)
    return worst


def case_dot(lib, rng, W, K, reverse=False, gather=False, ws=None):
    ak, bk = reversed_legs(DOT_DIMS[K]) if reverse else (np.arange(K, dtype=np.int32), np.arange(K, dtype=np.int32))
    A, B = dot_operands(rng, W, K, gather, ws)
    out = run_dot(lib, W, K, ak, bk, A, B)
    worst = check_dot(W, K, ak, bk, A, B, out)
    WORST[("dot", K >= 8192)] = max(WORST.get(("dot", K >= 8192), 0.0), worst)
    return out, (ak, bk, A, B)


def case_dot_regrowth(lib, rng, K=131072):
    """One context on the split path at W = 4, then W = 300 (the partial-sum buffer grows), then W = 4 again. Runs in a
    thread of its own: each host thread gets a fresh default context, so the buffer starts empty."""
    errors = []

    def body():
        try:
            for W in (4, 300, 4):
                case_dot(lib, rng, W, K, ws=97)
        except BaseException as e:        # re-raised in the calling thread
            errors.append(e)

    t = threading.Thread(target=body)
    t.start()
    t.join()
    if errors:
        raise errors[0]


def case_dot_determinism(lib, rng, W, K):
    out, (ak, bk, A, B) = case_dot(lib, rng, W, K, reverse=K in DOT_DIMS)
    same(run_dot(lib, W, K, ak, bk, A, B), out, "two identical traces")
