"""Checks of the two factorisation steps of the boundary-MPS compression, shared by the host-simulation and GPU suites.

Every boundary-MPS absorption is a forward chain of R factors (Engine::chain_step) and a backward sweep of truncations
(Engine::truncated_right_vectors). peps_test_chain_step / peps_test_truncated_right_vectors run exactly these two steps
on host matrices inside a context, so they see its walker count, its number type (real, or complex through the real
embedding [[Ar, -Ai], [Ai, Ar]]) and the environment switches its constructor reads.

The references are float64 numpy. Inputs are built with a known answer where possible: Theta = U diag(s) V^H with Haar
U and V (QR of a real or complex Gaussian), so the truth is V, not LAPACK's answer."""
import ctypes as C
import math

import numpy as np

from oracle.bmps import truncation_dim
from peps_b200 import _lib

W = 3
U_EPS = 2.2e-16


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double)) if a is not None else None


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32)) if a is not None else None


def make_ctx(lib, walkers, complex_):
    """A context of `walkers` walkers (the lattice only fixes a valid engine; no TPS is loaded). Environment switches
    must be set before this call: the engine reads them in its constructor."""
    cfg = _lib.PepsConfig(2, 2, 2, 1, walkers, 0, 1, 1, 0.0)
    h = C.c_void_p()
    assert lib.peps_create(C.byref(h), C.byref(cfg)) == 0, lib.peps_last_error(None)
    if complex_:
        assert lib.peps_set_complex(h) == 0, lib.peps_last_error(h)
    return h


class Ctx:
    def __init__(self, lib, walkers, complex_):
        self.lib, self.complex_ = lib, complex_
        self.h = make_ctx(lib, walkers, complex_)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.lib.peps_destroy(self.h)


def _planes(a):
    return np.ascontiguousarray(a.real, dtype=np.float64), np.ascontiguousarray(a.imag, dtype=np.float64)


def run_chain_step(ctx, a, eps=0.0, row_cnt=None, row_scale=0, rank_hint=0, reduce_tall=True):
    """r [W][cap][n] (complex in a complex context), rows, cnt [W], tri."""
    lib, cx = ctx.lib, ctx.complex_
    nw, m, n = a.shape
    cap = min(2 * m, 2 * n) if cx else min(m, n)
    are, aim = _planes(a)
    rre, rim = np.empty((nw, cap, n)), np.empty((nw, cap, n))
    rows, tri = C.c_int32(), C.c_int32()
    cnt = np.empty(nw, dtype=np.int32)
    rc = None if row_cnt is None else np.ascontiguousarray(row_cnt, dtype=np.int32)
    ok = lib.peps_test_chain_step(ctx.h, m, n, _dp(are), _dp(aim) if cx else None, _ip(rc), row_scale, rank_hint, eps,
                                  int(reduce_tall), _dp(rre), _dp(rim) if cx else None, C.byref(rows), _ip(cnt), C.byref(tri))
    assert ok == 0, lib.peps_last_error(ctx.h)
    r = rre + 1j * rim if cx else rre
    return r, rows.value, cnt, tri.value


def run_truncation(ctx, th, dmin, dmax, terr, held):
    """B [W][min(dmax, rows, cols)][cols] (complex in a complex context), kept [W]."""
    lib, cx = ctx.lib, ctx.complex_
    nw, nr, nc = th.shape
    tcap = min(dmax, nr, nc)
    tre, tim = _planes(th)
    bre, bim = np.empty((nw, tcap, nc)), np.empty((nw, tcap, nc))
    kept = np.empty(nw, dtype=np.int32)
    ok = lib.peps_test_truncated_right_vectors(ctx.h, nr, nc, _dp(tre), _dp(tim) if cx else None, dmin, dmax, terr, int(held),
                                               _dp(bre), _dp(bim) if cx else None, _ip(kept))
    assert ok == 0, lib.peps_last_error(ctx.h)
    return (bre + 1j * bim if cx else bre), kept


# ---- inputs ------------------------------------------------------------------------------------------------------------
def gaussian(rng, shape, complex_):
    g = rng.standard_normal(shape)
    return g + 1j * rng.standard_normal(shape) if complex_ else g


def haar(rng, n, k, complex_):
    """n x k with orthonormal columns (QR of a Gaussian)."""
    q, _ = np.linalg.qr(gaussian(rng, (n, k), complex_))
    return q


def with_spectrum(rng, m, n, s, complex_):
    """A = U diag(s) V^H (len(s) <= min(m, n)); returns A and V."""
    k = len(s)
    u, v = haar(rng, m, k, complex_), haar(rng, n, k, complex_)
    return (u * s) @ v.conj().T, v


def round_up(x, g):
    return (x + g - 1) // g * g


def gram(x):
    return x.conj().T @ x


# ---- chain step --------------------------------------------------------------------------------------------------------
def check_gram(r, a, tol=1e-12):
    ref = gram(a)
    scale = np.max(np.abs(ref))
    err = np.max(np.abs(gram(r) - ref))
    assert err <= tol * scale, f"|r^H r - A^H A|_max = {err:.3e} > {tol:g} * {scale:.3e}"


def check_zero_rows(r, rows, cnt):
    for w in range(r.shape[0]):
        assert 0 <= cnt[w] <= rows
        assert np.all(r[w][cnt[w]:] == 0.0), f"walker {w}: rows >= cnt = {cnt[w]} of r are not exactly zero"
    assert np.all(np.isfinite(r))


def chain_full_rank(lib, complex_, m, n):
    """C1: full-rank A, eps = 0 (no deflation): r^H r = A^H A; a real r is upper trapezoidal with all min(m, n) rows."""
    rng = np.random.default_rng(10 + m + 7 * n)
    a = gaussian(rng, (W, m, n), complex_)
    with Ctx(lib, W, complex_) as ctx:
        r, rows, cnt, tri = run_chain_step(ctx, a)
    if complex_:
        assert rows == min(2 * m, 2 * n) and tri == 0
    else:
        kk = min(m, n)
        assert rows == kk and tri == 1
        for w in range(W):
            assert np.all(np.tril(r[w][:, :kk], -1) == 0.0), "the strictly lower part of a real R must be exactly zero"
    assert np.all(cnt == rows)
    check_zero_rows(r, rows, cnt)
    for w in range(W):
        check_gram(r[w], a[w])


def exact_rank_batch(rng, m, n, ranks, complex_):
    """A[w] = U_r S V_r^H of exact rank ranks[w], singular values from 1 down to 1e-3."""
    a = np.zeros((W, m, n), dtype=complex if complex_ else float)
    for w, rk in enumerate(ranks):
        a[w] = with_spectrum(rng, m, n, np.logspace(0, -3, rk), complex_)[0]
    return a


def check_exact_rank(r, rows, cnt, tri, a, ranks, complex_):
    m, n = a.shape[1:]
    kk = min(2 * m, 2 * n) if complex_ else min(m, n)
    gran = 32 if kk >= 128 else 8
    if kk < 16:                                        # too small to deflate: the plain R factor
        assert rows == kk
    elif complex_:
        assert 2 * max(ranks) <= rows <= round_up(2 * max(ranks), gran), (rows, ranks)
        assert tri == 0
    else:
        # Weyl: cnt[w] >= rank. Equality is not guaranteed: the column presort is not a pivoting, and when the leading
        # block of the presorted columns is ill-conditioned (sigma_r = 1e-3 here) the rows just past the rank carry
        # rounding amplified by its condition number, which can exceed eps times the largest row norm (observed:
        # cnt = 41 for rank 40 at 128 x 128 on the host simulation). The Gram bound below still holds.
        assert all(c >= rk for c, rk in zip(cnt, ranks)), f"cnt {list(cnt)} below the exact ranks {list(ranks)}"
        # ... but the deflation must act: a few rows past the rank at most (a step that kept every row would pass the
        # bounds above)
        assert all(c <= rk + 8 for c, rk in zip(cnt, ranks) if rk < kk), f"cnt {list(cnt)} far above the ranks {list(ranks)}"
        print("exact ranks", list(ranks), "cnt", [int(c) for c in cnt])
        assert rows == min(kk, round_up(int(max(cnt)), gran))
        assert tri == 0
    check_zero_rows(r, rows, cnt)
    for w in range(W):
        check_gram(r[w], a[w])


def chain_exact_rank(lib, complex_, m, n, ranks, eps=1e-13):
    """C2: exact-rank A through the rank-revealing step (column presort, early stop, per-walker cnt, gran rounding)."""
    rng = np.random.default_rng(20 + m + 3 * n)
    a = exact_rank_batch(rng, m, n, ranks, complex_)
    with Ctx(lib, W, complex_) as ctx:
        r, rows, cnt, tri = run_chain_step(ctx, a, eps=eps)
    check_exact_rank(r, rows, cnt, tri, a, ranks, complex_)
    return rows, cnt


def chain_graded(lib, complex_, m, n, eps):
    """C3: sigma_i = 10^(-i/16). Every dropped row is below eps * sigma_1, so the Gram matrix moves by at most
    kk eps^2 sigma_1^2 (kk: the smaller side of the factorised matrix, the embedding for complex states) and, by Weyl,
    every singular value above sqrt(kk) eps sigma_1 survives."""
    rng = np.random.default_rng(30 + m + 5 * n)
    k = min(m, n)
    s = 10.0 ** (-np.arange(k) / 16.0)
    a = np.stack([with_spectrum(rng, m, n, s, complex_)[0] for _ in range(W)])
    with Ctx(lib, W, complex_) as ctx:
        r, rows, cnt, tri = run_chain_step(ctx, a, eps=eps)
    kk = min(2 * m, 2 * n) if complex_ else k
    check_zero_rows(r, rows, cnt)
    for w in range(W):
        err = np.linalg.norm(gram(a[w]) - gram(r[w]), 2)
        assert err <= kk * eps ** 2 + 1e-12, f"walker {w}: |A^H A - r^H r|_2 = {err:.3e}"
        if not complex_:
            assert cnt[w] >= int(np.sum(s > math.sqrt(kk) * eps)), (cnt[w], eps)


def chain_row_hint(lib, m, n, o, rc, eps):
    """C4 (real contexts: the complex branch drops the hint): rows >= rc[w] * o of A[w] are zero. The hinted step
    skips them and must give the unhinted answer."""
    rng = np.random.default_rng(40 + m + n)
    a = rng.standard_normal((W, m, n))
    for w in range(W):
        a[w][rc[w] * o:] = 0.0
    with Ctx(lib, W, False) as ctx:
        r0, rows0, cnt0, tri0 = run_chain_step(ctx, a, eps=eps)
        r1, rows1, cnt1, tri1 = run_chain_step(ctx, a, eps=eps, row_cnt=rc, row_scale=o)
    assert (rows1, tri1) == (rows0, tri0) and list(cnt1) == list(cnt0)
    assert np.max(np.abs(r1 - r0)) <= 1e-12 * np.max(np.abs(r0))
    check_zero_rows(r1, rows1, cnt1)
    for w in range(W):
        check_gram(r1[w], a[w])


def chain_zero_walker(lib, complex_, m, n, eps):
    """C5: an all-zero walker inside a batch gives an exactly zero, finite r and leaves the other walkers alone."""
    rng = np.random.default_rng(50 + m + n)
    a = gaussian(rng, (W, m, n), complex_)
    a[1] = 0.0
    with Ctx(lib, W, complex_) as ctx:
        r, rows, cnt, tri = run_chain_step(ctx, a, eps=eps)
    with Ctx(lib, 2, complex_) as ctx:
        r2, rows2, cnt2, tri2 = run_chain_step(ctx, a[[0, 2]], eps=eps)
    assert np.all(np.isfinite(r)) and np.all(r[1] == 0.0)
    assert rows == rows2 and tri == tri2 and [cnt[0], cnt[2]] == list(cnt2)
    for w, w2 in ((0, 0), (2, 1)):
        assert np.max(np.abs(r[w] - r2[w2])) <= 1e-12 * np.max(np.abs(r2[w2]))
        check_gram(r[w], a[w])
    check_zero_rows(r, rows, cnt)


def chain_tall(lib, complex_, m, n, eps, reduce_tall=True):
    """C6: matrices taller than one two-stage CAQR takes (PEPS_QR_MAX_ROWS lowers the limit) are reduced by row chunks
    first (reduce_tall), or handed to one CAQR whatever their height (reduce_tall = 0, the MPS-only chain)."""
    rng = np.random.default_rng(60 + m + n)
    k = min(m, n)
    if eps == 0.0:
        a = gaussian(rng, (W, m, n), complex_)
    else:
        ranks = [max(1, k // 5), max(1, k // 2), k]
        a = exact_rank_batch(rng, m, n, ranks, complex_)
    with Ctx(lib, W, complex_) as ctx:
        r, rows, cnt, tri = run_chain_step(ctx, a, eps=eps, reduce_tall=reduce_tall)
    if eps == 0.0:
        assert rows == (min(2 * m, 2 * n) if complex_ else k) and tri == (0 if complex_ else 1)
        check_zero_rows(r, rows, cnt)
        for w in range(W):
            check_gram(r[w], a[w])
    else:
        check_exact_rank(r, rows, cnt, tri, a, ranks, complex_)


def chain_determinism(lib, complex_, m, n):
    """C7: the same call twice gives bit-identical r, rows and cnt."""
    rng = np.random.default_rng(70)
    a = exact_rank_batch(rng, m, n, [min(m, n) // 4, min(m, n) // 2, min(m, n)], complex_)
    with Ctx(lib, W, complex_) as ctx:
        r0, rows0, cnt0, tri0 = run_chain_step(ctx, a, eps=1e-13)
        r1, rows1, cnt1, tri1 = run_chain_step(ctx, a, eps=1e-13)
    assert (rows0, tri0) == (rows1, tri1) and np.array_equal(cnt0, cnt1)
    assert np.array_equal(r0, r1)


# ---- truncation step ---------------------------------------------------------------------------------------------------
def truncate_both(ctx, th, dmin, dmax, terr):
    """The writer path (held = 0, SVD compression) and the held-tensor path (held = 1, variational sweeps) must agree
    bit for bit."""
    b0, k0 = run_truncation(ctx, th, dmin, dmax, terr, held=False)
    b1, k1 = run_truncation(ctx, th, dmin, dmax, terr, held=True)
    assert np.array_equal(k0, k1)
    assert np.array_equal(b0, b1), "held = 0 and held = 1 differ"
    return b0, k0


def known_svd_batch(rng, nr, nc, complex_, decay=0.93):
    th = np.zeros((W, nr, nc), dtype=complex if complex_ else float)
    vs, ss = [], []
    k = min(nr, nc)
    for w in range(W):
        s = np.sort(decay ** np.arange(k) * (1 + 0.02 * rng.random(k)))[::-1]
        th[w], v = with_spectrum(rng, nr, nc, s, complex_)
        vs.append(v)
        ss.append(s)
    return th, vs, ss


def check_kept_vectors(th, b, t, v, s):
    """b (tcap x nc): t orthonormal rows of V_t^H, zero rows beyond."""
    bt = b[:t]
    assert np.all(np.isfinite(b))
    assert np.max(np.abs(bt @ bt.conj().T - np.eye(t))) < 1e-12
    assert np.all(b[t:] == 0.0), "rows >= kept must be exactly zero"
    # the discarded weight: fails if b held V^T (unconjugated) instead of V^H
    tail = float(np.sum(s[t:] ** 2))
    resid = np.linalg.norm(th - th @ bt.conj().T @ bt) ** 2
    assert abs(resid - tail) <= 1e-10 * tail + 1e-24 * float(np.sum(s ** 2)), (resid, tail)
    # the kept subspace; conditioning ~ eps * s_1 / gap at the cut
    gap = s[t - 1] - (s[t] if t < len(s) else 0.0)
    p_ref = v[:, :t] @ v[:, :t].conj().T
    assert np.max(np.abs(bt.conj().T @ bt - p_ref)) < 50 * U_EPS * s[0] / gap + 1e-13
    # rows in singular-value order, like the reference's Vt: the variational compression compares the singular values of
    # a bond position by position between sweeps
    sv = np.linalg.norm(th @ bt.conj().T, axis=0)
    assert np.all(sv[1:] <= sv[:-1] + 1e-12 * s[0]), f"kept rows are not sorted by singular value: {sv}"


def trunc_known_svd(lib, complex_, nr, nc, dmin, dmax, terr):
    """T1: kept = the TensorToolkit rule on the true spectrum; B = V_t^H."""
    rng = np.random.default_rng(100 + nr + 3 * nc + dmax)
    th, vs, ss = known_svd_batch(rng, nr, nc, complex_)
    with Ctx(lib, W, complex_) as ctx:
        b, kept = truncate_both(ctx, th, dmin, dmax, terr)
    for w in range(W):
        t = truncation_dim(ss[w], dmin, dmax, terr)
        assert kept[w] == t, (w, kept[w], t)
        check_kept_vectors(th[w], b[w], t, vs[w], ss[w])


def trunc_odd_cut(lib, complex_, nr, nc, t):
    """T2: trunc_err between the two copies of s_t in the real embedding: the rule on the embedding keeps 2t - 1
    values, and the complex basis must still hold t vectors."""
    rng = np.random.default_rng(200 + nr + nc + t)
    th, vs, ss = known_svd_batch(rng, nr, nc, complex_, decay=0.8)
    terr = [(0.75 * s[t - 1] ** 2 + np.sum(s[t:] ** 2)) / np.sum(s ** 2) for s in ss]
    for w in range(W):
        assert truncation_dim(ss[w], 1, nc, terr[w]) == t
    for w in range(W):                                 # one trunc_err per call: the walkers share it
        with Ctx(lib, W, complex_) as ctx:
            b, kept = truncate_both(ctx, th, 1, min(nr, nc), terr[w])
        assert kept[w] == t, (kept[w], t)
        check_kept_vectors(th[w], b[w], t, vs[w], ss[w])


def trunc_rank_below_dmin(lib, complex_, nr, nc, ranks, dmin, dmax):
    """T3: rank(Theta[w]) = ranks[w] < dmin (0 = an all-zero walker). The rule on s padded with zeros keeps dmin. The
    first rank rows span the row space; every other row is exactly zero, or orthonormal to the rest and annihilated by
    Theta -- both give the same contraction. Returns which of the two the path produced."""
    rng = np.random.default_rng(300 + nr + nc)
    th = np.zeros((W, nr, nc), dtype=complex if complex_ else float)
    vs = []
    for w, rk in enumerate(ranks):
        if rk:
            th[w], v = with_spectrum(rng, nr, nc, np.logspace(0, -1, rk), complex_)
        else:
            v = np.zeros((nc, 0))
        vs.append(v)
    with Ctx(lib, W, complex_) as ctx:
        b, kept = truncate_both(ctx, th, dmin, dmax, 0.0)
    assert np.all(np.isfinite(b)), "NaN / Inf in B"
    extra = set()
    for w, rk in enumerate(ranks):
        assert kept[w] == min(dmin, nr, nc) == truncation_dim(np.zeros(min(nr, nc)) if rk == 0 else
                                                               np.r_[np.logspace(0, -1, rk), np.zeros(min(nr, nc) - rk)],
                                                               dmin, dmax, 0.0)
        bw = b[w]
        assert np.all(bw[kept[w]:] == 0.0)
        if rk:
            br = bw[:rk]
            assert np.max(np.abs(br @ br.conj().T - np.eye(rk))) < 1e-12
            assert np.max(np.abs(br.conj().T @ br - vs[w] @ vs[w].conj().T)) < 1e-12
        rest = bw[rk:kept[w]]
        for i, row in enumerate(rest):
            if np.all(row == 0.0):
                extra.add("zero")
                continue
            extra.add("orthonormal")
            full = bw[:rk + i + 1]
            assert np.max(np.abs(full @ full.conj().T - np.eye(rk + i + 1))) < 1e-12
            assert np.linalg.norm(th[w] @ row.conj()) <= 1e-12 * max(1.0, np.linalg.norm(th[w], 2))
    return extra


def trunc_identity(lib, complex_, nr, nc, dmin):
    """T4: rows >= cols and cols <= dmin: nothing can be truncated, B is the identity."""
    rng = np.random.default_rng(400 + nr + nc)
    th = gaussian(rng, (W, nr, nc), complex_)
    with Ctx(lib, W, complex_) as ctx:
        b, kept = truncate_both(ctx, th, dmin, dmin + 3, 0.0)
    assert np.all(kept == nc)
    for w in range(W):
        assert np.array_equal(b[w], np.eye(nc))       # the imaginary plane is exactly zero as well


def trunc_mixed_batch(lib, complex_, nr, nc, dmin, dmax, terr):
    """T5: walkers with different spectra and kept counts; each must come out as it does alone, row by row in
    singular-value order, up to the unit factor a singular vector is fixed by (a sign; a phase for complex states: the
    basis Jacobi settles on in each exact pair of singular values of the real embedding depends on the rotation order,
    which depends on the largest row count in the batch)."""
    rng = np.random.default_rng(500 + nr + nc)
    k = min(nr, nc)
    th = np.zeros((W, nr, nc), dtype=complex if complex_ else float)
    for w, d in enumerate((0.3, 0.5, 0.7)):
        th[w] = with_spectrum(rng, nr, nc, d ** np.arange(k), complex_)[0]
    with Ctx(lib, W, complex_) as ctx:
        b, kept = truncate_both(ctx, th, dmin, dmax, terr)
    assert len(set(kept.tolist())) == W, f"the walkers should keep different counts: {kept}"
    for w in range(W):
        with Ctx(lib, 1, complex_) as ctx:
            b1, k1 = truncate_both(ctx, th[w:w + 1], dmin, dmax, terr)
        assert kept[w] == k1[0]
        assert np.all(b[w][kept[w]:] == 0.0)
        for i in range(kept[w]):
            ov = np.vdot(b1[0][i], b[w][i])
            ph = ov / abs(ov)
            assert np.max(np.abs(b[w][i] - ph * b1[0][i])) <= 1e-12, f"walker {w}, row {i} differs from its run alone"


def trunc_determinism(lib, complex_, nr, nc, dmin, dmax, terr):
    """T7: the same call twice gives bit-identical B and kept."""
    rng = np.random.default_rng(700)
    th, _, _ = known_svd_batch(rng, nr, nc, complex_)
    with Ctx(lib, W, complex_) as ctx:
        b0, k0 = run_truncation(ctx, th, dmin, dmax, terr, held=False)
        b1, k1 = run_truncation(ctx, th, dmin, dmax, terr, held=False)
    assert np.array_equal(k0, k1) and np.array_equal(b0, b1)


# ---- a consumer of the row order -----------------------------------------------------------------------------------------
def variational_convergence_real_vs_complex(lib, rows=5, cols=5, D=3, chi=5, W=2, tol=1e-6, max_iter=10):
    """The two-site variational compression stops once the singular values of the last bond, compared position by
    position with those of the previous sweep, move by less than tol. That needs the kept rows in singular-value order.
    A real-valued state in a complex context must stop after the same sweeps as in a real context (counted by the
    truncations, peps_stat 4) and give the same amplitudes; with tol = 0 both run every sweep."""
    from oracle import vmc
    from peps_b200.api import BMPSTruncateParams, SplitIndexTPS, WalkerBatch
    tps = vmc.random_tps(rows, cols, 2, D, seed=33)
    cfgs = np.stack([vmc.shuffled_half_filled_config(rows, cols, 8 + w) for w in range(W)])
    calls, amps = {}, {}
    for t in (tol, 0.0):
        for cx in (False, True):
            b = WalkerBatch(rows, cols, 2, D, W, BMPSTruncateParams.Variational2Site(1, chi, 0.0, t, max_iter), lib=lib)
            if cx:
                b.set_complex()
            b.set_tps(SplitIndexTPS(tps))
            b.set_configs(cfgs)
            b.init_walkers()
            calls[t, cx] = b.stat(4)
            amps[t, cx] = b.amplitudes_c() if cx else b.amplitudes()
            b.close()
    assert calls[tol, False] < calls[0.0, False], "the real context should converge before max_iter sweeps"
    assert calls[tol, True] == calls[tol, False], f"complex context: {calls[tol, True]} truncations, real: {calls[tol, False]}"
    assert calls[0.0, True] == calls[0.0, False]
    for t in (tol, 0.0):
        assert np.max(np.abs(amps[t, True] / amps[t, False] - 1)) < 1e-10
