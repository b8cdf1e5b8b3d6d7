// Walker-batched factorisations used by the boundary-MPS absorption:
//   * caqr()          communication-avoiding R-only Householder QR (flat tree over row blocks, compact-WY
//                     trailing updates as batched contractions on the DMMA pipe). Replaces the reference's
//                     QR(tmp2, ldims, ...) in BMPS::MultiplyMPOSVDCompress_ (bmps_impl.h:817-821); Q is never
//                     formed because the truncation sweep below only needs the R chain.
//   * truncate_rows() one-sided block Jacobi on the rows of Theta followed by the TensorToolkit truncation
//                     rule; returns the kept right singular vectors. Replaces SVD(...) in
//                     BMPS::RightCanonicalizeTruncate (bmps_impl.h:225-263).
// Backend-agnostic host code.
#pragma once
#include <cstdio>
#include <algorithm>
#include <cstdlib>
#include <vector>
#include "tensor.h"

namespace peps {

struct LinalgCtx {
  int W = 0;
  Pool *pool = nullptr;
  Planner *planner = nullptr;
  double *offmax = nullptr;      // [W]
  int32_t *done = nullptr;       // [W]
  std::vector<int32_t> done_host;
  // statistics
  long jacobi_sweeps = 0, jacobi_calls = 0, qr_calls = 0;
  long jacobi_rounds = 0;
  long rows_in = 0, rows_kept = 0;   // Jacobi row counts before / after deflation (summed over calls)
  double deflation_eps = 1e-13;      // rows of R below eps * (largest row norm) are treated as zero (perturbs Theta by <= sqrt(rows) * eps * |Theta|)
  bool presort_columns = true;       // PEPS_PRESORT_COLS=0 switches the column pre-sorting of truncate_rows off
  bool qr_early_stop = true;         // PEPS_QR_EARLY_STOP=0 switches the early termination of the rank-revealing QRs off
  bool z2_sectors = false;           // fermion mode: rows of Theta fall into two parity sectors with disjoint column supports
  int qr_stop_stride = 3;            // trailing-norm check every n-th panel (PEPS_QR_STOP_STRIDE): 1 -> 29.2, 2 -> 29.2, 3 -> 29.4 samples/s, off -> 28.8
  bool small_svd = true;             // PEPS_SMALL_SVD=0 switches the single-CTA SVD path of truncate_rows off
  long small_svd_calls = 0;
  double jacobi_tol = 1e-14;
  int jacobi_inner_sweeps = 1;
  int jacobi_max_sweeps = 40;
};

constexpr size_t kPanelSmemBudget = 150 * 1024;   // bytes for the panel itself
constexpr size_t kJacobiSmemBudget = 168 * 1024;   // panel only; the kernel adds ~56 KB of Gram / rotation state

struct QRLayout { int nb = 0, rb = 0, nrb = 0, m_pad = 0; };
// tallest matrix handed to one two-stage CAQR (the flat tree takes 18 x 576 rows); PEPS_QR_MAX_ROWS lowers it (tests)
inline int qr_max_rows() {
  const char *e = std::getenv("PEPS_QR_MAX_ROWS");      // read per call: cheap next to a factorisation, and tests toggle it
  const int v = e ? std::atoi(e) : 8192;
  return (v < 64 || v > 8192) ? 8192 : v;
}

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

// Preferred row-block height of the CAQR flat tree (PEPS_QR_RB overrides; multiple of 32). Blocks of 256 rows: the panel
// kernel runs two CTAs per SM and the trailing update uses the column-streaming kernel (reflector block resident in
// shared memory); matrices taller than 18 x 256 rows fall back to taller blocks automatically.
inline int qr_pref_rb() {
  static int v = -1;
  if (v < 0) {
    const char *e = std::getenv("PEPS_QR_RB");
    v = e ? std::atoi(e) : 256;
    if (v < 32 || v % 32 != 0) v = 256;
  }
  return v;
}

inline QRLayout qr_layout(int m, int n) {
  (void)n;
  QRLayout L;
  const int nb = 32;
  const int rbmax = (int)(kPanelSmemBudget / (sizeof(double) * nb)) / nb * nb;     // 576 rows: the register panel kernel
  int rb0 = std::min(std::min(rbmax, round_up(m, nb)), std::max(nb, qr_pref_rb() / nb * nb));
  int nrb = (m + rb0 - 1) / rb0;
  const int nrb_max = rbmax / nb;               // the stacked stage-2 panel (nrb * nb rows) must fit the same kernel
  if (nrb > nrb_max) nrb = nrb_max;
  int rb = round_up((m + nrb - 1) / nrb, nb);
  if (rb > rbmax) throw std::runtime_error("qr_layout: matrix too tall for a two-stage CAQR (needs a deeper tree)");
  L.nb = nb; L.rb = rb; L.nrb = (m + rb - 1) / rb; L.m_pad = L.nrb * rb;
  return L;
}

inline GettDesc make_desc(Planner &pl, const std::vector<int32_t> &am, const std::vector<int32_t> &ak,
                          const std::vector<int32_t> &bk, const std::vector<int32_t> &bn,
                          const std::vector<int32_t> &cm, const std::vector<int32_t> &cn, int a_kfast, int b_nfast) {
  GettDesc d;
  d.M = (int)am.size(); d.K = (int)ak.size(); d.N = (int)bn.size();
  d.am = pl.upload(am); d.ak = pl.upload(ak); d.bk = pl.upload(bk); d.bn = pl.upload(bn);
  d.cm = pl.upload(cm); d.cn = pl.upload(cn);
  d.a_kfast = a_kfast; d.b_nfast = b_nfast;
  return d;
}

inline std::vector<int32_t> iota_scaled(int n, int scale, int base = 0) {
  std::vector<int32_t> v((size_t)n);
  for (int i = 0; i < n; ++i) v[(size_t)i] = base + i * scale;
  return v;
}

// In-place R-only QR of A[w] (m x n, row-major, leading dimension n, walker stride ws; the buffer holds
// L.m_pad rows, rows >= m zero). On return rows [0, min(m,n)) hold R (upper trapezoidal), everything else
// in the buffer is zero.
// Early termination of a rank-revealing factorisation (columns pre-sorted by norm, rows of R below eps * max dropped by
// the caller afterwards): once the trailing block of a walker is below 0.1 * eps * (largest column norm) in Frobenius
// norm, every R row still to come would be dropped anyway -- the walker's remaining panels are skipped (device-side
// flags, no host round trip). Rows >= the stopping column then hold the negligible unfactored block instead of R rows /
// zeros; the caller's deflation discards them (their norms are below its threshold by construction).
struct QRStop {
  const double *colnorm2 = nullptr;      // [W][n] squared column norms before the factorisation
  const int32_t *colorder = nullptr;     // [W][n] columns by descending norm
  double eps = 0.0;                      // the caller's deflation threshold (0 disables)
  int first_col = 0;                     // start checking once this many columns are factorised (a rank hint)
};

inline void caqr(LinalgCtx &cx, double *A, long ws, int m, int n, const QRLayout &L, const int32_t *row_cnt = nullptr,
                 int row_scale = 0, const QRStop *stop = nullptr) {
  const int W = cx.W, nb = L.nb, rb = L.rb, nrb = L.nrb, lda = n;
  const int kk = std::min(m, n);
  ++cx.qr_calls;
  if (m <= 1) return;
  Planner &pl = *cx.planner;
  double *Vw = (double *)cx.pool->get(sizeof(double) * (size_t)W * nrb * rb * nb);
  double *Tw = (double *)cx.pool->get(sizeof(double) * (size_t)W * nrb * nb * nb);
  std::vector<int32_t> rowtab1((size_t)nrb * rb);
  for (int b = 0; b < nrb; ++b)
    for (int s = 0; s < rb; ++s) rowtab1[(size_t)b * rb + s] = b * rb + s;
  const int32_t *rowtab1_d = pl.upload(rowtab1);
  // stage-1 row blocks are contiguous: the trailing update fetches its tiles through a tile descriptor when it can
  TileMap tmap;
  const bool have_tmap = (rb % 64 == 0) && nb == 32 && be_make_tile_map(&tmap, A, ws, lda, L.m_pad, n, W, rb / 8, 8);
  // row blocks of <= 256 rows: descriptor with whole-block boxes for the column-streaming trailing update
  TileMap tmapc;
  const bool have_tmapc = rb <= 256 && rb % 16 == 0 && nb == 32 && be_make_tile_map(&tmapc, A, ws, lda, L.m_pad, n, W, rb, 8);
  const int npanel = (kk + nb - 1) / nb;
  const bool stopping = stop && stop->eps > 0.0 && cx.qr_early_stop && npanel > 2;
  int32_t *stopped = nullptr;
  double *stop_acc = nullptr;
  if (stopping) {
    stopped = (int32_t *)cx.pool->get(sizeof(int32_t) * (size_t)W);
    stop_acc = (double *)cx.pool->get(sizeof(double) * (size_t)W);
    be_memset0(stopped, sizeof(int32_t) * (size_t)W);
    be_memset0(stop_acc, sizeof(double) * (size_t)W);
  }
  for (int p = 0; p < npanel; ++p) {
    const int col0 = p * nb, pw = std::min(nb, kk - col0), c1 = col0 + pw, ntrail = n - c1;
    // row blocks above the one holding the diagonal are finished; the diagonal block skips its rows above col0
    const int b0 = col0 / rb, nact = nrb - b0;
    PanelArgs pa;
    pa.A = A; pa.ws = ws; pa.lda = lda; pa.rowtab = rowtab1_d + (size_t)b0 * rb; pa.R = rb; pa.skip0 = col0 - b0 * rb; pa.NI = nact;
    pa.col0 = col0; pa.pw = pw; pa.nbw = nb; pa.Vw = Vw; pa.Tw = Tw; pa.W = W;
    pa.row_cnt = row_cnt; pa.row_scale = row_scale;        // stage 1 only: all-zero row blocks of a walker are skipped
    pa.stopped = stopped;
    be_panel_qr(pa);
    if (ntrail > 0) {
      ApplyArgs ap;
      ap.A = A; ap.ws = ws; ap.lda = lda; ap.rowtab = pa.rowtab; ap.R = rb; ap.NI = nact; ap.col1 = c1; ap.ntrail = ntrail;
      ap.nbw = nb; ap.Vw = Vw; ap.Tw = Tw; ap.W = W;
      if (have_tmap) { ap.tmap = &tmap; ap.row0 = b0 * rb; }
      if (have_tmapc) { ap.tmap_cols = &tmapc; ap.row0 = b0 * rb; }
      ap.row_cnt = row_cnt; ap.row_scale = row_scale; ap.stopped = stopped;
      be_apply_reflector(ap);
    }
    if (nact > 1) {
      // stage 2: stack the local R blocks of the active row blocks and factorise them; update the same rows of the
      // trailing matrix
      const int R2 = nact * pw;
      std::vector<int32_t> rowtab2((size_t)R2);
      for (int b = 0; b < nact; ++b)
        for (int i = 0; i < pw; ++i) rowtab2[(size_t)b * pw + i] = (b0 + b) * rb + (b == 0 ? pa.skip0 : 0) + i;
      PanelArgs p2 = pa;
      p2.rowtab = pl.upload(rowtab2); p2.R = R2; p2.skip0 = 0; p2.NI = 1; p2.row_cnt = nullptr;
      be_panel_qr(p2);
      if (ntrail > 0) {
        ApplyArgs ap;
        ap.A = A; ap.ws = ws; ap.lda = lda; ap.rowtab = p2.rowtab; ap.R = R2; ap.NI = 1; ap.col1 = c1; ap.ntrail = ntrail;
        ap.nbw = nb; ap.Vw = Vw; ap.Tw = Tw; ap.W = W; ap.stopped = stopped;
        be_apply_reflector(ap);
      }
    }
    // the exact trailing norm is a full pass over the trailing block: every `stop_stride`-th panel only (PEPS_QR_STOP_STRIDE)
    if (stopping && ntrail > 0 && c1 < m && c1 >= stop->first_col && p + 1 < npanel && (p % cx.qr_stop_stride) == cx.qr_stop_stride - 1)
      be_trailing_check(A, ws, lda, c1, m, c1, n, stop->colnorm2, stop->colorder, n, 0.01 * stop->eps * stop->eps, stop_acc, stopped, W);
  }
  if (stopping) { cx.pool->put(stopped); cx.pool->put(stop_acc); }
  cx.pool->put(Vw);
  cx.pool->put(Tw);
}

struct JacobiLayout { int bs = 0, nblk = 0, nr_pad = 0; };

inline int jacobi_max_bs() {
  static int v = -1;
  if (v < 0) {
    const char *e = std::getenv("PEPS_JACOBI_BS");
    v = e ? std::atoi(e) : 16;
    if (v != 4 && v != 8 && v != 16) v = 16;
  }
  return v;
}

inline JacobiLayout jacobi_layout(int nr, int nc) {
  JacobiLayout J;
  int ncp = round_up(nc, 8);
  for (int bs : {16, 8, 4}) {
    if (bs > jacobi_max_bs()) continue;
    size_t bytes = (size_t)2 * bs * (ncp + 4) * sizeof(double);
    if (bytes > kJacobiSmemBudget && bs != 4) continue;
    if (bytes > kJacobiSmemBudget) throw std::runtime_error("jacobi_layout: rows too long for the shared-memory panel");
    if (bs > 4 && nr <= bs) continue;            // prefer one pair covering everything for tiny problems
    J.bs = bs;
    break;
  }
  int nblk = (nr + J.bs - 1) / J.bs;
  if (nblk < 2) nblk = 2;
  if (nblk & 1) ++nblk;
  J.nblk = nblk; J.nr_pad = nblk * J.bs;
  return J;
}

// Rows the Theta buffer must provide for truncate_rows(nr, nc).
inline int truncate_buffer_rows(int nr, int nc) {
  return nr > 1 ? std::max(nr, qr_layout(nr, nc).m_pad) : nr;
}

// Theta[w]: nr x nc (leading dimension nc) inside a zero-padded buffer of truncate_buffer_rows(nr,nc) rows.
// Writes B[w] (tcap x nc): the kept right singular vectors (rows), zero rows beyond kept[w].
//   1. R-only QR of Theta (Drmac-Veselic preconditioning: the rows of R are far closer to orthogonal than the
//      rows of Theta, which roughly halves the Jacobi sweeps; Theta and R share right singular vectors).
//   2. rows of R below deflation_eps * max row norm are dropped (backward-stable perturbation); the surviving
//      rows, sorted by norm, form the Jacobi problem (graded spectra shrink it by a large factor).
//   3. one-sided block Jacobi on those rows, then the TensorToolkit truncation rule on the row norms.
inline void truncate_rows(LinalgCtx &cx, double *G, long ws, int nr, int nc, int dmin, int dmax, double trunc_err,
                          int tcap, double *B, long wb, int32_t *kept) {
  const int W = cx.W;
  const int nsv = std::min(nr, nc);
  // 0. columns sorted by decreasing norm (a cheap stand-in for the column pivoting of the preconditioning QR): R comes
  //    out graded along its diagonal and the row Jacobi below needs about half the sweeps (12 -> 6.5 on the boundary
  //    spectra of the bench state). The kept right singular vectors are un-permuted at the end.
  const bool presort = cx.presort_columns && nr > 1 && nc > 1;
  double *Gin = G;
  int32_t *cord = nullptr;
  if (presort) {
    const int brows = truncate_buffer_rows(nr, nc);
    double *cn2 = (double *)cx.pool->get(sizeof(double) * (size_t)W * nc);
    int32_t *ccnt = (int32_t *)cx.pool->get(sizeof(int32_t) * (size_t)W);
    cord = (int32_t *)cx.pool->get(sizeof(int32_t) * (size_t)W * nc);
    be_col_norms2(G, ws, nc, nr, nc, cn2, W);
    be_rank_rows(cn2, nc, 0.0, cord, ccnt, W);
    G = (double *)cx.pool->get(sizeof(double) * (size_t)W * brows * nc);
    if (brows > nr) be_memset0(G, sizeof(double) * (size_t)W * brows * nc);
    be_permute_cols(Gin, ws, nc, nr, nc, cord, 1, G, (long)brows * nc, nc, W);
    ws = (long)brows * nc;
    cx.pool->put(ccnt);
    QRStop st;
    st.colnorm2 = cn2; st.colorder = cord; st.eps = cx.deflation_eps; st.first_col = std::max(0, std::min(dmax, nsv) - 32);
    if (nr > 1) caqr(cx, G, ws, nr, nc, qr_layout(nr, nc), nullptr, 0, &st);
    cx.pool->put(cn2);
  } else if (nr > 1) {
    caqr(cx, G, ws, nr, nc, qr_layout(nr, nc));
  }
  const int kk = nsv;
  double *n2a = (double *)cx.pool->get(sizeof(double) * (size_t)W * kk);
  int32_t *ord = (int32_t *)cx.pool->get(sizeof(int32_t) * (size_t)W * kk);
  int32_t *cnt = (int32_t *)cx.pool->get(sizeof(int32_t) * (size_t)W);
  be_row_norms2(G, ws, nc, kk, nc, n2a, W);
  be_rank_rows(n2a, kk, cx.deflation_eps * cx.deflation_eps, ord, cnt, W);
  cx.done_host.resize((size_t)W);
  be_d2h(cx.done_host.data(), cnt, sizeof(int32_t) * W);
  int nr_eff = 1;
  for (int w = 0; w < W; ++w) nr_eff = std::max(nr_eff, (int)cx.done_host[(size_t)w]);
  cx.rows_in += kk; cx.rows_kept += nr_eff;
  if (cx.small_svd && nr_eff >= 2 && round_up(nr_eff, 8) <= kSmallSvdMaxN && round_up(nc, 32) <= (int)(kPanelSmemBudget / (sizeof(double) * 32)) / 32 * 32) {
    // Second preconditioning + single-CTA Jacobi (Drmac-Veselic): the surviving rows G2 (nr_eff x nc) are factorised
    // G2^T = Q Rt by a tall-skinny QR whose reflectors are KEPT; the one-sided Jacobi runs on the small square factor
    // Rt (n2 x n2, resident in shared memory, all sweeps and the convergence test on the device: no host round trip
    // per sweep); the kept left singular vectors Y of Rt are mapped back by B^T = Q [Y; 0] (reflectors applied in
    // reverse order) and un-permuted. Rows of B: orthonormal to rounding (Q is a product of reflectors, Y comes out
    // of Jacobi with high relative accuracy).
    ++cx.jacobi_calls; ++cx.small_svd_calls;
    const int n2 = round_up(nr_eff, 8), nb = 32;
    const int rb = round_up(nc, 32), kk2 = std::min(nc, n2), npanel = (kk2 + nb - 1) / nb;      // ONE row block (<= 576 rows)
    const long wsT = (long)rb * n2, wsC = (long)rb * tcap;
    double *GT = (double *)cx.pool->get(sizeof(double) * (size_t)W * wsT);
    be_memset0(GT, sizeof(double) * (size_t)W * wsT);
    be_gather_rows_transposed(G, ws, nc, nc, kk, ord, cnt, GT, wsT, n2, W);
    double *Vall = (double *)cx.pool->get(sizeof(double) * (size_t)npanel * W * rb * nb);
    double *Tall = (double *)cx.pool->get(sizeof(double) * (size_t)npanel * W * nb * nb);
    const int32_t *rowtab = cx.planner->upload(iota_scaled(rb, 1));
    TileMap tmT, tmC;
    const bool mapT = (rb % 64 == 0) && be_make_tile_map(&tmT, GT, wsT, n2, rb, n2, W, rb / 8, 8);
    for (int p = 0; p < npanel; ++p) {
      const int col0 = p * nb, pw = std::min(nb, kk2 - col0), c1 = col0 + pw, ntrail = n2 - c1;
      PanelArgs pa;
      pa.A = GT; pa.ws = wsT; pa.lda = n2; pa.rowtab = rowtab; pa.R = rb; pa.skip0 = col0; pa.NI = 1;
      pa.col0 = col0; pa.pw = pw; pa.nbw = nb; pa.Vw = Vall + (size_t)p * W * rb * nb; pa.Tw = Tall + (size_t)p * W * nb * nb; pa.W = W;
      be_panel_qr(pa);
      if (ntrail > 0) {
        ApplyArgs ap;
        ap.A = GT; ap.ws = wsT; ap.lda = n2; ap.rowtab = rowtab; ap.R = rb; ap.NI = 1; ap.col1 = c1; ap.ntrail = ntrail;
        ap.nbw = nb; ap.Vw = pa.Vw; ap.Tw = pa.Tw; ap.W = W;
        if (mapT) { ap.tmap = &tmT; ap.row0 = 0; }
        be_apply_reflector(ap);
      }
    }
    double *C0 = (double *)cx.pool->get(sizeof(double) * (size_t)W * wsC);
    be_memset0(C0, sizeof(double) * (size_t)W * wsC);
    SmallSvdArgs sa;
    sa.Rt = GT; sa.ws = wsT; sa.ld = n2; sa.n2 = n2; sa.count = cnt; sa.nsv = nsv; sa.dmin = dmin; sa.dmax = dmax;
    sa.trunc_err = trunc_err; sa.tcap = tcap; sa.tol = cx.jacobi_tol; sa.max_sweeps = cx.jacobi_max_sweeps;
    sa.out = C0; sa.wo = wsC; sa.kept = kept; sa.sweeps = nullptr; sa.W = W;
    be_svd_small(sa);
    const bool mapC = (rb % 64 == 0) && be_make_tile_map(&tmC, C0, wsC, tcap, rb, tcap, W, rb / 8, 8);
    for (int p = npanel - 1; p >= 0; --p) {
      ApplyArgs ap;
      ap.A = C0; ap.ws = wsC; ap.lda = tcap; ap.rowtab = rowtab; ap.R = rb; ap.NI = 1; ap.col1 = 0; ap.ntrail = tcap;
      ap.nbw = nb; ap.Vw = Vall + (size_t)p * W * rb * nb; ap.Tw = Tall + (size_t)p * W * nb * nb; ap.W = W; ap.notrans = 1;
      if (mapC) { ap.tmap = &tmC; ap.row0 = 0; }
      be_apply_reflector(ap);
    }
    be_transpose_permute(C0, wsC, nc, tcap, presort ? cord : nullptr, B, wb, W);
    for (void *p : {(void *)GT, (void *)Vall, (void *)Tall, (void *)C0, (void *)n2a, (void *)ord, (void *)cnt}) cx.pool->put(p);
    if (presort) { cx.pool->put(cord); cx.pool->put(G); }
    return;
  }
  JacobiLayout J = jacobi_layout(nr_eff, nc);
  double *G2 = (double *)cx.pool->get(sizeof(double) * (size_t)W * J.nr_pad * nc);
  const long ws2 = (long)J.nr_pad * nc;
  be_gather_rows(G, ws, nc, nc, kk, ord, cnt, G2, ws2, J.nr_pad, W);
  long ws2cur = ws2;
  // Z2 sectors (fermion mode): regroup the rows so that every block of the Jacobi schedule is sector-pure and skip the block
  // pairs of different sectors (exactly orthogonal: disjoint column supports); half of the block pairs remain.
  int32_t *bsec = nullptr, *cwin = nullptr, *cord2 = nullptr;
  const bool sectors = cx.z2_sectors && nr_eff > 2 * J.bs;
  if (sectors) {
    JacobiLayout Jz = J;
    Jz.nblk = (nr_eff + J.bs - 1) / J.bs + 1;                       // one extra block: each sector is padded to whole blocks
    if (Jz.nblk & 1) ++Jz.nblk;
    Jz.nr_pad = Jz.nblk * J.bs;
    double *Gz = (double *)cx.pool->get(sizeof(double) * (size_t)W * Jz.nr_pad * nc);
    be_memset0(Gz, sizeof(double) * (size_t)W * Jz.nr_pad * nc);
    bsec = (int32_t *)cx.pool->get(sizeof(int32_t) * (size_t)W * Jz.nblk);
    cwin = (int32_t *)cx.pool->get(sizeof(int32_t) * (size_t)W * 4);
    cord2 = (int32_t *)cx.pool->get(sizeof(int32_t) * (size_t)W * nc);       // column order: presort composed with the sector grouping
    be_sector_arrange(G2, ws2, nc, nc, cnt, J.bs, Jz.nblk, Gz, (long)Jz.nr_pad * nc, bsec, presort ? cord : nullptr, cord2, cwin, W);
    cx.pool->put(G2);
    G2 = Gz; J = Jz; ws2cur = (long)Jz.nr_pad * nc; nr_eff = Jz.nr_pad;
  }
  if (nr_eff > 1) {
    ++cx.jacobi_calls;
    be_fill(cx.offmax, 0.0, W);
    be_memset0(cx.done, sizeof(int32_t) * W);
    JacobiArgs ja;
    ja.G = G2; ja.ws = ws2cur; ja.ld = nc; ja.nr_pad = J.nr_pad; ja.nc = nc; ja.bs = J.bs; ja.nblk = J.nblk;
    ja.tol = cx.jacobi_tol; ja.inner_sweeps = cx.jacobi_inner_sweeps; ja.offmax = cx.offmax; ja.done = cx.done; ja.W = W;
    ja.nactive = W;
    ja.bsec = bsec; ja.cwin = cwin;
    for (int sweep = 0; sweep < cx.jacobi_max_sweeps; ++sweep) {
      for (int round = 0; round < ja.nblk - 1; ++round) {
        ja.round = round;
        be_jacobi_round(ja);
      }
      ++cx.jacobi_sweeps;
      cx.jacobi_rounds += ja.nblk - 1;
      be_jacobi_flags(cx.offmax, cx.done, ja.tol, W);
      be_d2h(cx.done_host.data(), cx.done, sizeof(int32_t) * W);
      int nact = 0;
      for (int w = 0; w < W; ++w) nact += cx.done_host[(size_t)w] ? 0 : 1;
      ja.nactive = nact;
      if (nact == 0 && ja.bsec) {
        // sector phase converged: finish with unrestricted sweeps over ALL pairs at a looser threshold. Cross-sector pairs
        // are orthogonal to rounding noise (1e-16 .. 1e-14 relative), a mislabelled row would show O(1e-3 .. 1) overlaps:
        // pairs below 1e-11 leave after their Gram matrix (no rotation), anything above is rotated -- a wrong label costs
        // time, never accuracy (an unrotated 1e-11 overlap perturbs a kept vector by <= 1e-11, below the 1e-10 parity bar).
        ja.bsec = nullptr;
        ja.tol = std::max(cx.jacobi_tol, 1e-11);
        be_memset0(cx.done, sizeof(int32_t) * W);
        ja.nactive = W;
        continue;
      }
      if (nact == 0) break;
      // dynamic deflation: after a sweep the row norms track the singular values far better than the rows of R
      // did; rows that fell below deflation_eps * max are dropped and the problem is re-compacted when that
      // removes at least one block pair worth of work.
      if (!sectors && nr_eff > 2 * ja.bs && sweep + 1 < cx.jacobi_max_sweeps) {
        be_row_norms2(G2, ws2cur, nc, nr_eff, nc, n2a, W);
        be_rank_rows(n2a, nr_eff, cx.deflation_eps * cx.deflation_eps, ord, cnt, W);
        std::vector<int32_t> ch((size_t)W);
        be_d2h(ch.data(), cnt, sizeof(int32_t) * W);
        int ne = 1;
        for (int w = 0; w < W; ++w) ne = std::max(ne, (int)ch[(size_t)w]);
        JacobiLayout Jn = jacobi_layout(ne, nc);
        if (Jn.bs == ja.bs && Jn.nblk + 2 <= ja.nblk) {
          double *G3 = (double *)cx.pool->get(sizeof(double) * (size_t)W * Jn.nr_pad * nc);
          be_gather_rows(G2, ws2cur, nc, nc, nr_eff, ord, cnt, G3, (long)Jn.nr_pad * nc, Jn.nr_pad, W);
          cx.pool->put(G2);
          G2 = G3; ws2cur = (long)Jn.nr_pad * nc; nr_eff = ne;
          ja.G = G2; ja.ws = ws2cur; ja.nr_pad = Jn.nr_pad; ja.nblk = Jn.nblk;
        }
      }
    }
  }
  double *n2b = (double *)cx.pool->get(sizeof(double) * (size_t)W * nr_eff);
  int32_t *ord2 = (int32_t *)cx.pool->get(sizeof(int32_t) * (size_t)W * tcap);
  be_row_norms2(G2, ws2cur, nc, nr_eff, nc, n2b, W);
  be_select_truncate(n2b, nr_eff, nsv, dmin, dmax, trunc_err, tcap, ord2, kept, W);
  if (presort || cord2) {
    double *Bp = (double *)cx.pool->get(sizeof(double) * (size_t)W * tcap * nc);
    be_gather_rows_normalized(G2, ws2cur, nc, nc, n2b, nr_eff, ord2, kept, tcap, Bp, (long)tcap * nc, W);
    be_permute_cols(Bp, (long)tcap * nc, nc, tcap, nc, cord2 ? cord2 : cord, 0, B, wb, nc, W);
    cx.pool->put(Bp);
    if (presort) { cx.pool->put(cord); cx.pool->put(G); }
  } else {
    be_gather_rows_normalized(G2, ws2cur, nc, nc, n2b, nr_eff, ord2, kept, tcap, B, wb, W);
  }
  for (void *p : {(void *)n2a, (void *)ord, (void *)cnt, (void *)G2, (void *)n2b, (void *)ord2}) cx.pool->put(p);
  if (bsec) { cx.pool->put(bsec); cx.pool->put(cwin); cx.pool->put(cord2); }
}

}  // namespace peps
