// Device-op interface of the B200 VMC sampling library.
//
// Every function here is one batched device operation over W walkers. The product implementation is
// backend_cuda.cu (hand-written sm_100a kernels). tests/hostsim/backend_host.cpp implements the same
// interface with plain loops for CPU-side tests of the host orchestration (engine.cpp); it is never
// linked into the product library.
#pragma once
#include <cstddef>
#include <cstdint>

namespace peps {

// Base address of one batched operand: element base for (walker w, inner batch b) is
//   p + w*ws + b*bs + (gidx ? gidx[w*gws] * gs : 0)
// The gather term is the fused "physical-slice gather" of the reference's
// TensorNetwork2D::UpdateSiteTensor (tensor_network_2d_basic_impl.h:82-108): the site tensor of walker
// w is read straight out of the shared SplitIndexTPS at slice config[w][site].
struct Operand {
  double *p = nullptr;
  long ws = 0;
  long bs = 0;
  const int32_t *gidx = nullptr;
  int gws = 0;
  long gs = 0;
};
inline Operand mkop(double *p, long ws, long bs = 0) {
  Operand o; o.p = p; o.ws = ws; o.bs = bs; return o;
}
inline Operand mkgather(double *p, const int32_t *gidx, int gws, long gs) {
  Operand o; o.p = p; o.gidx = gidx; o.gws = gws; o.gs = gs; return o;
}

// C(m,n) = alpha * sum_k A(m,k) B(k,n) + beta * C(m,n) with separable addressing
//   A(m,k) = A.base + am[m] + ak[k],  B(k,n) = B.base + bk[k] + bn[n],  C(m,n) = C.base + cm[m] + cn[n]
// (tables live in device memory; they encode any pairwise tensor contraction without a transpose pass).
struct GettDesc {
  int M = 0, N = 0, K = 0;
  const int32_t *am = nullptr, *ak = nullptr, *bk = nullptr, *bn = nullptr, *cm = nullptr, *cn = nullptr;
  int a_kfast = 0;   // 1: A's unit-stride index is a contracted one
  int b_nfast = 1;   // 1: B's unit-stride index is a free one
  // 1: consecutive PAIRS (2i, 2i+1) along the operand's fast index are adjacent in memory and every pair starts at an
  // even element offset (so a 16-byte copy / store moves a pair when the operand base is 16-byte aligned). For A the
  // fast index is K when a_kfast else M; for B it is N when b_nfast else K; for C it is N.
  int a_vec2 = 0, b_vec2 = 0, c_vec2 = 0;
  // Optional structural-zero hints (device tables, may be null): A(m,k) == 0 for k < klo_m[m], B(k,n) == 0 for
  // k < klo_n[n] (the R factors of the forward chain are upper trapezoidal). A backend may start the K loop of a tile
  // at the largest K step below both bounds; ignoring the hints gives the same result. work = executed / nominal flops.
  const int32_t *klo_m = nullptr, *klo_n = nullptr;
  double work = 1.0;
  // Optional per-walker zero tails (device arrays, may be null): A(m, .) == 0 for every m >= m_cnt[w] * m_scale, B(., n)
  // == 0 for every n >= n_cnt[w] * n_scale. Output tiles entirely inside a tail are written as zeros without touching
  // the operands. Ignoring the hints gives the same result.
  const int32_t *m_cnt = nullptr, *n_cnt = nullptr;
  int m_scale = 0, n_scale = 0;
};

// ---- backend context / memory / stream -----------------------------------------------------------------
// A backend context owns the device ordinal, the stream, the launch counter and the profiler of one engine. Every
// other be_* call acts on the context BOUND to the calling host thread. The C ABI binds the engine's context at every
// entry point, so a peps_ctx may be created in one thread and used from another (one thread at a time), and several
// contexts (also on different devices) may be interleaved in one thread.
struct BeCtx;
BeCtx *be_ctx_create(int device);         // throws without a CUDA device: the product has no CPU fallback
void be_ctx_bind(BeCtx *c);               // cudaSetDevice(c->device) when needed + makes c current for this thread
void be_ctx_destroy(BeCtx *c);
void be_init(int device);                 // binds a per-thread default context (stand-alone kernel tests)
const char *be_name();                    // "cuda-sm_100a" or "hostsim"
void *be_malloc(size_t bytes);
void be_free(void *p);
void be_memset0(void *p, size_t bytes);
void be_h2d(void *dst, const void *src, size_t bytes);
void be_d2h(void *dst, const void *src, size_t bytes);
void be_d2d(void *dst, const void *src, size_t bytes);
void be_sync();
void *be_stream();                        // cudaStream_t of the context (nullptr on hostsim)
long be_launch_count();                   // number of kernels launched so far (for bench.py gpu_launches)

// ---- per-kernel-class device timing (CUDA events on the launching stream) -----------------------------
enum KernelClass { KC_GETT = 0, KC_DOT, KC_PANEL, KC_JACOBI, KC_SMALL, KC_APPLY, KC_COUNT };
void be_profile_enable(int on);           // when on, every launch is bracketed by an event pair
// Synchronises, folds all pending event pairs into the per-class totals and returns them (arrays of KC_COUNT);
// `reset` clears the totals afterwards. flops = useful FP64 flops the launches of that class executed.
void be_profile_collect(double *ms, long *launches, double *flops, int reset);

// ---- tensor contraction ----------------------------------------------------------------------------
void be_gett(const GettDesc &d, Operand A, Operand B, Operand C, double alpha, double beta, int W, int NB);
// out[w] = sum_k A(ak[k]) * B(bk[k])
void be_dot(int K, const int32_t *ak, const int32_t *bk, Operand A, Operand B, double *out, int W);

// ---- dense helpers ---------------------------------------------------------------------------------
void be_fill(double *p, double v, long n);
// dst[w][r][c] = src[w][r][c] for r < rows, c < cols (row strides lds/ldd, walker strides ws/wd)
void be_copy2d(double *dst, long wd, long ldd, const double *src, long ws, long lds, int rows, int cols, int W);
// dst[w][t][c] = (t == c) for t < rows, c < cols
void be_set_identity(double *dst, long wd, int rows, int cols, int W);

// ---- communication-avoiding R-only QR: one panel step -----------------------------------------------
// For every (walker w, item it): gather the rows rowtab[it*R + s] (s = skip..R-1, skip = (it==0 ? skip0 : 0))
// of panel columns [col0, col0+pw) of the row-major matrix Abase + w*ws (leading dimension lda), Householder-
// factorise the (R-skip) x pw panel, write R (upper triangle on the first pw active rows, zeros below) back in
// place, and emit the explicit reflector block V (unit lower trapezoid, [w][it][R][nbw], skipped slots and columns
// >= pw zero) and the compact-WY factor T ([w][it][nbw][nbw], upper triangular):  Q^T C = C - V T^T (V^T C).
struct PanelArgs {
  double *A; long ws; int lda;
  const int32_t *rowtab; int R; int skip0; int NI;
  int col0, pw, nbw;
  double *Vw, *Tw;
  int W;
  // Optional per-walker row limit (device array, may be null): rows >= row_cnt[w] * row_scale of A[w] are exactly zero
  // on entry (the walker's rank-revealing chain kept fewer rows than the batch maximum the buffers are sized for). An
  // item whose FIRST row (rowtab[it * R]) is at or beyond the limit is skipped: it would produce V = 0, R = 0. The
  // trailing update must be called with the same limit. Only meaningful for items of ascending contiguous rows.
  const int32_t *row_cnt = nullptr;
  int row_scale = 0;
  // Optional early-termination flags (device, may be null): walkers with stopped[w] != 0 are skipped entirely -- their
  // trailing matrix is already numerically zero (be_trailing_check), the R rows not computed would be dropped anyway.
  const int32_t *stopped = nullptr;
};
void be_panel_qr(const PanelArgs &a);
// Early termination of a rank-revealing QR: acc[w] += |A[w][row0:nrows, col0:ncols]|_F^2 (rows / columns of the trailing
// block), then stopped[w] = (acc[w] <= thresh2 * colnorm2[w][colorder[w][0]]) and acc[w] = 0. Walkers already stopped
// are not read again. colnorm2 / colorder: squared column norms of the matrix before the factorisation and their
// descending order (the largest one bounds the largest row norm of R from below).
void be_trailing_check(const double *A, long ws, int lda, int row0, int nrows, int col0, int ncols, const double *colnorm2,
                       const int32_t *colorder, int n, double thresh2, double *acc, int32_t *stopped, int W);

// Trailing update of one CAQR panel step: for every (walker, item) C <- C - V T^T (V^T C) where C are the rows
// rowtab[it*R + s] (s < R) and columns [col1, col1 + ntrail) of A, and V / T are the blocks emitted by
// be_panel_qr. One fused kernel (C tile resident in shared memory) instead of two contractions.
// Opaque tile descriptor of a walker-batched row-major matrix (a CUtensorMap on the CUDA backend): lets a kernel
// fetch a (box_rows x box_cols) tile of walker w with one TMA instruction. be_make_tile_map returns false when the
// backend or the shape (alignment, box limits) cannot use it; callers then leave ApplyArgs::tmap null.
struct TileMap { alignas(64) unsigned char blob[128]; };
bool be_make_tile_map(TileMap *tm, const double *A, long ws, int lda, int rows, int cols, int W, int box_rows, int box_cols);
struct ApplyArgs {
  double *A; long ws; int lda;
  const int32_t *rowtab; int R; int NI;
  int col1, ntrail, nbw;
  const double *Vw, *Tw;
  int W;
  // optional fast path: the rows of item `it` are the contiguous range [row0 + it*R, row0 + (it+1)*R) and tmap
  // describes A with boxes of (R/8 rows x 8 columns)
  const TileMap *tmap = nullptr;
  int row0 = 0;
  // optional second descriptor of the same matrix with boxes of (R rows x 8 columns): selects the column-streaming
  // kernel for contiguous row blocks of R <= 256 rows (V resident in shared memory, one 8-column chunk per warp in flight)
  const TileMap *tmap_cols = nullptr;
  // 0: C <- Q^T C = C - V T^T (V^T C)  (factorisation);  1: C <- Q C = C - V T (V^T C)  (forming / applying Q)
  int notrans = 0;
  // same meaning as PanelArgs::row_cnt / row_scale: items starting at or beyond the walker's limit are skipped
  const int32_t *row_cnt = nullptr;
  int row_scale = 0;
  const int32_t *stopped = nullptr;     // PanelArgs::stopped
};
void be_apply_reflector(const ApplyArgs &a);

// ---- one-sided block Jacobi on the ROWS of G[w] (nr_pad x nc, leading dimension ld) ----------------------
// One round of the round-robin block-pair schedule: block pairs (I,J) of `round` are loaded, their
// (2*bs)x(2*bs) Gram matrix is diagonalised by cyclic two-sided Jacobi (inner_sweeps sweeps) and the
// rotation is applied to the 2*bs rows, larger norms sorted to the lower row index.
// offmax[w] is max'ed with the largest |g_pq|/sqrt(g_pp g_qq) seen (before rotation).
// Walkers with done[w] != 0 are skipped.
struct JacobiArgs {
  double *G; long ws; int ld; int nr_pad; int nc; int bs; int nblk; int round;
  double tol; int inner_sweeps; double *offmax; const int32_t *done; int W;
  int nactive = 0;   // walkers not yet converged (host-side count, for flop accounting only)
  // Z2 sectors (fermion mode): bsec[w][b] = sector (0 / 1, 2 = empty) of row block b; block pairs of different sectors are
  // orthogonal to rounding (disjoint column supports) and are skipped -- which also keeps every block sector-pure; the
  // driver finishes with unrestricted sweeps, so a wrong label costs time, never accuracy
  const int32_t *bsec = nullptr;
  // cwin[w] = {c0, width} of sector 0, {c0, width} of sector 1: the column window a same-sector block pair works on
  // (the columns are sorted by sector; outside its window a row holds rounding noise). Ignored without bsec.
  const int32_t *cwin = nullptr;
};
void be_jacobi_round(const JacobiArgs &a);
// done[w] = (offmax[w] <= tol); offmax[w] = 0 for the next sweep. Returns nothing (host reads done[]).
void be_jacobi_flags(double *offmax, int32_t *done, double tol, int W);
// Fermion mode: the rows of src[w] (count[w] valid rows of nc columns, leading dimension ld) fall into two parity sectors with
// disjoint column supports -- up to rounding noise, so labels compare weights: a row is in sector 0 when it carries more
// weight on the sector-0 columns (the support of row 0, re-estimated once by column majority) than off them; dst[w] (zero-initialised by the caller, nblk * bs rows) receives the rows of
// sector 0 from row 0 on and the rows of sector 1 from the next multiple of bs on, each in their original order;
// bsec[w][b] = 0 / 1 / 2 (empty) per block of bs rows. The COLUMNS are regrouped too (sector-0 columns first, original
// order kept inside a sector): cord_out[w][new column] = cord_in[w][old column] (cord_in null = identity) composes the
// caller's column permutation with it, cwin[w] = the two column windows (JacobiArgs::cwin).
void be_sector_arrange(const double *src, long ws, int ld, int nc, const int32_t *count, int bs, int nblk, double *dst, long wd,
                       int32_t *bsec, const int32_t *cord_in, int32_t *cord_out, int32_t *cwin, int W);
// norms2[w][c] = |G[w][:nr][c]|^2   (column norms)
void be_col_norms2(const double *G, long ws, int ld, int nr, int nc, double *norms2, int W);
// dst[w][r][j] = src[w][r][order[w][j]]  (gather = 1)   or   dst[w][r][order[w][j]] = src[w][r][j]  (gather = 0)
// for r < nr, j < nc; order[w] is a permutation of [0, nc)
void be_permute_cols(const double *src, long ws, int lds, int nr, int nc, const int32_t *order, int gather,
                     double *dst, long wd, int ldd, int W);
// norms2[w][r] = |G[w][r][:]|^2
void be_row_norms2(const double *G, long ws, int ld, int nr, int nc, double *norms2, int W);
// order[w][rank] = row index sorted by norm descending (ties by index), for all nr rows;
// count[w] = number of rows with norms2 > defl2 * max_row(norms2)   (numerical row rank used to shrink the
// Jacobi problem: the dropped rows perturb Theta by <= sqrt(nr * defl2) * |Theta|, a backward-stable amount).
void be_rank_rows(const double *norms2, int nr, double defl2, int32_t *order, int32_t *count, int W);
// dst[w][r][:] = (r < count[w]) ? src[w][order[w][r]][:] : 0     for r < nr_dst
void be_gather_rows(const double *src, long ws, int ld, int nc, int nr_src, const int32_t *order, const int32_t *count,
                    double *dst, long wd, int nr_dst, int W);
// Rank rows by norm (descending, ties by index); kept[w] by the TensorToolkit truncation rule over the
// nsv = min(nr_true, nc) largest values, capped at tcap; order[w][t] = row index of rank t (t < tcap).
void be_select_truncate(const double *norms2, int nr, int nsv, int dmin, int dmax, double trunc_err, int tcap,
                        int32_t *order, int32_t *kept, int W);
// B[w][t][c] = G[w][order[w][t]][c] / norm  for t < kept[w], else 0   (t < tcap, c < nc)
void be_gather_rows_normalized(const double *G, long ws, int ld, int nc, const double *norms2, int nr,
                               const int32_t *order, const int32_t *kept, int tcap, double *B, long wb, int W);

// ---- small-matrix SVD path of the truncation (second preconditioning + single-CTA Jacobi) ---------------------------
// dst[w][c][r] = (r < count[w]) ? src[w][order[w][r]][c] : 0   for c < nc, r < n2 (dst: row-major, leading dimension
// n2, walker stride wd; rows c >= nc of dst are not touched): the numerically non-zero rows of R, sorted by norm,
// written TRANSPOSED so that their LQ factorisation is a tall-skinny QR.
void be_gather_rows_transposed(const double *src, long ws, int ld, int nc, int nr_src, const int32_t *order,
                               const int32_t *count, double *dst, long wd, int n2, int W);
// One-sided Jacobi SVD of the n2 x n2 upper-triangular factor Rt[w] (row-major, leading dimension ld; only the
// leading count[w] columns are non-zero), one CTA per walker with the whole factor resident in shared memory, all
// sweeps and the convergence test on the device. The COLUMNS of Rt are rotated until mutually orthogonal
// (|x.y| <= tol |x||y| for every pair during one whole sweep), giving Rt J = Y Sigma; the TensorToolkit truncation rule
// (dmin, dmax, trunc_err over nsv singular values) picks kept[w]; out[w][i][t] = Y[i][rank t] for i < n2, t < kept[w]
// and 0 for kept[w] <= t < tcap (row-major, leading dimension tcap, walker stride wo): the kept LEFT singular
// vectors of Rt, i.e. the kept right singular vectors of the gathered rows in the basis of the QR's Q.
// sweeps[w] (may be null) receives the number of sweeps walker w needed.
struct SmallSvdArgs {
  const double *Rt; long ws; int ld; int n2; const int32_t *count;
  int nsv, dmin, dmax; double trunc_err; int tcap;
  double tol; int max_sweeps;
  double *out; long wo; int32_t *kept; int32_t *sweeps; int W;
};
constexpr int kSmallSvdMaxN = 128;        // largest n2 the kernel holds in shared memory
void be_svd_small(const SmallSvdArgs &a);
// B[w][t][order ? order[w][j] : j] = C0[w][j][t]   for j < nc, t < tcap  (C0 leading dimension tcap, B leading dim nc)
void be_transpose_permute(const double *C0, long wc, int nc, int tcap, const int32_t *order, double *B, long wb, int W);

// ---- Monte Carlo state kernels ---------------------------------------------------------------------
// std::mt19937(seed[w]) for every walker: mt[w][624], idx[w] = 624
void be_mt_seed(uint32_t *mt, int32_t *idx, const uint32_t *seeds, int W);
// MCUpdateSquareNNExchangeOBC::TwoSiteNNUpdateLocalImpl decision (square_nn_updater.h:146-188) for all walkers:
// skip if cfg equal; accept if |psi_b| >= |psi_a| else iff uniform01 < (|psi_b|/|psi_a|)^2 (draw only then);
// on accept swap cfg[s1], cfg[s2], amplitude = psi_b, accepted[w] += 1.
// jastrow != nullptr: MCUpdateSquareNNExchangeJastrowDressedTJ (square_nn_updater.h:380-438): abs_ratio = |psi_b * jastrow[w]| /
// |psi_a|, accept iff abs_ratio >= 1 or uniform01 < abs_ratio^2 (the draw happens only then); the cached amplitude stays the PEPS part.
void be_nn_exchange_decide(int32_t *cfg, int nsites, int s1, int s2, const double *psi_b, double *amp,
                           uint32_t *mt, int32_t *idx, int32_t *accepted, int W, const double *jastrow = nullptr);
// Jastrow factor exp(sum_{i<j} v_ij n_i n_j) (vmc_basic/jastrow_factor.h:34-121): ratio[w] of exchanging the states of s1 and s2,
// 1 when the two densities are equal, else exp(field(empty site) - field(filled site)) with field(i) = sum_{j != i} v[i][j] n_j
// over the sites in row-major order (JastrowFieldAtSite). dens[phys] = density of a physical state, v = [nsites][nsites].
void be_jastrow_ratio(const int32_t *cfg, int nsites, int s1, int s2, const int32_t *dens, const double *v, double *ratio, int W);
// x[w] *= s[w]
void be_scale(double *x, const double *s, int W);
// EvaluateBondEnergy of SquareSpinOneHalfXXZModelMixIn (square_spin_onehalf_xxz_obc.h:72-104):
// eloc[w] += (c1==c2) ? 0.25 jz : -0.25 jz + (psi_ex[w] * (1/psi[w])) * 0.5 jxy
void be_xxz_bond_energy(const int32_t *cfg, int nsites, int s1, int s2, const double *psi_ex, const double *psi,
                        double jz, double jxy, double *eloc, int W);
// EvaluateOnSiteOffDiagEnergy of TransverseFieldIsingSquareOBC (transverse_field_ising_square_obc.h:191-204):
// eloc[w] += coef * psi_ex[w] * (1 / psi[w])
void be_ratio_accumulate(const double *psi_ex, const double *psi, double coef, double *eloc, int W);
// eloc[w] += -h00 * (cfg[w][0] - 0.5)
void be_xxz_onsite_energy(const int32_t *cfg, int nsites, double h00, double *eloc, int W);
// ---- table-driven model terms (seam B2 as data: square_nnn_energy_solver.h:171-198 EvaluateBondEnergy) -----------------
// A term acts on `nsite` (1 or 2) sites with local state index p = c1 (* phys + c2). Tables (device): diag[p] = <p|H|p>;
// for slot t < T: target[p*T + t] = local state p' with <p'|H|p> != 0 (or -1), coef[p*T + t] = <p'|H|p>.
// be_term_targets: idx_a[w], idx_b[w] = physical indices of target slot t of walker w's local state (its own state when the
// slot is empty), coefw[w] = the matrix element (0 when empty). s2 < 0: one-site term.
void be_term_targets(const int32_t *cfg, int nsites, int s1, int s2, int phys, const int32_t *target, const double *coef, int T,
                     int t, int32_t *idx_a, int32_t *idx_b, double *coefw, int W);
// eloc[w] += (diag ? diag[p_w] : 0) + (coefw ? coefw[w] * (psi_ex[w] * (1 / psi[w])) : 0)
void be_term_accumulate(const int32_t *cfg, int nsites, int s1, int s2, int phys, const double *diag, const double *coefw,
                        const double *psi_ex, const double *psi, double *eloc, int W);

// ---- complex (c128) tensors as split planes ----------------------------------------------------------------------------
// A complex walker-batched tensor is two real planes (re, im). Contractions are four real be_gett launches; the
// factorisations run on the REAL EMBEDDING M = [[Ar, -Ai], [Ai, Ar]] (2m x 2n) of a complex m x n matrix A:
//   * any real R with R^T R = M^T M gives the complex factor r = (R1 - i R2) / sqrt(2) with r^H r = A^H A, where R1 | R2 are
//     the two column halves of R (be_split_r);
//   * the singular values of M are those of A twice over, and its kept right singular subspace is invariant under
//     J (multiplication by i): be_complex_basis turns 2 t real orthonormal vectors b into t complex orthonormal ones by
//     pivoted Gram-Schmidt of z = b[:n] + i b[n:] (the Gram matrix of the z has eigenvalues 2 and 0 only).
// M[w] (2m x 2n, leading dimension 2n, walker stride wm) <- planes Ar / Ai [w] (m x n, leading dimension n, stride wa)
void be_embed_complex(const double *Ar, const double *Ai, long wa, int m, int n, double *M, long wm, int W);
// planes (rows x n, stride wo) <- R[w] (rows x 2n, leading dimension 2n, stride wr): re = R[:, :n] / sqrt2, im = -R[:, n:] / sqrt2
void be_split_r(const double *R, long wr, int rows, int n, double *outr, double *outi, long wo, int W);
// Bm[w]: tcap2 x 2n real (leading dimension 2n, stride wb), kept2[w] orthonormal rows (the rest zero). Writes planes
// Br / Bi [w] (tcap x n, stride wo): keptc[w] = (kept2[w] + 1) / 2 orthonormal complex rows = rows of Vt = V^H (the
// CONJUGATES of the right singular vectors z, Theta = U S V^H), zero rows beyond; keptc is written back. One CTA per walker, modified Gram-Schmidt with pivoting, twice.
void be_complex_basis(double *Bm, long wb, int tcap2, int n, const int32_t *kept2, double *Br, double *Bi, long wo, int tcap,
                      int32_t *keptc, int W);
// out[w] (planes outr / outi) = (d0 - d1) + i (d2 + d3) for the four real dots of a bilinear complex dot product
void be_complex_combine(const double *d0, const double *d1, const double *d2, const double *d3, double *outr, double *outi, int W);
// complex twins of the Monte Carlo kernels: amplitudes / energies as planes [2][W]; |psi| = hypot(re, im)
// jastrow != nullptr: the Jastrow-dressed acceptance of be_nn_exchange_decide with |psi_b * jastrow| = hypot of the scaled planes
void be_nn_exchange_decide_c(int32_t *cfg, int nsites, int s1, int s2, const double *pbr, const double *pbi, double *ampr,
                             double *ampi, uint32_t *mt, int32_t *idx, int32_t *accepted, int W, const double *jastrow = nullptr);
// eloc += (c1 == c2) ? 0.25 jz : -0.25 jz + conj(psi_ex / psi) * 0.5 jxy     (square_spin_onehalf_xxz_obc.h:72-104)
void be_xxz_bond_energy_c(const int32_t *cfg, int nsites, int s1, int s2, const double *exr, const double *exi, const double *pr,
                          const double *pi, double jz, double jxy, double *er, double *ei, int W);
// complex twins of be_ratio_accumulate / be_term_accumulate: the reference conjugates every amplitude ratio that enters E_loc
// (transverse_field_ising_square_obc.h:191-204, square_nnn_energy_solver.h:171-198): e += coef * conj(psi_ex / psi)
void be_ratio_accumulate_c(const double *exr, const double *exi, const double *pr, const double *pi, double coef, double *er,
                           double *ei, int W);
// e += (diag ? diag[p_w] : 0) + (coefw ? coefw[w] * conj(psi_ex[w] / psi[w]) : 0)   (tables are real)
void be_term_accumulate_c(const int32_t *cfg, int nsites, int s1, int s2, int phys, const double *diag, const double *coefw,
                          const double *exr, const double *exi, const double *pr, const double *pi, double *er, double *ei, int W);
// O* = conj(hole / psi) (mc_energy_grad_evaluator.h:245-272): osum += O*, eosum += conj(E_loc) O*; all arrays as planes
void be_accumulate_ostar_c(const double *hr, const double *hi, long hole_stride, const int32_t *hole_off, const int32_t *site_size,
                           const int32_t *tps_off, const int32_t *cfg, int nsites, const double *ampr, const double *ampi,
                           const double *er, const double *ei, double *osr, double *osi, double *eor, double *eoi, int W);

// ---- fermionic (fZ2-graded) tensors as sign-dressed dense tensors ---------------------------------------------------
// A graded network of parity-conserving site tensors equals a bosonic network of dressed tensors (engine.h, "fermion
// mode"). Per site the device TPS holds FERMION_VARIANTS * phys slices: variant v, state s at slice v * phys + s.
//   v = 0..5: horizontal machinery, leg-sign masks {0, U, R, R|U, R|D, R|D|U};  v = 6, 7: vertical machinery, {0, L}.
constexpr int FERMION_VARIANTS = 8;
// Jordan-Wigner bits and gather indices of the current configurations (one thread per walker):
//   jw_h[w][site] = parity of the sites left of `site` in its row, jw_v = above it in its column;
//   gidx_h = jw_h * phys + cfg,  gidx_v = (6 + jw_v) * phys + cfg.
void be_fermion_gather(const int32_t *cfg, int rows, int cols, int phys, const int32_t *phys_par, int32_t *gidx_h,
                       int32_t *gidx_v, int32_t *jw_h, int32_t *jw_v, int W);
// Replacement slices and signed matrix element of target slot t of a two-site term on (s1, s2) (square_spinless_fermion.h:
// 118-211, square_tJ_model.h:300-345: psi_ex / psi along one contraction path). kind 0: horizontal NN bond, 1: vertical
// NN bond, 2: diagonal s1 = left-up, s2 = right-down, 3: diagonal s1 = left-down, s2 = right-up (kinds 0, 2, 3 in the
// horizontal machinery, 1 in the vertical). target == nullptr: the exchange of the two states with element 1 (updater).
// A target that moves a fermion (both site parities flip) gets the leg-sign masks and the Jordan-Wigner sign of the hop;
// parity-preserving targets keep the canonical masks; empty slots give the walker's own slices and coefw = 0.
#if defined(__CUDACC__)
#define PEPS_HD __host__ __device__
#else
#define PEPS_HD
#endif
// one walker of be_fermion_targets (shared by the CUDA kernel and the test-only host simulation)
PEPS_HD inline void fermion_target_one(const int32_t *c, const int32_t *jh, const int32_t *jv, int s1, int s2, int phys,
                                       const int32_t *par, int kind, const int32_t *target, const double *coef, int T, int t,
                                       int32_t &idx_a, int32_t &idx_b, double &coefw) {
  const int c1 = c[s1], c2 = c[s2], p = c1 * phys + c2;
  int tg;
  double cf;
  if (target) { tg = target[p * T + t]; cf = tg < 0 ? 0.0 : coef[p * T + t]; }
  else { tg = c1 != c2 ? c2 * phys + c1 : -1; cf = tg < 0 ? 0.0 : 1.0; }
  const int n1 = tg < 0 ? c1 : tg / phys, n2 = tg < 0 ? c2 : tg % phys;
  const int moved = (par[c1] ^ par[n1]) & (par[c2] ^ par[n2]);
  int va, vb, neg = 0;
  if (kind == 1) { va = 6 + jv[s1]; vb = 6 + (jv[s2] ^ moved); }
  else if (kind == 0 || !moved) { va = jh[s1]; vb = jh[s2] ^ moved; }
  else if (kind == 2) { va = 2 + jh[s1]; vb = jh[s2] ^ 1; neg = jh[s2]; }
  else { va = jh[s1]; vb = 4 + jh[s2]; neg = jh[s1]; }
  idx_a = va * phys + n1;
  idx_b = vb * phys + n2;
  coefw = neg ? -cf : cf;
}
void be_fermion_targets(const int32_t *cfg, int nsites, int s1, int s2, int phys, const int32_t *phys_par,
                        const int32_t *jw_h, const int32_t *jw_v, int kind, const int32_t *target, const double *coef,
                        int T, int t, int32_t *idx_a, int32_t *idx_b, double *coefw, int W);
// CalGTenForFermionicTensors + ActFermionPOps (utility/helpers.h:57-67, mc_energy_grad_evaluator.h:259-266) on the holes
// of the horizontal machinery: psi_site = <hole, dressed site tensor>; hole <- hole * sign[jw_h] * amp[w] / psi_site, so
// that hole / amp is O* = conj(d psi / d T) / conj(psi_site) in the user's (undressed) tensor entries.
// sign: [2][hole_stride] (+1 / -1 per element for jw_h = 0 / 1); gtps_off[site]: offset of the site's dressed slices.
void be_fermion_finish_holes(double *holes, long hole_stride, const int32_t *hole_off, const int32_t *site_size,
                             const double *gtps, const int64_t *gtps_off, const int32_t *gidx_h, const int32_t *jw_h,
                             int nsites, const double *sign, const double *amp, int W);

// complex twin: holes / dressed tensors / amplitudes as planes (the im plane of gtps starts gtps_im_off doubles after the
// re plane); psi_site = bilinear <hole, tensor>, hole <- hole * sign * amp / psi_site in complex arithmetic, so that
// conj(hole / amp) = conj(d psi / d T) / conj(psi_site) (be_accumulate_ostar_c).
void be_fermion_finish_holes_c(double *hr, double *hi, long hole_stride, const int32_t *hole_off, const int32_t *site_size,
                               const double *gtps, long gtps_im_off, const int64_t *gtps_off, const int32_t *gidx_h,
                               const int32_t *jw_h, int nsites, const double *sign, const double *ampr, const double *ampi, int W);

// O* accumulation (mc_energy_grad_evaluator.h:245-272) for one sample of all walkers:
//   o = (1/amp[w]) * hole[w][e];  osum[slot(site,cfg[w][site]) + e] += o;  eosum[...] += eloc[w] * o
// holes: [W][hole_stride]; per site: offset hole_off[site], size site_size[site]; TPS slot of (site, s) at
// tps_off[site] + s*site_size[site].
void be_accumulate_ostar(const double *holes, long hole_stride, const int32_t *hole_off, const int32_t *site_size,
                         const int32_t *tps_off, const int32_t *cfg, int nsites, int phys, const double *amp,
                         const double *eloc, double *osum, double *eosum, int W);

// ---- stochastic reconfiguration: device-resident O* sample store and the S-matrix-free matvec ---------------
// (optimizer/stochastic_reconfiguration_smatrix.h:45-91). A stored sample i keeps O*_i as the [hole_stride] vector
// of its sampled physical slices plus the configuration that says which TPS slots they occupy.
// store: ostar[i][e] = holes[w][e] / amp[w], cfgs[i][:] = cfg[w][:] for i = first + w.
void be_sr_store(const double *holes, long hole_stride, const double *amp, const int32_t *cfg, int nsites,
                 double *ostar, int32_t *cfgs, long first, int W);
// Complex states through the real embedding: with O*_i = conj(hole / amp) = o_r + i o_i, the real-linear map v -> sum_i
// <O*_i, v> O*_i on planar vectors [v_r ; v_i] is sum_i (x_i x_i^T + y_i y_i^T) with x_i = [o_r ; o_i] and y_i = J x_i =
// [-o_i ; o_r]: the REAL kernels below run on 2 N samples of a lattice with 2 nsites "sites" (re plane, im plane).
// ostar: [2 cap][2 hole_stride], row first + w = x, row cap + first + w = y; cfgs: [2 cap][2 nsites] = the configuration twice.
void be_sr_store_c(const double *hr, const double *hi, long hole_stride, const double *ampr, const double *ampi, const int32_t *cfg,
                   int nsites, double *ostar, int32_t *cfgs, long first, long cap, int W);
// delta[i] = (O*_i . v) - mean_dot_v  for i < n   (O*_i . v sums over the sampled slot of every site)
void be_sr_dots(const double *ostar, const int32_t *cfgs, long hole_stride, const int32_t *hole_off,
                const int32_t *site_size, const int32_t *tps_off, int nsites, const double *v, double mean_dot_v,
                double *delta, long n);
// out[slot] = sum_i delta[i] O*_i[slot]   over the full TPS-shaped vector (slots a sample does not occupy get 0)
void be_sr_accumulate(const double *ostar, const int32_t *cfgs, long hole_stride, const int32_t *hole_off,
                      const int32_t *site_size, const int32_t *tps_off, int nsites, int phys, const double *delta,
                      double *out, long n);

// ---- MinSR: the natural gradient solved in sample space (N x N) instead of parameter space -------------------------
// Masked Gram of two row sets of the store that share the configurations `cfgs` (n rows each, hole layout):
//   G[i][j] = sum_site [cfgs_i(site) == cfgs_j(site)] <left_i[site block], right_j[site block]>     (i, j < n)
// G is row-major n x n. Only the tiles of the upper triangle are computed (DMMA, the K loop walks the sites and folds a
// per-site accumulator under the mask at each site boundary, split-K over site ranges reduced in a fixed order: two
// calls give bit-identical G); the lower triangle is G[j][i] = lower_sign * G[i][j]. lower_sign = -1 declares G
// antisymmetric (the cross Gram <y_i, x_j> of a complex store) and sets its diagonal to 0. site_size_host: the site sizes
// on the host (the split-K ranges are chosen from them).
void be_sr_gram(const double *left, const double *right, const int32_t *cfgs, long hole_stride, const int32_t *hole_off,
                const int32_t *site_size, const int32_t *site_size_host, int nsites, long n, double lower_sign, double *G);
// T[i][j] = scale * (G[i][j] - a[i] - sign * a[j] + c)   (sign = -1: antisymmetric result, diagonal set to 0)
void be_minsr_centre(const double *G, const double *a, double c, double sign, long n, double scale, double *T);
// M = Tr + shift I (n x n, Ti null) or the real embedding [[Tr, -Ti], [Ti, Tr]] + shift I (2n x 2n), row-major
void be_minsr_embed(const double *Tr, const double *Ti, long n, double shift, double *M);
// Cholesky factor M = L L^T (m x m, row-major) in place: blocked right-looking, 32-column panels, trailing update on
// DMMA; only the lower triangle is read and written. info[0] = 0, or the 1-based index of the first non-positive pivot.
void be_chol(double *M, long m, int32_t *info);
// b <- (L L^T)^{-1} b with the factor of be_chol (forward then backward substitution)
void be_chol_solve(const double *L, long m, double *b);


// ---- device-resident vector algebra of the SR conjugate-gradient solver (TPS-shaped vectors of n doubles) ----------
// out[i] = ca * a[i] + cb * b[i]   (b may be null: out = ca * a; out may alias a or b)
void be_vec_lincomb(double *out, double ca, const double *a, double cb, const double *b, long n);
// result[0] = sum_i a[i] * b[i]    (device scalar; fixed-shape two-stage reduction: deterministic)
void be_vec_dot(const double *a, const double *b, long n, double *result);

}  // namespace peps
