// TEST-ONLY host simulation of peps_b200/csrc/backend.h.
//
// This file is never linked into the product library (libpeps_b200.so has no CPU path and throws when no
// CUDA device is present). It exists so that `-m "not gpu"` tests can exercise the HOST orchestration
// (engine.cpp: stack discipline, contraction sequences, sweep/energy control flow, the C ABI) in the build
// container, which has no GPU. Every op is the plain-loop statement of the semantics documented in
// backend.h; the GPU parity tests compare the CUDA kernels against the oracle, not against this file.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <stdexcept>
#include <vector>
#include "../../peps_b200/csrc/backend.h"

namespace peps {

static long g_launches = 0;
struct BeCtx { int device; };
BeCtx *be_ctx_create(int device) { return new BeCtx{device}; }
void be_ctx_bind(BeCtx *) {}
void be_ctx_destroy(BeCtx *c) { delete c; }
void be_init(int) {}
const char *be_name() { return "hostsim"; }
void *be_malloc(size_t bytes) { return std::malloc(bytes ? bytes : 8); }
void be_free(void *p) { std::free(p); }
void be_memset0(void *p, size_t bytes) { std::memset(p, 0, bytes); }
void be_h2d(void *d, const void *s, size_t b) { std::memcpy(d, s, b); }
void be_d2h(void *d, const void *s, size_t b) { std::memcpy(d, s, b); }
void be_d2d(void *d, const void *s, size_t b) { std::memcpy(d, s, b); }
void be_sync() {}
void *be_stream() { return nullptr; }
long be_launch_count() { return g_launches; }
void be_profile_enable(int) {}
void be_profile_collect(double *ms, long *launches, double *flops, int) {
  for (int c = 0; c < KC_COUNT; ++c) { if (ms) ms[c] = 0; if (launches) launches[c] = 0; if (flops) flops[c] = 0; }
}

static const double *obase(const Operand &o, int w, int b) {
  const double *p = o.p + (long)w * o.ws + (long)b * o.bs;
  if (o.gidx) p += (long)o.gidx[(long)w * o.gws] * o.gs;
  return p;
}

void be_gett(const GettDesc &d, Operand A, Operand B, Operand C, double alpha, double beta, int W, int NB) {
  ++g_launches;
  for (int w = 0; w < W; ++w)
    for (int b = 0; b < NB; ++b) {
      const double *Ab = obase(A, w, b), *Bb = obase(B, w, b);
      double *Cb = const_cast<double *>(obase(C, w, b));
      std::vector<double> out((size_t)d.M * d.N);
      // per-walker zero tails are honoured per element AND verified: a wrong limit fails the host-logic tests
      const int mlim = d.m_cnt ? d.m_cnt[w] * d.m_scale : d.M, nlim = d.n_cnt ? d.n_cnt[w] * d.n_scale : d.N;
      for (int m = 0; m < d.M; ++m)
        for (int k = 0; k < d.K; ++k)
          if (m >= mlim && Ab[d.am[m] + d.ak[k]] != 0.0) throw std::logic_error("hostsim gett: m_cnt tail of A is not zero");
      for (int n = 0; n < d.N; ++n)
        for (int k = 0; k < d.K; ++k)
          if (n >= nlim && Bb[d.bk[k] + d.bn[n]] != 0.0) throw std::logic_error("hostsim gett: n_cnt tail of B is not zero");
      for (int m = 0; m < d.M; ++m)
        for (int n = 0; n < d.N; ++n) {
          double s = 0.0;
          if (m >= mlim || n >= nlim) { out[(size_t)m * d.N + n] = 0.0; continue; }
          // structural-zero hints are honoured PER ELEMENT here (the strictest reading): a wrong hint table shows up
          // as a parity failure of the host-logic tests
          int k0 = 0;
          if (d.klo_m) k0 = std::max(k0, (int)d.klo_m[m]);
          if (d.klo_n) k0 = std::max(k0, (int)d.klo_n[n]);
          for (int k = k0; k < d.K; ++k) s += Ab[d.am[m] + d.ak[k]] * Bb[d.bk[k] + d.bn[n]];
          out[(size_t)m * d.N + n] = s;
        }
      for (int m = 0; m < d.M; ++m)
        for (int n = 0; n < d.N; ++n) {
          double *cp = Cb + d.cm[m] + d.cn[n];
          double v = alpha * out[(size_t)m * d.N + n];
          if (beta != 0.0) v += beta * (*cp);
          *cp = v;
        }
    }
}

void be_dot(int K, const int32_t *ak, const int32_t *bk, Operand A, Operand B, double *out, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w) {
    const double *Ab = obase(A, w, 0), *Bb = obase(B, w, 0);
    double s = 0.0;
    for (int k = 0; k < K; ++k) s += Ab[ak[k]] * Bb[bk[k]];
    out[w] = s;
  }
}

void be_fill(double *p, double v, long n) { ++g_launches; for (long i = 0; i < n; ++i) p[i] = v; }
void be_copy2d(double *dst, long wd, long ldd, const double *src, long ws, long lds, int rows, int cols, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w)
    for (int r = 0; r < rows; ++r)
      for (int c = 0; c < cols; ++c) dst[w * wd + r * ldd + c] = src[w * ws + r * lds + c];
}
void be_set_identity(double *dst, long wd, int rows, int cols, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w)
    for (int r = 0; r < rows; ++r)
      for (int c = 0; c < cols; ++c) dst[w * wd + (long)r * cols + c] = (r == c) ? 1.0 : 0.0;
}

void be_trailing_check(const double *A, long ws, int lda, int row0, int nrows, int col0, int ncols, const double *colnorm2,
                       const int32_t *colorder, int n, double thresh2, double *acc, int32_t *stopped, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w) {
    if (stopped[w]) continue;
    double s2 = 0.0;
    for (int r = row0; r < nrows; ++r)
      for (int c = col0; c < ncols; ++c) { const double v = A[w * ws + (long)r * lda + c]; s2 += v * v; }
    stopped[w] = (s2 <= thresh2 * colnorm2[(long)w * n + colorder[(long)w * n]]) ? 1 : 0;
    acc[w] = 0.0;
  }
}
void be_panel_qr(const PanelArgs &a) {
  ++g_launches;
  const int R = a.R, pw = a.pw, nbw = a.nbw;
  for (int w = 0; w < a.W; ++w)
    for (int it = 0; it < a.NI; ++it) {
      if (a.stopped && a.stopped[w]) continue;
      const int skip = (it == 0) ? a.skip0 : 0, nact = R - skip;
      double *Aw = a.A + (long)w * a.ws;
      const int32_t *rows = a.rowtab + (long)it * R;
      if (a.row_cnt && rows[0] >= a.row_cnt[w] * a.row_scale) {       // skipped item: verify that it really is all zero
        for (int r = 0; r < R; ++r)
          for (int c = 0; c < a.lda; ++c)
            if (Aw[(long)rows[r] * a.lda + c] != 0.0) throw std::logic_error("hostsim panel: skipped row block is not zero");
        continue;
      }
      std::vector<double> P((size_t)nact * pw), tau((size_t)pw, 0.0), V((size_t)nact * pw, 0.0), T((size_t)pw * pw, 0.0);
      auto at = [&](int r, int c) -> double & { return P[(size_t)r * pw + c]; };
      for (int r = 0; r < nact; ++r)
        for (int c = 0; c < pw; ++c) at(r, c) = Aw[(long)rows[skip + r] * a.lda + a.col0 + c];
      for (int j = 0; j < pw; ++j) {
        if (j >= nact) continue;
        double xn2 = 0.0;
        for (int r = j + 1; r < nact; ++r) xn2 += at(r, j) * at(r, j);
        double alpha = at(j, j), beta = alpha, tj = 0.0, sj = 0.0;
        if (xn2 > 0.0) {
          double nrm = std::sqrt(alpha * alpha + xn2);
          beta = (alpha >= 0.0) ? -nrm : nrm;
          tj = (beta - alpha) / beta;
          sj = 1.0 / (alpha - beta);
        }
        tau[(size_t)j] = tj;
        V[(size_t)j * pw + j] = 1.0;
        for (int r = j + 1; r < nact; ++r) V[(size_t)r * pw + j] = at(r, j) * sj;
        if (tj != 0.0)
          for (int c = j + 1; c < pw; ++c) {
            double wv = at(j, c);
            for (int r = j + 1; r < nact; ++r) wv += V[(size_t)r * pw + j] * at(r, c);
            double f = tj * wv;
            at(j, c) -= f;
            for (int r = j + 1; r < nact; ++r) at(r, c) -= f * V[(size_t)r * pw + j];
          }
        at(j, j) = beta;
        for (int r = j + 1; r < nact; ++r) at(r, j) = 0.0;
      }
      for (int j = 0; j < pw; ++j) {
        T[(size_t)j * pw + j] = tau[(size_t)j];
        std::vector<double> s((size_t)j, 0.0);
        for (int b2 = 0; b2 < j; ++b2)
          for (int r = 0; r < nact; ++r) s[(size_t)b2] += V[(size_t)r * pw + b2] * V[(size_t)r * pw + j];
        for (int a2 = 0; a2 < j; ++a2) {
          double v = 0.0;
          for (int b2 = a2; b2 < j; ++b2) v += T[(size_t)a2 * pw + b2] * s[(size_t)b2];
          T[(size_t)a2 * pw + j] = -tau[(size_t)j] * v;
        }
      }
      for (int r = 0; r < nact; ++r)
        for (int c = 0; c < pw; ++c) Aw[(long)rows[skip + r] * a.lda + a.col0 + c] = (r <= c) ? at(r, c) : 0.0;
      double *Vo = a.Vw + ((long)w * a.NI + it) * (long)R * nbw;
      double *To = a.Tw + ((long)w * a.NI + it) * (long)nbw * nbw;
      for (long e = 0; e < (long)R * nbw; ++e) Vo[e] = 0.0;
      for (long e = 0; e < (long)nbw * nbw; ++e) To[e] = 0.0;
      for (int r = 0; r < nact; ++r)
        for (int c = 0; c < pw; ++c) Vo[(long)(skip + r) * nbw + c] = V[(size_t)r * pw + c];
      for (int a2 = 0; a2 < pw; ++a2)
        for (int b2 = a2; b2 < pw; ++b2) To[(long)a2 * nbw + b2] = T[(size_t)a2 * pw + b2];
    }
}

bool be_make_tile_map(TileMap *, const double *, long, int, int, int, int, int, int) { return false; }
void be_apply_reflector(const ApplyArgs &a) {
  ++g_launches;
  for (int w = 0; w < a.W; ++w)
    for (int it = 0; it < a.NI; ++it) {
      double *Aw = a.A + (long)w * a.ws;
      const int32_t *rows = a.rowtab + (long)it * a.R;
      if (a.row_cnt && rows[0] >= a.row_cnt[w] * a.row_scale) continue;
      if (a.stopped && a.stopped[w]) continue;
      const double *V = a.Vw + ((long)w * a.NI + it) * (long)a.R * a.nbw;
      const double *T = a.Tw + ((long)w * a.NI + it) * (long)a.nbw * a.nbw;
      std::vector<double> Wm((size_t)a.nbw * a.ntrail, 0.0), W2((size_t)a.nbw * a.ntrail, 0.0);
      for (int r = 0; r < a.R; ++r)
        for (int c = 0; c < a.nbw; ++c) {
          double v = V[(long)r * a.nbw + c];
          if (v == 0.0) continue;
          for (int tcol = 0; tcol < a.ntrail; ++tcol) Wm[(size_t)c * a.ntrail + tcol] += v * Aw[(long)rows[r] * a.lda + a.col1 + tcol];
        }
      for (int c = 0; c < a.nbw; ++c)          // W2 = T^T W   (notrans: T W)
        for (int b2 = (a.notrans ? c : 0); b2 < (a.notrans ? a.nbw : c + 1); ++b2) {
          double tv = a.notrans ? T[(long)c * a.nbw + b2] : T[(long)b2 * a.nbw + c];
          if (tv == 0.0) continue;
          for (int tcol = 0; tcol < a.ntrail; ++tcol) W2[(size_t)c * a.ntrail + tcol] += tv * Wm[(size_t)b2 * a.ntrail + tcol];
        }
      for (int r = 0; r < a.R; ++r)
        for (int tcol = 0; tcol < a.ntrail; ++tcol) {
          double s = 0.0;
          for (int c = 0; c < a.nbw; ++c) s += V[(long)r * a.nbw + c] * W2[(size_t)c * a.ntrail + tcol];
          Aw[(long)rows[r] * a.lda + a.col1 + tcol] -= s;
        }
    }
}

static void rr_pair(int nblk, int round, int q, int &I, int &J) {
  const int n1 = nblk - 1;
  if (q == 0) { I = n1; J = round % n1; }
  else { I = (round + q) % n1; J = (round - q + n1) % n1; }
}

void be_sector_arrange(const double *src, long ws, int ld, int nc, const int32_t *count, int bs, int nblk, double *dst, long wd,
                       int32_t *bsec, const int32_t *cord_in, int32_t *cord_out, int32_t *cwin, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w) {
    const int n = std::min((int)count[w], nblk * bs);
    const double *S = src + (long)w * ws;
    std::vector<int> colA((size_t)nc, 0), lab((size_t)std::max(n, 1), 1);
    double mx = 0.0;
    for (int c = 0; c < nc && n > 0; ++c) mx = std::max(mx, std::fabs(S[c]));
    for (int c = 0; c < nc; ++c) colA[(size_t)c] = (n > 0 && std::fabs(S[c]) > 1e-8 * mx);
    for (int pass = 0; pass < 2; ++pass) {
      for (int r = 0; r < n; ++r) {
        double in = 0.0, out = 0.0;
        for (int c = 0; c < nc; ++c) { const double v = std::fabs(S[(long)r * ld + c]); if (colA[(size_t)c]) in += v; else out += v; }
        lab[(size_t)r] = in >= out ? 0 : 1;
      }
      if (pass == 0)
        for (int c = 0; c < nc; ++c) {
          double wa = 0.0, wb = 0.0;
          for (int r = 0; r < n; ++r) { const double v = std::fabs(S[(long)r * ld + c]); if (lab[(size_t)r] == 0) wa += v; else wb += v; }
          colA[(size_t)c] = wa >= wb;
        }
    }
    int nA = 0, nB = 0;
    for (int r = 0; r < n; ++r) nA += (lab[(size_t)r] == 0);
    const int baseB = (nA + bs - 1) / bs * bs;
    int ia = 0;
    double *D = dst + (long)w * wd;
    int cA = 0;
    for (int c = 0; c < nc; ++c) cA += colA[(size_t)c];
    std::vector<int> cpos((size_t)nc);
    int ja = 0, jb = cA;
    for (int c = 0; c < nc; ++c) cpos[(size_t)c] = colA[(size_t)c] ? ja++ : jb++;
    for (int c = 0; c < nc; ++c) cord_out[(long)w * nc + cpos[(size_t)c]] = cord_in ? cord_in[(long)w * nc + c] : c;
    cwin[(long)w * 4 + 0] = 0; cwin[(long)w * 4 + 1] = std::min(nc, (cA + 1) & ~1);
    cwin[(long)w * 4 + 2] = cA & ~1; cwin[(long)w * 4 + 3] = nc - (cA & ~1);
    for (int r = 0; r < n; ++r) {
      const int p = lab[(size_t)r] == 0 ? ia++ : baseB + nB++;
      if (p < nblk * bs) for (int c = 0; c < nc; ++c) D[(long)p * ld + cpos[(size_t)c]] = S[(long)r * ld + c];
    }
    const int blkA = (nA + bs - 1) / bs, blkB = (nB + bs - 1) / bs;
    for (int b = 0; b < nblk; ++b) bsec[(long)w * nblk + b] = b < blkA ? 0 : (b < blkA + blkB ? 1 : 2);
    if (std::getenv("PEPS_DEBUG_SECTORS")) std::fprintf(stderr, "[sectors] w=%d n=%d nc=%d nA=%d nB=%d\n", w, n, nc, nA, nB);
  }
}
void be_jacobi_round(const JacobiArgs &a) {
  ++g_launches;
  const int bs = a.bs, n2 = 2 * bs, nc = a.nc;
  for (int w = 0; w < a.W; ++w) {
    if (a.done[w]) continue;
    double *Gw = a.G + (long)w * a.ws;
    for (int q = 0; q < a.nblk / 2; ++q) {
      int I, J;
      rr_pair(a.nblk, a.round, q, I, J);
      if (a.bsec) {
        const int sI = a.bsec[(long)w * a.nblk + I], sJ = a.bsec[(long)w * a.nblk + J];
        if (sI != sJ || sI == 2) continue;
      }
      int lo = std::min(I, J), hi = std::max(I, J);
      int c0 = 0, nc = a.nc;
      if (a.bsec && a.cwin) { const int sI = a.bsec[(long)w * a.nblk + I]; c0 = a.cwin[(long)w * 4 + 2 * sI]; nc = a.cwin[(long)w * 4 + 2 * sI + 1]; if (nc <= 0) continue; }
      double *Gw = a.G + (long)w * a.ws + c0;
      auto grow = [&](int r) { return (r < bs) ? lo * bs + r : hi * bs + (r - bs); };
      std::vector<double> Ps((size_t)n2 * nc), G((size_t)n2 * n2), Wm((size_t)n2 * n2, 0.0);
      for (int r = 0; r < n2; ++r)
        for (int c = 0; c < nc; ++c) Ps[(size_t)r * nc + c] = Gw[(long)grow(r) * a.ld + c];
      for (int p = 0; p < n2; ++p)
        for (int qq = 0; qq < n2; ++qq) {
          double s = 0.0;
          for (int c = 0; c < nc; ++c) s += Ps[(size_t)p * nc + c] * Ps[(size_t)qq * nc + c];
          G[(size_t)p * n2 + qq] = s;
        }
      for (int r = 0; r < n2; ++r) Wm[(size_t)r * n2 + r] = 1.0;
      double mx = 0.0;
      for (int p = 0; p < n2; ++p)
        for (int qq = p + 1; qq < n2; ++qq) {
          double gpp = G[(size_t)p * n2 + p], gqq = G[(size_t)qq * n2 + qq], gpq = std::fabs(G[(size_t)p * n2 + qq]);
          if (gpp > 0.0 && gqq > 0.0 && gpq > 0.0) mx = std::max(mx, gpq / std::sqrt(gpp * gqq));
        }
      a.offmax[w] = std::max(a.offmax[w], mx);
      for (int sw = 0; sw < a.inner_sweeps; ++sw)
        for (int rd = 0; rd < n2 - 1; ++rd) {
          std::vector<double> cs((size_t)n2);
          std::vector<int> pr((size_t)n2);
          for (int t = 0; t < n2 / 2; ++t) {
            int p, qq;
            rr_pair(n2, rd, t, p, qq);
            if (p > qq) std::swap(p, qq);
            double app = G[(size_t)p * n2 + p], aqq = G[(size_t)qq * n2 + qq], apq = G[(size_t)p * n2 + qq];
            double c = 1.0, s = 0.0;
            if (apq * apq > a.tol * a.tol * std::fabs(app * aqq) && apq != 0.0) {
              double d = aqq - app, r = std::sqrt(d * d + 4.0 * apq * apq);
              double tt = (d >= 0.0) ? (2.0 * apq) / (d + r) : (-2.0 * apq) / (r - d);
              c = 1.0 / std::sqrt(1.0 + tt * tt);
              s = c * tt;
            }
            cs[(size_t)t] = c; cs[(size_t)(n2 / 2 + t)] = s;
            pr[(size_t)(2 * t)] = p; pr[(size_t)(2 * t + 1)] = qq;
          }
          for (int k = 0; k < n2 / 2; ++k) {
            int p = pr[(size_t)(2 * k)], qq = pr[(size_t)(2 * k + 1)];
            double c = cs[(size_t)k], s = cs[(size_t)(n2 / 2 + k)];
            for (int i = 0; i < n2; ++i) {
              double gp = G[(size_t)i * n2 + p], gq = G[(size_t)i * n2 + qq];
              G[(size_t)i * n2 + p] = c * gp - s * gq;
              G[(size_t)i * n2 + qq] = s * gp + c * gq;
              double wp = Wm[(size_t)i * n2 + p], wq = Wm[(size_t)i * n2 + qq];
              Wm[(size_t)i * n2 + p] = c * wp - s * wq;
              Wm[(size_t)i * n2 + qq] = s * wp + c * wq;
            }
          }
          for (int k = 0; k < n2 / 2; ++k) {
            int p = pr[(size_t)(2 * k)], qq = pr[(size_t)(2 * k + 1)];
            double c = cs[(size_t)k], s = cs[(size_t)(n2 / 2 + k)];
            for (int i = 0; i < n2; ++i) {
              double gp = G[(size_t)p * n2 + i], gq = G[(size_t)qq * n2 + i];
              G[(size_t)p * n2 + i] = c * gp - s * gq;
              G[(size_t)qq * n2 + i] = s * gp + c * gq;
            }
          }
        }
      std::vector<int> perm((size_t)n2);
      for (int t = 0; t < n2; ++t) {
        double mine = G[(size_t)t * n2 + t];
        int rank = 0;
        for (int j = 0; j < n2; ++j) {
          double o = G[(size_t)j * n2 + j];
          rank += (o > mine) || (o == mine && j < t);
        }
        perm[(size_t)rank] = t;
      }
      for (int r = 0; r < n2; ++r)
        for (int c = 0; c < nc; ++c) {
          double s = 0.0;
          for (int k = 0; k < n2; ++k) s += Wm[(size_t)k * n2 + perm[(size_t)r]] * Ps[(size_t)k * nc + c];
          Gw[(long)grow(r) * a.ld + c] = s;
        }
    }
  }
}
void be_jacobi_flags(double *offmax, int32_t *done, double tol, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w) { done[w] = offmax[w] <= tol; offmax[w] = 0.0; }
}
void be_col_norms2(const double *G, long ws, int ld, int nr, int nc, double *norms2, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w)
    for (int c = 0; c < nc; ++c) {
      double s = 0.0;
      for (int r = 0; r < nr; ++r) s += G[w * ws + (long)r * ld + c] * G[w * ws + (long)r * ld + c];
      norms2[(long)w * nc + c] = s;
    }
}
void be_permute_cols(const double *src, long ws, int lds, int nr, int nc, const int32_t *order, int gather,
                     double *dst, long wd, int ldd, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w)
    for (int r = 0; r < nr; ++r)
      for (int j = 0; j < nc; ++j) {
        const int o = order[(long)w * nc + j];
        if (gather) dst[w * wd + (long)r * ldd + j] = src[w * ws + (long)r * lds + o];
        else dst[w * wd + (long)r * ldd + o] = src[w * ws + (long)r * lds + j];
      }
}
void be_row_norms2(const double *G, long ws, int ld, int nr, int nc, double *norms2, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w)
    for (int r = 0; r < nr; ++r) {
      double s = 0.0;
      for (int c = 0; c < nc; ++c) s += G[w * ws + (long)r * ld + c] * G[w * ws + (long)r * ld + c];
      norms2[(long)w * nr + r] = s;
    }
}
void be_rank_rows(const double *norms2, int nr, double defl2, int32_t *order, int32_t *count, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w) {
    const double *x = norms2 + (long)w * nr;
    double mx = 0.0;
    for (int r = 0; r < nr; ++r) mx = std::max(mx, x[r]);
    int cnt = 0;
    for (int r = 0; r < nr; ++r) {
      int rank = 0;
      for (int j = 0; j < nr; ++j) rank += (x[j] > x[r]) || (x[j] == x[r] && j < r);
      order[(long)w * nr + rank] = r;
      cnt += x[r] > defl2 * mx;
    }
    count[w] = cnt;
  }
}
void be_gather_rows(const double *src, long ws, int ld, int nc, int nr_src, const int32_t *order, const int32_t *count,
                    double *dst, long wd, int nr_dst, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w)
    for (int r = 0; r < nr_dst; ++r) {
      double *out = dst + (long)w * wd + (long)r * nc;
      if (r >= count[w] || r >= nr_src) { for (int c = 0; c < nc; ++c) out[c] = 0.0; continue; }
      const double *x = src + (long)w * ws + (long)order[(long)w * nr_src + r] * ld;
      for (int c = 0; c < nc; ++c) out[c] = x[c];
    }
}
void be_select_truncate(const double *norms2, int nr, int nsv, int dmin, int dmax, double trunc_err, int tcap,
                        int32_t *order, int32_t *kept, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w) {
    const double *x = norms2 + (long)w * nr;
    std::vector<double> srt((size_t)nr);
    for (int r = 0; r < nr; ++r) {
      int rank = 0;
      for (int j = 0; j < nr; ++j) rank += (x[j] > x[r]) || (x[j] == x[r] && j < r);
      srt[(size_t)rank] = x[r];
      if (rank < tcap) order[(long)w * tcap + rank] = r;
    }
    int n = nsv, k = n;
    if (n > dmin) {
      double total = 0.0;
      for (int i = 0; i < n && i < nr; ++i) total += srt[(size_t)i];
      double kept_sum = total;
      while (k > dmin) {
        double sv2 = (k - 1 < nr) ? srt[(size_t)(k - 1)] : 0.0;
        if (k <= dmax && total > 0.0 && (1.0 - (kept_sum - sv2) / total) > trunc_err) break;
        kept_sum -= sv2;
        --k;
      }
    }
    kept[w] = std::min(k, tcap);
  }
}
void be_gather_rows_normalized(const double *G, long ws, int ld, int nc, const double *norms2, int nr,
                               const int32_t *order, const int32_t *kept, int tcap, double *B, long wb, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w)
    for (int t = 0; t < tcap; ++t) {
      double *out = B + (long)w * wb + (long)t * nc;
      if (t >= kept[w] || t >= nr) { for (int c = 0; c < nc; ++c) out[c] = 0.0; continue; }
      int src = order[(long)w * tcap + t];
      double n2 = norms2[(long)w * nr + src];
      double inv = n2 > 0.0 ? 1.0 / std::sqrt(n2) : 0.0;
      for (int c = 0; c < nc; ++c) out[c] = G[w * ws + (long)src * ld + c] * inv;
    }
}

void be_mt_seed(uint32_t *mt, int32_t *idx, const uint32_t *seeds, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w) {
    uint32_t *s = mt + (long)w * 624;
    s[0] = seeds[w];
    for (int i = 1; i < 624; ++i) s[i] = 1812433253u * (s[i - 1] ^ (s[i - 1] >> 30)) + (uint32_t)i;
    idx[w] = 624;
  }
}
static uint32_t mt_next(uint32_t *s, int32_t &i) {
  if (i >= 624) {
    for (int k = 0; k < 624; ++k) {
      uint32_t y = (s[k] & 0x80000000u) | (s[(k + 1) % 624] & 0x7fffffffu);
      s[k] = s[(k + 397) % 624] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
    }
    i = 0;
  }
  uint32_t y = s[i++];
  y ^= y >> 11; y ^= (y << 7) & 0x9d2c5680u; y ^= (y << 15) & 0xefc60000u; y ^= y >> 18;
  return y;
}
void be_nn_exchange_decide(int32_t *cfg, int nsites, int s1, int s2, const double *psi_b, double *amp,
                           uint32_t *mt, int32_t *idx, int32_t *accepted, int W, const double *jastrow) {
  ++g_launches;
  for (int w = 0; w < W; ++w) {
    int32_t *c = cfg + (long)w * nsites;
    int c1 = c[s1], c2 = c[s2];
    if (c1 == c2) continue;
    double pb = psi_b[w], pa = amp[w];
    bool ok;
    double div = 0.0;
    if (jastrow) { div = std::fabs(pb * jastrow[w]) / std::fabs(pa); ok = div >= 1.0; }
    else ok = std::fabs(pb) >= std::fabs(pa);
    if (!ok) {
      if (!jastrow) div = std::fabs(pb) / std::fabs(pa);
      double P = div * div;
      uint32_t x0 = mt_next(mt + (long)w * 624, idx[w]);
      uint32_t x1 = mt_next(mt + (long)w * 624, idx[w]);
      double r = ((double)x0 + (double)x1 * 4294967296.0) / 18446744073709551616.0;
      if (r >= 1.0) r = std::nextafter(1.0, 0.0);
      ok = r < P;
    }
    if (ok) { c[s1] = c2; c[s2] = c1; amp[w] = pb; accepted[w] += 1; }
  }
}
void be_jastrow_ratio(const int32_t *cfg, int nsites, int s1, int s2, const int32_t *dens, const double *v, double *ratio, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w) {
    const int32_t *c = cfg + (long)w * nsites;
    const int n1 = dens[c[s1]], n2 = dens[c[s2]];
    if (n1 == n2) { ratio[w] = 1.0; continue; }
    double f1 = 0.0, f2 = 0.0;
    for (int j = 0; j < nsites; ++j) {
      if (j != s1) f1 += v[(long)s1 * nsites + j] * (double)dens[c[j]];
      if (j != s2) f2 += v[(long)s2 * nsites + j] * (double)dens[c[j]];
    }
    ratio[w] = n1 < n2 ? std::exp(f1 - f2) : std::exp(f2 - f1);
  }
}
void be_scale(double *x, const double *s, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w) x[w] *= s[w];
}
void be_ratio_accumulate(const double *psi_ex, const double *psi, double coef, double *eloc, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w) eloc[w] += coef * (psi_ex[w] * (1.0 / psi[w]));
}
void be_xxz_bond_energy(const int32_t *cfg, int nsites, int s1, int s2, const double *psi_ex, const double *psi,
                        double jz, double jxy, double *eloc, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w) {
    const int32_t *c = cfg + (long)w * nsites;
    double e;
    if (c[s1] == c[s2]) e = 0.25 * jz;
    else { double inv = 1.0 / psi[w]; e = -0.25 * jz + (psi_ex[w] * inv) * 0.5 * jxy; }
    eloc[w] += e;
  }
}
void be_term_targets(const int32_t *cfg, int nsites, int s1, int s2, int phys, const int32_t *target, const double *coef, int T,
                     int t, int32_t *idx_a, int32_t *idx_b, double *coefw, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w) {
    const int32_t *c = cfg + (long)w * nsites;
    const int c1 = c[s1], c2 = s2 >= 0 ? c[s2] : 0;
    const int p = s2 >= 0 ? c1 * phys + c2 : c1;
    const int tg = target[p * T + t];
    idx_a[w] = tg < 0 ? c1 : (s2 >= 0 ? tg / phys : tg);
    if (idx_b) idx_b[w] = tg < 0 ? c2 : tg % phys;
    coefw[w] = tg < 0 ? 0.0 : coef[p * T + t];
  }
}
void be_term_accumulate(const int32_t *cfg, int nsites, int s1, int s2, int phys, const double *diag, const double *coefw,
                        const double *psi_ex, const double *psi, double *eloc, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w) {
    const int32_t *c = cfg + (long)w * nsites;
    const int p = s2 >= 0 ? c[s1] * phys + c[s2] : c[s1];
    double e = diag ? diag[p] : 0.0;
    if (coefw && coefw[w] != 0.0) e += coefw[w] * (psi_ex[w] * (1.0 / psi[w]));
    eloc[w] += e;
  }
}
// ---- complex (c128) tensors as split planes (backend.h) -----------------------------------------------------------------
void be_embed_complex(const double *Ar, const double *Ai, long wa, int m, int n, double *M, long wm, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w)
    for (long r = 0; r < m; ++r)
      for (long c = 0; c < n; ++c) {
        const double a = Ar[(long)w * wa + r * n + c], b = Ai[(long)w * wa + r * n + c];
        double *Mw = M + (long)w * wm;
        Mw[r * 2 * n + c] = a; Mw[r * 2 * n + n + c] = -b;
        Mw[(r + m) * 2 * n + c] = b; Mw[(r + m) * 2 * n + n + c] = a;
      }
}
void be_split_r(const double *R, long wr, int rows, int n, double *outr, double *outi, long wo, int W) {
  ++g_launches;
  const double s = 0.70710678118654752440;
  for (int w = 0; w < W; ++w)
    for (long r = 0; r < rows; ++r)
      for (long c = 0; c < n; ++c) {
        outr[(long)w * wo + r * n + c] = s * R[(long)w * wr + r * 2 * n + c];
        outi[(long)w * wo + r * n + c] = -s * R[(long)w * wr + r * 2 * n + n + c];
      }
}
void be_complex_basis(double *Bm, long wb, int tcap2, int n, const int32_t *kept2, double *Br, double *Bi, long wo, int tcap,
                      int32_t *keptc, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w) {
    double *B = Bm + (long)w * wb, *outr = Br + (long)w * wo, *outi = Bi + (long)w * wo;
    const int k2 = std::min((int)kept2[w], tcap2), kc = std::min((k2 + 1) / 2, tcap);
    for (long e = 0; e < (long)tcap * n; ++e) { outr[e] = 0.0; outi[e] = 0.0; }
    std::vector<double> res((size_t)std::max(k2, 0));
    for (int q = 0; q < kc; ++q) {
      double best = -1.0;
      for (int j = 0; j < k2; ++j) {
        double sq = 0.0;
        for (int c = 0; c < 2 * n; ++c) sq += B[(long)j * 2 * n + c] * B[(long)j * 2 * n + c];
        res[(size_t)j] = sq;
        best = std::max(best, sq);
      }
      if (best < 1e-10) break;                               // subspace exhausted: the remaining rows stay zero
      // pivot: the first candidate (rows of Bm are sorted by singular value) whose residual is at least half the largest
      int p = 0;
      while (res[(size_t)p] < 0.5 * best) ++p;
      best = res[(size_t)p];
      const double inv = 1.0 / std::sqrt(best);
      for (int c = 0; c < n; ++c) { outr[(long)q * n + c] = inv * B[(long)p * 2 * n + c]; outi[(long)q * n + c] = inv * B[(long)p * 2 * n + n + c]; }
      for (int prev = 0; prev < q; ++prev) {
        double cr = 0.0, ci = 0.0;
        for (int c = 0; c < n; ++c) {
          const double ar = outr[(long)prev * n + c], ai = outi[(long)prev * n + c], br = outr[(long)q * n + c], bi = outi[(long)q * n + c];
          cr += ar * br + ai * bi; ci += ar * bi - ai * br;
        }
        for (int c = 0; c < n; ++c) {
          const double ar = outr[(long)prev * n + c], ai = outi[(long)prev * n + c];
          outr[(long)q * n + c] -= cr * ar - ci * ai;
          outi[(long)q * n + c] -= cr * ai + ci * ar;
        }
      }
      double nn = 0.0;
      for (int c = 0; c < n; ++c) nn += outr[(long)q * n + c] * outr[(long)q * n + c] + outi[(long)q * n + c] * outi[(long)q * n + c];
      const double nv = nn > 0.0 ? 1.0 / std::sqrt(nn) : 0.0;
      for (int c = 0; c < n; ++c) { outr[(long)q * n + c] *= nv; outi[(long)q * n + c] *= nv; }
      for (int j = 0; j < k2; ++j) {
        double cr = 0.0, ci = 0.0;
        for (int c = 0; c < n; ++c) {
          const double ar = outr[(long)q * n + c], ai = outi[(long)q * n + c], br = B[(long)j * 2 * n + c], bi = B[(long)j * 2 * n + n + c];
          cr += ar * br + ai * bi; ci += ar * bi - ai * br;
        }
        for (int c = 0; c < n; ++c) {
          const double ar = outr[(long)q * n + c], ai = outi[(long)q * n + c];
          B[(long)j * 2 * n + c] -= cr * ar - ci * ai;
          B[(long)j * 2 * n + n + c] -= cr * ai + ci * ar;
        }
      }
    }
    for (long e = 0; e < (long)tcap * n; ++e) outi[e] = -outi[e];     // rows of Vt = V^H: conjugates of the right singular vectors
    keptc[w] = kc;
  }
}
void be_complex_combine(const double *d0, const double *d1, const double *d2, const double *d3, double *outr, double *outi, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w) { outr[w] = d0[w] - d1[w]; outi[w] = d2[w] + d3[w]; }
}
void be_nn_exchange_decide_c(int32_t *cfg, int nsites, int s1, int s2, const double *pbr, const double *pbi, double *ampr,
                             double *ampi, uint32_t *mt, int32_t *idx, int32_t *accepted, int W, const double *jastrow) {
  ++g_launches;
  for (int w = 0; w < W; ++w) {
    int32_t *c = cfg + (long)w * nsites;
    const int c1 = c[s1], c2 = c[s2];
    if (c1 == c2) continue;
    const double j = jastrow ? jastrow[w] : 1.0;
    const double ab = jastrow ? std::hypot(pbr[w] * j, pbi[w] * j) : std::hypot(pbr[w], pbi[w]), aa = std::hypot(ampr[w], ampi[w]);
    bool ok = jastrow ? ab / aa >= 1.0 : ab >= aa;
    if (!ok) {
      const double div = ab / aa, P = div * div;
      uint32_t x0 = mt_next(mt + (long)w * 624, idx[w]);
      uint32_t x1 = mt_next(mt + (long)w * 624, idx[w]);
      double r = ((double)x0 + (double)x1 * 4294967296.0) / 18446744073709551616.0;
      if (r >= 1.0) r = std::nextafter(1.0, 0.0);
      ok = r < P;
    }
    if (ok) { c[s1] = c2; c[s2] = c1; ampr[w] = pbr[w]; ampi[w] = pbi[w]; accepted[w] += 1; }
  }
}
void be_xxz_bond_energy_c(const int32_t *cfg, int nsites, int s1, int s2, const double *exr, const double *exi, const double *pr,
                          const double *pi, double jz, double jxy, double *er, double *ei, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w) {
    const int32_t *c = cfg + (long)w * nsites;
    if (c[s1] == c[s2]) { er[w] += 0.25 * jz; continue; }
    const double d = pr[w] * pr[w] + pi[w] * pi[w];
    const double rr = (exr[w] * pr[w] + exi[w] * pi[w]) / d, ri = (exi[w] * pr[w] - exr[w] * pi[w]) / d;
    er[w] += -0.25 * jz + rr * 0.5 * jxy;
    ei[w] += -ri * 0.5 * jxy;
  }
}
void be_ratio_accumulate_c(const double *exr, const double *exi, const double *pr, const double *pi, double coef, double *er,
                           double *ei, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w) {
    const double d = pr[w] * pr[w] + pi[w] * pi[w];
    const double rr = (exr[w] * pr[w] + exi[w] * pi[w]) / d, ri = (exi[w] * pr[w] - exr[w] * pi[w]) / d;
    er[w] += coef * rr;
    ei[w] += -coef * ri;
  }
}
void be_term_accumulate_c(const int32_t *cfg, int nsites, int s1, int s2, int phys, const double *diag, const double *coefw,
                          const double *exr, const double *exi, const double *pr, const double *pi, double *er, double *ei, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w) {
    const int32_t *c = cfg + (long)w * nsites;
    const int p = s2 >= 0 ? c[s1] * phys + c[s2] : c[s1];
    double e_r = diag ? diag[p] : 0.0, e_i = 0.0;
    if (coefw && coefw[w] != 0.0) {
      const double d = pr[w] * pr[w] + pi[w] * pi[w];
      const double rr = (exr[w] * pr[w] + exi[w] * pi[w]) / d, ri = (exi[w] * pr[w] - exr[w] * pi[w]) / d;
      e_r += coefw[w] * rr;
      e_i -= coefw[w] * ri;
    }
    er[w] += e_r;
    ei[w] += e_i;
  }
}
void be_fermion_finish_holes_c(double *hr, double *hi, long hole_stride, const int32_t *hole_off, const int32_t *site_size,
                               const double *gtps, long gtps_im_off, const int64_t *gtps_off, const int32_t *gidx_h,
                               const int32_t *jw_h, int nsites, const double *sign, const double *ampr, const double *ampi, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w)
    for (int site = 0; site < nsites; ++site) {
      const int sz = site_size[site];
      double *a = hr + (long)w * hole_stride + hole_off[site], *b = hi + (long)w * hole_stride + hole_off[site];
      const double *tr = gtps + gtps_off[site] + (long)gidx_h[(long)w * nsites + site] * sz, *ti = tr + gtps_im_off;
      double pr = 0.0, pi = 0.0;
      for (int e = 0; e < sz; ++e) { pr += a[e] * tr[e] - b[e] * ti[e]; pi += a[e] * ti[e] + b[e] * tr[e]; }
      const double d = pr * pr + pi * pi;
      const double fr = (ampr[w] * pr + ampi[w] * pi) / d, fi = (ampi[w] * pr - ampr[w] * pi) / d;
      const double *sg = sign + (long)jw_h[(long)w * nsites + site] * hole_stride + hole_off[site];
      for (int e = 0; e < sz; ++e) {
        const double x = a[e] * sg[e], y = b[e] * sg[e];
        a[e] = x * fr - y * fi;
        b[e] = x * fi + y * fr;
      }
    }
}
void be_accumulate_ostar_c(const double *hr, const double *hi, long hole_stride, const int32_t *hole_off, const int32_t *site_size,
                           const int32_t *tps_off, const int32_t *cfg, int nsites, const double *ampr, const double *ampi,
                           const double *er, const double *ei, double *osr, double *osi, double *eor, double *eoi, int W) {
  ++g_launches;
  for (int site = 0; site < nsites; ++site)
    for (int e = 0; e < site_size[site]; ++e)
      for (int w = 0; w < W; ++w) {
        const int c = cfg[(long)w * nsites + site];
        const double d = ampr[w] * ampr[w] + ampi[w] * ampi[w];
        const double a = hr[(long)w * hole_stride + hole_off[site] + e], b = hi[(long)w * hole_stride + hole_off[site] + e];
        const double qr = (a * ampr[w] + b * ampi[w]) / d, qi = (b * ampr[w] - a * ampi[w]) / d;
        const double orr = qr, oi = -qi;
        const long slot = tps_off[site] + (long)c * site_size[site] + e;
        osr[slot] += orr; osi[slot] += oi;
        eor[slot] += er[w] * orr + ei[w] * oi;
        eoi[slot] += er[w] * oi - ei[w] * orr;
      }
}
void be_fermion_gather(const int32_t *cfg, int rows, int cols, int phys, const int32_t *par, int32_t *gh, int32_t *gv,
                       int32_t *jh, int32_t *jv, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w) {
    const long base = (long)w * rows * cols;
    for (int r = 0; r < rows; ++r)
      for (int c = 0; c < cols; ++c) {
        const long i = base + r * cols + c;
        int left = 0, above = 0;
        for (int k = 0; k < c; ++k) left ^= par[cfg[base + r * cols + k]];
        for (int k = 0; k < r; ++k) above ^= par[cfg[base + k * cols + c]];
        jh[i] = left; jv[i] = above;
        gh[i] = left * phys + cfg[i];
        gv[i] = (6 + above) * phys + cfg[i];
      }
  }
}
void be_fermion_targets(const int32_t *cfg, int nsites, int s1, int s2, int phys, const int32_t *phys_par,
                        const int32_t *jw_h, const int32_t *jw_v, int kind, const int32_t *target, const double *coef,
                        int T, int t, int32_t *idx_a, int32_t *idx_b, double *coefw, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w) {
    const long o = (long)w * nsites;
    fermion_target_one(cfg + o, jw_h + o, jw_v + o, s1, s2, phys, phys_par, kind, target, coef, T, t, idx_a[w], idx_b[w], coefw[w]);
  }
}
void be_fermion_finish_holes(double *holes, long hole_stride, const int32_t *hole_off, const int32_t *site_size,
                             const double *gtps, const int64_t *gtps_off, const int32_t *gidx_h, const int32_t *jw_h,
                             int nsites, const double *sign, const double *amp, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w)
    for (int site = 0; site < nsites; ++site) {
      const int sz = site_size[site];
      double *h = holes + (long)w * hole_stride + hole_off[site];
      const double *t = gtps + gtps_off[site] + (long)gidx_h[(long)w * nsites + site] * sz;
      double psi = 0.0;
      for (int e = 0; e < sz; ++e) psi += h[e] * t[e];
      const double f = amp[w] / psi;
      const double *sg = sign + (long)jw_h[(long)w * nsites + site] * hole_stride + hole_off[site];
      for (int e = 0; e < sz; ++e) h[e] = h[e] * sg[e] * f;
    }
}
void be_xxz_onsite_energy(const int32_t *cfg, int nsites, double h00, double *eloc, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w) eloc[w] += -h00 * ((double)cfg[(long)w * nsites] - 0.5);
}
void be_accumulate_ostar(const double *holes, long hole_stride, const int32_t *hole_off, const int32_t *site_size,
                         const int32_t *tps_off, const int32_t *cfg, int nsites, int phys, const double *amp,
                         const double *eloc, double *osum, double *eosum, int W) {
  ++g_launches;
  (void)phys;
  for (int site = 0; site < nsites; ++site)
    for (int e = 0; e < site_size[site]; ++e)
      for (int w = 0; w < W; ++w) {
        int s = cfg[(long)w * nsites + site];
        double o = (1.0 / amp[w]) * holes[(long)w * hole_stride + hole_off[site] + e];
        long slot = tps_off[site] + (long)s * site_size[site] + e;
        osum[slot] += o;
        eosum[slot] += eloc[w] * o;
      }
}


void be_sr_store_c(const double *hr, const double *hi, long hole_stride, const double *ampr, const double *ampi, const int32_t *cfg,
                   int nsites, double *ostar, int32_t *cfgs, long first, long cap, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w) {
    const double d = ampr[w] * ampr[w] + ampi[w] * ampi[w];
    const double *a = hr + (long)w * hole_stride, *b = hi + (long)w * hole_stride;
    double *x = ostar + (first + w) * 2 * hole_stride, *y = ostar + (cap + first + w) * 2 * hole_stride;
    for (long e = 0; e < hole_stride; ++e) {
      const double qr = (a[e] * ampr[w] + b[e] * ampi[w]) / d, qi = (b[e] * ampr[w] - a[e] * ampi[w]) / d;
      const double o_r = qr, o_i = -qi;
      x[e] = o_r; x[hole_stride + e] = o_i;
      y[e] = -o_i; y[hole_stride + e] = o_r;
    }
    for (int s = 0; s < 2 * nsites; ++s) {
      const int32_t c = cfg[(long)w * nsites + (s % nsites)];
      cfgs[(first + w) * 2 * nsites + s] = c;
      cfgs[(cap + first + w) * 2 * nsites + s] = c;
    }
  }
}
void be_sr_store(const double *holes, long hole_stride, const double *amp, const int32_t *cfg, int nsites,
                 double *ostar, int32_t *cfgs, long first, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w) {
    for (long e = 0; e < hole_stride; ++e) ostar[(first + w) * hole_stride + e] = (1.0 / amp[w]) * holes[(long)w * hole_stride + e];
    for (int s = 0; s < nsites; ++s) cfgs[(first + w) * nsites + s] = cfg[(long)w * nsites + s];
  }
}
void be_sr_dots(const double *ostar, const int32_t *cfgs, long hole_stride, const int32_t *hole_off,
                const int32_t *site_size, const int32_t *tps_off, int nsites, const double *v, double mean_dot_v,
                double *delta, long n) {
  ++g_launches;
  for (long i = 0; i < n; ++i) {
    double acc = 0.0;
    for (int site = 0; site < nsites; ++site)
      for (int e = 0; e < site_size[site]; ++e)
        acc += ostar[i * hole_stride + hole_off[site] + e] * v[tps_off[site] + (long)cfgs[i * nsites + site] * site_size[site] + e];
    delta[i] = acc - mean_dot_v;
  }
}
void be_sr_accumulate(const double *ostar, const int32_t *cfgs, long hole_stride, const int32_t *hole_off,
                      const int32_t *site_size, const int32_t *tps_off, int nsites, int phys, const double *delta,
                      double *out, long n) {
  ++g_launches;
  for (int site = 0; site < nsites; ++site)
    for (int e = 0; e < site_size[site]; ++e) {
      for (int s = 0; s < phys; ++s) out[tps_off[site] + (long)s * site_size[site] + e] = 0.0;
      for (long i = 0; i < n; ++i)
        out[tps_off[site] + (long)cfgs[i * nsites + site] * site_size[site] + e] += delta[i] * ostar[i * hole_stride + hole_off[site] + e];
    }
}

void be_gather_rows_transposed(const double *src, long ws, int ld, int nc, int nr_src, const int32_t *order,
                               const int32_t *count, double *dst, long wd, int n2, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w)
    for (int c = 0; c < nc; ++c)
      for (int r = 0; r < n2; ++r)
        dst[w * wd + (long)c * n2 + r] = (r < count[w] && r < nr_src) ? src[w * ws + (long)order[(long)w * nr_src + r] * ld + c] : 0.0;
}
static int host_truncation_rule(const std::vector<double> &srt, int nsv, int dmin, int dmax, double trunc_err, int tcap) {
  const int nr = (int)srt.size();
  int n = nsv, k = n;
  if (n > dmin) {
    double total = 0.0;
    for (int i = 0; i < n && i < nr; ++i) total += srt[(size_t)i];
    double kept_sum = total;
    while (k > dmin) {
      double sv2 = (k - 1 < nr) ? srt[(size_t)(k - 1)] : 0.0;
      if (k <= dmax && total > 0.0 && (1.0 - (kept_sum - sv2) / total) > trunc_err) break;
      kept_sum -= sv2;
      --k;
    }
  }
  return std::min(k, tcap);
}
void be_svd_small(const SmallSvdArgs &a) {
  ++g_launches;
  const int n = a.n2;
  for (int w = 0; w < a.W; ++w) {
    std::vector<std::vector<double>> X((size_t)n, std::vector<double>((size_t)n));
    for (int k = 0; k < n; ++k)
      for (int i = 0; i < n; ++i) X[(size_t)k][(size_t)i] = a.Rt[w * a.ws + (long)i * a.ld + k];
    int sweeps = 0;
    for (; sweeps < a.max_sweeps; ++sweeps) {
      double off = 0.0;
      for (int p = 0; p < n; ++p)
        for (int q = p + 1; q < n; ++q) {
          double app = 0, aqq = 0, apq = 0;
          for (int i = 0; i < n; ++i) { app += X[p][i] * X[p][i]; aqq += X[q][i] * X[q][i]; apq += X[p][i] * X[q][i]; }
          if (app <= 0.0 || aqq <= 0.0 || apq == 0.0) continue;
          off = std::max(off, std::fabs(apq) / std::sqrt(app * aqq));
          if (apq * apq <= a.tol * a.tol * app * aqq) continue;
          const double zeta = (aqq - app) / (2.0 * apq);
          const double t = (zeta >= 0 ? 1.0 : -1.0) / (std::fabs(zeta) + std::sqrt(1.0 + zeta * zeta));
          const double c = 1.0 / std::sqrt(1.0 + t * t), sn = c * t;
          for (int i = 0; i < n; ++i) {
            const double x = X[p][i], y = X[q][i];
            X[p][i] = c * x - sn * y;
            X[q][i] = sn * x + c * y;
          }
        }
      if (off <= a.tol) { ++sweeps; break; }
    }
    if (a.sweeps) a.sweeps[w] = sweeps;
    std::vector<double> n2v((size_t)n);
    for (int k = 0; k < n; ++k) { double s2 = 0; for (int i = 0; i < n; ++i) s2 += X[k][i] * X[k][i]; n2v[(size_t)k] = s2; }
    std::vector<int> perm((size_t)n);
    for (int k = 0; k < n; ++k) {
      int rank = 0;
      for (int j = 0; j < n; ++j) rank += (n2v[j] > n2v[k]) || (n2v[j] == n2v[k] && j < k);
      perm[(size_t)rank] = k;
    }
    std::vector<double> srt((size_t)n);
    for (int r = 0; r < n; ++r) srt[(size_t)r] = n2v[(size_t)perm[(size_t)r]];
    const int kept = host_truncation_rule(srt, a.nsv, a.dmin, a.dmax, a.trunc_err, a.tcap);
    a.kept[w] = kept;
    for (int i = 0; i < n; ++i)
      for (int t = 0; t < a.tcap; ++t) {
        double v = 0.0;
        if (t < kept && t < n && srt[(size_t)t] > 0.0) v = X[(size_t)perm[(size_t)t]][(size_t)i] / std::sqrt(srt[(size_t)t]);
        a.out[w * a.wo + (long)i * a.tcap + t] = v;
      }
  }
}
void be_transpose_permute(const double *C0, long wc, int nc, int tcap, const int32_t *order, double *B, long wb, int W) {
  ++g_launches;
  for (int w = 0; w < W; ++w)
    for (int j = 0; j < nc; ++j)
      for (int t = 0; t < tcap; ++t)
        B[w * wb + (long)t * nc + (order ? order[(long)w * nc + j] : j)] = C0[w * wc + (long)j * tcap + t];
}
void be_vec_lincomb(double *out, double ca, const double *a, double cb, const double *b, long n) {
  ++g_launches;
  for (long i = 0; i < n; ++i) out[i] = ca * a[i] + (b ? cb * b[i] : 0.0);
}
void be_vec_dot(const double *a, const double *b, long n, double *result) {
  ++g_launches;
  double s = 0.0;
  for (long i = 0; i < n; ++i) s += a[i] * b[i];
  result[0] = s;
}

}  // namespace peps
