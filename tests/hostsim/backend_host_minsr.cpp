// TEST-ONLY host simulation of the MinSR device ops of peps_b200/csrc/backend.h (be_sr_gram, be_minsr_centre,
// be_minsr_embed, be_chol, be_chol_solve): plain loops, linked into the host-simulation library next to
// backend_host.cpp and never into the product library.
#include <cmath>
#include <cstdint>
#include "../../peps_b200/csrc/backend.h"

namespace peps {

void be_sr_gram(const double *left, const double *right, const int32_t *cfgs, long hole_stride, const int32_t *hole_off,
                const int32_t *site_size, const int32_t *, int nsites, long n, double lower_sign, double *G) {
  for (long i = 0; i < n; ++i)
    for (long j = i; j < n; ++j) {
      double acc = 0.0;
      for (int site = 0; site < nsites; ++site) {
        if (cfgs[i * nsites + site] != cfgs[j * nsites + site]) continue;
        const double *a = left + i * hole_stride + hole_off[site], *b = right + j * hole_stride + hole_off[site];
        for (int e = 0; e < site_size[site]; ++e) acc += a[e] * b[e];
      }
      G[i * n + j] = acc;
      G[j * n + i] = lower_sign * acc;
      if (i == j && lower_sign < 0) G[i * n + i] = 0.0;
    }
}
void be_minsr_centre(const double *G, const double *a, double c, double sign, long n, double scale, double *T) {
  for (long i = 0; i < n; ++i)
    for (long j = 0; j < n; ++j) T[i * n + j] = (sign < 0 && i == j) ? 0.0 : scale * (G[i * n + j] - a[i] - sign * a[j] + c);
}
void be_minsr_embed(const double *Tr, const double *Ti, long n, double shift, double *M) {
  const long m = Ti ? 2 * n : n;
  for (long i = 0; i < m; ++i)
    for (long j = 0; j < m; ++j) {
      const long bi = i / n, bj = j / n, ii = i % n, jj = j % n;
      const double v = (bi == bj) ? Tr[ii * n + jj] : (bi > bj ? Ti[ii * n + jj] : -Ti[ii * n + jj]);
      M[i * m + j] = v + (i == j ? shift : 0.0);
    }
}
void be_chol(double *M, long m, int32_t *info) {
  info[0] = 0;
  for (long j = 0; j < m; ++j) {
    double d = M[j * m + j];
    for (long p = 0; p < j; ++p) d -= M[j * m + p] * M[j * m + p];
    if (!(d > 0.0)) { if (!info[0]) info[0] = (int32_t)(j + 1); d = 1.0; }
    d = std::sqrt(d);
    M[j * m + j] = d;
    for (long i = j + 1; i < m; ++i) {
      double s = M[i * m + j];
      for (long p = 0; p < j; ++p) s -= M[i * m + p] * M[j * m + p];
      M[i * m + j] = s / d;
    }
  }
}
void be_chol_solve(const double *L, long m, double *b) {
  for (long i = 0; i < m; ++i) {
    double s = b[i];
    for (long j = 0; j < i; ++j) s -= L[i * m + j] * b[j];
    b[i] = s / L[i * m + i];
  }
  for (long i = m - 1; i >= 0; --i) {
    double s = b[i];
    for (long j = i + 1; j < m; ++j) s -= L[j * m + i] * b[j];
    b[i] = s / L[i * m + i];
  }
}

}  // namespace peps
