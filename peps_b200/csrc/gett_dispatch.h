// Kernel selection of be_gett: which contraction kernel, tile and copy widths a call gets. A pure host-side function of the
// call's arguments, shared by the CUDA launch (backend_cuda.cu) and the peps_test_gett entry point (c_api.cpp), so the
// variant a test reports is the one the launch takes.
#pragma once
#include <cstdint>
#include <cstdlib>
#include "backend.h"

namespace peps {

enum GettKernel { GETT_NONE = 0, GETT_SMALL = 1, GETT_LARGE = 2 };
struct GettVariant {
  int kernel = GETT_NONE;        // GETT_NONE: nothing is launched (empty call)
  int tile_m = 0, tile_n = 0;    // CTA tile
  int akf = 0, bkf = 0;          // A / B tiles stored contracted-fast (GettDesc::a_kfast, !GettDesc::b_nfast)
  int avec = 0, bvec = 0, cvec = 0;   // 16-byte copies of A / B / C (large-tile kernel only)
};

constexpr int GETT_LARGE_TILE_N = 64;      // N extent of every gett_large_kernel tile

// A 16-byte copy of an element pair moves (2i, 2i+1) of walker w only when the walker's base is 16-byte aligned.
inline bool gett_operand_aligned2(const Operand &o) {
  return ((reinterpret_cast<uintptr_t>(o.p) & 15) == 0) && ((o.ws & 1) == 0) && ((o.bs & 1) == 0) &&
         (o.gidx == nullptr || (o.gs & 1) == 0);
}

inline GettVariant gett_variant(const GettDesc &d, const Operand &A, const Operand &B, const Operand &C, int W, int NB) {
  GettVariant v;
  if (d.M <= 0 || d.N <= 0 || W <= 0 || NB <= 0) return v;
  static const bool use_large = []() { const char *e = std::getenv("PEPS_GETT_LARGE"); return e ? std::atoi(e) != 0 : true; }();
  v.akf = d.a_kfast != 0;
  v.bkf = d.b_nfast == 0;
  if (use_large && d.M > 32 && d.N > 32 && d.K >= 8) {
    v.kernel = GETT_LARGE;
    v.avec = d.a_vec2 && gett_operand_aligned2(A);
    v.bvec = d.b_vec2 && gett_operand_aligned2(B);
    v.cvec = d.c_vec2 && gett_operand_aligned2(C);
    // 128-row tiles unless that leaves fewer than two CTAs per SM: then 64-row tiles double the CTA count
    const long ctas128 = (long)((d.M + 127) / 128) * ((d.N + GETT_LARGE_TILE_N - 1) / GETT_LARGE_TILE_N) * NB * W;
    v.tile_m = (ctas128 < 2L * 148 || d.M <= 96) ? 64 : 128;
    v.tile_n = GETT_LARGE_TILE_N;
    return v;
  }
  v.kernel = GETT_SMALL;
  if (d.M > 32 && d.N > 32) { v.tile_m = 64; v.tile_n = 64; }
  else if (d.M > 32) { v.tile_m = 64; v.tile_n = 16; }
  else if (d.N > 32) { v.tile_m = 16; v.tile_n = 64; }
  else { v.tile_m = 32; v.tile_n = 32; }
  return v;
}

}  // namespace peps
