// sm_100a implementation of backend.h: hand-written kernels for the walker-batched VMC sampling path.
//
// Kernel inventory (DESIGN.md section 4 gives the roofline of each):
//   gett_kernel        walker-batched FP64 tensor contraction on the DMMA pipe (mma.sync m8n8k4.f64), operands
//                      addressed through separable offset tables so no transpose pass ever touches HBM; the
//                      physical-index slice of the sampled site is gathered straight from the shared TPS.
//   dot_kernel         rank-3 inner product closing a trace.
//   panel_qr_kernel    one panel of the communication-avoiding R-only Householder QR, panel resident in smem.
//   jacobi_round_kernel one round of one-sided block Jacobi (Gram + rotation on DMMA, panel resident in smem).
//   small kernels      row norms, truncation/selection, RNG + Metropolis decision, energies, O* accumulation.
//   sr_gram_kernel     MinSR: masked Gram of the O* store on the DMMA pipe (per-site mask folded at site boundaries).
//   chol_*_kernel      MinSR: blocked Cholesky (trailing update on DMMA) and the two triangular solves.
#include <cuda.h>
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <stdexcept>
#include <algorithm>
#include <string>
#include <type_traits>
#include <unordered_map>
#include <map>
#include <mutex>
#include <utility>
#include <vector>
#include "backend.h"
#include "gett_dispatch.h"

namespace peps {

// Stream, launch counter, profiler and per-device kernel attributes live in a backend context (BeCtx) owned by the
// engine. Every C-ABI entry binds its context to the calling thread first (be_ctx_bind: cudaSetDevice + current
// pointer), so a context may be created in one host thread and driven from another, and contexts on different
// devices can coexist in one thread. Contexts driven from different host threads run on different streams, so
// their kernels overlap on the GPU.
#define CUDA_CHECK(x)                                                                              \
  do {                                                                                             \
    cudaError_t e_ = (x);                                                                          \
    if (e_ != cudaSuccess)                                                                         \
      throw std::runtime_error(std::string("CUDA error: ") + cudaGetErrorString(e_) + " at " +     \
                               __FILE__ + ":" + std::to_string(__LINE__));                         \
  } while (0)

// ---- per-class event timing --------------------------------------------------------------------------
struct Profiler {
  bool on = false;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pending[KC_COUNT];
  std::vector<cudaEvent_t> pool;
  double ms[KC_COUNT] = {0}, flops[KC_COUNT] = {0};
  long launches[KC_COUNT] = {0};
  cudaEvent_t get() {
    if (!pool.empty()) { cudaEvent_t e = pool.back(); pool.pop_back(); return e; }
    cudaEvent_t e;
    CUDA_CHECK(cudaEventCreate(&e));
    return e;
  }
};
struct BeCtx {
  int device = 0;
  cudaStream_t stream = nullptr;
  long launches = 0;
  Profiler prof;
  double *dot_part = nullptr;                          // partial sums of the K-split trace closure
  double *vdot_part = nullptr;                         // partial sums of be_vec_dot
  size_t dot_part_cap = 0;
  double *gram_part = nullptr;                         // split-K partial tiles of be_sr_gram
  size_t gram_part_cap = 0;
  int32_t *gram_split = nullptr;                       // site ranges of the split-K slices
  int gram_split_cap = 0;
};
static thread_local BeCtx *g_cx = nullptr;
static thread_local int g_cur_device = -1;
static inline BeCtx &cx() {
  if (!g_cx) throw std::runtime_error("peps_b200: no backend context bound to this thread");
  return *g_cx;
}
#define g_stream (cx().stream)
#define g_prof (cx().prof)

BeCtx *be_ctx_create(int device) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0)
    throw std::runtime_error("peps_b200: no CUDA device available; the product has no CPU fallback");
  if (device < 0 || device >= n) throw std::invalid_argument("peps_b200: CUDA device ordinal out of range");
  CUDA_CHECK(cudaSetDevice(device));
  g_cur_device = device;
  BeCtx *c = new BeCtx();
  c->device = device;
  cudaError_t se = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
  if (se != cudaSuccess) { delete c; throw std::runtime_error(std::string("CUDA error: ") + cudaGetErrorString(se)); }
  return c;
}
void be_ctx_bind(BeCtx *c) {
  if (c && g_cur_device != c->device) { CUDA_CHECK(cudaSetDevice(c->device)); g_cur_device = c->device; }
  g_cx = c;
}
void be_ctx_destroy(BeCtx *c) {
  if (!c) return;
  if (g_cur_device != c->device) { cudaSetDevice(c->device); g_cur_device = c->device; }
  cudaStreamSynchronize(c->stream);
  for (int k = 0; k < KC_COUNT; ++k)
    for (auto &pr : c->prof.pending[k]) { cudaEventDestroy(pr.first); cudaEventDestroy(pr.second); }
  for (cudaEvent_t ev : c->prof.pool) cudaEventDestroy(ev);
  if (c->dot_part) cudaFree(c->dot_part);
  if (c->vdot_part) cudaFree(c->vdot_part);
  if (c->gram_part) cudaFree(c->gram_part);
  if (c->gram_split) cudaFree(c->gram_split);
  cudaStreamDestroy(c->stream);
  if (g_cx == c) g_cx = nullptr;
  delete c;
}
// stand-alone kernel tests (peps_test_*): one default context per host thread and device
void be_init(int device) {
  static thread_local std::unordered_map<int, BeCtx *> defaults;
  auto it = defaults.find(device);
  if (it == defaults.end()) it = defaults.emplace(device, be_ctx_create(device)).first;
  be_ctx_bind(it->second);
}

static inline void post_launch() {
  ++cx().launches;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) throw std::runtime_error(std::string("kernel launch failed: ") + cudaGetErrorString(e));
}
// dynamic shared memory opt-in, remembered per context (= per device)
// The attribute is a property of (device, kernel) shared by every context of the process, and setting it REPLACES the
// previous value: the largest size ever requested is kept in a process-wide table (contexts on several host threads
// ask for different sizes of the same kernel concurrently).
template <class K>
static inline void ensure_smem(K kern, size_t smem) {
  static std::mutex mu;
  static std::map<std::pair<int, const void *>, size_t> table;
  std::lock_guard<std::mutex> lock(mu);
  size_t &have = table[{cx().device, (const void *)kern}];
  if (smem > have) {
    CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    have = smem;
  }
}

struct LaunchScope {          // brackets one kernel launch
  int c; cudaEvent_t s = nullptr;
  LaunchScope(int cls, double fl) : c(cls) {
    g_prof.launches[c] += 1;
    g_prof.flops[c] += fl;
    if (g_prof.on) { s = g_prof.get(); cudaEventRecord(s, g_stream); }
  }
  ~LaunchScope() {
    if (s) { cudaEvent_t e = g_prof.get(); cudaEventRecord(e, g_stream); g_prof.pending[c].push_back({s, e}); }
  }
};
void be_profile_enable(int on) { g_prof.on = on != 0; }
void be_profile_collect(double *ms, long *launches, double *flops, int reset) {
  CUDA_CHECK(cudaStreamSynchronize(g_stream));
  for (int c = 0; c < KC_COUNT; ++c) {
    for (auto &pr : g_prof.pending[c]) {
      float t = 0.f;
      cudaEventElapsedTime(&t, pr.first, pr.second);
      g_prof.ms[c] += t;
      g_prof.pool.push_back(pr.first);
      g_prof.pool.push_back(pr.second);
    }
    g_prof.pending[c].clear();
    if (ms) ms[c] = g_prof.ms[c];
    if (launches) launches[c] = g_prof.launches[c];
    if (flops) flops[c] = g_prof.flops[c];
    if (reset) { g_prof.ms[c] = 0; g_prof.launches[c] = 0; g_prof.flops[c] = 0; }
  }
}

const char *be_name() { return "cuda-sm_100a"; }
void *be_malloc(size_t bytes) {
  void *p = nullptr;
  CUDA_CHECK(cudaMalloc(&p, bytes ? bytes : 8));
  return p;
}
void be_free(void *p) { if (p) cudaFree(p); }
void be_memset0(void *p, size_t bytes) { CUDA_CHECK(cudaMemsetAsync(p, 0, bytes, g_stream)); }
void be_h2d(void *dst, const void *src, size_t bytes) {
  CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, g_stream));
  CUDA_CHECK(cudaStreamSynchronize(g_stream));
}
void be_d2h(void *dst, const void *src, size_t bytes) {
  CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, g_stream));
  CUDA_CHECK(cudaStreamSynchronize(g_stream));
}
void be_d2d(void *dst, const void *src, size_t bytes) {
  CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, g_stream));
}
void be_sync() { CUDA_CHECK(cudaStreamSynchronize(g_stream)); }
void *be_stream() { return (void *)g_stream; }
long be_launch_count() { return cx().launches; }

// =====================================================================================================
// gett: walker-batched FP64 contraction on the tensor (DMMA) pipe
// =====================================================================================================
__device__ __forceinline__ void dmma8x8x4(double &c0, double &c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

__device__ __forceinline__ const double *operand_base(const Operand &o, int w, int b) {
  const double *p = o.p + (long)w * o.ws + (long)b * o.bs;
  if (o.gidx) p += (long)o.gidx[(long)w * o.gws] * o.gs;
  return p;
}

constexpr int GETT_THREADS = 128;
constexpr int GETT_BK = 16;

// CTA tile (16*WMT) x (16*WNT), 2x2 warps, each warp (8*WMT) x (8*WNT) made of m8n8k4 DMMA tiles.
template <int WMT, int WNT>
__global__ void __launch_bounds__(GETT_THREADS, 3)
gett_kernel(GettDesc d, Operand A, Operand B, Operand C, double alpha, double beta) {
  constexpr int BM = 16 * WMT, BN = 16 * WNT, BK = GETT_BK;
  constexpr int LDA = BM + 4, LDB = BN + 4;       // +4 doubles: conflict-free DMMA fragment loads
  constexpr int NA = BM * BK / GETT_THREADS, NBv = BN * BK / GETT_THREADS;
  __shared__ double As[2][BK * LDA];         // double buffered: one barrier per K step
  __shared__ double Bs[2][BK * LDB];

  const int tiles_m = (d.M + BM - 1) / BM;
  const int tm = blockIdx.x % tiles_m, tn = blockIdx.x / tiles_m;
  const int m0 = tm * BM, n0 = tn * BN;
  const int w = blockIdx.z, bb = blockIdx.y;
  const double *Ab = operand_base(A, w, bb);
  const double *Bb = operand_base(B, w, bb);
  double *Cb = const_cast<double *>(operand_base(C, w, bb));
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int wm = warp >> 1, wn = warp & 1;
  if ((d.m_cnt && m0 >= d.m_cnt[w] * d.m_scale) || (d.n_cnt && n0 >= d.n_cnt[w] * d.n_scale)) {
    for (int e = t; e < BM * BN; e += GETT_THREADS) {
      const int m = m0 + e / BN, n = n0 + e % BN;
      if (m < d.M && n < d.N) { double *cp = Cb + d.cm[m] + d.cn[n]; *cp = (beta != 0.0) ? beta * (*cp) : 0.0; }
    }
    return;
  }

  // per-thread loader coordinates (fixed part hoisted out of the K loop)
  int a_ml[NA], a_kl[NA], a_off[NA];
#pragma unroll
  for (int i = 0; i < NA; ++i) {
    int e = t + i * GETT_THREADS;
    if (d.a_kfast) { a_kl[i] = e % BK; a_ml[i] = e / BK; } else { a_ml[i] = e % BM; a_kl[i] = e / BM; }
    int m = m0 + a_ml[i];
    a_off[i] = (m < d.M) ? d.am[m] : -1;
  }
  int b_nl[NBv], b_kl[NBv], b_off[NBv];
#pragma unroll
  for (int i = 0; i < NBv; ++i) {
    int e = t + i * GETT_THREADS;
    if (d.b_nfast) { b_nl[i] = e % BN; b_kl[i] = e / BN; } else { b_kl[i] = e % BK; b_nl[i] = e / BK; }
    int n = n0 + b_nl[i];
    b_off[i] = (n < d.N) ? d.bn[n] : -1;
  }

  double acc[WMT][WNT][2];
#pragma unroll
  for (int i = 0; i < WMT; ++i)
#pragma unroll
    for (int j = 0; j < WNT; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

  double ra[NA], rb[NBv];
  auto load_global = [&](int k0) {
#pragma unroll
    for (int i = 0; i < NA; ++i) {
      int k = k0 + a_kl[i];
      ra[i] = (a_off[i] >= 0 && k < d.K) ? __ldg(Ab + a_off[i] + d.ak[k]) : 0.0;
    }
#pragma unroll
    for (int i = 0; i < NBv; ++i) {
      int k = k0 + b_kl[i];
      rb[i] = (b_off[i] >= 0 && k < d.K) ? __ldg(Bb + b_off[i] + d.bk[k]) : 0.0;
    }
  };
  auto store_smem = [&](int buf) {
#pragma unroll
    for (int i = 0; i < NA; ++i) As[buf][a_kl[i] * LDA + a_ml[i]] = ra[i];
#pragma unroll
    for (int i = 0; i < NBv; ++i) Bs[buf][b_kl[i] * LDB + b_nl[i]] = rb[i];
  };

  const int nk = (d.K + BK - 1) / BK;
  int kt0 = 0;
  if (d.klo_m != nullptr || d.klo_n != nullptr) {      // structural zeros: skip the K steps below both bounds
    __shared__ int s_klo[2];
    if (t < 2) s_klo[t] = 0x7fffffff;
    __syncthreads();
    int vm = 0x7fffffff, vn = 0x7fffffff;
    if (d.klo_m) { for (int i = t; i < BM; i += GETT_THREADS) if (m0 + i < d.M) vm = min(vm, d.klo_m[m0 + i]); } else vm = 0;
    if (d.klo_n) { for (int i = t; i < BN; i += GETT_THREADS) if (n0 + i < d.N) vn = min(vn, d.klo_n[n0 + i]); } else vn = 0;
    atomicMin(&s_klo[0], vm);
    atomicMin(&s_klo[1], vn);
    __syncthreads();
    kt0 = min(nk, max(s_klo[0], s_klo[1]) / BK);
  }
  if (kt0 < nk) {
    load_global(kt0 * BK);
    store_smem(0);
  }
  __syncthreads();
  int cur = 0;
  for (int kt = kt0; kt < nk; ++kt) {
    if (kt + 1 < nk) load_global((kt + 1) * BK);
#pragma unroll
    for (int kk = 0; kk < BK; kk += 4) {
      double af[WMT], bf[WNT];
      const int kr = kk + (lane & 3), rr = lane >> 2;
#pragma unroll
      for (int i = 0; i < WMT; ++i) af[i] = As[cur][kr * LDA + wm * 8 * WMT + i * 8 + rr];
#pragma unroll
      for (int j = 0; j < WNT; ++j) bf[j] = Bs[cur][kr * LDB + wn * 8 * WNT + j * 8 + rr];
#pragma unroll
      for (int i = 0; i < WMT; ++i)
#pragma unroll
        for (int j = 0; j < WNT; ++j) dmma8x8x4(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
    }
    if (kt + 1 < nk) store_smem(cur ^ 1);      // the other buffer: nobody reads it during this step
    __syncthreads();
    cur ^= 1;
  }
  // epilogue
#pragma unroll
  for (int i = 0; i < WMT; ++i) {
    int m = m0 + wm * 8 * WMT + i * 8 + (lane >> 2);
    if (m >= d.M) continue;
    int cmo = d.cm[m];
#pragma unroll
    for (int j = 0; j < WNT; ++j) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        int n = n0 + wn * 8 * WNT + j * 8 + 2 * (lane & 3) + h;
        if (n >= d.N) continue;
        double *cp = Cb + cmo + d.cn[n];
        double v = alpha * acc[i][j][h];
        if (beta != 0.0) v += beta * (*cp);
        *cp = v;
      }
    }
  }
}

// ---- large-tile contraction kernel -----------------------------------------------------------------------
// CTA tile 128 (M) x 64 (N), 8 warps as 4 x 2, warp tile 32 x 32 (4 x 4 DMMA m8n8k4 tiles, 16 accumulator pairs); or,
// when the launch would otherwise leave SMs idle, 64 x 64 with 8 warps as 2 x 4 (warp tile 32 x 16).
// Operand tiles travel global -> shared with cp.async (LDGSTS: no register staging, the copy engine zero-fills the
// ragged edges) through a 3-stage ring, one barrier per K step of 16; 16-byte copies wherever the planner proved that
// pairs along the operand's unit-stride index are contiguous and aligned (GettDesc::a_vec2 / b_vec2), 8-byte copies
// through the offset tables otherwise (true gathers). Each operand tile is laid out in shared memory along ITS OWN
// unit-stride index -- [k][m] (+4 pad) when the free index is fast, [m][k] (+4 pad) when the contracted index is fast --
// so both the copy writes and the DMMA fragment reads are bank-conflict free in either case.
constexpr int GL_BN = GETT_LARGE_TILE_N, GL_BK = 16, GL_THREADS = 256;
constexpr int GL_LDB = GL_BN + 4, GL_LDK = GL_BK + 4;
__host__ __device__ constexpr int gl_a_elems(int bm, bool akf) { return akf ? bm * GL_LDK : GL_BK * (bm + 4); }
__host__ __device__ constexpr int gl_b_elems(bool bkf) { return bkf ? GL_BN * GL_LDK : GL_BK * GL_LDB; }
// ring depth: four stages when two CTAs of that size still share an SM (the K = 64 contractions then have every K step in
// flight from the start), three otherwise
__host__ __device__ constexpr int gl_stages(int bm, bool akf, bool bkf) {
  return (size_t)4 * (gl_a_elems(bm, akf) + gl_b_elems(bkf)) * sizeof(double) <= 113 * 1024 ? 4 : 3;
}
__host__ __device__ constexpr size_t gl_smem(int bm, bool akf, bool bkf) {
  return (size_t)gl_stages(bm, akf, bkf) * (gl_a_elems(bm, akf) + gl_b_elems(bkf)) * sizeof(double);
}

__device__ __forceinline__ void cp_async16(void *dst, const void *src, bool valid) {
  const unsigned saddr = (unsigned)__cvta_generic_to_shared(dst);
  const int sz = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(saddr), "l"(src), "r"(sz));
}
__device__ __forceinline__ void cp_async8(void *dst, const void *src, bool valid) {
  const unsigned saddr = (unsigned)__cvta_generic_to_shared(dst);
  const int sz = valid ? 8 : 0;
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(saddr), "l"(src), "r"(sz));
}

// AKF: A's unit-stride index is a contracted one (tile stored [m][k]); BKF: likewise for B (tile stored [n][k]).
// WGM: warps along M (4: 128 x 64 tile, 2: 64 x 64 tile)
template <bool AKF, bool BKF, int WGM>
__global__ void __launch_bounds__(GL_THREADS, 2)
gett_large_kernel(GettDesc d, Operand A, Operand B, Operand C, double alpha, double beta, int avec, int bvec, int cvec) {
  constexpr int GL_BM = 32 * WGM, GL_LDA = GL_BM + 4, GL_A_ELEMS = gl_a_elems(GL_BM, AKF), GL_B_ELEMS = gl_b_elems(BKF);
  constexpr int GL_STAGES = gl_stages(GL_BM, AKF, BKF);
  constexpr int WGN = 8 / WGM, NT = GL_BN / (8 * WGN);        // warps along N, 8-column tiles per warp (4 or 2)
  constexpr int APT = GL_BM * GL_BK / 2 / GL_THREADS;        // A pairs per thread (4 or 2)
  extern __shared__ __align__(16) double gl_sm[];
  double *As = gl_sm;                                        // [STAGES][GL_A_ELEMS]
  double *Bs = gl_sm + GL_STAGES * GL_A_ELEMS;               // [STAGES][GL_B_ELEMS]
  const int tiles_m = (d.M + GL_BM - 1) / GL_BM;
  const int tm = blockIdx.x % tiles_m, tn = blockIdx.x / tiles_m;
  const int m0 = tm * GL_BM, n0 = tn * GL_BN;
  const int w = blockIdx.z, bb = blockIdx.y;
  const double *Ab = operand_base(A, w, bb);
  const double *Bb = operand_base(B, w, bb);
  double *Cb = const_cast<double *>(operand_base(C, w, bb));
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int wm = warp / WGN, wn = warp % WGN;
  if ((d.m_cnt && m0 >= d.m_cnt[w] * d.m_scale) || (d.n_cnt && n0 >= d.n_cnt[w] * d.n_scale)) {
    // the whole tile lies in this walker's zero tail: C = beta * C (+ 0)
    for (int e = t; e < GL_BM * GL_BN; e += GL_THREADS) {
      const int m = m0 + e / GL_BN, n = n0 + e % GL_BN;
      if (m < d.M && n < d.N) { double *cp = Cb + d.cm[m] + d.cn[n]; *cp = (beta != 0.0) ? beta * (*cp) : 0.0; }
    }
    return;
  }

  // ---- loader coordinates: the free-index part of every offset is fixed for the whole K loop -------------------
  // A tile = BM * 8 pairs: free-fast -> pair (m2 = q % (BM/2), k = q / (BM/2)); contracted-fast -> pair (k2 = q % 8, m = q / 8)
  int a_fo[APT][2];      // offsets of the (up to) two elements of pair i along the free index (-1: outside M)
  int a_kl[APT];         // first K index of pair i inside the K step
  int a_so[APT];         // shared-memory offset of pair i
#pragma unroll
  for (int i = 0; i < APT; ++i) {
    const int q = t + i * GL_THREADS;
    if (AKF) {
      const int kp = q & 7, ml = q >> 3, m = m0 + ml;
      a_kl[i] = 2 * kp; a_so[i] = ml * GL_LDK + 2 * kp;
      a_fo[i][0] = (m < d.M) ? d.am[m] : -1; a_fo[i][1] = a_fo[i][0];
    } else {
      const int mp = q % (GL_BM / 2), kl = q / (GL_BM / 2), m = m0 + 2 * mp;
      a_kl[i] = kl; a_so[i] = kl * GL_LDA + 2 * mp;
      a_fo[i][0] = (m < d.M) ? d.am[m] : -1; a_fo[i][1] = (m + 1 < d.M) ? d.am[m + 1] : -1;
    }
  }
  // B tile = 512 pairs: free-fast -> pair (n2 = q % 32, k = q / 32); contracted-fast -> pair (k2 = q % 8, n = q / 8)
  int b_fo[2][2], b_kl[2], b_so[2];
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int q = t + i * GL_THREADS;
    if (BKF) {
      const int kp = q & 7, nl = q >> 3, n = n0 + nl;
      b_kl[i] = 2 * kp; b_so[i] = nl * GL_LDK + 2 * kp;
      b_fo[i][0] = (n < d.N) ? d.bn[n] : -1; b_fo[i][1] = b_fo[i][0];
    } else {
      const int np = q & 31, kl = q >> 5, n = n0 + 2 * np;
      b_kl[i] = kl; b_so[i] = kl * GL_LDB + 2 * np;
      b_fo[i][0] = (n < d.N) ? d.bn[n] : -1; b_fo[i][1] = (n + 1 < d.N) ? d.bn[n + 1] : -1;
    }
  }
  auto issue = [&](int kt, int stage) {
    const int k0 = kt * GL_BK;
    double *as = As + stage * GL_A_ELEMS, *bs = Bs + stage * GL_B_ELEMS;
#pragma unroll
    for (int i = 0; i < APT; ++i) {
      const int k = k0 + a_kl[i];
      if (AKF) {                                   // the pair runs along K: (k, k+1) of one row m
        const bool v0 = a_fo[i][0] >= 0 && k < d.K, v1 = a_fo[i][0] >= 0 && k + 1 < d.K;
        const int o0 = v0 ? a_fo[i][0] + d.ak[k] : 0;
        if (avec) cp_async16(as + a_so[i], Ab + o0, v0);
        else {
          cp_async8(as + a_so[i], Ab + o0, v0);
          cp_async8(as + a_so[i] + 1, Ab + (v1 ? a_fo[i][0] + d.ak[k + 1] : 0), v1);
        }
      } else {                                     // the pair runs along M: (m, m+1) at one k
        const bool kin = k < d.K;
        const int ko = kin ? d.ak[k] : 0;
        const bool v0 = kin && a_fo[i][0] >= 0, v1 = kin && a_fo[i][1] >= 0;
        if (avec) cp_async16(as + a_so[i], Ab + (v0 ? a_fo[i][0] + ko : 0), v0);
        else {
          cp_async8(as + a_so[i], Ab + (v0 ? a_fo[i][0] + ko : 0), v0);
          cp_async8(as + a_so[i] + 1, Ab + (v1 ? a_fo[i][1] + ko : 0), v1);
        }
      }
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int k = k0 + b_kl[i];
      if (BKF) {
        const bool v0 = b_fo[i][0] >= 0 && k < d.K, v1 = b_fo[i][0] >= 0 && k + 1 < d.K;
        const int o0 = v0 ? b_fo[i][0] + d.bk[k] : 0;
        if (bvec) cp_async16(bs + b_so[i], Bb + o0, v0);
        else {
          cp_async8(bs + b_so[i], Bb + o0, v0);
          cp_async8(bs + b_so[i] + 1, Bb + (v1 ? b_fo[i][0] + d.bk[k + 1] : 0), v1);
        }
      } else {
        const bool kin = k < d.K;
        const int ko = kin ? d.bk[k] : 0;
        const bool v0 = kin && b_fo[i][0] >= 0, v1 = kin && b_fo[i][1] >= 0;
        if (bvec) cp_async16(bs + b_so[i], Bb + (v0 ? b_fo[i][0] + ko : 0), v0);
        else {
          cp_async8(bs + b_so[i], Bb + (v0 ? b_fo[i][0] + ko : 0), v0);
          cp_async8(bs + b_so[i] + 1, Bb + (v1 ? b_fo[i][1] + ko : 0), v1);
        }
      }
    }
  };

  const int nk = (d.K + GL_BK - 1) / GL_BK;
  int kt0 = 0;
  if (d.klo_m != nullptr || d.klo_n != nullptr) {      // structural zeros: skip the K steps below both bounds
    __shared__ int s_klo[2];
    if (t < 2) s_klo[t] = 0x7fffffff;
    __syncthreads();
    int vm = 0x7fffffff, vn = 0x7fffffff;
    if (d.klo_m) { for (int i = t; i < GL_BM; i += GL_THREADS) if (m0 + i < d.M) vm = min(vm, d.klo_m[m0 + i]); } else vm = 0;
    if (d.klo_n) { for (int i = t; i < GL_BN; i += GL_THREADS) if (n0 + i < d.N) vn = min(vn, d.klo_n[n0 + i]); } else vn = 0;
    atomicMin(&s_klo[0], vm);
    atomicMin(&s_klo[1], vn);
    __syncthreads();
    kt0 = min(nk, max(s_klo[0], s_klo[1]) / GL_BK);
  }

  double acc[4][NT][2];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < NT; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

  // fragment base offsets inside a stage
  const int fr = lane >> 2, fk = lane & 3;
  const int a_frag = AKF ? (wm * 32 + fr) * GL_LDK + fk : fk * GL_LDA + wm * 32 + fr;
  const int b_frag = BKF ? (wn * 8 * NT + fr) * GL_LDK + fk : fk * GL_LDB + wn * 8 * NT + fr;
  constexpr int A_I = AKF ? 8 * GL_LDK : 8, A_K = AKF ? 1 : GL_LDA;     // strides per 8-row tile / per k
  constexpr int B_J = BKF ? 8 * GL_LDK : 8, B_K = BKF ? 1 : GL_LDB;

#pragma unroll
  for (int s = 0; s < GL_STAGES - 1; ++s) {
    if (kt0 + s < nk) issue(kt0 + s, s);
    asm volatile("cp.async.commit_group;\n" ::);
  }
  for (int kt = kt0; kt < nk; ++kt) {
    asm volatile("cp.async.wait_group %0;\n" ::"n"(GL_STAGES - 2));
    __syncthreads();                                 // stage kt has landed for everyone; stage kt-1 is free again
    {
      const int nxt = kt + GL_STAGES - 1;
      if (nxt < nk) issue(nxt, (nxt - kt0) % GL_STAGES);
      asm volatile("cp.async.commit_group;\n" ::);
    }
    const int stage = (kt - kt0) % GL_STAGES;
    const double *as = As + stage * GL_A_ELEMS + a_frag, *bs = Bs + stage * GL_B_ELEMS + b_frag;
#pragma unroll
    for (int kk = 0; kk < GL_BK; kk += 4) {
      double af[4], bf[NT];
#pragma unroll
      for (int i = 0; i < 4; ++i) af[i] = as[kk * A_K + i * A_I];
#pragma unroll
      for (int j = 0; j < NT; ++j) bf[j] = bs[kk * B_K + j * B_J];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < NT; ++j) dmma8x8x4(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
    }
  }
  asm volatile("cp.async.wait_group 0;\n" ::);
  // epilogue: lane (fr, fk) holds C[row fr][cols 2 fk, 2 fk + 1] of every 8x8 tile; the offset-table entries of the
  // lane's rows and columns are fetched together up front (one latency instead of one per tile)
  int cmo[4], cno[NT][2];
#pragma unroll
  for (int i = 0; i < 4; ++i) { const int m = m0 + wm * 32 + i * 8 + fr; cmo[i] = (m < d.M) ? d.cm[m] : -1; }
#pragma unroll
  for (int j = 0; j < NT; ++j) {
    const int n = n0 + wn * 8 * NT + j * 8 + 2 * fk;
    cno[j][0] = (n < d.N) ? d.cn[n] : -1;
    cno[j][1] = (n + 1 < d.N) ? d.cn[n + 1] : -1;
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    if (cmo[i] < 0) continue;
#pragma unroll
    for (int j = 0; j < NT; ++j) {
      if (cno[j][0] < 0) continue;
      double v0 = alpha * acc[i][j][0], v1 = alpha * acc[i][j][1];
      if (cvec) {                                    // the two columns are adjacent and 16-byte aligned in C
        double2 *cp = reinterpret_cast<double2 *>(Cb + cmo[i] + cno[j][0]);
        if (beta != 0.0) { const double2 o = *cp; v0 += beta * o.x; v1 += beta * o.y; }
        *cp = make_double2(v0, v1);
      } else {
        double *cp = Cb + cmo[i] + cno[j][0];
        if (beta != 0.0) v0 += beta * (*cp);
        *cp = v0;
        if (cno[j][1] >= 0) {
          double *cq = Cb + cmo[i] + cno[j][1];
          if (beta != 0.0) v1 += beta * (*cq);
          *cq = v1;
        }
      }
    }
  }
}

void be_gett(const GettDesc &d, Operand A, Operand B, Operand C, double alpha, double beta, int W, int NB) {
  const GettVariant v = gett_variant(d, A, B, C, W, NB);
  if (v.kernel == GETT_NONE) return;
  LaunchScope scope(KC_GETT, 2.0 * d.M * d.N * d.K * (double)W * NB * d.work);
  if (v.kernel == GETT_LARGE) {
    const int tn = (d.N + GL_BN - 1) / GL_BN;
    const int bm = v.tile_m;
    const bool half = bm == 64;
    dim3 grid(((d.M + bm - 1) / bm) * tn, NB, W);
    const bool akf = v.akf != 0, bkf = v.bkf != 0;
    const size_t smem = gl_smem(bm, akf, bkf);
    auto go = [&](auto kern) {
      ensure_smem(kern, smem);
      kern<<<grid, GL_THREADS, smem, g_stream>>>(d, A, B, C, alpha, beta, v.avec, v.bvec, v.cvec);
    };
    if (half) {
      if (akf && bkf) go(gett_large_kernel<true, true, 2>);
      else if (akf) go(gett_large_kernel<true, false, 2>);
      else if (bkf) go(gett_large_kernel<false, true, 2>);
      else go(gett_large_kernel<false, false, 2>);
    } else {
      if (akf && bkf) go(gett_large_kernel<true, true, 4>);
      else if (akf) go(gett_large_kernel<true, false, 4>);
      else if (bkf) go(gett_large_kernel<false, true, 4>);
      else go(gett_large_kernel<false, false, 4>);
    }
    post_launch();
    return;
  }
  auto launch = [&](auto kern, int BM, int BN) {
    int tiles = ((d.M + BM - 1) / BM) * ((d.N + BN - 1) / BN);
    dim3 grid(tiles, NB, W);
    kern<<<grid, GETT_THREADS, 0, g_stream>>>(d, A, B, C, alpha, beta);
    post_launch();
  };
  if (v.tile_m == 64 && v.tile_n == 64) launch(gett_kernel<4, 4>, 64, 64);
  else if (v.tile_m == 64) launch(gett_kernel<4, 1>, 64, 16);
  else if (v.tile_n == 64) launch(gett_kernel<1, 4>, 64 / 4, 64);
  else launch(gett_kernel<2, 2>, 32, 32);
}

// =====================================================================================================
// dot
// =====================================================================================================
// K is split over blockIdx.y (the NNN traces contract 262 k elements per walker); the partial sums are combined in a
// fixed order by a second tiny kernel, so the result does not depend on scheduling.
__global__ void dot_kernel(int K, int kchunk, const int32_t *ak, const int32_t *bk, Operand A, Operand B, double *part) {
  const int w = blockIdx.x, sidx = blockIdx.y;
  const double *Ab = operand_base(A, w, 0);
  const double *Bb = operand_base(B, w, 0);
  __shared__ double red[256];
  double s = 0.0;
  const int k1 = min(K, (sidx + 1) * kchunk);
  for (int k = sidx * kchunk + threadIdx.x; k < k1; k += blockDim.x) s += Ab[ak[k]] * Bb[bk[k]];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int h = blockDim.x / 2; h > 0; h >>= 1) {
    if (threadIdx.x < h) red[threadIdx.x] += red[threadIdx.x + h];
    __syncthreads();
  }
  if (threadIdx.x == 0) part[(long)w * gridDim.y + sidx] = red[0];
}
__global__ void dot_finish_kernel(const double *part, int nsplit, double *out, int W) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= W) return;
  double s = 0.0;
  for (int i = 0; i < nsplit; ++i) s += part[(long)w * nsplit + i];
  out[w] = s;
}
void be_dot(int K, const int32_t *ak, const int32_t *bk, Operand A, Operand B, double *out, int W) {
  LaunchScope scope(KC_DOT, 2.0 * K * W);
  const int nsplit = std::max(1, std::min(32, K / 4096));
  if (nsplit == 1) {
    dot_kernel<<<dim3(W, 1), 256, 0, g_stream>>>(K, K, ak, bk, A, B, out);
    post_launch();
    return;
  }
  double *&part = cx().dot_part;
  size_t &part_cap = cx().dot_part_cap;
  if ((size_t)W * 32 > part_cap) {
    if (part) { CUDA_CHECK(cudaStreamSynchronize(g_stream)); cudaFree(part); }
    part_cap = (size_t)W * 32;
    CUDA_CHECK(cudaMalloc(&part, sizeof(double) * part_cap));
  }
  const int kchunk = (K + nsplit - 1) / nsplit;
  dot_kernel<<<dim3(W, nsplit), 256, 0, g_stream>>>(K, kchunk, ak, bk, A, B, part);
  ++cx().launches;
  dot_finish_kernel<<<(W + 127) / 128, 128, 0, g_stream>>>(part, nsplit, out, W);
  post_launch();
}

// =====================================================================================================
// dense helpers
// =====================================================================================================
__global__ void fill_kernel(double *p, double v, long n) {
  long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  long stride = (long)gridDim.x * blockDim.x;
  for (; i < n; i += stride) p[i] = v;
}
void be_fill(double *p, double v, long n) {
  if (n <= 0) return;
  int blocks = (int)((n + 255) / 256 < 148L * 8 ? (n + 255) / 256 : 148L * 8);
  LaunchScope scope(KC_SMALL, 0.0);
  fill_kernel<<<blocks, 256, 0, g_stream>>>(p, v, n);
  post_launch();
}
__global__ void copy2d_kernel(double *dst, long wd, long ldd, const double *src, long ws, long lds, int rows,
                              int cols) {
  const int w = blockIdx.y;
  long n = (long)rows * cols;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    int r = (int)(i / cols), c = (int)(i % cols);
    dst[w * wd + r * ldd + c] = src[w * ws + r * lds + c];
  }
}
void be_copy2d(double *dst, long wd, long ldd, const double *src, long ws, long lds, int rows, int cols, int W) {
  long n = (long)rows * cols;
  if (n <= 0) return;
  int bx = (int)((n + 255) / 256 < 64 ? (n + 255) / 256 : 64);
  LaunchScope scope(KC_SMALL, 0.0);
  copy2d_kernel<<<dim3(bx, W), 256, 0, g_stream>>>(dst, wd, ldd, src, ws, lds, rows, cols);
  post_launch();
}
__global__ void identity_kernel(double *dst, long wd, int rows, int cols) {
  const int w = blockIdx.y;
  long n = (long)rows * cols;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    int r = (int)(i / cols), c = (int)(i % cols);
    dst[w * wd + i] = (r == c) ? 1.0 : 0.0;
  }
}
void be_set_identity(double *dst, long wd, int rows, int cols, int W) {
  long n = (long)rows * cols;
  int bx = (int)((n + 255) / 256 < 64 ? (n + 255) / 256 : 64);
  LaunchScope scope(KC_SMALL, 0.0);
  identity_kernel<<<dim3(bx, W), 256, 0, g_stream>>>(dst, wd, rows, cols);
  post_launch();
}

// =====================================================================================================
// CAQR panel
// =====================================================================================================
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

constexpr int PQR_THREADS = 256;

__global__ void __launch_bounds__(PQR_THREADS) panel_qr_kernel(PanelArgs a) {
  extern __shared__ double sm[];
  const int it = blockIdx.x, w = blockIdx.y;
  if (a.row_cnt && a.rowtab[(long)it * a.R] >= a.row_cnt[w] * a.row_scale) return;     // all-zero item of this walker
  if (a.stopped && a.stopped[w]) return;                                                // factorisation of this walker already terminated
  const int R = a.R, pw = a.pw, nbw = a.nbw;
  const int skip = (it == 0) ? a.skip0 : 0;
  const int nact = R - skip;
  const int LDP = R + 1;
  double *P = sm;                               // [nbw][LDP] column-major panel
  double *S = P + (size_t)nbw * LDP;            // [nbw][nbw]
  double *T = S + nbw * nbw;                    // [nbw][nbw]
  double *tau = T + nbw * nbw;                  // [nbw]
  double *scal = tau + nbw;                     // [nbw]
  double *beta = scal + nbw;                    // [nbw]
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5, nwarp = PQR_THREADS / 32;
  double *Aw = a.A + (long)w * a.ws;
  const int32_t *rows = a.rowtab + (long)it * R;

  // 1. gather the panel
  for (int e = t; e < nact * pw; e += PQR_THREADS) {
    int r = e / pw, c = e % pw;
    P[c * LDP + r] = Aw[(long)rows[skip + r] * a.lda + a.col0 + c];
  }
  __syncthreads();

  // 2. Householder columns (LAPACK dgeqr2 / dlarfg conventions)
  for (int j = 0; j < pw; ++j) {
    double tj = 0.0, sj = 0.0, bj = 0.0;
    if (j < nact) {
      const double *x = P + j * LDP;
      double part = 0.0;
      for (int r = j + 1 + lane; r < nact; r += 32) part += x[r] * x[r];
      double xn2 = warp_sum(part);
      double alpha = x[j];
      bj = alpha;
      if (xn2 > 0.0) {
        double nrm = sqrt(alpha * alpha + xn2);
        bj = (alpha >= 0.0) ? -nrm : nrm;
        tj = (bj - alpha) / bj;
        sj = 1.0 / (alpha - bj);
      }
      if (tj != 0.0) {
        for (int c = j + 1 + warp; c < pw; c += nwarp) {
          double *y = P + c * LDP;
          double pr = 0.0;
          for (int r = j + 1 + lane; r < nact; r += 32) pr += x[r] * y[r];
          double wv = warp_sum(pr) * sj + y[j];
          double f = tj * wv;
          for (int r = j + 1 + lane; r < nact; r += 32) y[r] -= f * sj * x[r];
          if (lane == 0) y[j] -= f;
        }
      }
    }
    if (t == 0) { tau[j] = tj; scal[j] = sj; beta[j] = bj; }
    __syncthreads();
  }

  // 3. S = R-part extraction happens at write-back; build V in place: column c rows > c scaled, keep the
  //    R entries (rows <= c) in registers? They live in P rows <= c of column c: copy them to S scratch first.
  //    Rpart[r][c] (r <= c < pw) is stashed in T temporarily (nbw x nbw), then T is rebuilt after S.
  for (int e = t; e < nbw * nbw; e += PQR_THREADS) {
    int r = e / nbw, c = e % nbw;
    double v = 0.0;
    if (c < pw && r <= c && r < nact) v = (r == c) ? beta[c] : P[c * LDP + r];
    T[e] = v;                                   // T holds Rpart for now
  }
  __syncthreads();
  // write R part + zeros to A now (panel columns, all active rows)
  for (int e = t; e < nact * pw; e += PQR_THREADS) {
    int r = e / pw, c = e % pw;
    double v = (r < nbw && r <= c) ? T[r * nbw + c] : 0.0;
    Aw[(long)rows[skip + r] * a.lda + a.col0 + c] = v;
  }
  __syncthreads();
  // V in place
  for (int e = t; e < nact * pw; e += PQR_THREADS) {
    int c = e / nact, r = e % nact;
    double v;
    if (r < c) v = 0.0;
    else if (r == c) v = 1.0;
    else v = P[c * LDP + r] * scal[c];
    P[c * LDP + r] = v;
  }
  __syncthreads();
  // S = V^T V (strict upper part)
  for (int pidx = warp; pidx < pw * pw; pidx += nwarp) {
    int ca = pidx / pw, cb = pidx % pw;
    if (ca >= cb) continue;
    const double *x = P + ca * LDP, *y = P + cb * LDP;
    double pr = 0.0;
    for (int r = cb + lane; r < nact; r += 32) pr += x[r] * y[r];
    pr = warp_sum(pr);
    if (lane == 0) S[ca * nbw + cb] = pr;
  }
  __syncthreads();
  // T (forward, columnwise): T[j][j] = tau_j; T[0:j, j] = -tau_j * T[0:j,0:j] * S[0:j, j]
  for (int e = t; e < nbw * nbw; e += PQR_THREADS) T[e] = 0.0;
  __syncthreads();
  if (warp == 0) {
    for (int j = 0; j < pw; ++j) {
      double tj = tau[j];
      double v = 0.0;
      if (lane < j) {
        for (int b2 = lane; b2 < j; ++b2) v += T[lane * nbw + b2] * S[b2 * nbw + j];
        v *= -tj;
      }
      __syncwarp();
      if (lane < j) T[lane * nbw + j] = v;
      if (lane == j) T[j * nbw + j] = tj;
      __syncwarp();
    }
  }
  __syncthreads();
  // 4. emit V and T
  double *Vo = a.Vw + ((long)w * a.NI + it) * (long)R * nbw;
  double *To = a.Tw + ((long)w * a.NI + it) * (long)nbw * nbw;
  for (int e = t; e < skip * nbw; e += PQR_THREADS) Vo[e] = 0.0;
  for (int e = t; e < nact * nbw; e += PQR_THREADS) {
    int r = e / nbw, c = e % nbw;
    Vo[(long)(skip + r) * nbw + c] = (c < pw) ? P[c * LDP + r] : 0.0;
  }
  for (int e = t; e < nbw * nbw; e += PQR_THREADS) To[e] = T[e];
}

static size_t panel_smem_bytes(int R, int nbw) {
  return ((size_t)nbw * (R + 1) + 2 * (size_t)nbw * nbw + 3 * nbw) * sizeof(double);
}

// Register-resident variant: warp w owns the CPW = NBW/8 panel columns w, w+8, ... (cyclic, so the work stays
// balanced as the factorisation advances), lane l owns rows l, l+32, ... (RPL of them): every Householder update is
// FMA work out of registers. All reflectors live in shared memory (vcols, column-major V) and are published with a
// per-column ready flag, so there is no block barrier in the column loop: the owner of column j+1 applies
// reflector j to that column first, builds and publishes reflector j+1, and only then catches up on its other
// columns, while every other warp runs at its own pace. A warp reduces the dot products of all its columns
// together (interleaved shuffles). S = V^T V falls out of the same dot products; T is emitted for the trailing
// update (C - V T^T (V^T C)), so V T^T is never formed.
// Optional phase clocks of CTA (0,0) (development aid: build with -DPEPS_KERNEL_CLOCKS, run with PEPS_PANEL_CLK=n)
#ifdef PEPS_KERNEL_CLOCKS
__device__ long long g_panel_clk[8 + 32 * 8];
#define PANEL_CLK(i) do { if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) g_panel_clk[i] = clock64(); } while (0)
#define COL_CLK(j, k) do { if (blockIdx.x == 0 && blockIdx.y == 0 && lane == 0) g_panel_clk[8 + (j) * 8 + (k)] = clock64(); } while (0)
#else
#define PANEL_CLK(i) do { } while (0)
#define COL_CLK(j, k) do { } while (0)
#endif
template <int NBW, int RPL, int MINB>
__global__ void __launch_bounds__(PQR_THREADS, MINB) panel_qr_reg_kernel(PanelArgs a) {
  extern __shared__ double sm[];
  PANEL_CLK(0);
  constexpr int CPW = NBW / 8;
  constexpr int LDT = NBW + 1, LDSS = NBW + 1;
  constexpr int RP = RPL * 32;
  const int it = blockIdx.x, w = blockIdx.y;
  if (a.row_cnt && a.rowtab[(long)it * a.R] >= a.row_cnt[w] * a.row_scale) return;     // all-zero item of this walker
  if (a.stopped && a.stopped[w]) return;                                                // factorisation of this walker already terminated
  const int R = a.R, pw = a.pw, nbw = a.nbw;
  const int skip = (it == 0) ? a.skip0 : 0;
  const int nact = R - skip;
  double *vcols = sm;                      // [NBW][RP]
  double *S = vcols + (size_t)NBW * RP;    // [NBW][LDSS]
  double *Tt = S + NBW * LDSS;             // [NBW][LDT]   T[a][b]
  volatile double *tau_s = Tt + NBW * LDT; // [NBW]
  double *Rd = const_cast<double *>(tau_s) + NBW;   // [NBW]
  long *roff = reinterpret_cast<long *>(Rd + NBW);  // [RP] global offset of active row r
  volatile int *ready = reinterpret_cast<volatile int *>(roff + RP);   // [NBW]
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  double *Aw = a.A + (long)w * a.ws;
  const int32_t *rows = a.rowtab + (long)it * R;
  for (int r = t; r < RP; r += PQR_THREADS) roff[r] = (r < nact) ? (long)rows[skip + r] * a.lda + a.col0 : 0;
  for (int e = t; e < NBW * LDSS; e += PQR_THREADS) S[e] = 0.0;
  for (int e = t; e < NBW * LDT; e += PQR_THREADS) Tt[e] = 0.0;
  if (t < NBW) { tau_s[t] = 0.0; Rd[t] = 0.0; ready[t] = 0; }
  __syncthreads();

  // The panel travels global <-> registers through a swizzled staging tile (the reflector buffer, idle at both ends
  // of the kernel): global accesses are whole panel rows (coalesced), the register tile picks its strided elements
  // out of shared memory without bank conflicts. Element (r, c) sits at r * NBW + (c ^ (r % NBW)).
  double *stage = vcols;
  constexpr int RPI = 32 / NBW;             // panel rows per warp-wide access
  for (int r0 = warp * RPI; r0 < RP; r0 += 8 * RPI) {
    const int r = r0 + lane / NBW, c = lane % NBW;
    double *dstp = stage + (size_t)r * NBW + (c ^ (r & (NBW - 1)));
    if (r < nact && c < pw) {
      const unsigned saddr = (unsigned)__cvta_generic_to_shared(dstp);
      asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(saddr), "l"(Aw + roff[r] + c));
    } else {
      *dstp = 0.0;
    }
  }
  asm volatile("cp.async.commit_group;\n" ::);
  asm volatile("cp.async.wait_group 0;\n" ::);
  __syncthreads();
  double P[CPW][RPL];
#pragma unroll
  for (int i = 0; i < RPL; ++i) {
    const int r = lane + 32 * i;
#pragma unroll
    for (int cc = 0; cc < CPW; ++cc) P[cc][i] = stage[(size_t)r * NBW + ((warp + 8 * cc) ^ (r & (NBW - 1)))];
  }
  __syncthreads();                          // the tile is about to be overwritten by reflector 0

  // builds reflector j from column j (owned by this warp as LOCAL column CJ, a compile-time index: a run-time index
  // into the register tile turns every element access into a branch tree on the critical path), publishes it;
  // P keeps [R | 1 | v]
  auto build = [&](int j, auto cj_c) {
    constexpr int CJ = decltype(cj_c)::value;
    double *vb = vcols + (size_t)j * RP;
    double n0 = 0.0, n1 = 0.0, n2 = 0.0, n3 = 0.0, alpha = 0.0;
#pragma unroll
    for (int i = 0; i < RPL; ++i) {        // selects only (rows >= nact hold zeros): a branch per element costs ~60 cycles
      const double v = P[CJ][i];
      const int r = lane + 32 * i;
      alpha = (r == j) ? v : alpha;
      const double vm = (r > j) ? v : 0.0;
      if ((i & 3) == 0) n0 = fma(vm, vm, n0); else if ((i & 3) == 1) n1 = fma(vm, vm, n1);
      else if ((i & 3) == 2) n2 = fma(vm, vm, n2); else n3 = fma(vm, vm, n3);
    }
    double xn2 = (n0 + n1) + (n2 + n3);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {     // norm and the diagonal entry travel together
      xn2 += __shfl_xor_sync(0xffffffffu, xn2, o);
      alpha += __shfl_xor_sync(0xffffffffu, alpha, o);
    }
    COL_CLK(j, 3);
    double bj = alpha, tj = 0.0, sj = 0.0;
    if (xn2 > 0.0) {
      const double s2 = alpha * alpha + xn2;
      const double rs = rsqrt(s2);
      const double nrm = s2 * rs;
      bj = (alpha >= 0.0) ? -nrm : nrm;
      const double inv_b = (alpha >= 0.0) ? -rs : rs;
      tj = 1.0 - alpha * inv_b;            // (beta - alpha) / beta
      sj = 1.0 / (alpha - bj);
    }
    COL_CLK(j, 4);
#pragma unroll
    for (int i = 0; i < RPL; ++i) {
      const int r = lane + 32 * i;
      const double pm = P[CJ][i] * sj;
      const double v = (r > j) ? pm : ((r == j) ? 1.0 : 0.0);
      vb[r] = v;
      P[CJ][i] = (r >= j) ? v : P[CJ][i];
    }
    if (lane == 0) { tau_s[j] = tj; Rd[j] = bj; }
    COL_CLK(j, 5);
    __syncwarp();
    __threadfence_block();
    if (lane == 0) ready[j] = 1;
  };
  // look-ahead of the owner of column jn: apply reflector j (v, tj) to that column alone, then build reflector jn
  auto lookahead = [&](int jn, const double (&v)[RPL], double tj, auto cn_c) {
    constexpr int CN = decltype(cn_c)::value;
    double d0 = 0.0, d1 = 0.0, d2 = 0.0, d3 = 0.0;
#pragma unroll
    for (int i = 0; i < RPL; ++i) {
      const double q = v[i] * P[CN][i];
      if ((i & 3) == 0) d0 += q; else if ((i & 3) == 1) d1 += q; else if ((i & 3) == 2) d2 += q; else d3 += q;
    }
    const double f = tj * warp_sum((d0 + d1) + (d2 + d3));
    COL_CLK(jn, 1);
#pragma unroll
    for (int i = 0; i < RPL; ++i) P[CN][i] -= f * v[i];
    COL_CLK(jn, 2);
    build(jn, cn_c);
    COL_CLK(jn, 6);
  };

  PANEL_CLK(1);
  if (warp == 0 && pw > 0) build(0, std::integral_constant<int, 0>{});
  for (int j = 0; j < pw; ++j) {
    while (ready[j] == 0) __nanosleep(40);
    __threadfence_block();
    const double *vb = vcols + (size_t)j * RP;
    const double tj = tau_s[j];
    double v[RPL];
#pragma unroll
    for (int i = 0; i < RPL; ++i) v[i] = vb[lane + 32 * i];
    const int jn = j + 1;
    const bool own_next = (jn < pw) && (warp == (jn & 7));
    if (own_next) {                         // publish reflector j+1 early; the other columns catch up below
      COL_CLK(jn, 7);
      switch (jn >> 3) {
        case 0: lookahead(jn, v, tj, std::integral_constant<int, 0>{}); break;
        case 1: if constexpr (CPW > 1) lookahead(jn, v, tj, std::integral_constant<int, 1>{}); break;
        case 2: if constexpr (CPW > 2) lookahead(jn, v, tj, std::integral_constant<int, 2>{}); break;
        default: if constexpr (CPW > 3) lookahead(jn, v, tj, std::integral_constant<int, 3>{}); break;
      }
    }
    // all remaining columns of this warp together: dots, one interleaved reduction, updates / S entries
    double d[CPW][2];
#pragma unroll
    for (int cc = 0; cc < CPW; ++cc) d[cc][0] = d[cc][1] = 0.0;
#pragma unroll
    for (int i = 0; i < RPL; ++i) {
#pragma unroll
      for (int cc = 0; cc < CPW; ++cc) d[cc][i & 1] += v[i] * P[cc][i];
    }
    double dot[CPW];
#pragma unroll
    for (int cc = 0; cc < CPW; ++cc) dot[cc] = d[cc][0] + d[cc][1];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
      for (int cc = 0; cc < CPW; ++cc) dot[cc] += __shfl_xor_sync(0xffffffffu, dot[cc], o);
    }
#pragma unroll
    for (int cc = 0; cc < CPW; ++cc) {
      const int c = warp + 8 * cc;
      if (c >= pw || c == j || (own_next && c == jn)) continue;
      if (c > j) {
        const double f = tj * dot[cc];
        if (f != 0.0) {
#pragma unroll
          for (int i = 0; i < RPL; ++i) P[cc][i] -= f * v[i];
        }
      } else if (lane == 0) {
        S[c * LDSS + j] = dot[cc];
      }
    }
  }
  PANEL_CLK(2);
  __syncthreads();
  PANEL_CLK(3);

  // T = (strict_upper(S) + diag(1/tau))^-1, built block-recursively so that the whole CTA works on it:
  //   8x8 diagonal blocks by the column recurrence T[a][j] = -tau_j sum_{a<=b<j} T[a][b] S[b][j] (one lane per row),
  //   then T12 = -T11 (S12 T22) for block sizes 8, 16, ... (X = S12 T22 staged in the dead reflector buffer).
  {
    if (warp < NBW / 8 && lane < 8) {
      const int base = warp * 8;
      double trow[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const double tj = (base + j < pw) ? tau_s[base + j] : 0.0;
        double acc = 0.0;
#pragma unroll
        for (int b2 = 0; b2 < j; ++b2) acc += trow[b2] * S[(base + b2) * LDSS + base + j];   // trow[b2] = 0 for b2 < lane
        trow[j] = (j == lane) ? tj : ((j > lane) ? -tj * acc : 0.0);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) Tt[(base + lane) * LDT + base + j] = trow[j];
    }
    __syncthreads();
    double *X = vcols;                     // [NBW][LDT] scratch
#pragma unroll 1
    for (int bs = 8; bs < NBW; bs *= 2) {
      const int nel = (NBW / (2 * bs)) * bs * bs;
      for (int e = t; e < nel; e += PQR_THREADS) {
        const int m = e / (bs * bs), aa = (e / bs) % bs, c = e % bs, base = m * 2 * bs;
        const double *Sr = S + (base + aa) * LDSS + base + bs, *Tc = Tt + (base + bs) * LDT + base + bs + c;
        double x0 = 0.0, x1 = 0.0;
        int k = 0;
        for (; k + 1 <= c; k += 2) { x0 += Sr[k] * Tc[k * LDT]; x1 += Sr[k + 1] * Tc[(k + 1) * LDT]; }
        if (k <= c) x0 += Sr[k] * Tc[k * LDT];
        X[(base + aa) * LDT + c] = x0 + x1;
      }
      __syncthreads();
      for (int e = t; e < nel; e += PQR_THREADS) {
        const int m = e / (bs * bs), aa = (e / bs) % bs, c = e % bs, base = m * 2 * bs;
        const double *Tr = Tt + (base + aa) * LDT + base, *Xc = X + base * LDT + c;
        double x0 = 0.0, x1 = 0.0;
        int k = aa;
        for (; k + 1 < bs; k += 2) { x0 += Tr[k] * Xc[k * LDT]; x1 += Tr[k + 1] * Xc[(k + 1) * LDT]; }
        if (k < bs) x0 += Tr[k] * Xc[k * LDT];
        Tt[(base + aa) * LDT + base + bs + c] = -(x0 + x1);
      }
      __syncthreads();
    }
  }
  PANEL_CLK(4);
  // emit R (in place, zeros below it) and V through the staging tile
#pragma unroll
  for (int i = 0; i < RPL; ++i) {
    const int r = lane + 32 * i;
#pragma unroll
    for (int cc = 0; cc < CPW; ++cc) stage[(size_t)r * NBW + ((warp + 8 * cc) ^ (r & (NBW - 1)))] = P[cc][i];
  }
  __syncthreads();
  double *Vo = a.Vw + ((long)w * a.NI + it) * (long)R * nbw;
  for (int e = t; e < skip * nbw; e += PQR_THREADS) Vo[e] = 0.0;
  for (int e = t; e < nact * NBW; e += PQR_THREADS) {
    const int r = e / NBW, c = e % NBW;
    const double pv = stage[(size_t)r * NBW + (c ^ (r & (NBW - 1)))];
    Vo[(long)(skip + r) * nbw + c] = (c < pw && r >= c) ? pv : 0.0;
    if (c < pw) Aw[roff[r] + c] = (r < c) ? pv : ((r == c) ? Rd[c] : 0.0);
  }
  double *To = a.Tw + ((long)w * a.NI + it) * (long)nbw * nbw;
  for (int e = t; e < NBW * NBW; e += PQR_THREADS) To[e] = Tt[(e / NBW) * LDT + (e % NBW)];
  PANEL_CLK(5);
}

template <int NBW, int RPL>
static size_t panel_reg_smem_bytes(int nact_max) {
  (void)nact_max;
  return ((size_t)(NBW + 1) * RPL * 32 + 2 * (size_t)NBW * (NBW + 1) + 2 * NBW) * sizeof(double) + NBW * sizeof(int) + 16;
}

void be_panel_qr(const PanelArgs &a) {
  LaunchScope scope(KC_PANEL, 4.0 * a.R * a.pw * a.pw * (double)a.NI * a.W);
  auto launch_reg = [&](auto kern, size_t smem) {
    ensure_smem(kern, smem);
    kern<<<dim3(a.NI, a.W), PQR_THREADS, smem, g_stream>>>(a);
  };
  const int R = a.R;
  // panels of <= 256 rows: 64 KB tile and <= 128 registers, two CTAs share an SM and hide each other's reflector chain
  // panels of <= 128 rows (PEPS_QR_RB=128): 16 panel values per thread, up to four CTAs per SM
  if (a.nbw == 32 && R <= 128) launch_reg(panel_qr_reg_kernel<32, 4, 4>, panel_reg_smem_bytes<32, 4>(R));
  else if (a.nbw == 32 && R <= 256) launch_reg(panel_qr_reg_kernel<32, 8, 2>, panel_reg_smem_bytes<32, 8>(R));
  else if (a.nbw == 32 && R <= 512) launch_reg(panel_qr_reg_kernel<32, 16, 1>, panel_reg_smem_bytes<32, 16>(R));
  else if (a.nbw == 32 && R <= 576) launch_reg(panel_qr_reg_kernel<32, 18, 1>, panel_reg_smem_bytes<32, 18>(R));
  else if (a.nbw == 16 && R <= 512) launch_reg(panel_qr_reg_kernel<16, 16, 1>, panel_reg_smem_bytes<16, 16>(R));
  else if (a.nbw == 16 && R <= 1184) launch_reg(panel_qr_reg_kernel<16, 37, 1>, panel_reg_smem_bytes<16, 37>(R));
  else {
    size_t smem = panel_smem_bytes(a.R, a.nbw);
    ensure_smem(panel_qr_kernel, smem);
    panel_qr_kernel<<<dim3(a.NI, a.W), PQR_THREADS, smem, g_stream>>>(a);
  }
  post_launch();
#ifdef PEPS_KERNEL_CLOCKS
  static const int dbg = std::getenv("PEPS_PANEL_CLK") ? std::atoi(std::getenv("PEPS_PANEL_CLK")) : 0;
  static int shown = 0;
  if (dbg && a.nbw == 32 && R > 256 && R <= 512 && shown < dbg) {
    ++shown;
    long long h[8 + 32 * 8];
    CUDA_CHECK(cudaStreamSynchronize(g_stream));
    CUDA_CHECK(cudaMemcpyFromSymbol(h, g_panel_clk, sizeof(h)));
    if (shown == 1)
      for (int j = 2; j < 32; ++j) {
        const long long *c = h + 8 + j * 8, *pc = h + 8 + (j - 1) * 8;
        fprintf(stderr, "[col %2d] since prev publish: vload=%lld dot+sum=%lld upd=%lld norm=%lld rsq/div=%lld scale+sts=%lld fence=%lld | period=%lld\n",
                j, c[7] - pc[6], c[1] - c[7], c[2] - c[1], c[3] - c[2], c[4] - c[3], c[5] - c[4], c[6] - c[5], c[6] - pc[6]);
      }
    fprintf(stderr, "[panel clk] R=%d pw=%d NI=%d W=%d load=%lld cols=%lld wait=%lld T=%lld emit=%lld\n", R, a.pw, a.NI, a.W,
            h[1] - h[0], h[2] - h[1], h[3] - h[2], h[4] - h[3], h[5] - h[4]);
  }
#endif
}

// Fused trailing update of one CAQR panel step (see backend.h ApplyArgs): the C tile (R rows x NBW columns) stays
// in shared memory; W = V^T C is accumulated on the DMMA pipe with the row range split over the 8 warps, then
// C - V T^T W is formed tile-row by tile-row and written back. V fragments are read straight from L2.
// Each warp brings in its own 64-row slice with one bulk copy (TMA) per row, completion counted on the warp's own
// mbarrier: a warp starts its share of V^T C as soon as ITS rows have landed, there is no block-wide wait on the load.
#ifdef PEPS_KERNEL_CLOCKS
__device__ long long g_apply_clk[8];
#define APPLY_CLK(i) do { if (blockIdx.x == gridDim.x - 1 && blockIdx.y == gridDim.y - 1 && blockIdx.z == gridDim.z - 1 && threadIdx.x == 0) g_apply_clk[i] = clock64(); } while (0)   // the LAST CTA: warm caches
#else
#define APPLY_CLK(i) do { } while (0)
#endif
__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity) {
  asm volatile(
      "{\n.reg .pred p;\nWAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\nbra WAIT_%=;\nDONE_%=:\n}\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, unsigned bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                   (unsigned)__cvta_generic_to_shared(dst)), "l"(src), "r"(bytes), "r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}

__device__ __forceinline__ void bulk_s2g(void *dst, const void *src, unsigned bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;\n" ::"l"(dst), "r"((unsigned)__cvta_generic_to_shared(src)),
               "r"(bytes) : "memory");
}

__device__ __forceinline__ void tma_load_3d(void *dst, const void *tmap, int x, int y, int z, uint64_t *bar) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];\n" ::"r"(
                   (unsigned)__cvta_generic_to_shared(dst)), "l"(tmap), "r"(x), "r"(y), "r"(z), "r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}

// TM = true: the rows of an item are contiguous and `tm` describes the matrix: each warp fetches its row slice with
// four TMA tile loads (8 columns x slice rows each) into a chunked tile layout [column chunk][row][8], which the DMMA
// fragment loads read without bank conflicts and without padding; no row-offset table at all.
template <int NBW, int MINB, bool TM>
__global__ void __launch_bounds__(256, MINB) apply_reflector_kernel(ApplyArgs a, const __grid_constant__ TileMap tm) {
  extern __shared__ __align__(16) double sm[];
  APPLY_CLK(0);
  constexpr int TN = NBW, MT = NBW / 8, NT = NBW / 8, LDC = TN + 4, LDW = TN + 4, NTILE = MT * NT;
  const int ct = blockIdx.x, it = blockIdx.y, w = blockIdx.z;
  if (a.row_cnt && a.rowtab[(long)it * a.R] >= a.row_cnt[w] * a.row_scale) return;     // all-zero item of this walker
  if (a.stopped && a.stopped[w]) return;
  const int R = a.R, R8 = (R + 7) & ~7, nbw = a.nbw;
  double *Cs = sm;                               // [R8][LDC], or [NBW/8][R8][8] with tile descriptors
  auto csi = [&](int r, int c) -> size_t {
    if constexpr (TM) return ((size_t)(c >> 3) * R8 + r) * 8 + (c & 7);
    else return (size_t)r * LDC + c;
  };
  double *part = Cs + (size_t)R8 * LDC;          // [4][NTILE][64]
  double *Wsm = part + 4 * NTILE * 64;           // [NBW][LDW] = -(V^T C)
  long *roff = reinterpret_cast<long *>(Wsm + NBW * LDW);   // [R8]
  uint64_t *bars = reinterpret_cast<uint64_t *>(roff + R8); // [8] one per warp
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  double *Aw = a.A + (long)w * a.ws;
  const int32_t *rows = a.rowtab + (long)it * R;
  const double *V = a.Vw + ((long)w * a.NI + it) * (long)R * nbw;
  const double *Tg = a.Tw + ((long)w * a.NI + it) * (long)nbw * nbw;
  const int cbase = a.col1 + ct * TN;
  const int ncols = min(TN, a.ntrail - ct * TN);
  const int kslice = ((R8 / 8) + 7) & ~7;        // rows per warp (whole 8-row tiles)
  const int k0 = min(R8, warp * kslice), k1 = min(R8, k0 + kslice);
  // 16-byte granularity everywhere? (bulk copies and paired stores need it; the 8-byte path below covers the rest)
  const bool wide = (((a.lda | cbase | ncols) & 1) == 0) && ((a.ws & 1) == 0) && ((reinterpret_cast<uintptr_t>(a.A) & 15) == 0);

  double tpre[(NBW * NBW + 255) / 256];          // T, fetched now, staged in shared memory after V^T C
#pragma unroll
  for (int u = 0; u < (NBW * NBW + 255) / 256; ++u) tpre[u] = (t + u * 256 < NBW * NBW) ? __ldg(Tg + t + u * 256) : 0.0;

  // 0. C tile -> shared memory, each warp its own row slice
  if (lane == 0) mbar_init(&bars[warp], 1);
  if constexpr (!TM) { for (int r = k0 + lane; r < k1; r += 32) roff[r] = (r < R) ? (long)rows[r] * a.lda + cbase : -1; }
  APPLY_CLK(6);
  asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  __syncwarp();
  APPLY_CLK(7);
  if constexpr (TM) {
    if (lane == 0 && k1 > k0) {
      mbar_expect_tx(&bars[warp], (unsigned)((k1 - k0) * NBW * 8));
#pragma unroll
      for (int j = 0; j < NBW / 8; ++j)
        tma_load_3d(Cs + ((size_t)j * R8 + k0) * 8, &tm, cbase + 8 * j, a.row0 + it * R + k0, w, &bars[warp]);
    }
    APPLY_CLK(1);
    if (k1 > k0) mbar_wait(&bars[warp], 0);
  } else if (wide) {
    const int nvalid = max(0, min(k1, R) - k0);
    if (lane == 0) mbar_expect_tx(&bars[warp], (unsigned)(nvalid * ncols * 8));
    __syncwarp();
    for (int r = k0 + lane; r < k1; r += 32) {
      double *dstp = Cs + (size_t)r * LDC;
      if (r < R) {
        bulk_g2s(dstp, Aw + roff[r], (unsigned)(ncols * 8), &bars[warp]);
        for (int c = ncols; c < LDC; ++c) dstp[c] = 0.0;
      } else {
        for (int c = 0; c < LDC; ++c) dstp[c] = 0.0;
      }
    }
    APPLY_CLK(1);
    mbar_wait(&bars[warp], 0);
  } else {
    for (int r = k0; r < k1; ++r) {
      const long o = roff[r];
      double *dstp = Cs + (size_t)r * LDC + lane;
      if (lane < TN) {
        if (o >= 0 && lane < ncols) {
          const unsigned saddr = (unsigned)__cvta_generic_to_shared(dstp);
          asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(saddr), "l"(Aw + o + lane));
        } else {
          *dstp = 0.0;
        }
      }
      if (lane < LDC - TN) Cs[(size_t)r * LDC + TN + lane] = 0.0;
    }
    asm volatile("cp.async.commit_group;\n" ::);
    APPLY_CLK(1);
    asm volatile("cp.async.wait_group 0;\n" ::);
  }
  __syncwarp();
  APPLY_CLK(2);

  double *Wraw = part;                        // [NBW][LDW] raw W = V^T C (inside the partial-sum scratch)
  {
    // A. partial W = V^T C over this warp's row slice
    double acc[MT][NT][2];
#pragma unroll
    for (int i = 0; i < MT; ++i)
#pragma unroll
      for (int j = 0; j < NT; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
#pragma unroll 4
    for (int k = k0; k < k1; k += 4) {      // unrolled so that several k-steps of V fragments are in flight from L2
      const int kr = k + (lane & 3);
      double af[MT], bf[NT];
#pragma unroll
      for (int i = 0; i < MT; ++i) af[i] = (kr < R) ? __ldg(V + (long)kr * nbw + i * 8 + (lane >> 2)) : 0.0;
#pragma unroll
      for (int j = 0; j < NT; ++j) bf[j] = Cs[csi(kr, j * 8 + (lane >> 2))];
#pragma unroll
      for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < NT; ++j) dmma8x8x4(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
    }
    APPLY_CLK(3);
    const int eo = (lane >> 2) * 8 + 2 * (lane & 3);
    if (warp >= 4) {
#pragma unroll
      for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < NT; ++j) {
          double *g = part + ((size_t)(warp - 4) * NTILE + i * NT + j) * 64 + eo;
          g[0] = acc[i][j][0]; g[1] = acc[i][j][1];
        }
    }
    __syncthreads();
    if (warp < 4) {
#pragma unroll
      for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < NT; ++j) {
          double *g = part + ((size_t)warp * NTILE + i * NT + j) * 64 + eo;
          acc[i][j][0] += g[0]; acc[i][j][1] += g[1];
        }
      __syncwarp();
#pragma unroll
      for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < NT; ++j) {
          double *g = part + ((size_t)warp * NTILE + i * NT + j) * 64 + eo;
          g[0] = acc[i][j][0]; g[1] = acc[i][j][1];
        }
    }
    __syncthreads();
    double wv[(NTILE * 64 + 255) / 256];
#pragma unroll
    for (int u = 0; u < (NTILE * 64 + 255) / 256; ++u) {
      const int e = t + u * 256;
      double v = 0.0;
      if (e < NTILE * 64) {
#pragma unroll
        for (int g = 0; g < 4; ++g) v += part[((size_t)g * NTILE + (e >> 6)) * 64 + (e & 63)];
      }
      wv[u] = v;
    }
    __syncthreads();
#pragma unroll
    for (int u = 0; u < (NTILE * 64 + 255) / 256; ++u) {
      const int e = t + u * 256;
      if (e < NTILE * 64) {
        const int tile = e >> 6, rr = (e >> 3) & 7, cc = e & 7;
        Wraw[((tile / NT) * 8 + rr) * LDW + (tile % NT) * 8 + cc] = wv[u];
      }
    }
  }
  {
    // Wsm = -(T^T W):  (T^T W)[a][c] = sum_{b <= a} T[b][a] W[b][c]     (T staged in shared memory)
    double *Tsm = Wraw + NBW * LDW;            // [NBW][LDW], still inside the partial-sum scratch
#pragma unroll
    for (int u = 0; u < (NBW * NBW + 255) / 256; ++u) {
      const int e = t + u * 256;
      if (e < NBW * NBW) Tsm[(e / NBW) * LDW + (e % NBW)] = tpre[u];
    }
    __syncthreads();
    for (int e = t; e < NBW * TN; e += 256) {
      const int aa = e / TN, c = e % TN;
      double v0 = 0.0, v1 = 0.0;
      if (a.notrans) {                                 // (T W)[a][c] = sum_{b >= a} T[a][b] W[b][c]: applies Q instead of Q^T
        for (int b2 = aa; b2 < NBW; ++b2) v0 += Tsm[aa * LDW + b2] * Wraw[b2 * LDW + c];
      } else {
        int b2 = 0;
        for (; b2 + 1 <= aa; b2 += 2) {
          v0 += Tsm[b2 * LDW + aa] * Wraw[b2 * LDW + c];
          v1 += Tsm[(b2 + 1) * LDW + aa] * Wraw[(b2 + 1) * LDW + c];
        }
        if (b2 <= aa) v0 += Tsm[b2 * LDW + aa] * Wraw[b2 * LDW + c];
      }
      Wsm[aa * LDW + c] = -(v0 + v1);
    }
    __syncthreads();
  }

  APPLY_CLK(4);
  // C. C <- C + V (-(T^T W)) over the warp's own row slice, written straight back to global memory; the V fragments
  // of the next 8-row tile are fetched while the current one is on the DMMA pipe
  {
    double bw[NBW / 4][NT];
#pragma unroll
    for (int ks = 0; ks < NBW / 4; ++ks)
#pragma unroll
      for (int j = 0; j < NT; ++j) bw[ks][j] = Wsm[(ks * 4 + (lane & 3)) * LDW + j * 8 + (lane >> 2)];
    double afn[NBW / 4];
    auto fetch = [&](int rt) {
      const int r = rt * 8 + (lane >> 2);
      const double *vt = V + (long)r * nbw + (lane & 3);
#pragma unroll
      for (int ks = 0; ks < NBW / 4; ++ks) afn[ks] = (r < R) ? __ldg(vt + ks * 4) : 0.0;
    };
    if (k0 < k1) fetch(k0 / 8);
    for (int rt = k0 / 8; rt < k1 / 8; ++rt) {
      const int r = rt * 8 + (lane >> 2);
      double af[NBW / 4];
#pragma unroll
      for (int ks = 0; ks < NBW / 4; ++ks) af[ks] = afn[ks];
      if (rt + 1 < k1 / 8) fetch(rt + 1);
      double acc[NT][2];
#pragma unroll
      for (int j = 0; j < NT; ++j) {
        acc[j][0] = Cs[csi(r, j * 8 + 2 * (lane & 3))];
        acc[j][1] = Cs[csi(r, j * 8 + 2 * (lane & 3) + 1)];
      }
#pragma unroll
      for (int ks = 0; ks < NBW / 4; ++ks)
#pragma unroll
        for (int j = 0; j < NT; ++j) dmma8x8x4(acc[j][0], acc[j][1], af[ks], bw[ks][j]);
      if (r < R) {
        // registers -> global directly (a TMA store out of the resident tile was measured slower: 15.0 vs 16.9 TF/s,
        // the CTA then has to wait for the bulk read of its tile before it can retire)
        double *dst;
        if constexpr (TM) dst = Aw + (long)(a.row0 + it * R + r) * a.lda + cbase; else dst = Aw + roff[r];
#pragma unroll
        for (int j = 0; j < NT; ++j) {
          const int c = j * 8 + 2 * (lane & 3);
          if (wide) {
            if (c < ncols) *reinterpret_cast<double2 *>(dst + c) = make_double2(acc[j][0], acc[j][1]);
          } else {
            if (c < ncols) dst[c] = acc[j][0];
            if (c + 1 < ncols) dst[c + 1] = acc[j][1];
          }
        }
      }
    }
  }
  APPLY_CLK(5);
}

// Column-streaming trailing update for contiguous row blocks of R <= 256 rows (R % 16 == 0, 32-wide panels).
// The round-1 kernel above keeps a (512 x 32) C tile resident and streams V twice from L2 per tile (once per DMMA phase):
// 524 KB of L2 -> SM traffic per 2.1 MFLOP, one CTA per SM whose load, V^T C, T^T W, C - V W and store phases do not
// overlap. Here the REFLECTOR block V (R x 32) and T live in shared memory for the whole CTA, and each warp streams
// 8-column chunks of the trailing matrix through its own (R x 8) buffer: TMA load of the chunk -> W = V^T C (DMMA, no
// cross-warp reduction: a warp owns all R rows of its 8 columns) -> -(T^T W) (DMMA, warp-private) -> C + V W (DMMA) ->
// stores straight from registers -> TMA load of the warp's next chunk. No block-wide barrier after the prologue: the
// eight warps drift apart, so one warp's load latency and serial steps are covered by the others' DMMA work, and V is
// read from L2 once per CTA instead of twice per tile.
constexpr int AC_LDV = 36, AC_LDT = 36;
static size_t apply_cols_smem_bytes(int R) {
  return ((size_t)R * AC_LDV + 32 * AC_LDT + 8 * ((size_t)R * 8 + 256)) * sizeof(double) + 9 * sizeof(uint64_t);
}
__global__ void __launch_bounds__(256, 1) apply_cols_kernel(ApplyArgs a, const __grid_constant__ TileMap tm, int nchunk, int cper) {
  extern __shared__ __align__(128) double acs[];
  const int R = a.R;
  double *Vs = acs;                                   // [R][36]
  double *Ts = Vs + (size_t)R * AC_LDV;               // [32][36]
  double *wbase = Ts + 32 * AC_LDT;
  const int wstride = R * 8 + 256;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5, fr = lane >> 2, fk = lane & 3;
  double *Cw = wbase + (size_t)warp * wstride;        // [R][8] this warp's chunk of the trailing matrix
  double *Ww = Cw + (size_t)R * 8;                    // [32][8] this warp's W
  uint64_t *bars = reinterpret_cast<uint64_t *>(wbase + (size_t)8 * wstride);   // [0..7] chunk barriers, [8] V
  const int cs = blockIdx.x, it = blockIdx.y, w = blockIdx.z;
  if (a.row_cnt && a.row0 + it * R >= a.row_cnt[w] * a.row_scale) return;               // all-zero row block of this walker
  if (a.stopped && a.stopped[w]) return;
  const double *V = a.Vw + ((long)w * a.NI + it) * (long)R * 32;
  const double *Tg = a.Tw + ((long)w * a.NI + it) * 1024L;
  double *Aw = a.A + (long)w * a.ws;
  const int row_base = a.row0 + it * R;
  const int c_lo = cs * cper, c_hi = min(nchunk, c_lo + cper);
  if (lane == 0) mbar_init(&bars[warp], 1);
  if (t == 0) mbar_init(&bars[8], 1);
  asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  __syncthreads();
  if (t == 0) mbar_expect_tx(&bars[8], (unsigned)(R * 256));
  int chunk = c_lo + warp;
  if (chunk < c_hi && lane == 0) {
    mbar_expect_tx(&bars[warp], (unsigned)(R * 64));
    tma_load_3d(Cw, &tm, a.col1 + 8 * chunk, row_base, w, &bars[warp]);
  }
  __syncthreads();
  for (int r = t; r < R; r += 256) bulk_g2s(Vs + (size_t)r * AC_LDV, V + (long)r * 32, 256u, &bars[8]);
  for (int e = t; e < 1024; e += 256) Ts[(e >> 5) * AC_LDT + (e & 31)] = __ldg(Tg + e);
  __syncthreads();
  mbar_wait(&bars[8], 0);
  unsigned ph = 0;
  for (; chunk < c_hi; chunk += 8) {
    mbar_wait(&bars[warp], ph);
    ph ^= 1;
    // A. W = V^T C over all R rows of the warp's 8 columns
    double acc[4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = 0.0;
#pragma unroll 4
    for (int k = 0; k < R; k += 4) {
      const int kr = k + fk;
      const double bf = Cw[kr * 8 + fr];
      const double *vr = Vs + (size_t)kr * AC_LDV + fr;
#pragma unroll
      for (int i = 0; i < 4; ++i) dmma8x8x4(acc[i][0], acc[i][1], vr[8 * i], bf);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) *reinterpret_cast<double2 *>(Ww + (i * 8 + fr) * 8 + 2 * fk) = make_double2(acc[i][0], acc[i][1]);
    __syncwarp();
    // T. Ww <- -(T^T W)   (notrans: -(T W))
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = 0.0;
#pragma unroll
    for (int ks = 0; ks < 8; ++ks) {
      const double bf = Ww[(ks * 4 + fk) * 8 + fr];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const double af = a.notrans ? Ts[(i * 8 + fr) * AC_LDT + ks * 4 + fk] : Ts[(ks * 4 + fk) * AC_LDT + i * 8 + fr];
        dmma8x8x4(acc[i][0], acc[i][1], af, bf);
      }
    }
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 4; ++i) *reinterpret_cast<double2 *>(Ww + (i * 8 + fr) * 8 + 2 * fk) = make_double2(-acc[i][0], -acc[i][1]);
    __syncwarp();
    double bw[8];
#pragma unroll
    for (int ks = 0; ks < 8; ++ks) bw[ks] = Ww[(ks * 4 + fk) * 8 + fr];
    // C. C <- C + V (-(T^T W)), two 8-row tiles in flight, stores straight from registers
    const int gcol = a.col1 + 8 * chunk + 2 * fk;
    const bool colok = gcol < a.col1 + a.ntrail;
    for (int rt = 0; rt < R / 8; rt += 2) {
      const int r0 = rt * 8 + fr, r1 = r0 + 8;
      double2 c0 = *reinterpret_cast<const double2 *>(Cw + r0 * 8 + 2 * fk);
      double2 c1 = *reinterpret_cast<const double2 *>(Cw + r1 * 8 + 2 * fk);
      const double *v0 = Vs + (size_t)r0 * AC_LDV + fk, *v1 = Vs + (size_t)r1 * AC_LDV + fk;
#pragma unroll
      for (int ks = 0; ks < 8; ++ks) {
        dmma8x8x4(c0.x, c0.y, v0[4 * ks], bw[ks]);
        dmma8x8x4(c1.x, c1.y, v1[4 * ks], bw[ks]);
      }
      if (colok) {
        *reinterpret_cast<double2 *>(Aw + (long)(row_base + r0) * a.lda + gcol) = c0;
        *reinterpret_cast<double2 *>(Aw + (long)(row_base + r1) * a.lda + gcol) = c1;
      }
    }
    __syncwarp();
    if (chunk + 8 < c_hi && lane == 0) {
      asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
      mbar_expect_tx(&bars[warp], (unsigned)(R * 64));
      tma_load_3d(Cw, &tm, a.col1 + 8 * (chunk + 8), row_base, w, &bars[warp]);
    }
  }
}

template <int NBW>
static size_t apply_smem_bytes(int R) {
  int R8 = (R + 7) & ~7;
  return ((size_t)R8 * (NBW + 4) + 4 * (size_t)(NBW / 8) * (NBW / 8) * 64 + (size_t)NBW * (NBW + 4) + (size_t)R8 + 8) * sizeof(double);
}
bool be_make_tile_map(TileMap *tm, const double *A, long ws, int lda, int rows, int cols, int W, int box_rows, int box_cols) {
  typedef CUresult (*EncodeFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                               const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeFn encode = []() -> EncodeFn {
    if (const char *e = std::getenv("PEPS_TILE_MAPS")) if (std::atoi(e) == 0) return nullptr;
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) return nullptr;
    return (EncodeFn)fn;
  }();
  static_assert(sizeof(CUtensorMap) <= sizeof(TileMap), "TileMap too small");
  if (!encode) return false;
  if ((lda & 1) || (ws & 1) || (reinterpret_cast<uintptr_t>(A) & 15) || box_rows < 1 || box_rows > 256 || box_cols < 2 ||
      box_cols > 256 || (box_cols & 1))
    return false;
  cuuint64_t gdim[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)W};
  cuuint64_t gstr[2] = {(cuuint64_t)lda * 8, (cuuint64_t)ws * 8};
  cuuint32_t box[3] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult rc = encode(reinterpret_cast<CUtensorMap *>(tm), CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, const_cast<double *>(A), gdim, gstr, box, estr,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return rc == CUDA_SUCCESS;
}

void be_apply_reflector(const ApplyArgs &a) {
  if (a.ntrail <= 0) return;
  LaunchScope scope(KC_APPLY, 4.0 * a.R * a.nbw * (double)a.ntrail * a.NI * a.W);
  static const TileMap no_map{};
  static const bool use_cols = []() { const char *e = std::getenv("PEPS_APPLY_COLS"); return e ? std::atoi(e) != 0 : true; }();
  if (use_cols && a.tmap_cols != nullptr && a.nbw == 32 && a.R <= 256 && a.R % 16 == 0 && (a.col1 & 1) == 0 && (a.lda & 1) == 0) {
    const int nchunk = (a.ntrail + 7) / 8;
    const int csplit = std::max(1, std::min(8, (nchunk + 12) / 24));
    const int cper = (nchunk + csplit - 1) / csplit;
    const size_t smem = apply_cols_smem_bytes(a.R);
    ensure_smem(apply_cols_kernel, smem);
    apply_cols_kernel<<<dim3((nchunk + cper - 1) / cper, a.NI, a.W), 256, smem, g_stream>>>(a, *a.tmap_cols, nchunk, cper);
    post_launch();
    return;
  }
  auto launch = [&](auto kern, size_t smem, int tn, const TileMap &tmap) {
    ensure_smem(kern, smem);
    kern<<<dim3((a.ntrail + tn - 1) / tn, a.NI, a.W), 256, smem, g_stream>>>(a, tmap);
  };
  // TMA boxes must start on a 16-byte boundary in global memory: an odd first trailing column rules the tile path out
  const bool tile = a.tmap != nullptr && a.nbw == 32 && a.R % 64 == 0 && (a.col1 & 1) == 0;
  // row blocks of <= 256 rows: the resident tile is <= 112 KB, two CTAs share an SM and overlap load / DMMA / store
  const bool small = apply_smem_bytes<32>(a.R) <= 112 * 1024;
  if (a.nbw == 32 && tile && small) launch(apply_reflector_kernel<32, 2, true>, apply_smem_bytes<32>(a.R), 32, *a.tmap);
  else if (a.nbw == 32 && tile) launch(apply_reflector_kernel<32, 1, true>, apply_smem_bytes<32>(a.R), 32, *a.tmap);
  else if (a.nbw == 32 && small) launch(apply_reflector_kernel<32, 2, false>, apply_smem_bytes<32>(a.R), 32, no_map);
  else if (a.nbw == 32) launch(apply_reflector_kernel<32, 1, false>, apply_smem_bytes<32>(a.R), 32, no_map);
  else if (a.nbw == 16) launch(apply_reflector_kernel<16, 1, false>, apply_smem_bytes<16>(a.R), 16, no_map);
  else if (a.nbw == 8) launch(apply_reflector_kernel<8, 1, false>, apply_smem_bytes<8>(a.R), 8, no_map);
  else throw std::runtime_error("be_apply_reflector: unsupported panel width");
  post_launch();
#ifdef PEPS_KERNEL_CLOCKS
  static const int dbg = std::getenv("PEPS_APPLY_CLK") ? std::atoi(std::getenv("PEPS_APPLY_CLK")) : 0;
  static int shown = 0;
  if (dbg && a.nbw == 32 && a.R == 512 && a.ntrail >= 256 && shown < dbg) {
    ++shown;
    long long h[8];
    CUDA_CHECK(cudaStreamSynchronize(g_stream));
    CUDA_CHECK(cudaMemcpyFromSymbol(h, g_apply_clk, sizeof(h)));
    fprintf(stderr, "[apply clk] R=%d ntrail=%d NI=%d W=%d roff=%lld fence=%lld issue=%lld wait=%lld A=%lld reduce+T=%lld C=%lld\n", a.R, a.ntrail, a.NI, a.W,
            h[6] - h[0], h[7] - h[6], h[1] - h[7], h[2] - h[1], h[3] - h[2], h[4] - h[3], h[5] - h[4]);
  }
#endif
}

// Early termination of the rank-revealing factorisations (backend.h be_trailing_check)
__global__ void trailing_norm_kernel(const double *A, long ws, int lda, int row0, int nrows, int col0, int ncols, double *acc,
                                     const int32_t *stopped) {
  const int w = blockIdx.y;
  if (stopped[w]) return;
  const double *Aw = A + (long)w * ws;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  double s0 = 0.0, s1 = 0.0;
  for (int r = row0 + blockIdx.x * nwarp + warp; r < nrows; r += gridDim.x * nwarp) {
    const double *x = Aw + (long)r * lda;
    int c = col0 + lane;
    for (; c + 32 < ncols; c += 64) { const double a = x[c], b = x[c + 32]; s0 = fma(a, a, s0); s1 = fma(b, b, s1); }
    if (c < ncols) { const double a = x[c]; s0 = fma(a, a, s0); }
  }
  double s = warp_sum(s0 + s1);
  __shared__ double red[8];
  if (lane == 0) red[warp] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < nwarp; ++i) t += red[i];
    if (t != 0.0) atomicAdd(acc + w, t);
  }
}
__global__ void trailing_decide_kernel(const double *colnorm2, const int32_t *colorder, int n, double thresh2, double *acc,
                                       int32_t *stopped, int W) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= W || stopped[w]) return;
  stopped[w] = (acc[w] <= thresh2 * colnorm2[(long)w * n + colorder[(long)w * n]]) ? 1 : 0;
  acc[w] = 0.0;
}
void be_trailing_check(const double *A, long ws, int lda, int row0, int nrows, int col0, int ncols, const double *colnorm2,
                       const int32_t *colorder, int n, double thresh2, double *acc, int32_t *stopped, int W) {
  if (nrows <= row0 || ncols <= col0) return;
  LaunchScope scope(KC_SMALL, 0.0);
  const int bx = std::max(1, std::min(16, (nrows - row0 + 63) / 64));
  trailing_norm_kernel<<<dim3(bx, W), 256, 0, g_stream>>>(A, ws, lda, row0, nrows, col0, ncols, acc, stopped);
  ++cx().launches;
  trailing_decide_kernel<<<(W + 127) / 128, 128, 0, g_stream>>>(colnorm2, colorder, n, thresh2, acc, stopped, W);
  post_launch();
}

// =====================================================================================================
// block Jacobi round
// =====================================================================================================
constexpr int JAC_THREADS = 256;
constexpr int JAC_KGROUPS = 4;          // K (column) split of the Gram matrix across warp pairs

__host__ __device__ __forceinline__ void rr_pair(int nblk, int round, int q, int &I, int &J) {
  // round-robin tournament on nblk (even) players: player nblk-1 is fixed
  const int n1 = nblk - 1;
  if (q == 0) { I = n1; J = round % n1; }
  else { I = (round + q) % n1; J = (round - q + n1) % n1; }
}

// Jacobi rotation (c, s) annihilating a_pq of [[app, apq], [apq, aqq]] (p < q), Rutishauser's small-angle choice.
// The tangent only steers the iteration (an error eps in it leaves eps * a_pq behind, which the next visit removes),
// so it is evaluated in FP32 with the approximate SFU instructions on exponent-normalised inputs; c = 1/sqrt(1 + t^2)
// and s = c t are then formed in FP64 (float seed + two Newton steps: 1e-7 -> 2e-14 -> 1e-27) so the rotation is
// orthogonal to double rounding. Branch-free: this sits on the critical path of every rotation set.
__device__ __forceinline__ void jacobi_cs(double app, double aqq, double apq, double tol2, double &c, double &s) {
  const double d = aqq - app, b2 = 2.0 * apq;
  const double m = fmax(fabs(d), fabs(b2));
  // scale = 2^-(exponent of m): keeps the FP32 evaluation away from overflow / underflow
  const int ex = ((__double2hiint(m) >> 20) & 0x7ff) - 1023;
  const double scale = __hiloint2double((1023 - ex) << 20, 0);
  const float df = (float)(d * scale), bf = (float)(b2 * scale);
  float rf;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rf) : "f"(fmaf(df, df, bf * bf)));
  float tf = __fdividef(bf, fabsf(df) + rf);
  tf = (df >= 0.0f) ? tf : -tf;
  float yf;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(yf) : "f"(fmaf(tf, tf, 1.0f)));
  const double t = (double)tf;
  const double hx = -0.5 * fma(t, t, 1.0);
  double y = (double)yf;
  y = y * fma(hx, y * y, 1.5);
  y = y * fma(hx, y * y, 1.5);
  const bool rot = (apq * apq > tol2 * fabs(app * aqq)) && (apq != 0.0);     // also discards the 0/0 of an all-zero block
  c = rot ? y : 1.0;
  s = rot ? y * t : 0.0;
}

// Systolic (Brent-Luk) round-robin ordering on 2*NP slots: slots [0, NP) are the "top" row, [NP, 2NP) the "bottom"
// row, pair k is always (slot k, slot NP + k). After a rotation set the index in slot s moves to slot jac_mu(s):
// top[0] stays, everything else advances one step along top[1] -> ... -> top[NP-1] -> bot[NP-1] -> ... -> bot[0] ->
// top[1]. All pairs meet once in 2NP-1 sets, and every shared-memory access of a rotation set is a contiguous run.
__device__ __forceinline__ int jac_mu(int s, int NP) {
  if (s == 0) return 0;
  if (s < NP - 1) return s + 1;
  if (s == NP - 1) return 2 * NP - 1;
  if (s == NP) return 1;
  return s - 1;
}
__device__ __forceinline__ int jac_mu_inv(int s, int NP) {
  if (s == 0) return 0;
  if (s == 1) return NP;
  if (s < NP) return s - 1;
  if (s < 2 * NP - 1) return s + 1;
  return NP - 1;
}

// One round of one-sided block Jacobi for one block pair. N2 = 2*bs rows resident in shared memory.
//   load -> Gram (DMMA, K split over warp pairs) -> cyclic two-sided Jacobi on the N2 x N2 Gram matrix with one
//   barrier per rotation set (the angles of set r+1 are computed by 16 threads while the others apply set r)
//   -> rows <- W^T rows on the DMMA pipe -> store.
#ifdef PEPS_KERNEL_CLOCKS
__device__ long long g_jac_clk[32];
#define JAC_CLK(i) do { if (blockIdx.x == gridDim.x - 1 && blockIdx.y == gridDim.y - 1 && threadIdx.x == 0) g_jac_clk[i] = clock64(); } while (0)
#define JAC_CLK_T(tid, i) do { if (blockIdx.x == gridDim.x - 1 && blockIdx.y == gridDim.y - 1 && threadIdx.x == (tid)) g_jac_clk[i] = clock64(); } while (0)
#else
#define JAC_CLK(i) do { } while (0)
#define JAC_CLK_T(tid, i) do { } while (0)
#endif
template <int N2>
__global__ void __launch_bounds__(JAC_THREADS) jacobi_round_kernel(JacobiArgs a) {
  extern __shared__ __align__(16) double sm[];
  JAC_CLK(0);
  constexpr int T2 = N2 / 8;
  constexpr int NT = T2 * (T2 + 1) / 2;
  constexpr int LG = N2 + 1;
  constexpr int NP = N2 / 2;
  constexpr int bs = N2 / 2;
  const int w = blockIdx.y;
  if (a.done[w]) return;
  const int LDS = ((a.nc + 7) & ~7) + 4;             // shared-memory row stride: sized by the full width
  double *Ps = sm;                                   // [N2][LDS]
  double *Gpart = Ps + (size_t)N2 * LDS;             // [JAC_KGROUPS][NT][64]
  double *Gm = Gpart + JAC_KGROUPS * NT * 64;        // [2][N2][LG]
  double *Wm = Gm + 2 * N2 * LG;                     // [2][N2][LG]
  double *coef = Wm + 2 * N2 * LG;                   // [2][2][N2]: (a_i, b_i) double buffered
  int *perm = (int *)(coef + 4 * N2);                // [N2]
  __shared__ double red[JAC_THREADS / 32];
  __shared__ int tile_p[NT], tile_q[NT];
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5, nwarp = JAC_THREADS / 32;

  int I, J;
  rr_pair(a.nblk, a.round, blockIdx.x, I, J);
  int c0 = 0, nc = a.nc;                             // column window of this block pair
  if (a.bsec) {                                      // Z2 sectors: cross-sector and empty block pairs are no-ops
    const int sI = a.bsec[(long)w * a.nblk + I], sJ = a.bsec[(long)w * a.nblk + J];
    if (sI != sJ || sI == 2) return;
    if (a.cwin) {                                    // the rows of a sector live on that sector's columns (sorted first / last)
      c0 = a.cwin[(long)w * 4 + 2 * sI]; nc = a.cwin[(long)w * 4 + 2 * sI + 1];
      if (nc <= 0) return;
    }
  }
  const int ncp = (nc + 7) & ~7;
  const int lo = min(I, J), hi = max(I, J);
  double *Gw = a.G + (long)w * a.ws + c0;
  const double tol2 = a.tol * a.tol;

  // 0. schedule tables
  if (t < NT) {
    int idx = 0;
    for (int p = 0; p < T2; ++p)
      for (int q = p; q < T2; ++q) { if (idx == t) { tile_p[t] = p; tile_q[t] = q; } ++idx; }
  }
  JAC_CLK(1);
  // 1. load the two row blocks (zero padded columns): one bulk copy (TMA) per row when the rows are 16-byte granular
  const bool wide = ((nc & 1) == 0) && ((c0 & 1) == 0) && ((a.ld & 1) == 0) && ((a.ws & 1) == 0) && ((reinterpret_cast<uintptr_t>(a.G) & 15) == 0);
  __shared__ uint64_t ld_bar;
  if (wide) {
    if (t == 0) {
      mbar_init(&ld_bar, 1);
      asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
      mbar_expect_tx(&ld_bar, (unsigned)(N2 * nc * 8));
    }
    __syncthreads();
    if (t < N2) {
      const int grow = (t < bs) ? lo * bs + t : hi * bs + (t - bs);
      bulk_g2s(Ps + (size_t)t * LDS, Gw + (long)grow * a.ld, (unsigned)(nc * 8), &ld_bar);
    }
    for (int e = t; e < N2 * (LDS - nc); e += JAC_THREADS) Ps[(size_t)(e / (LDS - nc)) * LDS + nc + e % (LDS - nc)] = 0.0;
    mbar_wait(&ld_bar, 0);
  } else {
    for (int r = warp; r < N2; r += nwarp) {
      const int grow = (r < bs) ? lo * bs + r : hi * bs + (r - bs);
      for (int c = lane; c < LDS; c += 32) Ps[(size_t)r * LDS + c] = (c < nc) ? Gw[(long)grow * a.ld + c] : 0.0;
    }
  }
  __syncthreads();
  JAC_CLK(2);

  // 2. Gram matrix on the DMMA pipe: warp (kg, half) accumulates its half of the upper tiles over its K slice
  {
    const int kg = warp >> 1, half = warp & 1;
    const int kq = ((ncp / JAC_KGROUPS) + 3) & ~3;
    const int k0 = kg * kq, k1 = min(ncp, k0 + kq);
    constexpr int MAXT = (NT + 1) / 2;
    double acc[MAXT][2];
    const double *ap[MAXT], *bp[MAXT];
#pragma unroll
    for (int i = 0; i < MAXT; ++i) {
      acc[i][0] = acc[i][1] = 0.0;
      int ti = 2 * i + half;
      int tp = (ti < NT) ? tile_p[ti] : 0, tq = (ti < NT) ? tile_q[ti] : 0;
      ap[i] = Ps + (size_t)(tp * 8 + (lane >> 2)) * LDS + (lane & 3);
      bp[i] = Ps + (size_t)(tq * 8 + (lane >> 2)) * LDS + (lane & 3);
    }
    for (int k = k0; k < k1; k += 4) {
#pragma unroll
      for (int i = 0; i < MAXT; ++i)
        if (2 * i + half < NT) dmma8x8x4(acc[i][0], acc[i][1], ap[i][k], bp[i][k]);
    }
#pragma unroll
    for (int i = 0; i < MAXT; ++i) {
      int ti = 2 * i + half;
      if (ti < NT) {
        double *g = Gpart + ((size_t)kg * NT + ti) * 64 + (lane >> 2) * 8 + 2 * (lane & 3);
        g[0] = acc[i][0]; g[1] = acc[i][1];
      }
    }
  }
  __syncthreads();
  JAC_CLK(3);
  for (int e = t; e < NT * 64; e += JAC_THREADS) {
    int ti = e >> 6, rr = (e >> 3) & 7, cc = e & 7;
    double v = 0.0;
#pragma unroll
    for (int kg = 0; kg < JAC_KGROUPS; ++kg) v += Gpart[((size_t)kg * NT + ti) * 64 + (e & 63)];
    int r = tile_p[ti] * 8 + rr, c = tile_q[ti] * 8 + cc;
    Gm[r * LG + c] = v;
    Gm[c * LG + r] = v;
  }
  for (int e = t; e < N2 * N2; e += JAC_THREADS) {
    int r = e / N2, c = e % N2;
    Wm[r * LG + c] = (r == c) ? 1.0 : 0.0;
  }
  __syncthreads();

  // 3. convergence measure before rotating: max g_pq^2 / (g_pp g_qq)
  {
    double mx = 0.0;
    for (int e = t; e < N2 * N2; e += JAC_THREADS) {
      int p = e / N2, q = e % N2;
      if (p < q) {
        double gpp = Gm[p * LG + p], gqq = Gm[q * LG + q], gpq = Gm[p * LG + q];
        if (gpp > 0.0 && gqq > 0.0 && gpq != 0.0) mx = fmax(mx, gpq * gpq / (gpp * gqq));
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if (lane == 0) red[warp] = mx;
    __syncthreads();
    if (t == 0) {
      for (int i = 1; i < nwarp; ++i) mx = fmax(mx, red[i]);
      mx = sqrt(mx);
      if (mx > 0.0) atomicMax((unsigned long long *)(a.offmax + w), (unsigned long long)__double_as_longlong(mx));
      red[0] = mx;
    }
    __syncthreads();
    if (red[0] <= a.tol) return;       // the 2*bs rows are already mutually orthogonal: nothing to rotate
  }

  JAC_CLK(4);
  // 4. cyclic two-sided Jacobi on Gm accumulating Wm, one barrier per rotation set. Thread (ki, kj) owns the 2x2
  //    block {p_i, q_i} x {p_j, q_j} of G (and of W): the four outputs need exactly the four inputs it loads.
  //    Slots are in the systolic order above, so nothing in the loop depends on the set index.
  const int nrounds = a.inner_sweeps * (N2 - 1);
  if (t < NP) {
    double c, s;
    jacobi_cs(Gm[t * LG + t], Gm[(NP + t) * LG + NP + t], Gm[t * LG + NP + t], tol2, c, s);
    coef[t] = c; coef[NP + t] = s;
  }
  // angle thread k: the indices that will form pair k after the move sit in slots po, qo now
  const int po = jac_mu_inv(t < NP ? t : 0, NP), qo = jac_mu_inv(NP + (t < NP ? t : 0), NP);
  const int aka = po % NP, akb = qo % NP;
  const bool selp = po < NP, selq = qo < NP;
  // update thread(s): block (ka, kb) -> rows {ka, NP+ka} x columns {kb, NP+kb}, written to the moved slots
  __syncthreads();
  int cur = 0;
  for (int g = 0; g < nrounds; ++g) {
    const double *Gc = Gm + cur * N2 * LG, *Wc = Wm + cur * N2 * LG, *cf = coef + cur * 2 * N2;
    double *Gn = Gm + (cur ^ 1) * N2 * LG, *Wn = Wm + (cur ^ 1) * N2 * LG, *cfn = coef + (cur ^ 1) * 2 * N2;
    if (t < NP) {
      // warp 0: angles of the NEXT rotation set, from the three entries of J^T G J each of its pairs will see
      if (g + 1 < nrounds) {
        const int pa = aka, qa = NP + aka, pb = akb, qb = NP + akb;
        const double ca = cf[aka], sa = cf[NP + aka], cb = cf[akb], sb = cf[NP + akb];
        const double gaa = Gc[pa * LG + pa], gab = Gc[pa * LG + qa], gba = Gc[qa * LG + pa], gbb = Gc[qa * LG + qa];
        const double haa = Gc[pb * LG + pb], hab = Gc[pb * LG + qb], hba = Gc[qb * LG + pb], hbb = Gc[qb * LG + qb];
        const double xpp = Gc[pa * LG + pb], xpq = Gc[pa * LG + qb], xqp = Gc[qa * LG + pb], xqq = Gc[qa * LG + qb];
        if (g == 3) JAC_CLK(10);
        // column of the rotation of pair a that lands on p (rows pa, qa); likewise for q in pair b
        const double ua0 = selp ? ca : sa, ua1 = selp ? -sa : ca;
        const double ub0 = selq ? cb : sb, ub1 = selq ? -sb : cb;
        const double npp = ua0 * (gaa * ua0 + gab * ua1) + ua1 * (gba * ua0 + gbb * ua1);
        const double nqq = ub0 * (haa * ub0 + hab * ub1) + ub1 * (hba * ub0 + hbb * ub1);
        const double npq = ua0 * (xpp * ub0 + xpq * ub1) + ua1 * (xqp * ub0 + xqq * ub1);
        double c, s;
        if (g == 3) JAC_CLK(11);
        jacobi_cs(npp, nqq, npq, tol2, c, s);
        cfn[t] = c; cfn[NP + t] = s;
        if (g == 3) JAC_CLK(12);
      }
    } else if (t >= 32) {
      // warps 1..7: G <- J^T G J and W <- W J by 2x2 blocks (four inputs, four outputs each)
      if (g == 3) JAC_CLK_T(32, 16);
      for (int e = t - 32; e < NP * NP; e += JAC_THREADS - 32) {
        const int ka = e / NP, kb = e % NP;
        const int pa = ka, qa = NP + ka, pb = kb, qb = NP + kb;
        const int mpa = jac_mu(pa, NP), mqa = jac_mu(qa, NP), mpb = jac_mu(pb, NP), mqb = jac_mu(qb, NP);
        const double ca = cf[ka], sa = cf[NP + ka], cb = cf[kb], sb = cf[NP + kb];
        const double g_pp = Gc[pa * LG + pb], g_pq = Gc[pa * LG + qb], g_qp = Gc[qa * LG + pb], g_qq = Gc[qa * LG + qb];
        const double w_pp = Wc[pa * LG + pb], w_pq = Wc[pa * LG + qb], w_qp = Wc[qa * LG + pb], w_qq = Wc[qa * LG + qb];
        if (g == 3 && e < 224) JAC_CLK_T(32, 17);
        const double r_pp = ca * g_pp - sa * g_qp, r_pq = ca * g_pq - sa * g_qq;     // rows: J^T G
        const double r_qp = sa * g_pp + ca * g_qp, r_qq = sa * g_pq + ca * g_qq;
        Gn[mpa * LG + mpb] = cb * r_pp - sb * r_pq; Gn[mpa * LG + mqb] = sb * r_pp + cb * r_pq;   // columns: (.) J
        Gn[mqa * LG + mpb] = cb * r_qp - sb * r_qq; Gn[mqa * LG + mqb] = sb * r_qp + cb * r_qq;
        // W <- W J: rows pa, qa of W are just two arbitrary (fixed) rows here; columns (pb, qb) rotate and move
        Wn[pa * LG + mpb] = cb * w_pp - sb * w_pq; Wn[pa * LG + mqb] = sb * w_pp + cb * w_pq;
        Wn[qa * LG + mpb] = cb * w_qp - sb * w_qq; Wn[qa * LG + mqb] = sb * w_qp + cb * w_qq;
        if (g == 3 && e < 224) JAC_CLK_T(32, 18);
      }
      if (g == 3) JAC_CLK_T(32, 19);
    }
    if (g == 3) JAC_CLK(13);
    __syncthreads();
    if (g == 3) JAC_CLK(14);
    if (g == 2) JAC_CLK(9);
    cur ^= 1;
  }
  const double *Gf = Gm + cur * N2 * LG, *Wf = Wm + cur * N2 * LG;
  JAC_CLK(5);

  // 5. permutation: new row r takes rotated direction perm[r], sorted by diagonal descending
  if (t < N2) {
    double mine = Gf[t * LG + t];
    int rank = 0;
    for (int j = 0; j < N2; ++j) {
      double o = Gf[j * LG + j];
      rank += (o > mine) || (o == mine && j < t);
    }
    perm[rank] = t;
  }
  __syncthreads();

  JAC_CLK(6);
  // 6. apply: Pnew[r][c] = sum_k W[k][perm[r]] * Ps[k][c] on the DMMA pipe, in place per 8-column slice
  {
    double af[T2][N2 / 4];
#pragma unroll
    for (int mt = 0; mt < T2; ++mt) {
      const int col = perm[mt * 8 + (lane >> 2)];
#pragma unroll
      for (int ks = 0; ks < N2 / 4; ++ks) af[mt][ks] = Wf[(ks * 4 + (lane & 3)) * LG + col];
    }
    const int nslice = ncp / 8;
    for (int sl = warp; sl < nslice; sl += nwarp) {
      double acc[T2][2];
#pragma unroll
      for (int mt = 0; mt < T2; ++mt) { acc[mt][0] = 0.0; acc[mt][1] = 0.0; }
      const double *bcol = Ps + (size_t)(lane & 3) * LDS + sl * 8 + (lane >> 2);
#pragma unroll
      for (int ks = 0; ks < N2 / 4; ++ks) {
        double bfrag = bcol[(size_t)ks * 4 * LDS];
#pragma unroll
        for (int mt = 0; mt < T2; ++mt) dmma8x8x4(acc[mt][0], acc[mt][1], af[mt][ks], bfrag);
      }
      __syncwarp();
#pragma unroll
      for (int mt = 0; mt < T2; ++mt) {
        double2 v; v.x = acc[mt][0]; v.y = acc[mt][1];
        *reinterpret_cast<double2 *>(Ps + (size_t)(mt * 8 + (lane >> 2)) * LDS + sl * 8 + 2 * (lane & 3)) = v;
      }
    }
  }
  __syncthreads();
  JAC_CLK(7);

  // 7. store (bulk copies straight out of shared memory; the CTA waits until its tile has been read)
  if (wide) {
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
    __syncthreads();
    if (t < N2) {
      const int grow = (t < bs) ? lo * bs + t : hi * bs + (t - bs);
      bulk_s2g(Gw + (long)grow * a.ld, Ps + (size_t)t * LDS, (unsigned)(nc * 8));
      asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
      asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
    }
  } else {
    for (int r = warp; r < N2; r += nwarp) {
      const int grow = (r < bs) ? lo * bs + r : hi * bs + (r - bs);
      for (int c = lane; c < nc; c += 32) Gw[(long)grow * a.ld + c] = Ps[(size_t)r * LDS + c];
    }
  }
  JAC_CLK(8);
}

static size_t jacobi_smem_bytes(int bs, int nc) {
  int n2 = 2 * bs, ncp = (nc + 7) & ~7, t2 = n2 / 8, nt = t2 * (t2 + 1) / 2;
  size_t doubles = (size_t)n2 * (ncp + 4) + (size_t)JAC_KGROUPS * nt * 64 + 4 * (size_t)n2 * (n2 + 1) + 4 * n2;
  return doubles * sizeof(double) + n2 * sizeof(int) + 16;
}
void be_jacobi_round(const JacobiArgs &a) {
  size_t smem = jacobi_smem_bytes(a.bs, a.nc);
  LaunchScope scope(KC_JACOBI, 3.0 * (2.0 * a.bs) * (2.0 * a.bs) * a.nc * (a.nblk / 2) * (double)a.nactive);
  auto launch = [&](auto kern) {
    ensure_smem(kern, smem);
    kern<<<dim3(a.nblk / 2, a.W), JAC_THREADS, smem, g_stream>>>(a);
  };
  if (a.bs == 16) launch(jacobi_round_kernel<32>);
  else if (a.bs == 8) launch(jacobi_round_kernel<16>);
  else if (a.bs == 4) launch(jacobi_round_kernel<8>);
  else throw std::runtime_error("be_jacobi_round: unsupported block size");
  post_launch();
#ifdef PEPS_KERNEL_CLOCKS
  static const int dbg = std::getenv("PEPS_JACOBI_CLK") ? std::atoi(std::getenv("PEPS_JACOBI_CLK")) : 0;
  static int shown = 0, seen = 0;
  if (dbg && a.bs == 16 && a.nc == 512 && (++seen % 97) == 0 && shown < dbg) {
    ++shown;
    long long h[32];
    CUDA_CHECK(cudaStreamSynchronize(g_stream));
    CUDA_CHECK(cudaMemcpyFromSymbol(h, g_jac_clk, sizeof(h)));
    fprintf(stderr, "[jacobi clk] nblk=%d W=%d tables=%lld load=%lld gram=%lld reduce+conv=%lld rotations=%lld perm=%lld apply=%lld store=%lld\n", a.nblk, a.W,
            h[1] - h[0], h[2] - h[1], h[3] - h[2], h[4] - h[3], h[5] - h[4], h[6] - h[5], h[7] - h[6], h[8] - h[7]);
    fprintf(stderr, "[jacobi upd ] since barrier: start=%lld loads=%lld compute+stores=%lld second_element=%lld\n", h[16] - h[9], h[17] - h[16], h[18] - h[17], h[19] - h[18]);
    fprintf(stderr, "[jacobi set] loads=%lld entries=%lld cs=%lld to_barrier=%lld barrier=%lld\n", h[10] - h[9], h[11] - h[10], h[12] - h[11], h[13] - h[12], h[14] - h[13]);
  }
#endif
}

__global__ void jacobi_flags_kernel(double *offmax, int32_t *done, double tol, int W) {
  int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w < W) {
    done[w] = (offmax[w] <= tol) ? 1 : 0;
    offmax[w] = 0.0;
  }
}
// one CTA per walker; labels / column marks in shared memory (rows <= 2048, columns <= 4096). In floating point the
// sector structure holds up to rounding noise only (a Householder QR puts R rows at pivot POSITIONS, which mixes in noise),
// so the labels compare weights: a row belongs to sector 0 when it carries more weight on the sector-0 columns than off
// them; the sector-0 columns start as the support of row 0 (largest norm) and are re-estimated once by column majority.
__global__ void __launch_bounds__(1024) sector_arrange_kernel(const double *src, long ws, int ld, int nc, const int32_t *count, int bs,
                                                             int nblk, double *dst, long wd, int32_t *bsec, const int32_t *cord_in,
                                                             int32_t *cord_out, int32_t *cwin) {
  extern __shared__ int sa_sm[];
  int *colA = sa_sm;              // [nc] column belongs to the sector of row 0
  int *lab = colA + nc;           // [nrows] 0 = sector of row 0, 1 = other
  int *pos = lab + nblk * bs;     // [nrows] destination row
  int *cpos = pos + nblk * bs;    // [nc] destination column: sector-0 columns first
  __shared__ double s_red[32];
  const int w = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5, NT = blockDim.x, NW = blockDim.x >> 5;
  const int n = min(count[w], nblk * bs);
  const double *S = src + (long)w * ws;
  double mx = 0.0;
  for (int c = t; c < nc; c += NT) mx = fmax(mx, n > 0 ? fabs(S[c]) : 0.0);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if (lane == 0) s_red[warp] = mx;
  __syncthreads();
  mx = 0.0;
  for (int i = 0; i < NW; ++i) mx = fmax(mx, s_red[i]);
  for (int c = t; c < nc; c += NT) colA[c] = (n > 0 && fabs(S[c]) > 1e-8 * mx) ? 1 : 0;
  __syncthreads();
  for (int pass = 0; pass < 2; ++pass) {
    for (int r = warp; r < n; r += NW) {
      double in = 0.0, out = 0.0;
      for (int c = lane; c < nc; c += 32) { const double v = fabs(S[(long)r * ld + c]); if (colA[c]) in += v; else out += v; }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) { in += __shfl_xor_sync(0xffffffffu, in, o); out += __shfl_xor_sync(0xffffffffu, out, o); }
      if (lane == 0) lab[r] = in >= out ? 0 : 1;
    }
    __syncthreads();
    if (pass == 0) {
      for (int c = t; c < nc; c += NT) {
        double wa = 0.0, wb = 0.0;
        for (int r = 0; r < n; ++r) { const double v = fabs(S[(long)r * ld + c]); if (lab[r] == 0) wa += v; else wb += v; }
        colA[c] = wa >= wb ? 1 : 0;
      }
      __syncthreads();
    }
  }
  if (t == 0) {
    int nA = 0, nB = 0;
    for (int r = 0; r < n; ++r) nA += (lab[r] == 0);
    const int baseB = (nA + bs - 1) / bs * bs;
    int ia = 0;
    for (int r = 0; r < n; ++r) { if (lab[r] == 0) pos[r] = ia++; else pos[r] = baseB + nB++; }
    const int blkA = (nA + bs - 1) / bs, blkB = (nB + bs - 1) / bs;
    for (int b = 0; b < nblk; ++b) bsec[(long)w * nblk + b] = b < blkA ? 0 : (b < blkA + blkB ? 1 : 2);
    int cA = 0;
    for (int c = 0; c < nc; ++c) cA += colA[c];
    int ja = 0, jb = cA;
    for (int c = 0; c < nc; ++c) cpos[c] = colA[c] ? ja++ : jb++;
    // windows with even starts and widths (16-byte row copies): a window may take in one column of the other sector,
    // where the rows of this sector hold rounding noise only
    int32_t *cw = cwin + (long)w * 4;
    cw[0] = 0; cw[1] = min(nc, (cA + 1) & ~1);
    cw[2] = cA & ~1; cw[3] = nc - cw[2];
    if ((nc & 1) && (cw[3] & 1)) { /* odd full width: the kernel's scalar path handles odd windows */ }
  }
  __syncthreads();
  for (int c = t; c < nc; c += NT) cord_out[(long)w * nc + cpos[c]] = cord_in ? cord_in[(long)w * nc + c] : c;
  double *D = dst + (long)w * wd;
  for (int r = warp; r < n; r += NW) {
    const int p = pos[r];
    if (p < nblk * bs)
      for (int c = lane; c < nc; c += 32) D[(long)p * ld + cpos[c]] = S[(long)r * ld + c];
  }
}
void be_sector_arrange(const double *src, long ws, int ld, int nc, const int32_t *count, int bs, int nblk, double *dst, long wd,
                       int32_t *bsec, const int32_t *cord_in, int32_t *cord_out, int32_t *cwin, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  const size_t smem = sizeof(int) * (2 * (size_t)nc + 2 * (size_t)nblk * bs);
  if (smem > 96 * 1024) throw std::runtime_error("be_sector_arrange: matrix too large for the label tables");
  ensure_smem(sector_arrange_kernel, smem);
  sector_arrange_kernel<<<W, 1024, smem, g_stream>>>(src, ws, ld, nc, count, bs, nblk, dst, wd, bsec, cord_in, cord_out, cwin);
  post_launch();
}
void be_jacobi_flags(double *offmax, int32_t *done, double tol, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  jacobi_flags_kernel<<<(W + 127) / 128, 128, 0, g_stream>>>(offmax, done, tol, W);
  post_launch();
}

// column norms: a CTA owns 32 columns, its 8 warps stride over the rows (256-byte coalesced reads), partial sums are
// combined in a fixed order (deterministic)
__global__ void col_norms2_kernel(const double *G, long ws, int ld, int nr, int nc, double *norms2) {
  __shared__ double part[8][33];
  const int w = blockIdx.y, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + lane;
  double s0 = 0.0, s1 = 0.0;
  if (c < nc) {
    const double *x = G + (long)w * ws + c;
    int r = warp;
    for (; r + 8 < nr; r += 16) {
      const double a = x[(long)r * ld], b = x[(long)(r + 8) * ld];
      s0 += a * a; s1 += b * b;
    }
    if (r < nr) { const double a = x[(long)r * ld]; s0 += a * a; }
  }
  part[warp][lane] = s0 + s1;
  __syncthreads();
  if (warp == 0 && c < nc) {
    double t = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += part[k][lane];
    norms2[(long)w * nc + c] = t;
  }
}
void be_col_norms2(const double *G, long ws, int ld, int nr, int nc, double *norms2, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  col_norms2_kernel<<<dim3((nc + 31) / 32, W), 256, 0, g_stream>>>(G, ws, ld, nr, nc, norms2);
  post_launch();
}
__global__ void permute_cols_kernel(const double *src, long ws, int lds, int nr, int nc, const int32_t *order, int gather,
                                    double *dst, long wd, int ldd) {
  const int w = blockIdx.y, r = blockIdx.x;
  const double *x = src + (long)w * ws + (long)r * lds;
  double *y = dst + (long)w * wd + (long)r * ldd;
  const int32_t *o = order + (long)w * nc;
  if (gather) { for (int j = threadIdx.x; j < nc; j += blockDim.x) y[j] = x[o[j]]; }
  else { for (int j = threadIdx.x; j < nc; j += blockDim.x) y[o[j]] = x[j]; }
}
void be_permute_cols(const double *src, long ws, int lds, int nr, int nc, const int32_t *order, int gather,
                     double *dst, long wd, int ldd, int W) {
  if (nr <= 0) return;
  LaunchScope scope(KC_SMALL, 0.0);
  permute_cols_kernel<<<dim3(nr, W), 128, 0, g_stream>>>(src, ws, lds, nr, nc, order, gather, dst, wd, ldd);
  post_launch();
}
__global__ void row_norms2_kernel(const double *G, long ws, int ld, int nr, int nc, double *norms2) {
  const int w = blockIdx.y;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= nr) return;
  const double *x = G + (long)w * ws + (long)warp * ld;
  double s = 0.0;
  for (int c = lane; c < nc; c += 32) s += x[c] * x[c];
  s = warp_sum(s);
  if (lane == 0) norms2[(long)w * nr + warp] = s;
}
void be_row_norms2(const double *G, long ws, int ld, int nr, int nc, double *norms2, int W) {
  int wpb = 8;
  LaunchScope scope(KC_SMALL, 0.0);
  row_norms2_kernel<<<dim3((nr + wpb - 1) / wpb, W), wpb * 32, 0, g_stream>>>(G, ws, ld, nr, nc, norms2);
  post_launch();
}

__global__ void rank_rows_kernel(const double *norms2, int nr, double defl2, int32_t *order, int32_t *count) {
  const int w = blockIdx.x;
  const double *x = norms2 + (long)w * nr;
  __shared__ double smax[256];
  double mx = 0.0;
  for (int r = threadIdx.x; r < nr; r += blockDim.x) mx = fmax(mx, x[r]);
  smax[threadIdx.x] = mx;
  __syncthreads();
  for (int h = blockDim.x / 2; h > 0; h >>= 1) {
    if (threadIdx.x < h) smax[threadIdx.x] = fmax(smax[threadIdx.x], smax[threadIdx.x + h]);
    __syncthreads();
  }
  mx = smax[0];
  __syncthreads();
  int cnt = 0;
  for (int r = threadIdx.x; r < nr; r += blockDim.x) {
    double mine = x[r];
    int rank = 0;
    for (int j = 0; j < nr; ++j) {
      double o = x[j];
      rank += (o > mine) || (o == mine && j < r);
    }
    order[(long)w * nr + rank] = r;
    cnt += (mine > defl2 * mx) ? 1 : 0;
  }
  __shared__ int scnt[256];
  scnt[threadIdx.x] = cnt;
  __syncthreads();
  for (int h = blockDim.x / 2; h > 0; h >>= 1) {
    if (threadIdx.x < h) scnt[threadIdx.x] += scnt[threadIdx.x + h];
    __syncthreads();
  }
  if (threadIdx.x == 0) count[w] = scnt[0];
}
void be_rank_rows(const double *norms2, int nr, double defl2, int32_t *order, int32_t *count, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  rank_rows_kernel<<<W, 256, 0, g_stream>>>(norms2, nr, defl2, order, count);
  post_launch();
}
__global__ void gather_rows_plain_kernel(const double *src, long ws, int ld, int nc, int nr_src, const int32_t *order,
                                         const int32_t *count, double *dst, long wd) {
  const int w = blockIdx.y, r = blockIdx.x;
  double *out = dst + (long)w * wd + (long)r * nc;
  if (r >= count[w] || r >= nr_src) {
    for (int c = threadIdx.x; c < nc; c += blockDim.x) out[c] = 0.0;
    return;
  }
  const double *x = src + (long)w * ws + (long)order[(long)w * nr_src + r] * ld;
  for (int c = threadIdx.x; c < nc; c += blockDim.x) out[c] = x[c];
}
void be_gather_rows(const double *src, long ws, int ld, int nc, int nr_src, const int32_t *order, const int32_t *count,
                    double *dst, long wd, int nr_dst, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  gather_rows_plain_kernel<<<dim3(nr_dst, W), 128, 0, g_stream>>>(src, ws, ld, nc, nr_src, order, count, dst, wd);
  post_launch();
}

__global__ void select_truncate_kernel(const double *norms2, int nr, int nsv, int dmin, int dmax, double trunc_err,
                                       int tcap, int32_t *order, int32_t *kept) {
  extern __shared__ double srt[];   // sorted squared singular values
  const int w = blockIdx.x;
  const double *x = norms2 + (long)w * nr;
  for (int r = threadIdx.x; r < nr; r += blockDim.x) {
    double mine = x[r];
    int rank = 0;
    for (int j = 0; j < nr; ++j) {
      double o = x[j];
      rank += (o > mine) || (o == mine && j < r);
    }
    srt[rank] = mine;
    if (rank < tcap) order[(long)w * tcap + rank] = r;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int n = nsv;           // singular values beyond the nr rows present are exact zeros
    int k = n;
    if (n > dmin) {
      double total = 0.0;
      for (int i = 0; i < n && i < nr; ++i) total += srt[i];
      double kept_sum = total;
      while (k > dmin) {
        double sv2 = (k - 1 < nr) ? srt[k - 1] : 0.0;
        if (k <= dmax && total > 0.0 && (1.0 - (kept_sum - sv2) / total) > trunc_err) break;
        kept_sum -= sv2;
        --k;
      }
    }
    if (k > tcap) k = tcap;
    kept[w] = k;
  }
}
void be_select_truncate(const double *norms2, int nr, int nsv, int dmin, int dmax, double trunc_err, int tcap,
                        int32_t *order, int32_t *kept, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  select_truncate_kernel<<<W, 256, nr * sizeof(double), g_stream>>>(norms2, nr, nsv, dmin, dmax, trunc_err, tcap,
                                                                   order, kept);
  post_launch();
}

__global__ void gather_rows_kernel(const double *G, long ws, int ld, int nc, const double *norms2, int nr,
                                   const int32_t *order, const int32_t *kept, int tcap, double *B, long wb) {
  const int w = blockIdx.y, tr = blockIdx.x;
  double *out = B + (long)w * wb + (long)tr * nc;
  if (tr >= kept[w] || tr >= nr) {
    for (int c = threadIdx.x; c < nc; c += blockDim.x) out[c] = 0.0;
    return;
  }
  int src = order[(long)w * tcap + tr];
  double n2 = norms2[(long)w * nr + src];
  double inv = (n2 > 0.0) ? 1.0 / sqrt(n2) : 0.0;
  const double *x = G + (long)w * ws + (long)src * ld;
  for (int c = threadIdx.x; c < nc; c += blockDim.x) out[c] = x[c] * inv;
}
void be_gather_rows_normalized(const double *G, long ws, int ld, int nc, const double *norms2, int nr,
                               const int32_t *order, const int32_t *kept, int tcap, double *B, long wb, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  gather_rows_kernel<<<dim3(tcap, W), 128, 0, g_stream>>>(G, ws, ld, nc, norms2, nr, order, kept, tcap, B, wb);
  post_launch();
}

// =====================================================================================================
// small-matrix SVD path of the truncation
// =====================================================================================================
__global__ void gather_rows_transposed_kernel(const double *src, long ws, int ld, int nc, int nr_src, const int32_t *order,
                                              const int32_t *count, double *dst, long wd, int n2) {
  __shared__ double tile[32][33];
  const int w = blockIdx.z, c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;      // 32 x 8
  const int cnt = min(count[w], nr_src);
  for (int rr = ty; rr < 32; rr += 8) {
    const int r = r0 + rr, c = c0 + tx;
    double v = 0.0;
    if (r < cnt && c < nc) v = src[(long)w * ws + (long)order[(long)w * nr_src + r] * ld + c];
    tile[rr][tx] = v;
  }
  __syncthreads();
  for (int cc = ty; cc < 32; cc += 8) {
    const int c = c0 + cc, r = r0 + tx;
    if (c < nc && r < n2) dst[(long)w * wd + (long)c * n2 + r] = tile[tx][cc];
  }
}
void be_gather_rows_transposed(const double *src, long ws, int ld, int nc, int nr_src, const int32_t *order,
                               const int32_t *count, double *dst, long wd, int n2, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  gather_rows_transposed_kernel<<<dim3((nc + 31) / 32, (n2 + 31) / 32, W), 256, 0, g_stream>>>(src, ws, ld, nc, nr_src, order, count, dst, wd, n2);
  post_launch();
}

__global__ void transpose_permute_kernel(const double *C0, long wc, int nc, int tcap, const int32_t *order, double *B, long wb) {
  __shared__ double tile[32][33];
  const int w = blockIdx.z, j0 = blockIdx.x * 32, t0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int jj = ty; jj < 32; jj += 8) {
    const int j = j0 + jj, t = t0 + tx;
    tile[jj][tx] = (j < nc && t < tcap) ? C0[(long)w * wc + (long)j * tcap + t] : 0.0;
  }
  __syncthreads();
  for (int tt = ty; tt < 32; tt += 8) {
    const int t = t0 + tt, j = j0 + tx;
    if (t < tcap && j < nc) {
      const int col = order ? order[(long)w * nc + j] : j;
      B[(long)w * wb + (long)t * nc + col] = tile[tx][tt];
    }
  }
}
void be_transpose_permute(const double *C0, long wc, int nc, int tcap, const int32_t *order, double *B, long wb, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  transpose_permute_kernel<<<dim3((nc + 31) / 32, (tcap + 31) / 32, W), 256, 0, g_stream>>>(C0, wc, nc, tcap, order, B, wb);
  post_launch();
}

// One-sided Jacobi SVD of a small square factor, one CTA per walker (see backend.h SmallSvdArgs). The n2 column vectors
// of Rt live in shared memory as rows X[k][.] (leading dimension NCAP + 8: 16-byte accesses of consecutive vectors hit
// disjoint bank groups). A rotation set pairs the vectors by the round-robin tournament; four lanes own one pair: each
// lane keeps NCAP/4 elements of both vectors in registers between the dot products and the rotation, so a set moves
// every vector through shared memory exactly once in each direction. The pair's Gram entries are summed over the four
// lanes by two shuffles. After a rotation the vector with the larger norm goes to the lower index (de Rijk), which keeps
// the singular values nearly sorted and speeds up convergence. A sweep without any rotation ends the iteration.
constexpr int SVS_THREADS = 256;
template <int NCAP>
__global__ void __launch_bounds__(SVS_THREADS, 1) svd_small_kernel(SmallSvdArgs a) {
  extern __shared__ __align__(16) double svs_sm[];
  constexpr int LDX = NCAP + 8;
  constexpr int NCH = NCAP / 8;                      // 8-element chunks per vector; lane j of a group owns elements 8i+2j, 8i+2j+1
  double *X = svs_sm;                                // [NCAP][LDX]
  double *nrm = X + (size_t)NCAP * LDX;              // [NCAP] squared norms, then sorted
  double *srt = nrm + NCAP;                          // [NCAP]
  int *perm = reinterpret_cast<int *>(srt + NCAP);   // [NCAP]
  __shared__ int s_kept;
  const int w = blockIdx.x;
  const int t = threadIdx.x, lane4 = t & 3, group = t >> 2;
  const unsigned gmask = 0xFu << ((t & 31) & ~3);       // the four lanes of this pair: groups of a warp may diverge
  const int n2 = a.n2;
  const int cnt = min(a.count[w], n2);
  const int nact = (cnt + 1) & ~1;                   // vectors taking part (even); beyond cnt they are zero
  const int nch = (nact + 7) >> 3;                   // chunks that can hold non-zeros (Rt is upper triangular)
  const double *Rw = a.Rt + (long)w * a.ws;
  const double tol2 = a.tol * a.tol;

  // load: X[k][i] = Rt[i][k]
  for (int e = t; e < NCAP * LDX; e += SVS_THREADS) X[e] = 0.0;
  __syncthreads();
  for (int e = t; e < n2 * n2; e += SVS_THREADS) {
    const int i = e / n2, k = e - i * n2;
    if (k >= i && k < nact) X[(size_t)k * LDX + i] = Rw[(long)i * a.ld + k];
  }
  __syncthreads();

  int sweeps = 0;
  if (nact >= 2) {
    const int npair = nact >> 1;
    for (; sweeps < a.max_sweeps; ++sweeps) {
      int rotated = 0;
      for (int step = 0; step < nact - 1; ++step) {
        for (int pr = group; pr < npair; pr += SVS_THREADS / 4) {
          int I, J;
          rr_pair(nact, step, pr, I, J);
          const int p = min(I, J), q = max(I, J);
          double2 *xp = reinterpret_cast<double2 *>(X + (size_t)p * LDX) + lane4;
          double2 *xq = reinterpret_cast<double2 *>(X + (size_t)q * LDX) + lane4;
          double2 vp[NCH], vq[NCH];
          double app = 0.0, aqq = 0.0, apq = 0.0, app1 = 0.0, aqq1 = 0.0, apq1 = 0.0;   // two partial sums each: the
#pragma unroll                                                                            // FMA chains are on the critical path
          for (int i = 0; i < NCH; ++i) {
            if (i < nch) {
              vp[i] = xp[4 * i]; vq[i] = xq[4 * i];
              app = fma(vp[i].x, vp[i].x, app); app1 = fma(vp[i].y, vp[i].y, app1);
              aqq = fma(vq[i].x, vq[i].x, aqq); aqq1 = fma(vq[i].y, vq[i].y, aqq1);
              apq = fma(vp[i].x, vq[i].x, apq); apq1 = fma(vp[i].y, vq[i].y, apq1);
            }
          }
          app += app1; aqq += aqq1; apq += apq1;
#pragma unroll
          for (int o = 1; o <= 2; o <<= 1) {
            app += __shfl_xor_sync(gmask, app, o);
            aqq += __shfl_xor_sync(gmask, aqq, o);
            apq += __shfl_xor_sync(gmask, apq, o);
          }
          double c, s;
          jacobi_cs(app, aqq, apq, tol2, c, s);
          if (s != 0.0) {                              // uniform over the four lanes of the pair
            rotated = 1;
            const double tg = s / c;
            const bool swap = (app - tg * apq) < (aqq + tg * apq);      // larger norm to the lower index
            double2 *dp = swap ? xq : xp, *dq = swap ? xp : xq;
#pragma unroll
            for (int i = 0; i < NCH; ++i) {
              if (i < nch) {
                double2 np, nq;
                np.x = c * vp[i].x - s * vq[i].x; np.y = c * vp[i].y - s * vq[i].y;
                nq.x = s * vp[i].x + c * vq[i].x; nq.y = s * vp[i].y + c * vq[i].y;
                dp[4 * i] = np; dq[4 * i] = nq;
              }
            }
          }
        }
        __syncthreads();
      }
      if (!__syncthreads_or(rotated)) { ++sweeps; break; }
    }
  }
  if (a.sweeps && t == 0) a.sweeps[w] = sweeps;

  // squared norms, ranking (descending, ties by index), truncation rule
  for (int k = group; k < NCAP; k += SVS_THREADS / 4) {
    double s2 = 0.0;
    if (k < nact) {
      const double2 *xk = reinterpret_cast<const double2 *>(X + (size_t)k * LDX) + lane4;
#pragma unroll
      for (int i = 0; i < NCH; ++i) if (i < nch) { const double2 v = xk[4 * i]; s2 = fma(v.x, v.x, s2); s2 = fma(v.y, v.y, s2); }
    }
    s2 += __shfl_xor_sync(gmask, s2, 1);
    s2 += __shfl_xor_sync(gmask, s2, 2);
    if (lane4 == 0) nrm[k] = s2;
  }
  __syncthreads();
  if (t < NCAP) {
    const double mine = nrm[t];
    int rank = 0;
    for (int j = 0; j < NCAP; ++j) { const double o = nrm[j]; rank += (o > mine) || (o == mine && j < t); }
    perm[rank] = t; srt[rank] = mine;
  }
  __syncthreads();
  if (t == 0) {
    const int n = a.nsv;
    int k = n;
    if (n > a.dmin) {
      double total = 0.0;
      for (int i = 0; i < n && i < NCAP; ++i) total += srt[i];
      double kept_sum = total;
      while (k > a.dmin) {
        const double sv2 = (k - 1 < NCAP) ? srt[k - 1] : 0.0;
        if (k <= a.dmax && total > 0.0 && (1.0 - (kept_sum - sv2) / total) > a.trunc_err) break;
        kept_sum -= sv2;
        --k;
      }
    }
    if (k > a.tcap) k = a.tcap;
    s_kept = k;
    a.kept[w] = k;
  }
  __syncthreads();
  const int kept = s_kept;
  double *out = a.out + (long)w * a.wo;
  for (int e = t; e < n2 * a.tcap; e += SVS_THREADS) {
    const int i = e / a.tcap, tt = e - i * a.tcap;
    double v = 0.0;
    if (tt < kept && tt < NCAP) {
      const double s2 = srt[tt];
      if (s2 > 0.0) v = X[(size_t)perm[tt] * LDX + i] * (1.0 / sqrt(s2));
    }
    out[(long)i * a.tcap + tt] = v;
  }
}
template <int NCAP>
static size_t svd_small_smem() { return ((size_t)NCAP * (NCAP + 8) + 2 * NCAP) * sizeof(double) + NCAP * sizeof(int) + 16; }
void be_svd_small(const SmallSvdArgs &a) {
  if (a.n2 > kSmallSvdMaxN || a.n2 < 1 || (a.n2 & 7)) throw std::runtime_error("be_svd_small: n2 must be a multiple of 8 in [8, 128]");
  // model flops of one sweep: n(n-1)/2 pairs x (3 dots + rotation) x n elements x 2 flops ~ 7 n^3
  LaunchScope scope(KC_JACOBI, 7.0 * a.n2 * a.n2 * a.n2 * 4.0 * (double)a.W);
  auto launch = [&](auto kern, size_t smem) {
    ensure_smem(kern, smem);
    kern<<<a.W, SVS_THREADS, smem, g_stream>>>(a);
  };
  if (a.n2 <= 32) launch(svd_small_kernel<32>, svd_small_smem<32>());
  else if (a.n2 <= 64) launch(svd_small_kernel<64>, svd_small_smem<64>());
  else launch(svd_small_kernel<128>, svd_small_smem<128>());
  post_launch();
}

// =====================================================================================================
// Monte Carlo state kernels
// =====================================================================================================
__global__ void mt_seed_kernel(uint32_t *mt, int32_t *idx, const uint32_t *seeds, int W) {
  int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= W) return;
  uint32_t *s = mt + (long)w * 624;
  s[0] = seeds[w];
  for (int i = 1; i < 624; ++i) s[i] = 1812433253u * (s[i - 1] ^ (s[i - 1] >> 30)) + (uint32_t)i;
  idx[w] = 624;
}
void be_mt_seed(uint32_t *mt, int32_t *idx, const uint32_t *seeds, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  mt_seed_kernel<<<(W + 63) / 64, 64, 0, g_stream>>>(mt, idx, seeds, W);
  post_launch();
}

__device__ uint32_t mt_next(uint32_t *s, int32_t &i) {
  if (i >= 624) {
    for (int k = 0; k < 624; ++k) {
      uint32_t y = (s[k] & 0x80000000u) | (s[(k + 1) % 624] & 0x7fffffffu);
      s[k] = s[(k + 397) % 624] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
    }
    i = 0;
  }
  uint32_t y = s[i++];
  y ^= y >> 11;
  y ^= (y << 7) & 0x9d2c5680u;
  y ^= (y << 15) & 0xefc60000u;
  y ^= y >> 18;
  return y;
}
// libstdc++ generate_canonical<double,53> on mt19937: (x0 + x1 * 2^32) / 2^64 with one rounding of the sum
__device__ double mt_uniform01(uint32_t *s, int32_t &i) {
  uint32_t x0 = mt_next(s, i);
  uint32_t x1 = mt_next(s, i);
  double sum = (double)x0 + (double)x1 * 4294967296.0;
  double r = sum / 18446744073709551616.0;
  if (r >= 1.0) r = 0.99999999999999988897769753748434595763683319091796875;  // nextafter(1, 0)
  return r;
}

__global__ void nn_exchange_decide_kernel(int32_t *cfg, int nsites, int s1, int s2, const double *psi_b,
                                          double *amp, uint32_t *mt, int32_t *idx, int32_t *accepted, int W, const double *jastrow) {
  int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= W) return;
  int32_t *c = cfg + (long)w * nsites;
  int c1 = c[s1], c2 = c[s2];
  if (c1 == c2) return;
  double pb = psi_b[w], pa = amp[w];
  bool ok;
  double div = 0.0;
  if (jastrow) { div = fabs(pb * jastrow[w]) / fabs(pa); ok = div >= 1.0; }
  else ok = fabs(pb) >= fabs(pa);
  if (!ok) {
    if (!jastrow) div = fabs(pb) / fabs(pa);
    double P = div * div;
    int32_t i = idx[w];
    double u = mt_uniform01(mt + (long)w * 624, i);
    idx[w] = i;
    ok = (u < P);
  }
  if (ok) {
    c[s1] = c2; c[s2] = c1;
    amp[w] = pb;
    accepted[w] += 1;
  }
}
void be_nn_exchange_decide(int32_t *cfg, int nsites, int s1, int s2, const double *psi_b, double *amp,
                           uint32_t *mt, int32_t *idx, int32_t *accepted, int W, const double *jastrow) {
  LaunchScope scope(KC_SMALL, 0.0);
  nn_exchange_decide_kernel<<<(W + 63) / 64, 64, 0, g_stream>>>(cfg, nsites, s1, s2, psi_b, amp, mt, idx, accepted, W, jastrow);
  post_launch();
}
__global__ void jastrow_ratio_kernel(const int32_t *cfg, int nsites, int s1, int s2, const int32_t *dens, const double *v,
                                     double *ratio, int W) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= W) return;
  const int32_t *c = cfg + (long)w * nsites;
  const int n1 = dens[c[s1]], n2 = dens[c[s2]];
  if (n1 == n2) { ratio[w] = 1.0; return; }
  double f1 = 0.0, f2 = 0.0;
  for (int j = 0; j < nsites; ++j) {
    const double nj = (double)dens[c[j]];
    if (j != s1) f1 += v[(long)s1 * nsites + j] * nj;
    if (j != s2) f2 += v[(long)s2 * nsites + j] * nj;
  }
  ratio[w] = n1 < n2 ? exp(f1 - f2) : exp(f2 - f1);
}
void be_jastrow_ratio(const int32_t *cfg, int nsites, int s1, int s2, const int32_t *dens, const double *v, double *ratio, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  jastrow_ratio_kernel<<<(W + 63) / 64, 64, 0, g_stream>>>(cfg, nsites, s1, s2, dens, v, ratio, W);
  post_launch();
}
__global__ void scale_kernel(double *x, const double *s, int W) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w < W) x[w] *= s[w];
}
void be_scale(double *x, const double *s, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  scale_kernel<<<(W + 127) / 128, 128, 0, g_stream>>>(x, s, W);
  post_launch();
}

__global__ void xxz_bond_energy_kernel(const int32_t *cfg, int nsites, int s1, int s2, const double *psi_ex,
                                       const double *psi, double jz, double jxy, double *eloc, int W) {
  int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= W) return;
  const int32_t *c = cfg + (long)w * nsites;
  double e;
  if (c[s1] == c[s2]) e = 0.25 * jz;
  else {
    double inv_psi = 1.0 / psi[w];
    double ratio = psi_ex[w] * inv_psi;
    e = -0.25 * jz + ratio * 0.5 * jxy;
  }
  eloc[w] += e;
}
void be_xxz_bond_energy(const int32_t *cfg, int nsites, int s1, int s2, const double *psi_ex, const double *psi,
                        double jz, double jxy, double *eloc, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  xxz_bond_energy_kernel<<<(W + 127) / 128, 128, 0, g_stream>>>(cfg, nsites, s1, s2, psi_ex, psi, jz, jxy, eloc, W);
  post_launch();
}
__global__ void ratio_accumulate_kernel(const double *psi_ex, const double *psi, double coef, double *eloc, int W) {
  int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w < W) eloc[w] += coef * (psi_ex[w] * (1.0 / psi[w]));
}
void be_ratio_accumulate(const double *psi_ex, const double *psi, double coef, double *eloc, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  ratio_accumulate_kernel<<<(W + 127) / 128, 128, 0, g_stream>>>(psi_ex, psi, coef, eloc, W);
  post_launch();
}
__global__ void term_targets_kernel(const int32_t *cfg, int nsites, int s1, int s2, int phys, const int32_t *target, const double *coef,
                                    int T, int t, int32_t *idx_a, int32_t *idx_b, double *coefw, int W) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= W) return;
  const int32_t *c = cfg + (long)w * nsites;
  const int c1 = c[s1], c2 = s2 >= 0 ? c[s2] : 0;
  const int p = s2 >= 0 ? c1 * phys + c2 : c1;
  const int tg = target[p * T + t];
  idx_a[w] = tg < 0 ? c1 : (s2 >= 0 ? tg / phys : tg);
  if (idx_b) idx_b[w] = tg < 0 ? c2 : tg % phys;
  coefw[w] = tg < 0 ? 0.0 : coef[p * T + t];
}
void be_term_targets(const int32_t *cfg, int nsites, int s1, int s2, int phys, const int32_t *target, const double *coef, int T,
                     int t, int32_t *idx_a, int32_t *idx_b, double *coefw, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  term_targets_kernel<<<(W + 127) / 128, 128, 0, g_stream>>>(cfg, nsites, s1, s2, phys, target, coef, T, t, idx_a, idx_b, coefw, W);
  post_launch();
}
__global__ void term_accumulate_kernel(const int32_t *cfg, int nsites, int s1, int s2, int phys, const double *diag,
                                       const double *coefw, const double *psi_ex, const double *psi, double *eloc, int W) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= W) return;
  const int32_t *c = cfg + (long)w * nsites;
  const int p = s2 >= 0 ? c[s1] * phys + c[s2] : c[s1];
  double e = diag ? diag[p] : 0.0;
  if (coefw && coefw[w] != 0.0) e += coefw[w] * (psi_ex[w] * (1.0 / psi[w]));
  eloc[w] += e;
}
void be_term_accumulate(const int32_t *cfg, int nsites, int s1, int s2, int phys, const double *diag, const double *coefw,
                        const double *psi_ex, const double *psi, double *eloc, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  term_accumulate_kernel<<<(W + 127) / 128, 128, 0, g_stream>>>(cfg, nsites, s1, s2, phys, diag, coefw, psi_ex, psi, eloc, W);
  post_launch();
}
__global__ void xxz_onsite_kernel(const int32_t *cfg, int nsites, double h00, double *eloc, int W) {
  int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w < W) eloc[w] += -h00 * ((double)cfg[(long)w * nsites] - 0.5);
}
void be_xxz_onsite_energy(const int32_t *cfg, int nsites, double h00, double *eloc, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  xxz_onsite_kernel<<<(W + 127) / 128, 128, 0, g_stream>>>(cfg, nsites, h00, eloc, W);
  post_launch();
}

// =====================================================================================================
// complex (c128) tensors as split planes (backend.h)
// =====================================================================================================
__global__ void embed_complex_kernel(const double *Ar, const double *Ai, long wa, int m, int n, double *M, long wm) {
  const int w = blockIdx.y;
  const double *ar = Ar + (long)w * wa, *ai = Ai + (long)w * wa;
  double *Mw = M + (long)w * wm;
  for (long e = blockIdx.x * (long)blockDim.x + threadIdx.x; e < (long)m * n; e += (long)gridDim.x * blockDim.x) {
    const long r = e / n, c = e - r * n;
    const double a = ar[e], b = ai[e];
    Mw[r * 2 * n + c] = a;  Mw[r * 2 * n + n + c] = -b;
    Mw[(r + m) * 2 * n + c] = b;  Mw[(r + m) * 2 * n + n + c] = a;
  }
}
void be_embed_complex(const double *Ar, const double *Ai, long wa, int m, int n, double *M, long wm, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  embed_complex_kernel<<<dim3(64, W), 256, 0, g_stream>>>(Ar, Ai, wa, m, n, M, wm);
  post_launch();
}
__global__ void split_r_kernel(const double *R, long wr, int rows, int n, double *outr, double *outi, long wo) {
  const int w = blockIdx.y;
  const double *Rw = R + (long)w * wr;
  const double s = 0.70710678118654752440;
  for (long e = blockIdx.x * (long)blockDim.x + threadIdx.x; e < (long)rows * n; e += (long)gridDim.x * blockDim.x) {
    const long r = e / n, c = e - r * n;
    outr[(long)w * wo + e] = s * Rw[r * 2 * n + c];
    outi[(long)w * wo + e] = -s * Rw[r * 2 * n + n + c];
  }
}
void be_split_r(const double *R, long wr, int rows, int n, double *outr, double *outi, long wo, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  split_r_kernel<<<dim3(32, W), 256, 0, g_stream>>>(R, wr, rows, n, outr, outi, wo);
  post_launch();
}
// one CTA per walker; the 2t candidate vectors stay in Bm (global / L2), z_j = Bm[j][:n] + i Bm[j][n:]
__global__ void __launch_bounds__(256) complex_basis_kernel(double *Bm, long wb, int tcap2, int n, const int32_t *kept2, double *Br,
                                                            double *Bi, long wo, int tcap, int32_t *keptc) {
  __shared__ double red[256], red2[256];
  __shared__ int s_piv;
  __shared__ double s_cr, s_ci;
  const int w = blockIdx.x, t = threadIdx.x;
  double *B = Bm + (long)w * wb;
  double *outr = Br + (long)w * wo, *outi = Bi + (long)w * wo;
  const int k2 = min(kept2[w], tcap2);
  const int kc = min((k2 + 1) / 2, tcap);
  int kc_done = kc;
  for (long e = t; e < (long)tcap * n; e += 256) { outr[e] = 0.0; outi[e] = 0.0; }
  __syncthreads();
  for (int q = 0; q < kc; ++q) {
    // pivot: the first remaining candidate whose residual is at least half the largest. The rows of Bm are sorted by
    // singular value and the residuals of a clean pair basis are ~1 or ~0, so the complex rows come out sorted as well
    // (the largest residual alone would break ties between unit rows by rounding).
    double best = -1.0;
    for (int j = t; j < k2; j += 256) {
      double s = 0.0;
      for (int c = 0; c < 2 * n; ++c) { const double v = B[(long)j * 2 * n + c]; s = fma(v, v, s); }
      best = fmax(best, s);
    }
    red[t] = best;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) { if (t < s) red[t] = fmax(red[t], red[t + s]); __syncthreads(); }
    const double mx = red[0];
    __syncthreads();
    double first = -1.0; int fi = k2;
    for (int j = t; j < k2; j += 256) {
      double s = 0.0;
      for (int c = 0; c < 2 * n; ++c) { const double v = B[(long)j * 2 * n + c]; s = fma(v, v, s); }
      if (s >= 0.5 * mx) { first = s; fi = j; break; }
    }
    red[t] = first; red2[t] = (double)fi;
    __syncthreads();
    if (t == 0) {
      double b = -1.0; int p = -1;
      for (int i = 0; i < 256; ++i) if ((int)red2[i] < k2 && (p < 0 || (int)red2[i] < p)) { b = red[i]; p = (int)red2[i]; }
      s_piv = p; s_cr = b;
    }
    __syncthreads();
    const int p = s_piv;
    // candidates are unit rows (or zero rows beyond the numerical rank); once the best residual is rounding noise the
    // subspace is exhausted: the remaining rows stay ZERO, exactly like the zero-padded rows of the real path (a normalised
    // noise vector would be a spurious direction)
    if (p < 0 || mx < 1e-10) { kc_done = q; break; }
    const double inv = 1.0 / sqrt(s_cr);
    // q-th basis vector = normalised pivot; re-orthogonalised against the previous ones (second Gram-Schmidt pass)
    for (int c = t; c < n; c += 256) { outr[(long)q * n + c] = inv * B[(long)p * 2 * n + c]; outi[(long)q * n + c] = inv * B[(long)p * 2 * n + n + c]; }
    __syncthreads();
    for (int prev = 0; prev < q; ++prev) {
      double cr = 0.0, ci = 0.0;                 // <u_prev, u_q> = sum conj(u_prev) u_q
      for (int c = t; c < n; c += 256) {
        const double ar = outr[(long)prev * n + c], ai = outi[(long)prev * n + c], br = outr[(long)q * n + c], bi2 = outi[(long)q * n + c];
        cr += ar * br + ai * bi2; ci += ar * bi2 - ai * br;
      }
      red[t] = cr; red2[t] = ci;
      __syncthreads();
      for (int s = 128; s > 0; s >>= 1) { if (t < s) { red[t] += red[t + s]; red2[t] += red2[t + s]; } __syncthreads(); }
      cr = red[0]; ci = red2[0];
      __syncthreads();
      for (int c = t; c < n; c += 256) {
        const double ar = outr[(long)prev * n + c], ai = outi[(long)prev * n + c];
        outr[(long)q * n + c] -= cr * ar - ci * ai;
        outi[(long)q * n + c] -= cr * ai + ci * ar;
      }
      __syncthreads();
    }
    {
      double s = 0.0;
      for (int c = t; c < n; c += 256) { const double a = outr[(long)q * n + c], b = outi[(long)q * n + c]; s += a * a + b * b; }
      red[t] = s;
      __syncthreads();
      for (int st = 128; st > 0; st >>= 1) { if (t < st) red[t] += red[t + st]; __syncthreads(); }
      const double nv = red[0] > 0.0 ? 1.0 / sqrt(red[0]) : 0.0;
      __syncthreads();
      for (int c = t; c < n; c += 256) { outr[(long)q * n + c] *= nv; outi[(long)q * n + c] *= nv; }
      __syncthreads();
    }
    // project u_q out of every candidate: z_j -= <u_q, z_j> u_q   (complex; the pivot itself becomes ~0)
    for (int j = 0; j < k2; ++j) {
      double cr = 0.0, ci = 0.0;
      for (int c = t; c < n; c += 256) {
        const double ar = outr[(long)q * n + c], ai = outi[(long)q * n + c], br = B[(long)j * 2 * n + c], bi2 = B[(long)j * 2 * n + n + c];
        cr += ar * br + ai * bi2; ci += ar * bi2 - ai * br;
      }
      red[t] = cr; red2[t] = ci;
      __syncthreads();
      for (int s = 128; s > 0; s >>= 1) { if (t < s) { red[t] += red[t + s]; red2[t] += red2[t + s]; } __syncthreads(); }
      cr = red[0]; ci = red2[0];
      __syncthreads();
      for (int c = t; c < n; c += 256) {
        const double ar = outr[(long)q * n + c], ai = outi[(long)q * n + c];
        B[(long)j * 2 * n + c] -= cr * ar - ci * ai;
        B[(long)j * 2 * n + n + c] -= cr * ai + ci * ar;
      }
      __syncthreads();
    }
  }
  // the MPS tensor is Vt = V^H: its rows are the CONJUGATES of the right singular vectors z (Theta = U S V^H)
  __syncthreads();
  for (long e = t; e < (long)kc_done * n; e += 256) outi[e] = -outi[e];
  if (t == 0) keptc[w] = kc;                       // the kept count follows the truncation rule; rows beyond kc_done are zero
}
void be_complex_basis(double *Bm, long wb, int tcap2, int n, const int32_t *kept2, double *Br, double *Bi, long wo, int tcap,
                      int32_t *keptc, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  complex_basis_kernel<<<W, 256, 0, g_stream>>>(Bm, wb, tcap2, n, kept2, Br, Bi, wo, tcap, keptc);
  post_launch();
}
__global__ void complex_combine_kernel(const double *d0, const double *d1, const double *d2, const double *d3, double *outr,
                                       double *outi, int W) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w < W) { outr[w] = d0[w] - d1[w]; outi[w] = d2[w] + d3[w]; }
}
void be_complex_combine(const double *d0, const double *d1, const double *d2, const double *d3, double *outr, double *outi, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  complex_combine_kernel<<<(W + 127) / 128, 128, 0, g_stream>>>(d0, d1, d2, d3, outr, outi, W);
  post_launch();
}
__global__ void nn_exchange_decide_c_kernel(int32_t *cfg, int nsites, int s1, int s2, const double *pbr, const double *pbi,
                                            double *ampr, double *ampi, uint32_t *mt, int32_t *idx, int32_t *accepted, int W,
                                            const double *jastrow) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= W) return;
  int32_t *c = cfg + (long)w * nsites;
  const int c1 = c[s1], c2 = c[s2];
  if (c1 == c2) return;
  const double j = jastrow ? jastrow[w] : 1.0;
  const double ab = jastrow ? hypot(pbr[w] * j, pbi[w] * j) : hypot(pbr[w], pbi[w]), aa = hypot(ampr[w], ampi[w]);
  bool ok = jastrow ? ab / aa >= 1.0 : ab >= aa;
  if (!ok) {
    const double div = ab / aa, P = div * div;
    int32_t i = idx[w];
    const double u = mt_uniform01(mt + (long)w * 624, i);
    idx[w] = i;
    ok = u < P;
  }
  if (ok) { c[s1] = c2; c[s2] = c1; ampr[w] = pbr[w]; ampi[w] = pbi[w]; accepted[w] += 1; }
}
void be_nn_exchange_decide_c(int32_t *cfg, int nsites, int s1, int s2, const double *pbr, const double *pbi, double *ampr,
                             double *ampi, uint32_t *mt, int32_t *idx, int32_t *accepted, int W, const double *jastrow) {
  LaunchScope scope(KC_SMALL, 0.0);
  nn_exchange_decide_c_kernel<<<(W + 63) / 64, 64, 0, g_stream>>>(cfg, nsites, s1, s2, pbr, pbi, ampr, ampi, mt, idx, accepted, W, jastrow);
  post_launch();
}
__global__ void ratio_accumulate_c_kernel(const double *exr, const double *exi, const double *pr, const double *pi, double coef,
                                          double *er, double *ei, int W) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= W) return;
  const double d = pr[w] * pr[w] + pi[w] * pi[w];
  const double rr = (exr[w] * pr[w] + exi[w] * pi[w]) / d, ri = (exi[w] * pr[w] - exr[w] * pi[w]) / d;   // psi_ex / psi
  er[w] += coef * rr;
  ei[w] += -coef * ri;                                                                                   // conj
}
void be_ratio_accumulate_c(const double *exr, const double *exi, const double *pr, const double *pi, double coef, double *er,
                           double *ei, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  ratio_accumulate_c_kernel<<<(W + 127) / 128, 128, 0, g_stream>>>(exr, exi, pr, pi, coef, er, ei, W);
  post_launch();
}
__global__ void term_accumulate_c_kernel(const int32_t *cfg, int nsites, int s1, int s2, int phys, const double *diag,
                                         const double *coefw, const double *exr, const double *exi, const double *pr,
                                         const double *pi, double *er, double *ei, int W) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= W) return;
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
void be_term_accumulate_c(const int32_t *cfg, int nsites, int s1, int s2, int phys, const double *diag, const double *coefw,
                          const double *exr, const double *exi, const double *pr, const double *pi, double *er, double *ei, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  term_accumulate_c_kernel<<<(W + 127) / 128, 128, 0, g_stream>>>(cfg, nsites, s1, s2, phys, diag, coefw, exr, exi, pr, pi, er, ei, W);
  post_launch();
}
__global__ void xxz_bond_energy_c_kernel(const int32_t *cfg, int nsites, int s1, int s2, const double *exr, const double *exi,
                                         const double *pr, const double *pi, double jz, double jxy, double *er, double *ei, int W) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= W) return;
  const int32_t *c = cfg + (long)w * nsites;
  if (c[s1] == c[s2]) { er[w] += 0.25 * jz; return; }
  const double d = pr[w] * pr[w] + pi[w] * pi[w];
  const double rr = (exr[w] * pr[w] + exi[w] * pi[w]) / d, ri = (exi[w] * pr[w] - exr[w] * pi[w]) / d;   // psi_ex / psi
  er[w] += -0.25 * jz + rr * 0.5 * jxy;
  ei[w] += -ri * 0.5 * jxy;                                                                              // conj
}
void be_xxz_bond_energy_c(const int32_t *cfg, int nsites, int s1, int s2, const double *exr, const double *exi, const double *pr,
                          const double *pi, double jz, double jxy, double *er, double *ei, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  xxz_bond_energy_c_kernel<<<(W + 127) / 128, 128, 0, g_stream>>>(cfg, nsites, s1, s2, exr, exi, pr, pi, jz, jxy, er, ei, W);
  post_launch();
}
__global__ void accumulate_ostar_c_kernel(const double *hr, const double *hi, long hole_stride, const int32_t *hole_off,
                                          const int32_t *site_size, const int32_t *tps_off, const int32_t *cfg, int nsites,
                                          const double *ampr, const double *ampi, const double *er, const double *ei, double *osr,
                                          double *osi, double *eor, double *eoi, int W) {
  const int site = blockIdx.y;
  const int sz = site_size[site];
  const long ho = hole_off[site], to = tps_off[site];
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < sz; e += gridDim.x * blockDim.x)
    for (int w = 0; w < W; ++w) {                       // fixed walker order
      const int c = cfg[(long)w * nsites + site];
      const double d = ampr[w] * ampr[w] + ampi[w] * ampi[w];
      const double a = hr[(long)w * hole_stride + ho + e], b = hi[(long)w * hole_stride + ho + e];
      const double qr = (a * ampr[w] + b * ampi[w]) / d, qi = (b * ampr[w] - a * ampi[w]) / d;          // hole / psi
      const double orr = qr, oi = -qi;                                                                  // O* = conj
      const long slot = to + (long)c * sz + e;
      osr[slot] += orr; osi[slot] += oi;
      eor[slot] += er[w] * orr + ei[w] * oi;            // conj(E) O* = (er - i ei)(or + i oi)
      eoi[slot] += er[w] * oi - ei[w] * orr;
    }
}
void be_accumulate_ostar_c(const double *hr, const double *hi, long hole_stride, const int32_t *hole_off, const int32_t *site_size,
                           const int32_t *tps_off, const int32_t *cfg, int nsites, const double *ampr, const double *ampi,
                           const double *er, const double *ei, double *osr, double *osi, double *eor, double *eoi, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  accumulate_ostar_c_kernel<<<dim3(16, nsites), 256, 0, g_stream>>>(hr, hi, hole_stride, hole_off, site_size, tps_off, cfg, nsites,
                                                                  ampr, ampi, er, ei, osr, osi, eor, eoi, W);
  post_launch();
}

// =====================================================================================================
// fermion mode (sign-dressed dense tensors; backend.h)
// =====================================================================================================
__global__ void fermion_gather_kernel(const int32_t *cfg, int rows, int cols, int phys, const int32_t *par, int32_t *gh,
                                      int32_t *gv, int32_t *jh, int32_t *jv, int W) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= W) return;
  const long base = (long)w * rows * cols;
  for (int r = 0; r < rows; ++r) {
    int acc = 0;
    for (int c = 0; c < cols; ++c) {
      const long i = base + r * cols + c;
      jh[i] = acc;
      gh[i] = acc * phys + cfg[i];
      acc ^= par[cfg[i]];
    }
  }
  for (int c = 0; c < cols; ++c) {
    int acc = 0;
    for (int r = 0; r < rows; ++r) {
      const long i = base + r * cols + c;
      jv[i] = acc;
      gv[i] = (6 + acc) * phys + cfg[i];
      acc ^= par[cfg[i]];
    }
  }
}
void be_fermion_gather(const int32_t *cfg, int rows, int cols, int phys, const int32_t *phys_par, int32_t *gidx_h,
                       int32_t *gidx_v, int32_t *jw_h, int32_t *jw_v, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  fermion_gather_kernel<<<(W + 63) / 64, 64, 0, g_stream>>>(cfg, rows, cols, phys, phys_par, gidx_h, gidx_v, jw_h, jw_v, W);
  post_launch();
}
__global__ void fermion_targets_kernel(const int32_t *cfg, int nsites, int s1, int s2, int phys, const int32_t *par,
                                       const int32_t *jh, const int32_t *jv, int kind, const int32_t *target,
                                       const double *coef, int T, int t, int32_t *idx_a, int32_t *idx_b, double *coefw, int W) {
  const int w = blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= W) return;
  const long o = (long)w * nsites;
  fermion_target_one(cfg + o, jh + o, jv + o, s1, s2, phys, par, kind, target, coef, T, t, idx_a[w], idx_b[w], coefw[w]);
}
void be_fermion_targets(const int32_t *cfg, int nsites, int s1, int s2, int phys, const int32_t *phys_par,
                        const int32_t *jw_h, const int32_t *jw_v, int kind, const int32_t *target, const double *coef,
                        int T, int t, int32_t *idx_a, int32_t *idx_b, double *coefw, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  fermion_targets_kernel<<<(W + 127) / 128, 128, 0, g_stream>>>(cfg, nsites, s1, s2, phys, phys_par, jw_h, jw_v, kind, target,
                                                                coef, T, t, idx_a, idx_b, coefw, W);
  post_launch();
}
// one CTA per (site, walker): fixed-order tree reduction of <hole, dressed tensor>, then the rescale of the hole
__global__ void fermion_finish_holes_kernel(double *holes, long hole_stride, const int32_t *hole_off, const int32_t *site_size,
                                            const double *gtps, const int64_t *gtps_off, const int32_t *gidx_h,
                                            const int32_t *jw_h, int nsites, const double *sign, const double *amp) {
  __shared__ double red[256];
  const int site = blockIdx.x, w = blockIdx.y;
  const int sz = site_size[site];
  double *h = holes + (long)w * hole_stride + hole_off[site];
  const double *t = gtps + gtps_off[site] + (long)gidx_h[(long)w * nsites + site] * sz;
  double acc = 0.0;
  for (int e = threadIdx.x; e < sz; e += blockDim.x) acc += h[e] * t[e];
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int s = blockDim.x / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
    __syncthreads();
  }
  const double f = amp[w] / red[0];
  const double *sg = sign + (long)jw_h[(long)w * nsites + site] * hole_stride + hole_off[site];
  for (int e = threadIdx.x; e < sz; e += blockDim.x) h[e] = h[e] * sg[e] * f;
}
void be_fermion_finish_holes(double *holes, long hole_stride, const int32_t *hole_off, const int32_t *site_size,
                             const double *gtps, const int64_t *gtps_off, const int32_t *gidx_h, const int32_t *jw_h,
                             int nsites, const double *sign, const double *amp, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  fermion_finish_holes_kernel<<<dim3(nsites, W), 256, 0, g_stream>>>(holes, hole_stride, hole_off, site_size, gtps, gtps_off,
                                                                     gidx_h, jw_h, nsites, sign, amp);
  post_launch();
}

// complex twin: two fixed-order tree reductions (re, im of the bilinear <hole, tensor>), complex rescale
__global__ void fermion_finish_holes_c_kernel(double *hr, double *hi, long hole_stride, const int32_t *hole_off,
                                              const int32_t *site_size, const double *gtps, long gtps_im_off,
                                              const int64_t *gtps_off, const int32_t *gidx_h, const int32_t *jw_h, int nsites,
                                              const double *sign, const double *ampr, const double *ampi) {
  __shared__ double redr[256], redi[256];
  const int site = blockIdx.x, w = blockIdx.y;
  const int sz = site_size[site];
  double *a = hr + (long)w * hole_stride + hole_off[site], *b = hi + (long)w * hole_stride + hole_off[site];
  const double *tr = gtps + gtps_off[site] + (long)gidx_h[(long)w * nsites + site] * sz, *ti = tr + gtps_im_off;
  double accr = 0.0, acci = 0.0;
  for (int e = threadIdx.x; e < sz; e += blockDim.x) {
    accr += a[e] * tr[e] - b[e] * ti[e];
    acci += a[e] * ti[e] + b[e] * tr[e];
  }
  redr[threadIdx.x] = accr; redi[threadIdx.x] = acci;
  __syncthreads();
  for (int s = blockDim.x / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) { redr[threadIdx.x] += redr[threadIdx.x + s]; redi[threadIdx.x] += redi[threadIdx.x + s]; }
    __syncthreads();
  }
  const double pr = redr[0], pi = redi[0], d = pr * pr + pi * pi;
  const double fr = (ampr[w] * pr + ampi[w] * pi) / d, fi = (ampi[w] * pr - ampr[w] * pi) / d;          // amp / psi_site
  const double *sg = sign + (long)jw_h[(long)w * nsites + site] * hole_stride + hole_off[site];
  for (int e = threadIdx.x; e < sz; e += blockDim.x) {
    const double x = a[e] * sg[e], y = b[e] * sg[e];
    a[e] = x * fr - y * fi;
    b[e] = x * fi + y * fr;
  }
}
void be_fermion_finish_holes_c(double *hr, double *hi, long hole_stride, const int32_t *hole_off, const int32_t *site_size,
                               const double *gtps, long gtps_im_off, const int64_t *gtps_off, const int32_t *gidx_h,
                               const int32_t *jw_h, int nsites, const double *sign, const double *ampr, const double *ampi, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  fermion_finish_holes_c_kernel<<<dim3(nsites, W), 256, 0, g_stream>>>(hr, hi, hole_stride, hole_off, site_size, gtps, gtps_im_off,
                                                                       gtps_off, gidx_h, jw_h, nsites, sign, ampr, ampi);
  post_launch();
}

template <int PHYS>
__global__ void accumulate_ostar_kernel(const double *holes, long hole_stride, const int32_t *hole_off,
                                        const int32_t *site_size, const int32_t *tps_off, const int32_t *cfg,
                                        int nsites, int phys, const double *amp, const double *eloc, double *osum,
                                        double *eosum, int W) {
  const int site = blockIdx.y;
  const int sz = site_size[site];
  const long ho = hole_off[site], to = tps_off[site];
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < sz; e += gridDim.x * blockDim.x) {
    double ao[PHYS], aeo[PHYS];
#pragma unroll
    for (int s = 0; s < PHYS; ++s) { ao[s] = (s < phys) ? osum[to + (long)s * sz + e] : 0.0; aeo[s] = (s < phys) ? eosum[to + (long)s * sz + e] : 0.0; }
    for (int w = 0; w < W; ++w) {                     // fixed walker order: the sums do not depend on scheduling
      const int c = cfg[(long)w * nsites + site];
      const double inv = 1.0 / amp[w];
      const double o = inv * holes[(long)w * hole_stride + ho + e];
      const double eo = eloc[w] * o;
#pragma unroll
      for (int s = 0; s < PHYS; ++s) { ao[s] += (c == s) ? o : 0.0; aeo[s] += (c == s) ? eo : 0.0; }
    }
#pragma unroll
    for (int s = 0; s < PHYS; ++s)
      if (s < phys) { osum[to + (long)s * sz + e] = ao[s]; eosum[to + (long)s * sz + e] = aeo[s]; }
  }
}
void be_accumulate_ostar(const double *holes, long hole_stride, const int32_t *hole_off, const int32_t *site_size,
                         const int32_t *tps_off, const int32_t *cfg, int nsites, int phys, const double *amp,
                         const double *eloc, double *osum, double *eosum, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  if (phys <= 2)
    accumulate_ostar_kernel<2><<<dim3(16, nsites), 256, 0, g_stream>>>(holes, hole_stride, hole_off, site_size, tps_off,
                                                                       cfg, nsites, phys, amp, eloc, osum, eosum, W);
  else if (phys <= 4)
    accumulate_ostar_kernel<4><<<dim3(16, nsites), 256, 0, g_stream>>>(holes, hole_stride, hole_off, site_size, tps_off,
                                                                       cfg, nsites, phys, amp, eloc, osum, eosum, W);
  else throw std::runtime_error("be_accumulate_ostar: physical dimension > 4 is not supported");
  post_launch();
}


// =====================================================================================================
// stochastic reconfiguration (HBM-bound: every O* sample is read once per kernel)
// =====================================================================================================
__global__ void sr_store_kernel(const double *holes, long hole_stride, const double *amp, const int32_t *cfg, int nsites,
                                double *ostar, int32_t *cfgs, long first) {
  const int w = blockIdx.y;
  const double inv = 1.0 / amp[w];
  const double *src = holes + (long)w * hole_stride;
  double *dst = ostar + (first + w) * hole_stride;
  for (long e = blockIdx.x * (long)blockDim.x + threadIdx.x; e < hole_stride; e += (long)gridDim.x * blockDim.x)
    dst[e] = inv * src[e];
  if (blockIdx.x == 0)
    for (int s = threadIdx.x; s < nsites; s += blockDim.x) cfgs[(first + w) * nsites + s] = cfg[(long)w * nsites + s];
}
void be_sr_store(const double *holes, long hole_stride, const double *amp, const int32_t *cfg, int nsites,
                 double *ostar, int32_t *cfgs, long first, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  sr_store_kernel<<<dim3(32, W), 256, 0, g_stream>>>(holes, hole_stride, amp, cfg, nsites, ostar, cfgs, first);
  post_launch();
}

__global__ void sr_store_c_kernel(const double *hr, const double *hi, long hole_stride, const double *ampr, const double *ampi,
                                  const int32_t *cfg, int nsites, double *ostar, int32_t *cfgs, long first, long cap) {
  const int w = blockIdx.y;
  const double d = ampr[w] * ampr[w] + ampi[w] * ampi[w];
  const double *a = hr + (long)w * hole_stride, *b = hi + (long)w * hole_stride;
  double *x = ostar + (first + w) * 2 * hole_stride, *y = ostar + (cap + first + w) * 2 * hole_stride;
  for (long e = blockIdx.x * (long)blockDim.x + threadIdx.x; e < hole_stride; e += (long)gridDim.x * blockDim.x) {
    const double qr = (a[e] * ampr[w] + b[e] * ampi[w]) / d, qi = (b[e] * ampr[w] - a[e] * ampi[w]) / d;   // hole / amp
    const double o_r = qr, o_i = -qi;                                                                      // O* = conj
    x[e] = o_r; x[hole_stride + e] = o_i;
    y[e] = -o_i; y[hole_stride + e] = o_r;
  }
  if (blockIdx.x == 0)
    for (int s = threadIdx.x; s < 2 * nsites; s += blockDim.x) {
      const int32_t c = cfg[(long)w * nsites + (s % nsites)];
      cfgs[(first + w) * 2 * nsites + s] = c;
      cfgs[(cap + first + w) * 2 * nsites + s] = c;
    }
}
void be_sr_store_c(const double *hr, const double *hi, long hole_stride, const double *ampr, const double *ampi, const int32_t *cfg,
                   int nsites, double *ostar, int32_t *cfgs, long first, long cap, int W) {
  LaunchScope scope(KC_SMALL, 0.0);
  sr_store_c_kernel<<<dim3(32, W), 256, 0, g_stream>>>(hr, hi, hole_stride, ampr, ampi, cfg, nsites, ostar, cfgs, first, cap);
  post_launch();
}

__global__ void sr_dots_kernel(const double *ostar, const int32_t *cfgs, long hole_stride, const int32_t *hole_off,
                               const int32_t *site_size, const int32_t *tps_off, int nsites, const double *v,
                               double mean_dot_v, double *delta) {
  const long i = blockIdx.x;
  const double *o = ostar + i * hole_stride;
  const int32_t *c = cfgs + i * nsites;
  __shared__ double red[256];
  double acc = 0.0;
  for (int site = 0; site < nsites; ++site) {
    const int sz = site_size[site];
    const double *os = o + hole_off[site];
    const double *vs = v + tps_off[site] + (long)c[site] * sz;
    for (int e = threadIdx.x; e < sz; e += blockDim.x) acc += os[e] * vs[e];
  }
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int h = blockDim.x / 2; h > 0; h >>= 1) {
    if (threadIdx.x < h) red[threadIdx.x] += red[threadIdx.x + h];
    __syncthreads();
  }
  if (threadIdx.x == 0) delta[i] = red[0] - mean_dot_v;
}
void be_sr_dots(const double *ostar, const int32_t *cfgs, long hole_stride, const int32_t *hole_off,
                const int32_t *site_size, const int32_t *tps_off, int nsites, const double *v, double mean_dot_v,
                double *delta, long n) {
  if (n <= 0) return;
  LaunchScope scope(KC_SMALL, 2.0 * hole_stride * (double)n);
  sr_dots_kernel<<<(unsigned)n, 256, 0, g_stream>>>(ostar, cfgs, hole_stride, hole_off, site_size, tps_off, nsites, v,
                                                    mean_dot_v, delta);
  post_launch();
}

// out[slot(site, s) + e] = sum_i [cfg_i(site) == s] delta[i] O*_i[hole_off(site) + e]: one thread per element of the
// hole layout, `PHYS` register accumulators, eight samples in flight per thread (the sample loop is the HBM stream:
// consecutive threads read consecutive elements of the same sample; the configuration entry and delta[i] are uniform
// per block and come out of L1). Deterministic: a fixed summation order per element.
template <int PHYS>
__global__ void __launch_bounds__(256) sr_accumulate_kernel(const double *__restrict__ ostar, const int32_t *__restrict__ cfgs,
                                                          long hole_stride, const int32_t *hole_off, const int32_t *site_size,
                                                          const int32_t *tps_off, int nsites, int phys,
                                                          const double *__restrict__ delta, double *out, long n) {
  const int site = blockIdx.y;
  const int sz = site_size[site];
  const long ho = hole_off[site], to = tps_off[site];
  const int32_t *cs = cfgs + site;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < sz; e += gridDim.x * blockDim.x) {
    double acc[PHYS];
#pragma unroll
    for (int s = 0; s < PHYS; ++s) acc[s] = 0.0;
    const double *col = ostar + ho + e;
    long i = 0;
    for (; i + 8 <= n; i += 8) {
      double o[8], d[8];
      int c[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        o[u] = col[(i + u) * hole_stride];
        c[u] = cs[(i + u) * nsites];
        d[u] = delta[i + u];
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const double t = d[u] * o[u];
#pragma unroll
        for (int s = 0; s < PHYS; ++s) acc[s] += (c[u] == s) ? t : 0.0;
      }
    }
    for (; i < n; ++i) {
      const double t = delta[i] * col[i * hole_stride];
      const int c = cs[i * nsites];
#pragma unroll
      for (int s = 0; s < PHYS; ++s) acc[s] += (c == s) ? t : 0.0;
    }
#pragma unroll
    for (int s = 0; s < PHYS; ++s)
      if (s < phys) out[to + (long)s * sz + e] = acc[s];
  }
}
void be_sr_accumulate(const double *ostar, const int32_t *cfgs, long hole_stride, const int32_t *hole_off,
                      const int32_t *site_size, const int32_t *tps_off, int nsites, int phys, const double *delta,
                      double *out, long n) {
  LaunchScope scope(KC_SMALL, 2.0 * hole_stride * (double)n);
  auto launch = [&](auto kern) {
    kern<<<dim3(16, nsites), 256, 0, g_stream>>>(ostar, cfgs, hole_stride, hole_off, site_size, tps_off, nsites, phys, delta, out, n);
  };
  if (phys <= 2) launch(sr_accumulate_kernel<2>);
  else if (phys <= 4) launch(sr_accumulate_kernel<4>);
  else throw std::runtime_error("be_sr_accumulate: physical dimension > 4 is not supported");
  post_launch();
}

// =====================================================================================================
// MinSR: masked Gram of the O* store (DMMA), centring, blocked Cholesky and the triangular solves
// =====================================================================================================
// CTA tile 64 x 64 of G, 2 x 2 warps of 32 x 32 (4 x 4 m8n8k4 DMMA tiles each). The K loop walks the sites of the
// CTA's split-K range in 16-element chunks (zero-padded at the end of a site), double-buffered through cp.async. Every
// chunk also brings the site's configuration entries of the tile's 64 rows and 64 columns. Products accumulate in a
// per-site register tile that is folded into the running total at the site boundary where cfg_i(site) == cfg_j(site).
constexpr int GR_BM = 64, GR_BK = 16, GR_THREADS = 128, GR_LD = GR_BM + 4;
struct GramStage {
  double a[GR_BK * GR_LD];
  double b[GR_BK * GR_LD];
  int32_t c[2 * GR_BM];
};
__device__ __forceinline__ void cp_async4(void *dst, const void *src, bool valid) {
  const unsigned saddr = (unsigned)__cvta_generic_to_shared(dst);
  const int sz = valid ? 4 : 0;
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(saddr), "l"(src), "r"(sz));
}
__global__ void __launch_bounds__(GR_THREADS)
sr_gram_kernel(const double *__restrict__ left, const double *__restrict__ right, const int32_t *__restrict__ cfgs,
               long hole_stride, const int32_t *__restrict__ hole_off, const int32_t *__restrict__ site_size, int nsites,
               const int32_t *__restrict__ split, long n, int tiles, double *__restrict__ part) {
  __shared__ GramStage st[2];
  int ti = 0, idx = blockIdx.x;                      // upper-triangle tile (ti <= tj), row by row
  while (idx >= tiles - ti) { idx -= tiles - ti; ++ti; }
  const int tj = ti + idx;
  const long r0 = (long)ti * GR_BM, c0 = (long)tj * GR_BM;
  const int s_end = split[blockIdx.y + 1];
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5, wm = warp >> 1, wn = warp & 1;
  const int lk = t & 15, lr = t >> 4;                // loader: k = t % 16, rows t / 16 + 8 i
  auto issue = [&](int stage, int site, int k0) {
    GramStage &S = st[stage];
    const int sz = site_size[site];
    const long ho = hole_off[site];
    const bool kv = k0 + lk < sz;
#pragma unroll
    for (int i = 0; i < GR_BM / 8; ++i) {
      const int r = lr + 8 * i;
      const bool va = kv && r0 + r < n, vb = kv && c0 + r < n;
      cp_async8(&S.a[lk * GR_LD + r], va ? left + (r0 + r) * hole_stride + ho + k0 + lk : left, va);
      cp_async8(&S.b[lk * GR_LD + r], vb ? right + (c0 + r) * hole_stride + ho + k0 + lk : right, vb);
    }
    const long g = t < GR_BM ? r0 + t : c0 + (t - GR_BM);
    cp_async4(&S.c[t], g < n ? cfgs + g * nsites + site : cfgs, g < n);
    asm volatile("cp.async.commit_group;\n" ::);
  };
  double acc[4][4][2], tot[4][4][2];
#pragma unroll
  for (int mt = 0; mt < 4; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) acc[mt][nt][0] = acc[mt][nt][1] = tot[mt][nt][0] = tot[mt][nt][1] = 0.0;
  int site = split[blockIdx.y], k0 = 0, stage = 0;
  issue(0, site, 0);
  for (;;) {
    int nsite = site, nk0 = k0 + GR_BK;
    if (nk0 >= site_size[site]) { nsite = site + 1; nk0 = 0; }
    const bool more = nsite < s_end;
    if (more) {
      issue(stage ^ 1, nsite, nk0);
      asm volatile("cp.async.wait_group 1;\n" ::);
    } else {
      asm volatile("cp.async.wait_group 0;\n" ::);
    }
    __syncthreads();
    const GramStage &S = st[stage];
#pragma unroll
    for (int kk = 0; kk < GR_BK; kk += 4) {
      double a[4], b[4];
      const int kr = (kk + (lane & 3)) * GR_LD + (lane >> 2);
#pragma unroll
      for (int q = 0; q < 4; ++q) { a[q] = S.a[kr + wm * 32 + q * 8]; b[q] = S.b[kr + wn * 32 + q * 8]; }
#pragma unroll
      for (int mt = 0; mt < 4; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) dmma8x8x4(acc[mt][nt][0], acc[mt][nt][1], a[mt], b[nt]);
    }
    if (nsite != site) {                             // site boundary: fold the site's products under the mask
#pragma unroll
      for (int mt = 0; mt < 4; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt)
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            const int r = wm * 32 + mt * 8 + (lane >> 2), c = wn * 32 + nt * 8 + (lane & 3) * 2 + i;
            if (S.c[r] == S.c[GR_BM + c]) tot[mt][nt][i] += acc[mt][nt][i];
            acc[mt][nt][i] = 0.0;
          }
    }
    __syncthreads();                                 // the stage is refilled by the issue of the next step
    if (!more) break;
    site = nsite; k0 = nk0; stage ^= 1;
  }
  double *P = part + (size_t)blockIdx.y * n * n;
#pragma unroll
  for (int mt = 0; mt < 4; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const long r = r0 + wm * 32 + mt * 8 + (lane >> 2), c = c0 + wn * 32 + nt * 8 + (lane & 3) * 2 + i;
        if (r < n && c < n) P[r * n + c] = tot[mt][nt][i];
      }
}
// G[i][j] = sum over the split-K slices in slice order (i <= j), mirrored with lower_sign below the diagonal
__global__ void sr_gram_reduce_kernel(const double *__restrict__ part, int nsplit, long n, double sign, double *__restrict__ G) {
  const size_t nn = (size_t)n * n;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < nn; e += (size_t)gridDim.x * blockDim.x) {
    const long i = (long)(e / n), j = (long)(e % n);
    if (i == j && sign < 0) { G[e] = 0.0; continue; }
    const size_t src = i <= j ? e : (size_t)j * n + i;
    double s = 0.0;
    for (int p = 0; p < nsplit; ++p) s += part[p * nn + src];
    G[e] = i <= j ? s : sign * s;
  }
}
void be_sr_gram(const double *left, const double *right, const int32_t *cfgs, long hole_stride, const int32_t *hole_off,
                const int32_t *site_size, const int32_t *site_size_host, int nsites, long n, double lower_sign, double *G) {
  if (n <= 0 || nsites <= 0) return;
  const int tiles = (int)((n + GR_BM - 1) / GR_BM);
  const long ntile = (long)tiles * (tiles + 1) / 2;
  int sms = 148;
  CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, cx().device));
  // split-K: contiguous site ranges of about equal padded length, enough slices for ~4 CTAs per SM
  std::vector<long> kp((size_t)nsites);
  long ktot = 0;
  for (int s = 0; s < nsites; ++s) { kp[(size_t)s] = (site_size_host[s] + GR_BK - 1) / GR_BK * GR_BK; ktot += kp[(size_t)s]; }
  const int want = (int)std::min<long>(std::min(nsites, 16), std::max<long>(1, (4L * sms + ntile - 1) / ntile));
  std::vector<int32_t> split{0};
  long run = 0;
  for (int s = 0; s + 1 < nsites; ++s) {
    run += kp[(size_t)s];
    if ((int)split.size() < want && run * want >= ktot * (long)split.size()) split.push_back(s + 1);
  }
  split.push_back(nsites);
  const int nsplit = (int)split.size() - 1;
  BeCtx &c = cx();
  const size_t need = (size_t)nsplit * n * n;
  if (need > c.gram_part_cap || nsplit + 1 > c.gram_split_cap) {
    CUDA_CHECK(cudaStreamSynchronize(g_stream));
    if (need > c.gram_part_cap) {
      if (c.gram_part) cudaFree(c.gram_part);
      CUDA_CHECK(cudaMalloc(&c.gram_part, sizeof(double) * need));
      c.gram_part_cap = need;
    }
    if (nsplit + 1 > c.gram_split_cap) {
      if (c.gram_split) cudaFree(c.gram_split);
      CUDA_CHECK(cudaMalloc(&c.gram_split, sizeof(int32_t) * 17));
      c.gram_split_cap = 17;
    }
  }
  be_h2d(c.gram_split, split.data(), sizeof(int32_t) * split.size());
  {
    LaunchScope scope(KC_GETT, 2.0 * GR_BM * GR_BM * (double)ktot * ntile);
    sr_gram_kernel<<<dim3((unsigned)ntile, (unsigned)nsplit), GR_THREADS, 0, g_stream>>>(
        left, right, cfgs, hole_stride, hole_off, site_size, nsites, c.gram_split, n, tiles, c.gram_part);
    post_launch();
  }
  LaunchScope scope(KC_SMALL, (double)nsplit * n * n);
  const int blocks = (int)std::min<long>(((long)n * n + 255) / 256, 148L * 16);
  sr_gram_reduce_kernel<<<blocks, 256, 0, g_stream>>>(c.gram_part, nsplit, n, lower_sign, G);
  post_launch();
}

__global__ void minsr_centre_kernel(const double *G, const double *a, double c, double sign, long n, double scale, double *T) {
  const size_t nn = (size_t)n * n;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < nn; e += (size_t)gridDim.x * blockDim.x) {
    const long i = (long)(e / n), j = (long)(e % n);
    T[e] = (sign < 0 && i == j) ? 0.0 : scale * (G[e] - a[i] - sign * a[j] + c);
  }
}
void be_minsr_centre(const double *G, const double *a, double c, double sign, long n, double scale, double *T) {
  if (n <= 0) return;
  LaunchScope scope(KC_SMALL, 0.0);
  const int blocks = (int)std::min<long>(((long)n * n + 255) / 256, 148L * 16);
  minsr_centre_kernel<<<blocks, 256, 0, g_stream>>>(G, a, c, sign, n, scale, T);
  post_launch();
}
__global__ void minsr_embed_kernel(const double *Tr, const double *Ti, long n, double shift, double *M) {
  const long m = Ti ? 2 * n : n;
  const size_t mm = (size_t)m * m;
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < mm; e += (size_t)gridDim.x * blockDim.x) {
    const long i = (long)(e / m), j = (long)(e % m);
    const long bi = i / n, bj = j / n, ii = i % n, jj = j % n;   // blocks [[Tr, -Ti], [Ti, Tr]]
    double v = (bi == bj) ? Tr[ii * n + jj] : (bi > bj ? Ti[ii * n + jj] : -Ti[ii * n + jj]);
    M[e] = v + (i == j ? shift : 0.0);
  }
}
void be_minsr_embed(const double *Tr, const double *Ti, long n, double shift, double *M) {
  if (n <= 0) return;
  LaunchScope scope(KC_SMALL, 0.0);
  const long m = Ti ? 2 * n : n;
  const int blocks = (int)std::min<long>((m * m + 255) / 256, 148L * 16);
  minsr_embed_kernel<<<blocks, 256, 0, g_stream>>>(Tr, Ti, n, shift, M);
  post_launch();
}

// Panel step k0 of the blocked Cholesky: every CTA factorises the kb x kb diagonal block in shared memory (one warp,
// right-looking) and solves its 128 rows below it, L21 = A21 L11^{-T} (one row per thread, in registers); CTA 0 writes
// the factorised block back and records the first non-positive pivot.
constexpr int CH_NB = 32;
__global__ void __launch_bounds__(128) chol_panel_kernel(double *M, long m, long k0, int kb, int32_t *info) {
  __shared__ double Ld[CH_NB][CH_NB + 1];
  const int t = threadIdx.x;
  for (int e = t; e < CH_NB * CH_NB; e += blockDim.x) {
    const int i = e / CH_NB, j = e % CH_NB;
    Ld[i][j] = (i < kb && j <= i) ? M[(k0 + i) * m + k0 + j] : (i == j ? 1.0 : 0.0);
  }
  __syncthreads();
  if (t < 32) {
    for (int j = 0; j < kb; ++j) {
      double d = Ld[j][j];
      if (!(d > 0.0)) {                              // not positive definite (or NaN): flag it, keep the arithmetic finite
        if (blockIdx.x == 0 && t == 0 && info[0] == 0) info[0] = (int32_t)(k0 + j + 1);
        d = 1.0;
      }
      d = sqrt(d);
      __syncwarp();
      if (t == j) Ld[j][j] = d;
      if (t > j && t < kb) Ld[t][j] /= d;
      __syncwarp();
      if (t > j && t < kb)
        for (int k = j + 1; k <= t; ++k) Ld[t][k] -= Ld[t][j] * Ld[k][j];
      __syncwarp();
    }
  }
  __syncthreads();
  if (blockIdx.x == 0)
    for (int e = t; e < kb * kb; e += blockDim.x) {
      const int i = e / kb, j = e % kb;
      if (j <= i) M[(k0 + i) * m + k0 + j] = Ld[i][j];
    }
  const long r = k0 + kb + (long)blockIdx.x * blockDim.x + t;
  if (r >= m) return;
  double *row = M + r * m + k0;
  double x[CH_NB];
#pragma unroll
  for (int j = 0; j < CH_NB; ++j) x[j] = j < kb ? row[j] : 0.0;
#pragma unroll
  for (int j = 0; j < CH_NB; ++j) {
    double s = x[j];
#pragma unroll
    for (int p = 0; p < j; ++p) s -= x[p] * Ld[j][p];
    x[j] = s / Ld[j][j];
  }
#pragma unroll
  for (int j = 0; j < CH_NB; ++j)
    if (j < kb) row[j] = x[j];
}
// Trailing update A22 -= L21 L21^T on the lower-triangle 64 x 64 tiles of the rows / columns [k0 + kb, m) (DMMA, K = kb)
__global__ void __launch_bounds__(GR_THREADS) chol_update_kernel(double *M, long m, long k0, int kb) {
  __shared__ double As[CH_NB * GR_LD], Bs[CH_NB * GR_LD];
  int ti = 0, idx = blockIdx.x;                      // lower-triangle tile (tj <= ti), row by row
  while (idx > ti) { idx -= ti + 1; ++ti; }
  const int tj = idx;
  const long k1 = k0 + kb, r0 = k1 + (long)ti * GR_BM, c0 = k1 + (long)tj * GR_BM;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5, wm = warp >> 1, wn = warp & 1;
  for (int e = t; e < GR_BM * CH_NB; e += GR_THREADS) {
    const int r = e / CH_NB, k = e % CH_NB;
    As[k * GR_LD + r] = (k < kb && r0 + r < m) ? M[(r0 + r) * m + k0 + k] : 0.0;
    Bs[k * GR_LD + r] = (k < kb && c0 + r < m) ? M[(c0 + r) * m + k0 + k] : 0.0;
  }
  __syncthreads();
  double acc[4][4][2];
#pragma unroll
  for (int mt = 0; mt < 4; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) acc[mt][nt][0] = acc[mt][nt][1] = 0.0;
#pragma unroll
  for (int kk = 0; kk < CH_NB; kk += 4) {
    double a[4], b[4];
    const int kr = (kk + (lane & 3)) * GR_LD + (lane >> 2);
#pragma unroll
    for (int q = 0; q < 4; ++q) { a[q] = As[kr + wm * 32 + q * 8]; b[q] = Bs[kr + wn * 32 + q * 8]; }
#pragma unroll
    for (int mt = 0; mt < 4; ++mt)
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) dmma8x8x4(acc[mt][nt][0], acc[mt][nt][1], a[mt], b[nt]);
  }
#pragma unroll
  for (int mt = 0; mt < 4; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const long r = r0 + wm * 32 + mt * 8 + (lane >> 2), c = c0 + wn * 32 + nt * 8 + (lane & 3) * 2 + i;
        if (r < m && c <= r) M[r * m + c] -= acc[mt][nt][i];
      }
}
void be_chol(double *M, long m, int32_t *info) {
  CUDA_CHECK(cudaMemsetAsync(info, 0, sizeof(int32_t), g_stream));
  for (long k0 = 0; k0 < m; k0 += CH_NB) {
    const int kb = (int)std::min<long>(CH_NB, m - k0);
    const long below = m - k0 - kb;
    {
      LaunchScope scope(KC_PANEL, (double)kb * kb * kb / 3.0 + (double)below * kb * kb);
      chol_panel_kernel<<<(unsigned)std::max<long>(1, (below + 127) / 128), 128, 0, g_stream>>>(M, m, k0, kb, info);
      post_launch();
    }
    if (below > 0) {
      const long tiles = (below + GR_BM - 1) / GR_BM, ntile = tiles * (tiles + 1) / 2;
      LaunchScope scope(KC_GETT, 2.0 * GR_BM * GR_BM * CH_NB * (double)ntile);
      chol_update_kernel<<<(unsigned)ntile, GR_THREADS, 0, g_stream>>>(M, m, k0, kb);
      post_launch();
    }
  }
}
// One CTA: forward substitution L y = b, then backward L^T z = y, in 32-row blocks. The off-block products are
// warp-parallel dot products (forward: a warp per row of L; backward: lanes over the block's columns, warps over the
// rows below, summed over warps in a fixed order); the 32 x 32 diagonal blocks are solved by one warp with shuffles.
__global__ void __launch_bounds__(1024) chol_solve_kernel(const double *__restrict__ L, long m, double *b) {
  __shared__ double part[32][33];
  __shared__ double sblk[32];
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const long nb = (m + 31) / 32;
  for (long I = 0; I < nb; ++I) {
    const long i0 = I * 32;
    const int kb = (int)(m - i0 < 32 ? m - i0 : 32);
    if (warp < kb) {
      const double *row = L + (i0 + warp) * m;
      double s = 0.0;
      for (long j = lane; j < i0; j += 32) s += row[j] * b[j];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0) sblk[warp] = b[i0 + warp] - s;
    }
    __syncthreads();
    if (warp == 0) {
      double v = lane < kb ? sblk[lane] : 0.0;
      for (int j = 0; j < kb; ++j) {
        const double yj = __shfl_sync(0xffffffffu, v, j) / L[(i0 + j) * m + i0 + j];
        if (lane == j) v = yj;
        else if (lane > j && lane < kb) v -= L[(i0 + lane) * m + i0 + j] * yj;
      }
      if (lane < kb) b[i0 + lane] = v;
    }
    __syncthreads();
  }
  for (long I = nb - 1; I >= 0; --I) {
    const long i0 = I * 32;
    const int kb = (int)(m - i0 < 32 ? m - i0 : 32);
    double s = 0.0;
    if (lane < kb)
      for (long j = i0 + kb + warp; j < m; j += 32) s += L[j * m + i0 + lane] * b[j];
    part[warp][lane] = s;
    __syncthreads();
    if (warp == 0) {
      double tot = 0.0;
      for (int w = 0; w < 32; ++w) tot += part[w][lane];
      double v = lane < kb ? b[i0 + lane] - tot : 0.0;
      for (int j = kb - 1; j >= 0; --j) {
        const double zj = __shfl_sync(0xffffffffu, v, j) / L[(i0 + j) * m + i0 + j];
        if (lane == j) v = zj;
        else if (lane < j) v -= L[(i0 + j) * m + i0 + lane] * zj;
      }
      if (lane < kb) b[i0 + lane] = v;
    }
    __syncthreads();
  }
}
void be_chol_solve(const double *L, long m, double *b) {
  if (m <= 0) return;
  LaunchScope scope(KC_SMALL, 2.0 * (double)m * m);
  chol_solve_kernel<<<1, 1024, 0, g_stream>>>(L, m, b);
  post_launch();
}

// ---- vector algebra of the device-resident CG ----------------------------------------------------------
__global__ void vec_lincomb_kernel(double *out, double ca, const double *a, double cb, const double *b, long n) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x)
    out[i] = b ? ca * a[i] + cb * b[i] : ca * a[i];
}
void be_vec_lincomb(double *out, double ca, const double *a, double cb, const double *b, long n) {
  if (n <= 0) return;
  LaunchScope scope(KC_SMALL, 0.0);
  const int blocks = (int)std::min<long>((n + 255) / 256, 148L * 8);
  vec_lincomb_kernel<<<blocks, 256, 0, g_stream>>>(out, ca, a, cb, b, n);
  post_launch();
}
constexpr int VDOT_BLOCKS = 296;
__global__ void vec_dot_part_kernel(const double *a, const double *b, long n, double *part) {
  __shared__ double red[256];
  double s0 = 0.0, s1 = 0.0;
  long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  const long stride = (long)gridDim.x * blockDim.x;
  for (; i + stride < n; i += 2 * stride) { s0 += a[i] * b[i]; s1 += a[i + stride] * b[i + stride]; }
  if (i < n) s0 += a[i] * b[i];
  red[threadIdx.x] = s0 + s1;
  __syncthreads();
  for (int h = blockDim.x / 2; h > 0; h >>= 1) {
    if (threadIdx.x < h) red[threadIdx.x] += red[threadIdx.x + h];
    __syncthreads();
  }
  if (threadIdx.x == 0) part[blockIdx.x] = red[0];
}
__global__ void vec_dot_finish_kernel(const double *part, int nb, double *result) {
  __shared__ double red[512];
  red[threadIdx.x] = (threadIdx.x < nb) ? part[threadIdx.x] : 0.0;
  __syncthreads();
  for (int h = blockDim.x / 2; h > 0; h >>= 1) {
    if (threadIdx.x < h) red[threadIdx.x] += red[threadIdx.x + h];
    __syncthreads();
  }
  if (threadIdx.x == 0) result[0] = red[0];
}
void be_vec_dot(const double *a, const double *b, long n, double *result) {
  LaunchScope scope(KC_SMALL, 2.0 * (double)n);
  double *&part = cx().vdot_part;
  if (!part) CUDA_CHECK(cudaMalloc(&part, sizeof(double) * VDOT_BLOCKS));
  vec_dot_part_kernel<<<VDOT_BLOCKS, 256, 0, g_stream>>>(a, b, n, part);
  ++cx().launches;
  vec_dot_finish_kernel<<<1, 512, 0, g_stream>>>(part, VDOT_BLOCKS, result);
  post_launch();
}

}  // namespace peps
