// See engine.h. Backend-agnostic host orchestration of the walker-batched VMC sampling path.
#include "engine.h"
#include <algorithm>
#include <array>
#include <cmath>
#include <complex>
#include <cstdio>
#include <cstdlib>
#include <limits>
#include <type_traits>

namespace peps {

Engine::Engine(const EngineConfig &c)
    : rows_(c.rows), cols_(c.cols), phys_(c.phys), D_(c.D), W_(c.walkers), nsites_(c.rows * c.cols),
      dmin_(c.dmin), dmax_(c.dmax), terr_(c.trunc_err) {
  if (rows_ < 2 || cols_ < 2) throw std::invalid_argument("Engine: lattice must be at least 2x2");
  if (W_ < 1 || phys_ < 1 || D_ < 1) throw std::invalid_argument("Engine: bad sizes");
  bectx_ = be_ctx_create(c.device);
  be_ctx_bind(bectx_);
  row_mod_.assign((size_t)rows_, 1);
  col_mod_.assign((size_t)cols_, 1);
  la_.W = W_; la_.pool = &pool_; la_.planner = &planner_;
  if (const char *e = std::getenv("PEPS_DEFLATION_EPS")) la_.deflation_eps = std::atof(e);
  if (const char *e = std::getenv("PEPS_BMPS_MEMO")) memo_on_ = std::atoi(e) != 0;
  if (const char *e = std::getenv("PEPS_PRESORT_COLS")) la_.presort_columns = std::atoi(e) != 0;
  if (const char *e = std::getenv("PEPS_CHAIN_EPS")) chain_eps_ = std::atof(e);
  if (const char *e = std::getenv("PEPS_SMALL_SVD")) la_.small_svd = std::atoi(e) != 0;
  if (const char *e = std::getenv("PEPS_QR_EARLY_STOP")) la_.qr_early_stop = std::atoi(e) != 0;
  if (const char *e = std::getenv("PEPS_QR_STOP_STRIDE")) la_.qr_stop_stride = std::max(1, std::atoi(e));
  la_.offmax = (double *)be_malloc(sizeof(double) * W_);
  la_.done = (int32_t *)be_malloc(sizeof(int32_t) * W_);
  tps_off_h_.resize((size_t)nsites_);
  site_size_h_.resize((size_t)nsites_);
  site_dims_h_.resize((size_t)nsites_);
  hole_off_h_.resize((size_t)nsites_);
  long off = 0, hoff = 0;
  for (int r = 0; r < rows_; ++r)
    for (int cc = 0; cc < cols_; ++cc) {
      int s = r * cols_ + cc;
      std::array<int, 4> d = {cc == 0 ? 1 : D_, r == rows_ - 1 ? 1 : D_, cc == cols_ - 1 ? 1 : D_, r == 0 ? 1 : D_};
      site_dims_h_[(size_t)s] = d;
      site_size_h_[(size_t)s] = d[0] * d[1] * d[2] * d[3];
      tps_off_h_[(size_t)s] = off;
      hole_off_h_[(size_t)s] = hoff;
      off += (long)phys_ * site_size_h_[(size_t)s];
      hoff += site_size_h_[(size_t)s];
    }
  tps_total_ = off;
  hole_stride_ = hoff;
  tps_ = (double *)be_malloc(sizeof(double) * tps_total_);
  gtps_ = tps_;
  gtps_total_ = tps_total_;
  gtps_off_h_ = tps_off_h_;
  osum_ = (double *)be_malloc(sizeof(double) * tps_total_);
  eosum_ = (double *)be_malloc(sizeof(double) * tps_total_);
  be_memset0(osum_, sizeof(double) * tps_total_);
  be_memset0(eosum_, sizeof(double) * tps_total_);
  std::vector<int32_t> t32((size_t)nsites_), h32((size_t)nsites_);
  for (int s = 0; s < nsites_; ++s) { t32[(size_t)s] = (int32_t)tps_off_h_[(size_t)s]; h32[(size_t)s] = (int32_t)hole_off_h_[(size_t)s]; }
  tps_off_d_ = (int32_t *)be_malloc(sizeof(int32_t) * nsites_);
  site_size_d_ = (int32_t *)be_malloc(sizeof(int32_t) * nsites_);
  hole_off_d_ = (int32_t *)be_malloc(sizeof(int32_t) * nsites_);
  be_h2d(tps_off_d_, t32.data(), sizeof(int32_t) * nsites_);
  be_h2d(site_size_d_, site_size_h_.data(), sizeof(int32_t) * nsites_);
  be_h2d(hole_off_d_, h32.data(), sizeof(int32_t) * nsites_);
  cfg_ = (int32_t *)be_malloc(sizeof(int32_t) * (size_t)W_ * nsites_);
  be_memset0(cfg_, sizeof(int32_t) * (size_t)W_ * nsites_);
  amp_ = (double *)be_malloc(sizeof(double) * W_);
  mt_ = (uint32_t *)be_malloc(sizeof(uint32_t) * (size_t)W_ * 624);
  mtidx_ = (int32_t *)be_malloc(sizeof(int32_t) * W_);
  accepted_ = (int32_t *)be_malloc(sizeof(int32_t) * W_);
  eloc_ = (double *)be_malloc(sizeof(double) * W_);
  psi_tmp_ = (double *)be_malloc(sizeof(double) * W_);
  psi_row_ = (double *)be_malloc(sizeof(double) * W_);
  kept_ = (int32_t *)be_malloc(sizeof(int32_t) * W_);
  holes_ = (double *)be_malloc(sizeof(double) * (size_t)W_ * hole_stride_);
  be_memset0(holes_, sizeof(double) * (size_t)W_ * hole_stride_);
  be_memset0(amp_, sizeof(double) * W_);
  be_memset0(eloc_, sizeof(double) * W_);
  std::vector<uint32_t> seeds((size_t)W_);
  for (int w = 0; w < W_; ++w) seeds[(size_t)w] = 5489u + (uint32_t)w;
  seed_rng(seeds.data());
}

Engine::~Engine() {
  be_ctx_bind(bectx_);
  be_sync();
  for (int p = 0; p < 4; ++p) {
    for (auto &b : bmps_[p]) release(b);
    for (auto &t : bten_[p]) release(t);
    for (auto &t : bten2_[p]) release(t);
  }
  for (void *p : {(void *)tps_, (void *)osum_, (void *)eosum_, (void *)tps_off_d_, (void *)site_size_d_, (void *)hole_off_d_,
                  (void *)cfg_, (void *)amp_, (void *)mt_, (void *)mtidx_, (void *)accepted_, (void *)eloc_, (void *)psi_tmp_,
                  (void *)psi_row_, (void *)kept_, (void *)holes_, (void *)la_.offmax, (void *)la_.done, (void *)sr_ostar_,
                  (void *)sr_cfgs_, (void *)sr_delta_, (void *)sr_eloc_, (void *)psi_list_d_, (void *)term_ia_, (void *)term_ib_, (void *)term_cw_, (void *)idx_const_, (void *)idx_flip_, (void *)psi_alt_, (void *)bond_rec_, (void *)idx_perm_,
                  (void *)(fermion_ ? gtps_ : nullptr), (void *)gtps_off_d_, (void *)gidx_[0], (void *)gidx_[1], (void *)jw_[0],
                  (void *)jw_[1], (void *)phys_par_d_, (void *)fsign_, (void *)psi_loc_, (void *)jastrow_v_, (void *)jr_, (void *)dens_d_, (void *)sr_desc2_, (void *)fs_target_d_, (void *)fs_coef_d_, (void *)site_rec_})
    be_free(p);
  for (auto &t : term_) { be_free(t.diag); be_free(t.target); be_free(t.coef); }
  be_free(pin_.diag); be_free(pin_.target); be_free(pin_.coef);
  pool_.release_all();
  planner_.release_all();
  be_ctx_destroy(bectx_);
}

void Engine::site_dims(int r, int c, int out[4]) const {
  for (int i = 0; i < 4; ++i) out[i] = site_dims_h_[(size_t)(r * cols_ + c)][(size_t)i];
}
void Engine::set_tps(const double *host) {
  be_h2d(tps_, host, sizeof(double) * tps_total_);
  if (complex_) be_memset0(tps_ + tps_total_, sizeof(double) * tps_total_);     // a real state in a complex context
  tps_loaded_ = true;
  if (fermion_) {
    dress_plane(host, gtps_);
    if (complex_) be_memset0(gtps_ + gtps_total_, sizeof(double) * gtps_total_);
  }
  touch_all();
}
// fermion mode: FERMION_VARIANTS sign patterns per site (backend.h) of one plane of the user's tensors
void Engine::dress_plane(const double *host, double *dst) {
  {
    std::vector<double> g((size_t)(tps_total_ * FERMION_VARIANTS));
    static const int vmask[FERMION_VARIANTS] = {0, 8, 4, 12, 6, 14, 0, 1};     // bits: L = 1, D = 2, R = 4, U = 8
    for (int site = 0; site < nsites_; ++site) {
      const auto &d = site_dims_h_[(size_t)site];
      const int sz = site_size_h_[(size_t)site];
      const std::vector<int32_t> *par = &leg_par_h_[(size_t)site * 4];
      for (int v = 0; v < FERMION_VARIANTS; ++v) {
        const bool vert = v >= 6;
        int e = 0;
        for (int l = 0; l < d[0]; ++l)
          for (int dd = 0; dd < d[1]; ++dd)
            for (int r = 0; r < d[2]; ++r)
              for (int u = 0; u < d[3]; ++u, ++e) {
                const int pl = par[0][(size_t)l], pd = par[1][(size_t)dd], pr = par[2][(size_t)r], pu = par[3][(size_t)u];
                int q = vert ? (pl & pd) ^ (pl & pr) ^ (pl & pu) ^ pl ^ pd : (pl & pd) ^ (pl & pr) ^ (pd & pr) ^ pl ^ pd;
                if (vmask[v] & 1) q ^= pl;
                if (vmask[v] & 2) q ^= pd;
                if (vmask[v] & 4) q ^= pr;
                if (vmask[v] & 8) q ^= pu;
                const double sg = q ? -1.0 : 1.0;
                for (int p = 0; p < phys_; ++p)
                  g[(size_t)(gtps_off_h_[(size_t)site] + ((long)v * phys_ + p) * sz + e)] =
                      sg * host[tps_off_h_[(size_t)site] + (long)p * sz + e];
              }
      }
    }
    be_h2d(dst, g.data(), sizeof(double) * g.size());
  }
}
void Engine::get_tps(double *host) { be_d2h(host, tps_, sizeof(double) * tps_total_); }
void Engine::scale_tps(double f) {
  std::vector<double> h((size_t)tps_total_ * (complex_ ? 2 : 1));
  be_d2h(h.data(), tps_, sizeof(double) * h.size());
  for (auto &x : h) x *= f;
  if (complex_) set_tps_c(h.data(), h.data() + tps_total_);
  else set_tps(h.data());
}
void Engine::set_configs(const int32_t *host) {
  // every entry is used as the physical-slice index of a gather operand: reject anything outside [0, phys)
  for (size_t i = 0; i < (size_t)W_ * nsites_; ++i)
    if (host[i] < 0 || host[i] >= phys_)
      throw std::invalid_argument("set_configs: entry " + std::to_string(host[i]) + " of walker " + std::to_string(i / nsites_) +
                                  " is outside [0, phys = " + std::to_string(phys_) + ")");
  be_h2d(cfg_, host, sizeof(int32_t) * (size_t)W_ * nsites_);
  refresh_gather();
  touch_all();
}
void Engine::get_configs(int32_t *host) { be_d2h(host, cfg_, sizeof(int32_t) * (size_t)W_ * nsites_); }
void Engine::seed_rng(const uint32_t *seeds) {
  uint32_t *d = (uint32_t *)pool_.get(sizeof(uint32_t) * W_);
  be_h2d(d, seeds, sizeof(uint32_t) * W_);
  be_mt_seed(mt_, mtidx_, d, W_);
  be_sync();
  pool_.put(d);
}
void Engine::set_rng_state(const uint32_t *mt, const int32_t *idx) {
  be_h2d(mt_, mt, sizeof(uint32_t) * (size_t)W_ * 624);
  be_h2d(mtidx_, idx, sizeof(int32_t) * W_);
}
void Engine::get_rng_state(uint32_t *mt, int32_t *idx) {
  be_d2h(mt, mt_, sizeof(uint32_t) * (size_t)W_ * 624);
  be_d2h(idx, mtidx_, sizeof(int32_t) * W_);
}
void Engine::get_amplitudes(double *host) { be_d2h(host, amp_, sizeof(double) * W_); }
void Engine::get_holes(double *host) { be_d2h(host, holes_, sizeof(double) * (size_t)W_ * hole_stride_); }
long Engine::stat(int which) const {
  switch (which) {
    case 0: return n_absorb_;
    case 1: return n_bten_;
    case 2: return n_trace_;
    case 3: return la_.jacobi_sweeps;
    case 4: return la_.jacobi_calls;
    case 5: return la_.qr_calls;
    case 6: return be_launch_count();
    case 7: return (long)pool_.total_bytes();
    case 8: return la_.rows_in;
    case 9: return la_.rows_kept;
    case 10: return la_.jacobi_rounds;
    case 11: return n_memo_hits_;
    case 12: return chain_rows_in_;
    case 13: return chain_rows_kept_;
    case 14: return la_.small_svd_calls;
    default: return -1;
  }
}

// ---------------------------------------------------------------------------------------------------
// tensors
// ---------------------------------------------------------------------------------------------------
BT Engine::alloc(std::initializer_list<int> dims) {
  BT t;
  t.rank = (int)dims.size();
  long n = 1;
  int i = 0;
  for (int d : dims) { t.d[i++] = d; n *= d; }
  t.n = n;
  t.p = (double *)pool_.get(sizeof(double) * (size_t)W_ * n * (complex_ ? 2 : 1));
  return t;
}
BT Engine::ones111() {
  BT t = alloc({1, 1, 1});
  be_fill(t.p, 1.0, W_);
  if (complex_) be_memset0(imag(t), sizeof(double) * W_);
  return t;
}
void Engine::release(BT &t) {
  if (t.p) pool_.put(t.p);
  t.p = nullptr;
}
void Engine::release(BMPSv &v) {
  for (auto &t : v) release(t);
  v.clear();
}
TRef Engine::ref(const BT &t) const {
  TRef r;
  r.op = mkop(t.p, t.n);
  if (complex_) r.opi = mkop(imag(t), t.n);
  r.rank = t.rank;
  for (int i = 0; i < t.rank; ++i) r.d[i] = t.d[i];
  return r;
}
TRef Engine::site_ref(int site, int cfg_site) const {
  TRef r;
  if (fermion_ && cfg_site != site) throw std::logic_error("fermion mode: exchanged tensors need explicit dressed slices");
  r.op = mkgather(gtps_ + gtps_off_h_[(size_t)site], (fermion_ ? gidx_[gmode_] : cfg_) + cfg_site, nsites_, site_size_h_[(size_t)site]);
  if (complex_) r.opi = mkgather(gtps_ + gtps_total_ + gtps_off_h_[(size_t)site], (fermion_ ? gidx_[gmode_] : cfg_) + cfg_site, nsites_, site_size_h_[(size_t)site]);
  r.rank = 4;
  for (int i = 0; i < 4; ++i) r.d[i] = site_dims_h_[(size_t)site][(size_t)i];
  return r;
}
template <class H>
static GettDesc with_hints(GettDesc d, const H *h) {
  if (h) {
    d.klo_m = h->klo_m; d.klo_n = h->klo_n; d.work = h->work;
    d.m_cnt = h->m_cnt; d.m_scale = h->m_scale; d.n_cnt = h->n_cnt; d.n_scale = h->n_scale;
  }
  return d;
}
TRef Engine::site_ref_idx(int site, const int32_t *idx, int stride) const {
  TRef r;
  r.op = mkgather(gtps_ + gtps_off_h_[(size_t)site], idx, stride, site_size_h_[(size_t)site]);
  if (complex_) r.opi = mkgather(gtps_ + gtps_total_ + gtps_off_h_[(size_t)site], idx, stride, site_size_h_[(size_t)site]);
  r.rank = 4;
  for (int i = 0; i < 4; ++i) r.d[i] = site_dims_h_[(size_t)site][(size_t)i];
  return r;
}
BT Engine::einsum(const std::string &spec, const TRef &a, const TRef &b, const KHints *h, bool conj_b) {
  const Plan &pl = planner_.get(spec, a.d, a.rank, b.d, b.rank);
  BT out;
  out.rank = (int)pl.outdims.size();
  for (int i = 0; i < out.rank; ++i) out.d[i] = pl.outdims[(size_t)i];
  out.n = pl.outn;
  out.p = (double *)pool_.get(sizeof(double) * (size_t)W_ * out.n * (complex_ ? 2 : 1));
  if (!complex_) {
    be_gett(with_hints(pl.d, h), a.op, b.op, mkop(out.p, out.n), 1.0, 0.0, W_, 1);
    return out;
  }
  // (ar + i ai)(br + i s bi), s = -1 for conj(b): four real products on the split planes (no structural-zero hints)
  const double sb = conj_b ? -1.0 : 1.0;
  const Operand cr = mkop(out.p, out.n), ci = mkop(imag(out), out.n);
  be_gett(pl.d, a.op, b.op, cr, 1.0, 0.0, W_, 1);
  be_gett(pl.d, a.opi, b.opi, cr, -sb, 1.0, W_, 1);
  be_gett(pl.d, a.op, b.opi, ci, sb, 0.0, W_, 1);
  be_gett(pl.d, a.opi, b.op, ci, 1.0, 1.0, W_, 1);
  return out;
}
void Engine::einsum_into(const std::string &spec, const TRef &a, const TRef &b, Operand c, const long *sc, double alpha,
                         double beta, const KHints *h, const Operand *c_im) {
  const Plan &pl = planner_.get(spec, a.d, a.rank, b.d, b.rank, nullptr, nullptr, sc);
  if (!complex_) { be_gett(with_hints(pl.d, h), a.op, b.op, c, alpha, beta, W_, 1); return; }
  if (!c_im || alpha != 1.0 || beta != 0.0) throw std::logic_error("einsum_into: this contraction is not available for complex states");
  be_gett(pl.d, a.op, b.op, c, 1.0, 0.0, W_, 1);
  be_gett(pl.d, a.opi, b.opi, c, -1.0, 1.0, W_, 1);
  be_gett(pl.d, a.op, b.opi, *c_im, 1.0, 0.0, W_, 1);
  be_gett(pl.d, a.opi, b.op, *c_im, 1.0, 1.0, W_, 1);
}
// r[k][e][a] is an R factor: r[k][col] == 0 for col = e*A + a < k. First possibly non-zero K index per row / column of
// the three contractions that consume it (K enumerations: a; (e,p) with p = `inner`; (e,a)).
const Engine::KHints &Engine::r_hints(int which, int k, int e, int a, int p, int b) {
  std::array<int, 6> key = {which, k, e, a, p, b};
  auto it = hints_.find(key);
  if (it != hints_.end()) return it->second;
  std::vector<int32_t> tab;
  int K = 0;
  if (which == 0) {                       // N = (k, e), K = a
    K = a;
    tab.resize((size_t)e * k);
    for (int ee = 0; ee < e; ++ee)
      for (int kk = 0; kk < k; ++kk) tab[(size_t)kk * e + ee] = std::min(a, std::max(0, kk - ee * a));
  } else if (which == 1) {                // M = (k, b), K = (e, p): tmp1[e][k][.][.] == 0 for e < floor(k / A)
    K = e * p;
    tab.resize((size_t)k * b);
    for (int kk = 0; kk < k; ++kk)
      for (int bb = 0; bb < b; ++bb) tab[(size_t)kk * b + bb] = std::min(K, p * (kk / a));
  } else {                                // M = k, K = (e, a)
    K = e * a;
    tab.resize((size_t)k);
    for (int kk = 0; kk < k; ++kk) tab[(size_t)kk] = std::min(K, kk);
  }
  KHints h;
  const int32_t *dev = planner_.upload(tab);
  // executed fraction at the kernel's granularity (64-wide tiles, K steps of 16)
  double done = 0.0, total = 0.0;
  for (size_t t0 = 0; t0 < tab.size(); t0 += 64) {
    int lo = K;
    for (size_t i = t0; i < std::min(tab.size(), t0 + 64); ++i) lo = std::min(lo, (int)tab[i]);
    done += K - std::min(K, lo / 16 * 16);
    total += K;
  }
  h.work = total > 0 ? done / total : 1.0;
  if (which == 0) h.klo_n = dev; else h.klo_m = dev;
  return hints_.emplace(key, h).first->second;
}
std::string Engine::site_labels(int post, char pre, char toward, char next, char away) {
  std::string s(4, '?');
  s[(size_t)((post + 3) % 4)] = pre;
  s[(size_t)post] = toward;
  s[(size_t)((post + 1) % 4)] = next;
  s[(size_t)((post + 2) % 4)] = away;
  return s;
}
std::vector<int> Engine::slice_sites(int num, int orient) const {
  std::vector<int> v;
  if (orient == HORIZONTAL) for (int c = 0; c < cols_; ++c) v.push_back(num * cols_ + c);
  else for (int r = 0; r < rows_; ++r) v.push_back(r * cols_ + num);
  return v;
}

// ---------------------------------------------------------------------------------------------------
// BMPS::MultiplyMPOSVDCompress_ (bmps_impl.h:756-862), restated as an R-chain + right-to-left truncation:
//   forward  : r_{i+1} = R factor of [r_i (x) mps_i (x) mpo_i] as a (k,o) x (f,b) matrix      (:778-850, R only)
//   backward : Theta_i = r_i . X_i with X_i = mps_i (x) mpo_i (x) E_{i+1}; the kept right singular vectors of
//              Theta_i are res[i] (= Vt of :235-238); E_i = X_i . res[i]^T carries the truncated right part
//              (the reference carries the same information as U.S absorbed into res[i-1], :251-254).
// In exact arithmetic both give the same truncated MPS up to the gauge of each kept subspace.
// ---------------------------------------------------------------------------------------------------
Engine::BMPSv Engine::absorb(const BMPSv &mps, const std::vector<int> &sites_in, int post) {
  // BMPS::MultiplyMPO (bmps_impl.h:404-437): N == 2 always takes the SVD path
  if (scheme_ != 0 && mps.size() > 2) return absorb_variational(mps, sites_in, post, scheme_ == 2);
  return absorb_svd(mps, sites_in, post);
}
// One step of the forward R chain (engine.h). A complex A is factorised through its real embedding M = [[Ar, -Ai], [Ai, Ar]]
// (2m x 2n): any real R with R^T R = M^T M gives the complex factor (R1 - i R2) / sqrt(2) (backend.h). reduce_tall = false
// hands the matrix to one CAQR whatever its height (the MPS-only chain of compress_mps, at most 2 chi D rows).
template <class Write>
Engine::ChainStep Engine::chain_step(int m_in, int n_in, Write &&write, const int32_t *rc, int o, int rk, double eps,
                                     bool reduce_tall) {
  ChainStep out;
  int m = complex_ ? 2 * m_in : m_in;
  const int n = complex_ ? 2 * n_in : n_in, kk = std::min(m, n);
  // a matrix is reduced by row chunks when it is taller than one two-stage CAQR takes and has more rows than columns
  // (the R factor of a wider one has all its rows). A matrix of more than qr_max_rows() rows that is not reduced (m <= n),
  // and the chunks of a matrix with n >= qr_max_rows(), go to qr_layout as they are, which throws above its 18 x 576
  // rows; no product shape comes near (n is at most 2 chi D, 1024 at chi = 64, D = 8).
  auto tall = [&](int rows) { return reduce_tall && rows > qr_max_rows() && rows > n; };
  QRLayout L;
  if (!tall(m)) L = qr_layout(m, n);
  else { L.m_pad = m; L.nb = 32; }                     // reduced by row chunks below
  long wsA = (long)L.m_pad * n;
  auto padded = [&] {
    double *p = (double *)pool_.get(sizeof(double) * (size_t)W_ * wsA);
    if (L.m_pad > m) be_memset0(p, sizeof(double) * (size_t)W_ * wsA);
    return p;
  };
  double *A;
  if (!complex_) {
    A = padded();
    write(mkop(A, wsA), nullptr);
  } else {
    const long wa = (long)m_in * n_in;
    double *Ar = (double *)pool_.get(sizeof(double) * (size_t)W_ * wa), *Ai = (double *)pool_.get(sizeof(double) * (size_t)W_ * wa);
    const Operand ci = mkop(Ai, wa);
    write(mkop(Ar, wa), &ci);
    A = padded();
    be_embed_complex(Ar, Ai, wa, m_in, n_in, A, wsA, W_);
    pool_.put(Ar); pool_.put(Ai);
    rc = nullptr; o = 0; rk *= 2;                      // no zero-tail hints through the embedding; its rank doubles
  }
  // Matrices taller than the two-stage CAQR takes (the real embeddings of the complex path at the headline size) are
  // reduced first: R factors of row chunks, stacked (one more tree level, R^T R unchanged). Chunks have more rows than
  // columns, so every pass shrinks the matrix (chunks of at most n rows would stack back to the same height forever).
  auto reduce = [&](double *&Ap) {
    while (tall(m)) {
      const int nchunk = (m + qr_max_rows() - 1) / qr_max_rows();
      const int chunk = std::max(round_up((m + nchunk - 1) / nchunk, 32), round_up(n + 1, 32));
      int stacked = 0;
      for (int c = 0; c * chunk < m; ++c) stacked += std::min(std::min(chunk, m - c * chunk), n);
      QRLayout Ls;
      if (!tall(stacked)) Ls = qr_layout(stacked, n);
      else { Ls.m_pad = stacked; Ls.nb = 32; }
      const long wsS = (long)Ls.m_pad * n;
      double *S = (double *)pool_.get(sizeof(double) * (size_t)W_ * wsS);
      be_memset0(S, sizeof(double) * (size_t)W_ * wsS);
      int off = 0;
      for (int c = 0; c * chunk < m; ++c) {
        const int rows_c = std::min(chunk, m - c * chunk), kkc = std::min(rows_c, n);
        QRLayout Lc = qr_layout(rows_c, n);
        const long wsC = (long)Lc.m_pad * n;
        double *buf = (double *)pool_.get(sizeof(double) * (size_t)W_ * wsC);
        if (Lc.m_pad > rows_c) be_memset0(buf, sizeof(double) * (size_t)W_ * wsC);
        be_copy2d(buf, wsC, n, Ap + (long)c * chunk * n, wsA, n, rows_c, n, W_);
        caqr(la_, buf, wsC, rows_c, n, Lc);
        be_copy2d(S + (long)off * n, wsS, n, buf, wsC, n, kkc, n, W_);
        off += kkc;
        pool_.put(buf);
      }
      pool_.put(Ap);
      Ap = S; wsA = wsS; m = stacked; L = Ls; rc = nullptr; o = 0;
    }
  };
  double *R;                                           // the factor: rows x n at R, walker stride wsR
  long wsR;
  int rows;
  const bool deflate = eps > 0.0 && kk >= 16;
  if (deflate) {
    // Rank-revealing step of the R chain. Columns sorted by norm (pivoting-lite) grade the rows of R; rows below
    // eps * (largest row norm) are dropped, a backward-stable perturbation of the left part of relative size
    // <= sqrt(rows) * eps. The exact MPO x MPS product has bond dimension D*chi, its numerical rank is a
    // fraction of that, and every later step of the chain (and Theta = r X) shrinks with it.
    double *cn2 = (double *)pool_.get(sizeof(double) * (size_t)W_ * std::max(n, kk));
    int32_t *ord = (int32_t *)pool_.get(sizeof(int32_t) * (size_t)W_ * std::max(n, kk));
    int32_t *cord = (int32_t *)pool_.get(sizeof(int32_t) * (size_t)W_ * n);
    int32_t *cnt = (int32_t *)pool_.get(sizeof(int32_t) * (size_t)W_);
    be_col_norms2(A, wsA, n, m, n, cn2, W_);
    be_rank_rows(cn2, n, 0.0, cord, cnt, W_);
    double *Ap = padded();
    be_permute_cols(A, wsA, n, m, n, cord, 1, Ap, wsA, n, W_);
    pool_.put(A);
    reduce(Ap);
    QRStop st;                                         // early termination: the rank of r_{i+1} is close to that of r_i
    st.colnorm2 = cn2; st.colorder = cord; st.eps = eps; st.first_col = std::max(0, std::min(rk, kk) - 96);
    caqr(la_, Ap, wsA, m, n, L, rc, o, &st);
    be_row_norms2(Ap, wsA, n, kk, n, cn2, W_);
    be_rank_rows(cn2, kk, eps * eps, ord, cnt, W_);
    std::vector<int32_t> ch((size_t)W_);
    be_d2h(ch.data(), cnt, sizeof(int32_t) * W_);
    rows = 1;
    for (int w = 0; w < W_; ++w) rows = std::max(rows, (int)ch[(size_t)w]);
    const int gran = kk >= 128 ? 32 : 8;               // few distinct shapes: plans, tables and pool buffers are keyed by size
    rows = std::min(kk, (rows + gran - 1) / gran * gran);
    chain_rows_in_ += kk; chain_rows_kept_ += rows;
    wsR = (long)rows * n;
    double *Rg = (double *)pool_.get(sizeof(double) * (size_t)W_ * wsR);
    be_gather_rows(Ap, wsA, n, n, kk, ord, cnt, Rg, wsR, rows, W_);
    R = (double *)pool_.get(sizeof(double) * (size_t)W_ * wsR);
    be_permute_cols(Rg, wsR, n, rows, n, cord, 0, R, wsR, n, W_);
    out.cnt = cnt;                                     // rows >= cnt[w] of the factor are zero (be_gather_rows)
    for (void *p : {(void *)cn2, (void *)ord, (void *)cord, (void *)Ap, (void *)Rg}) pool_.put(p);
  } else {
    reduce(A);
    caqr(la_, A, wsA, m, n, L, rc, o);
    R = A; wsR = wsA; rows = kk;
    out.tri = true;
  }
  if (complex_) {
    out.r = alloc({rows, n_in});
    be_split_r(R, wsR, rows, n_in, out.r.p, imag(out.r), out.r.n, W_);
    pool_.put(R);
    if (out.cnt) pool_.put(out.cnt);
    out.cnt = nullptr; out.tri = false;                // the structural-zero hints of the contractions are real-only
  } else if (!deflate) {
    out.r = alloc({rows, n});
    be_copy2d(out.r.p, out.r.n, n, R, wsR, n, rows, n, W_);
    pool_.put(R);
  } else {
    out.r.p = R; out.r.rank = 2; out.r.d[0] = rows; out.r.d[1] = n; out.r.n = wsR;
  }
  return out;
}

// One truncation step (engine.h). A complex Theta is truncated through its real embedding: the singular values come in
// exact pairs (keep 2 dmin .. 2 dmax), the kept right singular subspace is J-invariant and be_complex_basis turns its 2t
// real vectors into t complex ones (backend.h).
template <class Theta>
BT Engine::truncated_right_vectors(int rows, int cols, Theta &&theta, int dmin, int dmax, double terr) {
  constexpr bool held = std::is_same<typename std::decay<Theta>::type, BT>::value;     // a tensor, else a writer
  if (keeps_every_column(rows, cols, dmin)) {
    // nothing can be truncated and the row space is the whole space: any orthonormal basis is the same gauge class
    BT B = alloc({cols, cols});
    be_set_identity(B.p, B.n, cols, cols, W_);
    if (complex_) be_memset0(imag(B), sizeof(double) * (size_t)W_ * B.n);
    return B;
  }
  const int tcap = std::min(dmax, std::min(rows, cols));
  BT B = alloc({tcap, cols});
  if (!complex_) {
    const int brows = truncate_buffer_rows(rows, cols);
    const long ws = (long)brows * cols;
    double *G = (double *)pool_.get(sizeof(double) * (size_t)W_ * ws);
    if (brows > rows) be_memset0(G, sizeof(double) * (size_t)W_ * ws);
    if constexpr (held) be_copy2d(G, ws, cols, theta.p, theta.n, cols, rows, cols, W_);
    else theta(mkop(G, ws), nullptr);
    truncate_rows(la_, G, ws, rows, cols, dmin, dmax, terr, tcap, B.p, B.n, kept_);
    pool_.put(G);
    return B;
  }
  double *Tr, *Ti;                                     // the planes of Theta, walker stride wt
  long wt;
  if constexpr (held) {
    Tr = theta.p; Ti = imag(theta); wt = theta.n;
  } else {
    wt = (long)rows * cols;
    Tr = (double *)pool_.get(sizeof(double) * (size_t)W_ * wt); Ti = (double *)pool_.get(sizeof(double) * (size_t)W_ * wt);
    const Operand ci = mkop(Ti, wt);
    theta(mkop(Tr, wt), &ci);
  }
  const int rows2 = 2 * rows, cols2 = 2 * cols;
  const int brows2 = truncate_buffer_rows(rows2, cols2);
  const long ws2 = (long)brows2 * cols2;
  double *GM = (double *)pool_.get(sizeof(double) * (size_t)W_ * ws2);
  if (brows2 > rows2) be_memset0(GM, sizeof(double) * (size_t)W_ * ws2);
  be_embed_complex(Tr, Ti, wt, rows, cols, GM, ws2, W_);
  if constexpr (!held) { pool_.put(Tr); pool_.put(Ti); }
  const int dmax2 = (int)std::min<long>(2L * dmax, std::numeric_limits<int>::max()), dmin2 = (int)std::min<long>(2L * dmin, dmax2);
  const int tcap2 = std::min(dmax2, std::min(rows2, cols2));
  double *Bm = (double *)pool_.get(sizeof(double) * (size_t)W_ * tcap2 * cols2);
  truncate_rows(la_, GM, ws2, rows2, cols2, dmin2, dmax2, terr, tcap2, Bm, (long)tcap2 * cols2, kept_);
  be_complex_basis(Bm, (long)tcap2 * cols2, tcap2, cols, kept_, B.p, imag(B), B.n, tcap, kept_, W_);
  pool_.put(GM); pool_.put(Bm);
  return B;
}

void Engine::test_chain_step(int m, int n, const double *a_re, const double *a_im, const int32_t *row_cnt, int row_scale,
                             int rank_hint, double eps, bool reduce_tall, double *r_re, double *r_im, int *rows_out,
                             int32_t *cnt_out, int *tri_out) {
  BT A = alloc({m, n});
  be_h2d(A.p, a_re, sizeof(double) * (size_t)W_ * A.n);
  if (complex_) be_h2d(imag(A), a_im, sizeof(double) * (size_t)W_ * A.n);
  int32_t *rc = nullptr;
  if (row_cnt) {
    rc = (int32_t *)pool_.get(sizeof(int32_t) * (size_t)W_);
    be_h2d(rc, row_cnt, sizeof(int32_t) * (size_t)W_);
  }
  ChainStep cs = chain_step(m, n, [&](Operand c, const Operand *c_im) {
    be_copy2d(c.p, c.ws, n, A.p, A.n, n, m, n, W_);
    if (c_im) be_copy2d(c_im->p, c_im->ws, n, imag(A), A.n, n, m, n, W_);
  }, rc, row_scale, rank_hint, eps, reduce_tall);
  const int rows = cs.r.d[0], cap = complex_ ? std::min(2 * m, 2 * n) : std::min(m, n);
  std::vector<double> h((size_t)W_ * cs.r.n);
  for (int pl = 0; pl < (complex_ ? 2 : 1); ++pl) {
    double *out = pl ? r_im : r_re;
    be_d2h(h.data(), pl ? imag(cs.r) : cs.r.p, sizeof(double) * h.size());
    std::fill(out, out + (size_t)W_ * cap * n, 0.0);
    for (int w = 0; w < W_; ++w)
      std::copy(h.begin() + (long)w * cs.r.n, h.begin() + (long)w * cs.r.n + (long)rows * n, out + (size_t)w * cap * n);
  }
  *rows_out = rows;
  *tri_out = cs.tri ? 1 : 0;
  if (cs.cnt) be_d2h(cnt_out, cs.cnt, sizeof(int32_t) * (size_t)W_);
  else std::fill(cnt_out, cnt_out + W_, rows);
  release(cs.r);
  release(A);
  pool_.put(cs.cnt);
  pool_.put(rc);
}

void Engine::test_truncated_right_vectors(int rows, int cols, const double *th_re, const double *th_im, int dmin, int dmax,
                                          double terr, bool held, double *b_re, double *b_im, int32_t *kept_out) {
  BT T = alloc({rows, cols});
  be_h2d(T.p, th_re, sizeof(double) * (size_t)W_ * T.n);
  if (complex_) be_h2d(imag(T), th_im, sizeof(double) * (size_t)W_ * T.n);
  BT B = held ? truncated_right_vectors(rows, cols, T, dmin, dmax, terr)
              : truncated_right_vectors(rows, cols, [&](Operand c, const Operand *c_im) {
                  be_copy2d(c.p, c.ws, cols, T.p, T.n, cols, rows, cols, W_);
                  if (c_im) be_copy2d(c_im->p, c_im->ws, cols, imag(T), T.n, cols, rows, cols, W_);
                }, dmin, dmax, terr);
  be_d2h(b_re, B.p, sizeof(double) * (size_t)W_ * B.n);
  if (complex_) be_d2h(b_im, imag(B), sizeof(double) * (size_t)W_ * B.n);
  if (keeps_every_column(rows, cols, dmin)) std::fill(kept_out, kept_out + W_, cols);     // the shortcut does not write kept_
  else be_d2h(kept_out, kept_, sizeof(int32_t) * (size_t)W_);
  release(B);
  release(T);
}

Engine::BMPSv Engine::absorb_svd(const BMPSv &mps, const std::vector<int> &sites_in, int post) {
  ++n_absorb_;
  const int N = (int)mps.size();
  std::vector<int> sites(sites_in);
  if (post == RIGHT || post == UP) std::reverse(sites.begin(), sites.end());      // bmps_impl.h:694-699
  const std::string sl = site_labels(post, 'e', 'p', 'f', 'o');
  auto sdim = [&](int site, char l) { return site_dims_h_[(size_t)site][sl.find(l)]; };
  std::vector<BT> r((size_t)N);
  std::vector<char> r_tri((size_t)N, 0);     // r_i is an upper-trapezoidal R factor (structural-zero hints apply)
  // per-walker number of non-zero rows of r_i (device, null = all rows): rows beyond it are exact zeros, so the row blocks
  // / tiles they fill are skipped per walker in the next chain step (the buffers are sized by the batch maximum)
  std::vector<int32_t *> r_cnt((size_t)N, nullptr);
  r[0] = ones111();
  for (int i = 0; i < N - 1; ++i) {
    const int site = sites[(size_t)i];
    TRef sref = tn_site(site);
    const bool tri = r_tri[(size_t)i] != 0;
    const int rk = r[(size_t)i].d[0], re = r[(size_t)i].d[1], ra = r[(size_t)i].d[2];
    const int pd = mps[(size_t)i].d[1], bd = mps[(size_t)i].d[2];
    const int32_t *rc = r_cnt[(size_t)i];
    KHints h1, h2;
    if (tri) { h1 = r_hints(0, rk, re, ra, pd, bd); h2 = r_hints(1, rk, re, ra, pd, bd); }
    if (rc) { h1.n_cnt = rc; h1.n_scale = re; h2.m_cnt = rc; h2.m_scale = bd; }
    BT tmp1 = einsum("apb,kea->kepb", ref(mps[(size_t)i]), ref(r[(size_t)i]), (tri || rc) ? &h1 : nullptr);   // bmps_impl.h:806
    const int k = r[(size_t)i].d[0], o = sdim(site, 'o'), f = sdim(site, 'f'), b = mps[(size_t)i].d[2];
    ChainStep cs = chain_step(k * o, f * b, [&](Operand c, const Operand *c_im) {
      einsum_into("kepb," + sl + "->kofb", ref(tmp1), sref, c, nullptr, 1.0, 0.0, (tri || rc) ? &h2 : nullptr, c_im);   // bmps_impl.h:807
      release(tmp1);
    }, rc, o, rk, chain_eps_, true);                                                        // bmps_impl.h:817-821
    BT &rn = r[(size_t)i + 1] = cs.r;
    rn.rank = 3; rn.d[1] = f; rn.d[2] = b;
    r_cnt[(size_t)i + 1] = cs.cnt;
    r_tri[(size_t)i + 1] = cs.tri ? 1 : 0;
  }
  BMPSv res((size_t)N);
  BT E = ones111();                                                                      // E[f,b,j]
  for (int i = N - 1; i >= 1; --i) {                                                     // bmps_impl.h:853-857
    const int site = sites[(size_t)i];
    BT Y = einsum("apb,fbj->apfj", ref(mps[(size_t)i]), ref(E));
    BT X = einsum("apfj," + sl + "->eaoj", ref(Y), tn_site(site));
    release(Y);
    const bool tri = r_tri[(size_t)i] != 0;
    const int32_t *rc = r_cnt[(size_t)i];
    BT B = truncated_right_vectors(r[(size_t)i].d[0], X.d[2] * X.d[3], [&](Operand c, const Operand *c_im) {
      KHints h3;
      if (tri) h3 = r_hints(2, r[(size_t)i].d[0], r[(size_t)i].d[1], r[(size_t)i].d[2], 0, 0);
      if (rc) { h3.m_cnt = rc; h3.m_scale = 1; }
      einsum_into("kea,eaoj->koj", ref(r[(size_t)i]), ref(X), c, nullptr, 1.0, 0.0, (tri || rc) ? &h3 : nullptr, c_im);
    }, dmin_, dmax_, terr_);
    B.rank = 3; B.d[1] = X.d[2]; B.d[2] = X.d[3];
    BT En = einsum("eaoj,toj->eat", ref(X), ref(B), nullptr, /*conj_b=*/true);     // U S = Theta Vt^H (bmps_impl.h:251-254)
    release(X);
    release(E);
    E = En;
    res[(size_t)i] = B;
  }
  {
    const int site = sites[0];
    BT Y = einsum("apb,fbj->apfj", ref(mps[0]), ref(E));
    BT X = einsum("apfj," + sl + "->eaoj", ref(Y), tn_site(site));
    release(Y);
    release(E);
    BT first = X;                   // (e=1, a=1, o, j) viewed as (1, o, j)
    first.rank = 3;
    first.d[0] = 1; first.d[1] = X.d[2]; first.d[2] = X.d[3];
    res[0] = first;
  }
  for (auto &t : r) release(t);
  for (int32_t *c : r_cnt) if (c) pool_.put(c);
  return res;
}

// ---------------------------------------------------------------------------------------------------
// variational compression: BMPS::MultiplyMPO2SiteVariationalCompress_ / 1Site (bmps_impl.h:864-995 / 997-1172)
// ---------------------------------------------------------------------------------------------------
// The bond-dimension reduction of MakeVariationalInitGuess_ (bmps_impl.h:1197-1201: Centralize(N-1) + RightCanonicalize-
// Truncate(i, dmin, dmax, terr) for i = N-1..1), restated like absorb_svd: forward R chain, backward truncation.
Engine::BMPSv Engine::compress_mps(const BMPSv &mps, int dmin, int dmax, double terr) {
  const int N = (int)mps.size();
  std::vector<BT> r((size_t)N);
  r[0] = alloc({1, 1});
  be_fill(r[0].p, 1.0, W_);
  if (complex_) be_memset0(imag(r[0]), sizeof(double) * W_);
  for (int i = 0; i < N - 1; ++i) {
    r[(size_t)i + 1] = chain_step(r[(size_t)i].d[0] * mps[(size_t)i].d[1], mps[(size_t)i].d[2], [&](Operand c, const Operand *c_im) {
      einsum_into("ka,apb->kpb", ref(r[(size_t)i]), ref(mps[(size_t)i]), c, nullptr, 1.0, 0.0, nullptr, c_im);
    }, nullptr, 0, 0, 0.0, false).r;
  }
  BMPSv res((size_t)N);
  BT E = alloc({1, 1});
  be_fill(E.p, 1.0, W_);
  if (complex_) be_memset0(imag(E), sizeof(double) * W_);
  for (int i = N - 1; i >= 1; --i) {
    BT X = einsum("apb,bj->apj", ref(mps[(size_t)i]), ref(E));
    BT B = truncated_right_vectors(r[(size_t)i].d[0], X.d[1] * X.d[2], [&](Operand c, const Operand *c_im) {
      einsum_into("ka,apj->kpj", ref(r[(size_t)i]), ref(X), c, nullptr, 1.0, 0.0, nullptr, c_im);
    }, dmin, dmax, terr);
    B.rank = 3; B.d[1] = X.d[1]; B.d[2] = X.d[2];
    BT En = einsum("apj,tpj->at", ref(X), ref(B), nullptr, /*conj_b=*/true);       // U S = Theta Vt^H
    release(X); release(E);
    E = En;
    res[(size_t)i] = B;
  }
  res[0] = einsum("apb,bj->apj", ref(mps[0]), ref(E));
  release(E);
  for (auto &t : r) release(t);
  return res;
}
Engine::BMPSv Engine::absorb_variational(const BMPSv &mps, const std::vector<int> &sites_in, int post, bool one_site) {
  const int N = (int)mps.size();
  std::vector<int> sites(sites_in);
  if (post == RIGHT || post == UP) std::reverse(sites.begin(), sites.end());
  const std::string sli = site_labels(post, 'e', 'p', 'f', 'o'), slj = site_labels(post, 'f', 'q', 'g', 'u');
  // initial guess (:1176-1212): the boundary reduced to bond dimension <= 2, multiplied with SVD compression
  BMPSv small = compress_mps(mps, 1, 2, 0.0);
  const int dmin0 = dmin_, dmax0 = dmax_; const double terr0 = terr_;
  if (one_site) { dmin_ = dmax_; terr_ = 0.0; }
  BMPSv res = absorb_svd(small, sites_in, post);
  dmin_ = dmin0; dmax_ = dmax0; terr_ = terr0;
  release(small);
  std::vector<BT> lenvs, renvs;
  lenvs.push_back(ones111());
  renvs.push_back(ones111());
  auto right2 = [&](int j, const BT &renv) {              // R2[f,b,u,j] = mps_j . renv . site_j   (:896-897)
    BT r1 = einsum("bqc,cgj->bqgj", ref(mps[(size_t)j]), ref(renv));
    BT r2 = einsum("bqgj," + slj + "->fbuj", ref(r1), tn_site(sites[(size_t)j]));
    release(r1);
    return r2;
  };
  auto left2 = [&](int i2, const BT &lenv) {              // L2[k,o,f,b] = lenv . mps_i . site_i    (:893-894)
    BT l1 = einsum("kea,apb->kepb", ref(lenv), ref(mps[(size_t)i2]));
    BT l2 = einsum("kepb," + sli + "->kofb", ref(l1), tn_site(sites[(size_t)i2]));
    release(l1);
    return l2;
  };
  for (int i = N - 1; i > 1; --i) {                       // GrowRightEnvironments_ (:731-743)
    BT r2 = right2(i, renvs.back());
    renvs.push_back(einsum("fbuj,tuj->bft", ref(r2), ref(res[(size_t)i]), nullptr, /*conj_b=*/true));   // res_dag (:885)
    release(r2);
  }
  // per-row squared norms of a batched (rows x nc) matrix view, complex: |re|^2 + |im|^2
  auto row_norms2 = [&](const BT &x, int rows, int nc, std::vector<double> &h) {
    double *n2 = (double *)pool_.get(sizeof(double) * (size_t)W_ * rows);
    h.assign((size_t)W_ * rows, 0.0);
    be_row_norms2(x.p, x.n, nc, rows, nc, n2, W_);
    be_d2h(h.data(), n2, sizeof(double) * h.size());
    if (complex_) {
      std::vector<double> hi(h.size());
      be_row_norms2(imag(x), x.n, nc, rows, nc, n2, W_);
      be_d2h(hi.data(), n2, sizeof(double) * hi.size());
      for (size_t q = 0; q < h.size(); ++q) h[q] += hi[q];
    }
    pool_.put(n2);
  };
  // one two-site sweep; returns the batch maximum of sum |s - s_last| / s_0 over the last bond when `track`
  std::vector<double> s_last;                             // [W][t] singular values of the last bond of the previous sweep
  int s_last_t = -1;
  auto sweep_two_site = [&](int d0, int d1, bool track) -> double {
    for (int i = 0; i < N - 2; ++i) {                     // res[i] = U (:891-918)
      BT l2 = left2(i, lenvs.back()), r2 = right2(i + 1, renvs.back());
      BT thT = einsum("kofb,fbuj->ujko", ref(l2), ref(r2));
      BT U = truncated_right_vectors(thT.d[0] * thT.d[1], thT.d[2] * thT.d[3], thT, d0, d1, terr_);
      BT Ut = U; Ut.rank = 3; Ut.d[0] = U.d[0]; Ut.d[1] = l2.d[0]; Ut.d[2] = l2.d[1];     // (t, k, o)
      lenvs.push_back(einsum("kofb,tko->tfb", ref(l2), ref(Ut), nullptr, /*conj_b=*/true));
      release(thT); release(l2); release(r2); release(U);
      release(renvs.back()); renvs.pop_back();
    }
    double diff = 0.0;
    for (int i = N - 2; i > 0; --i) {                     // res[i+1] = Vt (:920-947)
      BT l2 = left2(i, lenvs.back()), r2 = right2(i + 1, renvs.back());
      BT th = einsum("kofb,fbuj->kouj", ref(l2), ref(r2));
      BT V = truncated_right_vectors(th.d[0] * th.d[1], th.d[2] * th.d[3], th, d0, d1, terr_);
      BT Vt = V; Vt.rank = 3; Vt.d[0] = V.d[0]; Vt.d[1] = r2.d[2]; Vt.d[2] = r2.d[3];      // (t, u, j)
      if (track && i == 1) {                              // singular values of this bond: column norms of theta V^T
        BT us = einsum("kouj,tuj->tko", ref(th), ref(Vt), nullptr, /*conj_b=*/true);
        const int t = us.d[0], nc = us.d[1] * us.d[2];
        std::vector<double> h;
        row_norms2(us, t, nc, h);
        release(us);
        for (auto &x : h) x = std::sqrt(x);
        if (s_last_t == t) {
          for (int w = 0; w < W_; ++w) {
            double d = 0.0;
            for (int q = 0; q < t; ++q) d += std::fabs(h[(size_t)w * t + q] - s_last[(size_t)w * t + q]);
            diff = std::max(diff, d / h[(size_t)w * t]);
          }
        } else {
          diff = std::numeric_limits<double>::infinity();
        }
        s_last = h; s_last_t = t;
      }
      release(res[(size_t)i + 1]);
      res[(size_t)i + 1] = Vt;
      renvs.push_back(einsum("fbuj,tuj->bft", ref(r2), ref(Vt), nullptr, /*conj_b=*/true));
      release(th); release(l2); release(r2);
      release(lenvs.back()); lenvs.pop_back();
    }
    return diff;
  };
  auto finish_two_site = [&](bool keep_renv) {            // sites 0, 1: res[0] = U S, res[1] = Vt (:963-988)
    BT l2 = left2(0, lenvs.back()), r2 = right2(1, renvs.back());
    BT th = einsum("kofb,fbuj->kouj", ref(l2), ref(r2));
    BT V = truncated_right_vectors(th.d[0] * th.d[1], th.d[2] * th.d[3], th, dmin_, dmax_, terr_);
    BT Vt = V; Vt.rank = 3; Vt.d[0] = V.d[0]; Vt.d[1] = r2.d[2]; Vt.d[2] = r2.d[3];
    release(res[0]); release(res[1]);
    res[0] = einsum("kouj,tuj->kot", ref(th), ref(Vt), nullptr, /*conj_b=*/true);      // U S = theta Vt^H
    res[1] = Vt;
    if (keep_renv) renvs.push_back(einsum("fbuj,tuj->bft", ref(r2), ref(Vt), nullptr, /*conj_b=*/true));       // :1108-1110
    release(th); release(l2); release(r2);
  };
  if (!one_site) {
    for (int it = 0; it < var_iter_; ++it) {
      const double diff = sweep_two_site(dmin_, dmax_, true);
      if (it > 0 && diff < var_tol_) break;              // every walker converged (:949-960)
    }
    finish_two_site(false);
  } else {
    sweep_two_site(dmax_, dmax_, false);                  // fixes the bond dimensions at D_max (:1021-1085)
    finish_two_site(true);
    double last = 0.0;
    for (int it = 0; it < var_iter_; ++it) {
      for (int i = 0; i < N - 1; ++i) {                   // res[i] = Q of (L2 . renv) (:1116-1131); any orthonormal basis of
        BT l2 = left2(i, lenvs.back());                   // the same column space is the same MPS up to the bond gauge
        BT aT = einsum("kofb,bft->tko", ref(l2), ref(renvs.back()));
        const int t = aT.d[0], nc = aT.d[1] * aT.d[2];
        BT Q = truncated_right_vectors(t, nc, aT, std::min(t, nc), std::min(t, nc), 0.0);
        BT Qt = Q; Qt.rank = 3; Qt.d[0] = Q.d[0]; Qt.d[1] = l2.d[0]; Qt.d[2] = l2.d[1];  // (t', k, o)
        lenvs.push_back(einsum("kofb,tko->tfb", ref(l2), ref(Qt), nullptr, /*conj_b=*/true));
        release(aT); release(l2); release(Q);
        release(renvs.back()); renvs.pop_back();
      }
      double r_norm = 0.0;
      for (int i = N - 1; i > 0; --i) {                   // :1133-1151
        BT r2 = right2(i, renvs.back());
        BT a = einsum("fbuj,kfb->kuj", ref(r2), ref(lenvs.back()));
        const int k = a.d[0], nc = a.d[1] * a.d[2];
        if (i == 1) {                                     // r.Get2Norm() of the last QR = |a|_F, batch maximum of the change
          std::vector<double> h;
          row_norms2(a, k, nc, h);
          for (int w = 0; w < W_; ++w) { double s2 = 0; for (int q = 0; q < k; ++q) s2 += h[(size_t)w * k + q]; r_norm = std::max(r_norm, std::sqrt(s2)); }
        }
        BT Q = truncated_right_vectors(k, nc, a, std::min(k, nc), std::min(k, nc), 0.0);
        BT Qt = Q; Qt.rank = 3; Qt.d[0] = Q.d[0]; Qt.d[1] = r2.d[2]; Qt.d[2] = r2.d[3];     // (t, u, j)
        release(res[(size_t)i]);
        res[(size_t)i] = Qt;
        renvs.push_back(einsum("fbuj,tuj->bft", ref(r2), ref(Qt), nullptr, /*conj_b=*/true));
        release(a); release(r2);
        release(lenvs.back()); lenvs.pop_back();
      }
      if (it > 0 && std::fabs(r_norm - last) / std::fabs(r_norm) <= var_tol_) break;
      last = r_norm;
    }
    BT l2 = left2(0, lenvs.back());                       // :1161-1166
    release(res[0]);
    res[0] = einsum("kofb,bft->kot", ref(l2), ref(renvs.back()));
    release(l2);
  }
  for (auto &t : lenvs) release(t);
  for (auto &t : renvs) release(t);
  ++n_absorb_;
  return res;
}

// ---------------------------------------------------------------------------------------------------
// contractor
// ---------------------------------------------------------------------------------------------------
void Engine::contractor_init() {                       // impl/bmps_contractor_init.h:25-70
  for (int p = 0; p < 4; ++p) {
    for (auto &b : bmps_[p]) release(b);
    bmps_[p].clear();
    for (auto &m : memo_[p]) release(m.second.v);
    memo_[p].clear();
    stamp_[p].assign(1, 1);                            // the vacuum BMPS depends on nothing
    for (auto &t : bten_[p]) release(t);
    bten_[p].clear();
    for (auto &t : bten2_[p]) release(t);
    bten2_[p].clear();
    int n = (p == UP || p == DOWN) ? cols_ : rows_;
    BMPSv vac;
    for (int i = 0; i < n; ++i) vac.push_back(ones111());
    bmps_[p].push_back(vac);
  }
}
const Engine::BMPSv &Engine::bmps_at_slice(int pos, int logical) const {   // bmps_contractor.h:985-999
  if (pos == DOWN) return bmps_[DOWN].at((size_t)(rows_ - 1 - logical));
  if (pos == RIGHT) return bmps_[RIGHT].at((size_t)(cols_ - 1 - logical));
  return bmps_[pos].at((size_t)logical);
}
const BT &Engine::bten_at_slice(int pos, int logical) const {              // bmps_contractor.h:1001-1009
  if (pos == DOWN) return bten_[DOWN].at((size_t)(rows_ - 1 - logical));
  if (pos == RIGHT) return bten_[RIGHT].at((size_t)(cols_ - 1 - logical));
  return bten_[pos].at((size_t)logical);
}
bool Engine::slices_unchanged_since(int pos, int k, long stamp) const {
  // bmps_[pos][k] depends on: UP rows [0,k), DOWN rows [rows-k,rows), LEFT cols [0,k), RIGHT cols [cols-k,cols)
  if (stamp <= 0) return false;
  for (int i = 0; i < k; ++i) {
    long mod = pos == UP ? row_mod_[(size_t)i] : pos == DOWN ? row_mod_[(size_t)(rows_ - 1 - i)]
             : pos == LEFT ? col_mod_[(size_t)i] : col_mod_[(size_t)(cols_ - 1 - i)];
    if (mod > stamp) return false;
  }
  return true;
}
void Engine::touch_site(int site) {
  ++epoch_;
  row_mod_[(size_t)(site / cols_)] = epoch_;
  col_mod_[(size_t)(site % cols_)] = epoch_;
}
void Engine::touch_all() {
  ++epoch_;
  std::fill(row_mod_.begin(), row_mod_.end(), epoch_);
  std::fill(col_mod_.begin(), col_mod_.end(), epoch_);
  purge_memo();
}
void Engine::purge_memo() {
  for (int p = 0; p < 4; ++p)
    for (auto it = memo_[p].begin(); it != memo_[p].end();) {
      if (slices_unchanged_since(p, it->first, it->second.stamp)) { ++it; continue; }
      release(it->second.v);
      it = memo_[p].erase(it);
    }
}
void Engine::push_grown(int pos, int mpo_num, int orient) {
  mode_for_bmps(pos);
  const int k = (int)bmps_[pos].size();
  auto it = memo_[pos].find(k);
  if (it != memo_[pos].end()) {
    const bool ok = slices_unchanged_since(pos, k, it->second.stamp);
    if (ok) {
      bmps_[pos].push_back(std::move(it->second.v));
      stamp_[pos].push_back(it->second.stamp);
      ++n_memo_hits_;
    } else {
      release(it->second.v);
    }
    memo_[pos].erase(it);
    if (ok) return;
  }
  const bool pred_ok = k == 1 || slices_unchanged_since(pos, k - 1, stamp_[pos].back());
  bmps_[pos].push_back(absorb(bmps_[pos].back(), slice_sites(mpo_num, orient), pos));
  stamp_[pos].push_back(pred_ok ? epoch_ : 0);
}
void Engine::grow_bmps_step(int pos) {                 // grow.h:32-48
  int existed = (int)bmps_[pos].size();
  int mpo_num = (pos == UP || pos == LEFT) ? existed - 1 : (pos == DOWN ? rows_ - existed : cols_ - existed);
  int orient = (pos == UP || pos == DOWN) ? HORIZONTAL : VERTICAL;
  push_grown(pos, mpo_num, orient);
}
void Engine::grow_full_bmps(int pos) {                 // grow.h:50-86
  int existed = (int)bmps_[pos].size();
  if (pos == DOWN) for (int row = rows_ - existed; row > 0; --row) push_grown(pos, row, HORIZONTAL);
  else if (pos == UP) for (int row = existed - 1; row < rows_ - 1; ++row) push_grown(pos, row, HORIZONTAL);
  else if (pos == LEFT) for (int col = existed - 1; col < cols_ - 1; ++col) push_grown(pos, col, VERTICAL);
  else for (int col = cols_ - existed; col > 0; --col) push_grown(pos, col, VERTICAL);
}
void Engine::park_or_release_top(int pos) {
  const int k = (int)bmps_[pos].size() - 1;
  if (memo_on_ && slices_unchanged_since(pos, k, stamp_[pos].back())) {
    auto it = memo_[pos].find(k);
    if (it != memo_[pos].end()) { release(it->second.v); memo_[pos].erase(it); }
    memo_[pos].emplace(k, Memo{std::move(bmps_[pos].back()), stamp_[pos].back()});
  } else {
    release(bmps_[pos].back());
  }
  bmps_[pos].pop_back();
  stamp_[pos].pop_back();
}
void Engine::delete_inner_bmps(int pos) {              // bmps_contractor.h:320-324
  while (bmps_[pos].size() > 1) park_or_release_top(pos);
  purge_memo();
}
void Engine::grow_bmps_for_row(int row) {              // grow.h:88-104
  for (int rb = rows_ - (int)bmps_[DOWN].size(); rb > row; --rb) push_grown(DOWN, rb, HORIZONTAL);
  for (int rb = (int)bmps_[UP].size() - 1; rb < row; ++rb) push_grown(UP, rb, HORIZONTAL);
}
void Engine::grow_bmps_for_col(int col) {              // grow.h:106-122
  for (int cb = cols_ - (int)bmps_[RIGHT].size(); cb > col; --cb) push_grown(RIGHT, cb, VERTICAL);
  for (int cb = (int)bmps_[LEFT].size() - 1; cb < col; ++cb) push_grown(LEFT, cb, VERTICAL);
}
void Engine::shift_bmps_window(int pos) {              // grow.h:143-148
  park_or_release_top(pos);
  grow_bmps_step(opposite(pos));
}
void Engine::init_bten(int pos) {                      // init.h:72-120
  for (auto &t : bten_[pos]) release(t);
  bten_[pos].clear();
  bten_[pos].push_back(ones111());
}
BT Engine::bten_step(const BT &bten, const BT &mps1, const TRef &site, const BT &mps2, int post) {   // grow.h:577-579
  ++n_bten_;
  const std::string sl = site_labels(post, 'p', 'y', 'f', 'o');
  BT tmp1 = einsum("apx,xyz->apyz", ref(mps1), ref(bten));
  BT tmp2 = einsum("apyz," + sl + "->zafo", ref(tmp1), site);
  release(tmp1);
  BT out = einsum("zafo,zfb->aob", ref(tmp2), ref(mps2));
  release(tmp2);
  return out;
}
void Engine::bten_operands(int post, int slice, int bten_size, const BT *&mps1, const BT *&mps2, int &site) const {
  const int pre_post = (post + 3) % 4, next_post = (post + 1) % 4;
  const int n = (post == LEFT || post == RIGHT) ? cols_ : rows_;
  mps1 = &bmps_at_slice(pre_post, slice).at((size_t)(n - bten_size));
  mps2 = &bmps_at_slice(next_post, slice).at((size_t)(bten_size - 1));
  if (post == LEFT) site = slice * cols_ + (bten_size - 1);
  else if (post == RIGHT) site = slice * cols_ + (n - bten_size);
  else if (post == UP) site = (bten_size - 1) * cols_ + slice;
  else site = (n - bten_size) * cols_ + slice;
}
void Engine::grow_full_bten(int pos, int slice, int remain, bool init) {     // grow.h:243-373
  if (init) init_bten(pos);
  mode_for_bten(pos);
  const int n = (pos == LEFT || pos == RIGHT) ? cols_ : rows_;
  for (int i = (int)bten_[pos].size() - 1; i < n - remain; ++i) {
    const BT *m1, *m2; int site;
    bten_operands(pos, slice, i + 1, m1, m2, site);
    bten_[pos].push_back(bten_step(bten_[pos].back(), *m1, tn_site(site), *m2, pos));
  }
}
void Engine::grow_bten_step(int post) {                // grow.h:529-582
  mode_for_bten(post);
  int slice = (post == LEFT || post == RIGHT) ? (int)bmps_[UP].size() - 1 : (int)bmps_[LEFT].size() - 1;
  const BT *m1, *m2; int site;
  bten_operands(post, slice, (int)bten_[post].size(), m1, m2, site);
  bten_[post].push_back(bten_step(bten_[post].back(), *m1, tn_site(site), *m2, post));
}
void Engine::shift_bten_window(int pos) {              // grow.h:517-521
  release(bten_[pos].back());
  bten_[pos].pop_back();
  grow_bten_step(opposite(pos));
}
void Engine::nn_trace(int ra, int ca, int rb, int cb, int orient, int cfg_site_a, int cfg_site_b, double *psi_out) {
  ++n_trace_;                                          // trace.h:90-205
  gmode_ = orient;
  int first, second, slice, ia, ib, n;
  if (orient == HORIZONTAL) { first = LEFT; second = RIGHT; slice = ra; ia = ca; ib = cb; n = cols_; }
  else { first = UP; second = DOWN; slice = ca; ia = ra; ib = rb; n = rows_; }
  const BT *m1, *m2; int site;
  bten_operands(first, slice, ia + 1, m1, m2, site);
  BT half_a = bten_step(bten_[first].at((size_t)ia), *m1, site_ref(ra * cols_ + ca, cfg_site_a), *m2, first);
  bten_operands(second, slice, n - ib, m1, m2, site);
  BT half_b = bten_step(bten_at_slice(second, ib), *m1, site_ref(rb * cols_ + cb, cfg_site_b), *m2, second);
  reverse_dot(half_a, half_b, psi_out);             // Contract(tmp2,{0,1,2}, tmp5,{2,1,0})  trace.h:202
  release(half_a);
  release(half_b);
}
void Engine::nn_trace_idx(int ra, int ca, int rb, int cb, int orient, const int32_t *idx_a, const int32_t *idx_b, int stride,
                          double *psi_out) {
  ++n_trace_;
  int first, second, slice, ia, ib, n;
  if (orient == HORIZONTAL) { first = LEFT; second = RIGHT; slice = ra; ia = ca; ib = cb; n = cols_; }
  else { first = UP; second = DOWN; slice = ca; ia = ra; ib = rb; n = rows_; }
  const BT *m1, *m2; int site;
  bten_operands(first, slice, ia + 1, m1, m2, site);
  BT half_a = bten_step(bten_[first].at((size_t)ia), *m1, site_ref_idx(ra * cols_ + ca, idx_a, stride), *m2, first);
  bten_operands(second, slice, n - ib, m1, m2, site);
  BT half_b = bten_step(bten_at_slice(second, ib), *m1, site_ref_idx(rb * cols_ + cb, idx_b, stride), *m2, second);
  reverse_dot(half_a, half_b, psi_out);
  release(half_a);
  release(half_b);
}
void Engine::tnn_trace_idx(int r, int c, int orient, const int32_t *idx0, const int32_t *idx1, const int32_t *idx2, int stride,
                           double *psi_out) {                                                     // trace.h:326-420
  ++n_trace_;
  const int first = orient == HORIZONTAL ? LEFT : UP, second = opposite(first);
  const int slice = orient == HORIZONTAL ? r : c, i0 = orient == HORIZONTAL ? c : r;
  const int32_t *idx[3] = {idx0, idx1, idx2};
  BT cur;
  for (int step = 0; step < 3; ++step) {
    const BT *m1, *m2; int site;
    bten_operands(first, slice, i0 + step + 1, m1, m2, site);
    BT nxt = bten_step(step == 0 ? bten_[first].at((size_t)i0) : cur, *m1, site_ref_idx(site, idx[step], stride), *m2, first);
    if (step > 0) release(cur);
    cur = nxt;
  }
  reverse_dot(cur, bten_at_slice(second, i0 + 2), psi_out);
  release(cur);
}
void Engine::probe_tnn_trace(int r, int c, int orient, const int32_t *cfg3_host, double *psi_host) {
  int32_t *d = (int32_t *)pool_.get(sizeof(int32_t) * (size_t)W_ * 3);
  be_h2d(d, cfg3_host, sizeof(int32_t) * (size_t)W_ * 3);
  if (orient == HORIZONTAL) {
    grow_bmps_for_row(r);
    init_bten(LEFT);
    for (int k = 0; k < c; ++k) grow_bten_step(LEFT);
    grow_full_bten(RIGHT, r, c + 3, true);
  } else {
    grow_bmps_for_col(c);
    init_bten(UP);
    for (int k = 0; k < r; ++k) grow_bten_step(UP);
    grow_full_bten(DOWN, c, r + 3, true);
  }
  tnn_trace_idx(r, c, orient, d, d + 1, d + 2, 3, psi_tmp_);
  be_d2h(psi_host, psi_tmp_, sizeof(double) * sw());
  pool_.put(d);
}
void Engine::one_site_trace(int r, int c, const int32_t *idx, int stride, double *psi_out) {     // trace.h:30-88
  ++n_trace_;
  const BT *m1, *m2; int site;
  bten_operands(LEFT, r, c + 1, m1, m2, site);
  BT half = bten_step(bten_[LEFT].at((size_t)c), *m1, site_ref_idx(r * cols_ + c, idx, stride), *m2, LEFT);
  reverse_dot(half, bten_at_slice(RIGHT, c), psi_out);
  release(half);
}
// out[w] = sum over all indices of a[i0,i1,...] * b[...,i1,i0] (b has the reversed leg order of a)
void Engine::reverse_dot(const BT &a, const BT &b, double *out) {
  const long n = a.n;
  // index tables depend on the shape only: built once per shape
  std::array<int, 7> key = {a.rank, a.d[0], a.d[1], a.d[2], a.d[3], a.d[4], a.d[5]};
  auto it = rdot_tabs_.find(key);
  if (it == rdot_tabs_.end()) {
    std::vector<int32_t> ak((size_t)n), bk((size_t)n);
    std::vector<long> bstride((size_t)a.rank);
    {
      // b dims are a's reversed: b index order (i_{r-1}, ..., i_0); stride of i_k in b
      long acc = 1;
      for (int k = 0; k < a.rank; ++k) { bstride[(size_t)k] = acc; acc *= a.d[k]; }
    }
    for (long k = 0; k < n; ++k) {
      long rem = k, off = 0;
      for (int ax = a.rank - 1; ax >= 0; --ax) {
        long idx = rem % a.d[ax];
        rem /= a.d[ax];
        off += idx * bstride[(size_t)ax];
      }
      ak[(size_t)k] = (int32_t)k;
      bk[(size_t)k] = (int32_t)off;
    }
    it = rdot_tabs_.emplace(key, std::make_pair(planner_.upload(ak), planner_.upload(bk))).first;
  }
  if (!complex_) { be_dot((int)n, it->second.first, it->second.second, mkop(a.p, a.n), mkop(b.p, b.n), out, W_); return; }
  // bilinear complex dot: (ar.br - ai.bi) + i (ar.bi + ai.br); out is planar [2][W]
  double *d = (double *)pool_.get(sizeof(double) * 4 * (size_t)W_);
  const Operand ar = mkop(a.p, a.n), ai = mkop(imag(a), a.n), br = mkop(b.p, b.n), bi = mkop(imag(b), b.n);
  be_dot((int)n, it->second.first, it->second.second, ar, br, d, W_);
  be_dot((int)n, it->second.first, it->second.second, ai, bi, d + W_, W_);
  be_dot((int)n, it->second.first, it->second.second, ar, bi, d + 2 * W_, W_);
  be_dot((int)n, it->second.first, it->second.second, ai, br, d + 3 * W_, W_);
  be_complex_combine(d, d + W_, d + 2 * W_, d + 3 * W_, out, out + W_, W_);
  pool_.put(d);
}

// ---------------------------------------------------------------------------------------------------
// two-row environments (BTen2) and next-nearest-neighbour traces
// ---------------------------------------------------------------------------------------------------
void Engine::init_bten2(int pos) {                     // init.h:130-186
  for (auto &t : bten2_[pos]) release(t);
  bten2_[pos].clear();
  BT t = alloc({1, 1, 1, 1});
  be_fill(t.p, 1.0, W_);
  if (complex_) be_memset0(imag(t), sizeof(double) * W_);
  bten2_[pos].push_back(t);
}
const BT &Engine::bten2_at_slice(int pos, int logical) const {
  if (pos == DOWN) return bten2_[DOWN].at((size_t)(rows_ - 1 - logical));
  if (pos == RIGHT) return bten2_[RIGHT].at((size_t)(cols_ - 1 - logical));
  return bten2_[pos].at((size_t)logical);
}
BT Engine::bten2_step(const BT &bten2, const BT &mps1, const TRef &site1, const TRef &site2, const BT &mps2, int post) {
  // helpers.h:151-180 / grow.h:497-511: site1 sits next to the BMPS at pre_post, site2 next to the one at next_post
  ++n_bten_;
  const std::string sl1 = site_labels(post, 'p', 'y', 'n', 'o');
  const std::string sl2 = site_labels(post, 'n', 'v', 'f', 'q');
  BT tmp1 = einsum("apx,xyvz->apyvz", ref(mps1), ref(bten2));
  BT tmp2 = einsum("apyvz," + sl1 + "->vzaon", ref(tmp1), site1);
  release(tmp1);
  BT tmp3 = einsum("vzaon," + sl2 + "->zaofq", ref(tmp2), site2);
  release(tmp2);
  BT out = einsum("zaofq,zfb->aoqb", ref(tmp3), ref(mps2));
  release(tmp3);
  return out;
}
void Engine::bten2_operands(int post, int slice1, int bten_size, const BT *&mps1, const BT *&mps2, int &site1, int &site2) const {
  const int n = (post == LEFT || post == RIGHT) ? cols_ : rows_;
  const int s1 = slice1, s2 = slice1 + 1;
  const BMPSv *b1, *b2;
  if (post == LEFT) { b1 = &bmps_at_slice(UP, s1); b2 = &bmps_at_slice(DOWN, s2); site1 = s1 * cols_ + bten_size - 1; site2 = s2 * cols_ + bten_size - 1; }
  else if (post == RIGHT) { b1 = &bmps_at_slice(DOWN, s2); b2 = &bmps_at_slice(UP, s1); site1 = s2 * cols_ + n - bten_size; site2 = s1 * cols_ + n - bten_size; }
  else if (post == UP) { b1 = &bmps_at_slice(RIGHT, s2); b2 = &bmps_at_slice(LEFT, s1); site1 = (bten_size - 1) * cols_ + s2; site2 = (bten_size - 1) * cols_ + s1; }
  else { b1 = &bmps_at_slice(LEFT, s1); b2 = &bmps_at_slice(RIGHT, s2); site1 = (n - bten_size) * cols_ + s1; site2 = (n - bten_size) * cols_ + s2; }
  mps1 = &b1->at((size_t)(n - bten_size));
  mps2 = &b2->at((size_t)(bten_size - 1));
}
void Engine::grow_full_bten2(int pos, int slice1, int remain, bool init) {       // grow.h:375-515
  if (init) init_bten2(pos);
  mode_for_bten(pos);
  const int n = (pos == LEFT || pos == RIGHT) ? cols_ : rows_;
  for (int i = (int)bten2_[pos].size() - 1; i < n - remain; ++i) {
    const BT *m1, *m2; int s1, s2;
    bten2_operands(pos, slice1, i + 1, m1, m2, s1, s2);
    bten2_[pos].push_back(bten2_step(bten2_[pos].back(), *m1, site_ref(s1, s1), site_ref(s2, s2), *m2, pos));
  }
}
void Engine::grow_bten2_step(int post, int slice1) {   // grow.h:447-493
  mode_for_bten(post);
  const BT *m1, *m2; int s1, s2;
  bten2_operands(post, slice1, (int)bten2_[post].size(), m1, m2, s1, s2);
  bten2_[post].push_back(bten2_step(bten2_[post].back(), *m1, site_ref(s1, s1), site_ref(s2, s2), *m2, post));
}
void Engine::shift_bten2_window(int pos, int slice1) { // grow.h:523-527
  release(bten2_[pos].back());
  bten2_[pos].pop_back();
  grow_bten2_step(opposite(pos), slice1);
}
void Engine::nnn_trace(int row1, int col1, int dir, double *psi_out, int orient) {   // trace.h:207-324
  const int row2 = row1 + 1, col2 = col1 + 1;
  const int s11 = row1 * cols_ + col1, s21 = row2 * cols_ + col1, s12 = row1 * cols_ + col2, s22 = row2 * cols_ + col2;
  // configuration index each of the four plaquette tensors gathers: the two sites on the diagonal exchange theirs
  int g11 = s11, g21 = s21, g12 = s12, g22 = s22;
  if (dir == 0) { g11 = s22; g22 = s11; } else { g21 = s12; g12 = s21; }
  nnn_trace_refs(row1, col1, orient, site_ref(s11, g11), site_ref(s21, g21), site_ref(s12, g12), site_ref(s22, g22), psi_out);
}
void Engine::nnn_trace_refs(int row1, int col1, int orient, const TRef &t11, const TRef &t21, const TRef &t12, const TRef &t22,
                            double *psi_out) {
  ++n_trace_;
  const int row2 = row1 + 1, col2 = col1 + 1;
  const BT *m1, *m2; int a, b;
  BT half_a, half_b;
  if (orient == HORIZONTAL) {                          // two-row environments LEFT | RIGHT (:218-281)
    bten2_operands(LEFT, row1, col1 + 1, m1, m2, a, b);
    half_a = bten2_step(bten2_[LEFT].at((size_t)col1), *m1, t11, t21, *m2, LEFT);
    bten2_operands(RIGHT, row1, cols_ - col2, m1, m2, a, b);
    half_b = bten2_step(bten2_at_slice(RIGHT, col2), *m1, t22, t12, *m2, RIGHT);
  } else {                                             // two-column environments UP | DOWN (:282-324)
    bten2_operands(UP, col1, row1 + 1, m1, m2, a, b);
    half_a = bten2_step(bten2_[UP].at((size_t)row1), *m1, t12, t11, *m2, UP);
    bten2_operands(DOWN, col1, rows_ - row2, m1, m2, a, b);
    half_b = bten2_step(bten2_at_slice(DOWN, row2), *m1, t21, t22, *m2, DOWN);
  }
  reverse_dot(half_a, half_b, psi_out);                // Contract(tmp[3],{0,1,2,3}, tmp[7],{3,2,1,0})
  release(half_a);
  release(half_b);
}
// ReplaceSqrt5DistTwoSiteTrace (trace.h:426-536) with the two corner sites EXCHANGING their physical indices: a 2 x 3
// (HORIZONTAL) or 3 x 2 (VERTICAL) plaquette, two environment steps from the first side, one from the other.
void Engine::sqrt5_trace(int row1, int col1, int dir, int orient, double *psi_out) {
  ++n_trace_;
  const BT *m1, *m2; int a, b;
  auto S = [&](int r, int c) { return r * cols_ + c; };
  BT h1, h2, hb;
  if (orient == HORIZONTAL) {
    const int row2 = row1 + 1, col2 = col1 + 1, col3 = col1 + 2;
    int g[2][3];
    for (int r = 0; r < 2; ++r) for (int c = 0; c < 3; ++c) g[r][c] = S(row1 + r, col1 + c);
    if (dir == 0) std::swap(g[0][0], g[1][2]); else std::swap(g[1][0], g[0][2]);
    bten2_operands(LEFT, row1, col1 + 1, m1, m2, a, b);
    h1 = bten2_step(bten2_[LEFT].at((size_t)col1), *m1, site_ref(S(row1, col1), g[0][0]), site_ref(S(row2, col1), g[1][0]), *m2, LEFT);
    bten2_operands(LEFT, row1, col2 + 1, m1, m2, a, b);
    h2 = bten2_step(h1, *m1, site_ref(S(row1, col2), g[0][1]), site_ref(S(row2, col2), g[1][1]), *m2, LEFT);
    bten2_operands(RIGHT, row1, cols_ - col3, m1, m2, a, b);
    hb = bten2_step(bten2_at_slice(RIGHT, col3), *m1, site_ref(S(row2, col3), g[1][2]), site_ref(S(row1, col3), g[0][2]), *m2, RIGHT);
  } else {
    const int row2 = row1 + 1, row3 = row1 + 2, col2 = col1 + 1;
    int g[3][2];
    for (int r = 0; r < 3; ++r) for (int c = 0; c < 2; ++c) g[r][c] = S(row1 + r, col1 + c);
    if (dir == 0) std::swap(g[0][0], g[2][1]); else std::swap(g[2][0], g[0][1]);
    bten2_operands(UP, col1, row1 + 1, m1, m2, a, b);
    h1 = bten2_step(bten2_[UP].at((size_t)row1), *m1, site_ref(S(row1, col2), g[0][1]), site_ref(S(row1, col1), g[0][0]), *m2, UP);
    bten2_operands(UP, col1, row2 + 1, m1, m2, a, b);
    h2 = bten2_step(h1, *m1, site_ref(S(row2, col2), g[1][1]), site_ref(S(row2, col1), g[1][0]), *m2, UP);
    bten2_operands(DOWN, col1, rows_ - row3, m1, m2, a, b);
    hb = bten2_step(bten2_at_slice(DOWN, row3), *m1, site_ref(S(row3, col1), g[2][0]), site_ref(S(row3, col2), g[2][1]), *m2, DOWN);
  }
  reverse_dot(h2, hb, psi_out);                        // Contract(tmp[11],{0,1,2,3}, tmp[7],{3,2,1,0})  (:534)
  release(h1); release(h2); release(hb);
}
// test probes: grow the two-slice environments around the plaquette, then evaluate the exchange trace
void Engine::probe_plaquette_trace(int kind, int row1, int col1, int dir, int orient, double *psi_host) {
  const int span = kind == 0 ? 2 : 3;                  // plaquette extent along the MPS orientation
  if (orient == HORIZONTAL) {
    grow_bmps_for_row(row1);                           // UP stack to row1, DOWN stack to rows below row1
    grow_full_bten2(LEFT, row1, cols_ - col1, true);
    grow_full_bten2(RIGHT, row1, col1 + span, true);
  } else {
    grow_bmps_for_col(col1);
    grow_full_bten2(UP, col1, rows_ - row1, true);
    grow_full_bten2(DOWN, col1, row1 + span, true);
  }
  if (kind == 0) nnn_trace(row1, col1, dir, psi_tmp_, orient); else sqrt5_trace(row1, col1, dir, orient, psi_tmp_);
  be_d2h(psi_host, psi_tmp_, sizeof(double) * sw());
}
void Engine::punch_hole(int r, int c, int orient) {    // grow.h:150-183
  const BT *up, *down, *left, *right;
  if (orient == HORIZONTAL) {
    up = &bmps_at_slice(UP, r).at((size_t)(cols_ - 1 - c));
    down = &bmps_at_slice(DOWN, r).at((size_t)c);
    left = &bten_[LEFT].at((size_t)c);
    right = &bten_at_slice(RIGHT, c);
  } else {
    up = &bten_[UP].at((size_t)r);
    down = &bten_at_slice(DOWN, r);
    left = &bmps_at_slice(LEFT, c).at((size_t)r);
    right = &bmps_at_slice(RIGHT, c).at((size_t)(rows_ - 1 - r));
  }
  BT tmp1 = einsum("xlz,zdb->xldb", ref(*left), ref(*down));
  BT tmp2 = einsum("brz,zux->brux", ref(*right), ref(*up));
  const int site = r * cols_ + c;
  const Operand hi = mkop(holes_ + (long)W_ * hole_stride_ + hole_off_h_[(size_t)site], hole_stride_);
  einsum_into("xldb,brux->ldru", ref(tmp1), ref(tmp2), mkop(holes_ + hole_off_h_[(size_t)site], hole_stride_), nullptr, 1.0, 0.0,
              nullptr, complex_ ? &hi : nullptr);
  release(tmp1);
  release(tmp2);
}

// ---------------------------------------------------------------------------------------------------
// walker-level operations
// ---------------------------------------------------------------------------------------------------
void Engine::evaluate_amplitude() {                    // wave_function_component.h:187-212
  grow_bmps_for_row(0);
  grow_full_bten(RIGHT, 0, 2, true);
  init_bten(LEFT);
  nn_trace(0, 0, 0, 1, HORIZONTAL, 0, 1, amp_);
}
void Engine::init_walkers() {                          // wave_function_component.h:155-162
  contractor_init();
  evaluate_amplitude();
}

// ---------------------------------------------------------------------------------------------------
// the lattice traversal shared by the updaters and the energy solvers
// ---------------------------------------------------------------------------------------------------
template <class Start, class Visit, class End>
void Engine::line_pass(int orient, int reach, Start &&start, Visit &&visit, End &&end) {   // bond_traversal_mixin.h:112-143
  const bool h = orient == HORIZONTAL;
  const int lines = h ? rows_ : cols_, n = h ? cols_ : rows_;
  generate_bmps_approach(h ? UP : LEFT);
  for (int line = 0; line < lines; ++line) {
    init_bten(h ? LEFT : UP);
    grow_full_bten(h ? RIGHT : DOWN, line, reach, true);
    start(line);
    for (int pos = 0; pos <= n - reach; ++pos) {
      if (pos > 0) shift_bten_window(h ? RIGHT : DOWN);
      visit(line, pos);
    }
    end(line);
    if (line < lines - 1) shift_bmps_window(h ? DOWN : RIGHT);
  }
}
template <class Start, class Step>
void Engine::sweep_lines(int reach, Start &&start, Step &&step) {         // square_nn_updater.h:29-81
  line_pass(HORIZONTAL, reach, [&](int row) { start(row, 0, HORIZONTAL); }, [&](int row, int col) { step(row, col, HORIZONTAL); },
            [](int) {});
  delete_inner_bmps(LEFT);
  delete_inner_bmps(RIGHT);
  line_pass(VERTICAL, reach, [&](int col) { start(0, col, VERTICAL); }, [&](int col, int row) { step(row, col, VERTICAL); },
            [](int) {});
  delete_inner_bmps(UP);
}
template <class Visit>
void Engine::nnn_row_pass(int row, Visit &&visit) {                        // square_nnn_energy_solver.h:203-265
  if (row >= rows_ - 1) return;
  init_bten2(LEFT);
  grow_full_bten2(RIGHT, row, 2, true);
  for (int col = 0; col < cols_ - 1; ++col) {
    visit(col);
    shift_bten2_window(RIGHT, row);
  }
}
Engine::PsiList::PsiList(Engine &e, double *host) : e(e), host(host) {
  if (host && !e.psi_list_d_) e.psi_list_d_ = (double *)be_malloc(sizeof(double) * (size_t)(e.rows_ + e.cols_) * e.sw());
}
void Engine::PsiList::record(const double *psi) {
  if (host) be_d2d(e.psi_list_d_ + (size_t)n * e.sw(), psi, sizeof(double) * e.sw());
  ++n;
}
void Engine::PsiList::download() {
  if (host) be_d2h(host, e.psi_list_d_, sizeof(double) * (size_t)n * e.sw());
}

// MCUpdateSquareNNExchangeOBC (square_nn_updater.h:29-81, 146-188). Fermion mode: same visit order, decisions and draws;
// the exchanged tensors are the dressed slices of be_fermion_targets, the gather indices follow every decision.
void Engine::sweep(int nsweeps, double *accept_rate_host) {
  auto step = [&](int ra, int ca, int orient) {
    const int rb = orient == VERTICAL ? ra + 1 : ra, cb = orient == HORIZONTAL ? ca + 1 : ca;
    const int s1 = ra * cols_ + ca, s2 = rb * cols_ + cb;
    if (fermion_) {
      be_fermion_targets(cfg_, nsites_, s1, s2, phys_, phys_par_d_, jw_[0], jw_[1], orient, nullptr, nullptr, 0, 0, term_ia_, term_ib_, term_cw_, W_);
      nn_trace_idx(ra, ca, rb, cb, orient, term_ia_, term_ib_, 1, psi_tmp_);
    } else {
      nn_trace(ra, ca, rb, cb, orient, s2, s1, psi_tmp_);                     // :164-166 (masked in the decide kernel)
    }
    exchange_decide(s1, s2, psi_tmp_, jastrow_for(s1, s2));
    refresh_gather();
    touch_site(s1); touch_site(s2);
  };
  for (int sw = 0; sw < nsweeps; ++sw) {
    be_memset0(accepted_, sizeof(int32_t) * W_);
    sweep_lines(2, [](int, int, int) {}, step);
  }
  if (accept_rate_host) {
    std::vector<int32_t> acc((size_t)W_);
    be_d2h(acc.data(), accepted_, sizeof(int32_t) * W_);
    const double bond_num = (double)(cols_ * (rows_ - 1) + rows_ * (cols_ - 1));
    for (int w = 0; w < W_; ++w) accept_rate_host[w] = (double)acc[(size_t)w] / bond_num;
  }
}

namespace {
// std::mt19937 on the host, in the state layout of the device streams (624 words + index)
struct HostMT {
  uint32_t mt[624];
  int idx;
  uint32_t next() {
    if (idx >= 624) {
      for (int k = 0; k < 624; ++k) {
        uint32_t y = (mt[k] & 0x80000000u) | (mt[(k + 1) % 624] & 0x7fffffffu);
        mt[k] = mt[(k + 397) % 624] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
      }
      idx = 0;
    }
    uint32_t y = mt[idx++];
    y ^= y >> 11; y ^= (y << 7) & 0x9d2c5680u; y ^= (y << 15) & 0xefc60000u; y ^= y >> 18;
    return y;
  }
  // std::uniform_real_distribution<long double>(a, b)(engine) of libstdc++: generate_canonical<long double, 64> takes
  // two 32-bit draws, exact in the x87 significand
  long double uniform(long double a, long double b) {
    const long double x0 = (long double)next(), x1 = (long double)next();
    long double u = (x0 + x1 * 4294967296.0L) / (4294967296.0L * 4294967296.0L);
    if (u >= 1.0L) u = std::nextafter(1.0L, 0.0L);
    return u * (b - a) + a;
  }
};
// SuwaTodoStateUpdate (suwa_todo_update.h:53-113): geometric allocation on the cumulative weights, heaviest state first
int suwa_todo(int init, std::vector<double> w, HostMT &rng) {
  const int n = (int)w.size();
  int imax = 0;
  for (int i = 1; i < n; ++i) if (w[(size_t)i] > w[(size_t)imax]) imax = i;
  if (imax != 0) std::swap(w[0], w[(size_t)imax]);
  if (init == imax) init = 0; else if (init == 0) init = imax;
  std::vector<long double> cum((size_t)n);
  cum[0] = (long double)w[0];
  for (int i = 1; i < n; ++i) cum[(size_t)i] = cum[(size_t)i - 1] + (long double)w[(size_t)i];
  const long double total = cum.back();
  long double start = (init == 0 ? 0.0L : cum[(size_t)init - 1]) + (long double)w[0];
  if (start >= total) start -= total;
  long double x = rng.uniform(start, std::nextafter(start + (long double)w[(size_t)init], start));
  if (x >= total) x -= total;
  int fin = (int)(std::upper_bound(cum.begin(), cum.end(), x) - cum.begin());
  if (imax != 0) { if (fin == 0) fin = imax; else if (fin == imax) fin = 0; }
  return fin;
}
// the per-walker device streams ([W][624] words, [W] indices) as host generators for the Suwa-Todo draws, and back
std::vector<HostMT> download_rng(const uint32_t *mt_d, const int32_t *idx_d, int W) {
  std::vector<uint32_t> mt((size_t)W * 624);
  std::vector<int32_t> idx((size_t)W);
  be_d2h(mt.data(), mt_d, sizeof(uint32_t) * mt.size());
  be_d2h(idx.data(), idx_d, sizeof(int32_t) * idx.size());
  std::vector<HostMT> rng((size_t)W);
  for (int w = 0; w < W; ++w) {
    std::copy(mt.begin() + (size_t)w * 624, mt.begin() + (size_t)(w + 1) * 624, rng[(size_t)w].mt);
    rng[(size_t)w].idx = idx[(size_t)w];
  }
  return rng;
}
void upload_rng(const std::vector<HostMT> &rng, uint32_t *mt_d, int32_t *idx_d) {
  std::vector<uint32_t> mt(rng.size() * 624);
  std::vector<int32_t> idx(rng.size());
  for (size_t w = 0; w < rng.size(); ++w) {
    std::copy(rng[w].mt, rng[w].mt + 624, mt.begin() + w * 624);
    idx[w] = rng[w].idx;
  }
  be_h2d(mt_d, mt.data(), sizeof(uint32_t) * mt.size());
  be_h2d(idx_d, idx.data(), sizeof(int32_t) * idx.size());
}
}  // namespace

void Engine::ensure_idx_const() {
  if (idx_const_) return;
  const int d = phys_;
  idx_const_ = (int32_t *)be_malloc(sizeof(int32_t) * (size_t)d * W_);
  std::vector<int32_t> h((size_t)d * W_);
  for (int s = 0; s < d; ++s) for (int w = 0; w < W_; ++w) h[(size_t)s * W_ + w] = s;
  be_h2d(idx_const_, h.data(), sizeof(int32_t) * h.size());
}
void Engine::sweep_full_space(int nsweeps, double *accept_rate_host) {
  const int d = phys_, nst = d * d;
  ensure_idx_const();
  ensure_psi_alt(nst);
  // fermion mode ("work for both fermion and boson", square_nn_updater.h:251): every target state through the dressed
  // replacement rule of be_fermion_targets (a full table: slot t = local state t where both site parities change together,
  // empty otherwise -- those amplitudes vanish for parity-conserving tensors and get weight 0)
  if (fermion_ && !fs_target_d_) {
    std::vector<int32_t> tg((size_t)nst * nst);
    std::vector<double> cf((size_t)nst * nst, 1.0);
    for (int p = 0; p < nst; ++p)
      for (int q = 0; q < nst; ++q) {
        const bool ok = (phys_par_h_[(size_t)(p / d)] ^ phys_par_h_[(size_t)(q / d)]) == (phys_par_h_[(size_t)(p % d)] ^ phys_par_h_[(size_t)(q % d)]);
        tg[(size_t)p * nst + q] = ok ? q : -1;
      }
    fs_target_d_ = (int32_t *)be_malloc(sizeof(int32_t) * tg.size());
    fs_coef_d_ = (double *)be_malloc(sizeof(double) * cf.size());
    be_h2d(fs_target_d_, tg.data(), sizeof(int32_t) * tg.size());
    be_h2d(fs_coef_d_, cf.data(), sizeof(double) * cf.size());
  }
  std::vector<int32_t> cfg((size_t)W_ * nsites_);
  const size_t S = sw();                                                 // complex: every amplitude array is [re W][im W]
  std::vector<double> amp(S), alt((size_t)nst * S);
  be_d2h(cfg.data(), cfg_, sizeof(int32_t) * cfg.size());
  be_d2h(amp.data(), amp_, sizeof(double) * amp.size());
  std::vector<HostMT> rng = download_rng(mt_, mtidx_, W_);
  std::vector<int> accepted((size_t)W_);
  auto bond = [&](int ra, int ca, int orient) {                          // TwoSiteNNUpdateLocalImpl (:257-291)
    const int rb = orient == VERTICAL ? ra + 1 : ra, cb = orient == HORIZONTAL ? ca + 1 : ca;
    const int s1 = ra * cols_ + ca, s2 = rb * cols_ + cb;
    for (int a = 0; a < d; ++a)
      for (int b = 0; b < d; ++b) {
        if (fermion_) {
          be_fermion_targets(cfg_, nsites_, s1, s2, phys_, phys_par_d_, jw_[0], jw_[1], orient == HORIZONTAL ? 0 : 1, fs_target_d_, fs_coef_d_,
                             nst, a * d + b, term_ia_, term_ib_, term_cw_, W_);
          nn_trace_idx(ra, ca, rb, cb, orient, term_ia_, term_ib_, 1, psi_alt_ + (size_t)(a * d + b) * S);
        } else {
          nn_trace_idx(ra, ca, rb, cb, orient, idx_const_ + (size_t)a * W_, idx_const_ + (size_t)b * W_, 1,
                       psi_alt_ + (size_t)(a * d + b) * S);
        }
      }
    be_d2h(alt.data(), psi_alt_, sizeof(double) * alt.size());
    bool any = false;
    std::vector<double> wt((size_t)nst);
    for (int w = 0; w < W_; ++w) {
      int32_t *c = cfg.data() + (size_t)w * nsites_;
      const int init = c[s1] * d + c[s2];
      if (!complex_) {
        const double a0 = amp[(size_t)w];
        for (int i = 0; i < nst; ++i) {
          const double r = (i == init ? a0 : alt[(size_t)i * W_ + w]) / a0;
          wt[(size_t)i] = r * r;                                         // std::norm(alternative_psi / amplitude)
        }
      } else {
        const std::complex<double> a0(amp[(size_t)w], amp[(size_t)W_ + w]);
        for (int i = 0; i < nst; ++i) {
          const std::complex<double> x(alt[(size_t)i * S + w], alt[(size_t)i * S + W_ + w]);
          wt[(size_t)i] = std::norm((i == init ? a0 : x) / a0);
        }
      }
      if (fermion_)
        for (int i = 0; i < nst; ++i)
          if ((phys_par_h_[(size_t)(init / d)] ^ phys_par_h_[(size_t)(i / d)]) != (phys_par_h_[(size_t)(init % d)] ^ phys_par_h_[(size_t)(i % d)]))
            wt[(size_t)i] = 0.0;
      const int fin = suwa_todo(init, wt, rng[(size_t)w]);
      if (fin != init) {
        c[s1] = fin / d; c[s2] = fin % d;
        amp[(size_t)w] = alt[(size_t)fin * S + w];
        if (complex_) amp[(size_t)W_ + w] = alt[(size_t)fin * S + W_ + w];
        ++accepted[(size_t)w];
        any = true;
      }
    }
    if (any) {
      be_h2d(cfg_, cfg.data(), sizeof(int32_t) * cfg.size());
      be_h2d(amp_, amp.data(), sizeof(double) * amp.size());
      refresh_gather();
    }
    touch_site(s1); touch_site(s2);
  };
  for (int sw = 0; sw < nsweeps; ++sw) {
    std::fill(accepted.begin(), accepted.end(), 0);
    sweep_lines(2, [](int, int, int) {}, bond);
  }
  upload_rng(rng, mt_, mtidx_);
  if (accept_rate_host) {
    const double bond_num = (double)(cols_ * (rows_ - 1) + rows_ * (cols_ - 1));
    for (int w = 0; w < W_; ++w) accept_rate_host[w] = accepted[(size_t)w] / bond_num;
  }
}

void Engine::sweep_three_site(int nsweeps, double *accept_rate_host) {
  if (rows_ < 3 || cols_ < 3) throw std::invalid_argument("the 3-site updater needs a lattice of at least 3x3");
  const int maxp = 6;
  if (!idx_perm_) idx_perm_ = (int32_t *)be_malloc(sizeof(int32_t) * (size_t)maxp * W_ * 3);
  ensure_psi_alt(maxp);
  std::vector<int32_t> cfg((size_t)W_ * nsites_), perm_h((size_t)maxp * W_ * 3);
  const size_t S = sw();                                               // complex: every amplitude array is [re W][im W]
  std::vector<double> amp(S), alt((size_t)maxp * S);
  be_d2h(cfg.data(), cfg_, sizeof(int32_t) * cfg.size());
  std::vector<HostMT> rng = download_rng(mt_, mtidx_, W_);
  std::vector<int> accepted((size_t)W_);
  auto refresh_amplitude = [&](int r, int c, int orient) {            // :39-42, :66-69
    const int s0 = r * cols_ + c, step = orient == HORIZONTAL ? 1 : cols_;
    const int32_t *own = fermion_ ? gidx_[orient] : cfg_;            // fermion mode: the dressed slices of the machinery
    tnn_trace_idx(r, c, orient, own + s0, own + s0 + step, own + s0 + 2 * step, nsites_, amp_);
    be_d2h(amp.data(), amp_, sizeof(double) * amp.size());
  };
  // fermion mode: gather index of `state` at the k-th site of the triple when the sites before it carry `st[0..k-1]`: the
  // Jordan-Wigner bit follows the new states (the triple's parity is conserved, later sites are unaffected)
  auto dressed = [&](const int32_t *cw, int r, int c, int orient, const std::array<int, 3> &st, int k) -> int32_t {
    if (!fermion_) return st[(size_t)k];
    int bit = 0;
    if (orient == HORIZONTAL) for (int x = 0; x < c; ++x) bit ^= phys_par_h_[(size_t)cw[r * cols_ + x]];
    else for (int y = 0; y < r; ++y) bit ^= phys_par_h_[(size_t)cw[y * cols_ + c]];
    for (int q = 0; q < k; ++q) bit ^= phys_par_h_[(size_t)st[(size_t)q]];
    return (int32_t)(((orient == HORIZONTAL ? 0 : 6) + bit) * phys_ + st[(size_t)k]);
  };
  auto triple = [&](int r, int c, int orient) {                       // TNN3SiteUpdateImpl (:108-158)
    const int s0 = r * cols_ + c, step = orient == HORIZONTAL ? 1 : cols_;
    const int st[3] = {s0, s0 + step, s0 + 2 * step};
    std::vector<std::vector<std::array<int, 3>>> perms((size_t)W_);
    std::vector<int> init((size_t)W_, -1);
    int nslots = 0;
    for (int w = 0; w < W_; ++w) {
      const int32_t *cw = cfg.data() + (size_t)w * nsites_;
      std::array<int, 3> sp = {cw[st[0]], cw[st[1]], cw[st[2]]};
      if (sp[0] == sp[1] && sp[1] == sp[2]) continue;                  // no draw for a uniform triple
      std::array<int, 3> srt = sp;
      std::sort(srt.begin(), srt.end());
      do { perms[(size_t)w].push_back(srt); } while (std::next_permutation(srt.begin(), srt.end()));
      init[(size_t)w] = (int)(std::find(perms[(size_t)w].begin(), perms[(size_t)w].end(), sp) - perms[(size_t)w].begin());
      nslots = std::max(nslots, (int)perms[(size_t)w].size());
    }
    if (nslots == 0) return;
    for (int s = 0; s < nslots; ++s)
      for (int w = 0; w < W_; ++w) {
        const int32_t *cw = cfg.data() + (size_t)w * nsites_;
        const bool has = s < (int)perms[(size_t)w].size();
        const std::array<int, 3> own = {cw[st[0]], cw[st[1]], cw[st[2]]};
        const std::array<int, 3> &use = has ? perms[(size_t)w][(size_t)s] : own;
        for (int k = 0; k < 3; ++k) perm_h[((size_t)s * W_ + w) * 3 + k] = dressed(cw, r, c, orient, use, k);
      }
    be_h2d(idx_perm_, perm_h.data(), sizeof(int32_t) * (size_t)nslots * W_ * 3);
    for (int s = 0; s < nslots; ++s) {
      const int32_t *ix = idx_perm_ + (size_t)s * W_ * 3;
      tnn_trace_idx(r, c, orient, ix, ix + 1, ix + 2, 3, psi_alt_ + (size_t)s * S);
    }
    be_d2h(alt.data(), psi_alt_, sizeof(double) * (size_t)nslots * S);
    bool any = false;
    for (int w = 0; w < W_; ++w) {
      const int np = (int)perms[(size_t)w].size();
      if (np == 0) continue;
      std::vector<double> psis((size_t)np), psii((size_t)np, 0.0), wt((size_t)np);
      double mx = 0.0;
      for (int i = 0; i < np; ++i) {
        const bool own = i == init[(size_t)w];
        psis[(size_t)i] = own ? amp[(size_t)w] : alt[(size_t)i * S + w];
        if (complex_) psii[(size_t)i] = own ? amp[(size_t)W_ + w] : alt[(size_t)i * S + W_ + w];
        mx = std::max(mx, complex_ ? std::hypot(psis[(size_t)i], psii[(size_t)i]) : std::fabs(psis[(size_t)i]));
      }
      for (int i = 0; i < np; ++i) {                                   // std::norm(psis[i] / psi_abs_max)
        const double q = psis[(size_t)i] / mx, qi = psii[(size_t)i] / mx;
        wt[(size_t)i] = complex_ ? q * q + qi * qi : q * q;
      }
      const int fin = suwa_todo(init[(size_t)w], wt, rng[(size_t)w]);
      if (fin == init[(size_t)w]) continue;
      int32_t *cw = cfg.data() + (size_t)w * nsites_;
      for (int k = 0; k < 3; ++k) cw[st[k]] = perms[(size_t)w][(size_t)fin][(size_t)k];
      amp[(size_t)w] = psis[(size_t)fin];
      if (complex_) amp[(size_t)W_ + w] = psii[(size_t)fin];
      ++accepted[(size_t)w];
      any = true;
    }
    if (any) {
      be_h2d(cfg_, cfg.data(), sizeof(int32_t) * cfg.size());
      be_h2d(amp_, amp.data(), sizeof(double) * amp.size());
      refresh_gather();
    }
    for (int k = 0; k < 3; ++k) touch_site(st[k]);
  };
  for (int sw = 0; sw < nsweeps; ++sw) {                                // square_3site_updater.h:29-97
    std::fill(accepted.begin(), accepted.end(), 0);
    sweep_lines(3, refresh_amplitude, triple);
  }
  upload_rng(rng, mt_, mtidx_);
  if (accept_rate_host) {
    const double total = (double)(cols_ * (rows_ - 2) + rows_ * (cols_ - 2));
    for (int w = 0; w < W_; ++w) accept_rate_host[w] = accepted[(size_t)w] / total;
  }
}

void Engine::energy_and_holes_tfim(bool calc_holes, double *eloc_host, double *psi_list_host) {
  require_boson("the transverse-field Ising solver");
  // TransverseFieldIsingSquareOBC::CalEnergyAndHolesImplParsed (transverse_field_ising_square_obc.h:208-247)
  if (phys_ != 2) throw std::invalid_argument("transverse-field Ising model needs phys = 2");
  std::vector<int32_t> cfg((size_t)W_ * nsites_), flip((size_t)W_ * nsites_);
  be_d2h(cfg.data(), cfg_, sizeof(int32_t) * cfg.size());
  std::vector<double> diag((size_t)W_);
  for (int w = 0; w < W_; ++w) {                                          // CalDiagTermEnergy (:160-182)
    const int32_t *c = cfg.data() + (size_t)w * nsites_;
    double e = 0.0;
    for (int r = 0; r < rows_; ++r) for (int cc = 0; cc < cols_ - 1; ++cc) e += (c[r * cols_ + cc] == c[r * cols_ + cc + 1]) ? -1 : 1;
    for (int cc = 0; cc < cols_; ++cc) for (int r = 0; r < rows_ - 1; ++r) e += (c[r * cols_ + cc] == c[(r + 1) * cols_ + cc]) ? -1 : 1;
    diag[(size_t)w] = e;
  }
  for (size_t i = 0; i < cfg.size(); ++i) flip[i] = 1 - cfg[i];
  if (!idx_flip_) idx_flip_ = (int32_t *)be_malloc(sizeof(int32_t) * flip.size());
  be_h2d(idx_flip_, flip.data(), sizeof(int32_t) * flip.size());
  be_memset0(eloc_, sizeof(double) * sw());
  PsiList psi_list(*this, psi_list_host);
  line_pass(HORIZONTAL, 1,
            [&](int row) {
              nn_trace(row, 0, row, 1, HORIZONTAL, row * cols_, row * cols_ + 1, psi_row_);
              psi_list.record(psi_row_);
            },
            [&](int row, int col) {
              if (calc_holes) punch_hole(row, col, HORIZONTAL);
              one_site_trace(row, col, idx_flip_ + row * cols_ + col, nsites_, psi_tmp_);      // :191-204
              ratio_acc(psi_tmp_, psi_row_, -tfim_h_, eloc_);
            },
            [](int) {});
  psi_list.download();
  std::vector<double> e((size_t)W_);
  be_d2h(e.data(), eloc_, sizeof(double) * W_);
  for (int w = 0; w < W_; ++w) e[(size_t)w] += diag[(size_t)w];
  be_h2d(eloc_, e.data(), sizeof(double) * W_);
  if (eloc_host) std::copy(e.begin(), e.end(), eloc_host);
}

void Engine::energy_and_holes(bool calc_holes, double *eloc_host, double *psi_list_host) {
  if (jastrow_on_ && !(fermion_ || tables_on_)) throw std::logic_error("Jastrow dressing needs a table-driven model (peps_set_model_term)");
  if (jastrow_on_ && !tables_exchange_only_) throw std::logic_error("Jastrow dressing supports exchange terms only");
  const bool xxz = !fermion_ && !tables_on_;
  if (xxz && tfim_) { energy_and_holes_tfim(calc_holes, eloc_host, psi_list_host); return; }
  if (xxz && phys_ != 2) throw std::invalid_argument("the XXZ / J1-J2 energy solvers need phys = 2");
  energy_pass(calc_holes, eloc_host, psi_list_host);
}

// The traversal of SquareNNNModelEnergySolver (square_nnn_energy_solver.h:79-315, bond_traversal_mixin.h:112-143) for the
// built-in XXZ / J1-J2 model (SquareSpinOneHalfXXZModelMixIn) and for the table models, bosons and fermions. The results go
// to eloc_, to the bond's record while measure() runs (bond_target), or to the site's record while measure_site_term() runs.
void Engine::energy_pass(bool calc_holes, double *eloc_host, double *psi_list_host) {
  const bool xxz = !fermion_ && !tables_on_;                        // the built-in model: no table is set
  const TermTable &nn = term_[0], &nnn = term_[1], &on = term_[2];
  // bosons divide by one psi per line (psi_row_). Fermions recompute psi per bond by Trace (NN) and once per plaquette by
  // ReplaceNNNSiteTrace with the original tensors (NNN), so that psi_ex / psi runs along one contraction path (psi_loc_).
  double *const psi = fermion_ ? psi_loc_ : psi_row_;
  be_memset0(eloc_, sizeof(double) * sw());
  PsiList psi_list(*this, psi_list_host);
  // one table term on (s1, s2), s2 < 0 on-site: the diagonal element + one replacement trace per target slot, masked per
  // walker; trace(idx_a, idx_b, out) evaluates the amplitude with the replacement physical indices
  auto term = [&](const TermTable &tt, int s1, int s2, int kind, double *dst, auto &&trace) {
    if (tt.T == 0) { term_acc(s1, s2, tt.diag, nullptr, nullptr, psi, dst); return; }
    for (int t = 0; t < tt.T; ++t) {
      if (fermion_)
        be_fermion_targets(cfg_, nsites_, s1, s2, phys_, phys_par_d_, jw_[0], jw_[1], kind, tt.target, tt.coef, tt.T, t, term_ia_, term_ib_, term_cw_, W_);
      else
        be_term_targets(cfg_, nsites_, s1, s2, phys_, tt.target, tt.coef, tt.T, t, term_ia_, s2 >= 0 ? term_ib_ : nullptr, term_cw_, W_);
      if (s2 >= 0) if (const double *jr = jastrow_for(s1, s2)) be_scale(term_cw_, jr, W_);
      trace(term_ia_, term_ib_, psi_tmp_);
      term_acc(s1, s2, t == 0 ? tt.diag : nullptr, term_cw_, psi_tmp_, psi, dst);
    }
  };
  auto line_start = [&](int ra, int ca, int rb, int cb, int orient) {
    if (fermion_) return;
    nn_trace(ra, ca, rb, cb, orient, ra * cols_ + ca, rb * cols_ + cb, psi_row_);
    psi_list.record(psi_row_);
  };
  auto bond = [&](int row, int col, int orient) {                    // (row, col) - its right / lower neighbour
    const int r2 = orient == VERTICAL ? row + 1 : row, c2 = orient == HORIZONTAL ? col + 1 : col;
    const int s1 = row * cols_ + col, s2 = r2 * cols_ + c2;
    double *const dst = bond_target(orient, row, col);
    if (xxz) {
      nn_trace(row, col, r2, c2, orient, s2, s1, psi_tmp_);
      bond_energy(s1, s2, psi_tmp_, psi_row_, jz_, jxy_, dst);
      return;
    }
    if (fermion_) {
      if (!nn.set) return;
      nn_trace(row, col, r2, c2, orient, s1, s2, psi_loc_);                                // Trace(tn, site1, site2, orient)
      if ((orient == HORIZONTAL ? col : row) == 0) psi_list.record(psi_loc_);
    }
    auto tr = [&](const int32_t *ia, const int32_t *ib, double *out) { nn_trace_idx(row, col, r2, c2, orient, ia, ib, 1, out); };
    if (nn.set) term(nn, s1, s2, orient, dst, tr);
    if (pin_.set && s1 == pin_s1_ && s2 == pin_s2_) term(pin_, s1, s2, orient, dst, tr);
  };
  auto plaquette = [&](int row, int col) {
    const int s11 = row * cols_ + col, s21 = s11 + cols_, s12 = s11 + 1, s22 = s21 + 1;
    if (fermion_) {
      gmode_ = HORIZONTAL;
      nnn_trace_refs(row, col, HORIZONTAL, site_ref(s11, s11), site_ref(s21, s21), site_ref(s12, s12), site_ref(s22, s22), psi_loc_);
    }
    for (int dir = 0; dir < 2; ++dir) {                              // (row,col) - (row+1,col+1), then (row+1,col) - (row,col+1)
      const int s1 = dir == 0 ? s11 : s21, s2 = dir == 0 ? s22 : s12;
      double *const dst = bond_target(2 + dir, row, col);
      if (xxz) {
        nnn_trace(row, col, dir, psi_tmp_);
        bond_energy(s1, s2, psi_tmp_, psi_row_, jz2_, jxy2_, dst);
        continue;
      }
      term(nnn, s1, s2, 2 + dir, dst, [&](const int32_t *ia, const int32_t *ib, double *out) {
        auto ref = [&](int s) { return s == s1 ? site_ref_idx(s, ia, 1) : s == s2 ? site_ref_idx(s, ib, 1) : site_ref(s, s); };
        gmode_ = HORIZONTAL;                                                   // read by site_ref in fermion mode only
        nnn_trace_refs(row, col, HORIZONTAL, ref(s11), ref(s21), ref(s12), ref(s22), out);
      });
    }
  };
  line_pass(HORIZONTAL, 1, [&](int row) { line_start(row, 0, row, 1, HORIZONTAL); },
            [&](int row, int col) {
              if (calc_holes) punch_hole(row, col, HORIZONTAL);
              const int s = row * cols_ + col;
              if (on.set) term(on, s, -1, 0, rec_sites_ ? site_rec_ + (size_t)s * sw() : eloc_,
                               [&](const int32_t *ia, const int32_t *, double *out) { one_site_trace(row, col, ia, 1, out); });
              if (col < cols_ - 1) bond(row, col, HORIZONTAL);
            },
            [&](int row) {
              if (xxz ? (jz2_ != 0.0 || jxy2_ != 0.0) : nnn.set) nnn_row_pass(row, [&](int col) { plaquette(row, col); });
              if (xxz && rec_bonds_ && row == rows_ / 2) row_corr_hook(row);          // bond_traversal_mixin.h:96-98
            });
  if (fermion_ && calc_holes) {
    if (complex_)
      be_fermion_finish_holes_c(holes_, holes_ + (long)W_ * hole_stride_, hole_stride_, hole_off_d_, site_size_d_, gtps_, gtps_total_,
                                gtps_off_d_, gidx_[HORIZONTAL], jw_[HORIZONTAL], nsites_, fsign_, amp_, amp_ + W_, W_);
    else
      be_fermion_finish_holes(holes_, hole_stride_, hole_off_d_, site_size_d_, gtps_, gtps_off_d_, gidx_[HORIZONTAL], jw_[HORIZONTAL],
                              nsites_, fsign_, amp_, W_);
  }
  line_pass(VERTICAL, 2, [&](int col) { line_start(0, col, 1, col, VERTICAL); }, [&](int col, int row) { bond(row, col, VERTICAL); },
            [](int) {});
  if (xxz) be_xxz_onsite_energy(cfg_, nsites_, h00_, eloc_, W_);               // the site-0 pinning term
  psi_list.download();
  if (eloc_host) be_d2h(eloc_host, eloc_, sizeof(double) * W_);
}

void Engine::set_model_term(int kind, int T, const double *diag, const int32_t *target, const double *coef) {
  if (kind < 0 || kind > 2) throw std::invalid_argument("set_model_term: kind must be 0 (NN), 1 (NNN) or 2 (on-site)");
  if (T < 0 || !diag || (T > 0 && (!target || !coef))) throw std::invalid_argument("set_model_term: null table");
  const int np = kind == 2 ? phys_ : phys_ * phys_;
  for (int i = 0; i < np * T; ++i)
    if (target[i] >= np) throw std::invalid_argument("set_model_term: target state out of range");
  if (fermion_) {
    if (kind == 2 && T > 0) throw std::invalid_argument("set_model_term: fermion mode supports diagonal on-site terms only");
    if (kind != 2) check_two_site_table(T, target);
  }
  for (int p = 0; kind != 2 && p < np; ++p)
    for (int tt = 0; tt < T; ++tt) {
      const int tg = target[p * T + tt];
      if (tg >= 0 && tg != (p % phys_) * phys_ + p / phys_) tables_exchange_only_ = false;
    }
  if (kind == 2 && T > 0) tables_exchange_only_ = false;
  be_sync();
  upload_table(term_[kind], np, T, diag, target, coef);
  if (!term_ia_) {
    term_ia_ = (int32_t *)be_malloc(sizeof(int32_t) * W_);
    term_ib_ = (int32_t *)be_malloc(sizeof(int32_t) * W_);
    term_cw_ = (double *)be_malloc(sizeof(double) * W_);
  }
  tables_on_ = true;
}
// fermion mode: both site parities of a two-site target change together (a hop or a pair) or not at all
void Engine::check_two_site_table(int T, const int32_t *target) const {
  for (int p = 0; p < phys_ * phys_; ++p)
    for (int t = 0; t < T; ++t) {
      const int tg = target[p * T + t];
      if (tg < 0) continue;
      const int d1 = phys_par_h_[(size_t)(p / phys_)] ^ phys_par_h_[(size_t)(tg / phys_)];
      const int d2 = phys_par_h_[(size_t)(p % phys_)] ^ phys_par_h_[(size_t)(tg % phys_)];
      if (d1 != d2) throw std::invalid_argument("fermion mode needs two-site targets that move one fermion between the two sites, create / annihilate a pair, or keep both parities");
    }
}
void Engine::free_table(TermTable &t) {
  be_free(t.diag); be_free(t.target); be_free(t.coef);
  t = TermTable();
}
void Engine::upload_table(TermTable &t, int np, int T, const double *diag, const int32_t *target, const double *coef) {
  free_table(t);
  t.T = T; t.set = true;
  t.diag = (double *)be_malloc(sizeof(double) * np);
  be_h2d(t.diag, diag, sizeof(double) * np);
  if (T > 0) {
    t.target = (int32_t *)be_malloc(sizeof(int32_t) * (size_t)np * T);
    t.coef = (double *)be_malloc(sizeof(double) * (size_t)np * T);
    be_h2d(t.target, target, sizeof(int32_t) * (size_t)np * T);
    be_h2d(t.coef, coef, sizeof(double) * (size_t)np * T);
  }
}
void Engine::set_bond_pin(int s1, int s2, int T, const double *diag, const int32_t *target, const double *coef) {
  be_sync();
  if (T <= 0) { free_table(pin_); pin_s1_ = pin_s2_ = -1; return; }
  if (!diag || !target || !coef) throw std::invalid_argument("set_bond_pin: null table");
  const bool horizontal = s2 == s1 + 1 && s1 >= 0 && (s1 % cols_) < cols_ - 1 && s2 < nsites_;
  const bool vertical = s2 == s1 + cols_ && s1 >= 0 && s2 < nsites_;
  if (!horizontal && !vertical)                       // ValidateSingletPairPinningBondInLattice_ (square_tJ_model.h:240-250)
    throw std::invalid_argument("set_bond_pin: (site1, site2) must be a nearest-neighbour bond inside the lattice, site1 the left / upper site");
  const int np = phys_ * phys_;
  for (int i = 0; i < np * T; ++i)
    if (target[i] >= np) throw std::invalid_argument("set_bond_pin: target state out of range");
  if (fermion_) check_two_site_table(T, target);
  if (!tables_on_) throw std::logic_error("set_bond_pin: needs a table-driven model (peps_set_model_term) first");
  upload_table(pin_, np, T, diag, target, coef);
  pin_s1_ = s1; pin_s2_ = s2;
  tables_exchange_only_ = false;
}
template <class Body>
void Engine::with_term_table(int kind, int T, const double *diag, const int32_t *target, const double *coef, Body &&body) {
  be_sync();
  TermTable saved[3] = {term_[0], term_[1], term_[2]}, saved_pin = pin_;
  const bool s_on = tables_on_, s_ex = tables_exchange_only_, s_j = jastrow_on_;
  for (auto &t : term_) t = TermTable();
  pin_ = TermTable();
  auto restore = [&]() {
    be_sync();
    free_table(term_[kind]);
    for (int k = 0; k < 3; ++k) term_[k] = saved[k];
    pin_ = saved_pin;
    tables_on_ = s_on; tables_exchange_only_ = s_ex; jastrow_on_ = s_j;
    rec_sites_ = false;
  };
  try {
    set_model_term(kind, T, diag, target, coef);
    jastrow_on_ = false;
    body();
  } catch (...) { restore(); throw; }
  restore();
}
void Engine::measure_bond_term(int T, const double *diag, const int32_t *target, const double *coef, double *out_h, double *out_v) {
  if (T < 0 || !diag || (T > 0 && (!target || !coef))) throw std::invalid_argument("measure_bond_term: null table");
  with_term_table(0, T, diag, target, coef, [&]() { measure(nullptr, out_h, out_v, nullptr, nullptr, nullptr); });
}
void Engine::measure_site_term(int T, const double *diag, const int32_t *target, const double *coef, double *out) {
  require_boson("measure_site_term");
  if (T < 0 || !diag || !out || (T > 0 && (!target || !coef))) throw std::invalid_argument("measure_site_term: null table");
  const size_t S = sw();
  with_term_table(2, T, diag, target, coef, [&]() {
    if (!site_rec_) site_rec_ = (double *)be_malloc(sizeof(double) * (size_t)nsites_ * S);
    be_memset0(site_rec_, sizeof(double) * (size_t)nsites_ * S);
    rec_sites_ = true;
    energy_pass(false, nullptr, nullptr);
    std::vector<double> rec((size_t)nsites_ * S);
    be_d2h(rec.data(), site_rec_, sizeof(double) * rec.size());
    const int np = complex_ ? 2 : 1;                    // complex context: planar output (real block, imaginary block)
    for (int pl = 0; pl < np; ++pl)
      for (int w = 0; w < W_; ++w)
        for (int s = 0; s < nsites_; ++s)
          out[(size_t)pl * W_ * nsites_ + (size_t)w * nsites_ + s] = rec[(size_t)s * S + (size_t)pl * W_ + w];
  });
}
void Engine::clear_model_terms() {
  be_sync();
  for (auto &t : term_) free_table(t);
  free_table(pin_); pin_s1_ = pin_s2_ = -1;
  tables_on_ = false;
  tables_exchange_only_ = true;
}

// ---------------------------------------------------------------------------------------------------
// fermion mode (engine.h: set_fermion)
// ---------------------------------------------------------------------------------------------------
void Engine::bond_energy(int s1, int s2, const double *psi_ex, const double *psi, double jz, double jxy, double *target) {
  if (complex_) be_xxz_bond_energy_c(cfg_, nsites_, s1, s2, psi_ex, psi_ex + W_, psi, psi + W_, jz, jxy, target, target + W_, W_);
  else be_xxz_bond_energy(cfg_, nsites_, s1, s2, psi_ex, psi, jz, jxy, target, W_);
}
void Engine::set_complex() {
  if (complex_) return;
  if (fermion_ || tps_loaded_)
    throw std::logic_error("set_complex: call right after construction, before set_fermion / set_tps");
  be_sync();
  // per-walker scalar buffers allocated lazily so far are real-sized: drop them, they come back as planes
  be_free(psi_alt_); psi_alt_ = nullptr; psi_alt_slots_ = 0;
  be_free(psi_list_d_); psi_list_d_ = nullptr;
  be_free(bond_rec_); bond_rec_ = nullptr;
  be_free(site_rec_); site_rec_ = nullptr;
  if (sr_cap_ > 0) sr_reserve(0);
  auto grow = [&](double *&p, size_t n) { be_free(p); p = (double *)be_malloc(sizeof(double) * 2 * n); be_memset0(p, sizeof(double) * 2 * n); };
  grow(tps_, (size_t)tps_total_); gtps_ = tps_;
  grow(osum_, (size_t)tps_total_); grow(eosum_, (size_t)tps_total_);
  grow(amp_, (size_t)W_); grow(eloc_, (size_t)W_); grow(psi_tmp_, (size_t)W_); grow(psi_row_, (size_t)W_);
  grow(holes_, (size_t)W_ * hole_stride_);
  for (int p = 0; p < 4; ++p) {                     // tensors allocated so far are real-sized: drop them
    for (auto &b : bmps_[p]) release(b);
    bmps_[p].clear(); stamp_[p].clear();
    for (auto &m : memo_[p]) release(m.second.v);
    memo_[p].clear();
    for (auto &t : bten_[p]) release(t);
    bten_[p].clear();
    for (auto &t : bten2_[p]) release(t);
    bten2_[p].clear();
  }
  complex_ = true;
  touch_all();
}
void Engine::set_tps_c(const double *re, const double *im) {
  if (!complex_) throw std::logic_error("set_tps_c: the context is real (peps_set_complex)");
  be_h2d(tps_, re, sizeof(double) * tps_total_);
  be_h2d(tps_ + tps_total_, im, sizeof(double) * tps_total_);
  tps_loaded_ = true;
  if (fermion_) { dress_plane(re, gtps_); dress_plane(im, gtps_ + gtps_total_); }
  touch_all();
}
void Engine::get_planar(int what, double *re, double *im) {
  const double *p; size_t n;
  switch (what) {
    case 0: p = amp_; n = (size_t)W_; break;
    case 1: p = eloc_; n = (size_t)W_; break;
    case 2: p = holes_; n = (size_t)W_ * hole_stride_; break;
    case 3: p = osum_; n = (size_t)tps_total_; break;
    case 4: p = eosum_; n = (size_t)tps_total_; break;
    case 5: p = tps_; n = (size_t)tps_total_; break;
    default: throw std::invalid_argument("get_planar: unknown array");
  }
  if (re) be_d2h(re, p, sizeof(double) * n);
  if (im) {
    if (complex_) be_d2h(im, p + n, sizeof(double) * n);
    else std::fill(im, im + n, 0.0);
  }
}
void Engine::set_fermion(const int32_t *phys_par, const int32_t *leg_par) {
  if (!phys_par || !leg_par) throw std::invalid_argument("set_fermion: null table");
  if (fermion_) throw std::logic_error("set_fermion: already in fermion mode");
  if (tables_on_) throw std::logic_error("set_fermion: call it before set_model_term");
  for (int p = 0; p < phys_; ++p)
    if (phys_par[p] != 0 && phys_par[p] != 1) throw std::invalid_argument("set_fermion: parities must be 0 or 1");
  be_sync();
  phys_par_h_.assign(phys_par, phys_par + phys_);
  leg_par_h_.assign((size_t)nsites_ * 4, {});
  long pos = 0;
  for (int site = 0; site < nsites_; ++site)
    for (int k = 0; k < 4; ++k) {
      const int d = site_dims_h_[(size_t)site][(size_t)k];
      auto &v = leg_par_h_[(size_t)site * 4 + (size_t)k];
      v.assign(leg_par + pos, leg_par + pos + d);
      for (int x : v) if (x != 0 && x != 1) throw std::invalid_argument("set_fermion: parities must be 0 or 1");
      pos += d;
    }
  // the two ends of a bond must carry the same parities; boundary legs are even
  for (int r = 0; r < rows_; ++r)
    for (int c = 0; c < cols_; ++c) {
      const int s = r * cols_ + c;
      if (c + 1 < cols_ && leg_par_h_[(size_t)s * 4 + 2] != leg_par_h_[(size_t)(s + 1) * 4 + 0])
        throw std::invalid_argument("set_fermion: R / L parities of a horizontal bond differ");
      if (r + 1 < rows_ && leg_par_h_[(size_t)s * 4 + 1] != leg_par_h_[(size_t)(s + cols_) * 4 + 3])
        throw std::invalid_argument("set_fermion: D / U parities of a vertical bond differ");
      if ((c == 0 && leg_par_h_[(size_t)s * 4 + 0][0]) || (r == rows_ - 1 && leg_par_h_[(size_t)s * 4 + 1][0]) ||
          (c == cols_ - 1 && leg_par_h_[(size_t)s * 4 + 2][0]) || (r == 0 && leg_par_h_[(size_t)s * 4 + 3][0]))
        throw std::invalid_argument("set_fermion: boundary legs must be even");
    }
  fermion_ = true;
  la_.z2_sectors = true;
  if (const char *e = std::getenv("PEPS_Z2_SECTORS")) la_.z2_sectors = std::atoi(e) != 0;
  gtps_off_h_.resize((size_t)nsites_);
  for (int s = 0; s < nsites_; ++s) gtps_off_h_[(size_t)s] = tps_off_h_[(size_t)s] * FERMION_VARIANTS;
  gtps_total_ = tps_total_ * FERMION_VARIANTS;
  gtps_ = (double *)be_malloc(sizeof(double) * (size_t)gtps_total_ * (complex_ ? 2 : 1));
  be_memset0(gtps_, sizeof(double) * (size_t)gtps_total_ * (complex_ ? 2 : 1));
  if (complex_) la_.z2_sectors = false;               // the sector labels are those of Theta, not of its real embedding
  std::vector<int64_t> o64(gtps_off_h_.begin(), gtps_off_h_.end());
  gtps_off_d_ = (int64_t *)be_malloc(sizeof(int64_t) * nsites_);
  be_h2d(gtps_off_d_, o64.data(), sizeof(int64_t) * nsites_);
  for (int m = 0; m < 2; ++m) {
    gidx_[m] = (int32_t *)be_malloc(sizeof(int32_t) * (size_t)W_ * nsites_);
    jw_[m] = (int32_t *)be_malloc(sizeof(int32_t) * (size_t)W_ * nsites_);
  }
  phys_par_d_ = (int32_t *)be_malloc(sizeof(int32_t) * phys_);
  be_h2d(phys_par_d_, phys_par_h_.data(), sizeof(int32_t) * phys_);
  psi_loc_ = (double *)be_malloc(sizeof(double) * sw());
  if (!term_ia_) {
    term_ia_ = (int32_t *)be_malloc(sizeof(int32_t) * W_);
    term_ib_ = (int32_t *)be_malloc(sizeof(int32_t) * W_);
    term_cw_ = (double *)be_malloc(sizeof(double) * W_);
  }
  // sign of d psi_H / d T per element: (-1)^(l d + l r + d r + l + d + u J_H)
  std::vector<double> sg((size_t)hole_stride_ * 2);
  for (int site = 0; site < nsites_; ++site) {
    const auto &d = site_dims_h_[(size_t)site];
    const std::vector<int32_t> *par = &leg_par_h_[(size_t)site * 4];
    long e = hole_off_h_[(size_t)site];
    for (int l = 0; l < d[0]; ++l)
      for (int dd = 0; dd < d[1]; ++dd)
        for (int r = 0; r < d[2]; ++r)
          for (int u = 0; u < d[3]; ++u, ++e) {
            const int pl = par[0][(size_t)l], pd = par[1][(size_t)dd], pr = par[2][(size_t)r], pu = par[3][(size_t)u];
            const int q = (pl & pd) ^ (pl & pr) ^ (pd & pr) ^ pl ^ pd;
            sg[(size_t)e] = q ? -1.0 : 1.0;
            sg[(size_t)(hole_stride_ + e)] = (q ^ pu) ? -1.0 : 1.0;
          }
  }
  fsign_ = (double *)be_malloc(sizeof(double) * sg.size());
  be_h2d(fsign_, sg.data(), sizeof(double) * sg.size());
  refresh_gather();
  touch_all();
  if (tps_loaded_) {                                    // a state uploaded before the switch: dress it now
    std::vector<double> h((size_t)tps_total_ * (complex_ ? 2 : 1));
    be_d2h(h.data(), tps_, sizeof(double) * h.size());
    if (complex_) set_tps_c(h.data(), h.data() + tps_total_);
    else set_tps(h.data());
  }
}
void Engine::set_jastrow(const double *v, const int32_t *density) {
  if (!v || !density) throw std::invalid_argument("set_jastrow: null table");
  for (int i = 0; i < nsites_; ++i)
    for (int j = 0; j < i; ++j)
      if (v[(size_t)i * nsites_ + j] != v[(size_t)j * nsites_ + i]) throw std::invalid_argument("set_jastrow: v must be symmetric");
  be_sync();
  if (!jastrow_v_) {
    jastrow_v_ = (double *)be_malloc(sizeof(double) * (size_t)nsites_ * nsites_);
    jr_ = (double *)be_malloc(sizeof(double) * W_);
    dens_d_ = (int32_t *)be_malloc(sizeof(int32_t) * phys_);
  }
  be_h2d(jastrow_v_, v, sizeof(double) * (size_t)nsites_ * nsites_);
  be_h2d(dens_d_, density, sizeof(int32_t) * phys_);
  jastrow_on_ = true;
}
void Engine::refresh_gather() {
  if (fermion_) be_fermion_gather(cfg_, rows_, cols_, phys_, phys_par_d_, gidx_[HORIZONTAL], gidx_[VERTICAL], jw_[HORIZONTAL], jw_[VERTICAL], W_);
}

double *Engine::bond_target(int kind, int row, int col) {
  if (!rec_bonds_) return eloc_;
  const int nh = rows_ * (cols_ - 1), nv = (rows_ - 1) * cols_, nd = (rows_ - 1) * (cols_ - 1);
  const int idx = kind == 0 ? row * (cols_ - 1) + col : kind == 1 ? nh + row * cols_ + col
                : kind == 2 ? nh + nv + row * (cols_ - 1) + col : nh + nv + nd + row * (cols_ - 1) + col;
  return bond_rec_ + (size_t)idx * sw();
}
void Engine::upload_flipped_configs() {
  std::vector<int32_t> cfg((size_t)W_ * nsites_);
  be_d2h(cfg.data(), cfg_, sizeof(int32_t) * cfg.size());
  for (auto &c : cfg) c = 1 - c;
  if (!idx_flip_) idx_flip_ = (int32_t *)be_malloc(sizeof(int32_t) * cfg.size());
  be_h2d(idx_flip_, cfg.data(), sizeof(int32_t) * cfg.size());
}
// MeasureSpinOneHalfOffDiagOrderInRow (square_spin_onehalf_xxz_obc.h:22-60), lock step over the walkers: the tensor at
// (row, cols/4) is replaced by its flipped slice (tn.UpdateSiteTensor), the LEFT environment regrown across it, then
// one ReplaceOneSiteTrace with the flipped slice per site to the right. Ratios for equal spins are masked on the host.
void Engine::row_corr_hook(int row) {
  const int c1 = cols_ / 4, s1 = row * cols_ + c1, nc = cols_ / 2;
  const int nh = rows_ * (cols_ - 1), nv = (rows_ - 1) * cols_, nd = (rows_ - 1) * (cols_ - 1);
  double *corr = bond_rec_ + (size_t)(nh + nv + 2 * nd) * sw();
  auto truncate_left = [&]() {                                   // EraseEnvsAfterUpdate on the BTen stacks (:556-560)
    while ((int)bten_[LEFT].size() > c1 + 1) { release(bten_[LEFT].back()); bten_[LEFT].pop_back(); }
    while ((int)bten_[RIGHT].size() > cols_ - c1) { release(bten_[RIGHT].back()); bten_[RIGHT].pop_back(); }
  };
  override_site_ = s1; override_idx_ = idx_flip_ + s1; override_stride_ = nsites_;
  truncate_left();
  grow_bten_step(LEFT);
  grow_full_bten(RIGHT, row, c1 + 2, false);
  for (int i = 1; i <= nc; ++i) {
    const int c2 = c1 + i, s2 = row * cols_ + c2;
    one_site_trace(row, c2, idx_flip_ + s2, nsites_, psi_tmp_);
    ratio_acc(psi_tmp_, psi_row_, 1.0, corr + (size_t)(i - 1) * sw());
    shift_bten_window(RIGHT);
  }
  override_site_ = -1;
  truncate_left();
}
void Engine::measure(double *energy, double *e_h, double *e_v, double *e_dr, double *e_ur, double *row_corr) {
  // fermion mode: the same registry (energy, bond energies of the table model); the spin-1/2 row correlator is zero
  const bool builtin_xxz = !fermion_ && !tables_on_;   // table models (bosons and fermions) record their bond energies only
  if (builtin_xxz && tfim_) throw std::invalid_argument("measure: bond observables are defined for the XXZ / J1-J2 solvers and for table models");
  if (builtin_xxz && phys_ != 2) throw std::invalid_argument("measure: spin-1/2 observables need phys = 2");
  const int nh = rows_ * (cols_ - 1), nv = (rows_ - 1) * cols_, nd = (rows_ - 1) * (cols_ - 1), ncr = cols_ / 2;
  const int nb = nh + nv + 2 * nd;
  const size_t S = sw();
  const int np = complex_ ? 2 : 1;        // complex context: every output array is planar, its real block then its imaginary block
  if (!bond_rec_) bond_rec_ = (double *)be_malloc(sizeof(double) * (size_t)(nb + ncr) * S);
  be_memset0(bond_rec_, sizeof(double) * (size_t)(nb + ncr) * S);
  if (builtin_xxz) upload_flipped_configs();
  rec_bonds_ = true;
  try {
    energy_and_holes(false, nullptr, nullptr);            // with recording on, eloc_ only receives the on-site term
  } catch (...) { rec_bonds_ = false; override_site_ = -1; throw; }
  rec_bonds_ = false;
  std::vector<double> onsite(S);
  be_d2h(onsite.data(), eloc_, sizeof(double) * S);
  std::vector<double> rec((size_t)(nb + ncr) * S);
  be_d2h(rec.data(), bond_rec_, sizeof(double) * rec.size());
  auto scatter = [&](double *dst, int first, int count) {
    if (!dst) return;
    for (int pl = 0; pl < np; ++pl)
      for (int w = 0; w < W_; ++w)
        for (int i = 0; i < count; ++i)
          dst[(size_t)pl * W_ * count + (size_t)w * count + i] = rec[(size_t)(first + i) * S + (size_t)pl * W_ + w];
  };
  scatter(e_h, 0, nh); scatter(e_v, nh, nv); scatter(e_dr, nh + nv, nd); scatter(e_ur, nh + nv + nd, nd);
  if (row_corr) {
    std::vector<int32_t> cfg((size_t)W_ * nsites_);
    be_d2h(cfg.data(), cfg_, sizeof(int32_t) * cfg.size());
    const int row = rows_ / 2, c1 = cols_ / 4;
    for (int pl = 0; pl < np; ++pl)
      for (int w = 0; w < W_; ++w)
        for (int i = 0; i < ncr; ++i) {
          const int32_t *c = cfg.data() + (size_t)w * nsites_;
          const bool equal = c[row * cols_ + c1] == c[row * cols_ + c1 + i + 1];
          row_corr[(size_t)pl * W_ * ncr + (size_t)w * ncr + i] = (equal || !builtin_xxz) ? 0.0 : rec[(size_t)(nb + i) * S + (size_t)pl * W_ + w];
        }
  }
  if (energy)
    for (int pl = 0; pl < np; ++pl)
      for (int w = 0; w < W_; ++w) {
        double e = 0.0;
        for (int i = 0; i < nb; ++i) e += rec[(size_t)i * S + (size_t)pl * W_ + w];
        energy[(size_t)pl * W_ + w] = e + onsite[(size_t)pl * W_ + w];
      }
}
void Engine::measure_structure_factor(double *out_host) {
  require_boson("the structure-factor measurement");
  if (phys_ != 2) throw std::invalid_argument("measure_structure_factor: S+ S- correlators are defined for spin-1/2 (phys = 2)");
  ensure_idx_const();
  const int32_t *up_idx = idx_const_ + (size_t)1 * W_, *dn_idx = idx_const_;     // spin-up / spin-down slices for every walker
  const long npairs = structure_factor_pairs();
  const size_t S = sw();                                                           // complex: [pair][re W | im W]
  double *vals = (double *)pool_.get(sizeof(double) * (size_t)npairs * S);         // [pair][W]
  be_memset0(vals, sizeof(double) * (size_t)npairs * S);
  generate_bmps_approach(UP);                                  // the full DOWN stack (structure_factor...h:118)
  long pair = 0;
  for (int y1 = 0; y1 < rows_ - 1; ++y1) {
    while ((int)bmps_[UP].size() <= y1) grow_bmps_step(UP);    // main_walker.Evolve(row y1 - 1): the UP stack itself
    const BMPSv &main = bmps_[UP].at((size_t)y1);
    for (int x1 = 0; x1 < cols_; ++x1) {
      // excited row: S+ at (y1, x1) = the spin-up slice for every walker (a no-op where the spin is already up; those
      // walkers' values are masked below like the reference's zeros)
      override_site_ = y1 * cols_ + x1; override_idx_ = up_idx; override_stride_ = 1;
      BMPSv exc;
      try { exc = absorb(main, slice_sites(y1, HORIZONTAL), UP); } catch (...) { override_site_ = -1; pool_.put(vals); throw; }
      override_site_ = -1;
      for (int y2 = y1 + 1; y2 < rows_; ++y2) {
        const BMPSv &bottom = bmps_at_slice(DOWN, y2);
        std::vector<BT> left;                                  // InitBTenLeft over the whole row (bmps_walker.h)
        left.push_back(ones111());
        for (int x = 0; x < cols_; ++x)
          left.push_back(bten_step(left.back(), exc.at((size_t)(cols_ - 1 - x)), site_ref(y2 * cols_ + x, y2 * cols_ + x), bottom.at((size_t)x), LEFT));
        BT right = ones111();
        for (int x2 = cols_ - 1; x2 >= 0; --x2) {
          const int s2 = y2 * cols_ + x2;
          BT half = bten_step(left.at((size_t)x2), exc.at((size_t)(cols_ - 1 - x2)), site_ref_idx(s2, dn_idx, 1), bottom.at((size_t)x2), LEFT);
          reverse_dot(half, right, vals + (size_t)(pair + x2) * S);              // TraceWithBTen
          release(half);
          if (x2 > 0) {                                                           // GrowBTenRightStep
            BT nr = bten_step(right, bottom.at((size_t)x2), site_ref(s2, s2), exc.at((size_t)(cols_ - 1 - x2)), RIGHT);
            release(right);
            right = nr;
          }
        }
        release(right);
        for (auto &t : left) release(t);
        pair += cols_;
        if (y2 < rows_ - 1) {
          BMPSv nxt = absorb(exc, slice_sites(y2, HORIZONTAL), UP);
          release(exc);
          exc = std::move(nxt);
        }
      }
      release(exc);
    }
  }
  // mask on the host: S+ needs a down spin at the source, S- an up spin at the target; transpose to [W][pair]
  // (complex context: out_host is planar, the [W][pair] real block followed by the imaginary block)
  std::vector<double> h((size_t)npairs * S);
  std::vector<int32_t> cfg((size_t)W_ * nsites_);
  be_d2h(h.data(), vals, sizeof(double) * h.size());
  be_d2h(cfg.data(), cfg_, sizeof(int32_t) * cfg.size());
  pool_.put(vals);
  long p = 0;
  for (int y1 = 0; y1 < rows_ - 1; ++y1)
    for (int x1 = 0; x1 < cols_; ++x1)
      for (int y2 = y1 + 1; y2 < rows_; ++y2)
        for (int x2 = 0; x2 < cols_; ++x2, ++p)
          for (int w = 0; w < W_; ++w) {
            const int32_t *c = cfg.data() + (size_t)w * nsites_;
            const bool ok = c[y1 * cols_ + x1] == 0 && c[y2 * cols_ + x2] == 1;
            out_host[(size_t)w * npairs + p] = ok ? h[(size_t)p * S + w] : 0.0;
            if (complex_) out_host[(size_t)W_ * npairs + (size_t)w * npairs + p] = ok ? h[(size_t)p * S + W_ + w] : 0.0;
          }
}
void Engine::zero_accumulators() {
  be_memset0(osum_, sizeof(double) * tps_total_ * (complex_ ? 2 : 1));
  be_memset0(eosum_, sizeof(double) * tps_total_ * (complex_ ? 2 : 1));
}
void Engine::accumulate_ostar() {                      // mc_energy_grad_evaluator.h:245-272
  if (complex_) {
    be_accumulate_ostar_c(holes_, holes_ + (long)W_ * hole_stride_, hole_stride_, hole_off_d_, site_size_d_, tps_off_d_, cfg_, nsites_, amp_,
                          amp_ + W_, eloc_, eloc_ + W_, osum_, osum_ + tps_total_, eosum_, eosum_ + tps_total_, W_);
    if (sr_on_) {
      if (sr_count_ + W_ > sr_cap_) throw std::runtime_error("SR sample store is full (peps_sr_reserve)");
      be_sr_store_c(holes_, holes_ + (long)W_ * hole_stride_, hole_stride_, amp_, amp_ + W_, cfg_, nsites_, sr_ostar_, sr_cfgs_, sr_count_,
                    sr_cap_, W_);
      be_d2d(sr_eloc_ + sr_count_, eloc_, sizeof(double) * W_);
      be_d2d(sr_eloc_ + sr_cap_ + sr_count_, eloc_ + W_, sizeof(double) * W_);
      sr_count_ += W_;
    }
    return;
  }
  be_accumulate_ostar(holes_, hole_stride_, hole_off_d_, site_size_d_, tps_off_d_, cfg_, nsites_, phys_, amp_, eloc_,
                      osum_, eosum_, W_);
  if (sr_on_) {                                        // Ostar_samples.emplace_back(...)  (:273-277)
    if (sr_count_ + W_ > sr_cap_) throw std::runtime_error("SR sample store is full (peps_sr_reserve)");
    be_sr_store(holes_, hole_stride_, amp_, cfg_, nsites_, sr_ostar_, sr_cfgs_, sr_count_, W_);
    be_d2d(sr_eloc_ + sr_count_, eloc_, sizeof(double) * W_);
    sr_count_ += W_;
  }
}
void Engine::sr_reserve(long max_samples) {
  if (max_samples < 0) throw std::invalid_argument("sr_reserve: negative capacity");
  be_sync();
  be_free(sr_ostar_); be_free(sr_cfgs_); be_free(sr_delta_); be_free(sr_eloc_);
  sr_ostar_ = nullptr; sr_cfgs_ = nullptr; sr_delta_ = nullptr; sr_eloc_ = nullptr;
  sr_cap_ = max_samples; sr_count_ = 0;
  const size_t k = complex_ ? 4 : 1;                   // complex: x and y samples of doubled length (real embedding)
  if (max_samples > 0) {
    sr_ostar_ = (double *)be_malloc(sizeof(double) * (size_t)max_samples * hole_stride_ * k);
    sr_cfgs_ = (int32_t *)be_malloc(sizeof(int32_t) * (size_t)max_samples * nsites_ * k);
    sr_delta_ = (double *)be_malloc(sizeof(double) * (size_t)max_samples * (complex_ ? 2 : 1));
    sr_eloc_ = (double *)be_malloc(sizeof(double) * (size_t)max_samples * (complex_ ? 2 : 1));
  }
  if (complex_ && !sr_desc2_) {
    std::vector<int32_t> d((size_t)6 * nsites_);
    for (int s = 0; s < nsites_; ++s) {
      d[(size_t)s] = (int32_t)hole_off_h_[(size_t)s];
      d[(size_t)(nsites_ + s)] = (int32_t)(hole_stride_ + hole_off_h_[(size_t)s]);
      d[(size_t)(2 * nsites_ + s)] = d[(size_t)(3 * nsites_ + s)] = site_size_h_[(size_t)s];
      d[(size_t)(4 * nsites_ + s)] = (int32_t)tps_off_h_[(size_t)s];
      d[(size_t)(5 * nsites_ + s)] = (int32_t)(tps_total_ + tps_off_h_[(size_t)s]);
    }
    sr_desc2_ = (int32_t *)be_malloc(sizeof(int32_t) * d.size());
    be_h2d(sr_desc2_, d.data(), sizeof(int32_t) * d.size());
  }
}
// complex states: v, out planar [2][tps_total]; the x samples are centred with Re(mean . v), the y samples with Im
void Engine::sr_matvec_device_c(const double *v_dev, double mean_re, double mean_im, double *out_dev) {
  if (!complex_) throw std::logic_error("sr_matvec_device_c: the context is real");
  const int32_t *ho2 = sr_desc2_, *ss2 = sr_desc2_ + 2 * nsites_, *to2 = sr_desc2_ + 4 * nsites_;
  const long hs2 = 2 * hole_stride_;
  const int ns2 = 2 * nsites_;
  const double *oy = sr_ostar_ + (size_t)sr_cap_ * hs2;
  const int32_t *cy = sr_cfgs_ + (size_t)sr_cap_ * ns2;
  double *tmp = (double *)pool_.get(sizeof(double) * 2 * (size_t)tps_total_);
  be_sr_dots(sr_ostar_, sr_cfgs_, hs2, ho2, ss2, to2, ns2, v_dev, mean_re, sr_delta_, sr_count_);
  be_sr_dots(oy, cy, hs2, ho2, ss2, to2, ns2, v_dev, mean_im, sr_delta_ + sr_cap_, sr_count_);
  be_sr_accumulate(sr_ostar_, sr_cfgs_, hs2, ho2, ss2, to2, ns2, phys_, sr_delta_, out_dev, sr_count_);
  be_sr_accumulate(oy, cy, hs2, ho2, ss2, to2, ns2, phys_, sr_delta_ + sr_cap_, tmp, sr_count_);
  be_vec_lincomb(out_dev, 1.0, out_dev, 1.0, tmp, 2 * (long)tps_total_);
  pool_.put(tmp);
}
void Engine::sr_matvec_device(const double *v_dev, double mean_dot_v, double *out_dev) {
  require_real("sr_matvec with a real mean (peps_sr_matvec_c takes the planar vectors of a complex context)");
  // SRSMatrix::operator* without the 1/(N ranks) factor and the diagonal shift (applied by the caller after the
  // cross-GPU all-reduce): stochastic_reconfiguration_smatrix.h:60-66
  be_sr_dots(sr_ostar_, sr_cfgs_, hole_stride_, hole_off_d_, site_size_d_, tps_off_d_, nsites_, v_dev, mean_dot_v,
             sr_delta_, sr_count_);
  be_sr_accumulate(sr_ostar_, sr_cfgs_, hole_stride_, hole_off_d_, site_size_d_, tps_off_d_, nsites_, phys_, sr_delta_,
                   out_dev, sr_count_);
}
void Engine::sr_matvec_host_c(const double *v, double mean_re, double mean_im, double *out) {
  const size_t bytes = sizeof(double) * 2 * (size_t)tps_total_;
  double *vd = (double *)pool_.get(bytes);
  double *od = (double *)pool_.get(bytes);
  be_h2d(vd, v, bytes);
  sr_matvec_device_c(vd, mean_re, mean_im, od);
  be_d2h(out, od, bytes);
  pool_.put(vd);
  pool_.put(od);
}
void Engine::sr_matvec_host(const double *v, double mean_dot_v, double *out) {
  double *vd = (double *)pool_.get(sizeof(double) * tps_total_);
  double *od = (double *)pool_.get(sizeof(double) * tps_total_);
  be_h2d(vd, v, sizeof(double) * tps_total_);
  sr_matvec_device(vd, mean_dot_v, od);
  be_d2h(out, od, sizeof(double) * tps_total_);
  pool_.put(vd);
  pool_.put(od);
}
Engine::CGOutcome Engine::sr_natural_gradient(const double *gradient_host, const double *ostar_mean_host, long total_samples,
                                              double diag_shift, const CGParams &prm, const double *init_guess_host,
                                              AllReduceFn allreduce, void *user, double *x_host) {
  if (total_samples <= 0) throw std::invalid_argument("sr_natural_gradient: total_samples must be positive");
  // complex context: planar vectors of 2 tps_total doubles; the real dot of two planar vectors is Re <a, b>, which is all
  // the Hermitian CG needs (alpha, beta real); <mean, x> = dot(MEAN, x) + i dot(MEANJ, x) with MEANJ = J mean = [-m_i ; m_r]
  const long n = tps_total_ * (complex_ ? 2 : 1);
  const size_t bytes = sizeof(double) * (size_t)n;
  enum { B = 0, MEAN, X, R, P, AP, RPREV, BEST, MEANJ, NV };
  double *v[NV];
  for (auto &p : v) p = (double *)pool_.get(bytes);
  double *scal = (double *)pool_.get(sizeof(double) * 2);
  CGOutcome out;
  auto dot = [&](const double *a, const double *b2) {
    double h = 0.0;
    be_vec_dot(a, b2, n, scal);
    be_d2h(&h, scal, sizeof(double));
    return h;
  };
  // SRSMatrix::operator* (stochastic_reconfiguration_smatrix.h:45-91): local sum on the device, all-reduce of the
  // device buffer, 1/N and the diagonal shift
  auto matvec = [&](const double *x, double *y) {
    ++out.matvecs;
    const double mean_dot_v = dot(v[MEAN], x);
    if (complex_) sr_matvec_device_c(x, mean_dot_v, dot(v[MEANJ], x), y);
    else sr_matvec_device(x, mean_dot_v, y);
    if (allreduce) {
      be_sync();
      if (allreduce(user, y, (size_t)n) != 0) throw std::runtime_error("sr_natural_gradient: the all-reduce callback failed");
    }
    be_vec_lincomb(y, 1.0 / (double)total_samples, y, diag_shift, x, n);
  };
  auto finish = [&](const double *x, double rsq, int iters, int reason) {
    be_d2h(x_host, x, bytes);
    out.iterations = iters; out.residual_norm = std::sqrt(rsq); out.reason = reason;
    for (auto &p : v) pool_.put(p);
    pool_.put(scal);
    return out;
  };
  be_h2d(v[B], gradient_host, bytes);
  be_h2d(v[MEAN], ostar_mean_host, bytes);
  if (complex_) {
    be_d2d(v[MEANJ] + tps_total_, v[MEAN], bytes / 2);                   // im plane <- m_r
    be_vec_lincomb(v[MEANJ], -1.0, v[MEAN] + tps_total_, 0.0, nullptr, tps_total_);      // re plane <- -m_i
  }
  if (init_guess_host) be_h2d(v[X], init_guess_host, bytes); else be_memset0(v[X], bytes);
  const double rhs_sq = dot(v[B], v[B]);
  const double tol_sq = std::max(prm.rel_tol * prm.rel_tol * rhs_sq, prm.abs_tol * prm.abs_tol);
  matvec(v[X], v[AP]);
  be_vec_lincomb(v[R], 1.0, v[B], -1.0, v[AP], n);                       // r = b - A x0
  double r_sq = dot(v[R], v[R]);
  if (r_sq <= tol_sq) return finish(v[X], r_sq, 0, 0);
  be_d2d(v[P], v[R], bytes); be_d2d(v[BEST], v[X], bytes); be_d2d(v[RPREV], v[R], bytes);
  double best_sq = r_sq, rkp1 = r_sq;
  int stagnation = 0;
  const double eps = 2.220446049250313e-16;
  for (int k = 0; k < prm.max_iter; ++k) {
    const double rk = rkp1;
    matvec(v[P], v[AP]);
    const double pap = dot(v[P], v[AP]);
    if (!(std::isfinite(pap) && pap > 0.0)) return finish(v[BEST], best_sq, k, 3);          // kIndefiniteMatrix
    const double alpha = rk / pap;
    be_vec_lincomb(v[X], 1.0, v[X], alpha, v[P], n);
    if (alpha * alpha * dot(v[P], v[P]) < eps * eps * dot(v[X], v[X])) {
      if (++stagnation >= 3) return finish(v[BEST], best_sq, k + 1, 2);                    // kStagnated
    } else {
      stagnation = 0;
    }
    if (prm.recompute > 0 && (k % prm.recompute) == prm.recompute - 1) {
      matvec(v[X], v[AP]);
      be_vec_lincomb(v[R], 1.0, v[B], -1.0, v[AP], n);
    } else {
      be_vec_lincomb(v[R], 1.0, v[R], -alpha, v[AP], n);
    }
    rkp1 = dot(v[R], v[R]);
    if (!std::isfinite(rkp1)) return finish(v[BEST], best_sq, k + 1, 4);                   // kNumericalBreakdown
    if (rkp1 < best_sq) { be_d2d(v[BEST], v[X], bytes); best_sq = rkp1; }
    if (rkp1 <= tol_sq) return finish(v[X], rkp1, k + 1, 0);                               // kConverged
    if (k > 0 && std::fabs(dot(v[RPREV], v[R])) > prm.ortho * rkp1) {                      // orthogonality restart
      be_d2d(v[P], v[R], bytes); be_d2d(v[RPREV], v[R], bytes);
      continue;
    }
    be_d2d(v[RPREV], v[R], bytes);
    const double beta = rkp1 / rk;
    if (!std::isfinite(beta)) return finish(v[BEST], best_sq, k + 1, 4);
    be_vec_lincomb(v[P], 1.0, v[R], beta, v[P], n);
  }
  return finish(v[BEST], best_sq, prm.max_iter, 1);                                        // kMaxIterations
}
// MinSR centring: with a_i = <O*_i, Obar> and c = <Obar, Obar>, T = (G - a 1^T - 1 a^T + c 1 1^T) / N. A complex store
// holds x_i = [o_r; o_i] and y_i = J x_i; <y_i, y_j> = <x_i, x_j> and <x_i, y_j> = -<y_i, x_j>, so Re T comes from the
// Gram of the x rows and Im T = <y~_i, x~_j> / N = (<y_i, x_j> + f_i - f_j) / N with f_i = <x_i, J Obar>.
void Engine::minsr_centred_t(double *tr, double *ti, double *obar, double *gdiag_host) {
  const long N = sr_count_;
  const bool cx = complex_;
  const int32_t *ho = cx ? sr_desc2_ : hole_off_d_, *ss = cx ? sr_desc2_ + 2 * nsites_ : site_size_d_,
                *to = cx ? sr_desc2_ + 4 * nsites_ : tps_off_d_;
  const long hs = cx ? 2 * hole_stride_ : hole_stride_;
  const int ns = cx ? 2 * nsites_ : nsites_;
  const long tl = tps_total_ * (cx ? 2 : 1);
  std::vector<int32_t> ssh((size_t)ns);
  for (int s = 0; s < ns; ++s) ssh[(size_t)s] = site_size_h_[(size_t)(s % nsites_)];
  double *a = (double *)pool_.get(sizeof(double) * (size_t)N);
  double *G = (double *)pool_.get(sizeof(double) * (size_t)N * N);
  double *scal = (double *)pool_.get(sizeof(double));
  be_fill(a, 1.0 / (double)N, N);                                     // Obar = sum_i O*_i / N (one accumulate pass)
  be_sr_accumulate(sr_ostar_, sr_cfgs_, hs, ho, ss, to, ns, phys_, a, obar, N);
  be_sr_dots(sr_ostar_, sr_cfgs_, hs, ho, ss, to, ns, obar, 0.0, a, N);
  double c = 0.0;
  be_vec_dot(obar, obar, tl, scal);
  be_d2h(&c, scal, sizeof(double));
  be_sr_gram(sr_ostar_, sr_ostar_, sr_cfgs_, hs, ho, ss, ssh.data(), ns, N, 1.0, G);
  if (gdiag_host) {
    std::vector<double> g((size_t)N * N);
    be_d2h(g.data(), G, sizeof(double) * g.size());
    for (long i = 0; i < N; ++i) gdiag_host[i] = g[(size_t)(i * N + i)];
  }
  be_minsr_centre(G, a, c, 1.0, N, 1.0 / (double)N, tr);
  if (cx) {
    double *objt = (double *)pool_.get(sizeof(double) * (size_t)tl);
    be_d2d(objt + tps_total_, obar, sizeof(double) * tps_total_);                            // J Obar = [-Obar_i; Obar_r]
    be_vec_lincomb(objt, -1.0, obar + tps_total_, 0.0, nullptr, tps_total_);
    be_sr_dots(sr_ostar_, sr_cfgs_, hs, ho, ss, to, ns, objt, 0.0, a, N);                     // a = f
    be_vec_lincomb(a, -1.0, a, 0.0, nullptr, N);                                             // a = -f
    be_sr_gram(sr_ostar_ + (size_t)sr_cap_ * hs, sr_ostar_, sr_cfgs_, hs, ho, ss, ssh.data(), ns, N, -1.0, G);
    be_minsr_centre(G, a, 0.0, -1.0, N, 1.0 / (double)N, ti);
    pool_.put(objt);
  }
  pool_.put(a); pool_.put(G); pool_.put(scal);
}
void Engine::sr_minsr_tmatrix(double *t_host, double *gdiag_host) {
  const long N = sr_count_;
  if (N <= 0) throw std::invalid_argument("sr_minsr_tmatrix: the O* store is empty (collect samples with peps_sr_collect first)");
  const size_t nn = (size_t)N * N;
  double *t = (double *)pool_.get(sizeof(double) * nn * (complex_ ? 2 : 1));
  double *obar = (double *)pool_.get(sizeof(double) * (size_t)tps_total_ * (complex_ ? 2 : 1));
  minsr_centred_t(t, complex_ ? t + nn : nullptr, obar, gdiag_host);
  if (t_host) be_d2h(t_host, t, sizeof(double) * nn * (complex_ ? 2 : 1));
  pool_.put(t); pool_.put(obar);
}
void Engine::sr_minsr_natural_gradient(long total_samples, double diag_shift, double *x_host, double *energy_mean_host) {
  const long N = sr_count_;
  if (!(diag_shift > 0.0))
    throw std::invalid_argument("sr_minsr_natural_gradient: diag_shift must be positive (the centred T has the all-ones vector in "
                                "its null space, so T + diag_shift is singular at diag_shift = 0)");
  if (N <= 0) throw std::invalid_argument("sr_minsr_natural_gradient: the O* store is empty (Evaluate with collect_sr_buffers first)");
  if (total_samples != N)
    throw std::invalid_argument("sr_minsr_natural_gradient: total_samples (" + std::to_string(total_samples) + ") differs from the " +
                                std::to_string(N) + " samples in this context's store; MinSR needs every sample on one GPU");
  const bool cx = complex_;
  const size_t nn = (size_t)N * N;
  const long m = cx ? 2 * N : N, tl = tps_total_ * (cx ? 2 : 1);
  const double rs = 1.0 / std::sqrt((double)N);
  double *t = (double *)pool_.get(sizeof(double) * nn * (cx ? 2 : 1));
  double *obar = (double *)pool_.get(sizeof(double) * (size_t)tl);
  minsr_centred_t(t, cx ? t + nn : nullptr, obar, nullptr);
  // e_i = conj(E_i - Ebar) / sqrt(N), Ebar the plain mean (complex: the real embedding [Re; -Im])
  std::vector<double> eh((size_t)m), rhs((size_t)m);
  be_d2h(eh.data(), sr_eloc_, sizeof(double) * (size_t)N);
  if (cx) be_d2h(eh.data() + N, sr_eloc_ + sr_cap_, sizeof(double) * (size_t)N);
  double emean[2] = {0.0, 0.0};
  for (int p = 0; p < (cx ? 2 : 1); ++p) {
    for (long i = 0; i < N; ++i) emean[p] += eh[(size_t)(p * N + i)];
    emean[p] /= (double)N;
    for (long i = 0; i < N; ++i) rhs[(size_t)(p * N + i)] = (p ? -1.0 : 1.0) * (eh[(size_t)(p * N + i)] - emean[p]) * rs;
  }
  double *M = (double *)pool_.get(sizeof(double) * (size_t)m * m);
  double *z = (double *)pool_.get(sizeof(double) * (size_t)m);
  int32_t *info = (int32_t *)pool_.get(sizeof(int32_t));
  be_minsr_embed(t, cx ? t + nn : nullptr, N, diag_shift, M);
  be_chol(M, m, info);
  int32_t ih = 0;
  be_d2h(&ih, info, sizeof(int32_t));
  auto release = [&] { pool_.put(t); pool_.put(obar); pool_.put(M); pool_.put(z); pool_.put(info); };
  if (ih != 0) {
    release();
    throw std::runtime_error("sr_minsr_natural_gradient: non-positive Cholesky pivot " + std::to_string(ih) + " of T + diag_shift (" +
                             std::to_string(m) + " x " + std::to_string(m) + "); increase diag_shift");
  }
  be_h2d(z, rhs.data(), sizeof(double) * (size_t)m);
  be_chol_solve(M, m, z);
  std::vector<double> zh((size_t)m);
  be_d2h(zh.data(), z, sizeof(double) * (size_t)m);
  double zs[2] = {0.0, 0.0};
  for (long i = 0; i < m; ++i) zs[i / N] += zh[(size_t)i];
  // x = (sum_i z_i O*_i - (sum_i z_i) Obar) / sqrt(N); complex: x rows with z[:N], y rows (centred by J Obar) with z[N:]
  double *x = (double *)pool_.get(sizeof(double) * (size_t)tl);
  if (!cx) {
    be_sr_accumulate(sr_ostar_, sr_cfgs_, hole_stride_, hole_off_d_, site_size_d_, tps_off_d_, nsites_, phys_, z, x, N);
    be_vec_lincomb(x, rs, x, -zs[0] * rs, obar, tl);
  } else {
    const int32_t *ho2 = sr_desc2_, *ss2 = sr_desc2_ + 2 * nsites_, *to2 = sr_desc2_ + 4 * nsites_;
    const long hs2 = 2 * hole_stride_;
    const int ns2 = 2 * nsites_;
    double *tmp = (double *)pool_.get(sizeof(double) * (size_t)tl);
    be_sr_accumulate(sr_ostar_, sr_cfgs_, hs2, ho2, ss2, to2, ns2, phys_, z, x, N);
    be_sr_accumulate(sr_ostar_ + (size_t)sr_cap_ * hs2, sr_cfgs_ + (size_t)sr_cap_ * ns2, hs2, ho2, ss2, to2, ns2, phys_, z + N, tmp, N);
    be_vec_lincomb(x, rs, x, rs, tmp, tl);
    be_vec_lincomb(x, 1.0, x, -zs[0] * rs, obar, tl);
    // - zs[1] rs J Obar: re plane += zs[1] rs Obar_i, im plane -= zs[1] rs Obar_r
    be_vec_lincomb(x, 1.0, x, zs[1] * rs, obar + tps_total_, tps_total_);
    be_vec_lincomb(x + tps_total_, 1.0, x + tps_total_, -zs[1] * rs, obar, tps_total_);
    pool_.put(tmp);
  }
  be_d2h(x_host, x, sizeof(double) * (size_t)tl);
  if (energy_mean_host) { energy_mean_host[0] = emean[0]; if (cx) energy_mean_host[1] = emean[1]; }
  pool_.put(x);
  release();
}
void Engine::get_accumulators(double *osum_host, double *eosum_host) {
  if (osum_host) be_d2h(osum_host, osum_, sizeof(double) * tps_total_);
  if (eosum_host) be_d2h(eosum_host, eosum_, sizeof(double) * tps_total_);
}

long Engine::bmps_tensor(int pos, int k, int i, double *out_host, int dims[3]) {
  const BT &t = bmps_[pos].at((size_t)k).at((size_t)i);
  for (int a = 0; a < 3; ++a) dims[a] = t.d[a];
  if (out_host) be_d2h(out_host, t.p, sizeof(double) * (size_t)W_ * t.n);
  return t.n;
}
void Engine::probe_trace_row(int row, double *psi_host) {
  grow_bmps_for_row(row);
  init_bten(LEFT);
  grow_full_bten(RIGHT, row, 2, true);
  nn_trace(row, 0, row, 1, HORIZONTAL, row * cols_, row * cols_ + 1, psi_tmp_);
  be_d2h(psi_host, psi_tmp_, sizeof(double) * sw());
}

}  // namespace peps
