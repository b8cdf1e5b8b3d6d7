// extern "C" surface of libpeps_b200 (include/peps_b200.h). Exceptions never cross the ABI: every entry point
// catches, stores the message in the context (or a thread-local slot) and returns non-zero.
#include <cmath>
#include <cstring>
#include <memory>
#include <string>
#include <vector>
#include "../../include/peps_b200.h"
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include "engine.h"

using namespace peps;

struct peps_ctx {
  std::unique_ptr<Engine> eng;
  std::string err;
};
static thread_local std::string g_err;

// Every entry point first binds the context's device and stream to the calling host thread (Engine::bind), so a
// context may be driven from any thread (one at a time) and contexts on different devices may be interleaved.
#define GUARD(ctx, ...)                                    \
  try {                                                    \
    if (ctx) (ctx)->eng->bind();                           \
    __VA_ARGS__;                                           \
    return 0;                                              \
  } catch (const std::exception &e) {                      \
    if (ctx) (ctx)->err = e.what(); else g_err = e.what(); \
    return 1;                                              \
  } catch (...) {                                          \
    if (ctx) (ctx)->err = "unknown error"; else g_err = "unknown error"; \
    return 1;                                              \
  }

extern "C" {

const char *peps_backend_name(void) { return be_name(); }

int peps_create(peps_ctx **out, const peps_config *cfg) {
  peps_ctx *ctx = nullptr;
  try {
    if (!out || !cfg) throw std::invalid_argument("peps_create: null argument");
    ctx = new peps_ctx();
    EngineConfig ec;
    ec.rows = cfg->rows; ec.cols = cfg->cols; ec.phys = cfg->phys; ec.D = cfg->D; ec.walkers = cfg->walkers;
    ec.device = cfg->device; ec.dmin = cfg->dmin; ec.dmax = cfg->dmax; ec.trunc_err = cfg->trunc_err;
    ctx->eng.reset(new Engine(ec));
    *out = ctx;
    return 0;
  } catch (const std::exception &e) {
    g_err = e.what();
    delete ctx;
    if (out) *out = nullptr;
    return 1;
  }
}
void peps_destroy(peps_ctx *ctx) { delete ctx; }
const char *peps_last_error(peps_ctx *ctx) { return ctx ? ctx->err.c_str() : g_err.c_str(); }

size_t peps_tps_size(peps_ctx *ctx) { return ctx->eng->tps_size(); }
size_t peps_tps_site_offset(peps_ctx *ctx, int32_t row, int32_t col) { return (size_t)ctx->eng->site_offset(row, col); }
int peps_set_tps(peps_ctx *ctx, const double *h, size_t n) {
  GUARD(ctx, { if (n != ctx->eng->tps_size()) throw std::invalid_argument("peps_set_tps: size mismatch"); ctx->eng->set_tps(h); })
}
int peps_get_tps(peps_ctx *ctx, double *h, size_t n) {
  GUARD(ctx, { if (n != ctx->eng->tps_size()) throw std::invalid_argument("peps_get_tps: size mismatch"); ctx->eng->get_tps(h); })
}
int peps_set_truncation(peps_ctx *ctx, int32_t dmin, int32_t dmax, double terr) {
  GUARD(ctx, { if (dmin < 1 || dmax < dmin) throw std::invalid_argument("peps_set_truncation: need 1 <= dmin <= dmax"); ctx->eng->set_truncation(dmin, dmax, terr); })
}
int peps_set_compress_scheme(peps_ctx *ctx, int32_t scheme, double tol, int32_t max_iter) { GUARD(ctx, ctx->eng->set_compress_scheme(scheme, tol, max_iter)) }
int peps_set_jacobi(peps_ctx *ctx, double tol, int32_t inner, int32_t maxs) { GUARD(ctx, ctx->eng->set_jacobi(tol, inner, maxs)) }
int peps_set_deflation(peps_ctx *ctx, double eps) { GUARD(ctx, { if (eps < 0) throw std::invalid_argument("peps_set_deflation: eps < 0"); ctx->eng->set_deflation(eps); }) }
int peps_set_chain_deflation(peps_ctx *ctx, double eps) { GUARD(ctx, { if (eps < 0) throw std::invalid_argument("peps_set_chain_deflation: eps < 0"); ctx->eng->set_chain_deflation(eps); }) }
int peps_set_model_xxz(peps_ctx *ctx, double jz, double jxy, double h00) { GUARD(ctx, { ctx->eng->set_model_kind_xxz(); ctx->eng->set_model_xxz(jz, jxy, h00); ctx->eng->set_model_nnn(0.0, 0.0); }) }
int peps_set_model_j1j2_xxz(peps_ctx *ctx, double jz, double jxy, double jz2, double jxy2, double h00) {
  GUARD(ctx, { ctx->eng->set_model_kind_xxz(); ctx->eng->set_model_xxz(jz, jxy, h00); ctx->eng->set_model_nnn(jz2, jxy2); })
}
int peps_set_model_tfim(peps_ctx *ctx, double h) { GUARD(ctx, ctx->eng->set_model_tfim(h)) }
int peps_set_model_term(peps_ctx *ctx, int32_t kind, int32_t T, const double *diag, const int32_t *target, const double *coef) {
  GUARD(ctx, ctx->eng->set_model_term(kind, T, diag, target, coef))
}
int peps_clear_model_terms(peps_ctx *ctx) { GUARD(ctx, ctx->eng->clear_model_terms()) }
int peps_set_complex(peps_ctx *ctx) { GUARD(ctx, ctx->eng->set_complex()) }
int peps_set_tps_c(peps_ctx *ctx, const double *re, const double *im, size_t n) {
  GUARD(ctx, { if (n != ctx->eng->tps_size()) throw std::invalid_argument("peps_set_tps_c: wrong element count"); ctx->eng->set_tps_c(re, im); })
}
int peps_get_planar(peps_ctx *ctx, int32_t what, double *re, double *im) { GUARD(ctx, ctx->eng->get_planar(what, re, im)) }
int peps_set_jastrow(peps_ctx *ctx, const double *v, const int32_t *density) { GUARD(ctx, ctx->eng->set_jastrow(v, density)) }
int peps_clear_jastrow(peps_ctx *ctx) { GUARD(ctx, ctx->eng->clear_jastrow()) }
int peps_set_fermion(peps_ctx *ctx, const int32_t *phys_par, const int32_t *leg_par, size_t n_leg_par) {
  GUARD(ctx, {
    Engine &e = *ctx->eng;
    size_t need = 0;
    for (int r = 0; r < e.rows(); ++r)
      for (int c = 0; c < e.cols(); ++c) { int d[4]; e.site_dims(r, c, d); need += (size_t)(d[0] + d[1] + d[2] + d[3]); }
    if (n_leg_par != need) throw std::invalid_argument("peps_set_fermion: leg_par must hold " + std::to_string(need) + " entries");
    e.set_fermion(phys_par, leg_par);
  })
}
int peps_set_configs(peps_ctx *ctx, const int32_t *c) { GUARD(ctx, ctx->eng->set_configs(c)) }
int peps_get_configs(peps_ctx *ctx, int32_t *c) { GUARD(ctx, ctx->eng->get_configs(c)) }
int peps_seed_rng(peps_ctx *ctx, const uint32_t *s) { GUARD(ctx, ctx->eng->seed_rng(s)) }
int peps_set_rng_state(peps_ctx *ctx, const uint32_t *mt, const int32_t *idx) { GUARD(ctx, ctx->eng->set_rng_state(mt, idx)) }
int peps_get_rng_state(peps_ctx *ctx, uint32_t *mt, int32_t *idx) { GUARD(ctx, ctx->eng->get_rng_state(mt, idx)) }
int peps_init_walkers(peps_ctx *ctx) { GUARD(ctx, ctx->eng->init_walkers()) }
int peps_get_amplitudes(peps_ctx *ctx, double *a) { GUARD(ctx, ctx->eng->get_amplitudes(a)) }

int peps_normalize_state_order1(peps_ctx *ctx, double max_abs_override, double *site_factor_out) {
  GUARD(ctx, {
    Engine &e = *ctx->eng;
    double mx = max_abs_override;
    if (!(mx > 0.0)) {
      std::vector<double> a((size_t)e.walkers()), ai((size_t)e.walkers());
      e.get_planar(0, a.data(), ai.data());            // |psi| = hypot(re, im) (imaginary plane zero for real states)
      mx = 0.0;
      for (size_t k = 0; k < a.size(); ++k) mx = std::max(mx, std::hypot(a[k], ai[k]));
    }
    if (!(mx > 0.0) || !std::isfinite(mx)) throw std::runtime_error("peps_normalize_state_order1: amplitudes are zero or not finite");
    double scale = 1.0 / mx;
    double f = std::pow(scale, 1.0 / double(e.rows() * e.cols()));
    e.scale_tps(f);
    e.init_walkers();
    if (site_factor_out) *site_factor_out = f;
  })
}

int peps_sweep(peps_ctx *ctx, int32_t n, double *acc) { GUARD(ctx, ctx->eng->sweep(n, acc)) }
int peps_set_updater(peps_ctx *ctx, int32_t kind) { GUARD(ctx, ctx->eng->set_updater(kind)) }
int peps_sweep_three_site(peps_ctx *ctx, int32_t n, double *acc) { GUARD(ctx, ctx->eng->sweep_three_site(n, acc)) }
int peps_sweep_full_space(peps_ctx *ctx, int32_t n, double *acc) { GUARD(ctx, ctx->eng->sweep_full_space(n, acc)) }
int peps_energy_and_holes(peps_ctx *ctx, int32_t calc_holes, double *eloc, double *psi_list) {
  GUARD(ctx, ctx->eng->energy_and_holes(calc_holes != 0, eloc, psi_list))
}
int peps_measure(peps_ctx *ctx, double *energy, double *e_h, double *e_v, double *e_dr, double *e_ur, double *row_corr) {
  GUARD(ctx, ctx->eng->measure(energy, e_h, e_v, e_dr, e_ur, row_corr))
}
int64_t peps_structure_factor_pairs(peps_ctx *ctx) { return ctx->eng->structure_factor_pairs(); }
int peps_measure_bond_term(peps_ctx *ctx, int32_t T, const double *diag, const int32_t *target, const double *coef, double *out_h, double *out_v) {
  GUARD(ctx, ctx->eng->measure_bond_term(T, diag, target, coef, out_h, out_v))
}
int peps_measure_site_term(peps_ctx *ctx, int32_t T, const double *diag, const int32_t *target, const double *coef, double *out) {
  GUARD(ctx, ctx->eng->measure_site_term(T, diag, target, coef, out))
}
int peps_set_bond_pin(peps_ctx *ctx, int32_t site1, int32_t site2, int32_t T, const double *diag, const int32_t *target, const double *coef) {
  GUARD(ctx, ctx->eng->set_bond_pin(site1, site2, T, diag, target, coef))
}
int peps_measure_structure_factor(peps_ctx *ctx, double *out) { GUARD(ctx, ctx->eng->measure_structure_factor(out)) }
size_t peps_holes_stride(peps_ctx *ctx) { return (size_t)ctx->eng->holes_stride(); }
int peps_get_holes(peps_ctx *ctx, double *h) { GUARD(ctx, ctx->eng->get_holes(h)) }
int peps_zero_accumulators(peps_ctx *ctx) { GUARD(ctx, ctx->eng->zero_accumulators()) }
int peps_accumulate_ostar(peps_ctx *ctx) { GUARD(ctx, ctx->eng->accumulate_ostar()) }
int peps_get_accumulators(peps_ctx *ctx, double *o, double *eo, size_t n) {
  GUARD(ctx, { if (n != ctx->eng->tps_size()) throw std::invalid_argument("peps_get_accumulators: size mismatch"); ctx->eng->get_accumulators(o, eo); })
}
double *peps_ostar_sum_device(peps_ctx *ctx) { return ctx->eng->osum_device(); }
double *peps_eloc_ostar_sum_device(peps_ctx *ctx) { return ctx->eng->eosum_device(); }
int peps_sample(peps_ctx *ctx, int32_t sweeps, double *eloc, double *acc) {
  GUARD(ctx, {
    ctx->eng->step_sweep(sweeps, acc);
    ctx->eng->energy_and_holes(true, eloc, nullptr);
    ctx->eng->accumulate_ostar();
  })
}
int peps_sr_reserve(peps_ctx *ctx, int64_t n) { GUARD(ctx, ctx->eng->sr_reserve((long)n)) }
int peps_sr_collect(peps_ctx *ctx, int32_t on) { GUARD(ctx, ctx->eng->sr_collect(on != 0)) }
int peps_sr_clear(peps_ctx *ctx) { GUARD(ctx, ctx->eng->sr_clear()) }
int64_t peps_sr_count(peps_ctx *ctx) { return ctx->eng->sr_count(); }
int peps_sr_matvec(peps_ctx *ctx, const double *v, double mean_dot_v, double *out, size_t n) {
  GUARD(ctx, { if (n != ctx->eng->tps_size()) throw std::invalid_argument("peps_sr_matvec: size mismatch"); ctx->eng->sr_matvec_host(v, mean_dot_v, out); })
}
int peps_sr_matvec_c(peps_ctx *ctx, const double *v, double mean_re, double mean_im, double *out, size_t n) {
  GUARD(ctx, { if (n != 2 * ctx->eng->tps_size()) throw std::invalid_argument("peps_sr_matvec_c: size mismatch (planar vectors of 2 * peps_tps_size() doubles)"); ctx->eng->sr_matvec_host_c(v, mean_re, mean_im, out); })
}
int peps_sr_matvec_device(peps_ctx *ctx, const double *v, double mean_dot_v, double *out) { GUARD(ctx, ctx->eng->sr_matvec_device(v, mean_dot_v, out)) }
int peps_sr_natural_gradient(peps_ctx *ctx, const double *gradient, const double *ostar_mean, int64_t total_samples, double diag_shift,
                             const peps_cg_params *prm, const double *init_guess, peps_allreduce_fn allreduce, void *user, double *x_out,
                             int32_t *iterations, double *residual_norm, int32_t *reason) {
  GUARD(ctx, {
    if (!gradient || !ostar_mean || !x_out) throw std::invalid_argument("peps_sr_natural_gradient: null argument");
    Engine::CGParams p;
    if (prm) { p.max_iter = prm->max_iter; p.rel_tol = prm->relative_tolerance; p.abs_tol = prm->absolute_tolerance;
               p.recompute = prm->residual_recompute_interval; p.ortho = prm->orthogonality_threshold; }
    Engine::CGOutcome o = ctx->eng->sr_natural_gradient(gradient, ostar_mean, (long)total_samples, diag_shift, p, init_guess, allreduce, user, x_out);
    if (iterations) *iterations = o.iterations;
    if (residual_norm) *residual_norm = o.residual_norm;
    if (reason) *reason = o.reason;
  })
}
int peps_sr_minsr_natural_gradient(peps_ctx *ctx, int64_t total_samples, double diag_shift, double *x_out, double *energy_mean_out) {
  GUARD(ctx, {
    if (!x_out) throw std::invalid_argument("peps_sr_minsr_natural_gradient: null x_out");
    ctx->eng->sr_minsr_natural_gradient((long)total_samples, diag_shift, x_out, energy_mean_out);
  })
}
int peps_sr_minsr_tmatrix(peps_ctx *ctx, double *t_out, size_t n) {
  GUARD(ctx, {
    const size_t N = (size_t)ctx->eng->sr_count(), want = N * N * (ctx->eng->is_complex() ? 2 : 1);
    if (n != want) throw std::invalid_argument("peps_sr_minsr_tmatrix: size mismatch (N * N doubles, 2 * N * N in a complex context, N = peps_sr_count)");
    ctx->eng->sr_minsr_tmatrix(t_out, nullptr);
  })
}
int peps_sr_minsr_gram_diag(peps_ctx *ctx, double *g_out, size_t n) {
  GUARD(ctx, {
    if (n != (size_t)ctx->eng->sr_count()) throw std::invalid_argument("peps_sr_minsr_gram_diag: size mismatch (peps_sr_count doubles)");
    ctx->eng->sr_minsr_tmatrix(nullptr, g_out);
  })
}
int peps_probe_trace_row(peps_ctx *ctx, int32_t row, double *psi) { GUARD(ctx, ctx->eng->probe_trace_row(row, psi)) }
int peps_probe_tnn_trace(peps_ctx *ctx, int32_t row, int32_t col, int32_t orient, const int32_t *cfg3, double *psi) {
  GUARD(ctx, {
    const int n = orient == 0 ? ctx->eng->cols() : ctx->eng->rows(), i0 = orient == 0 ? col : row;
    if (orient < 0 || orient > 1 || row < 0 || col < 0 || row >= ctx->eng->rows() || col >= ctx->eng->cols() || i0 + 2 >= n)
      throw std::invalid_argument("peps_probe_tnn_trace: the three sites do not fit the lattice");
    ctx->eng->probe_tnn_trace(row, col, orient, cfg3, psi);
  })
}
int peps_probe_plaquette_trace(peps_ctx *ctx, int32_t kind, int32_t row, int32_t col, int32_t dir, int32_t orient, double *psi) {
  GUARD(ctx, {
    Engine &e = *ctx->eng;
    const int span = kind == 0 ? 2 : 3;
    const int h = orient == 0 ? 2 : span, wd = orient == 0 ? span : 2;
    if (kind < 0 || kind > 1 || dir < 0 || dir > 1 || orient < 0 || orient > 1 || row < 0 || col < 0 || row + h > e.rows() || col + wd > e.cols())
      throw std::invalid_argument("peps_probe_plaquette_trace: the plaquette does not fit the lattice");
    e.probe_plaquette_trace(kind, row, col, dir, orient, psi);
  })
}
int32_t peps_bmps_stack_size(peps_ctx *ctx, int32_t pos) { return ctx->eng->bmps_stack_size(pos); }
int peps_get_bmps_tensor(peps_ctx *ctx, int32_t pos, int32_t k, int32_t i, double *out, int32_t dims[3]) {
  GUARD(ctx, { int d[3]; ctx->eng->bmps_tensor(pos, k, i, out, d); for (int a = 0; a < 3; ++a) dims[a] = d[a]; })
}
int64_t peps_stat(peps_ctx *ctx, int32_t which) { return ctx->eng->stat(which); }
int peps_sync(peps_ctx *ctx) { GUARD(ctx, be_sync()) }
int peps_profile_enable(peps_ctx *ctx, int32_t on) { GUARD(ctx, be_profile_enable(on)) }
int peps_profile_get(peps_ctx *ctx, double *ms, int64_t *launches, double *flops, int32_t reset) {
  GUARD(ctx, {
    long l[KC_COUNT];
    be_profile_collect(ms, l, flops, reset);
    if (launches) for (int c = 0; c < KC_COUNT; ++c) launches[c] = l[c];
  })
}
void *peps_stream(peps_ctx *ctx) {
  try { ctx->eng->bind(); return be_stream(); } catch (...) { return nullptr; }
}

// ---- stand-alone kernel tests -----------------------------------------------------------------------
int peps_test_qr_r(int32_t device, int32_t W, int32_t m, int32_t n, const double *a, double *r_out) {
  peps_ctx *nullctx = nullptr;
  GUARD(nullctx, {
    be_init(device);
    Pool pool; Planner planner; LinalgCtx cx;
    cx.W = W; cx.pool = &pool; cx.planner = &planner;
    QRLayout L = qr_layout(m, n);
    double *A = (double *)pool.get(sizeof(double) * (size_t)W * L.m_pad * n);
    be_memset0(A, sizeof(double) * (size_t)W * L.m_pad * n);
    double *tmp = (double *)pool.get(sizeof(double) * (size_t)W * m * n);
    be_h2d(tmp, a, sizeof(double) * (size_t)W * m * n);
    be_copy2d(A, (long)L.m_pad * n, n, tmp, (long)m * n, n, m, n, W);
    caqr(cx, A, (long)L.m_pad * n, m, n, L);
    int kk = std::min(m, n);
    double *R = (double *)pool.get(sizeof(double) * (size_t)W * kk * n);
    be_copy2d(R, (long)kk * n, n, A, (long)L.m_pad * n, n, kk, n, W);
    be_d2h(r_out, R, sizeof(double) * (size_t)W * kk * n);
  })
}

int peps_test_truncate(int32_t device, int32_t W, int32_t nr, int32_t nc, int32_t dmin, int32_t dmax, double trunc_err,
                       const double *theta, double *b_out, int32_t *kept_out, int32_t *sweeps_out) {
  peps_ctx *nullctx = nullptr;
  GUARD(nullctx, {
    be_init(device);
    Pool pool; Planner planner; LinalgCtx cx;
    cx.W = W; cx.pool = &pool; cx.planner = &planner;
    if (const char *e = std::getenv("PEPS_PRESORT_COLS")) cx.presort_columns = std::atoi(e) != 0;
    if (const char *e = std::getenv("PEPS_SMALL_SVD")) cx.small_svd = std::atoi(e) != 0;
    if (const char *e = std::getenv("PEPS_QR_EARLY_STOP")) cx.qr_early_stop = std::atoi(e) != 0;
    if (const char *e = std::getenv("PEPS_Z2_SECTORS")) cx.z2_sectors = std::atoi(e) != 0;     // test hook: block-diagonal Theta
    cx.offmax = (double *)pool.get(sizeof(double) * W);
    cx.done = (int32_t *)pool.get(sizeof(int32_t) * W);
    int brows = truncate_buffer_rows(nr, nc);
    double *G = (double *)pool.get(sizeof(double) * (size_t)W * brows * nc);
    be_memset0(G, sizeof(double) * (size_t)W * brows * nc);
    double *tmp = (double *)pool.get(sizeof(double) * (size_t)W * nr * nc);
    be_h2d(tmp, theta, sizeof(double) * (size_t)W * nr * nc);
    be_copy2d(G, (long)brows * nc, nc, tmp, (long)nr * nc, nc, nr, nc, W);
    int tcap = std::min(dmax, std::min(nr, nc));
    double *B = (double *)pool.get(sizeof(double) * (size_t)W * tcap * nc);
    int32_t *kept = (int32_t *)pool.get(sizeof(int32_t) * W);
    truncate_rows(cx, G, (long)brows * nc, nr, nc, dmin, dmax, trunc_err, tcap, B, (long)tcap * nc, kept);
    be_d2h(b_out, B, sizeof(double) * (size_t)W * tcap * nc);
    be_d2h(kept_out, kept, sizeof(int32_t) * W);
    if (sweeps_out) *sweeps_out = (int32_t)cx.jacobi_sweeps;
  })
}

int peps_test_einsum(int32_t device, int32_t W, const char *spec, const int32_t *dims_a, int32_t rank_a,
                     const int32_t *dims_b, int32_t rank_b, const double *a, const double *b, double *c) {
  peps_ctx *nullctx = nullptr;
  GUARD(nullctx, {
    be_init(device);
    Pool pool; Planner planner;
    int da[6], db[6];
    long na = 1, nb = 1;
    for (int i = 0; i < rank_a; ++i) { da[i] = dims_a[i]; na *= da[i]; }
    for (int i = 0; i < rank_b; ++i) { db[i] = dims_b[i]; nb *= db[i]; }
    const Plan &pl = planner.get(spec, da, rank_a, db, rank_b);
    double *A = (double *)pool.get(sizeof(double) * (size_t)W * na);
    double *Bp = (double *)pool.get(sizeof(double) * (size_t)W * nb);
    double *C = (double *)pool.get(sizeof(double) * (size_t)W * pl.outn);
    be_h2d(A, a, sizeof(double) * (size_t)W * na);
    be_h2d(Bp, b, sizeof(double) * (size_t)W * nb);
    be_gett(pl.d, mkop(A, na), mkop(Bp, nb), mkop(C, pl.outn), 1.0, 0.0, W, 1);
    if (const char *e = std::getenv("PEPS_EINSUM_TIME")) {      // development aid: device time of `e` repetitions
      const int reps = std::max(1, std::atoi(e));
      be_profile_enable(1);
      double ms[KC_COUNT]; long ln[KC_COUNT]; double fl[KC_COUNT];
      be_profile_collect(ms, ln, fl, 1);
      for (int r = 0; r < reps; ++r) be_gett(pl.d, mkop(A, na), mkop(Bp, nb), mkop(C, pl.outn), 1.0, 0.0, W, 1);
      be_sync();
      be_profile_collect(ms, ln, fl, 1);
      be_profile_enable(0);
      std::fprintf(stderr, "[einsum] %s W=%d M=%d K=%d N=%d: %.1f us per call, %.2f TFLOP/s\n", spec, W, pl.d.M, pl.d.K, pl.d.N,
                   1e3 * ms[KC_GETT] / reps, fl[KC_GETT] / (ms[KC_GETT] * 1e9));
    }
    be_d2h(c, C, sizeof(double) * (size_t)W * pl.outn);
  })
}

}  // extern "C"
