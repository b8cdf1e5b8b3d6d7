// C++ host-side wrapper over the C ABI (include/peps_b200.h), mirroring the reference's interface names for the
// VMC sampling path so existing drivers keep their shape:
//   qlpeps::BMPSTruncateParams            one_dim_tn/boundary_mps/bmps.h:47-98
//   qlpeps::MonteCarloParams              algorithm/vmc_update/monte_carlo_peps_params.h:37-92
//   qlpeps::MCEnergyGradEvaluator         algorithm/vmc_update/mc_energy_grad_evaluator.h:57-330
//   evaluator callback (seam B1)          algorithm/vmc_update/vmc_peps_optimizer.h:155-157
// Errors from the ABI become std::runtime_error, like the reference's own failure paths
// (bmps_impl.h:839-843, square_nnn_energy_solver.h:148-150). Header-only; link against libpeps_b200.so.
#pragma once
#include <cmath>
#include <complex>
#include <cstdint>
#include <functional>
#include <limits>
#include <map>
#include <stdexcept>
#include <string>
#include <tuple>
#include <vector>
#include "peps_b200.h"

namespace peps_b200 {

struct BMPSTruncateParams {
  size_t D_min = 1, D_max = 1;
  double trunc_err = 0.0;
  static BMPSTruncateParams SVD(size_t dmin, size_t dmax, double err) { return {dmin, dmax, err}; }
};

struct MonteCarloParams {
  size_t num_samples = 0, num_warmup_sweeps = 0, sweeps_between_samples = 1;
  std::vector<int32_t> initial_config;   // rows*cols physical indices (row-major); replicated to every walker
  bool is_warmed_up = false;
};

struct XXZModel { double jz = 1.0, jxy = 1.0, pinning00 = 0.0; };   // SquareSpinOneHalfXXZModelOBC(jz, jxy, pinning)
struct J1J2XXZModel { double jz = 1.0, jxy = 1.0, jz2 = 0.0, jxy2 = 0.0, pinning00 = 0.0; };   // SquareSpinOneHalfJ1J2XXZModelOBC
struct TransverseFieldIsingModel { double h = 1.0; };                 // TransverseFieldIsingSquareOBC(h)
// ---- seam B2 as data ------------------------------------------------------------------------------------------------
// A model term as tables (peps_set_model_term). ProbeTwoSiteTerm / ProbeOneSiteTerm build them from a reference-style
// bond-energy functor: the reference's mix-in hook
//   EvaluateBondEnergy(site1, site2, cfg1, cfg2, orient, tn, contractor, sitps1, sitps2, inv_psi)
// (model_solvers/base/square_nnn_energy_solver.h:171-198) is pure arithmetic on (cfg1, cfg2), the couplings and the
// amplitude ratios psi(S')/psi(S) it obtains through contractor.ReplaceNNSiteTrace(...) * inv_psi. The probe calls the
// functor with a recording `ratio(c1', c2')` callback: once returning 0 (-> the diagonal element), then once per recorded
// target with an indicator ratio (-> the matrix element). Any model whose bond energy is linear in the ratios -- every
// model of the reference -- becomes a table, and the engine needs no patch.
struct ModelTerm {
  int32_t kind = 0;                    // 0 NN bonds, 1 NNN links, 2 on-site
  int32_t T = 0;                       // target slots per local state
  std::vector<double> diag, coef;      // [np], [np * T]
  std::vector<int32_t> target;         // [np * T], -1 = unused
};
// f(c1, c2, ratio) -> bond energy, ratio(c1', c2') = psi(S with (c1,c2) -> (c1',c2')) / psi(S)
inline ModelTerm ProbeTwoSiteTerm(int32_t kind, int phys,
                                  const std::function<double(int, int, const std::function<double(int, int)> &)> &f) {
  const int np = phys * phys;
  std::vector<std::vector<int>> tg((size_t)np);
  std::vector<std::vector<double>> cf((size_t)np);
  ModelTerm m;
  m.kind = kind; m.diag.assign((size_t)np, 0.0);
  for (int p = 0; p < np; ++p) {
    std::vector<int> seen;
    m.diag[(size_t)p] = f(p / phys, p % phys, [&](int a, int b) { int q = a * phys + b; if (q != p) { bool k = false; for (int s : seen) k |= (s == q); if (!k) seen.push_back(q); } return 0.0; });
    for (int q : seen) {
      const double v = f(p / phys, p % phys, [&](int a, int b) { return (a * phys + b == q) ? 1.0 : 0.0; }) - m.diag[(size_t)p];
      if (v != 0.0) { tg[(size_t)p].push_back(q); cf[(size_t)p].push_back(v); }
    }
    m.T = std::max<int32_t>(m.T, (int32_t)tg[(size_t)p].size());
  }
  m.target.assign((size_t)np * std::max(m.T, 1), -1); m.coef.assign((size_t)np * std::max(m.T, 1), 0.0);
  for (int p = 0; p < np; ++p)
    for (size_t t = 0; t < tg[(size_t)p].size(); ++t) { m.target[(size_t)p * m.T + t] = tg[(size_t)p][t]; m.coef[(size_t)p * m.T + t] = cf[(size_t)p][t]; }
  return m;
}
// f(c, ratio) -> on-site energy, ratio(c') = psi(S with c -> c') / psi(S)
inline ModelTerm ProbeOneSiteTerm(int phys, const std::function<double(int, const std::function<double(int)> &)> &f) {
  ModelTerm m;
  m.kind = 2; m.diag.assign((size_t)phys, 0.0);
  std::vector<std::vector<int>> tg((size_t)phys);
  std::vector<std::vector<double>> cf((size_t)phys);
  for (int p = 0; p < phys; ++p) {
    std::vector<int> seen;
    m.diag[(size_t)p] = f(p, [&](int q) { if (q != p) { bool k = false; for (int s : seen) k |= (s == q); if (!k) seen.push_back(q); } return 0.0; });
    for (int q : seen) {
      const double v = f(p, [&](int a) { return a == q ? 1.0 : 0.0; }) - m.diag[(size_t)p];
      if (v != 0.0) { tg[(size_t)p].push_back(q); cf[(size_t)p].push_back(v); }
    }
    m.T = std::max<int32_t>(m.T, (int32_t)tg[(size_t)p].size());
  }
  m.target.assign((size_t)phys * std::max(m.T, 1), -1); m.coef.assign((size_t)phys * std::max(m.T, 1), 0.0);
  for (int p = 0; p < phys; ++p)
    for (size_t t = 0; t < tg[(size_t)p].size(); ++t) { m.target[(size_t)p * m.T + t] = tg[(size_t)p][t]; m.coef[(size_t)p * m.T + t] = cf[(size_t)p][t]; }
  return m;
}
// SquareSpinOneHalfXXZModelMixIn::EvaluateBondEnergy (square_spin_onehalf_xxz_obc.h:72-104) written against the probe
inline ModelTerm XXZBondTerm(int32_t kind, double jz, double jxy) {
  return ProbeTwoSiteTerm(kind, 2, [=](int c1, int c2, const std::function<double(int, int)> &ratio) {
    if (c1 == c2) return 0.25 * jz;
    return -0.25 * jz + ratio(c2, c1) * 0.5 * jxy;
  });
}

// SquareSpinlessFermion::EvaluateBondEnergy / EvaluateNNNEnergy (square_spinless_fermion.h:118-211) against the probe:
// states 0 = occupied, 1 = empty; the ratio is psi_ex / psi along one contraction path (fermion mode of the engine).
inline ModelTerm SpinlessFermionBondTerm(double t, double V) {
  return ProbeTwoSiteTerm(0, 2, [=](int c1, int c2, const std::function<double(int, int)> &ratio) {
    const double e = V * double(1 - c1) * double(1 - c2);
    return c1 == c2 ? e : -t * ratio(c2, c1) + e;
  });
}
inline ModelTerm SpinlessFermionNNNTerm(double t2) {
  return ProbeTwoSiteTerm(1, 2, [=](int c1, int c2, const std::function<double(int, int)> &ratio) {
    return c1 == c2 ? 0.0 : -t2 * ratio(c2, c1);
  });
}
// SquaretJModelMixIn::EvaluateBondEnergy (square_tJ_model.h:300-345): 0 = up, 1 = down, 2 = empty
inline ModelTerm tJBondTerm(double t, double J, double V) {
  return ProbeTwoSiteTerm(0, 3, [=](int c1, int c2, const std::function<double(int, int)> &ratio) {
    if (c1 == c2) return c1 == 2 ? 0.0 : V;
    if (c1 == 2 || c2 == 2) return -t * ratio(c2, c1);
    return (-0.5 + ratio(c2, c1) * 0.5) * J + V;
  });
}
// SquaretJModelMixIn::EvaluateNNNEnergy (square_tJ_model.h:424-460): t2 hopping when exactly one site is empty
inline ModelTerm tJNNNTerm(double t2) {
  return ProbeTwoSiteTerm(1, 3, [=](int c1, int c2, const std::function<double(int, int)> &ratio) {
    if (c1 == c2 || (c1 != 2 && c2 != 2)) return 0.0;
    return -t2 * ratio(c2, c1);
  });
}
// EvaluateBondSingletPairFortJModel (square_tJ_model.h:546-602) against the probe: delta_dag (which = 0), delta (which = 1)
// or the pinning source delta_pin * (delta_dag + delta) (which = 2; SetSingletPairPinningField, :86-137, 256-289)
inline ModelTerm tJSingletPairTerm(int which, double delta_pin = 1.0) {
  const double s = 1.0 / std::sqrt(2.0);
  return ProbeTwoSiteTerm(0, 3, [=](int c1, int c2, const std::function<double(int, int)> &ratio) {
    double dd = 0.0, d = 0.0;
    if (c1 == 2 && c2 == 2) dd = (ratio(0, 1) - ratio(1, 0)) * s;
    else if (c1 == 0 && c2 == 1) d = ratio(2, 2) * s;
    else if (c1 == 1 && c2 == 0) d = -ratio(2, 2) * s;
    return which == 0 ? dd : which == 1 ? d : delta_pin * (dd + d);
  });
}
// EvaluateTotalOnsiteEnergy of the t-J models (square_tJ_model.h:248-262): -mu per electron
inline ModelTerm tJOnsiteTerm(double mu) {
  return ProbeOneSiteTerm(3, [=](int c, const std::function<double(int)> &) { return c == 2 ? 0.0 : -mu; });
}
// Parities of a QLTensor<T, fZ2QN> SplitIndexTPS for WalkerBatch::SetFermion: phys_par[s] = parity of physical state s,
// leg_par = per site (row-major) the parity of every index value of the L, D, R, U legs, concatenated.
struct FermionParities {
  std::vector<int32_t> phys_par, leg_par;
};

// ---- runtime parameter packs (algorithm/vmc_update/monte_carlo_peps_params.h) and their free functions -----------------
struct ConfigurationRescueParams {
  bool enabled = true;
  double amplitude_min_threshold = std::numeric_limits<double>::min();
  double amplitude_max_threshold = std::numeric_limits<double>::max();
};
// CheckWaveFunctionAmplitudeValidity (vmc_basic/wave_function_component.h:393-401)
inline bool CheckWaveFunctionAmplitudeValidity(double amplitude, double min_threshold, double max_threshold) {
  const double a = std::fabs(amplitude);
  return !std::isnan(a) && !std::isinf(a) && a > min_threshold && a < max_threshold;
}
// ComputePsiConsistencySummaryAligned (algorithm/vmc_update/psi_consistency.h:76-130): {psi_mean, psi_rel_err}
inline std::pair<double, double> ComputePsiConsistencySummaryAligned(const std::vector<double> &psi) {
  if (psi.empty()) return {0.0, 0.0};
  size_t ri = 0;
  for (size_t i = 0; i < psi.size(); ++i) if (std::fabs(psi[i]) > std::fabs(psi[ri])) ri = i;
  const bool ref_valid = std::fabs(psi[ri]) > 1e-14;
  std::vector<double> al(psi);
  double mean = 0.0;
  for (auto &v : al) { if (ref_valid && v * psi[ri] < 0.0) v = -v; mean += v; }
  mean /= (double)psi.size();
  const double denom = std::max(std::fabs(mean), std::numeric_limits<double>::epsilon());
  double dev = 0.0;
  for (double v : al) dev = std::max(dev, std::fabs(v - mean));
  return {mean, dev / denom};
}

enum class Updater : int32_t { NNExchange = 0, NNFullSpace = 1, TNN3SiteExchange = 2 };   // MCUpdateSquareNNExchangeOBC / ...NNFullSpaceUpdateOBC / MCUpdateSquareTNN3SiteExchange

class WalkerBatch {
 public:
  WalkerBatch(int rows, int cols, int phys, int D, int walkers, const BMPSTruncateParams &t, int device = 0)
      : rows_(rows), cols_(cols), walkers_(walkers) {
    peps_config c{rows, cols, phys, D, walkers, device, (int32_t)t.D_min, (int32_t)t.D_max, t.trunc_err};
    if (peps_create(&h_, &c) != 0) throw std::runtime_error(peps_last_error(nullptr));
  }
  ~WalkerBatch() { if (h_) peps_destroy(h_); }
  WalkerBatch(const WalkerBatch &) = delete;
  WalkerBatch &operator=(const WalkerBatch &) = delete;
  size_t tps_size() const { return peps_tps_size(h_); }
  int walkers() const { return walkers_; }
  void SetTPS(const std::vector<double> &flat) { ck(peps_set_tps(h_, flat.data(), flat.size())); }
  // QLTEN_Complex states (SplitIndexTPS<QLTEN_Complex, QNT>): SetComplex on the fresh batch (before SetFermion / SetTPS); the
  // ABI moves planes, this wrapper std::complex<double>
  using cplx = std::complex<double>;
  void SetComplex() { ck(peps_set_complex(h_)); complex_ = true; }
  bool is_complex() const { return complex_; }
  void SetTPS(const std::vector<cplx> &flat) {
    std::vector<double> re(flat.size()), im(flat.size());
    for (size_t i = 0; i < flat.size(); ++i) { re[i] = flat[i].real(); im[i] = flat[i].imag(); }
    ck(peps_set_tps_c(h_, re.data(), im.data(), re.size()));
  }
  // what: 0 amplitudes, 1 local energies, 2 holes, 3 sum O*, 4 sum conj(E_loc) O*, 5 the state (peps_get_planar)
  std::vector<cplx> Planar(int what, size_t n) {
    std::vector<double> re(n), im(n);
    ck(peps_get_planar(h_, what, re.data(), im.data()));
    std::vector<cplx> out(n);
    for (size_t i = 0; i < n; ++i) out[i] = cplx(re[i], im[i]);
    return out;
  }
  std::vector<cplx> AmplitudesComplex() { return Planar(0, (size_t)walkers_); }
  std::vector<cplx> LocalEnergiesComplex() { return Planar(1, (size_t)walkers_); }
  void Accumulators(std::vector<cplx> &osum, std::vector<cplx> &eosum) { osum = Planar(3, tps_size()); eosum = Planar(4, tps_size()); }
  std::vector<double> GetTPS() { std::vector<double> v(tps_size()); ck(peps_get_tps(h_, v.data(), v.size())); return v; }
  void SetModel(const XXZModel &m) { ck(peps_set_model_xxz(h_, m.jz, m.jxy, m.pinning00)); }
  void SetModel(const J1J2XXZModel &m) { ck(peps_set_model_j1j2_xxz(h_, m.jz, m.jxy, m.jz2, m.jxy2, m.pinning00)); }
  void SetModel(const TransverseFieldIsingModel &m) { ck(peps_set_model_tfim(h_, m.h)); }
  // table-driven model (seam B2 as data): one call per term; ClearModelTerms returns to the built-in solvers
  void SetModelTerm(const ModelTerm &m) { ck(peps_set_model_term(h_, m.kind, m.T, m.diag.data(), m.target.data(), m.coef.data())); }
  void ClearModelTerms() { ck(peps_clear_model_terms(h_)); }
  // SquaretJModelMixIn::SetSingletPairPinningField as data (peps_set_bond_pin): `m` (a kind-0 ModelTerm, e.g.
  // tJSingletPairPinningTerm(delta)) acts on the one NN bond (site1, site2), row-major site indices, site1 the left / upper site
  void SetBondPin(int site1, int site2, const ModelTerm &m) { ck(peps_set_bond_pin(h_, site1, site2, m.T, m.diag.data(), m.target.data(), m.coef.data())); }
  void ClearBondPin() { ck(peps_set_bond_pin(h_, 0, 1, 0, nullptr, nullptr, nullptr)); }
  // EvaluateBondSC-style observable as data (peps_measure_bond_term): values on the horizontal [W][rows][cols-1] and the
  // vertical [W][rows-1][cols] bonds (real contexts)
  std::pair<std::vector<double>, std::vector<double>> MeasureBondTerm(const ModelTerm &m) {
    std::vector<double> h((size_t)walkers_ * rows_ * (cols_ - 1)), v((size_t)walkers_ * (rows_ - 1) * cols_);
    ck(peps_measure_bond_term(h_, m.T, m.diag.data(), m.target.data(), m.coef.data(), h.data(), v.data()));
    return {h, v};
  }
  // fZ2-graded tensors (peps_set_fermion): once, before SetTPS and SetModelTerm
  // JastrowDress: v[nsites * nsites] symmetric, density[phys] (peps_set_jastrow)
  void SetJastrow(const std::vector<double> &v, const std::vector<int32_t> &density) { ck(peps_set_jastrow(h_, v.data(), density.data())); }
  void SetFermion(const FermionParities &p) { ck(peps_set_fermion(h_, p.phys_par.data(), p.leg_par.data(), p.leg_par.size())); }
  std::vector<double> EnergyAndHoles(bool calc_holes) {
    std::vector<double> e((size_t)walkers_);
    ck(peps_energy_and_holes(h_, calc_holes ? 1 : 0, e.data(), nullptr));
    return e;
  }
  // MonteCarloEngine::EnsureConfigurationValidity (monte_carlo_engine.h:340-414) with walkers as ranks: invalid walkers
  // take the first valid walker's configuration; returns the rescued walkers, throws when disabled / nobody is valid.
  std::vector<int> EnsureConfigurationValidity(const ConfigurationRescueParams &rp = ConfigurationRescueParams()) {
    std::vector<double> amp = Amplitudes();
    std::vector<int> bad;
    int src = -1;
    for (int w = 0; w < walkers_; ++w) {
      if (CheckWaveFunctionAmplitudeValidity(amp[(size_t)w], rp.amplitude_min_threshold, rp.amplitude_max_threshold)) { if (src < 0) src = w; }
      else bad.push_back(w);
    }
    if (bad.empty()) return bad;
    if (!rp.enabled) throw std::runtime_error("invalid configurations and configuration rescue is disabled");
    if (src < 0) throw std::runtime_error("all walkers have invalid configurations: check bond dimension, truncation cutoff, initial configuration");
    std::vector<int32_t> cfg = GetConfigs();
    const size_t ns = (size_t)rows_ * cols_;
    for (int w : bad) std::copy(cfg.begin() + (size_t)src * ns, cfg.begin() + (size_t)(src + 1) * ns, cfg.begin() + (size_t)w * ns);
    SetConfigs(cfg);
    InitWalkers();
    for (double a : Amplitudes())
      if (!CheckWaveFunctionAmplitudeValidity(a, rp.amplitude_min_threshold, rp.amplitude_max_threshold))
        throw std::runtime_error("rescue FAILED: the valid configuration of another walker is not valid here");
    return bad;
  }
  void SetUpdater(Updater u) { updater_ = u; ck(peps_set_updater(h_, (int32_t)u)); }
  void SetChainDeflation(double eps) { ck(peps_set_chain_deflation(h_, eps)); }
  // EvaluateObservables (base/square_nnn_model_measurement_solver.h:33-214): per-walker arrays, see peps_measure
  struct Observables { std::vector<double> energy, bond_energy_h, bond_energy_v, bond_energy_dr, bond_energy_ur, row_corr; };
  Observables Measure() {
    Observables o;
    const size_t W = (size_t)walkers_, r = (size_t)rows_, c = (size_t)cols_;
    o.energy.resize(W); o.bond_energy_h.resize(W * r * (c - 1)); o.bond_energy_v.resize(W * (r - 1) * c);
    o.bond_energy_dr.resize(W * (r - 1) * (c - 1)); o.bond_energy_ur.resize(W * (r - 1) * (c - 1)); o.row_corr.resize(W * (c / 2));
    ck(peps_measure(h_, o.energy.data(), o.bond_energy_h.data(), o.bond_energy_v.data(), o.bond_energy_dr.data(),
                    o.bond_energy_ur.data(), o.row_corr.data()));
    return o;
  }
  void SetConfigs(const std::vector<int32_t> &cfg) { ck(peps_set_configs(h_, cfg.data())); }
  std::vector<int32_t> GetConfigs() { std::vector<int32_t> v((size_t)walkers_ * rows_ * cols_); ck(peps_get_configs(h_, v.data())); return v; }
  void SeedRNG(const std::vector<uint32_t> &seeds) { ck(peps_seed_rng(h_, seeds.data())); }
  void InitWalkers() { ck(peps_init_walkers(h_)); }
  std::vector<double> Amplitudes() { std::vector<double> v((size_t)walkers_); ck(peps_get_amplitudes(h_, v.data())); return v; }
  double NormalizeStateOrder1(double max_abs_override = 0.0) { double f = 0; ck(peps_normalize_state_order1(h_, max_abs_override, &f)); return f; }
  std::vector<double> StepSweep(int n) {
    std::vector<double> a((size_t)walkers_);
    ck(updater_ == Updater::NNFullSpace ? peps_sweep_full_space(h_, n, a.data())
       : updater_ == Updater::TNN3SiteExchange ? peps_sweep_three_site(h_, n, a.data()) : peps_sweep(h_, n, a.data()));
    return a;
  }
  void ZeroAccumulators() { ck(peps_zero_accumulators(h_)); }
  void Sample(int sweeps_between_samples, std::vector<double> &eloc, std::vector<double> &accept) {
    eloc.resize((size_t)walkers_); accept.resize((size_t)walkers_);
    ck(peps_sample(h_, sweeps_between_samples, eloc.data(), accept.data()));
  }
  void Accumulators(std::vector<double> &osum, std::vector<double> &eosum) {
    osum.resize(tps_size()); eosum.resize(tps_size());
    ck(peps_get_accumulators(h_, osum.data(), eosum.data(), osum.size()));
  }
  // ---- stochastic reconfiguration: the O* samples of the walker loop stay in HBM (peps_sr_*; the reference keeps
  // Ostar_samples as vector<SplitIndexTPS> on the host, mc_energy_grad_evaluator.h:273-277)
  void SrReserve(size_t max_walker_samples) { ck(peps_sr_reserve(h_, (int64_t)max_walker_samples)); }
  void SrCollect(bool on) { ck(peps_sr_collect(h_, on ? 1 : 0)); }
  void SrClear() { ck(peps_sr_clear(h_)); }
  size_t SrCount() { return (size_t)peps_sr_count(h_); }
  // local, unnormalised sum_i (O*_i . v - mean_dot_v) O*_i  (SRSMatrix::operator*, stochastic_reconfiguration_smatrix.h:60-65)
  std::vector<double> SrMatvec(const std::vector<double> &v, double mean_dot_v) {
    std::vector<double> out(v.size());
    ck(peps_sr_matvec(h_, v.data(), mean_dot_v, out.data(), v.size()));
    return out;
  }
  // MeasureStructureFactor (structure_factor_measurement_mixin.h:89-228): raw S+S- overlaps [W][pairs], pairs in the
  // reference's order (y1, x1, y2 > y1, x2)
  std::vector<double> MeasureStructureFactor() {
    std::vector<double> out((size_t)walkers_ * (size_t)peps_structure_factor_pairs(h_));
    ck(peps_measure_structure_factor(h_, out.data()));
    return out;
  }
  int rows() const { return rows_; }
  int cols() const { return cols_; }
  peps_ctx *handle() { return h_; }

 private:
  void ck(int rc) { if (rc != 0) throw std::runtime_error(peps_last_error(h_)); }
  peps_ctx *h_ = nullptr;
  int rows_, cols_, walkers_;
  bool complex_ = false;
  Updater updater_ = Updater::NNExchange;
};

struct EvaluateResult {               // MCEnergyGradEvaluator::Result (mc_energy_grad_evaluator.h:66-75)
  double energy = 0, energy_error = 0, gradient_norm = 0;
  std::vector<double> gradient;       // packed like the TPS
  std::vector<double> accept_rates_avg;
  std::vector<double> energy_samples; // [walkers][samples_per_walker]
  std::vector<double> Ostar_mean;     // with collect_sr_buffers: mean O* (packed), and the global sample count
  size_t total_samples = 0;
};

struct ConjugateGradientParams {      // optimizer/optimizer_params.h:50-57
  int max_iter = 100;
  double relative_tolerance = 1e-4, absolute_tolerance = 0.0;
  int residual_recompute_interval = 20;
  double orthogonality_threshold = 0.5;
};

struct EvaluateResultComplex {        // the same for TenElemT = QLTEN_Complex
  std::complex<double> energy = 0;
  double energy_error = 0, gradient_norm = 0;
  std::vector<std::complex<double>> gradient;
  std::vector<double> accept_rates_avg;
  std::vector<std::complex<double>> energy_samples;
};

// MeanAndBinnedErrorSqrtNUniformBin with walkers in the role of ranks (monte_carlo_tools/statistics.h:146-225)
inline std::pair<double, double> BinnedMean(const std::vector<double> &es, size_t walkers, size_t n) {
  if (n == 0) return {0.0, 0.0};
  size_t bin = std::max<size_t>(1, (size_t)std::sqrt((double)n)), nb = n / bin;
  std::vector<double> means;
  for (size_t w = 0; w < walkers; ++w)
    for (size_t i = 0; i < nb; ++i) {
      double s = 0;
      for (size_t k = 0; k < bin; ++k) s += es[w * n + i * bin + k];
      means.push_back(s / (double)bin);
    }
  if (means.empty()) return {0.0, 0.0};
  double mean = 0;
  for (double m : means) mean += m;
  mean /= (double)means.size();
  if (means.size() == 1) return {mean, std::numeric_limits<double>::infinity()};
  double var = 0;
  for (double m : means) var += (m - mean) * (m - mean);
  var /= (double)means.size();
  return {mean, std::sqrt(var / ((double)means.size() - 1.0))};
}

class MCEnergyGradEvaluator {
 public:
  MCEnergyGradEvaluator(const MonteCarloParams &mc, const BMPSTruncateParams &trunc, int rows, int cols, int phys, int D,
                        int walkers, const XXZModel &model, uint32_t seed, int device = 0)
      : mc_(mc), batch_(rows, cols, phys, D, walkers, trunc, device) {
    batch_.SetModel(model);
    std::vector<int32_t> cfg;
    for (int w = 0; w < walkers; ++w) cfg.insert(cfg.end(), mc.initial_config.begin(), mc.initial_config.end());
    batch_.SetConfigs(cfg);
    std::vector<uint32_t> seeds((size_t)walkers);
    for (int w = 0; w < walkers; ++w) seeds[(size_t)w] = seed + (uint32_t)w;
    batch_.SeedRNG(seeds);
  }
  // Models given as data (seam B2) and, with `fermion`, fZ2-graded states: e.g. {SpinlessFermionBondTerm(t, V),
  // SpinlessFermionNNNTerm(t2)} or {tJBondTerm(t, J, V), tJOnsiteTerm(mu)} with the parities of the SplitIndexTPS
  // (SquareSpinlessFermion / SquaretJ*Model runs of the reference, BASELINE config #4)
  MCEnergyGradEvaluator(const MonteCarloParams &mc, const BMPSTruncateParams &trunc, int rows, int cols, int phys, int D,
                        int walkers, const std::vector<ModelTerm> &terms, uint32_t seed, const FermionParities *fermion = nullptr,
                        int device = 0)
      : mc_(mc), batch_(rows, cols, phys, D, walkers, trunc, device) {
    if (fermion) batch_.SetFermion(*fermion);
    for (const auto &t : terms) batch_.SetModelTerm(t);
    std::vector<int32_t> cfg;
    for (int w = 0; w < walkers; ++w) cfg.insert(cfg.end(), mc.initial_config.begin(), mc.initial_config.end());
    batch_.SetConfigs(cfg);
    std::vector<uint32_t> seeds((size_t)walkers);
    for (int w = 0; w < walkers; ++w) seeds[(size_t)w] = seed + (uint32_t)w;
    batch_.SeedRNG(seeds);
  }
  // Evaluate(state): state fan-out, RefreshWavefunctionComponent, the walker loop, energy binning, gradient.
  // collect_sr_buffers (mc_energy_grad_evaluator.h:181-183, 273-277): keep the O* samples in HBM for CalculateNaturalGradient
  EvaluateResult Evaluate(const std::vector<double> &packed_tps, bool collect_sr_buffers = false) {
    batch_.SetTPS(packed_tps);
    batch_.InitWalkers();
    const size_t W = (size_t)batch_.walkers();
    const size_t n = std::max<size_t>(1, (mc_.num_samples + W - 1) / W);
    batch_.ZeroAccumulators();
    if (collect_sr_buffers) {
      if (sr_cap_ < n * W) { batch_.SrReserve(n * W); sr_cap_ = n * W; }
      batch_.SrClear();
    }
    batch_.SrCollect(collect_sr_buffers);
    EvaluateResult r;
    r.energy_samples.assign(W * n, 0.0);
    double acc = 0;
    std::vector<double> e, a;
    for (size_t s = 0; s < n; ++s) {
      batch_.Sample((int)mc_.sweeps_between_samples, e, a);
      for (size_t w = 0; w < W; ++w) { r.energy_samples[w * n + s] = e[w]; acc += a[w]; }
    }
    std::vector<double> osum, eosum;
    batch_.Accumulators(osum, eosum);
    auto me = BinnedMean(r.energy_samples, W, n);
    r.energy = me.first; r.energy_error = me.second;
    r.gradient.resize(osum.size());
    for (size_t i = 0; i < osum.size(); ++i) {
      r.gradient[i] = (eosum[i] - r.energy * osum[i]) / (double)(n * W);
      r.gradient_norm += r.gradient[i] * r.gradient[i];
    }
    r.accept_rates_avg = {acc / (double)(n * W)};
    batch_.SrCollect(false);
    if (collect_sr_buffers) {
      r.Ostar_mean.resize(osum.size());
      for (size_t i = 0; i < osum.size(); ++i) r.Ostar_mean[i] = osum[i] / (double)(n * W);
      r.total_samples = n * W;
    }
    return r;
  }
  // Optimizer::CalculateNaturalGradient (optimizer/optimizer_impl.h:1031-1089) on the samples of the last
  // Evaluate(state, true): solves (S + diag_shift) x = gradient with the reference's CG loop on the device
  // (peps_sr_natural_gradient; single GPU here -- pass an all-reduce callback through the C ABI for several).
  // Returns {natural gradient (packed), CG iterations, residual norm}; throws on an indefinite matrix / breakdown.
  std::tuple<std::vector<double>, int, double> CalculateNaturalGradient(const EvaluateResult &r, double diag_shift,
                                                                          const ConjugateGradientParams &cg = ConjugateGradientParams(),
                                                                          const std::vector<double> *init_guess = nullptr) {
    if (r.total_samples == 0) throw std::runtime_error("CalculateNaturalGradient: Evaluate(state, collect_sr_buffers = true) first");
    peps_cg_params p{cg.max_iter, cg.relative_tolerance, cg.absolute_tolerance, cg.residual_recompute_interval, cg.orthogonality_threshold};
    std::vector<double> x(r.gradient.size());
    int32_t it = 0, reason = 0;
    double resid = 0.0;
    if (peps_sr_natural_gradient(batch_.handle(), r.gradient.data(), r.Ostar_mean.data(), (int64_t)r.total_samples, diag_shift, &p,
                                 init_guess ? init_guess->data() : nullptr, nullptr, nullptr, x.data(), &it, &resid, &reason) != 0)
      throw std::runtime_error(peps_last_error(batch_.handle()));
    if (reason == 3 || reason == 4) throw std::runtime_error("CG solver terminated: indefinite matrix / numerical breakdown");
    return std::make_tuple(x, (int)it, resid);
  }
  // MinSR (optimizer/minsr_scalapack.h), the minimum-step form of SR, on the samples of the last Evaluate(state, true):
  // x = (S + diag_shift)^{-1} g_c solved in sample space by a device Cholesky of the N x N matrix T + diag_shift
  // (peps_sr_minsr_natural_gradient). g_c uses the PLAIN mean of the stored local energies, so it equals r.gradient when the
  // samples per walker are a multiple of floor(sqrt(samples per walker)). Single GPU. Returns {natural gradient (packed),
  // energy mean}; throws for diag_shift <= 0 or a non-positive Cholesky pivot.
  std::tuple<std::vector<double>, double> CalculateNaturalGradientMinSR(const EvaluateResult &r, double diag_shift) {
    if (r.total_samples == 0) throw std::runtime_error("CalculateNaturalGradientMinSR: Evaluate(state, collect_sr_buffers = true) first");
    std::vector<double> x(r.gradient.size());
    double em = 0.0;
    if (peps_sr_minsr_natural_gradient(batch_.handle(), (int64_t)r.total_samples, diag_shift, x.data(), &em) != 0)
      throw std::runtime_error(peps_last_error(batch_.handle()));
    return std::make_tuple(x, em);
  }
  // EvaluateEnergyOnly (mc_energy_grad_evaluator.h:331-392): the step-selector trial -- StepSweep + CalEnergy per sample, no
  // holes / O* / gradient. Returns {energy, energy_error, mean acceptance rate}.
  std::tuple<double, double, double> EvaluateEnergyOnly(const std::vector<double> &packed_tps) {
    batch_.SetTPS(packed_tps);
    batch_.InitWalkers();
    const size_t W = (size_t)batch_.walkers();
    const size_t n = std::max<size_t>(1, (mc_.num_samples + W - 1) / W);
    std::vector<double> es(W * n);
    double acc = 0;
    for (size_t s = 0; s < n; ++s) {
      for (double a : batch_.StepSweep((int)mc_.sweeps_between_samples)) acc += a;
      const std::vector<double> e = batch_.EnergyAndHoles(false);
      for (size_t w = 0; w < W; ++w) es[w * n + s] = e[w];
    }
    auto me = BinnedMean(es, W, n);
    return std::make_tuple(me.first, me.second, acc / (double)(n * W));
  }
  // Evaluate for a QLTEN_Complex state (batch().SetComplex() first): E_loc = ... conj(psi_ex / psi), gradient =
  // sum conj(E_loc) O* / N - conj(E) sum O* / N (mc_energy_grad_evaluator.h:245-309); error bar from the real parts
  EvaluateResultComplex Evaluate(const std::vector<std::complex<double>> &packed_tps) {
    if (!batch_.is_complex()) throw std::runtime_error("Evaluate(complex state): call batch().SetComplex() right after construction");
    using cplx = std::complex<double>;
    batch_.SetTPS(packed_tps);
    batch_.InitWalkers();
    const size_t W = (size_t)batch_.walkers();
    const size_t n = std::max<size_t>(1, (mc_.num_samples + W - 1) / W);
    batch_.ZeroAccumulators();
    EvaluateResultComplex r;
    r.energy_samples.assign(W * n, cplx(0));
    std::vector<double> re(W * n), im(W * n), e, a;
    double acc = 0;
    for (size_t s = 0; s < n; ++s) {
      batch_.Sample((int)mc_.sweeps_between_samples, e, a);
      const std::vector<cplx> ec = batch_.LocalEnergiesComplex();
      for (size_t w = 0; w < W; ++w) { r.energy_samples[w * n + s] = ec[w]; re[w * n + s] = ec[w].real(); im[w * n + s] = ec[w].imag(); acc += a[w]; }
    }
    std::vector<cplx> osum, eosum;
    batch_.Accumulators(osum, eosum);
    auto mr = BinnedMean(re, W, n), mi = BinnedMean(im, W, n);
    r.energy = cplx(mr.first, mi.first); r.energy_error = mr.second;
    r.gradient.resize(osum.size());
    for (size_t i = 0; i < osum.size(); ++i) {
      r.gradient[i] = (eosum[i] - std::conj(r.energy) * osum[i]) / (double)(n * W);
      r.gradient_norm += std::norm(r.gradient[i]);
    }
    r.accept_rates_avg = {acc / (double)(n * W)};
    return r;
  }
  WalkerBatch &batch() { return batch_; }

 private:
  MonteCarloParams mc_;
  WalkerBatch batch_;
  size_t sr_cap_ = 0;
};

// MCPEPSMeasurer (algorithm/vmc_update/monte_carlo_peps_measurer_impl.h:172-257) on a prepared WalkerBatch (state, model,
// updater, configurations and seeds set by the caller): warm up, then per sample `sweeps_between_samples` sweeps +
// EvaluateObservables; a walker plays the role of a rank: per-walker sample means, then mean and standard error across the
// walkers (GatherStatisticListOfData, monte_carlo_tools/statistics.h:288-339). Keys: energy, bond_energy_h / _v / _dr / _ur,
// row_corr (the SmSp_row / SpSm_row channel of each walker), and SpSm_cross_raw with enable_structure_factor.
class MCPEPSMeasurer {
 public:
  using Stats = std::map<std::string, std::pair<std::vector<double>, std::vector<double>>>;   // key -> (mean, stderr)
  MCPEPSMeasurer(WalkerBatch &batch, const MonteCarloParams &mc, bool enable_structure_factor = false)
      : b_(batch), mc_(mc), sf_(enable_structure_factor) {}
  Stats Execute() {
    const size_t W = (size_t)b_.walkers();
    if (!mc_.is_warmed_up && mc_.num_warmup_sweeps > 0) b_.StepSweep((int)mc_.num_warmup_sweeps);
    const size_t nper = std::max<size_t>(1, (mc_.num_samples + W - 1) / W);
    std::map<std::string, std::vector<double>> sums;
    auto add = [&](const std::string &k, const std::vector<double> &v) {
      auto &s = sums[k];
      if (s.empty()) s.assign(v.size(), 0.0);
      for (size_t i = 0; i < v.size(); ++i) s[i] += v[i];
    };
    for (size_t s = 0; s < nper; ++s) {
      b_.StepSweep((int)mc_.sweeps_between_samples);
      WalkerBatch::Observables o = b_.Measure();
      add("energy", o.energy); add("bond_energy_h", o.bond_energy_h); add("bond_energy_v", o.bond_energy_v);
      add("bond_energy_dr", o.bond_energy_dr); add("bond_energy_ur", o.bond_energy_ur); add("row_corr", o.row_corr);
      if (sf_) add("SpSm_cross_raw", b_.MeasureStructureFactor());
    }
    Stats out;
    for (auto &kv : sums) {
      const size_t per = kv.second.size() / W;
      std::vector<double> mean(per, 0.0), err(per, std::numeric_limits<double>::infinity());
      for (size_t w = 0; w < W; ++w) for (size_t i = 0; i < per; ++i) mean[i] += kv.second[w * per + i] / (double)nper / (double)W;
      if (W > 1)
        for (size_t i = 0; i < per; ++i) {
          double v = 0.0;
          for (size_t w = 0; w < W; ++w) { const double d = kv.second[w * per + i] / (double)nper - mean[i]; v += d * d; }
          err[i] = std::sqrt(v / ((double)W * ((double)W - 1.0)));
        }
      out[kv.first] = {mean, err};
    }
    samples_per_walker_ = nper;
    return out;
  }
  size_t samples_per_walker() const { return samples_per_walker_; }

 private:
  WalkerBatch &b_;
  MonteCarloParams mc_;
  bool sf_;
  size_t samples_per_walker_ = 0;
};

// Seam B1: adapts the evaluator to `std::function<std::tuple<T, SITPS, double>(const SITPS&)>`
// (VMCPEPSOptimizer::SetEnergyEvaluator). `pack` flattens the caller's SplitIndexTPS, `unpack` builds one back.
template <class SITPS>
std::function<std::tuple<double, SITPS, double>(const SITPS &)> MakeEnergyEvaluator(
    MCEnergyGradEvaluator &ev, std::function<std::vector<double>(const SITPS &)> pack,
    std::function<SITPS(const std::vector<double> &, const SITPS &like)> unpack) {
  return [&ev, pack, unpack](const SITPS &state) {
    EvaluateResult r = ev.Evaluate(pack(state));
    return std::make_tuple(r.energy, unpack(r.gradient, state), r.energy_error);
  };
}

}  // namespace peps_b200
