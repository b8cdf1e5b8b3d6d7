// Walker-batched boundary-MPS engine: every walker (Markov chain) runs the reference's contraction
// sequence in lock step; walkers differ only in which physical slice of the shared SplitIndexTPS each site
// operand gathers, in the Metropolis decisions and in the RNG stream. Host code drives the (walker-uniform)
// control flow and launches one batched device op per reference tensor operation.
//
// Reference call graph mirrored here (include/qlpeps/...):
//   BMPS::MultiplyMPOSVDCompress_            one_dim_tn/boundary_mps/bmps_impl.h:756-862      -> absorb()
//   BMPSContractor grow/shift/delete          two_dim_tn/tensor_network_2d/bmps/impl/bmps_contractor_grow.h
//   BMPSContractor traces / PunchHole         .../impl/bmps_contractor_trace.h:11-205, grow.h:150-183
//   TPSWaveFunctionComponent::EvaluateAmplitude  vmc_basic/wave_function_component.h:187-212
//   MCUpdateSquareNNExchangeOBC sweep         vmc_basic/configuration_update_strategies/square_nn_updater.h:29-188
//   SquareNNNModelEnergySolver (NN) + XXZ     algorithm/vmc_update/model_solvers/base/square_nnn_energy_solver.h:79-315
//   MCEnergyGradEvaluator accumulation        algorithm/vmc_update/mc_energy_grad_evaluator.h:205-282
#pragma once
#include <array>
#include <memory>
#include <string>
#include <vector>
#include "linalg.h"
#include "tensor.h"
#include <map>
#include <stdexcept>

namespace peps {

enum Pos { LEFT = 0, DOWN = 1, RIGHT = 2, UP = 3 };
enum Orient { HORIZONTAL = 0, VERTICAL = 1 };
inline int opposite(int p) { return (p + 2) % 4; }

struct TRef {           // operand view with dims
  Operand op;
  Operand opi;          // imaginary plane (complex mode)
  int rank = 0;
  int d[6] = {1, 1, 1, 1, 1, 1};
};

struct EngineConfig {
  int rows = 0, cols = 0, phys = 2, D = 0, walkers = 0, device = 0;
  int dmin = 1, dmax = 1;
  double trunc_err = 0.0;
};

class Engine {
 public:
  explicit Engine(const EngineConfig &c);
  ~Engine();

  // ---- state upload / download
  size_t tps_size() const { return (size_t)tps_total_; }
  long site_offset(int r, int c) const { return tps_off_h_[(size_t)(r * cols_ + c)]; }
  void site_dims(int r, int c, int out[4]) const;
  void set_tps(const double *host);
  void get_tps(double *host);
  void scale_tps(double f);
  void set_configs(const int32_t *host);
  void get_configs(int32_t *host);
  void seed_rng(const uint32_t *seeds);
  void set_rng_state(const uint32_t *mt, const int32_t *idx);
  void get_rng_state(uint32_t *mt, int32_t *idx);
  void get_amplitudes(double *host);
  void set_truncation(int dmin, int dmax, double terr) { dmin_ = dmin; dmax_ = dmax; terr_ = terr; touch_all(); }
  // BMPSTruncateParams::Variational2Site / Variational1Site (one_dim_tn/boundary_mps/bmps.h:81-97): scheme 0 = SVD
  // compression, 1 = two-site, 2 = one-site variational; the batch iterates until EVERY walker meets convergence_tol
  void set_compress_scheme(int scheme, double tol, int max_iter) {
    if (scheme < 0 || scheme > 2 || max_iter < 1) throw std::invalid_argument("set_compress_scheme: scheme in {0,1,2}, max_iter >= 1");
    scheme_ = scheme; var_tol_ = tol; var_iter_ = max_iter; touch_all();
  }
  void set_jacobi(double tol, int inner, int max_sweeps) {
    la_.jacobi_tol = tol; la_.jacobi_inner_sweeps = inner; la_.jacobi_max_sweeps = max_sweeps; touch_all();
  }

  // ---- the hot path
  void init_walkers();                                // contractor.Init + EvaluateAmplitude for all walkers
  void evaluate_amplitude();
  void sweep(int nsweeps, double *accept_rate_host);  // accept_rate_host[W] (last sweep), may be null
  // MCUpdateSquareNNFullSpaceUpdateOBC (square_nn_updater.h:253-293): all phys^2 local states of a bond by batched
  // ReplaceNNSiteTrace on the device, Suwa-Todo choice (long double prefix sums + one long double draw per bond,
  // suwa_todo_update.h:53-113) on the host from the per-walker mt19937 streams
  void sweep_full_space(int nsweeps, double *accept_rate_host);
  // MCUpdateSquareTNN3SiteExchange (square_3site_updater.h:23-160): permutations of the spins of three consecutive
  // sites by batched ReplaceTNNSiteTrace (one trace per permutation slot, per-walker physical indices), Suwa-Todo
  // choice on the host; the cached amplitude is refreshed by a three-site trace at every row / column start
  void sweep_three_site(int nsweeps, double *accept_rate_host);
  // MonteCarloEngine::StepSweep with the configured updater (0 = NN exchange, 1 = NN full space, 2 = 3-site exchange)
  void set_updater(int kind) { if (kind < 0 || kind > 2) throw std::invalid_argument("unknown updater"); updater_ = kind; }
  void step_sweep(int nsweeps, double *accept_rate_host) {
    if (updater_ == 1) sweep_full_space(nsweeps, accept_rate_host);
    else if (updater_ == 2) sweep_three_site(nsweeps, accept_rate_host);
    else sweep(nsweeps, accept_rate_host);
  }
  void energy_and_holes(bool calc_holes, double *eloc_host, double *psi_list_host);
  // SquareNNNModelMeasurementSolver::EvaluateObservables (base/square_nnn_model_measurement_solver.h:33-214) for the
  // XXZ / J1-J2 models: the bond traversal without holes, every bond energy kept. Host outputs (any may be null):
  // energy[W], e_h[W][rows][cols-1], e_v[W][rows-1][cols], e_dr / e_ur[W][rows-1][cols-1] (zeros without NNN terms).
  // row_corr[W][cols/2]: MeasureSpinOneHalfOffDiagOrderInRow (square_spin_onehalf_xxz_obc.h:22-60) on row rows/2 from
  // site (rows/2, cols/4): conj(psi(both spins flipped) / psi) per distance, 0 where the two spins are equal.
  void measure(double *energy, double *e_h, double *e_v, double *e_dr, double *e_ur, double *row_corr);
  // StructureFactorMeasurementMixin::MeasureStructureFactor (model_solvers/base/structure_factor_measurement_mixin.h:
  // 89-228): S+(y1,x1) S-(y2,x2) overlaps for all pairs with y2 > y1 by excited-state propagation of the UP boundary.
  // out[W][npairs], pair order (y1, x1, y2, x2) with x2 fastest; RAW overlaps, 0 where S+ / S- annihilate (spin-1/2 only).
  long structure_factor_pairs() const { return (long)cols_ * cols_ * (rows_ * (rows_ - 1) / 2); }
  void measure_structure_factor(double *out_host);
  void zero_accumulators();
  void accumulate_ostar();                            // uses holes/eloc/amplitude of the last energy_and_holes
  void get_accumulators(double *osum_host, double *eosum_host);
  double *osum_device() { return osum_; }
  double *eosum_device() { return eosum_; }
  // SR: O* sample store (optimizer/stochastic_reconfiguration_smatrix.h). reserve() allocates capacity for
  // `max_samples` walker-samples; while collecting, accumulate_ostar() also appends O*_w and its configuration.
  void sr_reserve(long max_samples);
  void sr_clear() { sr_count_ = 0; }
  void sr_collect(bool on) { sr_on_ = on; }
  long sr_count() const { return sr_count_; }
  // out = sum_i (O*_i . v - mean_dot_v) O*_i over the stored samples (device pointers, TPS-shaped vectors)
  void sr_matvec_device(const double *v_dev, double mean_dot_v, double *out_dev);
  void sr_matvec_host(const double *v, double mean_dot_v, double *out);
  void sr_matvec_host_c(const double *v, double mean_re, double mean_im, double *out);   // complex context, planar vectors
  // Optimizer::CalculateNaturalGradient (optimizer/optimizer_impl.h:1031-1089) with every CG vector resident in HBM:
  // solves (S + diag_shift) x = gradient by the reference's conjugate-gradient loop (utility/conjugate_gradient_solver.h:
  // 181-276: best-iterate tracking, stagnation / NaN / indefiniteness exits, orthogonality restart, periodic residual
  // recomputation). S v = (1/total_samples) allreduce(sum_i (O*_i . v - mean . v) O*_i) + diag_shift v; `allreduce`
  // (may be null on a single GPU) sums a DEVICE buffer in place over all GPUs (NCCL on the device pointer).
  struct CGParams { int max_iter = 100; double rel_tol = 1e-4, abs_tol = 0.0; int recompute = 20; double ortho = 0.5; };
  struct CGOutcome { int iterations = 0; double residual_norm = 0.0; int reason = 0; long matvecs = 0; };
  typedef int (*AllReduceFn)(void *user, double *device_buf, size_t n);
  CGOutcome sr_natural_gradient(const double *gradient_host, const double *ostar_mean_host, long total_samples,
                                double diag_shift, const CGParams &prm, const double *init_guess_host, AllReduceFn allreduce,
                                void *user, double *x_host);
  // MinSR, the minimum-step form of SR (optimizer/minsr_scalapack.h), on the same store: the solve runs in sample space.
  // With X_i = (O*_i - Obar) / sqrt(N), e_i = conj(E_i - Ebar) / sqrt(N) and T = X X^H (N x N),
  //   x = X^H (T + diag_shift)^{-1} e = (S + diag_shift)^{-1} g_c,   g_c = (1/N) sum_i conj(E_i - Ebar) (O*_i - Obar).
  // Obar and Ebar (the PLAIN mean of the stored local energies) come from the store itself, so g_c equals the evaluator's
  // gradient exactly when its binned energy mean equals the plain mean (samples per walker a multiple of floor(sqrt(n))).
  // Single GPU: total_samples must equal the stored count; diag_shift > 0. x_host: TPS-shaped (planar in a complex
  // context); energy_mean_host: Ebar (1 or 2 doubles).
  void sr_minsr_natural_gradient(long total_samples, double diag_shift, double *x_host, double *energy_mean_host);
  // The centred T of the stored samples (complex: Re T then Im T, N x N each, row-major); gdiag_host (may be null):
  // the uncentred Gram diagonal G_ii = |O*_i|^2.
  void sr_minsr_tmatrix(double *t_host, double *gdiag_host);
  void set_model_xxz(double jz, double jxy, double h00) {
    if (phys_ != 2) throw std::invalid_argument("spin-1/2 XXZ / J1-J2 models need phys = 2");
    jz_ = jz; jxy_ = jxy; h00_ = h00;
  }
  void set_deflation(double eps) { la_.deflation_eps = eps; touch_all(); }
  // rows of the forward R chain below eps * (largest row norm) are dropped (0 = keep the full D*chi rows)
  void set_chain_deflation(double eps) { chain_eps_ = eps; touch_all(); }
  // SquareSpinOneHalfJ1J2XXZModelOBC couplings (model_solvers/square_spin_onehalf_j1j2_xxz_obc.h:34-113); 0 disables NNN
  void set_model_nnn(double jz2, double jxy2) { jz2_ = jz2; jxy2_ = jxy2; }
  // TransverseFieldIsingSquareOBC(h) (model_solvers/transverse_field_ising_square_obc.h:28-247); phys must be 2
  void set_model_tfim(double h) {
    if (phys_ != 2) throw std::invalid_argument("the transverse-field Ising model needs phys = 2");
    tfim_ = true; tfim_h_ = h;
  }
  void set_model_kind_xxz() { tfim_ = false; }
  // Seam B2 as data: a model given by the matrix elements of its local terms instead of an engine branch (the data a
  // user's EvaluateBondEnergy / EvaluateNNNEnergy / EvaluateTotalOnsiteEnergy mix-in encodes, square_nnn_energy_solver.h:
  // 171-198). kind: 0 = NN bonds (both orientations), 1 = NNN (both diagonals), 2 = on-site. Local state p = c1 (* phys +
  // c2) with site1 the left / upper site (diagonals: the left site of the link). diag[p] = <p|H|p>; slot t < T:
  // target[p*T+t] = p' (or -1), coef[p*T+t] = <p|H|p'>. Setting any term switches the table-driven solver on.
  void set_model_term(int kind, int T, const double *diag, const int32_t *target, const double *coef);
  void clear_model_terms();
  // A two-site operator given by its table, measured on every NN bond of the current configurations: out_h[W][rows][cols-1],
  // out_v[W][rows-1][cols] = sum_p' <p|O|p'> conj(psi(p') / psi) -- the data form of a model's EvaluateBondSC hook
  // (base/square_nnn_model_measurement_solver.h:116-131; t-J: delta_dag / delta of square_tJ_model.h:546-602 as two
  // tables). Runs the measurement traversal with the operator in place of the model (Jastrow dressing off).
  void measure_bond_term(int T, const double *diag, const int32_t *target, const double *coef, double *out_h, double *out_v);
  // The one-site analogue: out[W][rows][cols] = sum_p' <p|O|p'> conj(psi(p') / psi) for a one-site operator given by its table
  // (layout of kind 2 of set_model_term), e.g. sigma_x of the transverse-field Ising measurement solver
  // (transverse_field_ising_square_obc.h:95-100: sigma_x(site) = -ex_term / h). Bosonic contexts.
  void measure_site_term(int T, const double *diag, const int32_t *target, const double *coef, double *out);
  // An extra table term on ONE NN bond (s1 = left / upper site, s2 = s1 + 1 or s1 + cols), added to the energy: the
  // singlet-pair pinning field of the t-J models (square_tJ_model.h:86-137, 256-289) as data. T = 0 clears it.
  void set_bond_pin(int s1, int s2, int T, const double *diag, const int32_t *target, const double *coef);
  // Fermion mode (fZ2-graded tensors, BASELINE config #4): the graded network is evaluated as a bosonic network of
  // sign-dressed site tensors, B = T * (-1)^q with q_H = l d + l r + d r + l + d + u J_H for the row machinery (UP / DOWN
  // boundary MPS, LEFT / RIGHT BTen, BTen2) and q_V = l d + l r + l u + l + d + l J_V for the column machinery; J_H / J_V =
  // parity of the sites left of / above the site (a Jordan-Wigner bit per walker and site, part of the gather index). The
  // boundary MPS differ from the reference's graded ones (bmps_impl.h:21-96, 756-862 fermionic branches) by diagonal sign
  // gauges only. phys_par[phys] = fermion parity of each physical state; leg_par = for every site (row-major) the parities
  // of the index values of its L, D, R, U legs, concatenated (site_dims entries each). Call before set_tps; models are
  // given by set_model_term tables (kinds 0 / 1 / 2) whose off-diagonal targets either move one fermion between the two
  // sites or keep both site parities. Derivation and checks: oracle/fermion.py, tests/test_fermion_oracle.py.
  void set_fermion(const int32_t *phys_par, const int32_t *leg_par);
  // Complex (QLTEN_Complex) states: tensors become two real planes (re, im), a contraction four real launches of the
  // contraction kernel, the factorisations run on the real embedding [[Ar, -Ai], [Ai, Ar]] (backend.h "complex tensors as
  // split planes"). Call right after construction. Built for the headline path: amplitude, NN-exchange sweep, XXZ /
  // J1-J2 local energy, holes / O* and the two accumulators; per-walker scalars and the accumulators are planar
  // ([2][..], imaginary plane second). The other updaters / solvers, SR and the fermion mode stay real-only.
  void set_complex();
  bool is_complex() const { return complex_; }
  void set_tps_c(const double *re, const double *im);
  void dress_plane(const double *host, double *dst);
  void get_planar(int what, double *re, double *im);   // 0 amplitudes, 1 eloc, 2 holes, 3 osum, 4 eosum
  // Jastrow-dressed wave function psi(S) = psi_PEPS(S) exp(sum_{i<j} v_ij n_i n_j) (TPSWaveFunctionComponent<..., JastrowDress>,
  // vmc_basic/wave_function_component.h:107-135, vmc_basic/jastrow_factor.h): v = [nsites][nsites] symmetric (diagonal ignored),
  // density[phys] = particle number of a physical state. The NN exchange sweep takes the Jastrow ratio into the acceptance
  // (MCUpdateSquareNNExchangeJastrowDressedTJ, square_nn_updater.h:380-438; the cached amplitude stays the PEPS part) and the
  // table-driven / fermionic energy solvers multiply every exchange matrix element by it (square_tJ_model.h:352-410, 480-520).
  void set_jastrow(const double *v, const int32_t *density);
  void clear_jastrow() { jastrow_on_ = false; }
  bool fermion() const { return fermion_; }

  // ---- probes used by the parity tests (per-walker values of reference contractor calls)
  int bmps_stack_size(int pos) const { return (int)bmps_[pos].size(); }
  long bmps_tensor(int pos, int k, int i, double *out_host, int dims[3]);  // copy one BMPS tensor of all walkers
  void probe_trace_row(int row, double *psi_host);                         // grows what is needed, Trace(tn,{row,0},HORIZONTAL)
  void get_holes(double *host);
  long holes_stride() const { return hole_stride_; }
  int walkers() const { return W_; }
  int rows() const { return rows_; }
  int cols() const { return cols_; }
  long stat(int which) const;
  const char *backend() const { return be_name(); }
  // makes this engine's backend context (device + stream) current for the calling host thread
  void bind() const { be_ctx_bind(bectx_); }

  // ---- contractor API (walker-batched restatement of BMPSContractor)
  void contractor_init();
  void grow_bmps_step(int pos);
  void grow_full_bmps(int pos);
  void delete_inner_bmps(int pos);
  void generate_bmps_approach(int post) { delete_inner_bmps(post); grow_full_bmps(opposite(post)); }
  void grow_bmps_for_row(int row);
  void grow_bmps_for_col(int col);
  void shift_bmps_window(int pos);
  void init_bten(int pos);
  void grow_full_bten(int pos, int slice, int remain, bool init);
  void grow_bten_step(int post);
  void shift_bten_window(int pos);
  // psi_out[w] = ReplaceNNSiteTrace(site_a, site_b, tensors sitps(site_a)[cfg(cfg_a)], sitps(site_b)[cfg(cfg_b)])
  void nn_trace(int ra, int ca, int rb, int cb, int orient, int cfg_site_a, int cfg_site_b, double *psi_out);
  void punch_hole(int r, int c, int orient);          // into the holes buffer
  // psi_out[w] = ReplaceOneSiteTrace({r,c}, sitps({r,c})[idx[w*stride]], HORIZONTAL) (trace.h:30-88)
  void one_site_trace(int r, int c, const int32_t *idx, int stride, double *psi_out);
  // psi_out[w] = ReplaceTNNSiteTrace({r,c}, orient, slices idx0/1/2[w*stride] of the three consecutive sites) (trace.h:326-420)
  void tnn_trace_idx(int r, int c, int orient, const int32_t *idx0, const int32_t *idx1, const int32_t *idx2, int stride,
                     double *psi_out);
  // test probe: grows the environments of the row (HORIZONTAL) / column (VERTICAL) of `site` and evaluates the three-site
  // trace starting there with the physical indices cfg3[w][0..2] (host array)
  void probe_tnn_trace(int r, int c, int orient, const int32_t *cfg3_host, double *psi_host);
  // ReplaceNNSiteTrace with explicit physical indices (device arrays) instead of entries of the configuration
  void nn_trace_idx(int ra, int ca, int rb, int cb, int orient, const int32_t *idx_a, const int32_t *idx_b, int stride,
                    double *psi_out);
  // two-row environments and next-nearest-neighbour traces (init.h:130-186, grow.h:375-527, trace.h:207-281)
  void init_bten2(int pos);
  void grow_full_bten2(int pos, int slice1, int remain, bool init);
  void grow_bten2_step(int post, int slice1);
  void shift_bten2_window(int pos, int slice1);
  // psi_out[w] = ReplaceNNNSiteTrace({row1,col1}, dir, orient, exchanged tensors); dir 0 = LEFTUP_TO_RIGHTDOWN
  void nnn_trace(int row1, int col1, int dir, double *psi_out, int orient = HORIZONTAL);
  // psi_out[w] = ReplaceSqrt5DistTwoSiteTrace({row1,col1}, dir, orient, exchanged tensors) (trace.h:426-536)
  void sqrt5_trace(int row1, int col1, int dir, int orient, double *psi_out);
  // kind 0: NNN plaquette (2 x 2), 1: sqrt(5)-distance plaquette (2 x 3 / 3 x 2); grows the environments first
  void probe_plaquette_trace(int kind, int row1, int col1, int dir, int orient, double *psi_host);
  // test probes of the two factorisation steps of the boundary-MPS compression on host matrices (one plane, or re / im
  // planes in a complex context): chain_step on A[w] (m x n); r_out [W][cap][n] per plane, cap = min(m, n) (complex:
  // min(2m, 2n)), zero rows beyond rows_out; cnt_out[w] = the step's cnt (rows_out when it has none); tri_out = its tri.
  void test_chain_step(int m, int n, const double *a_re, const double *a_im, const int32_t *row_cnt, int row_scale,
                       int rank_hint, double eps, bool reduce_tall, double *r_re, double *r_im, int *rows_out,
                       int32_t *cnt_out, int *tri_out);
  // truncated_right_vectors of Theta[w] (rows x cols), through a writer (held = false) or a held tensor (held = true);
  // b_out [W][min(dmax, rows, cols)][cols] per plane; kept_out[w] = kept_ after the call (cols for the identity shortcut)
  void test_truncated_right_vectors(int rows, int cols, const double *th_re, const double *th_im, int dmin, int dmax,
                                    double terr, bool held, double *b_re, double *b_im, int32_t *kept_out);

 private:
  using BMPSv = std::vector<BT>;
  BT alloc(std::initializer_list<int> dims);
  BT ones111();
  void release(BT &t);
  void release(BMPSv &v);
  TRef ref(const BT &t) const;
  TRef site_ref(int site, int cfg_site) const;
  TRef site_ref_idx(int site, const int32_t *idx, int stride) const;
  void energy_and_holes_tfim(bool calc_holes, double *eloc_host, double *psi_list_host);
  // the energy solver's bond traversal (square_nnn_energy_solver.h:79-315) for the XXZ / J1-J2 model and the table models:
  // per site of the H pass the holes, the on-site term and the horizontal bond; per row the NNN plaquettes and (XXZ model,
  // under measure()) the row correlator; then the vertical bonds, and the XXZ model's site-0 pinning term last
  void energy_pass(bool calc_holes, double *eloc_host, double *psi_list_host);
  // One pass of the bond traversal (bond_traversal_mixin.h:112-143) over the rows (HORIZONTAL) or the columns (VERTICAL).
  // Per line: start(line) once the environments are grown, visit(line, pos) for pos = 0 .. n - reach with the BTen window
  // shifted between consecutive visits, end(line) before the boundary MPS moves to the next line. The boundary-MPS memo
  // hits only while every pass drops and regrows the stacks in this order.
  template <class Start, class Visit, class End>
  void line_pass(int orient, int reach, Start &&start, Visit &&visit, End &&end);
  // One Monte Carlo sweep (square_nn_updater.h:29-81): a HORIZONTAL then a VERTICAL line pass; start(r, c, orient) at the
  // first site of every line, step(r, c, orient) on every window of `reach` sites starting at (r, c)
  template <class Start, class Step>
  void sweep_lines(int reach, Start &&start, Step &&step);
  // the next-nearest-neighbour plaquettes between `row` and `row + 1` (square_nnn_energy_solver.h:203-265): visit(col)
  // for col = 0 .. cols - 2 on the BTen2 window; nothing on the last row
  template <class Visit>
  void nnn_row_pass(int row, Visit &&visit);
  // the psi list of energy_and_holes: one psi per line, kept on the device, one download at the end (no sync per line)
  struct PsiList {
    Engine &e;
    double *host;
    int n = 0;
    PsiList(Engine &e, double *host);
    void record(const double *psi);
    void download();
  };
  // runs body() with the table (kind, T, diag, target, coef) as the only model term (no pin, Jastrow dressing off);
  // the model's tables and flags are restored (and site recording switched off) afterwards, also when body() throws
  template <class Body>
  void with_term_table(int kind, int T, const double *diag, const int32_t *target, const double *coef, Body &&body);
  void refresh_gather();
  void require_boson(const char *what) const {
    if (fermion_) throw std::logic_error(std::string(what) + " is not available in fermion mode");
  }
  bool fermion_ = false, tps_loaded_ = false;
  bool complex_ = false;
  double *imag(const BT &t) const { return t.p + (long)W_ * t.n; }
  // doubles of one per-walker scalar array ([W], or the two planes [2][W] of a complex context)
  size_t sw() const { return (size_t)W_ * (complex_ ? 2 : 1); }
  // eloc-style accumulations on real arrays or planes: dst += coef * conj(psi_ex / psi)  /  the table term of be_term_accumulate
  void ratio_acc(const double *psi_ex, const double *psi, double coef, double *dst) {
    if (complex_) be_ratio_accumulate_c(psi_ex, psi_ex + W_, psi, psi + W_, coef, dst, dst + W_, W_);
    else be_ratio_accumulate(psi_ex, psi, coef, dst, W_);
  }
  void term_acc(int s1, int s2, const double *diag, const double *coefw, const double *psi_ex, const double *psi, double *dst) {
    if (complex_)
      be_term_accumulate_c(cfg_, nsites_, s1, s2, phys_, diag, coefw, psi_ex, psi_ex ? psi_ex + W_ : nullptr, psi, psi + W_, dst, dst + W_, W_);
    else be_term_accumulate(cfg_, nsites_, s1, s2, phys_, diag, coefw, psi_ex, psi, dst, W_);
  }
  void exchange_decide(int s1, int s2, const double *psi_b, const double *jastrow) {
    if (complex_) be_nn_exchange_decide_c(cfg_, nsites_, s1, s2, psi_b, psi_b + W_, amp_, amp_ + W_, mt_, mtidx_, accepted_, W_, jastrow);
    else be_nn_exchange_decide(cfg_, nsites_, s1, s2, psi_b, amp_, mt_, mtidx_, accepted_, W_, jastrow);
  }
  void require_real(const char *what) const {
    if (complex_) throw std::logic_error(std::string(what) + " is not available for complex states");
  }
  // One step of the forward R chain: r (rows x n, either number type) with r^H r = A^H A for the m x n matrix A that
  // write(c, c_im) fills (real context: c = the zero-padded factorisation buffer, c_im null; complex: c / *c_im = the two
  // planes). eps > 0: rank-revealing step, rows below eps * (largest row norm) are dropped. rc / o: per-walker zero-tail
  // hint of the rows of A (null = none); rk: rank of the previous factor (early-stop hint); reduce_tall: matrices taller
  // than qr_max_rows() are reduced by row chunks first. cnt (device, null = all rows): rows >= cnt[w] of r are zero; tri:
  // r is upper trapezoidal. Both hint the next step's contractions (real contexts only).
  struct ChainStep { BT r; int32_t *cnt = nullptr; bool tri = false; };
  template <class Write>
  ChainStep chain_step(int m, int n, Write &&write, const int32_t *rc, int o, int rk, double eps, bool reduce_tall);
  void bond_energy(int s1, int s2, const double *psi_ex, const double *psi, double jz, double jxy, double *target);
  bool jastrow_on_ = false, tables_exchange_only_ = true;
  double *jastrow_v_ = nullptr, *jr_ = nullptr;   // [nsites][nsites], [W]
  int32_t *dens_d_ = nullptr;                      // [phys]
  const double *jastrow_for(int s1, int s2) {      // Jastrow ratio of exchanging s1 and s2 for every walker (null when off)
    if (!jastrow_on_) return nullptr;
    be_jastrow_ratio(cfg_, nsites_, s1, s2, dens_d_, jastrow_v_, jr_, W_);
    return jr_;
  }
  mutable int gmode_ = HORIZONTAL;        // machinery whose dressing tn_site() / site_ref() gather (fermion mode)
  void mode_for_bmps(int pos) const { gmode_ = (pos == UP || pos == DOWN) ? HORIZONTAL : VERTICAL; }
  void mode_for_bten(int pos) const { gmode_ = (pos == LEFT || pos == RIGHT) ? HORIZONTAL : VERTICAL; }
  double *gtps_ = nullptr;                // gathered TPS: == tps_ for bosons; FERMION_VARIANTS * phys dressed slices per site
  long gtps_total_ = 0;                   // doubles of one plane of gtps_ (complex: the im plane follows the re plane)
  std::vector<long> gtps_off_h_;
  int64_t *gtps_off_d_ = nullptr;
  int32_t *gidx_[2] = {nullptr, nullptr}; // [W][nsites] gather index per machinery (fermion mode)
  int32_t *jw_[2] = {nullptr, nullptr};   // [W][nsites] Jordan-Wigner bits
  int32_t *phys_par_d_ = nullptr;
  std::vector<int32_t> phys_par_h_;
  std::vector<std::vector<int32_t>> leg_par_h_;   // [site * 4 + leg]
  double *fsign_ = nullptr;               // [2][hole_stride] sign of d psi / d T per element for J_H = 0 / 1
  double *psi_loc_ = nullptr;             // [W] psi of the current bond / plaquette along the same contraction path
  struct TermTable { bool set = false; int T = 0; double *diag = nullptr; int32_t *target = nullptr; double *coef = nullptr; };
  TermTable term_[3];
  double *site_rec_ = nullptr;            // [nsites][W] (planes in a complex context): per-site records of measure_site_term
  bool rec_sites_ = false;
  TermTable pin_;                         // extra term on the NN bond (pin_s1_, pin_s2_)
  int pin_s1_ = -1, pin_s2_ = -1;
  void upload_table(TermTable &t, int np, int T, const double *diag, const int32_t *target, const double *coef);
  void check_two_site_table(int T, const int32_t *target) const;
  static void free_table(TermTable &t);
  bool tables_on_ = false;
  int32_t *term_ia_ = nullptr, *term_ib_ = nullptr;   // [W] replacement physical indices of the current target slot
  double *term_cw_ = nullptr;                          // [W] matrix element of the current target slot
  void nnn_trace_refs(int row1, int col1, int orient, const TRef &t11, const TRef &t21, const TRef &t12, const TRef &t22,
                      double *psi_out);
  // structural-zero hints for contractions with an upper-trapezoidal R factor of the forward chain (backend.h GettDesc)
  struct KHints {
    const int32_t *klo_m = nullptr, *klo_n = nullptr; double work = 1.0;
    const int32_t *m_cnt = nullptr, *n_cnt = nullptr; int m_scale = 0, n_scale = 0;   // per-walker zero tails (backend.h GettDesc)
  };
  // which: 0 = "apb,kea->kepb" (hint on N = (k,e)), 1 = "kepb,<site>->kofb" (hint on M = (k,b)), 2 = "kea,eaoj->koj" (M = k)
  const KHints &r_hints(int which, int k, int e, int a, int p, int b);
  BT einsum(const std::string &spec, const TRef &a, const TRef &b, const KHints *h = nullptr, bool conj_b = false);
  void einsum_into(const std::string &spec, const TRef &a, const TRef &b, Operand c, const long *sc = nullptr,
                   double alpha = 1.0, double beta = 0.0, const KHints *h = nullptr, const Operand *c_im = nullptr);
  BMPSv absorb(const BMPSv &mps, const std::vector<int> &sites, int post);
  // variational compression (bmps_impl.h:864-1260)
  BMPSv absorb_svd(const BMPSv &mps, const std::vector<int> &sites, int post);
  BMPSv absorb_variational(const BMPSv &mps, const std::vector<int> &sites, int post, bool one_site);
  BMPSv compress_mps(const BMPSv &mps, int dmin, int dmax, double terr);
  // kept right singular vectors of the rows x cols matrix Theta[w]: B (tcap, cols), rows of V^H. theta is either the
  // tensor holding Theta or a writer write(c, c_im) that fills it (real context: c = the zero-padded buffer truncate_rows
  // takes, c_im null; complex: c / *c_im = the two planes); the writer is not called when nothing can be truncated.
  template <class Theta>
  BT truncated_right_vectors(int rows, int cols, Theta &&theta, int dmin, int dmax, double terr);
  // the identity shortcut of truncated_right_vectors: nothing can be truncated and the row space is the whole space
  static bool keeps_every_column(int rows, int cols, int dmin) { return rows >= cols && cols <= dmin; }
  int scheme_ = 0;                 // CompressMPSScheme: 0 SVD_COMPRESS, 1 VARIATION2Site, 2 VARIATION1Site
  double var_tol_ = 1e-12;
  int var_iter_ = 10;
  BT bten_step(const BT &bten, const BT &mps1, const TRef &site, const BT &mps2, int post);
  BT bten2_step(const BT &bten2, const BT &mps1, const TRef &site1, const TRef &site2, const BT &mps2, int post);
  void bten2_operands(int post, int slice1, int bten_size, const BT *&mps1, const BT *&mps2, int &site1, int &site2) const;
  const BT &bten2_at_slice(int pos, int logical) const;
  void reverse_dot(const BT &a, const BT &b, double *out);
  std::vector<int> slice_sites(int num, int orient) const;
  const BMPSv &bmps_at_slice(int pos, int logical) const;
  const BT &bten_at_slice(int pos, int logical) const;
  void bten_operands(int post, int slice, int bten_size, const BT *&mps1, const BT *&mps2, int &site) const;
  static std::string site_labels(int post, char pre, char toward, char next, char away);

  BeCtx *bectx_ = nullptr;
  int rows_, cols_, phys_, D_, W_, nsites_;
  int dmin_, dmax_;
  double terr_;
  double jz_ = 1.0, jxy_ = 1.0, h00_ = 0.0, jz2_ = 0.0, jxy2_ = 0.0;
  int updater_ = 0;
  double *bond_rec_ = nullptr;     // [n_h + n_v + 2 n_d + cols/2][W] per-bond energies (+ row correlator) of the last measure()
  int override_site_ = -1;         // site whose tensor is temporarily replaced (tn.UpdateSiteTensor): slice override_idx_[w * override_stride_]
  const int32_t *override_idx_ = nullptr;
  int override_stride_ = 0;
  TRef tn_site(int site) const {
    return site == override_site_ ? site_ref_idx(site, override_idx_, override_stride_) : site_ref(site, site);
  }
  void ensure_idx_const();
  void upload_flipped_configs();
  void row_corr_hook(int row);
  bool rec_bonds_ = false;
  double *bond_target(int kind, int row, int col);   // where a bond energy is accumulated (eloc_ unless recording)
  bool tfim_ = false;
  double tfim_h_ = 0.0;
  int32_t *idx_const_ = nullptr;   // [phys][W]: idx_const_[s*W + w] = s
  int32_t *idx_flip_ = nullptr;    // [W][nsites]: 1 - config
  int32_t *fs_target_d_ = nullptr;   // fermion mode, full-space updater: [phys^2][phys^2] target table (parity-consistent states)
  double *fs_coef_d_ = nullptr;
  int32_t *idx_perm_ = nullptr;    // [6][W][3]: physical indices of permutation slot s of walker w (3-site updater)
  double *psi_alt_ = nullptr;      // [psi_alt_slots_][W] amplitudes of the alternative local states of an update
  int psi_alt_slots_ = 0;
  void ensure_psi_alt(int slots) {
    if (slots <= psi_alt_slots_) return;
    be_sync();
    be_free(psi_alt_);
    psi_alt_ = (double *)be_malloc(sizeof(double) * (size_t)slots * sw());
    psi_alt_slots_ = slots;
  }
  Pool pool_;
  Planner planner_;
  LinalgCtx la_;

  // TPS: per site, phys slices of (dl,dd,dr,du) row-major; site s slice p at tps_ + tps_off[s] + p*site_size[s]
  double *tps_ = nullptr;
  long tps_total_ = 0;
  std::vector<long> tps_off_h_;
  std::vector<int> site_size_h_;
  std::vector<std::array<int, 4>> site_dims_h_;
  int32_t *tps_off_d_ = nullptr, *site_size_d_ = nullptr, *hole_off_d_ = nullptr;

  int32_t *cfg_ = nullptr;        // [W][nsites]
  double *amp_ = nullptr;         // [W]
  uint32_t *mt_ = nullptr;        // [W][624]
  int32_t *mtidx_ = nullptr;      // [W]
  int32_t *accepted_ = nullptr;   // [W]
  double *eloc_ = nullptr;        // [W]
  double *psi_tmp_ = nullptr;     // [W]
  double *psi_row_ = nullptr;     // [W]
  double *psi_list_d_ = nullptr;  // [(rows + cols)][W] psi list of the last energy_and_holes (downloaded once)
  double *holes_ = nullptr;       // [W][hole_stride]
  long hole_stride_ = 0;
  std::vector<long> hole_off_h_;
  double *osum_ = nullptr, *eosum_ = nullptr;   // [tps_total]
  int32_t *kept_ = nullptr;       // [W] rows kept by the last truncation

  double *sr_ostar_ = nullptr;    // [sr_cap_][hole_stride]
  int32_t *sr_cfgs_ = nullptr;    // [sr_cap_][nsites]
  double *sr_delta_ = nullptr;    // [sr_cap_]
  double *sr_eloc_ = nullptr;     // [sr_cap_] local energy of every stored sample (complex: planes [2][sr_cap_])
  // MinSR: centred T (planes tr / ti, N x N) and Obar (TPS-shaped, planar when complex) of the stored samples
  void minsr_centred_t(double *tr, double *ti, double *obar, double *gdiag_host);
  // complex context: the store holds the real embedding (backend.h be_sr_store_c): [2 sr_cap_] rows of 2 hole_stride doubles,
  // configurations twice, and the doubled site descriptors (re plane sites, then im plane sites) of the planar TPS layout
  int32_t *sr_desc2_ = nullptr;   // [3][2 nsites]: hole_off2, site_size2, tps_off2
  void sr_matvec_device_c(const double *v_dev, double mean_re, double mean_im, double *out_dev);
  long sr_cap_ = 0, sr_count_ = 0;
  bool sr_on_ = false;

  std::map<std::array<int, 6>, KHints> hints_;
  std::map<std::array<int, 7>, std::pair<const int32_t *, const int32_t *>> rdot_tabs_;
  std::vector<BMPSv> bmps_[4];
  // Boundary-MPS memo. The reference drops stack entries (DeleteInnerBMPS, ShiftBMPSWindow) and later regrows them
  // from unchanged configurations: the LEFT stack finished by the sweep's vertical pass is rebuilt column by column
  // by the energy solver's vertical pass, and the DOWN stack consumed by the energy solver's horizontal pass is
  // rebuilt by the next sweep. Absorption is deterministic, so a dropped entry whose rows/columns have not been
  // touched since it was computed IS the tensor the regrowth would produce: it is parked here and handed back.
  struct Memo { BMPSv v; long stamp; };
  std::vector<long> stamp_[4];                // epoch at which bmps_[pos][k] was computed (0 = built on a stale entry)
  std::map<int, Memo> memo_[4];               // deleted entries by stack index
  std::vector<long> row_mod_, col_mod_;       // epoch of the last possible configuration change per row / column
  long epoch_ = 1, n_memo_hits_ = 0;
  bool memo_on_ = true;                       // PEPS_BMPS_MEMO=0 disables (A/B tests)
  bool slices_unchanged_since(int pos, int k, long stamp) const;
  void touch_site(int site);
  void touch_all();
  void purge_memo();
  void park_or_release_top(int pos);
  void push_grown(int pos, int mpo_num, int orient);
  std::vector<BT> bten_[4];
  std::vector<BT> bten2_[4];
  long n_absorb_ = 0, n_bten_ = 0, n_trace_ = 0;
  double chain_eps_ = 1e-13;       // PEPS_CHAIN_EPS (same threshold as the truncation deflation)
  long chain_rows_in_ = 0, chain_rows_kept_ = 0;
};

}  // namespace peps
