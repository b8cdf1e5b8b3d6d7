/*
 * peps_b200 -- C ABI of the B200-native VMC sampling hot path of QuantumLiquids/PEPS.
 *
 * The reference has no FFI; its seams are C++ template contracts (SURVEY.md section 8b). Each entry point
 * below names the reference interface it replaces (paths relative to /root/reference/include/qlpeps/).
 * One context owns W walkers (= the reference's MPI ranks, algorithm/vmc_update/monte_carlo_engine.h:563)
 * on one GPU. All calls are stream-ordered on the context's stream and return 0 on success; on failure
 * they return non-zero and peps_last_error() describes the fault (no exception crosses the ABI).
 *
 * Threading: a context owns its CUDA device ordinal and stream. Every entry point binds them to the calling host
 * thread first (cudaSetDevice + the context's stream), so a context may be created in one thread and used from
 * another, and contexts on different devices may be interleaved in one thread. A context is NOT re-entrant: at most
 * one host thread may be inside a call on a given context at any time. Different contexts may be driven concurrently
 * from different threads (their kernels overlap on the GPU).
 *
 * Data conventions: real FP64; site tensor legs (L, D, R, U) row-major (tensor_network_2d.h:38-46);
 * edge legs have dimension 1; configurations are int32 [W][rows][cols].
 */
#ifndef PEPS_B200_H
#define PEPS_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct peps_ctx peps_ctx;

typedef struct {
  int32_t rows, cols;      /* lattice Ly x Lx */
  int32_t phys;            /* physical dimension d */
  int32_t D;               /* PEPS bond dimension (uniform; edge legs are 1) */
  int32_t walkers;         /* Markov chains batched on this GPU */
  int32_t device;          /* CUDA device ordinal */
  int32_t dmin, dmax;      /* BMPSTruncateParams::D_min / D_max (one_dim_tn/boundary_mps/bmps.h:47-98) */
  double trunc_err;        /* BMPSTruncateParams::trunc_err */
} peps_config;

/* Library / build identification ("cuda-sm_100a"). */
const char *peps_backend_name(void);

/* TPSWaveFunctionComponent + MonteCarloEngine construction (vmc_basic/wave_function_component.h:155-162,
 * algorithm/vmc_update/monte_carlo_engine.h:422-427) for W walkers. */
int peps_create(peps_ctx **out, const peps_config *cfg);
void peps_destroy(peps_ctx *ctx);
const char *peps_last_error(peps_ctx *ctx);

/* Number of doubles of the packed SplitIndexTPS (two_dim_tn/tps/split_index_tps.h:80-607):
 * sites row-major, per site `phys` tensors (L,D,R,U) row-major. */
size_t peps_tps_size(peps_ctx *ctx);
/* Offset (in doubles) of tensor (row, col, phys index 0); phys slices are contiguous after it. */
size_t peps_tps_site_offset(peps_ctx *ctx, int32_t row, int32_t col);
/* MonteCarloEngine::AssignState / the evaluator's state broadcast (mc_energy_grad_evaluator.h:152-161). */
int peps_set_tps(peps_ctx *ctx, const double *host_tps, size_t n);
int peps_get_tps(peps_ctx *ctx, double *host_tps, size_t n);
/* BMPSContractor::SetTruncateParams (two_dim_tn/tensor_network_2d/bmps/bmps_contractor.h:216-230). */
int peps_set_truncation(peps_ctx *ctx, int32_t dmin, int32_t dmax, double trunc_err);
/* BMPSTruncateParams::compress_scheme (one_dim_tn/boundary_mps/bmps.h:31-35, 54-97): 0 = SVD_COMPRESS (default),
 * 1 = VARIATION2Site, 2 = VARIATION1Site (bmps_impl.h:864-1172) with convergence_tol and iter_max; boundaries of two sites
 * always take the SVD path (:416). The batch sweeps until EVERY walker meets convergence_tol (lock step), and the
 * orthonormal factors are the kept singular vectors instead of LAPACK's U / Householder Q: the same boundary MPS up to the
 * gauge of each bond. */
int peps_set_compress_scheme(peps_ctx *ctx, int32_t scheme, double convergence_tol, int32_t iter_max);
/* Convergence control of the Jacobi truncation kernel (no reference counterpart: LAPACK gesdd there). */
int peps_set_jacobi(peps_ctx *ctx, double tol, int32_t inner_sweeps, int32_t max_sweeps);
/* Rows of the QR-preconditioned Theta below eps * (largest row norm) are dropped before / between Jacobi sweeps
 * (default 1e-13; a backward-stable perturbation of relative size <= sqrt(rows) * eps). 0 disables deflation. */
int peps_set_deflation(peps_ctx *ctx, double eps);
/* Rank-revealing step of the forward R chain of a row absorption (no reference counterpart: the reference keeps the
 * full D*chi bond of the exact MPO x MPS product until the SVD sweep): rows of the column-sorted R factor below
 * eps * (largest row norm) are dropped (default 1e-13; the Gram matrix R^T R changes by <= rows * eps^2 relative).
 * 0 keeps every row. */
int peps_set_chain_deflation(peps_ctx *ctx, double eps);
/* SquareSpinOneHalfXXZModelOBC(jz, jxy, pinning00) (model_solvers/square_spin_onehalf_xxz_obc.h:174-328). */
int peps_set_model_xxz(peps_ctx *ctx, double jz, double jxy, double pinning00);
/* SquareSpinOneHalfJ1J2XXZModelOBC(jz, jxy, jz2, jxy2, pinning00) (model_solvers/square_spin_onehalf_j1j2_xxz_obc.h:34-113):
 * next-nearest-neighbour couplings evaluated through BTen2 + ReplaceNNNSiteTrace in the horizontal pass
 * (base/square_nnn_energy_solver.h:203-265). jz2 = jxy2 = 0 switches the NNN pass off. */
int peps_set_model_j1j2_xxz(peps_ctx *ctx, double jz, double jxy, double jz2, double jxy2, double pinning00);
/* TransverseFieldIsingSquareOBC(h): H = -sum_<ij> sz_i sz_j - h sum_i sx_i, one ReplaceOneSiteTrace per site in the
 * horizontal pass (model_solvers/transverse_field_ising_square_obc.h:149-247; BASELINE config #1). phys must be 2. */
int peps_set_model_tfim(peps_ctx *ctx, double h);

/* Seam B2 as data -- a user model without an engine patch. The reference's model mix-ins implement
 * EvaluateBondEnergy(site1, site2, cfg1, cfg2, orient, tn, contractor, ..., inv_psi), EvaluateNNNEnergy(...) and
 * EvaluateTotalOnsiteEnergy(config) (model_solvers/base/square_nnn_energy_solver.h:31-36, 171-198): pure arithmetic on the
 * local configuration, the couplings and amplitude ratios psi(S')/psi(S) of locally modified configurations. Here the same
 * information is uploaded as tables and the engine runs the reference's traversal (:79-315, base/bond_traversal_mixin.h:
 * 112-143) with one batched replacement trace per target slot. kind: 0 = nearest-neighbour bonds (both orientations),
 * 1 = next-nearest-neighbour links (both diagonals), 2 = on-site. Local state p = c1 (* phys + c2), site1 = the left /
 * upper site of the bond (diagonals: the left site of the link). diag[p] = <p|H|p>; for slot t < T: target[p*T + t] = a
 * local state p' != p with <p|H|p'> != 0 (or -1 when the slot is unused), coef[p*T + t] = <p|H|p'>.
 *   E_loc += diag[p] + sum_t coef[p][t] * psi(S with p -> p'_t) / psi(S)
 * Setting any term switches the table-driven solver on (it replaces the built-in XXZ / J1-J2 / TFIM branches, which are
 * reproduced exactly by their tables: include/peps_b200.hpp XXZBondTerm, TFIMTerms); peps_clear_model_terms switches
 * back. Works for any phys (spin-1, t-J-like bosonic parts, ...). */
int peps_set_model_term(peps_ctx *ctx, int32_t kind, int32_t T, const double *diag, const int32_t *target, const double *coef);
int peps_clear_model_terms(peps_ctx *ctx);
/* An extra table term on ONE nearest-neighbour bond, added to the local energy by the table-driven / fermionic solvers: the
 * singlet-pair pinning field of the t-J models, SquaretJModelMixIn::SetSingletPairPinningField + EvaluateSingletPairPinningEnergy_
 * (model_solvers/square_tJ_model.h:86-137, 256-289), as data: delta * (delta_dag + delta) of EvaluateBondSingletPairFortJModel
 * (:546-602) is the table {(E,E) -> (up,dn): +delta/sqrt2, (E,E) -> (dn,up): -delta/sqrt2, (up,dn) -> (E,E): +delta/sqrt2,
 * (dn,up) -> (E,E): -delta/sqrt2}. site1 = row-major index of the left / upper site, site2 = site1 + 1 or site1 + cols; a bond
 * outside the lattice is an error (ValidateSingletPairPinningBondInLattice_, :240-250). Same table layout as kind 0 of
 * peps_set_model_term; T = 0 clears the pin; peps_clear_model_terms clears it too. Call after the model terms. */
int peps_set_bond_pin(peps_ctx *ctx, int32_t site1, int32_t site2, int32_t T, const double *diag, const int32_t *target, const double *coef);

/* Fermionic (fZ2-graded) tensors -- QLTensor<T, fZ2QN> states of the reference (BASELINE config #4: SquareSpinlessFermion,
 * model_solvers/square_spinless_fermion.h:51-213; SquaretJNNModel / SquaretJVModel, model_solvers/square_tJ_model.h:85-420).
 * phys_par[phys]: fermion parity of every physical state (spinless fermion {1, 0}: 0 = occupied, 1 = empty; t-J {1, 1, 0}).
 * leg_par: for every site in row-major order the parity of every index value of its L, D, R, U legs, concatenated
 * (n_leg_par = sum over sites of dL + dD + dR + dU; the `qnval` of the sector an index value belongs to in the .qlten
 * header). The TPS is uploaded by peps_set_tps as dense (L, D, R, U) blocks with the dim-1 parity leg dropped, exactly as
 * for bosons. Call once, before peps_set_tps and peps_set_model_term. The engine then evaluates the graded network of the
 * reference (fermionic branches of bmps_impl.h:21-96, 756-862, bmps_contractor_trace.h:90-205, grow.h:150-183) as an
 * ordinary network of sign-dressed site tensors (DESIGN.md, "Fermions"): same |psi|, same Markov chain, psi_ex / psi per
 * bond along one contraction path (square_nnn_energy_solver.h:143-310), O* = Pi(R*) of utility/helpers.h:57-67 and
 * mc_energy_grad_evaluator.h:259-266 as the Euclidean gradient of log psi* in the uploaded tensor entries. Models are
 * tables (peps_set_model_term); an off-diagonal target must either move one fermion between the two sites of the term or
 * keep both site parities (hopping, spin exchange). Updater: NN exchange (peps_sweep). */
int peps_set_fermion(peps_ctx *ctx, const int32_t *phys_par, const int32_t *leg_par, size_t n_leg_par);

/* Complex states (QLTEN_Complex instantiations of the reference: SplitIndexTPS<QLTEN_Complex, QNT>, every test of
 * tests/CMakeLists.txt:57-83 is compiled for both element types). peps_set_complex switches a fresh context (before the
 * first peps_set_tps*) to complex arithmetic: tensors live as two real planes, a contraction is four launches of the real
 * contraction kernel, the boundary-MPS factorisations run on the real embedding [[Ar, -Ai], [Ai, Ar]] of their matrices
 * (DESIGN.md section 11). Covered: amplitude, the three updaters (|psi| = hypot; Suwa-Todo weights std::norm), every energy
 * solver (XXZ / J1-J2, transverse-field Ising, table models, fermion mode: call peps_set_complex BEFORE peps_set_fermion) with
 * conj(psi_ex / psi) (square_spin_onehalf_xxz_obc.h:72-104), holes and O* = conj(hole / psi), sum O*, sum conj(E_loc) O*
 * (mc_energy_grad_evaluator.h:245-272), measurement (structure factor included), the SR store / matvec / natural gradient,
 * SVD and variational boundary compression. Conventions of a complex context:
 *   - peps_set_tps_c uploads the two planes of the packed state; peps_get_planar reads per-walker / state-shaped results as
 *     planes: what = 0 amplitudes [W], 1 local energies [W] (after peps_energy_and_holes), 2 holes [W][holes_stride] (the
 *     raw environment; O* = conj(hole / amplitude); fermion mode: the finished hole), 3 sum O*, 4 sum conj(E_loc) O*
 *     [tps_size], 5 the state [tps_size]. The real getters return the real planes.
 *   - the psi list of peps_energy_and_holes holds (rows+cols) entries of 2 W doubles (re[W] then im[W]);
 *   - every output array of peps_measure is planar: its real block followed by its imaginary block (twice the real size);
 *   - the accumulator device pointers address 2 * tps_size doubles (re plane, im plane);
 *   - the peps_probe_* calls return 2 W doubles (re[W], im[W]). */
int peps_set_complex(peps_ctx *ctx);
int peps_set_tps_c(peps_ctx *ctx, const double *re, const double *im, size_t n);
int peps_get_planar(peps_ctx *ctx, int32_t what, double *re, double *im);

/* Jastrow-dressed wave function psi(S) = psi_PEPS(S) * exp(sum_{i<j} v_ij n_i n_j): TPSWaveFunctionComponent<..., JastrowDress>
 * (vmc_basic/wave_function_component.h:107-135) with JastrowFactor (vmc_basic/jastrow_factor.h:34-121). v: [nsites][nsites]
 * symmetric, row-major site index, diagonal ignored; density[phys]: particle number of each physical state (t-J: {1, 1, 0}).
 * peps_sweep then is MCUpdateSquareNNExchangeJastrowDressedTJ (square_nn_updater.h:380-438: the Jastrow ratio enters the
 * acceptance, the cached amplitude stays the PEPS part) and the table-driven / fermionic energy solvers multiply every
 * exchange matrix element by the Jastrow ratio (square_tJ_model.h:352-410). Needs a model given by peps_set_model_term whose
 * off-diagonal targets are exchanges of the two local states. */
int peps_set_jastrow(peps_ctx *ctx, const double *v, const int32_t *density);
int peps_clear_jastrow(peps_ctx *ctx);

/* Configuration per walker (vmc_basic/configuration.h:57), int32 [W][rows][cols]. */
int peps_set_configs(peps_ctx *ctx, const int32_t *cfg);
int peps_get_configs(peps_ctx *ctx, int32_t *cfg);
/* MonteCarloSweepUpdaterBase(unsigned seed): std::mt19937(seed[w]) per walker
 * (vmc_basic/configuration_update_strategies/monte_carlo_sweep_updater_base.h:37). */
int peps_seed_rng(peps_ctx *ctx, const uint32_t *seeds);
/* Raw std::mt19937 state, [W][624] words + [W] next index, interchangeable with a host engine. */
int peps_set_rng_state(peps_ctx *ctx, const uint32_t *mt, const int32_t *idx);
int peps_get_rng_state(peps_ctx *ctx, uint32_t *mt, int32_t *idx);

/* contractor.Init(tn) + EvaluateAmplitude() for every walker (wave_function_component.h:155-212). */
int peps_init_walkers(peps_ctx *ctx);
/* TPSWaveFunctionComponent::amplitude per walker. */
int peps_get_amplitudes(peps_ctx *ctx, double *amp);
/* MonteCarloEngine::NormalizeStateOrder1 (monte_carlo_engine.h:206-240) over this context's walkers:
 * returns the per-site factor applied; pass max_abs_override > 0 to use a cross-GPU maximum. */
int peps_normalize_state_order1(peps_ctx *ctx, double max_abs_override, double *site_factor_out);

/* MonteCarloEngine::StepSweep(n) with MCUpdateSquareNNExchangeOBC
 * (configuration_update_strategies/square_nn_updater.h:29-81,146-188); accept_rates[W] of the last sweep. */
int peps_sweep(peps_ctx *ctx, int32_t nsweeps, double *accept_rates);
/* MonteCarloEngine::StepSweep(n) with MCUpdateSquareNNFullSpaceUpdateOBC (square_nn_updater.h:253-293): all phys^2
 * local states of every bond (no Sz conservation), Suwa-Todo choice (monte_carlo_tools/suwa_todo_update.h:53-113) with
 * the reference's long double prefix sums and draw, taken on the host from the same per-walker mt19937 streams. */
int peps_sweep_full_space(peps_ctx *ctx, int32_t nsweeps, double *accept_rates);
/* MonteCarloEngine::StepSweep(n) with MCUpdateSquareTNN3SiteExchange (configuration_update_strategies/
 * square_3site_updater.h:23-160): permutations of the spins on three consecutive sites through ReplaceTNNSiteTrace,
 * Suwa-Todo choice; the cached amplitude is refreshed by a three-site trace at every row / column start. */
int peps_sweep_three_site(peps_ctx *ctx, int32_t nsweeps, double *accept_rates);
/* Selects the updater peps_sample steps with: 0 = MCUpdateSquareNNExchangeOBC (default), 1 = MCUpdateSquareNNFullSpaceUpdateOBC,
 * 2 = MCUpdateSquareTNN3SiteExchange. */
int peps_set_updater(peps_ctx *ctx, int32_t kind);
/* ModelEnergySolver::CalEnergyAndHoles<calchols> (algorithm/vmc_update/model_energy_solver.h:69-100 ->
 * model_solvers/base/square_nnn_energy_solver.h:79-315). eloc[W]; psi_list[(rows+cols)][W] may be NULL. */
int peps_energy_and_holes(peps_ctx *ctx, int32_t calc_holes, double *eloc, double *psi_list);
/* SquareNNNModelMeasurementSolver::EvaluateObservables for the XXZ / J1-J2 models
 * (model_solvers/base/square_nnn_model_measurement_solver.h:33-214; registry keys energy, bond_energy_h,
 * bond_energy_v, bond_energy_dr, bond_energy_ur; spin_z is config - 1/2 and needs no device work): the bond traversal
 * of the energy solver without holes. Host outputs per walker, any may be NULL: energy[W], e_h[W][rows][cols-1],
 * e_v[W][rows-1][cols], e_dr / e_ur[W][rows-1][cols-1], and row_corr[W][cols/2] = the off-diagonal correlator of
 * MeasureSpinOneHalfOffDiagOrderInRow (model_solvers/square_spin_onehalf_xxz_obc.h:22-60) on row rows/2 from site
 * (rows/2, cols/4): conj(psi(both spins flipped) / psi), 0 for equal spins (registry keys SmSp_row / SpSm_row by the
 * spin at the first site, :264-291). */
int peps_measure(peps_ctx *ctx, double *energy, double *e_h, double *e_v, double *e_dr, double *e_ur, double *row_corr);
/* A two-site operator given as a table (layout of kind 0 of peps_set_model_term), evaluated on every nearest-neighbour bond of
 * the current configurations: out_h[W][rows][cols-1], out_v[W][rows-1][cols] = sum_p' <p|O|p'> conj(psi(p') / psi). The data
 * form of a model's EvaluateBondSC hook (base/square_nnn_model_measurement_solver.h:116-131): for the t-J models the pair
 * (delta_dag, delta) of EvaluateBondSingletPairFortJModel (square_tJ_model.h:546-602) is two tables and
 * SC_bond_singlet_h / _v = (conj(delta_dag) + delta) / 2. Works for bosonic contexts and in fermion mode (hops, pair
 * creation / annihilation, parity-preserving targets); complex contexts return planar arrays. The model and its state are
 * untouched. */
int peps_measure_bond_term(peps_ctx *ctx, int32_t T, const double *diag, const int32_t *target, const double *coef, double *out_h, double *out_v);
/* The one-site analogue (table layout of kind 2 of peps_set_model_term): out[W][rows][cols] = sum_p' <p|O|p'> conj(psi(p') / psi),
 * e.g. sigma_x of TransverseFieldIsingSquareOBC::EvaluateObservables (model_solvers/transverse_field_ising_square_obc.h:95-100,
 * sigma_x(site) = -ex_term / h = conj(psi_flip / psi)) with the table {0 -> 1: 1, 1 -> 0: 1}. Bosonic contexts; planar output in a
 * complex context. */
int peps_measure_site_term(peps_ctx *ctx, int32_t T, const double *diag, const int32_t *target, const double *coef, double *out);
/* StructureFactorMeasurementMixin::MeasureStructureFactor (model_solvers/base/structure_factor_measurement_mixin.h:89-228,
 * registry key SpSm_cross): all-pairs S+(y1,x1) S-(y2,x2) overlaps with y2 > y1 by "excited state propagation" -- the UP
 * boundary is forked at row y1 (BMPSContractor::BMPSWalker, bmps/impl/bmps_walker.h), absorbs the row with S+ applied and
 * is propagated through the rows below; every target is closed against the DOWN stack through LEFT / RIGHT environments.
 * out[W][pairs], pairs = cols^2 * rows (rows - 1) / 2 in the order (y1, x1, y2, x2), x2 fastest; RAW overlaps like the
 * reference (divide by the amplitude), 0 where S+ or S- annihilates the walker's configuration. phys must be 2. */
int64_t peps_structure_factor_pairs(peps_ctx *ctx);
int peps_measure_structure_factor(peps_ctx *ctx, double *out);
/* Hole tensors of the last call: [W][stride], per site (L,D,R,U) at the site's hole offset. */
size_t peps_holes_stride(peps_ctx *ctx);
int peps_get_holes(peps_ctx *ctx, double *holes);

/* MCEnergyGradEvaluator accumulation (mc_energy_grad_evaluator.h:245-272): Ostar_sum += O*, ELocConj_Ostar_sum
 * += E_loc O*, O* = hole / amplitude at the sampled physical index. */
int peps_zero_accumulators(peps_ctx *ctx);
int peps_accumulate_ostar(peps_ctx *ctx);
int peps_get_accumulators(peps_ctx *ctx, double *ostar_sum, double *eloc_ostar_sum, size_t n);
/* Device pointers of the two accumulators (for NCCL all-reduce by the caller; mc_energy_grad_evaluator.h:296-310). */
double *peps_ostar_sum_device(peps_ctx *ctx);
double *peps_eloc_ostar_sum_device(peps_ctx *ctx);
/* One VMC sample for all walkers = StepSweep(sweeps_between_samples) + CalEnergyAndHoles<true> + accumulation
 * (the loop body of mc_energy_grad_evaluator.h:205-282). eloc[W], accept_rates[W] may be NULL. */
int peps_sample(peps_ctx *ctx, int32_t sweeps_between_samples, double *eloc, double *accept_rates);

/* ---- stochastic reconfiguration (optimizer/stochastic_reconfiguration_smatrix.h:45-91) ------------------------
 * The reference keeps Ostar_samples as vector<SplitIndexTPS> on the host (mc_energy_grad_evaluator.h:273-277); here
 * they stay in HBM. peps_sr_reserve sizes the store in walker-samples; while peps_sr_collect(1) is set every
 * peps_accumulate_ostar / peps_sample appends the O* of all walkers. peps_sr_matvec returns the LOCAL, unnormalised
 * sum_i (O*_i . v - mean_dot_v) O*_i (TPS-shaped vectors); the caller all-reduces it over GPUs, divides by the total
 * sample count and adds diag_shift * v, exactly the tail of SRSMatrix::operator* (:66,:86-88). */
int peps_sr_reserve(peps_ctx *ctx, int64_t max_walker_samples);
int peps_sr_collect(peps_ctx *ctx, int32_t on);
int peps_sr_clear(peps_ctx *ctx);
int64_t peps_sr_count(peps_ctx *ctx);
int peps_sr_matvec(peps_ctx *ctx, const double *v_host, double mean_dot_v, double *out_host, size_t n);
int peps_sr_matvec_device(peps_ctx *ctx, const double *v_dev, double mean_dot_v, double *out_dev);
/* Complex context (peps_set_complex): TPS-shaped vectors are planar, peps_tps_size() real parts followed by peps_tps_size()
 * imaginary parts; <O*_i, v> is the conjugating inner product of SplitIndexTPS::operator* and mean_dot_v = <Obar, v> is
 * complex. The store keeps the real embedding of the samples, so the same HBM-streaming kernels serve both cases. In a
 * complex context peps_sr_natural_gradient takes / returns planar arrays of 2 * peps_tps_size() doubles. */
int peps_sr_matvec_c(peps_ctx *ctx, const double *v_host, double mean_dot_v_re, double mean_dot_v_im, double *out_host, size_t n);

/* Optimizer::CalculateNaturalGradient (optimizer/optimizer_impl.h:1031-1089) on the device-resident sample store: solves
 * (S + diag_shift) x = gradient with the reference's conjugate-gradient loop (utility/conjugate_gradient_solver.h:181-276
 * and its MPI form :355-611: best-iterate tracking, stagnation / NaN / indefiniteness exits, orthogonality restart,
 * periodic residual recomputation). Every CG vector stays in HBM; per iteration the only host traffic is a handful of
 * scalars. `allreduce` (NULL on a single GPU) must sum `n` doubles at DEVICE pointer `device_buf` in place over all
 * GPUs and return 0 once the result is complete (ncclAllReduce on the pointer + stream synchronisation): it replaces
 * the reference's master/slave broadcast-and-reduce of the matvec (SRSMatrix::operator* :60-88 under MPI). The vector
 * algebra is duplicated on every GPU, so no broadcast of the iterate is needed. gradient / ostar_mean / init_guess
 * (may be NULL = 0) / x_out are host arrays of peps_tps_size() doubles, identical on every rank. reason: 0 converged,
 * 1 max iterations, 2 stagnated, 3 indefinite matrix, 4 numerical breakdown (the reference's TerminationReason). */
typedef int (*peps_allreduce_fn)(void *user, double *device_buf, size_t n);
typedef struct {
  int32_t max_iter;                     /* ConjugateGradientParams (optimizer/optimizer_params.h:50-57) */
  double relative_tolerance, absolute_tolerance;
  int32_t residual_recompute_interval;
  double orthogonality_threshold;
} peps_cg_params;
int peps_sr_natural_gradient(peps_ctx *ctx, const double *gradient, const double *ostar_mean, int64_t total_samples,
                             double diag_shift, const peps_cg_params *params, const double *init_guess,
                             peps_allreduce_fn allreduce, void *user, double *x_out, int32_t *iterations,
                             double *residual_norm, int32_t *reason);

/* MinSR, the minimum-step form of SR (optimizer/minsr_scalapack.h; its equivalence with SR: test_sr_vs_minsr_equivalence.cpp),
 * on the same device-resident store: the linear system is solved in sample space. With X_i = (O*_i - Obar) / sqrt(N),
 * e_i = conj(E_i - Ebar) / sqrt(N) and the N x N matrix T = X X^H,
 *   x = X^H (T + diag_shift)^{-1} e = (S + diag_shift)^{-1} g_c,   g_c = (1/N) sum_i conj(E_i - Ebar) (O*_i - Obar)
 * (push-through identity, exact for diag_shift > 0): one masked Gram on the DMMA pipe, a device Cholesky of T + diag_shift
 * (complex: of the real 2N embedding [[Re T, -Im T], [Im T, Re T]]) and two passes over the store; no tolerance, no
 * iteration count. Obar and Ebar are computed from the store (Ebar = the PLAIN mean of the local energies stored with the
 * samples), so g_c equals the evaluator's gradient exactly when its binned energy mean equals the plain mean, i.e. when
 * the samples per walker are a multiple of floor(sqrt(samples per walker)). Single GPU: total_samples must equal
 * peps_sr_count. x_out: peps_tps_size() doubles (planar 2 * peps_tps_size() in a complex context); energy_mean_out (may be
 * NULL): Ebar, 1 double (2 in a complex context: re, im). Errors: diag_shift <= 0, an empty store, a count mismatch, a
 * non-positive Cholesky pivot. The store is left unchanged. */
int peps_sr_minsr_natural_gradient(peps_ctx *ctx, int64_t total_samples, double diag_shift, double *x_out, double *energy_mean_out);
/* Probes of the MinSR matrices (tests, timing): the centred T (row-major N x N; a complex context returns Re T then Im T,
 * n = 2 N^2), and the uncentred Gram diagonal G_ii = |O*_i|^2 (n = N), whose largest value over the largest T_ii measures
 * the cancellation of forming T from the uncentred Gram. */
int peps_sr_minsr_tmatrix(peps_ctx *ctx, double *t_out, size_t n);
int peps_sr_minsr_gram_diag(peps_ctx *ctx, double *g_out, size_t n);

/* ---- probes for the parity tests ------------------------------------------------------------------ */
/* BMPSContractor::GrowBMPSForRow + InitBTen/GrowFullBTen + Trace(tn,{row,0},HORIZONTAL) (trace.h:11-28). */
int peps_probe_trace_row(peps_ctx *ctx, int32_t row, double *psi);
/* BMPSContractor::ReplaceTNNSiteTrace (bmps/impl/bmps_contractor_trace.h:326-420): amplitude with the three consecutive
 * sites starting at (row, col) along `orient` (0 = HORIZONTAL, 1 = VERTICAL) set to the physical indices
 * cfg3[w][0..2]; grows the environments it needs first. The building block of MCUpdateSquareTNN3SiteExchange. */
int peps_probe_tnn_trace(peps_ctx *ctx, int32_t row, int32_t col, int32_t orient, const int32_t *cfg3, double *psi);
/* BMPSContractor::ReplaceNNNSiteTrace (kind 0, bmps/impl/bmps_contractor_trace.h:207-324, both MPS orientations) and
 * ReplaceSqrt5DistTwoSiteTrace (kind 1, :426-536): amplitude with the two corner sites of the plaquette whose upper-left
 * site is (row, col) EXCHANGING their physical indices. dir 0 = LEFTUP_TO_RIGHTDOWN, 1 = LEFTDOWN_TO_RIGHTUP; orient
 * 0 = HORIZONTAL (2 x 2 / 2 x 3 plaquette between two-row environments), 1 = VERTICAL (2 x 2 / 3 x 2 between two-column
 * environments). Grows InitBTen2 / GrowFullBTen2 (init.h:130-186, grow.h:375-515) first. */
int peps_probe_plaquette_trace(peps_ctx *ctx, int32_t kind, int32_t row, int32_t col, int32_t dir, int32_t orient, double *psi);
/* Size of bmps_set_[position]; copy of tensor i of stack entry k, [W][d0][d1][d2]; dims returned. */
int32_t peps_bmps_stack_size(peps_ctx *ctx, int32_t position);
int peps_get_bmps_tensor(peps_ctx *ctx, int32_t position, int32_t k, int32_t i, double *out, int32_t dims[3]);
/* Counters: 0 absorptions, 1 BTen steps, 2 traces, 3 Jacobi sweeps, 4 Jacobi calls, 5 QR calls,
 * 6 kernel launches, 7 pooled device bytes. */
int64_t peps_stat(peps_ctx *ctx, int32_t which);
/* Per-kernel-class device timing with CUDA events on the launching stream. Classes: 0 contraction (gett),
 * 1 trace dot, 2 CAQR panel, 3 Jacobi round, 4 small kernels, 5 CAQR trailing update. peps_profile_get syncs and
 * fills arrays of 6. */
int peps_profile_enable(peps_ctx *ctx, int32_t on);
int peps_profile_get(peps_ctx *ctx, double *ms, int64_t *launches, double *flops, int32_t reset);
/* Stream synchronisation and the context's cudaStream_t (for CUDA-event timing by the caller). */
int peps_sync(peps_ctx *ctx);
void *peps_stream(peps_ctx *ctx);

/* ---- stand-alone kernels exposed for unit parity tests ---------------------------------------------- */
/* R factor of W matrices (m x n row-major): out [W][min(m,n)][n]. */
int peps_test_qr_r(int32_t device, int32_t W, int32_t m, int32_t n, const double *a, double *r_out);
/* Truncated right singular vectors of W matrices (nr x nc): b_out [W][tcap][nc], kept_out [W]; total Jacobi sweeps. */
int peps_test_truncate(int32_t device, int32_t W, int32_t nr, int32_t nc, int32_t dmin, int32_t dmax, double trunc_err,
                       const double *theta, double *b_out, int32_t *kept_out, int32_t *sweeps_out);
/* One step of the boundary-MPS R chain on the context's walkers (its number type and environment settings; no TPS needed):
 * A[w] is m x n (a_re, plus a_im in a complex context). r_re / r_im [W][cap][n] receive r with r^H r = A^H A up to the
 * dropped rows (eps > 0: rank-revealing step, rows below eps * largest row norm dropped), cap = min(m, n), min(2m, 2n) in a
 * complex context; rows >= rows_out are zero. row_cnt (may be NULL): rows >= row_cnt[w] * row_scale of A[w] are zero;
 * rank_hint: rank of the previous factor (early-stop start); reduce_tall: tall matrices are reduced by row chunks first.
 * cnt_out[w]: rows >= cnt_out[w] of r[w] are exactly zero; tri_out: r is upper trapezoidal. */
int peps_test_chain_step(peps_ctx *ctx, int32_t m, int32_t n, const double *a_re, const double *a_im, const int32_t *row_cnt,
                         int32_t row_scale, int32_t rank_hint, double eps, int32_t reduce_tall, double *r_re, double *r_im,
                         int32_t *rows_out, int32_t *cnt_out, int32_t *tri_out);
/* One truncation step of the boundary-MPS compression on the context's walkers: the kept right singular vectors (rows of
 * V^H) of Theta[w] (rows x cols, th_re / th_im) by the TensorToolkit rule (dmin, dmax, trunc_err). held = 0 fills the
 * factorisation buffer through a writer (SVD compression), held = 1 hands over a tensor holding Theta (variational sweeps).
 * b_re / b_im [W][min(dmax, rows, cols)][cols]; kept_out [W]: rows kept, rows beyond are zero. */
int peps_test_truncated_right_vectors(peps_ctx *ctx, int32_t rows, int32_t cols, const double *th_re, const double *th_im,
                                      int32_t dmin, int32_t dmax, double trunc_err, int32_t held, double *b_re, double *b_im,
                                      int32_t *kept_out);
/* Batched einsum of two tensors per walker (spec like "apb,kea->kepb"), host buffers. */
int peps_test_einsum(int32_t device, int32_t W, const char *spec, const int32_t *dims_a, int32_t rank_a,
                     const int32_t *dims_b, int32_t rank_b, const double *a, const double *b, double *c);

#ifdef __cplusplus
}
#endif
#endif /* PEPS_B200_H */
