"""Host-side mirror of the reference's plugin / operator interface for the VMC sampling path.

Names, argument meaning and error behaviour follow the reference (paths relative to
/root/reference/include/qlpeps/):

  BMPSTruncateParams            one_dim_tn/boundary_mps/bmps.h:47-98
  MonteCarloParams              algorithm/vmc_update/monte_carlo_peps_params.h:37-92
  Configuration                 vmc_basic/configuration.h:57
  SplitIndexTPS                 two_dim_tn/tps/split_index_tps.h:80-607 (dense, real FP64)
  SquareSpinOneHalfXXZModelOBC  algorithm/vmc_update/model_solvers/square_spin_onehalf_xxz_obc.h:174-328
  MCUpdateSquareNNExchange      vmc_basic/configuration_update_strategies/square_nn_updater.h:146-188
  MCEnergyGradEvaluator         algorithm/vmc_update/mc_energy_grad_evaluator.h:57-330

The one structural difference: the reference runs ONE Markov chain per MPI rank
(monte_carlo_engine.h:563); here ``walkers`` chains are batched per GPU, so "rank" in the reference's
formulas reads "walker" (times the number of GPUs when a torch.distributed group is given).

All arithmetic happens behind the C ABI (include/peps_b200.h); numpy here only packs / unpacks buffers.
"""
import ctypes as C
import math
from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np

from . import _lib


class PepsError(RuntimeError):
    """Non-zero status from the C ABI (the reference throws std::runtime_error / std::invalid_argument)."""


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _ip(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32))


def _up(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint32))


@dataclass
class BMPSTruncateParams:
    D_min: int = 1
    D_max: int = 2 ** 31 - 1
    trunc_err: float = 0.0
    compress_scheme: int = 0            # CompressMPSScheme: 0 SVD_COMPRESS, 1 VARIATION2Site, 2 VARIATION1Site
    convergence_tol: float = 0.0
    iter_max: int = 1

    @staticmethod
    def SVD(d_min, d_max, trunc_error):
        return BMPSTruncateParams(int(d_min), int(d_max), float(trunc_error))

    @staticmethod
    def Variational2Site(d_min, d_max, trunc_error, convergence_tol, iter_max):
        return BMPSTruncateParams(int(d_min), int(d_max), float(trunc_error), 1, float(convergence_tol), int(iter_max))

    @staticmethod
    def Variational1Site(d_min, d_max, trunc_error, convergence_tol, iter_max):
        return BMPSTruncateParams(int(d_min), int(d_max), float(trunc_error), 2, float(convergence_tol), int(iter_max))


class Configuration:
    """rows x cols grid of physical indices."""

    def __init__(self, rows_or_array, cols=None):
        if cols is None:
            self.data = np.array(rows_or_array, dtype=np.int32)
        else:
            self.data = np.zeros((rows_or_array, cols), dtype=np.int32)

    def rows(self):
        return self.data.shape[0]

    def cols(self):
        return self.data.shape[1]

    def __call__(self, site):
        return int(self.data[site[0], site[1]])

    def __eq__(self, other):
        return np.array_equal(self.data, other.data)

    def Random(self, occupancy, seed=None):
        """Configuration::Random(occupancy_num) (vmc_basic/configuration.h:127-164): occupancy[s] sites in state s, shuffled.
        The reference draws from std::random_device (not reproducible); here an optional seed makes the draw repeatable."""
        occ = [int(x) for x in occupancy]
        if sum(occ) != self.data.size:
            raise ValueError("Configuration.Random: the occupancy numbers must add up to the number of sites")
        flat = np.concatenate([np.full(n, s_, dtype=np.int32) for s_, n in enumerate(occ)])
        np.random.default_rng(seed).shuffle(flat)
        self.data = flat.reshape(self.data.shape)
        return self

    def Sum(self):
        return int(self.data.sum())


@dataclass
class PsiConsistencyWarningParams:
    """algorithm/vmc_update/monte_carlo_peps_params.h (RuntimeParams::psi_consistency)."""
    enabled: bool = True
    master_only: bool = False
    threshold: float = 1e-3
    max_warnings: int = 50
    max_print_elems: int = 8


@dataclass
class ConfigurationRescueParams:
    """RuntimeParams::config_rescue: amplitudes with |psi| <= min or >= max (or NaN / inf) are invalid."""
    enabled: bool = True
    amplitude_min_threshold: float = np.finfo(np.float64).tiny
    amplitude_max_threshold: float = np.finfo(np.float64).max


def check_wavefunction_amplitude_validity(amplitudes, min_threshold, max_threshold):
    """CheckWaveFunctionAmplitudeValidity (vmc_basic/wave_function_component.h:393-401), element-wise over walkers."""
    a = np.abs(np.asarray(amplitudes))
    with np.errstate(invalid="ignore"):
        return np.isfinite(a) & (a > min_threshold) & (a < max_threshold)


def compute_psi_consistency_summary_aligned(psi_list):
    """ComputePsiConsistencySummaryAligned (algorithm/vmc_update/psi_consistency.h:76-130): (psi_mean, psi_rel_err) of
    one configuration's list of contraction results, signs aligned to the element of largest magnitude."""
    psi = np.asarray(psi_list)
    if psi.size == 0:
        return 0.0, 0.0
    ref = psi[int(np.argmax(np.abs(psi)))]
    aligned = psi.copy()
    if abs(ref) > 1e-14:
        aligned = np.where(np.real(psi * np.conj(ref / abs(ref))) < 0.0, -psi, psi)    # unit phase of ref: no overflow for huge amplitudes
    mean = np.sum(aligned) / psi.size
    denom = max(abs(mean), np.finfo(np.float64).eps)
    return mean, float(np.max(np.abs(aligned - mean)) / denom)


@dataclass
class MonteCarloParams:
    num_samples: int
    num_warmup_sweeps: int
    sweeps_between_samples: int
    initial_config: Optional[Configuration] = None
    is_warmed_up: bool = False


class SplitIndexTPS:
    """tps(r, c)[s] = dense (L, D, R, U) array; also the gradient / O* vector type (vector-space ops)."""

    def __init__(self, tensors):
        self.t = tensors
        self.rows_, self.cols_ = len(tensors), len(tensors[0])

    def rows(self):
        return self.rows_

    def cols(self):
        return self.cols_

    def PhysicalDim(self):
        return len(self.t[0][0])

    def __call__(self, site):
        return self.t[site[0]][site[1]]

    def bond_dim(self):
        return max(max(x.shape) for row in self.t for site in row for x in site)

    def pack(self):
        dt = np.complex128 if np.iscomplexobj(self.t[0][0][0]) else np.float64
        return np.concatenate([np.ascontiguousarray(x, dtype=dt).ravel() for row in self.t for site in row for x in site])

    @staticmethod
    def unpack(flat, like):
        out, pos = [], 0
        for row in like.t:
            orow = []
            for site in row:
                osite = []
                for x in site:
                    osite.append(np.array(flat[pos:pos + x.size]).reshape(x.shape))
                    pos += x.size
                orow.append(osite)
            out.append(orow)
        return SplitIndexTPS(out)

    def _like(self, tensors):
        """A vector with this one's index structure (subclasses keep their extra structure, e.g. the fermion parities)."""
        return SplitIndexTPS(tensors)

    def _zip(self, other, fn):
        return self._like([[[fn(a, b) for a, b in zip(sa, sb)] for sa, sb in zip(ra, rb)]
                           for ra, rb in zip(self.t, other.t)])

    def __add__(self, o):
        return self._zip(o, lambda a, b: a + b)

    def __sub__(self, o):
        return self._zip(o, lambda a, b: a - b)

    def __mul__(self, s):
        if isinstance(s, SplitIndexTPS):           # operator*(SITPS, SITPS) = sum conj(a) b  (split_index_tps.h:370-377)
            return sum(np.vdot(a, b) for ra, rb in zip(self.t, s.t) for sa, sb in zip(ra, rb) for a, b in zip(sa, sb))
        return self._like([[[x * s for x in site] for site in row] for row in self.t])

    __rmul__ = __mul__

    def NormSquare(self):
        return float(sum(np.sum(np.abs(x) ** 2) for row in self.t for site in row for x in site))


class FermionSplitIndexTPS(SplitIndexTPS):
    """SplitIndexTPS<T, fZ2QN>: dense (L, D, R, U) blocks (the dim-1 parity leg dropped) plus the fermion parity of
    every index value (par[r][c] = [pL, pD, pR, pU]) and of every physical state (phys_par). The vector-space operations
    are those of the dense container; gradients / O* come back in the same entries."""

    def __init__(self, tensors, par, phys_par):
        super().__init__(tensors)
        self.par = par
        self.phys_par = tuple(int(x) for x in phys_par)

    def _like(self, tensors):
        return FermionSplitIndexTPS(tensors, self.par, self.phys_par)

    def leg_par_flat(self):
        return np.ascontiguousarray(np.concatenate([np.asarray(p, dtype=np.int32).ravel()
                                                    for row in self.par for site in row for p in site]), dtype=np.int32)

    @staticmethod
    def unpack(flat, like):
        d = SplitIndexTPS.unpack(flat, like)
        return FermionSplitIndexTPS(d.t, like.par, like.phys_par)

    @staticmethod
    def random(rows, cols, D, seed, phys_par=(1, 0), n_odd=None):
        """Parity-conserving uniform [-1, 1) tensors; every bond has D//2 (or n_odd) odd index values, placed last
        (SURVEY.md 8d.1, config #4: 'even/odd blocks D/2 each')."""
        rng = np.random.default_rng(seed)
        n_odd = D // 2 if n_odd is None else n_odd
        bp = np.array([0] * (D - n_odd) + [1] * n_odd, dtype=np.int32)
        one = np.zeros(1, dtype=np.int32)
        T = [[None] * cols for _ in range(rows)]
        par = [[None] * cols for _ in range(rows)]
        for r in range(rows):
            for c in range(cols):
                ps = [bp if c > 0 else one, bp if r < rows - 1 else one, bp if c < cols - 1 else one, bp if r > 0 else one]
                tot = (ps[0][:, None, None, None] + ps[1][None, :, None, None] + ps[2][None, None, :, None]
                       + ps[3][None, None, None, :]) % 2
                par[r][c] = ps
                T[r][c] = [rng.uniform(-1.0, 1.0, tot.shape) * (tot == pp) for pp in phys_par]
        return FermionSplitIndexTPS(T, par, phys_par)


@dataclass
class SquareSpinOneHalfXXZModelOBC:
    jz: float = 1.0
    jxy: float = 1.0
    pinning00: float = 0.0


@dataclass
class SquareSpinOneHalfJ1J2XXZModelOBC:
    """model_solvers/square_spin_onehalf_j1j2_xxz_obc.h:34-113; the one-argument reference ctor (j2) is
    SquareSpinOneHalfJ1J2XXZModelOBC(1, 1, j2, j2, 0)."""
    jz: float = 1.0
    jxy: float = 1.0
    jz2: float = 0.0
    jxy2: float = 0.0
    pinning00: float = 0.0


class TableModel:
    """A model given by local Hamiltonian matrices (seam B2 as data, include/peps_b200.h peps_set_model_term): h2 /
    h2_nnn are (d*d, d*d) matrices in the basis p = c1*d + c2 (site1 = left / upper site; diagonals: left site of the
    link), h1 is (d, d). What a reference-style EvaluateBondEnergy / EvaluateNNNEnergy / EvaluateTotalOnsiteEnergy mix-in
    (square_nnn_energy_solver.h:171-198) computes, with its matrix elements as data."""

    bond_pin = None         # (site1, site2, H): an extra two-site term on ONE NN bond (peps_set_bond_pin)
    enable_sc_measurement = False   # t-J measurement solvers: also record SC_bond_singlet_h / _v (MCPEPSMeasurer)

    def SetSingletPairPinningField(self, site1, site2, delta):
        """SquaretJModelMixIn::SetSingletPairPinningField (square_tJ_model.h:109-133): delta * (delta_dag + delta) on one NN
        bond of a t-J model (states 0 = up, 1 = down, 2 = empty); the two sites in either order."""
        if not np.isfinite(delta):
            raise ValueError("Singlet pair pinning delta must be finite.")
        (r1, c1), (r2, c2) = site1, site2
        if abs(r1 - r2) + abs(c1 - c2) != 1:
            raise ValueError("Singlet pair pinning field requires a nearest-neighbor bond.")
        if (r2, c2) < (r1, c1):
            (r1, c1), (r2, c2) = (r2, c2), (r1, c1)
        dd, d = TableModel.tj_singlet_pair_tables()
        self.bond_pin = ((r1, c1), (r2, c2), delta * (dd + d))
        return self

    def ClearSingletPairPinningField(self):
        self.bond_pin = None
        return self

    @staticmethod
    def tj_singlet_pair_tables():
        """(delta_dag, delta) of EvaluateBondSingletPairFortJModel (square_tJ_model.h:546-602) as 9x9 tables in the basis
        p = c1*3 + c2: value = sum_p' H[p, p'] conj(psi(p') / psi)."""
        s = 1.0 / np.sqrt(2.0)
        dd, d = np.zeros((9, 9)), np.zeros((9, 9))
        dd[8, 1], dd[8, 3] = s, -s             # (E, E) -> (up, dn) - (dn, up)
        d[1, 8], d[3, 8] = s, -s               # (up, dn) -> (E, E);  (dn, up) -> -(E, E)
        return dd, d

    def __init__(self, phys, h2=None, h2_nnn=None, h1=None):
        self.phys, self.h2, self.h2_nnn, self.h1 = phys, h2, h2_nnn, h1

    @staticmethod
    def tables(H):
        H = np.asarray(H, dtype=np.float64)
        n = H.shape[0]
        off = [[q for q in range(n) if q != p and H[p, q] != 0.0] for p in range(n)]
        T = max((len(o) for o in off), default=0)
        target = -np.ones((n, max(T, 1)), dtype=np.int32)
        coef = np.zeros((n, max(T, 1)))
        for p, o in enumerate(off):
            for t, q in enumerate(o):
                target[p, t], coef[p, t] = q, H[p, q]
        return T, np.ascontiguousarray(np.diag(H)), target, coef

    @staticmethod
    def xxz(jz=1.0, jxy=1.0, jz2=0.0, jxy2=0.0, pinning00=None):
        """SquareSpinOneHalfXXZModelMixIn (square_spin_onehalf_xxz_obc.h:72-140) as tables; cfg 0/1, Sz = cfg - 1/2."""
        def bond(a, b):
            H = np.diag([0.25 * a, -0.25 * a, -0.25 * a, 0.25 * a])
            H[1, 2] = H[2, 1] = 0.5 * b
            return H
        return TableModel(2, bond(jz, jxy), bond(jz2, jxy2) if (jz2 or jxy2) else None)

    @staticmethod
    def spinless_fermion(t, t2=0.0, V=0.0):
        """SquareSpinlessFermion(t, t2, V) (model_solvers/square_spinless_fermion.h:51-213) as tables; 0 = occupied,
        1 = empty. The hop amplitude is the matrix element in the engine's fermion mode: the Jordan-Wigner sign of the
        move is supplied by the contraction (psi_ex / psi along one path), as in the reference."""
        h2 = np.zeros((4, 4))
        h2[0, 0] = V
        h2[1, 2] = h2[2, 1] = -t
        h2n = None
        if t2 != 0.0:
            h2n = np.zeros((4, 4))
            h2n[1, 2] = h2n[2, 1] = -t2
        return TableModel(2, h2, h2n)

    @staticmethod
    def tj(t, J, V=0.0, mu=0.0, t2=0.0):
        """SquaretJNNModel(t, J, mu) / SquaretJVModel(t, t2, J, V, mu) / SquaretJNNNModel (model_solvers/square_tJ_model.h:
        300-345, NNN hopping :424-460); 0 = up, 1 = down, 2 = empty."""
        h2 = np.zeros((9, 9))
        for a in (0, 1):
            h2[a * 3 + a, a * 3 + a] = V
            h2[a * 3 + 2, 2 * 3 + a] = h2[2 * 3 + a, a * 3 + 2] = -t
        h2[1, 1] = h2[3, 3] = -0.5 * J + V
        h2[1, 3] = h2[3, 1] = 0.5 * J
        h1 = np.diag([-mu, -mu, 0.0]) if mu != 0.0 else None
        h2n = None
        if t2 != 0.0:
            h2n = np.zeros((9, 9))
            for a in (0, 1):
                h2n[a * 3 + 2, 2 * 3 + a] = h2n[2 * 3 + a, a * 3 + 2] = -t2
        return TableModel(3, h2, h2n, h1)

    @staticmethod
    def tfim(h):
        """TransverseFieldIsingSquareOBC (transverse_field_ising_square_obc.h:149-247): -sz sz bonds, -h sx on-site."""
        return TableModel(2, np.diag([-1.0, 1.0, 1.0, -1.0]), None, np.array([[0.0, -h], [-h, 0.0]]))


@dataclass
class MCUpdateSquareTNN3SiteExchange:
    """square_3site_updater.h:23-160: permutations of the spins on three consecutive sites, Suwa-Todo choice."""
    seed: int = 5489
    kind = 2


@dataclass
class TransverseFieldIsingSquareOBC:
    """model_solvers/transverse_field_ising_square_obc.h:28-247: H = -sum_<ij> sz_i sz_j - h sum_i sx_i."""
    h: float = 1.0


@dataclass
class MCUpdateSquareNNExchange:
    """Explicit-seed constructor of the reference updater; walker w draws from std::mt19937(seed + w)."""
    seed: int = 5489
    kind = 0


@dataclass
class MCUpdateSquareNNFullSpaceUpdate:
    """square_nn_updater.h:253-293: all phys^2 local states per bond, Suwa-Todo choice (no Sz conservation)."""
    seed: int = 5489
    kind = 1


class WalkerBatch:
    """Thin RAII wrapper over a peps_ctx: W walkers of one lattice on one GPU."""

    def __init__(self, rows, cols, phys, D, walkers, trunc: BMPSTruncateParams, device=0, lib=None):
        self.lib = lib if lib is not None else _lib.load()
        self.rows, self.cols, self.phys, self.D, self.W = rows, cols, phys, D, walkers
        cfg = _lib.PepsConfig(rows, cols, phys, D, walkers, device, trunc.D_min, min(trunc.D_max, 2 ** 31 - 1), trunc.trunc_err)
        h = C.c_void_p()
        if self.lib.peps_create(C.byref(h), C.byref(cfg)) != 0:
            raise PepsError(self.lib.peps_last_error(None).decode())
        self.h = h
        self.tps_size = self.lib.peps_tps_size(self.h)
        if trunc.compress_scheme != 0:
            self._ck(self.lib.peps_set_compress_scheme(self.h, trunc.compress_scheme, trunc.convergence_tol, trunc.iter_max))

    def close(self):
        if getattr(self, "h", None):
            self.lib.peps_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise PepsError(self.lib.peps_last_error(self.h).decode())

    # state
    def set_fermion(self, ftps):
        """Switch the context to fZ2-graded tensors (peps_set_fermion); before set_tps / set_model."""
        pp = np.ascontiguousarray(ftps.phys_par, dtype=np.int32)
        lp = ftps.leg_par_flat()
        self._ck(self.lib.peps_set_fermion(self.h, _ip(pp), _ip(lp), lp.size))
        self.phys_par = tuple(int(x) for x in ftps.phys_par)

    # complex (QLTEN_Complex) states: planar arrays across the ABI, numpy complex here
    def set_complex(self):
        """Switch a fresh context to complex arithmetic (peps_set_complex): before the first set_tps."""
        self._ck(self.lib.peps_set_complex(self.h))
        self.is_complex = True

    def _planar(self, what, shape):
        re, im = np.empty(shape), np.empty(shape)
        self._ck(self.lib.peps_get_planar(self.h, what, _dp(re), _dp(im)))
        return re + 1j * im

    def amplitudes_c(self):
        return self._planar(0, self.W)

    def eloc_c(self):
        return self._planar(1, self.W)

    def holes_c(self):
        """Raw environments PunchHole(site) per walker; the reference's hole_res is their conjugate (Dag)."""
        return self._planar(2, (self.W, self.lib.peps_holes_stride(self.h)))

    def accumulators_c(self):
        return self._planar(3, self.tps_size), self._planar(4, self.tps_size)

    def set_jastrow(self, v, density):
        """JastrowDress (wave_function_component.h:107-135): v[nsites][nsites] symmetric, density[phys]."""
        n = self.rows * self.cols
        v = np.ascontiguousarray(v, dtype=np.float64).reshape(n, n)
        d = np.ascontiguousarray(density, dtype=np.int32).reshape(self.phys)
        self._ck(self.lib.peps_set_jastrow(self.h, _dp(v), _ip(d)))

    def set_tps(self, tps):
        if getattr(self, "is_complex", False):
            flat = (np.concatenate([np.asarray(x, dtype=np.complex128).ravel() for row in tps.t for site in row for x in site])
                    if isinstance(tps, SplitIndexTPS) else np.asarray(tps, dtype=np.complex128).ravel())
            if flat.size != self.tps_size:
                raise PepsError(f"TPS has {flat.size} elements, context expects {self.tps_size}")
            re, im = np.ascontiguousarray(flat.real), np.ascontiguousarray(flat.imag)
            self._ck(self.lib.peps_set_tps_c(self.h, _dp(re), _dp(im), re.size))
            return
        flat = tps.pack() if isinstance(tps, SplitIndexTPS) else np.ascontiguousarray(tps, dtype=np.float64)
        if flat.size != self.tps_size:
            raise PepsError(f"TPS has {flat.size} elements, context expects {self.tps_size}")
        self._ck(self.lib.peps_set_tps(self.h, _dp(flat), flat.size))

    def get_tps_flat(self):
        if getattr(self, "is_complex", False):
            return self._planar(5, self.tps_size)
        out = np.empty(self.tps_size)
        self._ck(self.lib.peps_get_tps(self.h, _dp(out), out.size))
        return out

    def set_truncation(self, trunc):
        self._ck(self.lib.peps_set_truncation(self.h, trunc.D_min, trunc.D_max, trunc.trunc_err))
        self._ck(self.lib.peps_set_compress_scheme(self.h, trunc.compress_scheme, trunc.convergence_tol, max(1, trunc.iter_max)))

    def set_jacobi(self, tol=1e-14, inner_sweeps=1, max_sweeps=40):
        self._ck(self.lib.peps_set_jacobi(self.h, tol, inner_sweeps, max_sweeps))

    def set_deflation(self, eps):
        self._ck(self.lib.peps_set_deflation(self.h, eps))

    def set_updater(self, updater):
        self.updater_kind = int(getattr(updater, "kind", updater))
        self._ck(self.lib.peps_set_updater(self.h, self.updater_kind))

    def set_chain_deflation(self, eps):
        self._ck(self.lib.peps_set_chain_deflation(self.h, eps))

    def set_model(self, model):
        if isinstance(model, TableModel):
            self._ck(self.lib.peps_clear_model_terms(self.h))
            for kind, H in ((0, model.h2), (1, model.h2_nnn), (2, model.h1)):
                if H is None:
                    continue
                T, diag, target, coef = TableModel.tables(H)
                self._ck(self.lib.peps_set_model_term(self.h, kind, T, _dp(diag), _ip(target), _dp(coef)))
            if model.bond_pin is not None:
                (r1, c1), (r2, c2), H = model.bond_pin
                T, diag, target, coef = TableModel.tables(H)
                self._ck(self.lib.peps_set_bond_pin(self.h, r1 * self.cols + c1, r2 * self.cols + c2, T, _dp(diag), _ip(target), _dp(coef)))
            return
        self._ck(self.lib.peps_clear_model_terms(self.h))
        if isinstance(model, TransverseFieldIsingSquareOBC):
            self._ck(self.lib.peps_set_model_tfim(self.h, model.h))
        elif hasattr(model, "jz2"):
            self._ck(self.lib.peps_set_model_j1j2_xxz(self.h, model.jz, model.jxy, model.jz2, model.jxy2, model.pinning00))
        else:
            self._ck(self.lib.peps_set_model_xxz(self.h, model.jz, model.jxy, model.pinning00))

    def set_configs(self, cfgs):
        a = np.ascontiguousarray(cfgs, dtype=np.int32).reshape(self.W, self.rows, self.cols)
        self._ck(self.lib.peps_set_configs(self.h, _ip(a)))

    def get_configs(self):
        a = np.empty((self.W, self.rows, self.cols), dtype=np.int32)
        self._ck(self.lib.peps_get_configs(self.h, _ip(a)))
        return a

    def seed_rng(self, seeds):
        a = np.ascontiguousarray(seeds, dtype=np.uint32).reshape(self.W)
        self._ck(self.lib.peps_seed_rng(self.h, _up(a)))

    def get_rng_state(self):
        mt = np.empty((self.W, 624), dtype=np.uint32)
        idx = np.empty(self.W, dtype=np.int32)
        self._ck(self.lib.peps_get_rng_state(self.h, _up(mt), _ip(idx)))
        return mt, idx

    def set_rng_state(self, mt, idx):
        mt = np.ascontiguousarray(mt, dtype=np.uint32)
        idx = np.ascontiguousarray(idx, dtype=np.int32)
        self._ck(self.lib.peps_set_rng_state(self.h, _up(mt), _ip(idx)))

    # hot path
    def init_walkers(self):
        self._ck(self.lib.peps_init_walkers(self.h))

    def amplitudes(self):
        a = np.empty(self.W)
        self._ck(self.lib.peps_get_amplitudes(self.h, _dp(a)))
        return a

    def normalize_state_order1(self, max_abs_override=0.0):
        f = C.c_double()
        self._ck(self.lib.peps_normalize_state_order1(self.h, max_abs_override, C.byref(f)))
        return f.value

    def sweep(self, n=1):
        """StepSweep with the updater chosen by set_updater (NN exchange unless told otherwise)."""
        acc = np.empty(self.W)
        kind = getattr(self, "updater_kind", 0)
        f = {0: self.lib.peps_sweep, 1: self.lib.peps_sweep_full_space, 2: self.lib.peps_sweep_three_site}[kind]
        self._ck(f(self.h, n, _dp(acc)))
        return acc

    def energy_and_holes(self, calc_holes=True, want_psi=False):
        """CalEnergyAndHoles for every walker. Complex context: returns complex E_loc (and psi list) -- the psi list crosses
        the ABI as [entry][re W | im W], E_loc is read back through peps_get_planar."""
        cx = getattr(self, "is_complex", False)
        e = np.empty(self.W)
        psi = np.empty((self.rows + self.cols, 2 if cx else 1, self.W)) if want_psi else None
        self._ck(self.lib.peps_energy_and_holes(self.h, int(calc_holes), _dp(e), _dp(psi) if want_psi else None))
        if cx:
            e = self.eloc_c()
            psi = psi[:, 0] + 1j * psi[:, 1] if want_psi else None
        elif want_psi:
            psi = psi[:, 0]
        return (e, psi) if want_psi else e

    def measure(self):
        """One EvaluateObservables call for every walker (model_solvers/base/square_nnn_model_measurement_solver.h:
        33-214): dict of per-walker arrays under the reference's registry keys."""
        W, r, c = self.W, self.rows, self.cols
        npl = 2 if getattr(self, "is_complex", False) else 1         # complex context: planar arrays (re block, im block)
        e = np.empty((npl, W))
        eh, ev = np.empty((npl, W, r, c - 1)), np.empty((npl, W, r - 1, c))
        edr, eur = np.empty((npl, W, r - 1, c - 1)), np.empty((npl, W, r - 1, c - 1))
        corr = np.empty((npl, W, c // 2))
        self._ck(self.lib.peps_measure(self.h, _dp(e), _dp(eh), _dp(ev), _dp(edr), _dp(eur), _dp(corr)))
        e, eh, ev, edr, eur, corr = [(a[0] + 1j * a[1]) if npl == 2 else a[0] for a in (e, eh, ev, edr, eur, corr)]
        cfg = self.get_configs()
        if getattr(self, "phys_par", None) is not None:        # fermion models: requires_density_measurement (charge)
            out = {"energy": e, "charge": np.asarray(self.phys_par, dtype=float)[cfg], "bond_energy_h": eh,
                   "bond_energy_v": ev, "bond_energy_dr": edr, "bond_energy_ur": eur}
            if self.phys_par == (1, 1, 0):                     # t-J: CalSpinSzImpl (square_tJ_model.h:233-236): up, down, empty
                out["spin_z"] = np.array([0.5, -0.5, 0.0])[cfg]
            return out
        sz = cfg.astype(float) - 0.5
        first_down = (cfg[:, r // 2, c // 4] == 0)[:, None]          # EvaluateOffDiagOrderInRow channel split (:281-287)
        flat = sz.reshape(W, -1)
        iu = np.triu_indices(flat.shape[1])
        return {"energy": e, "spin_z": sz, "bond_energy_h": eh, "bond_energy_v": ev,
                "bond_energy_dr": edr, "bond_energy_ur": eur,
                "SmSp_row": np.where(first_down, 0.0, corr), "SpSm_row": np.where(first_down, corr, 0.0),
                "SzSz_all2all": flat[:, iu[0]] * flat[:, iu[1]]}

    def measure_bond_observable(self, H):
        """A two-site operator as a (d*d, d*d) table on every NN bond (peps_measure_bond_term): (horizontal [W][rows][cols-1],
        vertical [W][rows-1][cols]) of sum_p' H[p, p'] conj(psi(p') / psi)."""
        W, r, c = self.W, self.rows, self.cols
        npl = 2 if getattr(self, "is_complex", False) else 1
        T, diag, target, coef = TableModel.tables(H)
        oh, ov = np.empty((npl, W, r, c - 1)), np.empty((npl, W, r - 1, c))
        self._ck(self.lib.peps_measure_bond_term(self.h, T, _dp(diag), _ip(target), _dp(coef), _dp(oh), _dp(ov)))
        return (oh[0] + 1j * oh[1], ov[0] + 1j * ov[1]) if npl == 2 else (oh[0], ov[0])

    def measure_site_observable(self, H1):
        """A one-site operator as a (d, d) table on every site (peps_measure_site_term): [W][rows][cols] of
        sum_p' H1[p, p'] conj(psi(p') / psi)."""
        npl = 2 if getattr(self, "is_complex", False) else 1
        T, diag, target, coef = TableModel.tables(H1)
        out = np.empty((npl, self.W, self.rows, self.cols))
        self._ck(self.lib.peps_measure_site_term(self.h, T, _dp(diag), _ip(target), _dp(coef), _dp(out)))
        return out[0] + 1j * out[1] if npl == 2 else out[0]

    def measure_tfim(self):
        """TransverseFieldIsingSquareOBC::EvaluateObservables (transverse_field_ising_square_obc.h:60-146): energy, spin_z,
        sigma_x (per site) and SzSz_row along the middle row."""
        cfg = self.get_configs()
        sz = cfg.astype(float) - 0.5
        row, c1 = self.rows // 2, self.cols // 4
        return {"energy": self.energy_and_holes(False), "spin_z": sz,
                "sigma_x": self.measure_site_observable(np.array([[0.0, 1.0], [1.0, 0.0]])),
                "SzSz_row": np.stack([sz[:, row, c1] * sz[:, row, c1 + i] for i in range(1, self.cols // 2 + 1)], axis=1)}

    def measure_sc_bond_singlet(self):
        """SC_bond_singlet_h / _v of the t-J measurement solvers (base/square_nnn_model_measurement_solver.h:116-131):
        (conj(delta_dag) + delta) / 2 per bond."""
        dd, d = TableModel.tj_singlet_pair_tables()
        ddh, ddv = self.measure_bond_observable(dd)
        dh, dv = self.measure_bond_observable(d)
        return (np.conj(ddh) + dh) / 2.0, (np.conj(ddv) + dv) / 2.0

    def measure_structure_factor(self):
        """MeasureStructureFactor (structure_factor_measurement_mixin.h:89-228): (pairs [n][4] = (y1, x1, y2, x2),
        values [W][n]) -- raw S+S- overlaps; the registry key SpSm_cross holds value / amplitude."""
        n = int(self.lib.peps_structure_factor_pairs(self.h))
        cx = getattr(self, "is_complex", False)
        out = np.empty((2 if cx else 1, self.W, n))
        self._ck(self.lib.peps_measure_structure_factor(self.h, _dp(out)))
        out = out[0] + 1j * out[1] if cx else out[0]
        pairs = np.array([(y1, x1, y2, x2) for y1 in range(self.rows - 1) for x1 in range(self.cols)
                          for y2 in range(y1 + 1, self.rows) for x2 in range(self.cols)], dtype=np.int32)
        return pairs, out

    def holes(self):
        n = self.lib.peps_holes_stride(self.h)
        a = np.empty((self.W, n))
        self._ck(self.lib.peps_get_holes(self.h, _dp(a)))
        return a

    def zero_accumulators(self):
        self._ck(self.lib.peps_zero_accumulators(self.h))

    def accumulate_ostar(self):
        self._ck(self.lib.peps_accumulate_ostar(self.h))

    def accumulators(self):
        o, eo = np.empty(self.tps_size), np.empty(self.tps_size)
        self._ck(self.lib.peps_get_accumulators(self.h, _dp(o), _dp(eo), o.size))
        return o, eo

    def sample(self, sweeps_between_samples=1):
        e, acc = np.empty(self.W), np.empty(self.W)
        self._ck(self.lib.peps_sample(self.h, sweeps_between_samples, _dp(e), _dp(acc)))
        return e, acc

    # stochastic reconfiguration store
    def sr_reserve(self, max_walker_samples):
        self._ck(self.lib.peps_sr_reserve(self.h, int(max_walker_samples)))

    def sr_collect(self, on=True):
        self._ck(self.lib.peps_sr_collect(self.h, int(on)))

    def sr_clear(self):
        self._ck(self.lib.peps_sr_clear(self.h))

    def sr_count(self):
        return int(self.lib.peps_sr_count(self.h))

    def sr_matvec(self, v, mean_dot_v):
        if getattr(self, "is_complex", False):             # planar across the ABI, numpy complex here
            v = np.asarray(v, dtype=np.complex128)
            pv = np.ascontiguousarray(np.concatenate([v.real, v.imag]))
            out = np.empty(2 * self.tps_size)
            m = complex(mean_dot_v)
            self._ck(self.lib.peps_sr_matvec_c(self.h, _dp(pv), m.real, m.imag, _dp(out), out.size))
            return out[:self.tps_size] + 1j * out[self.tps_size:]
        v = np.ascontiguousarray(v, dtype=np.float64)
        out = np.empty(self.tps_size)
        self._ck(self.lib.peps_sr_matvec(self.h, _dp(v), float(mean_dot_v), _dp(out), out.size))
        return out

    # probes
    def _probe_out(self):
        return np.empty((2 if getattr(self, "is_complex", False) else 1, self.W))    # complex context: planar (re[W], im[W])

    @staticmethod
    def _probe_val(a):
        return a[0] + 1j * a[1] if a.shape[0] == 2 else a[0]

    def probe_trace_row(self, row):
        a = self._probe_out()
        self._ck(self.lib.peps_probe_trace_row(self.h, row, _dp(a)))
        return self._probe_val(a)

    def probe_tnn_trace(self, row, col, orient, cfg3):
        """ReplaceTNNSiteTrace for every walker: cfg3[w] = physical indices of the three consecutive sites."""
        c3 = np.ascontiguousarray(cfg3, dtype=np.int32).reshape(self.W, 3)
        a = self._probe_out()
        self._ck(self.lib.peps_probe_tnn_trace(self.h, row, col, orient, _ip(c3), _dp(a)))
        return self._probe_val(a)

    def probe_plaquette_trace(self, kind, row, col, direction, orient):
        """kind 0: ReplaceNNNSiteTrace, 1: ReplaceSqrt5DistTwoSiteTrace, the two corner sites exchanging their spins."""
        a = self._probe_out()
        self._ck(self.lib.peps_probe_plaquette_trace(self.h, kind, row, col, direction, orient, _dp(a)))
        return self._probe_val(a)

    def bmps_stack_size(self, pos):
        return self.lib.peps_bmps_stack_size(self.h, pos)

    def bmps_tensor(self, pos, k, i):
        dims = np.zeros(3, dtype=np.int32)
        self._ck(self.lib.peps_get_bmps_tensor(self.h, pos, k, i, None, _ip(dims)))
        out = np.empty((self.W, int(dims[0]), int(dims[1]), int(dims[2])))
        self._ck(self.lib.peps_get_bmps_tensor(self.h, pos, k, i, _dp(out), _ip(dims)))
        return out

    def stat(self, which):
        return int(self.lib.peps_stat(self.h, which))

    KERNEL_CLASSES = ("gett", "dot", "panel_qr", "jacobi_round", "small", "apply_reflector")

    def profile_enable(self, on=True):
        self._ck(self.lib.peps_profile_enable(self.h, int(on)))

    def profile_get(self, reset=True):
        ms = np.zeros(6)
        fl = np.zeros(6)
        ln = np.zeros(6, dtype=np.int64)
        self._ck(self.lib.peps_profile_get(self.h, _dp(ms), ln.ctypes.data_as(C.POINTER(C.c_int64)), _dp(fl), int(reset)))
        return {k: dict(ms=float(ms[i]), launches=int(ln[i]), flops=float(fl[i])) for i, k in enumerate(self.KERNEL_CLASSES)}

    def sync(self):
        self._ck(self.lib.peps_sync(self.h))

    def stream(self):
        return self.lib.peps_stream(self.h)

    def accumulator_device_ptrs(self):
        return self.lib.peps_ostar_sum_device(self.h), self.lib.peps_eloc_ostar_sum_device(self.h)


class MCPEPSMeasurer:
    """MCPEPSMeasurer (algorithm/vmc_update/monte_carlo_peps_measurer_impl.h:172-257): warm up, then per sample
    `sweeps_between_samples` sweeps + EvaluateObservables; a walker plays the role of a rank: per-walker sample means,
    then mean and standard error across walkers (GatherStatisticListOfData, monte_carlo_tools/statistics.h:288-339).
    Built keys: energy, spin_z, bond_energy_h / _v / _dr / _ur, SmSp_row / SpSm_row, SzSz_all2all and, with
    enable_structure_factor, SpSm_cross (all pairs with y2 > y1; self.sf_pairs lists (y1, x1, y2, x2))."""

    def __init__(self, mc_params, trunc, tps, model, updater, walkers, device=0, lib=None, enable_structure_factor=False):
        rows, cols = tps.rows(), tps.cols()
        self.mc = mc_params
        self.model = model
        self.is_complex = bool(np.iscomplexobj(tps.t[0][0][0]))
        self.enable_structure_factor = enable_structure_factor      # StructureFactorMeasurementMixin::SetEnableStructureFactor
        self.batch = WalkerBatch(rows, cols, tps.PhysicalDim(), tps.bond_dim(), walkers, trunc, device, lib)
        if self.is_complex:
            self.batch.set_complex()
        if isinstance(tps, FermionSplitIndexTPS):              # config #4: fZ2 states, keys energy / charge / bond energies
            self.batch.set_fermion(tps)
        self.batch.set_tps(tps)
        self.batch.set_model(model)
        self.batch.set_updater(updater)
        self.batch.set_configs(np.broadcast_to(np.asarray(mc_params.initial_config.data, dtype=np.int32),
                                               (walkers, rows, cols)).copy())
        self.batch.seed_rng(np.arange(walkers, dtype=np.uint32) + np.uint32(updater.seed))
        self.batch.init_walkers()
        self.has_nnn = (hasattr(model, "jz2") and (model.jz2 != 0.0 or model.jxy2 != 0.0)) or \
                       (isinstance(model, TableModel) and model.h2_nnn is not None)

    def Execute(self):
        b, W = self.batch, self.batch.W
        if not self.mc.is_warmed_up:
            for _ in range(self.mc.num_warmup_sweeps):
                b.sweep(1)
        nper = max(1, -(-self.mc.num_samples // W))
        sums = None
        for _ in range(nper):
            b.sweep(self.mc.sweeps_between_samples)
            obs = b.measure_tfim() if isinstance(self.model, TransverseFieldIsingSquareOBC) else b.measure()
            if getattr(self.model, "enable_sc_measurement", False):  # t-J solvers: ModelType::enable_sc_measurement
                obs["SC_bond_singlet_h"], obs["SC_bond_singlet_v"] = b.measure_sc_bond_singlet()
            if self.enable_structure_factor:                         # registry key SpSm_cross: overlap / amplitude
                self.sf_pairs, raw = b.measure_structure_factor()
                obs["SpSm_cross"] = raw / (b.amplitudes_c() if self.is_complex else b.amplitudes())[:, None]
            if sums is None:
                sums = {k: np.zeros_like(v, dtype=complex if np.iscomplexobj(v) else float) for k, v in obs.items()}
            for k, v in obs.items():
                sums[k] += v
        out = {}
        for k, v in sums.items():
            if k in ("bond_energy_dr", "bond_energy_ur") and not self.has_nnn:
                continue
            per_walker = v / nper
            mean = per_walker.mean(axis=0)
            err = (np.sqrt((np.abs(per_walker - mean) ** 2).sum(axis=0) / (W * (W - 1))) if W > 1
                   else np.full(np.shape(mean), np.inf))
            out[k] = (mean, err)
        self.results = out
        self.samples_per_walker = nper
        return out

    def DumpData(self, path=""):
        """MCPEPSMeasurer::DumpData: stats CSVs + metadata.txt of the last Execute() (see dump_measurement_stats)."""
        b = self.batch
        meta = {"total_samples_requested": self.mc.num_samples, "samples_per_rank": self.samples_per_walker,
                "samples_scheduled_total": self.samples_per_walker * b.W, "samples_collected_total": self.samples_per_walker * b.W,
                "mpi_size": b.W, "warmup_sweeps": self.mc.num_warmup_sweeps, "sweeps_between_samples": self.mc.sweeps_between_samples,
                "initial_config_warmed_up": "true" if self.mc.is_warmed_up else "false", "lx": b.cols, "ly": b.rows,
                "boundary_condition": "Open", "peps_bond_dimension": b.D}
        dump_measurement_stats(self.results, path, meta)


class _CudaView:
    """__cuda_array_interface__ wrapper of a device pointer owned by the library (zero-copy torch view)."""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": "<f8", "data": (int(ptr), False), "version": 3}


def _csv(x):
    """ToCsvString (monte_carlo_peps_measurer_impl.h:24-36): scientific, max_digits10 = 17 significant digits; complex values
    as the stream form of std::complex, (re,im)."""
    if isinstance(x, (complex, np.complexfloating)):
        return "(%.16e,%.16e)" % (x.real, x.imag)
    return "%.16e" % float(x)


def dump_measurement_stats(results, path, meta=None):
    """MCPEPSMeasurer::DumpData (monte_carlo_peps_measurer_impl.h:266-330, 396-440, 544-620): ``<path>/stats/<key>_mean.csv``
    + ``_stderr.csv`` for observables registered with a 2-D shape (one lattice row per line), ``<path>/stats/<key>.csv``
    with the header ``index,mean,stderr`` for everything else, and ``<path>/metadata.txt``. ``results``: {key: (mean,
    stderr)} as returned by MCPEPSMeasurer.Execute()."""
    import os
    base = (path.rstrip("/") + "/") if path else "./"
    stats = base + "stats/"
    os.makedirs(stats, exist_ok=True)
    for key, (mean, err) in results.items():
        mean = np.asarray(mean, dtype=complex if np.iscomplexobj(mean) else float)      # QLTEN_Complex runs keep complex means
        err = np.asarray(err, dtype=float)
        if mean.ndim == 2:
            for suffix, arr in (("_mean.csv", mean), ("_stderr.csv", err)):
                with open(stats + key + suffix, "w") as f:
                    for row in arr:
                        f.write(",".join(_csv(v) for v in row) + "\n")
        else:
            with open(stats + key + ".csv", "w") as f:
                f.write("index,mean,stderr\n")
                for i, (m, e) in enumerate(zip(mean.ravel(), err.ravel())):
                    f.write(f"{i},{_csv(m)},{_csv(e)}\n")
    with open(base + "metadata.txt", "w") as f:
        f.write("format_version 1\n")
        for k, v in (meta or {}).items():
            f.write(f"{k} {v}\n")
        f.write(f"registered_observables {len(results)}\n")
        f.write(f"stats_path {base}stats\n")


@dataclass
class EvaluateResult:
    """MCEnergyGradEvaluator::Result (mc_energy_grad_evaluator.h:66-75)."""
    energy: float
    energy_error: float
    gradient: SplitIndexTPS
    gradient_norm: float
    accept_rates_avg: List[float]
    energy_samples: np.ndarray = field(default=None)
    Ostar_mean: Optional[SplitIndexTPS] = None       # set when SR buffers were collected (O* samples stay in HBM)
    total_samples: int = 0


def combine_energy_bins(energy_samples):
    """MeanAndBinnedErrorSqrtNUniformBin over all walkers (vmc_basic/monte_carlo_tools/statistics.h:146-225):
    per walker bins of floor(sqrt(N)) samples, incomplete tail bin discarded, mean / stderr over all bin means.
    energy_samples: [walkers_total][N]."""
    es = np.asarray(energy_samples, dtype=np.float64)
    n = es.shape[1]
    if n == 0:
        return 0.0, 0.0
    bin_size = max(1, int(math.sqrt(n)))
    nb = n // bin_size
    means = []
    for w in range(es.shape[0]):
        for i in range(nb):
            s = 0.0
            for x in es[w, i * bin_size:(i + 1) * bin_size]:
                s += float(x)
            means.append(s / bin_size)
    if not means:
        return 0.0, 0.0
    mean = 0.0
    for m in means:
        mean += m
    mean /= len(means)
    if len(means) == 1:
        return mean, float("inf")
    var = sum((m - mean) ** 2 for m in means) / len(means)
    return mean, math.sqrt(var / (len(means) - 1))


class MCEnergyGradEvaluator:
    """Evaluate(state) -> (energy, gradient, error): the B1 seam of SURVEY.md section 8b.

    ``dist`` is an optional initialised torch.distributed module with world_size > 1: energies are all-gathered
    and the two accumulators all-reduced (NCCL on the GPU, gloo in CPU tests), replacing the reference's
    Gather/Gatherv + per-tensor MPI_Send/Recv (mc_energy_grad_evaluator.h:292-310).
    """

    def __init__(self, mc_params: MonteCarloParams, trunc: BMPSTruncateParams, tps: SplitIndexTPS, model, updater,
                 walkers, configs=None, device=0, lib=None, dist=None, rank=0, world_size=1, config_rescue=None,
                 psi_consistency=None):
        self.mc, self.trunc, self.model, self.updater = mc_params, trunc, model, updater
        self.config_rescue = config_rescue or ConfigurationRescueParams()
        self.psi_consistency = psi_consistency or PsiConsistencyWarningParams()
        self.psi_warnings = []                 # (sample index, walker, psi_rel_err) above the threshold, up to max_warnings
        self.rescued = []                      # walkers whose configuration was replaced by EnsureConfigurationValidity
        self.state = tps                       # the device holds its own copy (set_tps below and in every Evaluate(state))
        self.dist, self.rank, self.world_size = dist, rank, world_size
        self.batch = WalkerBatch(tps.rows(), tps.cols(), tps.PhysicalDim(), tps.bond_dim(), walkers, trunc, device, lib)
        self.is_complex = bool(np.iscomplexobj(tps.t[0][0][0]))    # QLTEN_Complex state: complex arithmetic on the device
        if self.is_complex:
            self.batch.set_complex()
        if isinstance(tps, FermionSplitIndexTPS):
            self.batch.set_fermion(tps)
        self.batch.set_model(model)
        self.batch.set_updater(updater)
        self.batch.set_tps(tps)
        if configs is None:
            if mc_params.initial_config is None:
                raise PepsError("MCEnergyGradEvaluator: initial configuration required")
            configs = np.broadcast_to(mc_params.initial_config.data, (walkers,) + mc_params.initial_config.data.shape)
        self.batch.set_configs(configs)
        base = updater.seed + rank * walkers
        self.batch.seed_rng(np.arange(base, base + walkers, dtype=np.uint64).astype(np.uint32))
        self.batch.init_walkers()
        self.warmed_up = mc_params.is_warmed_up

    def EnsureConfigurationValidity(self):
        """MonteCarloEngine::EnsureConfigurationValidity (monte_carlo_engine.h:340-414), walkers playing the ranks: a
        walker whose amplitude is NaN / inf / outside (min, max) takes the configuration of the FIRST valid walker (in
        global walker order over all GPUs) and is re-evaluated; the batch is then marked as not warmed up (walkers run in
        lock step, so the warm-up sweeps are repeated for all of them). Raises when rescue is disabled or no walker on any
        GPU is valid. Returns the list of rescued local walkers."""
        b = self.batch
        rp = self.config_rescue
        valid = check_wavefunction_amplitude_validity(self._amps(), rp.amplitude_min_threshold, rp.amplitude_max_threshold)
        src_cfg, n_valid_global, n_total = None, int(valid.sum()), b.W * self.world_size
        cfgs = b.get_configs()
        if self.dist is not None and self.world_size > 1:
            import torch
            dev = "cuda" if self.dist.get_backend() == "nccl" else "cpu"
            first = int(np.argmax(valid)) if valid.any() else -1
            mine = torch.tensor([int(valid.sum()), first], dtype=torch.int64, device=dev)
            allv = [torch.empty_like(mine) for _ in range(self.world_size)]
            self.dist.all_gather(allv, mine)
            allv = [t.cpu().numpy() for t in allv]
            n_valid_global = int(sum(t[0] for t in allv))
            src_rank = next((r for r, t in enumerate(allv) if t[1] >= 0), -1)
            if n_valid_global < n_total and src_rank >= 0:
                buf = torch.from_numpy(cfgs[int(allv[src_rank][1])].astype(np.int32) if self.rank == src_rank
                                       else np.zeros((b.rows, b.cols), dtype=np.int32)).to(dev)
                self.dist.broadcast(buf, src=src_rank)
                src_cfg = buf.cpu().numpy()
        elif valid.any():
            src_cfg = cfgs[int(np.argmax(valid))]
        if n_valid_global == n_total:
            return []
        if not rp.enabled:
            raise PepsError(f"{n_total - n_valid_global}/{n_total} walkers have invalid configurations and configuration rescue is disabled")
        if n_valid_global == 0 or src_cfg is None:
            raise PepsError(f"all {n_total} walkers have invalid configurations: check bond dimension, truncation cutoff, initial configuration")
        bad = np.flatnonzero(~valid)
        if bad.size:
            cfgs[bad] = src_cfg
            b.set_configs(cfgs)
            b.init_walkers()                   # TryConstructWavefunction_ for the rescued walkers (monte_carlo_engine.h:396)
            again = check_wavefunction_amplitude_validity(self._amps(), rp.amplitude_min_threshold, rp.amplitude_max_threshold)
            if not again.all():
                raise PepsError("rescue FAILED: the valid configuration of another walker is not valid here (TPS or truncation parameter issue)")
            self.warmed_up = False
        self.rescued = [int(w) for w in bad]
        return self.rescued

    def WarmUp(self):
        """MonteCarloEngine::WarmUp (monte_carlo_engine.h:146-173)."""
        if not self.warmed_up:
            for _ in range(self.mc.num_warmup_sweeps):
                self.batch.sweep(1)
            self.warmed_up = True
        amps = self._amps()
        bad = (not np.all(np.isfinite(amps))) or bool(np.any(amps == 0))
        mx = float("inf") if bad else float(np.max(np.abs(amps)))
        if self.dist is not None and self.world_size > 1:
            mx = self._allreduce_max(mx)       # an illegal amplitude on any rank shows up as inf on every rank: all raise together
        if not math.isfinite(mx):
            raise PepsError("Amplitude is still not legal after warm up")
        self.batch.normalize_state_order1(mx)
        self.state = type(self.state).unpack(self.batch.get_tps_flat(), self.state)

    def _amps(self):
        return self.batch.amplitudes_c() if self.is_complex else self.batch.amplitudes()

    def _allreduce_max(self, x):
        import torch
        t = torch.tensor([x], dtype=torch.float64)
        if self.dist.get_backend() == "nccl":
            t = t.cuda()
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.cpu()[0])

    def Evaluate(self, state: Optional[SplitIndexTPS] = None, collect_sr_buffers: bool = False) -> EvaluateResult:
        b = self.batch
        if state is not None:                  # always re-upload: the caller may have edited the tensors in place
            self.state = state
            b.set_tps(state)
        b.init_walkers()                       # engine_.RefreshWavefunctionComponent()  (:164)
        n = self.samples_per_walker()
        b.zero_accumulators()
        if collect_sr_buffers:                 # collect_sr_buffers_ of the reference evaluator (:181-183, :273-277)
            if getattr(self, "_sr_cap", 0) < n * b.W:   # reallocate only when the store is too small
                b.sr_reserve(n * b.W)
                self._sr_cap = n * b.W
            b.sr_clear()
        b.sr_collect(collect_sr_buffers)
        energies = np.empty((b.W, n), dtype=complex if self.is_complex else float)
        accept = np.zeros(b.W)
        pc = self.psi_consistency
        for s in range(n):                     # the walker loop (:205-282), all walkers in lock step
            if pc.enabled:                     # psi list of the energy solver -> consistency summary (psi_consistency.h)
                acc = b.sweep(self.mc.sweeps_between_samples)
                e, psi = b.energy_and_holes(True, True)
                b.accumulate_ostar()
                for w in range(b.W):
                    _, rel = compute_psi_consistency_summary_aligned(psi[:, w])
                    if rel > pc.threshold and len(self.psi_warnings) < pc.max_warnings:
                        self.psi_warnings.append((s, w, rel))
            else:
                e, acc = b.sample(self.mc.sweeps_between_samples)
                if self.is_complex:
                    e = b.eloc_c()
            if not np.all(np.isfinite(e)):     # zero amplitude: std::runtime_error in the reference solver (square_nnn_energy_solver.h:148-150)
                raise PepsError("local energy is not finite (zero or illegal amplitude): run EnsureConfigurationValidity / WarmUp first")
            energies[:, s] = e
            accept += acc
        all_e = energies
        if self.dist is not None and self.world_size > 1:
            import torch
            nccl = self.dist.get_backend() == "nccl"
            dev = "cuda" if nccl else "cpu"
            if nccl:
                # NCCL all-reduce straight on the device pointers of the two accumulators (peps_ostar_sum_device /
                # peps_eloc_ostar_sum_device): the gradient sums never pass through host memory before the reduction
                b.sync()
                for ptr in b.accumulator_device_ptrs():        # complex: both planes of an accumulator are contiguous
                    self.dist.all_reduce(torch.as_tensor(_CudaView(ptr, b.tps_size * (2 if self.is_complex else 1)), device="cuda"))
                torch.cuda.synchronize()
                osum, eosum = b.accumulators_c() if self.is_complex else b.accumulators()
            else:
                osum, eosum = b.accumulators_c() if self.is_complex else b.accumulators()
                host = np.ascontiguousarray(np.stack([osum, eosum]))
                buf = torch.from_numpy(host.view(np.float64))          # complex sums reduce as (re, im) pairs
                self.dist.all_reduce(buf)
                osum, eosum = host
            mine = torch.from_numpy(np.ascontiguousarray(energies).view(np.float64)).to(dev)
            gathered = [torch.empty_like(mine) for _ in range(self.world_size)]
            self.dist.all_gather(gathered, mine)
            all_e = np.concatenate([g.cpu().numpy() for g in gathered], axis=0)
            if self.is_complex:
                all_e = np.ascontiguousarray(all_e).view(np.complex128)
        elif self.is_complex:
            osum, eosum = b.accumulators_c()
        else:
            osum, eosum = b.accumulators()
        if self.is_complex:                    # complex mean of the bin means, error bar from the real parts
            er, err = combine_energy_bins(all_e.real)
            ei, _ = combine_energy_bins(all_e.imag)
            energy = complex(er, ei)
        else:
            energy, err = combine_energy_bins(all_e)
        total_walkers = all_e.shape[0]
        grad_flat = (eosum - np.conj(energy) * osum) / (n * total_walkers)        # (:296-309)
        grad = type(self.state).unpack(grad_flat, self.state)
        b.sr_collect(False)
        res = EvaluateResult(energy, err, grad, grad.NormSquare(), [float(np.mean(accept / n))], all_e)
        if collect_sr_buffers:
            res.Ostar_mean = type(self.state).unpack(osum / (n * total_walkers), self.state)
            res.total_samples = n * total_walkers
        return res

    def EvaluateEnergyOnly(self, state: Optional[SplitIndexTPS] = None):
        """MCEnergyGradEvaluator::EvaluateEnergyOnly (mc_energy_grad_evaluator.h:331-392), the step-selector trial: the same
        chains with CalEnergy (no holes, no O*, no gradient reduction). Returns (energy, energy_error, accept_rates_avg)."""
        b = self.batch
        if state is not None:
            self.state = state
            b.set_tps(state)
        b.init_walkers()
        n = self.samples_per_walker()
        energies = np.empty((b.W, n), dtype=complex if self.is_complex else float)
        accept = np.zeros(b.W)
        for s in range(n):
            accept += b.sweep(self.mc.sweeps_between_samples)
            e = b.energy_and_holes(False)
            if not np.all(np.isfinite(e)):
                raise PepsError("local energy is not finite (zero or illegal amplitude): run EnsureConfigurationValidity / WarmUp first")
            energies[:, s] = e
        all_e = energies
        if self.dist is not None and self.world_size > 1:
            import torch
            dev = "cuda" if self.dist.get_backend() == "nccl" else "cpu"
            mine = torch.from_numpy(np.ascontiguousarray(energies).view(np.float64)).to(dev)
            gathered = [torch.empty_like(mine) for _ in range(self.world_size)]
            self.dist.all_gather(gathered, mine)
            all_e = np.concatenate([g.cpu().numpy() for g in gathered], axis=0)
            if self.is_complex:
                all_e = np.ascontiguousarray(all_e).view(np.complex128)
        if self.is_complex:
            er, err = combine_energy_bins(all_e.real)
            energy = complex(er, combine_energy_bins(all_e.imag)[0])
        else:
            energy, err = combine_energy_bins(all_e)
        return energy, err, [float(np.mean(accept / n))]

    def CalculateNaturalGradient(self, result: EvaluateResult, diag_shift, cg_params=None, init_guess=None):
        """Optimizer::CalculateNaturalGradient (optimizer/optimizer_impl.h:1031-1089) against the O* samples kept in
        HBM by the last Evaluate(collect_sr_buffers=True). Returns (natural_gradient, cg_iterations, residual_norm)."""
        from . import sr
        cb = None
        if self.dist is not None and self.world_size > 1:
            cb = sr.device_allreduce_callback(self.dist)      # NCCL on the device pointer of the matvec output
        r = sr.calculate_natural_gradient(self.batch, result.gradient.pack(), result.Ostar_mean.pack(), result.total_samples,
                                          diag_shift, cg_params or sr.ConjugateGradientParams(),
                                          None if init_guess is None else init_guess.pack(), cb)
        return type(self.state).unpack(r.x, self.state), r.iterations, r.residual_norm

    def CalculateNaturalGradientMinSR(self, result: EvaluateResult, diag_shift):
        """MinSR (optimizer/minsr_scalapack.h), the minimum-step form of SR, on the O* samples kept in HBM by the last
        Evaluate(collect_sr_buffers=True): x = (S + diag_shift)^{-1} g_c solved in sample space by a device Cholesky of the
        N x N matrix T + diag_shift (sr.calculate_natural_gradient_minsr). Returns (natural_gradient, energy_mean) with
        energy_mean the plain mean of the stored local energies; g_c equals result.gradient when the samples per walker are
        a multiple of floor(sqrt(samples per walker)) (then the binned mean is the plain mean). Single GPU only."""
        from . import sr
        if self.world_size > 1:
            raise PepsError("CalculateNaturalGradientMinSR: MinSR needs every O* sample on one GPU (world_size > 1 is not "
                            "supported; use CalculateNaturalGradient)")
        if result.total_samples == 0:
            raise PepsError("CalculateNaturalGradientMinSR: Evaluate(state, collect_sr_buffers=True) first")
        x, em = sr.calculate_natural_gradient_minsr(self.batch, result.total_samples, diag_shift)
        return type(self.state).unpack(x, self.state), em

    def samples_per_walker(self):
        """SamplesPerRank = ceil(total / ranks) (monte_carlo_engine.h:97-98) with ranks = walkers * GPUs."""
        total = self.batch.W * self.world_size
        return max(1, -(-self.mc.num_samples // total))
