"""Stochastic reconfiguration on top of the device-resident O* sample store.

The product path is ``calculate_natural_gradient`` -> ``peps_sr_natural_gradient`` (C ABI): the whole CG loop runs in the
engine with every vector resident in HBM and the cross-GPU sum done by NCCL on the device pointer of the matvec
output. ``conjugate_gradient`` / ``SRSMatrix`` below are the host-side statement of the same loop (numpy vectors,
matvec through ``peps_sr_matvec``) kept for single-matvec checks and as the readable form of:
  * ConjugateGradientSolver        utility/conjugate_gradient_solver.h:181-276 (serial form; with several GPUs every rank
                                   runs the identical vector updates on the all-reduced matvec, so the reference's
                                   master/slave broadcast of v, :355-611, is not needed)
  * ConjugateGradientParams        optimizer/optimizer_params.h:50-57
  * SRSMatrix::operator*           optimizer/stochastic_reconfiguration_smatrix.h:45-91 (the sum over samples runs in the
                                   CUDA kernels sr_dots / sr_accumulate; normalisation + diag_shift here)
  * Optimizer::CalculateNaturalGradient  optimizer/optimizer_impl.h:1031-1089
``calculate_natural_gradient_minsr`` -> ``peps_sr_minsr_natural_gradient`` is the minimum-step form of SR
(optimizer/minsr_scalapack.h) on the same store: a direct solve in sample space, no tolerance, no iteration count.
"""
import math
from dataclasses import dataclass

import numpy as np

CONVERGED, MAX_ITERATIONS, STAGNATED, INDEFINITE_MATRIX, NUMERICAL_BREAKDOWN = range(5)
REASONS = ("kConverged", "kMaxIterations", "kStagnated", "kIndefiniteMatrix", "kNumericalBreakdown")


@dataclass
class ConjugateGradientParams:
    max_iter: int = 100
    relative_tolerance: float = 1e-4
    absolute_tolerance: float = 0.0
    residual_recompute_interval: int = 20
    orthogonality_threshold: float = 0.5


@dataclass
class CGResult:
    x: np.ndarray
    residual_norm: float
    iterations: int
    reason: int


def conjugate_gradient(matvec, b, x0, params: ConjugateGradientParams) -> CGResult:
    """Line-by-line restatement of the reference's serial solver (best-iterate tracking, stagnation / NaN /
    indefiniteness exits, orthogonality restart, periodic residual recomputation)."""
    nrm2 = lambda v: float(np.dot(v, v))
    rhs_norm_sq = nrm2(b)
    tol_sq = max(params.relative_tolerance ** 2 * rhs_norm_sq, params.absolute_tolerance ** 2)
    r = b - matvec(x0)
    r_norm_sq = nrm2(r)
    if r_norm_sq <= tol_sq:
        return CGResult(x0, math.sqrt(r_norm_sq), 0, CONVERGED)
    p, x, best_x = r.copy(), x0.copy(), x0.copy()
    best_sq = r_norm_sq
    r_prev = r.copy()
    rkp1 = r_norm_sq
    stagnation = 0
    eps = np.finfo(np.float64).eps
    for k in range(params.max_iter):
        rk = rkp1
        ap = matvec(p)
        pap = float(np.dot(p, ap))
        if not (math.isfinite(pap) and pap > 0.0):
            return CGResult(best_x, math.sqrt(best_sq), k, INDEFINITE_MATRIX)
        alpha = rk / pap
        x = x + alpha * p
        if alpha * alpha * nrm2(p) < eps * eps * nrm2(x):
            stagnation += 1
            if stagnation >= 3:
                return CGResult(best_x, math.sqrt(best_sq), k + 1, STAGNATED)
        else:
            stagnation = 0
        ri = params.residual_recompute_interval
        if ri > 0 and (k % ri) == ri - 1:
            r = b - matvec(x)
        else:
            r = r - alpha * ap
        rkp1 = nrm2(r)
        if not math.isfinite(rkp1):
            return CGResult(best_x, math.sqrt(best_sq), k + 1, NUMERICAL_BREAKDOWN)
        if rkp1 < best_sq:
            best_x, best_sq = x.copy(), rkp1
        if rkp1 <= tol_sq:
            return CGResult(x, math.sqrt(rkp1), k + 1, CONVERGED)
        if k > 0:
            if abs(float(np.dot(r_prev, r))) > params.orthogonality_threshold * rkp1:
                p = r.copy()
                r_prev = r.copy()
                continue
        r_prev = r.copy()
        beta = rkp1 / rk
        if not math.isfinite(beta):
            return CGResult(best_x, math.sqrt(best_sq), k + 1, NUMERICAL_BREAKDOWN)
        p = r + beta * p
    return CGResult(best_x, math.sqrt(best_sq), params.max_iter, MAX_ITERATIONS)


class SRSMatrix:
    """S v = (1/N_total) sum_i (O*_i . v - Obar . v) O*_i + diag_shift v with the samples resident in HBM."""

    def __init__(self, batch, ostar_mean_flat, total_samples, diag_shift=0.0, allreduce=None):
        self.batch, self.mean, self.n, self.diag_shift, self.allreduce = batch, ostar_mean_flat, total_samples, diag_shift, allreduce

    def __call__(self, v):
        mean_dot_v = np.vdot(self.mean, v) if np.iscomplexobj(self.mean) else float(np.dot(self.mean, v))   # conj(mean) . v
        out = self.batch.sr_matvec(v, mean_dot_v)
        if self.allreduce is not None:
            out = self.allreduce(out)
        out = out * (1.0 / float(self.n))
        if self.diag_shift != 0.0:
            out = out + self.diag_shift * v
        return out


def device_allreduce_callback(dist):
    """peps_allreduce_fn for an initialised torch.distributed module: wraps the DEVICE pointer handed over by the engine
    (NCCL: a zero-copy CUDA tensor view, reduced in place over NVLink; gloo in the CPU tests of the host logic, where the
    'device' buffer of the host simulation is ordinary memory)."""
    import ctypes as C
    import torch
    from . import _lib

    nccl = dist.get_backend() == "nccl"

    def cb(_user, ptr, n):
        try:
            if nccl:
                class _Cai:
                    __cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (ptr, False), "version": 3}
                t = torch.as_tensor(_Cai(), device="cuda")
                dist.all_reduce(t)
                torch.cuda.synchronize()
            else:
                arr = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_double)), shape=(n,))
                t = torch.from_numpy(arr)
                dist.all_reduce(t)
            return 0
        except Exception as exc:                      # never let an exception cross the C ABI
            import sys
            print("all-reduce callback failed:", exc, file=sys.stderr)
            return 1
    return _lib.ALLREDUCE_FN(cb)


def calculate_natural_gradient(batch, gradient_flat, ostar_mean_flat, total_samples, diag_shift, cg_params, init_guess=None,
                               allreduce_cb=None):
    """Optimizer::CalculateNaturalGradient: solves (S + diag_shift) x = gradient on the device (all CG vectors in HBM);
    raises on indefinite / breakdown like the reference, returns the best iterate on non-convergence.
    ``allreduce_cb``: a _lib.ALLREDUCE_FN (see device_allreduce_callback) or None on a single GPU."""
    import ctypes as C
    from . import _lib
    cx = bool(getattr(batch, "is_complex", False))          # complex context: planar arrays (re block, im block) across the ABI
    pk = (lambda a: np.ascontiguousarray(np.concatenate([np.asarray(a).real, np.asarray(a).imag]), dtype=np.float64)) if cx \
        else (lambda a: np.ascontiguousarray(a, dtype=np.float64))
    g, m = pk(gradient_flat), pk(ostar_mean_flat)
    x0 = None if init_guess is None else pk(init_guess)
    x = np.empty_like(g)
    prm = _lib.PepsCGParams(cg_params.max_iter, cg_params.relative_tolerance, cg_params.absolute_tolerance,
                            cg_params.residual_recompute_interval, cg_params.orthogonality_threshold)
    it, reason, resid = C.c_int32(), C.c_int32(), C.c_double()
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    cb = allreduce_cb if allreduce_cb is not None else C.cast(None, _lib.ALLREDUCE_FN)
    batch._ck(batch.lib.peps_sr_natural_gradient(batch.h, dp(g), dp(m), int(total_samples), float(diag_shift), C.byref(prm),
                                                 dp(x0) if x0 is not None else None, cb, None, dp(x), C.byref(it),
                                                 C.byref(resid), C.byref(reason)))
    if cx:
        x = x[:x.size // 2] + 1j * x[x.size // 2:]
    res = CGResult(x, resid.value, it.value, reason.value)
    if res.reason in (INDEFINITE_MATRIX, NUMERICAL_BREAKDOWN):
        raise RuntimeError(f"CG solver terminated: {REASONS[res.reason]} iterations={res.iterations} residual_norm={res.residual_norm}")
    return res


def calculate_natural_gradient_minsr(batch, total_samples, diag_shift):
    """MinSR on the device-resident store (single GPU). With X_i = (O*_i - Obar) / sqrt(N), e_i = conj(E_i - Ebar) / sqrt(N)
    and T = X X^H (N x N), returns ``(x, energy_mean)`` with

        x = X^H (T + diag_shift)^{-1} e = (S + diag_shift)^{-1} g_c,   g_c = (1/N) sum_i conj(E_i - Ebar) (O*_i - Obar),

    exact for diag_shift > 0 (push-through identity). Obar and Ebar come from the store itself; Ebar is the PLAIN mean of the
    stored local energies, so g_c equals ``EvaluateResult.gradient`` exactly when the evaluator's binned mean equals the
    plain mean, i.e. when the samples per walker are a multiple of floor(sqrt(samples per walker)). ``x`` is the packed
    TPS vector (complex in a complex context), ``energy_mean`` is Ebar."""
    import ctypes as C
    cx = bool(getattr(batch, "is_complex", False))
    x = np.empty(batch.tps_size * (2 if cx else 1))
    em = np.zeros(2)
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    batch._ck(batch.lib.peps_sr_minsr_natural_gradient(batch.h, int(total_samples), float(diag_shift), dp(x), dp(em)))
    if cx:
        return x[:x.size // 2] + 1j * x[x.size // 2:], complex(em[0], em[1])
    return x, float(em[0])


def minsr_tmatrix(batch):
    """The centred N x N matrix T = X X^H of the stored samples (complex in a complex context): a probe for tests and timing."""
    import ctypes as C
    cx = bool(getattr(batch, "is_complex", False))
    n = batch.sr_count()
    t = np.empty(n * n * (2 if cx else 1))
    batch._ck(batch.lib.peps_sr_minsr_tmatrix(batch.h, t.ctypes.data_as(C.POINTER(C.c_double)), t.size))
    t = t.reshape(-1, n, n)
    return t[0] + 1j * t[1] if cx else t[0]


def minsr_gram_diag(batch):
    """The uncentred Gram diagonal G_ii = |O*_i|^2 of the stored samples."""
    import ctypes as C
    g = np.empty(batch.sr_count())
    batch._ck(batch.lib.peps_sr_minsr_gram_diag(batch.h, g.ctypes.data_as(C.POINTER(C.c_double)), g.size))
    return g
