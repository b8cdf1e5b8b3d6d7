"""VMC optimisation + measurement of the square-lattice Heisenberg model (OBC) on the B200 path -- the flow of the reference's
integration test tests/integration_tests/test_square_heisenberg_obc.cpp (3 x 4, SR with CG, then MCPEPSMeasurer; its pass
criterion is |E - E_ED| < 1e-3 with E_ED = -6.691680193514947 at D = 6 after a simple-update start).

Usage on a B200:  python examples/heisenberg_vmc_optimize.py [--iters 40] [--D 4]
"""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from peps_b200 import sr                                                        # noqa: E402
from peps_b200.api import (BMPSTruncateParams, Configuration, MCEnergyGradEvaluator, MCPEPSMeasurer, MonteCarloParams,   # noqa: E402
                           MCUpdateSquareNNExchange, SplitIndexTPS, SquareSpinOneHalfXXZModelOBC)

E_ED_3x4 = -6.691680193514947           # tests/integration_tests/test_square_heisenberg_obc.cpp:38


def optimize(state, rows, cols, chi, walkers, samples, iters, step, diag_shift=1e-3, seed=1, lib=None, log=print, init=None,
             model=None, solver="sr"):
    """`model`: any model of peps_b200.api (default Heisenberg); a FermionSplitIndexTPS state runs in fermion mode.
    `solver`: "sr" (conjugate gradient in parameter space) or "minsr" (direct solve in sample space, one GPU)."""
    if solver not in ("sr", "minsr"):
        raise ValueError(f"unknown solver {solver!r}: 'sr' or 'minsr'")
    model = model if model is not None else SquareSpinOneHalfXXZModelOBC(1.0, 1.0, 0.0)
    init = init if init is not None else Configuration(rows, cols).Random([rows * cols // 2, rows * cols - rows * cols // 2], seed=seed)
    mc = MonteCarloParams(num_samples=samples, num_warmup_sweeps=20, sweeps_between_samples=1, initial_config=init)
    ev = MCEnergyGradEvaluator(mc, BMPSTruncateParams.SVD(chi, 2 * chi, 1e-15), state, model, MCUpdateSquareNNExchange(seed=seed),
                               walkers, lib=lib)
    ev.EnsureConfigurationValidity()
    ev.WarmUp()
    state = ev.state
    cg = sr.ConjugateGradientParams(max_iter=100, relative_tolerance=3e-3, residual_recompute_interval=20)
    energies = []
    for it in range(iters):
        res = ev.Evaluate(state, collect_sr_buffers=True)
        if solver == "minsr":
            nat, _ = ev.CalculateNaturalGradientMinSR(res, diag_shift)
            how = "MinSR"
        else:
            nat, cg_iters, _ = ev.CalculateNaturalGradient(res, diag_shift, cg)
            how = f"CG {cg_iters} its"
        state = state - nat * step
        energies.append(float(np.real(res.energy)))
        log(f"iter {it:3d}  E = {res.energy:+.8f} +- {res.energy_error:.2e}  {how}  accept {res.accept_rates_avg[0]:.2f}")
    return energies, state


def measure(state, rows, cols, chi, walkers, samples, seed=7, lib=None, init=None, model=None):
    model = model if model is not None else SquareSpinOneHalfXXZModelOBC(1.0, 1.0, 0.0)
    init = init if init is not None else Configuration(rows, cols).Random([rows * cols // 2, rows * cols - rows * cols // 2], seed=seed)
    mc = MonteCarloParams(num_samples=samples, num_warmup_sweeps=50, sweeps_between_samples=1, initial_config=init)
    return MCPEPSMeasurer(mc, BMPSTruncateParams.SVD(chi, 2 * chi, 1e-15), state, model, MCUpdateSquareNNExchange(seed=seed),
                          walkers, lib=lib).Execute()


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=40)
    ap.add_argument("--D", type=int, default=4)
    ap.add_argument("--walkers", type=int, default=64)
    ap.add_argument("--samples", type=int, default=5120)
    a = ap.parse_args()
    rows, cols = 4, 3
    rng = np.random.default_rng(3)
    t = [[[rng.random((a.D if c > 0 else 1, a.D if r < rows - 1 else 1, a.D if c < cols - 1 else 1, a.D if r > 0 else 1)) - 0.3
           for _ in range(2)] for c in range(cols)] for r in range(rows)]
    energies, state = optimize(SplitIndexTPS(t), rows, cols, max(6, a.D), a.walkers, a.samples, a.iters, 0.1)
    obs = measure(state, rows, cols, max(6, a.D), a.walkers, 10 * a.samples)
    print(f"measured E = {obs['energy'][0]:+.6f} +- {obs['energy'][1]:.1e};  ED {E_ED_3x4:+.6f}")
