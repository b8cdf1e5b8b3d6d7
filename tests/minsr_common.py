"""Shared MinSR scenarios: the same checks run on the host simulation (test_minsr.py) and on the GPU (test_gpu_minsr.py).

Each scenario evaluates a state with collect_sr_buffers, rebuilds the dense O* samples from the oracle chains (the same
Markov chains: same seeds), and checks MinSR against the dense (S + shift)^{-1} g, the dense sample-space MinSR
(minsr_dense), the probe's centred T and the product CG."""
import numpy as np

from oracle import vmc, sr as osr
from peps_b200 import sr
from peps_b200.api import (BMPSTruncateParams, SplitIndexTPS, MCEnergyGradEvaluator, MonteCarloParams,
                           SquareSpinOneHalfXXZModelOBC, MCUpdateSquareNNExchange)


def minsr_dense(ostars, obar, elocs, diag_shift):
    """Dense statement of MinSR (optimizer/minsr_scalapack.h): X_i = (O*_i - obar) / sqrt(N), e_i = conj(E_i - Ebar) / sqrt(N)
    with Ebar the plain mean, T = X X^H (T_ij = <X_i, X_j> = sum conj(X_i) X_j), x = X^T (T + diag_shift I)^{-1} e, i.e.
    x = sum_i z_i X_i. Returns (x, T)."""
    o = np.asarray(ostars)
    n = o.shape[0]
    e = np.asarray(elocs)
    x_rows = (o - obar) / np.sqrt(n)
    t = np.conj(x_rows) @ x_rows.T
    z = np.linalg.solve(t + diag_shift * np.eye(n), np.conj(e - e.mean()) / np.sqrt(n))
    return x_rows.T @ z, t


def store_order(a, W, n):
    """[W * n, ...] in walker-major order -> the store's order (sample s of walker w at s * W + w)."""
    a = np.asarray(a)
    return a.reshape((W, n) + a.shape[1:]).swapaxes(0, 1).reshape((W * n,) + a.shape[1:])


def boson_scenario(lib, rows=3, cols=3, D=2, W=3, n=4, chi=4, complex_=False):
    """test_sr.py::sr_scenario's setup (real) or parity_common.run_complex_sr's (complex): evaluator, result, dense O* rows
    and local energies, both in store order."""
    if complex_:
        from parity_common import complex_tps
        tps_l = complex_tps(rows, cols, D, 8)
    else:
        tps_l = vmc.random_tps(rows, cols, 2, D, seed=8)
    cfgs = np.stack([vmc.shuffled_half_filled_config(rows, cols, 60 + w) for w in range(W)])
    mc = MonteCarloParams(num_samples=n * W, num_warmup_sweeps=0, sweeps_between_samples=1, is_warmed_up=True)
    ev = MCEnergyGradEvaluator(mc, BMPSTruncateParams.SVD(chi, chi, 0.0), SplitIndexTPS(tps_l), SquareSpinOneHalfXXZModelOBC(1, 1, 0),
                               MCUpdateSquareNNExchange(31), walkers=W, configs=cfgs, lib=lib)
    res = ev.Evaluate(collect_sr_buffers=True)
    model = vmc.XXZModel()
    ostars = []
    for w in range(W):
        wk = vmc.Walker(tps_l, cfgs[w], (chi, chi, 0.0))
        up = vmc.NNExchangeUpdater(31 + w)
        for _ in range(n):
            up.sweep(tps_l, wk)
            _, holes, _ = model.energy_and_holes(tps_l, wk, True)
            inv = np.conj(1.0 / wk.amplitude)
            sample = {(r, c): (int(wk.config[r, c]), holes[r][c] * inv) for r in range(rows) for c in range(cols)}
            ostars.append(osr.dense_ostar(sample, tps_l))
    return ev, res, store_order(ostars, W, n), store_order(res.energy_samples.reshape(-1), W, n)


def fermion_scenario(lib, W=3, n=4):
    """test_fermion_hostsim.py::test_fermion_sr_natural_gradient's fZ2 state and chains."""
    from oracle import fermion as F
    from peps_b200.api import FermionSplitIndexTPS, TableModel, Configuration
    from parity_common import fermion_configs
    rows, cols, D, trunc = 3, 3, 2, (4, 4, 0.0)
    f = F.FermionTPS.random(rows, cols, D, 13)
    ftps = FermionSplitIndexTPS(f.T, f.par, f.phys_par)
    cfgs = fermion_configs(rows, cols, W, 2)
    ev = MCEnergyGradEvaluator(MonteCarloParams(n * W, 0, 1, Configuration(cfgs[0]), True), BMPSTruncateParams.SVD(*trunc), ftps,
                               TableModel.spinless_fermion(1.0, 0.5, 0.2), MCUpdateSquareNNExchange(seed=41), W, configs=cfgs, lib=lib)
    res = ev.Evaluate(collect_sr_buffers=True)
    omodel = F.SpinlessFermionModel(1.0, 0.5, 0.2)
    ostars = []
    for w in range(W):
        wk = F.FermionWalker(f, cfgs[w], trunc)
        up = F.FermionNNExchangeUpdater(41 + w)
        for _ in range(n):
            up.sweep(wk)
            _, ost, _ = omodel.energy_and_holes(wk, True)
            dense = [[[np.zeros_like(x) for x in site] for site in row] for row in f.T]
            for r in range(rows):
                for c in range(cols):
                    dense[r][c][int(wk.config[r, c])] = ost[r][c]
            ostars.append(np.concatenate([x.ravel() for row in dense for site in row for x in site]))
    return ev, res, store_order(ostars, W, n), store_order(res.energy_samples.reshape(-1), W, n)


def check_minsr(ev, res, ostars, elocs, shift=1e-3, cg_tol=1e-8):
    """MinSR == dense (S + shift)^{-1} g (1e-10), == the dense sample-space MinSR, probe T == oracle T (1e-12 of max|T|),
    == the product CG at relative_tolerance 1e-12 (cg_tol). Returns x."""
    o = np.asarray(ostars)
    N = o.shape[0]
    assert ev.batch.sr_count() == N == res.total_samples
    obar = o.mean(axis=0)
    nat, em = ev.CalculateNaturalGradientMinSR(res, shift)
    x = nat.pack()
    g = res.gradient.pack()
    oc = o - obar
    s_dense = oc.T @ oc.conj() / N + shift * np.eye(obar.size)
    x_dense = np.linalg.solve(s_dense, g)
    scale = np.max(np.abs(x_dense))
    assert np.max(np.abs(x - x_dense)) < 1e-10 * scale, np.max(np.abs(x - x_dense)) / scale
    x_or, t_or = minsr_dense(o, obar, elocs, shift)
    assert np.max(np.abs(x - x_or)) < 1e-10 * scale
    assert abs(em - np.mean(elocs)) < 1e-12 * max(1.0, abs(em))
    assert abs(em - res.energy) < 1e-12 * max(1.0, abs(em))        # n per walker is a multiple of the bin size here
    t = sr.minsr_tmatrix(ev.batch)
    assert np.max(np.abs(t - t_or)) < 1e-12 * np.max(np.abs(t_or)), np.max(np.abs(t - t_or)) / np.max(np.abs(t_or))
    cg, _, _ = ev.CalculateNaturalGradient(res, shift, sr.ConjugateGradientParams(max_iter=500, relative_tolerance=1e-12))
    assert np.max(np.abs(x - cg.pack())) < cg_tol * scale, np.max(np.abs(x - cg.pack())) / scale
    return x


def check_errors(ev, res, lib):
    """Clear errors for shift <= 0, a wrong total_samples, world_size > 1 and an empty store; MinSR leaves the store and a
    later CG solve unchanged."""
    import pytest
    from peps_b200.api import PepsError
    params = sr.ConjugateGradientParams(max_iter=200, relative_tolerance=1e-10)
    before, it0, r0 = ev.CalculateNaturalGradient(res, 1e-3, params)
    count = ev.batch.sr_count()
    for bad in (0.0, -1e-3):
        with pytest.raises(PepsError, match="diag_shift must be positive"):
            ev.CalculateNaturalGradientMinSR(res, bad)
    with pytest.raises(PepsError, match="differs from the"):
        sr.calculate_natural_gradient_minsr(ev.batch, res.total_samples + 1, 1e-3)
    ev.CalculateNaturalGradientMinSR(res, 1e-3)
    assert ev.batch.sr_count() == count
    after, it1, r1 = ev.CalculateNaturalGradient(res, 1e-3, params)
    assert it0 == it1 and r0 == r1 and np.array_equal(before.pack(), after.pack())
    ws = ev.world_size
    ev.world_size = 2
    try:
        with pytest.raises(PepsError, match="world_size > 1"):
            ev.CalculateNaturalGradientMinSR(res, 1e-3)
    finally:
        ev.world_size = ws
    ev.batch.sr_clear()
    with pytest.raises(PepsError, match="store is empty"):
        sr.calculate_natural_gradient_minsr(ev.batch, 0, 1e-3)
    with pytest.raises(PepsError, match="store is empty"):
        sr.minsr_tmatrix(ev.batch)
