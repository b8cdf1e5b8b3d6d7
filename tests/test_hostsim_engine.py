"""CPU tests of the HOST logic (engine.cpp orchestration, C ABI, Python mirror) using the test-only host simulation
of the device ops. The CUDA kernels themselves are checked on the GPU box by tests/test_gpu_parity.py."""
import numpy as np
import pytest

import hostsim_lib
from parity_common import run_pipeline_parity, run_gradient_parity
from peps_b200 import _lib
from peps_b200.api import (BMPSTruncateParams, SplitIndexTPS, WalkerBatch, MCEnergyGradEvaluator, MonteCarloParams,
                           Configuration, SquareSpinOneHalfXXZModelOBC, MCUpdateSquareNNExchange, PepsError)
from oracle import vmc
from helpers import load_golden_tps, exact_summation


@pytest.fixture(scope="module")
def lib():
    return hostsim_lib.load()


def test_backend_is_hostsim(lib):
    assert lib.peps_backend_name() == b"hostsim"


@pytest.mark.parametrize("rows,cols,D,trunc", [
    (4, 4, 3, (6, 6, 0.0)),          # fixed-shape truncation (the bench setting Dmin = Dmax = chi)
    (3, 5, 2, (4, 4, 0.0)),          # ragged lattice
    (4, 4, 3, (2, 7, 1e-6)),         # walker-dependent kept dimension (Dmin < Dmax, trunc_err > 0)
    (2, 2, 4, (1, 100, 0.0)),        # smallest lattice, no truncation
])
def test_pipeline_parity_hostsim(lib, rows, cols, D, trunc):
    run_pipeline_parity(lib, rows, cols, D, 3, trunc, nsweeps=2)


def test_pipeline_parity_signed_tps(lib):
    run_pipeline_parity(lib, 4, 4, 3, 2, (9, 9, 0.0), nsweeps=2, signed=True, seed=5)


@pytest.mark.parametrize("rows,cols,D,trunc", [(4, 4, 3, (6, 6, 0.0)), (3, 5, 2, (4, 4, 0.0))])
def test_j1j2_pipeline_parity_hostsim(lib, rows, cols, D, trunc):
    """J1-J2 model (BASELINE config #3): BTen2 growth + NNN traces in the energy pass."""
    run_pipeline_parity(lib, rows, cols, D, 3, trunc, nsweeps=2, j2=0.5)


def test_pinning00_pipeline_parity_hostsim(lib):
    """SquareSpinOneHalfXXZModelOBC with a pinning field on site (0, 0): E_loc includes -h00 Sz(0,0)."""
    run_pipeline_parity(lib, 4, 4, 3, 3, (6, 6, 0.0), nsweeps=2, pinning00=0.37)


@pytest.mark.parametrize("rows,cols,D,trunc", [(4, 4, 2, (2, 4, 1e-14)), (3, 4, 3, (5, 5, 0.0))])
def test_tfim_full_space_pipeline_parity_hostsim(lib, rows, cols, D, trunc):
    """BASELINE config #1 path: transverse-field Ising solver (ReplaceOneSiteTrace per site) + full-space NN updater
    with the Suwa-Todo choice (long double prefix sums, one long double draw per bond)."""
    run_pipeline_parity(lib, rows, cols, D, 3, trunc, nsweeps=2, tfim_h=0.5)


@pytest.mark.parametrize("rows,cols,D,trunc", [(4, 4, 3, (6, 6, 0.0)), (3, 5, 2, (2, 4, 1e-10))])
def test_three_site_updater_pipeline_parity_hostsim(lib, rows, cols, D, trunc):
    """MCUpdateSquareTNN3SiteExchange (square_3site_updater.h:23-160): chains bit-identical to the oracle's, amplitudes
    (refreshed by the three-site trace at every row / column start), energies and holes to 1e-10."""
    run_pipeline_parity(lib, rows, cols, D, 3, trunc, nsweeps=2, three_site=True)


def test_tfim_golden_2x2_energy_through_abi(lib):
    """K4 (TFIM) through the C ABI: exact summation over all 16 configurations of the 2x2 simple-update fixture."""
    from peps_b200.api import TransverseFieldIsingSquareOBC
    tps, z = load_golden_tps("tfim2x2_double_su")
    cfgs = np.array([[int(b) for b in format(k, "04b")] for k in range(16)]).reshape(16, 2, 2)
    b = WalkerBatch(2, 2, 2, tps[0][0][0].shape[2], 16, BMPSTruncateParams.SVD(1, 8, 1e-16), lib=lib)
    b.set_tps(SplitIndexTPS(tps))
    b.set_configs(cfgs)
    b.set_model(TransverseFieldIsingSquareOBC(1.0))
    b.init_walkers()
    e = b.energy_and_holes(True)
    wt = b.amplitudes() ** 2
    assert abs(np.sum(wt * e) / np.sum(wt) - float(z["exp_energy"])) < 1e-10


def test_bmps_memo_is_exact_and_saves_one_stack_per_sample(lib, monkeypatch):
    """The LEFT stack finished by the sweep's vertical pass is handed back to the energy solver's vertical pass, and
    the DOWN stack consumed by the energy solver's horizontal pass to the next sweep, instead of being re-absorbed
    (engine.h: Memo). Same chains, energies and holes bit for bit; (cols-1) + (rows-1) fewer absorptions per sample."""
    rows, cols, D, W = 4, 5, 3, 3
    tps = vmc.random_tps(rows, cols, 2, D, seed=11)
    cfgs = np.stack([vmc.shuffled_half_filled_config(rows, cols, 50 + w) for w in range(W)])
    out = {}
    for memo in ("1", "0"):
        monkeypatch.setenv("PEPS_BMPS_MEMO", memo)
        b = WalkerBatch(rows, cols, 2, D, W, BMPSTruncateParams.SVD(5, 5, 0.0), lib=lib)
        b.set_tps(SplitIndexTPS(tps))
        b.set_configs(cfgs)
        b.seed_rng(np.arange(W, dtype=np.uint32) + 3)
        b.init_walkers()
        rec = []
        a0 = b.stat(0)
        for _ in range(3):
            b.sweep(1)
            e = b.energy_and_holes(True)
            rec.append((b.get_configs().copy(), e.copy(), b.holes().copy(), b.amplitudes().copy()))
        out[memo] = (rec, b.stat(0) - a0, b.stat(11))
    for (c1, e1, h1, a1), (c0, e0, h0, a0) in zip(out["1"][0], out["0"][0]):
        assert np.array_equal(c1, c0) and np.array_equal(e1, e0) and np.array_equal(h1, h0) and np.array_equal(a1, a0)
    total = 3 * (4 * (rows - 1) + 4 * (cols - 1)) - (rows - 1)     # the first sweep starts on init_walkers' DOWN stack
    assert out["0"][1] == total and out["0"][2] == 0
    hits = 3 * (cols - 1) + 2 * (rows - 1)
    assert out["1"][2] == hits and out["1"][1] == total - hits


def test_gradient_accumulation_parity_hostsim(lib):
    run_gradient_parity(lib, 3, 4, 2, 3, (4, 4, 0.0), nsamples=4)


def test_golden_2x2_energy_through_abi(lib):
    """K4 through the C ABI: exact summation over the six Sz=0 configurations of the 2x2 simple-update fixture."""
    tps, z = load_golden_tps("heis2x2_double_su")
    import itertools
    cfgs = np.array([np.array(b).reshape(2, 2) for b in itertools.product([0, 1], repeat=4) if sum(b) == 2])
    b = WalkerBatch(2, 2, 2, 4, len(cfgs), BMPSTruncateParams.SVD(1, 100, 0.0), lib=lib)
    b.set_tps(SplitIndexTPS(tps))
    b.set_configs(cfgs)
    b.init_walkers()
    amp = b.amplitudes()
    e = b.energy_and_holes(True)
    energy = float(np.sum(amp ** 2 * e) / np.sum(amp ** 2))
    assert abs(energy - float(z["exp_energy"])) < 1e-10
    # gradient through the accumulators equals the oracle's exact-summation gradient
    holes = b.holes()
    e_ref, g_ref = exact_summation(tps, vmc.XXZModel())
    wsum = np.sum(amp ** 2)
    s_o = np.zeros(b.tps_size)
    s_eo = np.zeros(b.tps_size)
    site_size = 16
    for w in range(len(cfgs)):
        for s in range(4):
            slot = s * 2 * site_size + int(cfgs[w].ravel()[s]) * site_size
            inc = amp[w] * holes[w, s * site_size:(s + 1) * site_size]
            s_o[slot:slot + site_size] += inc
            s_eo[slot:slot + site_size] += e[w] * inc
    grad = (s_eo - energy * s_o) / wsum
    assert np.max(np.abs(grad - SplitIndexTPS(g_ref).pack())) < 1e-12


def test_evaluator_mirror_runs(lib):
    tps = SplitIndexTPS(vmc.random_tps(3, 3, 2, 2, seed=4))
    mc = MonteCarloParams(num_samples=12, num_warmup_sweeps=2, sweeps_between_samples=1,
                          initial_config=Configuration(vmc.neel_config(3, 3)))
    ev = MCEnergyGradEvaluator(mc, BMPSTruncateParams.SVD(4, 4, 0.0), tps, SquareSpinOneHalfXXZModelOBC(1, 1, 0),
                               MCUpdateSquareNNExchange(7), walkers=4, lib=lib)
    ev.WarmUp()
    assert np.isclose(np.max(np.abs(ev.batch.amplitudes())), 1.0, rtol=0.3)
    res = ev.Evaluate()
    assert res.energy_samples.shape == (4, 3)
    assert np.isfinite(res.energy) and np.isfinite(res.gradient_norm)
    assert res.gradient.pack().shape == tps.pack().shape


def test_evaluator_mirror_tfim_full_space(lib):
    """examples/transverse_field_ising_vmc_optimize.cpp-style evaluator: TFIM h = 0.5, full-space updater."""
    from peps_b200.api import TransverseFieldIsingSquareOBC, MCUpdateSquareNNFullSpaceUpdate
    tps = SplitIndexTPS(vmc.random_tps(3, 3, 2, 2, seed=9))
    mc = MonteCarloParams(num_samples=12, num_warmup_sweeps=2, sweeps_between_samples=2,
                          initial_config=Configuration(vmc.neel_config(3, 3)))
    ev = MCEnergyGradEvaluator(mc, BMPSTruncateParams.SVD(2, 4, 1e-14), tps, TransverseFieldIsingSquareOBC(0.5),
                               MCUpdateSquareNNFullSpaceUpdate(3), walkers=4, lib=lib)
    res = ev.Evaluate()
    assert res.energy_samples.shape == (4, 3)
    assert np.isfinite(res.energy) and np.isfinite(res.gradient_norm)
    assert not np.all(ev.batch.get_configs().sum(axis=(1, 2)) == 4)      # Sz is not conserved by this updater


@pytest.mark.parametrize("j2", [0.0, 0.5])
def test_measure_bond_energies_parity_hostsim(lib, j2):
    """EvaluateObservables (base/square_nnn_model_measurement_solver.h:33-214): every bond energy against the oracle."""
    from peps_b200.api import SquareSpinOneHalfJ1J2XXZModelOBC
    rows, cols, D, W = 3, 4, 2, 3
    tps = vmc.random_tps(rows, cols, 2, D, seed=31)
    cfgs = np.stack([vmc.shuffled_half_filled_config(rows, cols, 70 + w) for w in range(W)])
    b = WalkerBatch(rows, cols, 2, D, W, BMPSTruncateParams.SVD(4, 4, 0.0), lib=lib)
    b.set_tps(SplitIndexTPS(tps))
    b.set_configs(cfgs)
    b.set_model(SquareSpinOneHalfJ1J2XXZModelOBC(1.0, 0.8, j2, 0.7 * j2, 0.3))
    b.init_walkers()
    obs = b.measure()
    model = vmc.XXZModel(1.0, 0.8, 0.3, j2, 0.7 * j2)
    for w in range(W):
        ref = model.measure(tps, vmc.Walker(tps, cfgs[w], (4, 4, 0.0)))
        for k, v in ref.items():
            assert np.allclose(obs[k][w], v, rtol=1e-10, atol=1e-12), (k, w)
    e = b.energy_and_holes(False)
    assert np.allclose(e, obs["energy"], rtol=1e-12)          # the recording pass leaves the energy path untouched


def test_measurer_mirror_on_golden_4x4(lib):
    """MCPEPSMeasurer on the reference's 4x4 D=8 Heisenberg fixture (slow_tests/test_boson_mc_peps_measure.cpp:31-76):
    energy near e0 = -9.18912 and nearest-neighbour bond energies near the ED <S_i.S_j> of the reference's
    ed_reference table (corner bond -0.4618, tests/test_data/ed_reference/square_heisenberg_4x4_obc_ed.json)."""
    from peps_b200.api import MCPEPSMeasurer
    tps, z = load_golden_tps("heis4x4_D8_double")
    mc = MonteCarloParams(num_samples=48, num_warmup_sweeps=3, sweeps_between_samples=1,
                          initial_config=Configuration(z["configs"][0]))
    m = MCPEPSMeasurer(mc, BMPSTruncateParams.SVD(8, 8, 0.0), SplitIndexTPS(tps), SquareSpinOneHalfXXZModelOBC(1, 1, 0),
                       MCUpdateSquareNNExchange(11), walkers=8, lib=lib)
    out = m.Execute()
    e, err = out["energy"]
    assert abs(e - float(z["exp_e0_state"])) < max(5 * err, 0.4)
    eh = out["bond_energy_h"][0]
    assert eh.shape == (4, 3) and abs(eh[0, 0] - (-0.4618)) < 0.25
    assert abs(eh.sum() + out["bond_energy_v"][0].sum() - e) < 1e-9
    assert np.allclose(out["spin_z"][0].sum(), 0.0)
    assert "bond_energy_dr" not in out


@pytest.mark.parametrize("orient", [0, 1])
def test_three_site_trace_parity_hostsim(lib, orient):
    """ReplaceTNNSiteTrace (trace.h:326-420) against the oracle and against amplitudes from scratch."""
    rows, cols, D, W = 4, 5, 2, 3
    tps = vmc.random_tps(rows, cols, 2, D, seed=8)
    cfgs = np.stack([vmc.shuffled_half_filled_config(rows, cols, 20 + w) for w in range(W)])
    b = WalkerBatch(rows, cols, 2, D, W, BMPSTruncateParams.SVD(1, 64, 0.0), lib=lib)
    b.set_tps(SplitIndexTPS(tps))
    b.set_configs(cfgs)
    b.init_walkers()
    r0, c0 = (2, 1) if orient == 0 else (1, 3)
    sites = [(r0, c0 + k) if orient == 0 else (r0 + k, c0) for k in range(3)]
    new = np.array([[1, 0, 1], [0, 0, 1], [1, 1, 0]], dtype=np.int32)
    psi = b.probe_tnn_trace(r0, c0, orient, new)
    for w in range(W):
        cf = cfgs[w].copy()
        for k, st in enumerate(sites):
            cf[st] = new[w, k]
        ref = vmc.Walker(tps, cf, (1, 64, 0.0)).amplitude
        assert abs(psi[w] / ref - 1) < 1e-10


def test_error_paths(lib):
    with pytest.raises(PepsError):
        WalkerBatch(1, 4, 2, 2, 1, BMPSTruncateParams.SVD(2, 2, 0.0), lib=lib)     # lattice too small
    b = WalkerBatch(2, 2, 2, 2, 1, BMPSTruncateParams.SVD(2, 2, 0.0), lib=lib)
    with pytest.raises(PepsError):
        b.set_tps(np.zeros(3))
    with pytest.raises(PepsError):
        b.set_truncation(BMPSTruncateParams.SVD(3, 2, 0.0))


def test_rng_state_roundtrip_matches_std_mt19937(lib):
    from oracle.mt19937 import MT19937
    b = WalkerBatch(2, 2, 2, 2, 2, BMPSTruncateParams.SVD(2, 2, 0.0), lib=lib)
    b.seed_rng([42, 43])
    mt, idx = b.get_rng_state()
    for w, seed in enumerate((42, 43)):
        ref, ridx = MT19937(seed).state()
        assert list(mt[w]) == ref and idx[w] == ridx
    b.set_rng_state(mt, idx)
    mt2, idx2 = b.get_rng_state()
    assert np.array_equal(mt, mt2) and np.array_equal(idx, idx2)


@pytest.mark.parametrize("rb", ["32", "64", "512"])
def test_caqr_host_logic_with_diagonal_crossing_row_blocks(rb):
    """linalg.h:caqr with row blocks shorter than the matrix is wide (the diagonal walks through several blocks; blocks
    above it are finished and skipped): R^T R = A^T A and the LAPACK diagonal, through the host simulation.
    Run in a subprocess because the block height is read once per process (PEPS_QR_RB)."""
    import subprocess, sys, textwrap
    code = textwrap.dedent("""
        import sys, ctypes as C, numpy as np
        sys.path.insert(0, %r); sys.path.insert(0, %r)
        import hostsim_lib
        lib = hostsim_lib.load()
        dp = lambda x: x.ctypes.data_as(C.POINTER(C.c_double))
        rng = np.random.default_rng(5)
        for (m, n) in [(200, 96), (96, 96), (70, 130), (300, 40)]:
            W = 2
            a = rng.standard_normal((W, m, n)); kk = min(m, n); r = np.empty((W, kk, n))
            assert lib.peps_test_qr_r(0, W, m, n, dp(a), dp(r)) == 0
            for w in range(W):
                assert np.max(np.abs(np.tril(r[w][:, :kk], -1))) == 0.0
                ref = a[w].T @ a[w]
                assert np.max(np.abs(r[w].T @ r[w] - ref)) < 1e-12 * np.max(np.abs(ref)), (m, n)
                rr = np.linalg.qr(a[w], mode="r")
                assert np.max(np.abs(np.abs(np.diag(r[w])) - np.abs(np.diag(rr)))) < 1e-11 * np.max(np.abs(rr))
        print("ok")
    """) % (hostsim_lib.ROOT, hostsim_lib.ROOT + "/tests")
    import os
    env = dict(os.environ, PEPS_QR_RB=rb)
    out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


def test_chain_deflation_keeps_amplitudes(lib):
    """Rank-revealing step of the forward R chain (engine.cpp: absorb): dropping the rows of the column-sorted R factor
    below 1e-14 of the largest one shrinks the chain and leaves amplitudes, energies and holes unchanged to 1e-10."""
    rows, cols, D, W = 4, 6, 3, 2
    tps = vmc.random_tps(rows, cols, 2, D, seed=17)
    cfgs = np.stack([vmc.shuffled_half_filled_config(rows, cols, 90 + w) for w in range(W)])
    out = {}
    for eps in (0.0, 1e-14, 1e-4):
        b = WalkerBatch(rows, cols, 2, D, W, BMPSTruncateParams.SVD(9, 9, 0.0), lib=lib)
        b.set_chain_deflation(eps)
        b.set_tps(SplitIndexTPS(tps))
        b.set_configs(cfgs)
        b.init_walkers()
        e = b.energy_and_holes(True)
        out[eps] = (b.amplitudes().copy(), e.copy(), b.holes().copy(), b.stat(12), b.stat(13))
    a0, e0, h0, in0, kept0 = out[0.0]
    a1, e1, h1, in1, kept1 = out[1e-14]
    assert in0 == 0 and in1 > 0 and kept1 <= in1
    a2, _, _, in2, kept2 = out[1e-4]
    assert kept2 < in2 and np.max(np.abs(a2 / a0 - 1)) < 1e-2     # a coarse threshold really shortens the chain
    assert np.max(np.abs(a1 / a0 - 1)) < 1e-10
    assert np.max(np.abs(e1 - e0) / np.maximum(1, np.abs(e0))) < 1e-10
    assert np.max(np.abs(h1 - h0)) < 1e-10 * np.max(np.abs(h0))
    for w in range(W):
        ref = vmc.Walker(tps, cfgs[w], (9, 9, 0.0)).amplitude
        assert abs(a1[w] / ref - 1) < 1e-10


def test_plaquette_traces_hostsim():
    """ReplaceNNNSiteTrace (both MPS orientations) and ReplaceSqrt5DistTwoSiteTrace through the C ABI (host-simulated
    device ops) against amplitudes of the exchanged configurations evaluated from scratch by the oracle."""
    from parity_common import run_plaquette_trace_parity
    run_plaquette_trace_parity(hostsim_lib.load())


def test_configuration_rescue_and_psi_consistency_hostsim():
    """EnsureConfigurationValidity (monte_carlo_engine.h:340-414) with walkers as ranks: a TPS whose spin-1 slice at
    site (0,0) is zero makes every configuration with that spin up illegal (amplitude exactly 0); such walkers take the
    first valid walker's configuration. Psi-consistency summaries (psi_consistency.h:76-130) stay below the threshold
    for an exact contraction and fire for a strongly truncated one."""
    from peps_b200.api import (MCEnergyGradEvaluator, MonteCarloParams, SquareSpinOneHalfXXZModelOBC, MCUpdateSquareNNExchange,
                               ConfigurationRescueParams, PsiConsistencyWarningParams, PepsError, BMPSTruncateParams, SplitIndexTPS,
                               compute_psi_consistency_summary_aligned, check_wavefunction_amplitude_validity)
    lib = hostsim_lib.load()
    tl = vmc.random_tps(3, 3, 2, 2, seed=4)
    tl[0][0][1] = np.zeros_like(tl[0][0][1])
    tps = SplitIndexTPS(tl)
    good = np.array([[0, 1, 0], [1, 0, 1], [0, 1, 1]])       # spin 0 at (0,0): legal
    bad = np.array([[1, 0, 1], [0, 1, 0], [1, 0, 0]])        # spin 1 at (0,0): amplitude 0
    cfgs = np.stack([bad, good, bad, good])
    mc = MonteCarloParams(num_samples=8, num_warmup_sweeps=1, sweeps_between_samples=1, is_warmed_up=True)
    ev = MCEnergyGradEvaluator(mc, BMPSTruncateParams.SVD(4, 4, 0.0), tps, SquareSpinOneHalfXXZModelOBC(1, 1, 0),
                               MCUpdateSquareNNExchange(3), walkers=4, configs=cfgs, lib=lib)
    amp = ev.batch.amplitudes()
    assert amp[0] == 0.0 and amp[2] == 0.0 and amp[1] != 0.0
    assert list(check_wavefunction_amplitude_validity(amp, 2.3e-308, 1.7e308)) == [False, True, False, True]
    assert ev.EnsureConfigurationValidity() == [0, 2]
    c = ev.batch.get_configs()
    assert np.array_equal(c[0], good) and np.array_equal(c[2], good) and not ev.warmed_up
    assert np.all(ev.batch.amplitudes() != 0.0)
    assert ev.EnsureConfigurationValidity() == []
    # disabled rescue / nobody valid -> error like the reference's abort
    ev2 = MCEnergyGradEvaluator(mc, BMPSTruncateParams.SVD(4, 4, 0.0), tps, SquareSpinOneHalfXXZModelOBC(1, 1, 0),
                                MCUpdateSquareNNExchange(3), walkers=2, configs=np.stack([bad, good]), lib=lib,
                                config_rescue=ConfigurationRescueParams(enabled=False))
    with pytest.raises(PepsError):
        ev2.EnsureConfigurationValidity()
    ev3 = MCEnergyGradEvaluator(mc, BMPSTruncateParams.SVD(4, 4, 0.0), tps, SquareSpinOneHalfXXZModelOBC(1, 1, 0),
                                MCUpdateSquareNNExchange(3), walkers=2, configs=np.stack([bad, bad]), lib=lib)
    with pytest.raises(PepsError):
        ev3.EnsureConfigurationValidity()
    # psi consistency: exact contraction -> no warnings; chi = 1 on a D = 3 state -> closures disagree -> warnings
    assert compute_psi_consistency_summary_aligned([1.0, -1.0 - 1e-9, 1.0])[1] < 1e-8
    t2 = SplitIndexTPS(vmc.random_tps(4, 4, 2, 3, seed=9, signed=True))
    cf = np.stack([vmc.shuffled_half_filled_config(4, 4, 40 + w) for w in range(2)])
    for chi, expect in ((200, False), (1, True)):
        e4 = MCEnergyGradEvaluator(MonteCarloParams(4, 0, 1, is_warmed_up=True), BMPSTruncateParams.SVD(1, chi, 0.0), t2,
                                   SquareSpinOneHalfXXZModelOBC(1, 1, 0), MCUpdateSquareNNExchange(3), walkers=2, configs=cf,
                                   lib=lib, psi_consistency=PsiConsistencyWarningParams(threshold=1e-6))
        e4.Evaluate()
        assert (len(e4.psi_warnings) > 0) == expect


def test_table_model_hostsim():
    from parity_common import run_table_model_parity
    run_table_model_parity(hostsim_lib.load())


def test_oracle_table_model_equals_brute_force():
    """The oracle's generic TableModel (reference traversal with matrix elements as data) equals
    E_loc = sum_S' <S|H|S'> psi(S') / psi(S) evaluated term by term from scratch amplitudes (spin-1, d = 3)."""
    from parity_common import spin_one_matrices
    rows, cols, d = 2, 3, 3
    h2, h2n, h1 = spin_one_matrices()
    tps = vmc.random_tps(rows, cols, d, 2, seed=7)
    cfg = np.array([[0, 2, 1], [1, 1, 0]])
    trunc = (1, 1000, 0.0)
    amp = lambda c: vmc.Walker(tps, c, trunc).amplitude
    psi = amp(cfg)
    e, _, _ = vmc.TableModel(d, h2, h2n, h1).energy_and_holes(tps, vmc.Walker(tps, cfg, trunc), False)

    def two(H, s1, s2):
        p = cfg[s1] * d + cfg[s2]
        tot = 0.0
        for q in range(d * d):
            if H[p, q] != 0.0:
                c2 = cfg.copy(); c2[s1], c2[s2] = q // d, q % d
                tot += H[p, q] * amp(c2) / psi
        return tot
    ref = 0.0
    for r in range(rows):
        for c in range(cols):
            p = cfg[r, c]
            for q in range(d):
                if h1[p, q] != 0.0:
                    c2 = cfg.copy(); c2[r, c] = q
                    ref += h1[p, q] * amp(c2) / psi
            if c < cols - 1:
                ref += two(h2, (r, c), (r, c + 1))
            if r < rows - 1:
                ref += two(h2, (r, c), (r + 1, c))
            if r < rows - 1 and c < cols - 1:
                ref += two(h2n, (r, c), (r + 1, c + 1)) + two(h2n, (r + 1, c), (r, c + 1))
    assert abs(e - ref) < 1e-11 * max(1.0, abs(ref))


def test_structure_factor_hostsim_and_brute_force():
    """All-pairs S+S- overlaps: engine (host-simulated device ops) == oracle restatement of MeasureStructureFactor, and
    the oracle == amplitudes of the doubly flipped configurations evaluated from scratch (exact contraction)."""
    from parity_common import run_structure_factor_parity
    run_structure_factor_parity(hostsim_lib.load())
    rows, cols = 3, 3
    tps = vmc.random_tps(rows, cols, 2, 2, seed=3)
    cfg = vmc.shuffled_half_filled_config(rows, cols, 2)
    trunc = (1, 1000, 0.0)
    for (y1, x1, y2, x2, v) in vmc.measure_structure_factor(tps, vmc.Walker(tps, cfg, trunc)):
        if cfg[y1, x1] == 0 and cfg[y2, x2] == 1:
            c2 = cfg.copy(); c2[y1, x1] = 1; c2[y2, x2] = 0
            ref = vmc.Walker(tps, c2, trunc).amplitude
            assert abs(v / ref - 1) < 1e-11
        else:
            assert v == 0.0


@pytest.mark.parametrize("scheme", [1, 2])
def test_variational_compression_hostsim(scheme):
    from parity_common import run_variational_parity
    print(run_variational_parity(hostsim_lib.load(), scheme))


@pytest.mark.parametrize("complex_", [False, True])
def test_tfim_measurement_parity_hostsim(lib, complex_):
    from parity_common import run_tfim_measure_parity
    run_tfim_measure_parity(lib, complex_)
