"""MinSR (the minimum-step form of SR, solved in sample space) on the host simulation of the device ops: equivalence with
SR on the dense matrices and the product CG (real, complex, fZ2 fermion states; D = 3 with odd site sizes), the error
paths, the C++ wrapper, and an optimisation run. The same checks run on the GPU in test_gpu_minsr.py."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

import hostsim_lib
import minsr_common as mc
from oracle import vmc
from peps_b200 import sr
from peps_b200.api import (BMPSTruncateParams, SplitIndexTPS, MCEnergyGradEvaluator, MonteCarloParams, Configuration,
                           SquareSpinOneHalfXXZModelOBC, MCUpdateSquareNNExchange)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_minsr_equals_sr_real_hostsim():
    mc.check_minsr(*mc.boson_scenario(hostsim_lib.load()))


def test_minsr_equals_sr_complex_hostsim():
    mc.check_minsr(*mc.boson_scenario(hostsim_lib.load(), complex_=True))


def test_minsr_equals_sr_fermion_hostsim():
    mc.check_minsr(*mc.fermion_scenario(hostsim_lib.load()))


def test_minsr_equals_sr_odd_site_sizes_hostsim():
    """D = 3: corner blocks of 9, edge blocks of 27 doubles; N = 5 * 4 = 20 samples."""
    mc.check_minsr(*mc.boson_scenario(hostsim_lib.load(), D=3, W=5, n=4, chi=9))


@pytest.mark.parametrize("complex_", [False, True])
def test_minsr_errors_and_store_unchanged_hostsim(complex_):
    ev, res, _, _ = mc.boson_scenario(hostsim_lib.load(), complex_=complex_)
    mc.check_errors(ev, res, hostsim_lib.load())


def test_minsr_dense_push_through():
    """minsr_common.minsr_dense: the sample-space solve equals the parameter-space solve (S + shift)^{-1} g (complex samples)."""
    rng = np.random.default_rng(1)
    o = rng.standard_normal((7, 30)) + 1j * rng.standard_normal((7, 30))
    e = rng.standard_normal(7) + 1j * rng.standard_normal(7)
    obar = o.mean(0)
    x, t = mc.minsr_dense(o, obar, e, 1e-2)
    g = ((np.conj(e - e.mean()))[:, None] * (o - obar)).sum(0) / 7
    s = (o - obar).T @ (o - obar).conj() / 7 + 1e-2 * np.eye(30)
    assert np.allclose(x, np.linalg.solve(s, g), rtol=0, atol=1e-12 * np.max(np.abs(x)))
    assert np.allclose(t, t.conj().T) and np.max(np.abs(t.sum(1))) < 1e-12 * np.max(np.abs(t))


def test_cpp_wrapper_minsr_matches_python_mirror():
    libdir, libfile = os.path.join(ROOT, "tests", "hostsim"), "libpeps_hostsim.so"
    lib = hostsim_lib.load()
    tps = SplitIndexTPS(vmc.random_tps(3, 3, 2, 2, seed=4))
    cfg = vmc.neel_config(3, 3)
    W, chi, ns, seed, shift = 3, 4, 12, 21, 1e-3
    with tempfile.TemporaryDirectory() as td:
        exe = os.path.join(td, "cpp_minsr")
        subprocess.check_call(["g++", "-std=c++17", "-O1", os.path.join(ROOT, "tests", "cpp", "test_cpp_minsr.cpp"), "-o", exe,
                               "-L" + libdir, "-l:" + libfile, "-Wl,-rpath," + libdir])
        flat = tps.pack()
        inp = f"3 3 2 2 {W} {chi} {ns} {seed} {shift!r}\n{flat.size}\n" + " ".join(repr(float(x)) for x in flat) + "\n" + \
              " ".join(str(int(c)) for c in cfg.ravel()) + "\n"
        x2, em, count = map(float, subprocess.run([exe], input=inp, capture_output=True, text=True, check=True).stdout.split())
    m = MonteCarloParams(num_samples=ns, num_warmup_sweeps=0, sweeps_between_samples=1, initial_config=Configuration(cfg),
                         is_warmed_up=True)
    ev = MCEnergyGradEvaluator(m, BMPSTruncateParams.SVD(chi, chi, 0.0), tps, SquareSpinOneHalfXXZModelOBC(1, 1, 0),
                               MCUpdateSquareNNExchange(seed), walkers=W, lib=lib)
    res = ev.Evaluate(collect_sr_buffers=True)
    nat, em_py = ev.CalculateNaturalGradientMinSR(res, shift)
    assert int(count) == ev.batch.sr_count() == ns
    assert abs(x2 - nat.NormSquare()) < 1e-12 * nat.NormSquare()
    assert abs(em - em_py) < 1e-12 * max(1.0, abs(em_py))


def test_heisenberg_vmc_optimize_minsr_hostsim():
    """examples/heisenberg_vmc_optimize.py with solver="minsr" on the 2x2 K4 fixture: the same descent as the SR run of
    test_examples.py (-1.9952 towards the exact -2)."""
    import sys
    sys.path.insert(0, os.path.join(ROOT, "examples"))
    import heisenberg_vmc_optimize as ex
    from helpers import load_golden_tps
    lib = hostsim_lib.load()
    tps, z = load_golden_tps("heis2x2_double_su")
    e_start = float(z["exp_energy"])
    energies, state = ex.optimize(SplitIndexTPS(tps), 2, 2, chi=16, walkers=16, samples=1600, iters=6, step=0.3, lib=lib,
                                  log=lambda *_: None, init=Configuration(np.array([[0, 1], [1, 0]])), solver="minsr")
    obs = ex.measure(state, 2, 2, chi=16, walkers=16, samples=3200, lib=lib)
    e_final, err = float(obs["energy"][0]), float(obs["energy"][1])
    assert -2.0 - 4 * err - 1e-9 <= e_final < e_start - 1e-3, (e_start, energies, e_final, err)
