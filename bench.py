#!/usr/bin/env python
"""bench.py -- VMC samples/s of the walker-batched sampling hot path (BASELINE.json metric).

One "step" = one VMC sample for every walker on every GPU: `sweeps_between_samples` NN-exchange Metropolis sweeps +
CalEnergyAndHoles<true> + O* accumulation (the loop body of the reference's MCEnergyGradEvaluator::Evaluate,
algorithm/vmc_update/mc_energy_grad_evaluator.h:205-282). Workload: BASELINE.json's headline configuration,
10x10 Heisenberg, D=8, chi=64 (Dmin=Dmax=chi, trunc_err=0), synthetic random positive TPS (SURVEY.md section 8d.1).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--walkers W_per_gpu] [--impl ours|reference] [--dump-outputs DIR]

Prints ONE JSON line on rank 0. `value` is timed with CUDA events on the library's stream with the TPS, the
configurations and the RNG state resident in HBM; `e2e` goes through the public evaluator-style call with host
buffers (TPS upload from pinned memory, walker refresh, sample, download of energies and both accumulators).
The `--impl reference` arm times the oracle port of the reference's CPU algorithm (oracle/) on the host cores.
`--dump-outputs DIR` writes the outputs of the last timed step as .npy files (see dump_outputs), so that two builds can
be compared output for output.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (L, D, chi)
    "heisenberg_10x10_D8_chi64": (10, 8, 64),
    "heisenberg_8x8_D6_chi36": (8, 6, 36),
    "heisenberg_4x4_D4_chi8": (4, 4, 8),
}
TPS_SEED = 20260101
CFG_SEED0 = 1000
RNG_SEED0 = 7

# algorithmic flop model per sample per walker (SURVEY.md section 8d.2 / Appendix A; factorisation counts are
# LAPACK model counts, not executed counts)
MODEL_FLOPS = {"heisenberg_10x10_D8_chi64": dict(gemm=2.96e11, qr=1.18e12, svd=9.80e11, total=2.45e12),
               "heisenberg_8x8_D6_chi36": dict(gemm=1.08e10, qr=2.88e10, svd=3.18e10, total=7.1e10),
               "heisenberg_4x4_D4_chi8": dict(gemm=2.43e6, qr=1.23e6, svd=1.88e6, total=5.5e6)}


SIGNED_TPS = False


def make_inputs(L, D, n_walkers, first_walker):
    from oracle import vmc
    tps = vmc.random_tps(L, L, 2, D, seed=TPS_SEED, signed=SIGNED_TPS)
    cfgs = np.stack([vmc.shuffled_half_filled_config(L, L, CFG_SEED0 + first_walker + w) for w in range(n_walkers)])
    seeds = np.arange(RNG_SEED0 + first_walker, RNG_SEED0 + first_walker + n_walkers, dtype=np.uint32)
    return tps, cfgs, seeds


# ---------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference algorithm on the host cores
# ---------------------------------------------------------------------------------------------------------
# One process == one Markov chain with one BLAS thread (the reference runs one chain per MPI rank with
# hp_numeric::SetTensorManipulationThreads(1)); `cores` processes run side by side.
#   * calibration (once): every process runs ONE REAL FULL SAMPLE of its chain (MC sweep + CalEnergyAndHoles<true>) and
#     times it, then times the bounded slice below -> slice_fraction = t_slice / t_full_sample, both measured.
#   * step: every process re-runs the bounded slice = one bulk boundary-MPS absorption (BMPS::MultiplyMPO of row L/2
#     into the UP boundary that already holds rows 0..L/2-1: full D*chi bond, QR chain + truncating SVD sweep), the
#     unit that carries ~90 % of a sample's flops. The parent times the step by wall clock over all processes.
#   samples/s = cores * slice_fraction / t_step.
CAL_FILE = os.path.join(ROOT, "profiles", "cpu_slice_calibration.json")
_W = {}


def _cpu_init(L, D, chi, counter):
    try:
        from threadpoolctl import threadpool_limits
        _W["limiter"] = threadpool_limits(limits=1)
    except Exception:
        pass
    with counter.get_lock():
        wid = counter.value
        counter.value += 1
    from oracle import vmc
    from oracle.bmps import multiply_mpo, vacuum_bmps, UP
    tps, cfgs, _ = make_inputs(L, D, 1, 100000 + wid)
    tn = vmc.project(tps, cfgs[0])
    mps = vacuum_bmps(L)
    for k in range(L // 2):                        # UP boundary with rows 0 .. L/2-1 absorbed
        mps = multiply_mpo(mps, [tn[k][c] for c in range(L)], UP, chi, chi, 0.0)
    _W.update(L=L, D=D, chi=chi, wid=wid, tps=tps, cfg=cfgs[0], tn=tn, mps=mps)


def _cpu_slice(_):
    from oracle.bmps import multiply_mpo, UP
    L, chi, tn = _W["L"], _W["chi"], _W["tn"]
    t0 = time.perf_counter()
    multiply_mpo(_W["mps"], [tn[L // 2][c] for c in range(L)], UP, chi, chi, 0.0)
    return time.perf_counter() - t0


def _cpu_full_sample(_):
    from oracle import vmc
    chi = _W["chi"]
    wk = vmc.Walker(_W["tps"], _W["cfg"], (chi, chi, 0.0))
    up = vmc.NNExchangeUpdater(RNG_SEED0 + 100000 + _W["wid"])
    t0 = time.perf_counter()
    up.sweep(_W["tps"], wk)
    vmc.XXZModel().energy_and_holes(_W["tps"], wk, True)
    t_full = time.perf_counter() - t0
    return t_full, _cpu_slice(0)


class CpuArm:
    def __init__(self, L, D, chi, cores):
        import multiprocessing as mp
        ctx = mp.get_context("spawn")
        self.cores = cores
        self.pool = ctx.Pool(cores, initializer=_cpu_init, initargs=(L, D, chi, ctx.Value("i", 0)))
        self.pool.map(_cpu_slice, range(cores), chunksize=1)          # also forces every worker through its setup

    def calibrate(self):
        res = self.pool.map(_cpu_full_sample, range(self.cores), chunksize=1)
        t_full = float(np.mean([r[0] for r in res]))
        t_slice = float(np.mean([r[1] for r in res]))
        return dict(t_full_sample_s=t_full, t_slice_s=t_slice, slice_fraction=t_slice / t_full, cores=self.cores)

    def step(self):
        t0 = time.perf_counter()
        self.pool.map(_cpu_slice, range(self.cores), chunksize=1)
        return time.perf_counter() - t0

    def close(self):
        self.pool.terminate()


SLICE_TEXT = ("one bulk boundary-MPS absorption (BMPS::MultiplyMPO of row L/2, full D*chi bond) per process and step; "
              "samples/s = cores * slice_fraction / t_step with slice_fraction = t_slice / t_full_sample, both timed "
              "on this host (one real full sample per process: MC sweep + CalEnergyAndHoles<true>)")


def cpu_baseline_quick(L, D, chi, cores, nsteps=3):
    """cpu_baseline of the main arm: a few slice steps; the slice fraction comes from the calibration the reference arm
    measured on the GPU box (profiles/cpu_slice_calibration.json) or is measured now if that file is missing."""
    arm = CpuArm(L, D, chi, cores)
    try:
        cal = None
        if os.path.exists(CAL_FILE):
            c = json.load(open(CAL_FILE))
            if c.get("workload") == [L, D, chi]:
                cal = c
        src = "profiles/cpu_slice_calibration.json (measured by `bench.py --impl reference` on the B200 box host)"
        if cal is None:
            cal = arm.calibrate()
            src = "measured in this run"
        ts = [arm.step() for _ in range(nsteps)]
    finally:
        arm.close()
    t = float(np.mean(ts))
    return cores * cal["slice_fraction"] / t, dict(t_step_s=t, slice_fraction=cal["slice_fraction"], slice_fraction_source=src,
                                                   t_full_sample_s=cal.get("t_full_sample_s"))


def workload_config(args, world):
    """The `config` object of the JSON line: the same for the product arm and the reference arm (the driver compares them)."""
    L, D, chi = WORKLOADS[args.workload]
    return {"workload": args.workload, "lattice": f"{L}x{L}", "D": D, "chi": chi, "walkers_per_gpu": args.walkers,
            "streams_per_gpu": args.streams, "trunc": "Dmin=Dmax=chi, trunc_err=0",
            "model": "Heisenberg NN (XXZ jz=jxy=1)" if args.j2 == 0.0 else f"J1-J2 Heisenberg (j2={args.j2})",
            "sweeps_between_samples": 1,
            "tps": ("uniform[-1,1)" if args.signed else "uniform[0,1)") + f" seed {TPS_SEED}, NormalizeAllSite + order-1 rescale",
            "l2": "per-step working set (walkers x ~60 MB of BMPS stacks + scratch) exceeds the 126 MB L2",
            "parallelism": f"walkers sharded over {world} GPU(s); NCCL all-reduce of the two accumulators",
            "algorithm": "reference call sequence; exact boundary-MPS memo (6(L-1) absorptions per sample instead of "
                         "8(L-1), bit-identical); R-only QR chain with rows below 1e-13 of the largest dropped; "
                         "column-sorted preconditioning QR, second (LQ) preconditioning with kept reflectors and a single-CTA "
                         "one-sided Jacobi on the small square factor (block Jacobi on the rows when more than 128 "
                         "rows survive the deflation) (DESIGN.md section 2); the CPU arm runs the reference's own algorithm "
                         "(full SVD-compression absorptions) on the same workload"}


def run_reference_arm(args, rank):
    if rank != 0:
        return
    L, D, chi = WORKLOADS[args.workload]
    cores = os.cpu_count() or 1
    arm = CpuArm(L, D, chi, cores)
    try:
        cal = arm.calibrate()
        for _ in range(args.warmup):
            arm.step()
        ts = [arm.step() for _ in range(args.steps)]
    finally:
        arm.close()
    t = float(np.mean(ts))
    value = cores * cal["slice_fraction"] / t
    line = {"impl": "reference", "metric": "vmc_samples_per_s", "value": value, "unit": "samples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, args.gpus),
            "cpu_baseline": {"value": value, "unit": "samples/s", "cores": cores, "kind": "port", "sample": SLICE_TEXT,
                             "detail": dict(cal, workload=[L, D, chi], t_step_s=t,
                                            whole_sample_check_samples_per_s=cores / cal["t_full_sample_s"])},
            "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------
# clocks sampler
# ---------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.lines, self.proc, self.device = [], None, device

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except ValueError:
                continue
            for nm, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measure_fp64_peak(torch, n=4096, reps=6):
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    (a @ b); torch.cuda.synchronize()
    best = 0.0
    for _ in range(reps):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(); (a @ b); e.record(); torch.cuda.synchronize()
        best = max(best, 2 * n ** 3 / (s.elapsed_time(e) * 1e-3) / 1e12)
    del a, b
    return best


class LaneSet:
    """S host threads, each owning one context (= one CUDA stream) with W/S walkers of the same state: kernels of
    different contexts overlap on the GPU (the per-lane host round trips -- one per chain / truncation step -- are hidden
    behind the other lanes' kernels)."""

    def __init__(self, L, D, chi, W, S, device, tps, cfgs, seeds, j2=0.0, rank=0, world=1, dist=None, torch=None, model=None,
                 complex_=False):
        import queue
        from peps_b200.api import BMPSTruncateParams, SplitIndexTPS, FermionSplitIndexTPS, WalkerBatch
        S = max(1, min(S, W))
        while W % S:
            S -= 1
        self.L, self.D, self.chi, self.W, self.S, self.Ws = L, D, chi, W, S, W // S
        self.sit = tps if isinstance(tps, SplitIndexTPS) else SplitIndexTPS(tps)
        self.torch, self.dist, self.world = torch, dist, world
        outer = self

        class Lane(threading.Thread):
            def __init__(self, i):
                super().__init__(daemon=True)
                self.i, self.q, self.r, self.b = i, queue.Queue(), queue.Queue(), None
                self.start()

            def run(self):
                while True:
                    fn = self.q.get()
                    if fn is None:
                        return
                    try:
                        self.r.put(("ok", fn(self)))
                    except Exception as exc:      # surface worker failures on the main thread
                        self.r.put(("err", exc))

        self.lanes = [Lane(i) for i in range(S)]

        def setup(ln):
            sl = slice(ln.i * outer.Ws, (ln.i + 1) * outer.Ws)
            ln.b = WalkerBatch(L, L, 2, D, outer.Ws, BMPSTruncateParams.SVD(chi, chi, 0.0), device=device)
            if complex_:
                ln.b.set_complex()                    # QLTEN_Complex states: split planes (DESIGN.md section 11)
            if isinstance(outer.sit, FermionSplitIndexTPS):
                ln.b.set_fermion(outer.sit)           # fZ2-graded tensors (BASELINE config #4)
            ln.b.set_tps(outer.sit)
            if model is not None:
                ln.b.set_model(model)
            if j2 != 0.0:
                from peps_b200.api import SquareSpinOneHalfJ1J2XXZModelOBC
                ln.b.set_model(SquareSpinOneHalfJ1J2XXZModelOBC(1.0, 1.0, j2, j2, 0.0))
            ln.b.set_configs(cfgs[sl])
            ln.b.seed_rng(seeds[sl])
            ln.b.init_walkers()
            return float(np.max(np.abs(ln.b.amplitudes_c() if complex_ else ln.b.amplitudes())))

        mx = max(self.on_all(setup))
        if world > 1:
            t = torch.tensor([mx], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            mx = float(t.item())
        self.on_all(lambda ln: ln.b.normalize_state_order1(mx))     # MonteCarloEngine::NormalizeStateOrder1
        self.on_all(lambda ln: ln.b.zero_accumulators())

    def on_all(self, fn):
        for ln in self.lanes:
            ln.q.put(fn)
        out = []
        for ln in self.lanes:
            st, v = ln.r.get()
            if st == "err":
                raise v
            out.append(v)
        return out

    def barrier(self):
        self.on_all(lambda ln: ln.b.sync())
        if self.torch is not None:
            self.torch.cuda.synchronize()
            if self.world > 1:
                self.dist.barrier()

    def samples(self, n):
        """n samples on every lane; returns the last sample's (local energies, acceptance rates) of every walker."""
        def run(ln):
            last = None
            for _ in range(n):
                last = ln.b.sample(1)
            ln.b.sync()
            return last
        res = self.on_all(run)
        return np.concatenate([r[0] for r in res]), np.concatenate([r[1] for r in res])

    def timed_samples(self, n):
        """n samples on every lane between two CUDA events recorded with the device idle; returns (ms, energies)."""
        torch = self.torch
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        ev0.record()
        e, _ = self.samples(n)
        torch.cuda.synchronize()
        ev1.record()
        self.barrier()
        return ev0.elapsed_time(ev1), e

    def stat_sum(self, which):
        return sum(self.on_all(lambda ln: ln.b.stat(which)))

    def close(self):
        def fin(ln):
            ln.b.close()
        self.on_all(fin)
        for ln in self.lanes:
            ln.q.put(None)


def secondary_lines(torch, device, D_chi, walkers, streams):
    """Non-favourable companions of the headline (VERDICT r1 item 6): the J1-J2 model of BASELINE config #3, the signed
    [-1,1) TPS (flat boundary spectra: nothing deflates, the Jacobi fallback path runs) and a PHYSICAL state (the
    reference's converged 4x4 D=8 Heisenberg fixture at chi = 16 and 64). One warm-up + one timed step each, fewer walkers
    than the headline: indicative samples/s plus the fractions of rows the rank-revealing steps keep."""
    global SIGNED_TPS
    from oracle import vmc
    L, D, chi = D_chi
    out = []

    def run(name, L, D, chi, W, S, tps, j2=0.0, model=None, note=None, complex_=False):
        cfgs = np.stack([vmc.shuffled_half_filled_config(L, L, CFG_SEED0 + w) for w in range(W)])
        seeds = np.arange(RNG_SEED0, RNG_SEED0 + W, dtype=np.uint32)
        try:
            ls = LaneSet(L, D, chi, W, S, device, tps, cfgs, seeds, j2=j2, torch=torch, model=model, complex_=complex_)
        except Exception as exc:                     # noqa: BLE001  (a companion line must not take the others down)
            out.append({"name": name, "error": repr(exc)[:300]})
            return
        try:
            ls.samples(1)
            r0 = [ls.stat_sum(k) for k in (8, 9, 12, 13, 4, 14)]
            ms, e = ls.timed_samples(1)
            r1 = [ls.stat_sum(k) for k in (8, 9, 12, 13, 4, 14)]
            d = [b - a for a, b in zip(r0, r1)]
            out.append({"name": name, "lattice": f"{L}x{L}", "D": D, "chi": chi, "walkers": W, "streams": ls.S,
                        "samples_per_s": W / (ms * 1e-3), "ms_per_step": ms, "mean_eloc": float(np.mean(e)),
                        "truncation_rows_kept_frac": d[1] / max(d[0], 1), "chain_rows_kept_frac": d[3] / max(d[2], 1),
                        "small_svd_path_frac": d[5] / max(d[4], 1), **({"note": note} if note else {})})
        except Exception as exc:                     # noqa: BLE001
            out.append({"name": name, "error": repr(exc)[:300]})
        finally:
            ls.close()

    SIGNED_TPS = False
    tps = vmc.random_tps(L, L, 2, D, seed=TPS_SEED)
    run("j1j2_j2=0.5", L, D, chi, walkers, streams, tps, j2=0.5)
    run("signed_tps", L, D, chi, walkers, streams, vmc.random_tps(L, L, 2, D, seed=TPS_SEED, signed=True),
        note="throughput stress line only: a chi-truncated contraction of a uniform[-1,1) state is ill-conditioned at this size (row "
             "closures of ONE configuration differ by ~10x in the oracle too, CUDA vs oracle share no digits); parity of this code "
             "path is asserted where it is well-posed (8x8 D=6 chi=36 signed: 1e-9, tests/test_gpu_parity.py)")
    # BASELINE config #4: 8x8 spinless fermions, fZ2 tensors with even / odd blocks of D/2, chi = 64 (SURVEY.md 8d.1)
    from peps_b200.api import FermionSplitIndexTPS, TableModel
    run("fermion_spinless_8x8_D8_chi64_fZ2", 8, 8, 64, walkers, streams, FermionSplitIndexTPS.random(8, 8, 8, TPS_SEED),
        model=TableModel.spinless_fermion(1.0, 0.0, 0.0),
        note="BASELINE config #4: fZ2-graded state evaluated as a sign-dressed dense network (DESIGN.md section 9); random "
             "parity-conserving tensors are full rank, so the sector-aware block-Jacobi truncation path runs")
    # complex (QLTEN_Complex) state at BASELINE config #2's size: uniform [0,1) real parts + uniform [-0.5,0.5) imaginary parts
    rng = np.random.default_rng(TPS_SEED)
    ctps = vmc.random_tps(8, 8, 2, 6, seed=TPS_SEED, dtype=np.complex128)
    for row in ctps:
        for site in row:
            for k in range(len(site)):
                site[k] = site[k] + 1j * (rng.random(site[k].shape) - 0.5) * np.max(np.abs(site[k]))
    run("complex_heisenberg_8x8_D6_chi36", 8, 6, 36, walkers, streams, vmc.normalize_all_site(ctps), complex_=True,
        note="QLTEN_Complex state on split planes: four real contraction launches per complex contraction, factorisations on "
             "the real embedding (DESIGN.md section 11)")
    gold = os.path.join(ROOT, "tests", "golden", "heis4x4_D8_double.npz")
    if os.path.exists(gold):
        z = np.load(gold)
        phys = [[[z[f"t_{r}_{c}_{s}"] for s in range(2)] for c in range(4)] for r in range(4)]
        for c in (16, 64):
            run(f"physical_heisenberg_4x4_D8_fixture_chi{c}", 4, 8, c, 296, streams, phys)
    return out


def run_sr_bench(args, torch, device):
    """--sr: the stochastic-reconfiguration matvec on the device-resident O* store (SRSMatrix::operator*,
    optimizer/stochastic_reconfiguration_smatrix.h:45-91), the HBM-bound piece next to the sampling path: every stored O*
    sample is streamed twice per matvec (sr_dots, sr_accumulate). Reports GB/s against the measured HBM bandwidth and the
    device-resident CG (peps_sr_natural_gradient) iterations/s."""
    import ctypes as C
    from oracle import vmc
    from peps_b200.api import BMPSTruncateParams, SplitIndexTPS, WalkerBatch
    from peps_b200 import sr
    L, D, chi = WORKLOADS[args.workload]
    W = 148
    tps, cfgs, seeds = make_inputs(L, D, W, 0)
    b = WalkerBatch(L, L, 2, D, W, BMPSTruncateParams.SVD(chi, chi, 0.0), device=device)
    b.set_tps(SplitIndexTPS(tps)); b.set_configs(cfgs); b.seed_rng(seeds); b.init_walkers()
    b.normalize_state_order1()
    reps = max(1, -(-args.sr_samples // W))
    b.sr_reserve(reps * W)
    b.sr_collect(True)
    b.zero_accumulators()
    b.sample(1)                                   # one real sample of every walker ...
    for _ in range(reps - 1):
        b.accumulate_ostar()                      # ... replicated into the store (the kernels only see bytes)
    b.sr_collect(False)
    ns = b.sr_count()
    stride = int(b.lib.peps_holes_stride(b.h))
    P = b.tps_size
    v = torch.randn(P, dtype=torch.float64, device="cuda")
    out = torch.empty(P, dtype=torch.float64, device="cuda")
    call = lambda: b._ck(b.lib.peps_sr_matvec_device(b.h, C.c_void_p(v.data_ptr()), 0.1, C.c_void_p(out.data_ptr())))
    for _ in range(3):
        call()
    b.sync()
    # L2 flush between timed matvecs is unnecessary: the store (ns * stride * 8 bytes) is far larger than the 126 MB L2
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    b.sync(); torch.cuda.synchronize()
    t0 = time.perf_counter()
    n_it = 20
    for _ in range(n_it):
        call()
    b.sync()
    dt = (time.perf_counter() - t0) / n_it
    bytes_per = 2.0 * ns * stride * 8 + 2.0 * P * 8 + ns * L * L * 4 * 2
    peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
    peak = float(peaks.get("hbm_gbs", 6548.8))
    # device-resident CG on the same store
    osum, _ = b.accumulators()
    g = np.random.default_rng(0).standard_normal(P)
    t1 = time.perf_counter()
    res = sr.calculate_natural_gradient(b, g, osum / ns, ns, 1e-3, sr.ConjugateGradientParams(max_iter=30, relative_tolerance=1e-14))
    cg_dt = time.perf_counter() - t1
    line = {"metric": "sr_matvec_GBps", "value": bytes_per / dt / 1e9, "unit": "GB/s", "n_gpus": 1, "higher_is_better": True,
            "dtype": "f64", "data": "synthetic", "config": {"workload": args.workload, "stored_samples": ns, "ostar_doubles_per_sample": stride,
                                                              "store_GB": ns * stride * 8 / 1e9, "l2": "store >> 126 MB L2"},
            "ms_per_matvec": dt * 1e3,
            "roofline": {"bound": "hbm", "achieved": bytes_per / dt / 1e9, "peak": peak, "unit": "GB/s", "frac": bytes_per / dt / 1e9 / peak,
                         "bytes_per_matvec": bytes_per, "peak_source": "MEASURED_PEAKS.json hbm_gbs"},
            "cg": {"iterations": res.iterations, "seconds": cg_dt, "iterations_per_s": res.iterations / cg_dt, "reason": sr.REASONS[res.reason],
                   "note": "every CG vector resident in HBM; two matvec-class passes over the store per iteration"}}
    print(json.dumps(line))
    b.close()


def dump_outputs(directory, ls, energies, accept, accumulators=None):
    """--dump-outputs: what a caller of the timed loop holds after its last step, as float64 DIR/<name>.npy (rank 0's
    walkers in lane order): that sample's local energy and acceptance rate per walker, the walkers' configurations, and the
    gradient accumulators sum O* and sum E_loc O* over every sample since they were zeroed (warm-up included), summed over
    the lanes, or the all-reduced ones when several GPUs run. Inputs are seeded, so equal arguments give equal inputs."""
    os.makedirs(directory, exist_ok=True)
    if accumulators is None:
        per_lane = ls.on_all(lambda ln: ln.b.accumulators())
        accumulators = (sum(p[0] for p in per_lane), sum(p[1] for p in per_lane))
    out = {"eloc": energies, "accept_rate": accept, "configs": np.concatenate(ls.on_all(lambda ln: ln.b.get_configs())),
           "ostar_sum": accumulators[0], "eloc_ostar_sum": accumulators[1]}
    for name, a in out.items():
        np.save(os.path.join(directory, name + ".npy"), np.asarray(a, dtype=np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--walkers", type=int, default=148, help="walkers (Markov chains) per GPU")
    ap.add_argument("--j2", type=float, default=0.0, help="next-nearest-neighbour coupling (J1-J2 model, BASELINE config #3); 0 = NN Heisenberg headline")
    ap.add_argument("--workload", default="heisenberg_10x10_D8_chi64", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--signed", action="store_true", help="uniform [-1,1) TPS entries (cancellation stress variant of SURVEY.md 8d.1)")
    ap.add_argument("--e2e-steps", type=int, default=1)
    ap.add_argument("--secondary", type=int, default=1, help="also time the J1-J2 / signed / physical-state companions (N=1 only)")
    ap.add_argument("--secondary-walkers", type=int, default=74)
    ap.add_argument("--sr", action="store_true", help="time the SR matvec / CG on the device-resident O* store instead of the sampling path")
    ap.add_argument("--sr-samples", type=int, default=2048)
    ap.add_argument("--streams", type=int, default=4, help="host threads / CUDA streams sharing the walkers of a GPU")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what their last step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.sr or args.impl == "reference"):
        ap.error("--dump-outputs writes the outputs of the sampling path; it does not apply to --sr or --impl reference")

    global SIGNED_TPS
    SIGNED_TPS = args.signed
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    if args.sr:
        run_sr_bench(args, torch, local_rank)
        return
    from peps_b200.api import SplitIndexTPS
    L, D, chi = WORKLOADS[args.workload]
    W = args.walkers
    tps, cfgs, seeds = make_inputs(L, D, W, rank * W)
    sit = SplitIndexTPS(tps)
    dev = torch.device("cuda", local_rank)
    ls = LaneSet(L, D, chi, W, args.streams, local_rank, sit, cfgs, seeds, j2=args.j2, rank=rank, world=world,
                 dist=dist if world > 1 else None, torch=torch)
    lanes, S, Ws, on_all, barrier = ls.lanes, ls.S, ls.Ws, ls.on_all, ls.barrier

    # accumulators as torch views for the NCCL all-reduce of [sum O*, sum E_loc O*]
    n_par = lanes[0].b.tps_size

    class _Cai:
        def __init__(self, ptr, n):
            self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (ptr, False), "version": 3}

    views = []
    for ln in lanes:
        p_o, p_eo = ln.b.accumulator_device_ptrs()
        views.append((torch.as_tensor(_Cai(p_o, n_par), device=dev), torch.as_tensor(_Cai(p_eo, n_par), device=dev)))

    for _ in range(args.warmup):
        on_all(lambda ln: ln.b.sample(1))
    barrier()
    launches0 = ls.stat_sum(6)
    stats0 = [ls.stat_sum(k) for k in (8, 9, 12, 13, 4, 14)]
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()                                      # device idle on both sides of the timed region
    energies, accept = ls.samples(args.steps)
    if world > 1:                                     # gradient reduction of the iteration (NCCL over NVLink)
        acc_o = torch.stack([v[0] for v in views]).sum(0)
        acc_eo = torch.stack([v[1] for v in views]).sum(0)
        dist.all_reduce(acc_o)
        dist.all_reduce(acc_eo)
    torch.cuda.synchronize()
    ev1.record()
    barrier()
    elapsed_ms = ev0.elapsed_time(ev1)
    clk = clocks.stop() if rank == 0 else None
    launches = ls.stat_sum(6) - launches0
    stats1 = [ls.stat_sum(k) for k in (8, 9, 12, 13, 4, 14)]
    dstat = [b_ - a_ for a_, b_ in zip(stats0, stats1)]
    if args.dump_outputs and rank == 0:               # before the profiled step below moves the chains on
        dump_outputs(args.dump_outputs, ls, energies, accept,
                     (acc_o.cpu().numpy(), acc_eo.cpu().numpy()) if world > 1 else None)
    # one more step of the same loop with every launch bracketed by a CUDA-event pair on the launching stream:
    # per-kernel-class device time and useful flops for the roofline (kept out of `value`: the 2 x ~100k event
    # records per step cost about 10 % of a step)

    def profiled(ln):
        ln.b.profile_enable(True)
        ln.b.profile_get(True)
        ln.b.sample(1)
        pr = ln.b.profile_get(True)
        ln.b.profile_enable(False)
        return pr

    prs = []
    for ln in lanes:                                   # one lane at a time: per-launch durations free of overlap
        ln.q.put(profiled)
        st, v = ln.r.get()
        if st == "err":
            raise v
        prs.append(v)
    prof = {k: {f: sum(p[k][f] for p in prs) for f in ("ms", "launches", "flops")} for k in prs[0]}
    if world > 1:
        t = torch.tensor([elapsed_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    total_samples = W * world * args.steps
    value = total_samples / (elapsed_ms * 1e-3)

    # ---- end-to-end through the evaluator-style public call with host buffers
    flat = torch.from_numpy(sit.pack()).pin_memory()
    h2d = flat.numel() * 8 * S
    E2E_SAMPLES = 4                                   # samples per walker and Evaluate call (the reference's examples take tens per rank)
    d2h = (2 * n_par * 8 + 2 * E2E_SAMPLES * Ws * 8) * S

    def e2e_step(ln):
        for _ in range(args.e2e_steps):
            ln.b.set_tps(flat.numpy())                # state fan-out (mc_energy_grad_evaluator.h:161)
            ln.b.init_walkers()                       # RefreshWavefunctionComponent (:164)
            ln.b.zero_accumulators()
            for _s in range(E2E_SAMPLES):
                e, acc = ln.b.sample(1)               # per-walker energies come back to the host every sample
            osum, eosum = ln.b.accumulators()
        return None

    barrier()
    t0 = time.perf_counter()
    on_all(e2e_step)
    barrier()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = W * world * args.e2e_steps * E2E_SAMPLES / e2e_s if args.e2e_steps else 0.0

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel
    # The lanes of the timed loop hold W/S walkers each, so a launch profiled with its lane running ALONE covers a fraction of
    # the SMs (the other lanes fill the rest in the timed loop): those per-lane figures stay in `per_lane`. The kernel's own
    # roofline position is measured on launches of the full batch: the same W walkers in ONE lane (one warm-up sample, then
    # one sample with every launch bracketed by a CUDA-event pair on its stream, the kernel alone on the GPU).
    ls.close()
    lane_prof = prof
    full = LaneSet(L, D, chi, W, 1, local_rank, sit, cfgs, seeds, j2=args.j2, torch=torch)
    full.samples(1)
    full.lanes[0].q.put(profiled)
    st, prof = full.lanes[0].r.get()
    if st == "err":
        raise prof
    full.close()
    dom = max(prof.items(), key=lambda kv: kv[1]["ms"])
    dom_name, dom_p = dom
    fp64_peak = measure_fp64_peak(torch)
    achieved = dom_p["flops"] / max(dom_p["ms"], 1e-9) / 1e9            # TFLOP/s of useful FP64 work in that kernel class
    step_ms = elapsed_ms / args.steps
    mf = MODEL_FLOPS[args.workload]
    lane_dom = lane_prof[dom_name]
    traffic = None       # dram bytes of the benchmarked launches are not measured in-run; ncu captures: profiles/r2_ncu_*.txt
    roofline = {"kernel": dom_name, "bound": "tensor", "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s",
                "frac": achieved / fp64_peak,
                "peak_source": "cuBLAS DGEMM 4096^3 through torch.matmul, measured in this run (MEASURED_PEAKS.json carries no FP64 figure)",
                "traffic": traffic,
                "traffic_note": "not measured in-run; ncu --set full on six consecutive full-batch launches of this kernel inside a real "
                                "148-walker sample (profiles/r2_ncu_final_apply_cols_kernel.txt): 1.1-1.25 ms launches (3256-4884 CTAs) "
                                "read 1.5-1.7 GB and write 1.3-1.5 GB of DRAM -- the trailing matrix streams through once (read ~ "
                                "write, no re-reads) -- with the DMMA pipe 59-63 % active and 31-33 % of the DRAM bandwidth in use",
                "measured_on": f"one extra sample of the same workload with all {W} walkers in one lane (full-batch launches, the kernel alone "
                               "on the GPU), every launch bracketed by a CUDA-event pair on its stream; `per_lane` holds the same "
                               f"measurement on the timed loop's own lanes ({Ws} walkers each, one lane at a time)",
                "launches": dom_p["launches"], "avg_launch_us": 1e3 * dom_p["ms"] / max(dom_p["launches"], 1),
                "share_of_step": dom_p["ms"] / max(sum(v["ms"] for v in prof.values()), 1e-9),
                "per_class_ms": {k: round(v["ms"], 1) for k, v in prof.items()},
                "per_class_tflops": {k: (v["flops"] / max(v["ms"], 1e-9) / 1e9) for k, v in prof.items()},
                "per_class_frac": {k: (v["flops"] / max(v["ms"], 1e-9) / 1e9) / fp64_peak for k, v in prof.items() if v["flops"] > 0},
                "per_lane": {"walkers_per_launch": Ws, "achieved": lane_dom["flops"] / max(lane_dom["ms"], 1e-9) / 1e9,
                             "frac": lane_dom["flops"] / max(lane_dom["ms"], 1e-9) / 1e9 / fp64_peak,
                             "per_class_ms": {k: round(v["ms"], 1) for k, v in lane_prof.items()},
                             "per_class_tflops": {k: (v["flops"] / max(v["ms"], 1e-9) / 1e9) for k, v in lane_prof.items()}},
                "whole_path": {"model_flops_per_sample": mf["total"], "model_tflops": value * mf["total"] / world / 1e12,
                               "frac_of_fp64_peak": value * mf["total"] / world / 1e12 / fp64_peak,
                               "contraction_model_tflops": value * mf["gemm"] / world / 1e12}}

    secondary = None
    if args.secondary and world == 1:
        try:                                         # companions must never take the headline line down with them
            secondary = secondary_lines(torch, local_rank, (L, D, chi), args.secondary_walkers, 2)
        except Exception as exc:                     # noqa: BLE001
            secondary = [{"name": "secondary lines failed", "error": repr(exc)[:300]}]
    cpu = None
    if not args.no_cpu_baseline and world == 1:      # the CPU arm is timed at N=1 only (rank 0, all host cores)
        cores = os.cpu_count() or 1
        v, detail = cpu_baseline_quick(L, D, chi, cores)
        cpu = {"value": v, "unit": "samples/s", "cores": cores, "kind": "port",
               "sample": "oracle port, one chain + one BLAS thread per core: " + SLICE_TEXT, "detail": detail}

    line = {"metric": "vmc_samples_per_s", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, world),
            "rank_revealing": {"chain_rows_kept_frac": dstat[3] / max(dstat[2], 1), "truncation_rows_kept_frac": dstat[1] / max(dstat[0], 1),
                               "small_svd_path_frac": dstat[5] / max(dstat[4], 1),
                               "note": "the positive synthetic TPS has low numerical rank; see `secondary` for J1-J2, the signed state and a physical state"},
            "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": args.e2e_steps, "call": "Evaluate-style call with host buffers: set_tps (pinned) + init_walkers + 4 samples per walker (energies to the host each) + download of both accumulators"},
            "gpu_launches": int(launches), "clocks": clk, "roofline": roofline, "cpu_baseline": cpu, "secondary": secondary,
            "mean_eloc": float(np.mean(energies))}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
