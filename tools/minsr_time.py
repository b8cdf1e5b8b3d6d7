#!/usr/bin/env python
"""MinSR against CG on the device-resident O* store at the headline workload (10x10, D=8, chi=64, 148 walkers, 14 samples
per walker = 2072 stored samples of 278 784 doubles: a 4.6 GB store, far larger than the 126 MB L2, so no flush is needed).

Prints one JSON line: the Gram / Cholesky + solve / total MinSR times (kernel times from a torch.profiler pass of their
own, total call time from a host clock around synchronous calls after warm-up), the Gram kernel's executed and useful
(masked) TF/s against a cuBLAS DGEMM measured in the same run, CG time and iterations to relative tolerances 1e-4, 1e-8 and
1e-12 on the same store, max|x_minsr - x_cg| / max|x|, max G_ii / max T_ii, and the card's name and power limit.
    python tools/minsr_time.py [--walkers 148] [--samples 14] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as exc:                      # noqa: BLE001
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"not read ({exc!r})"}


def dgemm_tflops(torch, n=8192, reps=10):
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    for _ in range(3):
        torch.matmul(a, b)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        torch.matmul(a, b)
    e1.record()
    torch.cuda.synchronize()
    return 2.0 * n ** 3 * reps / (e0.elapsed_time(e1) * 1e-3) / 1e12


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--walkers", type=int, default=148)
    ap.add_argument("--samples", type=int, default=14, help="samples per walker (14 x 148 = 2072)")
    ap.add_argument("--shift", type=float, default=1e-3)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from oracle import vmc
    from peps_b200 import sr
    from peps_b200.api import BMPSTruncateParams, SplitIndexTPS, WalkerBatch
    L, D, chi, W = 10, 8, 64, a.walkers
    tps = vmc.random_tps(L, L, 2, D, seed=20260101)
    b = WalkerBatch(L, L, 2, D, W, BMPSTruncateParams.SVD(chi, chi, 0.0))
    b.set_tps(SplitIndexTPS(tps))
    b.set_configs(np.stack([vmc.shuffled_half_filled_config(L, L, 1000 + w) for w in range(W)]))
    b.seed_rng(np.arange(7, 7 + W, dtype=np.uint32))
    b.init_walkers()
    b.normalize_state_order1()
    b.sr_reserve(W * a.samples)
    b.sr_collect(True)
    b.zero_accumulators()
    cfgs, elocs = [], []
    t0 = time.perf_counter()
    for _ in range(a.samples):                   # real samples: one sweep between them
        e, _ = b.sample(1)
        cfgs.append(b.get_configs().reshape(W, -1))
        elocs.append(e)
    t_sampling = time.perf_counter() - t0
    b.sr_collect(False)
    N = b.sr_count()
    stride = int(b.lib.peps_holes_stride(b.h))
    sizes = np.array([t[0].size for row in tps for t in row])
    cfg = np.concatenate(cfgs)                   # store order
    # flops of the Gram: executed = upper-triangle 64 x 64 tiles over the 16-padded K; useful = pairs agreeing per site
    tiles = -(-N // 64)
    k_pad = int(np.sum(-(-sizes // 16) * 16))
    gram_exec = 2.0 * 64 * 64 * k_pad * tiles * (tiles + 1) / 2
    n1 = cfg.sum(axis=0).astype(float)
    n0 = N - n1
    gram_useful = float(np.sum(2.0 * sizes * (n0 * (n0 + 1) / 2 + n1 * (n1 + 1) / 2)))
    # warm-up, then host-clock timing of the synchronous calls
    x, em = sr.calculate_natural_gradient_minsr(b, N, a.shift)
    T = sr.minsr_tmatrix(b)
    times, ttimes = [], []
    for _ in range(a.reps):
        b.sync()
        t0 = time.perf_counter()
        x2, _ = sr.calculate_natural_gradient_minsr(b, N, a.shift)
        times.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        sr.minsr_tmatrix(b)
        ttimes.append(time.perf_counter() - t0)
    bit_identical = bool(np.array_equal(x, x2))
    # kernel times in a profiler pass of their own
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sr.calculate_natural_gradient_minsr(b, N, a.shift)
        b.sync()
        torch.cuda.synchronize()
    from torch.autograd import DeviceType
    kt = {}
    for evt in prof.events():
        if evt.device_type != DeviceType.CUDA:
            continue
        dt = evt.time_range.elapsed_us()
        for key in ("sr_gram_kernel", "sr_gram_reduce_kernel", "chol_panel_kernel", "chol_update_kernel", "chol_solve_kernel",
                    "minsr_embed_kernel", "minsr_centre_kernel", "sr_accumulate_kernel", "sr_dots_kernel"):
            if key in evt.name:
                kt[key] = kt.get(key, 0.0) + dt / 1e3          # us -> ms
    gram_ms = kt.get("sr_gram_kernel", 0.0) + kt.get("sr_gram_reduce_kernel", 0.0)
    chol_ms = sum(kt.get(k, 0.0) for k in ("minsr_embed_kernel", "chol_panel_kernel", "chol_update_kernel", "chol_solve_kernel"))
    gdiag = sr.minsr_gram_diag(b)
    # CG on the same store and the same right-hand side g_c (plain energy mean)
    osum, eosum = b.accumulators()
    obar = osum / N
    g = eosum / N - em * obar
    cg = {}
    for tol in (1e-4, 1e-8, 1e-12):
        b.sync()
        t0 = time.perf_counter()
        r = sr.calculate_natural_gradient(b, g, obar, N, a.shift, sr.ConjugateGradientParams(max_iter=5000, relative_tolerance=tol))
        cg[f"{tol:g}"] = {"ms": (time.perf_counter() - t0) * 1e3, "iterations": r.iterations, "reason": sr.REASONS[r.reason],
                          "max_abs_diff_vs_minsr_rel": float(np.max(np.abs(x - r.x)) / np.max(np.abs(x)))}
    dg = dgemm_tflops(torch)
    total_ms = float(np.median(times)) * 1e3
    line = {
        "metric": "minsr_ms", "value": total_ms, "unit": "ms", "higher_is_better": False, "dtype": "f64",
        "card": card(),
        "config": {"workload": "heisenberg_10x10_D8_chi64", "walkers": W, "samples_per_walker": a.samples, "stored_samples": N,
                   "ostar_doubles_per_sample": stride, "store_GB": N * stride * 8 / 1e9, "diag_shift": a.shift,
                   "sampling_s": t_sampling, "l2": "store >> 126 MB L2"},
        "minsr_total_ms_median": total_ms, "minsr_total_ms_all": [t * 1e3 for t in times],
        "tmatrix_probe_ms_median": float(np.median(ttimes)) * 1e3,
        "gram_ms": gram_ms, "cholesky_solve_ms": chol_ms, "kernel_ms": kt,
        "gram_tflops_executed": gram_exec / (kt.get("sr_gram_kernel", float("nan")) * 1e-3) / 1e12,
        "gram_tflops_useful": gram_useful / (kt.get("sr_gram_kernel", float("nan")) * 1e-3) / 1e12,
        "gram_flops_executed": gram_exec, "gram_flops_useful": gram_useful,
        "cublas_dgemm_tflops_8192": dg,
        "cg": cg,
        "max_Gii_over_max_Tii": float(np.max(gdiag) / np.max(np.diag(T))),
        "minsr_bit_identical_two_calls": bit_identical,
        "energy_mean_plain": em,
    }
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")
    b.close()


if __name__ == "__main__":
    main()
