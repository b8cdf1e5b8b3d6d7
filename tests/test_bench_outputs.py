"""bench.py --dump-outputs writes what the timed loop computed in its last step: after --warmup + --steps samples every
walker holds the configuration, acceptance rate and local energy of the oracle chain with the same seeds, and the
accumulators hold the oracle's sum O* and sum E_loc O* over all those samples and walkers."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_bench_dump_outputs_match_the_oracle_chains(tmp_path):
    import bench
    from oracle import vmc
    from parity_common import flat_holes
    workload, W, warmup, steps = "heisenberg_4x4_D4_chi8", 4, 1, 2
    out = tmp_path / "out"
    run = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--walkers", str(W),
                          "--streams", "2", "--warmup", str(warmup), "--steps", str(steps), "--secondary", "0",
                          "--no-cpu-baseline", "--e2e-steps", "0", "--dump-outputs", str(out)],
                         cwd=tmp_path, capture_output=True, text=True, check=True)
    assert json.loads(run.stdout.strip().splitlines()[-1])["steps"] == steps
    d = {n: np.load(out / f"{n}.npy") for n in ("eloc", "accept_rate", "configs", "ostar_sum", "eloc_ostar_sum")}
    assert all(a.dtype == np.float64 for a in d.values())
    L, D, chi = bench.WORKLOADS[workload]
    tps, cfgs, seeds = bench.make_inputs(L, D, W, 0)
    trunc = (chi, chi, 0.0)
    # the benchmark rescales the state by NormalizeStateOrder1 over the initial amplitudes of all its walkers
    tps, _ = vmc.normalize_state_order1(tps, [vmc.Walker(tps, cfgs[w], trunc).amplitude for w in range(W)])
    osum, eosum = np.zeros_like(d["ostar_sum"]), np.zeros_like(d["eloc_ostar_sum"])
    for w in range(W):
        wk = vmc.Walker(tps, cfgs[w], trunc)
        up = vmc.NNExchangeUpdater(int(seeds[w]))
        for _ in range(warmup + steps):
            acc = up.sweep(tps, wk)[0]
            e, holes, _ = vmc.XXZModel().energy_and_holes(tps, wk, True)
            ost = flat_holes(holes, L, L) / wk.amplitude
            off = hoff = 0
            for r in range(L):
                for c in range(L):
                    sz = tps[r][c][0].size
                    s = int(wk.config[r, c])
                    osum[off + s * sz: off + (s + 1) * sz] += ost[hoff:hoff + sz]
                    eosum[off + s * sz: off + (s + 1) * sz] += e * ost[hoff:hoff + sz]
                    off += 2 * sz
                    hoff += sz
        assert np.array_equal(d["configs"][w], wk.config), f"walker {w}"
        assert d["accept_rate"][w] == acc, (w, d["accept_rate"][w], acc)
        assert abs(d["eloc"][w] - e) < 1e-10 * max(1.0, abs(e)), (w, d["eloc"][w], e)
    assert off == osum.size
    for k, ref in (("ostar_sum", osum), ("eloc_ostar_sum", eosum)):
        assert np.max(np.abs(d[k] - ref)) < 1e-9 * np.max(np.abs(ref)), k
