"""MinSR through the CUDA library: the equivalence checks of test_minsr.py (real, complex, fZ2, D = 3), the error paths, a
size test that exercises the Gram kernel's tiling and split-K, and run-to-run bit identity."""
import numpy as np
import pytest

import minsr_common as mc
from oracle import vmc
from peps_b200 import sr
from peps_b200.api import BMPSTruncateParams, SplitIndexTPS, WalkerBatch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    from peps_b200 import _lib
    l = _lib.load()
    assert l.peps_backend_name() == b"cuda-sm_100a"
    return l


def test_minsr_equals_sr_real_gpu(lib):
    mc.check_minsr(*mc.boson_scenario(lib))


def test_minsr_equals_sr_complex_gpu(lib):
    mc.check_minsr(*mc.boson_scenario(lib, complex_=True))


def test_minsr_equals_sr_fermion_gpu(lib):
    mc.check_minsr(*mc.fermion_scenario(lib))


def test_minsr_equals_sr_odd_site_sizes_gpu(lib):
    """D = 3 (site blocks of 9 / 27 / 81 doubles, zero-padded K chunks); N = 20 * 4 = 80 samples: two Gram tiles per side,
    the second one partial."""
    mc.check_minsr(*mc.boson_scenario(lib, D=3, W=20, n=4, chi=9))


@pytest.mark.parametrize("complex_", [False, True])
def test_minsr_errors_and_store_unchanged_gpu(lib, complex_):
    ev, res, _, _ = mc.boson_scenario(lib, complex_=complex_)
    mc.check_errors(ev, res, lib)


def test_minsr_tmatrix_size_and_bit_identity_gpu(lib):
    """6x6, D = 4, 125 walkers x 9 samples = 1125 stored samples (18 Gram tiles per side, the last partial; several split-K
    slices): the device T equals a float64 numpy Gram of the same samples expanded to the TPS layout, and two MinSR calls
    give bit-identical results."""
    L, D, W, n, chi = 6, 4, 125, 9, 8
    tps_l = vmc.random_tps(L, L, 2, D, seed=5)
    b = WalkerBatch(L, L, 2, D, W, BMPSTruncateParams.SVD(chi, chi, 0.0), lib=lib)
    b.set_tps(SplitIndexTPS(tps_l))
    b.set_configs(np.stack([vmc.shuffled_half_filled_config(L, L, 200 + w) for w in range(W)]))
    b.seed_rng(np.arange(11, 11 + W, dtype=np.uint32))
    b.init_walkers()
    b.normalize_state_order1()
    b.sr_reserve(W * n)
    b.sr_collect(True)
    b.zero_accumulators()
    sizes = [t[0].size for row in tps_l for t in row]
    rows = []
    for _ in range(n):
        b.sample(1)
        h, amp, cfg = b.holes(), b.amplitudes(), b.get_configs().reshape(W, -1)
        assert h.shape[1] == sum(sizes)
        dense = np.zeros((W, b.tps_size))
        ho = to = 0
        for s, sz in enumerate(sizes):
            for w in range(W):
                dense[w, to + cfg[w, s] * sz: to + (cfg[w, s] + 1) * sz] = h[w, ho:ho + sz] / amp[w]
            ho += sz
            to += 2 * sz
        rows.append(dense)
    b.sr_collect(False)
    o = np.concatenate(rows)                     # store order: sample-major, walkers inside
    N = o.shape[0]
    assert b.sr_count() == N == W * n
    oc = o - o.mean(0)
    t_ref = oc @ oc.T / N
    t = sr.minsr_tmatrix(b)
    assert np.max(np.abs(t - t_ref)) < 1e-12 * np.max(np.abs(t_ref)), np.max(np.abs(t - t_ref)) / np.max(np.abs(t_ref))
    g = sr.minsr_gram_diag(b)
    assert np.max(np.abs(g - np.einsum("ij,ij->i", o, o))) < 1e-12 * np.max(g)
    x1, e1 = sr.calculate_natural_gradient_minsr(b, N, 1e-3)
    x2, e2 = sr.calculate_natural_gradient_minsr(b, N, 1e-3)
    assert np.array_equal(x1, x2) and e1 == e2
    assert np.array_equal(t, sr.minsr_tmatrix(b))
    b.close()
