"""The contraction and trace-closure checks of tests/gett_common.py on the test-only host simulation, at small shapes.
They check the references, the test entry points, the host twin and the kernel selection of be_gett (a host function the
host simulation shares with the GPU backend); tests/test_gpu_gett.py runs the full case list against the CUDA kernels."""
import zlib

import numpy as np
import pytest

import hostsim_lib
import gett_common as gc

SMALL, LARGE = gc.KERNEL_SMALL, gc.KERNEL_LARGE
LAYOUT = pytest.mark.parametrize("a_kfast,b_nfast", gc.LAYOUTS, ids=["akf-bnf", "akf-bkf", "amf-bnf", "amf-bkf"])
AB = pytest.mark.parametrize("alpha,beta", gc.ALPHA_BETA, ids=[f"{a:g},{b:g}" for a, b in gc.ALPHA_BETA])


@pytest.fixture(scope="module")
def lib():
    return hostsim_lib.load()


@pytest.fixture
def rng(request):
    return np.random.default_rng(zlib.crc32(request.node.name.encode()))


@AB
@pytest.mark.parametrize("M,N,K,target", [(20, 30, 50, (SMALL, 32, 32)), (50, 20, 9, (SMALL, 64, 16)), (9, 50, 1, (SMALL, 16, 64)),
                                          (40, 40, 5, (SMALL, 64, 64)), (37, 41, 67, (LARGE, 64, 64))])
def test_gett_reference(lib, rng, M, N, K, target, alpha, beta):
    gc.case_reference(lib, rng, 2, M, N, K, True, True, alpha, beta, target)


@pytest.mark.parametrize("W,M,N,K,target", [(3, 200, 130, 8, (LARGE, 64, 64)), (50, 200, 130, 8, (LARGE, 128, 64)),
                                            (49, 200, 130, 8, (LARGE, 64, 64)), (100, 96, 130, 8, (LARGE, 64, 64)),
                                            (3, 33, 33, 8, (LARGE, 64, 64)), (3, 100, 100, 7, (SMALL, 64, 64)),
                                            (3, 32, 100, 8, (SMALL, 16, 64)), (3, 100, 32, 8, (SMALL, 64, 16))])
def test_gett_dispatch(lib, rng, W, M, N, K, target):
    """128-row tiles from 296 CTAs of that size on (M > 96), the small-tile kernel for M or N <= 32 or K < 8."""
    gc.case_reference(lib, rng, W, M, N, K, False, True, 1.0, 0.0, target)


@LAYOUT
def test_gett_reference_layouts(lib, rng, a_kfast, b_nfast):
    gc.case_reference(lib, rng, 3, 37, 41, 19, a_kfast, b_nfast, -1.0, 1.0, (LARGE, 64, 64), pads=(1, 2, 0),
                      ws_pads=(3, 0, 1))


def test_gett_layouts_agree(lib, rng):
    gc.case_layouts(lib, rng, 2, 40, 34, 18, LARGE, 64, 64)


@LAYOUT
def test_gett_copy_paths(lib, rng, a_kfast, b_nfast):
    gc.case_copy_paths(lib, rng, 2, 40, 34, 18, a_kfast, b_nfast, LARGE, 64, 64)


@pytest.mark.parametrize("kind", ["offset", "per_row", "skip", "m_only", "n_only", "weak"])
def test_gett_hints(lib, rng, kind):
    gc.case_hints(lib, rng, 2, 140, 70, 260, False, True, kind, (LARGE, 64, 64), tile_m=64)


@pytest.mark.parametrize("side,scale", [("m", 3), ("n", 2)])
@pytest.mark.parametrize("alpha,beta", [(1.0, 0.0), (-1.0, 1.0)], ids=["1,0", "-1,1"])
def test_gett_zero_tails(lib, rng, side, scale, alpha, beta):
    gc.case_tails(lib, rng, 6, 50, 44, 12, True, True, side, scale, alpha, beta, (LARGE, 64, 64))


@pytest.mark.parametrize("which", ["A", "B"])
@pytest.mark.parametrize("gs_pad", [0, 1], ids=["even", "odd"])
def test_gett_gather(lib, rng, which, gs_pad):
    gc.case_gather(lib, rng, 5, 36, 40, 16, which, gs_pad, target=(LARGE, 64, 64))


def test_gett_deterministic(lib, rng):
    gc.case_determinism(lib, rng, 2, 40, 34, 18, True, False, (LARGE, 64, 64))


@pytest.mark.parametrize("which,post", [("kepb", 0), ("kofb", 0), ("kofb", 1), ("koj", 0)])
def test_gett_chain_contractions(lib, rng, which, post):
    gc.case_headline(lib, rng, which, 6, 2, 4, post, (SMALL, 32, 32))


@pytest.mark.parametrize("W", [1, 37])
@pytest.mark.parametrize("K", [1, 255, 8191, 8192, 12289])
def test_dot(lib, rng, K, W):
    gc.case_dot(lib, rng, W, K, reverse=K in gc.DOT_DIMS, ws=None if K < 8192 else 97)


@pytest.mark.parametrize("K", [255, 8192])
def test_dot_gather(lib, rng, K):
    gc.case_dot(lib, rng, 5, K, gather=True)


def test_dot_regrowth(lib, rng):
    gc.case_dot_regrowth(lib, rng, K=8192)


def test_dot_deterministic(lib, rng):
    gc.case_dot_determinism(lib, rng, 3, 8192)


def test_gett_rejects_out_of_bounds_tables(lib, rng):
    """The entry point checks every address the tables can form before anything runs."""
    call = gc.dense_call(rng, 2, 8, 8, 8)
    with pytest.raises(AssertionError, match="outside the buffer"):
        gc.run(lib, call.but(ak=call.ak + 1000))
