"""The contraction kernels (be_gett) and the trace closure (be_dot) on the GPU against float64 references
(tests/gett_common.py). Every case that targets a kernel variant asserts the variant the backend reports, so a change of
the dispatch cannot move a case off its target quietly. Run on the GPU box with ``-m gpu``.

Large-tile kernel gett_large_kernel<AKF, BKF, WGM>: 128-row tiles (WGM = 4) are chosen when the call has at least 296
CTAs of that size, so the 200 x 130 cases (six 128 x 64 tiles per walker) run 50 walkers for them and 3 for the 64-row
tiles. The ring is three stages deep for <true, *, 4> and four for the others."""
import zlib

import numpy as np
import pytest

import gett_common as gc

pytestmark = pytest.mark.gpu

SMALL, LARGE = gc.KERNEL_SMALL, gc.KERNEL_LARGE
W_TILE = {64: 3, 128: 50}          # walkers of the 200 x 130 cases per tile height
LAYOUT = pytest.mark.parametrize("a_kfast,b_nfast", gc.LAYOUTS, ids=["akf-bnf", "akf-bkf", "amf-bnf", "amf-bkf"])
TILE = pytest.mark.parametrize("tile", [64, 128])
AB = pytest.mark.parametrize("alpha,beta", gc.ALPHA_BETA, ids=[f"{a:g},{b:g}" for a, b in gc.ALPHA_BETA])


@pytest.fixture(scope="module")
def lib():
    from peps_b200 import _lib
    l = _lib.load()
    assert l.peps_backend_name() == b"cuda-sm_100a"
    return l


@pytest.fixture
def rng(request):
    return np.random.default_rng(zlib.crc32(request.node.name.encode()))


@pytest.fixture(scope="module", autouse=True)
def worst_error_report():
    """Prints the largest |C - ref| / bound seen per kernel variant (visible with -s)."""
    yield
    print("\nlargest error / bound per variant (kernel, tile_m, tile_n, akf, bkf, avec, bvec, cvec):")
    for k in sorted(gc.WORST, key=str):
        print(f"  {k}: {gc.WORST[k]:.3g}")


# ---- small-tile kernel gett_kernel<WMT, WNT> ------------------------------------------------------------------------
SMALL_SHAPES = [(20, 30, 50, 32, 32), (32, 32, 200, 32, 32), (100, 20, 50, 64, 16), (20, 100, 50, 16, 64),
                (100, 100, 5, 64, 64), (33, 70, 7, 64, 64), (300, 30, 1, 64, 16)]


@AB
@pytest.mark.parametrize("M,N,K,tm,tn", SMALL_SHAPES)
def test_gpu_small_reference(lib, rng, M, N, K, tm, tn, alpha, beta):
    gc.case_reference(lib, rng, 3, M, N, K, True, True, alpha, beta, (SMALL, tm, tn))


@LAYOUT
@pytest.mark.parametrize("M,N,K,tm,tn", [(20, 30, 50, 32, 32), (100, 20, 50, 64, 16), (20, 100, 50, 16, 64), (100, 100, 5, 64, 64)])
def test_gpu_small_layouts(lib, rng, a_kfast, b_nfast, M, N, K, tm, tn):
    gc.case_reference(lib, rng, 3, M, N, K, a_kfast, b_nfast, -1.0, 1.0, (SMALL, tm, tn), pads=(1, 2, 0), ws_pads=(3, 0, 1))


@pytest.mark.parametrize("kind", ["offset", "per_row", "skip", "m_only", "weak"])
def test_gpu_small_hints(lib, rng, kind):
    gc.case_hints(lib, rng, 3, 150, 20, 300, False, True, kind, (SMALL, 64, 16), tile_m=64)


@pytest.mark.parametrize("side,scale", [("m", 3), ("n", 2)])
def test_gpu_small_tails(lib, rng, side, scale):
    gc.case_tails(lib, rng, 12, 100, 30, 40, True, True, side, scale, -1.0, 1.0, (SMALL, 64, 16))


@pytest.mark.parametrize("which", ["A", "B"])
def test_gpu_small_gather(lib, rng, which):
    gc.case_gather(lib, rng, 9, 20, 100, 24, which, 1, target=(SMALL, 16, 64))


# ---- large-tile kernel gett_large_kernel<AKF, BKF, WGM>: all eight variants ----------------------------------------
@AB
@TILE
@LAYOUT
def test_gpu_large_reference_ragged(lib, rng, a_kfast, b_nfast, tile, alpha, beta):
    """M, N, K odd and no multiple of any tile: 8-byte copies, ragged edges in every direction."""
    gc.case_reference(lib, rng, W_TILE[tile], 201, 131, 67, a_kfast, b_nfast, alpha, beta, (LARGE, tile, 64))


@TILE
def test_gpu_large_layouts_agree(lib, rng, tile):
    gc.case_layouts(lib, rng, W_TILE[tile], 200, 130, 70, LARGE, tile, 64)


@TILE
@LAYOUT
def test_gpu_large_copy_paths(lib, rng, a_kfast, b_nfast, tile):
    gc.case_copy_paths(lib, rng, W_TILE[tile], 200, 130, 70, a_kfast, b_nfast, LARGE, tile, 64)


@TILE
@pytest.mark.parametrize("a_kfast,b_nfast", [(True, False), (False, True)], ids=["akf-bkf", "amf-bnf"])
@pytest.mark.parametrize("K", [8, 32, 48, 64, 1000])
def test_gpu_large_k_steps(lib, rng, K, a_kfast, b_nfast, tile):
    """K = 8 (the smallest K of the large kernel, one K step), fewer K steps than the ring depth (2), equal to the
    three-stage (3) and the four-stage ring (4), and many more (63, the last one ragged)."""
    gc.case_reference(lib, rng, W_TILE[tile], 200, 130, K, a_kfast, b_nfast, -1.0, 1.0, (LARGE, tile, 64))


@TILE
@pytest.mark.parametrize("a_kfast,b_nfast", [(True, False), (False, True)], ids=["akf-bkf", "amf-bnf"])
@pytest.mark.parametrize("kind", ["offset", "per_row", "skip", "m_only", "n_only", "weak"])
def test_gpu_large_hints(lib, rng, kind, a_kfast, b_nfast, tile):
    gc.case_hints(lib, rng, W_TILE[tile], 200, 130, 300, a_kfast, b_nfast, kind, (LARGE, tile, 64), tile_m=tile)


@pytest.mark.parametrize("beta", [0.0, -1.0])
@TILE
def test_gpu_large_hints_skip_beta(lib, rng, tile, beta):
    gc.case_hints(lib, rng, W_TILE[tile], 200, 130, 300, True, True, "skip", (LARGE, tile, 64), alpha=0.5, beta=beta,
                  tile_m=tile)


@pytest.mark.parametrize("alpha,beta", [(1.0, 0.0), (-1.0, 1.0), (0.5, -2.0)], ids=["1,0", "-1,1", "0.5,-2"])
@pytest.mark.parametrize("side,scale", [("m", 3), ("n", 2)])
@TILE
def test_gpu_large_tails(lib, rng, tile, side, scale, alpha, beta):
    gc.case_tails(lib, rng, W_TILE[tile], 200, 130, 40, True, False, side, scale, alpha, beta, (LARGE, tile, 64))


@TILE
@pytest.mark.parametrize("which", ["A", "B"])
@pytest.mark.parametrize("gs_pad", [0, 1], ids=["even", "odd"])
def test_gpu_large_gather(lib, rng, which, gs_pad, tile):
    """gs even: 16-byte copies of the gathered operand; gs odd: 8-byte copies."""
    call, _, var = gc.case_gather(lib, rng, W_TILE[tile], 200, 130, 40, which, gs_pad, b_nfast=True, a_kfast=False,
                                  target=(LARGE, tile, 64), alpha=-1.0, beta=1.0)
    assert var[5 if which == "A" else 6] == (1 - gs_pad)


def test_gpu_large_deterministic(lib, rng):
    gc.case_determinism(lib, rng, 50, 200, 130, 300, True, False, (LARGE, 128, 64))


# ---- the hinted chain contractions of absorb_svd at the benchmark's D = 8, chi = 64, 37 walkers per context ----------
@pytest.mark.parametrize("which,post", [("kepb", 0), ("kofb", 0), ("kofb", 1), ("koj", 0)])
def test_gpu_chain_contractions(lib, rng, which, post):
    var = gc.case_headline(lib, rng, which, 37, 8, 64, post, (LARGE, 128, 64))
    if which == "koj":
        assert var[3:5] == (1, 0)        # gett_large_kernel<true, false, 4>: the three-stage ring


# ---- trace closure -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("W", [1, 37, 129, 300])
@pytest.mark.parametrize("K", [1, 255, 8191, 8192, 12289, 131072, 262144])
def test_gpu_dot(lib, rng, K, W):
    """One slice (K < 8192), two (8192), a ragged last chunk (12289 = 3 x 4097 - 2) and 32 (131072, 262144); W = 129 and
    300 need several blocks of the finishing kernel. Large traces use overlapping walker windows (stride 97)."""
    gc.case_dot(lib, rng, W, K, reverse=K in gc.DOT_DIMS, ws=None if K * W <= 2 ** 22 else 97)


@pytest.mark.parametrize("K", [255, 12289, 262144])
def test_gpu_dot_gather(lib, rng, K):
    gc.case_dot(lib, rng, 37, K, gather=True)


def test_gpu_dot_regrowth(lib, rng):
    gc.case_dot_regrowth(lib, rng)


def test_gpu_dot_deterministic(lib, rng):
    gc.case_dot_determinism(lib, rng, 37, 262144)
