"""The boundary-MPS chain step and truncation step through the CUDA library, against dense float64 references
(tests/factor_steps_common.py), real and complex, at the sizes the boundary MPS reaches in the benchmarked workloads:
the 8x8, D=6, chi=36 sample (Theta of 216 columns, 432 in the real embedding of a complex state) and chi=64 (embeddings
of 1024 columns, truncated by block Jacobi). Run on the GPU box with ``-m gpu``."""
import pytest

import factor_steps_common as fs

pytestmark = pytest.mark.gpu

CX = pytest.mark.parametrize("complex_", [False, True], ids=["real", "complex"])


@pytest.fixture(scope="module")
def lib():
    from peps_b200 import _lib
    l = _lib.load()
    assert l.peps_backend_name() == b"cuda-sm_100a"
    return l


@CX
@pytest.mark.parametrize("m,n", [(18, 18), (37, 5), (5, 37), (1000, 96), (512, 512), (4096, 512)])
def test_gpu_chain_step_full_rank(lib, complex_, m, n):
    fs.chain_full_rank(lib, complex_, m, n)


@CX
@pytest.mark.parametrize("env", [None, ("PEPS_QR_EARLY_STOP", "0"), ("PEPS_QR_STOP_STRIDE", "1")], ids=["default", "nostop", "stride1"])
@pytest.mark.parametrize("m,n,ranks", [(512, 512, (40, 200, 512)), (4096, 512, (40, 200, 512)), (512, 512, (40, 200, 300))])
def test_gpu_chain_step_exact_rank(lib, monkeypatch, complex_, env, m, n, ranks):
    if env:
        monkeypatch.setenv(*env)
    fs.chain_exact_rank(lib, complex_, m, n, ranks)


@CX
@pytest.mark.parametrize("eps", [1e-4, 1e-8])
@pytest.mark.parametrize("m,n", [(37, 5), (1000, 96), (512, 512)])
def test_gpu_chain_step_graded_spectrum(lib, complex_, m, n, eps):
    fs.chain_graded(lib, complex_, m, n, eps)


@pytest.mark.parametrize("eps", [0.0, 1e-13])
@pytest.mark.parametrize("m,n,o,rc", [(128, 64, 8, (16, 5, 10)), (1296, 216, 6, (216, 100, 37))])
def test_gpu_chain_step_row_hint(lib, m, n, o, rc, eps):
    fs.chain_row_hint(lib, m, n, o, list(rc), eps)


@CX
@pytest.mark.parametrize("eps", [0.0, 1e-13])
@pytest.mark.parametrize("m,n", [(40, 24), (1000, 96), (512, 512)])
def test_gpu_chain_step_zero_walker(lib, complex_, m, n, eps):
    fs.chain_zero_walker(lib, complex_, m, n, eps)


@pytest.mark.parametrize("eps", [0.0, 1e-13])
def test_gpu_chain_step_tall_complex(lib, eps):
    """A complex 4608 x 64 matrix: its 9216-row embedding is taller than one two-stage CAQR takes."""
    fs.chain_tall(lib, True, 4608, 64, eps)


@CX
@pytest.mark.parametrize("eps", [0.0, 1e-13])
def test_gpu_chain_step_tall_reduction_forced(lib, monkeypatch, complex_, eps):
    monkeypatch.setenv("PEPS_QR_MAX_ROWS", "64")
    fs.chain_tall(lib, complex_, 600, 96, eps)


@CX
def test_gpu_chain_step_tall_without_reduction(lib, monkeypatch, complex_):
    """The MPS-only chain of compress_mps (reduce_tall = 0): chi D x chi at chi = 64, D = 8, handed to one CAQR even
    above the (lowered) height limit."""
    monkeypatch.setenv("PEPS_QR_MAX_ROWS", "64")
    fs.chain_tall(lib, complex_, 512, 64, 0.0, reduce_tall=False)


@CX
def test_gpu_chain_step_deterministic(lib, complex_):
    fs.chain_determinism(lib, complex_, 4096, 512)


@CX
@pytest.mark.parametrize("nr,nc,dmin,dmax,terr", [(3, 3, 2, 2, 0.0), (64, 64, 8, 8, 0.0), (8, 512, 8, 8, 0.0),
                                                   (512, 64, 16, 16, 0.0), (40, 72, 4, 30, 1e-6), (100, 37, 10, 20, 1e-3),
                                                   (216, 216, 36, 36, 0.0), (432, 216, 36, 36, 0.0), (512, 512, 64, 64, 0.0)])
def test_gpu_truncation_known_svd(lib, complex_, nr, nc, dmin, dmax, terr):
    fs.trunc_known_svd(lib, complex_, nr, nc, dmin, dmax, terr)


@pytest.mark.parametrize("nr,nc", [(512, 512), (1024, 512)])
def test_gpu_truncation_known_svd_complex_chi64(lib, nr, nc):
    """Embeddings of 1024 / 2048 rows and 1024 columns: the block Jacobi path with 8-row blocks."""
    fs.trunc_known_svd(lib, True, nr, nc, 64, 64, 0.0)


@CX
@pytest.mark.parametrize("nr,nc,t", [(48, 40, 7), (432, 216, 36)])
def test_gpu_truncation_odd_embedded_cut(lib, complex_, nr, nc, t):
    fs.trunc_odd_cut(lib, complex_, nr, nc, t)


@CX
@pytest.mark.parametrize("small_svd", ["1", "0"])
@pytest.mark.parametrize("nr,nc,ranks,dmin,dmax", [(40, 30, (3, 5, 0), 8, 12), (432, 216, (10, 30, 0), 36, 36)])
def test_gpu_truncation_rank_below_dmin(lib, monkeypatch, complex_, small_svd, nr, nc, ranks, dmin, dmax):
    monkeypatch.setenv("PEPS_SMALL_SVD", small_svd)
    print(fs.trunc_rank_below_dmin(lib, complex_, nr, nc, ranks, dmin, dmax))


@CX
@pytest.mark.parametrize("nr,nc,dmin", [(12, 5, 6), (5, 5, 5), (72, 36, 36)])
def test_gpu_truncation_identity_shortcut(lib, complex_, nr, nc, dmin):
    fs.trunc_identity(lib, complex_, nr, nc, dmin)


@CX
@pytest.mark.parametrize("nr,nc,dmin,dmax,terr", [(64, 48, 2, 30, 1e-6), (432, 216, 4, 36, 1e-6)])
def test_gpu_truncation_mixed_batch(lib, complex_, nr, nc, dmin, dmax, terr):
    fs.trunc_mixed_batch(lib, complex_, nr, nc, dmin, dmax, terr)


@CX
@pytest.mark.parametrize("env", [("PEPS_SMALL_SVD", "1"), ("PEPS_SMALL_SVD", "0"), ("PEPS_PRESORT_COLS", "0")],
                         ids=["small_svd", "block_jacobi", "no_presort"])
@pytest.mark.parametrize("nr,nc,dmin,dmax,terr", [(64, 64, 8, 8, 0.0), (100, 37, 10, 20, 1e-3), (216, 216, 36, 36, 0.0)])
def test_gpu_truncation_paths(lib, monkeypatch, complex_, env, nr, nc, dmin, dmax, terr):
    monkeypatch.setenv(*env)
    fs.trunc_known_svd(lib, complex_, nr, nc, dmin, dmax, terr)


@CX
@pytest.mark.parametrize("nr,nc", [(64, 48), (512, 512)])
def test_gpu_truncation_deterministic(lib, complex_, nr, nc):
    fs.trunc_determinism(lib, complex_, nr, nc, 4, 64, 1e-8)


def test_gpu_complex_variational_convergence_matches_real(lib):
    fs.variational_convergence_real_vs_complex(lib)
