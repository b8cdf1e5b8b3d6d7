"""The boundary-MPS chain step and truncation step on the test-only host simulation of the device ops, against dense
float64 references (tests/factor_steps_common.py), real and complex. Small shapes; tests/test_gpu_factor_steps.py runs
the same checks at the benchmarked sizes on the GPU."""
import pytest

import hostsim_lib
import factor_steps_common as fs

CX = pytest.mark.parametrize("complex_", [False, True], ids=["real", "complex"])


@pytest.fixture(scope="module")
def lib():
    return hostsim_lib.load()


@CX
@pytest.mark.parametrize("m,n", [(18, 18), (37, 5), (5, 37), (128, 96)])
def test_chain_step_full_rank(lib, complex_, m, n):
    fs.chain_full_rank(lib, complex_, m, n)


@CX
@pytest.mark.parametrize("env", [None, ("PEPS_QR_EARLY_STOP", "0"), ("PEPS_QR_STOP_STRIDE", "1")], ids=["default", "nostop", "stride1"])
@pytest.mark.parametrize("m,n,ranks", [(128, 128, (12, 40, 128)), (128, 96, (20, 50, 96)), (128, 128, (12, 40, 60))])
def test_chain_step_exact_rank(lib, monkeypatch, complex_, env, m, n, ranks):
    if env:
        monkeypatch.setenv(*env)
    fs.chain_exact_rank(lib, complex_, m, n, ranks)


@CX
@pytest.mark.parametrize("eps", [1e-4, 1e-8])
@pytest.mark.parametrize("m,n", [(18, 18), (37, 5), (128, 96)])
def test_chain_step_graded_spectrum(lib, complex_, m, n, eps):
    fs.chain_graded(lib, complex_, m, n, eps)


@pytest.mark.parametrize("eps", [0.0, 1e-13])
def test_chain_step_row_hint(lib, eps):
    fs.chain_row_hint(lib, 128, 64, 8, [16, 5, 10], eps)


@CX
@pytest.mark.parametrize("eps", [0.0, 1e-13])
@pytest.mark.parametrize("m,n", [(40, 24), (128, 96)])
def test_chain_step_zero_walker(lib, complex_, m, n, eps):
    fs.chain_zero_walker(lib, complex_, m, n, eps)


@CX
@pytest.mark.parametrize("eps", [0.0, 1e-13])
def test_chain_step_tall_reduction(lib, monkeypatch, complex_, eps):
    monkeypatch.setenv("PEPS_QR_MAX_ROWS", "64")
    fs.chain_tall(lib, complex_, 600, 96, eps)


@CX
def test_chain_step_tall_without_reduction(lib, monkeypatch, complex_):
    """The MPS-only chain of compress_mps (reduce_tall = 0) hands a matrix taller than the limit to one CAQR."""
    monkeypatch.setenv("PEPS_QR_MAX_ROWS", "64")
    fs.chain_tall(lib, complex_, 96, 24, 0.0, reduce_tall=False)


@CX
def test_chain_step_deterministic(lib, complex_):
    fs.chain_determinism(lib, complex_, 128, 96)


@CX
@pytest.mark.parametrize("nr,nc,dmin,dmax,terr", [(3, 3, 2, 2, 0.0), (64, 64, 8, 8, 0.0), (8, 128, 8, 8, 0.0),
                                                   (128, 64, 16, 16, 0.0), (40, 72, 4, 30, 1e-6), (100, 37, 10, 20, 1e-3)])
def test_truncation_known_svd(lib, complex_, nr, nc, dmin, dmax, terr):
    fs.trunc_known_svd(lib, complex_, nr, nc, dmin, dmax, terr)


@CX
def test_truncation_odd_embedded_cut(lib, complex_):
    fs.trunc_odd_cut(lib, complex_, 48, 40, 7)


@CX
@pytest.mark.parametrize("small_svd", ["1", "0"])
def test_truncation_rank_below_dmin(lib, monkeypatch, complex_, small_svd):
    monkeypatch.setenv("PEPS_SMALL_SVD", small_svd)
    print(fs.trunc_rank_below_dmin(lib, complex_, 40, 30, (3, 5, 0), 8, 12))


@CX
@pytest.mark.parametrize("nr,nc,dmin", [(12, 5, 6), (5, 5, 5)])
def test_truncation_identity_shortcut(lib, complex_, nr, nc, dmin):
    fs.trunc_identity(lib, complex_, nr, nc, dmin)


@CX
def test_truncation_mixed_batch(lib, complex_):
    fs.trunc_mixed_batch(lib, complex_, 64, 48, 2, 30, 1e-6)


@CX
@pytest.mark.parametrize("env", [("PEPS_SMALL_SVD", "1"), ("PEPS_SMALL_SVD", "0"), ("PEPS_PRESORT_COLS", "0")],
                         ids=["small_svd", "block_jacobi", "no_presort"])
@pytest.mark.parametrize("nr,nc,dmin,dmax,terr", [(64, 64, 8, 8, 0.0), (100, 37, 10, 20, 1e-3)])
def test_truncation_paths(lib, monkeypatch, complex_, env, nr, nc, dmin, dmax, terr):
    monkeypatch.setenv(*env)
    fs.trunc_known_svd(lib, complex_, nr, nc, dmin, dmax, terr)


@CX
def test_truncation_deterministic(lib, complex_):
    fs.trunc_determinism(lib, complex_, 64, 48, 4, 16, 1e-8)


def test_complex_variational_convergence_matches_real(lib):
    fs.variational_convergence_real_vs_complex(lib)
