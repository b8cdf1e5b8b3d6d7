"""ctypes binding of the C ABI declared in include/peps_b200.h.

``load()`` opens the in-tree CUDA library (building it on first use if a compiler is present). There is no
CPU fallback: on a machine without a CUDA device ``peps_create`` fails with a clear error.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libpeps_b200.so")


class PepsConfig(C.Structure):
    _fields_ = [("rows", C.c_int32), ("cols", C.c_int32), ("phys", C.c_int32), ("D", C.c_int32),
                ("walkers", C.c_int32), ("device", C.c_int32), ("dmin", C.c_int32), ("dmax", C.c_int32),
                ("trunc_err", C.c_double)]


class PepsCGParams(C.Structure):
    _fields_ = [("max_iter", C.c_int32), ("relative_tolerance", C.c_double), ("absolute_tolerance", C.c_double),
                ("residual_recompute_interval", C.c_int32), ("orthogonality_threshold", C.c_double)]


class PepsTestOperand(C.Structure):
    """peps_test_operand: one host-buffer operand of peps_test_gett / peps_test_dot."""
    _fields_ = [("data", C.POINTER(C.c_double)), ("len", C.c_int64), ("off", C.c_int64), ("ws", C.c_int64),
                ("gidx", C.POINTER(C.c_int32)), ("gidx_len", C.c_int64), ("gws", C.c_int32), ("gs", C.c_int64)]


# int (*peps_allreduce_fn)(void *user, double *device_buf, size_t n)
ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_size_t)

_P = C.c_void_p
_D = C.POINTER(C.c_double)
_I = C.POINTER(C.c_int32)
_U = C.POINTER(C.c_uint32)
_TO = C.POINTER(PepsTestOperand)

# name -> (restype, argtypes); the single source of truth used by tests to check the exported symbols
SIGNATURES = {
    "peps_backend_name": (C.c_char_p, []),
    "peps_create": (C.c_int, [C.POINTER(_P), C.POINTER(PepsConfig)]),
    "peps_destroy": (None, [_P]),
    "peps_last_error": (C.c_char_p, [_P]),
    "peps_tps_size": (C.c_size_t, [_P]),
    "peps_tps_site_offset": (C.c_size_t, [_P, C.c_int32, C.c_int32]),
    "peps_set_tps": (C.c_int, [_P, _D, C.c_size_t]),
    "peps_get_tps": (C.c_int, [_P, _D, C.c_size_t]),
    "peps_set_truncation": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_double]),
    "peps_set_compress_scheme": (C.c_int, [_P, C.c_int32, C.c_double, C.c_int32]),
    "peps_set_jacobi": (C.c_int, [_P, C.c_double, C.c_int32, C.c_int32]),
    "peps_set_deflation": (C.c_int, [_P, C.c_double]),
    "peps_set_model_xxz": (C.c_int, [_P, C.c_double, C.c_double, C.c_double]),
    "peps_set_chain_deflation": (C.c_int, [_P, C.c_double]),
    "peps_set_model_j1j2_xxz": (C.c_int, [_P, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double]),
    "peps_set_model_term": (C.c_int, [_P, C.c_int32, C.c_int32, _D, _I, _D]),
    "peps_clear_model_terms": (C.c_int, [_P]),
    "peps_set_bond_pin": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, _D, _I, _D]),
    "peps_measure_bond_term": (C.c_int, [_P, C.c_int32, _D, _I, _D, _D, _D]),
    "peps_measure_site_term": (C.c_int, [_P, C.c_int32, _D, _I, _D, _D]),
    "peps_set_fermion": (C.c_int, [_P, _I, _I, C.c_size_t]),
    "peps_set_jastrow": (C.c_int, [_P, _D, _I]),
    "peps_set_complex": (C.c_int, [_P]),
    "peps_set_tps_c": (C.c_int, [_P, _D, _D, C.c_size_t]),
    "peps_get_planar": (C.c_int, [_P, C.c_int32, _D, _D]),
    "peps_clear_jastrow": (C.c_int, [_P]),
    "peps_set_configs": (C.c_int, [_P, _I]),
    "peps_get_configs": (C.c_int, [_P, _I]),
    "peps_seed_rng": (C.c_int, [_P, _U]),
    "peps_set_rng_state": (C.c_int, [_P, _U, _I]),
    "peps_get_rng_state": (C.c_int, [_P, _U, _I]),
    "peps_init_walkers": (C.c_int, [_P]),
    "peps_get_amplitudes": (C.c_int, [_P, _D]),
    "peps_normalize_state_order1": (C.c_int, [_P, C.c_double, _D]),
    "peps_sweep": (C.c_int, [_P, C.c_int32, _D]),
    "peps_sweep_full_space": (C.c_int, [_P, C.c_int32, _D]),
    "peps_sweep_three_site": (C.c_int, [_P, C.c_int32, _D]),
    "peps_measure": (C.c_int, [_P, _D, _D, _D, _D, _D, _D]),
    "peps_set_updater": (C.c_int, [_P, C.c_int32]),
    "peps_set_model_tfim": (C.c_int, [_P, C.c_double]),
    "peps_energy_and_holes": (C.c_int, [_P, C.c_int32, _D, _D]),
    "peps_structure_factor_pairs": (C.c_int64, [_P]),
    "peps_measure_structure_factor": (C.c_int, [_P, _D]),
    "peps_holes_stride": (C.c_size_t, [_P]),
    "peps_get_holes": (C.c_int, [_P, _D]),
    "peps_zero_accumulators": (C.c_int, [_P]),
    "peps_accumulate_ostar": (C.c_int, [_P]),
    "peps_get_accumulators": (C.c_int, [_P, _D, _D, C.c_size_t]),
    "peps_ostar_sum_device": (C.c_void_p, [_P]),
    "peps_eloc_ostar_sum_device": (C.c_void_p, [_P]),
    "peps_sample": (C.c_int, [_P, C.c_int32, _D, _D]),
    "peps_sr_reserve": (C.c_int, [_P, C.c_int64]),
    "peps_sr_collect": (C.c_int, [_P, C.c_int32]),
    "peps_sr_clear": (C.c_int, [_P]),
    "peps_sr_count": (C.c_int64, [_P]),
    "peps_sr_matvec": (C.c_int, [_P, _D, C.c_double, _D, C.c_size_t]),
    "peps_sr_matvec_device": (C.c_int, [_P, C.c_void_p, C.c_double, C.c_void_p]),
    "peps_sr_matvec_c": (C.c_int, [_P, _D, C.c_double, C.c_double, _D, C.c_size_t]),
    "peps_sr_natural_gradient": (C.c_int, [_P, _D, _D, C.c_int64, C.c_double, C.POINTER(PepsCGParams), _D, ALLREDUCE_FN,
                                           C.c_void_p, _D, C.POINTER(C.c_int32), _D, C.POINTER(C.c_int32)]),
    "peps_sr_minsr_natural_gradient": (C.c_int, [_P, C.c_int64, C.c_double, _D, _D]),
    "peps_sr_minsr_tmatrix": (C.c_int, [_P, _D, C.c_size_t]),
    "peps_sr_minsr_gram_diag": (C.c_int, [_P, _D, C.c_size_t]),
    "peps_probe_trace_row": (C.c_int, [_P, C.c_int32, _D]),
    "peps_probe_tnn_trace": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, _I, _D]),
    "peps_probe_plaquette_trace": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _D]),
    "peps_bmps_stack_size": (C.c_int32, [_P, C.c_int32]),
    "peps_get_bmps_tensor": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, _D, _I]),
    "peps_stat": (C.c_int64, [_P, C.c_int32]),
    "peps_sync": (C.c_int, [_P]),
    "peps_profile_enable": (C.c_int, [_P, C.c_int32]),
    "peps_profile_get": (C.c_int, [_P, _D, C.POINTER(C.c_int64), _D, C.c_int32]),
    "peps_stream": (C.c_void_p, [_P]),
    "peps_test_qr_r": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, _D, _D]),
    "peps_test_truncate": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_double,
                                     _D, _D, _I, _I]),
    "peps_test_chain_step": (C.c_int, [_P, C.c_int32, C.c_int32, _D, _D, _I, C.c_int32, C.c_int32, C.c_double, C.c_int32,
                                       _D, _D, _I, _I, _I]),
    "peps_test_truncated_right_vectors": (C.c_int, [_P, C.c_int32, C.c_int32, _D, _D, C.c_int32, C.c_int32, C.c_double,
                                                    C.c_int32, _D, _D, _I]),
    "peps_test_einsum": (C.c_int, [C.c_int32, C.c_int32, C.c_char_p, _I, C.c_int32, _I, C.c_int32, _D, _D, _D]),
    "peps_test_gett": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _I, _I, _I, _I, _I, _I, C.c_int32,
                                 C.c_int32, _I, _I, _I, C.c_int32, _I, C.c_int32, C.c_double, C.c_double, _TO, _TO, _TO, _D,
                                 _I]),
    "peps_test_dot": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, _I, _I, _TO, _TO, _D]),
}


def bind(path):
    """dlopen ``path`` and attach the prototypes."""
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


_lib = None


def load():
    """The product library. Raises if it has not been built (``python peps_b200/build.py`` or
    ``__graft_entry__.build()``)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            from . import build as _build
            _build.build_cuda()
        _lib = bind(LIB_PATH)
    return _lib
