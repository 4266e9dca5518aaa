"""ctypes binding of include/sbn_b200.h, sbn_b200_gp.h and sbn_b200_patterns.h (the C ABI of libsbn_b200.so).

Loading is explicit and loud: if the CUDA library has not been built, importing
this module raises -- there is no Python/NumPy fallback for any compute call.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SBNB_LIBRARY") or os.path.join(_HERE, "lib", "libsbn_b200.so")  # (override: development aid)


class SbnbError(RuntimeError):
    """A failed C-ABI call; mirrors the reference's Failwith -> RuntimeError."""

    def __init__(self, code, message):
        super().__init__(message)
        self.code = code


class TreeBatchStruct(ctypes.Structure):
    _fields_ = [
        ("tree_count", ctypes.c_int32),
        ("node_count", ctypes.c_int32),
        ("parent_ids", ctypes.POINTER(ctypes.c_int32)),
        ("branch_lengths", ctypes.POINTER(ctypes.c_double)),
        ("rates", ctypes.POINTER(ctypes.c_double)),
        ("node_heights", ctypes.POINTER(ctypes.c_double)),
        ("node_bounds", ctypes.POINTER(ctypes.c_double)),
        ("height_ratios", ctypes.POINTER(ctypes.c_double)),
        ("rate_count", ctypes.c_int32),
    ]


class GradientOutStruct(ctypes.Structure):
    _fields_ = [
        ("log_likelihood", ctypes.POINTER(ctypes.c_double)),
        ("branch_lengths", ctypes.POINTER(ctypes.c_double)),
        ("substitution_model", ctypes.POINTER(ctypes.c_double)),
        ("site_model", ctypes.POINTER(ctypes.c_double)),
        ("ratios_root_height", ctypes.POINTER(ctypes.c_double)),
        ("clock_model", ctypes.POINTER(ctypes.c_double)),
    ]


# Every symbol include/sbn_b200.h declares: (restype, argtypes).
_P = ctypes.POINTER
_c = ctypes
SIGNATURES = {
    "sbnb_compress_site_patterns": (_c.c_int, [_c.c_int32, _c.c_int64, _c.c_char_p, _c.c_int32, _P(_c.c_uint8),
                                               _P(_c.c_double), _P(_c.c_int64), _P(_c.c_double)]),
    "sbnb_compress_site_patterns_encoded": (_c.c_int, [_c.c_int32, _c.c_int64, _c.c_char_p, _c.c_int32, _c.c_int32,
                                                       _P(_c.c_uint8), _P(_c.c_double), _P(_c.c_int64),
                                                       _P(_c.c_double)]),
    "sbnb_last_error": (_c.c_char_p, []),
    "sbnb_device_count": (_c.c_int, []),
    "sbnb_engine_create": (_c.c_int, [_c.c_char_p, _c.c_char_p, _c.c_char_p, _c.c_int32, _c.c_int64,
                                      _P(_c.c_uint8), _P(_c.c_double), _c.c_int32, _P(_c.c_void_p)]),
    "sbnb_engine_create_multi": (_c.c_int, [_c.c_char_p, _c.c_char_p, _c.c_char_p, _c.c_int32, _c.c_int64,
                                            _P(_c.c_uint8), _P(_c.c_double), _P(_c.c_int32), _c.c_int32,
                                            _c.c_int32, _P(_c.c_void_p)]),
    "sbnb_engine_create_encoded": (_c.c_int, [_c.c_char_p, _c.c_char_p, _c.c_char_p, _c.c_int32, _c.c_int64,
                                              _P(_c.c_uint8), _c.c_int32, _P(_c.c_double), _c.c_int32,
                                              _P(_c.c_void_p)]),
    "sbnb_engine_create_multi_encoded": (_c.c_int, [_c.c_char_p, _c.c_char_p, _c.c_char_p, _c.c_int32, _c.c_int64,
                                                    _P(_c.c_uint8), _c.c_int32, _P(_c.c_double), _P(_c.c_int32),
                                                    _c.c_int32, _c.c_int32, _P(_c.c_void_p)]),
    "sbnb_engine_device_count": (_c.c_int32, [_c.c_void_p]),
    "sbnb_engine_set_substitution_gradient": (_c.c_int, [_c.c_void_p, _c.c_int32]),
    "sbnb_engine_destroy": (None, [_c.c_void_p]),
    "sbnb_engine_param_count": (_c.c_int32, [_c.c_void_p]),
    "sbnb_engine_param_block": (_c.c_int, [_c.c_void_p, _c.c_char_p, _P(_c.c_int32), _P(_c.c_int32)]),
    "sbnb_engine_category_count": (_c.c_int32, [_c.c_void_p]),
    "sbnb_log_likelihoods_unrooted": (_c.c_int, [_c.c_void_p, _P(TreeBatchStruct), _P(_c.c_double),
                                                 _c.c_int32, _P(_c.c_double)]),
    "sbnb_log_likelihoods_rooted": (_c.c_int, [_c.c_void_p, _P(TreeBatchStruct), _P(_c.c_double),
                                               _c.c_int32, _P(_c.c_double)]),
    "sbnb_unrooted_log_likelihoods_of_rooted": (_c.c_int, [_c.c_void_p, _P(TreeBatchStruct),
                                                           _P(_c.c_double), _c.c_int32, _P(_c.c_double)]),
    "sbnb_site_log_likelihoods_unrooted": (_c.c_int, [_c.c_void_p, _P(TreeBatchStruct), _P(_c.c_double),
                                                      _c.c_int32, _P(_c.c_double), _P(_c.c_double)]),
    "sbnb_site_log_likelihoods_rooted": (_c.c_int, [_c.c_void_p, _P(TreeBatchStruct), _P(_c.c_double),
                                                    _c.c_int32, _P(_c.c_double), _P(_c.c_double)]),
    "sbnb_gradients_unrooted": (_c.c_int, [_c.c_void_p, _P(TreeBatchStruct), _P(_c.c_double),
                                           _c.c_int32, _P(GradientOutStruct)]),
    "sbnb_gradients_rooted": (_c.c_int, [_c.c_void_p, _P(TreeBatchStruct), _P(_c.c_double),
                                         _c.c_int32, _P(GradientOutStruct)]),
    "sbnb_batch_stage": (_c.c_int, [_c.c_void_p, _P(TreeBatchStruct), _P(_c.c_double), _c.c_int32,
                                    _P(_c.c_void_p)]),
    "sbnb_batch_run": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_int32, _c.c_int32]),
    "sbnb_batch_fetch": (_c.c_int, [_c.c_void_p, _c.c_void_p, _P(_c.c_double), _P(_c.c_double),
                                    _P(_c.c_double)]),
    "sbnb_batch_device_results": (_c.c_int, [_c.c_void_p, _P(_c.c_void_p), _P(_c.c_void_p), _P(_c.c_void_p)]),
    "sbnb_batch_fetch_substitution_sums": (_c.c_int, [_c.c_void_p, _c.c_void_p, _P(_c.c_double)]),
    "sbnb_finish_gradients_analytic": (_c.c_int, [_c.c_char_p, _c.c_char_p, _c.c_char_p, _c.c_int32,
                                                  _P(TreeBatchStruct), _c.c_int32, _P(_c.c_double), _P(_c.c_double),
                                                  _P(_c.c_double), _P(_c.c_double), _P(_c.c_double),
                                                  _P(GradientOutStruct)]),
    "sbnb_batch_fetch_site_log_likelihoods": (_c.c_int, [_c.c_void_p, _c.c_void_p, _P(_c.c_double)]),
    "sbnb_batch_fetch_invariant_sums": (_c.c_int, [_c.c_void_p, _c.c_void_p, _P(_c.c_double)]),
    "sbnb_finish_gradients_invariant": (_c.c_int, [_c.c_char_p, _c.c_char_p, _c.c_char_p, _c.c_int32,
                                                   _P(TreeBatchStruct), _c.c_int32, _P(_c.c_double), _P(_c.c_double),
                                                   _P(_c.c_double), _P(_c.c_double), _P(_c.c_double), _P(_c.c_double),
                                                   _P(GradientOutStruct)]),
    "sbnb_finish_gradients": (_c.c_int, [_c.c_char_p, _c.c_char_p, _c.c_char_p, _c.c_int32, _P(TreeBatchStruct),
                                         _c.c_int32, _c.c_int32, _P(_c.c_double), _P(_c.c_double),
                                         _P(_c.c_double), _P(GradientOutStruct)]),
    "sbnb_finish_log_likelihoods_rooted": (_c.c_int, [_c.c_int32, _P(TreeBatchStruct), _P(_c.c_double)]),
    "sbnb_batch_destroy": (None, [_c.c_void_p, _c.c_void_p]),
    "sbnb_batch_evaluation_count": (_c.c_int32, [_c.c_void_p]),
    "sbnb_engine_stream": (_c.c_void_p, [_c.c_void_p]),
    "sbnb_engine_launch_count": (_c.c_int64, [_c.c_void_p]),
    "sbnb_batch_algorithmic_bytes": (_c.c_double, [_c.c_void_p, _c.c_int32]),
    "sbnb_engine_transfer_bytes": (_c.c_int, [_c.c_void_p, _P(_c.c_int64), _P(_c.c_int64)]),
    "sbnb_engine_walk_timing": (_c.c_int, [_c.c_void_p, _P(_c.c_double), _P(_c.c_int64), _c.c_int32]),
    "sbnb_engine_set_pattern_range": (_c.c_int, [_c.c_void_p, _c.c_int64, _c.c_int64]),
    "sbnb_debug_tree_program": (_c.c_int, [_P(_c.c_int32), _c.c_int32, _c.c_int32, _P(_c.c_int32),
                                           _P(_c.c_int32), _P(_c.c_int32)]),
    "sbnb_debug_model_tables": (_c.c_int, [_c.c_char_p, _c.c_char_p, _c.c_char_p] + [_P(_c.c_double)] * 9),
    "sbnb_debug_substitution_derivatives": (_c.c_int, [_c.c_char_p, _c.c_char_p, _c.c_char_p, _P(_c.c_double),
                                                       _P(_c.c_double), _P(_c.c_double), _P(_c.c_int32)]),
}

# Every symbol include/sbn_b200_gp.h declares.
_QUARTET = [_c.c_void_p, _c.c_int32] + [_P(_c.c_int32), _c.c_int32] * 4
_GP_GET = (_c.c_int, [_c.c_void_p, _P(_c.c_double)])
SIGNATURES.update({
    "sbnb_gp_create": (_c.c_int, [_c.c_int32, _c.c_int64, _P(_c.c_uint8), _P(_c.c_double), _c.c_int64, _c.c_int32,
                                  _c.c_int32, _c.c_double, _P(_c.c_double), _P(_c.c_double), _c.c_int32,
                                  _P(_c.c_double), _c.c_int32, _P(_c.c_void_p)]),
    "sbnb_gp_create_encoded": (_c.c_int, [_c.c_int32, _c.c_int64, _P(_c.c_uint8), _c.c_int32, _P(_c.c_double),
                                          _c.c_int64, _c.c_int32, _c.c_int32, _c.c_double, _P(_c.c_double),
                                          _P(_c.c_double), _c.c_int32, _P(_c.c_double), _c.c_int32,
                                          _P(_c.c_void_p)]),
    "sbnb_gp_destroy": (None, [_c.c_void_p]),
    "sbnb_gp_process_operations": (_c.c_int, [_c.c_void_p, _P(_c.c_int32), _c.c_int64]),
    "sbnb_gp_set_substitution_model": (_c.c_int, [_c.c_void_p, _c.c_char_p, _P(_c.c_double), _c.c_int32]),
    "sbnb_gp_set_site_model": (_c.c_int, [_c.c_void_p, _c.c_char_p, _P(_c.c_double), _c.c_int32]),
    "sbnb_gp_category_count": (_c.c_int32, [_c.c_void_p]),
    "sbnb_gp_schedule_program": (_c.c_int, [_c.c_int32, _c.c_int32, _P(_c.c_int32), _c.c_int64, _P(_c.c_int32),
                                          _P(_c.c_int64)]),
    "sbnb_gp_set_branch_lengths": _GP_GET,
    "sbnb_gp_set_branch_lengths_to_constant": (_c.c_int, [_c.c_void_p, _c.c_double]),
    "sbnb_gp_get_branch_lengths": _GP_GET,
    "sbnb_gp_reset_log_marginal_likelihood": (_c.c_int, [_c.c_void_p]),
    "sbnb_gp_get_log_marginal_likelihood": _GP_GET,
    "sbnb_gp_get_per_gpcsp_log_likelihoods": (_c.c_int, [_c.c_void_p, _c.c_int32, _c.c_int32, _P(_c.c_double)]),
    "sbnb_gp_get_per_gpcsp_components_of_full_log_marginal": _GP_GET,
    "sbnb_gp_get_log_likelihood_matrix": _GP_GET,
    "sbnb_gp_get_sbn_parameters": _GP_GET,
    "sbnb_gp_set_sbn_parameters": _GP_GET,
    "sbnb_gp_get_hybrid_marginals": _GP_GET,
    "sbnb_gp_set_hybrid_marginals": _GP_GET,
    "sbnb_gp_log_likelihood_and_derivative": (_c.c_int, [_c.c_void_p, _c.c_int32, _c.c_int32, _c.c_int32,
                                                         _P(_c.c_double)]),
    "sbnb_gp_transition_matrix": (_c.c_int, [_c.c_void_p, _c.c_double, _P(_c.c_double)]),
    "sbnb_gp_quartet_hybrid_likelihoods": (_c.c_int, _QUARTET + [_P(_c.c_double)]),
    "sbnb_gp_process_quartet_hybrid_request": (_c.c_int, _QUARTET),
    "sbnb_gp_get_plv": (_c.c_int, [_c.c_void_p, _c.c_int32, _P(_c.c_double)]),
    "sbnb_gp_get_rescaling_counts": (_c.c_int, [_c.c_void_p, _P(_c.c_int32)]),
    "sbnb_gp_launch_count": (_c.c_int64, [_c.c_void_p]),
    "sbnb_gp_last_kernel_ms": (_c.c_double, [_c.c_void_p]),
    "sbnb_gp_debug_launch_plan": (_c.c_int, [_c.c_void_p, _P(_c.c_int32)]),
})

MODE_LOG_LIKELIHOOD = 0
MODE_BRANCH_GRADIENT = 1
STAGE_ROOTED = 1
STAGE_SUBSTITUTION_FD = 2
STAGE_SUBSTITUTION_ANALYTIC = 4
STAGE_SITE_LOG_LIKELIHOODS = 8
SUBSTITUTION_SUMS = 20
INVARIANT_SUMS = 5  # +I: D, then E_A..E_T (sbnb_batch_fetch_invariant_sums)
SHARD_TREES = 0
TIPS_STATES = 0
TIPS_NUCLEOTIDE_MASKS = 1
TIP_ENCODINGS = {"states": TIPS_STATES, "masks": TIPS_NUCLEOTIDE_MASKS}
SHARD_PATTERNS = 1
SUBSTITUTION_ANALYTIC = 0
SUBSTITUTION_FINITE_DIFFERENCES = 1

_lib = None


def load():
    """Loads libsbn_b200.so and binds every declared symbol; raises if missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} has not been built (run `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C libsbn_b200/csrc`). libsbn_b200 has no CPU fallback."
        )
    lib = ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_GLOBAL)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export it
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def check(code):
    if code != 0:
        message = load().sbnb_last_error()
        # (backslashreplace: no message byte can turn the SbnbError into a UnicodeDecodeError)
        raise SbnbError(code, message.decode(errors="backslashreplace") if message else f"libsbn_b200 error {code}")


def as_double_ptr(array):
    if array is None:
        return None
    assert array.dtype == np.float64 and array.flags["C_CONTIGUOUS"]
    return array.ctypes.data_as(_P(_c.c_double))


def tip_encoding(name):
    """'states' (0..3 = ACGT, >= 4 gap) or 'masks' (nucleotide masks 1..15) -> SBNB_TIPS_*."""
    if name not in TIP_ENCODINGS:
        raise RuntimeError("tip_encoding must be 'states' or 'masks'.")
    return TIP_ENCODINGS[name]


def as_int32_ptr(array):
    if array is None:
        return None
    assert array.dtype == np.int32 and array.flags["C_CONTIGUOUS"]
    return array.ctypes.data_as(_P(_c.c_int32))
