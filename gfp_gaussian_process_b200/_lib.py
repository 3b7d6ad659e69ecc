"""ctypes binding of libggp_b200.so (include/ggp_b200.h).

The shared library is the product; this module only marshals numpy arrays into the C ABI.  There is no
Python or CPU fallback: if the library is missing, or no CUDA device is present, calls raise.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GGP_B200_LIB", os.path.join(_HERE, "libggp_b200.so"))   # override: A/B-testing kernel builds

GGP_OK, GGP_ERR_BAD_ARG, GGP_ERR_NAN, GGP_ERR_CUDA, GGP_ERR_NOMEM = range(5)
N_PARAMS = 11
GGP_MODE_STRICT, GGP_MODE_FAST = 0, 1

c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)
c_int64_p = C.POINTER(C.c_int64)


class ForestDesc(C.Structure):
    _fields_ = [
        ("n_cells", C.c_int64),
        ("n_ctp", C.c_int64),
        ("cell_offset", c_int64_p),
        ("parent", c_int32_p),
        ("daughter1", c_int32_p),
        ("daughter2", c_int32_p),
        ("time", c_double_p),
        ("log_length", c_double_p),
        ("fp", c_double_p),
        ("segment", c_int32_p),
        ("noise_model", C.c_int32),
        ("division_model", C.c_int32),
        ("fp_auto", C.c_double),
        ("init_f", C.c_double * 4),
        ("init_r", C.c_double * 4),
        ("compute_init", C.c_int32),
        ("device", C.c_int32),
    ]


class NanInfo(C.Structure):
    _fields_ = [("cell", C.c_int64), ("t_index", C.c_int64)]


# every entry point include/ggp_b200.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "ggp_forest_create": (C.c_int, [C.POINTER(ForestDesc), C.POINTER(C.c_void_p)]),
    "ggp_forest_destroy": (None, [C.c_void_p]),
    "ggp_forest_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "ggp_forest_upload_series": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ggp_forest_n_cells": (C.c_int64, [C.c_void_p]),
    "ggp_forest_n_ctp": (C.c_int64, [C.c_void_p]),
    "ggp_forest_n_roots": (C.c_int64, [C.c_void_p]),
    "ggp_forest_n_generations": (C.c_int64, [C.c_void_p]),
    "ggp_forest_get_init": (C.c_int, [C.c_void_p, c_double_p, c_double_p]),
    "ggp_correlation_sums": (C.c_int, [C.c_void_p, c_double_p, C.c_int32, C.c_double, C.c_double, C.c_int32, C.c_double, C.c_int32,
                                       c_double_p, c_double_p, c_int64_p]),
    "ggp_group_create": (C.c_int, [C.POINTER(ForestDesc), c_int32_p, C.c_int32, C.POINTER(C.c_void_p)]),
    "ggp_group_destroy": (None, [C.c_void_p]),
    "ggp_group_size": (C.c_int32, [C.c_void_p]),
    "ggp_group_is_contiguous": (C.c_int32, [C.c_void_p]),
    "ggp_group_member": (C.c_void_p, [C.c_void_p, C.c_int32]),
    "ggp_group_member_cells": (C.c_int64, [C.c_void_p, C.c_int32, c_int64_p]),
    "ggp_group_member_ctp": (C.c_int64, [C.c_void_p, C.c_int32, c_int64_p]),
    "ggp_group_set_mode": (C.c_int, [C.c_void_p, C.c_int32]),
    "ggp_group_loglik": (C.c_int, [C.c_void_p, c_double_p, C.c_int32, c_double_p, c_double_p, c_double_p, C.POINTER(NanInfo)]),
    "ggp_group_loglik_grad": (C.c_int, [C.c_void_p, c_double_p, C.c_int32, c_int32_p, C.c_int32, c_double_p, c_double_p,
                                        C.POINTER(NanInfo)]),
    "ggp_group_loglik_hess": (C.c_int, [C.c_void_p, c_double_p, C.c_int32, c_int32_p, C.c_int32, c_double_p, c_double_p,
                                        c_double_p, C.POINTER(NanInfo)]),
    "ggp_group_loglik_tree_grad": (C.c_int, [C.c_void_p, c_double_p, C.c_int32, c_int32_p, C.c_int32, c_double_p, c_double_p,
                                             c_double_p, c_double_p, C.POINTER(NanInfo)]),
    "ggp_group_n_roots": (C.c_int64, [C.c_void_p]),
    "ggp_simulate": (C.c_int, [C.c_void_p, c_double_p, C.c_int32, C.c_uint64, C.c_int32, c_double_p, c_double_p, c_double_p]),
    "ggp_group_simulate": (C.c_int, [C.c_void_p, c_double_p, C.c_int32, C.c_uint64, C.c_int32, c_double_p, c_double_p, c_double_p]),
    "ggp_group_predict": (C.c_int, [C.c_void_p, c_double_p, C.c_int32, c_double_p, c_double_p, c_double_p]),
    "ggp_group_predict14": (C.c_int, [C.c_void_p, c_double_p, C.c_int32, c_double_p, c_double_p, c_double_p]),
    "ggp_group_joints": (C.c_int, [C.c_void_p, c_double_p, C.c_int32, C.c_double, C.c_int64, C.c_int64, C.c_int64, c_int64_p,
                                   c_int64_p, c_int64_p, c_double_p]),
    "ggp_group_correlation_sums": (C.c_int, [C.c_void_p, c_double_p, C.c_int32, C.c_double, C.c_double, C.c_int32, C.c_double, C.c_int32,
                                             c_double_p, c_double_p, c_int64_p]),
    "ggp_forest_set_mode": (C.c_int, [C.c_void_p, C.c_int32]),
    "ggp_forest_get_mode": (C.c_int32, [C.c_void_p]),
    "ggp_last_fast_nodes": (C.c_int32, [C.c_void_p]),
    "ggp_last_strict_reruns": (C.c_int64, [C.c_void_p]),
    "ggp_init_stats": (C.c_int, [C.POINTER(ForestDesc), c_double_p, c_double_p]),
    "ggp_loglik": (C.c_int, [C.c_void_p, c_double_p, C.c_int32, c_double_p, c_double_p, c_double_p, C.POINTER(NanInfo)]),
    "ggp_loglik_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "ggp_loglik_grad": (C.c_int, [C.c_void_p, c_double_p, C.c_int32, c_int32_p, C.c_int32, c_double_p, c_double_p, C.POINTER(NanInfo)]),
    "ggp_loglik_hess": (C.c_int, [C.c_void_p, c_double_p, C.c_int32, c_int32_p, C.c_int32, c_double_p, c_double_p, c_double_p,
                                  C.POINTER(NanInfo)]),
    "ggp_loglik_tree_grad": (C.c_int, [C.c_void_p, c_double_p, C.c_int32, c_int32_p, C.c_int32, c_double_p, c_double_p, c_double_p,
                                       c_double_p, C.POINTER(NanInfo)]),
    "ggp_sync_kernel_ms": (C.c_int, [C.c_void_p, c_double_p]),
    "ggp_predict": (C.c_int, [C.c_void_p, c_double_p, C.c_int32, c_double_p, c_double_p, c_double_p]),
    "ggp_predict14": (C.c_int, [C.c_void_p, c_double_p, C.c_int32, c_double_p, c_double_p, c_double_p]),
    "ggp_backward_cell_state": (C.c_int, [C.c_void_p, c_double_p]),
    "ggp_joints": (C.c_int, [C.c_void_p, c_double_p, C.c_int32, C.c_double, C.c_int64, C.c_int64, C.c_int64, c_int64_p, c_int64_p, c_int64_p, c_double_p]),
    "ggp_last_kernel_ms": (C.c_double, [C.c_void_p]),
    "ggp_last_launch_count": (C.c_int64, [C.c_void_p]),
    "ggp_last_error": (C.c_char_p, []),
    "ggp_version": (C.c_char_p, []),
    "ggp_math_eval": (C.c_int, [C.c_int32, C.c_int32, C.c_int64, c_double_p, c_double_p, c_double_p]),
    "ggp_fp64_peak": (C.c_int, [C.c_int32, c_double_p]),
    "ggp_propagate_eval": (C.c_int, [C.c_int32, C.c_int64, c_double_p, c_double_p, c_double_p, c_double_p, c_double_p]),
}

_lib = None


def load():
    """Load libggp_b200.so (built in-tree by __graft_entry__.build()).  Raises if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
                "There is no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


class GgpError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"ggp error {code}: {msg}")
        self.code = code


def check(rc, allow=()):
    if rc != GGP_OK and rc not in allow:
        raise GgpError(rc, load().ggp_last_error().decode())
    return rc
