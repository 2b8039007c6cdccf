"""ctypes binding of libamg1d.so (include/amg1d.h).

There is no CPU fallback: importing this module without the built CUDA library raises, and every
non-zero status from the library raises ``Amg1dError`` with the library's own message.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("AMG1D_LIB") or os.path.join(_HERE, "libamg1d.so")   # AMG1D_LIB: tuning builds

OK, ERR_ARG, ERR_CUDA, ERR_NCCL, ERR_NOMEM, ERR_STATE, ERR_UNSUPPORTED = range(7)
VEC_X, VEC_B, VEC_R = 0, 1, 2
MAX_COLS = 8                     # AMG1D_MAX_COLS: right-hand sides of one multi-column set

_pd = C.POINTER(C.c_double)
_pi64 = C.POINTER(C.c_int64)
_h = C.c_void_p

# name -> (restype, argtypes); the test-suite checks this table against include/amg1d.h
PROTOTYPES = {
    "amg1d_create": (C.c_int, [C.POINTER(_h), C.c_int, C.c_int, C.c_void_p]),
    "amg1d_destroy": (C.c_int, [_h]),
    "amg1d_last_error": (C.c_char_p, [_h]),
    "amg1d_version": (C.c_int, []),
    "amg1d_nccl_unique_id": (C.c_int, [C.c_void_p]),
    "amg1d_create_dist": (C.c_int, [C.POINTER(_h), C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                    C.c_void_p]),
    "amg1d_set_level": (C.c_int, [_h, C.c_int, C.c_int64, C.c_int, _pd, _pd, _pd, _pd, C.c_int,
                                  _pi64, C.c_int64]),
    "amg1d_set_level_flux": (C.c_int, [_h, C.c_int, C.c_int64, C.c_int, _pd, _pd, _pd, _pd, _pd, _pd, _pd,
                                       _pd, _pd, _pd, C.c_int]),
    "amg1d_coarsen_level": (C.c_int, [_h, C.c_int, _pd, C.c_int]),
    "amg1d_coarsen_level_galerkin": (C.c_int, [_h, C.c_int, C.c_int64, C.c_int, _pi64, C.c_int64]),
    "amg1d_get_level": (C.c_int, [_h, C.c_int, _pd, _pd, _pd, _pd]),
    "amg1d_set_level_smoother": (C.c_int, [_h, C.c_int, _pd, _pd, _pd]),
    "amg1d_set_level_pattern": (C.c_int, [_h, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int, _pd,
                                          _pd, _pd, _pd, C.c_int]),
    "amg1d_set_transfer": (C.c_int, [_h, C.c_int, C.c_int64, C.c_int, C.c_int, _pi64, _pd, _pd]),
    "amg1d_set_transfer_pattern": (C.c_int, [_h, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int,
                                             C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _pd, _pd]),
    "amg1d_finalize": (C.c_int, [_h]),
    "amg1d_vcycle": (C.c_int, [_h, _pd, _pd, C.c_int, C.c_int, C.c_double]),
    "amg1d_solve": (C.c_int, [_h, _pd, _pd, C.c_int, C.c_double, C.c_int, C.c_int, C.c_double,
                              C.POINTER(C.c_int), _pd, _pd, _pd]),
    "amg1d_ldiv": (C.c_int, [_h, _pd, _pd, C.c_int, C.c_int, C.c_double]),
    "amg1d_vcycle_batch": (C.c_int, [_h, C.c_int, C.POINTER(_pd), C.POINTER(_pd), C.c_int, C.c_int, C.c_int,
                                     C.c_double]),
    "amg1d_pcg": (C.c_int, [_h, _pd, _pd, C.c_int, C.c_double, C.c_int, C.c_int, C.c_double,
                            C.POINTER(C.c_int), _pd]),
    "amg1d_apply_smoother": (C.c_int, [_h, C.c_int, _pd, _pd, C.c_int64, C.c_double]),
    "amg1d_smoother_solve": (C.c_int, [_h, C.c_int, _pd, _pd, C.c_int, C.c_double, C.c_double,
                                       C.POINTER(C.c_int), _pd, _pd, _pd]),
    "amg1d_matvec": (C.c_int, [_h, C.c_int, _pd, _pd]),
    "amg1d_residual": (C.c_int, [_h, C.c_int, _pd, _pd, _pd]),
    "amg1d_restrict": (C.c_int, [_h, C.c_int, _pd, _pd]),
    "amg1d_prolong": (C.c_int, [_h, C.c_int, _pd, _pd]),
    "amg1d_coarse_solve": (C.c_int, [_h, _pd, _pd]),
    "amg1d_direct_solve": (C.c_int, [_h, C.c_int, _pd, _pd]),
    "amg1d_dev_set_problem": (C.c_int, [_h, _pd, _pd]),
    "amg1d_dev_fill_rhs_random": (C.c_int, [_h, C.c_uint64]),
    "amg1d_dev_assemble_rhs": (C.c_int, [_h, C.c_int, C.c_int, _pd, _pd, C.c_int, C.c_int, _pd, C.c_double,
                                         C.c_double, _pd, C.c_int, _pi64, _pd, C.POINTER(C.c_int)]),
    "amg1d_dev_get_rhs": (C.c_int, [_h, _pd]),
    "amg1d_dev_solve": (C.c_int, [_h, C.c_int, C.c_double, C.c_int, C.c_int, C.c_double, C.POINTER(C.c_int), _pd]),
    "amg1d_dev_pcg": (C.c_int, [_h, C.c_int, C.c_double, C.c_int, C.c_int, C.c_double, C.POINTER(C.c_int), _pd]),
    "amg1d_dev_vcycle": (C.c_int, [_h, C.c_int, C.c_int, C.c_double, C.c_int]),
    "amg1d_dev_residual_norm": (C.c_int, [_h, _pd]),
    "amg1d_dev_rhs_norm": (C.c_int, [_h, _pd]),
    "amg1d_dev_get_solution": (C.c_int, [_h, _pd]),
    "amg1d_dev_set_problems": (C.c_int, [_h, C.c_int, _pd, _pd]),
    "amg1d_dev_fill_rhs_random_multi": (C.c_int, [_h, C.c_int, C.c_uint64]),
    "amg1d_dev_vcycle_multi": (C.c_int, [_h, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int]),
    "amg1d_dev_residual_norms": (C.c_int, [_h, _pd]),
    "amg1d_dev_solve_multi": (C.c_int, [_h, C.c_int, C.c_double, C.c_int, C.c_int, C.c_double, C.POINTER(C.c_int),
                                        _pd]),
    "amg1d_dev_pcg_multi": (C.c_int, [_h, C.c_int, C.c_double, C.c_int, C.c_int, C.c_double, C.POINTER(C.c_int),
                                      _pd]),
    "amg1d_dev_get_solutions": (C.c_int, [_h, _pd]),
    "amg1d_synchronize": (C.c_int, [_h]),
    "amg1d_stream": (C.c_void_p, [_h]),
    "amg1d_dev_ptr": (C.c_void_p, [_h, C.c_int, C.c_int]),
    "amg1d_set_option": (C.c_int, [_h, C.c_char_p, C.c_int64]),
    "amg1d_get_info": (C.c_int64, [_h, C.c_char_p]),
    "amg1d_get_profile": (C.c_int, [_h, C.c_int, C.c_int, _pd, C.POINTER(C.c_int)]),
    "amg1d_host_alloc": (C.c_int, [C.POINTER(C.c_void_p), C.c_int64]),
    "amg1d_host_free": (C.c_int, [C.c_void_p]),
}


class Amg1dError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"libamg1d error {code}: {message}")
        self.code = code


_lib = None


def load():
    """Load libamg1d.so (built in-tree by ``__graft_entry__.build()``); raise if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: the CUDA library is not built. Run "
            "`python -c 'import __graft_entry__ as g; g.build()'` at the repo root. "
            "There is no CPU fallback for the V-cycle.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)      # AttributeError here = header / library mismatch
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(handle, code):
    if code != OK:
        msg = load().amg1d_last_error(handle)
        raise Amg1dError(code, msg.decode() if msg else "")


def dptr(a):
    """Pointer to a C-contiguous float64 numpy array (None -> NULL)."""
    if a is None:
        return None
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_pd)


def iptr(a):
    if a is None:
        return None
    assert a.dtype == np.int64 and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_pi64)


def f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def i64(a):
    return np.ascontiguousarray(a, dtype=np.int64)
