"""ctypes binding of include/lpb200.h (the C ABI of liblpb200.so).

The library is built in-tree by ``lp_b200/build.py`` (``__graft_entry__.build()``).  There is no
Python or CPU fallback: if the shared library is missing, loading raises ``LibraryNotBuilt``.
"""
from __future__ import annotations

import ctypes as C
import os
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_lib", "liblpb200.so")

LPB_OK = 0
LPB_ERR_UNCONSTRAINED = 1
LPB_ERR_NUMERICAL_PROBLEM = 2
LPB_ERR_INVALID_PARAMETER = 3
LPB_ERR_INCOMPATIBLE_INPUT_DIMENSIONS = 4
LPB_ERR_INFEASIBLE = 5
LPB_ERR_UNBOUNDED = 6
LPB_ERR_ITERATION_LIMIT_EXCEEDED = 7
LPB_ERR_CUDA = -1
LPB_ERR_NCCL = -2
LPB_ERR_NO_DEVICE = -3
LPB_ERR_BAD_ARGUMENT = -4
LPB_ERR_UNSUPPORTED = -5

LPB_SOLVER_CHOLESKY = 0
LPB_SOLVER_INVERSE = 1
LPB_SOLVER_LEAST_SQUARES = 2

LPB_MEM_HOST = 0
LPB_MEM_DEVICE = 1
LPB_TRACE_COLS = 16

c_double_p = C.POINTER(C.c_double)
c_int64_p = C.POINTER(C.c_int64)
c_int32_p = C.POINTER(C.c_int32)


class LibraryNotBuilt(RuntimeError):
    pass


class lpb_options(C.Structure):
    _fields_ = [("tol", C.c_double), ("disp", C.c_int32), ("ip", C.c_int32), ("solver_type", C.c_int32),
                ("reserved", C.c_int32), ("alpha0", C.c_double), ("max_iter", C.c_int64)]


class lpb_residual_scalars(C.Structure):
    _fields_ = [("nrm_rp", C.c_double), ("nrm_rd", C.c_double), ("cx", C.c_double), ("by", C.c_double),
                ("xz", C.c_double)]


class lpb_direction_in(C.Structure):
    _fields_ = [("corrector", C.c_int32), ("ip", C.c_int32), ("eta", C.c_double), ("gamma", C.c_double),
                ("mu", C.c_double), ("alpha", C.c_double)]


class lpb_direction_out(C.Structure):
    _fields_ = [("cu", C.c_double), ("bv", C.c_double), ("cp", C.c_double), ("bq", C.c_double),
                ("nan_pq", C.c_int32), ("reserved", C.c_int32)]


class lpb_profile(C.Structure):
    _fields_ = [("total_ms", C.c_double), ("syrk_ms", C.c_double), ("potrf_ms", C.c_double),
                ("solve_ms", C.c_double), ("sweep_ms", C.c_double), ("vector_ms", C.c_double),
                ("comm_ms", C.c_double), ("launches", C.c_int64), ("iterations", C.c_int64),
                ("syrk_launches", C.c_int64), ("potrf_launches", C.c_int64),
                ("syrk_cols", C.c_int64)]


# name -> (restype, argtypes); must list EVERY symbol include/lpb200.h declares
# (tests/test_abi.py checks the two against each other).
SIGNATURES = {
    "lpb_options_default": (None, [C.POINTER(lpb_options)]),
    "lpb_options_validate": (C.c_int, [C.POINTER(lpb_options)]),
    "lpb_strerror": (C.c_char_p, [C.c_int]),
    "lpb_last_error": (C.c_char_p, []),
    "lpb_abi_version": (C.c_int, []),
    "lpb_device_count": (C.c_int, []),
    "lpb_slack_dims": (C.c_int, [C.c_int64] * 7 + [c_int64_p] * 3),
    "lpb_build_slack_form": (C.c_int, [C.c_void_p, C.c_int64,
                                       C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_int64,
                                       C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_int64,
                                       C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "lpb_host_alloc": (C.c_int, [C.POINTER(C.c_void_p), C.c_uint64]),
    "lpb_host_free": (C.c_int, [C.c_void_p]),
    "lpb_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                             C.c_void_p, C.c_double, C.c_int, C.c_void_p]),
    "lpb_set_problem": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_double, C.c_int]),
    "lpb_create_bare": (C.c_int, [C.POINTER(C.c_void_p), C.c_int64, C.c_int64, C.c_void_p]),
    "lpb_destroy": (C.c_int, [C.c_void_p]),
    "lpb_nccl_unique_id": (C.c_int, [C.c_void_p]),
    "lpb_comm_ready": (C.c_int, [C.c_int, C.c_int]),
    "lpb_peer_export": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]),
    "lpb_peer_import": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "lpb_comm_finalize": (C.c_int, []),
    "lpb_create_sharded": (C.c_int, [C.POINTER(C.c_void_p), C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                     C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_double, C.c_int,
                                     C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "lpb_create_sharded_synthetic": (C.c_int, [C.POINTER(C.c_void_p), C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                               C.c_uint64, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "lpb_download_problem": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "lpb_solve": (C.c_int, [C.c_void_p, C.POINTER(lpb_options), C.c_void_p, c_double_p, c_int64_p]),
    "lpb_trace": (C.c_int64, [C.c_void_p, C.c_void_p, C.c_int64]),
    "lpb_blind_start": (C.c_int, [C.c_void_p]),
    "lpb_residuals": (C.c_int, [C.c_void_p, C.c_double, C.c_double, C.POINTER(lpb_residual_scalars)]),
    "lpb_form_and_factor": (C.c_int, [C.c_void_p]),
    "lpb_direction": (C.c_int, [C.c_void_p, C.POINTER(lpb_direction_in), C.c_double, C.c_double,
                                C.POINTER(lpb_direction_out)]),
    "lpb_assemble_delta": (C.c_int, [C.c_void_p, C.c_double, c_double_p]),
    "lpb_do_step": (C.c_int, [C.c_void_p, C.c_double, C.c_int]),
    "lpb_extract_x": (C.c_int, [C.c_void_p, C.c_double, C.c_void_p, c_double_p]),
    "lpb_solve_batched": (C.c_int, [C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.POINTER(lpb_options), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_int, C.c_void_p]),
    "lpb_solve_many": (C.c_int, [C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.POINTER(lpb_options), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_int, C.c_void_p]),
    "lpb_k_syrk_adat": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                                  C.c_void_p, C.c_int64]),
    "lpb_k_potrf": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, c_int32_p]),
    "lpb_k_potrs": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64]),
    "lpb_k_gemv_n": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "lpb_k_gemv_t": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "lpb_release_workspaces": (C.c_int, []),
    "lpb_get_profile": (C.c_int, [C.c_void_p, C.POINTER(lpb_profile)]),
    "lpb_launch_count": (C.c_int64, [C.c_void_p]),
    "lpb_measure_dmma_peak": (C.c_int, [C.c_void_p, C.c_double, c_double_p]),
    "lpb_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int64]),
    "lpb_debug_read": (C.c_int64, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64]),
    "lpb_debug_counter": (C.c_int64, [C.c_void_p, C.c_char_p]),
    "lpb_presolve_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int64, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p,
                                      C.c_void_p, C.c_int64, C.c_int]),
    "lpb_presolve_info": (C.c_int, [C.c_void_p, c_int64_p, c_int64_p, c_int64_p, c_int64_p, c_int64_p, c_int32_p]),
    "lpb_presolve_get": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "lpb_presolve_restore_x": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "lpb_presolve_destroy": (C.c_int, [C.c_void_p]),
}

_lib = None


def _preload_nccl():
    """liblpb200.so needs `libnccl.so.2`.  A process that also imports torch must end up with ONE NCCL, and it
    has to be torch's bundled one (newer than the system library; torch fails to import against the older
    one: "undefined symbol ncclDevCommCreate").  Loading the bundled copy first, when there is one, makes the
    order of `import torch` and the first lp_b200 call irrelevant."""
    for base in sys.path:
        cand = os.path.join(base, "nvidia", "nccl", "lib", "libnccl.so.2")
        if os.path.exists(cand):
            try:
                C.CDLL(cand, mode=C.RTLD_GLOBAL)
            except OSError:
                pass
            return


def load():
    """dlopen liblpb200.so (once) and attach the prototypes.  Raises LibraryNotBuilt if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LibraryNotBuilt(
            "%s not found: run `python -c 'import __graft_entry__ as g; g.build()'` (or "
            "`python -m lp_b200.build`) first. There is no CPU fallback." % LIB_PATH)
    _preload_nccl()
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.lpb_abi_version() != 1:
        raise RuntimeError("liblpb200.so ABI version mismatch")
    _lib = lib
    return lib


def last_error() -> str:
    s = load().lpb_last_error()
    return s.decode() if s else ""


def strerror(code: int) -> str:
    return load().lpb_strerror(code).decode()
