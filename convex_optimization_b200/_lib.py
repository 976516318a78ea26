# -*- coding: utf-8 -*-
"""ctypes binding of libb200lasso.so (C ABI: include/b200lasso.h) and its build recipe.

There is no CPU fallback: importing this module never fails, but the first call that
needs the library raises ``RuntimeError`` when the shared object is missing, and every
compute entry point of the library itself fails without a CUDA device.
"""
import ctypes
import os
import subprocess
import sys

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)
# B200L_LIB selects another build of the library (e.g. an older one, to compare outputs)
LIB_PATH = os.environ.get("B200L_LIB") or os.path.join(_PKG, "libb200lasso.so")
SRC = os.path.join(_PKG, "csrc", "b200lasso.cu")
INCLUDE = os.path.join(_ROOT, "include")
HEADER = os.path.join(INCLUDE, "b200lasso.h")

F32, F64 = 0, 1
NTRACE = 16
NTTRACE = 96
IPC_HANDLE_BYTES = 64
ROWMAJOR, TRANSPOSED = 0, 1

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3",
              "-std=c++17", "-Xcompiler", "-fPIC", "-shared"]


def build(force=False, verbose=False):
    """Compile csrc/b200lasso.cu for sm_100a into the in-tree libb200lasso.so."""
    if (not force and os.path.exists(LIB_PATH)
            and os.path.getmtime(LIB_PATH) >= max(os.path.getmtime(SRC),
                                                  os.path.getmtime(HEADER))):
        return LIB_PATH
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc] + NVCC_FLAGS + ["-I", INCLUDE, SRC, "-o", LIB_PATH]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed:\n%s\n%s" % (" ".join(cmd), proc.stderr))
    if verbose:
        sys.stderr.write(proc.stderr)
    return LIB_PATH


_c_int = ctypes.c_int
_c_i32 = ctypes.c_int32
_c_i64 = ctypes.c_int64
_c_dbl = ctypes.c_double
_p = ctypes.c_void_p
_pd = ctypes.POINTER(ctypes.c_double)
_pi32 = ctypes.POINTER(ctypes.c_int32)
_pi64 = ctypes.POINTER(ctypes.c_int64)
_pint = ctypes.POINTER(ctypes.c_int)

# name -> (restype, argtypes); must list every symbol include/b200lasso.h declares
PROTOTYPES = {
    "b200l_last_error": (ctypes.c_char_p, []),
    "b200l_abi_version": (_c_int, []),
    "b200l_device_count": (_c_int, [_pint]),
    "b200l_device_info": (_c_int, [_c_int, ctypes.c_char_p, _c_int, _pint, _pint, _pint]),
    "b200l_ctx_create": (_c_int, [ctypes.POINTER(_p), _c_int, _c_int, _c_i64, _c_i64, _c_i32, _c_int]),
    "b200l_ctx_destroy": (_c_int, [_p]),
    "b200l_ctx_ld": (_c_int, [_p, _pi64]),
    "b200l_ctx_set_stream": (_c_int, [_p, _p]),
    "b200l_ctx_bind_A": (_c_int, [_p, _p]),
    "b200l_diag_ata": (_c_int, [_p, _pd]),
    "b200l_gemv_t": (_c_int, [_p, _c_i32, _pd, _pd]),
    "b200l_gemv_n": (_c_int, [_p, _c_i32, _pd, _pd]),
    "b200l_set_problem": (_c_int, [_p, _pd]),
    "b200l_reset": (_c_int, [_p]),
    "b200l_set_x": (_c_int, [_p, _pd]),
    "b200l_restart_counters": (_c_int, [_p]),
    "b200l_get_x": (_c_int, [_p, _pd]),
    "b200l_get_r": (_c_int, [_p, _pd]),
    "b200l_run": (_c_int, [_p, _pi32, _c_i64, _c_dbl, _c_dbl, _pd, _pd, _pi64, _pi32, _pd]),
    "b200l_run_config": (_c_int, [_p, _pi32, _pi32, _pi32, _pi32, _pi32, _pi32]),
    "b200l_set_tuning": (_c_int, [_p, _c_i32, _c_i32]),
    "b200l_run_traced": (_c_int, [_p, _c_i64, _c_dbl, ctypes.POINTER(ctypes.c_uint64),
                         ctypes.POINTER(ctypes.c_uint64), _pi32, _pd]),
    "b200l_set_wait_limit": (_c_int, [_p, _c_dbl]),
    "b200l_debug_flags": (_c_int, [_p, _c_i32]),
    "b200l_gen_gaussian": (_c_int, [_p, ctypes.c_uint64, _c_i32, _c_i32]),
    "b200l_row_sumsq": (_c_int, [_p, _pd]),
    "b200l_scale_rows": (_c_int, [_p, _pd]),
    "b200l_comm_export": (_c_int, [_p, _c_i32, _c_i32, _p, _c_i32]),
    "b200l_comm_connect": (_c_int, [_p, _p, _c_i32]),
    "b200l_comm_destroy": (_c_int, [_p]),
    "b200l_objective": (_c_int, [_p, _c_dbl, _pd]),
    "b200l_objective_terms": (_c_int, [_p, _pd, _pd]),
    "b200l_gemv_t_dev": (_c_int, [_p, _c_i32, _p, _p]),
    "b200l_gemv_n_dev": (_c_int, [_p, _c_i32, _p, _p]),
    "b200l_set_diag": (_c_int, [_p, _pd]),
    "b200l_comm_close_peers": (_c_int, [_p]),
    "b200l_comm_inbox_bytes": (_c_int, [_p, _c_i32, _pi64]),
    "b200l_comm_attach": (_c_int, [_p, _c_i32, _c_i32, ctypes.POINTER(_p), _p]),
}

_lib = None


def load():
    """Return the loaded library (ctypes.CDLL) with prototypes set; raise if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "libb200lasso.so is not built (%s). Run `python -c 'import __graft_entry__ as g; "
            "g.build()'` or convex_optimization_b200._lib.build(). There is no CPU fallback."
            % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.b200l_abi_version() != 1:
        raise RuntimeError("libb200lasso.so ABI version mismatch")
    _lib = lib
    return lib


class B200LassoError(RuntimeError):
    pass


def check(rc):
    if rc != 0:
        msg = load().b200l_last_error()
        raise B200LassoError(msg.decode("utf-8", "replace") if msg else "b200lasso failure")


def dptr(arr):
    """double* of a C-contiguous float64 numpy array."""
    return arr.ctypes.data_as(_pd)
