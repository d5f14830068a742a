"""ctypes binding of libnsgpu.so (include/nsgpu.h).  PyTorch is not required.

The library is built in-tree by ``build()`` (nvcc, sm_100a).  There is no CPU fallback: if the shared
object is missing or no CUDA device is present the calls raise ``NsgpuError``.
"""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libnsgpu.so")
_lib = None

c_i32p = ctypes.POINTER(ctypes.c_int32)
c_i64p = ctypes.POINTER(ctypes.c_int64)
c_f64p = ctypes.POINTER(ctypes.c_double)
c_ctx = ctypes.c_void_p


class NsgpuError(RuntimeError):
    pass


# name -> (restype, argtypes): every symbol include/nsgpu.h declares
SIGNATURES = {
    "nsgpu_version": (ctypes.c_int, []),
    "nsgpu_create": (ctypes.c_int, [ctypes.POINTER(c_ctx), ctypes.c_int]),
    "nsgpu_destroy": (ctypes.c_int, [c_ctx]),
    "nsgpu_last_error": (ctypes.c_char_p, [c_ctx]),
    "nsgpu_set_mesh": (ctypes.c_int, [c_ctx, ctypes.c_int, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_void_p]),
    "nsgpu_set_space": (ctypes.c_int, [c_ctx, ctypes.c_int, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64]),
    "nsgpu_set_form": (ctypes.c_int, [c_ctx, ctypes.c_int] + [ctypes.c_double] * 5),
    "nsgpu_set_bcs": (ctypes.c_int, [c_ctx, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "nsgpu_build_pattern": (ctypes.c_int, [c_ctx, c_i64p]),
    "nsgpu_get_pattern": (ctypes.c_int, [c_ctx, ctypes.c_void_p, ctypes.c_void_p]),
    "nsgpu_pattern_sizes": (ctypes.c_int, [c_ctx, c_i64p, c_i64p]),
    "nsgpu_owned_nnz": (ctypes.c_int, [c_ctx, c_i64p]),
    "nsgpu_residual": (ctypes.c_int, [c_ctx, ctypes.c_void_p, ctypes.c_void_p]),
    "nsgpu_jacobian": (ctypes.c_int, [c_ctx, ctypes.c_void_p, ctypes.c_void_p]),
    "nsgpu_jacobian_residual": (ctypes.c_int, [c_ctx, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "nsgpu_spmv": (ctypes.c_int, [c_ctx, ctypes.c_void_p, ctypes.c_void_p]),
    "nsgpu_tfqmr": (ctypes.c_int, [c_ctx, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_double, ctypes.c_double, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                   ctypes.POINTER(ctypes.c_int), c_f64p, c_f64p]),
    "nsgpu_tfqmr_dev": (ctypes.c_int, [c_ctx, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_double, ctypes.c_double, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                       ctypes.POINTER(ctypes.c_int), c_f64p, c_f64p]),
    "nsgpu_ilu_apply": (ctypes.c_int, [c_ctx, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "nsgpu_ilu_colours": (ctypes.c_int, [c_ctx, ctypes.c_void_p, ctypes.POINTER(ctypes.c_int32)]),
    "nsgpu_pilu_apply": (ctypes.c_int, [c_ctx, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "nsgpu_pilu_colours": (ctypes.c_int, [c_ctx, ctypes.c_void_p, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32)]),
    "nsgpu_axpy_dev": (ctypes.c_int, [c_ctx, ctypes.c_double, ctypes.c_void_p, ctypes.c_void_p]),
    "nsgpu_norm_dev": (ctypes.c_int, [c_ctx, ctypes.c_void_p, c_f64p]),
    "nsgpu_dot_dev": (ctypes.c_int, [c_ctx, ctypes.c_void_p, ctypes.c_void_p, c_f64p]),
    "nsgpu_values_norm": (ctypes.c_int, [c_ctx, c_f64p]),
    "nsgpu_set_values": (ctypes.c_int, [c_ctx, ctypes.c_void_p]),
    "nsgpu_get_values": (ctypes.c_int, [c_ctx, ctypes.c_void_p]),
    "nsgpu_jacobian_residual_dev": (ctypes.c_int, [c_ctx, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]),
    "nsgpu_spmv_dev": (ctypes.c_int, [c_ctx, ctypes.c_void_p, ctypes.c_void_p]),
    "nsgpu_values_dev": (ctypes.c_int, [c_ctx, ctypes.POINTER(ctypes.c_void_p)]),
    "nsgpu_sync": (ctypes.c_int, [c_ctx]),
    "nsgpu_stream": (ctypes.c_void_p, [c_ctx]),
    "nsgpu_dev_alloc": (ctypes.c_int, [c_ctx, ctypes.c_int64, ctypes.POINTER(ctypes.c_void_p)]),
    "nsgpu_dev_free": (ctypes.c_int, [c_ctx, ctypes.c_void_p]),
    "nsgpu_memcpy_h2d": (ctypes.c_int, [c_ctx, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64]),
    "nsgpu_memcpy_d2h": (ctypes.c_int, [c_ctx, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64]),
    "nsgpu_host_alloc_pinned": (ctypes.c_int, [ctypes.c_int64, ctypes.POINTER(ctypes.c_void_p)]),
    "nsgpu_host_free_pinned": (ctypes.c_int, [ctypes.c_void_p]),
    "nsgpu_last_kernel_name": (ctypes.c_char_p, [c_ctx]),
    "nsgpu_last_spmv_name": (ctypes.c_char_p, [c_ctx]),
    "nsgpu_set_option": (ctypes.c_int, [c_ctx, ctypes.c_char_p, ctypes.c_int64]),
    "nsgpu_timers": (ctypes.c_int, [c_ctx, c_f64p, ctypes.c_int]),
    "nsgpu_fp64_peak": (ctypes.c_int, [c_ctx, c_f64p]),
    "nsgpu_launch_count": (ctypes.c_int64, [c_ctx]),
    "nsgpu_last_kernel_ms": (ctypes.c_int, [c_ctx, c_f64p]),
    "nsgpu_timer_start": (ctypes.c_int, [c_ctx]),
    "nsgpu_timer_stop": (ctypes.c_int, [c_ctx, c_f64p]),
    "nsgpu_comm_unique_id": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64]),
    "nsgpu_comm_init": (ctypes.c_int, [c_ctx, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]),
    "nsgpu_set_halo": (ctypes.c_int, [c_ctx, ctypes.c_int] + [ctypes.c_void_p] * 5),
    "nsgpu_set_row_exchange": (ctypes.c_int, [c_ctx, ctypes.c_int] + [ctypes.c_void_p] * 5),
    "nsgpu_set_col_ghosts": (ctypes.c_int, [c_ctx, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "nsgpu_local_sizes": (ctypes.c_int, [c_ctx, c_i64p, c_i64p, c_i64p]),
    "nsgpu_get_rows": (ctypes.c_int, [c_ctx, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64]),
    "nsgpu_add_pattern_entries": (ctypes.c_int, [c_ctx, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p]),
    "nsgpu_trace_setup": (ctypes.c_int, [c_ctx, ctypes.c_void_p, ctypes.c_double]),
    "nsgpu_trace_velocity": (ctypes.c_int, [c_ctx, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "nsgpu_trace_run": (ctypes.c_int, [c_ctx, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int] + [ctypes.c_double] * 6 + [ctypes.c_int64] + [ctypes.c_void_p] * 4),
}


def build(verbose=False):
    """Compile libnsgpu.so for sm_100a with nvcc (cross-compiles without a GPU)."""
    r = subprocess.run(["make", "-C", os.path.join(_HERE, "csrc"), "-j8"], capture_output=not verbose, text=True)
    if r.returncode != 0:
        raise NsgpuError("building libnsgpu.so failed:\n" + (r.stdout or "") + (r.stderr or ""))
    return LIB_PATH


def load():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NsgpuError(f"{LIB_PATH} is missing: run __graft_entry__.build() (nvcc, sm_100a). There is no CPU fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def check(ctx, rc, what=""):
    if rc != 0:
        msg = load().nsgpu_last_error(ctx)
        raise NsgpuError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")
