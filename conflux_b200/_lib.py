"""ctypes binding of libconflux_b200.so (the C ABI declared in include/conflux_b200.h).

The product path fails loudly when the CUDA library is missing or no device is visible -- there is no CPU
fallback and nothing here imports oracle/."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libconflux_b200.so")
_lib = None

c_double_p = ctypes.POINTER(ctypes.c_double)
c_int_p = ctypes.POINTER(ctypes.c_int)


class ConfluxError(RuntimeError):
    pass


# every exported symbol of include/conflux_b200.h (checked by tests/test_abi.py)
SYMBOLS = [
    "cflx_last_error", "cflx_version", "cflx_device_count", "cflx_get_unique_id", "cflx_comm_create",
    "cflx_comm_barrier", "cflx_comm_destroy", "cflx_host_alloc", "cflx_host_free", "cflx_auto_grid", "cflx_lu_dims", "cflx_init_matrix_host",
    "cflx_lu_create", "cflx_lu_info", "cflx_lu_set_local", "cflx_lu_queue_next_local", "cflx_lu_factor", "cflx_lu_get_factors",
    "cflx_lu_get_permutation", "cflx_lu_residual", "cflx_lu_validate", "cflx_lu_solve", "cflx_lu_launch_count", "cflx_lu_uses_tcgen05", "cflx_lu_set_profiling", "cflx_lu_phase_ms", "cflx_lu_timeline",
    "cflx_lu_set_kernel_timing", "cflx_lu_trailing_stats", "cflx_lu_destroy", "cflx_chol_auto_grid", "cflx_chol_auto_tile", "cflx_chol_dims", "cflx_chol_init_matrix_host",
    "cflx_chol_create", "cflx_chol_info", "cflx_chol_set_local", "cflx_chol_factor", "cflx_chol_get_local", "cflx_chol_validate",
    "cflx_chol_launch_count", "cflx_chol_destroy", "cflx_dbg_gemm_tn", "cflx_dbg_panel", "cflx_dbg_trsm", "cflx_dbg_trsm_left_upper", "cflx_dbg_potrf_tile", "cflx_dbg_push_pivots", "cflx_dbg_ozaki_gemm", "cflx_dbg_umma_peak", "cflx_dbg_last_panel_cycles", "cflx_dbg_fp64_peak", "cflx_dbg_fp64_peak_ex",
]


def _preload_nccl():
    """libconflux_b200.so needs `libnccl.so.2`.  PyTorch bundles a newer NCCL under the same soname; if ours were
    loaded first a later `import torch` would bind to the older system library and fail to resolve its symbols, so
    the bundled one (when present) is loaded first and shared by both."""
    import sys
    for d in sys.path:
        cand = os.path.join(d, "nvidia", "nccl", "lib", "libnccl.so.2")
        if os.path.exists(cand):
            try:
                ctypes.CDLL(cand, mode=ctypes.RTLD_GLOBAL)
                return cand
            except OSError:
                pass
    return None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ConfluxError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(conflux_b200 has no CPU fallback)")
        _preload_nccl()
        L = ctypes.CDLL(LIB_PATH)
        L.cflx_last_error.restype = ctypes.c_char_p
        L.cflx_version.restype = ctypes.c_char_p
        L.cflx_comm_destroy.restype = None
        L.cflx_lu_destroy.restype = None
        L.cflx_comm_destroy.argtypes = [ctypes.c_void_p]
        L.cflx_lu_destroy.argtypes = [ctypes.c_void_p]
        L.cflx_comm_barrier.argtypes = [ctypes.c_void_p]
        L.cflx_comm_create.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int,
                                       ctypes.POINTER(ctypes.c_void_p)]
        L.cflx_lu_create.argtypes = [ctypes.c_void_p] + [ctypes.c_int] * 6 + [ctypes.POINTER(ctypes.c_void_p)]
        L.cflx_host_alloc.argtypes = [ctypes.c_size_t, ctypes.POINTER(ctypes.c_void_p)]
        L.cflx_host_free.argtypes = [ctypes.c_void_p]
        L.cflx_lu_info.argtypes = [ctypes.c_void_p, c_int_p]
        L.cflx_lu_set_local.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        L.cflx_lu_queue_next_local.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        L.cflx_lu_factor.argtypes = [ctypes.c_void_p, c_double_p]
        L.cflx_lu_get_factors.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        L.cflx_lu_get_permutation.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        L.cflx_lu_residual.argtypes = [ctypes.c_void_p, c_double_p]
        L.cflx_lu_validate.argtypes = [ctypes.c_void_p, c_double_p, c_double_p]
        L.cflx_lu_solve.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, c_double_p]
        L.cflx_lu_uses_tcgen05.argtypes = [ctypes.c_void_p]
        L.cflx_lu_launch_count.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64), ctypes.c_int]
        L.cflx_lu_set_profiling.argtypes = [ctypes.c_void_p, ctypes.c_int]
        L.cflx_lu_phase_ms.argtypes = [ctypes.c_void_p, c_double_p]
        L.cflx_lu_timeline.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_int]
        L.cflx_lu_set_kernel_timing.argtypes = [ctypes.c_void_p, ctypes.c_int]
        L.cflx_lu_trailing_stats.argtypes = [ctypes.c_void_p, c_double_p, c_double_p]
        L.cflx_chol_destroy.restype = None
        L.cflx_chol_destroy.argtypes = [ctypes.c_void_p]
        L.cflx_chol_auto_grid.argtypes = [ctypes.c_int, ctypes.c_int, c_int_p]
        L.cflx_chol_auto_tile.argtypes = [ctypes.c_int] * 3
        L.cflx_chol_dims.argtypes = [ctypes.c_int] * 5 + [c_int_p]
        L.cflx_chol_init_matrix_host.argtypes = [ctypes.c_int] * 6 + [ctypes.c_void_p]
        L.cflx_chol_create.argtypes = [ctypes.c_void_p] + [ctypes.c_int] * 5 + [ctypes.POINTER(ctypes.c_void_p)]
        L.cflx_chol_info.argtypes = [ctypes.c_void_p, c_int_p]
        L.cflx_chol_set_local.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        L.cflx_chol_factor.argtypes = [ctypes.c_void_p, c_double_p]
        L.cflx_chol_get_local.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        L.cflx_chol_validate.argtypes = [ctypes.c_void_p, c_double_p, c_double_p]
        L.cflx_chol_launch_count.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64), ctypes.c_int]
        L.cflx_init_matrix_host.argtypes = [ctypes.c_int] * 8 + [ctypes.c_void_p]
        L.cflx_dbg_gemm_tn.argtypes = [ctypes.c_int] * 3 + [ctypes.c_void_p] * 3 + [ctypes.c_double] * 2 + [
            ctypes.c_void_p, ctypes.c_int, c_double_p]
        L.cflx_dbg_panel.argtypes = [ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 4 + [ctypes.c_int, c_double_p]
        L.cflx_dbg_trsm.argtypes = [ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 5
        L.cflx_dbg_trsm_left_upper.argtypes = [ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 3
        L.cflx_dbg_potrf_tile.argtypes = [ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 4
        L.cflx_dbg_push_pivots.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int,
                                           ctypes.c_void_p, ctypes.c_void_p]
        L.cflx_dbg_ozaki_gemm.argtypes = [ctypes.c_int] * 3 + [ctypes.c_void_p] * 8 + [ctypes.c_int, c_double_p, c_double_p]
        L.cflx_dbg_umma_peak.argtypes = [ctypes.c_int, ctypes.c_int, c_double_p]
        L.cflx_dbg_fp64_peak.argtypes = [ctypes.c_int, c_double_p]
        L.cflx_dbg_fp64_peak_ex.argtypes = [ctypes.c_int, c_double_p, c_double_p]
        _lib = L
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = lib().cflx_last_error().decode(errors="replace")
        raise ConfluxError(f"{what} failed with status {rc}: {msg}")
