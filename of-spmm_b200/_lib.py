"""ctypes binding of libofspmm_b200.so (include/ofspmm.h).

The product path has no CPU fallback: if the CUDA library is missing this module raises
``OfspmmLibraryError`` at load time, and every status code other than OFSPMM_OK raises
``OfspmmError`` — the Python mirror of the glue's CHECK / LOG(FATAL) on a non-zero status
(reference convention: oneflow/core/device/cuda_util.h:54-57).
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libofspmm_b200.so")

DTYPE_FLOAT, DTYPE_INT32, DTYPE_INT64, DTYPE_BFLOAT16 = 2, 5, 6, 11
# value dtype of a pattern matrix: every stored entry is 1.0, no values array (val must be NULL)
VAL_UNIT = 0x100

EXPORTS = (
    "ofspmm_fwd_workspace_bytes", "ofspmm_fwd", "ofspmm_fwd_strided", "ofspmm_bwd_b_workspace_bytes", "ofspmm_bwd_b",
    "ofspmm_bwd_b_transient_workspace_bytes", "ofspmm_bwd_b_transient",
    "ofspmm_sddmm_workspace_bytes", "ofspmm_sddmm", "ofspmm_partition", "ofspmm_partition_host",
    "ofspmm_row_hist", "ofspmm_csr_transpose_workspace_bytes", "ofspmm_csr_transpose",
    "ofspmm_fwd_host_workspace_bytes", "ofspmm_fwd_host", "ofspmm_strerror", "ofspmm_version",
    "ofspmm_launch_count", "ofspmm_fwd_variant", "ofspmm_variant_name",
    "ofspmm_fwd_ex_workspace_bytes", "ofspmm_fwd_ex", "ofspmm_plan_bytes", "ofspmm_plan_build",
    "ofspmm_choose_variant", "ofspmm_bwd_b_cached_workspace_bytes", "ofspmm_bwd_b_cached", "ofspmm_sddmm_ex",
    "ofspmm_gather_rows", "ofspmm_scatter_add_rows", "ofspmm_permute_values", "ofspmm_scatter_add_rows_f32",
    "ofspmm_cast_from_f32", "ofspmm_coo_to_csr_workspace_bytes", "ofspmm_coo_to_csr", "ofspmm_csr_expand_rows",
    "ofspmm_csr_normalize", "ofspmm_signal_peers", "ofspmm_pull_rows_multi", "ofspmm_combine_rows_multi",
    "ofspmm_sample_neighbors_workspace_bytes", "ofspmm_sample_neighbors",
)

# ofspmm_opts.flags / variant codes (include/ofspmm.h)
FWD_ACCUMULATE, FWD_BIAS, FWD_RELU, ORDER_DYNAMIC, ORDER_STATIC, FWD_ACC32_IN, FWD_ACC32_OUT = 1, 2, 4, 8, 16, 32, 64
FWD_MEAN = 128
VARIANT_AUTO, VARIANT_ITEMS64, VARIANT_ROWPAR, VARIANT_ROWS, VARIANT_EXPLICIT = 0, 1, 2, 4, 0x100


class OfspmmLibraryError(ImportError):
    pass


class OfspmmError(RuntimeError):
    def __init__(self, status: int, where: str):
        self.status = status
        msg = lib().ofspmm_strerror(status).decode()
        super().__init__(f"{where}: ofspmm status {status} ({msg})")


class CsrStruct(ctypes.Structure):
    """struct ofspmm_csr (include/ofspmm.h)."""
    _fields_ = [("rows", ctypes.c_int64), ("cols", ctypes.c_int64), ("nnz", ctypes.c_int64),
                ("crow", ctypes.c_void_p), ("col", ctypes.c_void_p), ("val", ctypes.c_void_p),
                ("idx_dtype", ctypes.c_int32), ("val_dtype", ctypes.c_int32)]


class PullSeg(ctypes.Structure):
    """struct ofspmm_pull_seg."""
    _fields_ = [("src", ctypes.c_void_p), ("list", ctypes.c_void_p), ("flag", ctypes.c_void_p),
                ("count", ctypes.c_int64), ("dst_row", ctypes.c_int64)]


class CombineSeg(ctypes.Structure):
    """struct ofspmm_combine_seg."""
    _fields_ = [("src", ctypes.c_void_p), ("inv", ctypes.c_void_p), ("flag", ctypes.c_void_p)]


class OptsStruct(ctypes.Structure):
    """struct ofspmm_opts (include/ofspmm.h)."""
    _fields_ = [("flags", ctypes.c_uint32), ("tasks_per_warp", ctypes.c_int32), ("variant", ctypes.c_int32),
                ("reserve_ctas_per_sm", ctypes.c_int32), ("plan", ctypes.c_void_p), ("plan_bytes", ctypes.c_size_t),
                ("bias", ctypes.c_void_p), ("acc32", ctypes.c_void_p)]


_LIB = None


def lib() -> ctypes.CDLL:
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise OfspmmLibraryError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C of-spmm_b200/csrc`).  There is no CPU fallback on this path.")
    try:
        L = ctypes.CDLL(LIB_PATH)
    except OSError as e:  # pragma: no cover
        raise OfspmmLibraryError(f"cannot load {LIB_PATH}: {e}") from e
    i64, i32, vp, sz = ctypes.c_int64, ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t
    csr_p = ctypes.POINTER(CsrStruct)
    L.ofspmm_fwd_workspace_bytes.argtypes = [i64, i64, i64, i64, i32]
    L.ofspmm_fwd_workspace_bytes.restype = sz
    L.ofspmm_fwd.argtypes = [csr_p, vp, vp, i64, i32, vp, sz, vp]
    L.ofspmm_fwd.restype = i32
    L.ofspmm_fwd_strided.argtypes = [csr_p, vp, i64, vp, i64, i64, i32, vp, sz, vp]
    L.ofspmm_fwd_strided.restype = i32
    L.ofspmm_bwd_b_workspace_bytes.argtypes = [i64, i64, i64, i64, i32, i32]
    L.ofspmm_bwd_b_workspace_bytes.restype = sz
    L.ofspmm_bwd_b.argtypes = [csr_p, csr_p, vp, vp, i64, i32, vp, sz, vp]
    L.ofspmm_bwd_b.restype = i32
    L.ofspmm_bwd_b_transient_workspace_bytes.argtypes = [i64, i64, i64, i64, i32, i32, i32]
    L.ofspmm_bwd_b_transient_workspace_bytes.restype = sz
    L.ofspmm_bwd_b_transient.argtypes = [csr_p, vp, vp, i64, i32, vp, sz, vp]
    L.ofspmm_bwd_b_transient.restype = i32
    L.ofspmm_sddmm_workspace_bytes.argtypes = [i64, i64, i64, i64, i32]
    L.ofspmm_sddmm_workspace_bytes.restype = sz
    L.ofspmm_sddmm.argtypes = [csr_p, vp, vp, vp, i64, i32, vp, sz, vp]
    L.ofspmm_sddmm.restype = i32
    L.ofspmm_partition.argtypes = [vp, i32, i64, i64, i64, vp, vp, vp]
    L.ofspmm_partition.restype = i32
    L.ofspmm_partition_host.argtypes = [vp, i32, i64, i64, i64, vp, vp]
    L.ofspmm_partition_host.restype = i32
    L.ofspmm_row_hist.argtypes = [vp, i32, i64, vp, vp]
    L.ofspmm_row_hist.restype = i32
    L.ofspmm_csr_transpose_workspace_bytes.argtypes = [i64, i64, i64, i32]
    L.ofspmm_csr_transpose_workspace_bytes.restype = sz
    L.ofspmm_csr_transpose.argtypes = [csr_p, vp, vp, vp, vp, vp, sz, vp]
    L.ofspmm_csr_transpose.restype = i32
    L.ofspmm_fwd_host_workspace_bytes.argtypes = [i64, i64, i64, i64, i32, i32, i32]
    L.ofspmm_fwd_host_workspace_bytes.restype = sz
    L.ofspmm_fwd_host.argtypes = [csr_p, vp, vp, i64, i32, vp, sz, vp]
    L.ofspmm_fwd_host.restype = i32
    L.ofspmm_strerror.argtypes = [i32]
    L.ofspmm_strerror.restype = ctypes.c_char_p
    L.ofspmm_version.restype = i32
    L.ofspmm_launch_count.restype = ctypes.c_uint64
    L.ofspmm_fwd_variant.argtypes = [i64, i64, i64, i32]
    L.ofspmm_fwd_variant.restype = ctypes.c_char_p
    opts_p = ctypes.POINTER(OptsStruct)
    L.ofspmm_variant_name.argtypes = [i32, i64, i64, i64, i32]
    L.ofspmm_variant_name.restype = ctypes.c_char_p
    L.ofspmm_fwd_ex_workspace_bytes.argtypes = [i64, i64, i64, i64, i32, i32]
    L.ofspmm_fwd_ex_workspace_bytes.restype = sz
    L.ofspmm_fwd_ex.argtypes = [csr_p, vp, i64, vp, i64, i64, i32, opts_p, vp, sz, vp]
    L.ofspmm_fwd_ex.restype = i32
    L.ofspmm_plan_bytes.argtypes = [i64, i64, i64, i32, i32]
    L.ofspmm_plan_bytes.restype = sz
    L.ofspmm_plan_build.argtypes = [vp, i32, i64, i64, i64, i32, i32, vp, sz, vp]
    L.ofspmm_plan_build.restype = i32
    L.ofspmm_choose_variant.argtypes = [ctypes.POINTER(ctypes.c_int64), i64, i64, i64, i32]
    L.ofspmm_choose_variant.restype = i32
    L.ofspmm_bwd_b_cached_workspace_bytes.argtypes = [i64, i64, i64, i64, i32, i32]
    L.ofspmm_bwd_b_cached_workspace_bytes.restype = sz
    L.ofspmm_bwd_b_cached.argtypes = [csr_p, vp, vp, vp, vp, vp, i64, i32, opts_p, vp, sz, vp]
    L.ofspmm_bwd_b_cached.restype = i32
    L.ofspmm_sddmm_ex.argtypes = [csr_p, vp, vp, vp, i64, i32, opts_p, vp, sz, vp]
    L.ofspmm_sddmm_ex.restype = i32
    L.ofspmm_scatter_add_rows_f32.argtypes = [vp, i64, vp, i64, vp, i32, i64, i64, i64, i32, i32, vp]
    L.ofspmm_scatter_add_rows_f32.restype = i32
    L.ofspmm_cast_from_f32.argtypes = [vp, vp, i64, i32, vp]
    L.ofspmm_cast_from_f32.restype = i32
    L.ofspmm_coo_to_csr_workspace_bytes.argtypes = [i64, i64, i64]
    L.ofspmm_coo_to_csr_workspace_bytes.restype = sz
    L.ofspmm_coo_to_csr.argtypes = [vp, vp, vp, i64, i64, i64, i32, i32, vp, vp, vp, vp, vp, sz, vp]
    L.ofspmm_coo_to_csr.restype = i32
    L.ofspmm_csr_expand_rows.argtypes = [vp, i32, i64, vp, vp]
    L.ofspmm_csr_expand_rows.restype = i32
    L.ofspmm_csr_normalize.argtypes = [vp, vp, vp, i32, i64, i64, i32, vp, vp]
    L.ofspmm_csr_normalize.restype = i32
    L.ofspmm_signal_peers.argtypes = [ctypes.POINTER(ctypes.c_void_p), i32, ctypes.c_uint64, vp]
    L.ofspmm_signal_peers.restype = i32
    L.ofspmm_pull_rows_multi.argtypes = [vp, i64, i64, ctypes.POINTER(PullSeg), i32, ctypes.c_uint64, i64, i32, i32, i32, vp]
    L.ofspmm_pull_rows_multi.restype = i32
    L.ofspmm_combine_rows_multi.argtypes = [vp, i64, i64, ctypes.POINTER(CombineSeg), i32, ctypes.c_uint64, i64, i64, i32, i32, vp]
    L.ofspmm_combine_rows_multi.restype = i32
    L.ofspmm_permute_values.argtypes = [vp, i32, vp, i32, i64, vp, vp]
    L.ofspmm_permute_values.restype = i32
    L.ofspmm_gather_rows.argtypes = [vp, i64, vp, i64, vp, i32, i64, i64, i64, i32, i32, vp]
    L.ofspmm_gather_rows.restype = i32
    L.ofspmm_scatter_add_rows.argtypes = [vp, i64, vp, i64, vp, i32, i64, i64, i64, i32, i32, vp]
    L.ofspmm_scatter_add_rows.restype = i32
    L.ofspmm_sample_neighbors_workspace_bytes.argtypes = [i64, i64, i32]
    L.ofspmm_sample_neighbors_workspace_bytes.restype = sz
    L.ofspmm_sample_neighbors.argtypes = [csr_p, vp, i64, i64, ctypes.c_uint64, i64, vp, vp, vp, vp, vp, vp, sz, vp]
    L.ofspmm_sample_neighbors.restype = i32
    _LIB = L
    return L


def check(status: int, where: str) -> None:
    if status != 0:
        raise OfspmmError(status, where)


def launch_count() -> int:
    return int(lib().ofspmm_launch_count())
