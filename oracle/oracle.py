"""ctypes/numpy front-end of the CPU oracle (oracle/ofspmm_oracle.c).  TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this module.  The product package ``of-spmm_b200`` never does.

PARITY UNPINNED by the reference: /root/reference holds no SpMM op, test or golden vector
(SURVEY.md §0.1, §8c).  The oracle is pinned instead against scipy.sparse and torch.sparse_csr
(tests/golden/make_golden.py, tests/test_oracle.py).
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import tempfile
from typing import Optional, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "ofspmm_oracle.c")
_OUT = os.path.join(_HERE, "_build")

_c_i64 = ctypes.c_int64
_c_int = ctypes.c_int
_vp = ctypes.c_void_p


def build(native: bool = False, force: bool = False, out: str = _OUT) -> str:
    """Compile the oracle with gcc into ``out`` if the shared object is missing or older than its source."""
    so = os.path.join(out, "libofspmm_oracle_native.so" if native else "libofspmm_oracle.so")
    if not force and os.path.exists(so) and os.path.getmtime(so) >= os.path.getmtime(_SRC):
        return so
    os.makedirs(out, exist_ok=True)
    march = "-march=native" if native else "-march=x86-64-v3"
    cmd = ["gcc", "-O3", "-fPIC", "-shared", "-pthread", "-std=c11", march, "-o", so, _SRC, "-lm"]
    subprocess.run(cmd, check=True, capture_output=True)
    return so


_LIBS = {}


def lib(native: bool = False) -> ctypes.CDLL:
    if native not in _LIBS:
        if native:
            # A -march=native build is only valid on the host that compiles it, and bench.py (the CPU
            # baseline) must not write into the tree, which may be read-only.  So each process compiles
            # it (about a second of gcc) in a temporary directory that is gone as soon as the library is
            # loaded: nothing is left behind, however the process ends.
            with tempfile.TemporaryDirectory(prefix="ofspmm_oracle_") as d:
                L = ctypes.CDLL(build(native=True, out=d))
        else:
            L = ctypes.CDLL(build())
        for fn in ("oracle_spmm_f32", "oracle_spmm_f64", "oracle_spmm_absmax", "oracle_spmm_t_f32",
                   "oracle_spmm_t_f64", "oracle_sddmm_f32"):
            getattr(L, fn).argtypes = [_c_i64, _c_i64, _c_i64, _vp, _vp, _vp, _vp, _vp, _c_int]
            getattr(L, fn).restype = None
        L.oracle_spmm_f32_mt.argtypes = [_c_i64, _c_i64, _c_i64, _vp, _vp, _vp, _vp, _vp, _c_int, _c_int]
        L.oracle_spmm_f32_mt.restype = _c_int
        L.oracle_spmm_t_f32_mt.argtypes = [_c_i64, _c_i64, _c_i64, _vp, _vp, _vp, _vp, _vp, _c_int, _c_int]
        L.oracle_spmm_t_f32_mt.restype = _c_int
        L.oracle_spmm_t_absmax.argtypes = [_c_i64, _c_i64, _c_i64, _vp, _vp, _vp, _vp, _vp, _vp, _c_int]
        L.oracle_spmm_t_absmax.restype = None
        L.oracle_sddmm_f64.argtypes = [_c_i64, _c_i64, _c_i64, _vp, _vp, _vp, _vp, _vp, _vp, _c_int]
        L.oracle_sddmm_f64.restype = None
        L.oracle_merge_path_partition.argtypes = [_vp, _c_int, _c_i64, _c_i64, _c_i64, _vp, _vp]
        L.oracle_merge_path_partition.restype = None
        L.oracle_row_blocks.argtypes = [_vp, _c_int, _c_i64, _c_i64, _c_i64, _vp]
        L.oracle_row_blocks.restype = None
        L.oracle_row_hist.argtypes = [_vp, _c_int, _c_i64, _vp]
        L.oracle_row_hist.restype = None
        L.oracle_csr_transpose.argtypes = [_c_i64, _c_i64, _vp, _vp, _vp, _c_int, _vp, _vp, _vp, _vp]
        L.oracle_csr_transpose.restype = None
        L.oracle_bf16_to_f32.argtypes = [_vp, _vp, _c_i64]
        L.oracle_f32_to_bf16.argtypes = [_vp, _vp, _c_i64]
        L.oracle_balanced_split.argtypes = [_c_i64, _c_i64, _c_i64, _vp, _vp]
        _LIBS[native] = L
    return _LIBS[native]


def _p(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(_vp)


def _idx(crow: np.ndarray, col: np.ndarray) -> Tuple[np.ndarray, np.ndarray, int]:
    if crow.dtype == np.int64 or col.dtype == np.int64:
        return (np.ascontiguousarray(crow, np.int64), np.ascontiguousarray(col, np.int64), 1)
    return (np.ascontiguousarray(crow, np.int32), np.ascontiguousarray(col, np.int32), 0)


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(a, np.float32)


# ------------------------------------------------------------------ bf16

def bf16_to_f32(a_u16: np.ndarray) -> np.ndarray:
    a = np.ascontiguousarray(a_u16, np.uint16)
    out = np.empty(a.shape, np.float32)
    lib().oracle_bf16_to_f32(_p(a), _p(out), a.size)
    return out


def f32_to_bf16(a_f32: np.ndarray) -> np.ndarray:
    a = _f32(a_f32)
    out = np.empty(a.shape, np.uint16)
    lib().oracle_f32_to_bf16(_p(a), _p(out), a.size)
    return out


# ------------------------------------------------------------------ forward

def spmm_f32(crow, col, val, B, K: Optional[int] = None, threads: int = 1, native: bool = False):
    """oracle-A: sequential fp32 CSR·dense (``threads``>1 = equal-row-count split)."""
    crow, col, i64 = _idx(np.asarray(crow), np.asarray(col))
    val, B = _f32(val), _f32(B)
    M, N = crow.size - 1, B.shape[1]
    K = B.shape[0] if K is None else K
    C = np.empty((M, N), np.float32)
    L = lib(native)
    if threads == 1:
        L.oracle_spmm_f32(M, K, N, _p(crow), _p(col), _p(val), _p(B), _p(C), i64)
    else:
        L.oracle_spmm_f32_mt(M, K, N, _p(crow), _p(col), _p(val), _p(B), _p(C), i64, threads)
    return C


def spmm_f64(crow, col, val, B, K: Optional[int] = None):
    """oracle-B: fp64-accumulated ground truth from the fp32 inputs."""
    crow, col, i64 = _idx(np.asarray(crow), np.asarray(col))
    val, B = _f32(val), _f32(B)
    M, N = crow.size - 1, B.shape[1]
    K = B.shape[0] if K is None else K
    C = np.empty((M, N), np.float64)
    lib().oracle_spmm_f64(M, K, N, _p(crow), _p(col), _p(val), _p(B), _p(C), i64)
    return C


def spmm_absmax(crow, col, val, B, K: Optional[int] = None):
    crow, col, i64 = _idx(np.asarray(crow), np.asarray(col))
    val, B = _f32(val), _f32(B)
    M, N = crow.size - 1, B.shape[1]
    K = B.shape[0] if K is None else K
    out = np.empty((M, N), np.float32)
    lib().oracle_spmm_absmax(M, K, N, _p(crow), _p(col), _p(val), _p(B), _p(out), i64)
    return out


def spmm_bf16(crow, col, val, B_u16, K: Optional[int] = None):
    """oracle-A for bf16 dense data: fp32 accumulate over the bf16-exact inputs, one final RNE
    rounding to bf16 (the reference's half-precision convention, SURVEY.md §8a3).  ``val`` is fp32
    or uint16-bf16.  Returns uint16 bf16 bits."""
    val = np.asarray(val)
    val32 = bf16_to_f32(val) if val.dtype == np.uint16 else _f32(val)
    return f32_to_bf16(spmm_f32(crow, col, val32, bf16_to_f32(B_u16), K))


# ------------------------------------------------------------------ backward wrt B

def spmm_t_f32(crow, col, val, dY, K: int, threads: int = 1, native: bool = False):
    crow, col, i64 = _idx(np.asarray(crow), np.asarray(col))
    val, dY = _f32(val), _f32(dY)
    M, N = crow.size - 1, dY.shape[1]
    dB = np.empty((K, N), np.float32)
    L = lib(native)
    if threads == 1:
        L.oracle_spmm_t_f32(M, K, N, _p(crow), _p(col), _p(val), _p(dY), _p(dB), i64)
    else:
        L.oracle_spmm_t_f32_mt(M, K, N, _p(crow), _p(col), _p(val), _p(dY), _p(dB), i64, threads)
    return dB


def spmm_t_f64(crow, col, val, dY, K: int):
    crow, col, i64 = _idx(np.asarray(crow), np.asarray(col))
    val, dY = _f32(val), _f32(dY)
    M, N = crow.size - 1, dY.shape[1]
    dB = np.empty((K, N), np.float64)
    lib().oracle_spmm_t_f64(M, K, N, _p(crow), _p(col), _p(val), _p(dY), _p(dB), i64)
    return dB


def spmm_t_absmax(crow, col, val, dY, K: int):
    crow, col, i64 = _idx(np.asarray(crow), np.asarray(col))
    val, dY = _f32(val), _f32(dY)
    M, N = crow.size - 1, dY.shape[1]
    amax = np.empty((K, N), np.float32)
    cnt = np.empty((K,), np.int64)
    lib().oracle_spmm_t_absmax(M, K, N, _p(crow), _p(col), _p(val), _p(dY), _p(amax), _p(cnt), i64)
    return amax, cnt


# ------------------------------------------------------------------ SDDMM

def sddmm_f32(crow, col, dY, B):
    crow, col, i64 = _idx(np.asarray(crow), np.asarray(col))
    dY, B = _f32(dY), _f32(B)
    M, N, K = crow.size - 1, B.shape[1], B.shape[0]
    out = np.empty((col.size,), np.float32)
    lib().oracle_sddmm_f32(M, K, N, _p(crow), _p(col), _p(dY), _p(B), _p(out), i64)
    return out


def sddmm_f64(crow, col, dY, B):
    crow, col, i64 = _idx(np.asarray(crow), np.asarray(col))
    dY, B = _f32(dY), _f32(B)
    M, N, K = crow.size - 1, B.shape[1], B.shape[0]
    out = np.empty((col.size,), np.float64)
    aabs = np.empty((col.size,), np.float64)
    lib().oracle_sddmm_f64(M, K, N, _p(crow), _p(col), _p(dY), _p(B), _p(out), _p(aabs), i64)
    return out, aabs


# ------------------------------------------------------------------ partitioner / histogram / transpose

def merge_path_partition(crow, P: int):
    crow = np.asarray(crow)
    i64 = 1 if crow.dtype == np.int64 else 0
    crow = np.ascontiguousarray(crow, np.int64 if i64 else np.int32)
    M, nnz = crow.size - 1, int(crow[-1])
    rows = np.empty((P + 1,), np.int64)
    nzs = np.empty((P + 1,), np.int64)
    lib().oracle_merge_path_partition(_p(crow), i64, M, nnz, P, _p(rows), _p(nzs))
    return rows, nzs


def row_blocks(crow, P: int):
    crow = np.asarray(crow)
    i64 = 1 if crow.dtype == np.int64 else 0
    crow = np.ascontiguousarray(crow, np.int64 if i64 else np.int32)
    M, nnz = crow.size - 1, int(crow[-1])
    b = np.empty((P + 1,), np.int64)
    lib().oracle_row_blocks(_p(crow), i64, M, nnz, P, _p(b))
    return b


def row_hist(crow):
    crow = np.asarray(crow)
    i64 = 1 if crow.dtype == np.int64 else 0
    crow = np.ascontiguousarray(crow, np.int64 if i64 else np.int32)
    h = np.empty((32,), np.int64)
    lib().oracle_row_hist(_p(crow), i64, crow.size - 1, _p(h))
    return h


def csr_transpose(crow, col, val, K: int):
    crow, col, i64 = _idx(np.asarray(crow), np.asarray(col))
    val = _f32(val)
    M = crow.size - 1
    nnz = col.size
    t_crow = np.empty((K + 1,), np.int64)
    t_col = np.empty((nnz,), np.int64)
    t_val = np.empty((nnz,), np.float32)
    t_perm = np.empty((nnz,), np.int64)
    lib().oracle_csr_transpose(M, K, _p(crow), _p(col), _p(val), i64, _p(t_crow), _p(t_col),
                               _p(t_val), _p(t_perm))
    return t_crow, t_col, t_val, t_perm


def balanced_split(total: int, parts: int, idx: int):
    b = ctypes.c_int64()
    e = ctypes.c_int64()
    lib().oracle_balanced_split(total, parts, idx, ctypes.byref(b), ctypes.byref(e))
    return b.value, e.value


# ------------------------------------------------------------------ tolerance (SURVEY.md §8c)

def fp32_tolerance(ref64: np.ndarray, amax: np.ndarray, lens: np.ndarray, rtol: float = 1e-5):
    """|got - ref64| <= rtol*|ref64| + 2^-23 * len_i * amax_ij  (row-length-scaled atol)."""
    return rtol * np.abs(ref64) + (2.0 ** -23) * lens.astype(np.float64)[:, None] * amax.astype(np.float64)
