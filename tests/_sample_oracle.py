"""ctypes/numpy front-end of the neighbour-sampling oracle (tests/c/sample_oracle.c).  TEST
INFRASTRUCTURE ONLY: imported by the sampling tests, never by the product package.

The shared object is compiled with gcc once per process into a temporary directory that is removed
as soon as the library is loaded, so nothing is written into the source tree."""
from __future__ import annotations

import ctypes
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "c", "sample_oracle.c")
_LIB = None
_i64, _int, _vp, _u64 = ctypes.c_int64, ctypes.c_int, ctypes.c_void_p, ctypes.c_uint64
U64_MASK = 2 ** 64 - 1


def lib() -> ctypes.CDLL:
    global _LIB
    if _LIB is None:
        with tempfile.TemporaryDirectory(prefix="ofspmm_sample_oracle_") as d:
            so = os.path.join(d, "libsample_oracle.so")
            subprocess.run(["gcc", "-O2", "-fPIC", "-shared", "-std=c11", "-o", so, _SRC], check=True, capture_output=True)
            L = ctypes.CDLL(so)
        L.oracle_sample_key.argtypes = [_u64, _i64, _i64]
        L.oracle_sample_key.restype = _u64
        L.oracle_sample_neighbors.argtypes = [_i64, _vp, _i64, _vp, _vp, _vp, _int, _i64, _u64, _vp, _vp, _vp, _vp, _vp]
        L.oracle_sample_neighbors.restype = None
        _LIB = L
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data_as(_vp)


def sample_key(seed: int, v: int, j: int) -> int:
    """key(s, v, j) = mix(mix(s ^ v) + j) of ofspmm_sample_neighbors, as an unsigned int."""
    return int(lib().oracle_sample_key(seed & U64_MASK, v, j))


def sample_neighbors_rows(rows: int, dst, seg_off, seg_col, seg_val, fanout: int, seed: int):
    """ofspmm_sample_neighbors on a square A of ``rows`` rows, given only the destinations' rows: row
    dst[i] is seg_col / seg_val[seg_off[i]:seg_off[i+1]].  ``seg_val`` float32, uint16 (bf16 bits) or
    None.  Returns (blk_crow, blk_col, blk_val, src_nodes, counts), int64 index arrays; values keep
    their dtype and bits."""
    dst = np.ascontiguousarray(dst, np.int64)
    seg_off = np.ascontiguousarray(seg_off, np.int64)
    seg_col = np.ascontiguousarray(seg_col, np.int64)
    n = dst.size
    vbytes = 0 if seg_val is None else np.asarray(seg_val).dtype.itemsize
    seg_val = None if seg_val is None else np.ascontiguousarray(seg_val)
    cap = max(int(seg_off[-1]) if seg_off.size else 0, 1)   # the kept entries are a subset of the rows given
    blk_crow = np.empty(n + 1, np.int64)
    blk_col = np.empty(cap, np.int64)
    blk_val = np.empty(cap, seg_val.dtype) if seg_val is not None else None
    src = np.empty(n + cap, np.int64)
    counts = np.zeros(3, np.int64)
    lib().oracle_sample_neighbors(rows, _p(dst), n, _p(seg_off), _p(seg_col), _p(seg_val), vbytes, fanout,
                                  seed & U64_MASK, _p(blk_crow), _p(blk_col), _p(blk_val), _p(src), _p(counts))
    nnz, num_src = int(counts[0]), int(counts[1])
    return blk_crow, blk_col[:nnz], None if blk_val is None else blk_val[:nnz], src[:num_src], counts


def sample_neighbors(crow, col, val, dst, fanout: int, seed: int):
    """ofspmm_sample_neighbors on the whole square CSR (crow, col, val) (see sample_neighbors_rows)."""
    crow = np.asarray(crow, np.int64)
    col = np.asarray(col, np.int64)
    rows = crow.size - 1
    dst = np.asarray(dst, np.int64)
    ok = (dst >= 0) & (dst < rows)
    d = np.where(ok, dst, 0)
    b, e = crow[d], np.where(ok, crow[np.minimum(d + 1, rows)], crow[d])
    seg_off = np.concatenate([[0], np.cumsum(e - b)])
    take = np.concatenate([np.arange(x, y) for x, y in zip(b, e)] + [np.zeros(0, np.int64)])
    seg_val = None if val is None else np.asarray(val)[take]
    return sample_neighbors_rows(rows, dst, seg_off, col[take], seg_val, fanout, seed)
