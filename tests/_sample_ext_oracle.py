"""ctypes/numpy front-end of the weighted / with-replacement sampling oracle
(tests/c/sample_ext_oracle.c).  TEST INFRASTRUCTURE ONLY: imported by the sampling tests, never by
the product package.

The shared object is compiled with gcc (-ffp-contract=off, so that every fp64 step of the keys is
the one written) once per process into a temporary directory that is removed as soon as the library
is loaded, so nothing is written into the source tree."""
from __future__ import annotations

import ctypes
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "c", "sample_ext_oracle.c")
_LIB = None
_i64, _int, _vp, _u64, _d = ctypes.c_int64, ctypes.c_int, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_double
U64_MASK = 2 ** 64 - 1


def lib() -> ctypes.CDLL:
    global _LIB
    if _LIB is None:
        with tempfile.TemporaryDirectory(prefix="ofspmm_sample_ext_oracle_") as d:
            so = os.path.join(d, "libsample_ext_oracle.so")
            subprocess.run(["gcc", "-O2", "-fPIC", "-shared", "-std=c11", "-ffp-contract=off", "-o", so, _SRC, "-lm"],
                           check=True, capture_output=True)
            L = ctypes.CDLL(so)
        L.oracle_neglog.argtypes = [_d]
        L.oracle_neglog.restype = _d
        L.oracle_neglog_array.argtypes = [_vp, _i64, _vp]
        L.oracle_neglog_array.restype = None
        L.oracle_weighted_key.argtypes = [_u64, _i64, _i64, _d]
        L.oracle_weighted_key.restype = _u64
        L.oracle_sample_neighbors_ex.argtypes = [_i64, _vp, _i64, _vp, _vp, _vp, _vp, _int, _vp, _int, _int, _i64, _u64,
                                                 _vp, _vp, _vp, _vp, _vp, _vp]
        L.oracle_sample_neighbors_ex.restype = None
        _LIB = L
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data_as(_vp)


def neglog(u: np.ndarray) -> np.ndarray:
    """The sampler's -ln u (of-spmm_b200/csrc/sample_key.h) on a float64 array."""
    u = np.ascontiguousarray(u, np.float64)
    out = np.empty_like(u)
    lib().oracle_neglog_array(_p(u), u.size, _p(out))
    return out


def weighted_key(seed: int, v: int, j: int, w: float) -> int:
    """The weighted key bits of position j of row v (all ones for an ineligible weight)."""
    return int(lib().oracle_weighted_key(seed & U64_MASK, v, j, float(w)))


def _pbytes(prob):
    return 0 if prob is None else np.asarray(prob).dtype.itemsize


def sample_neighbors_ex_rows(rows: int, dst, seg_off, seg_base, seg_col, seg_val, seg_prob, replace: bool, fanout: int,
                             seed: int):
    """ofspmm_sample_neighbors_ex on a square A of ``rows`` rows, given only the destinations' rows:
    row dst[i] is seg_col / seg_val / seg_prob[seg_off[i]:seg_off[i+1]] and starts at entry
    seg_base[i] of A.  ``seg_val`` / ``seg_prob`` float32, uint16 (bf16 bits) or None.  Returns
    (blk_crow, blk_col, blk_val, blk_eid, src_nodes, counts)."""
    dst = np.ascontiguousarray(dst, np.int64)
    seg_off = np.ascontiguousarray(seg_off, np.int64)
    seg_base = np.ascontiguousarray(seg_base, np.int64)
    seg_col = np.ascontiguousarray(seg_col, np.int64)
    n = dst.size
    vbytes = 0 if seg_val is None else np.asarray(seg_val).dtype.itemsize
    seg_val = None if seg_val is None else np.ascontiguousarray(seg_val)
    seg_prob = None if seg_prob is None else np.ascontiguousarray(seg_prob)
    total = int(seg_off[-1]) if seg_off.size else 0
    cap = max(n * max(fanout, 0) if replace and fanout != -1 else total, 1)
    blk_crow = np.empty(n + 1, np.int64)
    blk_col = np.empty(cap, np.int64)
    blk_val = np.empty(cap, seg_val.dtype) if seg_val is not None else None
    blk_eid = np.empty(cap, np.int64)
    src = np.empty(n + cap, np.int64)
    counts = np.zeros(3, np.int64)
    lib().oracle_sample_neighbors_ex(rows, _p(dst), n, _p(seg_off), _p(seg_base), _p(seg_col), _p(seg_val), vbytes,
                                     _p(seg_prob), _pbytes(seg_prob), int(bool(replace)), fanout, seed & U64_MASK,
                                     _p(blk_crow), _p(blk_col), _p(blk_val), _p(blk_eid), _p(src), _p(counts))
    nnz, num_src = int(counts[0]), int(counts[1])
    return (blk_crow, blk_col[:nnz], None if blk_val is None else blk_val[:nnz], blk_eid[:nnz], src[:num_src], counts)


def sample_neighbors_ex(crow, col, val, dst, fanout: int, seed: int, prob=None, replace: bool = False):
    """ofspmm_sample_neighbors_ex on the whole square CSR (crow, col, val) with weights ``prob``
    (see sample_neighbors_ex_rows)."""
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
    seg_prob = None if prob is None else np.asarray(prob)[take]
    return sample_neighbors_ex_rows(rows, dst, seg_off, b, col[take], seg_val, seg_prob, replace, fanout, seed)
