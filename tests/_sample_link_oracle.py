"""ctypes/numpy front-end of the link-prediction oracle (tests/c/sample_link_oracle.c, compiled
together with tests/c/sample_ext_oracle.c, whose weighted key it shares).  TEST INFRASTRUCTURE ONLY:
imported by the link-prediction tests, never by the product package.

The shared object is built with gcc (-ffp-contract=off) once per process in a temporary directory
that is removed as soon as the library is loaded, so nothing is written into the source tree."""
from __future__ import annotations

import ctypes
import os
import subprocess
import tempfile

import numpy as np

_C = os.path.join(os.path.dirname(os.path.abspath(__file__)), "c")
_LIB = None
_i64, _int, _vp, _u64, _u32, _i32 = ctypes.c_int64, ctypes.c_int, ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int32
U64_MASK = 2 ** 64 - 1


def lib() -> ctypes.CDLL:
    global _LIB
    if _LIB is None:
        with tempfile.TemporaryDirectory(prefix="ofspmm_sample_link_oracle_") as d:
            so = os.path.join(d, "libsample_link_oracle.so")
            subprocess.run(["gcc", "-O2", "-fPIC", "-shared", "-std=c11", "-ffp-contract=off", "-o", so,
                            os.path.join(_C, "sample_link_oracle.c"), os.path.join(_C, "sample_ext_oracle.c"), "-lm"],
                           check=True, capture_output=True)
            L = ctypes.CDLL(so)
        L.oracle_take_row.argtypes = [_i64, _i64, _i64, _vp, _int, _int, _i64, _u64, _vp, _i64, _vp]
        L.oracle_take_row.restype = _i64
        L.oracle_edge_ids.argtypes = [_i64, _vp, _vp, _i64, _vp, _vp, _vp, _vp]
        L.oracle_edge_ids.restype = None
        L.oracle_negative_sample.argtypes = [_i64, _i64, _vp, _i64, _vp, _vp, _vp, _i64, _u64, _u32, _i32, _vp, _vp]
        L.oracle_negative_sample.restype = None
        _LIB = L
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data_as(_vp)


def _segments(crow, col, rows_of):
    """The rows rows_of[i] of the CSR (empty for an id outside [0, rows)): (seg_off, seg_base, seg_col)."""
    crow = np.asarray(crow, np.int64)
    rows = crow.size - 1
    r = np.asarray(rows_of, np.int64)
    ok = (r >= 0) & (r < rows)
    d = np.where(ok, r, 0)
    b = crow[d]
    e = np.where(ok, crow[np.minimum(d + 1, rows)], b)
    seg_off = np.concatenate([[0], np.cumsum(e - b)]).astype(np.int64)
    take = np.concatenate([np.arange(x, y) for x, y in zip(b, e)] + [np.zeros(0, np.int64)]).astype(np.int64)
    return seg_off, b.astype(np.int64), np.ascontiguousarray(np.asarray(col)[take], np.int64)


def take_row(v: int, base: int, deg: int, seed: int, excl, prob=None, replace=False, fanout=-1):
    """Offsets j of row v (``deg`` entries from position ``base``) that the sampler takes, in block
    order, with the sorted exclusion list ``excl`` (int64) and the row's weights ``prob``."""
    excl = np.ascontiguousarray(excl, np.int64)
    prob = None if prob is None else np.ascontiguousarray(prob)
    out = np.empty(max(deg, fanout if replace else 0, 1), np.int64)
    n = lib().oracle_take_row(v, base, deg, _p(prob), 0 if prob is None else prob.dtype.itemsize, int(bool(replace)),
                              fanout, seed & U64_MASK, _p(excl), excl.size, _p(out))
    return out[:n]


def sample_neighbors_excl(crow, col, val, dst, fanout: int, seed: int, excl, prob=None, replace: bool = False):
    """ofspmm_sample_neighbors_ex with OFSPMM_SAMPLE_EXCLUDE on the square CSR (crow, col, val) for
    distinct valid destinations: the rows from oracle_take_row, then the block's relabel as the
    header states it (out-of-range columns dropped; src_nodes = dst, then the other sampled ids
    ascending).  Returns (blk_crow, blk_col, blk_val, blk_eid, src_nodes)."""
    crow = np.asarray(crow, np.int64)
    col = np.asarray(col, np.int64)
    rows = crow.size - 1
    excl = np.unique(np.asarray(excl, np.int64))
    blk_crow, gcol, eids = [0], [], []
    for v in np.asarray(dst, np.int64):
        b, e = int(crow[v]), int(crow[v + 1])
        p = None if prob is None else np.asarray(prob)[b:e]
        js = take_row(int(v), b, e - b, seed, excl, p, replace, fanout)
        pos = b + js
        c = col[pos]
        keep = (c >= 0) & (c < rows)
        gcol.append(c[keep])
        eids.append(pos[keep])
        blk_crow.append(blk_crow[-1] + int(keep.sum()))
    gcol = np.concatenate(gcol + [np.zeros(0, np.int64)])
    eid = np.concatenate(eids + [np.zeros(0, np.int64)])
    dst = np.asarray(dst, np.int64)
    new = np.setdiff1d(np.unique(gcol), dst)
    src = np.concatenate([dst, new])
    where = {int(x): i for i, x in enumerate(src)}
    blk_col = np.array([where[int(c)] for c in gcol], np.int64)
    blk_val = None if val is None else np.asarray(val)[eid]
    return np.asarray(blk_crow, np.int64), blk_col, blk_val, eid, src


def edge_ids(crow, col, u, v):
    """ofspmm_edge_ids: position of the first entry (u[i], v[i]) of A, -1 if none."""
    u = np.ascontiguousarray(u, np.int64)
    v = np.ascontiguousarray(v, np.int64)
    seg_off, seg_base, seg_col = _segments(crow, col, u)
    eid = np.empty(u.size, np.int64)
    lib().oracle_edge_ids(len(crow) - 1, _p(u), _p(v), u.size, _p(seg_off), _p(seg_base), _p(seg_col), _p(eid))
    return eid


def negative_sample(crow, col, cols: int, src, k: int, seed: int, exclude_edges=True, exclude_self=True, max_trials=8,
                    segments=None):
    """ofspmm_negative_sample: (neg (len(src) x k), counts [-1 slots, invalid sources]).  ``segments``:
    the sources' rows as (begin, end, seg_col), row of src[i] = seg_col[begin[i]:end[i]], for a
    matrix too large to pass whole (crow then only gives the row count)."""
    src = np.ascontiguousarray(src, np.int64)
    if segments is None:
        seg_off, _, seg_col = _segments(crow, col, src)
        begin, end = seg_off[:-1].copy(), seg_off[1:].copy()
    else:
        begin, end, seg_col = (np.ascontiguousarray(a, np.int64) for a in segments)
    neg = np.empty(max(src.size * k, 1), np.int64)
    counts = np.zeros(2, np.int64)
    flags = (1 if exclude_edges else 0) | (2 if exclude_self else 0)
    lib().oracle_negative_sample(len(crow) - 1, cols, _p(src), src.size, _p(begin), _p(end), _p(seg_col), k,
                                 seed & U64_MASK, flags, max_trials, _p(neg), _p(counts))
    return neg[:src.size * k].reshape(src.size, k), counts
