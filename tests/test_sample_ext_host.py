"""CPU tests of weighted / with-replacement neighbour sampling and edge ids: the fp64 -ln of the
weighted keys against numpy.log, the oracle (tests/c/sample_ext_oracle.c) against a brute-force
Python restatement of the definitions in include/ofspmm.h, the C ABI's option validation and
workspace query, and the Python argument checks, none of which needs a GPU."""
import ctypes
import os
import sys
from importlib import import_module

import numpy as np
import pytest
import torch

import ofspmm_b200 as ofs
from oracle import oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import _sample_ext_oracle as SEO  # noqa: E402

_lib = import_module("of-spmm_b200._lib")
sampling = import_module("of-spmm_b200.sampling")
G = ofs.graphs
M64 = (1 << 64) - 1


# ------------------------------------------------------------------ neglog

def _u(m):
    return (np.asarray(m, np.uint64) + np.uint64(1)).astype(np.float64) * 2.0 ** -53


def test_neglog_within_4_ulp_of_numpy_log():
    """Over 10.5e6 distinct inputs (m+1)·2^-53: both ends of the domain, the values just below 1,
    both sides of every reduction boundary (2^-e and sqrt(2)/2·2^-e) and random ones."""
    rng = np.random.default_rng(5)
    parts = [np.arange(0, 1 << 21), (1 << 53) - 1 - np.arange(0, 1 << 22), rng.integers(0, 1 << 53, 1 << 22)]
    for e in range(1, 53):
        for c in (2.0 ** (53 - e), np.sqrt(0.5) * 2.0 ** (53 - e)):
            parts.append(np.clip(int(c) + np.arange(-2000, 2000), 0, (1 << 53) - 1))
    m = np.unique(np.concatenate(parts).astype(np.uint64))
    assert m.size >= 10_000_000
    u = _u(m)
    got = SEO.neglog(u)
    ref = -np.log(u)
    ulp = np.spacing(np.maximum(np.abs(ref), np.finfo(np.float64).tiny))
    err = np.abs(got - ref) / ulp
    assert float(err.max()) <= 4.0, (float(err.max()), float(u[np.argmax(err)]))
    assert (got >= 0).all() and not np.signbit(got).any()


def test_neglog_of_one_is_zero():
    assert SEO.neglog(np.array([1.0]))[0] == 0.0
    assert not np.signbit(SEO.neglog(np.array([1.0]))[0])
    assert SEO.lib().oracle_neglog(1.0) == 0.0


def test_neglog_monotone_on_dense_sweeps():
    """Consecutive inputs below 1, at the bottom of the domain and across the sqrt(2)/2 and 1/2
    boundaries: non-increasing."""
    starts = [(1 << 53) - (1 << 21), 0, int(np.sqrt(0.5) * 2.0 ** 53) - (1 << 20), (1 << 52) - (1 << 20),
              int(np.sqrt(0.5) * 2.0 ** 40) - (1 << 20)]
    for s in starts:
        m = np.arange(s, s + (1 << 21), dtype=np.uint64)
        m = m[m < (1 << 53)]
        v = SEO.neglog(_u(m))
        assert (np.diff(v) <= 0).all(), s


# ------------------------------------------------------------------ oracle vs brute force

def _x(seed, v, j):
    return sampling.mix64((sampling.mix64((seed ^ v) & M64) + j) & M64)


def _widen(p):
    p = np.asarray(p)
    if p.dtype == np.uint16:
        return (p.astype(np.uint32) << 16).view(np.float32).astype(np.float64)
    return p.astype(np.float64)


def _wkeys(seed, v, w):
    """bits(neglog(U_j) / w_j) for the eligible j, the division done by numpy in fp64."""
    js = [j for j in range(w.size) if 0 < w[j] < np.inf]
    u = np.array([((_x(seed, v, j) >> 11) + 1) * 2.0 ** -53 for j in js], np.float64)
    keys = (SEO.neglog(u) / w[js]).view(np.uint64) if js else np.zeros(0, np.uint64)
    return js, [int(k) for k in keys]


def brute_force(crow, col, val, dst, fanout, seed, prob=None, replace=False):
    rows = len(crow) - 1
    dst = [int(x) for x in dst]
    kc, kv, ke, row_len, invalid = [], [], [], [], 0
    w_all = None if prob is None else _widen(prob)
    for v in dst:
        if not (0 <= v < rows) or dst.count(v) != 1:
            invalid += 1
            row_len.append(0)
            continue
        b, e = int(crow[v]), int(crow[v + 1])
        deg = e - b
        if replace and fanout != -1:
            take = [(_x(seed, v, t) * deg) >> 64 for t in range(fanout if deg > 0 else 0)]
        elif prob is not None:
            js, keys = _wkeys(seed, v, w_all[b:e])
            k = len(js) if fanout == -1 else min(len(js), fanout)
            take = sorted(j for _, j in sorted(zip(keys, js))[:k])
        else:
            keys = [_x(seed, v, j) for j in range(deg)]
            k = deg if fanout == -1 else min(deg, fanout)
            take = sorted(sorted(range(deg), key=lambda j: (keys[j], j))[:k])
        n = 0
        for j in take:
            c = int(col[b + j])
            if 0 <= c < rows:
                kc.append(c)
                kv.append(None if val is None else val[b + j])
                ke.append(b + j)
                n += 1
        row_len.append(n)
    tail = sorted(set(kc) - set(dst))
    local = [dst.index(c) if c in dst else len(dst) + tail.index(c) for c in kc]
    blk_crow = np.concatenate([[0], np.cumsum(row_len)]).astype(np.int64)
    vals = None if val is None else np.array(kv, dtype=np.asarray(val).dtype)
    return blk_crow, np.array(local, np.int64), vals, np.array(ke, np.int64), np.array(dst + tail, np.int64), invalid


def _graph(rng, rows, max_deg):
    lens = rng.integers(0, max_deg + 1, rows)
    lens[rng.integers(0, rows, max(1, rows // 8))] = 0
    crow = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    col = rng.integers(0, rows, int(crow[-1]))
    if col.size > 4:
        col[1::5] = col[0:-1:5][: col[1::5].size]                   # repeated columns
        pick = rng.integers(0, col.size, max(1, col.size // 10))
        col[pick] = np.where(rng.random(pick.size) < 0.5, -1, rows)  # out-of-range columns
    val = rng.standard_normal(col.size).astype(np.float32)
    return crow, col, val


def _weights(rng, n, kind):
    """Graded positive weights with zeros, negatives, NaN and +-inf mixed in; fp32 or bf16 bits."""
    w = rng.exponential(1.0, n).astype(np.float32) * np.float32(10.0) ** rng.integers(-3, 4, n).astype(np.float32)
    special = np.array([0.0, -0.0, -1.5, np.nan, np.inf, -np.inf, 1e-40], np.float32)
    pick = rng.random(n) < 0.3
    w[pick] = special[rng.integers(0, special.size, int(pick.sum()))]
    return O.f32_to_bf16(w) if kind == "bf16" else w


MODES = ["weighted_fp32", "weighted_bf16", "replace", "uniform"]


@pytest.mark.parametrize("fanout", [0, 1, 3, -1])
@pytest.mark.parametrize("mode", MODES)
def test_oracle_matches_brute_force(mode, fanout):
    rng = np.random.default_rng([fanout + 1, MODES.index(mode), 77])
    for trial in range(6):
        rows = int(rng.integers(1, 40))
        crow, col, val = _graph(rng, rows, 9)
        prob = _weights(rng, col.size, mode.split("_")[1]) if mode.startswith("weighted") else None
        if trial % 3 == 1:
            val = O.f32_to_bf16(val)
        elif trial % 3 == 2:
            val = None
        dst = rng.permutation(rows)[: int(rng.integers(0, rows + 1))]
        seed = int(rng.integers(0, 2 ** 63)) * 2 + trial
        replace = mode == "replace"
        want = brute_force(crow, col, val, dst, fanout, seed, prob, replace)
        bc, bcol, bval, beid, src, counts = SEO.sample_neighbors_ex(crow, col, val, dst, fanout, seed, prob, replace)
        assert np.array_equal(bc, want[0]) and np.array_equal(bcol, want[1]) and np.array_equal(src, want[4])
        assert np.array_equal(beid, want[3])
        assert counts.tolist() == [bc[-1], src.size, 0]
        assert np.array_equal(col[beid], src[bcol])                        # the edge-id invariants
        if val is not None:
            assert np.array_equal(bval.view(np.uint8), want[2].view(np.uint8))
            assert np.array_equal(np.asarray(val)[beid].view(np.uint8), bval.view(np.uint8))


def test_weighted_rows_with_few_eligible_entries():
    """npos < fanout: every eligible entry is taken, no ineligible one; a row of ineligible weights
    gives an empty row."""
    crow = np.array([0, 5, 8, 8], np.int64)
    col = np.array([0, 1, 2, 0, 1, 2, 0, 1], np.int64)
    prob = np.array([0.0, 2.0, np.nan, -1.0, 3.0, 0.0, -np.inf, np.inf], np.float32)
    bc, bcol, _, beid, src, counts = SEO.sample_neighbors_ex(crow, col, None, [0, 1, 2], 3, 9, prob)
    assert np.diff(bc).tolist() == [2, 0, 0] and beid.tolist() == [1, 4]
    assert counts[2] == 0 and src[bcol].tolist() == [1, 1]


def test_replace_draws_use_python_int_mulhi():
    crow = np.array([0, 7, 7, 10], np.int64)
    col = np.array([0, 1, 2, 0, 1, 2, 0, 2, 1, 0], np.int64)
    seed, fanout = 0xDEADBEEF12345, 25
    _, bcol, _, beid, src, _ = SEO.sample_neighbors_ex(crow, col, None, [0, 1, 2], fanout, seed, None, True)
    want = [(_x(seed, 0, t) * 7 >> 64) for t in range(fanout)] + [7 + (_x(seed, 2, t) * 3 >> 64) for t in range(fanout)]
    assert beid.tolist() == want
    assert np.array_equal(col[beid], src[bcol])


def test_weighted_key_is_bits_of_neglog_over_weight():
    rng = np.random.default_rng(3)
    for _ in range(200):
        seed, v, j = int(rng.integers(0, 2 ** 63)), int(rng.integers(0, 2 ** 31)), int(rng.integers(0, 10 ** 6))
        w = float(rng.exponential(2.0))
        u = ((_x(seed, v, j) >> 11) + 1) * 2.0 ** -53
        assert SEO.weighted_key(seed, v, j, w) == int(np.array([SEO.neglog(np.array([u]))[0] / w]).view(np.uint64)[0])
    for bad in (0.0, -0.0, -2.0, float("nan"), float("inf"), float("-inf")):
        assert SEO.weighted_key(1, 2, 3, bad) == M64


# ------------------------------------------------------------------ C ABI without a GPU

def _opts(flags=0, prob_dtype=0, prob=None):
    return ctypes.byref(_lib.SampleOptsStruct(flags, prob_dtype, prob))


def test_sample_ex_abi_validation_without_gpu():
    L = _lib.lib()
    crow = np.zeros(5, np.int32)
    dst = np.zeros(2, np.int32)
    buf = np.zeros(64, np.int64)
    p = buf.ctypes.data
    eid_ws = L.ofspmm_sample_neighbors_ex_workspace_bytes(2, 8, _lib.DTYPE_INT32, _opts(_lib.SAMPLE_EDGE_IDS))
    A = _lib.CsrStruct(4, 4, 0, crow.ctypes.data, None, None, _lib.DTYPE_INT32, _lib.VAL_UNIT)

    def call(opts, blk_eid=None, cap=8, ws_bytes=eid_ws):
        return L.ofspmm_sample_neighbors_ex(ctypes.byref(A), opts, dst.ctypes.data, 2, 3, 1, cap, p, p, None, blk_eid,
                                            p, p, p, ws_bytes, None)

    assert call(_opts(4)) == 1                                                  # unknown flag bit
    assert call(_opts(1 << 31)) == 1
    assert call(_opts(_lib.SAMPLE_REPLACE, _lib.DTYPE_FLOAT, p)) == 1           # replace with prob
    assert call(_opts(0, _lib.DTYPE_INT32, p)) == 1                             # prob dtype not FLOAT / BF16
    assert call(_opts(0, 0, p)) == 1
    assert call(_opts(0), blk_eid=p) == 1                                       # blk_eid without EDGE_IDS
    assert call(None, blk_eid=p) == 1
    assert call(_opts(_lib.SAMPLE_REPLACE), blk_eid=p) == 1
    assert call(_opts(_lib.SAMPLE_EDGE_IDS)) == 1                               # EDGE_IDS without blk_eid
    assert call(_opts(_lib.SAMPLE_EDGE_IDS | _lib.SAMPLE_REPLACE)) == 1
    assert call(_opts(_lib.SAMPLE_EDGE_IDS), blk_eid=p, ws_bytes=eid_ws - 1) == 3   # workspace sized with EDGE_IDS
    assert L.ofspmm_sample_neighbors_ex(None, None, dst.ctypes.data, 2, 3, 1, 8, p, p, None, None, p, p, p,
                                        eid_ws, None) == 1


def test_sample_ex_workspace_query():
    L = _lib.lib()
    I64 = _lib.DTYPE_INT64
    q = L.ofspmm_sample_neighbors_ex_workspace_bytes
    base = L.ofspmm_sample_neighbors_workspace_bytes(1000, 25_000, I64)
    assert q(1000, 25_000, I64, None) == base == q(1000, 25_000, I64, _opts())
    # the options that do not add a buffer keep the size; prob is not read by the query
    assert q(1000, 25_000, I64, _opts(_lib.SAMPLE_REPLACE)) == base
    assert q(1000, 25_000, I64, _opts(0, _lib.DTYPE_FLOAT, 0x1000)) == base
    assert q(1000, 25_000, I64, _opts(0, _lib.DTYPE_BFLOAT16, 0x1000)) == base
    e = q(1000, 25_000, I64, _opts(_lib.SAMPLE_EDGE_IDS))
    assert e >= base + 8 * 25_000
    assert q(1000, 25_000, _lib.DTYPE_INT32, _opts(_lib.SAMPLE_EDGE_IDS)) == e
    assert q(0, 0, I64, _opts(_lib.SAMPLE_EDGE_IDS)) > 0
    # bad arguments: 0
    assert q(-1, 8, I64, None) == 0 and q(2, -1, I64, None) == 0 and q(2, 8, 9, None) == 0
    assert q(2, 8, I64, _opts(4)) == 0
    assert q(2, 8, I64, _opts(_lib.SAMPLE_REPLACE, _lib.DTYPE_FLOAT, 0x1000)) == 0
    assert q(2, 8, I64, _opts(0, _lib.DTYPE_INT64, 0x1000)) == 0
    # batch-sized: linear in num_dst + cap, independent of any graph
    e2 = q(2000, 50_000, I64, _opts(_lib.SAMPLE_EDGE_IDS))
    e0 = q(0, 0, I64, _opts(_lib.SAMPLE_EDGE_IDS))
    assert e2 - e0 <= 2.2 * (e - e0)


def test_ops_and_sampling_reject_cpu_tensors_and_bad_options():
    crow = torch.tensor([0, 1, 2], dtype=torch.int32)
    col = torch.tensor([1, 0], dtype=torch.int32)
    w = torch.tensor([1.0, 2.0])
    d = torch.tensor([0])
    with pytest.raises(ofs.OpInferError, match="device type cpu"):
        ofs.sample_neighbors(crow, col, None, 2, 2, d, 1, 0, prob=w)
    with pytest.raises(ofs.OpInferError, match="device type cpu"):
        ofs.sample_neighbors(crow, col, None, 2, 2, d, 1, 0, replace=True, return_eid=True)
    with pytest.raises(ofs.OpInferError, match="with replacement"):
        ofs.sample_neighbors(crow, col, None, 2, 2, d, 1, 0, prob=w, replace=True)
    with pytest.raises(ofs.OpInferError, match="nnz float32 / bfloat16 weights"):
        ofs.sample_neighbors(crow, col, None, 2, 2, d, 1, 0, prob=torch.ones(3))
    with pytest.raises(ofs.OpInferError, match="nnz float32 / bfloat16 weights"):
        ofs.sample_neighbors(crow, col, None, 2, 2, d, 1, 0, prob=torch.ones(2, dtype=torch.float64))
    P = G.CsrMatrix(crow, col, None, 2, 2)
    with pytest.raises(ofs.OpInferError, match="device type cpu"):
        ofs.sample_blocks(P, d, [1], 0, prob=w, edge_ids=True)
    with pytest.raises(ofs.OpInferError, match="with replacement"):
        ofs.sample_blocks(P, d, [1], 0, prob=w, replace=True)
    assert sampling.Block(P, d).eid is None
