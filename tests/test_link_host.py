"""CPU tests of the link-prediction pieces: the oracle (tests/c/sample_link_oracle.c) against a
brute-force Python restatement of the definitions in include/ofspmm.h (sampling with an exclusion
list in the three modes, negative sampling, edge lookup), the C ABI's validation of the new entry
points, flag and fields, the workspace query with exclusion, and the autograd wiring of
``edge_score`` and the assembly of a ``LinkBatch`` on CPU stand-ins; none needs a GPU."""
import ctypes
import os
import sys
from importlib import import_module

import numpy as np
import pytest
import torch

import ofspmm_b200 as ofs

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import _sample_ext_oracle as SEO  # noqa: E402
import _sample_link_oracle as SLO  # noqa: E402

_lib = import_module("of-spmm_b200._lib")
sampling = import_module("of-spmm_b200.sampling")
F = import_module("of-spmm_b200.functional")
G = ofs.graphs
M64 = (1 << 64) - 1


def _x(seed, v, j):
    return sampling.mix64((sampling.mix64((seed ^ v) & M64) + j) & M64)


def _graph(seed=4, rows=40):
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, 14, rows)
    lens[::7] = 0
    crow = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    col = np.concatenate([np.sort(rng.choice(rows, int(n), replace=False)) for n in lens] + [np.zeros(0, int)])
    w = rng.exponential(1.0, col.size).astype(np.float32)
    w[rng.random(col.size) < 0.2] = 0.0
    return crow, col.astype(np.int64), w


# ------------------------------------------------------------------ oracle vs brute force

def _brute_take(v, b, deg, seed, excl, w=None, replace=False, fanout=-1):
    excl = set(int(e) for e in excl)
    elig = [j for j in range(deg) if b + j not in excl]
    if replace and fanout != -1:
        return [elig[(_x(seed, v, t) * len(elig)) >> 64] for t in range(fanout if elig else 0)]
    if w is not None:
        js = [j for j in elig if 0 < w[j] < np.inf]
        keys = [SEO.weighted_key(seed, v, j, float(w[j])) for j in js]
    else:
        js = elig
        keys = [_x(seed, v, j) for j in js]
    k = len(js) if fanout == -1 else min(len(js), fanout)
    return sorted(j for _, j in sorted(zip(keys, js))[:k])


@pytest.mark.parametrize("mode", ["uniform", "weighted", "replace"])
@pytest.mark.parametrize("fanout", [-1, 0, 1, 3, 25])
def test_take_row_matches_brute_force(mode, fanout):
    crow, col, w = _graph()
    rng = np.random.default_rng(fanout + 7)
    excl = np.unique(rng.choice(col.size, col.size // 3, replace=False))
    excl = np.unique(np.concatenate([excl, np.arange(crow[3], crow[4]), [0, col.size - 1]]))   # a whole row
    seed = 0xC0FFEE + fanout
    for v in range(crow.size - 1):
        b, e = int(crow[v]), int(crow[v + 1])
        wr = w[b:e] if mode == "weighted" else None
        got = SLO.take_row(v, b, e - b, seed, excl, wr, mode == "replace", fanout)
        want = _brute_take(v, b, e - b, seed, excl, wr, mode == "replace", fanout)
        assert got.tolist() == want, (v, mode)
        assert not set((b + got).tolist()) & set(excl.tolist())


@pytest.mark.parametrize("mode", ["uniform", "weighted", "replace"])
def test_empty_exclusion_is_the_sampler_without_it(mode):
    """The oracle with an empty list equals sample_ext_oracle's (the definitions without exclusion)."""
    crow, col, w = _graph(seed=9)
    dst = np.array([5, 1, 2, 9, 30, 17])
    prob = w if mode == "weighted" else None
    a = SLO.sample_neighbors_excl(crow, col, None, dst, 3, 77, [], prob, mode == "replace")
    rc, rcol, _, reid, rsrc, _ = SEO.sample_neighbors_ex(crow, col, None, dst, 3, 77, prob, mode == "replace")
    assert np.array_equal(a[0], rc) and np.array_equal(a[1], rcol) and np.array_equal(a[3], reid)
    assert np.array_equal(a[4], rsrc)


def test_negative_sample_oracle_matches_brute_force():
    crow, col, _ = _graph(seed=11)
    rows = crow.size - 1
    src = np.array([3, 3, 0, 8, -1, rows, 12])
    k, seed, trials = 4, 0xABCDEF, 3
    edges = {(u, int(c)) for u in range(rows) for c in col[crow[u]:crow[u + 1]]}
    for ex_e in (False, True):
        for ex_s in (False, True):
            neg, counts = SLO.negative_sample(crow, col, rows, src, k, seed, ex_e, ex_s, trials)
            want, failed = [], 0
            for i, u in enumerate(src):
                for t in range(k):
                    c = -1
                    for r in range(trials if 0 <= u < rows else 0):
                        p = (sampling.mix64((sampling.mix64((seed ^ i) & M64) + r * k + t) & M64) * rows) >> 64
                        if (ex_s and p == u) or (ex_e and (int(u), p) in edges):
                            continue
                        c = p
                        break
                    want.append(c)
                    failed += c < 0
            assert neg.ravel().tolist() == want
            assert counts.tolist() == [failed, 2]
    neg, _ = SLO.negative_sample(crow, col, rows, src, k, seed)
    assert neg[0].tolist() != neg[1].tolist()   # keyed by position: a repeated source differs


def test_edge_ids_oracle_matches_dictionary():
    crow, col, _ = _graph(seed=13)
    rows = crow.size - 1
    first = {}
    for u in range(rows):
        for p in range(crow[u], crow[u + 1]):
            first.setdefault((u, int(col[p])), p)
    rng = np.random.default_rng(2)
    u = np.concatenate([rng.integers(-2, rows + 2, 300), [c[0] for c in list(first)[:50]]])
    v = np.concatenate([rng.integers(-2, rows + 2, 300), [c[1] for c in list(first)[:50]]])
    got = SLO.edge_ids(crow, col, u, v)
    assert got.tolist() == [first.get((int(a), int(b)), -1) for a, b in zip(u, v)]
    assert (got[300:] >= 0).all()


# ------------------------------------------------------------------ C ABI without a GPU

def _sopts(flags=0, exclude=None, num_exclude=0):
    return ctypes.byref(_lib.SampleOptsStruct(flags, 0, None, exclude, num_exclude))


def test_sample_exclude_abi_validation_and_workspace():
    L = _lib.lib()
    crow = np.zeros(5, np.int32)
    dst = np.zeros(2, np.int32)
    buf = np.zeros(64, np.int64)
    p = buf.ctypes.data
    ws = L.ofspmm_sample_neighbors_ex_workspace_bytes(2, 8, _lib.DTYPE_INT32, None)
    A = _lib.CsrStruct(4, 4, 0, crow.ctypes.data, None, None, _lib.DTYPE_INT32, _lib.VAL_UNIT)

    def call(opts):
        return L.ofspmm_sample_neighbors_ex(ctypes.byref(A), opts, dst.ctypes.data, 2, 3, 1, 8, p, p, None, None,
                                            p, p, p, ws, None)

    X = _lib.SAMPLE_EXCLUDE
    assert X == 8
    assert call(_sopts(4)) == 1 and call(_sopts(16)) == 1 and call(_sopts(X | 16, p, 1)) == 1   # unknown flags
    assert call(_sopts(X, None, 3)) == 1                 # NULL list with entries
    assert call(_sopts(X, p, -1)) == 1                   # negative size
    assert call(_sopts(X | _lib.SAMPLE_REPLACE, None, -5)) == 1
    q = L.ofspmm_sample_neighbors_ex_workspace_bytes
    for idt in (_lib.DTYPE_INT32, _lib.DTYPE_INT64):
        for nd, cap in ((0, 0), (2, 8), (1000, 25_000)):
            for fl in (0, _lib.SAMPLE_REPLACE, _lib.SAMPLE_EDGE_IDS):
                base = q(nd, cap, idt, _sopts(fl))
                assert base > 0
                assert q(nd, cap, idt, _sopts(fl | X, p, 123)) == base == q(nd, cap, idt, _sopts(fl | X, None, 0))
                # the fields are not read without the flag
                assert q(nd, cap, idt, _sopts(fl, None, -7)) == base
    assert q(2, 8, _lib.DTYPE_INT32, _sopts(X, None, 3)) == 0 and q(2, 8, _lib.DTYPE_INT32, _sopts(X, p, -1)) == 0


def test_edge_ids_and_negative_sample_abi_validation():
    L = _lib.lib()
    crow = np.zeros(5, np.int64)
    ids = np.zeros(4, np.int64)
    cnt = np.zeros(2, np.int64)
    sq = _lib.CsrStruct(4, 4, 0, crow.ctypes.data, None, None, _lib.DTYPE_INT64, _lib.VAL_UNIT)
    rect = _lib.CsrStruct(4, 6, 0, crow.ctypes.data, None, None, _lib.DTYPE_INT64, _lib.VAL_UNIT)
    bad_idx = _lib.CsrStruct(4, 4, 0, crow.ctypes.data, None, None, _lib.DTYPE_FLOAT, _lib.VAL_UNIT)
    p = ids.ctypes.data

    def neg(A=sq, n=4, k=2, flags=3, trials=8, src=p, out=p, counts=cnt.ctypes.data):
        return L.ofspmm_negative_sample(ctypes.byref(A) if A is not None else None, src, n, k, 1, flags, trials, out,
                                        counts, None)

    assert neg(trials=0) == 1 and neg(trials=-3) == 1          # max_trials < 1
    assert neg(k=-1) == 1                                      # k < 0
    assert neg(flags=4) == 1 and neg(flags=0x80000000) == 1    # unknown flags
    assert neg(A=rect, flags=2) == 1 and neg(A=rect, flags=3) == 1   # EXCLUDE_SELF on a rectangular A
    assert neg(n=-1) == 1 and neg(counts=None) == 1 and neg(src=None) == 1 and neg(out=None) == 1
    assert neg(A=None) == 1 and neg(A=bad_idx) == 2
    assert neg(n=1 << 40, k=1 << 30) == 5                      # num_src * k slots overflow

    def eids(A=sq, n=4, u=p, v=p, out=p):
        return L.ofspmm_edge_ids(ctypes.byref(A) if A is not None else None, u, v, n, out, None)

    assert eids(n=-1) == 1 and eids(u=None) == 1 and eids(v=None) == 1 and eids(out=None) == 1
    assert eids(A=None) == 1 and eids(A=bad_idx) == 2
    assert eids(n=0, u=None, v=None, out=None) == 0            # nothing to do: no launch, no device


def test_python_link_ops_reject_cpu_tensors_and_bad_arguments():
    crow = torch.tensor([0, 1, 2], dtype=torch.int32)
    col = torch.tensor([1, 0], dtype=torch.int32)
    s = torch.tensor([0, 1])
    with pytest.raises(ofs.OpInferError, match="device type cpu"):
        ofs.edge_ids(crow, col, 2, 2, s, s)
    with pytest.raises(ofs.OpInferError, match="device type cpu"):
        ofs.negative_sample(crow, col, 2, 2, s, 3, 0)
    with pytest.raises(ofs.OpInferError, match="device type cpu"):
        ofs.sample_neighbors(crow, col, None, 2, 2, s, 1, 0, exclude_eid=torch.tensor([0]))
    with pytest.raises(ValueError, match="exclude must be"):
        ofs.sample_link_batch(G.CsrMatrix(crow, col, None, 2, 2), torch.tensor([0]), 1, [2], 0, exclude="both")


# ------------------------------------------------------------------ edge_score wiring and LinkBatch assembly

class _DenseKernels:
    """CPU stand-in for functional.OpsKernels: the pair matrix as a dense matrix with repeated entries
    summed, dense torch arithmetic."""

    def __init__(self, rows_of):
        self.rows_of = rows_of
        self.calls = []

    def _dense(self, a_col, a_val, m, k):
        return torch.zeros(m, k, dtype=a_val.dtype).index_put((self.rows_of, a_col.long()), a_val, accumulate=True)

    def fwd(self, a_crow, a_col, a_val, b, m, k, bias, relu, plan):
        self.calls.append("fwd")
        return self._dense(a_col, a_val, m, k) @ b

    def grad_b(self, a_crow, a_col, a_val, dy, m, k, plan):
        self.calls.append("grad_b")
        return self._dense(a_col, a_val, m, k).t() @ dy

    def sddmm(self, a_crow, a_col, dy, b, m, k, val_dtype, plan):
        self.calls.append("sddmm")
        return (dy[self.rows_of] * b[a_col.long()]).sum(1).to(val_dtype)


def test_edge_score_autograd_wiring_cpu():
    torch.manual_seed(0)
    crow = torch.tensor([0, 3, 3, 5, 9], dtype=torch.int32)           # row 1: every negative failed
    col = torch.tensor([2, 0, 0, 1, 4, 3, 3, 3, 0], dtype=torch.int32)  # repeats in rows 0 and 3
    rows_of = torch.repeat_interleave(torch.arange(4), (crow[1:] - crow[:-1]).long())
    hr = torch.randn(4, 6, dtype=torch.float64, requires_grad=True)
    hc = torch.randn(5, 6, dtype=torch.float64, requires_grad=True)
    K = _DenseKernels(rows_of)
    s = F.edge_score(crow, col, hr, hc, 4, 5, kernels=K)
    w = torch.randn(s.shape, dtype=torch.float64)
    (s * w).sum().backward()
    assert K.calls == ["sddmm", "fwd", "grad_b"]
    hr2, hc2 = hr.detach().clone().requires_grad_(), hc.detach().clone().requires_grad_()
    ref = (hr2[rows_of] * hc2[col.long()]).sum(1)
    (ref * w).sum().backward()
    assert torch.allclose(s, ref) and torch.allclose(hr.grad, hr2.grad) and torch.allclose(hc.grad, hc2.grad)
    # only the inputs that need a gradient get one
    K2 = _DenseKernels(rows_of)
    F.edge_score(crow, col, hr.detach(), hc, 4, 5, kernels=K2).sum().backward()
    assert K2.calls == ["sddmm", "grad_b"]
    with pytest.raises(ofs.OpInferError):
        F.edge_score(crow, col, hr[:3], hc, 4, 5, kernels=K)


def test_link_pairs_assembly_cpu():
    u = torch.tensor([7, 2, 7, 4])
    v = torch.tensor([3, 9, 3, 4])
    neg = torch.tensor([[1, -1, 9], [-1, -1, -1], [5, 5, -1], [0, 2, 8]])
    seeds, pair, src_local, labels = sampling.link_pairs(u, v, neg)
    assert seeds.tolist() == [0, 1, 2, 3, 4, 5, 7, 8, 9]
    assert pair.crow.dtype == torch.int32 and pair.col.dtype == torch.int32 and pair.val is None
    assert pair.crow.tolist() == [0, 3, 4, 7, 11] and (pair.rows, pair.cols) == (4, 9)
    got = seeds[pair.col.long()].tolist()
    assert got == [3, 1, 9, 9, 3, 5, 5, 4, 0, 2, 8]
    assert labels.tolist() == [1, 0, 0, 1, 1, 0, 0, 1, 0, 0, 0]
    assert seeds[src_local].tolist() == u.tolist()
    # k = 0: one entry per row, the positive
    seeds, pair, src_local, labels = sampling.link_pairs(u, v, neg[:, :0])
    assert pair.crow.tolist() == [0, 1, 2, 3, 4] and labels.tolist() == [1, 1, 1, 1]
    assert seeds.tolist() == [2, 3, 4, 7, 9]
