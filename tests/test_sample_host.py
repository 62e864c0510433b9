"""CPU tests of neighbour sampling: the oracle against a brute-force numpy restatement of the
definition in include/ofspmm.h, the key function against ``graphs._mix64_``, and the C ABI's
argument validation and workspace query, none of which needs a GPU."""
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
import _sample_oracle as SO  # noqa: E402

_lib = import_module("of-spmm_b200._lib")
sampling = import_module("of-spmm_b200.sampling")
G = ofs.graphs
U64 = 2 ** 64


def _signed(x: int) -> int:
    x %= U64
    return x - U64 if x >= 2 ** 63 else x


def _keys(seed: int, v: int, deg: int) -> np.ndarray:
    """key(s, v, j) for j < deg through graphs._mix64_ (int64 bits), as uint64."""
    h0 = G._mix64_(torch.tensor([_signed(seed ^ v)], dtype=torch.int64))
    k = G._mix64_(h0 + torch.arange(deg, dtype=torch.int64))
    return k.numpy().view(np.uint64)


def brute_force(crow, col, val, dst, fanout, seed):
    rows = len(crow) - 1
    dst = [int(x) for x in dst]
    kept_cols, kept_vals, row_len, invalid = [], [], [], 0
    for v in dst:
        if not (0 <= v < rows) or dst.count(v) != 1:
            invalid += 1
            row_len.append(0)
            continue
        b, e = int(crow[v]), int(crow[v + 1])
        deg = e - b
        k = deg if fanout == -1 else min(deg, fanout)
        keys = _keys(seed, v, deg)
        order = sorted(range(deg), key=lambda j: (int(keys[j]), j))[:k]
        n = 0
        for j in sorted(order):
            c = int(col[b + j])
            if 0 <= c < rows:
                kept_cols.append(c)
                kept_vals.append(None if val is None else val[b + j])
                n += 1
        row_len.append(n)
    tail = sorted(set(kept_cols) - set(dst))
    src = dst + tail
    local = [dst.index(c) if c in dst else len(dst) + tail.index(c) for c in kept_cols]
    blk_crow = np.concatenate([[0], np.cumsum(row_len)]).astype(np.int64)
    vals = None if val is None else np.array(kept_vals, dtype=np.asarray(val).dtype)
    return blk_crow, np.array(local, np.int64), vals, np.array(src, np.int64), invalid


def _graph(rng, rows, max_deg, bad_cols=False, dup_cols=False):
    lens = rng.integers(0, max_deg + 1, rows)
    lens[rng.integers(0, rows, max(1, rows // 8))] = 0          # empty rows
    crow = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    col = rng.integers(0, rows, int(crow[-1]))
    if dup_cols and col.size > 4:
        col[1::5] = col[0:-1:5][: col[1::5].size]                 # repeated columns inside rows
    if bad_cols and col.size > 4:
        pick = rng.integers(0, col.size, max(1, col.size // 10))
        col[pick] = np.where(rng.random(pick.size) < 0.5, -1 - rng.integers(0, 3, pick.size), rows + rng.integers(0, 3, pick.size))
    val = rng.standard_normal(col.size).astype(np.float32)
    return crow, col, val


CASES = ["plain", "bad_cols", "dup_cols", "pattern", "bf16"]


@pytest.mark.parametrize("fanout", [0, 1, 3, -1])
@pytest.mark.parametrize("case", CASES)
def test_oracle_matches_brute_force(fanout, case):
    rng = np.random.default_rng([fanout + 1, CASES.index(case)])
    for trial in range(6):
        rows = int(rng.integers(1, 40))
        crow, col, val = _graph(rng, rows, 8, bad_cols=case == "bad_cols", dup_cols=case == "dup_cols")
        if case == "pattern":
            val = None
        elif case == "bf16":
            val = O.f32_to_bf16(val)
        dst = rng.permutation(rows)[: int(rng.integers(0, rows + 1))]    # unsorted, distinct
        seed = int(rng.integers(0, 2 ** 63)) * 2 + trial
        want = brute_force(crow, col, val, dst, fanout, seed)
        bc, bcol, bval, src, counts = SO.sample_neighbors(crow, col, val, dst, fanout, seed)
        assert np.array_equal(bc, want[0]) and np.array_equal(bcol, want[1]) and np.array_equal(src, want[3])
        assert counts.tolist() == [bc[-1], src.size, 0]
        if val is not None:
            assert bval.dtype == want[2].dtype and np.array_equal(bval.view(np.uint8), want[2].view(np.uint8))


def test_oracle_row_lengths_around_k():
    """Rows of deg < k, = k and = k + 1 (k = 3): the first two are copied whole, the last loses one."""
    crow = np.array([0, 2, 5, 9, 9], np.int64)
    col = np.array([1, 2, 0, 1, 3, 0, 1, 2, 3], np.int64)
    bc, bcol, _, src, counts = SO.sample_neighbors(crow, col, None, [0, 1, 2, 3], 3, 17)
    assert np.diff(bc).tolist() == [2, 3, 3, 0]
    assert src.tolist() == [0, 1, 2, 3] and counts[2] == 0
    want = brute_force(crow, col, None, [0, 1, 2, 3], 3, 17)
    assert np.array_equal(bcol, want[1])


def test_oracle_counts_invalid_destinations():
    crow, col, val = _graph(np.random.default_rng(3), 20, 6)
    dst = [4, 25, 7, 4, -1, 9]          # 25 and -1 out of range; 4 repeated (both occurrences)
    bc, bcol, _, src, counts = SO.sample_neighbors(crow, col, val, dst, 2, 5)
    assert counts[2] == 4
    assert np.diff(bc)[[0, 1, 3, 4]].tolist() == [0, 0, 0, 0]
    assert src[:6].tolist() == dst
    want = brute_force(crow, col, val, dst, 2, 5)
    assert want[4] == 4 and np.array_equal(bc, want[0]) and np.array_equal(bcol, want[1])


def test_key_matches_graphs_mix64():
    rng = np.random.default_rng(11)
    for _ in range(50):
        seed = int(rng.integers(0, 2 ** 63)) * 2 + int(rng.integers(0, 2))
        v = int(rng.integers(0, 2 ** 40))
        deg = int(rng.integers(1, 40))
        keys = _keys(seed, v, deg)
        assert [SO.sample_key(seed, v, j) for j in range(deg)] == [int(k) for k in keys]
        assert sampling.mix64(seed) == int(G._mix64_(torch.tensor([_signed(seed)])).numpy().view(np.uint64)[0])
    assert sampling.hop_seed(7, 2) == sampling.mix64(9)


# ------------------------------------------------------------------ C ABI without a GPU

def _csr(rows=4, cols=4, nnz=0, idx=_lib.DTYPE_INT32, vd=_lib.VAL_UNIT, crow=None):
    return _lib.CsrStruct(rows, cols, nnz, crow, None, None, idx, vd)


def test_sample_abi_validation_without_gpu():
    L = _lib.lib()
    crow = np.zeros(5, np.int32)
    dst = np.zeros(2, np.int32)
    buf = np.zeros(64, np.int64)
    p = buf.ctypes.data
    ws_need = L.ofspmm_sample_neighbors_workspace_bytes(2, 8, _lib.DTYPE_INT32)
    A = _csr(crow=crow.ctypes.data)

    def call(A_ref, fanout=3, cap=8, blk_crow=p, blk_col=p, blk_val=None, src=p, counts=p, ws=p, ws_bytes=ws_need,
             dstp=dst.ctypes.data, num_dst=2):
        return L.ofspmm_sample_neighbors(A_ref, dstp, num_dst, fanout, 1, cap, blk_crow, blk_col, blk_val, src,
                                         counts, ws, ws_bytes, None)

    assert call(None) == 1                                        # null csr
    assert call(ctypes.byref(A), blk_crow=None) == 1              # null outputs
    assert call(ctypes.byref(A), counts=None) == 1
    assert call(ctypes.byref(A), src=None) == 1
    assert call(ctypes.byref(A), blk_col=None) == 1
    assert call(ctypes.byref(A), dstp=None) == 1
    assert call(ctypes.byref(A), blk_val=p) == 1                  # values array for a pattern matrix
    Af = _csr(crow=crow.ctypes.data, vd=_lib.DTYPE_FLOAT)
    assert call(ctypes.byref(Af), blk_val=None) == 1              # ... and none for a valued one
    Ar = _csr(rows=4, cols=5, crow=crow.ctypes.data)
    assert call(ctypes.byref(Ar)) == 1                            # rows != cols
    assert call(ctypes.byref(A), fanout=-2) == 1
    assert call(ctypes.byref(A), num_dst=-1) == 1
    assert call(ctypes.byref(A), cap=2 ** 31 - 1) == 5            # cap >= 2^31 - 1
    assert call(ctypes.byref(A), ws_bytes=ws_need - 1) == 3       # workspace smaller than the query
    assert call(ctypes.byref(A), ws=None) == 3
    Ab = _csr(crow=crow.ctypes.data, idx=9)
    assert call(ctypes.byref(Ab)) == 2                            # not an index dtype
    assert L.ofspmm_sample_neighbors_workspace_bytes(-1, 8, _lib.DTYPE_INT32) == 0
    assert L.ofspmm_sample_neighbors_workspace_bytes(2, 8, 9) == 0


def test_sample_workspace_scales_with_batch_not_graph():
    """The query takes no size of A: a batch of 1e5 destinations x fanout 25 needs the same bytes for
    a papers100M-sized graph as for a small one, and grows linearly with num_dst + cap."""
    L = _lib.lib()
    w1 = L.ofspmm_sample_neighbors_workspace_bytes(100_000, 2_500_000, _lib.DTYPE_INT64)
    w2 = L.ofspmm_sample_neighbors_workspace_bytes(200_000, 5_000_000, _lib.DTYPE_INT64)
    w0 = L.ofspmm_sample_neighbors_workspace_bytes(0, 0, _lib.DTYPE_INT64)
    assert 0 < w0 < w1 < w2
    assert w1 < 200 * (100_000 + 2_500_000)          # bytes per destination / slot, not per row of A
    assert w2 - w0 <= 2.2 * (w1 - w0)
    assert L.ofspmm_sample_neighbors_workspace_bytes(100_000, 2_500_000, _lib.DTYPE_INT32) == w1


def test_sample_neighbors_rejects_cpu_tensors_and_bad_arguments():
    crow = torch.tensor([0, 1, 2], dtype=torch.int32)
    col = torch.tensor([1, 0], dtype=torch.int32)
    with pytest.raises(ofs.OpInferError, match="device type cpu"):
        ofs.sample_neighbors(crow, col, None, 2, 2, torch.tensor([0]), 1, 0)
    with pytest.raises(ofs.OpInferError, match="device type cpu"):
        ofs.sample_blocks(G.CsrMatrix(crow, col, None, 2, 2), torch.tensor([0]), [1], 0)
