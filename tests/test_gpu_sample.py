"""GPU tests of device neighbour sampling (``ofspmm_sample_neighbors``, ``ops.sample_neighbors``,
``sampling.sample_blocks``): bit-exact against the CPU oracle over index / value dtypes and fanouts
(hub rows included, so the multi-pass selection and the whole-CTA path run), structural properties
that need no oracle, determinism, uniformity, the C-ABI contract (CUDA-graph replay, capacity,
invalid destinations, empty batches), the 2^31-non-zero matrix, and 2-layer GraphSAGE on the blocks."""
import ctypes
import os
import sys
import gc
from importlib import import_module

import numpy as np
import pytest
import torch

import ofspmm_b200 as ofs
from oracle import oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import _sample_oracle as SO  # noqa: E402

pytestmark = pytest.mark.gpu

G = ofs.graphs
ops = import_module("of-spmm_b200.ops")
gcn = import_module("of-spmm_b200.gcn")
sampling = import_module("of-spmm_b200.sampling")
_lib = ofs._lib
DEV = "cuda:0"
HUB = 100_000


def _edge_graph(seed=7, rows=3000):
    """Rows of 0..60 entries (every 11th empty), rows of exactly 0..4 entries around small fanouts,
    one hub of 1e5 entries, rows of 4096 and 5000 entries (both sides of the whole-CTA threshold),
    repeated columns inside rows and columns outside [0, rows)."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, 61, rows)
    lens[::11] = 0
    lens[1:6] = [1, 2, 3, 4, 26]
    lens[17], lens[18], lens[19] = HUB, 4096, 5000
    crow = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    col = rng.integers(0, rows, int(crow[-1]))
    col[3::7] = col[2::7][: col[3::7].size]                       # repeated columns
    bad = rng.integers(0, col.size, col.size // 50)
    col[bad] = np.where(rng.random(bad.size) < 0.5, -1, rows + 1)  # out-of-range columns
    val = rng.standard_normal(col.size).astype(np.float32)
    dst = rng.permutation(rows)[:900]
    dst = np.concatenate([[17, 18, 19, 1, 2, 3, 4, 5, 0], dst[~np.isin(dst, [17, 18, 19, 1, 2, 3, 4, 5, 0])]])
    return crow, col, val, dst


@pytest.fixture(scope="module")
def EG():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return _edge_graph()


def _dev(crow, col, val, idx, vkind):
    t = torch.int32 if idx == "int32" else torch.int64
    c = torch.from_numpy(crow).to(t).to(DEV)
    k = torch.from_numpy(col).to(t).to(DEV)
    if vkind == "none":
        return c, k, None, None
    if vkind == "fp32":
        return c, k, torch.from_numpy(val).to(DEV), val
    bits = O.f32_to_bf16(val)
    return c, k, torch.from_numpy(bits.view(np.int16)).to(DEV).view(torch.bfloat16), bits


def _val_bits(t):
    if t is None:
        return None
    return t.cpu().view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32).numpy()


def _ref_bits(v):
    return None if v is None else v.view(np.int16 if v.dtype == np.uint16 else np.int32)


@pytest.mark.parametrize("fanout", [1, 3, 25, -1, HUB])
@pytest.mark.parametrize("vkind", ["fp32", "bf16", "none"])
@pytest.mark.parametrize("idx", ["int32", "int64"])
def test_bit_exact_vs_oracle(EG, idx, vkind, fanout):
    crow, col, val, dst = EG
    rows = crow.size - 1
    c, k, v, vref = _dev(crow, col, val, idx, vkind)
    d = torch.from_numpy(dst).to(DEV)
    seed = 0x9E3779B97F4A7C15 + 12345
    bc, bcol, bval, src = ops.sample_neighbors(c, k, v, rows, rows, d, fanout, seed)
    torch.cuda.synchronize()
    rc, rcol, rval, rsrc, counts = SO.sample_neighbors(crow, col, vref, dst, fanout, seed)
    assert counts[2] == 0
    assert bc.dtype == torch.int32 and bcol.dtype == torch.int32 and src.dtype == c.dtype
    assert np.array_equal(bc.cpu().numpy(), rc)
    assert np.array_equal(bcol.cpu().numpy(), rcol)
    assert np.array_equal(src.cpu().numpy(), rsrc)
    if vkind == "none":
        assert bval is None
    else:
        assert bval.dtype == v.dtype and np.array_equal(_val_bits(bval), _ref_bits(rval))


def test_structural_properties():
    A = G.reddit_like(256, seed=2).to(DEV)
    seeds = torch.randperm(A.rows, generator=torch.Generator().manual_seed(1))[:300].to(DEV).to(torch.int32)
    fanout = 7
    bc, bcol, _, src = ops.sample_neighbors(A.crow, A.col, None, A.rows, A.cols, seeds, fanout, 99)
    deg = (A.crow[1:] - A.crow[:-1]).long()[seeds.long()]
    assert torch.equal(torch.diff(bc).long(), torch.clamp(deg, max=fanout))     # no invalid columns here
    assert torch.equal(src[:seeds.numel()], seeds)
    tail = src[seeds.numel():]
    assert bool((tail[1:] > tail[:-1]).all())                                   # unique and ascending
    assert not bool(torch.isin(tail, seeds).any())
    glob = src.long()[bcol.long()]
    crow_h, col_h, bc_h, glob_h = A.crow.cpu().numpy(), A.col.cpu().numpy(), bc.cpu().numpy(), glob.cpu().numpy()
    used = np.zeros(src.numel(), bool)
    for i, v in enumerate(seeds.cpu().numpy()):
        row = set(col_h[crow_h[v]:crow_h[v + 1]].tolist())
        got = glob_h[bc_h[i]:bc_h[i + 1]]
        assert set(got.tolist()) <= row and len(set(got.tolist())) == got.size
        used[bcol.cpu().numpy()[bc_h[i]:bc_h[i + 1]]] = True
    assert used[seeds.numel():].all()                                          # every new source node is used


def test_determinism_and_seed_dependence(EG):
    crow, col, val, dst = EG
    rows = crow.size - 1
    c, k, v, _ = _dev(crow, col, val, "int64", "fp32")
    d = torch.from_numpy(dst).to(DEV)
    a = ops.sample_neighbors(c, k, v, rows, rows, d, 25, 1)
    b = ops.sample_neighbors(c, k, v, rows, rows, d, 25, 1)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    hub = torch.tensor([17], device=DEV)
    h1 = ops.sample_neighbors(c, k, v, rows, rows, hub, 25, 1)[1]
    h2 = ops.sample_neighbors(c, k, v, rows, rows, hub, 25, 2)[1]
    s1 = ops.sample_neighbors(c, k, v, rows, rows, hub, 25, 1)[3]
    s2 = ops.sample_neighbors(c, k, v, rows, rows, hub, 25, 2)[3]
    assert not torch.equal(s1[h1.long()], s2[h2.long()])


def test_uniformity_chi_square():
    """A 200-entry row sampled with k = 10 under seeds 0..3999: the per-position counts pass a
    chi-square test at the 0.999 quantile (199 degrees of freedom).  Fixed seeds: no flakes."""
    from scipy.stats import chi2
    deg, k, n = 200, 10, 4000
    crow = torch.tensor([0, deg] + [deg] * deg, dtype=torch.int32, device=DEV)
    col = torch.arange(1, deg + 1, dtype=torch.int32, device=DEV)        # position j holds node j + 1
    dst = torch.tensor([0], dtype=torch.int32, device=DEV)
    hits = torch.zeros(deg + 1, dtype=torch.int64, device=DEV)
    for s in range(n):
        bc, bcol, _, src = ops.sample_neighbors(crow, col, None, deg + 1, deg + 1, dst, k, s)
        assert bcol.numel() == k
        hits.index_add_(0, src.long()[bcol.long()], torch.ones(k, dtype=torch.int64, device=DEV))
    obs = hits[1:].cpu().numpy().astype(np.float64)
    exp = n * k / deg
    stat = float(((obs - exp) ** 2 / exp).sum())
    assert stat < chi2.ppf(0.999, deg - 1), stat


# ------------------------------------------------------------------ C ABI contract

class _Call:
    """Buffers of one ofspmm_sample_neighbors call, with a guard band after every output."""
    GUARD = 64

    def __init__(self, crow, col, val, rows, dst, fanout, seed, cap):
        self.keep = (crow, col, val, dst)
        self.A = ops._csr_struct(crow, col, val, rows, rows)
        self.dst, self.fanout, self.seed, self.cap = dst, fanout, seed, cap
        n, g = dst.numel(), self.GUARD
        self.blk_crow = torch.full((n + 1 + g,), -7, dtype=torch.int32, device=DEV)
        self.blk_col = torch.full((cap + g,), -7, dtype=torch.int32, device=DEV)
        self.blk_val = torch.full((cap + g,), -7.0, dtype=val.dtype, device=DEV) if val is not None else None
        self.src = torch.full((n + cap + g,), -7, dtype=crow.dtype, device=DEV)
        self.counts = torch.full((3,), -7, dtype=torch.int64, device=DEV)
        L = _lib.lib()
        self.ws_bytes = L.ofspmm_sample_neighbors_workspace_bytes(n, cap, ops._INDEX[crow.dtype])
        self.ws = torch.empty(self.ws_bytes, dtype=torch.uint8, device=DEV)

    def __call__(self):
        L = _lib.lib()
        return L.ofspmm_sample_neighbors(ctypes.byref(self.A), ops._ptr(self.dst), self.dst.numel(), self.fanout,
                                         self.seed, self.cap, self.blk_crow.data_ptr(), self.blk_col.data_ptr(),
                                         None if self.blk_val is None else self.blk_val.data_ptr(), self.src.data_ptr(),
                                         self.counts.data_ptr(), self.ws.data_ptr(), self.ws_bytes,
                                         torch.cuda.current_stream().cuda_stream)

    def outputs(self):
        """The written part of every output (sizes from counts), and counts."""
        n = self.dst.numel()
        nnz, num_src = (int(x) for x in self.counts[:2].tolist())
        outs = (self.blk_crow[:n + 1], self.blk_col[:nnz], None if self.blk_val is None else self.blk_val[:nnz],
                self.src[:num_src], self.counts)
        return [t.clone() for t in outs if t is not None]


def _ecg(EG, idx="int32"):
    crow, col, val, dst = EG
    c, k, v, _ = _dev(crow, col, val, idx, "fp32")
    return c, k, v, crow.size - 1, torch.from_numpy(dst).to(c.dtype).to(DEV)


def test_cuda_graph_replay_equals_eager(EG):
    c, k, v, rows, d = _ecg(EG)
    call = _Call(c, k, v, rows, d, 25, 77, d.numel() * 25)
    assert call() == 0
    torch.cuda.synchronize()
    eager = call.outputs()
    for t in (call.blk_crow, call.blk_col, call.blk_val, call.src, call.counts):
        t.fill_(-3)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            assert call() == 0
    torch.cuda.current_stream().wait_stream(s)
    for t in (call.blk_crow, call.blk_col, call.blk_val, call.src, call.counts):
        t.fill_(-5)
    graph.replay()
    torch.cuda.synchronize()
    for x, y in zip(eager, call.outputs()):
        assert torch.equal(x, y)
    assert int(eager[-1][0]) > 0


def test_capacity_exceeded_reports_size_and_writes_nothing_past_capacity(EG):
    c, k, v, rows, d = _ecg(EG)
    full = _Call(c, k, v, rows, d, 25, 3, d.numel() * 25)
    assert full() == 0
    torch.cuda.synchronize()
    deg = (c[1:] - c[:-1]).long()[d.long()]
    need = int(torch.clamp(deg, max=25).sum())
    small = _Call(c, k, v, rows, d, 25, 3, need - 1)
    assert small() == 0
    torch.cuda.synchronize()
    assert int(small.counts[0]) == need and int(small.counts[2]) == 0
    n, g, cap = d.numel(), _Call.GUARD, need - 1
    assert bool((small.blk_crow[n + 1:] == -7).all())
    assert bool((small.blk_col[cap:] == -7).all()) and bool((small.blk_val[cap:] == -7.0).all())
    assert bool((small.src[n + cap:] == -7).all())
    # the needed size is what a call with exactly that capacity fills
    exact = _Call(c, k, v, rows, d, 25, 3, need)
    assert exact() == 0
    torch.cuda.synchronize()
    assert torch.equal(exact.blk_crow[:n + 1], full.blk_crow[:n + 1])
    assert int(exact.counts[0]) == int(full.counts[0]) <= need


def test_invalid_destinations_are_counted(EG):
    crow, col, val, _ = EG
    rows = crow.size - 1
    c, k, v, _ = _dev(crow, col, val, "int64", "fp32")
    dst = np.array([5, rows, 17, 5, -3, 40, 17, 41], np.int64)     # out of range: 2; repeated: 5, 17 (x2 each)
    d = torch.from_numpy(dst).to(DEV)
    call = _Call(c, k, v, rows, d, 3, 11, dst.size * 3)
    assert call() == 0
    torch.cuda.synchronize()
    _, _, _, _, counts = SO.sample_neighbors(crow, col, val, dst, 3, 11)
    assert int(call.counts[2]) == counts[2] == 6
    bc = call.blk_crow[:dst.size + 1].cpu().numpy()
    assert (np.diff(bc)[[0, 1, 2, 3, 4, 6]] == 0).all()            # invalid ids read nothing
    assert bool((call.blk_crow[dst.size + 1:] == -7).all())
    with pytest.raises(ofs.OpInferError, match="out of range"):
        ops.sample_neighbors(c, k, v, rows, rows, d, 3, 11)


def test_empty_batch(EG):
    c, k, v, rows, _ = _ecg(EG)
    d = torch.empty(0, dtype=c.dtype, device=DEV)
    bc, bcol, bval, src = ops.sample_neighbors(c, k, v, rows, rows, d, 10, 0)
    assert bc.tolist() == [0] and bcol.numel() == 0 and bval.numel() == 0 and src.numel() == 0
    call = _Call(c, k, v, rows, d, 10, 0, 0)
    assert call() == 0
    torch.cuda.synchronize()
    assert call.counts.tolist() == [0, 0, 0] and int(call.blk_crow[0]) == 0
    assert bool((call.blk_crow[1:] == -7).all())


# ------------------------------------------------------------------ 2^31 + 2^25 non-zeros

@pytest.fixture(scope="module")
def WIDE():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    gc.collect()
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info(0)
    if free < 40e9:
        pytest.skip(f"needs 40 GB of free device memory for the 2^31-non-zero matrix, {free / 1e9:.0f} GB free")
    A = G.wide_csr(DEV)
    yield A, A.crow.cpu().numpy()
    del A
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


@pytest.mark.parametrize("fanout", [1, 25])
def test_wide_matrix_vs_oracle_on_its_rows(WIDE, fanout):
    A, crow_h = WIDE
    M = G.WIDE_M   # square view: the columns (< WIDE_K <= WIDE_M) index the same node set
    # the hub across 2^31, rows holding the out-of-range entries on both sides of 2^31, rows past
    # entry 2^31, rows long enough for the warp path's multi-pass selection, empty and 1-entry rows
    around = [int(np.searchsorted(crow_h, p, side="right")) - 1 for p, _ in G.WIDE_BAD]
    rows = [G.WIDE_HUB] + around + [G.WIDE_HUB + 1, G.WIDE_HUB + 2, M - 1, M - 2, 3, 5, 7, 1000, 2000, 98 * 97 + 3]
    rows += list(range(G.WIDE_HUB + 500, G.WIDE_HUB + 900))
    dst = np.array(list(dict.fromkeys(rows)), np.int64)
    d = torch.from_numpy(dst).to(DEV)
    seed = 2024
    bc, bcol, bval, src = ops.sample_neighbors(A.crow, A.col, A.val, M, M, d, fanout, seed)
    torch.cuda.synchronize()
    b, e = crow_h[dst], crow_h[dst + 1]
    seg_off = np.concatenate([[0], np.cumsum(e - b)])
    seg_col = np.concatenate([A.col[x:y].cpu().numpy() for x, y in zip(b, e)])
    seg_val = np.concatenate([A.val[x:y].cpu().numpy() for x, y in zip(b, e)])
    rc, rcol, rval, rsrc, counts = SO.sample_neighbors_rows(M, dst, seg_off, seg_col, seg_val, fanout, seed)
    assert counts[2] == 0 and int(e[0] - b[0]) == G.WIDE_HUB_LEN
    assert np.array_equal(bc.cpu().numpy(), rc)
    assert np.array_equal(bcol.cpu().numpy(), rcol)
    assert np.array_equal(src.cpu().numpy(), rsrc)
    assert np.array_equal(_val_bits(bval), _ref_bits(rval))


# ------------------------------------------------------------------ GraphSAGE on the blocks

def _sage_pair(in_dim=64, hidden=32, out_dim=16):
    l1 = gcn.SAGEConv(in_dim, hidden, activation="relu", seed=3, device=DEV)
    l2 = gcn.SAGEConv(hidden, out_dim, activation=None, seed=5, device=DEV)
    with torch.no_grad():
        l1.bias.uniform_(-0.5, 0.5, generator=torch.Generator(DEV).manual_seed(1))
        l2.bias.uniform_(-0.5, 0.5, generator=torch.Generator(DEV).manual_seed(2))
    return l1, l2


def test_full_fanout_blocks_equal_full_graph_sage():
    A = G.reddit_like(256, seed=2).to(DEV)
    P = G.CsrMatrix(A.crow, A.col, None, A.rows, A.cols)
    X = G.dense_operand(A.rows, 64, 8, DEV)
    seeds = torch.randperm(A.rows, generator=torch.Generator().manual_seed(4))[:128].to(DEV).to(torch.int32)
    l1, l2 = _sage_pair()
    with torch.no_grad():
        full = l2(P, l1(P, X))[seeds.long()]
        blocks = ofs.sample_blocks(P, seeds, [-1, -1], 5)
        assert torch.equal(blocks[-1].src_nodes[:seeds.numel()], seeds)
        h = X[blocks[0].src_nodes.long()]
        h = l1(blocks[0].adj, h)
        out = l2(blocks[1].adj, h)
    assert out.shape == full.shape
    assert torch.allclose(out, full, rtol=1e-4, atol=1e-4), float((out - full).abs().max())


def _dense_mean(adj):
    rows = torch.repeat_interleave(torch.arange(adj.rows, device=DEV), torch.diff(adj.crow).long())
    D = torch.zeros(adj.rows, adj.cols, dtype=torch.float64, device=DEV)
    D.index_put_((rows, adj.col.long()), torch.ones(rows.numel(), dtype=torch.float64, device=DEV), accumulate=True)
    cnt = D.sum(1, keepdim=True)
    return torch.where(cnt > 0, D / cnt.clamp(min=1), D)


def test_sampled_sage_forward_and_gradients_vs_fp64_autograd():
    A = G.reddit_like(64, seed=2).to(DEV)
    P = G.CsrMatrix(A.crow, A.col, None, A.rows, A.cols)
    X = G.dense_operand(A.rows, 64, 9, DEV)
    seeds = torch.randperm(A.rows, generator=torch.Generator().manual_seed(6))[:256].to(DEV)
    blocks = ofs.sample_blocks(P, seeds, [10, 5], 123)
    assert [b.adj.rows for b in blocks] == [blocks[1].src_nodes.numel(), seeds.numel()]
    # hop 0 (fanout 10) samples the seeds' neighbours: the last block; hop 1 (fanout 5) the first
    assert int(torch.diff(blocks[1].adj.crow).max()) <= 10 and int(torch.diff(blocks[0].adj.crow).max()) <= 5
    l1, l2 = _sage_pair()
    R = G.upstream_grad(seeds.numel(), 16, 3, DEV)
    h0 = X[blocks[0].src_nodes.long()]
    out = l2(blocks[1].adj, l1(blocks[0].adj, h0))
    (out * R).sum().backward()
    # fp64 dense reference on the same blocks
    W = {n: p.detach().double().requires_grad_(True) for n, p in
         (("n1", l1.weight_neigh), ("r1", l1.weight_root), ("b1", l1.bias),
          ("n2", l2.weight_neigh), ("r2", l2.weight_root), ("b2", l2.bias))}
    M1, M2 = _dense_mean(blocks[0].adj), _dense_mean(blocks[1].adj)
    x = h0.double()
    h1 = torch.relu(M1 @ x @ W["n1"] + x[:blocks[0].adj.rows] @ W["r1"] + W["b1"])
    ref = M2 @ h1 @ W["n2"] + h1[:blocks[1].adj.rows] @ W["r2"] + W["b2"]
    (ref * R.double()).sum().backward()
    assert torch.allclose(out.double(), ref, rtol=1e-4, atol=1e-4), float((out.double() - ref).abs().max())
    for name, p in (("n1", l1.weight_neigh), ("r1", l1.weight_root), ("b1", l1.bias),
                    ("n2", l2.weight_neigh), ("r2", l2.weight_root), ("b2", l2.bias)):
        g, gr = p.grad.double(), W[name].grad
        scale = float(gr.abs().max()) + 1e-12
        assert float((g - gr).abs().max()) <= 1e-4 * scale + 1e-5, (name, float((g - gr).abs().max()), scale)
