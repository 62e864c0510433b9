"""GPU tests of weighted and with-replacement neighbour sampling and of the edge ids
(``ofspmm_sample_neighbors_ex``, ``ops.sample_neighbors(prob=, replace=, return_eid=)``,
``sampling.sample_blocks``): bit-exact against the CPU oracle over index / value dtypes, modes and
fanouts on a graph with hub rows (whole-CTA path, split positive-weight count), equality of the
option-less calls with ``ofspmm_sample_neighbors``, chi-square tests of the distributions, the
C-ABI contract in the new modes, the 2^31-non-zero matrix, and learnable edge weights and
multi-edges on sampled blocks against fp64 autograd."""
import ctypes
import gc
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

pytestmark = pytest.mark.gpu

G = ofs.graphs
ops = import_module("of-spmm_b200.ops")
gcn = import_module("of-spmm_b200.gcn")
F = import_module("of-spmm_b200.functional")
_lib = ofs._lib
DEV = "cuda:0"
HUB = 100_000
SPECIAL = ("hub", 18, 19, 1, 2, 3, 4, 5, 0)


def _edge_graph(seed=8, rows=3000):
    """Rows of 0..60 entries (every 11th empty), rows of 1..4 and 26 entries, a hub of 1e5 entries,
    rows of 4096 and 5000 entries (both sides of the whole-CTA threshold), repeated and out-of-range
    columns; weights graded over six decades with zeros, negatives, NaN and infinities mixed in, and
    one long row (5000) and one short row (26) without any eligible weight."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, 61, rows)
    lens[::11] = 0
    lens[1:6] = [1, 2, 3, 4, 26]
    lens[17], lens[18], lens[19] = HUB, 4096, 5000
    crow = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    col = rng.integers(0, rows, int(crow[-1]))
    col[3::7] = col[2::7][: col[3::7].size]
    bad = rng.integers(0, col.size, col.size // 50)
    col[bad] = np.where(rng.random(bad.size) < 0.5, -1, rows + 1)
    val = rng.standard_normal(col.size).astype(np.float32)
    w = (rng.exponential(1.0, col.size) * 10.0 ** rng.integers(-3, 3, col.size)).astype(np.float32)
    special = np.array([0.0, -1.0, np.nan, np.inf, -np.inf], np.float32)
    pick = rng.random(col.size) < 0.2
    w[pick] = special[rng.integers(0, special.size, int(pick.sum()))]
    w[crow[19]:crow[20]] = -1.0
    w[crow[5]:crow[6]] = 0.0
    dst = rng.permutation(rows)[:900]
    first = [17, 18, 19, 1, 2, 3, 4, 5, 0]
    dst = np.concatenate([first, dst[~np.isin(dst, first)]])
    return crow, col, val, w, dst


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


def _prob(w, kind):
    if kind == "fp32":
        return torch.from_numpy(w).to(DEV), w
    bits = O.f32_to_bf16(w)
    return torch.from_numpy(bits.view(np.int16)).to(DEV).view(torch.bfloat16), bits


def _bits(t):
    if t is None:
        return None
    return t.cpu().view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32).numpy()


def _ref_bits(v):
    return None if v is None else v.view(np.int16 if v.dtype == np.uint16 else np.int32)


MODES = ["weighted_fp32", "weighted_bf16", "replace", "uniform_eid"]


@pytest.mark.parametrize("fanout", [1, 3, 25, -1, HUB])
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("vkind", ["fp32", "bf16", "none"])
@pytest.mark.parametrize("idx", ["int32", "int64"])
def test_bit_exact_vs_oracle(EG, idx, vkind, mode, fanout):
    crow, col, val, w, dst = EG
    if mode == "replace" and fanout == HUB:
        dst = dst[:40]          # 40 x 1e5 draws
    rows = crow.size - 1
    c, k, v, vref = _dev(crow, col, val, idx, vkind)
    p, pref = _prob(w, mode.split("_")[1]) if mode.startswith("weighted") else (None, None)
    replace = mode == "replace"
    d = torch.from_numpy(dst).to(DEV)
    seed = 0x9E3779B97F4A7C15 + 4242
    bc, bcol, bval, src, eid = ops.sample_neighbors(c, k, v, rows, rows, d, fanout, seed, prob=p, replace=replace,
                                                    return_eid=True)
    torch.cuda.synchronize()
    rc, rcol, rval, reid, rsrc, counts = SEO.sample_neighbors_ex(crow, col, vref, dst, fanout, seed, pref, replace)
    assert counts[2] == 0
    assert bc.dtype == torch.int32 and bcol.dtype == torch.int32 and src.dtype == c.dtype and eid.dtype == c.dtype
    assert np.array_equal(bc.cpu().numpy(), rc)
    assert np.array_equal(bcol.cpu().numpy(), rcol)
    assert np.array_equal(src.cpu().numpy(), rsrc)
    assert np.array_equal(eid.cpu().numpy(), reid)
    if vkind == "none":
        assert bval is None
    else:
        assert bval.dtype == v.dtype and np.array_equal(_bits(bval), _ref_bits(rval))
    # the invariants: A.col[eid] == src[blk_col], A.val[eid] == blk_val bit for bit
    assert torch.equal(k[eid.long()], src[bcol.long()])
    if v is not None:
        assert np.array_equal(_bits(v[eid.long()]), _bits(bval))
    if mode.startswith("weighted"):   # nothing ineligible is ever taken
        wt = p.float()[eid.long()]
        assert bool(((wt > 0) & torch.isfinite(wt)).all())


@pytest.mark.parametrize("idx", ["int32", "int64"])
def test_no_options_and_edge_ids_only_equal_the_plain_call(EG, idx):
    crow, col, val, _, dst = EG
    rows = crow.size - 1
    c, k, v, _ = _dev(crow, col, val, idx, "fp32")
    d = torch.from_numpy(dst).to(c.dtype).to(DEV)
    for fanout in (3, 25, -1):
        plain = _Call(c, k, v, rows, d, fanout, 5, None)
        assert plain() == 0
        for flags in (None, 0, _lib.SAMPLE_EDGE_IDS):
            ex = _Call(c, k, v, rows, d, fanout, 5, flags)
            assert ex() == 0
            torch.cuda.synchronize()
            o = ex.outputs()
            for x, y in zip(plain.outputs()[:5], o[:5]):
                assert torch.equal(x, y)
            if flags == _lib.SAMPLE_EDGE_IDS:
                bcol, src, eid = o[1], o[2], o[5]
                assert torch.equal(k[eid.long()], src[bcol.long()])
                assert torch.equal(v[eid.long()], o[4])
            else:
                assert o[5] is None


def test_weighted_k1_chi_square():
    """20 000 rows with the same graded weights 1..50, one weighted draw (k = 1) each: the per-position
    counts pass a chi-square test against w / sum(w) at the 0.999 quantile (49 degrees of freedom).
    Every row has its own keys (they depend on the row id); the seed is fixed: no flakes."""
    from scipy.stats import chi2
    deg, R = 50, 20_000
    crow = torch.arange(0, (R + 1) * deg, deg, dtype=torch.int32, device=DEV)
    col = torch.arange(deg, dtype=torch.int32, device=DEV).repeat(R)
    w = torch.arange(1, deg + 1, dtype=torch.float32, device=DEV).repeat(R)
    dst = torch.arange(R, dtype=torch.int32, device=DEV)
    A = max(R, deg)
    crow = torch.cat([crow, torch.full((A - R,), R * deg, dtype=torch.int32, device=DEV)])
    _, bcol, _, src, eid = ops.sample_neighbors(crow, col, None, A, A, dst, 1, 31337, prob=w, return_eid=True)
    assert eid.numel() == R
    pos = (eid.long() % deg)
    obs = torch.bincount(pos, minlength=deg).cpu().numpy().astype(np.float64)
    exp = R * np.arange(1, deg + 1) / (deg * (deg + 1) / 2)
    stat = float(((obs - exp) ** 2 / exp).sum())
    assert stat < chi2.ppf(0.999, deg - 1), stat


def test_replace_chi_square_uniform_positions():
    """5000 rows of 200 entries, 40 draws each: per-position counts against uniform, chi-square at the
    0.999 quantile (199 degrees of freedom); and a row holds repeats (multi-edges)."""
    from scipy.stats import chi2
    deg, R, k = 200, 5000, 40
    crow = torch.arange(0, (R + 1) * deg, deg, dtype=torch.int64, device=DEV)
    col = torch.arange(deg, dtype=torch.int64, device=DEV).repeat(R)
    dst = torch.arange(R, dtype=torch.int64, device=DEV)
    bc, _, _, _, eid = ops.sample_neighbors(crow, col, None, R, R, dst, k, 99, replace=True, return_eid=True)
    assert torch.equal(torch.diff(bc), torch.full((R,), k, dtype=torch.int32, device=DEV))
    obs = torch.bincount(eid % deg, minlength=deg).cpu().numpy().astype(np.float64)
    exp = R * k / deg
    stat = float(((obs - exp) ** 2 / exp).sum())
    assert stat < chi2.ppf(0.999, deg - 1), stat
    row0 = eid[:k].cpu().numpy()
    assert np.unique(row0).size < k   # 40 draws from 200: a repeat is all but certain (p ~ 0.98), seed fixed


# ------------------------------------------------------------------ C ABI contract in the new modes

class _Call:
    """Buffers of one ofspmm_sample_neighbors(_ex) call, with a guard band after every output.
    flags None: ofspmm_sample_neighbors; else the _ex call with these flags and weights `prob`."""
    GUARD = 64

    def __init__(self, crow, col, val, rows, dst, fanout, seed, flags, prob=None, cap=None):
        self.keep = (crow, col, val, dst, prob)
        self.A = ops._csr_struct(crow, col, val, rows, rows)
        n, g = dst.numel(), self.GUARD
        if cap is None:
            deg = (crow[1:] - crow[:-1]).long()[dst.long()]
            cap = int(deg.sum()) if fanout == -1 else dst.numel() * fanout
        self.dst, self.fanout, self.seed, self.cap, self.flags = dst, fanout, seed, cap, flags
        self.blk_crow = torch.full((n + 1 + g,), -7, dtype=torch.int32, device=DEV)
        self.blk_col = torch.full((cap + g,), -7, dtype=torch.int32, device=DEV)
        self.blk_val = torch.full((cap + g,), -7.0, dtype=val.dtype, device=DEV) if val is not None else None
        eid = flags is not None and flags & _lib.SAMPLE_EDGE_IDS
        self.blk_eid = torch.full((cap + g,), -7, dtype=crow.dtype, device=DEV) if eid else None
        self.src = torch.full((n + cap + g,), -7, dtype=crow.dtype, device=DEV)
        self.counts = torch.full((3,), -7, dtype=torch.int64, device=DEV)
        L = _lib.lib()
        if flags is None:
            self.opts = None
            self.ws_bytes = L.ofspmm_sample_neighbors_workspace_bytes(n, cap, ops._INDEX[crow.dtype])
        else:
            self.sopts = _lib.SampleOptsStruct(flags, ops._DENSE[prob.dtype] if prob is not None else 0,
                                               None if prob is None else prob.data_ptr())
            self.opts = ctypes.byref(self.sopts)
            self.ws_bytes = L.ofspmm_sample_neighbors_ex_workspace_bytes(n, cap, ops._INDEX[crow.dtype], self.opts)
        self.ws = torch.empty(self.ws_bytes, dtype=torch.uint8, device=DEV)

    def _ptr(self, t):
        return None if t is None else t.data_ptr()

    def __call__(self):
        L = _lib.lib()
        s = torch.cuda.current_stream().cuda_stream
        if self.flags is None:
            return L.ofspmm_sample_neighbors(ctypes.byref(self.A), ops._ptr(self.dst), self.dst.numel(), self.fanout,
                                             self.seed, self.cap, self.blk_crow.data_ptr(), self.blk_col.data_ptr(),
                                             self._ptr(self.blk_val), self.src.data_ptr(), self.counts.data_ptr(),
                                             self.ws.data_ptr(), self.ws_bytes, s)
        return L.ofspmm_sample_neighbors_ex(ctypes.byref(self.A), self.opts, ops._ptr(self.dst), self.dst.numel(),
                                            self.fanout, self.seed, self.cap, self.blk_crow.data_ptr(),
                                            self.blk_col.data_ptr(), self._ptr(self.blk_val), self._ptr(self.blk_eid),
                                            self.src.data_ptr(), self.counts.data_ptr(), self.ws.data_ptr(),
                                            self.ws_bytes, s)

    def buffers(self):
        return [t for t in (self.blk_crow, self.blk_col, self.blk_val, self.blk_eid, self.src, self.counts)
                if t is not None]

    def outputs(self):
        """(blk_crow, blk_col, src, counts, blk_val, blk_eid): the written part of each (None where absent)."""
        n = self.dst.numel()
        nnz, num_src = (int(x) for x in self.counts[:2].tolist())
        val = None if self.blk_val is None else self.blk_val[:nnz].clone()
        eid = None if self.blk_eid is None else self.blk_eid[:nnz].clone()
        return [self.blk_crow[:n + 1].clone(), self.blk_col[:nnz].clone(), self.src[:num_src].clone(),
                self.counts.clone(), val, eid]


CALL_MODES = {"weighted": lambda: _lib.SAMPLE_EDGE_IDS, "replace": lambda: _lib.SAMPLE_REPLACE | _lib.SAMPLE_EDGE_IDS,
              "eid": lambda: _lib.SAMPLE_EDGE_IDS}


def _mode_call(EG, mode, fanout, seed, cap=None, dst=None, idx="int32"):
    crow, col, val, w, d0 = EG
    rows = crow.size - 1
    c, k, v, _ = _dev(crow, col, val, idx, "fp32")
    d = torch.from_numpy(d0 if dst is None else dst).to(c.dtype).to(DEV)
    p = torch.from_numpy(w).to(DEV) if mode == "weighted" else None
    return _Call(c, k, v, rows, d, fanout, seed, CALL_MODES[mode](), prob=p, cap=cap)


def _eq(x, y):
    return (x is None and y is None) or torch.equal(x, y)


@pytest.mark.parametrize("mode", list(CALL_MODES))
def test_cuda_graph_replay_equals_eager(EG, mode):
    call = _mode_call(EG, mode, 25, 77)
    assert call() == 0
    torch.cuda.synchronize()
    eager = call.outputs()
    for t in call.buffers():
        t.fill_(-3)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            assert call() == 0
    torch.cuda.current_stream().wait_stream(s)
    for t in call.buffers():
        t.fill_(-5)
    graph.replay()
    torch.cuda.synchronize()
    for x, y in zip(eager, call.outputs()):
        assert _eq(x, y)
    assert int(eager[3][0]) > 0


@pytest.mark.parametrize("mode", list(CALL_MODES))
def test_capacity_exceeded_reports_size_and_writes_nothing_past_capacity(EG, mode):
    full = _mode_call(EG, mode, 25, 3)
    assert full() == 0
    torch.cuda.synchronize()
    c, d = full.keep[0], full.dst
    if mode == "replace":
        deg = (c[1:] - c[:-1]).long()[d.long()]
        need = int((deg > 0).sum()) * 25
    elif mode == "weighted":
        w = full.keep[4]
        ok = ((w > 0) & torch.isfinite(w)).long()
        cs = torch.cat([torch.zeros(1, dtype=torch.long, device=DEV), torch.cumsum(ok, 0)])
        npos = cs[c[1:].long()][d.long()] - cs[c[:-1].long()][d.long()]
        need = int(torch.clamp(npos, max=25).sum())
    else:
        deg = (c[1:] - c[:-1]).long()[d.long()]
        need = int(torch.clamp(deg, max=25).sum())
    small = _mode_call(EG, mode, 25, 3, cap=need - 1)
    assert small() == 0
    torch.cuda.synchronize()
    assert int(small.counts[0]) == need and int(small.counts[2]) == 0
    n, cap = d.numel(), need - 1
    assert bool((small.blk_crow[n + 1:] == -7).all())
    assert bool((small.blk_col[cap:] == -7).all()) and bool((small.blk_val[cap:] == -7.0).all())
    assert bool((small.blk_eid[cap:] == -7).all())
    assert bool((small.src[n + cap:] == -7).all())
    exact = _mode_call(EG, mode, 25, 3, cap=need)
    assert exact() == 0
    torch.cuda.synchronize()
    for x, y in zip(exact.outputs(), full.outputs()):
        assert _eq(x, y)


@pytest.mark.parametrize("mode", list(CALL_MODES))
def test_invalid_destinations_are_counted(EG, mode):
    crow, col, val, w, _ = EG
    rows = crow.size - 1
    dst = np.array([5, rows, 17, 5, -3, 40, 17, 41], np.int64)     # out of range: 2; repeated: 5, 17 (x2 each)
    call = _mode_call(EG, mode, 3, 11, cap=dst.size * 3, dst=dst, idx="int64")
    assert call() == 0
    torch.cuda.synchronize()
    prob = w if mode == "weighted" else None
    _, _, _, _, _, counts = SEO.sample_neighbors_ex(crow, col, val, dst, 3, 11, prob, mode == "replace")
    assert int(call.counts[2]) == counts[2] == 6
    bc = call.blk_crow[:dst.size + 1].cpu().numpy()
    assert (np.diff(bc)[[0, 1, 2, 3, 4, 6]] == 0).all()
    assert bool((call.blk_crow[dst.size + 1:] == -7).all())


@pytest.mark.parametrize("mode", list(CALL_MODES))
def test_empty_batch(EG, mode):
    call = _mode_call(EG, mode, 10, 0, cap=0, dst=np.zeros(0, np.int64))
    assert call() == 0
    torch.cuda.synchronize()
    assert call.counts.tolist() == [0, 0, 0] and int(call.blk_crow[0]) == 0
    assert bool((call.blk_crow[1:] == -7).all())
    crow, col, val, w, _ = EG
    c, k, v, _ = _dev(crow, col, val, "int32", "fp32")
    d = torch.empty(0, dtype=c.dtype, device=DEV)
    p = torch.from_numpy(w).to(DEV) if mode == "weighted" else None
    bc, bcol, bval, src, eid = ops.sample_neighbors(c, k, v, crow.size - 1, crow.size - 1, d, 10, 0, prob=p,
                                                    replace=mode == "replace", return_eid=True)
    assert bc.tolist() == [0] and bcol.numel() == 0 and bval.numel() == 0 and src.numel() == 0 and eid.numel() == 0


# ------------------------------------------------------------------ 2^31 + 2^25 non-zeros

@pytest.fixture(scope="module")
def WIDE():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    gc.collect()
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info(0)
    if free < 50e9:
        pytest.skip(f"needs 50 GB of free device memory for the 2^31-non-zero matrix, {free / 1e9:.0f} GB free")
    A = G.wide_csr(DEV)
    yield A, A.crow.cpu().numpy()
    del A
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


@pytest.mark.parametrize("mode", ["weighted", "eid"])
def test_wide_matrix_vs_oracle_on_its_rows(WIDE, mode):
    """prob = A.val (half the values negative: ineligible) on the hub across entry 2^31, the rows
    around the out-of-range entries and rows past 2^31; edge ids are int64 positions past 2^31."""
    A, crow_h = WIDE
    M = G.WIDE_M
    around = [int(np.searchsorted(crow_h, p, side="right")) - 1 for p, _ in G.WIDE_BAD]
    rows = [G.WIDE_HUB] + around + [G.WIDE_HUB + 1, G.WIDE_HUB + 2, M - 1, M - 2, 3, 5, 7, 1000, 2000]
    rows += list(range(G.WIDE_HUB + 500, G.WIDE_HUB + 700))
    dst = np.array(list(dict.fromkeys(rows)), np.int64)
    d = torch.from_numpy(dst).to(DEV)
    seed, fanout = 77, 25
    prob = A.val if mode == "weighted" else None
    bc, bcol, bval, src, eid = ops.sample_neighbors(A.crow, A.col, A.val, M, M, d, fanout, seed, prob=prob,
                                                    return_eid=True)
    torch.cuda.synchronize()
    b, e = crow_h[dst], crow_h[dst + 1]
    seg_off = np.concatenate([[0], np.cumsum(e - b)])
    seg_col = np.concatenate([A.col[x:y].cpu().numpy() for x, y in zip(b, e)])
    seg_val = np.concatenate([A.val[x:y].cpu().numpy() for x, y in zip(b, e)])
    rc, rcol, rval, reid, rsrc, counts = SEO.sample_neighbors_ex_rows(M, dst, seg_off, b, seg_col, seg_val,
                                                                      seg_val if prob is not None else None, False,
                                                                      fanout, seed)
    assert counts[2] == 0 and int(e[0] - b[0]) == G.WIDE_HUB_LEN
    assert np.array_equal(bc.cpu().numpy(), rc)
    assert np.array_equal(bcol.cpu().numpy(), rcol)
    assert np.array_equal(src.cpu().numpy(), rsrc)
    assert np.array_equal(eid.cpu().numpy(), reid)
    assert np.array_equal(_bits(bval), _ref_bits(rval))
    assert int(eid.max()) >= 1 << 31


# ------------------------------------------------------------------ end to end on the blocks

def _dense(adj, val):
    rows = torch.repeat_interleave(torch.arange(adj.rows, device=DEV), torch.diff(adj.crow).long())
    D = torch.zeros(adj.rows, adj.cols, dtype=torch.float64, device=DEV)
    return D.index_put((rows, adj.col.long()), val, accumulate=True)


def test_learnable_edge_weights_through_eid_vs_fp64_autograd():
    """sample_blocks(prob=A.val, edge_ids=True) on a Reddit-shaped graph, then a 2-layer aggregation
    spmm_csr(blk.crow, blk.col, w[blk.eid], h) with learnable full-graph edge weights w: forward and
    the gradients wrt w and X match fp64 dense autograd on the same blocks."""
    A = G.reddit_like(64, seed=2).to(DEV)
    seeds = torch.randperm(A.rows, generator=torch.Generator().manual_seed(6))[:256].to(DEV)
    blocks = ofs.sample_blocks(A, seeds, [10, 5], 7, prob=A.val, edge_ids=True)
    for blk in blocks:
        assert blk.eid is not None and blk.eid.numel() == blk.adj.nnz
        assert torch.equal(A.col[blk.eid.long()].long(), blk.src_nodes[blk.adj.col.long()].long())
        assert torch.equal(A.val[blk.eid.long()], blk.adj.val)
        assert bool((blk.adj.val > 0).all())           # negative weights are never sampled
    X = G.dense_operand(A.rows, 32, 9, DEV).requires_grad_(True)
    w = A.val.abs().clone().requires_grad_(True)
    R = G.upstream_grad(seeds.numel(), 32, 3, DEV)
    h = X[blocks[0].src_nodes.long()]
    for blk in blocks:
        h = F.spmm_csr(blk.adj.crow, blk.adj.col, w[blk.eid.long()], h, blk.adj.rows, blk.adj.cols)
    (h * R).sum().backward()
    X64 = X.detach().double().requires_grad_(True)
    w64 = w.detach().double().requires_grad_(True)
    h64 = X64[blocks[0].src_nodes.long()]
    for blk in blocks:
        h64 = _dense(blk.adj, w64[blk.eid.long()]) @ h64
    (h64 * R.double()).sum().backward()
    scale = float(h64.abs().max())
    assert float((h.double() - h64).abs().max()) <= 1e-4 * scale + 1e-5
    for g, gr in ((w.grad, w64.grad), (X.grad, X64.grad)):
        s = float(gr.abs().max()) + 1e-12
        assert float((g.double() - gr).abs().max()) <= 1e-4 * s + 1e-6, (float((g.double() - gr).abs().max()), s)
    assert int((w.grad != 0).sum()) > 0


def test_replace_blocks_sage_counts_multi_edges():
    """replace=True blocks fed to gcn.SAGEConv equal the fp64 mean with every repeated column counted
    (index_put_ with accumulate=True)."""
    A = G.reddit_like(64, seed=2).to(DEV)
    P = G.CsrMatrix(A.crow, A.col, None, A.rows, A.cols)
    X = G.dense_operand(A.rows, 64, 8, DEV)
    seeds = torch.randperm(A.rows, generator=torch.Generator().manual_seed(4))[:256].to(DEV)
    blocks = ofs.sample_blocks(P, seeds, [10, 5], 21, replace=True, edge_ids=True)
    dup = 0
    for b in blocks:
        key = torch.repeat_interleave(torch.arange(b.adj.rows, device=DEV), torch.diff(b.adj.crow).long()) * b.adj.cols
        dup += (key + b.adj.col.long()).numel() - torch.unique(key + b.adj.col.long()).numel()
    assert dup > 0                                   # multi-edges are present
    l1 = gcn.SAGEConv(64, 32, activation="relu", seed=3, device=DEV)
    l2 = gcn.SAGEConv(32, 16, activation=None, seed=5, device=DEV)
    with torch.no_grad():
        h0 = X[blocks[0].src_nodes.long()]
        out = l2(blocks[1].adj, l1(blocks[0].adj, h0))

        def mean(adj):
            D = _dense(adj, torch.ones(adj.nnz, dtype=torch.float64, device=DEV))
            cnt = D.sum(1, keepdim=True)
            return torch.where(cnt > 0, D / cnt.clamp(min=1), D)

        x = h0.double()
        h1 = torch.relu(mean(blocks[0].adj) @ x @ l1.weight_neigh.double() + x[:blocks[0].adj.rows] @ l1.weight_root.double()
                        + l1.bias.double())
        ref = (mean(blocks[1].adj) @ h1 @ l2.weight_neigh.double() + h1[:blocks[1].adj.rows] @ l2.weight_root.double()
               + l2.bias.double())
    assert torch.allclose(out.double(), ref, rtol=1e-4, atol=1e-4), float((out.double() - ref).abs().max())
