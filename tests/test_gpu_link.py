"""GPU tests of link prediction: edge exclusion in neighbour sampling (bit-exact against the CPU
oracle over index / value dtypes, modes and fanouts on a graph with hub rows; an empty list equals
the call without one), negative sampling (bit-exact, rejection checked with scipy, counts,
chi-square uniformity, exhausted trials, rectangular A, CUDA-graph replay), edge lookup, the
2^31-non-zero matrix, ``edge_score`` against fp64 autograd, and one link-prediction train step
against an fp64 dense re-implementation."""
import gc
import os
import sys
from importlib import import_module

import numpy as np
import pytest
import scipy.sparse as sp
import torch

import ofspmm_b200 as ofs
from oracle import oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import _sample_link_oracle as SLO  # noqa: E402

pytestmark = pytest.mark.gpu

G = ofs.graphs
ops = import_module("of-spmm_b200.ops")
gcn = import_module("of-spmm_b200.gcn")
F = import_module("of-spmm_b200.functional")
sampling = import_module("of-spmm_b200.sampling")
DEV = "cuda:0"
HUB = 100_000


def _hub_graph(seed=21, rows=3000):
    """Rows of 0..60 entries (every 11th empty), rows of 1..4 and 26 entries, a hub of 1e5 entries,
    rows of 4096 and 5000 entries (both sides of the whole-CTA threshold), out-of-range columns;
    weights with zeros, negatives and NaN mixed in."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, 61, rows)
    lens[::11] = 0
    lens[1:6] = [1, 2, 3, 4, 26]
    lens[17], lens[18], lens[19] = HUB, 4096, 5000
    crow = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    col = rng.integers(0, rows, int(crow[-1]))
    bad = rng.integers(0, col.size, col.size // 50)
    col[bad] = np.where(rng.random(bad.size) < 0.5, -1, rows + 1)
    val = rng.standard_normal(col.size).astype(np.float32)
    w = (rng.exponential(1.0, col.size) * 10.0 ** rng.integers(-2, 2, col.size)).astype(np.float32)
    pick = rng.random(col.size) < 0.15
    w[pick] = np.array([0.0, -1.0, np.nan], np.float32)[rng.integers(0, 3, int(pick.sum()))]
    dst = rng.permutation(rows)[:900]
    first = [17, 18, 19, 1, 2, 3, 4, 5, 0]
    dst = np.concatenate([first, dst[~np.isin(dst, first)]])
    nnz = col.size
    never = np.setdiff1d(np.arange(rows), dst)[:40]                 # rows that are never sampled
    ex = [rng.choice(nnz, nnz // 10, replace=False),                # 10 % of every row
          np.arange(crow[4], crow[6]),                              # rows 4 (4 entries) and 5 (26): k = 0
          crow[17] + rng.choice(HUB, 3000, replace=False),          # inside the hub
          np.arange(crow[18], crow[18] + 4000),                     # most of the 4096 row
          [0, nnz - 1]]
    ex += [np.arange(crow[v], crow[v + 1]) for v in never]
    return crow, col, val, w, dst, np.unique(np.concatenate(ex)).astype(np.int64)


@pytest.fixture(scope="module")
def HG():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return _hub_graph()


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
    return None if t is None else t.cpu().view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32).numpy()


def _ref_bits(v):
    return None if v is None else v.view(np.int16 if v.dtype == np.uint16 else np.int32)


MODES = ["uniform", "weighted_fp32", "weighted_bf16", "replace"]


@pytest.mark.parametrize("fanout", [-1, 0, 1, 5, 25])
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("vkind", ["fp32", "bf16", "none"])
@pytest.mark.parametrize("idx", ["int32", "int64"])
def test_exclusion_bit_exact_vs_oracle(HG, idx, vkind, mode, fanout):
    crow, col, val, w, dst, excl = HG
    rows = crow.size - 1
    c, k, v, vref = _dev(crow, col, val, idx, vkind)
    p, pref = _prob(w, mode.split("_")[1]) if mode.startswith("weighted") else (None, None)
    replace = mode == "replace"
    d = torch.from_numpy(dst).to(DEV)
    seed = 0x51A7E + fanout
    # the list is passed shuffled and with repeats: ops sorts and deduplicates it
    ex_t = torch.from_numpy(np.concatenate([excl[::-1], excl[:50]])).to(DEV)
    bc, bcol, bval, src, eid = ops.sample_neighbors(c, k, v, rows, rows, d, fanout, seed, prob=p, replace=replace,
                                                    return_eid=True, exclude_eid=ex_t)
    rc, rcol, rval, reid, rsrc = SLO.sample_neighbors_excl(crow, col, vref, dst, fanout, seed, excl, pref, replace)
    assert np.array_equal(bc.cpu().numpy(), rc)
    assert np.array_equal(bcol.cpu().numpy(), rcol)
    assert np.array_equal(src.cpu().numpy(), rsrc)
    assert np.array_equal(eid.cpu().numpy(), reid)
    if vkind == "none":
        assert bval is None
    else:
        assert np.array_equal(_bits(bval), _ref_bits(rval))
    # properties: nothing excluded is taken; a row without an excluded entry is the plain call's
    assert not np.isin(eid.cpu().numpy(), excl).any()
    pc, _, _, _, peid = ops.sample_neighbors(c, k, v, rows, rows, d, fanout, seed, prob=p, replace=replace,
                                             return_eid=True)
    pc, peid, bch, eidh = pc.cpu().numpy(), peid.cpu().numpy(), bc.cpu().numpy(), eid.cpu().numpy()
    hit = np.searchsorted(excl, crow[dst + 1]) - np.searchsorted(excl, crow[dst])
    clean = np.flatnonzero(hit == 0)
    assert clean.size > 50
    for i in clean:
        assert np.array_equal(eidh[bch[i]:bch[i + 1]], peid[pc[i]:pc[i + 1]])
    # dst[6], dst[7] = rows 4 and 5, wholly excluded: k = 0
    assert hit[6] == 4 and hit[7] == 26 and bch[6] == bch[7] == bch[8]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("idx", ["int32", "int64"])
def test_empty_exclusion_is_bit_identical(HG, idx, mode):
    crow, col, val, w, dst, _ = HG
    rows = crow.size - 1
    c, k, v, _ = _dev(crow, col, val, idx, "fp32")
    p = _prob(w, mode.split("_")[1])[0] if mode.startswith("weighted") else None
    d = torch.from_numpy(dst).to(DEV)
    for fanout in (-1, 1, 25):
        kw = dict(prob=p, replace=mode == "replace", return_eid=True)
        a = ops.sample_neighbors(c, k, v, rows, rows, d, fanout, 99, **kw)
        b = ops.sample_neighbors(c, k, v, rows, rows, d, fanout, 99, exclude_eid=torch.zeros(0, dtype=c.dtype,
                                                                                              device=DEV), **kw)
        for x, y in zip(a, b):
            assert torch.equal(x, y)


def test_sample_blocks_exclusion_applies_to_every_hop(HG):
    crow, col, val, _, dst, excl = HG
    rows = crow.size - 1
    c, k, v, _ = _dev(crow, col, val, "int64", "fp32")
    A = G.CsrMatrix(c, k, v, rows, rows)
    ex = torch.from_numpy(excl).to(DEV)
    blocks = ofs.sample_blocks(A, torch.from_numpy(dst[:200]).to(DEV), [10, 5, 3], 7, edge_ids=True, exclude_eid=ex)
    for b in blocks:
        assert not torch.isin(b.eid, ex).any()
        assert torch.equal(k[b.eid], b.src_nodes[b.adj.col.long()])


# ------------------------------------------------------------------ negative sampling and edge lookup

def _sorted_graph(rows=2000, cols=2000, seed=3, dense_row=None):
    """A CSR with sorted, distinct columns per row; ``dense_row`` holds every column but 3."""
    rng = np.random.default_rng(seed)
    m = sp.random(rows, cols, density=0.01, format="csr", random_state=seed)
    m.data[:] = 1
    if dense_row is not None:
        m = m.tolil()
        m[dense_row, :] = 1
        m[dense_row, [5, 77, 1500]] = 0
        m = m.tocsr()
        m.eliminate_zeros()
    m.sort_indices()
    del rng
    return m


def _negs(m, idx, src, k, seed, **kw):
    t = torch.int32 if idx == "int32" else torch.int64
    c = torch.from_numpy(m.indptr.astype(np.int64)).to(t).to(DEV)
    k_ = torch.from_numpy(m.indices.astype(np.int64)).to(t).to(DEV)
    neg, counts = ops.negative_sample(c, k_, m.shape[0], m.shape[1], torch.from_numpy(src).to(DEV), k, seed, **kw)
    return neg, counts, c, k_


@pytest.mark.parametrize("shape", [(2000, 2000), (1500, 2600)])
@pytest.mark.parametrize("idx", ["int32", "int64"])
def test_negative_sample_bit_exact_and_rejection(idx, shape):
    m = _sorted_graph(*shape, dense_row=7)
    rows, cols = m.shape
    rng = np.random.default_rng(1)
    src = np.concatenate([rng.integers(0, rows, 3000), [7, 7, -1, rows, rows + 5]])
    square = rows == cols
    for trials in (1, 8):
        neg, counts, *_ = _negs(m, idx, src, 5, 0xBEEF + trials, exclude_self=square, max_trials=trials)
        assert neg.dtype == (torch.int32 if idx == "int32" else torch.int64) and neg.shape == (src.size, 5)
        rneg, rcounts = SLO.negative_sample(m.indptr, m.indices, cols, src, 5, 0xBEEF + trials, True, square, trials)
        got = neg.cpu().numpy()
        assert np.array_equal(got, rneg)
        assert counts.cpu().tolist() == rcounts.tolist()
        assert rcounts[1] == 3 and (got[-3:] == -1).all()
        ok = got >= 0
        uu = np.broadcast_to(src[:, None], got.shape)[ok]
        vv = got[ok]
        assert (np.asarray(m[uu, vv]).ravel() == 0).all()        # no accepted pair is an edge of A
        if square:
            assert (uu != vv).all()                               # nor a self-loop
        assert rcounts[0] == (~ok).sum()
    # the near-complete row 7 exhausts its trials: most of its slots fail
    neg, _, _, _ = _negs(m, idx, np.array([7] * 50), 4, 5, max_trials=2, exclude_self=square)
    assert (neg.cpu().numpy() == -1).mean() > 0.9


def test_negative_sample_uniform_over_non_neighbours():
    """Chi-square: the accepted negatives of one row are uniform over its non-neighbours."""
    m = _sorted_graph(200, 200, seed=8)
    row = int(np.argmax(np.diff(m.indptr)))
    src = np.full(40_000, row)
    neg, _, _, _ = _negs(m, "int64", src, 5, 17)
    got = neg.cpu().numpy().ravel()
    got = got[got >= 0]
    allowed = np.setdiff1d(np.arange(200), np.concatenate([m.indices[m.indptr[row]:m.indptr[row + 1]], [row]]))
    assert np.isin(got, allowed).all()
    obs = np.bincount(got, minlength=200)[allowed]
    exp = got.size / allowed.size
    chi2 = float(((obs - exp) ** 2 / exp).sum())
    dof = allowed.size - 1
    assert chi2 < dof + 5 * np.sqrt(2 * dof), (chi2, dof)


def test_negative_sample_cuda_graph_replay():
    m = _sorted_graph(1000, 1000, seed=4)
    src = torch.from_numpy(np.random.default_rng(3).integers(-1, 1001, 4096)).to(DEV)
    c = torch.from_numpy(m.indptr.astype(np.int64)).to(DEV)
    k = torch.from_numpy(m.indices.astype(np.int64)).to(DEV)
    ref, ref_counts = ops.negative_sample(c, k, 1000, 1000, src, 3, 11)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.negative_sample(c, k, 1000, 1000, src, 3, 11)      # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        neg, counts = ops.negative_sample(c, k, 1000, 1000, src, 3, 11)
    for _ in range(3):
        neg.fill_(-7)
        counts.fill_(12345)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(neg, ref) and torch.equal(counts, ref_counts)


@pytest.mark.parametrize("idx", ["int32", "int64"])
def test_edge_ids_match_host_dictionary(idx):
    m = _sorted_graph(1500, 2600, seed=6)
    rows, cols = m.shape
    coo = m.tocoo()
    first = {(int(a), int(b)): p for p, (a, b) in enumerate(zip(np.repeat(np.arange(rows), np.diff(m.indptr)),
                                                                 m.indices))}
    rng = np.random.default_rng(0)
    sel = rng.integers(0, coo.nnz, 2000)
    u = np.concatenate([coo.row[sel], rng.integers(-3, rows + 3, 3000), [-1, rows, 0]])
    v = np.concatenate([coo.col[sel], rng.integers(-3, cols + 3, 3000), [0, 0, cols + 9]])
    t = torch.int32 if idx == "int32" else torch.int64
    c = torch.from_numpy(m.indptr.astype(np.int64)).to(t).to(DEV)
    k = torch.from_numpy(m.indices.astype(np.int64)).to(t).to(DEV)
    eid = ofs.edge_ids(c, k, rows, cols, torch.from_numpy(u).to(DEV), torch.from_numpy(v).to(DEV))
    assert eid.dtype == t
    want = [first.get((int(a), int(b)), -1) for a, b in zip(u, v)]
    assert eid.cpu().tolist() == want
    assert eid.cpu().tolist() == SLO.edge_ids(m.indptr, m.indices, u, v).tolist()
    assert (eid[:2000] >= 0).all()


# ------------------------------------------------------------------ 2^31 non-zeros

def test_wide_matrix_edge_ids_and_negative_rejection():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    gc.collect()
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info(0)
    if free < 40e9:
        pytest.skip(f"needs 40 GB of free device memory for a 2^31-non-zero matrix, {free / 1e9:.0f} GB free")
    A = G.wide_csr(DEV)
    crow_h = A.crow.cpu().numpy()
    hub = G.WIDE_HUB
    lens = np.diff(crow_h)
    after = [int(r) for r in np.flatnonzero(lens[hub + 1:] >= 2)[:3] + hub + 1]
    # the rows read here get their columns sorted (the lookup's precondition): the hub, which
    # straddles non-zero 2^31, and rows wholly above it
    rows_sel = [hub] + after
    for r in rows_sel:
        p0, p1 = int(crow_h[r]), int(crow_h[r + 1])
        A.col[p0:p1] = torch.sort(A.col[p0:p1])[0]
    seg_off, seg_col = [0], []
    for r in rows_sel:
        seg_col.append(A.col[int(crow_h[r]):int(crow_h[r + 1])].cpu().numpy())
        seg_off.append(seg_off[-1] + seg_col[-1].size)
    # lookup: entries on both sides of 2^31 in the hub, and in the rows after it
    hub_cols = seg_col[0]
    picks = [(1 << 31) - 3000 - int(crow_h[hub]), (1 << 31) + 3000 - int(crow_h[hub]), hub_cols.size - 1]
    u = [hub] * len(picks) + after + [hub, -1]
    v = [int(hub_cols[j]) for j in picks] + [int(seg_col[1][0]), int(seg_col[2][-1]), int(seg_col[3][0]), -5, 0]
    want = []
    for uu, vv in zip(u, v):
        if uu < 0:
            want.append(-1)
            continue
        i = rows_sel.index(uu)
        row = seg_col[i]
        j = int(np.searchsorted(row, vv))
        want.append(int(crow_h[uu]) + j if j < row.size and row[j] == vv else -1)
    eid = ofs.edge_ids(A.crow, A.col, G.WIDE_M, G.WIDE_K, torch.tensor(u, device=DEV), torch.tensor(v, device=DEV))
    got = eid.cpu().tolist()
    assert got == want
    assert sum(g >= 1 << 31 for g in got) >= 4
    # rejection: the hub (2^25 entries over 2^20 columns) holds nearly every column; the other
    # rows nearly none.  Bit-exact against the oracle on those rows.
    src = np.array([hub] * 8 + after * 4)
    row_of = {r: i for i, r in enumerate(rows_sel)}
    seg_off = np.asarray(seg_off)
    begin = np.array([seg_off[row_of[s]] for s in src])
    end = np.array([seg_off[row_of[s] + 1] for s in src])
    neg, counts = ofs.negative_sample(A.crow, A.col, G.WIDE_M, G.WIDE_K, torch.from_numpy(src).to(DEV), 4, 23,
                                      exclude_self=False, max_trials=4)
    rneg, rcounts = SLO.negative_sample(np.zeros(G.WIDE_M + 1), None, G.WIDE_K, src, 4, 23, True, False, 4,
                                        segments=(begin, end, np.concatenate(seg_col)))
    assert np.array_equal(neg.cpu().numpy(), rneg)
    assert counts.cpu().tolist() == rcounts.tolist()
    hub_set = set(hub_cols.tolist())
    assert all(x < 0 or x not in hub_set for x in rneg[:8].ravel())
    del A
    gc.collect()
    torch.cuda.empty_cache()


# ------------------------------------------------------------------ edge_score

@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_edge_score_vs_fp64_autograd(dtype):
    torch.manual_seed(5)
    lens = torch.tensor([4, 1, 6, 3, 1, 5] * 40)                    # rows of length 1: every negative failed
    rows, cols, n = lens.numel(), 300, 64
    crow = torch.zeros(rows + 1, dtype=torch.int32)
    crow[1:] = torch.cumsum(lens, 0)
    col = torch.randint(0, cols, (int(crow[-1]),), dtype=torch.int32)
    col[1::5] = col[0::5][: col[1::5].numel()]                       # repeated negatives
    rows_of = torch.repeat_interleave(torch.arange(rows), lens)
    hr = torch.randn(rows, n).to(dtype)
    hc = torch.randn(cols, n).to(dtype)
    a = hr.to(DEV).requires_grad_()
    b = hc.to(DEV).requires_grad_()
    s = ofs.edge_score(crow.to(DEV), col.to(DEV), a, b, rows, cols)
    assert s.dtype == dtype and s.shape == (col.numel(),)
    w = torch.randn(col.numel()).to(dtype)
    (s * w.to(DEV)).sum().backward()
    a64, b64 = hr.double().requires_grad_(), hc.double().requires_grad_()
    ref = (a64[rows_of] * b64[col.long()]).sum(1)
    (ref * w.double()).sum().backward()
    tol = dict(rtol=1e-4, atol=1e-4) if dtype == torch.float32 else dict(rtol=2e-2, atol=0.3)
    assert torch.allclose(s.double().cpu(), ref.detach(), **tol)
    assert torch.allclose(a.grad.double().cpu(), a64.grad, **tol)
    assert torch.allclose(b.grad.double().cpu(), b64.grad, **tol)


# ------------------------------------------------------------------ end to end

def _sym_graph(rows=3000, seed=12):
    rng = np.random.default_rng(seed)
    m = sp.random(rows, rows, density=0.004, format="csr", random_state=seed)
    m = ((m + m.T) > 0).astype(np.float32).tocsr()
    m.setdiag(0)
    m.eliminate_zeros()
    m.sort_indices()
    val = rng.random(m.nnz).astype(np.float32) + 0.5
    return m, val


def _batch(A, pos, seed, **kw):
    return ofs.sample_link_batch(A, pos, 3, [5, 4], seed, exclude="reverse", edge_ids=True, **kw)


def test_link_batch_is_deterministic_and_excludes_reverse_edges():
    m, val = _sym_graph()
    c = torch.from_numpy(m.indptr.astype(np.int64)).to(DEV)
    k = torch.from_numpy(m.indices.astype(np.int64)).to(DEV)
    A = G.CsrMatrix(c, k, torch.from_numpy(val).to(DEV), m.shape[0], m.shape[1])
    pos = torch.from_numpy(np.random.default_rng(2).choice(m.nnz, 256, replace=False)).to(DEV)
    b1, b2 = _batch(A, pos, 77), _batch(A, pos, 77)
    for x, y in ((b1.pair.crow, b2.pair.crow), (b1.pair.col, b2.pair.col), (b1.src_local, b2.src_local),
                 (b1.labels, b2.labels)):
        assert torch.equal(x, y)
    for x, y in zip(b1.blocks, b2.blocks):
        assert torch.equal(x.adj.crow, y.adj.crow) and torch.equal(x.adj.col, y.adj.col)
        assert torch.equal(x.src_nodes, y.src_nodes) and torch.equal(x.eid, y.eid)
    u = torch.searchsorted(c, pos, right=True) - 1
    v = k[pos]
    rev = ofs.edge_ids(c, k, A.rows, A.cols, v, u)
    assert (rev >= 0).all()                                     # symmetric graph: every reverse exists
    banned = torch.cat([pos, rev])
    for blk in b1.blocks:
        assert not torch.isin(blk.eid, banned).any()
    seeds = b1.seeds
    assert torch.equal(seeds, torch.unique(seeds)) and torch.equal(seeds[b1.src_local], u)
    pc = b1.pair.crow.long()
    assert torch.equal(seeds[b1.pair.col[pc[:-1]].long()], v)
    assert float(b1.labels.sum()) == 256


def test_link_prediction_train_step_matches_fp64_dense():
    """sample_link_batch(exclude="reverse") -> two SAGEConv layers on the blocks -> edge_score ->
    BCE-with-logits: the loss and every parameter gradient against an fp64 dense re-implementation."""
    torch.manual_seed(0)
    m, _ = _sym_graph()
    rows, nf, hid = m.shape[0], 16, 24
    c = torch.from_numpy(m.indptr.astype(np.int64)).to(DEV)
    k = torch.from_numpy(m.indices.astype(np.int64)).to(DEV)
    A = G.CsrMatrix(c, k, None, rows, rows)
    X = torch.randn(rows, nf, device=DEV)
    pos = torch.from_numpy(np.random.default_rng(4).choice(m.nnz, 128, replace=False)).to(DEV)
    batch = ofs.sample_link_batch(A, pos, 4, [6, 3], 31, exclude="reverse")
    layers = [gcn.SAGEConv(nf, hid, activation="relu", seed=3, device=DEV),
              gcn.SAGEConv(hid, hid, activation=None, seed=5, device=DEV)]
    h = X[batch.blocks[0].src_nodes]
    for layer, blk in zip(layers, batch.blocks):
        h = layer(blk.adj, h)
    p = batch.pair
    assert h.shape[0] == p.cols
    score = ofs.edge_score(p.crow, p.col, h[batch.src_local], h, p.rows, p.cols)
    loss = torch.nn.functional.binary_cross_entropy_with_logits(score, batch.labels)
    loss.backward()
    # fp64 dense re-implementation on the same blocks: out = act(mean(x_j) W_neigh + x_i W_root + b)
    params64 = [[q.detach().double().cpu().requires_grad_() for q in layer.parameters()] for layer in layers]
    h64 = X.double().cpu()[batch.blocks[0].src_nodes.cpu()]
    for layer, blk, (wn, wr, b) in zip(layers, batch.blocks, params64):
        adj = blk.adj
        rr = torch.repeat_interleave(torch.arange(adj.rows), (adj.crow[1:] - adj.crow[:-1]).long().cpu())
        D = torch.zeros(adj.rows, adj.cols, dtype=torch.float64)
        D.index_put_((rr, adj.col.long().cpu()), torch.ones(rr.numel(), dtype=torch.float64), accumulate=True)
        mean = D @ h64 / D.sum(1, keepdim=True).clamp_min(1)
        h64 = mean @ wn + h64[:adj.rows] @ wr + b
        if layer.activation == "relu":
            h64 = torch.relu(h64)
    rows_of = torch.repeat_interleave(torch.arange(p.rows), (p.crow[1:] - p.crow[:-1]).long().cpu())
    s64 = (h64[batch.src_local.cpu()][rows_of] * h64[p.col.long().cpu()]).sum(1)
    loss64 = torch.nn.functional.binary_cross_entropy_with_logits(s64, batch.labels.double().cpu())
    loss64.backward()
    assert abs(float(loss) - float(loss64)) < 1e-4 * max(1.0, abs(float(loss64)))
    for layer, ps in zip(layers, params64):
        for q, q64 in zip(layer.parameters(), ps):
            assert torch.allclose(q.grad.double().cpu(), q64.grad, rtol=1e-3, atol=1e-5)
