"""Mini-batch neighbour sampling for GraphSAGE-style training (DESIGN.md §3.8).

``sample_blocks`` turns a batch of seed nodes into one bipartite block per layer, sampled hop by hop
on the device by ``ofspmm_sample_neighbors``.  A block's adjacency is an ordinary ``CsrMatrix``
(rows = destination nodes, columns = local ids into ``src_nodes``), so the SpMM path and
``gcn.SAGEConv`` consume it unchanged:

    blocks = sample_blocks(A, seeds, [25, 10], rng_seed=step)
    h = X[blocks[0].src_nodes]
    for layer, blk in zip(layers, blocks):
        h = layer(blk.adj, h)            # h now has one row per blk.adj.rows destination
    # h[i] is the output of seeds[i]

``sample_link_batch`` builds a link-prediction batch on top of it: device negative sampling,
blocks sampled from the pairs' endpoints with the predicted edges (and their reverses) excluded,
and a pair matrix whose dot-product scores ``functional.edge_score`` computes:

    batch = sample_link_batch(A, pos_eid, k=5, fanouts=[25, 10], rng_seed=step, exclude="reverse")
    h = X[batch.blocks[0].src_nodes]
    for layer, blk in zip(layers, batch.blocks):
        h = layer(blk.adj, h)
    p = batch.pair
    score = edge_score(p.crow, p.col, h[batch.src_local], h, p.rows, p.cols)
    loss = F.binary_cross_entropy_with_logits(score, batch.labels)
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Sequence

import torch

from . import ops
from .graphs import CsrMatrix

# Salt of the negative-sampling seed ("NEG_SAMP"), which keeps its draws apart from the hop seeds.
_NEG_SALT = 0x4E45475F53414D50

_M64 = (1 << 64) - 1


def mix64(x: int) -> int:
    """The sampler's 64-bit mixer on a Python int (mod 2^64): multiply by 0x9E3779B97F4A7C15, then
    the splitmix64 finaliser — ``graphs._mix64_`` on one value."""
    x = (x * 0x9E3779B97F4A7C15) & _M64
    x ^= x >> 30
    x = (x * 0xBF58476D1CE4E5B9) & _M64
    x ^= x >> 27
    x = (x * 0x94D049BB133111EB) & _M64
    return x ^ (x >> 31)


def hop_seed(rng_seed: int, hop: int) -> int:
    """Seed of hop ``hop`` (0 = the hop that samples the seeds' neighbours): mix(rng_seed + hop)."""
    return mix64((rng_seed + hop) & _M64)


@dataclass
class Block:
    """One sampled layer: ``adj`` is ``num_dst x num_src`` (int32 CSR, ``val`` None for a pattern
    matrix), its columns index ``src_nodes`` (global ids, A's index dtype), and
    ``src_nodes[:adj.rows]`` are the destination nodes themselves.  ``eid`` (with ``edge_ids=True``)
    is the position in A of every entry of ``adj``, so ``w[eid]`` are the block's weights for
    per-edge parameters ``w`` of the full graph, with gradients flowing back to ``w``."""
    adj: CsrMatrix
    src_nodes: torch.Tensor
    eid: Optional[torch.Tensor] = None

    @property
    def dst_nodes(self) -> torch.Tensor:
        return self.src_nodes[:self.adj.rows]


def sample_blocks(A: CsrMatrix, seeds: torch.Tensor, fanouts: Sequence[int], rng_seed: int, *,
                  prob: Optional[torch.Tensor] = None, replace: bool = False, edge_ids: bool = False,
                  exclude_eid: Optional[torch.Tensor] = None) -> List[Block]:
    """Samples ``len(fanouts)`` hops from ``seeds`` (distinct node ids of the square CSR ``A``, on
    its device).  Hop h starts from the previous hop's ``src_nodes`` and samples at most
    ``fanouts[h]`` neighbours per node (-1: all) with seed ``hop_seed(rng_seed, h)``.

    Returns the blocks input layer first: ``blocks[0]`` consumes ``X[blocks[0].src_nodes]`` and
    ``blocks[-1].src_nodes[:len(seeds)] == seeds``.  Deterministic in (A, seeds, fanouts, rng_seed).
    A's values, if any, are carried into the blocks; ``A.val`` None samples the pattern.

    ``prob`` (nnz weights, e.g. ``A.val``): weighted sampling without replacement; ``replace``:
    ``fanouts[h]`` uniform draws per node with repeats kept; ``edge_ids``: every block carries
    ``eid`` (see ``ops.sample_neighbors``); ``exclude_eid``: positions in A that no block of any hop
    contains (DGL's ``exclude=``), sorted and deduplicated here."""
    blocks = []
    nodes = seeds
    if exclude_eid is not None:
        exclude_eid = torch.unique(exclude_eid.to(A.crow.dtype))
    for hop, fanout in enumerate(fanouts):
        crow, col, val, src, *eid = ops.sample_neighbors(A.crow, A.col, A.val, A.rows, A.cols, nodes, int(fanout),
                                                         hop_seed(rng_seed, hop), prob=prob, replace=replace,
                                                         return_eid=edge_ids, exclude_eid=exclude_eid)
        blocks.append(Block(CsrMatrix(crow, col, val, int(nodes.numel()), int(src.numel())), src,
                            eid[0] if edge_ids else None))
        nodes = src
    return blocks[::-1]


@dataclass
class LinkBatch:
    """One link-prediction batch.  ``pair`` is an int32 pattern CSR with one row per positive edge
    i: its first entry is the local id of the edge's destination, the others those of its negatives
    that did not fail; columns index the seed nodes ``blocks[-1].dst_nodes`` (the sorted distinct
    endpoints), and ``src_local[i]`` is the local id of the edge's source.  ``labels`` (float32, one
    per entry of ``pair``) is 1 at each row's first entry and 0 after it."""
    pair: CsrMatrix
    src_local: torch.Tensor
    labels: torch.Tensor
    blocks: List[Block]

    @property
    def seeds(self) -> torch.Tensor:
        return self.blocks[-1].dst_nodes


def link_pairs(u: torch.Tensor, v: torch.Tensor, neg: torch.Tensor):
    """The pair matrix of positive edges (u[i], v[i]) and their negatives neg[i] (-1: failed), over
    the sorted distinct endpoints.  Returns (seeds, pair, src_local, labels), see ``LinkBatch``."""
    n, k = int(u.numel()), int(neg.shape[1])
    ok = torch.cat([torch.ones(n, 1, dtype=torch.bool, device=u.device), neg >= 0], 1)
    ends = torch.cat([v.view(n, 1).to(neg.dtype), neg], 1)
    seeds = torch.unique(torch.cat([u.to(neg.dtype), ends[ok]]))
    local = torch.searchsorted(seeds, ends.clamp_min(0)).to(torch.int32)
    row_len = ok.sum(1)
    crow = torch.zeros(n + 1, dtype=torch.int32, device=u.device)
    crow[1:] = torch.cumsum(row_len, 0)
    col = local[ok].contiguous()   # row-major: each row's destination, then its negatives in draw order
    labels = torch.zeros(col.numel(), dtype=torch.float32, device=u.device)
    labels[crow[:-1].long()] = 1.0
    src_local = torch.searchsorted(seeds, u.to(neg.dtype))
    return seeds, CsrMatrix(crow, col, None, n, int(seeds.numel())), src_local, labels


def sample_link_batch(A: CsrMatrix, pos_eid: torch.Tensor, k: int, fanouts: Sequence[int], rng_seed: int, *,
                      exclude: Optional[str] = "self", prob: Optional[torch.Tensor] = None, replace: bool = False,
                      edge_ids: bool = False) -> LinkBatch:
    """A link-prediction batch for the positive edges at positions ``pos_eid`` of the square CSR
    ``A`` (DGL's ``EdgeDataLoader`` / PyG's ``LinkNeighborLoader``): edge i is (u_i, v_i) with u_i
    its row and v_i = A.col[pos_eid[i]]; ``k`` negatives per edge from ``ops.negative_sample``
    (rejecting edges of A and self-loops; failed draws are left out of ``pair``); blocks sampled as
    ``sample_blocks`` does from the sorted distinct endpoints.  ``exclude``: which edges no block
    contains, so that the model cannot read the labels through message passing: "self" the
    positive edges, "reverse" also their reverses (v_i, u_i) where A has them, None nothing.
    Deterministic in (A, pos_eid, k, fanouts, rng_seed)."""
    if exclude not in ("self", "reverse", None):
        raise ValueError(f"exclude must be 'self', 'reverse' or None, got {exclude!r}")
    pos_eid = pos_eid.to(A.crow.dtype)
    u = torch.searchsorted(A.crow, pos_eid, right=True) - 1
    v = A.col[pos_eid.long()]
    neg, _ = ops.negative_sample(A.crow, A.col, A.rows, A.cols, u, k, mix64((rng_seed ^ _NEG_SALT) & _M64))
    seeds, pair, src_local, labels = link_pairs(u, v, neg)
    excl = None
    if exclude is not None:
        excl = pos_eid
        if exclude == "reverse":
            rev = ops.edge_ids(A.crow, A.col, A.rows, A.cols, v, u)
            excl = torch.cat([pos_eid, rev[rev >= 0]])
    blocks = sample_blocks(A, seeds, fanouts, rng_seed, prob=prob, replace=replace, edge_ids=edge_ids,
                           exclude_eid=excl)
    return LinkBatch(pair, src_local, labels, blocks)
