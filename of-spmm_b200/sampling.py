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
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Sequence

import torch

from . import ops
from .graphs import CsrMatrix

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
                  prob: Optional[torch.Tensor] = None, replace: bool = False, edge_ids: bool = False) -> List[Block]:
    """Samples ``len(fanouts)`` hops from ``seeds`` (distinct node ids of the square CSR ``A``, on
    its device).  Hop h starts from the previous hop's ``src_nodes`` and samples at most
    ``fanouts[h]`` neighbours per node (-1: all) with seed ``hop_seed(rng_seed, h)``.

    Returns the blocks input layer first: ``blocks[0]`` consumes ``X[blocks[0].src_nodes]`` and
    ``blocks[-1].src_nodes[:len(seeds)] == seeds``.  Deterministic in (A, seeds, fanouts, rng_seed).
    A's values, if any, are carried into the blocks; ``A.val`` None samples the pattern.

    ``prob`` (nnz weights, e.g. ``A.val``): weighted sampling without replacement; ``replace``:
    ``fanouts[h]`` uniform draws per node with repeats kept; ``edge_ids``: every block carries
    ``eid`` (see ``ops.sample_neighbors``)."""
    blocks = []
    nodes = seeds
    for hop, fanout in enumerate(fanouts):
        crow, col, val, src, *eid = ops.sample_neighbors(A.crow, A.col, A.val, A.rows, A.cols, nodes, int(fanout),
                                                         hop_seed(rng_seed, hop), prob=prob, replace=replace,
                                                         return_eid=edge_ids)
        blocks.append(Block(CsrMatrix(crow, col, val, int(nodes.numel()), int(src.numel())), src,
                            eid[0] if edge_ids else None))
        nodes = src
    return blocks[::-1]
