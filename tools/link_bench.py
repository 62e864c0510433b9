"""Link-prediction benchmark (profiles/link_bench.md): the device pieces of a link-prediction batch
on the full-size Reddit-shaped graph and on R-MAT scale 24, with 1024 and 8192 positive edges, k in
{1, 5} negatives per edge and fanouts [25, 10].  For every (graph, batch, k) it reports

  * neg_ms        ofspmm_negative_sample (k negatives per positive edge, edges of A and self-loops
                  rejected, 8 trials), CUDA events around `--reps` back-to-back calls;
  * edge_ids_ms   ofspmm_edge_ids on the batch's reverse pairs (v, u), the same way;
  * kernel_ms     both hops of the blocks (ofspmm_sample_neighbors, uniform) from the batch's
                  endpoints: `plain` without exclusion, timed before and after `reverse`, the same
                  calls with the positive edges and their reverses excluded;
  * blocks_ms     wall time of sampling.sample_blocks on those seeds, without and with the exclusion;
  * batch_ms      wall time of sampling.sample_link_batch(exclude="reverse") (negatives, lookup,
                  assembly and blocks, device-to-host reads included);
  * step_ms       one link-prediction train step on the batch: feature gather, two SAGEConv layers,
                  edge_score, BCE-with-logits, backward.

The device name and power limit are read in the same process as the timings.  Writes one JSON
document to --out (default: stdout)."""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
from importlib import import_module

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import ofspmm_b200 as ofs  # noqa: E402
from sample_bench import AbiCall, DEV, _device_info, _events_ms, _wall_ms  # noqa: E402

ops = import_module("of-spmm_b200.ops")
gcn = import_module("of-spmm_b200.gcn")
sampling = import_module("of-spmm_b200.sampling")
G = ofs.graphs
_lib = ofs._lib


def bench_graph(name, A, batches, ks, fanouts, reps, feat, hidden):
    P = G.CsrMatrix(A.crow, A.col, None, A.rows, A.cols)
    gen = torch.Generator().manual_seed(0)
    X = torch.randn(A.rows, feat, device=DEV)
    l1 = gcn.SAGEConv(feat, hidden, activation="relu", seed=1, device=DEV)
    l2 = gcn.SAGEConv(hidden, hidden, activation=None, seed=2, device=DEV)
    L = _lib.lib()
    rows = []
    for bs in batches:
        pos = torch.randint(0, P.nnz, (bs,), generator=gen).unique().to(DEV).to(P.crow.dtype)
        u = (torch.searchsorted(P.crow, pos, right=True) - 1).to(P.crow.dtype)
        v = P.col[pos.long()]
        Astruct = ops._csr_struct(P.crow, P.col, None, P.rows, P.cols)
        eid = torch.empty_like(u)
        edge_ids_ms = _events_ms(lambda: _lib.check(L.ofspmm_edge_ids(
            ctypes.byref(Astruct), v.data_ptr(), u.data_ptr(), u.numel(), eid.data_ptr(),
            torch.cuda.current_stream().cuda_stream), "edge_ids"), reps)
        rev = eid[eid >= 0]
        excl = torch.unique(torch.cat([pos, rev]))
        for k in ks:
            neg = torch.empty((u.numel(), k), dtype=P.crow.dtype, device=DEV)
            counts = torch.empty(2, dtype=torch.int64, device=DEV)
            neg_ms = _events_ms(lambda: _lib.check(L.ofspmm_negative_sample(
                ctypes.byref(Astruct), u.data_ptr(), u.numel(), k, 12345, _lib.NEG_EXCLUDE_EDGES | _lib.NEG_EXCLUDE_SELF,
                8, neg.data_ptr(), counts.data_ptr(), torch.cuda.current_stream().cuda_stream), "negative_sample"), reps)
            failed = int(counts[0])
            seeds, pair, src_local, labels = sampling.link_pairs(u, v, neg)
            # the blocks' kernels, uniform mode: plain, then excluded, then plain again (same process)
            plain = [AbiCall(P, seeds, fanouts[0], sampling.hop_seed(0, 0))]
            blocks = ofs.sample_blocks(P, seeds, fanouts, 0)
            plain.append(AbiCall(P, blocks[-1].src_nodes, fanouts[1], sampling.hop_seed(0, 1)))
            xblocks = ofs.sample_blocks(P, seeds, fanouts, 0, exclude_eid=excl)
            excluded = [AbiCall(P, seeds, fanouts[0], sampling.hop_seed(0, 0), exclude=excl),
                        AbiCall(P, xblocks[-1].src_nodes, fanouts[1], sampling.hop_seed(0, 1), exclude=excl)]
            plain_before = _events_ms(lambda: [c() for c in plain], reps)
            excl_ms = _events_ms(lambda: [c() for c in excluded], reps)
            plain_after = _events_ms(lambda: [c() for c in plain], reps)
            blocks_ms = _wall_ms(lambda r: ofs.sample_blocks(P, seeds, fanouts, r), reps)
            xblocks_ms = _wall_ms(lambda r: ofs.sample_blocks(P, seeds, fanouts, r, exclude_eid=excl), reps)
            batch_ms = _wall_ms(lambda r: sampling.sample_link_batch(P, pos, k, fanouts, r, exclude="reverse"), reps)
            batch = sampling.sample_link_batch(P, pos, k, fanouts, 0, exclude="reverse")

            def step(r):
                for p in l1.parameters() + l2.parameters():
                    p.grad = None
                h = X[batch.blocks[0].src_nodes.long()]
                h = l2(batch.blocks[1].adj, l1(batch.blocks[0].adj, h))
                pr = batch.pair
                s = ofs.edge_score(pr.crow, pr.col, h[batch.src_local], h, pr.rows, pr.cols)
                torch.nn.functional.binary_cross_entropy_with_logits(s, batch.labels).backward()
            step_ms = _wall_ms(step, reps)
            row = {"graph": name, "positives": int(pos.numel()), "k": k, "fanouts": fanouts,
                   "reverse_found": int(rev.numel()), "excluded": int(excl.numel()), "neg_failed": failed,
                   "seeds": int(seeds.numel()), "block_nnz_plain": [b.adj.nnz for b in blocks],
                   "block_nnz_excluded": [b.adj.nnz for b in xblocks],
                   "neg_ms": round(neg_ms, 4), "edge_ids_ms": round(edge_ids_ms, 4),
                   "kernel_ms_plain_before": round(plain_before, 4), "kernel_ms_reverse": round(excl_ms, 4),
                   "kernel_ms_plain_after": round(plain_after, 4), "blocks_ms_plain": round(blocks_ms, 4),
                   "blocks_ms_reverse": round(xblocks_ms, 4), "batch_ms": round(batch_ms, 4),
                   "step_ms": round(step_ms, 4)}
            print(json.dumps(row), flush=True)
            rows.append(row)
            del blocks, xblocks, plain, excluded, batch
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--batches", type=int, nargs="+", default=[1024, 8192])
    ap.add_argument("--ks", type=int, nargs="+", default=[1, 5])
    ap.add_argument("--fanouts", type=int, nargs="+", default=[25, 10])
    ap.add_argument("--rmat-scale", type=int, default=24)
    ap.add_argument("--reddit-div", type=int, default=1, help="reddit_like scale divisor (1 = full size)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "the link-prediction benchmark runs on the GPU"
    doc = {"device": _device_info(), "reps": a.reps, "features": {"in": 128, "hidden": 128}, "results": []}
    print(json.dumps(doc["device"]), flush=True)
    A = G.reddit_like(a.reddit_div, seed=2, device=DEV)
    doc["results"] += bench_graph(f"reddit_like/{a.reddit_div}", A, a.batches, a.ks, a.fanouts, a.reps, 128, 128)
    del A
    torch.cuda.empty_cache()
    A = G.rmat_csr(a.rmat_scale, device=DEV)
    doc["results"] += bench_graph(f"rmat_{a.rmat_scale}", A, a.batches, a.ks, a.fanouts, a.reps, 128, 128)
    text = json.dumps(doc, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    else:
        print(text)


if __name__ == "__main__":
    main()
