"""Neighbour-sampling benchmark (profiles/sample_bench.md): device sampling for mini-batch GraphSAGE
on the full-size Reddit-shaped graph and on R-MAT scale 24 (hub rows stress the whole-CTA path),
batches of 1024 and 8192 seeds, fanouts [25, 10].  For every (graph, batch) it reports

  * kernel_ms     the C-ABI calls of both hops (ofspmm_sample_neighbors), CUDA events around
                  `--reps` back-to-back calls on fixed inputs, per batch;
  * blocks_ms     wall time of sampling.sample_blocks per batch (device-to-host reads included),
                  host clock around a synchronised loop over `--reps` seeds;
  * torch_ms      a torch-only sampler of the same definition (include/ofspmm.h), outputs checked
                  equal to the library's on both hops;
  * step_ms       one mini-batch 2-layer SAGE train step on the blocks (feature gather, forward,
                  backward), so that sampling is seen as a share of the step.

The device name and power limit are read in the same process as the timings.  Writes one JSON
document to --out (default: stdout)."""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import time
from importlib import import_module

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import ofspmm_b200 as ofs  # noqa: E402

ops = import_module("of-spmm_b200.ops")
gcn = import_module("of-spmm_b200.gcn")
sampling = import_module("of-spmm_b200.sampling")
G = ofs.graphs
_lib = ofs._lib
DEV = "cuda:0"


def _signed(x: int) -> int:
    x &= (1 << 64) - 1
    return x - (1 << 64) if x >= 1 << 63 else x


def torch_sample(crow, col, val, rows, dst, fanout, seed):
    """The sampling definition of include/ofspmm.h in plain torch on the device (valid, distinct dst)."""
    dev = crow.device
    d = dst.long()
    n = d.numel()
    b = crow[d].long()
    deg = crow[d + 1].long() - b
    k = deg if fanout == -1 else deg.clamp(max=fanout)
    total = int(deg.sum())
    row = torch.repeat_interleave(torch.arange(n, device=dev), deg, output_size=total)
    start = torch.cumsum(deg, 0) - deg
    j = torch.arange(total, device=dev) - start[row]
    pos = b[row] + j
    h0 = G._mix64_(torch.full((n,), _signed(seed), dtype=torch.int64, device=dev) ^ d)
    key = G._mix64_(h0[row] + j) ^ torch.iinfo(torch.int64).min   # unsigned order as signed order
    order = torch.argsort(key, stable=True)                       # ties keep ascending j
    order = order[torch.argsort(row[order], stable=True)]         # rows, each sorted by (key, j)
    rank = torch.empty_like(order)
    rank[order] = torch.arange(total, device=dev) - start[row[order]]
    c = col[pos].long()
    keep = (rank < k[row]) & (c >= 0) & (c < rows)
    kc = c[keep]
    blk_crow = torch.zeros(n + 1, dtype=torch.int32, device=dev)
    blk_crow[1:] = torch.cumsum(torch.bincount(row[keep], minlength=n), 0)
    uniq = torch.unique(kc)
    tail = uniq[~torch.isin(uniq, d)]
    src = torch.cat([d, tail]).to(crow.dtype)
    sd, perm = torch.sort(d)
    at = torch.searchsorted(sd, kc).clamp(max=max(n - 1, 0))
    local = torch.where(sd[at] == kc, perm[at], n + torch.searchsorted(tail, kc)).to(torch.int32)
    return blk_crow, local, (val[pos[keep]] if val is not None else None), src


def torch_blocks(A, seeds, fanouts, seed):
    out, nodes = [], seeds
    for h, f in enumerate(fanouts):
        r = torch_sample(A.crow, A.col, A.val, A.rows, nodes, f, sampling.hop_seed(seed, h))
        out.append(r)
        nodes = r[3]
    return out[::-1]


def _device_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


class AbiCall:
    """One preallocated ofspmm_sample_neighbors call (what the kernel timing launches)."""

    def __init__(self, A, dst, fanout, seed):
        self.keep = (A, dst)
        self.A = ops._csr_struct(A.crow, A.col, A.val, A.rows, A.cols)
        n = dst.numel()
        cap = min(n * fanout, A.nnz)
        self.args = (dst, n, fanout, seed, cap)
        self.bufs = [torch.empty(n + 1, dtype=torch.int32, device=DEV), torch.empty(cap, dtype=torch.int32, device=DEV),
                     None if A.val is None else torch.empty(cap, dtype=A.val.dtype, device=DEV),
                     torch.empty(n + cap, dtype=A.crow.dtype, device=DEV), torch.empty(3, dtype=torch.int64, device=DEV)]
        L = _lib.lib()
        self.ws_bytes = L.ofspmm_sample_neighbors_workspace_bytes(n, cap, ops._INDEX[A.crow.dtype])
        self.ws = torch.empty(self.ws_bytes, dtype=torch.uint8, device=DEV)

    def __call__(self):
        dst, n, fanout, seed, cap = self.args
        b = self.bufs
        _lib.check(_lib.lib().ofspmm_sample_neighbors(
            ctypes.byref(self.A), dst.data_ptr(), n, fanout, seed, cap, b[0].data_ptr(), b[1].data_ptr(),
            None if b[2] is None else b[2].data_ptr(), b[3].data_ptr(), b[4].data_ptr(), self.ws.data_ptr(),
            self.ws_bytes, torch.cuda.current_stream().cuda_stream), "sample_neighbors")


def _events_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def _wall_ms(fn, reps):
    fn(0)
    torch.cuda.synchronize()
    t = time.perf_counter()
    for r in range(reps):
        fn(r + 1)
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3 / reps


def bench_graph(name, A, batches, fanouts, reps, feat, hidden, classes):
    P = G.CsrMatrix(A.crow, A.col, None, A.rows, A.cols)   # GraphSAGE samples the pattern
    gen = torch.Generator().manual_seed(0)
    X = torch.randn(A.rows, feat, device=DEV)
    labels = torch.randint(0, classes, (A.rows,), device=DEV)
    l1 = gcn.SAGEConv(feat, hidden, activation="relu", seed=1, device=DEV)
    l2 = gcn.SAGEConv(hidden, classes, activation=None, seed=2, device=DEV)
    rows = []
    for bs in batches:
        seeds = torch.randperm(A.rows, generator=gen)[:bs].to(DEV)
        blocks = ofs.sample_blocks(P, seeds, fanouts, 0)
        # the torch sampler must produce the same blocks
        ref = torch_blocks(P, seeds.to(A.crow.dtype), fanouts, 0)
        same = all(torch.equal(b.adj.crow, r[0]) and torch.equal(b.adj.col, r[1]) and torch.equal(b.src_nodes, r[3])
                   for b, r in zip(blocks, ref))
        # kernel time: both hops through the C ABI on the inputs of this batch
        calls = [AbiCall(P, seeds.to(A.crow.dtype), fanouts[0], sampling.hop_seed(0, 0)),
                 AbiCall(P, blocks[-1].src_nodes, fanouts[1], sampling.hop_seed(0, 1))]
        kernel_ms = _events_ms(lambda: [c() for c in calls], reps)
        blocks_ms = _wall_ms(lambda r: ofs.sample_blocks(P, seeds, fanouts, r), reps)
        torch_ms = _wall_ms(lambda r: torch_blocks(P, seeds.to(A.crow.dtype), fanouts, r), max(3, reps // 4))

        def step(r):
            for p in l1.parameters() + l2.parameters():
                p.grad = None
            h = X[blocks[0].src_nodes.long()]
            out = l2(blocks[1].adj, l1(blocks[0].adj, h))
            torch.nn.functional.cross_entropy(out, labels[seeds]).backward()
        step_ms = _wall_ms(step, reps)
        row = {"graph": name, "batch": bs, "fanouts": fanouts,
               "block_rows": [b.adj.rows for b in blocks], "block_cols": [b.adj.cols for b in blocks],
               "block_nnz": [b.adj.nnz for b in blocks],
               "kernel_ms": round(kernel_ms, 4), "blocks_ms": round(blocks_ms, 4), "torch_ms": round(torch_ms, 4),
               "torch_equal": bool(same), "step_ms": round(step_ms, 4),
               "sampling_share": round(blocks_ms / (blocks_ms + step_ms), 4),
               "launches_per_batch": None}
        before = ofs.launch_count()
        ofs.sample_blocks(P, seeds, fanouts, 99)
        row["launches_per_batch"] = ofs.launch_count() - before
        print(json.dumps(row), flush=True)
        rows.append(row)
        del blocks, ref, calls
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--batches", type=int, nargs="+", default=[1024, 8192])
    ap.add_argument("--fanouts", type=int, nargs="+", default=[25, 10])
    ap.add_argument("--rmat-scale", type=int, default=24)
    ap.add_argument("--reddit-div", type=int, default=1, help="reddit_like scale divisor (1 = full size)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "the sampling benchmark runs on the GPU"
    doc = {"device": _device_info(), "reps": a.reps, "features": {"in": 128, "hidden": 128, "classes": 41}, "results": []}
    print(json.dumps(doc["device"]), flush=True)
    A = G.reddit_like(a.reddit_div, seed=2, device=DEV)
    doc["results"] += bench_graph(f"reddit_like/{a.reddit_div}", A, a.batches, a.fanouts, a.reps, 128, 128, 41)
    del A
    torch.cuda.empty_cache()
    A = G.rmat_csr(a.rmat_scale, device=DEV)
    doc["rmat_max_degree"] = int(torch.diff(A.crow).max())
    doc["results"] += bench_graph(f"rmat_{a.rmat_scale}", A, a.batches, a.fanouts, a.reps, 128, 128, 41)
    text = json.dumps(doc, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")
    else:
        print(text)


if __name__ == "__main__":
    main()
