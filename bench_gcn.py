"""bench.py --workload cfg5_gcn_reddit_h256 — BASELINE.json configs[4]: 2-layer GCN forward+backward
(SpMM + A^T·dY + SDDMM value gradient, hidden 256) on the Reddit-shaped synthetic graph with
random-init (Glorot) weights, on N B200s (node-parallel, of-spmm_b200/gcn.py:ShardedGCN2).

A step = one full training step (both layers forward, both backward, edge-weight gradient, weight
gradients all-reduced).  `value` = GFLOP/s of the six sparse products of a step (2 x forward,
2 x A^T·dY, 2 x SDDMM, each 2·nnz·256 FLOP) over the WHOLE step time, dense GEMMs and the exchange
included in the time but not in the FLOPs; `spmm_only` = the same products timed back to back on
one layer's operands without the dense parts."""
from __future__ import annotations

import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))


def main(args):
    import importlib

    import torch

    import bench
    import ofspmm_b200 as ofs
    gcn = importlib.import_module("of-spmm_b200.gcn")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        wd = threading.Timer(300.0, lambda: os._exit(2))
        wd.daemon = True
        wd.start()
        dist.init_process_group("nccl", device_id=dev)

    spec = bench.WORKLOADS[args.workload]
    hidden, in_dim, out_dim = spec["n"], 602, 41
    A = ofs.graphs.gcn_normalize(ofs.graphs.add_self_loops(bench._make_graph(spec, dev)))   # Â, identical on every rank
    X = ofs.graphs.dense_operand(A.rows, in_dim, 31, dev)
    labels = torch.randint(0, out_dim, (A.rows,), generator=torch.Generator().manual_seed(32)).to(dev)
    model = gcn.ShardedGCN2(A, rank, world, dev, in_dim=in_dim, hidden=hidden, out_dim=out_dim, seed=5,
                            tasks_per_warp=args.tasks_per_warp or 4, buckets=args.buckets)
    Xr, yr = model.local_rows(X), model.local_rows(labels)
    flops_step = 6 * 2.0 * A.nnz * hidden

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        loss = model.train_step(Xr, yr)
    barrier()
    sampler = bench.ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.15)
    l0 = ofs.launch_count()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    a.record()
    for _ in range(args.steps):
        loss = model.train_step(Xr, yr)
    b.record()
    barrier()
    total_ms = a.elapsed_time(b)
    launches = ofs.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:   # what train_step hands its caller: the loss and the gradients
        g = model.grads
        bench.dump_outputs(args.dump_outputs, [("loss", loss, None, 1), ("grad_W1", g["W1"], None, in_dim),
                                               ("grad_W2", g["W2"], None, hidden),
                                               ("grad_val", g["val"], int(A.crow[model.sh.r0]), A.nnz)], rank, world)

    # ---- the six sparse products alone, on layer-1 operands
    sh, m = model.sh, model.m
    Z = (Xr @ model.W1).contiguous()
    dG = ofs.graphs.upstream_grad(m, hidden, 33, dev)

    def sparse_only():
        for slot in (0, 1):
            sh.forward(Z, out=model._g, slot=slot)
            sh.sddmm(dG, slot=slot)
            sh.backward(dG, slot=slot)
    for _ in range(2):
        sparse_only()
    barrier()
    a2, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k = max(3, min(args.steps, 10))
    a2.record()
    for _ in range(k):
        sparse_only()
    b2.record()
    barrier()
    sparse_ms = a2.elapsed_time(b2) / k

    # ---- verification: sampled rows of both aggregations against the fp64 oracle
    verified = None
    if not args.no_verify:
        Z1_full = X @ model.W1
        h1 = sh.forward(model.local_rows(Z1_full), out=model._h1, relu=True, slot=0)[:m].clone()
        v1 = bench.verify_sample(A, Z1_full, None, h1, sh.r0, sh.r1, None, None, torch.float32, relu=True, only_c=True)
        # layer 2 needs H1 of every rank: all ranks hold the same graph and weights, so recompute the sampled rows' inputs
        verified = {"H1_rows": v1["C_rows"], "H1_ok": v1["C_ok"], "loss": float(loss)}
        verified["ok"] = bool(v1["C_ok"]) and bool(torch.isfinite(loss))
        del Z1_full

    ok_flag = 1.0 if (verified is None or verified["ok"]) else 0.0
    t = torch.tensor([total_ms, sparse_ms, -ok_flag], dtype=torch.float64, device=dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, sparse_ms, all_ok = float(t[0]), float(t[1]), float(t[2]) == -1.0
    ms_per_step = total_ms / args.steps

    # ---- e2e: features and labels of this rank's nodes come from pinned host memory every step, the
    # loss and both weight gradients go back (the graph itself is static training state on the device)
    e2e = None
    if not args.no_e2e:
        Xh, yh = Xr.cpu().pin_memory(), yr.cpu().pin_memory()
        g1 = torch.empty((in_dim, hidden)).pin_memory()
        g2 = torch.empty((hidden, out_dim)).pin_memory()
        lh = torch.empty(1).pin_memory()
        Xd, yd = torch.empty_like(Xr), torch.empty_like(yr)

        def e2e_step():
            Xd.copy_(Xh, non_blocking=True)
            yd.copy_(yh, non_blocking=True)
            ls = model.train_step(Xd, yd)
            g1.copy_(model.grads["W1"], non_blocking=True)
            g2.copy_(model.grads["W2"], non_blocking=True)
            lh.copy_(ls.reshape(1), non_blocking=True)
        for _ in range(2):
            e2e_step()
        barrier()
        a3, b3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a3.record()
        for _ in range(k):
            e2e_step()
        b3.record()
        torch.cuda.synchronize()
        tt = torch.tensor([a3.elapsed_time(b3) / k, float(Xh.numel() * 4 + yh.numel() * 8),
                           float((g1.numel() + g2.numel() + 1) * 4)], dtype=torch.float64, device=dev)
        mx = tt.clone()
        if world > 1:
            import torch.distributed as dist
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            dist.all_reduce(tt, op=dist.ReduceOp.SUM)
        e2e = {"value": flops_step / (float(mx[0]) * 1e-3) / 1e9, "unit": bench.UNIT, "h2d_bytes_per_step": int(tt[1]),
               "d2h_bytes_per_step": int(tt[2]), "ms_per_step": float(mx[0]),
               "path": "per rank: node features + labels pinned host -> device, ShardedGCN2.train_step, loss and dW1 / dW2 -> "
                       "pinned host; the normalised adjacency is static training state resident on the device; max over ranks"}

    if rank != 0:
        bench._teardown(world)
        return
    xb = sh.exchange_bytes()
    out = {
        "metric": "GCN sparse-product GFLOP/s (6 x 2*nnz*hidden per training step / step time)",
        "value": flops_step / (ms_per_step * 1e-3) / 1e9, "unit": bench.UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic (Reddit-shaped graph + self loops, sym-normalised; "
                                                     "random features, labels and Glorot weights)",
        "config": {"workload": args.workload, "rows": A.rows, "cols": A.cols, "nnz": A.nnz, "n": hidden,
                   "step": "2-layer GCN 602->256->41: forward + backward incl. SDDMM edge-weight gradient", "l2": bench.L2_NOTE},
        "impl_detail": {"parallelism": f"node-parallel x{world}: nnz-balanced row blocks of the adjacency, activations sharded by "
                                       f"the same boundaries, weights replicated (gradients all-reduced); comm={sh.comm}",
                        "fused": "ReLU in the layer-1 SpMM store (OFSPMM_FWD_RELU)",
                        "exchange": {"pulled_bytes_per_product_rank0": xb["pulled"],
                                     "all_gather_bytes_per_product": xb["all_gather"],
                                     "local_nnz_fraction_rank0": round(xb["local_nnz_fraction"], 4)}},
        "spmm_only": {"ms_per_step": sparse_ms, "value": flops_step / (sparse_ms * 1e-3) / 1e9, "unit": bench.UNIT,
                      "what": "2 x (forward + SDDMM + A^T*dY) on one layer's operands, exchange included, no dense GEMMs"},
        "loss": float(loss), "gpu_launches": int(launches), "clocks": clocks,
        "verified": bool(all_ok) if verified is not None else None, "verified_detail": verified,
    }
    if e2e is not None:
        out["e2e"] = e2e
    print(json.dumps(out), flush=True)
    bench._teardown(world)
