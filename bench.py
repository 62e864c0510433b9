#!/usr/bin/env python
"""bench.py — headline benchmark of the SpMM path (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME]
                    [--dump-outputs DIR]

A *step* is one pass of the hot path over the workload: SpMM forward C = A·B plus the A^T·dY
backward (BASELINE.json configs[1]: "forward + A^T·dY backward").  Default workload = configs[1]
(Reddit-shaped synthetic graph, 232 965 nodes, ~114.6 M nnz, dense N=128 fp32); configs[2] / [3] /
[4] are selectable with --workload.  For N>1 the same graph is partitioned into nnz-balanced row
blocks (one per rank), B / dB row-sharded, and every rank pulls only the B rows its block touches
out of the owners' HBM over NVLink while its local columns already compute (dist.ShardedSpmm;
strong scaling: total work fixed).

Prints ONE JSON line (rank 0).  `value` = GFLOP/s = flops of the whole job / max-over-ranks device
time, inputs resident in HBM.  `e2e` = the same metric through the public op API with pinned HOST
buffers, host<->device copies inside the timed region (max over ranks).  `roofline` is for the
dominant kernel (spmm_merge_kernel, forward) under the gather model M2 of SURVEY.md §8d, with the
ncu-measured DRAM and L2 bytes beside it; `cpu_baseline` is the oracle's OneFlow-style CPU loop on
this box's host cores; `verified` says that sampled rows of the timed outputs matched the oracle.

`--dump-outputs DIR` writes what the last timed step returned as DIR/<name>.npy, so that two builds
can be compared output for output on identical (seeded) inputs.  Once build() has run (it compiles
the CUDA library and the oracle), the benchmark writes nothing into the tree it runs from.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # no __pycache__ in the tree, which may be read-only

METRIC = "SpMM GFLOP/s (2*nnz*N/t), fwd + A^T*dY"
UNIT = "GFLOP/s"
STEP_DESC = "forward C=A*B + backward dB=A^T*dY"
L2_NOTE = ("inputs larger than L2 (CSR stream ~1 GB/step >> 126 MB); no flush between steps; cold-L2 forward "
           "reported as fwd_ms_cold_l2")
# L2 -> SM peak used for the second roofline entry: 184 L2 slices x 2 sectors/clk x 32 B x 1.964 GHz
# (ncu: lts__lts2xbar_cycles_active peak_sustained = 2 per slice, 184 slices active, profiles/r2_ncu_*.md)
L2_PEAK_GBS = 184 * 2 * 32 * 1.964
# --dump-outputs: all files together stay under 64 MB; the budget is split evenly between the outputs
DUMP_BYTES = 60 << 20

WORKLOADS = {
    "cfg2_reddit_n128_fp32": dict(kind="reddit", scale_div=1, n=128, dtype="fp32"),
    "cfg3_products_n256_bf16": dict(kind="products", scale_div=1, n=256, dtype="bf16"),
    "cfg4_rmat24_n128_fp32": dict(kind="rmat", scale=24, n=128, dtype="fp32"),
    "cfg1_uniform4096_n64_fp32": dict(kind="uniform", n=64, dtype="fp32"),
    "cfg5_gcn_reddit_h256": dict(kind="reddit", scale_div=1, n=256, dtype="fp32", gcn=True),
    "twin_reddit16_n128_fp32": dict(kind="reddit", scale_div=16, n=128, dtype="fp32"),
    "twin_rmat18_n128_fp32": dict(kind="rmat", scale=18, n=128, dtype="fp32"),
    "twin_gcn_reddit16_h256": dict(kind="reddit", scale_div=16, n=256, dtype="fp32", gcn=True),
}


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def _make_graph(spec, device):
    import ofspmm_b200 as ofs
    g = ofs.graphs
    if spec["kind"] == "reddit":
        return g.reddit_like(spec["scale_div"], seed=2, device=device)
    if spec["kind"] == "products":
        return g.products_like(spec["scale_div"], seed=3, device=device)
    if spec["kind"] == "rmat":
        return g.rmat_csr(spec["scale"], 16, seed=4, device=device)
    return g.uniform_csr(4096, 4096, 0.01, seed=1, device=device)


def _config(workload, A, n):
    """Identical in both arms (ours / reference) so the driver's same_config check holds."""
    return {"workload": workload, "rows": A.rows, "cols": A.cols, "nnz": A.nnz, "n": n, "step": STEP_DESC, "l2": L2_NOTE}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(self.idx)], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port (kind "port": the reference has no CPU SpMM kernel to compile,
# SURVEY.md §0.1) on all host cores

class CpuArm:
    """OneFlow-CPU-kernel-style loops (oracle/) on the FULL workload — no row-prefix extrapolation.
    Forward: rows split equally over the host threads (MultiThreadLoop + BalancedSplitter idiom,
    oneflow/core/thread/thread_manager.h:53-73).  A^T·dY: the same row-split loop on a CSR of A^T
    built once outside the timed region — the CPU twin of the cached transpose our op state holds,
    and unlike per-thread K x N accumulators it keeps scaling with the core count."""

    def __init__(self, A, B, dY, n):
        import numpy as np
        from oracle import oracle as O
        self.O, self.np = O, np
        try:
            O.lib(native=True)
            self.native = True
        except Exception:
            self.native = False
        self.cores = os.cpu_count() or 1
        self.crow, self.col, self.val = A.crow.cpu().numpy(), A.col.cpu().numpy(), A.val.float().cpu().numpy()
        self.B, self.dY = B.float().cpu().numpy(), dY.float().cpu().numpy()
        self.rows, self.cols, self.nnz, self.n = A.rows, A.cols, A.nnz, n
        t0 = time.perf_counter()
        tc, tcol, tv, _ = O.csr_transpose(self.crow, self.col, self.val, A.cols)
        self.t = (tc, tcol, tv)
        self.transpose_s = time.perf_counter() - t0

    def step(self, threads=None):
        th = threads or self.cores
        t0 = time.perf_counter()
        C = self.O.spmm_f32(self.crow, self.col, self.val, self.B, self.cols, threads=th, native=self.native)
        dB = self.O.spmm_f32(self.t[0], self.t[1], self.t[2], self.dY, self.rows, threads=th, native=self.native)
        secs = time.perf_counter() - t0
        self.last = (C, dB)
        return secs

    def single_thread_sample(self, frac=16):
        """The reference's default CPU_THREADING_RUNTIME is SEQ (CMakeLists.txt:54): the plain
        single-thread loops (forward + sequential scatter) on the first 1/frac of the rows."""
        rows1 = max(1, self.rows // frac)
        p1 = int(self.crow[rows1])
        t0 = time.perf_counter()
        self.O.spmm_f32(self.crow[:rows1 + 1], self.col[:p1], self.val[:p1], self.B, self.cols, threads=1, native=self.native)
        self.O.spmm_t_f32(self.crow[:rows1 + 1], self.col[:p1], self.val[:p1], self.dY[:rows1], self.cols, threads=1,
                          native=self.native)
        return 2.0 * 2.0 * p1 * self.n / max(time.perf_counter() - t0, 1e-9) / 1e9

    def describe(self, value, secs, reps):
        return {"value": value, "unit": UNIT, "cores": self.cores, "kind": "port",
                "sample": f"the full workload ({self.rows} rows, {self.nnz} nnz) x {reps} timed passes of {secs:.2f} s: fwd (rows "
                          f"split over {self.cores} threads) + A^T*dY (same loop on a CSR of A^T built once outside the timed "
                          f"region in {self.transpose_s:.1f} s, like the GPU arm's cached transpose); oracle built "
                          f"{'-march=native' if self.native else 'x86-64-v3'}"}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path.  /root/reference has
    no SpMM kernel and cannot be built offline (SURVEY.md §0.1-0.2), so this arm times the oracle
    port (OneFlow CPU-kernel idiom) on all host cores, every step the full workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    import ofspmm_b200 as ofs
    spec = WORKLOADS[args.workload]
    n = spec["n"]
    dev = "cuda:0" if torch.cuda.is_available() else "cpu"
    A = _make_graph(spec, dev)
    B = ofs.graphs.dense_operand(A.cols, n, 11, dev)
    dY = ofs.graphs.upstream_grad(A.rows, n, 12, dev)
    arm = CpuArm(A, B, dY, n)
    for _ in range(args.warmup):
        arm.step()
    times = [arm.step() for _ in range(args.steps)]
    if args.dump_outputs:
        C, dB = (torch.from_numpy(a) for a in arm.last)
        dump_outputs(args.dump_outputs, [("C", C, None, A.rows), ("dB", dB, None, A.cols)])
    secs = statistics.mean(times)
    flops = 2.0 * 2.0 * A.nnz * n
    v = flops / secs / 1e9
    base = arm.describe(v, secs, len(times))
    base["single_thread_value"] = arm.single_thread_sample()
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times),
        "warmup": args.warmup, "ms_per_step": secs * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": _config(args.workload, A, n),
        "impl_detail": {"parallelism": f"{arm.cores} host threads", "timed_passes": len(times),
                        "note": "every timed step is the full workload"},
        "cpu_baseline": base,
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------------
# verification of the timed outputs against the oracle (sampled rows, any size)

def verify_sample(A, B_full, dY_full, C_blk, r0, r1, dB_shard, shard_ids, dtype, nsample=256, seed=7, relu=False,
                  only_c=False):
    """>= nsample rows of C and of dB taken from the buffers the timed loop wrote, against the fp64
    oracle on exactly those rows (SURVEY.md §8c tolerances).  A / B_full / dY_full are the whole
    operands on this rank's device; C_blk = rows [r0, r1) of C; row i of dB_shard is row shard_ids[i]
    of dB (global ids, ascending — contiguous or block-cyclic ownership)."""
    import numpy as np
    import torch
    from oracle import oracle as O
    g = torch.Generator().manual_seed(seed)
    f32 = dtype == torch.float32
    res = {}
    # ---- C rows
    rows = torch.unique(torch.randint(r0, r1, (nsample,), generator=g)).to(A.crow.device)
    starts, ends = A.crow[rows].long(), A.crow[rows + 1].long()
    lens = ends - starts
    pos = torch.repeat_interleave(starts - torch.cumsum(lens, 0) + lens, lens) + torch.arange(int(lens.sum()), device=rows.device)
    col = A.col[pos].long()
    ok = (col >= 0) & (col < A.cols)
    ucol, inv = torch.unique(col[ok], return_inverse=True)
    mini_col = torch.full_like(col, -1)
    mini_col[ok] = inv
    crow = np.zeros(rows.numel() + 1, dtype=np.int64)
    crow[1:] = np.cumsum(lens.cpu().numpy())
    Bh = B_full[ucol].float().cpu().numpy() if ucol.numel() else np.zeros((1, B_full.shape[1]), np.float32)
    val = A.val[pos].float().cpu().numpy()
    want = O.spmm_f64(crow, mini_col.cpu().numpy(), val, Bh, max(1, ucol.numel()))
    amax = O.spmm_absmax(crow, mini_col.cpu().numpy(), val, Bh, max(1, ucol.numel()))
    if relu:
        want = np.maximum(want, 0.0)
    got = C_blk[(rows - r0)].float().cpu().numpy().astype(np.float64)
    tol = (O.fp32_tolerance(want, amax, np.diff(crow)) + 2.0 ** -21 * np.abs(want)) if f32 else (1e-2 * np.abs(want) + 2.0 ** -6 * amax)
    res["C_rows"] = int(rows.numel())
    res["C_ok"] = bool((np.abs(got - want) <= tol + 1e-30).all())
    if only_c:
        res["ok"] = res["C_ok"]
        return res
    # ---- dB rows (= columns of A): every non-zero of the sampled columns, over the whole matrix
    shard_ids = shard_ids.to(A.crow.device).long()
    pick = torch.unique(torch.randint(0, max(1, shard_ids.numel()), (nsample,), generator=g)).to(A.crow.device)
    cols_s = shard_ids[pick]                                   # ascending, like shard_ids
    hit = torch.isin(A.col, cols_s.to(A.col.dtype))
    p = torch.nonzero(hit).flatten()
    r_of = torch.searchsorted(A.crow.long(), p, right=True) - 1
    c_of = torch.searchsorted(cols_s, A.col[p].long())
    order = torch.argsort(c_of * (A.rows + 1) + r_of)
    p, r_of, c_of = p[order], r_of[order], c_of[order]
    urow, inv = torch.unique(r_of, return_inverse=True)
    tcrow = np.zeros(cols_s.numel() + 1, dtype=np.int64)
    tcrow[1:] = np.cumsum(torch.bincount(c_of, minlength=cols_s.numel()).cpu().numpy())
    dYh = dY_full[urow].float().cpu().numpy() if urow.numel() else np.zeros((1, dY_full.shape[1]), np.float32)
    tval = A.val[p].float().cpu().numpy()
    want = O.spmm_f64(tcrow, inv.cpu().numpy(), tval, dYh, max(1, urow.numel()))
    amax = O.spmm_absmax(tcrow, inv.cpu().numpy(), tval, dYh, max(1, urow.numel()))
    got = dB_shard[pick].float().cpu().numpy().astype(np.float64)
    # bf16 on several ranks: each rank's partial column sum is rounded to bf16 for transport
    tol = (O.fp32_tolerance(want, amax, np.diff(tcrow)) + 2.0 ** -20 * np.abs(want)) if f32 else \
        (1e-2 * np.abs(want) + 2.0 ** -7 * amax * (1 + np.sqrt(np.diff(tcrow)))[:, None])
    res["dB_rows"] = int(cols_s.numel())
    res["dB_ok"] = bool((np.abs(got - want) <= tol + 1e-30).all())
    res["ok"] = res["C_ok"] and res["dB_ok"]
    return res


def dump_outputs(path, outputs, rank=0, world=1):
    """--dump-outputs: each output as <path>/<name>.npy (float64 stays float64, everything else is
    written as float32).  ``outputs`` = [(name, tensor, where, rows)]: ``tensor`` holds rows of an
    output of ``rows`` rows in all; ``where`` says which — None (all of them, the same on every rank),
    an int (the global id of its first row, the rest follow contiguously) or a tensor of global row
    ids.  An output larger than its share of DUMP_BYTES is a seeded sample of its rows in ascending
    order, the same sample for every build and rank count.  Every rank calls this; rank 0 writes."""
    import math

    import numpy as np
    import torch
    share = DUMP_BYTES // len(outputs)
    for name, t, where, rows in outputs:
        dt = torch.float64 if t.dtype == torch.float64 else torch.float32
        row_bytes = math.prod(t.shape[1:]) * (8 if dt == torch.float64 else 4)
        sample = None
        if t.dim() > 0 and rows * row_bytes > share:
            g = torch.Generator().manual_seed(0)
            sample = torch.unique(torch.randint(0, rows, (max(1, share // row_bytes),), generator=g))
        if where is None:
            part = t if sample is None else t[sample.to(t.device)]
            part = part.detach().to(dt).cpu()
        else:
            if isinstance(where, int):
                ids = torch.arange(where, where + t.shape[0]) if sample is None else \
                    sample[(sample >= where) & (sample < where + t.shape[0])]
                pos = ids - where
            else:
                ids_all = where.cpu().long()
                pos = torch.arange(ids_all.numel()) if sample is None else torch.nonzero(torch.isin(ids_all, sample)).flatten()
                ids = ids_all[pos]
            pieces = [(ids, t[pos.to(t.device)].detach().to(dt).cpu())]
            if world > 1:
                import torch.distributed as dist
                gathered = [None] * world
                dist.all_gather_object(gathered, pieces[0])
                pieces = gathered
            ids = torch.cat([p[0] for p in pieces])
            part = torch.cat([p[1] for p in pieces])[torch.argsort(ids)]
        if rank == 0:
            os.makedirs(path, exist_ok=True)
            np.save(os.path.join(path, name + ".npy"), part.numpy())


# ------------------------------------------------------------------------------------------------
# e2e: host buffers in, host buffers out, copies inside the timed region

def _e2e_pipelined(args, ofs, ops, A, B, dY, n, dtype, dev, flops_step, blocks=8):
    """The CSR is streamed to the device in nnz-balanced row blocks (host twin of the partitioner);
    as soon as block i has landed, its forward rows C[r0:r1] = A_i·B and its contribution
    dB += A_i^T·dY_i (device transpose of the block, then the forward kernel in accumulate mode)
    run while block i+1 is still on the PCIe bus, and C blocks / dB go back on a third stream.
    Fresh inputs every step: nothing about the graph is cached across steps."""
    import torch
    host = {k: v.cpu().pin_memory() for k, v in dict(crow=A.crow, col=A.col, val=A.val, B=B, dY=dY).items()}
    C_h = torch.empty((A.rows, n), dtype=dtype).pin_memory()
    dB_h = torch.empty((A.cols, n), dtype=dtype).pin_memory()
    h2d = sum(v.numel() * v.element_size() for v in host.values())
    d2h = C_h.numel() * C_h.element_size() + dB_h.numel() * dB_h.element_size()
    d = {k: torch.empty_like(v, device=dev) for k, v in host.items()}
    C_d = torch.empty((A.rows, n), dtype=dtype, device=dev)
    dB_d = torch.empty((A.cols, n), dtype=dtype, device=dev)
    per_block_bwd = dtype == torch.float32   # fp32: dB accumulates block by block; bf16: one pass at the end
    bounds = ofs.row_blocks(host["crow"], A.nnz, blocks).tolist()      # host twin of the partitioner
    offs = [int(host["crow"][r]) for r in bounds]
    s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    torch.cuda.synchronize()

    def e2e_step():
        cur = torch.cuda.current_stream()
        s_in.wait_stream(cur)
        ev_in, ev_c = [], []
        with torch.cuda.stream(s_in):
            d["B"].copy_(host["B"], non_blocking=True)
            d["dY"].copy_(host["dY"], non_blocking=True)
            for i in range(blocks):
                r0, r1, p0, p1 = bounds[i], bounds[i + 1], offs[i], offs[i + 1]
                d["crow"][r0:r1 + 1].copy_(host["crow"][r0:r1 + 1], non_blocking=True)
                d["col"][p0:p1].copy_(host["col"][p0:p1], non_blocking=True)
                d["val"][p0:p1].copy_(host["val"][p0:p1], non_blocking=True)
                e = torch.cuda.Event()
                e.record(s_in)
                ev_in.append(e)
        first = True
        for i in range(blocks):
            r0, r1, p0, p1 = bounds[i], bounds[i + 1], offs[i], offs[i + 1]
            cur.wait_event(ev_in[i])
            if r1 > r0:
                crow_blk = d["crow"][r0:r1 + 1] - d["crow"][r0:r0 + 1]
                col_blk, val_blk = d["col"][p0:p1], d["val"][p0:p1]
                ops.spmm_csr_compute(crow_blk, col_blk, val_blk, d["B"], r1 - r0, A.cols, out=C_d[r0:r1])
                e = torch.cuda.Event()
                e.record(cur)
                ev_c.append((e, r0, r1))
                if per_block_bwd:
                    t = ops.csr_transpose(crow_blk, col_blk, val_blk, r1 - r0, A.cols)
                    ops.spmm_csr_compute(t[0], t[1], t[2], d["dY"][r0:r1], A.cols, r1 - r0, out=dB_d, accumulate=not first)
                    first = False
        if not per_block_bwd:   # 16-bit outputs: one pass over the whole A^T, a single rounding
            ops.spmm_csr_grad_b_transient_compute(d["crow"], d["col"], d["val"], d["dY"], A.rows, A.cols, out=dB_d)
        ev_b = torch.cuda.Event()
        ev_b.record(cur)
        with torch.cuda.stream(s_out):
            for e, r0, r1 in ev_c:
                s_out.wait_event(e)
                C_h[r0:r1].copy_(C_d[r0:r1], non_blocking=True)
            s_out.wait_event(ev_b)
            dB_h.copy_(dB_d, non_blocking=True)
        cur.wait_stream(s_out)

    for _ in range(3):
        e2e_step()
    torch.cuda.synchronize()
    k = max(3, min(args.steps, 10))
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(k):
        e2e_step()
    b.record()
    torch.cuda.synchronize()
    e2e_ms = a.elapsed_time(b) / k
    return ({"value": flops_step / (e2e_ms * 1e-3) / 1e9, "unit": UNIT, "h2d_bytes_per_step": h2d,
             "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms,
             "path": f"pinned host -> device in {blocks} nnz-balanced row blocks on a copy stream; per block, as it lands: "
                     "ofs spmm_csr (C rows) and csr_transpose + spmm_csr(accumulate) (dB += A_i^T*dY_i); C blocks / dB -> "
                     "pinned host on a third stream; nothing cached across steps"}, C_h, dB_h)


def _e2e_plugin_fwd(args, ofs, A, B, n, dtype, dev):
    """Forward only, through the C-ABI entry a host-tensor caller binds: ofspmm_fwd_host (host
    pointers in, host pointers out, staging carved from a caller-owned device workspace)."""
    import ctypes
    import torch
    L = ofs._lib.lib()
    crow, col, val, Bp = (t.cpu().pin_memory() for t in (A.crow, A.col, A.val, B))
    C_h = torch.empty((A.rows, n), dtype=dtype).pin_memory()
    dd = 2 if dtype == torch.float32 else 11
    cs = ofs._lib.CsrStruct(A.rows, A.cols, A.nnz, crow.data_ptr(), col.data_ptr(), val.data_ptr(), 5, 2)
    nbytes = L.ofspmm_fwd_host_workspace_bytes(A.rows, A.cols, A.nnz, n, dd, 5, 2)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream().cuda_stream

    def run():
        rc = L.ofspmm_fwd_host(ctypes.byref(cs), Bp.data_ptr(), C_h.data_ptr(), n, dd, ws.data_ptr(), nbytes, stream)
        assert rc == 0, rc
    for _ in range(2):
        run()
    torch.cuda.synchronize()
    k = 5
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(k):
        run()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / k
    h2d = sum(t.numel() * t.element_size() for t in (crow, col, val, Bp))
    return {"value": 2.0 * A.nnz * n / (ms * 1e-3) / 1e9, "unit": "GFLOP/s (forward only)", "ms_per_call": ms,
            "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": C_h.numel() * C_h.element_size(),
            "path": "ofspmm_fwd_host (C ABI): pinned host CSR + B -> device staging in the workspace, ofspmm_fwd, C -> pinned host"}


def _teardown(world):
    """Leave the process group without ever hanging the launcher: a watchdog force-exits if NCCL
    teardown does not return."""
    if world <= 1:
        return
    import torch.distributed as dist

    def _bail():
        sys.stdout.flush()
        os._exit(0)
    t = threading.Timer(20.0, _bail)
    t.daemon = True
    t.start()
    try:
        dist.destroy_process_group()
    except Exception:
        pass
    t.cancel()


def pick_runner(args, dmod, A, B, dY, n, dtype, rank, world, dev, compute=None, steps=10):
    """The sharded product for this workload at N > 1: by the byte-saving rule of
    ``dist.make_sharded`` and, where the rule says the exchange is dense (both schemes move the same
    bytes), by measurement at plan time.  ``compute`` / a CPU ``dev`` exist for the gloo test of
    this control flow (tests/test_bench_contract.py); the bench passes neither."""
    import torch
    import torch.distributed as dist
    cuda = torch.device(dev).type == "cuda"
    kw = dict(allgather_kw=dict(tasks_per_warp=args.tasks_per_warp or 2, static_order=not args.ag_dynamic_order),
              buckets=args.buckets, tasks_per_warp=args.tasks_per_warp or 4, pull_ctas=args.pull_ctas,
              shard_layout=args.layout, interleave=not args.no_interleave, combine_ctas=args.combine_ctas, compute=compute)
    tuned, saving = None, None
    dense = False
    if args.scheme == "auto":
        saving = dmod.needed_rows_saving(A, rank, world)
        dense = dtype == torch.float32 and saving < 0.25
    if args.scheme != "auto" or not dense or args.no_autotune:
        want = args.scheme if args.scheme != "auto" else ("allgather" if dense else "pull")
        runner, scheme, _ = dmod.make_sharded(A, n, dtype, rank, world, dev, scheme=want, **kw)
        return runner, scheme, saving, tuned

    # The exchange is dense (pulling only the needed rows saves nothing), so the two schemes move the
    # same bytes: settle it by measurement, at plan time, like any autotuner — untimed steps of each,
    # max over ranks, the same decision on every rank.  The needed-rows runner is the fallback if the
    # other one fails or disagrees with it.
    def sync():
        if cuda:
            torch.cuda.synchronize()

    def probe(r):
        b_in, dy_in = r.shard_rows(B), r.shard_rows_out(dY)
        for _ in range(3):
            r.step(b_in, dy_in)
        sync()
        dist.barrier()
        if cuda:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        t0 = time.perf_counter()
        for _ in range(steps):
            c, g = r.step(b_in, dy_in)
        if cuda:
            e1.record()
        sync()
        ms = e0.elapsed_time(e1) / steps if cuda else (time.perf_counter() - t0) * 1e3 / steps
        # the forward product alone (exchange included), for the record: an inference caller's number
        sync()
        dist.barrier()
        if cuda:
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record()
        t0 = time.perf_counter()
        for _ in range(steps):
            r.forward(b_in)
        if cuda:
            f1.record()
        sync()
        fms = f0.elapsed_time(f1) / steps if cuda else (time.perf_counter() - t0) * 1e3 / steps
        c, g = r.step(b_in, dy_in)                    # leave the buffers holding a full step's results
        sync()
        t = torch.tensor([ms, fms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1]), c, g

    runner, scheme, _ = dmod.make_sharded(A, n, dtype, rank, world, dev, scheme="pull", **kw)
    t_pull, f_pull, c_pull, g_pull = probe(runner)
    tuned = {"pull": t_pull, "pull_fwd_only": f_pull}
    # Candidates besides the plain needed-rows step: the same with the dB combine moved beside the
    # last forward pass (communication stream, 148 CTAs), and the collective scheme under three launch
    # policies of the products that run beside NCCL — round 1's measured optimum (static task order,
    # CTAs retire after 2 tasks per warp) and this round's default order with 2 and 4 tasks per warp.
    cands = []
    if args.tune_combine and not args.combine_ctas and not args.no_interleave:
        # opt-in: a second needed-rows runner (its own symmetric-memory buffers) alive beside the first
        cands.append(("pull[combine beside the last forward pass]", "pull", dict(kw, combine_ctas=148)))
    if args.tasks_per_warp or args.ag_dynamic_order:
        policies = [(args.tasks_per_warp or 2, not args.ag_dynamic_order)]
    else:
        policies = [(2, True), (2, False), (4, False)]
    for tpw, static in policies:
        cands.append((f"allgather[{'static' if static else 'dynamic'} order, {tpw} tasks/warp]", "allgather",
                      dict(kw, allgather_kw=dict(tasks_per_warp=tpw, static_order=static))))
    best_t, best_name, best_scheme = t_pull, None, "pull"
    other = c_ag = g_ag = None
    for name, sch, kw_c in cands:
        cand = None
        try:
            cand, _, _ = dmod.make_sharded(A, n, dtype, rank, world, dev, scheme=sch, **kw_c)
            t_ag, f_ag, c_ag, g_ag = probe(cand)
            tuned[name], tuned[name + " fwd_only"] = t_ag, f_ag
            # same inputs, independent exchange paths: they must agree to fp32 summation-order noise
            ok = torch.tensor([1.0], dtype=torch.float64, device=dev)
            ok *= float((c_ag - c_pull).abs().max()) <= 1e-4 * (float(c_pull.abs().max()) + 1e-30)
            if torch.equal(cand.shard_ids.cpu(), runner.shard_ids.cpu()):
                ok *= float((g_ag - g_pull).abs().max()) <= 1e-4 * (float(g_pull.abs().max()) + 1e-30)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            agree = bool(ok.item())
            tuned["schemes_agree"] = agree and tuned.get("schemes_agree", True)
            if agree and t_ag < best_t:
                best_t, best_name, best_scheme, other, cand = t_ag, name, sch, cand, other   # keep the best, drop the previous best
        except Exception as exc:  # pragma: no cover
            tuned[name + " error"] = repr(exc)[:200]
        del cand
        c_ag = g_ag = None
    if best_name is not None:
        runner, other, scheme = other, runner, best_scheme
        tuned["chosen"] = best_name
        if best_scheme == "allgather":
            tuned["allgather_policy"] = best_name
    else:
        tuned["chosen"] = "pull"
    del other, c_pull, g_pull, c_ag, g_ag
    import gc
    gc.collect()
    if cuda:
        torch.cuda.empty_cache()
    dist.barrier()
    return runner, scheme, saving, tuned



def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2_reddit_n128_fp32", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--tune-combine", action="store_true",
                    help="N>1, scheme auto: also time the needed-rows step with the combine beside the last forward pass")
    ap.add_argument("--no-autotune", action="store_true", help="N>1, scheme auto: decide by the byte-saving rule alone")
    ap.add_argument("--ag-dynamic-order", action="store_true", help="N>1, allgather: dynamic task order in the overlapped products")
    ap.add_argument("--scheme", default="auto", choices=["auto", "pull", "allgather"],
                    help="N>1: needed-rows pull over peer memory (default) or round 1's all-gather / reduce-scatter")
    ap.add_argument("--buckets", type=int, default=1, help="N>1, pull: remote column buckets (accumulate passes)")
    ap.add_argument("--tasks-per-warp", type=int, default=0,
                    help="N>1: CTAs of the overlapped products retire after k tasks (0: scheme default, 2 for allgather)")
    ap.add_argument("--pull-ctas", type=int, default=64, help="N>1, pull: grid cap of the peer-pull kernels")
    ap.add_argument("--no-interleave", action="store_true", help="N>1, pull: step = forward(); backward() back to back")
    ap.add_argument("--combine-ctas", type=int, default=0,
                    help="N>1, pull: >0 runs the dB combine beside the last forward pass with that many CTAs")
    ap.add_argument("--layout", default="auto", choices=["auto", "block", "cyclic"],
                    help="N>1, pull: ownership of B / dB rows (auto = block-cyclic when contiguous blocks would skew the egress)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (a seeded row sample of outputs "
                         "that would exceed 64 MB in all); bench_outputs/ in the tree is ignored by git")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(3, args.warmup)
    if args.impl == "reference":
        return run_reference(args)
    if WORKLOADS[args.workload].get("gcn"):
        import bench_gcn
        return bench_gcn.main(args)

    import torch
    import ofspmm_b200 as ofs
    ops = __import__("importlib").import_module("of-spmm_b200.ops")

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
        # a multi-rank run that stops making progress must not hold the box: hard exit after 5 min
        wd = threading.Timer(300.0, lambda: os._exit(2))
        wd.daemon = True
        wd.start()
        dist.init_process_group("nccl", device_id=dev)

    spec = WORKLOADS[args.workload]
    n = spec["n"]
    dtype = torch.float32 if spec["dtype"] == "fp32" else torch.bfloat16
    A = _make_graph(spec, dev)          # identical on every rank (seeded)
    B = ofs.graphs.dense_operand(A.cols, n, 11, dev, dtype)
    dY = ofs.graphs.upstream_grad(A.rows, n, 12, dev, dtype)
    s_dense = 4 if dtype == torch.float32 else 2
    alg = ofs.graphs.expected_alg_bytes(A.rows, A.cols, A.nnz, n, s_dense)
    flops_step = 2.0 * alg["flop"]      # forward + A^T·dY
    detail = {}

    if world > 1:
        dmod = __import__("importlib").import_module("of-spmm_b200.dist")
        runner, scheme, saving, tuned = pick_runner(args, dmod, A, B, dY, n, dtype, rank, world, dev)
        detail["scheme"] = {"requested": args.scheme, "used": scheme,
                            "needed_rows_saving_min_over_ranks": None if saving is None else round(saving, 4),
                            "autotune_ms_per_step": tuned,
                            "rule": "auto: 16-bit products, and graphs where pulling only the needed rows of B saves >= 25 % of an "
                                    "all-gather's bytes, take the needed-rows exchange over peer memory; fp32 products on graphs "
                                    "where every rank needs (nearly) every row are timed on both schemes before the timed region "
                                    "(10 steps each, max over ranks) and the faster one runs (profiles/r2_multigpu.md)"}
        if scheme == "pull":
            xb = runner.exchange_bytes()
            detail["step_order"] = ("interleaved" + (f", combine beside the last forward pass ({runner.combine_ctas} CTAs)"
                                                     if runner.combine_ctas else "")) if runner.interleave else "forward(); backward()"
            detail["shard_layout"] = runner.layout + (f" (blocks of {runner.cyc} rows dealt round-robin)" if runner.layout == "cyclic" else "")
            detail["exchange"] = {"pulled_bytes_per_product_rank0": xb["pulled"], "all_gather_bytes_per_product": xb["all_gather"],
                                  "local_nnz_fraction_rank0": round(xb["local_nnz_fraction"], 4)}
            parallelism = (f"row-block x{world} (nnz-balanced whole rows), B/dB row-sharded; needed-rows exchange over peer "
                           f"memory (comm={runner.comm}): local columns compute while {args.buckets} remote bucket(s) are pulled "
                           f"by one flag-synchronised TMA kernel (ofspmm_pull_rows_multi), then accumulate passes; dB partials "
                           f"published, then combined in rank order by one kernel (ofspmm_combine_rows_multi); the two "
                           f"products are interleaved in ShardedSpmm.step")
        else:
            parallelism = (f"row-block x{world} (nnz-balanced whole rows), B/dB row-sharded; ncclAllGather(B) hidden behind "
                           f"A^T*dY and ncclReduceScatter(dB) behind A*B, products launched as short-lived CTAs so the "
                           f"collectives get SMs ({(tuned or {}).get('allgather_policy') or f'{args.tasks_per_warp or 2} tasks/warp'}; "
                           f"comm={runner.comm})")
        B_in, dY_in = runner.shard_rows(B), runner.shard_rows_out(dY)
        step = lambda: runner.step(B_in, dY_in)
        fwd_only = lambda: runner.forward(B_in)
        plan_ms = None
        r0, r1, shard_ids = runner.r0, runner.r1, runner.shard_ids
        outputs = lambda: (runner._c, runner._db)
    else:
        t0 = time.perf_counter()
        plan = ops.SpmmPlan(A.crow, A.col, A.rows, A.cols, n, dtype, transpose=True)   # op state: built once
        torch.cuda.synchronize()
        plan_ms = (time.perf_counter() - t0) * 1e3
        C = torch.empty((A.rows, n), dtype=dtype, device=dev)
        dB = torch.empty((A.cols, n), dtype=dtype, device=dev)

        def fwd_only():
            ops.spmm_csr_compute(A.crow, A.col, A.val, B, A.rows, A.cols, out=C, plan=plan)

        def step():
            ops.spmm_csr_compute(A.crow, A.col, A.val, B, A.rows, A.cols, out=C, plan=plan)
            ops.spmm_csr_grad_b_compute(A.crow, A.col, A.val, dY, A.rows, A.cols, out=dB, plan=plan)
        parallelism = "single GPU"
        detail["variant"] = {"forward": plan.variant_name(), "backward (forward kernel on A^T)": plan.variant_name(True),
                             "chosen_from": "row-length histogram (ofspmm_row_hist -> ofspmm_choose_variant), plan built once",
                             "row_hist_log2": [int(x) for x in plan.hist.tolist()[:24]]}
        r0, r1, shard_ids = 0, A.rows, torch.arange(A.cols, device=dev)
        outputs = lambda: (C, dB)

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.15)
    launches0 = ofs.launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    barrier()
    ev[0].record()
    for i in range(args.steps):
        step()
    ev[1].record()
    barrier()
    total_ms = ev[0].elapsed_time(ev[1])
    launches = ofs.launch_count() - launches0
    if args.dump_outputs:
        c_out, db_out = outputs()
        dump_outputs(args.dump_outputs, [("C", c_out, r0, A.rows), ("dB", db_out, shard_ids, A.cols)], rank, world)
    # ---- the timed outputs are what gets verified (sampled rows vs the fp64 oracle)
    verified = None
    if not args.no_verify:
        c_out, db_out = outputs()
        verified = verify_sample(A, B, dY, c_out, r0, r1, db_out, shard_ids, dtype)
    # dominant kernel (forward): its own CUDA-event loop right after, same residency / clocks
    for _ in range(2):
        fwd_only()
    barrier()
    fa, fb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fa.record()
    for i in range(args.steps):
        fwd_only()
    fb.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    fwd_ms = fa.elapsed_time(fb) / args.steps

    ok_flag = 1.0 if (verified is None or verified["ok"]) else 0.0
    t = torch.tensor([total_ms, fwd_ms, -ok_flag], dtype=torch.float64, device=dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, fwd_ms, all_ok = float(t[0]), float(t[1]), float(t[2]) == -1.0
    ms_per_step = total_ms / args.steps
    value = flops_step / (ms_per_step * 1e-3) / 1e9

    # ---- cold-L2 forward (flush by writing 256 MB) for the record
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    cold = []
    for _ in range(min(5, args.steps)):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fwd_only(); b.record()
        torch.cuda.synchronize()
        cold.append(a.elapsed_time(b))
    del flush
    if world > 1:
        import torch.distributed as dist
        dist.barrier()

    # ---- e2e: pinned host buffers in and out, copies inside the timed region
    e2e, e2e_plugin = None, None
    if not args.no_e2e and world == 1:
        e2e, C_h, dB_h = _e2e_pipelined(args, ofs, ops, A, B, dY, n, dtype, dev, flops_step)
        if not args.no_verify:   # what came back to the host is checked too
            ve = verify_sample(A, B, dY, C_h.to(dev), 0, A.rows, dB_h.to(dev), torch.arange(A.cols, device=dev), dtype, seed=9)
            e2e["verified"] = ve["ok"]
        del C_h, dB_h
        if dtype == torch.float32:
            e2e_plugin = _e2e_plugin_fwd(args, ofs, A, B, n, dtype, dev)
    if not args.no_e2e and world > 1:
        # per rank: its CSR row block, B shard and dY block come from pinned host memory every step and
        # its C block / dB shard go back; time = max over ranks, bytes = sum over ranks.  Never let a
        # failure here cost the scaling numbers.
        try:
            import torch.distributed as dist
            blk = runner.A_blk
            host = {k: v.cpu().pin_memory() for k, v in dict(crow=blk.crow, col=blk.col, val=blk.val, B=B_in, dY=dY_in).items()}
            dst = dict(crow=blk.crow, col=blk.col, val=blk.val, B=B_in, dY=dY_in)
            C_h = torch.empty((blk.rows, n), dtype=dtype).pin_memory()
            dB_h = torch.empty((runner.shard, n), dtype=dtype).pin_memory()
            h2d = sum(v.numel() * v.element_size() for v in host.values())
            d2h = C_h.numel() * C_h.element_size() + dB_h.numel() * dB_h.element_size()

            def e2e_step():
                for key, src in host.items():
                    dst[key].copy_(src, non_blocking=True)
                if hasattr(runner, "update_values"):
                    runner.update_values(blk.val)          # the freshly copied values reach every sub-CSR
                c, g = runner.step(B_in, dY_in)
                C_h.copy_(c, non_blocking=True)
                dB_h.copy_(g, non_blocking=True)
            for _ in range(3):
                e2e_step()
            torch.cuda.synchronize()
            k = max(3, min(args.steps, 10))
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            dist.barrier()
            torch.cuda.synchronize()
            a.record()
            for _ in range(k):
                e2e_step()
            b.record()
            torch.cuda.synchronize()
            tt = torch.tensor([a.elapsed_time(b) / k, float(h2d), float(d2h)], dtype=torch.float64, device=dev)
            mx = tt.clone()
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            dist.all_reduce(tt, op=dist.ReduceOp.SUM)
            e2e_ms = float(mx[0])
            e2e = {"value": flops_step / (e2e_ms * 1e-3) / 1e9, "unit": UNIT, "h2d_bytes_per_step": int(tt[1]),
                   "d2h_bytes_per_step": int(tt[2]), "ms_per_step": e2e_ms,
                   "path": "per rank: pinned host -> device copies of its CSR row block (values re-split into the sub-CSRs), "
                           "B shard and dY block, the sharded step (structure plans cached: the graph is static across "
                           "steps), C block and dB shard -> pinned host; time = max over ranks, bytes = sum over ranks"}
        except Exception as exc:  # pragma: no cover
            e2e = {"value": None, "unit": UNIT, "h2d_bytes_per_step": None, "d2h_bytes_per_step": None,
                   "error": repr(exc)[:200]}

    if rank != 0:
        _teardown(world)
        return

    peak, peak_src = _peaks()
    fwd_bytes = alg["m2"] if world == 1 else alg["m2"] / world
    achieved = fwd_bytes / (fwd_ms * 1e-3) / 1e9
    traffic, l2_entry = None, None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")   # written by tools/ncu_summary.py from ncu --set full reports
    if world == 1 and os.path.exists(tpath):
        try:
            rec = json.load(open(tpath)).get(args.workload, {}).get("fwd")
            if rec:
                traffic = rec["dram_bytes"]
                l2_gbs = rec["l2_bytes"] / (fwd_ms * 1e-3) / 1e9
                l2_entry = {"bound": "l2", "achieved": l2_gbs, "peak": L2_PEAK_GBS, "unit": "GB/s", "frac": l2_gbs / L2_PEAK_GBS,
                            "traffic": rec["l2_bytes"], "kernel": rec["kernel"],
                            "peak_source": "ncu: 184 L2 slices x 2 sectors/clk x 32 B x 1.964 GHz (lts__lts2xbar peak_sustained)",
                            "dram_frac_of_measured_peak": rec["dram_bytes"] / (fwd_ms * 1e-3) / 1e9 / peak,
                            "l2_hit_pct": rec.get("l2_hit_pct"), "ncu_capture": rec.get("tag"),
                            "ncu_same_launch": {k: rec.get(k) for k in ("duration_ms_under_ncu", "l2_throughput_pct_ncu",
                                                                        "l2_slice_output_busy_pct_avg", "l2_slice_output_busy_pct_max",
                                                                        "dram_throughput_pct_ncu")}}
        except Exception:
            traffic = None
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32" if dtype == torch.float32 else "bf16", "data": "synthetic",
        "config": _config(args.workload, A, n),
        "impl_detail": dict(parallelism=parallelism, **detail),
        "fwd_ms": fwd_ms, "fwd_ms_cold_l2": statistics.mean(cold) if cold else None,
        "fwd_gflops": alg["flop"] / (fwd_ms * 1e-3) / 1e9,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "kernel": "spmm_merge_kernel (forward)", "peak_source": peak_src,
                     "model": "M2 gather model: nnz*(idx+val) + (M+1)*idx + nnz*N*s + M*N*s bytes per launch "
                              "(SURVEY.md 8d); B-row gathers are mostly L2 hits, so achieved may exceed the HBM copy "
                              "peak - `traffic` is the DRAM bytes ncu measured for one launch, roofline_l2 the resource "
                              "that binds when frac > 1",
                     "frac_of_nominal_8tbs": achieved / 8000.0,
                     "alg_bytes": fwd_bytes, "m1_compulsory_bytes": alg["m1"],
                     "m1_gbs": alg["m1"] / (fwd_ms * 1e-3) / 1e9 / max(1, world)},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "verified": bool(all_ok) if verified is not None else None,
        "verified_detail": verified,
        "reference_cuda_path": "n/a: the reference snapshot has no SpMM kernel and OneFlow does not build offline "
                               "(SURVEY.md 0.1-0.2); the CPU arm is `bench.py --impl reference`",
    }
    if l2_entry is not None:
        out["roofline_l2"] = l2_entry
    if plan_ms is not None:
        out["plan_ms_one_off"] = plan_ms
    if e2e is not None:
        out["e2e"] = e2e
    if e2e_plugin is not None:
        out["e2e_plugin_fwd"] = e2e_plugin
    if not args.no_cpu_baseline and world == 1:
        arm = CpuArm(A, B, dY, n)
        arm.step()
        ts = [arm.step() for _ in range(3)]
        secs = statistics.mean(ts)
        base = arm.describe(flops_step / secs / 1e9, secs, len(ts))
        base["single_thread_value"] = arm.single_thread_sample()
        out["cpu_baseline"] = base
    print(json.dumps(out), flush=True)
    _teardown(world)


if __name__ == "__main__":
    main()
