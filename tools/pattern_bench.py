"""Pattern matrices (no values array) against weighted ones, and the mean reduction, on the benchmark
graphs cfg2 (Reddit-shaped, N=128 fp32), cfg3 (products-shaped, N=256 bf16) and cfg4 (R-MAT-24,
N=128 fp32), built exactly as bench.py builds them.  Arms, alternated rep by rep, CUDA events around
each call, plan route (SpmmPlan with the histogram-chosen variant and cached A^T structure):

    fwd_weighted    C = A·B with A.val            fwd_pattern      C = A·B, a_val=None
    fwd_pattern_mean  reduce="mean"
    bwd_weighted    dB = A^T·dY (cached values)   bwd_pattern      dB = A^T·dY, a_val=None

Every compared pair is checked: pattern sum == weighted product with an all-ones array, bit for
bit (forward and A^T·dY); pattern mean == the pattern sum divided by the row lengths (within one
fp32 rounding pair).  Also reported: the M2 byte model (s_val = 0 for the pattern arms), the device
memory each side holds for A and its plan, the card name and power limit read in the same process.

    python tools/pattern_bench.py [--reps 20] [--warmup 5] [--out DIR]

The JSON goes to DIR/pattern_bench.json (default: a new temporary directory, printed at the end).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import torch  # noqa: E402

import ofspmm_b200 as ofs  # noqa: E402

ops = __import__("importlib").import_module("of-spmm_b200.ops")
G = ofs.graphs

CONFIGS = {
    "cfg2_reddit_n128_fp32": (lambda d: G.reddit_like(1, seed=2, device=d), 128, torch.float32),
    "cfg3_products_n256_bf16": (lambda d: G.products_like(1, seed=3, device=d), 256, torch.bfloat16),
    "cfg4_rmat24_n128_fp32": (lambda d: G.rmat_csr(24, 16, seed=4, device=d), 128, torch.float32),
}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True).stdout.strip().split(", ")
    return {"gpu": q[0], "power_limit_w": float(q[1])} if len(q) == 2 else {"gpu": torch.cuda.get_device_name(0)}


def nbytes(*ts):
    return sum(t.numel() * t.element_size() for t in ts if t is not None)


def time_arms(arms, reps, warmup):
    for _ in range(warmup):
        for f in arms.values():
            f()
    torch.cuda.synchronize()
    ms = {k: [] for k in arms}
    for _ in range(reps):
        for k, f in arms.items():            # alternated: one rep of every arm, then the next rep
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f()
            e1.record()
            e1.synchronize()
            ms[k].append(e0.elapsed_time(e1))
    return {k: {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v)} for k, v in ms.items()}


def bits(t):
    return t.view(torch.int32 if t.dtype == torch.float32 else torch.int16)


def run_config(name, reps, warmup):
    make, n, dt = CONFIGS[name]
    dev = "cuda:0"
    A = make(dev)
    B = G.dense_operand(A.cols, n, 11, dev, dt)
    dY = G.upstream_grad(A.rows, n, 12, dev, dt)
    plan_w = ops.SpmmPlan(A.crow, A.col, A.rows, A.cols, n, dt, transpose=True)
    plan_p = ops.SpmmPlan(A.crow, A.col, A.rows, A.cols, n, dt, transpose=True)
    C = torch.empty(A.rows, n, dtype=dt, device=dev)
    dB = torch.empty(A.cols, n, dtype=dt, device=dev)
    plan_w.transposed_values(A.val)        # the weighted plan route keeps A^T's values (part of its memory)
    arms = {
        "fwd_weighted": lambda: ops.spmm_csr_compute(A.crow, A.col, A.val, B, A.rows, A.cols, C, plan=plan_w),
        "fwd_pattern": lambda: ops.spmm_csr_compute(A.crow, A.col, None, B, A.rows, A.cols, C, plan=plan_p),
        "fwd_pattern_mean": lambda: ops.spmm_csr_compute(A.crow, A.col, None, B, A.rows, A.cols, C, plan=plan_p,
                                                         reduce="mean"),
        "bwd_weighted": lambda: ops.spmm_csr_grad_b_compute(A.crow, A.col, A.val, dY, A.rows, A.cols, out=dB, plan=plan_w),
        "bwd_pattern": lambda: ops.spmm_csr_grad_b_compute(A.crow, A.col, None, dY, A.rows, A.cols, out=dB, plan=plan_p),
    }
    t = time_arms(arms, reps, warmup)

    # outputs: pattern == explicit ones, bit for bit; mean == sum / len
    ones = torch.ones(A.nnz, dtype=torch.float32, device=dev)
    plan_o = ops.SpmmPlan(A.crow, A.col, A.rows, A.cols, n, dt, transpose=True)
    fp = ops.spmm_csr_compute(A.crow, A.col, None, B, A.rows, A.cols, plan=plan_p)
    fo = ops.spmm_csr_compute(A.crow, A.col, ones, B, A.rows, A.cols, plan=plan_o)
    bp = ops.spmm_csr_grad_b_compute(A.crow, A.col, None, dY, A.rows, A.cols, plan=plan_p)
    bo = ops.spmm_csr_grad_b_compute(A.crow, A.col, ones, dY, A.rows, A.cols, plan=plan_o)
    fm = ops.spmm_csr_compute(A.crow, A.col, None, B, A.rows, A.cols, plan=plan_p, reduce="mean")
    lens = A.row_lengths().to(dev).float().clamp(min=1)[:, None]
    mean_ref = fp.float() / lens
    mean_err = ((fm.float() - mean_ref).abs() / mean_ref.abs().clamp(min=1e-30)).max().item()
    del ones, plan_o
    checks = {"fwd_pattern_bits_equal_explicit_ones": bool(torch.equal(bits(fp), bits(fo))),
              "bwd_pattern_bits_equal_explicit_ones": bool(torch.equal(bits(bp), bits(bo))),
              "mean_max_rel_err_vs_sum_over_len": mean_err}

    s_dense, s_idx = (4 if dt == torch.float32 else 2), A.crow.element_size()
    m2_w = G.expected_alg_bytes(A.rows, A.cols, A.nnz, n, s_dense, 4, s_idx)["m2"]
    m2_p = G.expected_alg_bytes(A.rows, A.cols, A.nnz, n, s_dense, 0, s_idx)["m2"]
    struct = nbytes(A.crow, A.col, plan_w.part, plan_w.t_crow, plan_w.t_col, plan_w.t_perm, plan_w.t_part)
    mem = {"weighted_A_and_plan_bytes": struct + nbytes(A.val, plan_w._t_val),
           "pattern_A_and_plan_bytes": struct + nbytes(plan_p._t_val)}
    model = {"m2_bytes_weighted": m2_w, "m2_bytes_pattern": m2_p,
             "fwd_weighted_gbs": m2_w / t["fwd_weighted"]["median_ms"] / 1e6,
             "fwd_pattern_gbs": m2_p / t["fwd_pattern"]["median_ms"] / 1e6}
    spread = {k: (v["max_ms"] - v["min_ms"]) / v["median_ms"] for k, v in t.items()}
    res = {"config": name, "rows": A.rows, "cols": A.cols, "nnz": A.nnz, "n": n, "dtype": str(dt).replace("torch.", ""),
           "variant": plan_w.variant_name(), "times": t, "rel_spread": spread,
           "ratio_fwd_pattern_over_weighted": t["fwd_pattern"]["median_ms"] / t["fwd_weighted"]["median_ms"],
           "ratio_fwd_mean_over_sum": t["fwd_pattern_mean"]["median_ms"] / t["fwd_pattern"]["median_ms"],
           "ratio_bwd_pattern_over_weighted": t["bwd_pattern"]["median_ms"] / t["bwd_weighted"]["median_ms"],
           "checks": checks, "memory": mem, "byte_model": model}
    del A, B, dY, plan_w, plan_p, C, dB, fp, fo, bp, bo, fm
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None, help="output directory (default: a new temporary directory)")
    ap.add_argument("--configs", default=",".join(CONFIGS))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark times the GPU; there is nothing to measure without one"
    assert args.reps >= 20 and args.warmup >= 5
    out = {"card": card(), "reps": args.reps, "warmup": args.warmup,
           "method": "CUDA events per call, arms alternated rep by rep; inputs larger than L2, no flush",
           "results": [run_config(c, args.reps, args.warmup) for c in args.configs.split(",")]}
    out_dir = args.out or tempfile.mkdtemp(prefix="pattern_bench_")
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, "pattern_bench.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    for r in out["results"]:
        print(json.dumps({k: r[k] for k in ("config", "ratio_fwd_pattern_over_weighted", "ratio_fwd_mean_over_sum",
                                            "ratio_bwd_pattern_over_weighted", "checks", "rel_spread")}))
    print(json.dumps(out["card"]))
    print(f"wrote {path}")
    ok = all(r["checks"]["fwd_pattern_bits_equal_explicit_ones"] and r["checks"]["bwd_pattern_bits_equal_explicit_ones"]
             for r in out["results"])
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
