"""Cost of 64-bit task offsets: the forward on the wide test matrix (graphs.wide_csr: 2^31 + 2^25
non-zeros, int64 indices) against the two narrow row blocks it splits into at a task boundary,
which together do exactly the same tasks with 32-bit offsets.  N = 128 fp32, one explicit variant
for all three launches, the two sides alternated, CUDA events around each.  Prints one JSON line
with the card name and power limit read in the same process.

    python tools/wide_probe.py [--reps 20] [--warmup 3] > profiles/wide_probe.json
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import ofspmm_b200 as ofs  # noqa: E402

ops = __import__("importlib").import_module("of-spmm_b200.ops")
G, _lib = ofs.graphs, ofs._lib


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True).stdout.strip().split(", ")
    return {"gpu": q[0], "power_limit_w": float(q[1])} if len(q) == 2 else {"gpu": torch.cuda.get_device_name(0)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the probe times the GPU; there is nothing to measure without one"
    dev, n = "cuda:0", 128
    A = G.wide_csr(dev)
    M, K, nnz = A.rows, A.cols, A.nnz
    crow_h = A.crow.cpu().numpy()
    cand = np.arange(M // 4, M // 2)
    r = int(cand[(cand + crow_h[cand]) % 256 == 0][0])
    p = int(crow_h[r])
    blocks = [(A.crow[:r + 1], A.col[:p], A.val[:p], r), (A.crow[r:] - p, A.col[p:], A.val[p:], M - r)]
    hist = ops.row_hist(A.crow).cpu()
    v = _lib.lib().ofspmm_choose_variant((ctypes.c_int64 * 32)(*hist.tolist()), M, nnz, n, _lib.DTYPE_FLOAT)
    B = G.dense_operand(K, n, 31, dev)
    C = torch.empty(M, n, device=dev)
    # persistent plans and workspaces: the timed calls are the products alone
    wide = ops.SpmmPlan(A.crow, A.col, M, K, n, variant=v).prepared()
    narrow = [ops.SpmmPlan(c, k, m, K, n, variant=v).prepared() for c, k, _, m in blocks]
    outs = [C[:r], C[r:]]

    def run_wide():
        wide(A.val, B, C)

    def run_narrow():
        for f, (_, _, val, _), o in zip(narrow, blocks, outs):
            f(val, B, o)

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1)

    for _ in range(args.warmup):
        run_wide()
        run_narrow()
    tw, tn = [], []
    for _ in range(args.reps):
        tw.append(timed(run_wide))
        tn.append(timed(run_narrow))
    mw, mn = statistics.median(tw), statistics.median(tn)
    m2 = G.expected_alg_bytes(M, K, nnz, n, 4, 4, 8)["m2"]
    print(json.dumps({
        "probe": "wide_forward_vs_narrow_blocks", **card(), "rows": M, "cols": K, "nnz": nnz, "n": n,
        "dtype": "fp32", "idx": "int64", "split_row": r,
        "variant": _lib.lib().ofspmm_variant_name(v, M, nnz, n, _lib.DTYPE_FLOAT).decode(),
        "reps": args.reps, "wide_ms": round(mw, 3), "narrow_ms": round(mn, 3),
        "wide_ms_minmax": [round(min(tw), 3), round(max(tw), 3)],
        "narrow_ms_minmax": [round(min(tn), 3), round(max(tn), 3)],
        "wide_m2_gbs": round(m2 / mw / 1e6, 1), "narrow_m2_gbs": round(m2 / mn / 1e6, 1),
        "ratio_wide_over_narrow": round(mw / mn, 4), "target": 1.10,
        "l2": "B (512 MB) and the CSR stream exceed the 126 MB L2: no flush between passes",
    }))


if __name__ == "__main__":
    main()
