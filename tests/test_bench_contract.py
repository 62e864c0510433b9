"""The reference arm of bench.py (`--impl reference`) needs no GPU: check its one-line JSON contract
here, on BASELINE configs[0] (the reference's own CPU-runnable case)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None, extra_args=(), steps=2):
    env = dict(os.environ)
    env.update(extra_env or {})
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload",
                          "cfg1_uniform4096_n64_fp32", "--steps", str(steps), "--warmup", "3", *extra_args],
                         capture_output=True, text=True, env=env, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    return out.stdout.strip().splitlines()


def test_reference_arm_json_contract():
    lines = _run()
    assert len(lines) == 1                                   # exactly ONE JSON line
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["unit"] == "GFLOP/s" and j["higher_is_better"] is True
    assert j["metric"].startswith("SpMM GFLOP/s") and j["value"] > 0 and j["ms_per_step"] > 0
    assert j["config"]["workload"] == "cfg1_uniform4096_n64_fp32" and j["config"]["n"] == 64
    cb = j["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == j["value"] and "rows" in cb["sample"]
    assert j["e2e"] == {"value": j["value"], "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert j["vs_baseline"] is None and j["data"] == "synthetic"


def test_reference_arm_times_exactly_steps_passes():
    j = json.loads(_run(steps=7)[0])
    assert j["steps"] == j["impl_detail"]["timed_passes"] == 7
    assert "7 timed passes" in j["cpu_baseline"]["sample"]


def test_reference_arm_only_rank0_works_under_torchrun_env():
    # ranks != 0 exit 0 without output (the driver launches the arm with torchrun for N > 1)
    assert _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}) == []


def test_dump_outputs_writes_what_the_last_step_computed(tmp_path):
    import numpy as np
    sys.path.insert(0, ROOT)
    import ofspmm_b200 as ofs
    from oracle import oracle as O
    d = tmp_path / "out"
    # no visible GPU: the arm then builds its inputs with the CPU generators, as below
    assert len(_run({"CUDA_VISIBLE_DEVICES": ""}, ("--dump-outputs", str(d)))) == 1
    assert sorted(os.listdir(d)) == ["C.npy", "dB.npy"]
    C, dB = np.load(d / "C.npy"), np.load(d / "dB.npy")
    assert C.dtype == dB.dtype == np.float32 and C.shape == dB.shape == (4096, 64)
    # the inputs bench.py builds for this workload
    A = ofs.graphs.uniform_csr(4096, 4096, 0.01, seed=1)
    B, dY = ofs.graphs.dense_operand(A.cols, 64, 11).numpy(), ofs.graphs.upstream_grad(A.rows, 64, 12).numpy()
    crow, col, val = A.crow.numpy(), A.col.numpy(), A.val.numpy()
    C64 = O.spmm_f64(crow, col, val, B, A.cols)
    assert (np.abs(C - C64) <= O.fp32_tolerance(C64, O.spmm_absmax(crow, col, val, B, A.cols), np.diff(crow)) + 1e-30).all()
    dB64 = O.spmm_t_f64(crow, col, val, dY, A.cols)
    amax, cnt = O.spmm_t_absmax(crow, col, val, dY, A.cols)
    assert (np.abs(dB - dB64) <= O.fp32_tolerance(dB64, amax, cnt) + 1e-30).all()


def test_dump_outputs_row_sample_is_the_same_for_every_layout(tmp_path, monkeypatch):
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 4 * 100 * 8 * 4)       # 100 fp32 rows of 8 per output
    T = torch.arange(1000, dtype=torch.float32)[:, None].repeat(1, 8)   # row i holds i
    full, part = tmp_path / "full", tmp_path / "part"
    bench.dump_outputs(str(full), [("X", T, None, 1000), ("Y", T, torch.arange(1000), 1000),
                                   ("Z", T.double(), None, 1000), ("s", torch.tensor(2.5), None, 1)])
    X = np.load(full / "X.npy")
    ids = X[:, 0]
    assert X.dtype == np.float32 and 0 < len(ids) <= 100 and (np.diff(ids) > 0).all() and (X == ids[:, None]).all()
    assert np.array_equal(np.load(full / "Y.npy"), X)
    Z = np.load(full / "Z.npy")
    assert Z.dtype == np.float64 and 0 < len(Z) <= 50
    assert np.load(full / "s.npy") == np.float32(2.5)
    # what one rank of several holds (rows 300.. contiguous, or every third row) dumps the same rows
    bench.dump_outputs(str(part), [("X", T[300:], 300, 1000), ("Y", T[::3], torch.arange(0, 1000, 3), 1000),
                                   ("Z", T.double(), None, 1000), ("s", torch.tensor(2.5), None, 1)])
    assert np.array_equal(np.load(part / "X.npy"), X[ids >= 300])
    assert np.array_equal(np.load(part / "Y.npy"), X[ids % 3 == 0])


DUMP_TEST_BYTES = 2 * 300 * 8 * 4       # about 300 sampled rows of C and of dB (n = 8, fp32)


def _dump_worker(rank, world, port, layout, out, q):
    import importlib

    import torch
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import bench
        import ofspmm_b200 as ofs
        from test_dist_cpu import OracleCompute
        dmod = importlib.import_module("of-spmm_b200.dist")
        bench.DUMP_BYTES = DUMP_TEST_BYTES
        A = ofs.graphs.rmat_csr(10, 12, seed=4)
        B, dY = ofs.graphs.dense_operand(A.cols, 8, 5), ofs.graphs.upstream_grad(A.rows, 8, 6)
        sh = dmod.ShardedSpmm(A, 8, torch.float32, rank, world, "cpu", compute=OracleCompute(), shard_layout=layout,
                              cyclic_block=16)
        sh.step(sh.shard_rows(B), sh.shard_rows_out(dY))
        # the buffers and row ids bench.py dumps on several ranks
        bench.dump_outputs(out, [("C", sh._c, sh.r0, A.rows), ("dB", sh._db, sh.shard_ids, A.cols)], rank, world)
        q.put((rank, sh.r0, sh.r1, sh.shard_ids.tolist()))
        dist.barrier()
        dist.destroy_process_group()
    except Exception:
        import traceback
        q.put(("error", rank, traceback.format_exc()))


@pytest.mark.parametrize("layout", ["block", "cyclic"])
def test_dump_outputs_gathers_rows_of_every_rank(tmp_path, monkeypatch, layout):
    import socket

    import numpy as np
    import torch
    import torch.multiprocessing as mp
    sys.path.insert(0, ROOT)
    import bench
    import ofspmm_b200 as ofs
    from oracle import oracle as O
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    out = str(tmp_path / "ranks")
    procs = [ctx.Process(target=_dump_worker, args=(r, 2, port, layout, out, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=240) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
    for r in res:
        assert r[0] != "error", r[2]
    assert res[0][1] == 0 and res[0][2] == res[1][1] > 0                  # C: two contiguous row blocks
    if layout == "cyclic":
        assert res[0][3] != list(range(len(res[0][3])))                   # dB: non-contiguous row ids
    # the same outputs from one process, whole
    A = ofs.graphs.rmat_csr(10, 12, seed=4)
    B, dY = ofs.graphs.dense_operand(A.cols, 8, 5).numpy(), ofs.graphs.upstream_grad(A.rows, 8, 6).numpy()
    C = O.spmm_f32(A.crow.numpy(), A.col.numpy(), A.val.numpy(), B, A.cols)
    dB = O.spmm_t_f32(A.crow.numpy(), A.col.numpy(), A.val.numpy(), dY, A.cols)
    monkeypatch.setattr(bench, "DUMP_BYTES", DUMP_TEST_BYTES)
    whole = str(tmp_path / "whole")
    bench.dump_outputs(whole, [("C", torch.from_numpy(C), None, A.rows), ("dB", torch.from_numpy(dB), None, A.cols)])
    for name in ("C", "dB"):
        got, want = np.load(os.path.join(out, name + ".npy")), np.load(os.path.join(whole, name + ".npy"))
        assert got.shape == want.shape and 0 < got.shape[0] < 1024
        np.testing.assert_allclose(got, want, rtol=1e-5, atol=1e-5)


# ------------------------------------------------------------------ N > 1: which sharded product the bench runs

def _pick_worker(rank, world, port, scheme, no_autotune, graph, q):
    import argparse
    import importlib

    import torch
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import bench
        import ofspmm_b200 as ofs
        from test_dist_cpu import OracleCompute
        dmod = importlib.import_module("of-spmm_b200.dist")
        n = 8
        # "dense": every rank touches every column block (nothing saved); "banded": almost nothing remote
        if graph == "dense":
            A = ofs.graphs.uniform_csr(96, 96, 0.5, seed=3)
        else:
            idx = torch.arange(96)
            A = ofs.formats.coo_to_csr(idx, idx, torch.ones(96), (96, 96))
        B = ofs.graphs.dense_operand(A.cols, n, 5)
        dY = ofs.graphs.upstream_grad(A.rows, n, 6)
        args = argparse.Namespace(scheme=scheme, no_autotune=no_autotune, tasks_per_warp=0, ag_dynamic_order=False, buckets=1,
                                  pull_ctas=64, layout="auto", no_interleave=False, combine_ctas=0, tune_combine=True)
        runner, used, saving, tuned = bench.pick_runner(args, dmod, A, B, dY, n, torch.float32, rank, world, "cpu",
                                                        compute=OracleCompute(), steps=2)
        C, dB = runner.step(runner.shard_rows(B), runner.shard_rows_out(dY))
        q.put((rank, used, saving, tuned, type(runner).__name__, runner.r0, runner.r1, C.clone().numpy()))
        dist.barrier()
        dist.destroy_process_group()
    except Exception:
        import traceback
        q.put(("error", rank, traceback.format_exc()))


def _pick(world, scheme, no_autotune, graph):
    import socket

    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_pick_worker, args=(r, world, port, scheme, no_autotune, graph, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = [q.get(timeout=240) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
    for r in res:
        assert r[0] != "error", r[2]
    return sorted(res)


def test_pick_runner_dense_exchange_is_autotuned_and_sparse_is_not():
    import numpy as np
    sys.path.insert(0, ROOT)
    import ofspmm_b200 as ofs
    from oracle import oracle as O
    # dense exchange, fp32: both schemes are timed, they agree, every rank takes the same one
    res = _pick(2, "auto", False, "dense")
    used = {r[1] for r in res}
    assert len(used) == 1 and used <= {"pull", "allgather"}
    for r in res:
        assert r[2] < 0.25 and r[3]["schemes_agree"] is True
        assert set(r[3]) >= {"pull", "pull_fwd_only", "allgather[static order, 2 tasks/warp]",
                             "allgather[dynamic order, 2 tasks/warp]", "allgather[dynamic order, 4 tasks/warp]"}
        assert (r[1] == "allgather") == ("allgather_policy" in r[3]) and "chosen" in r[3]
        assert "pull[combine beside the last forward pass]" in r[3]
        assert not any(k.endswith("error") for k in r[3])
        assert r[4] == ("AllGatherSpmm" if r[1] == "allgather" else "ShardedSpmm")
    A = ofs.graphs.uniform_csr(96, 96, 0.5, seed=3)
    B = ofs.graphs.dense_operand(A.cols, 8, 5)
    ref = O.spmm_f64(A.crow.numpy(), A.col.numpy(), A.val.numpy(), B.numpy(), A.cols)
    got = np.concatenate([r[7] for r in res], axis=0)
    np.testing.assert_allclose(got, ref, rtol=1e-4, atol=1e-4)
    # the rule alone (no timing): dense -> all-gather
    assert {r[1] for r in _pick(2, "auto", True, "dense")} == {"allgather"}
    # sparse exchange (a diagonal: no remote row at all): needed-rows exchange, nothing timed
    for r in _pick(2, "auto", False, "banded"):
        assert r[1] == "pull" and r[2] > 0.9 and r[3] is None
    # an explicit request is honoured
    assert {r[1] for r in _pick(2, "pull", False, "dense")} == {"pull"}
