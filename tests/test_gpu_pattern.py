"""GPU tests of pattern matrices (a_val=None / OFSPMM_VAL_UNIT) and of the mean reduction.

The central oracle: a pattern product equals the same product with an explicit all-ones values
array, bit for bit.  The summation order depends only on (crow, n, dtype) and fma(1, x, acc) rounds
exactly like x + acc, so every kernel variant, index dtype, dense width and launch option must give
identical bits.  Masked slots and out-of-range columns must contribute 0, not 1."""
import gc
from importlib import import_module

import numpy as np
import pytest
import torch

import ofspmm_b200 as ofs
from oracle import oracle as O

pytestmark = pytest.mark.gpu

_lib = import_module("of-spmm_b200._lib")
ops = import_module("of-spmm_b200.ops")
F = import_module("of-spmm_b200.functional")
gcn = import_module("of-spmm_b200.gcn")
G = ofs.graphs
DEV = "cuda:0"
EX = _lib.VARIANT_EXPLICIT
VARIANTS = {"auto": None, "items64": EX | _lib.VARIANT_ITEMS64, "rowpar": EX | _lib.VARIANT_ROWPAR,
            "rows": EX | _lib.VARIANT_ROWS}


def _bits(t):
    return t.view(torch.int32 if t.dtype == torch.float32 else torch.int16)


def _same_bits(a, b):
    return torch.equal(_bits(a.contiguous()), _bits(b.contiguous()))


def _graph(idx=torch.int32, bad=True, M=3000, K=2000, seed=11):
    """Rows of 0..24 entries (about 10 % empty), two hub rows of 4000 entries (each spans ~16
    256-item tasks: exercises the carries and the fix-up), and, with ``bad``, columns outside
    [0, K) on both sides."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, 25, M)
    lens[rng.random(M) < 0.1] = 0
    lens[[7, M // 2]] = 4000
    lens[M - 1] = 0
    crow = np.concatenate([[0], np.cumsum(lens)])
    col = rng.integers(0, K, int(crow[-1]))
    if bad:
        pos = rng.choice(col.size, col.size // 200, replace=False)
        col[pos] = np.where(rng.random(pos.size) < 0.5, -3, K + 7)
    return G.CsrMatrix(torch.from_numpy(crow).to(idx), torch.from_numpy(col).to(idx),
                       torch.from_numpy(rng.uniform(-1, 1, col.size).astype(np.float32)), M, K)


@pytest.fixture(scope="module")
def graphs():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return {idx: _graph(idx).to(DEV) for idx in (torch.int32, torch.int64)}


def _ones(A, dtype):
    return torch.ones(A.nnz, dtype=dtype, device=DEV)


@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("dt", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("idx", [torch.int32, torch.int64])
@pytest.mark.parametrize("n", [1, 4, 20, 64, 128, 256])
def test_pattern_forward_equals_explicit_ones(graphs, variant, dt, idx, n):
    A = graphs[idx]
    B = G.dense_operand(A.cols, n, 5, DEV, dt)
    v = VARIANTS[variant]
    vals = [_ones(A, torch.float32)] + ([_ones(A, torch.bfloat16)] if dt == torch.bfloat16 else [])
    for reduce in ("sum", "mean"):
        got = ops.spmm_csr_compute(A.crow, A.col, None, B, A.rows, A.cols, variant=v, reduce=reduce)
        for ones in vals:
            ref = ops.spmm_csr_compute(A.crow, A.col, ones, B, A.rows, A.cols, variant=v, reduce=reduce)
            assert _same_bits(got, ref), (reduce, ones.dtype)


@pytest.mark.parametrize("mode", ["plan", "static", "tasks_per_warp", "strided", "bias_relu", "mean_bias_relu"])
@pytest.mark.parametrize("dt", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("n", [20, 64, 128])
def test_pattern_forward_options_equal_explicit_ones(graphs, mode, dt, n):
    A = graphs[torch.int32]
    ones = _ones(A, torch.float32)
    B = G.dense_operand(A.cols, n, 6, DEV, dt)
    kw = {}
    if mode == "plan":
        kw["plan"] = ops.SpmmPlan(A.crow, A.col, A.rows, A.cols, n, dt)
    elif mode == "static":
        kw["order"] = "static"
    elif mode == "tasks_per_warp":
        kw["tasks_per_warp"] = 2
    elif mode in ("bias_relu", "mean_bias_relu"):
        kw["bias"] = torch.linspace(-0.5, 0.5, n, device=DEV).to(dt)
        kw["relu"] = True
        kw["reduce"] = "mean" if mode == "mean_bias_relu" else "sum"
    if mode == "strided":
        Bw = G.dense_operand(A.cols, n + 12, 6, DEV, dt)
        B = Bw[:, 4:4 + n]
        out1 = torch.full((A.rows, n + 8), 7.0, device=DEV, dtype=dt)
        out2 = out1.clone()
        ops.spmm_csr_compute(A.crow, A.col, None, B, A.rows, A.cols, out1[:, 8:])
        ops.spmm_csr_compute(A.crow, A.col, ones, B, A.rows, A.cols, out2[:, 8:])
        assert _same_bits(out1, out2)
        return
    got = ops.spmm_csr_compute(A.crow, A.col, None, B, A.rows, A.cols, **kw)
    ref = ops.spmm_csr_compute(A.crow, A.col, ones, B, A.rows, A.cols, **kw)
    assert _same_bits(got, ref)


@pytest.mark.parametrize("dt", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("idx", [torch.int32, torch.int64])
@pytest.mark.parametrize("n", [4, 64, 128])
def test_grad_b_routes_equal_explicit_ones(graphs, dt, idx, n):
    A = graphs[idx]
    ones = _ones(A, torch.float32)
    dY = G.upstream_grad(A.rows, n, 8, DEV, dt)
    plan = ops.SpmmPlan(A.crow, A.col, A.rows, A.cols, n, dt, transpose=True)
    for route in ("plan", "regather", "transient", "transposed"):
        kw = {}
        if route in ("plan", "regather"):
            kw = {"plan": plan, "regather": route == "regather"}
        if route == "transposed":
            tc, tcol, _ = ops.csr_transpose(A.crow, A.col, None, A.rows, A.cols)
            _, _, tv = ops.csr_transpose(A.crow, A.col, ones, A.rows, A.cols)
            got = ops.spmm_csr_grad_b_compute(A.crow, A.col, None, dY, A.rows, A.cols, transposed=(tc, tcol, None))
            ref = ops.spmm_csr_grad_b_compute(A.crow, A.col, ones, dY, A.rows, A.cols, transposed=(tc, tcol, tv))
        else:
            got = ops.spmm_csr_grad_b_compute(A.crow, A.col, None, dY, A.rows, A.cols, **kw)
            ref = ops.spmm_csr_grad_b_compute(A.crow, A.col, ones, dY, A.rows, A.cols, **kw)
        assert _same_bits(got, ref), route
    assert plan._t_val is not None           # the weighted call cached A^T's values ...
    plan._t_val = None
    ops.spmm_csr_grad_b_compute(A.crow, A.col, None, dY, A.rows, A.cols, plan=plan)
    assert plan._t_val is None                # ... the pattern call caches none
    # atomic scatter: order-nondeterministic, against the fp64 oracle
    got = ops.spmm_csr_grad_b_compute(A.crow, A.col, None, dY, A.rows, A.cols, atomic=True).float().cpu().numpy()
    crow, col = A.crow.cpu().numpy(), A.col.cpu().numpy()
    one = np.ones(col.size, np.float32)
    dYh = dY.float().cpu().numpy()
    ref = O.spmm_t_f64(crow, col, one, dYh, A.cols)
    amax, cnt = O.spmm_t_absmax(crow, col, one, dYh, A.cols)
    tol = O.fp32_tolerance(ref, amax, cnt) + (2.0 ** -8 * np.abs(ref) if dt == torch.bfloat16 else 0) + 1e-30
    assert (np.abs(got - ref) <= tol).all()


def _mean_ref(A, B, bias=None, relu=False):
    crow, col = A.crow.cpu().numpy(), A.col.cpu().numpy()
    one = np.ones(col.size, np.float32)
    Bh = B.float().cpu().numpy()
    s = O.spmm_f64(crow, col, one, Bh, A.cols)
    amax = O.spmm_absmax(crow, col, one, Bh, A.cols)
    lens = np.diff(crow)
    d = np.maximum(lens, 1).astype(np.float64)[:, None]
    # fp32 summation bound on the sum, scaled by the division, plus the division's own rounding
    tol = O.fp32_tolerance(s, amax, lens) / d + 2.0 ** -22 * np.abs(s / d)
    out = s / d
    if bias is not None:
        out = out + bias.double().cpu().numpy()
    if relu:
        out = np.maximum(out, 0)
    return out, tol, lens


@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("dt", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("n", [4, 64, 256])
def test_mean_forward_against_oracle(graphs, weighted, dt, variant, n):
    A = graphs[torch.int32]
    B = G.dense_operand(A.cols, n, 12, DEV, dt)
    bias = torch.linspace(-0.25, 0.25, n, device=DEV).to(dt)
    val = (A.val.to(torch.bfloat16) if dt == torch.bfloat16 else A.val) if weighted else None
    v = VARIANTS[variant]
    got = ops.spmm_csr_compute(A.crow, A.col, val, B, A.rows, A.cols, variant=v, reduce="mean", bias=bias, relu=True)
    again = ops.spmm_csr_compute(A.crow, A.col, val, B, A.rows, A.cols, variant=v, reduce="mean", bias=bias, relu=True)
    assert _same_bits(got, again)
    crow, col = A.crow.cpu().numpy(), A.col.cpu().numpy()
    vh = val.float().cpu().numpy() if weighted else np.ones(col.size, np.float32)
    Bh = B.float().cpu().numpy()
    s = O.spmm_f64(crow, col, vh, Bh, A.cols)
    amax = O.spmm_absmax(crow, col, vh, Bh, A.cols)
    lens = np.diff(crow)
    d = np.maximum(lens, 1).astype(np.float64)[:, None]
    ref = np.maximum(s / d + bias.double().cpu().numpy(), 0)
    tol = O.fp32_tolerance(s, amax, lens) / d + 2.0 ** -22 * np.abs(s / d) + 2.0 ** -23 * np.abs(ref)
    if dt == torch.bfloat16:
        tol = tol + 2.0 ** -8 * np.abs(ref)
    err = np.abs(got.double().cpu().numpy() - ref)
    assert (err <= tol + 1e-30).all(), float((err - tol).max())
    empty = torch.from_numpy(lens == 0).to(DEV)
    assert _same_bits(got[empty], torch.relu(bias).expand(int(empty.sum()), n))


@pytest.mark.parametrize("weighted", [False, True])
def test_mean_matches_torch_sparse_mean(weighted):
    A = _graph(bad=False)
    B = G.dense_operand(A.cols, 64, 13)
    val = A.val if weighted else torch.ones(A.nnz)
    S = torch.sparse_csr_tensor(A.crow.long(), A.col.long(), val, size=(A.rows, A.cols))
    ref = torch.sparse.mm(S, B, reduce="mean")
    Ad = A.to(DEV)
    got = ops.spmm_csr_compute(Ad.crow, Ad.col, Ad.val if weighted else None, B.to(DEV), A.rows, A.cols, reduce="mean")
    assert torch.allclose(got.cpu(), ref, rtol=1e-5, atol=1e-5)
    assert torch.equal(got.cpu()[A.row_lengths() == 0], torch.zeros(int((A.row_lengths() == 0).sum()), 64))


def test_mean_alone_on_an_empty_matrix_gives_zeros():
    crow = torch.zeros(11, dtype=torch.int32, device=DEV)
    col = torch.zeros(0, dtype=torch.int32, device=DEV)
    B = torch.randn(6, 8, device=DEV)
    out = torch.full((10, 8), 5.0, device=DEV)
    ops.spmm_csr_compute(crow, col, None, B, 10, 6, out, reduce="mean")
    assert torch.equal(out, torch.zeros(10, 8, device=DEV))
    bias = torch.linspace(-1, 1, 8, device=DEV)
    out = ops.spmm_csr_compute(crow, col, None, B, 10, 6, reduce="mean", bias=bias, relu=True)
    assert torch.equal(out, torch.relu(bias).expand(10, 8))


@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("reduce", ["sum", "mean"])
@pytest.mark.parametrize("with_state", [False, True])
def test_spmm_csr_autograd_against_dense(weighted, reduce, with_state):
    A = G.uniform_csr(400, 300, 0.03, seed=4)
    lens = A.row_lengths()
    rows = torch.repeat_interleave(torch.arange(A.rows), lens)
    Ad = A.to(DEV)
    b = G.dense_operand(A.cols, 32, 3, DEV).requires_grad_(True)
    val = Ad.val.clone().requires_grad_(True) if weighted else None
    state = F.SpmmOpKernelState() if with_state else None
    out = ofs.spmm_csr(Ad.crow, Ad.col, val, b, A.rows, A.cols, state, reduce=reduce)
    w = torch.linspace(-1, 1, out.numel(), device=DEV).view_as(out)
    (out * w).sum().backward()
    v64 = (A.val.double() if weighted else torch.ones(A.nnz, dtype=torch.float64)).requires_grad_(weighted)
    dense = torch.zeros(A.rows, A.cols, dtype=torch.float64).index_put((rows, A.col.long()), v64)
    b64 = b.detach().double().cpu().requires_grad_(True)
    ref = dense @ b64
    if reduce == "mean":
        ref = ref / lens.double().clamp(min=1)[:, None]
    (ref * w.double().cpu()).sum().backward()
    close = lambda x, y: torch.allclose(x.double().cpu(), y, rtol=2e-4, atol=2e-6)  # noqa: E731
    assert close(out.detach(), ref.detach()) and close(b.grad, b64.grad)
    if weighted:
        assert close(val.grad, v64.grad)


@pytest.mark.parametrize("in_dim,out_dim,act", [(48, 16, "relu"), (48, 16, None), (16, 40, "relu")])
def test_sageconv_against_dense(in_dim, out_dim, act):
    A = G.uniform_csr(500, 500, 0.02, seed=6)
    lens = A.row_lengths()
    rows = torch.repeat_interleave(torch.arange(A.rows), lens)
    Ad = G.CsrMatrix(A.crow.to(DEV), A.col.to(DEV), None, A.rows, A.cols)
    conv = gcn.SAGEConv(in_dim, out_dim, activation=act, seed=2, device=DEV)
    with torch.no_grad():
        conv.bias.copy_(torch.linspace(-0.2, 0.2, out_dim))
    X = G.dense_operand(A.rows, in_dim, 4, DEV).requires_grad_(True)
    out = conv(Ad, X, state=F.SpmmOpKernelState())
    w = torch.linspace(-1, 1, out.numel(), device=DEV).view_as(out)
    (out * w).sum().backward()
    dense = torch.zeros(A.rows, A.cols, dtype=torch.float64).index_put((rows, A.col.long()),
                                                                      torch.ones(A.nnz, dtype=torch.float64))
    mean = dense / lens.double().clamp(min=1)[:, None]
    X64 = X.detach().double().cpu().requires_grad_(True)
    Wn = conv.weight_neigh.detach().double().cpu().requires_grad_(True)
    Wr = conv.weight_root.detach().double().cpu().requires_grad_(True)
    b64 = conv.bias.detach().double().cpu().requires_grad_(True)
    ref = mean @ X64 @ Wn + X64 @ Wr + b64
    if act == "relu":
        ref = torch.relu(ref)
    (ref * w.double().cpu()).sum().backward()
    close = lambda x, y: torch.allclose(x.double().cpu(), y, rtol=2e-4, atol=2e-5)  # noqa: E731
    assert close(out.detach(), ref.detach()) and close(X.grad, X64.grad)
    assert close(conv.weight_neigh.grad, Wn.grad) and close(conv.weight_root.grad, Wr.grad)
    assert close(conv.bias.grad, b64.grad)


def test_wide_pattern_forward_without_values():
    """2^31 + 2^25 int64 non-zeros, no values array: the case pattern matrices exist for."""
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info(0)
    if free < 60e9:
        pytest.skip(f"needs 60 GB of free device memory, {free / 1e9:.0f} GB free")
    A = G.wide_csr(DEV)
    A.val = None                              # the pattern matrix has no values
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    n = 32
    B = G.dense_operand(A.cols, n, 31, DEV)
    base = torch.cuda.memory_allocated(0)
    torch.cuda.reset_peak_memory_stats()
    C = ops.spmm_csr_compute(A.crow, A.col, None, B, A.rows, A.cols, reduce="mean")
    torch.cuda.synchronize()
    extra = torch.cuda.max_memory_allocated(0) - base
    assert extra < A.nnz * 4, f"the call allocated {extra / 1e9:.1f} GB, as much as a values array"
    crow_h = A.crow.cpu().numpy()
    rng = np.random.default_rng(5)
    rows_sel = np.unique(np.concatenate([[G.WIDE_HUB, 0, A.rows - 1], rng.choice(A.rows, 200, replace=False)]))
    lens = crow_h[rows_sel + 1] - crow_h[rows_sel]
    crow_s = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    col_s = np.concatenate([A.col[int(crow_h[i]):int(crow_h[i + 1])].cpu().numpy() for i in rows_sel]).astype(np.int64)
    one = np.ones(col_s.size, np.float32)
    Bh = B.cpu().numpy()
    s = O.spmm_f64(crow_s, col_s, one, Bh, A.cols)
    amax = O.spmm_absmax(crow_s, col_s, one, Bh, A.cols)
    d = np.maximum(lens, 1).astype(np.float64)[:, None]
    tol = O.fp32_tolerance(s, amax, lens) / d + 2.0 ** -22 * np.abs(s / d) + 1e-30
    got = C[torch.from_numpy(rows_sel).to(DEV)].double().cpu().numpy()
    assert (np.abs(got - s / d) <= tol).all()
    del A, B, C
    gc.collect()
    torch.cuda.empty_cache()
