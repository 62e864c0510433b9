"""CPU tests of pattern matrices (OFSPMM_VAL_UNIT: every stored entry is 1, no values array) and
of the mean reduction (OFSPMM_FWD_MEAN): argument validation of the C ABI, the workspace queries,
the `reduce=` argument, and the autograd wiring of the mean backward and of SAGEConv with a dense
CPU stand-in for the kernels, against dense float64 torch."""
import ctypes
from importlib import import_module

import pytest
import torch

import ofspmm_b200 as ofs

_lib = import_module("of-spmm_b200._lib")
ops = import_module("of-spmm_b200.ops")
F = import_module("of-spmm_b200.functional")
gcn = import_module("of-spmm_b200.gcn")

F32, BF16, I32, I64, UNIT = _lib.DTYPE_FLOAT, _lib.DTYPE_BFLOAT16, _lib.DTYPE_INT32, _lib.DTYPE_INT64, _lib.VAL_UNIT
OK, INVALID, UNSUPPORTED, WORKSPACE = 0, 1, 2, 3
M, K, NNZ, N = 5000, 4000, 100000, 64
FAKE = 1 << 20              # never dereferenced: every call below stops before touching memory


def _al(x):
    return (x + 255) // 256 * 256


def _csr(val=None, val_dtype=UNIT, idx=I32, nnz=NNZ):
    return _lib.CsrStruct(M, K, nnz, FAKE, FAKE, val, idx, val_dtype)


def _fwd_ex(A, flags=0, dd=F32, ws=None, wsb=0):
    o = _lib.OptsStruct()
    o.flags = flags
    o.bias = FAKE
    o.acc32 = FAKE
    return _lib.lib().ofspmm_fwd_ex(ctypes.byref(A), FAKE, N, FAKE, N, N, dd, ctypes.byref(o), ws, wsb, None)


def _entry_points(A, dd=F32):
    """Status of every entry point that takes a CSR, on fake operands and no workspace."""
    L = _lib.lib()
    return {
        "fwd": L.ofspmm_fwd(ctypes.byref(A), FAKE, FAKE, N, dd, None, 0, None),
        "fwd_strided": L.ofspmm_fwd_strided(ctypes.byref(A), FAKE, N, FAKE, N, N, dd, None, 0, None),
        "fwd_ex": _fwd_ex(A, 0, dd),
        "bwd_b_atomic": L.ofspmm_bwd_b(ctypes.byref(A), None, FAKE, FAKE, N, dd, None, 0, None),
        "bwd_b_transposed": L.ofspmm_bwd_b(ctypes.byref(A), ctypes.byref(_lib.CsrStruct(K, M, A.nnz, FAKE, FAKE, A.val,
                                                                                          A.idx_dtype, A.val_dtype)),
                                           FAKE, FAKE, N, dd, None, 0, None),
        "bwd_b_transient": L.ofspmm_bwd_b_transient(ctypes.byref(A), FAKE, FAKE, N, dd, None, 0, None),
        "bwd_b_cached": L.ofspmm_bwd_b_cached(ctypes.byref(A), FAKE, FAKE, FAKE, FAKE, FAKE, N, dd, None, None, 0, None),
        "csr_transpose": L.ofspmm_csr_transpose(ctypes.byref(A), FAKE, FAKE, None, FAKE, None, 0, None),
        "fwd_host": L.ofspmm_fwd_host(ctypes.byref(A), FAKE, FAKE, N, dd, None, 0, None),
    }


@pytest.mark.parametrize("dd", [F32, BF16])
@pytest.mark.parametrize("idx", [I32, I64])
def test_unit_is_accepted_by_every_product(dd, idx):
    """A pattern matrix with val NULL passes validation everywhere (with either dense dtype): a
    missing workspace is the only complaint."""
    r = _entry_points(_csr(idx=idx), dd)
    assert all(v == WORKSPACE for v in r.values()), r


def test_unit_with_a_values_array_is_rejected():
    r = _entry_points(_csr(val=FAKE))
    assert all(v == INVALID for v in r.values()), r


def test_weighted_matrix_still_needs_its_values():
    r = _entry_points(_csr(val=None, val_dtype=F32))
    assert r["fwd"] == r["bwd_b_transient"] == r["bwd_b_cached"] == r["fwd_host"] == INVALID
    assert r["csr_transpose"] == WORKSPACE       # the transpose never needed values


def test_transpose_of_a_pattern_matrix_takes_no_t_val():
    L = _lib.lib()
    A = _csr()
    assert L.ofspmm_csr_transpose(ctypes.byref(A), FAKE, FAKE, FAKE, FAKE, None, 0, None) == INVALID


@pytest.mark.parametrize("val,vd", [(None, UNIT), (FAKE, UNIT), (FAKE, F32)])
def test_sddmm_rejects_the_unit_dtype(val, vd):
    """For the SDDMM val_dtype is the dtype of dval: a pattern matrix has no values to differentiate."""
    L = _lib.lib()
    A = _csr(val=val, val_dtype=vd)
    o = _lib.OptsStruct()
    want = UNSUPPORTED if vd == UNIT else WORKSPACE
    assert L.ofspmm_sddmm(ctypes.byref(A), FAKE, FAKE, FAKE, N, F32, None, 0, None) == want
    assert L.ofspmm_sddmm_ex(ctypes.byref(A), FAKE, FAKE, FAKE, N, F32, ctypes.byref(o), None, 0, None) == want


@pytest.mark.parametrize("other", [_lib.FWD_ACCUMULATE, _lib.FWD_ACC32_IN, _lib.FWD_ACC32_OUT,
                                   _lib.FWD_ACC32_IN | _lib.FWD_ACC32_OUT])
@pytest.mark.parametrize("A", [_csr(), _csr(val=FAKE, val_dtype=F32)], ids=["pattern", "weighted"])
def test_mean_does_not_combine_with_accumulation(other, A):
    assert _fwd_ex(A, _lib.FWD_MEAN | other, BF16) == INVALID


@pytest.mark.parametrize("flags", [_lib.FWD_MEAN, _lib.FWD_MEAN | _lib.FWD_BIAS | _lib.FWD_RELU])
def test_mean_alone_and_with_the_epilogue_passes_validation(flags):
    for A in (_csr(), _csr(val=FAKE, val_dtype=F32)):
        assert _fwd_ex(A, flags) == WORKSPACE


def _fwd_ws(rows, nnz, n):
    items = 64 if -(-(rows + nnz) // 256) < 148 * 36 else 256
    P = -(-(rows + nnz) // items)
    return 256 + _al((P + 1) * 8) + _al(P * n * 4)


@pytest.mark.parametrize("nnz", [0, 1, 1000, 10 ** 6, 10 ** 8])
def test_unit_workspaces_hold_no_value_arrays(nnz):
    L = _lib.lib()
    for idx in (I32, I64):
        t_f = L.ofspmm_bwd_b_transient_workspace_bytes(M, K, nnz, N, F32, idx, F32)
        t_u = L.ofspmm_bwd_b_transient_workspace_bytes(M, K, nnz, N, F32, idx, UNIT)
        assert t_f - t_u == _al(max(nnz, 1) * 4)
        h_f = L.ofspmm_fwd_host_workspace_bytes(M, K, nnz, N, F32, idx, F32)
        h_u = L.ofspmm_fwd_host_workspace_bytes(M, K, nnz, N, F32, idx, UNIT)
        assert h_f - h_u == _al(nnz * 4)
    c_f = L.ofspmm_bwd_b_cached_workspace_bytes(M, K, nnz, N, F32, F32)
    c_b = L.ofspmm_bwd_b_cached_workspace_bytes(M, K, nnz, N, BF16, BF16)
    c_u = L.ofspmm_bwd_b_cached_workspace_bytes(M, K, nnz, N, F32, UNIT)
    assert c_f - c_u == _al(max(nnz, 1) * 4)
    assert c_u == _fwd_ws(K, nnz, N)
    assert c_b > L.ofspmm_bwd_b_cached_workspace_bytes(M, K, nnz, N, BF16, UNIT)


def test_queries_without_a_value_dtype_are_unchanged():
    L = _lib.lib()
    for nnz in (0, 1000, 10 ** 6):
        assert L.ofspmm_fwd_workspace_bytes(M, K, nnz, N, F32) == _fwd_ws(M, nnz, N)
        assert L.ofspmm_bwd_b_workspace_bytes(M, K, nnz, N, F32, 1) == _fwd_ws(K, nnz, N)
        assert L.ofspmm_sddmm_workspace_bytes(M, K, nnz, N, F32) == 256 + _al((-(-(M + nnz) // 256) + 1) * 8)


# ------------------------------------------------------------------ Python argument checks


def _graph(cols=50):
    A = ofs.graphs.uniform_csr(60, cols, 0.1, seed=3)
    crow = A.crow.clone()
    lens = A.row_lengths().clone()
    lens[[4, 17]] = 0                        # empty rows
    crow = torch.cat([torch.zeros(1, dtype=crow.dtype), torch.cumsum(lens, 0).to(crow.dtype)])
    keep = torch.cat([A.col[int(A.crow[i]):int(A.crow[i]) + int(lens[i])] for i in range(A.rows)])
    return ofs.graphs.CsrMatrix(crow, keep, torch.linspace(-1, 1, keep.numel()), 60, cols)


@pytest.mark.parametrize("bad", ["max", "Mean", "", None])
def test_reduce_argument_errors(bad):
    A = _graph()
    b = torch.randn(A.cols, 8)
    with pytest.raises(ops.OpInferError, match="reduce"):
        ops.spmm_csr_compute(A.crow, A.col, None, b, A.rows, A.cols, reduce=bad)
    with pytest.raises(ops.OpInferError, match="reduce"):
        F.spmm_csr(A.crow, A.col, None, b, A.rows, A.cols, reduce=bad)
    with pytest.raises(ops.OpInferError, match="reduce"):
        F.spmm_csr_bias_act(A.crow, A.col, None, b, A.rows, A.cols, kernels=_DenseKernels(A), reduce=bad)


def test_reduce_is_keyword_only():
    A = _graph()
    with pytest.raises(TypeError):
        F.spmm_csr(A.crow, A.col, None, torch.randn(A.cols, 4), A.rows, A.cols, None, "mean")


def test_mean_with_accumulate_is_an_argument_error():
    A = _graph()
    b = torch.randn(A.cols, 8)
    with pytest.raises(ops.OpInferError, match="mean"):
        ops.spmm_csr_compute(A.crow, A.col, None, b, A.rows, A.cols, torch.empty(A.rows, 8), accumulate=True,
                             reduce="mean")


def test_inv_row_lengths():
    crow = torch.tensor([0, 2, 2, 5, 6], dtype=torch.int32)
    assert torch.equal(ops.inv_row_lengths(crow).squeeze(1), torch.tensor([0.5, 0.0, 1 / 3, 1.0]))


# ------------------------------------------------------------------ autograd wiring on the CPU


class _DenseKernels:
    """CPU stand-in for functional.OpsKernels: dense float64-capable torch arithmetic, pattern
    matrices (a_val None = ones) and the mean reduction."""

    def __init__(self, A):
        self.rows_of = torch.repeat_interleave(torch.arange(A.rows), A.row_lengths())
        self.lens = A.row_lengths().to(torch.float64)
        self.calls = []

    def _dense(self, a_col, a_val, m, k, dtype):
        v = torch.ones(a_col.numel(), dtype=dtype) if a_val is None else a_val
        return torch.zeros(m, k, dtype=v.dtype).index_put((self.rows_of, a_col.long()), v, accumulate=True)

    def fwd(self, a_crow, a_col, a_val, b, m, k, bias, relu, plan, reduce="sum"):
        self.calls.append(("fwd", a_val is None, reduce, bias is not None, relu))
        out = self._dense(a_col, a_val, m, k, b.dtype) @ b
        if reduce == "mean":
            out = out / self.lens.clamp(min=1).to(out.dtype)[:, None]
        if bias is not None:
            out = out + bias
        return torch.relu(out) if relu else out

    def grad_b(self, a_crow, a_col, a_val, dy, m, k, plan):
        self.calls.append(("grad_b", a_val is None))
        return self._dense(a_col, a_val, m, k, dy.dtype).t() @ dy

    def sddmm(self, a_crow, a_col, dy, b, m, k, val_dtype, plan):
        self.calls.append(("sddmm",))
        return (dy[self.rows_of] * b[a_col.long()]).sum(1).to(val_dtype)


def _dense64(A, val):
    rows = torch.repeat_interleave(torch.arange(A.rows), A.row_lengths())
    v = torch.ones(A.nnz, dtype=torch.float64) if val is None else val
    return torch.zeros(A.rows, A.cols, dtype=torch.float64).index_put((rows, A.col.long()), v, accumulate=True)


@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("relu", [False, True])
def test_mean_backward_wiring(weighted, relu):
    A = _graph()
    K_ = _DenseKernels(A)
    b = torch.randn(A.cols, 6, dtype=torch.float64, generator=torch.Generator().manual_seed(1)).requires_grad_(True)
    bias = torch.linspace(-0.5, 0.5, 6, dtype=torch.float64).requires_grad_(True)
    val = A.val.double().requires_grad_(True) if weighted else None
    out = F.spmm_csr_bias_act(A.crow, A.col, val, b, A.rows, A.cols, bias, relu, kernels=K_, reduce="mean")
    w = torch.linspace(-1, 1, out.numel(), dtype=torch.float64).view_as(out)
    (out * w).sum().backward()
    assert K_.calls[0] == ("fwd", not weighted, "mean", True, relu)
    assert ("sddmm",) in K_.calls if weighted else ("sddmm",) not in K_.calls

    b64 = b.detach().clone().requires_grad_(True)
    bias64 = bias.detach().clone().requires_grad_(True)
    v64 = A.val.double().requires_grad_(True) if weighted else None
    lens = A.row_lengths().double().clamp(min=1)[:, None]
    ref = (_dense64(A, v64) @ b64) / lens + bias64
    ref = torch.relu(ref) if relu else ref
    (ref * w).sum().backward()
    # the backward's 1/len row scale is float32 (what the GPU path multiplies with)
    close = lambda a, r: torch.allclose(a, r, rtol=1e-6, atol=1e-6)  # noqa: E731
    assert torch.allclose(out, ref, rtol=1e-12, atol=1e-12)
    assert close(b.grad, b64.grad) and close(bias.grad, bias64.grad)
    if weighted:
        assert close(val.grad, v64.grad)
    empty = A.row_lengths() == 0
    assert torch.equal(out[empty], (torch.relu(bias) if relu else bias).detach().expand(int(empty.sum()), 6))


@pytest.mark.parametrize("in_dim,out_dim,act,bias", [(24, 16, "relu", True), (24, 16, None, True),
                                                      (12, 40, "relu", True), (12, 40, None, False)])
def test_sageconv_cpu_wiring(in_dim, out_dim, act, bias):
    A = _graph(cols=60)                                                 # square: X holds the root rows
    A = ofs.graphs.CsrMatrix(A.crow, A.col, None, A.rows, A.cols)      # no values anywhere
    K_ = _DenseKernels(A)
    conv = gcn.SAGEConv(in_dim, out_dim, bias=bias, activation=act, seed=3, device="cpu", dtype=torch.float64,
                        kernels=K_)
    assert conv.multiply_first == (out_dim <= in_dim)
    assert conv.aggregation_width() == min(in_dim, out_dim)
    with torch.no_grad():
        if conv.bias is not None:
            conv.bias.copy_(torch.linspace(-0.3, 0.3, out_dim))
    X = torch.randn(A.cols, in_dim, dtype=torch.float64, generator=torch.Generator().manual_seed(2)).requires_grad_(True)
    out = conv(A, X)
    fwd = [c for c in K_.calls if c[0] == "fwd"]
    assert fwd == [("fwd", True, "mean", conv.multiply_first and act is None and bias, False)]
    w = torch.linspace(-1, 1, out.numel(), dtype=torch.float64).view_as(out)
    (out * w).sum().backward()

    X64 = X.detach().clone().requires_grad_(True)
    Wn = conv.weight_neigh.detach().clone().requires_grad_(True)
    Wr = conv.weight_root.detach().clone().requires_grad_(True)
    b64 = conv.bias.detach().clone().requires_grad_(True) if bias else None
    mean = _dense64(A, None) / A.row_lengths().double().clamp(min=1)[:, None]
    ref = mean @ X64 @ Wn + X64[:A.rows] @ Wr
    if b64 is not None:
        ref = ref + b64
    if act == "relu":
        ref = torch.relu(ref)
    (ref * w).sum().backward()
    close = lambda a, b: torch.allclose(a, b, rtol=1e-6, atol=1e-6)  # noqa: E731  float32 1/len in the backward
    assert close(out, ref) and close(X.grad, X64.grad)
    assert close(conv.weight_neigh.grad, Wn.grad) and close(conv.weight_root.grad, Wr.grad)
    if bias:
        assert close(conv.bias.grad, b64.grad)
