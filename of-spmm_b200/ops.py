"""Host-side mirror of the OneFlow user-op pieces of SURVEY.md §8a (a2, a7): shape / dtype
inference with the reference's error behaviour, and the kernel-compute bodies that pull raw
pointers out of tensors and call the C ABI on the current stream.

Tensors are ``torch`` CUDA tensors — torch is only the memory / stream plumbing here; the maths is
all in libofspmm_b200.so.  Names follow the provisional op schema (`spmm_csr`,
`spmm_csr_grad_b`, `sddmm_csr`; inputs `a_crow, a_col, a_val, b`; attrs `a_rows, a_cols`).

Reference conventions mirrored:
  * InferLogicalTensorDesc / InferDataType with CHECK_*_OR_RETURN → Python exception
    (oneflow/user/ops/matmul_op.cpp:23-75, oneflow/user/ops/unsorted_segment_sum_op.cpp:66-78);
  * kernel selection by (device, dense dtype, index dtype); exactly one kernel may match
    (oneflow/core/framework/user_op_registry_manager.cpp:93-117) — here: CUDA only, no CPU kernel;
  * tmp_buffer sized by an InferTmpSizeFn (oneflow/user/kernels/unsorted_segment_sum_kernel.cpp:191-202)
    → the ``*_workspace_bytes`` queries, allocated from torch's stream-ordered caching allocator;
  * outputs are allocated uninitialised and fully overwritten by the kernel.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import CsrStruct, OptsStruct, check

_DENSE = {torch.float32: _lib.DTYPE_FLOAT, torch.bfloat16: _lib.DTYPE_BFLOAT16}
_INDEX = {torch.int32: _lib.DTYPE_INT32, torch.int64: _lib.DTYPE_INT64}


class OpInferError(RuntimeError):
    """What a failed CHECK_*_OR_RETURN in an op's Infer* function surfaces as in Python."""


def _chk(cond: bool, msg: str) -> None:
    if not cond:
        raise OpInferError(msg)


def _stream_ptr(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    if t is None or t.numel() == 0:
        return None if t is None else (t.data_ptr() or None)
    return t.data_ptr()


def _workspace(nbytes: int, device) -> Tuple[Optional[torch.Tensor], Optional[int]]:
    if nbytes == 0:
        return None, None
    w = torch.empty(nbytes, dtype=torch.uint8, device=device)
    return w, w.data_ptr()


def infer_spmm_csr(a_crow, a_col, a_val, b, a_rows: int, a_cols: int) -> Tuple[Tuple[int, int], torch.dtype]:
    """SpmmCsrOp::InferLogicalTensorDesc + InferDataType (SURVEY.md §8a2)."""
    _chk(a_crow.dim() == 1 and a_col.dim() == 1, "a_crow and a_col must be 1-D")
    _chk(b.dim() == 2, f"b must be 2-D (cols x n), got {b.dim()}-D")
    _chk(a_rows >= 0 and a_cols >= 0, "a_rows / a_cols must be non-negative")
    _chk(a_crow.numel() == a_rows + 1, f"a_crow must have a_rows+1 = {a_rows + 1} entries, got {a_crow.numel()}")
    _chk(b.shape[0] == a_cols, f"b has {b.shape[0]} rows but a_cols = {a_cols}")
    _chk(a_crow.dtype in _INDEX, f"a_crow must be an index dtype (int32/int64), got {a_crow.dtype}")
    _chk(a_col.dtype == a_crow.dtype, "a_col and a_crow must share one index dtype")
    _chk(b.dtype in _DENSE, f"b dtype {b.dtype} has no registered kernel (float32 / bfloat16)")
    if a_val is not None:
        _chk(a_val.dim() == 1 and a_val.numel() == a_col.numel(), "a_val and a_col must have nnz entries each")
        _chk(a_val.dtype in _DENSE, f"a_val dtype {a_val.dtype} unsupported")
        _chk(a_val.dtype == torch.float32 or b.dtype == torch.bfloat16,
             "bfloat16 a_val requires a bfloat16 dense operand")
    return (a_rows, int(b.shape[1])), b.dtype


def _check_device(*tensors) -> None:
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            # exactly one kernel is registered for this op and it is the CUDA one (no CPU kernel):
            raise OpInferError("spmm_csr: no kernel registered for device type cpu — tensors must be on a CUDA device")
        # 1-D tensors contiguous; dense 2-D operands row-major with unit inner stride (a column
        # slice of a wider matrix is fine: its row stride is passed on as the leading dimension)
        ok = t.is_contiguous() or (t.dim() == 2 and t.stride(1) == 1 and t.stride(0) >= t.shape[1])
        _chk(ok, "spmm_csr kernels take contiguous tensors (2-D operands: unit inner stride)")
        dev = dev or t.device
        _chk(t.device == dev, "all tensors must live on one device")


def _check_packed(*tensors) -> None:
    """Operands of the entry points that take no leading dimension (dy / b / out of
    `spmm_csr_grad_b` and `sddmm_csr`) must be packed row-major: a column-slice view would be read
    with the wrong row stride."""
    for t in tensors:
        if t is not None:
            _chk(t.is_contiguous(), "spmm_csr_grad_b / sddmm_csr take packed (contiguous) dense operands; "
                                    "call .contiguous() on column-slice views")


def _csr_struct(a_crow, a_col, a_val, rows: int, cols: int, val_dtype=None) -> CsrStruct:
    """``a_val`` None without a ``val_dtype`` is a pattern matrix (every stored entry 1.0)."""
    if a_val is not None:
        vd = _DENSE[a_val.dtype]
    else:
        vd = _DENSE[val_dtype] if val_dtype is not None else _lib.VAL_UNIT
    return CsrStruct(rows, cols, int(a_col.numel()), _ptr(a_crow), _ptr(a_col), _ptr(a_val),
                     _INDEX[a_crow.dtype], vd)


class SpmmPlan:
    """What the op keeps per CSR *structure* — the OpKernelState role
    (oneflow/user/kernels/stateful_opkernel.cpp:919-928), built once, outside any captured call:

      * the kernel variant chosen from the row-length histogram (``ofspmm_row_hist`` → host →
        ``ofspmm_choose_variant``) for this (structure, n, dtype);
      * the merge-path task partition of that variant (``ofspmm_plan_build``), so products skip
        the partition kernel;
      * optionally (``transpose=True``) the structure of A^T — ``t_crow, t_col, t_perm`` — with its
        own variant and partition, for the deterministic backward.  Values are never cached:
        ``spmm_csr_grad_b`` re-gathers them through ``t_perm`` on every call.

    The plan is read-only to the products and holds references to ``a_crow`` / ``a_col`` so their
    storage cannot be recycled under it."""

    def __init__(self, a_crow: torch.Tensor, a_col: torch.Tensor, a_rows: int, a_cols: int, n: int,
                 dtype: torch.dtype = torch.float32, transpose: bool = False, variant: Optional[int] = None):
        _check_device(a_crow, a_col)
        _chk(a_crow.dtype in _INDEX and a_col.dtype == a_crow.dtype, "a_crow / a_col must share an index dtype")
        _chk(a_crow.numel() == a_rows + 1, "a_crow must have a_rows+1 entries")
        _chk(dtype in _DENSE, f"dense dtype {dtype} unsupported")
        self.a_crow, self.a_col = a_crow, a_col
        self.rows, self.cols, self.n, self.dtype = a_rows, a_cols, int(n), dtype
        self.nnz = int(a_col.numel())
        self.key = (a_crow.data_ptr(), a_col.data_ptr(), a_crow._version, a_col._version, a_rows, a_cols, self.nnz)
        self.hist = None
        self.variant, self.part = self._build(a_crow, a_rows, self.nnz, variant)
        self.t_crow = self.t_col = self.t_perm = self.t_part = None
        self.t_variant = _lib.VARIANT_AUTO
        self._t_val, self._t_val_key = None, None
        self._inv_len = None
        if transpose:
            self.t_crow, self.t_col, _, self.t_perm = csr_transpose(a_crow, a_col, None, a_rows, a_cols, want_perm=True)
            self.t_variant, self.t_part = self._build(self.t_crow, a_cols, self.nnz, None)

    def _build(self, crow, rows, nnz, variant):
        L = _lib.lib()
        dd = _DENSE[self.dtype]
        with torch.cuda.device(crow.device):
            if variant is None:
                hist = row_hist(crow).cpu()                     # one D2H read, at plan time only
                if self.hist is None:
                    self.hist = hist
                arr = (ctypes.c_int64 * 32)(*hist.tolist())
                variant = L.ofspmm_choose_variant(arr, rows, nnz, self.n, dd)
            nbytes = L.ofspmm_plan_bytes(rows, nnz, self.n, dd, variant)
            part = torch.empty(nbytes, dtype=torch.uint8, device=crow.device)
            check(L.ofspmm_plan_build(_ptr(crow), _INDEX[crow.dtype], rows, nnz, self.n, dd, variant,
                                      part.data_ptr(), nbytes, _stream_ptr(crow)), "plan_build")
        return variant, part

    def matches(self, a_crow, a_col, a_rows, a_cols, n, dtype) -> bool:
        return (self.key == (a_crow.data_ptr(), a_col.data_ptr(), a_crow._version, a_col._version, a_rows, a_cols,
                             int(a_col.numel())) and self.n == int(n) and self.dtype == dtype)

    def transposed_values(self, a_val: torch.Tensor) -> torch.Tensor:
        """Values of A^T for ``a_val`` = a_val[t_perm].  Re-gathered whenever the tensor's identity or
        autograd version changed (in-place updates bump the version), reused otherwise — a proof of
        "unchanged" the C++ glue does not have, which therefore gathers on every call."""
        key = (a_val.data_ptr(), a_val._version, a_val.dtype)
        if self._t_val is None or self._t_val_key != key:
            out = torch.empty(self.nnz, dtype=a_val.dtype, device=a_val.device)
            with torch.cuda.device(a_val.device):
                check(_lib.lib().ofspmm_permute_values(_ptr(a_val), _DENSE[a_val.dtype], _ptr(self.t_perm),
                                                       _INDEX[self.t_perm.dtype], self.nnz, _ptr(out),
                                                       _stream_ptr(a_val)), "permute_values")
            self._t_val, self._t_val_key = out, key
        return self._t_val

    def inv_row_lengths(self) -> torch.Tensor:
        """(rows, 1) float32: 1 / (stored entries of each row), 0 for an empty row — the row scale of
        the mean aggregation's backward, computed once per structure."""
        if self._inv_len is None:
            self._inv_len = inv_row_lengths(self.a_crow)
        return self._inv_len

    def prepared(self, transposed: bool = False) -> "_Prepared":
        """Low-host-overhead launcher of A·B (or, ``transposed``, of A^T·dY on the cached structure)."""
        key = "_prep_t" if transposed else "_prep"
        p = getattr(self, key, None)
        if p is None:
            if transposed:
                p = _Prepared(self.t_crow, self.t_col, self.cols, self.rows, self.n, self.dtype, self.t_variant, self.t_part)
            else:
                p = _Prepared(self.a_crow, self.a_col, self.rows, self.cols, self.n, self.dtype, self.variant, self.part)
            setattr(self, key, p)
        return p

    def variant_name(self, transposed: bool = False) -> str:
        v = self.t_variant if transposed else self.variant
        r, c = (self.cols, self.rows) if transposed else (self.rows, self.cols)
        return _lib.lib().ofspmm_variant_name(v, r, self.nnz, self.n, _DENSE[self.dtype]).decode()


class _Prepared:
    """One forward-shaped product with everything that does not change between calls resolved once
    (CSR struct, variant, task partition, a persistent workspace, the opts struct): a call is a
    single ctypes call, ~10 us of host time instead of ~50 — which matters once 8 GPUs have cut the
    device time of a step to ~1 ms.  Built lazily by ``SpmmPlan.prepared``; never shared between
    streams that could run concurrently (it owns its workspace)."""

    def __init__(self, crow, col, rows: int, cols: int, n: int, dtype, variant: int, part: torch.Tensor):
        L = _lib.lib()
        self.L, self.n, self.rows, self.cols, self.dd = L, int(n), rows, cols, _DENSE[dtype]
        self.keep = (crow, col, part)
        self.A = CsrStruct(rows, cols, int(col.numel()), _ptr(crow), _ptr(col), None, _INDEX[crow.dtype], _lib.DTYPE_FLOAT)
        self.variant = variant
        with torch.cuda.device(crow.device):
            self.ws_bytes = L.ofspmm_fwd_ex_workspace_bytes(rows, cols, self.A.nnz, self.n, self.dd, variant)
            self.ws = torch.empty(max(self.ws_bytes, 16), dtype=torch.uint8, device=crow.device)
        self.opts = OptsStruct(0, 0, variant, 0, part.data_ptr(), part.numel(), None, None)
        self._byref_A, self._byref_o = ctypes.byref(self.A), ctypes.byref(self.opts)

    def __call__(self, val: torch.Tensor, b: torch.Tensor, out: torch.Tensor, flags: int = 0, bias=None, acc32=None,
                 reserve_ctas: int = 0, tasks_per_warp: int = 0) -> torch.Tensor:
        A, o = self.A, self.opts
        A.val = val.data_ptr() if val.numel() else None
        A.val_dtype = _DENSE[val.dtype]
        o.flags, o.tasks_per_warp, o.reserve_ctas_per_sm = flags, tasks_per_warp, reserve_ctas
        o.bias = bias.data_ptr() if bias is not None else None
        o.acc32 = acc32.data_ptr() if acc32 is not None else None
        ldb = b.stride(0) if b.shape[0] > 1 else self.n
        ldc = out.stride(0) if out.shape[0] > 1 else self.n
        check(self.L.ofspmm_fwd_ex(self._byref_A, b.data_ptr() if b.numel() else None, ldb, out.data_ptr(), ldc, self.n, self.dd,
                                   self._byref_o, self.ws.data_ptr(), self.ws_bytes,
                                   torch.cuda.current_stream(out.device).cuda_stream), "spmm_csr(prepared)")
        return out


def _opts(flags: int = 0, tasks_per_warp: int = 0, variant: int = 0, part: Optional[torch.Tensor] = None,
          bias: Optional[torch.Tensor] = None, acc32: Optional[torch.Tensor] = None, reserve_ctas: int = 0) -> OptsStruct:
    return OptsStruct(flags, tasks_per_warp, variant, reserve_ctas, part.data_ptr() if part is not None else None,
                      part.numel() if part is not None else 0, bias.data_ptr() if bias is not None else None,
                      acc32.data_ptr() if acc32 is not None else None)


def inv_row_lengths(a_crow: torch.Tensor) -> torch.Tensor:
    """(rows, 1) float32: 1 / (crow[i+1] - crow[i]), 0 for an empty row."""
    lens = (a_crow[1:] - a_crow[:-1]).to(torch.float32)
    return torch.where(lens > 0, 1.0 / lens.clamp(min=1), torch.zeros_like(lens)).unsqueeze(1)


def reduce_flag(reduce: str) -> int:
    """`reduce` argument -> OFSPMM_FWD_* bit ("sum": 0, "mean": OFSPMM_FWD_MEAN)."""
    _chk(reduce in ("sum", "mean"), f"reduce must be 'sum' or 'mean', got {reduce!r}")
    return _lib.FWD_MEAN if reduce == "mean" else 0


def _acc32_flags(acc32, acc32_in: bool, acc32_out: bool, rows: int, n: int, dt) -> int:
    if not (acc32_in or acc32_out):
        return 0
    _chk(dt != torch.float32, "acc32 passes are for 16-bit products (fp32 products accumulate in `out`)")
    _chk(acc32 is not None and acc32.dtype == torch.float32 and acc32.is_contiguous() and acc32.is_cuda
         and acc32.dim() == 2 and acc32.shape[0] >= rows and acc32.shape[1] == n,
         "acc32 must be a contiguous CUDA float32 tensor of shape (>= rows, n)")
    return (_lib.FWD_ACC32_IN if acc32_in else 0) | (_lib.FWD_ACC32_OUT if acc32_out else 0)


def spmm_csr_compute(a_crow, a_col, a_val, b, a_rows: int, a_cols: int,
                     out: Optional[torch.Tensor] = None, *, plan: Optional[SpmmPlan] = None,
                     accumulate: bool = False, bias: Optional[torch.Tensor] = None, relu: bool = False,
                     tasks_per_warp: int = 0, variant: Optional[int] = None, order: Optional[str] = None,
                     acc32: Optional[torch.Tensor] = None, acc32_in: bool = False, acc32_out: bool = False,
                     reserve_ctas: int = 0, reduce: str = "sum") -> torch.Tensor:
    """SpmmCsrKernel::Compute — out[a_rows, n] = A · b  (``accumulate``: out += A · b; ``bias`` /
    ``relu``: epilogue fused into the store, applied to the complete row sum).

    ``a_val`` None: pattern matrix, every stored entry is 1 and no values array is read.
    ``reduce="mean"``: each row sum is divided by the row's stored-entry count before bias / ReLU
    (an empty row gives 0; torch.sparse.mm(reduce="mean") semantics); not with ``accumulate`` or
    the ``acc32`` passes.

    ``plan`` supplies the histogram-chosen variant and the cached task partition; ``tasks_per_warp``
    > 0 launches short-lived CTAs (multi-GPU overlap); ``order`` in {None, "dynamic", "static"}.
    ``acc32`` (+ ``acc32_in`` / ``acc32_out``): fp32 running sums of a bf16 product that is computed
    in several passes — rounded to bf16 once, by the pass without ``acc32_out``."""
    mean = reduce_flag(reduce)
    _chk(not (mean and (accumulate or acc32_in or acc32_out)),
         "reduce='mean' divides the complete row sum: it cannot be combined with accumulate / acc32 passes")
    _check_device(a_crow, a_col, a_val, b, bias)
    (m, n), dt = infer_spmm_csr(a_crow, a_col, a_val, b, a_rows, a_cols)
    if out is None:
        _chk(not accumulate, "accumulate needs an `out` tensor to add to")
        out = torch.empty((m, n), dtype=dt, device=b.device)
    else:
        _chk(out.shape == (m, n) and out.dtype == dt and out.device == b.device,
             "out has the wrong shape / dtype / device")
        _check_device(out)
    if bias is not None:
        _chk(bias.dim() == 1 and bias.numel() == n and bias.dtype == dt and bias.is_contiguous(),
             "bias must be a contiguous vector of n elements of the dense dtype")
    if plan is not None:
        _chk(plan.matches(a_crow, a_col, a_rows, a_cols, n, dt), "plan was built for another CSR structure / n / dtype")
    L = _lib.lib()
    flags = mean | (_lib.FWD_ACCUMULATE if accumulate else 0) | (_lib.FWD_BIAS if bias is not None else 0) | \
            (_lib.FWD_RELU if relu else 0) | {None: 0, "dynamic": _lib.ORDER_DYNAMIC, "static": _lib.ORDER_STATIC}[order] | \
            _acc32_flags(acc32, acc32_in, acc32_out, m, n, dt)
    v = variant if variant is not None else (plan.variant if plan is not None else _lib.VARIANT_AUTO)
    part = plan.part if (plan is not None and v == plan.variant) else None
    with torch.cuda.device(b.device):
        A = _csr_struct(a_crow, a_col, a_val, a_rows, a_cols)
        nbytes = L.ofspmm_fwd_ex_workspace_bytes(a_rows, a_cols, A.nnz, n, _DENSE[dt], v)
        ws, wsp = _workspace(nbytes, b.device)
        ldb = b.stride(0) if b.shape[0] > 1 else max(n, 1)
        ldc = out.stride(0) if out.shape[0] > 1 else max(n, 1)
        o = _opts(flags, tasks_per_warp, v, part, bias, acc32 if (acc32_in or acc32_out) else None, reserve_ctas)
        rc = L.ofspmm_fwd_ex(ctypes.byref(A), _ptr(b), ldb, _ptr(out), ldc, n, _DENSE[dt], ctypes.byref(o), wsp, nbytes,
                             _stream_ptr(b))
        check(rc, "spmm_csr")
    return out


def spmm_csr_grad_b_compute(a_crow, a_col, a_val, dy, a_rows: int, a_cols: int,
                            transposed: Optional[Tuple[torch.Tensor, torch.Tensor, torch.Tensor]] = None,
                            out: Optional[torch.Tensor] = None, *, plan: Optional[SpmmPlan] = None,
                            atomic: bool = False, tasks_per_warp: int = 0, regather: bool = False,
                            acc32_out: Optional[torch.Tensor] = None, reserve_ctas: int = 0) -> torch.Tensor:
    """SpmmCsrGradBKernel::Compute — db[a_cols, n] = A^T · dy.  Routes, in order of preference:

      * ``plan`` with a transposed structure → forward kernel on the cached structure of A^T; the
        values are re-gathered through ``t_perm`` whenever ``a_val``'s (pointer, version) changed,
        or on every call with ``regather=True`` (= ``ofspmm_bwd_b_cached``, the glue's route);
      * ``transposed`` = (t_crow, t_col, t_val) from csr_transpose → forward kernel on that CSR;
      * default → ``ofspmm_bwd_b_transient`` (A^T built inside the workspace; deterministic and
        2-9x faster than the scatter on the BASELINE graphs);
      * ``atomic=True`` → the reference-style vector-atomic scatter (order-nondeterministic).

    ``a_val`` None: pattern matrix on every route; the plan route then caches no values of A^T."""
    _check_device(a_crow, a_col, a_val, dy)
    _chk(dy.dim() == 2 and dy.shape[0] == a_rows, f"dy must be (a_rows={a_rows}) x n")
    _check_packed(dy, out)
    infer_spmm_csr(a_crow, a_col, a_val, dy.new_empty((a_cols, dy.shape[1])), a_rows, a_cols)
    n, dt = int(dy.shape[1]), dy.dtype
    if out is None:
        out = torch.empty((a_cols, n), dtype=dt, device=dy.device)
    else:
        _chk(out.shape == (a_cols, n) and out.dtype == dt and out.device == dy.device, "out has the wrong shape / dtype / device")
    L = _lib.lib()
    _chk(acc32_out is None or (plan is not None and plan.t_crow is not None and not atomic and not regather),
         "acc32_out needs the plan route with cached transposed values")
    if plan is not None and plan.t_crow is not None and not atomic:
        _chk(plan.matches(a_crow, a_col, a_rows, a_cols, n, dt), "plan was built for another CSR structure / n / dtype")
        with torch.cuda.device(dy.device):
            if regather:   # the C ABI route the OneFlow glue uses: values gathered inside the call
                A = _csr_struct(a_crow, a_col, a_val, a_rows, a_cols)
                vs = {_lib.DTYPE_FLOAT: 4, _lib.DTYPE_BFLOAT16: 2, _lib.VAL_UNIT: 0}[A.val_dtype]
                nbytes = ((max(A.nnz, 1) * vs + 255) // 256) * 256 + \
                    L.ofspmm_fwd_ex_workspace_bytes(a_cols, a_rows, A.nnz, n, _DENSE[dt], plan.t_variant)
                nbytes = max(nbytes, L.ofspmm_bwd_b_cached_workspace_bytes(a_rows, a_cols, A.nnz, n, _DENSE[dt], A.val_dtype))
                ws, wsp = _workspace(nbytes, dy.device)
                o = _opts(0, tasks_per_warp, plan.t_variant, plan.t_part)
                check(L.ofspmm_bwd_b_cached(ctypes.byref(A), _ptr(plan.t_crow), _ptr(plan.t_col), _ptr(plan.t_perm),
                                            _ptr(dy), _ptr(out), n, _DENSE[dt], ctypes.byref(o), wsp, nbytes,
                                            _stream_ptr(dy)), "spmm_csr_grad_b(cached structure)")
            else:          # values of A^T kept while a_val's (pointer, version) is unchanged
                t_val = plan.transposed_values(a_val) if a_val is not None else None
                At = _csr_struct(plan.t_crow, plan.t_col, t_val, a_cols, a_rows)
                nbytes = L.ofspmm_fwd_ex_workspace_bytes(a_cols, a_rows, At.nnz, n, _DENSE[dt], plan.t_variant)
                ws, wsp = _workspace(nbytes, dy.device)
                # acc32_out: the fp32 sums go to that buffer instead of `out` (16-bit products whose
                # partial results are combined across ranks in fp32)
                fl = _acc32_flags(acc32_out, False, acc32_out is not None, a_cols, n, dt)
                o = _opts(fl, tasks_per_warp, plan.t_variant, plan.t_part, None, acc32_out, reserve_ctas)
                check(L.ofspmm_fwd_ex(ctypes.byref(At), _ptr(dy), n, _ptr(out), n, n, _DENSE[dt], ctypes.byref(o), wsp, nbytes,
                                      _stream_ptr(dy)), "spmm_csr_grad_b(cached structure + values)")
        return out
    if transposed is None and not atomic:
        return spmm_csr_grad_b_transient_compute(a_crow, a_col, a_val, dy, a_rows, a_cols, out=out)
    with torch.cuda.device(dy.device):
        A = _csr_struct(a_crow, a_col, a_val, a_rows, a_cols)
        At_ref = None
        if transposed is not None:
            t_crow, t_col, t_val = transposed
            _check_device(t_crow, t_col, t_val)
            _chk((t_val is None) == (a_val is None), "transposed values must be given exactly when a_val is")
            At = _csr_struct(t_crow, t_col, t_val, a_cols, a_rows)
            At_ref = ctypes.byref(At)
        nbytes = L.ofspmm_bwd_b_workspace_bytes(a_rows, a_cols, A.nnz, n, _DENSE[dt], 1 if transposed is not None else 0)
        ws, wsp = _workspace(nbytes, dy.device)
        check(L.ofspmm_bwd_b(ctypes.byref(A), At_ref, _ptr(dy), _ptr(out), n, _DENSE[dt], wsp, nbytes,
                             _stream_ptr(dy)), "spmm_csr_grad_b")
    return out


def sddmm_csr_compute(a_crow, a_col, dy, b, a_rows: int, a_cols: int,
                      val_dtype: torch.dtype = torch.float32,
                      out: Optional[torch.Tensor] = None, *, plan: Optional[SpmmPlan] = None) -> torch.Tensor:
    """SddmmCsrKernel::Compute — dval[p] = <dy[i,:], b[col[p],:]>."""
    _check_device(a_crow, a_col, dy, b)
    _check_packed(dy, b, out)
    infer_spmm_csr(a_crow, a_col, None, b, a_rows, a_cols)
    _chk(dy.dim() == 2 and dy.shape[0] == a_rows and dy.shape[1] == b.shape[1] and dy.dtype == b.dtype,
         "dy must be (a_rows x n) with b's dtype")
    _chk(val_dtype == torch.float32 or b.dtype == torch.bfloat16, "bfloat16 values require a bfloat16 dense operand")
    n, dt = int(b.shape[1]), b.dtype
    nnz = int(a_col.numel())
    if out is None:
        out = torch.empty((nnz,), dtype=val_dtype, device=b.device)
    L = _lib.lib()
    with torch.cuda.device(b.device):
        A = _csr_struct(a_crow, a_col, None, a_rows, a_cols, val_dtype)
        nbytes = L.ofspmm_sddmm_workspace_bytes(a_rows, a_cols, nnz, n, _DENSE[dt])
        ws, wsp = _workspace(nbytes, b.device)
        o = _opts(0, 0, 0, plan.part if plan is not None else None)
        check(L.ofspmm_sddmm_ex(ctypes.byref(A), _ptr(dy), _ptr(b), _ptr(out), n, _DENSE[dt], ctypes.byref(o), wsp, nbytes,
                                _stream_ptr(b)), "sddmm_csr")
    return out


def merge_path_partition(a_crow: torch.Tensor, nnz: int, parts: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Device merge-path partitioner: parts+1 (row, nz) split points as int64 tensors."""
    _check_device(a_crow)
    _chk(a_crow.dtype in _INDEX and a_crow.dim() == 1 and a_crow.numel() >= 1, "a_crow must be a 1-D index tensor")
    _chk(parts >= 1, "parts must be >= 1")
    rows = a_crow.numel() - 1
    out_row = torch.empty(parts + 1, dtype=torch.int64, device=a_crow.device)
    out_nz = torch.empty(parts + 1, dtype=torch.int64, device=a_crow.device)
    with torch.cuda.device(a_crow.device):
        check(_lib.lib().ofspmm_partition(_ptr(a_crow), _INDEX[a_crow.dtype], rows, nnz, parts,
                                          out_row.data_ptr(), out_nz.data_ptr(), _stream_ptr(a_crow)),
              "merge_path_partition")
    return out_row, out_nz


def merge_path_partition_host(a_crow: torch.Tensor, nnz: int, parts: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Host twin of the device partitioner (C ABI ofspmm_partition_host); CPU tensors."""
    _chk(not a_crow.is_cuda and a_crow.dtype in _INDEX and a_crow.is_contiguous(), "a_crow must be a contiguous CPU index tensor")
    rows = a_crow.numel() - 1
    out_row = torch.empty(parts + 1, dtype=torch.int64)
    out_nz = torch.empty(parts + 1, dtype=torch.int64)
    check(_lib.lib().ofspmm_partition_host(a_crow.data_ptr(), _INDEX[a_crow.dtype], rows, nnz, parts,
                                           out_row.data_ptr(), out_nz.data_ptr()), "merge_path_partition_host")
    return out_row, out_nz


def row_blocks(a_crow: torch.Tensor, nnz: int, parts: int) -> torch.Tensor:
    """Whole-row nnz-balanced row blocks for ``parts`` devices (SURVEY.md §8e): bounds[k] = the
    merge-path split row of diagonal k, bounds[0] = 0, bounds[parts] = rows."""
    rows, _ = (merge_path_partition if a_crow.is_cuda else merge_path_partition_host)(a_crow, nnz, parts)
    rows = rows.clone()
    rows[0] = 0
    rows[-1] = a_crow.numel() - 1
    return rows


def row_hist(a_crow: torch.Tensor) -> torch.Tensor:
    """32 log2 buckets of the row lengths (device)."""
    _check_device(a_crow)
    hist = torch.empty(32, dtype=torch.int64, device=a_crow.device)
    with torch.cuda.device(a_crow.device):
        check(_lib.lib().ofspmm_row_hist(_ptr(a_crow), _INDEX[a_crow.dtype], a_crow.numel() - 1,
                                         hist.data_ptr(), _stream_ptr(a_crow)), "row_hist")
    return hist


def csr_transpose(a_crow, a_col, a_val, a_rows: int, a_cols: int, want_perm: bool = False):
    """Device CSR → CSR of A^T (entries of a column in ascending row order).  Returns
    (t_crow, t_col, t_val[, t_perm])."""
    _check_device(a_crow, a_col, a_val)
    nnz = int(a_col.numel())
    dev = a_crow.device
    t_crow = torch.empty(a_cols + 1, dtype=a_crow.dtype, device=dev)
    t_col = torch.empty(nnz, dtype=a_crow.dtype, device=dev)
    t_val = torch.empty(nnz, dtype=a_val.dtype, device=dev) if a_val is not None else None
    t_perm = torch.empty(nnz, dtype=a_crow.dtype, device=dev) if want_perm else None
    L = _lib.lib()
    with torch.cuda.device(dev):
        A = _csr_struct(a_crow, a_col, a_val, a_rows, a_cols)
        nbytes = L.ofspmm_csr_transpose_workspace_bytes(a_rows, a_cols, nnz, _INDEX[a_crow.dtype])
        ws, wsp = _workspace(nbytes, dev)
        check(L.ofspmm_csr_transpose(ctypes.byref(A), _ptr(t_crow), _ptr(t_col), _ptr(t_val), _ptr(t_perm),
                                     wsp, nbytes, _stream_ptr(a_crow)), "csr_transpose")
    return (t_crow, t_col, t_val, t_perm) if want_perm else (t_crow, t_col, t_val)


def sample_neighbors(a_crow, a_col, a_val, a_rows: int, a_cols: int, dst: torch.Tensor, fanout: int,
                     rng_seed: int) -> Tuple[torch.Tensor, torch.Tensor, Optional[torch.Tensor], torch.Tensor]:
    """One fan-out-sampled bipartite block of the square CSR A (``ofspmm_sample_neighbors``): for
    each destination ``dst[i]``, at most ``fanout`` of its entries (all of them for -1), chosen by
    the keys of include/ofspmm.h — uniform without replacement, a pure function of
    (rng_seed, node, position).  Returns ``(blk_crow, blk_col, blk_val, src_nodes)``: an int32 CSR
    of len(dst) x len(src_nodes) whose columns index ``src_nodes`` (dst first, then the other
    sampled ids ascending); ``blk_val`` is None for a pattern matrix.  One device-to-host read (two
    with fanout -1); invalid destinations (out of range, repeated) raise."""
    _check_device(a_crow, a_col, a_val, dst)
    _chk(a_crow.dim() == 1 and a_col.dim() == 1 and dst.dim() == 1, "a_crow, a_col and dst must be 1-D")
    _chk(a_crow.dtype in _INDEX and a_col.dtype == a_crow.dtype, "a_crow / a_col must share an index dtype (int32/int64)")
    _chk(a_rows == a_cols, f"neighbour sampling needs a square matrix, got {a_rows} x {a_cols}")
    _chk(a_rows >= 0 and a_crow.numel() == a_rows + 1, f"a_crow must have a_rows+1 = {a_rows + 1} entries")
    _chk(fanout >= -1, f"fanout must be >= 0, or -1 for all neighbours, got {fanout}")
    if a_val is not None:
        _chk(a_val.dim() == 1 and a_val.numel() == a_col.numel() and a_val.dtype in _DENSE,
             "a_val must hold nnz float32 / bfloat16 values")
    _chk(not dst.is_floating_point() and not dst.is_complex(), f"dst must hold node ids, got {dst.dtype}")
    dev, idt = a_crow.device, a_crow.dtype
    dst = dst.to(idt).contiguous()
    num_dst, nnz = int(dst.numel()), int(a_col.numel())
    if fanout == -1:
        # the exact size: sum of the destinations' degrees (invalid ids count 0, read nothing)
        ok = (dst >= 0) & (dst < a_rows)
        d = torch.where(ok, dst, torch.zeros_like(dst)).long()
        deg = (a_crow[1:][d] - a_crow[:-1][d]) * ok if a_rows > 0 else torch.zeros_like(d)
        cap = int(deg.sum())
    else:
        cap = min(num_dst * fanout, nnz)   # at most one kept entry per non-zero of A
    blk_crow = torch.empty(num_dst + 1, dtype=torch.int32, device=dev)
    blk_col = torch.empty(cap, dtype=torch.int32, device=dev)
    blk_val = torch.empty(cap, dtype=a_val.dtype, device=dev) if a_val is not None else None
    src_nodes = torch.empty(num_dst + cap, dtype=idt, device=dev)
    counts = torch.empty(3, dtype=torch.int64, device=dev)
    L = _lib.lib()
    with torch.cuda.device(dev):
        A = _csr_struct(a_crow, a_col, a_val, a_rows, a_cols)
        nbytes = L.ofspmm_sample_neighbors_workspace_bytes(num_dst, cap, _INDEX[idt])
        ws, wsp = _workspace(nbytes, dev)
        check(L.ofspmm_sample_neighbors(ctypes.byref(A), _ptr(dst), num_dst, fanout, rng_seed & (2 ** 64 - 1), cap,
                                        _ptr(blk_crow), _ptr(blk_col), _ptr(blk_val), _ptr(src_nodes),
                                        counts.data_ptr(), wsp, nbytes, _stream_ptr(dst)), "sample_neighbors")
    nnz_blk, num_src, bad = counts.tolist()
    _chk(bad == 0, f"sample_neighbors: {bad} destination ids are out of range [0, {a_rows}) or repeated")
    return (blk_crow, blk_col[:nnz_blk], blk_val[:nnz_blk] if blk_val is not None else None, src_nodes[:num_src])


def spmm_csr_grad_b_transient_compute(a_crow, a_col, a_val, dy, a_rows: int, a_cols: int,
                                      out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """db = A^T · dy through route (3) of the C ABI (``ofspmm_bwd_b_transient``): A^T is built
    inside the workspace for this call only, then the forward kernel runs on it — deterministic,
    for callers that hold no op state (the default route of ``spmm_csr_grad_b_compute``)."""
    _check_device(a_crow, a_col, a_val, dy)
    _chk(dy.dim() == 2 and dy.shape[0] == a_rows and dy.is_contiguous(), f"dy must be contiguous (a_rows={a_rows}) x n")
    infer_spmm_csr(a_crow, a_col, a_val, dy.new_empty((a_cols, dy.shape[1])), a_rows, a_cols)
    n, dt = int(dy.shape[1]), dy.dtype
    if out is None:
        out = torch.empty((a_cols, n), dtype=dt, device=dy.device)
    L = _lib.lib()
    with torch.cuda.device(dy.device):
        A = _csr_struct(a_crow, a_col, a_val, a_rows, a_cols)
        nbytes = L.ofspmm_bwd_b_transient_workspace_bytes(a_rows, a_cols, A.nnz, n, _DENSE[dt], A.idx_dtype, A.val_dtype)
        ws, wsp = _workspace(nbytes, dy.device)
        check(L.ofspmm_bwd_b_transient(ctypes.byref(A), _ptr(dy), _ptr(out), n, _DENSE[dt], wsp, nbytes,
                                       _stream_ptr(dy)), "spmm_csr_grad_b(transient)")
    return out


def gather_rows(dst: torch.Tensor, src: torch.Tensor, index: Optional[torch.Tensor] = None, index_offset: int = 0,
                count: Optional[int] = None, max_ctas: int = 0) -> torch.Tensor:
    """dst[i, :] = src[index[i] - index_offset, :] (index None: rows 0..count-1).  ``src`` may be a
    peer-mapped tensor of another GPU (symmetric memory): the rows then travel over NVLink."""
    _check_device(dst, index)
    _chk(dst.dim() == 2 and src.dim() == 2 and dst.shape[1] == src.shape[1] and dst.dtype == src.dtype
         and dst.dtype in _DENSE and dst.stride(1) == 1 and src.stride(1) == 1, "gather_rows: 2-D operands of one dense dtype")
    count = int(index.numel() if index is not None else (dst.shape[0] if count is None else count))
    _chk(count <= dst.shape[0], "gather_rows: dst has fewer rows than indices")
    n = int(dst.shape[1])
    with torch.cuda.device(dst.device):
        check(_lib.lib().ofspmm_gather_rows(_ptr(dst), dst.stride(0) if dst.shape[0] > 1 else n, _ptr(src),
                                            src.stride(0) if src.shape[0] > 1 else n, _ptr(index),
                                            _INDEX[index.dtype] if index is not None else _lib.DTYPE_INT32, index_offset,
                                            count, n, _DENSE[dst.dtype], max_ctas, _stream_ptr(dst)), "gather_rows")
    return dst


def scatter_add_rows(dst: torch.Tensor, src: torch.Tensor, index: Optional[torch.Tensor] = None, index_offset: int = 0,
                     count: Optional[int] = None, max_ctas: int = 0) -> torch.Tensor:
    """dst[index[i] - index_offset, :] += src[i, :] for distinct indices (no atomics; deterministic)."""
    _check_device(dst, index)
    _chk(dst.dim() == 2 and src.dim() == 2 and dst.shape[1] == src.shape[1] and dst.dtype == src.dtype
         and dst.dtype in _DENSE and dst.stride(1) == 1 and src.stride(1) == 1, "scatter_add_rows: 2-D operands of one dense dtype")
    count = int(index.numel() if index is not None else (src.shape[0] if count is None else count))
    n = int(dst.shape[1])
    with torch.cuda.device(dst.device):
        check(_lib.lib().ofspmm_scatter_add_rows(_ptr(dst), dst.stride(0) if dst.shape[0] > 1 else n, _ptr(src),
                                                 src.stride(0) if src.shape[0] > 1 else n, _ptr(index),
                                                 _INDEX[index.dtype] if index is not None else _lib.DTYPE_INT32,
                                                 index_offset, count, n, _DENSE[dst.dtype], max_ctas, _stream_ptr(dst)),
              "scatter_add_rows")
    return dst


def scatter_add_rows_f32(dst: torch.Tensor, src: torch.Tensor, index: Optional[torch.Tensor] = None, index_offset: int = 0,
                         count: Optional[int] = None, max_ctas: int = 0) -> torch.Tensor:
    """fp32 dst[index[i] - index_offset, :] += float(src[i, :]) — src bf16 (or fp32) partial rows, e.g. a
    peer's; the sum over many contributors is rounded once at the end (``cast_from_f32``)."""
    _check_device(dst, index)
    _chk(dst.dtype == torch.float32 and dst.dim() == 2 and src.dim() == 2 and dst.shape[1] == src.shape[1]
         and src.dtype in _DENSE and dst.stride(1) == 1 and src.stride(1) == 1, "scatter_add_rows_f32: fp32 dst, dense src")
    count = int(index.numel() if index is not None else (src.shape[0] if count is None else count))
    n = int(dst.shape[1])
    with torch.cuda.device(dst.device):
        check(_lib.lib().ofspmm_scatter_add_rows_f32(_ptr(dst), dst.stride(0) if dst.shape[0] > 1 else n, _ptr(src),
                                                     src.stride(0) if src.shape[0] > 1 else n, _ptr(index),
                                                     _INDEX[index.dtype] if index is not None else _lib.DTYPE_INT32,
                                                     index_offset, count, n, _DENSE[src.dtype], max_ctas, _stream_ptr(dst)),
              "scatter_add_rows_f32")
    return dst


def cast_from_f32(dst: torch.Tensor, src: torch.Tensor) -> torch.Tensor:
    """dst = dtype(dst)(src) elementwise, src fp32, both contiguous with the same number of elements."""
    _check_device(dst, src)
    _chk(src.dtype == torch.float32 and dst.dtype in _DENSE and dst.is_contiguous() and src.is_contiguous()
         and dst.numel() == src.numel(), "cast_from_f32: contiguous fp32 source and dense destination of equal size")
    with torch.cuda.device(dst.device):
        check(_lib.lib().ofspmm_cast_from_f32(_ptr(src), _ptr(dst), dst.numel(), _DENSE[dst.dtype], _stream_ptr(dst)),
              "cast_from_f32")
    return dst
