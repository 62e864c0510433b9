"""Functional layer + autograd wiring — the mirror of SURVEY.md §8 rows a8 / a9.

``spmm_csr(a_crow, a_col, a_val, b, a_rows, a_cols)`` is the call a OneFlow user would make as
``flow._C.spmm_csr(...)`` (pattern: oneflow/core/functional/functional_api.yaml:1011-1015,
oneflow/core/functional/impl/nn_functor.cpp:290-323).  Gradients follow the grad-function pattern of
oneflow/core/autograd/gradient_funcs/matmul.cpp:36-104 and gather.cpp:29-72:

    Capture: remember which inputs need grad, save crow/col/val/b as needed
    Apply:   in_grads[a_val] = sddmm_csr(crow, col, dy, b)        iff a_val.requires_grad
             in_grads[b]     = spmm_csr_grad_b(crow, col, val, dy) iff b.requires_grad
             index inputs never get a gradient (ModifyInputArg: set_requires_grad(false),
             oneflow/user/ops/unsorted_segment_sum_op.cpp:71-78)

``a_val=None`` is a pattern matrix (every stored entry 1): only ``b`` gets a gradient.
``reduce="mean"`` divides each row by its stored-entry count; its backward scales dy row-wise by
1/len (``_mean_scale``) and then runs the same SDDMM and A^T·dy as the sum.
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import torch

from . import ops


class SpmmOpKernelState:
    """Per-op persistent data — the role OpKernelState plays in the reference
    (oneflow/user/kernels/stateful_opkernel.cpp:919-928): one ``ops.SpmmPlan`` per CSR *structure*
    (histogram-chosen kernel variants, cached task partitions, and the structure of A^T with its
    value permutation).  Values are never cached — the backward re-gathers ``a_val`` through
    ``t_perm`` on every call — so in-place updates of learnable edge weights are always seen.  The
    key holds the index tensors' data pointers, shapes and autograd versions, and the plan keeps
    the index tensors alive, so a recycled address cannot alias a different graph."""

    def __init__(self, transpose: bool = True) -> None:
        self._plan: Optional[ops.SpmmPlan] = None
        self._transpose = transpose

    def plan(self, a_crow, a_col, a_rows: int, a_cols: int, n: int, dtype) -> "ops.SpmmPlan":
        p = self._plan
        if p is None or not p.matches(a_crow, a_col, a_rows, a_cols, n, dtype):
            p = ops.SpmmPlan(a_crow, a_col, a_rows, a_cols, n, dtype, transpose=self._transpose)
            self._plan = p                               # one entry: the op sees one graph at a time
        return p

    def clear(self) -> None:
        self._plan = None


def _detach(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    return None if t is None else t.detach()


def _mean_scale(dz: torch.Tensor, a_crow: torch.Tensor, plan) -> torch.Tensor:
    """dz ⊙ (1/len) per row — the backward of the mean's division (0 for an empty row).  The 1/len
    vector is kept on the plan when the op has a state."""
    inv = plan.inv_row_lengths() if plan is not None else ops.inv_row_lengths(a_crow)
    return (dz * inv).to(dz.dtype).contiguous()


class _SpmmCsrFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a_crow, a_col, a_val, b, a_rows, a_cols, state, reduce):
        plan = state.plan(a_crow, a_col, a_rows, a_cols, b.shape[1], b.dtype) if state is not None else None
        out = ops.spmm_csr_compute(a_crow, a_col, _detach(a_val), b.detach(), a_rows, a_cols, plan=plan, reduce=reduce)
        # Capture (matmul.cpp:48-73): save only what Apply will read
        ctx.val_requires_grad = a_val is not None and a_val.requires_grad
        ctx.b_requires_grad = b.requires_grad
        ctx.a_rows, ctx.a_cols, ctx.state, ctx.reduce = a_rows, a_cols, state, reduce
        ctx.save_for_backward(a_crow, a_col, a_val, b if ctx.val_requires_grad else None)
        ctx.mark_non_differentiable(a_crow, a_col)
        return out

    @staticmethod
    def backward(ctx, dy):
        a_crow, a_col, a_val, b = ctx.saved_tensors
        dy = dy.contiguous()
        d_val = d_b = None
        plan = None
        if ctx.state is not None:
            plan = ctx.state.plan(a_crow, a_col, ctx.a_rows, ctx.a_cols, dy.shape[1], dy.dtype)
        if ctx.reduce == "mean":
            dy = _mean_scale(dy, a_crow, plan)
        if ctx.val_requires_grad:
            d_val = ops.sddmm_csr_compute(a_crow, a_col, dy, b, ctx.a_rows, ctx.a_cols, a_val.dtype, plan=plan)
        if ctx.b_requires_grad:
            # cached structure of A^T when the op has a state, transient transpose otherwise — both
            # deterministic; the atomic scatter is opt-in (ops.spmm_csr_grad_b_compute(atomic=True))
            d_b = ops.spmm_csr_grad_b_compute(a_crow, a_col, _detach(a_val), dy, ctx.a_rows, ctx.a_cols, plan=plan)
        return None, None, d_val, d_b, None, None, None, None


def spmm_csr(a_crow: torch.Tensor, a_col: torch.Tensor, a_val: Optional[torch.Tensor], b: torch.Tensor,
             a_rows: int, a_cols: int, state: Optional[SpmmOpKernelState] = None, *,
             reduce: str = "sum") -> torch.Tensor:
    """out[a_rows, n] = CSR(a_crow, a_col, a_val; a_rows x a_cols) @ b[a_cols, n].

    Differentiable wrt ``a_val`` (SDDMM) and ``b`` (A^T·dy).  ``state`` (optional) keeps the plan of
    the CSR structure (variant, task partition, structure of A^T); without it the partition is
    recomputed per call and the backward builds A^T transiently — still deterministic.
    ``a_val=None``: pattern matrix (every stored entry 1, no values array).  ``reduce="mean"``:
    row i is divided by its stored-entry count (torch.sparse.mm(reduce="mean")); empty rows give 0."""
    ops.reduce_flag(reduce)
    val_grad = a_val is not None and a_val.requires_grad
    if not (torch.is_grad_enabled() and (val_grad or b.requires_grad)):
        plan = state.plan(a_crow, a_col, a_rows, a_cols, b.shape[1], b.dtype) if state is not None else None
        return ops.spmm_csr_compute(a_crow, a_col, a_val, b, a_rows, a_cols, plan=plan, reduce=reduce)
    ops._check_device(a_crow, a_col, a_val, b)
    ops.infer_spmm_csr(a_crow, a_col, a_val, b, a_rows, a_cols)
    return _SpmmCsrFn.apply(a_crow, a_col, a_val, b, a_rows, a_cols, state, reduce)


def spmm_csr_grad_b(a_crow, a_col, a_val, dy, a_rows: int, a_cols: int, transposed=None, plan=None,
                    atomic: bool = False) -> torch.Tensor:
    """db[a_cols, n] = A^T @ dy (the op the grad function dispatches for ``b``)."""
    return ops.spmm_csr_grad_b_compute(a_crow, a_col, a_val, dy, a_rows, a_cols, transposed, plan=plan, atomic=atomic)


def sddmm_csr(a_crow, a_col, dy, b, a_rows: int, a_cols: int, val_dtype=torch.float32) -> torch.Tensor:
    """dval[p] = <dy[row(p), :], b[a_col[p], :]> (the op the grad function dispatches for ``a_val``)."""
    return ops.sddmm_csr_compute(a_crow, a_col, dy, b, a_rows, a_cols, val_dtype)


# ---------------------------------------------------------------------------------------------
# aggregation with the epilogue fused into the SpMM store (SURVEY.md §8f rank 2)

class OpsKernels:
    """The three device entry points an aggregation layer needs, bound to the C ABI.  Tests of the
    autograd wiring inject a CPU stand-in with the same three methods; the product path is this.
    ``fwd`` receives ``reduce="mean"`` as a keyword only for mean aggregations, so a stand-in that
    serves sum aggregations only needs no such argument."""

    def fwd(self, a_crow, a_col, a_val, b, a_rows, a_cols, bias, relu, plan, reduce="sum"):
        return ops.spmm_csr_compute(a_crow, a_col, a_val, b, a_rows, a_cols, plan=plan, bias=bias, relu=relu,
                                    reduce=reduce)

    def grad_b(self, a_crow, a_col, a_val, dy, a_rows, a_cols, plan):
        return ops.spmm_csr_grad_b_compute(a_crow, a_col, a_val, dy, a_rows, a_cols, plan=plan)

    def sddmm(self, a_crow, a_col, dy, b, a_rows, a_cols, val_dtype, plan):
        return ops.sddmm_csr_compute(a_crow, a_col, dy, b, a_rows, a_cols, val_dtype, plan=plan)


class _SpmmCsrEpilogueFn(torch.autograd.Function):
    """out = act(A·b + bias) with bias and ReLU applied where the row sum is stored
    (OFSPMM_FWD_BIAS | OFSPMM_FWD_RELU; precedent for a fused epilogue in the reference:
    oneflow/user/kernels/cublas_fused_mlp_kernel.cu).  Backward: dz = dy ⊙ [out > 0] (the mask comes
    from the saved OUTPUT, so the pre-activation is never materialised), dbias = Σ_rows dz,
    db = Aᵀ·dz, dval = sddmm(dz, b).  With ``reduce="mean"`` the product is divided row-wise by the
    stored-entry counts before the bias: dbias takes dz, then dz is scaled by 1/len for db / dval."""

    @staticmethod
    def forward(ctx, a_crow, a_col, a_val, b, bias, a_rows, a_cols, relu, state, kernels, reduce):
        plan = state.plan(a_crow, a_col, a_rows, a_cols, b.shape[1], b.dtype) if state is not None else None
        kw = {"reduce": reduce} if reduce != "sum" else {}
        out = kernels.fwd(a_crow, a_col, _detach(a_val), b.detach(), a_rows, a_cols,
                          None if bias is None else bias.detach(), relu, plan, **kw)
        need_val = a_val is not None and a_val.requires_grad
        ctx.need = (need_val, b.requires_grad, bias is not None and bias.requires_grad)
        ctx.a_rows, ctx.a_cols, ctx.state, ctx.relu, ctx.kernels = a_rows, a_cols, state, relu, kernels
        ctx.reduce = reduce
        ctx.save_for_backward(a_crow, a_col, a_val, b if need_val else None, out if relu else None)
        ctx.mark_non_differentiable(a_crow, a_col)
        return out

    @staticmethod
    def backward(ctx, dy):
        a_crow, a_col, a_val, b, out = ctx.saved_tensors
        need_val, need_b, need_bias = ctx.need
        dz = dy * (out > 0).to(dy.dtype) if ctx.relu else dy
        dz = dz.contiguous()
        plan = None
        if ctx.state is not None:
            plan = ctx.state.plan(a_crow, a_col, ctx.a_rows, ctx.a_cols, dz.shape[1], dz.dtype)
        d_val = d_b = d_bias = None
        if need_bias:
            d_bias = dz.float().sum(0).to(dz.dtype)
        if ctx.reduce == "mean":
            dz = _mean_scale(dz, a_crow, plan)
        if need_val:
            d_val = ctx.kernels.sddmm(a_crow, a_col, dz, b, ctx.a_rows, ctx.a_cols, a_val.dtype, plan)
        if need_b:
            d_b = ctx.kernels.grad_b(a_crow, a_col, _detach(a_val), dz, ctx.a_rows, ctx.a_cols, plan)
        return None, None, d_val, d_b, d_bias, None, None, None, None, None, None


def spmm_csr_bias_act(a_crow: torch.Tensor, a_col: torch.Tensor, a_val: Optional[torch.Tensor], b: torch.Tensor,
                      a_rows: int, a_cols: int, bias: Optional[torch.Tensor] = None, relu: bool = False,
                      state: Optional[SpmmOpKernelState] = None, kernels=None, *, reduce: str = "sum") -> torch.Tensor:
    """out[a_rows, n] = act(CSR(a_crow, a_col, a_val) @ b + bias), epilogue fused into the product's
    store; differentiable wrt ``a_val``, ``b`` and ``bias``.  ``a_val=None``: pattern matrix;
    ``reduce="mean"``: the product is divided row-wise by the stored-entry counts before the bias."""
    ops.reduce_flag(reduce)
    kernels = kernels or OpsKernels()
    if isinstance(kernels, OpsKernels):
        ops._check_device(a_crow, a_col, a_val, b)
        ops.infer_spmm_csr(a_crow, a_col, a_val, b, a_rows, a_cols)
    if bias is not None and (bias.dim() != 1 or bias.shape[0] != b.shape[1] or bias.dtype != b.dtype):
        raise ops.OpInferError(f"bias must be a 1-D tensor of {b.shape[1]} elements of dtype {b.dtype}")
    return _SpmmCsrEpilogueFn.apply(a_crow, a_col, a_val, b, bias, a_rows, a_cols, bool(relu), state, kernels, reduce)
