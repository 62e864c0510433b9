"""2-layer GCN on top of the SpMM op — the caller of the hot path in BASELINE.json configs[4]
("2-layer GCN forward+backward (SpMM + SDDMM value grad, hidden 256) on a Reddit-shaped synthetic
graph, random-init weights").  SURVEY.md §8f rank 2 ("next" row): a thin harness, not a framework —
dense X·W products are left to torch (cuBLAS, a plain library GEMM), every aggregation Â·H goes
through ``spmm_csr`` and therefore through the C ABI: forward ``ofspmm_fwd``, backward
``ofspmm_bwd_b`` on the cached transpose, and ``ofspmm_sddmm`` when the edge weights need a
gradient.

    H1  = relu( Â · (X · W1) )          aggregate at width `hidden`   (602 → 256: multiply first)
    out =       (Â · H1) · W2           aggregate at width `hidden`   (256 → 41: aggregate first)

so both aggregations run at the dense width BASELINE.md quotes for cfg5 (N = 256).
"""
from __future__ import annotations

import math
from typing import Callable, Optional

import torch

from .functional import SpmmOpKernelState, spmm_csr
from .graphs import CsrMatrix


def glorot(fan_in: int, fan_out: int, seed: int, device, dtype=torch.float32) -> torch.Tensor:
    g = torch.Generator(device="cpu")
    g.manual_seed(seed)
    bound = math.sqrt(6.0 / (fan_in + fan_out))
    w = (torch.rand(fan_in, fan_out, generator=g, dtype=torch.float32) * 2 - 1) * bound
    return w.to(device=device, dtype=dtype)


class GCNConv:
    """One graph-convolution layer  out = act(Â · X · W + bias)  — the module-level caller of the op
    (pattern: python/oneflow/nn/modules/linear.py; SURVEY.md §8f rank 2).

    * **Ordering by width**: the aggregation runs at the narrower of the two dense widths.
      ``multiply first``  (out_dim ≤ in_dim):  Z = X·W (cuBLAS), out = act(Â·Z + bias) with bias and
      ReLU **fused into the SpMM store** (one pass over the output, no pre-activation tensor);
      ``aggregate first`` (out_dim > in_dim):  G = Â·X, out = act(G·W + bias) — the epilogue
      follows the GEMM, so it is torch's.
    * Dropout acts on the layer input (torch): a mask in the SpMM store would need a device RNG
      stream per launch, which the C ABI does not carry.
    * The normalised adjacency is shared between layers: pass the same ``CsrMatrix`` and the same
      ``SpmmOpKernelState`` (plan, structure of Âᵀ) to every layer of a model.

    ``kernels``: None = the C ABI (``functional.OpsKernels``); the CPU tests inject a stand-in."""

    def __init__(self, in_dim: int, out_dim: int, bias: bool = True, activation: Optional[str] = "relu",
                 order: str = "auto", dropout: float = 0.0, seed: int = 0, device="cuda", dtype=torch.float32,
                 kernels=None):
        assert activation in (None, "relu") and order in ("auto", "multiply_first", "aggregate_first")
        self.in_dim, self.out_dim, self.activation, self.p = in_dim, out_dim, activation, float(dropout)
        self.multiply_first = order == "multiply_first" or (order == "auto" and out_dim <= in_dim)
        self.weight = glorot(in_dim, out_dim, seed, device, dtype).requires_grad_(True)
        self.bias = torch.zeros(out_dim, device=device, dtype=dtype).requires_grad_(True) if bias else None
        self.kernels = kernels
        self.training = True

    def parameters(self):
        return [p for p in (self.weight, self.bias) if p is not None]

    def aggregation_width(self) -> int:
        return self.out_dim if self.multiply_first else self.in_dim

    def __call__(self, A: CsrMatrix, X: torch.Tensor, val: Optional[torch.Tensor] = None,
                 state: Optional[SpmmOpKernelState] = None) -> torch.Tensor:
        from .functional import spmm_csr_bias_act
        val = A.val if val is None else val
        relu = self.activation == "relu"
        if self.p > 0:
            X = torch.nn.functional.dropout(X, self.p, self.training)
        if self.multiply_first:
            z = (X @ self.weight).contiguous()
            return spmm_csr_bias_act(A.crow, A.col, val, z, A.rows, A.cols, self.bias, relu, state, self.kernels)
        g = spmm_csr_bias_act(A.crow, A.col, val, X.contiguous(), A.rows, A.cols, None, False, state, self.kernels)
        out = g @ self.weight
        if self.bias is not None:
            out = out + self.bias
        return torch.relu(out) if relu else out


class SAGEConv:
    """GraphSAGE layer with the mean aggregator

        out = act(mean_{j∈N(i)} x_j · W_neigh + x_i · W_root + bias)

    on the PATTERN matrix of the graph (``A.crow``, ``A.col``; ``A.val`` is never read): the
    aggregation is ``spmm_csr(a_val=None, reduce="mean")``, so no values tensor exists anywhere.
    Rows of A are the destination nodes; their root features are the first ``A.rows`` rows of X.

    * **Ordering by width**, as in ``GCNConv``: the aggregation runs at the narrower width.
      ``multiply first`` (out_dim ≤ in_dim): mean(X·W_neigh); ``aggregate first``: mean(X)·W_neigh.
    * The root term is added with ``torch.addmm``.  The mean cannot accumulate into an existing
      output (the division would apply to it too), so the SpMM epilogue fuses only the bias, and
      only when there is no activation and the aggregation comes last (multiply first).
    * An isolated node (empty row) aggregates to 0 and keeps its root term.

    ``kernels``: None = the C ABI (``functional.OpsKernels``); the CPU tests inject a stand-in."""

    def __init__(self, in_dim: int, out_dim: int, bias: bool = True, activation: Optional[str] = "relu",
                 order: str = "auto", seed: int = 0, device="cuda", dtype=torch.float32, kernels=None):
        assert activation in (None, "relu") and order in ("auto", "multiply_first", "aggregate_first")
        self.in_dim, self.out_dim, self.activation = in_dim, out_dim, activation
        self.multiply_first = order == "multiply_first" or (order == "auto" and out_dim <= in_dim)
        self.weight_neigh = glorot(in_dim, out_dim, seed, device, dtype).requires_grad_(True)
        self.weight_root = glorot(in_dim, out_dim, seed + 1, device, dtype).requires_grad_(True)
        self.bias = torch.zeros(out_dim, device=device, dtype=dtype).requires_grad_(True) if bias else None
        self.kernels = kernels

    def parameters(self):
        return [p for p in (self.weight_neigh, self.weight_root, self.bias) if p is not None]

    def aggregation_width(self) -> int:
        return self.out_dim if self.multiply_first else self.in_dim

    def __call__(self, A: CsrMatrix, X: torch.Tensor, state: Optional[SpmmOpKernelState] = None) -> torch.Tensor:
        from .functional import spmm_csr_bias_act
        fuse_bias = self.bias if (self.multiply_first and self.activation is None) else None
        if self.multiply_first:
            z = (X @ self.weight_neigh).contiguous()
            h = spmm_csr_bias_act(A.crow, A.col, None, z, A.rows, A.cols, fuse_bias, False, state, self.kernels,
                                  reduce="mean")
        else:
            g = spmm_csr_bias_act(A.crow, A.col, None, X.contiguous(), A.rows, A.cols, None, False, state,
                                  self.kernels, reduce="mean")
            h = g @ self.weight_neigh
        out = torch.addmm(h, X[:A.rows], self.weight_root)
        if self.bias is not None and fuse_bias is None:
            out = out + self.bias
        return torch.relu(out) if self.activation == "relu" else out


class GCN2:
    """Two GCNConv layers sharing one normalised adjacency Â = (crow, col, val)."""

    def __init__(self, A: CsrMatrix, in_dim: int = 602, hidden: int = 256, out_dim: int = 41, seed: int = 5,
                 edge_weight_grad: bool = True, spmm: Optional[Callable] = None):
        dev = A.crow.device
        self.A = A
        self.val = A.val.detach().clone().requires_grad_(edge_weight_grad)
        self.W1 = glorot(in_dim, hidden, seed, dev).requires_grad_(True)
        self.W2 = glorot(hidden, out_dim, seed + 1, dev).requires_grad_(True)
        self.state = SpmmOpKernelState() if spmm is None else None   # cached Aᵀ for the backward
        self._spmm = spmm

    def parameters(self):
        return [p for p in (self.W1, self.W2, self.val) if p.requires_grad]

    def aggregate(self, H: torch.Tensor) -> torch.Tensor:
        A = self.A
        if self._spmm is not None:
            return self._spmm(A.crow, A.col, self.val, H, A.rows, A.cols)
        return spmm_csr(A.crow, A.col, self.val, H.contiguous(), A.rows, A.cols, self.state)

    def forward(self, X: torch.Tensor) -> torch.Tensor:
        h1 = torch.relu(self.aggregate(X @ self.W1))
        return self.aggregate(h1) @ self.W2

    def train_step(self, X: torch.Tensor, labels: torch.Tensor, lr: float = 0.0) -> torch.Tensor:
        """One forward + backward (cross-entropy on all nodes); optional plain SGD update."""
        for p in self.parameters():
            p.grad = None
        loss = torch.nn.functional.cross_entropy(self.forward(X), labels)
        loss.backward()
        if lr > 0:
            with torch.no_grad():
                for p in (self.W1, self.W2):
                    p -= lr * p.grad
        return loss.detach()

    def spmm_flops_per_step(self) -> int:
        """FLOPs of the sparse products in one train_step: 2 aggregations × (forward + Aᵀ·dY)
        [+ SDDMM when edge weights need a gradient], each 2·nnz·hidden."""
        per = 2 * self.A.nnz * self.W1.shape[1]
        return 2 * (2 + (1 if self.val.requires_grad else 0)) * per


class ShardedGCN2:
    """The same two GCNConv layers on N GPUs (BASELINE configs[4], 8 x B200): node-parallel — rank r
    owns the nnz-balanced row block of Â and the matching rows of X, H1, the logits and the labels;
    W1 / W2 are replicated, their gradients all-reduced.  Both aggregations and all four sparse
    gradients go through ONE ``dist.ShardedSpmm`` (needed-rows exchange over peer memory), built
    with ``shard_like_rows`` so the output block of layer 1 *is* the input shard of layer 2, and two
    buffer slots so the rows each layer pulled in the forward are still there for its SDDMM:

        forward   Z1 = X_r W1            H1_r = relu(Â_r · Z1)     [ReLU fused into the SpMM store]
                  G_r = Â_r · H1         logits_r = G_r W2
        backward  dG = dlogits W2ᵀ       dH1_r = (Âᵀ dG)_r          dval += sddmm(dG, H1)
                  dZ = dH1 ⊙ [H1 > 0]    dZ1_r = (Âᵀ dZ)_r          dval += sddmm(dZ, Z1)
                  dW2 = Σ_r G_rᵀ dlogits_r        dW1 = Σ_r X_rᵀ dZ1_r          (all-reduce)

    The backward is written out by hand (no autograd graph across the exchange)."""

    def __init__(self, A: CsrMatrix, rank: int, world: int, device, in_dim: int = 602, hidden: int = 256,
                 out_dim: int = 41, seed: int = 5, edge_weight_grad: bool = True, group=None, compute=None,
                 tasks_per_warp: int = 4, buckets: int = 1):
        import importlib
        dmod = importlib.import_module(__package__ + ".dist")
        self.rank, self.world, self.group, self.device = rank, world, group, device
        self.sh = dmod.ShardedSpmm(A, hidden, torch.float32, rank, world, device, shard_like_rows=True, slots=2,
                                   group=group, compute=compute, tasks_per_warp=tasks_per_warp, buckets=buckets)
        self.nodes = A.rows
        self.m = self.sh.r1 - self.sh.r0
        self.W1 = glorot(in_dim, hidden, seed, device)
        self.W2 = glorot(hidden, out_dim, seed + 1, device)
        self.edge_weight_grad = edge_weight_grad
        self.grads = {}
        self._h1 = torch.empty((self.m, hidden), dtype=torch.float32, device=device)
        self._g = torch.empty((self.m, hidden), dtype=torch.float32, device=device)

    def local_rows(self, T: torch.Tensor) -> torch.Tensor:
        return T[self.sh.r0:self.sh.r1].contiguous()

    def _all_reduce(self, t: torch.Tensor) -> torch.Tensor:
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(t, group=self.group)
        return t

    def train_step(self, X_r: torch.Tensor, labels_r: torch.Tensor, lr: float = 0.0) -> torch.Tensor:
        """One forward + backward on this rank's nodes; returns the global mean cross-entropy."""
        sh, m = self.sh, self.m
        z1 = X_r @ self.W1
        h1 = sh.forward(z1, out=self._h1, relu=True, slot=0)[:m]
        g = sh.forward(h1, out=self._g, slot=1)[:m]
        logits = g @ self.W2
        logp = torch.log_softmax(logits, dim=1)
        loss_sum = -logp.gather(1, labels_r[:, None]).sum()
        dlogits = (torch.exp(logp) - torch.nn.functional.one_hot(labels_r, logits.shape[1]).to(logp.dtype)) / self.nodes
        dW2 = g.t() @ dlogits
        dG = dlogits @ self.W2.t()
        dval = None
        if self.edge_weight_grad:
            dval = sh.sddmm(dG, slot=1)                       # against H1 rows pulled by the 2nd forward
        dH1 = sh.backward(dG, slot=1)[:m]
        dZ = dH1 * (h1 > 0)
        if self.edge_weight_grad:
            dval = dval + sh.sddmm(dZ, slot=0)                # against Z1 rows pulled by the 1st forward
        dZ1 = sh.backward(dZ, slot=0)[:m]
        dW1 = X_r.t() @ dZ1
        packed = torch.cat([dW1.flatten(), dW2.flatten(), loss_sum.reshape(1)])
        self._all_reduce(packed)
        n1 = dW1.numel()
        self.grads = {"W1": packed[:n1].view_as(dW1), "W2": packed[n1:n1 + dW2.numel()].view_as(dW2), "val": dval}
        if lr > 0:
            self.W1 -= lr * self.grads["W1"]
            self.W2 -= lr * self.grads["W2"]
        return packed[-1] / self.nodes

    def spmm_flops_per_step(self) -> int:
        per = 2 * self.sh.A_blk.nnz * self.W1.shape[1]        # this rank's block
        return 2 * (2 + (1 if self.edge_weight_grad else 0)) * per
