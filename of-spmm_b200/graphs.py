"""Seeded synthetic CSR generators for the BASELINE.json configs (SURVEY.md §8d).

All generators are torch-only and device-agnostic: the bench builds the full-size graphs on the
GPU (cfg2 ≈ 115 M, cfg4 ≈ 2^28 edge draws), the tests build down-scaled twins on the CPU.
Conventions: column indices sorted and unique within a row; ``crow``/``col`` int32; values fp32
``U(-1, 1)``.  The real Reddit / ogbn-products / Graph500 data are not available offline; node and
edge counts and degree clips are generator parameters (SURVEY.md §8d "Provenance").
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import torch


@dataclass
class CsrMatrix:
    """A = (crow[M+1], col[nnz], val[nnz]) of logical shape rows × cols."""
    crow: torch.Tensor
    col: torch.Tensor
    val: torch.Tensor
    rows: int
    cols: int

    @property
    def nnz(self) -> int:
        return int(self.col.numel())

    def to(self, device) -> "CsrMatrix":
        return CsrMatrix(self.crow.to(device), self.col.to(device), self.val.to(device),
                         self.rows, self.cols)

    def row_lengths(self) -> torch.Tensor:
        return (self.crow[1:] - self.crow[:-1]).to(torch.int64)

    def row_slice(self, r0: int, r1: int) -> "CsrMatrix":
        """Rows [r0, r1) as their own CSR (crow re-based to 0); all K columns kept."""
        p0, p1 = int(self.crow[r0]), int(self.crow[r1])
        return CsrMatrix((self.crow[r0:r1 + 1] - self.crow[r0]).contiguous(),
                         self.col[p0:p1].contiguous(), self.val[p0:p1].contiguous(),
                         r1 - r0, self.cols)

    def scipy(self):
        import scipy.sparse as sp
        return sp.csr_matrix((self.val.cpu().numpy(), self.col.cpu().numpy(),
                              self.crow.cpu().numpy()), shape=(self.rows, self.cols))


def _gen(seed: int, device) -> torch.Generator:
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    return g


def _keys_to_csr(keys: torch.Tensor, M: int, K: int, val: Optional[torch.Tensor],
                 g: torch.Generator) -> CsrMatrix:
    """keys = row*K + col, sorted and unique."""
    rows = torch.div(keys, K, rounding_mode="floor")
    col = (keys - rows * K).to(torch.int32)
    counts = torch.bincount(rows, minlength=M)
    crow = torch.zeros(M + 1, dtype=torch.int64, device=keys.device)
    crow[1:] = torch.cumsum(counts, 0)
    assert int(crow[-1]) < 2 ** 31, "nnz must fit int32 row offsets"
    if val is None:
        val = torch.rand(keys.numel(), generator=g, device=keys.device, dtype=torch.float32) * 2 - 1
    return CsrMatrix(crow.to(torch.int32), col, val, M, K)


def _sample_distinct(deg: torch.Tensor, K: int, sampler, max_rounds: int = 16) -> torch.Tensor:
    """Draw ``deg[i]`` distinct columns for every row i; returns sorted unique keys row*K+col.

    Duplicates inside a row are removed and topped up with fresh draws until every row has its
    requested count (or max_rounds is hit, which only happens if a row asks for more columns than
    its sampler can produce)."""
    M = deg.numel()
    dev = deg.device
    keys = torch.empty(0, dtype=torch.int64, device=dev)
    need = deg.clone()
    ar = torch.arange(M, device=dev)
    for rnd in range(max_rounds):
        if int(need.sum()) == 0:
            break
        rows = torch.repeat_interleave(ar, need)
        cols = sampler(rows, rnd)
        keys = torch.unique(torch.cat([keys, rows * K + cols]))
        have = torch.bincount(torch.div(keys, K, rounding_mode="floor"), minlength=M)
        need = (deg - have).clamp_(min=0)
    return keys


def uniform_csr(M: int, K: int, density: float, seed: int = 1, device="cpu") -> CsrMatrix:
    """cfg1: per-row nnz ~ Binomial(K, density), columns uniform without replacement."""
    g = _gen(seed, device)
    probs = torch.full((M,), float(density), device=device)
    deg = torch.binomial(torch.full((M,), float(K), device=device), probs, generator=g).to(torch.int64)
    deg.clamp_(max=K)

    def sampler(rows, rnd):
        return torch.randint(0, K, (rows.numel(),), generator=g, device=device, dtype=torch.int64)

    return _keys_to_csr(_sample_distinct(deg, K, sampler), M, K, None, g)


def lognormal_degrees(M: int, nnz: int, sigma: float, dmin: int, dmax: int,
                      g: torch.Generator, device) -> torch.Tensor:
    """Integer degrees ~ lognormal(sigma), clipped to [dmin, dmax], summing to exactly ``nnz``."""
    z = torch.randn(M, generator=g, device=device, dtype=torch.float64)
    w = torch.exp(sigma * z)
    dmax = min(dmax, max(dmin, nnz))
    deg = torch.full((M,), dmin, dtype=torch.int64, device=device)
    # water-filling: rescale the unclipped part a few times so the clipped sum hits the target
    scale = nnz / float(w.sum())
    for _ in range(30):
        deg = torch.clamp(torch.floor(w * scale).to(torch.int64), dmin, dmax)
        s = int(deg.sum())
        if s == nnz:
            break
        free = (deg > dmin) & (deg < dmax)
        denom = float((w * free).sum())
        if denom <= 0:
            break
        scale *= 1.0 + (nnz - s) / (denom * scale)
    # exact fix-up of the remainder on rows that still have room
    diff = nnz - int(deg.sum())
    if diff != 0:
        step = 1 if diff > 0 else -1
        room = (deg < dmax) if diff > 0 else (deg > dmin)
        idx = torch.nonzero(room).flatten()
        n = abs(diff)
        reps = (n + idx.numel() - 1) // max(1, idx.numel())
        perm = idx[torch.randperm(idx.numel(), generator=g, device=device)]
        for _ in range(reps):
            take = perm[: min(n, perm.numel())]
            deg[take] += step
            n -= take.numel()
            if n == 0:
                break
        deg.clamp_(dmin, dmax)
    return deg


def community_csr(M: int, nnz: int, sigma: float = 1.2, dmin: int = 1, dmax: int = 21657,
                  communities: int = 50, p_local: float = 0.7, seed: int = 2,
                  device="cpu") -> CsrMatrix:
    """cfg2 / cfg3 (Reddit- / ogbn-products-shaped): lognormal degrees summing to ``nnz``;
    ``p_local`` of a row's columns fall in the row's own community (contiguous id block), the
    rest are uniform over all columns."""
    g = _gen(seed, device)
    K = M
    deg = lognormal_degrees(M, nnz, sigma, dmin, min(dmax, K), g, device)
    csize = (M + communities - 1) // communities

    def sampler(rows, rnd):
        # top-up rounds >= 3 draw globally so rows wider than their community can still fill up
        n = rows.numel()
        local = torch.rand(n, generator=g, device=device) < (p_local if rnd < 3 else 0.0)
        base = torch.div(rows, csize, rounding_mode="floor") * csize
        width = torch.clamp(K - base, max=csize)
        u = torch.rand(n, generator=g, device=device, dtype=torch.float64)
        loc = base + torch.floor(u * width).to(torch.int64)
        glob = torch.randint(0, K, (n,), generator=g, device=device, dtype=torch.int64)
        return torch.where(local, loc, glob)

    return _keys_to_csr(_sample_distinct(deg, K, sampler), M, K, None, g)


def reddit_like(scale_div: int = 1, seed: int = 2, device="cpu") -> CsrMatrix:
    """cfg2: 232 965 nodes, 114 615 892 nnz, 50 communities.  ``scale_div`` > 1 gives the parity
    twin: nodes and nnz ÷ scale_div (same degree law and average degree), community *size* kept."""
    M = 232965 // scale_div
    nnz = 114615892 // scale_div
    return community_csr(M, nnz, 1.2, 1, min(21657, M), max(1, 50 // scale_div), 0.7, seed, device)


def products_like(scale_div: int = 1, seed: int = 3, device="cpu") -> CsrMatrix:
    """cfg3: 2 449 029 nodes, 123 718 280 nnz, 47 communities (twin: see reddit_like)."""
    M = 2449029 // scale_div
    nnz = 123718280 // scale_div
    return community_csr(M, nnz, 1.2, 1, min(17481, M), max(1, 47 // scale_div), 0.7, seed, device)


def rmat_csr(scale: int, edge_factor: int = 16, a: float = 0.57, b: float = 0.19, c: float = 0.19,
             seed: int = 4, device="cpu", chunk: int = 1 << 24) -> CsrMatrix:
    """cfg4: Graph500 R-MAT, 2^scale vertices, edge_factor·2^scale directed edge draws, no vertex
    permutation (hub skew stays at low ids), duplicate edges coalesced by summing their values."""
    g = _gen(seed, device)
    M = 1 << scale
    E = edge_factor * M
    ab, abc = a + b, a + b + c
    key_parts, val_parts = [], []
    for s in range(0, E, chunk):
        n = min(chunk, E - s)
        r = torch.zeros(n, dtype=torch.int64, device=device)
        col = torch.zeros(n, dtype=torch.int64, device=device)
        for _ in range(scale):
            u = torch.rand(n, generator=g, device=device)
            rbit = (u >= ab).to(torch.int64)
            cbit = (((u >= a) & (u < ab)) | (u >= abc)).to(torch.int64)
            r = (r << 1) | rbit
            col = (col << 1) | cbit
        key_parts.append(r * M + col)
        val_parts.append(torch.rand(n, generator=g, device=device, dtype=torch.float32) * 2 - 1)
    keys = torch.cat(key_parts)
    vals = torch.cat(val_parts)
    del key_parts, val_parts
    keys, order = torch.sort(keys)
    vals = vals[order]
    del order
    ukeys, counts = torch.unique_consecutive(keys, return_counts=True)
    del keys
    ends = torch.cumsum(counts, 0)
    csum = torch.cumsum(vals.to(torch.float64), 0)
    seg = csum[ends - 1]
    seg[1:] = seg[1:] - csum[ends[:-1] - 1]
    return _keys_to_csr(ukeys, M, M, seg.to(torch.float32), g)


def gcn_normalize(A: CsrMatrix) -> CsrMatrix:
    """Symmetric GCN normalisation val[p] = 1/sqrt(d_i · d_j) with d = row length (self loops are
    expected to be present already); used by the cfg5 harness."""
    d = A.row_lengths().clamp(min=1).to(torch.float32)
    rows = torch.repeat_interleave(torch.arange(A.rows, device=A.crow.device), A.row_lengths())
    val = torch.rsqrt(d[rows] * d[A.col.to(torch.int64)])
    return CsrMatrix(A.crow, A.col, val, A.rows, A.cols)


def add_self_loops(A: CsrMatrix) -> CsrMatrix:
    assert A.rows == A.cols
    dev = A.crow.device
    rows = torch.repeat_interleave(torch.arange(A.rows, device=dev), A.row_lengths())
    keys = torch.cat([rows * A.cols + A.col.to(torch.int64),
                      torch.arange(A.rows, device=dev) * (A.cols + 1)])
    keys = torch.unique(keys)
    return _keys_to_csr(keys, A.rows, A.cols, torch.ones(keys.numel(), device=dev), _gen(0, dev))


def dense_operand(K: int, N: int, seed: int, device="cpu", dtype=torch.float32) -> torch.Tensor:
    """B ~ N(0,1) fp32 (cast to ``dtype``)."""
    g = _gen(seed + 1000, device)
    return torch.randn(K, N, generator=g, device=device, dtype=torch.float32).to(dtype)


def upstream_grad(M: int, N: int, seed: int, device="cpu", dtype=torch.float32) -> torch.Tensor:
    """dY ~ U(0,1) (house style of the reference's autotest,
    python/oneflow/test_utils/automated_test_util/torch_flow_dual_object.py:1210-1212)."""
    g = _gen(seed + 2000, device)
    return torch.rand(M, N, generator=g, device=device, dtype=torch.float32).to(dtype)


# A matrix with more non-zeros than int32 offsets can count (2^31 + 2^25, int64 indices; 26 GB on
# the device).  Row WIDE_HUB holds 2^25 entries straddling non-zero 2^31; the rows before it are
# ~2000 long, the rows after it ~16; every 97th row is empty and every 89th has one entry.
WIDE_M, WIDE_K, WIDE_NNZ = 1 << 21, 1 << 20, (1 << 31) + (1 << 25)
WIDE_HUB, WIDE_HUB_START, WIDE_HUB_LEN = 1 << 20, (1 << 31) - (1 << 24), 1 << 25
# (position, column) of the entries outside [0, K), which every kernel skips: on both sides of 2^31
WIDE_BAD = ((1000, -1), ((1 << 31) - 5, -1), ((1 << 31) - 3, WIDE_K), ((1 << 31) + 7, -1),
            ((1 << 31) + 11, WIDE_K), (WIDE_NNZ - 2, WIDE_K))


def _wide_lengths(g: torch.Generator, n: int, total: int) -> torch.Tensor:
    idx = torch.arange(n)
    w = torch.rand(n, generator=g, dtype=torch.float64) + 0.5
    ones = idx % 89 == 5
    w[(idx % 97 == 3) | ones] = 0
    target = total - int(ones.sum())
    lens = torch.floor(w / w.sum() * target).to(torch.int64)
    lens[torch.nonzero(w > 0).flatten()[:target - int(lens.sum())]] += 1
    lens[ones] = 1
    return lens


def _mix64_(x: torch.Tensor) -> torch.Tensor:
    """In-place splitmix64 finaliser on int64 (wrapping products, logical shifts)."""
    x.mul_(-7046029254386353131)
    x.bitwise_xor_((x >> 30) & ((1 << 34) - 1))
    x.mul_(-4658895280553007687)
    x.bitwise_xor_((x >> 27) & ((1 << 37) - 1))
    x.mul_(-7723592293110705685)
    x.bitwise_xor_((x >> 31) & ((1 << 33) - 1))
    return x


def wide_csr(device="cuda", seed: int = 9, chunk: int = 1 << 26) -> CsrMatrix:
    """The WIDE_* matrix built on ``device`` in chunks: column and fp32 value of non-zero p are a
    hash of (seed, p), values k / 2^15 in [-1, 1)."""
    g = torch.Generator().manual_seed(seed)
    lens = torch.empty(WIDE_M, dtype=torch.int64)
    lens[:WIDE_HUB] = _wide_lengths(g, WIDE_HUB, WIDE_HUB_START)
    lens[WIDE_HUB] = WIDE_HUB_LEN
    lens[WIDE_HUB + 1:] = _wide_lengths(g, WIDE_M - WIDE_HUB - 1, WIDE_NNZ - WIDE_HUB_START - WIDE_HUB_LEN)
    crow = torch.zeros(WIDE_M + 1, dtype=torch.int64)
    crow[1:] = torch.cumsum(lens, 0)
    assert int(crow[-1]) == WIDE_NNZ and int(crow[WIDE_HUB]) == WIDE_HUB_START
    col = torch.empty(WIDE_NNZ, dtype=torch.int64, device=device)
    val = torch.empty(WIDE_NNZ, dtype=torch.float32, device=device)
    for p0 in range(0, WIDE_NNZ, chunk):
        p1 = min(WIDE_NNZ, p0 + chunk)
        x = _mix64_(torch.arange(p0, p1, dtype=torch.int64, device=device).add_(seed << 48))
        col[p0:p1] = (x >> 24) & (WIDE_K - 1)
        val[p0:p1] = ((x & 0xFFFF) - 32768).to(torch.float32).div_(32768.0)
        del x
    for p, c in WIDE_BAD:
        col[p] = c
    return CsrMatrix(crow.to(device), col, val, WIDE_M, WIDE_K)


def expected_alg_bytes(M: int, K: int, nnz: int, N: int, s_dense: int, s_val: int = 4,
                       s_idx: int = 4) -> dict:
    """SURVEY.md §8d: gather-model (M2) and compulsory (M1) byte counts for one SpMM."""
    csr = nnz * (s_idx + s_val) + (M + 1) * s_idx
    return {"m2": csr + nnz * N * s_dense + M * N * s_dense,
            "m1": csr + K * N * s_dense + M * N * s_dense,
            "flop": 2 * nnz * N}
