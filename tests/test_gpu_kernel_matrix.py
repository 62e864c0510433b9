"""Every forward, SDDMM and atomic A^T.dY kernel instantiation against the fp64 oracle.

The cases come from tests/_kernel_matrix.py, which mirrors the dispatch code: each call asserts
the kernel the mirror predicts through ofspmm_launch_count() (partition, merge kernel, fix-up when
the matrix has more than one task; one launch for the whole-row kernel) and, once per case, by the
kernel names torch.profiler records; and
tests/test_kernel_matrix_host.py checks that the cases reach every instantiation in the library.

The graphs are built to hit the places where such kernels go wrong: empty first and last rows and
runs of empty rows, rows that end or start exactly on a 64- or 256-item task boundary, hub rows
spanning many tasks (the fix-up kernel's binary search), and out-of-range columns (-1, cols, 2^30)
next to a NaN row 0 of B that no valid entry reads, so a wrongly masked index shows up as NaN.

Tolerances (oracle/oracle.py, SURVEY.md §8c):
  * fp32: O.fp32_tolerance, plus 2^-22 (|C_old| + |bias|) with accumulate or bias, plus
    2^-22 |s/len| for the mean;
  * bf16 outputs are rounded once from an fp32 result (include/ofspmm.h, DESIGN.md), so each element
    must be within tol32 + 1/2 ulp_bf16(|ref| + tol32) of the fp64 reference, tol32 the fp32 bound:
    a second rounding (a bf16 partial row, a bf16 round trip between acc32 passes) fails it.
"""
import os
import re
import subprocess
import sys
from functools import lru_cache

import numpy as np
import pytest
import torch

import ofspmm_b200 as ofs
from oracle import oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import _kernel_matrix as KM  # noqa: E402

pytestmark = pytest.mark.gpu
ops = __import__("importlib").import_module("of-spmm_b200.ops")
_lib = ofs._lib
DEV = "cuda:0"
TORCH = {KM.F32: torch.float32, KM.BF16: torch.bfloat16}
IDX = {KM.I32: torch.int32, KM.I64: torch.int64}


# ------------------------------------------------------------------ graphs

def matrix_graph(M=3000, K=2500, seed=5):
    """Rows of 0..29 entries; empty rows 0, M-1, 200..239 and 1500..1502; two hub rows of 3000
    entries (~12 256-item tasks each); rows adjusted so that rows start (S) and end (E) exactly on
    task boundaries; out-of-range columns only in rows 1000..1099 and in the second hub, so most
    tasks stay on the vectorised path.  Valid columns avoid 0 (B row 0 is NaN bait).  The merge
    items (rows + nnz) are a multiple of 256, so every task boundary is a diagonal k * items."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, 30, M)
    lens[rng.random(M) < 0.08] = 0
    fixed = np.zeros(M, dtype=bool)
    for lo, hi in ((0, 1), (200, 240), (1500, 1503), (M - 1, M)):
        lens[lo:hi] = 0
        fixed[lo:hi] = True
    hubs = (M - 400, M - 150)
    lens[list(hubs)] = 3000
    fixed[list(hubs)] = True
    # (diagonal, kind): S = a row starts at it (the previous one ended just before), E = a row's
    # last entry is the last item before it (its end marker falls into the next task)
    targets = [(256 * 20, "S"), (64 * 301, "S"), (256 * 120, "S"), (256 * 45, "E"), (64 * 401, "E"),
               (256 * 140, "E")]
    pos = 0
    for i in range(M):
        if not fixed[i]:
            for T, kind in targets:
                if kind == "S" and pos < T <= pos + lens[i] + 1:
                    lens[i] = T - pos - 1
                elif kind == "E" and pos < T <= pos + lens[i] + 1:
                    lens[i] = T - pos
        pos += int(lens[i]) + 1
    last = max(i for i in range(M - 300, M - 160) if not fixed[i])
    lens[last] += (-(M + int(lens.sum()))) % 256
    crow = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    nnz = int(crow[-1])
    col = rng.integers(1, K, nnz)
    rows_of = np.repeat(np.arange(M), lens)
    bad = ((rows_of >= 1000) & (rows_of < 1100) | (rows_of == hubs[1])) & (rng.random(nnz) < 0.1)
    choice = rng.integers(0, 3, int(bad.sum()))
    col[bad] = np.array([-1, K, 1 << 30])[choice]
    val = rng.uniform(-1, 1, nnz).astype(np.float32)
    return crow, col, val, M, K


def short_row_graph(M=6000, K=3000, seed=8):
    """Short rows only (0..12 entries, none near 512) and enough rows that the plan's histogram
    picks the whole-row kernel for widths up to 32 vectors."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, 13, M)
    lens[[0, M - 1]] = 0
    crow = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    col = rng.integers(1, K, int(crow[-1]))
    return crow, col, rng.uniform(-1, 1, col.size).astype(np.float32), M, K


def check_graph_shape(crow: torch.Tensor, ops_mod, strict: bool = True):
    lens = (crow[1:] - crow[:-1]).numpy()
    M, nnz = lens.size, int(crow[-1])
    assert lens[0] == 0 and lens[-1] == 0
    if not strict:
        return
    runs = np.flatnonzero(np.convolve(lens == 0, np.ones(3, dtype=int), "valid") == 3)
    assert runs.size > 0, "no run of empty rows"
    assert (lens > 5 * 256).sum() >= 2, "needs two hub rows over 5 tasks"
    assert (M + nnz) % 256 == 0
    c = crow.numpy()
    for items in (64, 256):
        r, z = ops_mod.merge_path_partition_host(crow, nnz, (M + nnz) // items)
        r, z = r.numpy()[1:-1], z.numpy()[1:-1]
        k = np.arange(1, r.size + 1)
        only = (k % 4 != 0) if items == 64 else np.ones(k.size, dtype=bool)
        nonempty = c[np.minimum(r + 1, M)] > c[r]
        starts = only & (z == c[r]) & nonempty & (r > 0) & (c[r] > c[np.maximum(r - 1, 0)])
        ends = only & (z == c[np.minimum(r + 1, M)]) & nonempty
        assert starts.any(), f"no row starts exactly on a {items}-item task boundary"
        assert ends.any(), f"no row ends exactly on a {items}-item task boundary"


class Graph:
    def __init__(self, crow, col, val, M, K, idx):
        self.M, self.K, self.idx = M, K, idx
        self.crow_np, self.col_np, self.val_np = crow, col, val
        self.lens = np.diff(crow)
        self.nnz = int(crow[-1])
        t = IDX[idx]
        self.crow = torch.from_numpy(crow).to(t).to(DEV)
        self.col = torch.from_numpy(col).to(t).to(DEV)
        self.val = {KM.F32: torch.from_numpy(val).to(DEV), KM.BF16: torch.from_numpy(val).to(DEV).to(torch.bfloat16),
                    KM.UNIT: None}
        # three sub-matrices (entries by position mod 3) for the bf16 fp32-accumulator passes
        self.parts = []
        pos = np.arange(self.nnz)
        rows_of = np.repeat(np.arange(M), self.lens)
        for r in range(3):
            m = pos % 3 == r
            pc = np.concatenate([[0], np.cumsum(np.bincount(rows_of[m], minlength=M))])
            self.parts.append((torch.from_numpy(pc).to(t).to(DEV), torch.from_numpy(col[m]).to(t).to(DEV),
                               {KM.F32: torch.from_numpy(val[m]).to(DEV),
                                KM.BF16: torch.from_numpy(val[m]).to(DEV).to(torch.bfloat16), KM.UNIT: None},
                               int(m.sum())))

    def val_f32(self, val_dtype):
        if val_dtype == KM.UNIT:
            return np.ones(self.nnz, np.float32)
        if val_dtype == KM.BF16:
            return torch.from_numpy(self.val_np).to(torch.bfloat16).float().numpy()
        return self.val_np


@pytest.fixture(scope="module")
def graphs():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    g = matrix_graph()
    return {idx: Graph(*g, idx) for idx in (KM.I32, KM.I64)}


@pytest.fixture(scope="module")
def short_graph():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return Graph(*short_row_graph(), KM.I32)


# ------------------------------------------------------------------ operands and references

@lru_cache(maxsize=None)
def _host_dense(rows, n, seed, dense, nan_row0=False):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(rows, n, generator=g, dtype=torch.float32)
    if nan_row0:
        x[0] = float("nan")
    return x.to(TORCH[dense])


def _carve(host, misaligned: bool):
    """Device copy of `host`; `misaligned`: a packed tensor carved one element into a larger buffer."""
    if not misaligned:
        return host.to(DEV)
    buf = torch.empty(host.numel() + 8, dtype=host.dtype, device=DEV)
    out = buf[1:1 + host.numel()].view(host.shape)
    out.copy_(host.to(DEV))
    return out


_REF = {}


def _fwd_ref(G, n, dense, val):
    """fp64 product, largest term per element; cached per (graph, n, input dtypes)."""
    key = ("fwd", id(G.crow_np), n, dense, val)
    if key not in _REF:
        B = _host_dense(G.K, n, 1, dense, True).float().numpy()
        v = G.val_f32(val)
        _REF[key] = (O.spmm_f64(G.crow_np, G.col_np, v, B, G.K), O.spmm_absmax(G.crow_np, G.col_np, v, B, G.K))
    return _REF[key]


def _ulp_bf16(x):
    e = np.floor(np.log2(np.maximum(np.abs(x), 2.0 ** -126)))
    return 2.0 ** (e - 7)


def _check(got, ref, tol32, dense, what):
    """fp32: |got - ref| <= tol32; bf16: faithful rounding of an fp32 result within tol32."""
    g = got.float().cpu().numpy().astype(np.float64)
    tol = tol32 + 1e-30
    if dense == KM.BF16:
        tol = tol32 + 0.5 * _ulp_bf16(np.abs(ref) + tol32)
    err = np.abs(g - ref)
    ok = err <= tol
    if not ok.all():
        i = np.argwhere(~ok)[0]
        raise AssertionError(f"{what}: {int((~ok).sum())} elements out of tolerance, first at {tuple(i)}: "
                             f"got {g[tuple(i)]!r} want {ref[tuple(i)]!r} tol {tol[tuple(i)]:.3e}")


def _launch(fn, want: KM.Launch, what):
    n0 = _lib.lib().ofspmm_launch_count()
    out = fn()
    assert _lib.lib().ofspmm_launch_count() - n0 == want.launches, f"{what}: launches != {want}"
    return out


def _mod(t):
    return t.data_ptr() % 16


# ------------------------------------------------------------------ forward

@pytest.mark.parametrize("case", KM.fwd_cases(), ids=lambda c: c.id)
def test_forward(graphs, case):
    G = graphs[case.idx]
    n, dense, val = case.n, case.dense, case.val
    dt = TORCH[dense]
    es = KM.ELEM_BYTES[dense]
    v = KM.FAMILIES[case.family]
    ref, amax = _fwd_ref(G, n, dense, val)
    lens = G.lens
    base_tol = O.fp32_tolerance(ref, amax, lens)
    B = _carve(_host_dense(G.K, n, 1, dense, True), case.misaligned == "B")
    bias = _carve(_host_dense(1, n, 3, dense)[0], case.misaligned == "bias")
    bias_np = bias.float().cpu().numpy().astype(np.float64)[None, :]
    a_val = G.val[val]

    def mirror(C, with_bias, nnz=G.nnz, ldc=None):
        return KM.fwd_launch(v, case.idx, dense, val, n, G.M, nnz, b_mod=_mod(B), c_mod=_mod(C),
                             bias_mod=_mod(bias) if with_bias else None, ldb=n, ldc=ldc)

    def run(out, crow=G.crow, col=G.col, av=a_val, **kw):
        return ops.spmm_csr_compute(crow, col, av, B, G.M, G.K, out=out, variant=v, **kw)

    # plain: the product, then the same into a strided C inside a NaN guard band (static task
    # order), then again (dynamic order): bitwise equal whenever the kernel is the same
    C = _carve(torch.empty(G.M, n, dtype=dt), case.misaligned == "C")
    want = mirror(C, False)
    _launch(lambda: run(C), want, "plain")
    _check(C, ref, base_tol, dense, f"{case.id} plain")
    pad = 16 // es
    off = 1 if case.misaligned == "C" else 0
    Cw = torch.full((G.M + 2, n + 2 * pad + off), float("nan"), dtype=dt, device=DEV)
    Cv = Cw[1:G.M + 1, pad + off:pad + off + n]
    want_g = mirror(Cv, False, ldc=Cw.stride(0))
    _launch(lambda: run(Cv, order="static"), want_g, "strided C")
    if want_g.kernel == want.kernel:
        assert torch.equal(Cv, C), f"{case.id}: strided C / static order changed bits"
    else:
        _check(Cv, ref, base_tol, dense, f"{case.id} strided C")
    guard = torch.ones_like(Cw, dtype=torch.bool)
    guard[1:G.M + 1, pad + off:pad + off + n] = False
    assert bool(torch.isnan(Cw[guard]).all()), f"{case.id}: write outside the rows / columns of C"
    # the repeat must launch the same kernel: an output of the same alignment as C
    C2 = _carve(torch.empty(G.M, n, dtype=dt), case.misaligned == "C")
    assert mirror(C2, False) == want
    _launch(lambda: run(C2), want, "repeat")
    assert torch.equal(C2, C), f"{case.id}: repeated call changed bits"

    # epilogue
    if dense == KM.F32:
        C_old = _host_dense(G.M, n, 4, dense).to(DEV)
        out = C_old.clone() if case.misaligned != "C" else _carve(C_old.cpu(), True)
        _launch(lambda: run(out, accumulate=True, bias=bias, relu=True), mirror(out, True), "acc+bias+relu")
        co = C_old.cpu().numpy().astype(np.float64)
        r = np.maximum(ref + co + bias_np, 0)
        _check(out, r, base_tol + 2.0 ** -22 * (np.abs(co) + np.abs(bias_np)), dense, f"{case.id} acc+bias+relu")
    else:
        # three passes over thirds of the entries, fp32 running sums in between, rounded once
        acc32 = torch.full((G.M, n), float("nan"), dtype=torch.float32, device=DEV)
        out = _carve(torch.full((G.M, n), float("nan"), dtype=dt), case.misaligned == "C")
        for i, (pc, pcol, pval, pnnz) in enumerate(G.parts):
            kw = dict(acc32=acc32, acc32_in=i > 0, acc32_out=i < 2)
            if i == 2:
                kw.update(bias=bias, relu=True)
            _launch(lambda: run(out, crow=pc, col=pcol, av=pval[val], **kw), mirror(out, i == 2, nnz=pnnz),
                    f"acc32 pass {i}")
        r = np.maximum(ref + bias_np, 0)
        _check(out, r, base_tol + 2.0 ** -22 * np.abs(bias_np), dense, f"{case.id} 3 acc32 passes+bias+relu")

    # mean, bias, relu
    out = _carve(torch.empty(G.M, n, dtype=dt), case.misaligned == "C")
    _launch(lambda: run(out, reduce="mean", bias=bias, relu=True), mirror(out, True), "mean")
    d = np.maximum(lens, 1).astype(np.float64)[:, None]
    s = ref / d
    r = np.maximum(s + bias_np, 0)
    tol = base_tol / d + 2.0 ** -22 * np.abs(s) + 2.0 ** -23 * np.abs(r) + 2.0 ** -22 * np.abs(bias_np)
    _check(out, r, tol, dense, f"{case.id} mean+bias+relu")


@pytest.mark.parametrize("dense,val", [(KM.F32, KM.F32), (KM.BF16, KM.BF16), (KM.F32, KM.UNIT)])
@pytest.mark.parametrize("nvec", [8, 16, 32])
def test_whole_row_kernel_under_a_plan(short_graph, dense, val, nvec):
    """A short-row graph: the plan's histogram picks the whole-row kernel (one launch, no task
    partition), which must agree with the oracle."""
    Gs = short_graph
    M, K = Gs.M, Gs.K
    n = nvec * KM.vec_width(dense)
    plan = ops.SpmmPlan(Gs.crow, Gs.col, M, K, n, TORCH[dense])
    assert plan.variant == KM.FAMILIES["rows"], hex(plan.variant)
    want = KM.fwd_launch(plan.variant, KM.I32, dense, val, n, M, Gs.nnz, plan=True)
    assert want.kernel[0] == "spmm_rows_kernel" and want.launches == 1
    B = _host_dense(K, n, 1, dense, True)
    ref, amax = _fwd_ref(Gs, n, dense, val)
    C = _launch(lambda: ops.spmm_csr_compute(Gs.crow, Gs.col, Gs.val[val], B.to(DEV), M, K, plan=plan), want, "plan")
    _check(C, ref, O.fp32_tolerance(ref, amax, Gs.lens), dense, f"whole rows under a plan n={n}")


# ------------------------------------------------------------------ A^T.dY

def _bwd_ref(G, n, dense, val):
    key = ("bwd", id(G.crow_np), n, dense, val)
    if key not in _REF:
        dY = _host_dense(G.M, n, 2, dense).float().numpy()
        v = G.val_f32(val)
        ref = O.spmm_t_f64(G.crow_np, G.col_np, v, dY, G.K)
        amax, cnt = O.spmm_t_absmax(G.crow_np, G.col_np, v, dY, G.K)
        _REF[key] = (ref, O.fp32_tolerance(ref, amax, cnt))
    return _REF[key]


@pytest.mark.parametrize("case", KM.atomic_cases(), ids=lambda c: c.id)
def test_atomic_grad_b(graphs, case):
    G = graphs[case.idx]
    ref, tol = _bwd_ref(G, case.n, case.dense, case.val)
    dY = _carve(_host_dense(G.M, case.n, 2, case.dense), case.misaligned == "dY")
    out = torch.empty(G.K, case.n, dtype=TORCH[case.dense], device=DEV)
    want = KM.atomic_launch(case.idx, case.dense, case.val, case.n, G.M, G.nnz, dy_mod=_mod(dY), out_mod=_mod(out))
    _launch(lambda: ops.spmm_csr_grad_b_compute(G.crow, G.col, G.val[case.val], dY, G.M, G.K, out=out, atomic=True),
            want, case.id)
    _check(out, ref, tol, case.dense, case.id)


@pytest.mark.parametrize("route", ["transient", "transposed", "cached"])
@pytest.mark.parametrize("idx", [KM.I32, KM.I64])
@pytest.mark.parametrize("n", [72, 520])
def test_grad_b_bf16_values_deterministic_routes(graphs, route, idx, n):
    """bf16-valued A on the routes that run the forward kernel on A^T."""
    G = graphs[idx]
    ref, tol = _bwd_ref(G, n, KM.BF16, KM.BF16)
    dY = _host_dense(G.M, n, 2, KM.BF16).to(DEV)
    a_val = G.val[KM.BF16]
    if route == "transient":
        got = ops.spmm_csr_grad_b_compute(G.crow, G.col, a_val, dY, G.M, G.K)
    elif route == "transposed":
        tr = ops.csr_transpose(G.crow, G.col, a_val, G.M, G.K)
        got = ops.spmm_csr_grad_b_compute(G.crow, G.col, a_val, dY, G.M, G.K, transposed=tr)
    else:
        plan = ops.SpmmPlan(G.crow, G.col, G.M, G.K, n, torch.bfloat16, transpose=True)
        got = ops.spmm_csr_grad_b_compute(G.crow, G.col, a_val, dY, G.M, G.K, plan=plan)
        again = ops.spmm_csr_grad_b_compute(G.crow, G.col, a_val, dY, G.M, G.K, plan=plan, regather=True)
        assert torch.equal(got, again)
    _check(got, ref, tol, KM.BF16, f"grad_b {route} bf16 values n={n}")


# ------------------------------------------------------------------ SDDMM

@pytest.mark.parametrize("case", KM.sddmm_cases(), ids=lambda c: c.id)
def test_sddmm(graphs, case):
    G = graphs[case.idx]
    n, dense = case.n, case.dense
    key = ("sddmm", id(G.crow_np), n, dense)
    if key not in _REF:
        r, aabs = O.sddmm_f64(G.crow_np, G.col_np, _host_dense(G.M, n, 2, dense).float().numpy(),
                              _host_dense(G.K, n, 1, dense, True).float().numpy())
        _REF[key] = (r, 1e-5 * np.abs(r) + 2.0 ** -23 * n * aabs)
    ref, tol = _REF[key]
    dY = _carve(_host_dense(G.M, n, 2, dense), case.misaligned == "dY")
    B = _carve(_host_dense(G.K, n, 1, dense, True), case.misaligned == "B")
    want = KM.sddmm_launch(case.idx, dense, case.val, n, G.M, G.nnz, b_mod=_mod(B), dy_mod=_mod(dY))
    got = _launch(lambda: ops.sddmm_csr_compute(G.crow, G.col, dY, B, G.M, G.K, val_dtype=TORCH[case.val]), want, case.id)
    _check(got, ref, tol, case.val, case.id)
    assert torch.equal(got, ops.sddmm_csr_compute(G.crow, G.col, dY, B, G.M, G.K, val_dtype=TORCH[case.val]))


# ------------------------------------------------------------------ kernel names

def _profiled_key(name: str):
    """KM.parse_demangled of a kernel name as torch.profiler reports it.  Demanglers differ in how
    they spell template values (`(int)8`, `(bool)1` against c++filt's `8`, `true`), and a name that
    arrives mangled is demangled with c++filt."""
    if name.startswith("_Z"):
        name = subprocess.run(["c++filt"], input=name, capture_output=True, text=True, check=True).stdout.strip()
    name = re.sub(r"\(bool\)([01])", lambda m: "true" if m.group(1) == "1" else "false", name)
    name = re.sub(r"\((?:int|unsigned int|long|unsigned long)\)(-?\d+)", r"\1", name)
    return KM.parse_demangled(name)


def _run_case(G, case):
    """The calls case_kernels accounts for, on operands of the case's alignment: the forward plain,
    with a bias and as a mean with a bias; the SDDMM; the atomic A^T.dY."""
    n, dense, val = case.n, case.dense, case.val
    dt = TORCH[dense]
    if case.op == "fwd":
        B = _carve(_host_dense(G.K, n, 1, dense, True), case.misaligned == "B")
        bias = _carve(_host_dense(1, n, 3, dense)[0], case.misaligned == "bias")
        v = KM.FAMILIES[case.family]
        for kw in ({}, dict(bias=bias, relu=True), dict(bias=bias, relu=True, reduce="mean")):
            C = _carve(torch.empty(G.M, n, dtype=dt), case.misaligned == "C")
            ops.spmm_csr_compute(G.crow, G.col, G.val[val], B, G.M, G.K, out=C, variant=v, **kw)
    elif case.op == "sddmm":
        dY = _carve(_host_dense(G.M, n, 2, dense), case.misaligned == "dY")
        B = _carve(_host_dense(G.K, n, 1, dense, True), case.misaligned == "B")
        ops.sddmm_csr_compute(G.crow, G.col, dY, B, G.M, G.K, val_dtype=TORCH[val])
    else:
        dY = _carve(_host_dense(G.M, n, 2, dense), case.misaligned == "dY")
        out = torch.empty(G.K, n, dtype=dt, device=DEV)
        ops.spmm_csr_grad_b_compute(G.crow, G.col, G.val[val], dY, G.M, G.K, out=out, atomic=True)


@pytest.mark.parametrize("case", list(KM.all_cases()), ids=lambda c: c.id)
def test_launched_kernel_names(graphs, case):
    """The kernels a case launches, by demangled name, are the ones the mirror predicts: a width
    that moves to another lane layout keeps the launch count and the result, but not the name."""
    G = graphs[case.idx]
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        _run_case(G, case)
        torch.cuda.synchronize()
    names = {e.name for e in prof.events()} | {k.name for e in prof.events() for k in getattr(e, "kernels", ())}
    got = {k for k in map(_profiled_key, names) if k is not None}
    want = KM.case_kernels(case, G.M, G.nnz)
    assert got == want, f"{case.id}: launched {sorted(map(KM.demangled, got))}, predicted {sorted(map(KM.demangled, want))}"
