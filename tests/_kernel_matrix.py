"""Which kernel instantiation a call launches: a pure-Python mirror of the dispatch code, and the
case matrix that reaches every instantiation.  Not a test module; imported by
tests/test_kernel_matrix_host.py (mirror against the library's variant names and against the
instantiations in the built library) and tests/test_gpu_kernel_matrix.py (every case against the
fp64 oracle).

Mirrored code:
  * lane layouts: internal.h (lane_layout, one ladder per LaneOp) and the layouts each launcher
    instantiates (dispatch_lanes in fwd_launch.cuh:launch_typed, fwd_rows.cu, sddmm.cu:launch_typed,
    bwd.cu:launch_typed);
  * type dispatch: launch.cuh (dispatch_dtypes, dispatch_index) as each launcher calls it;
  * forward: fwd.cu (resolve_variant, vec_rows_ok, rows_layout, launch_fwd), fwd_launch.cuh
    (launch_family, launch_typed, launch_full) and fwd_rows.cu (launch_family_rows);
  * SDDMM: sddmm.cu (launch_sddmm, launch_typed);
  * atomic A^T.dY: bwd.cu (launch_bwd_atomic, launch_typed, launch_one).

A kernel key is the demangled template argument list of the kernel the call launches, e.g.
("spmm_merge_kernel", "float", "float", "int", 4, 8, 1, True, False, 256, 4, "int2"): the same
spelling as `cuobjdump -sass` + `c++filt` give for the library, so a key can be looked up there.
Only narrow task partitions (int2 entries, nnz < 2^31 - 1) are mirrored: the wide (longlong2)
instantiations are exercised by tests/test_gpu_wide_nnz.py.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Iterator, Optional, Tuple

# public codes (include/ofspmm.h)
F32, BF16, I32, I64, UNIT = 2, 11, 5, 6, 0x100
VARIANT_ITEMS64, VARIANT_ROWPAR, VARIANT_ROWS, VARIANT_EXPLICIT = 1, 2, 4, 0x100

TASK_ITEMS, SMALL_TASK_ITEMS, WARPS = 256, 64, 4
SMALL_PROBLEM_TASKS = 148 * 36

FAMILIES = {
    "base": VARIANT_EXPLICIT,
    "items64": VARIANT_EXPLICIT | VARIANT_ITEMS64,
    "rowpar": VARIANT_EXPLICIT | VARIANT_ROWPAR,
    "rows": VARIANT_EXPLICIT | VARIANT_ROWS,
}
# (dense dtype, value dtype) pairs the libraries instantiate; SDDMM has no pattern matrices (its
# value dtype is the dtype of the dval output)
DTYPE_PAIRS = ((F32, F32), (BF16, F32), (BF16, BF16), (F32, UNIT), (BF16, UNIT))
SDDMM_DTYPE_PAIRS = ((F32, F32), (BF16, F32), (BF16, BF16))

CXX_DENSE = {F32: "float", BF16: "__nv_bfloat16"}
CXX_VAL = {F32: "float", BF16: "__nv_bfloat16", UNIT: "ofspmm::UnitVal"}
CXX_IDX = {I32: "int", I64: "long"}
ELEM_BYTES = {F32: 4, BF16: 2}

# the kernel templates the mirror accounts for, and the ones it leaves to other tests
KERNELS = ("spmm_merge_kernel", "spmm_fixup_kernel", "spmm_rows_kernel", "sddmm_merge_kernel",
           "sddmm_wide_kernel", "bwd_atomic_kernel")
WIDE_PARTITION = "longlong2"   # int64 matrices with >= 2^31 - 1 non-zeros: tests/test_gpu_wide_nnz.py


def num_tasks(rows: int, nnz: int, items: int) -> int:
    return (rows + nnz + items - 1) // items


def vec_width(dense: int) -> int:
    return 16 // ELEM_BYTES[dense]


def _rowpar_supported(n: int, dense: int) -> bool:
    v = vec_width(dense)
    return n % v == 0 and n // v <= 16


def _rows_supported(n: int, dense: int) -> bool:
    v = vec_width(dense)
    return n > 0 and n % v == 0 and n // v <= 32


def resolve_variant(variant: int, rows: int, nnz: int, n: int, dense: int) -> Tuple[int, bool, bool]:
    """fwd.cu:resolve_variant (narrow matrices) -> (items, whole_rows, row_parallel)."""
    if variant & VARIANT_EXPLICIT:
        if variant & VARIANT_ROWS:
            return SMALL_TASK_ITEMS, _rows_supported(n, dense), False
        if variant & VARIANT_ITEMS64:
            return SMALL_TASK_ITEMS, False, False
        if variant & VARIANT_ROWPAR and _rowpar_supported(n, dense):
            return TASK_ITEMS, False, True
        return TASK_ITEMS, False, False
    if num_tasks(rows, nnz, TASK_ITEMS) < SMALL_PROBLEM_TASKS:
        return SMALL_TASK_ITEMS, False, False
    return TASK_ITEMS, False, False


@dataclass(frozen=True)
class Launch:
    """What one call launches: `kernel` (its key), the column `panels` of its grid, the task count
    `tasks` of its partition (0 for the whole-row kernel), the `fixup` kernel key (forward with more
    than one task) and `launches`, the number ofspmm_launch_count() advances by."""
    kernel: tuple
    panels: int
    tasks: int
    fixup: Optional[tuple]
    launches: int


def _layout(n: int, aligned: bool, dense: int, ladder: tuple, scalar: tuple):
    """Shared shape of the launch_typed functions: (VEC, LPR, CH, panel columns) from the dense
    width.  `ladder` lists (max 16-byte vectors, LPR, CH) of the vector layouts, the last entry
    taking every wider row (max None); `scalar` the same for scalar lanes, in elements."""
    v = vec_width(dense)
    if aligned and n % v == 0:
        nvec = n // v
        for top, lpr, ch in ladder:
            if top is None or nvec <= top:
                return v, lpr, ch
    for top, lpr, ch in scalar:
        if top is None or n <= top:
            return 1, lpr, ch
    raise AssertionError("unreachable")


def _misaligned(*addr_mods: Optional[int]) -> bool:
    return any(m is not None and m % 16 for m in addr_mods)


FWD_LADDER = ((8, 8, 1), (16, 16, 1), (32, 32, 1), (64, 32, 2), (None, 32, 4))
FWD_SCALAR = ((32, 32, 1), (64, 32, 2), (128, 32, 4), (None, 32, 8))


def fwd_launch(variant: int, idx: int, dense: int, val: int, n: int, rows: int, nnz: int, *,
               b_mod: int = 0, c_mod: int = 0, bias_mod: Optional[int] = None,
               ldb: Optional[int] = None, ldc: Optional[int] = None, plan: bool = False) -> Launch:
    """Forward C = A.B (ofspmm_fwd_ex).  `*_mod` are the operand addresses modulo 16 (bias_mod None:
    no bias flag); `plan`: a task partition is passed in (no partition launch)."""
    ldb = n if ldb is None else ldb
    ldc = n if ldc is None else ldc
    v = vec_width(dense)
    items, whole, rowpar = resolve_variant(variant, rows, nnz, n, dense)
    aligned = not _misaligned(b_mod, c_mod, bias_mod)
    vec_rows = aligned and n % v == 0 and ldb % v == 0 and ldc % v == 0
    D, V, I = CXX_DENSE[dense], CXX_VAL[val], CXX_IDX[idx]
    if whole and idx == I32 and vec_rows and _rows_supported(n, dense):
        nvec = n // v
        lpr = 8 if nvec <= 8 else (16 if nvec <= 16 else 32)
        return Launch(("spmm_rows_kernel", D, V, v, lpr), 1, 0, None, 1)
    rowpar = rowpar and items == TASK_ITEMS and vec_rows
    if rowpar:
        VEC, LPR, CH = _layout(n, True, dense, ((8, 8, 1), (16, 16, 1)), ())
    else:
        VEC, LPR, CH = _layout(n, vec_rows, dense, FWD_LADDER, FWD_SCALAR)
    panels = 1
    if CH == 4 and VEC > 1:
        panels = (n // v + 127) // 128
    elif CH == 8:
        panels = (n + 255) // 256
    full = n % (LPR * VEC * CH) == 0
    P = num_tasks(rows, nnz, items)
    kernel = ("spmm_merge_kernel", D, V, I, VEC, LPR, CH, full, rowpar, items, WARPS, "int2")
    fixup = ("spmm_fixup_kernel", D, I, VEC, WARPS, "int2") if P > 1 else None
    return Launch(kernel, panels, P, fixup, (0 if plan else 1) + 1 + (fixup is not None))


def sddmm_launch(idx: int, dense: int, val: int, n: int, rows: int, nnz: int, *,
                 b_mod: int = 0, dy_mod: int = 0, plan: bool = False) -> Launch:
    """dval = SDDMM(dY, B) (ofspmm_sddmm_ex); `val` is the dtype of dval."""
    VEC, LPR, CH = _layout(n, not _misaligned(b_mod, dy_mod), dense,
                           ((8, 8, 1), (16, 16, 1), (32, 32, 1), (64, 32, 2), (128, 32, 4), (None, 0, 0)),
                           ((32, 32, 1), (128, 32, 4), (None, 0, 0)))
    D, V, I = CXX_DENSE[dense], CXX_VAL[val], CXX_IDX[idx]
    P = num_tasks(rows, nnz, TASK_ITEMS)
    if LPR == 0:
        kernel = ("sddmm_wide_kernel", D, V, I, VEC, TASK_ITEMS, WARPS, "int2")
    else:
        kernel = ("sddmm_merge_kernel", D, V, I, VEC, LPR, CH, n % (LPR * VEC * CH) == 0, TASK_ITEMS, WARPS, "int2")
    return Launch(kernel, 1, P, None, (0 if plan else 1) + 1)


def atomic_launch(idx: int, dense: int, val: int, n: int, rows: int, nnz: int, *, dy_mod: int = 0,
                  out_mod: int = 0) -> Launch:
    """dB = A^T.dY through the atomic scatter (ofspmm_bwd_b without A^T).  fp32 accumulates in dB
    itself (`out_mod`), bf16 in an aligned workspace and is cast once afterwards (one more launch)."""
    acc_mod = out_mod if dense == F32 else 0
    VEC, LPR, CH = _layout(n, not _misaligned(dy_mod, acc_mod), dense, FWD_LADDER, ((32, 32, 1), (128, 32, 4), (None, 32, 8)))
    panels = 1
    if CH == 4 and VEC > 1:
        panels = (n // VEC + 127) // 128
    elif CH == 8:
        panels = (n + 255) // 256
    D, V, I = CXX_DENSE[dense], CXX_VAL[val], CXX_IDX[idx]
    kernel = ("bwd_atomic_kernel", D, V, I, VEC, LPR, CH, TASK_ITEMS, WARPS, "int2")
    return Launch(kernel, panels, num_tasks(rows, nnz, TASK_ITEMS), None, 2 + (dense != F32))


LAYOUT_NAMES = {
    (8, 1): "vector-per-row(8 lanes x 16B, 4 nnz per step)",
    (16, 1): "vector-per-row(16 lanes x 16B, 2 nnz per step)",
    (32, 1): "warp-per-row(32 lanes x 16B)",
    (32, 2): "warp-per-row(32 lanes x 2 x 16B)",
    (32, 4): "warp-per-row(32 lanes x 4 x 16B, column panels)",
}


def variant_name(launch: Launch) -> str:
    """The `<schedule family>/<lane layout>` string ofspmm_variant_name reports for a forward key."""
    k = launch.kernel
    if k[0] == "spmm_rows_kernel":
        return f"whole_rows(one launch, no merge path)/group-per-row({k[4]} lanes x 16B, 4 gathers in flight)"
    _, _, _, _, vec, lpr, ch, _, rowpar, items, _, _ = k
    fam = ("merge_path(64-item tasks)" if items == SMALL_TASK_ITEMS else
           "merge_path(256-item tasks, row-parallel groups)" if rowpar else "merge_path(256-item tasks)")
    layout = "warp-per-row(scalar lanes, unaligned n)" if vec == 1 else LAYOUT_NAMES[(lpr, ch)]
    return f"{fam}/{layout}"


def demangled(key: tuple) -> str:
    """`void ofspmm::name<args>` as c++filt spells the kernel."""
    args = ", ".join(("true" if a else "false") if isinstance(a, bool) else str(a) for a in key[1:])
    return f"void ofspmm::{key[0]}<{args}>"


def parse_demangled(name: str) -> Optional[tuple]:
    """Inverse of `demangled` for the kernels in KERNELS (None for any other function)."""
    name = name.split("(")[0].strip()
    if name.startswith("void "):
        name = name[5:]
    if not name.startswith("ofspmm::") or "<" not in name:
        return None
    base, args = name[len("ofspmm::"):].split("<", 1)
    if base not in KERNELS:
        return None
    out = []
    for a in args.rstrip(">").split(","):
        a = a.strip()
        out.append(True if a == "true" else False if a == "false" else int(a) if a.lstrip("-").isdigit() else a)
    return (base, *out)


# ------------------------------------------------------------------ the case matrix

FP32_WIDTHS = (4, 20, 32, 36, 64, 100, 128, 132, 256, 260, 512, 640, 1024, 1028)
BF16_WIDTHS = (8, 40, 64, 72, 128, 200, 256, 264, 512, 520, 1024, 1032, 1280, 2048, 2056)
ODD_WIDTHS = (3, 33, 65, 129, 257, 513)
# scalar lanes with no masked lane (n a multiple of the scalar tile) happen only through a
# misaligned pointer: these widths are also run with one operand carved one element off
MISALIGNED_WIDTHS = (32, 64, 128, 256, 512)
FWD_MISALIGNED = ("B", "C", "bias")
SDDMM_MISALIGNED = ("B", "dY")


@dataclass(frozen=True)
class Case:
    op: str                 # "fwd" | "sddmm" | "atomic"
    family: str             # FAMILIES key ("-" for sddmm / atomic)
    idx: int
    dense: int
    val: int
    n: int
    misaligned: str = ""    # which operand is carved one element off ("" none)

    @property
    def id(self) -> str:
        dt = {F32: "f32", BF16: "bf16", UNIT: "unit"}
        s = f"{self.op}-{self.family}-{'i32' if self.idx == I32 else 'i64'}-{dt[self.dense]}-{dt[self.val]}-n{self.n}"
        return s + (f"-mis{self.misaligned}" if self.misaligned else "")


def _widths(dense: int):
    for n in (FP32_WIDTHS if dense == F32 else BF16_WIDTHS) + ODD_WIDTHS:
        yield n, ""


def fwd_case_launches(c: Case, rows: int, nnz: int):
    """Every launch the forward modes of one case make: (mode, Launch).  Modes: "plain" (also run
    with a strided, guard-banded C), "epilogue" (bias, plus ReLU and accumulate or the acc32 passes)
    and "mean" (with bias and ReLU).  The misaligned operand is the bias only where a bias is used."""
    b_mod = ELEM_BYTES[c.dense] if c.misaligned == "B" else 0
    c_mod = ELEM_BYTES[c.dense] if c.misaligned == "C" else 0
    bias_mod = ELEM_BYTES[c.dense] if c.misaligned == "bias" else 0
    v = FAMILIES[c.family]
    out = []
    for mode in ("plain", "epilogue", "mean"):
        bm = None if mode == "plain" else bias_mod
        out.append((mode, fwd_launch(v, c.idx, c.dense, c.val, c.n, rows, nnz, b_mod=b_mod, c_mod=c_mod, bias_mod=bm)))
    return out


def _select(cases_keys):
    """Keep a case when it reaches a (key, several panels) pair no earlier case of its group did."""
    seen, keep = set(), []
    for case, keys in cases_keys:
        new = {k for k in keys if k not in seen}
        if new:
            keep.append(case)
            seen |= new
    return keep


# a representative size for the case selection: several tasks, so every forward call stitches
SEL_ROWS, SEL_NNZ = 4000, 60000


def fwd_cases() -> list:
    """Per (index dtype, dtype pair), the families in FAMILIES order share one selection, so the
    row-parallel and whole-row families contribute their own kernels plus one width each that
    falls back to another family (row-parallel: a warp-wide row; whole-row: int64 indices or a row
    wider than 32 vectors)."""
    out = []
    for idx in (I32, I64):
        for dense, val in DTYPE_PAIRS:
            seen = set()
            for family in FAMILIES:
                cand = [Case("fwd", family, idx, dense, val, n) for n, _ in _widths(dense)]
                cand += [Case("fwd", family, idx, dense, val, n, FWD_MISALIGNED[i % 3])
                         for i, n in enumerate(MISALIGNED_WIDTHS)]
                for c in cand:
                    ks = {(L.kernel, L.panels > 1) for _, L in fwd_case_launches(c, SEL_ROWS, SEL_NNZ)}
                    if ks - seen:
                        out.append(c)
                        seen |= ks
                if family in ("rowpar", "rows"):
                    out.append(Case("fwd", family, idx, dense, val, 40 * vec_width(dense)))
    return out


def sddmm_cases() -> list:
    out = []
    for idx in (I32, I64):
        for dense, val in SDDMM_DTYPE_PAIRS:
            cand = [Case("sddmm", "-", idx, dense, val, n) for n, _ in _widths(dense)]
            cand += [Case("sddmm", "-", idx, dense, val, n, SDDMM_MISALIGNED[i % 2])
                     for i, n in enumerate(MISALIGNED_WIDTHS + (1024,))]
            out += _select([(c, {(sddmm_case_launch(c, SEL_ROWS, SEL_NNZ).kernel, False)}) for c in cand])
    return out


def sddmm_case_launch(c: Case, rows: int, nnz: int) -> Launch:
    es = ELEM_BYTES[c.dense]
    return sddmm_launch(c.idx, c.dense, c.val, c.n, rows, nnz, b_mod=es if c.misaligned == "B" else 0,
                        dy_mod=es if c.misaligned == "dY" else 0)


def atomic_cases() -> list:
    out = []
    for idx in (I32, I64):
        for dense, val in DTYPE_PAIRS:
            cand = [Case("atomic", "-", idx, dense, val, n) for n, _ in _widths(dense)]
            cand += [Case("atomic", "-", idx, dense, val, n, "dY") for n in MISALIGNED_WIDTHS]
            keyed = []
            for c in cand:
                L = atomic_case_launch(c, SEL_ROWS, SEL_NNZ)
                keyed.append((c, {(L.kernel, L.panels > 1)}))
            out += _select(keyed)
    return out


def atomic_case_launch(c: Case, rows: int, nnz: int) -> Launch:
    return atomic_launch(c.idx, c.dense, c.val, c.n, rows, nnz,
                         dy_mod=ELEM_BYTES[c.dense] if c.misaligned == "dY" else 0)


def all_cases() -> Iterator[Case]:
    yield from fwd_cases()
    yield from sddmm_cases()
    yield from atomic_cases()


def case_kernels(c: Case, rows: int = SEL_ROWS, nnz: int = SEL_NNZ) -> set:
    """Every kernel key a case launches (the fix-up kernel included)."""
    if c.op == "fwd":
        ks = set()
        for _, L in fwd_case_launches(c, rows, nnz):
            ks.add(L.kernel)
            if L.fixup:
                ks.add(L.fixup)
        return ks
    if c.op == "sddmm":
        return {sddmm_case_launch(c, rows, nnz).kernel}
    return {atomic_case_launch(c, rows, nnz).kernel}
