"""CPU checks of the dispatch mirror in tests/_kernel_matrix.py, against the built library:

  * the forward key the mirror predicts names the same schedule family and lane layout as
    ofspmm_variant_name() (int32 indices, 16-byte aligned operands: the cases the name describes);
  * the case matrix of tests/test_gpu_kernel_matrix.py launches every instantiation of the merge,
    fix-up, whole-row, SDDMM and atomic-scatter kernels in libofspmm_b200.so (except the wide-nnz
    ones, listed by name), and no case maps to a kernel the library does not have.

A template axis added to a kernel without a case that reaches it fails the second check."""
import os
import re
import shutil
import subprocess
import sys

import pytest

import ofspmm_b200 as ofs

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import _kernel_matrix as KM  # noqa: E402

_lib = ofs._lib


def _tool(name):
    for d in (os.environ.get("CUDA_HOME"), os.environ.get("CUDA_PATH"), "/usr/local/cuda"):
        if d and os.path.exists(os.path.join(d, "bin", name)):
            return os.path.join(d, "bin", name)
    return shutil.which(name)


@pytest.fixture(scope="module")
def L():
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("libofspmm_b200.so not built (make -C of-spmm_b200/csrc)")
    return _lib.lib()


@pytest.fixture(scope="module")
def instantiations(L):
    """Demangled names of the kernels of KM.KERNELS in the library (each once; a kernel compiled in
    several translation units appears once per unit in the SASS)."""
    cuobjdump, cxxfilt = _tool("cuobjdump"), shutil.which("c++filt")
    if cuobjdump is None or cxxfilt is None:
        pytest.skip("needs cuobjdump (CUDA toolkit) and c++filt")
    sass = subprocess.run([cuobjdump, "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    mangled = sorted(set(re.findall(r"Function : (\S+)", sass)))
    names = subprocess.run([cxxfilt], input="\n".join(mangled), capture_output=True, text=True, check=True).stdout
    keys = {}
    for d in names.splitlines():
        k = KM.parse_demangled(d)
        if k is not None:
            keys[k] = d
    return keys


def test_mirror_agrees_with_variant_name(L):
    """Every aligned int32 forward case: the mirror's family and layout == ofspmm_variant_name()."""
    checked = 0
    for c in KM.fwd_cases():
        if c.idx != KM.I32 or c.misaligned:
            continue
        v = KM.FAMILIES[c.family]
        want = KM.variant_name(KM.fwd_launch(v, c.idx, c.dense, c.val, c.n, KM.SEL_ROWS, KM.SEL_NNZ))
        got = L.ofspmm_variant_name(v, KM.SEL_ROWS, KM.SEL_NNZ, c.n, c.dense).decode()
        assert got == want, (c.id, got, want)
        checked += 1
    # AUTO without a histogram: the 64-item family below one task per resident warp
    for rows, nnz in ((4000, 60000), (1 << 20, 1 << 24)):
        for n in (64, 260):
            want = KM.variant_name(KM.fwd_launch(0, KM.I32, KM.F32, KM.F32, n, rows, nnz))
            assert L.ofspmm_variant_name(0, rows, nnz, n, KM.F32).decode() == want
    assert checked > 100


def test_mirror_details():
    """Spot checks of dispatch rules the variant name cannot show."""
    X, R = KM.VARIANT_EXPLICIT, KM.VARIANT_EXPLICIT | KM.VARIANT_ROWS
    rows, nnz = 4000, 60000
    # the whole-row kernel needs int32 indices and aligned operands; otherwise 64-item tasks
    assert KM.fwd_launch(R, KM.I32, KM.F32, KM.F32, 64, rows, nnz).kernel[0] == "spmm_rows_kernel"
    assert KM.fwd_launch(R, KM.I32, KM.F32, KM.F32, 64, rows, nnz).launches == 1
    for kw in (dict(idx=KM.I64), dict(b_mod=4), dict(bias_mod=8), dict(ldc=66)):
        idx = kw.pop("idx", KM.I32)
        Lc = KM.fwd_launch(R, idx, KM.F32, KM.F32, 64, rows, nnz, **kw)
        assert Lc.kernel[0] == "spmm_merge_kernel" and Lc.kernel[9] == 64 and Lc.launches == 3, kw
    # a misaligned bias matters only when the bias flag is set
    assert KM.fwd_launch(X, KM.I32, KM.F32, KM.F32, 64, rows, nnz, bias_mod=4).kernel[4] == 1
    assert KM.fwd_launch(X, KM.I32, KM.F32, KM.F32, 64, rows, nnz, bias_mod=None).kernel[4] == 4
    # column panels: 128 vectors per panel, 256 scalar columns per panel
    assert KM.fwd_launch(X, KM.I32, KM.F32, KM.F32, 1028, rows, nnz).panels == 3
    assert KM.fwd_launch(X, KM.I32, KM.BF16, KM.BF16, 1032, rows, nnz).panels == 2
    assert KM.fwd_launch(X, KM.I32, KM.F32, KM.F32, 513, rows, nnz).panels == 3
    assert KM.atomic_launch(KM.I32, KM.F32, KM.F32, 640, rows, nnz).panels == 2
    # one task: no fix-up launch
    assert KM.fwd_launch(X, KM.I32, KM.F32, KM.F32, 64, 10, 100).fixup is None


def test_cases_reach_every_kernel(instantiations):
    have = set(instantiations)
    narrow = {k for k in have if KM.WIDE_PARTITION not in k}
    wide = {k for k in have if KM.WIDE_PARTITION in k}
    # the wide-nnz instantiations are left to tests/test_gpu_wide_nnz.py: exactly these templates
    assert {k[0] for k in wide} == {"spmm_merge_kernel", "spmm_fixup_kernel", "sddmm_merge_kernel",
                                    "sddmm_wide_kernel", "bwd_atomic_kernel"}
    assert all(k[3] == "long" or k[0] == "spmm_fixup_kernel" and k[2] == "long" for k in wide)
    reached = set()
    for c in KM.all_cases():
        reached |= KM.case_kernels(c)
    missing = sorted(KM.demangled(k) for k in narrow - reached)
    phantom = sorted(KM.demangled(k) for k in reached - have)
    assert not phantom, f"cases map to {len(phantom)} kernels the library does not have: {phantom[:5]}"
    assert not missing, f"{len(missing)} kernel instantiations no case launches: {missing[:10]}"
    for name in KM.KERNELS:
        assert any(k[0] == name for k in narrow), f"no instantiation of {name} found in the library"
    # the parser reads back exactly the names c++filt printed
    for k, d in instantiations.items():
        assert KM.demangled(k) == d.split("(")[0].strip(), d


def test_task_boundary_graph_shapes():
    """The GPU matrix graphs have rows that end and rows that start exactly on 64- and 256-item
    task boundaries, empty first / last rows, runs of empty rows and hub rows over 5 tasks; checked
    with the library's host merge-path partition (so this also runs without a GPU)."""
    import torch
    import test_gpu_kernel_matrix as G
    ops = __import__("importlib").import_module("of-spmm_b200.ops")
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("libofspmm_b200.so not built")
    for make in (G.matrix_graph, G.short_row_graph):
        crow, col, val, M, K = make()
        G.check_graph_shape(torch.from_numpy(crow), ops, strict=make is G.matrix_graph)
