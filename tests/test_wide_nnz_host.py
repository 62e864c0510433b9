"""CPU tests of CSR matrices with 2^31-1 or more non-zeros ("wide", int64 indices): the workspace
and plan queries switch to 16-byte task partition entries exactly at the threshold and keep their
old values below it, the transpose scratch only shrank, the size limits that remain still return
OFSPMM_ERR_TOO_LARGE, and a wide int64 call now gets past validation (to the workspace check)."""
import ctypes
from importlib import import_module

import pytest

_lib = import_module("of-spmm_b200._lib")

F32, BF16, I32, I64 = _lib.DTYPE_FLOAT, _lib.DTYPE_BFLOAT16, _lib.DTYPE_INT32, _lib.DTYPE_INT64
OK, INVALID, WORKSPACE, TOO_LARGE = 0, 1, 3, 5
WIDE = 2 ** 31 - 1          # first nnz with 64-bit task offsets
M, K, N = 2 ** 21, 2 ** 20, 128
FAKE = 1 << 20              # never dereferenced: every call below stops before touching memory


def _al(x):
    return (x + 255) // 256 * 256


def _tasks(rows, nnz, items=256):
    return -(-(rows + nnz) // items)


def _entry(nnz):
    return 16 if nnz >= WIDE else 8


def _plan(rows, nnz, items=256):
    return _al((_tasks(rows, nnz, items) + 1) * _entry(nnz))


def _fwd(rows, nnz, n, dd):
    """Forward workspace of the AUTO variant: 64-item tasks when 256-item tasks cannot fill the
    GPU (148 SMs x 36 warps), never for wide matrices."""
    items = 64 if _tasks(rows, nnz) < 148 * 36 and nnz < WIDE else 256
    P = _tasks(rows, nnz, items)
    rowbuf = _al(P * n * 4)
    return 256 + _plan(rows, nnz, items) + rowbuf + (rowbuf if dd == BF16 else 0)


@pytest.mark.parametrize("nnz", [WIDE - 2, WIDE - 1, WIDE, 2 ** 31, 2 ** 31 + 2 ** 25, 2 ** 33])
@pytest.mark.parametrize("dd", [F32, BF16])
def test_queries_use_16_byte_entries_from_the_threshold_on(nnz, dd):
    L = _lib.lib()
    assert L.ofspmm_plan_bytes(M, nnz, N, dd, _lib.VARIANT_AUTO) == _plan(M, nnz)
    assert L.ofspmm_fwd_workspace_bytes(M, K, nnz, N, dd) == _fwd(M, nnz, N, dd)
    assert L.ofspmm_fwd_ex_workspace_bytes(M, K, nnz, N, dd, _lib.VARIANT_AUTO) == _fwd(M, nnz, N, dd)
    assert L.ofspmm_sddmm_workspace_bytes(M, K, nnz, N, dd) == 256 + _plan(M, nnz)
    vs = 4 if dd == F32 else 2
    assert L.ofspmm_bwd_b_cached_workspace_bytes(M, K, nnz, N, dd, F32 if dd == F32 else BF16) == \
        _al(nnz * vs) + _fwd(K, nnz, N, dd)
    atomic = _plan(M, nnz) + (0 if dd == F32 else _al(K * N * 4))
    assert L.ofspmm_bwd_b_workspace_bytes(M, K, nnz, N, dd, 0) == atomic
    assert L.ofspmm_bwd_b_workspace_bytes(M, K, nnz, N, dd, 1) == _fwd(K, nnz, N, dd)


@pytest.mark.parametrize("variant", [_lib.VARIANT_EXPLICIT | _lib.VARIANT_ROWS, _lib.VARIANT_EXPLICIT | _lib.VARIANT_ITEMS64])
def test_wide_matrices_fall_back_to_256_item_tasks(variant):
    """The whole-row kernel and 64-item tasks never serve a wide matrix: an explicit code for them
    is sized and named like the base family; below the threshold nothing changes."""
    L = _lib.lib()
    assert L.ofspmm_plan_bytes(M, WIDE, N, F32, variant) == _plan(M, WIDE)
    assert L.ofspmm_variant_name(variant, M, WIDE, N, F32).startswith(b"merge_path(256-item tasks)")
    below = L.ofspmm_plan_bytes(M, WIDE - 1, N, F32, variant)
    assert below == _al((_tasks(M, WIDE - 1, 64) + 1) * 8)
    rowpar = _lib.VARIANT_EXPLICIT | _lib.VARIANT_ROWPAR
    assert b"row-parallel" in L.ofspmm_variant_name(rowpar, M, WIDE, 32, F32)


@pytest.mark.parametrize("nnz", [0, 1000, 10 ** 6, 10 ** 8, 2 ** 31 + 2 ** 25])
@pytest.mark.parametrize("idx,cols", [(I32, K), (I64, K), (I64, 2 ** 33)])
def test_transpose_and_transient_workspace_only_shrank(nnz, idx, cols):
    """The transpose used to take four nnz-long index arrays plus the sort's own nnz-long buffers;
    it now takes at most one index array, two key arrays and the sort's small scratch."""
    L = _lib.lib()
    isz = 8 if idx == I64 else 4
    old_floor = 4 * _al(max(nnz, 1) * isz)          # lower bound of the former query
    t = L.ofspmm_csr_transpose_workspace_bytes(M, cols, nnz, idx)
    assert 0 < t < old_floor
    if nnz >= 10 ** 8:   # 32-bit keys whenever the column sentinel fits
        key = 4 if cols < WIDE else 8
        assert t >= _al(nnz * isz) + 2 * _al(nnz * key)
        assert t <= _al(nnz * isz) + 2 * _al(nnz * key) + nnz // 8
    tr = L.ofspmm_bwd_b_transient_workspace_bytes(M, cols, nnz, N, F32, idx, F32)
    fixed = _al((cols + 1) * isz) + _al(max(nnz, 1) * isz) + _al(max(nnz, 1) * 4) + _fwd(cols, nnz, N, F32)
    assert tr == fixed + _al(t)
    assert tr < fixed + old_floor


def _csr(rows, nnz, idx):
    return _lib.CsrStruct(rows, K, nnz, FAKE, FAKE, FAKE, idx, F32)


def _all_entry_points(A, ws=None, wsb=0):
    """Status of every CSR entry point on A with the given workspace (fake operands)."""
    L = _lib.lib()
    o = _lib.OptsStruct()
    r = {
        "fwd": L.ofspmm_fwd(ctypes.byref(A), FAKE, FAKE, N, F32, ws, wsb, None),
        "fwd_strided": L.ofspmm_fwd_strided(ctypes.byref(A), FAKE, N, FAKE, N, N, F32, ws, wsb, None),
        "fwd_ex": L.ofspmm_fwd_ex(ctypes.byref(A), FAKE, N, FAKE, N, N, F32, ctypes.byref(o), ws, wsb, None),
        "sddmm": L.ofspmm_sddmm(ctypes.byref(A), FAKE, FAKE, FAKE, N, F32, ws, wsb, None),
        "bwd_b": L.ofspmm_bwd_b(ctypes.byref(A), None, FAKE, FAKE, N, F32, ws, wsb, None),
        "bwd_b_transient": L.ofspmm_bwd_b_transient(ctypes.byref(A), FAKE, FAKE, N, F32, ws, wsb, None),
        "bwd_b_cached": L.ofspmm_bwd_b_cached(ctypes.byref(A), FAKE, FAKE, FAKE, FAKE, FAKE, N, F32, None, ws, wsb, None),
        "csr_transpose": L.ofspmm_csr_transpose(ctypes.byref(A), FAKE, FAKE, None, FAKE, ws, wsb, None),
        "plan_build": L.ofspmm_plan_build(FAKE, A.idx_dtype, A.rows, A.nnz, N, F32, 0, FAKE, 0, None),
    }
    return r


def test_wide_int64_call_reaches_the_workspace_check():
    """nnz = 2^31 with int64 indices passes validation: a null workspace is the only complaint."""
    r = _all_entry_points(_csr(M, 2 ** 31, I64))
    assert all(v == WORKSPACE for v in r.values()), r


@pytest.mark.parametrize("rows,nnz,idx", [
    (M, 2 ** 31 - 1, I32),          # int32 row offsets cannot count that many non-zeros
    (M, 2 ** 31, I32),
    (2 ** 31 - 1, 2 ** 31, I64),    # rows are still 32-bit
    (2 ** 31 - 1, 10, I64),
    (M, 2 ** 38, I64),              # 2^30 tasks of 256 items: beyond the task index range
])
def test_limits_that_remain(rows, nnz, idx):
    r = _all_entry_points(_csr(rows, nnz, idx))
    assert all(v == TOO_LARGE for v in r.values()), r


def test_largest_task_count_is_accepted():
    rows, nnz = 1, 2 ** 38 - 257     # (rows + nnz) / 256 = 2^30 - 1 tasks
    assert _tasks(rows, nnz) == 2 ** 30 - 1
    r = _all_entry_points(_csr(rows, nnz, I64))
    assert all(v == WORKSPACE for v in r.values()), r


def test_strerror_names_the_remaining_limits():
    msg = _lib.lib().ofspmm_strerror(TOO_LARGE).decode()
    assert "rows >= 2^31-1" in msg and "int32 indices" in msg
