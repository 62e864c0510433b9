"""CPU tests of the status every C entry point returns for invalid or degenerate arguments: unknown
dtype codes, zero sizes, null pointers and too-small workspaces.  Where several errors apply, the
one the library reports first is part of the contract (e.g. null CSR before bad dtype before
TOO_LARGE).

No call here reaches a kernel launch, so the file runs on any machine.  Where a launcher queries
the device before it looks at a dtype code, the status tells the two apart: NO_DEVICE without an
sm_100 GPU, UNSUPPORTED_DTYPE with one (``DEV_THEN_DTYPE``).  Calls that would reach their first
CUDA runtime call with host pointers are checked only without a GPU, where that call fails (CUDA)."""
import ctypes
from importlib import import_module

import numpy as np
import pytest
import torch

_lib = import_module("of-spmm_b200._lib")

OK, INVALID, DTYPE, WORKSPACE, CUDA, TOO_LARGE, NO_DEVICE = 0, 1, 2, 3, 4, 5, 6
F32, I32, I64, BF16, UNIT = _lib.DTYPE_FLOAT, _lib.DTYPE_INT32, _lib.DTYPE_INT64, _lib.DTYPE_BFLOAT16, _lib.VAL_UNIT
BAD = 9  # no dtype of the library

HAVE_B200 = torch.cuda.is_available() and torch.cuda.get_device_capability(0)[0] == 10
DEV_THEN_DTYPE = DTYPE if HAVE_B200 else NO_DEVICE
no_gpu_only = pytest.mark.skipif(torch.cuda.is_available(), reason="the call reaches a CUDA runtime call")

# a 256-byte aligned host buffer: stands in for every array argument, never read or written
_BUF = np.zeros(4096 + 256, np.uint8)
P = _BUF.ctypes.data + (-_BUF.ctypes.data) % 256
ODD = P + 4  # not 16-byte aligned


@pytest.fixture(scope="module")
def L():
    return _lib.lib()


def csr(rows=4, cols=4, nnz=8, idx=I32, vd=F32, crow=P, col=P, val=...):
    if val is ...:
        val = None if vd == UNIT else P
    return _lib.CsrStruct(rows, cols, nnz, crow, col, val, idx, vd)


def ref(A):
    return None if A is None else ctypes.byref(A)


# ---------------------------------------------------------------------------------------------
# utility entry points


def test_permute_values(L):
    def call(val=P, vd=F32, perm=P, idx=I32, nnz=4, out=P):
        return L.ofspmm_permute_values(val, vd, perm, idx, nnz, out, None)
    assert call(nnz=-1) == INVALID
    assert call(val=None) == INVALID
    assert call(perm=None, idx=BAD) == INVALID
    assert call(out=None) == INVALID
    assert call(idx=BAD) == DTYPE
    assert call(idx=BAD, nnz=0) == DTYPE
    assert call(vd=BAD, nnz=0) == OK
    assert call(val=None, perm=None, out=None, nnz=0) == OK
    assert call(vd=BAD) == DEV_THEN_DTYPE
    assert call(vd=UNIT) == DEV_THEN_DTYPE
    assert call(vd=BAD, idx=I64) == DEV_THEN_DTYPE


@pytest.mark.parametrize("name", ["ofspmm_gather_rows", "ofspmm_scatter_add_rows"])
def test_gather_and_scatter_rows(L, name):
    f = getattr(L, name)

    def call(dst=P, ld_dst=8, src=P, ld_src=8, lst=P, idx=I32, count=4, n=8, dense=F32):
        return f(dst, ld_dst, src, ld_src, lst, idx, 0, count, n, dense, 0, None)
    assert call(count=-1) == INVALID
    assert call(n=-1) == INVALID
    assert call(ld_dst=7) == INVALID
    assert call(ld_src=7) == INVALID
    assert call(dst=None) == INVALID
    assert call(src=None, idx=BAD) == INVALID
    assert call(idx=BAD) == DTYPE
    assert call(idx=BAD, count=0) == DTYPE
    assert call(lst=None, idx=BAD, dense=BAD) == DTYPE         # dense dtype checked before the device
    assert call(dense=BAD) == DTYPE
    assert call(dense=UNIT, idx=I64) == DTYPE
    assert call(dense=BAD, count=0) == OK
    assert call(dense=BAD, n=0, ld_dst=0, ld_src=0) == OK
    assert call(dst=None, src=None, count=0) == OK


def test_scatter_add_rows_f32(L):
    def call(dst=P, ld_dst=8, src=P, ld_src=8, lst=P, idx=I32, count=4, n=8, sd=BF16):
        return L.ofspmm_scatter_add_rows_f32(dst, ld_dst, src, ld_src, lst, idx, 0, count, n, sd, 0, None)
    assert call(count=-1) == INVALID
    assert call(ld_src=7) == INVALID
    assert call(src=None) == INVALID
    assert call(idx=BAD) == DTYPE
    assert call(sd=BAD) == DTYPE
    assert call(sd=BAD, lst=None, idx=BAD) == DTYPE
    assert call(sd=UNIT) == DTYPE
    assert call(sd=F32, idx=BAD) == DTYPE
    assert call(sd=F32, lst=None, idx=BAD, count=0) == OK
    assert call(sd=BAD, count=0) == OK
    assert call(sd=BAD, n=0) == OK


def test_cast_from_f32(L):
    def call(src=P, dst=P, count=4, dt=BF16):
        return L.ofspmm_cast_from_f32(src, dst, count, dt, None)
    assert call(count=-1) == INVALID
    assert call(src=None) == INVALID
    assert call(dst=None, dt=BAD) == INVALID
    assert call(dt=BAD, count=0) == OK
    assert call(src=None, dst=None, count=0) == OK
    assert call(dt=BAD) == DEV_THEN_DTYPE
    assert call(dt=I32) == DEV_THEN_DTYPE


def _pull_segs(*segs):
    arr = (_lib.PullSeg * max(1, len(segs)))()
    for i, (src, lst, flag, count) in enumerate(segs):
        arr[i] = _lib.PullSeg(src, lst, flag, count, 0)
    return arr


def test_pull_rows_multi(L):
    good = _pull_segs((P, P, P, 4))

    def call(dst=P, ld_dst=8, ld_src=8, segs=good, nseg=1, n=8, dense=F32, idx=I32):
        return L.ofspmm_pull_rows_multi(dst, ld_dst, ld_src, segs, nseg, 1, n, dense, idx, 0, None)
    assert call(n=-1) == INVALID
    assert call(ld_dst=7) == INVALID
    assert call(nseg=-1) == INVALID
    assert call(segs=None) == INVALID
    assert call(dst=None) == INVALID
    assert call(nseg=17, segs=(_lib.PullSeg * 17)()) == INVALID
    assert call(dense=BAD) == DTYPE
    assert call(dense=BAD, n=3, ld_dst=3, ld_src=3) == DTYPE       # dtype before the 16-byte check
    assert call(n=3, ld_dst=3, ld_src=3) == INVALID                 # rows of whole 16-byte units only
    assert call(dense=BF16, n=4, ld_dst=4, ld_src=4) == INVALID
    assert call(ld_src=6) == INVALID
    assert call(dst=ODD) == INVALID
    assert call(segs=_pull_segs((P, P, P, -1))) == INVALID
    assert call(segs=_pull_segs((None, P, P, 4))) == INVALID
    assert call(segs=_pull_segs((P, None, P, 4))) == INVALID
    assert call(segs=_pull_segs((P, P, None, 4))) == INVALID
    assert call(segs=_pull_segs((ODD, P, P, 4))) == INVALID
    assert call(segs=_pull_segs((ODD, None, None, 0)), idx=BAD) == INVALID
    assert call(segs=_pull_segs((None, None, None, 0)), idx=BAD) == OK   # no rows
    assert call(nseg=0, idx=BAD) == OK
    assert call(n=0, ld_dst=0, ld_src=0, idx=BAD) == OK
    assert call(idx=BAD) == DEV_THEN_DTYPE
    assert call(idx=BAD, ld_dst=16) == DEV_THEN_DTYPE               # register path (strided rows)


def test_combine_rows_multi(L):
    segs = (_lib.CombineSeg * 2)(_lib.CombineSeg(P, P, P), _lib.CombineSeg(P, None, P))

    def call(acc=P, ld_acc=8, ld_src=8, sg=segs, nseg=1, rows=4, n=8, sd=F32):
        return L.ofspmm_combine_rows_multi(acc, ld_acc, ld_src, sg, nseg, 1, rows, n, sd, 0, None)
    assert call(n=-1) == INVALID
    assert call(rows=-1) == INVALID
    assert call(ld_acc=7) == INVALID
    assert call(nseg=-1) == INVALID
    assert call(sg=None) == INVALID
    assert call(acc=None) == INVALID
    assert call(nseg=17, sg=(_lib.CombineSeg * 17)()) == INVALID
    assert call(sd=BAD) == DTYPE
    assert call(sd=UNIT) == DTYPE
    assert call(sd=BAD, n=3, ld_acc=3, ld_src=3) == DTYPE
    assert call(n=3, ld_acc=3, ld_src=3) == INVALID
    assert call(sd=BF16, n=4, ld_acc=4, ld_src=4) == INVALID
    assert call(sd=BF16, ld_acc=12) == INVALID                      # bf16: 32-byte accumulator units
    assert call(sd=BF16, acc=P + 16) == INVALID
    assert call(acc=ODD) == INVALID
    assert call(nseg=0) == OK
    assert call(rows=0, nseg=2) == OK
    assert call(n=0, ld_acc=0, ld_src=0, nseg=2) == OK
    assert call(nseg=2) == INVALID                                  # second segment without `inv`


def test_partition_and_row_hist(L):
    def part(crow=P, idx=I32, rows=4, nnz=8, parts=2, out_row=P, out_nz=P):
        return L.ofspmm_partition(crow, idx, rows, nnz, parts, out_row, out_nz, None)
    assert part(crow=None) == INVALID
    assert part(out_row=None, idx=BAD) == INVALID
    assert part(out_nz=None) == INVALID
    assert part(rows=-1) == INVALID
    assert part(nnz=-1, idx=BAD) == INVALID
    assert part(parts=0) == INVALID
    assert part(idx=BAD) == DTYPE
    assert part(idx=UNIT, rows=0, nnz=0) == DTYPE

    def hist(crow=P, idx=I32, rows=4, h=P):
        return L.ofspmm_row_hist(crow, idx, rows, h, None)
    assert hist(crow=None) == INVALID
    assert hist(h=None, idx=BAD) == INVALID
    assert hist(rows=-1, idx=BAD) == INVALID
    assert hist(idx=BAD) == DTYPE
    assert hist(idx=BAD, rows=0) == DTYPE


@no_gpu_only
def test_row_hist_zeroes_the_histogram_first(L):
    assert L.ofspmm_row_hist(P, I32, 0, P, None) == CUDA       # the memset precedes rows == 0
    assert L.ofspmm_row_hist(P, I64, 4, P, None) == CUDA


def test_expand_rows_and_normalize(L):
    def expand(crow=P, idx=I32, rows=4, out=P):
        return L.ofspmm_csr_expand_rows(crow, idx, rows, out, None)
    assert expand(rows=-1, idx=BAD) == INVALID
    assert expand(crow=None) == INVALID
    assert expand(out=None, idx=BAD) == INVALID
    assert expand(out=None, rows=0) == OK
    assert expand(idx=BAD) == DTYPE
    assert expand(idx=BAD, rows=0) == DTYPE
    assert expand(rows=0, idx=I64) == OK

    def norm(crow=P, col=P, val=P, idx=I32, rows=4, cols=4, mode=0, dinv=P):
        return L.ofspmm_csr_normalize(crow, col, val, idx, rows, cols, mode, dinv, None)
    assert norm(rows=-1) == INVALID
    assert norm(cols=-1, idx=BAD) == INVALID
    assert norm(crow=None) == INVALID
    assert norm(mode=2) == INVALID
    assert norm(dinv=None, idx=BAD) == WORKSPACE
    assert norm(dinv=None, mode=0, cols=5) == WORKSPACE
    assert norm(cols=5, idx=BAD) == INVALID                          # D^-1/2 A D^-1/2: square only
    assert norm(cols=5, mode=1, idx=BAD) == DTYPE
    assert norm(idx=BAD) == DTYPE
    assert norm(idx=BAD, rows=0, cols=0) == DTYPE
    assert norm(rows=0, cols=0, dinv=None) == OK
    assert norm(rows=0, cols=3, mode=1, idx=I64) == OK


def test_coo_to_csr(L):
    need = L.ofspmm_coo_to_csr_workspace_bytes(8, 4, 4)
    assert need > 0

    def call(row=P, col=P, val=P, nnz=8, rows=4, cols=4, co=0, idx=I32, crow=P, col_out=P, val_out=P, counts=P,
             ws=P, wsb=need):
        return L.ofspmm_coo_to_csr(row, col, val, nnz, rows, cols, co, idx, crow, col_out, val_out, counts, ws, wsb,
                                   None)
    assert call(nnz=-1) == INVALID
    assert call(rows=-1, idx=BAD) == INVALID
    assert call(co=3) == INVALID
    assert call(co=-1) == INVALID
    assert call(crow=None) == INVALID
    assert call(row=None, idx=BAD) == INVALID
    assert call(val_out=None) == INVALID
    assert call(idx=BAD) == DTYPE
    assert call(idx=BAD, nnz=2 ** 31 - 1) == DTYPE
    assert call(nnz=2 ** 31 - 1) == TOO_LARGE
    assert call(rows=2 ** 40, cols=2 ** 40) == TOO_LARGE
    assert call(idx=BAD, ws=None) == DTYPE
    assert call(wsb=need - 1) == WORKSPACE
    assert call(ws=None) == WORKSPACE
    assert call(idx=I64, wsb=need - 1) == WORKSPACE
    assert call(row=None, col=None, col_out=None, val_out=None, nnz=0, wsb=0) == WORKSPACE
    assert L.ofspmm_coo_to_csr_workspace_bytes(-1, 4, 4) == 0


def test_csr_transpose(L):
    def call(A, t_crow=P, t_col=P, t_val=P, t_perm=None, ws=P, wsb=None):
        if wsb is None and A is not None:
            wsb = max(0, L.ofspmm_csr_transpose_workspace_bytes(A.rows, A.cols, A.nnz, A.idx_dtype) - 1)
        return L.ofspmm_csr_transpose(ref(A), t_crow, t_col, t_val, t_perm, ws, wsb or 0, None)
    assert call(None) == INVALID
    assert call(csr(rows=-1, idx=BAD)) == INVALID
    assert call(csr(idx=BAD, rows=2 ** 31, crow=None)) == DTYPE
    assert call(csr(vd=BAD, rows=2 ** 31, crow=None)) == DTYPE
    assert call(csr(vd=UNIT, idx=I64, rows=2 ** 31, crow=None)) == TOO_LARGE
    assert call(csr(nnz=2 ** 31 - 1)) == TOO_LARGE
    assert call(csr(crow=None)) == INVALID
    assert call(csr(col=None)) == INVALID
    assert call(csr(val=None)) == WORKSPACE                     # the transpose needs no values of A
    assert call(csr(), t_crow=None) == INVALID
    assert call(csr(), t_col=None) == INVALID
    assert call(csr(nnz=0, col=None), t_col=None) == WORKSPACE
    assert call(csr(vd=UNIT), t_val=P) == INVALID
    assert call(csr(vd=UNIT), t_val=None) == WORKSPACE
    assert call(csr(vd=BF16, idx=I64), t_perm=P) == WORKSPACE
    assert call(csr(idx=I64, cols=2 ** 31)) == WORKSPACE         # 64-bit column keys
    assert call(csr(), ws=None, wsb=1 << 20) == WORKSPACE
    assert L.ofspmm_csr_transpose_workspace_bytes(4, 4, 8, BAD) == 0


def test_sample_neighbors(L):
    def call(A, dst=P, num_dst=2, fanout=3, cap=8, blk_crow=P, blk_col=P, blk_val=P, src=P, counts=P, ws=P, wsb=None):
        if wsb is None:
            wsb = L.ofspmm_sample_neighbors_workspace_bytes(num_dst, cap, I32) - 1
        return L.ofspmm_sample_neighbors(ref(A), dst, num_dst, fanout, 7, cap, blk_crow, blk_col, blk_val, src, counts,
                                         ws, wsb, None)
    assert call(None) == INVALID
    assert call(csr(vd=BAD)) == DTYPE
    assert call(csr(idx=BAD, rows=-1)) == INVALID
    assert call(csr(idx=I64, vd=BAD, rows=2 ** 31, cols=2 ** 31, crow=None)) == DTYPE
    assert call(csr(rows=2 ** 31, cols=2 ** 31, crow=None, idx=I64)) == TOO_LARGE
    assert call(csr(cols=5), cap=-1) == INVALID
    assert call(csr(), num_dst=2 ** 31, dst=None) == TOO_LARGE
    assert call(csr(), counts=None, cap=2 ** 31) == TOO_LARGE
    assert call(csr()) == WORKSPACE
    assert call(csr(vd=BF16, idx=I64)) == WORKSPACE
    assert call(csr(vd=UNIT), blk_val=None) == WORKSPACE
    assert call(csr(), ws=None, wsb=1 << 30) == WORKSPACE
    assert call(csr(), num_dst=0, cap=0, dst=None, blk_col=None, blk_val=None, src=None) == WORKSPACE


# ---------------------------------------------------------------------------------------------
# product entry points


def _opts(flags=0):
    return ctypes.byref(_lib.OptsStruct(flags, 0, 0, 0, None, 0, None, None))


FWD = {
    "fwd": lambda L, A, B, C, n, d, ws, wsb: L.ofspmm_fwd(ref(A), B, C, n, d, ws, wsb, None),
    "fwd_strided": lambda L, A, B, C, n, d, ws, wsb: L.ofspmm_fwd_strided(ref(A), B, n, C, n, n, d, ws, wsb, None),
    "fwd_ex": lambda L, A, B, C, n, d, ws, wsb: L.ofspmm_fwd_ex(ref(A), B, n, C, n, n, d, None, ws, wsb, None),
    "fwd_host": lambda L, A, B, C, n, d, ws, wsb: L.ofspmm_fwd_host(ref(A), B, C, n, d, ws, wsb, None),
}


def _fwd_need(L, name, A, n, d):
    if name == "fwd_host":
        return L.ofspmm_fwd_host_workspace_bytes(A.rows, A.cols, A.nnz, n, d, A.idx_dtype, A.val_dtype)
    return L.ofspmm_fwd_workspace_bytes(A.rows, A.cols, A.nnz, n, d)


@pytest.mark.parametrize("name", list(FWD))
def test_forward_entry_points(L, name):
    f = FWD[name]

    def call(A, B=P, C=P, n=8, d=F32, ws=P, wsb=None):
        if wsb is None and A is not None and A.rows >= 0 and A.nnz >= 0 and A.cols >= 0 and n >= 0:
            wsb = _fwd_need(L, name, A, n, d) - 1
        return f(L, A, B, C, n, d, ws, wsb or 0)
    assert call(None) == INVALID
    assert call(csr(rows=-1, idx=BAD)) == INVALID
    assert call(csr(nnz=-1)) == INVALID
    assert call(csr(idx=BAD, rows=2 ** 31, crow=None)) == DTYPE
    assert call(csr(vd=BAD, rows=2 ** 31, crow=None)) == DTYPE
    assert call(csr(vd=BF16, rows=2 ** 31, crow=None)) == TOO_LARGE   # dense dtype is checked later
    assert call(csr(rows=2 ** 31, crow=None), d=BAD) == TOO_LARGE
    assert call(csr(nnz=2 ** 31 - 1, crow=None)) == TOO_LARGE
    assert call(csr(crow=None), d=BAD) == INVALID
    assert call(csr(col=None), d=BAD) == INVALID
    assert call(csr(val=None), d=BAD) == INVALID
    assert call(csr(vd=UNIT, val=P), d=BAD) == INVALID
    assert call(csr(nnz=0, col=None, val=None), d=BAD) == DTYPE
    assert call(csr(), d=BAD) == DTYPE
    assert call(csr(), d=I32) == DTYPE
    assert call(csr(vd=BF16), d=F32) == DTYPE
    assert call(csr(), n=-1, C=None) == INVALID
    assert call(csr(), n=2 ** 31, C=None) == INVALID
    assert call(csr(), C=None) == INVALID
    assert call(csr(), B=None) == INVALID
    assert call(csr(rows=0, nnz=0), B=None, C=None) == OK
    assert call(csr(), n=0, B=None, C=None) == OK
    assert call(csr()) == WORKSPACE
    assert call(csr(vd=UNIT), d=BF16) == WORKSPACE
    assert call(csr(vd=BF16, idx=I64), d=BF16) == WORKSPACE
    assert call(csr(), ws=None, wsb=1 << 30) == WORKSPACE
    if name != "fwd_host":                                       # the host copy keeps its own alignment
        assert call(csr(), ws=ODD, wsb=1 << 30) == WORKSPACE


def test_forward_options(L):
    def call(A, flags, n=8):
        return L.ofspmm_fwd_ex(ref(A), P, n, P, n, n, F32, _opts(flags), P, 0, None)
    mean_acc = _lib.FWD_MEAN | _lib.FWD_ACCUMULATE
    assert call(csr(rows=0, nnz=0), mean_acc) == INVALID                  # before the empty-product exit
    assert call(csr(), _lib.FWD_MEAN | _lib.FWD_ACC32_IN) == INVALID
    assert call(csr(), _lib.FWD_BIAS) == INVALID                          # bias flag without a bias
    assert call(csr(), _lib.FWD_ACC32_IN | _lib.FWD_ACC32_OUT) == INVALID  # fp32 products accumulate in C
    assert call(csr(nnz=0), _lib.FWD_ACCUMULATE) == OK                    # += 0
    assert call(csr(), _lib.FWD_MEAN) == WORKSPACE


BWD = ("bwd_b", "bwd_b_transient", "bwd_b_cached")


def _bwd(L, name, A, dY=P, dB=P, n=8, d=F32, ws=P, wsb=0, At=None, t=(P, P, P)):
    if name == "bwd_b":
        return L.ofspmm_bwd_b(ref(A), ref(At), dY, dB, n, d, ws, wsb, None)
    if name == "bwd_b_transient":
        return L.ofspmm_bwd_b_transient(ref(A), dY, dB, n, d, ws, wsb, None)
    return L.ofspmm_bwd_b_cached(ref(A), *t, dY, dB, n, d, None, ws, wsb, None)


def _bwd_need(L, name, A, n, d):
    if name == "bwd_b":
        return L.ofspmm_bwd_b_workspace_bytes(A.rows, A.cols, A.nnz, n, d, 0)
    if name == "bwd_b_transient":
        return L.ofspmm_bwd_b_transient_workspace_bytes(A.rows, A.cols, A.nnz, n, d, A.idx_dtype, A.val_dtype)
    return L.ofspmm_bwd_b_cached_workspace_bytes(A.rows, A.cols, A.nnz, n, d, A.val_dtype)


@pytest.mark.parametrize("name", BWD)
def test_backward_entry_points(L, name):
    def call(A, **kw):
        return _bwd(L, name, A, **kw)
    assert call(None) == INVALID
    assert call(csr(cols=-1, idx=BAD)) == INVALID
    assert call(csr(idx=BAD, rows=2 ** 31, crow=None)) == DTYPE
    assert call(csr(vd=BAD, rows=2 ** 31, crow=None)) == DTYPE
    assert call(csr(rows=2 ** 31, crow=None), d=BAD) == TOO_LARGE
    assert call(csr(crow=None), d=BAD) == INVALID
    assert call(csr(val=None), d=BAD) == INVALID
    assert call(csr(), d=BAD, dB=None) == DTYPE
    assert call(csr(vd=BF16), d=F32, dB=None) == DTYPE
    assert call(csr(), n=-1, dB=None) == INVALID
    assert call(csr(), n=2 ** 31) == INVALID
    assert call(csr(cols=0), dB=None, dY=None) == OK
    assert call(csr(), n=0, dB=None, dY=None) == OK
    assert call(csr(), dB=None) == INVALID
    assert call(csr(), dY=None) == INVALID
    for A, d in ((csr(), F32), (csr(vd=BF16, idx=I64), BF16), (csr(vd=UNIT), F32), (csr(vd=UNIT, idx=I64), BF16)):
        need = _bwd_need(L, name, A, 8, d)
        assert call(A, d=d, wsb=need - 1) == WORKSPACE
        assert call(A, d=d, ws=None, wsb=need) == WORKSPACE
        assert call(A, d=d, ws=ODD, wsb=need) == WORKSPACE


def test_backward_route_checks(L):
    # bwd_b with a cached transpose: A^T is validated, then its shape, then its dtypes
    A = csr(rows=4, cols=6)
    assert _bwd(L, "bwd_b", A, At=csr(rows=6, cols=4, crow=None)) == INVALID
    assert _bwd(L, "bwd_b", A, At=csr(rows=6, cols=4, idx=BAD)) == DTYPE
    assert _bwd(L, "bwd_b", A, At=csr(rows=4, cols=6, idx=BAD)) == DTYPE
    assert _bwd(L, "bwd_b", A, At=csr(rows=4, cols=6)) == INVALID
    assert _bwd(L, "bwd_b", A, At=csr(rows=6, cols=4, nnz=7)) == INVALID
    assert _bwd(L, "bwd_b", A, At=csr(rows=6, cols=4, vd=BF16), d=F32) == DTYPE
    assert _bwd(L, "bwd_b", A, At=csr(rows=6, cols=4)) == WORKSPACE
    need = L.ofspmm_fwd_workspace_bytes(6, 4, 8, 8, F32)
    assert _bwd(L, "bwd_b", A, At=csr(rows=6, cols=4), wsb=need - 1) == WORKSPACE
    # cached route: the caller's A^T structure
    assert _bwd(L, "bwd_b_cached", A, t=(None, P, P)) == INVALID
    assert _bwd(L, "bwd_b_cached", A, t=(P, None, P)) == INVALID
    assert _bwd(L, "bwd_b_cached", A, t=(P, P, None)) == INVALID
    assert _bwd(L, "bwd_b_cached", A, t=(None, None, None), dB=None, n=0) == OK


@no_gpu_only
@pytest.mark.parametrize("name", ("bwd_b", "bwd_b_transient"))
def test_backward_empty_matrix_zeroes_db(L, name):
    # an empty A zeroes dB before the workspace is looked at; the cached route runs the forward
    assert _bwd(L, name, csr(nnz=0), ws=None) == CUDA
    assert _bwd(L, name, csr(rows=0, nnz=0), ws=None) == CUDA


@no_gpu_only
def test_backward_cached_empty_matrix(L):
    assert _bwd(L, "bwd_b_cached", csr(nnz=0), ws=None) == WORKSPACE
    assert _bwd(L, "bwd_b_cached", csr(nnz=0), wsb=1 << 30) == CUDA
    assert _bwd(L, "bwd_b", csr(nnz=0), At=csr(nnz=0), ws=None) == CUDA


def test_sddmm(L):
    def call(A, dY=P, B=P, dval=P, n=8, d=F32, ws=P, wsb=None, opts=None):
        if wsb is None and A is not None and A.rows >= 0 and A.nnz >= 0:
            wsb = L.ofspmm_sddmm_workspace_bytes(A.rows, A.cols, A.nnz, n, d) - 1
        return L.ofspmm_sddmm_ex(ref(A), dY, B, dval, n, d, opts, ws, wsb or 0, None)
    assert call(None) == INVALID
    assert call(csr(vd=UNIT, rows=-1)) == DTYPE                       # a pattern matrix: before anything else
    assert call(csr(rows=-1, idx=BAD)) == INVALID
    assert call(csr(idx=BAD, rows=2 ** 31, crow=None)) == DTYPE
    assert call(csr(vd=BAD)) == DTYPE
    assert call(csr(rows=2 ** 31, crow=None), d=BAD) == TOO_LARGE
    assert call(csr(crow=None), d=BAD) == INVALID
    assert call(csr(col=None), d=BAD) == INVALID
    assert call(csr(val=None), d=BAD) == DTYPE                       # A's values are not read
    assert call(csr(vd=BF16), d=F32) == DTYPE
    assert call(csr(), n=-1) == INVALID
    assert call(csr(nnz=0, col=None), dval=None, dY=None, B=None) == OK
    assert call(csr(), dval=None, n=0) == INVALID
    assert call(csr(), dY=None) == INVALID
    assert call(csr(), B=None) == INVALID
    assert call(csr()) == WORKSPACE
    assert call(csr(), ws=None, wsb=1 << 30) == WORKSPACE
    assert call(csr(), ws=ODD, wsb=1 << 30) == WORKSPACE
    assert call(csr(vd=BF16, idx=I64), d=BF16, opts=_opts()) == WORKSPACE
    assert L.ofspmm_sddmm(ref(csr(vd=UNIT)), P, P, P, 8, F32, P, 1 << 30, None) == DTYPE


@no_gpu_only
def test_sddmm_zero_width_zeroes_dval(L):
    assert L.ofspmm_sddmm_ex(ref(csr()), None, None, P, 0, F32, None, None, 0, None) == CUDA
    assert L.ofspmm_sddmm_ex(ref(csr(cols=0)), None, None, P, 8, F32, None, None, 0, None) == CUDA


@no_gpu_only
def test_forward_host_staging_copies_first(L):
    A = csr()
    need = L.ofspmm_fwd_host_workspace_bytes(4, 4, 8, 8, F32, I32, F32)
    assert L.ofspmm_fwd_host(ref(A), P, P, 8, F32, P, need, None) == CUDA
