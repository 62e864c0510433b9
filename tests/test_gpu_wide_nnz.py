"""GPU tests of a CSR matrix with 2^31 + 2^25 non-zeros and int64 indices ("wide": beyond what
int32 offsets can count), built on the device by ``graphs.wide_csr`` (26 GB).

Row r below is a task boundary (r + crow[r] is a multiple of the 256-item task size), so the tasks
of the wide product are exactly the tasks of the two row blocks [0, r) and [r, M) run as ordinary
(narrow) matrices, shifted by a constant: wide results must equal the concatenated block results
bit for bit, for every row and every non-zero, with no oracle.  A sample of rows, columns and
positions around 2^31 is also checked against the fp64 oracle.  The whole file stays below 120 GB
of device memory (``torch.cuda.max_memory_allocated``, reported after each stage)."""
import ctypes
import gc
from importlib import import_module

import numpy as np
import pytest
import torch

import ofspmm_b200 as ofs
from oracle import oracle as O

pytestmark = pytest.mark.gpu

G = ofs.graphs
ops = import_module("of-spmm_b200.ops")
gcn = import_module("of-spmm_b200.gcn")
_lib = ofs._lib
DEV = "cuda:0"
PEAK_LIMIT = 120e9
NEED_FREE = 115e9      # the file's own peak is ~109 GB
CHUNK = 1 << 27
M, K, NNZ = G.WIDE_M, G.WIDE_K, G.WIDE_NNZ
DD = {torch.float32: _lib.DTYPE_FLOAT, torch.bfloat16: _lib.DTYPE_BFLOAT16}


_BASE = [0]   # bytes other modules still hold when this one starts (not part of its peak)


def _stage(what):
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - _BASE[0]
    print(f"[wide] {what}: peak allocated {peak / 1e9:.1f} GB")
    assert peak <= PEAK_LIMIT, f"{what}: peak {peak / 1e9:.1f} GB > 120 GB"


def _release():
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def _B(n=128, dtype=torch.float32):
    return G.dense_operand(K, n, 31, DEV, dtype)


def _dY(n=128):
    return G.upstream_grad(M, n, 34, DEV)


@pytest.fixture(scope="module")
def W():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    # blocks the caching allocator kept from earlier modules are free for this one
    _release()
    free, _ = torch.cuda.mem_get_info(0)
    free += torch.cuda.memory_reserved(0) - torch.cuda.memory_allocated(0)
    if free < NEED_FREE:
        pytest.skip(f"needs {NEED_FREE / 1e9:.0f} GB of free device memory for a 2^31-non-zero matrix, "
                    f"{free / 1e9:.0f} GB free")
    _BASE[0] = torch.cuda.memory_allocated(0)
    torch.cuda.reset_peak_memory_stats()
    A = G.wide_csr(DEV)
    crow_h = A.crow.cpu().numpy()
    # split row: a task boundary in the first half, both blocks narrow (< 2^31-1 non-zeros)
    cand = np.arange(M // 4, M // 2)
    hit = cand[(cand + crow_h[cand]) % 256 == 0]
    assert hit.size > 0
    r = int(hit[0])
    assert crow_h[r] < 2 ** 31 - 1 and NNZ - crow_h[r] < 2 ** 31 - 1
    _stage("matrix built")
    yield dict(A=A, crow_h=crow_h, r=r)
    del A
    _release()


def _block(A, r0, r1, crow_h):
    """Rows [r0, r1) as a narrow CSR: views of col / val, crow re-based to 0."""
    p0, p1 = int(crow_h[r0]), int(crow_h[r1])
    return (A.crow[r0:r1 + 1] - p0), A.col[p0:p1], A.val[p0:p1], r1 - r0


def _variant(crow, rows, nnz, n, dtype):
    hist = ops.row_hist(crow).cpu()
    arr = (ctypes.c_int64 * 32)(*hist.tolist())
    return _lib.lib().ofspmm_choose_variant(arr, rows, nnz, n, DD[dtype])


def _fwd(crow, col, val, b, rows, cols, variant, **kw):
    return ops.spmm_csr_compute(crow, col, val, b, rows, cols, variant=variant, **kw)


ROWPAR = _lib.VARIANT_EXPLICIT | _lib.VARIANT_ROWPAR


@pytest.mark.parametrize("n,dtype,forced", [
    (128, torch.float32, None),
    (32, torch.float32, None),
    (32, torch.float32, ROWPAR),     # sub-warp groups owning whole rows
    (18, torch.float32, None),       # scalar lanes (rows not a whole number of 16-byte vectors)
    (256, torch.bfloat16, None),
])
@pytest.mark.parametrize("mode", ["plain", "bias_relu", "accumulate"])
def test_forward_equals_narrow_blocks_bit_for_bit(W, n, dtype, forced, mode):
    A, r, crow_h = W["A"], W["r"], W["crow_h"]
    v = forced if forced is not None else _variant(A.crow, M, NNZ, n, dtype)
    B = _B(n, dtype)
    kw, kw1, kw2 = {}, {}, {}
    if mode == "bias_relu":
        bias = G.dense_operand(1, n, 32, DEV, dtype)[0].contiguous()
        kw = kw1 = kw2 = dict(bias=bias, relu=True)
    elif mode == "accumulate":
        C0 = G.upstream_grad(M, n, 33, DEV, dtype)
        kw = dict(out=C0.clone(), accumulate=True)
        kw1 = dict(out=C0[:r].clone(), accumulate=True)
        kw2 = dict(out=C0[r:].clone(), accumulate=True)
        del C0
    C = _fwd(A.crow, A.col, A.val, B, M, K, v, **kw)
    c1, k1, v1, m1 = _block(A, 0, r, crow_h)
    c2, k2, v2, m2 = _block(A, r, M, crow_h)
    C1 = _fwd(c1, k1, v1, B, m1, K, v, **kw1)
    C2 = _fwd(c2, k2, v2, B, m2, K, v, **kw2)
    assert torch.equal(C[:r], C1) and torch.equal(C[r:], C2), \
        _lib.lib().ofspmm_variant_name(v, M, NNZ, n, DD[dtype]).decode()
    _stage(f"forward n={n} {dtype} {mode}")


def _rows_to_host(A, rows_sel, crow_h):
    """CSR of the selected rows, on the host (positions copied from the device)."""
    lens = crow_h[rows_sel + 1] - crow_h[rows_sel]
    crow_s = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    col = np.concatenate([A.col[int(crow_h[i]):int(crow_h[i + 1])].cpu().numpy() for i in rows_sel])
    val = np.concatenate([A.val[int(crow_h[i]):int(crow_h[i + 1])].cpu().numpy() for i in rows_sel])
    return crow_s, col.astype(np.int64), val, lens


def test_forward_against_oracle_on_sampled_rows(W):
    A, r, crow_h = W["A"], W["r"], W["crow_h"]
    B = _B()
    C = ops.spmm_csr_compute(A.crow, A.col, A.val, B, M, K)
    row_of = lambda p: int(np.searchsorted(crow_h, p, side="right") - 1)  # noqa: E731
    special = {G.WIDE_HUB, r, r - 1, row_of(2 ** 31 - 1), row_of(2 ** 31), row_of(1000), row_of(NNZ - 2),
               G.WIDE_HUB - 1, G.WIDE_HUB + 1, M - 1, 3, 5}
    rng = np.random.default_rng(3)
    rows_sel = np.array(sorted(special | set(rng.choice(M, 256 - len(special), replace=False).tolist())))
    assert (crow_h[rows_sel + 1] - crow_h[rows_sel] == 0).any() and (crow_h[rows_sel + 1] - crow_h[rows_sel] == 1).any()
    crow_s, col_s, val_s, lens = _rows_to_host(A, rows_sel, crow_h)
    Bh = B.cpu().numpy()
    ref = O.spmm_f64(crow_s, col_s, val_s, Bh, K)
    amax = O.spmm_absmax(crow_s, col_s, val_s, Bh, K)
    got = C[torch.from_numpy(rows_sel).to(DEV)].cpu().numpy().astype(np.float64)
    tol = O.fp32_tolerance(ref, amax, lens, rtol=1e-5) + 1e-30
    err = np.abs(got - ref)
    assert (err <= tol).all(), f"{(err > tol).sum()} outside tolerance, worst excess {float((err - tol).max()):.3e}"
    _stage("forward oracle")


def test_sddmm_equals_narrow_blocks_and_oracle(W):
    A, r, crow_h = W["A"], W["r"], W["crow_h"]
    B, dY, n = _B(), _dY(), 128
    dval = ops.sddmm_csr_compute(A.crow, A.col, dY, B, M, K)
    c1, k1, _, m1 = _block(A, 0, r, crow_h)
    c2, k2, _, m2 = _block(A, r, M, crow_h)
    d1 = ops.sddmm_csr_compute(c1, k1, dY[:r], B, m1, K)
    p = int(crow_h[r])
    assert torch.equal(dval[:p], d1)
    del d1
    d2 = ops.sddmm_csr_compute(c2, k2, dY[r:], B, m2, K)
    assert torch.equal(dval[p:], d2)
    del d2
    pos = np.array([2 ** 31 - 2, 2 ** 31 - 1, 2 ** 31, 2 ** 31 + 1, 2 ** 31 + 7, NNZ - 2, NNZ - 1])
    rows = np.searchsorted(crow_h, pos, side="right") - 1
    cols = A.col[torch.from_numpy(pos).to(DEV)].cpu().numpy()
    Bh, dYh = B.cpu().numpy().astype(np.float64), dY[torch.from_numpy(rows).to(DEV)].cpu().numpy().astype(np.float64)
    ok = (cols >= 0) & (cols < K)
    prod = dYh * Bh[np.where(ok, cols, 0)]
    ref = np.where(ok, prod.sum(1), 0.0)
    aabs = np.abs(prod).sum(1)
    got = dval[torch.from_numpy(pos).to(DEV)].cpu().numpy().astype(np.float64)
    assert (np.abs(got - ref) <= 1e-5 * np.abs(ref) + 2.0 ** -23 * n * aabs + 1e-30).all(), (got, ref)
    assert (got[~ok] == 0).all()
    _stage("sddmm")


def test_transpose_properties(W):
    A, crow_h = W["A"], W["crow_h"]
    t_crow, t_col, _, t_perm = ops.csr_transpose(A.crow, A.col, None, M, K, want_perm=True)
    _stage("transpose built")
    bad = len(G.WIDE_BAD)
    counts = torch.zeros(K, dtype=torch.int64, device=DEV)
    prev_key, prev_perm = None, None
    for q0 in range(0, NNZ, CHUNK):
        q1 = min(NNZ, q0 + CHUNK)
        c = A.col[q0:q1]
        ok = (c >= 0) & (c < K)
        counts += torch.bincount(c[ok], minlength=K)
        perm = t_perm[q0:q1]
        key = A.col[perm]
        key = torch.where((key >= 0) & (key < K), key, torch.full_like(key, K))
        if prev_key is not None:
            key = torch.cat([prev_key, key])
            perm = torch.cat([prev_perm, perm])
        # sorted by column (skipped entries last), stable: ascending position within a column
        assert (key[1:] >= key[:-1]).all()
        same = key[1:] == key[:-1]
        assert (perm[1:][same] > perm[:-1][same]).all()
        k2 = key[-(q1 - q0):] if prev_key is not None else key
        p2 = perm[-(q1 - q0):] if prev_perm is not None else perm
        want = torch.searchsorted(A.crow, p2, right=True) - 1
        want = torch.where(k2 < K, want, torch.full_like(want, -1))
        assert torch.equal(t_col[q0:q1], want)
        prev_key, prev_perm = key[-1:], perm[-1:]
    want_crow = torch.zeros(K + 1, dtype=torch.int64, device=DEV)
    want_crow[1:] = torch.cumsum(counts, 0)
    assert torch.equal(t_crow[:K], want_crow[:K]) and int(t_crow[K]) == NNZ
    assert int(want_crow[K]) == NNZ - bad
    assert (t_col[NNZ - bad:] == -1).all()
    assert t_perm[NNZ - bad:].cpu().tolist() == sorted(p for p, _ in G.WIDE_BAD)
    _stage("transpose checked")


def test_grad_b_routes(W):
    A, dY, n = W["A"], _dY(), 128
    _release()
    plan = ops.SpmmPlan(A.crow, A.col, M, K, n, torch.float32, transpose=True)
    t_crow, t_col, t_perm = plan.t_crow, plan.t_col, plan.t_perm
    dB = ops.spmm_csr_grad_b_compute(A.crow, A.col, A.val, dY, M, K, plan=plan, regather=True)
    _stage("grad_b cached")
    # forward on the wide A^T, and on its two narrow column blocks, with the cached route's variant
    t_val = torch.empty(NNZ, dtype=torch.float32, device=DEV)
    _lib.check(_lib.lib().ofspmm_permute_values(A.val.data_ptr(), _lib.DTYPE_FLOAT, t_perm.data_ptr(), _lib.DTYPE_INT64,
                                                NNZ, t_val.data_ptr(), torch.cuda.current_stream().cuda_stream), "permute")
    assert torch.equal(_fwd(t_crow, t_col, t_val, dY, K, M, plan.t_variant), dB)
    tc_h = t_crow.cpu().numpy()
    cand = np.arange(K // 4, 3 * K // 4)
    c = int(cand[(cand + tc_h[cand]) % 256 == 0][0])
    At = G.CsrMatrix(t_crow, t_col, t_val, K, M)
    b1, b2 = _block(At, 0, c, tc_h), _block(At, c, K, tc_h)
    assert torch.equal(_fwd(b1[0], b1[1], b1[2], dY, b1[3], M, plan.t_variant), dB[:c])
    assert torch.equal(_fwd(b2[0], b2[1], b2[2], dY, b2[3], M, plan.t_variant), dB[c:])
    _stage("A^T forward vs narrow blocks")
    del plan, At, b1, b2, t_val, t_crow, t_col, t_perm
    _release()
    dB_tr = ops.spmm_csr_grad_b_transient_compute(A.crow, A.col, A.val, dY, M, K)
    assert torch.equal(dB_tr, dB)
    del dB_tr
    _stage("grad_b transient")
    dB_at = ops.spmm_csr_grad_b_compute(A.crow, A.col, A.val, dY, M, K, atomic=True)
    cnt = torch.zeros(K, dtype=torch.int64, device=DEV)
    for q0 in range(0, NNZ, CHUNK):
        cc = A.col[q0:q0 + CHUNK]
        cnt += torch.bincount(cc[(cc >= 0) & (cc < K)], minlength=K)
    bound = float(A.val.abs().max()) * float(dY.abs().max())
    tol = 2e-5 * dB.abs().double() + 2.0 ** -22 * cnt.double()[:, None] * bound + 1e-30
    assert ((dB_at.double() - dB.double()).abs() <= tol).all()
    del dB_at
    _stage("grad_b atomic")
    # oracle on 256 sampled columns; their entries found on the device
    rng = np.random.default_rng(4)
    cols_s = np.unique(np.concatenate([[0, K - 1], rng.choice(K, 254, replace=False)]))
    cs = torch.from_numpy(cols_s).to(DEV)
    pos = torch.cat([torch.nonzero(torch.isin(A.col[q0:q0 + CHUNK], cs)).flatten() + q0
                     for q0 in range(0, NNZ, CHUNK)])
    rows = (torch.searchsorted(A.crow, pos, right=True) - 1).cpu().numpy()
    col_sub = torch.searchsorted(cs, A.col[pos]).cpu().numpy().astype(np.int64)
    val_sub = A.val[pos].cpu().numpy()
    crow_sub = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=M))]).astype(np.int64)
    dYh = dY.cpu().numpy()
    ref = O.spmm_t_f64(crow_sub, col_sub, val_sub, dYh, len(cols_s))
    amax, cnt_s = O.spmm_t_absmax(crow_sub, col_sub, val_sub, dYh, len(cols_s))
    got = dB[cs].cpu().numpy().astype(np.float64)
    tol = O.fp32_tolerance(ref, amax, cnt_s, rtol=1e-5) + 1e-30
    assert (np.abs(got - ref) <= tol).all()
    del dB
    _stage("grad_b oracle")


def test_spmm_csr_autograd_and_gcnconv(W):
    A, dY, B = W["A"], _dY(), _B()
    _release()

    def run():
        state = ofs.SpmmOpKernelState()
        v = A.val.detach().requires_grad_(True)
        b = B.detach().clone().requires_grad_(True)
        C = ofs.spmm_csr(A.crow, A.col, v, b, M, K, state)
        C.backward(dY)
        return C.detach(), b.grad, v.grad, state

    C, d_b, d_val, state = run()
    _stage("spmm_csr forward + backward")
    assert torch.equal(d_b, ops.spmm_csr_grad_b_compute(A.crow, A.col, A.val, dY, M, K, plan=state._plan))
    assert torch.equal(d_val, ops.sddmm_csr_compute(A.crow, A.col, dY, B, M, K))
    state.clear()
    del state
    _release()
    C2, d_b2, d_val2, state2 = run()
    assert torch.equal(C, C2) and torch.equal(d_b, d_b2) and torch.equal(d_val, d_val2)   # deterministic
    state2.clear()
    del C, C2, d_b, d_b2, d_val, d_val2, state2, dY, B
    _release()
    _stage("spmm_csr determinism")

    conv = gcn.GCNConv(64, 16, device=DEV, seed=6)
    X = G.dense_operand(K, 64, 35, DEV)
    st = ofs.SpmmOpKernelState()
    v = A.val.detach().requires_grad_(True)
    out = conv(A, X, val=v, state=st)
    want = ops.spmm_csr_compute(A.crow, A.col, A.val, (X @ conv.weight).detach().contiguous(), M, K,
                                bias=conv.bias.detach(), relu=True, plan=st._plan)
    assert torch.equal(out.detach(), want)
    out.square().sum().backward()
    assert torch.isfinite(conv.weight.grad).all() and torch.isfinite(conv.bias.grad).all()
    assert v.grad is not None and torch.isfinite(v.grad).all()
    st.clear()
    _stage("GCNConv forward + backward")
