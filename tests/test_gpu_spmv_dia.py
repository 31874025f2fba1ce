"""The offset-diagonal (DIA) copy of structured operators (csrc/spmv_dia.cuh): which operators get one, and that
streaming it gives bitwise the results of the CSR stream -- for mul!, cg! (Identity, Jacobi, iterator form) and
minres! -- under spmv_format 0 (DIA when present) vs 1 (always CSR)."""
import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu
SEED = 1234321


@pytest.fixture(scope="module")
def isb():
    import iterativesolvers_jl_b200 as m
    m.default_context()
    return m


def both_formats(isb, f):
    """f() under spmv_format 1 (CSR), then under 0 (auto)."""
    ctx = isb.default_context()
    L = isb.lib()
    try:
        assert L.b200_ctx_set_option(ctx._h, b"spmv_format", 1) == 0
        a = f()
        assert L.b200_ctx_set_option(ctx._h, b"spmv_format", 0) == 0
        b = f()
    finally:
        L.b200_ctx_set_option(ctx._h, b"spmv_format", 0)
    return a, b


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.int64 if a.dtype == np.float64 else np.int32)


def assert_bitwise(a, b):
    assert a.dtype == b.dtype and a.shape == b.shape
    assert np.array_equal(bits(a), bits(b))


def laplace_offsets(N, dims):
    return sorted({0} | {s * N ** k for k in range(dims) for s in (-1, 1)})


# ------------------------------------------------------------------ which operators get a DIA copy
def test_spmv_format_option(isb):
    import ctypes as C
    ctx = isb.default_context()
    L = isb.lib()
    v = C.c_int64(-1)
    assert L.b200_ctx_get_option(ctx._h, b"spmv_format", C.byref(v)) == 0 and v.value == 0
    assert L.b200_ctx_set_option(ctx._h, b"spmv_format", 2) != 0
    assert L.b200_ctx_get_option(ctx._h, b"spmv_format", C.byref(v)) == 0 and v.value == 0


# N, dims: m = 262144 and 512 (whole tiles), 1000, 10000 and 100 (ragged), 5 (tiny)
@pytest.mark.parametrize("N,dims", [(64, 3), (8, 3), (10, 3), (100, 2), (10, 2), (5, 1)])
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_laplacian_is_dia_and_bitwise(isb, oracle, N, dims, dtype):
    rng = np.random.default_rng(SEED)
    O = oracle.laplace_matrix(dtype, N, dims, base=1)
    A = isb.B200CSR.from_csc_arrays(O.colptr, O.rowval, O.nzval, O.shape, base=1)
    G = isb.B200CSR.laplacian(N, dims, dtype=dtype)                # the device generator gets the same copy
    assert A.format == "dia" and G.format == "dia"
    assert A.dia_offsets == laplace_offsets(N, dims) == G.dia_offsets
    x = rng.standard_normal(O.n).astype(dtype)
    y_csr, y_dia = both_formats(isb, lambda: A @ x)
    assert_bitwise(y_csr, y_dia)
    g_csr, g_dia = both_formats(isb, lambda: G @ x)
    assert_bitwise(g_csr, y_csr)
    assert_bitwise(g_dia, y_csr)
    yo = oracle.csc_spmv(O, x)
    if dtype == np.float64:
        assert_bitwise(y_dia, yo)
    else:
        np.testing.assert_allclose(y_dia, yo, rtol=1e-5, atol=1e-5)
    At = A.adjoint()                                                # the transpose is built by the same path
    assert At.format == "dia" and At.dia_offsets == A.dia_offsets


def test_advection_operator_bitwise(isb, oracle):
    M, _ = oracle.advection_dominated(N=20)
    A = isb.B200CSR.from_scipy(M)
    assert A.format == "dia" and len(A.dia_offsets) == 7
    x = np.random.default_rng(SEED).standard_normal(M.shape[0])
    y_csr, y_dia = both_formats(isb, lambda: A @ x)
    assert_bitwise(y_csr, y_dia)
    assert_bitwise(y_dia, oracle.csc_spmv(oracle.CSC.from_scipy(M), x))


def banded(n, offsets, keep, rng, drop_cols=()):
    """CSR (int32, sorted columns) of an n x n matrix with entries on `offsets`, each kept with probability `keep`;
    every entry of a column in drop_cols removed; a few stored entries explicit zeros."""
    rows, cols = [], []
    for o in offsets:
        i = np.arange(max(0, -o), min(n, n - o))
        k = rng.random(i.size) < keep
        rows.append(i[k])
        cols.append(i[k] + o)
    rows, cols = np.concatenate(rows), np.concatenate(cols)
    k = ~np.isin(cols, np.asarray(drop_cols, dtype=np.int64))
    rows, cols = rows[k], cols[k]
    vals = rng.standard_normal(rows.size)
    vals[rng.random(rows.size) < 0.05] = 0.0                        # explicit stored zeros
    M = sp.coo_matrix((vals, (rows, cols)), shape=(n, n)).tocsr()  # no duplicates: sum_duplicates keeps the zeros
    M.sort_indices()
    return M


def from_csr(isb, M):
    return isb.B200CSR.from_csr_slab(M.indptr.astype(np.int32), M.indices.astype(np.int32), M.data, M.shape[0])


def test_banded_with_holes_zeros_and_nonfinite_x(isb, oracle):
    rng = np.random.default_rng(SEED)
    n = 3000
    offs = [-700, -3, -1, 0, 2, 511]
    dead = rng.choice(n, 40, replace=False)                         # columns no stored entry reaches
    M = banded(n, offs, 0.9, rng, drop_cols=dead)
    A = from_csr(isb, M)
    assert A.format == "dia" and A.dia_offsets == offs
    assert M.nnz == A.nnz and np.count_nonzero(M.data == 0.0) > 0
    x = rng.standard_normal(n)
    x[dead[:20]] = np.nan                                           # reached only through clear (padded) slots
    x[dead[20:]] = np.inf
    live = np.setdiff1d(np.arange(n), dead)
    x[live[::97]] = np.inf                                          # reached through stored entries: Inf / NaN rows
    x[live[5::131]] = -np.inf
    y_csr, y_dia = both_formats(isb, lambda: A @ x)
    assert_bitwise(y_csr, y_dia)
    yo = oracle.csc_spmv(oracle.CSC.from_scipy(M), x)
    np.testing.assert_array_equal(y_dia, yo)                        # NaN == NaN here; finite values exact
    reached = np.zeros(n, bool)
    reached[M.indices] = True
    assert not reached[dead].any()
    assert np.isnan(y_dia).any() and np.isinf(y_dia).any() and np.isfinite(y_dia).sum() > n // 2


def test_eight_diagonals_dia_nine_csr(isb):
    rng = np.random.default_rng(SEED)
    n = 2000
    offs8 = [-300, -20, -2, -1, 0, 1, 5, 300]
    A8 = from_csr(isb, banded(n, offs8, 1.0, rng))
    assert A8.format == "dia" and A8.dia_offsets == offs8
    A9 = from_csr(isb, banded(n, offs8 + [600], 1.0, rng))
    assert A9.format == "csr" and A9.dia_offsets == []
    x = rng.standard_normal(n)
    for A in (A8, A9):
        y_csr, y_dia = both_formats(isb, lambda: A @ x)
        assert_bitwise(y_csr, y_dia)


def test_not_eligible_stays_csr(isb, oracle):
    rng = np.random.default_rng(SEED)
    M = sp.random(3000, 3000, density=0.002, random_state=5, format="csr", dtype=np.float64)
    assert isb.B200CSR.from_scipy(M).format == "csr"               # random sparse: many offsets
    R = sp.random(300, 500, density=0.01, random_state=6, format="csc", dtype=np.float64)
    assert isb.B200CSR.from_scipy(R).format == "csr"               # rectangular
    # a tridiagonal matrix with one row's columns stored out of order
    T = banded(1000, [-1, 0, 1], 1.0, rng)
    rp, ci, va = T.indptr.astype(np.int32), T.indices.astype(np.int32).copy(), T.data.copy()
    r = 500
    b, e = rp[r], rp[r + 1]
    ci[b:e], va[b:e] = ci[b:e][::-1].copy(), va[b:e][::-1].copy()
    A = isb.B200CSR.from_csr_slab(rp, ci, va, 1000)
    assert A.format == "csr"
    assert from_csr(isb, T).format == "dia"
    x = rng.standard_normal(1000)
    np.testing.assert_allclose(A @ x, T @ x, rtol=1e-14)


# ------------------------------------------------------------------ solvers: histories and x bitwise equal
def _no_persistent(isb):
    """64^3 = 2^18 rows would run cg! in the persistent small-operator kernel (CSR): switch it off."""
    ctx = isb.default_context()
    L = isb.lib()
    assert L.b200_ctx_set_option(ctx._h, b"cg_persistent", 0) == 0
    return lambda: L.b200_ctx_set_option(ctx._h, b"cg_persistent", 1)


@pytest.mark.parametrize("jacobi", [False, True])
def test_cg_bitwise_between_formats(isb, jacobi):
    ctx = isb.default_context()
    A = isb.B200CSR.laplacian(64, 3)
    assert A.format == "dia"
    n = A.m_local
    b = isb.DeviceArray.from_numpy(ctx, np.random.default_rng(SEED).standard_normal(n))
    restore = _no_persistent(isb)
    try:
        def run():
            Pl = isb.JacobiPrec(A.diag()) if jacobi else None
            x = isb.DeviceArray.zeros(ctx, n)
            x, h = isb.cg_(x, A, b, Pl=Pl, initially_zero=True, log=True, reltol=1e-8)
            return x.numpy(), np.asarray(h["resnorm"]), h.niters
        (xa, ha, na), (xb, hb, nb) = both_formats(isb, run)
    finally:
        restore()
    assert na == nb and na > 20
    assert_bitwise(ha, hb)
    assert_bitwise(xa, xb)


def test_cg_iterator_bitwise_between_formats(isb):
    ctx = isb.default_context()
    A = isb.B200CSR.laplacian(64, 3)
    n = A.m_local
    b = isb.DeviceArray.from_numpy(ctx, np.random.default_rng(SEED).standard_normal(n))
    restore = _no_persistent(isb)
    try:
        def run():
            x = isb.DeviceArray.zeros(ctx, n)
            it = isb.cg_iterator_(x, A, b, initially_zero=True, reltol=1e-8)
            res = np.concatenate([it.step(17), it.step(23)])
            out = it.x.numpy()
            it.close()
            return res, out
        (ra, xa), (rb, xb) = both_formats(isb, run)
    finally:
        restore()
    assert ra.size == 40
    assert_bitwise(ra, rb)
    assert_bitwise(xa, xb)


def test_minres_bitwise_between_formats(isb):
    ctx = isb.default_context()
    A = isb.B200CSR.laplacian(64, 3)
    n = A.m_local
    b = isb.DeviceArray.from_numpy(ctx, np.random.default_rng(SEED).standard_normal(n))

    def run():
        x = isb.DeviceArray.zeros(ctx, n)
        x, h = isb.minres_(x, A, b, initially_zero=True, log=True, maxiter=80)
        return x.numpy(), np.asarray(h["resnorm"])
    (xa, ha), (xb, hb) = both_formats(isb, run)
    assert ha.size > 20
    assert_bitwise(ha, hb)
    assert_bitwise(xa, xb)


def test_multi_gpu_operator_stays_csr():
    import os
    import socket
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip(f"needs 2 GPUs, {torch.cuda.device_count()} visible")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(root, "tests", "dia_dist_worker.py")]
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert out.returncode == 0 and "DIA_DIST_OK" in out.stdout, out.stdout[-4000:]
