"""The operator / preconditioner objects of the reference's duck-typed contract
(reference docs/src/getting_started.md:25-30, docs/src/preconditioning.md:5-15) on the device."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import check, lib
from .device import Context, DeviceArray, as_device_ptr, default_context, dtype_code


def _vp(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


class Identity:
    """No-op preconditioner, reference src/common.jl:28-32."""

    def _as_c(self, A):
        return _lib.Precond(_lib.PREC_IDENTITY, 0, None)


class JacobiPrec:
    """ldiv!(y, P, x) = y .= x ./ P.diagonal  (reference test/cg.jl:10-18).  `diagonal` may be a
    host array (uploaded once) or a DeviceArray."""

    def __init__(self, diagonal, ctx: Context | None = None):
        if isinstance(diagonal, DeviceArray):
            self.diagonal = diagonal
        else:
            self.diagonal = DeviceArray.from_numpy(ctx or default_context(), np.asarray(diagonal))

    def _as_c(self, A):
        if self.diagonal.dtype != A.dtype:
            raise TypeError("JacobiPrec diagonal eltype must match the operator")
        return _lib.Precond(_lib.PREC_JACOBI, 0, self.diagonal.ptr)

    def ldiv_(self, y: DeviceArray, x: DeviceArray):
        check(lib().b200_jacobi_ldiv(y.ctx._h, y.size, self.diagonal._p, x._p, y._p, y.code))
        return y


def precond_to_c(P, A):
    if P is None:
        return Identity()._as_c(A)
    if isinstance(P, FunctionPrec):        # B200_PREC_CALLBACK: `diag` carries the address of the b200_linop
        return _lib.Precond(_lib.PREC_CALLBACK, 0, C.cast(C.pointer(P.op._c), C.c_void_p))
    if hasattr(P, "_as_c"):
        return P._as_c(A)
    raise TypeError(f"unsupported preconditioner {type(P)}: the device path takes Identity() or JacobiPrec "
                    "(reference src/common.jl:28-32, test/cg.jl:14-18)")


class HaloPlan:
    """Host-side plan of the off-slab columns of a row-partitioned operator (multi-GPU).  Pure host
    code in the library; the exchange of the request lists goes through torch.distributed."""

    def __init__(self, rank: int, world: int, row_offsets):
        self.rank, self.world = rank, world
        self.row_offsets = np.ascontiguousarray(row_offsets, dtype=np.int64)
        assert self.row_offsets.shape == (world + 1,)
        self._h = C.c_void_p()
        check(lib().b200_halo_plan_create(rank, world, self.row_offsets.ctypes.data_as(C.POINTER(C.c_int64)),
                                          C.byref(self._h)))

    def scan_csr(self, rowptr: np.ndarray, colind: np.ndarray, base: int = 0):
        idx_bytes = rowptr.dtype.itemsize
        assert colind.dtype == rowptr.dtype and idx_bytes in (4, 8)
        m_local = int(self.row_offsets[self.rank + 1] - self.row_offsets[self.rank])
        check(lib().b200_halo_plan_scan(self._h, m_local, _vp(rowptr), _vp(colind), idx_bytes, base))
        return self

    def scan_laplacian(self, N: int, dims: int):
        check(lib().b200_halo_plan_scan_laplacian(self._h, N, dims))
        return self

    def recv_cols(self, owner: int) -> np.ndarray:
        n = lib().b200_halo_plan_recv_count(self._h, owner)
        out = np.empty(max(n, 0), dtype=np.int64)
        check(lib().b200_halo_plan_recv_cols(self._h, owner, _vp(out)))
        return out

    def set_send(self, peer: int, cols: np.ndarray):
        cols = np.ascontiguousarray(cols, dtype=np.int64)
        check(lib().b200_halo_plan_set_send(self._h, peer, _vp(cols), cols.size))

    def send_count(self, peer: int) -> int:
        return int(lib().b200_halo_plan_send_count(self._h, peer))

    def send_range(self, peer: int):
        """first local row when the rows `peer` asked for are one ascending contiguous range (then the CG update kernel
        stores them straight into the peer's halo), else None."""
        lo = C.c_int64(-1)
        r = int(lib().b200_halo_plan_send_range(self._h, peer, C.byref(lo)))
        if r < 0:
            raise ValueError("bad peer")
        return int(lo.value) if r == 1 else None

    @property
    def n_halo(self) -> int:
        return int(lib().b200_halo_plan_n_halo(self._h))

    def local_index(self, global_col: int) -> int:
        return int(lib().b200_halo_plan_local_index(self._h, global_col))

    def exchange(self):
        """every rank tells every owner which of its rows it needs (torch.distributed, any backend)."""
        import torch.distributed as dist
        mine = {o: self.recv_cols(o) for o in range(self.world) if o != self.rank}
        gathered = [None] * self.world
        dist.all_gather_object(gathered, mine)
        for peer in range(self.world):
            if peer != self.rank:
                self.set_send(peer, gathered[peer].get(self.rank, np.empty(0, dtype=np.int64)))
        return self

    def close(self):
        if self._h:
            lib().b200_halo_plan_destroy(self._h)
            self._h = C.c_void_p()


class B200CSR:
    """The operator A on the device (CSR int32, row slab).  Stands where the reference takes a
    SparseMatrixCSC: `mul!(y, A, x)`, `size(A, d)`, `eltype(A)` (SURVEY.md section 8b)."""

    def __init__(self, ctx: Context, handle):
        self.ctx, self._h = ctx, handle
        m, n, nnz, dt = C.c_int64(), C.c_int64(), C.c_int64(), C.c_int()
        rb, nh = C.c_int64(), C.c_int64()
        check(lib().b200_csr_info(handle, C.byref(m), C.byref(n), C.byref(nnz), C.byref(dt), C.byref(rb), C.byref(nh)))
        self.m_local, self.n_global, self.nnz, self.row_begin, self.n_halo = m.value, n.value, nnz.value, rb.value, nh.value
        self.dtype = np.dtype(np.float64 if dt.value == _lib.F64 else np.float32)
        self.code = dt.value
        # size(A, 1): row-partitioned (multi-GPU) operators are square; single-GPU ones may be rectangular (lsqr!/lsmr!)
        self.m_global = self.m_local if ctx.world == 1 else self.n_global
        self._adjoint = None

    # --- constructors -----------------------------------------------------------------------
    @classmethod
    def from_csc_arrays(cls, colptr, rowval, nzval, shape, base=0, ctx: Context | None = None):
        """from the three arrays of a SparseMatrixCSC{Tv,Ti} (base=1 for Julia's)."""
        ctx = ctx or default_context()
        colptr = np.ascontiguousarray(colptr)
        rowval = np.ascontiguousarray(rowval, dtype=colptr.dtype)
        nzval = np.ascontiguousarray(nzval)
        h = C.c_void_p()
        check(lib().b200_csr_from_csc(ctx._h, shape[0], shape[1], _vp(colptr), _vp(rowval), _vp(nzval),
                                      colptr.dtype.itemsize, dtype_code(nzval.dtype), base, C.byref(h)))
        return cls(ctx, h)

    @classmethod
    def from_scipy(cls, A, ctx: Context | None = None):
        """from any scipy.sparse matrix (converted to CSC = the reference's storage)."""
        A = A.tocsc()
        A.sort_indices()
        return cls.from_csc_arrays(A.indptr, A.indices, A.data, A.shape, 0, ctx)

    @classmethod
    def from_csr_slab(cls, rowptr, colind, vals, n_global, row_begin=0, base=0, plan: HaloPlan | None = None,
                      ctx: Context | None = None):
        ctx = ctx or default_context()
        rowptr = np.ascontiguousarray(rowptr)
        colind = np.ascontiguousarray(colind, dtype=rowptr.dtype)
        vals = np.ascontiguousarray(vals)
        h = C.c_void_p()
        check(lib().b200_csr_from_csr_slab(ctx._h, n_global, row_begin, rowptr.size - 1, _vp(rowptr), _vp(colind),
                                           _vp(vals), rowptr.dtype.itemsize, dtype_code(vals.dtype), base,
                                           plan._h if plan else None, C.byref(h)))
        return cls(ctx, h)

    @classmethod
    def laplacian(cls, N, dims, dtype=np.float64, row_begin=0, m_local=None, plan: HaloPlan | None = None,
                  ctx: Context | None = None):
        """laplace_matrix(T, N, dims) (reference test/laplace_matrix.jl) built on the device."""
        ctx = ctx or default_context()
        if m_local is None:
            m_local = N ** dims
        h = C.c_void_p()
        check(lib().b200_csr_laplacian(ctx._h, N, dims, dtype_code(dtype), row_begin, m_local,
                                       plan._h if plan else None, C.byref(h)))
        return cls(ctx, h)

    # --- reference operator contract ----------------------------------------------------------
    @property
    def shape(self):
        return (self.m_global, self.n_global)

    def adjoint(self) -> "B200CSR":
        """adjoint(A) as an operator of its own (what the reference stores as `adjoint(A)`, src/qmr.jl:54; used by
        mul!(y, A', x) in qmr!/lsqr!/lsmr!).  Built once on the device from the CSR of A and cached.  On multi-GPU
        contexts build it from the adjoint's own row slabs (from_csr_slab) and assign it with set_adjoint()."""
        if self._adjoint is None:
            h = C.c_void_p()
            check(lib().b200_csr_transpose(self.ctx._h, self._h, C.byref(h)))
            self._adjoint = B200CSR(self.ctx, h)
            self._adjoint._adjoint_of = self          # keeps A alive as long as A' is (not the other way round)
        return self._adjoint

    def set_adjoint(self, At: "B200CSR"):
        self._adjoint = At
        return self

    def set_adjoint_self(self):
        """for Hermitian operators: adjoint(A) is A (no second copy of the matrix)."""
        self._adjoint = self
        return self

    def size(self, d=None):
        return self.shape if d is None else self.shape[d - 1]

    def mul_(self, y, x):
        """mul!(y, A, x)."""
        if getattr(y, "shape", None) is not None and len(y.shape) == 2:
            check(lib().b200_spmm(self.ctx._h, self._h, as_device_ptr(x), x.shape[0], as_device_ptr(y), y.shape[0],
                                  y.shape[1]))
        else:
            check(lib().b200_spmv(self.ctx._h, self._h, as_device_ptr(x), as_device_ptr(y)))
        return y

    def __matmul__(self, x: np.ndarray) -> np.ndarray:
        """A * x with host arrays (convenience for tests)."""
        xd = DeviceArray.from_numpy(self.ctx, np.asarray(x, dtype=self.dtype))
        yd = DeviceArray(self.ctx, (self.m_local,) + tuple(xd.shape[1:]), self.dtype)
        self.mul_(yd, xd)
        return yd.numpy()

    @property
    def format(self) -> str:
        """"dia" if the SpMV streams the operator's offset-diagonal copy (spmv_format 0), else "csr"."""
        fmt = C.c_int()
        check(lib().b200_csr_format(self._h, C.byref(fmt), None, None))
        return "dia" if fmt.value == 1 else "csr"

    @property
    def dia_offsets(self) -> list:
        """the ascending col - row offsets of the DIA copy ([] for a CSR-only operator)."""
        nd = C.c_int()
        offs = (C.c_int64 * 8)()
        check(lib().b200_csr_format(self._h, None, C.byref(nd), offs))
        return [int(offs[d]) for d in range(nd.value)]

    def diag(self) -> DeviceArray:
        d = DeviceArray(self.ctx, self.m_local, self.dtype)
        check(lib().b200_csr_diag(self.ctx._h, self._h, d._p))
        return d

    def download(self):
        rowptr = np.empty(self.m_local + 1, dtype=np.int32)
        colind = np.empty(self.nnz, dtype=np.int32)
        vals = np.empty(self.nnz, dtype=self.dtype)
        check(lib().b200_csr_download(self.ctx._h, self._h, _vp(rowptr), _vp(colind), _vp(vals)))
        return rowptr, colind, vals

    def close(self):
        if getattr(self, "_adjoint", None) is not None and getattr(self._adjoint, "_adjoint_of", None) is self:
            self._adjoint.close()
        self._adjoint = None
        if self._h:
            lib().b200_csr_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class B200LinearOperator:
    """A matrix-free operator (or preconditioner) on device vectors: the reference's duck-typed contract
    `mul!(y, A, x)` / `size` / `eltype` (docs/src/getting_started.md:25-30; LinearMaps in test/cg.jl:71-77,
    test/lsqr.jl:36) carried through the C ABI as a `b200_linop` callback.

        mul(y, x)          enqueue y = A x on the context's stream; x, y are DeviceArray views (y never aliases x)
        adjoint_mul(y, x)  optional: y = A' x  (needed by qmr!/lsqr!/lsmr!)

    shape = (m, n) are the LOCAL lengths of y and x (on a single-GPU context also the global ones); on multi-GPU
    contexts pass `global_shape` and do the halo exchange inside `mul`."""

    def __init__(self, shape, dtype, mul, adjoint_mul=None, ctx: Context | None = None, global_shape=None):
        self.ctx = ctx or default_context()
        self.dtype = np.dtype(dtype)
        self.code = dtype_code(dtype)
        self.m_local, self.n_local = int(shape[0]), int(shape[1])
        gm, gn = global_shape if global_shape is not None else shape
        self.m_global, self.n_global = int(gm), int(gn)
        self._mul, self._adjoint_mul = mul, adjoint_mul
        self._exc = None
        self._adjoint = None
        self._cb = _lib.APPLY_FN(self._trampoline)            # keep the thunk alive as long as the operator
        self._c = _lib.LinOp(self._cb, None, self.m_local, self.n_local, self.n_global, self.m_global, self.code, 0)

    def _trampoline(self, user, x_ptr, y_ptr, stream):
        try:
            x = DeviceArray.view(self.ctx, x_ptr, self.n_local, self.dtype)
            y = DeviceArray.view(self.ctx, y_ptr, self.m_local, self.dtype)
            self._mul(y, x)
            return 0
        except BaseException as e:                            # never let an exception cross the C frames
            self._exc = e
            return 1

    def raise_pending(self):
        if self._exc is not None:
            e, self._exc = self._exc, None
            raise e

    @property
    def shape(self):
        return (self.m_global, self.n_global)

    def size(self, d=None):
        return self.shape if d is None else self.shape[d - 1]

    def mul_(self, y, x):
        self._mul(y, x)
        return y

    def adjoint(self) -> "B200LinearOperator":
        if self._adjoint is None:
            if self._adjoint_mul is None:
                raise TypeError("this operator has no adjoint_mul (needed by qmr!/lsqr!/lsmr!)")
            self._adjoint = B200LinearOperator((self.n_local, self.m_local), self.dtype, self._adjoint_mul, self._mul,
                                               self.ctx, (self.n_global, self.m_global))
            self._adjoint._adjoint = self
        return self._adjoint

    @classmethod
    def from_csr(cls, A: "B200CSR"):
        """a B200CSR seen through the callback interface: the descriptor's `apply` is the library's own SpMV thunk
        (b200_csr_as_linop), so no Python runs inside the iteration; `mul_` from Python still works."""
        n_loc = A.n_global if A.ctx.world == 1 else A.m_local
        op = cls((A.m_local, n_loc), A.dtype, lambda y, x: A.mul_(y, x),
                 (lambda y, x: A.adjoint().mul_(y, x)), A.ctx, A.shape)
        op._csr = A                                            # the descriptor points at the CSR handle
        check(lib().b200_csr_as_linop(A._h, C.byref(op._c)))
        return op


class FunctionPrec:
    """A preconditioner given as a function: ldiv(y, x) enqueues y = P \\ x on device vectors
    (`ldiv!(y, P, x)`, docs/src/preconditioning.md:5-15)."""

    def __init__(self, n, dtype, ldiv, ctx: Context | None = None):
        self.op = B200LinearOperator((n, n), dtype, ldiv, None, ctx)
