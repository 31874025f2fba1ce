"""ctypes binding of libb200krylov.so (the C ABI declared in include/b200krylov.h).

There is no fallback: if the shared library is missing or a call fails, this raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libb200krylov.so")

F64, F32 = 0, 1
ORTH_MGS, ORTH_CGS, ORTH_DGKS = 0, 1, 2
PREC_IDENTITY, PREC_JACOBI, PREC_CALLBACK = 0, 1, 2
ERR_INVALID = -1
ERR_BREAKDOWN = -5
ERR_CALLBACK = -7


class B200Error(RuntimeError):
    pass


class Precond(C.Structure):
    _fields_ = [("kind", C.c_int32), ("reserved", C.c_int32), ("diag", C.c_void_p)]


class Result(C.Structure):
    _fields_ = [("iters", C.c_int64), ("mvps", C.c_int64), ("isconverged", C.c_int32), ("status", C.c_int32),
                ("tol", C.c_double), ("residual", C.c_double), ("n_resnorm", C.c_int64)]


class CgOpts(C.Structure):
    _fields_ = [("abstol", C.c_double), ("reltol", C.c_double), ("maxiter", C.c_int64),
                ("initially_zero", C.c_int32), ("check_every", C.c_int32), ("Pl", Precond),
                ("fixed_iterations", C.c_int32), ("variant", C.c_int32)]


class GmresOpts(C.Structure):
    _fields_ = [("abstol", C.c_double), ("reltol", C.c_double), ("maxiter", C.c_int64), ("restart", C.c_int32),
                ("initially_zero", C.c_int32), ("orth_meth", C.c_int32), ("reserved", C.c_int32),
                ("Pl", Precond), ("Pr", Precond)]


class MinresOpts(C.Structure):
    _fields_ = [("abstol", C.c_double), ("reltol", C.c_double), ("maxiter", C.c_int64),
                ("initially_zero", C.c_int32), ("skew_hermitian", C.c_int32)]


class BicgstablOpts(C.Structure):
    _fields_ = [("abstol", C.c_double), ("reltol", C.c_double), ("max_mv_products", C.c_int64), ("l", C.c_int32),
                ("initial_zero", C.c_int32), ("Pl", Precond), ("r_shadow", C.c_void_p)]


class QmrOpts(C.Structure):
    _fields_ = [("abstol", C.c_double), ("reltol", C.c_double), ("maxiter", C.c_int64),
                ("initially_zero", C.c_int32), ("check_every", C.c_int32)]


class LsqOpts(C.Structure):
    _fields_ = [("damp", C.c_double), ("atol", C.c_double), ("btol", C.c_double), ("conlim", C.c_double),
                ("maxiter", C.c_int64), ("check_every", C.c_int32), ("reserved", C.c_int32)]


class LsqResult(C.Structure):
    _fields_ = [("iters", C.c_int64), ("mvps", C.c_int64), ("mtvps", C.c_int64), ("isconverged", C.c_int32),
                ("istop", C.c_int32), ("status", C.c_int32), ("reserved", C.c_int32), ("n_hist", C.c_int64),
                ("hist_stride", C.c_int64), ("atol", C.c_double), ("btol", C.c_double), ("ctol", C.c_double)]


class IdrsOpts(C.Structure):
    _fields_ = [("abstol", C.c_double), ("reltol", C.c_double), ("maxiter", C.c_int64), ("s", C.c_int32),
                ("smoothing", C.c_int32), ("Pl", Precond), ("P", C.c_void_p), ("ldp", C.c_int64),
                ("check_every", C.c_int32), ("reserved", C.c_int32)]


APPLY_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p)   # b200_apply_fn


class LinOp(C.Structure):
    _fields_ = [("apply", APPLY_FN), ("user", C.c_void_p), ("m_local", C.c_int64), ("n_local", C.c_int64),
                ("n_global", C.c_int64), ("m_global", C.c_int64), ("dtype", C.c_int32), ("reserved", C.c_int32)]


class SvdlOpts(C.Structure):
    _fields_ = [("nsv", C.c_int32), ("k", C.c_int32), ("j", C.c_int32), ("method", C.c_int32), ("maxiter", C.c_int64),
                ("tol", C.c_double), ("reltol", C.c_double), ("dolock", C.c_int32), ("reserved", C.c_int32)]


class SvdlResult(C.Structure):
    _fields_ = [("iters", C.c_int64), ("mvps", C.c_int64), ("mtvps", C.c_int64), ("isconverged", C.c_int32),
                ("k", C.c_int32), ("beta", C.c_double), ("tol", C.c_double)]


class PowmOpts(C.Structure):
    _fields_ = [("tol", C.c_double), ("maxiter", C.c_int64), ("shift", C.c_double), ("inverse", C.c_int32),
                ("check_every", C.c_int32)]


class LobpcgOpts(C.Structure):
    _fields_ = [("tol", C.c_double), ("maxiter", C.c_int64), ("largest", C.c_int32), ("blocksize", C.c_int32),
                ("P", Precond), ("fixed_iterations", C.c_int32), ("reserved", C.c_int32),
                ("trace_resnorm", C.c_void_p), ("trace_ritz", C.c_void_p), ("trace_cap", C.c_int64)]


class LobpcgResult(C.Structure):
    _fields_ = [("iterations", C.c_int64), ("converged", C.c_int32), ("status", C.c_int32)]


_P = C.c_void_p
_I64 = C.c_int64
_INT = C.c_int
_DBL = C.c_double

# name -> (restype, argtypes).  Every symbol include/b200krylov.h declares appears here
# (tests/test_abi.py cross-checks this table against the header).
SIGNATURES = {
    "b200_version": (_INT, []),
    "b200_last_error": (C.c_char_p, []),
    "b200_device_count": (_INT, [C.POINTER(_INT)]),
    "b200_ctx_create": (_INT, [_INT, C.POINTER(_P)]),
    "b200_nccl_unique_id": (_INT, [_P]),
    "b200_ctx_create_dist": (_INT, [_INT, _INT, _INT, _P, C.POINTER(_P)]),
    "b200_ctx_destroy": (_INT, [_P]),
    "b200_ctx_set_stream": (_INT, [_P, _P]),
    "b200_ctx_sync": (_INT, [_P]),
    "b200_ctx_info": (_INT, [_P, C.POINTER(_INT), C.POINTER(_INT), C.POINTER(_INT), C.POINTER(_INT)]),
    "b200_ctx_launch_count": (_I64, [_P]),
    "b200_ctx_timer_start": (_INT, [_P]),
    "b200_ctx_timer_stop": (_INT, [_P, C.POINTER(C.c_float)]),
    "b200_ctx_set_option": (_INT, [_P, C.c_char_p, _I64]),
    "b200_ctx_get_option": (_INT, [_P, C.c_char_p, C.POINTER(_I64)]),
    "b200_ctx_profile_enable": (_INT, [_P, _INT]),
    "b200_ctx_profile_read": (_INT, [_P, _INT, C.POINTER(_DBL), C.POINTER(_I64), _INT]),
    "b200_ctx_allreduce_f64": (_INT, [_P, C.POINTER(_DBL), _INT, _INT]),
    "b200_ctx_barrier": (_INT, [_P]),
    "b200_malloc": (_INT, [_P, C.c_size_t, C.POINTER(_P)]),
    "b200_free": (_INT, [_P, _P]),
    "b200_upload": (_INT, [_P, _P, _P, C.c_size_t]),
    "b200_download": (_INT, [_P, _P, _P, C.c_size_t]),
    "b200_host_alloc_pinned": (_INT, [C.c_size_t, C.POINTER(_P)]),
    "b200_host_free_pinned": (_INT, [_P]),
    "b200_csr_from_csc": (_INT, [_P, _I64, _I64, _P, _P, _P, _INT, _INT, _INT, C.POINTER(_P)]),
    "b200_csr_from_csr_slab": (_INT, [_P, _I64, _I64, _I64, _P, _P, _P, _INT, _INT, _INT, _P, C.POINTER(_P)]),
    "b200_csr_laplacian": (_INT, [_P, _I64, _INT, _INT, _I64, _I64, _P, C.POINTER(_P)]),
    "b200_csr_destroy": (_INT, [_P]),
    "b200_csr_info": (_INT, [_P, C.POINTER(_I64), C.POINTER(_I64), C.POINTER(_I64), C.POINTER(_INT),
                             C.POINTER(_I64), C.POINTER(_I64)]),
    "b200_csr_transpose": (_INT, [_P, _P, C.POINTER(_P)]),
    "b200_csr_format": (_INT, [_P, C.POINTER(_INT), C.POINTER(_INT), C.POINTER(_I64)]),
    "b200_csr_diag": (_INT, [_P, _P, _P]),
    "b200_csr_download": (_INT, [_P, _P, _P, _P, _P]),
    "b200_halo_plan_create": (_INT, [_INT, _INT, C.POINTER(_I64), C.POINTER(_P)]),
    "b200_halo_plan_scan": (_INT, [_P, _I64, _P, _P, _INT, _INT]),
    "b200_halo_plan_scan_laplacian": (_INT, [_P, _I64, _INT]),
    "b200_halo_plan_recv_count": (_I64, [_P, _INT]),
    "b200_halo_plan_recv_cols": (_INT, [_P, _INT, _P]),
    "b200_halo_plan_set_send": (_INT, [_P, _INT, _P, _I64]),
    "b200_halo_plan_send_count": (_I64, [_P, _INT]),
    "b200_halo_plan_send_range": (_INT, [_P, _INT, C.POINTER(_I64)]),
    "b200_halo_plan_n_halo": (_I64, [_P]),
    "b200_halo_plan_local_index": (_I64, [_P, _I64]),
    "b200_halo_plan_destroy": (_INT, [_P]),
    "b200_gen_laplace_nnz": (_I64, [_I64, _INT, _I64, _I64]),
    "b200_gen_laplace_csc_i64": (_I64, [_I64, _INT, _INT, _P, _P, _P]),
    "b200_gen_advection_csc_i64": (_I64, [_I64, _DBL, _INT, _P, _P, _P, _P]),
    "b200_gen_laplace_csr_slab_i32": (_I64, [_I64, _INT, _I64, _I64, _P, _P, _P]),
    "b200_mm_info": (_INT, [C.c_char_p, C.POINTER(_I64), C.POINTER(_I64), C.POINTER(_I64), C.POINTER(_INT),
                            C.POINTER(_INT)]),
    "b200_mm_read_csc_i64": (_INT, [C.c_char_p, _INT, _I64, _P, _P, _P]),
    "b200_spmv": (_INT, [_P, _P, _P, _P]),
    "b200_spmm": (_INT, [_P, _P, _P, _I64, _P, _I64, _INT]),
    "b200_dot": (_INT, [_P, _I64, _P, _P, _INT, C.POINTER(_DBL)]),
    "b200_nrm2": (_INT, [_P, _I64, _P, _INT, C.POINTER(_DBL)]),
    "b200_axpby": (_INT, [_P, _I64, _DBL, _P, _DBL, _P, _INT]),
    "b200_scal": (_INT, [_P, _I64, _DBL, _P, _INT]),
    "b200_copy": (_INT, [_P, _I64, _P, _P, _INT]),
    "b200_fill": (_INT, [_P, _I64, _DBL, _P, _INT]),
    "b200_jacobi_ldiv": (_INT, [_P, _I64, _P, _P, _P, _INT]),
    "b200_orthogonalize_and_normalize": (_INT, [_P, _I64, _P, _I64, _INT, _P, _P, _INT, _INT, C.POINTER(_DBL)]),
    "b200_hessenberg_ldiv": (_INT, [_P, _P, _INT, _INT, _P]),
    "b200_cg_solve": (_INT, [_P, _P, _P, _P, C.POINTER(CgOpts), C.POINTER(Result), _P, _I64]),
    "b200_cg_solve_host": (_INT, [_P, _P, _P, _P, C.POINTER(CgOpts), C.POINTER(Result), _P, _I64]),
    "b200_cg_iter_create": (_INT, [_P, _P, _P, _P, C.POINTER(CgOpts), _P, _P, _P, C.POINTER(_P)]),
    "b200_cg_iter_next": (_INT, [_P, _I64, C.POINTER(Result), _P, _I64]),
    "b200_cg_iter_destroy": (_INT, [_P]),
    "b200_chebyshev_solve": (_INT, [_P, _P, _P, _P, _DBL, _DBL, C.POINTER(CgOpts), C.POINTER(Result), _P, _I64]),
    "b200_chebyshev_solve_op": (_INT, [_P, C.POINTER(LinOp), _P, _P, _DBL, _DBL, C.POINTER(CgOpts), C.POINTER(Result), _P, _I64]),
    "b200_gmres_solve": (_INT, [_P, _P, _P, _P, C.POINTER(GmresOpts), C.POINTER(Result), _P, _I64]),
    "b200_gmres_solve_op": (_INT, [_P, C.POINTER(LinOp), _P, _P, C.POINTER(GmresOpts), C.POINTER(Result), _P, _I64]),
    "b200_gmres_iter_create": (_INT, [_P, _P, C.POINTER(LinOp), _P, _P, C.POINTER(GmresOpts), C.POINTER(_P)]),
    "b200_minres_iter_create": (_INT, [_P, _P, C.POINTER(LinOp), _P, _P, C.POINTER(MinresOpts), C.POINTER(_P)]),
    "b200_bicgstabl_iter_create": (_INT, [_P, _P, C.POINTER(LinOp), _P, _P, C.POINTER(BicgstablOpts), C.POINTER(_P)]),
    "b200_cg_iter_create_op": (_INT, [_P, _P, C.POINTER(LinOp), _P, _P, C.POINTER(CgOpts), C.POINTER(_P)]),
    "b200_iter_next": (_INT, [_P, _I64, C.POINTER(Result), _P, _I64]),
    "b200_iter_destroy": (_INT, [_P]),
    "b200_minres_solve": (_INT, [_P, _P, _P, _P, C.POINTER(MinresOpts), C.POINTER(Result), _P, _I64]),
    "b200_minres_solve_op": (_INT, [_P, C.POINTER(LinOp), _P, _P, C.POINTER(MinresOpts), C.POINTER(Result), _P, _I64]),
    "b200_bicgstabl_solve": (_INT, [_P, _P, _P, _P, C.POINTER(BicgstablOpts), C.POINTER(Result), _P, _I64]),
    "b200_bicgstabl_solve_op": (_INT, [_P, C.POINTER(LinOp), _P, _P, C.POINTER(BicgstablOpts), C.POINTER(Result), _P, _I64]),
    "b200_qmr_solve": (_INT, [_P, _P, _P, _P, _P, C.POINTER(QmrOpts), C.POINTER(Result), _P, _I64]),
    "b200_lsqr_solve": (_INT, [_P, _P, _P, _P, _P, C.POINTER(LsqOpts), C.POINTER(LsqResult), _P, _I64]),
    "b200_lsmr_solve": (_INT, [_P, _P, _P, _P, _P, C.POINTER(LsqOpts), C.POINTER(LsqResult), _P, _I64]),
    "b200_idrs_solve": (_INT, [_P, _P, _P, _P, C.POINTER(IdrsOpts), C.POINTER(Result), _P, _I64]),
    "b200_cg_solve_op": (_INT, [_P, C.POINTER(LinOp), C.POINTER(LinOp), _P, _P, C.POINTER(CgOpts), C.POINTER(Result), _P,
                                _I64]),
    "b200_qmr_solve_op": (_INT, [_P, C.POINTER(LinOp), C.POINTER(LinOp), _P, _P, C.POINTER(QmrOpts), C.POINTER(Result),
                                 _P, _I64]),
    "b200_lsqr_solve_op": (_INT, [_P, C.POINTER(LinOp), C.POINTER(LinOp), _P, _P, C.POINTER(LsqOpts),
                                  C.POINTER(LsqResult), _P, _I64]),
    "b200_lsmr_solve_op": (_INT, [_P, C.POINTER(LinOp), C.POINTER(LinOp), _P, _P, C.POINTER(LsqOpts),
                                  C.POINTER(LsqResult), _P, _I64]),
    "b200_idrs_solve_op": (_INT, [_P, C.POINTER(LinOp), _P, _P, C.POINTER(IdrsOpts), C.POINTER(Result), _P, _I64]),
    "b200_lobpcg_solve": (_INT, [_P, _P, _P, _I64, C.POINTER(LobpcgOpts), C.POINTER(LobpcgResult), _P, _P]),
    "b200_svdl": (_INT, [_P, _P, _P, _P, C.POINTER(SvdlOpts), C.POINTER(SvdlResult), _P, _P, _I64, _P, _I64, _P, _P, _P, _P,
                         _P]),
    "b200_svdl_op": (_INT, [_P, C.POINTER(LinOp), C.POINTER(LinOp), _P, C.POINTER(SvdlOpts), C.POINTER(SvdlResult), _P, _P,
                            _I64, _P, _I64, _P, _P, _P, _P, _P]),
    "b200_lobpcg_constraint_create": (_INT, [_P, _I64, _P, _I64, _INT, _INT, _INT, C.POINTER(_P)]),
    "b200_lobpcg_constraint_append": (_INT, [_P, _P, _P, _I64, _INT]),
    "b200_lobpcg_constraint_apply": (_INT, [_P, _P, _P, _I64, _INT]),
    "b200_lobpcg_constraint_info": (_INT, [_P, C.POINTER(_INT), C.POINTER(_INT)]),
    "b200_lobpcg_constraint_destroy": (_INT, [_P]),
    "b200_lobpcg_solve_constrained": (_INT, [_P, _P, _P, _I64, C.POINTER(LobpcgOpts), _P, C.POINTER(LobpcgResult), _P,
                                             _P]),
    "b200_csr_as_linop": (_INT, [_P, C.POINTER(LinOp)]),
    "b200_stationary": (_INT, [_P, _P, _P, _P, _INT, _DBL, _I64]),
    "b200_powm": (_INT, [_P, _P, C.POINTER(LinOp), _P, C.POINTER(PowmOpts), C.POINTER(Result), C.POINTER(C.c_double), _P, _I64]),
    "b200_lobpcg_solve_op": (_INT, [_P, C.POINTER(LinOp), C.POINTER(LinOp), _P, _I64, C.POINTER(LobpcgOpts), _P,
                                    C.POINTER(LobpcgResult), _P, _P]),
    "b200_lobpcg_constraint_create_b": (_INT, [_P, C.POINTER(LinOp), _I64, _P, _I64, _INT, _INT, _INT, C.POINTER(_P)]),
    "b200_dense_sygv_host": (_INT, [_INT, _P, _P, _P, _P]),
    "b200_debug_lobpcg_gram_rr": (_INT, [_P, _P, _I64, _INT, _P]),
}

_lib = None


def lib():
    """Load libb200krylov.so (built in-tree by `__graft_entry__.build()` / csrc/Makefile)."""
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            raise B200Error(f"{_SO} is missing: build it with `make -C iterativesolvers.jl_b200/csrc` "
                            "(there is no CPU or PyTorch fallback)")
        # libb200krylov.so needs libnccl.so.2.  If PyTorch's bundled NCCL exists, load THAT copy first so
        # that a later `import torch` (which needs its own, newer NCCL under the same soname) still works.
        import sysconfig
        bundled = os.path.join(sysconfig.get_paths()["purelib"], "nvidia", "nccl", "lib", "libnccl.so.2")
        if os.path.exists(bundled):
            C.CDLL(bundled, mode=C.RTLD_GLOBAL)
        _lib = C.CDLL(_SO)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(_lib, name)     # AttributeError if the library does not export it
            fn.restype = res
            fn.argtypes = args
    return _lib


def check(status: int):
    if status != 0:
        msg = lib().b200_last_error().decode(errors="replace")
        raise B200Error(f"libb200krylov error {status}: {msg}")
    return status
