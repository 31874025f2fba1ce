/*
 * b200krylov.h -- C ABI of the B200-native Krylov inner-loop engine (libb200krylov.so).
 *
 * This is the drop-in boundary behind IterativeSolvers.jl's cg!/gmres!/minres!/bicgstabl!/lobpcg!
 * entry points and its operator/preconditioner contract (mul!, ldiv!).  The reference has no FFI of
 * its own (it is pure Julia, duck-typed: docs/src/getting_started.md:25-30,
 * docs/src/preconditioning.md:5-15); every entry point below names the reference interface it
 * replaces (paths relative to the reference checkout).  INTEGRATION.md shows the Julia `ccall`
 * shim a maintainer would add.
 *
 * Conventions
 *   - extern "C", opaque handles, plain pointers and sizes; no C++ / torch types.
 *   - every function returns 0 on success, <0 on error (b200_last_error() has the message);
 *     nothing throws, nothing calls exit().  Non-convergence is NOT an error (reference
 *     src/cg.jl:238): it is reported through b200_result.isconverged.
 *   - all device work is ordered on the context's CUDA stream; one host thread per context.
 *   - `dtype`: B200_F64 or B200_F32 (the configs of BASELINE.json need no complex types).
 *   - device pointers are raw CUDA device addresses (cudaMalloc / torch tensor .data_ptr()).
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *     B200_ERR_CUDA.
 */
#ifndef B200KRYLOV_H
#define B200KRYLOV_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_API __attribute__((visibility("default")))

enum { B200_F64 = 0, B200_F32 = 1 };
/* storage the SpMV of an operator streams (b200_csr_format) */
enum { B200_FORMAT_CSR = 0, B200_FORMAT_DIA = 1 };

enum {
  B200_OK = 0,
  B200_ERR_INVALID = -1, /* bad argument (reference: throw("...") strings, src/lobpcg.jl:833-834) */
  B200_ERR_CUDA = -2,    /* CUDA runtime / launch failure, or no device                           */
  B200_ERR_NCCL = -3,
  B200_ERR_ALLOC = -4,
  B200_ERR_BREAKDOWN = -5, /* LAPACK-style failure: PosDefException (src/lobpcg.jl:380),
                              SingularException (src/bicgstabl.jl:123)                            */
  B200_ERR_UNSUPPORTED = -6,
  B200_ERR_CALLBACK = -7  /* a b200_linop callback returned non-zero                                   */
};

/* orth_meth of gmres! (reference src/orthogonalize.jl:5-8) */
enum { B200_ORTH_MGS = 0, B200_ORTH_CGS = 1, B200_ORTH_DGKS = 2 };

/* Pl / Pr kinds.  Identity() = reference src/common.jl:28-32; JACOBI = the diagonal
 * preconditioner idiom of reference test/cg.jl:14-18 (ldiv!(y,P,x) = y .= x ./ P.diagonal). */
enum { B200_PREC_IDENTITY = 0, B200_PREC_JACOBI = 1,
       B200_PREC_CALLBACK = 2 /* `diag` points to a b200_linop whose apply is ldiv!(y, Pl, x); accepted by
                                 the chebyshev / gmres / bicgstabl / idrs / lobpcg entry points (b200_cg_solve_op takes its callback as an
                                 argument as well) */ };

typedef struct b200_ctx b200_ctx;   /* device + stream (+ NCCL communicator)                     */
typedef struct b200_csr b200_csr;   /* the operator A: CSR int32 on device, row-partitioned       */
typedef struct b200_halo_plan b200_halo_plan; /* host-side plan of the off-slab columns           */

typedef struct {
  int32_t kind;       /* B200_PREC_*                                                              */
  int32_t reserved;
  const void *diag;   /* JACOBI: device pointer to the (local) diagonal, dtype of the operator    */
} b200_precond;

/* What the reference returns in ConvergenceHistory (src/history.jl:54-66) + solver exit state. */
typedef struct {
  int64_t iters;        /* niters(history)                                                        */
  int64_t mvps;         /* history.mvps  (quirks of SURVEY.md section 9 reproduced)               */
  int32_t isconverged;  /* converged(iterable) at exit                                            */
  int32_t status;       /* 0, or B200_ERR_BREAKDOWN if a NaN/breakdown was detected
                           (b200_cg_iter_next: 1 once done(it) holds).
                           DEVIATION from the reference, deliberate: a NaN residual norm (initial or
                           recurrence) ENDS the solve at that iteration with this status.  The
                           reference's done() (src/cg.jl:36: iteration >= maxiter || residual <= tol)
                           is false for NaN, so it keeps multiplying NaNs until maxiter (default
                           size(A,2) iterations); iters / mvps / the :resnorm length therefore differ
                           from the reference after a breakdown -- x is NaN in both.  Fixed-horizon
                           runs (opts.fixed_iterations) never stop early.                          */
  double tol;           /* max(reltol*||r0||, abstol)                                             */
  double residual;      /* iterable.residual at exit                                              */
  int64_t n_resnorm;    /* number of :resnorm entries written to the caller's history buffer      */
} b200_result;

/* ---------------------------------------------------------------- library / context */
B200_API int b200_version(void);
B200_API const char *b200_last_error(void);
B200_API int b200_device_count(int *count);

/* One context per (process, GPU).  world==1: no communicator. */
B200_API int b200_ctx_create(int device, b200_ctx **out);
/* Multi-GPU: one process per GPU; `nccl_id` = the 128-byte ncclUniqueId made by rank 0 with
 * b200_nccl_unique_id() and broadcast by the host program (torch.distributed / MPI / Julia
 * Distributed).  Row slabs of A and of every vector live on their owning rank. */
B200_API int b200_nccl_unique_id(void *out128);
B200_API int b200_ctx_create_dist(int device, int rank, int world, const void *nccl_id128, b200_ctx **out);
B200_API int b200_ctx_destroy(b200_ctx *ctx);
B200_API int b200_ctx_set_stream(b200_ctx *ctx, void *cuda_stream); /* borrow the caller's stream */
B200_API int b200_ctx_sync(b200_ctx *ctx);
B200_API int b200_ctx_info(const b200_ctx *ctx, int *device, int *rank, int *world, int *sm_count);
/* number of kernels this library has launched on the context since creation (bench evidence) */
B200_API int64_t b200_ctx_launch_count(const b200_ctx *ctx);
/* CUDA-event timing on the context's stream (ms between the two marks) */
B200_API int b200_ctx_timer_start(b200_ctx *ctx);
B200_API int b200_ctx_timer_stop(b200_ctx *ctx, float *ms);
/* Per-kernel-class timing inside the solvers: when enabled, the engines bracket each hot kernel
 * launch with CUDA events on the context's stream (slot 0: SpMV-class kernel, 1: vector update with
 * reduction, 2: vector update without reduction, 3: other).  read() synchronises and returns the
 * accumulated milliseconds and launch counts per slot since the last reset. */
B200_API int b200_ctx_profile_enable(b200_ctx *ctx, int on);
B200_API int b200_ctx_profile_read(b200_ctx *ctx, int slot, double *total_ms, int64_t *launches, int reset);
/* Tuning knobs (do not change results beyond floating-point summation order):
 *   "spmv_kernel": 0 = auto, 1 = sub-warp-per-row kernel, 2 = TMA-streamed kernel (when the tiles fit)
 *   "spmv_format": 0 (default) = operators that carry an offset-diagonal copy (b200_csr_format) stream it in the SpMV
 *           of mul!, cg! and minres! (bitwise the same results as the CSR: same row sums, same order); 1 = always the
 *           CSR.  Read at every launch, so one process can compare both on the same operator.
 *   "snake": 1 (default) = consecutive hot kernels of a solver sweep the rows in alternating directions so
 *           that each starts on the data the previous one touched last (L2 reuse); 0 = always ascending
 *   "orth_fused": 1 (default) = orthogonalize_and_normalize! (CGS / DGKS) is ONE cooperative launch (dots, update, norm,
 *           DGKS re-orthogonalisation rounds and the scaling separated by grid-wide barriers) and gmres! keeps H, the
 *           residual recurrence and the stopping test on the device, enqueueing a whole restart cycle per host
 *           synchronisation (single-GPU contexts); 0 = three kernels per orthogonalisation, host-side recurrences
 *   "pdl": 1 = the kernels of a cg! iteration are chained with programmatic dependent launch (griddepcontrol): the
 *           next kernel's blocks are resident when the previous one ends; 0 (default) = plain stream order, which
 *           measured faster on B200 with this driver (560 vs 520 iterations/s, 512^3 on 2 GPUs)
 *   "cg_persistent": 1 (default) = cg! on single-GPU operators of at most 2^18 rows runs its whole loop in ONE persistent
 *           cooperative kernel (grid-wide barriers between the phases of an iteration instead of three launches; same
 *           recurrence, same operation order); 0 = the streaming three-kernel iteration at every size
 *   "fold_push": 1 (default) = multi-GPU peer-memory cg! with Identity: the kernel that updates r stores r's boundary rows
 *           into the neighbours' halo segments itself and its finishing block raises the halo flags (one launch less
 *           per iteration; needs one contiguous row range per neighbour); 0 = separate push kernel
 *   "comm": 0 = auto, 1 = NCCL collectives, 2 = NVLink peer-memory collectives fused into the kernels
 *           (multi-GPU contexts; get "peer_ok" tells whether the peer buffers could be mapped)
 *   "lobpcg_mma": 1 (default) = fp32 LOBPCG blocks run the update and the Gram products as 3xTF32 tensor-core
 *           MMAs (fp32-level products, fp32 accumulate), the eight Rayleigh-Ritz Gram products of a step as
 *           tcgen05.mma with TMEM accumulators; 2 = the same with the legacy mma.sync Gram kernel;
 *           0 = CUDA-core kernels (always used for fp64) */
B200_API int b200_ctx_set_option(b200_ctx *ctx, const char *name, int64_t value);
B200_API int b200_ctx_get_option(const b200_ctx *ctx, const char *name, int64_t *value);
/* sum over ranks (no-op for world==1); used by hosts for max/sum of small host scalars */
B200_API int b200_ctx_allreduce_f64(b200_ctx *ctx, double *host_inout, int count, int op_max);
B200_API int b200_ctx_barrier(b200_ctx *ctx);

/* ---------------------------------------------------------------- device memory (similar / copyto!) */
B200_API int b200_malloc(b200_ctx *ctx, size_t bytes, void **dptr);
B200_API int b200_free(b200_ctx *ctx, void *dptr);
B200_API int b200_upload(b200_ctx *ctx, void *dst_dev, const void *src_host, size_t bytes);
B200_API int b200_download(b200_ctx *ctx, void *dst_host, const void *src_dev, size_t bytes);
B200_API int b200_host_alloc_pinned(size_t bytes, void **hptr);
B200_API int b200_host_free_pinned(void *hptr);

/* ---------------------------------------------------------------- the operator A
 * replaces: A::SparseMatrixCSC as used by mul!(y, A, x) at reference src/cg.jl:54,137,
 * src/gmres.jl:245,287, src/minres.jl:61,104, src/bicgstabl.jl:49,97,107, src/lobpcg.jl:125,129.
 */
/* From the three arrays of a host SparseMatrixCSC{Tv,Ti} (A.colptr, A.rowval, A.nzval;
 * idx_bytes = 8 for Int64 / 4 for Int32; base = 1 for Julia).  Single-GPU contexts only.
 * Uploads, transposes to CSR on the device, sorts columns inside each row. */
B200_API int b200_csr_from_csc(b200_ctx *ctx, int64_t m, int64_t n, const void *colptr, const void *rowval,
                               const void *nzval, int idx_bytes, int dtype, int base, b200_csr **out);
/* From a host CSR row slab: rows [row_begin, row_begin+m_local) of an n_global x n_global operator,
 * column indices GLOBAL.  world==1: row_begin=0, m_local=n_global, plan=NULL.
 * world>1: `plan` carries the halo exchange lists (see below). */
B200_API int b200_csr_from_csr_slab(b200_ctx *ctx, int64_t n_global, int64_t row_begin, int64_t m_local,
                                    const void *rowptr, const void *colind, const void *vals, int idx_bytes,
                                    int dtype, int base, const b200_halo_plan *plan, b200_csr **out);
/* laplace_matrix(T, N, dims) (reference test/laplace_matrix.jl:1-12) rows [row_begin,row_begin+m_local)
 * built directly on the device (bench input for sizes whose host copy would not fit the timed path). */
B200_API int b200_csr_laplacian(b200_ctx *ctx, int64_t N, int dims, int dtype, int64_t row_begin, int64_t m_local,
                                const b200_halo_plan *plan, b200_csr **out);
B200_API int b200_csr_destroy(b200_csr *A);
/* size(A,1) local, size(A,2) global, nnz local, eltype */
B200_API int b200_csr_info(const b200_csr *A, int64_t *m_local, int64_t *n_global, int64_t *nnz_local, int *dtype,
                           int64_t *row_begin, int64_t *n_halo);
/* Storage of the operator's SpMV under spmv_format 0.  Square single-GPU operators whose nonzeros lie on at most 8
 * diagonals (col - row offsets), and whose offset-diagonal (DIA) copy -- one value array per diagonal and a presence
 * byte per row -- is at most 0.8x the CSR bytes, get that copy at construction: *format = B200_FORMAT_DIA, *ndiag the
 * number of diagonals and offsets[0..ndiag) (room for 8) the ascending offsets.  Otherwise B200_FORMAT_CSR, ndiag 0.
 * Any output pointer may be NULL. */
B200_API int b200_csr_format(const b200_csr *A, int *format, int *ndiag, int64_t *offsets);
/* adjoint(A) as an operator (reference: `adjoint(A)` stored by LanczosDecomp src/qmr.jl:54 and used by
 * mul!(y, A', x) at src/qmr.jl:76, src/lsqr.jl:132,172, src/lsmr.jl:118,172).  Built on the device from the CSR of A
 * (real element types: adjoint == transpose).  Single-GPU contexts; on multi-GPU contexts pass the row slabs of A'
 * to b200_csr_from_csr_slab. */
B200_API int b200_csr_transpose(b200_ctx *ctx, const b200_csr *A, b200_csr **out);
/* diag(A) of the local rows into a device vector (JacobiPrec(diag(A)), reference test/cg.jl:57) */
B200_API int b200_csr_diag(b200_ctx *ctx, const b200_csr *A, void *diag_dev);
/* device CSR arrays back to the host (tests) */
B200_API int b200_csr_download(b200_ctx *ctx, const b200_csr *A, int32_t *rowptr, int32_t *colind, void *vals);

/* Host-side halo plan for row-partitioned operators (multi-GPU).  Pure host code: usable (and
 * tested) without a GPU.  row_offsets has world+1 entries (rank r owns [row_offsets[r], row_offsets[r+1])). */
B200_API int b200_halo_plan_create(int rank, int world, const int64_t *row_offsets, b200_halo_plan **out);
/* scan the slab's GLOBAL column indices and collect the off-slab columns, sorted, grouped by owner */
B200_API int b200_halo_plan_scan(b200_halo_plan *plan, int64_t m_local, const void *rowptr, const void *colind,
                                 int idx_bytes, int base);
/* analytic version for laplace_matrix(N, dims) slabs (no column array needed) */
B200_API int b200_halo_plan_scan_laplacian(b200_halo_plan *plan, int64_t N, int dims);
/* how many / which global columns this rank needs from `owner` (sorted ascending) */
B200_API int64_t b200_halo_plan_recv_count(const b200_halo_plan *plan, int owner);
B200_API int b200_halo_plan_recv_cols(const b200_halo_plan *plan, int owner, int64_t *cols_out);
/* tell the plan which of MY rows `peer` needs (global indices, the peer's recv_cols for me) */
B200_API int b200_halo_plan_set_send(b200_halo_plan *plan, int peer, const int64_t *cols, int64_t count);
B200_API int64_t b200_halo_plan_send_count(const b200_halo_plan *plan, int peer);
/* 1 (and *lo_local = first local row) when the rows `peer` asked for are ONE ascending contiguous range of this
 * rank's slab -- then the CG update kernel stores them straight into the peer's halo (no pack kernel); 0 otherwise
 * (empty, or scattered: packed and pushed by the halo kernel); -1 on bad arguments.  Slab-partitioned stencils
 * (the reference's laplace_matrix, test/laplace_matrix.jl:3-19) always give ranges. */
B200_API int b200_halo_plan_send_range(const b200_halo_plan *plan, int peer, int64_t *lo_local);
B200_API int64_t b200_halo_plan_n_halo(const b200_halo_plan *plan);
/* global column -> local extended index ([0,m_local) own rows, [m_local, m_local+n_halo) halo) */
B200_API int64_t b200_halo_plan_local_index(const b200_halo_plan *plan, int64_t global_col);
B200_API int b200_halo_plan_destroy(b200_halo_plan *plan);

/* Host generators of the reference's test/benchmark matrices (inputs for tests and bench.py):
 * laplace_matrix(Float64, N, dims) as SparseMatrixCSC{Float64,Int64} arrays (test/laplace_matrix.jl:1-12),
 * or as a CSR row slab with int32 columns.  Return nnz, or <0. */
B200_API int64_t b200_gen_laplace_nnz(int64_t N, int dims, int64_t row_begin, int64_t m_local);
B200_API int64_t b200_gen_laplace_csc_i64(int64_t N, int dims, int base, int64_t *colptr, int64_t *rowval,
                                          double *nzval);
/* advection_dominated(N, beta) of reference benchmark/advection_diffusion.jl:3-30 (matrix as CSC Int64 arrays and
 * the right-hand side b, which may be NULL).  Returns nnz, or <0. */
B200_API int64_t b200_gen_advection_csc_i64(int64_t N, double beta, int base, int64_t *colptr, int64_t *rowval,
                                            double *nzval, double *b);
B200_API int64_t b200_gen_laplace_csr_slab_i32(int64_t N, int dims, int64_t row_begin, int64_t m_local,
                                               int32_t *rowptr, int32_t *colind_global, double *vals);

/* Matrix Market ingestion (host code; SURVEY.md section 8f item 3): the reference's benchmark scripts load their
 * real-world operators with MatrixMarket.jl (benchmark/matrixmarket.jl:2,9-10).  `coordinate` format, field real /
 * integer / pattern, symmetry general / symmetric / skew-symmetric.  _info: dimensions, the number of nonzeros AFTER
 * expanding symmetric storage and summing duplicates, field (0 real, 1 integer, 2 pattern), symmetry (0, 1, 2).
 * _read_csc_i64: the three arrays of the SparseMatrixCSC{Float64,Int64} that mmread builds (rows ascending inside a
 * column; base = 1 for Julia) into caller-owned buffers: colptr n+1, rowval / nzval nnz_capacity >= nnz. */
B200_API int b200_mm_info(const char *path, int64_t *m, int64_t *n, int64_t *nnz, int *field, int *symmetry);
B200_API int b200_mm_read_csc_i64(const char *path, int base, int64_t nnz_capacity, int64_t *colptr, int64_t *rowval,
                                  double *nzval);

/* ---------------------------------------------------------------- L0: operator / vector algebra
 * (each Julia op of SURVEY.md section 8b is one call; x,y are LOCAL slabs on multi-GPU contexts,
 * reductions return the GLOBAL value on every rank)
 */
/* mul!(y, A, x)  -- y must not alias x */
B200_API int b200_spmv(b200_ctx *ctx, const b200_csr *A, const void *x_dev, void *y_dev);
/* mul!(Y, A, X) on column-major m x bs blocks (reference src/lobpcg.jl:124-131) */
B200_API int b200_spmm(b200_ctx *ctx, const b200_csr *A, const void *X_dev, int64_t ldx, void *Y_dev, int64_t ldy,
                       int bs);
/* dot(x, y), norm(x) (host result, synchronises) */
B200_API int b200_dot(b200_ctx *ctx, int64_t n, const void *x_dev, const void *y_dev, int dtype, double *result);
B200_API int b200_nrm2(b200_ctx *ctx, int64_t n, const void *x_dev, int dtype, double *result);
/* y .= a .* x .+ b .* y  (axpy!: b=1; broadcast update of src/cg.jl:51: a=1,x=r,b=beta) */
B200_API int b200_axpby(b200_ctx *ctx, int64_t n, double a, const void *x_dev, double b, void *y_dev, int dtype);
B200_API int b200_scal(b200_ctx *ctx, int64_t n, double a, void *x_dev, int dtype);           /* rmul! */
B200_API int b200_copy(b200_ctx *ctx, int64_t n, const void *x_dev, void *y_dev, int dtype);  /* copyto! */
B200_API int b200_fill(b200_ctx *ctx, int64_t n, double a, void *x_dev, int dtype);           /* fill! */
/* ldiv!(y, P::JacobiPrec, x): y .= x ./ diag  (y may alias x: ldiv!(P, x)) */
B200_API int b200_jacobi_ldiv(b200_ctx *ctx, int64_t n, const void *diag_dev, const void *x_dev, void *y_dev,
                              int dtype);

/* ---------------------------------------------------------------- L1: dense helper kernels */
/* orthogonalize_and_normalize!(V[:,1:k], w, h, method) -> nrm
 * (reference src/orthogonalize.jl:13-39 DGKS, :41-51 CGS, :67-79 MGS).
 * V: device, column-major, leading dimension ldv (local rows), k columns; w: device n_local;
 * h_host: k values out (host).  Fused: the k dots in one launch, the k axpys + norm in one launch. */
B200_API int b200_orthogonalize_and_normalize(b200_ctx *ctx, int64_t n_local, const void *V_dev, int64_t ldv, int k,
                                              void *w_dev, double *h_host, int method, int dtype, double *nrm);
/* ldiv!(FastHessenberg(H), rhs) (reference src/hessenberg.jl:15-46): H (m+1) x m column-major with
 * leading dimension ldh, rhs m+1; both device-resident fp64; mutated in place (single-block kernel). */
B200_API int b200_hessenberg_ldiv(b200_ctx *ctx, double *H_dev, int ldh, int m, double *rhs_dev);

/* ---------------------------------------------------------------- L2/L3: solver entry points
 * x is caller-owned and updated IN PLACE (reference src/cg.jl:241); b and A are never mutated.
 * resnorm_host (may be NULL) receives history[:resnorm]; capacity in entries.
 */
typedef struct {
  double abstol;            /* zero(real(eltype(b)))      src/cg.jl:210                            */
  double reltol;            /* sqrt(eps(real(eltype(b)))) src/cg.jl:211 -- pass <0 for that default */
  int64_t maxiter;          /* size(A,2)                  src/cg.jl:212 -- pass <0 for the default  */
  int32_t initially_zero;   /* src/cg.jl:125                                                       */
  int32_t check_every;      /* how many iterations are enqueued between host polls of the device-side
                               `done` flag (<=0: default).  Results do not depend on it: kernels of
                               iterations past `done` are no-ops.                                   */
  b200_precond Pl;          /* Identity -> CGIterable (src/cg.jl:43-66); else PCGIterable (:72-100) */
  int32_t fixed_iterations; /* bench only: ignore convergence, run exactly maxiter iterations      */
  int32_t variant;          /* reserved, must be 0                                                 */
} b200_cg_opts;

/* cg!(x, A, b; ...)  reference src/cg.jl:209-242.  x,b device pointers (local slabs). */
B200_API int b200_cg_solve(b200_ctx *ctx, const b200_csr *A, void *x_dev, const void *b_dev,
                           const b200_cg_opts *opts, b200_result *res, double *resnorm_host, int64_t resnorm_cap);
/* same call with HOST x,b (the end-to-end path: H2D of b and x, solve, D2H of x) */
B200_API int b200_cg_solve_host(b200_ctx *ctx, const b200_csr *A, void *x_host, const void *b_host,
                                const b200_cg_opts *opts, b200_result *res, double *resnorm_host,
                                int64_t resnorm_cap);

/* cg_iterator!(x, A, b; abstol, reltol, maxiter, statevars, Pl, initially_zero)  reference src/cg.jl:120-155:
 * the resumable form of the same engine.  u_dev, r_dev, c_dev are the caller-owned CGStateVariables
 * (src/cg.jl:114-118) or NULL (owned by the iterator).  Creation forms r = b - A x, u = 0, the residual and tol.
 * b200_cg_iter_next performs up to k calls of iterate(it) (src/cg.jl:43-66 / :72-100), stopping at done()
 * (src/cg.jl:36); on return x is complete, res->iters / mvps / residual / tol / isconverged describe the iterator,
 * res->status is 1 once done() holds, and resnorm_host (may be NULL; at most 4096 entries per call) receives the
 * residual after each iteration performed by this call. */
typedef struct b200_cg_iter b200_cg_iter;
B200_API int b200_cg_iter_create(b200_ctx *ctx, const b200_csr *A, void *x_dev, const void *b_dev,
                                 const b200_cg_opts *opts, void *u_dev, void *r_dev, void *c_dev,
                                 b200_cg_iter **out);
B200_API int b200_cg_iter_next(b200_cg_iter *it, int64_t k, b200_result *res, double *resnorm_host,
                               int64_t resnorm_cap);
B200_API int b200_cg_iter_destroy(b200_cg_iter *it);

/* chebyshev!(x, A, b, lmin, lmax; abstol, reltol, Pl, maxiter, initially_zero)  reference src/chebyshev.jl:131-160
 * (SURVEY.md section 8f item 2).  Uses the cg option block (abstol, reltol, maxiter, initially_zero, Pl). */
B200_API int b200_chebyshev_solve(b200_ctx *ctx, const b200_csr *A, void *x_dev, const void *b_dev,
                                  double lambda_min, double lambda_max, const b200_cg_opts *opts, b200_result *res,
                                  double *resnorm_host, int64_t resnorm_cap);


typedef struct {
  double abstol;            /* zero(real(eltype(b)))       src/qmr.jl:266                           */
  double reltol;            /* sqrt(eps(real(eltype(b))))  src/qmr.jl:267 -- pass <0 for that default */
  int64_t maxiter;          /* size(A, 2)                  src/qmr.jl:268 -- pass <0 for the default  */
  int32_t initially_zero;   /* src/qmr.jl:271                                                        */
  int32_t check_every;      /* iterations enqueued between host polls of the device-side done flag (<=0: 16) */
} b200_qmr_opts;
/* qmr!(x, A, b; abstol, reltol, maxiter, initially_zero)  reference src/qmr.jl:262-297 (SURVEY.md section 8f item 4).
 * At = adjoint(A) (b200_csr_transpose, or the adjoint's own row slabs on multi-GPU contexts).  res->mvps counts the
 * products with A and A' together; res->status = B200_ERR_BREAKDOWN after an exact Lanczos breakdown (delta == 0,
 * src/qmr.jl:84-86; see DESIGN.md for the one documented deviation there). */
B200_API int b200_qmr_solve(b200_ctx *ctx, const b200_csr *A, const b200_csr *At, void *x_dev, const void *b_dev,
                            const b200_qmr_opts *opts, b200_result *res, double *resnorm_host, int64_t resnorm_cap);

/* ---------------------------------------------------------------- matrix-free operators and preconditioners
 * The reference's operator contract is duck typing: anything with mul!(y, A, x), size and eltype
 * (docs/src/getting_started.md:25-30; test/cg.jl:71-77 and test/lsqr.jl:36 run the solvers on LinearMaps), and any
 * preconditioner with ldiv!(y, P, x) (docs/src/preconditioning.md:5-15).  A b200_linop is that contract at the C ABI:
 * `apply(user, x_dev, y_dev, cuda_stream)` must ENQUEUE y = A x (or y = P \ x) on the given stream (the context's)
 * without synchronising, for device vectors of n_local / m_local elements of `dtype`; y never aliases x; return 0.
 * The *_op entry points below run the same engines as their b200_csr twins -- all recurrence scalars stay in device
 * memory, the callback is simply the launch between two fused passes -- and on multi-GPU contexts the callback sees
 * the local slabs (halo exchange is the callback's business) while the engines allreduce their sums.  A callback may call
 * the operator-level functions (b200_spmv, b200_axpby, b200_jacobi_ldiv, ...) on the same context; starting another SOLVE
 * on that context from inside a callback is refused (B200_ERR_INVALID: the context's scratch belongs to the running solve) --
 * use a second context for nested solves.  The solver keeps a pointer to the descriptor for the duration of the call (the
 * iterables and the generalized LOBPCG constraint copy it). */
typedef int (*b200_apply_fn)(void *user, const void *x_dev, void *y_dev, void *cuda_stream);
typedef struct {
  b200_apply_fn apply;
  void *user;
  int64_t m_local;          /* length of y (local rows)                                                  */
  int64_t n_local;          /* length of x (local)                                                        */
  int64_t n_global;         /* size(A, 2): default maxiter (src/cg.jl:212)                                */
  int64_t m_global;         /* size(A, 1)                                                                 */
  int32_t dtype;            /* B200_F64 / B200_F32                                                        */
  int32_t reserved;
} b200_linop;
/* cg!(x, A, b; Pl, ...) for a general operator A and a general preconditioner (reference src/cg.jl:43-100,120-155,
 * 209-242): Pl = NULL uses opts->Pl (Identity -> CGIterable, Jacobi -> PCGIterable with the division fused into the
 * <c, r> pass); Pl != NULL is `ldiv!(c, Pl, r)` by callback.  opts->fixed_iterations / variant must be 0. */
B200_API int b200_cg_solve_op(b200_ctx *ctx, const b200_linop *A, const b200_linop *Pl, void *x_dev, const void *b_dev,
                              const b200_cg_opts *opts, b200_result *res, double *resnorm_host, int64_t resnorm_cap);
/* chebyshev! for a callback operator; opts->Pl: Identity, Jacobi or B200_PREC_CALLBACK (src/chebyshev.jl:37).
 * b200_chebyshev_solve with a callback preconditioner runs the same engine (csrc/chebyshev_core.h). */
B200_API int b200_chebyshev_solve_op(b200_ctx *ctx, const b200_linop *A, void *x_dev, const void *b_dev,
                                     double lambda_min, double lambda_max, const b200_cg_opts *opts, b200_result *res,
                                     double *resnorm_host, int64_t resnorm_cap);
/* powm!(B, x; shift, inverse, tol, maxiter) and invpowm!(B, x; shift, ...) = powm!(...; inverse = true) -- reference
 * src/simple.jl:118-151, :186 (beyond SURVEY section 8: the simple eigensolvers of the reference).  Exactly one of A and Aop
 * is non-NULL; for inverse iteration the operator applies inv(A - shift I) (:83-88).  x_dev: the normalised start vector,
 * overwritten by the eigenvector approximation.  *lambda_out = shift + (inverse ? 1/theta : theta), theta the Rayleigh
 * quotient (:51).  Up to maxiter + 1 iterations (done() tests `iteration > maxiter`, :27). */
typedef struct {
  double tol;               /* eps(real(T)) * size(B, 2)^3  src/simple.jl:119  (<0: default)                          */
  int64_t maxiter;          /* size(B, 1)                   src/simple.jl:120  (<0: default)                          */
  double shift;             /* src/simple.jl:121                                                                       */
  int32_t inverse;          /* src/simple.jl:122                                                                       */
  int32_t check_every;      /* iterations enqueued between host polls of the device-side done flag (<=0: 16)          */
} b200_powm_opts;
B200_API int b200_powm(b200_ctx *ctx, const b200_csr *A, const b200_linop *Aop, void *x_dev, const b200_powm_opts *opts,
                       b200_result *res, double *lambda_out, double *resnorm_host, int64_t resnorm_cap);
/* jacobi!(x, A, b; maxiter), gauss_seidel!, sor!(x, A, b, omega; maxiter), ssor! for sparse matrices -- reference
 * src/stationary_sparse.jl:203-424 (beyond SURVEY section 8: the stationary methods of the reference).  Exactly `maxiter`
 * iterations (<0: 10, the reference's default), no stopping test.  The sweeps are level-scheduled: every row performs the
 * reference's arithmetic in the reference's order (csrc/stationary_core.h).  A zero or missing diagonal entry is the
 * SingularException of DiagonalIndices (:19) -> B200_ERR_BREAKDOWN.  Single-GPU contexts; x_dev is updated in place. */
enum { B200_STATIONARY_JACOBI = 0, B200_STATIONARY_GAUSS_SEIDEL = 1, B200_STATIONARY_SOR = 2, B200_STATIONARY_SSOR = 3,
       /* OR-ed in: the arithmetic of the dense-matrix methods of src/stationary.jl (SOR relaxation written as
          x + w (t / a - x), :179; SSOR's backward half reading both triangles with the forward half's values, :247-258) for
          a dense matrix stored as CSR */
       B200_STATIONARY_DENSE_ARITHMETIC = 16 };
B200_API int b200_stationary(b200_ctx *ctx, const b200_csr *A, void *x_dev, const void *b_dev, int method, double omega,
                             int64_t maxiter);
/* qmr! / lsqr! / lsmr! / idrs! on callback operators (A and, where needed, At = adjoint(A)) */
B200_API int b200_qmr_solve_op(b200_ctx *ctx, const b200_linop *A, const b200_linop *At, void *x_dev, const void *b_dev,
                               const b200_qmr_opts *opts, b200_result *res, double *resnorm_host, int64_t resnorm_cap);

/* lsqr! / lsmr! share one option block and one result block. */
typedef struct {
  double damp;              /* lsqr: damp = 0 (src/lsqr.jl:91); lsmr: λ = 0 (src/lsmr.jl:90)                       */
  double atol, btol;        /* lsqr: sqrt(eps(real(T))) (src/lsqr.jl:91); lsmr: 1e-6 (src/lsmr.jl:89) -- <0: default */
  double conlim;            /* lsqr: 1/sqrt(eps) (src/lsqr.jl:92); lsmr: 1e8 (src/lsmr.jl:89) -- <0: default         */
  int64_t maxiter;          /* maximum(size(A)) (src/lsqr.jl:67, src/lsmr.jl:68) -- <0: default                      */
  int32_t check_every;      /* iterations enqueued between host polls of the device-side done flag (<=0: 16)        */
  int32_t reserved;
} b200_lsq_opts;
typedef struct {
  int64_t iters;            /* history.iters                                                                        */
  int64_t mvps, mtvps;      /* history.mvps / history.mtvps as the reference counts them (src/lsqr.jl:130,153,167;
                               src/lsmr.jl:160-161,164,170)                                                         */
  int32_t isconverged;      /* lsqr: istop > 0 (src/lsqr.jl:271); lsmr: istop not in (3, 6, 7) (src/lsmr.jl:285)      */
  int32_t istop;            /* the stopping rule that fired, 0..7                                                   */
  int32_t status;           /* 0, or B200_ERR_INVALID (lsqr: initial guess not finite, src/lsqr.jl:102-104)          */
  int32_t reserved;
  int64_t n_hist;           /* entries written to each history row                                                  */
  int64_t hist_stride;      /* distance between the rows of hist_host = min(hist_cap, maxiter)                      */
  double atol, btol, ctol;  /* history[:atol], [:btol], [:ctol]                                                     */
} b200_lsq_result;
/* lsqr!(x, A, b; damp, atol, btol, conlim, maxiter)  reference src/lsqr.jl:66-77, 90-275.
 * lsmr!(x, A, b; λ, atol, btol, conlim, maxiter)     reference src/lsmr.jl:67-82, 88-287.
 * A: m x n (rectangular allowed on single-GPU contexts), At = adjoint(A); x_dev: n values, updated in place;
 * b_dev: m values, not modified.  hist_host (may be NULL): 4 rows of res->hist_stride doubles --
 * row 0: history[:resnorm] (lsqr) / the ||r|| estimate (lsmr, not part of the reference's history),
 * row 1: [:anorm], row 2: [:rnorm], row 3: [:cnorm]; hist_cap = capacity per row the caller provides. */
B200_API int b200_lsqr_solve(b200_ctx *ctx, const b200_csr *A, const b200_csr *At, void *x_dev, const void *b_dev,
                             const b200_lsq_opts *opts, b200_lsq_result *res, double *hist_host, int64_t hist_cap);
B200_API int b200_lsmr_solve(b200_ctx *ctx, const b200_csr *A, const b200_csr *At, void *x_dev, const void *b_dev,
                             const b200_lsq_opts *opts, b200_lsq_result *res, double *hist_host, int64_t hist_cap);

B200_API int b200_lsqr_solve_op(b200_ctx *ctx, const b200_linop *A, const b200_linop *At, void *x_dev,
                                const void *b_dev, const b200_lsq_opts *opts, b200_lsq_result *res, double *hist_host,
                                int64_t hist_cap);
B200_API int b200_lsmr_solve_op(b200_ctx *ctx, const b200_linop *A, const b200_linop *At, void *x_dev,
                                const void *b_dev, const b200_lsq_opts *opts, b200_lsq_result *res, double *hist_host,
                                int64_t hist_cap);

typedef struct {
  double abstol, reltol;    /* src/idrs.jl:52-53 (reltol < 0: sqrt(eps(real(T))))                                  */
  int64_t maxiter;          /* size(A, 2)  src/idrs.jl:54 (<0: default)                                             */
  int32_t s;                /* dimension of the shadow space, default 8 (src/idrs.jl:50); 1..16                     */
  int32_t smoothing;        /* src/idrs.jl:112                                                                      */
  b200_precond Pl;          /* src/idrs.jl:51                                                                       */
  const void *P;            /* device, n_local x s column-major: the shadow vectors the reference draws with
                               rand!(copy(C)) (src/idrs.jl:132) -- the host passes the draw                        */
  int64_t ldp;
  int32_t check_every;      /* steps enqueued between host polls of the device-side done flag (<=0: 16)             */
  int32_t reserved;
} b200_idrs_opts;
/* idrs!(x, A, b; s, Pl, abstol, reltol, maxiter, smoothing)  reference src/idrs.jl:49-64, 112-145, 163-272. */
B200_API int b200_idrs_solve(b200_ctx *ctx, const b200_csr *A, void *x_dev, const void *b_dev,
                             const b200_idrs_opts *opts, b200_result *res, double *resnorm_host, int64_t resnorm_cap);
B200_API int b200_idrs_solve_op(b200_ctx *ctx, const b200_linop *A, void *x_dev, const void *b_dev,
                                const b200_idrs_opts *opts, b200_result *res, double *resnorm_host,
                                int64_t resnorm_cap);

typedef struct {
  double abstol, reltol;    /* src/gmres.jl:187-188                                                */
  int64_t maxiter;          /* size(A,2)           src/gmres.jl:190                                */
  int32_t restart;          /* min(20, size(A,2))  src/gmres.jl:189  (<=0: default)                */
  int32_t initially_zero;   /* src/gmres.jl:192                                                    */
  int32_t orth_meth;        /* B200_ORTH_*; reference default ModifiedGramSchmidt src/gmres.jl:194 */
  int32_t reserved;
  b200_precond Pl, Pr;      /* src/gmres.jl:185-186                                                */
} b200_gmres_opts;
/* gmres!(x, A, b; ...)  reference src/gmres.jl:184-222 */
B200_API int b200_gmres_solve(b200_ctx *ctx, const b200_csr *A, void *x_dev, const void *b_dev,
                              const b200_gmres_opts *opts, b200_result *res, double *resnorm_host,
                              int64_t resnorm_cap);
/* gmres! for a callback operator `mul!(y, A, x)`; opts->Pl / opts->Pr may be Identity, Jacobi or B200_PREC_CALLBACK
 * (`ldiv!(y, P, x)` by callback; src/gmres.jl:249,281,294,300,303).  b200_gmres_solve with a callback preconditioner runs
 * the same engine (csrc/gmres_core.h: Hessenberg matrix, residual recurrence and least-squares solve device-resident). */
B200_API int b200_gmres_solve_op(b200_ctx *ctx, const b200_linop *A, void *x_dev, const void *b_dev,
                                 const b200_gmres_opts *opts, b200_result *res, double *resnorm_host,
                                 int64_t resnorm_cap);

typedef struct {
  double abstol, reltol;    /* src/minres.jl:204-205                                               */
  int64_t maxiter;          /* src/minres.jl:206                                                   */
  int32_t initially_zero;   /* src/minres.jl:207                                                   */
  int32_t skew_hermitian;   /* src/minres.jl:201                                                   */
} b200_minres_opts;
/* minres!(x, A, b; ...)  reference src/minres.jl:200-237 */
B200_API int b200_minres_solve(b200_ctx *ctx, const b200_csr *A, void *x_dev, const void *b_dev,
                               const b200_minres_opts *opts, b200_result *res, double *resnorm_host,
                               int64_t resnorm_cap);
/* minres! for a callback operator `mul!(y, A, x)` (csrc/minres_core.h; src/minres.jl:61,104) */
B200_API int b200_minres_solve_op(b200_ctx *ctx, const b200_linop *A, void *x_dev, const void *b_dev,
                                  const b200_minres_opts *opts, b200_result *res, double *resnorm_host,
                                  int64_t resnorm_cap);

typedef struct {
  double abstol, reltol;    /* src/bicgstabl.jl:182-183                                            */
  int64_t max_mv_products;  /* size(A,2)  src/bicgstabl.jl:184                                     */
  int32_t l;                /* positional l = 2   src/bicgstabl.jl:181                             */
  int32_t initial_zero;     /* sic (no "ly")      src/bicgstabl.jl:32                              */
  b200_precond Pl;          /* src/bicgstabl.jl:187                                                */
  const void *r_shadow;     /* device vector; the reference draws rand(T,n) (src/bicgstabl.jl:38):
                               the host passes the draw so that runs are reproducible            */
} b200_bicgstabl_opts;
/* bicgstabl!(x, A, b, l; ...)  reference src/bicgstabl.jl:181-219 */
B200_API int b200_bicgstabl_solve(b200_ctx *ctx, const b200_csr *A, void *x_dev, const void *b_dev,
                                  const b200_bicgstabl_opts *opts, b200_result *res, double *resnorm_host,
                                  int64_t resnorm_cap);
/* bicgstabl! for a callback operator; opts->Pl may be Identity, Jacobi or B200_PREC_CALLBACK (`ldiv!(y, Pl, x)` by
 * callback; src/bicgstabl.jl:55,98,108).  b200_bicgstabl_solve with a callback preconditioner runs the same engine
 * (csrc/bicgstabl_core.h); l <= 8. */
B200_API int b200_bicgstabl_solve_op(b200_ctx *ctx, const b200_linop *A, void *x_dev, const void *b_dev,
                                     const b200_bicgstabl_opts *opts, b200_result *res, double *resnorm_host,
                                     int64_t resnorm_cap);

/* gmres_iterable! (src/gmres.jl:108-136), minres_iterable! (src/minres.jl:39-89), bicgstabl_iterator!
 * (src/bicgstabl.jl:27-73): the resumable forms ("the iterator is the solver", docs/src/iterators.md).  Exactly one of
 * A (device CSR) and Aop (callback operator) is non-NULL; the preconditioners travel in the option block (Identity,
 * Jacobi or B200_PREC_CALLBACK).  Creation performs the solver's setup (initial residual, tolerance); the iterable owns
 * its scratch, x_dev / b_dev (and r_shadow) stay the caller's.  b200_iter_next performs up to k calls of iterate()
 * (inner iterations for gmres, outer ones -- 2 l products -- for bicgstabl), stopping at done(); k = 0 reports the state.
 * res->iters / mvps / residual / tol / isconverged describe the iterable, res->status is 1 once done() holds, and
 * resnorm_host (may be NULL; at most 4096 entries per call) receives the residual norms of the iterations performed by
 * this call.  Results are identical to the one-shot *_solve_op engines for every chunking. */
typedef struct b200_iter b200_iter;
B200_API int b200_gmres_iter_create(b200_ctx *ctx, const b200_csr *A, const b200_linop *Aop, void *x_dev,
                                    const void *b_dev, const b200_gmres_opts *opts, b200_iter **out);
B200_API int b200_minres_iter_create(b200_ctx *ctx, const b200_csr *A, const b200_linop *Aop, void *x_dev,
                                     const void *b_dev, const b200_minres_opts *opts, b200_iter **out);
B200_API int b200_bicgstabl_iter_create(b200_ctx *ctx, const b200_csr *A, const b200_linop *Aop, void *x_dev,
                                        const void *b_dev, const b200_bicgstabl_opts *opts, b200_iter **out);
/* cg_iterator!(x, A, b, Pl; ...) (src/cg.jl:120-155) with a callback operator and / or a callback preconditioner; the
 * b200_csr + Identity / Jacobi form with caller-owned CGStateVariables is b200_cg_iter_create. */
B200_API int b200_cg_iter_create_op(b200_ctx *ctx, const b200_csr *A, const b200_linop *Aop, void *x_dev,
                                    const void *b_dev, const b200_cg_opts *opts, b200_iter **out);
B200_API int b200_iter_next(b200_iter *it, int64_t k, b200_result *res, double *resnorm_host, int64_t resnorm_cap);
B200_API int b200_iter_destroy(b200_iter *it);

typedef struct {
  double tol;               /* default_tolerance(T) = eps(real(T))^(3/10)  src/lobpcg.jl:751       */
  int64_t maxiter;          /* 200   src/lobpcg.jl:865                                             */
  int32_t largest;          /* src/lobpcg.jl:787                                                   */
  int32_t blocksize;        /* size(X0, 2)                                                         */
  b200_precond P;           /* src/lobpcg.jl:226-242 (RPreconditioner)                             */
  int32_t fixed_iterations; /* bench only: never soft-lock, run exactly maxiter steps              */
  int32_t reserved;
  /* log = true (src/lobpcg.jl:744-745, :881-884): the LOBPCGState of every iteration.  Host arrays (or NULL) with
   * `blocksize` doubles per iteration, row it-1 = residual norms / Ritz values after iteration it; at most trace_cap
   * rows are written (results.iterations says how many iterations ran). */
  double *trace_resnorm;
  double *trace_ritz;
  int64_t trace_cap;
} b200_lobpcg_opts;
typedef struct {
  int64_t iterations;       /* results.iterations  src/lobpcg.jl:890                               */
  int32_t converged;        /* all(residual_norms .<= tol)                                         */
  int32_t status;
} b200_lobpcg_result;
/* lobpcg(A, largest, X0; ...) -> LOBPCGResults  reference src/lobpcg.jl:787-839, 865-893.
 * X_dev: n_local x blocksize column-major (ld = ldx), overwritten with the Ritz vectors;
 * lambda_host, resnorm_host: blocksize values each. */
B200_API int b200_lobpcg_solve(b200_ctx *ctx, const b200_csr *A, void *X_dev, int64_t ldx,
                               const b200_lobpcg_opts *opts, b200_lobpcg_result *res, double *lambda_host,
                               double *resnorm_host);

/* svdl(A; nsv, k, j, tol, reltol, maxiter, method, vecs, dolock, v0)  reference src/svdl.jl:157-247 (SURVEY.md section
 * 8f item 4): singular values (and vectors) by Golub-Kahan-Lanczos bidiagonalisation with thick restart. */
typedef struct {
  int32_t nsv;              /* 6                          src/svdl.jl:158   (<=0: default)                          */
  int32_t k;                /* 2nsv Lanczos vectors       src/svdl.jl:158   (<=0: default; at most 64)              */
  int32_t j;                /* nsv vectors kept at restart src/svdl.jl:178  (<=0: default)                          */
  int32_t method;           /* 0 = :ritz (thickrestart! src/svdl.jl:376-404), 1 = :harmonic (harmonicrestart! :424-493) */
  int64_t maxiter;          /* minimum(size(A))           src/svdl.jl:159   (<0: default)                           */
  double tol, reltol;       /* sqrt(eps()) each           src/svdl.jl:158,179 (<0: default)                         */
  int32_t dolock;           /* src/svdl.jl:181, :214-221                                                            */
  int32_t reserved;
} b200_svdl_opts;
typedef struct {
  int64_t iters;            /* history.iters (one per restart, src/svdl.jl:189)                                     */
  int64_t mvps, mtvps;      /* products with A / A' as extend! counts them (src/svdl.jl:564, :582)                  */
  int32_t isconverged;      /* all(conv) reached (src/svdl.jl:222)                                                  */
  int32_t k;                /* size of the projected matrix B                                                       */
  double beta;              /* L.beta at exit                                                                       */
  double tol;               /* history[:tol]                                                                        */
} b200_svdl_result;
/* A: m x n operator, At = adjoint(A); v0_dev: n values (starting vector, a copy is normalised); sigma_host: nsv values
 * (F.S[1:nsv], :227).  U_dev (m x nsv, ld ldu) / V_dev (n x nsv, ld ldv): device, left / right singular vectors as the
 * reference forms them (L.P*F.U[:,1:l], L.Q[:,1:k]*F.V[:,1:l], :230-241) or NULL (vecs = :none).  Histories (host, may
 * be NULL): hist_ritz maxiter x k (:ritz), hist_resnorm maxiter x nsv (:resnorm = the error bounds of isconverged),
 * hist_conv maxiter x nsv (:conv), hist_betas maxiter (:betas); row `it` is written by iteration it+1.  B_host:
 * k x k column-major, the projected matrix L.B at exit (may be NULL). */
B200_API int b200_svdl(b200_ctx *ctx, const b200_csr *A, const b200_csr *At, const void *v0_dev,
                       const b200_svdl_opts *opts, b200_svdl_result *res, double *sigma_host, void *U_dev, int64_t ldu,
                       void *V_dev, int64_t ldv, double *hist_ritz, double *hist_resnorm, int32_t *hist_conv,
                       double *hist_betas, double *B_host);
B200_API int b200_svdl_op(b200_ctx *ctx, const b200_linop *A, const b200_linop *At, const void *v0_dev,
                          const b200_svdl_opts *opts, b200_svdl_result *res, double *sigma_host, void *U_dev,
                          int64_t ldu, void *V_dev, int64_t ldv, double *hist_ritz, double *hist_resnorm,
                          int32_t *hist_conv, double *hist_betas, double *B_host);

/* The constraint of lobpcg (`C` keyword, reference src/lobpcg.jl:829; struct Constraint :144-224): a basis Y the Ritz
 * vectors are kept orthogonal to.  Standard problem (B = I).  Y_dev: n_local x nc column-major (copied); `capacity`
 * >= nc columns are reserved for b200_lobpcg_constraint_append, which mirrors update! (:188-206: the Cholesky factor
 * of Y'Y is extended by an identity block -- the appended columns must be orthonormal and orthogonal to Y, as the
 * converged Ritz vectors of a constrained solve are); that is how the nev > blocksize driver (:925-962) deflates
 * the batches it has already computed.  _apply: X <- X - Y (Y'Y \ Y'X) on a column-major block (:212-224).
 * Errors: _create returns B200_ERR_BREAKDOWN ("PosDefException") when Y'Y is not positive definite.  The pivot rule
 * is a superset of LAPACK potrf's (!(d > 0), what cholesky! at :181-182 does): a pivot is also rejected when it is
 * below 4 nc eps of its diagonal entry, i.e. when Y is rank deficient up to rounding -- there potrf's answer depends on
 * the order of roundings and the accepted factor carries no correct digits. */
typedef struct b200_lobpcg_constraint b200_lobpcg_constraint;
B200_API int b200_lobpcg_constraint_create(b200_ctx *ctx, int64_t n_local, const void *Y_dev, int64_t ldy, int nc,
                                           int capacity, int dtype, b200_lobpcg_constraint **out);
B200_API int b200_lobpcg_constraint_append(b200_ctx *ctx, b200_lobpcg_constraint *c, const void *X_dev, int64_t ldx,
                                           int k);
B200_API int b200_lobpcg_constraint_apply(b200_ctx *ctx, const b200_lobpcg_constraint *c, void *X_dev, int64_t ldx,
                                          int bs);
B200_API int b200_lobpcg_constraint_info(const b200_lobpcg_constraint *c, int *nc, int *capacity);
B200_API int b200_lobpcg_constraint_destroy(b200_lobpcg_constraint *c);
/* lobpcg(A, largest, X0; C, ...): b200_lobpcg_solve with the constraint applied to the initial block (:868) and to the
 * preconditioned active residuals of every step (precond_constr! :564-569).  C == NULL is b200_lobpcg_solve. */
B200_API int b200_lobpcg_solve_constrained(b200_ctx *ctx, const b200_csr *A, void *X_dev, int64_t ldx,
                                           const b200_lobpcg_opts *opts, const b200_lobpcg_constraint *C,
                                           b200_lobpcg_result *res, double *lambda_host, double *resnorm_host);

/* The GENERAL form of lobpcg: generalized problem A x = lambda B x (B != NULL; reference src/lobpcg.jl:827-839 with the
 * B-blocks of :117-142, :262-338, :365-393), operators / preconditioner as callbacks (opts->P.kind = B200_PREC_CALLBACK:
 * `diag` points to the preconditioner's b200_linop), constraint in the B inner product.  Block sizes 1..16.  The standard
 * problem on a b200_csr with Identity / Jacobi is faster through b200_lobpcg_solve[_constrained] (tuned engine).
 * b200_csr_as_linop fills a b200_linop that applies a b200_csr (so that CSR and callback operators can be mixed);
 * b200_lobpcg_constraint_create_b is Constraint(Y, B, X) for B != nothing (:161-186); nc may be 0 with `capacity` columns
 * reserved for b200_lobpcg_constraint_append, which then also forms B * X for the new columns (update!, :188-206). */
B200_API int b200_csr_as_linop(const b200_csr *A, b200_linop *out);
B200_API int b200_lobpcg_solve_op(b200_ctx *ctx, const b200_linop *A, const b200_linop *B, void *X_dev, int64_t ldx,
                                  const b200_lobpcg_opts *opts, const b200_lobpcg_constraint *C, b200_lobpcg_result *res,
                                  double *lambda_host, double *resnorm_host);
B200_API int b200_lobpcg_constraint_create_b(b200_ctx *ctx, const b200_linop *B, int64_t n_local, const void *Y_dev,
                                             int64_t ldy, int nc, int capacity, int dtype, b200_lobpcg_constraint **out);

/* Test hook: the eight Rayleigh-Ritz Gram products (reference src/lobpcg.jl:586-605) of five row-major n x 16 fp32
 * device blocks X, R, AR, P, AP through one of the engine's kernels (variant 1: tcgen05.mma with TMEM accumulators,
 * variant 2: legacy mma.sync); out_host[p * 256 + i * 16 + j], products X'AR, X'R, R'AR, X'AP, X'P, R'P, AR'P, P'AP. */
B200_API int b200_debug_lobpcg_gram_rr(b200_ctx *ctx, const void *const *blk_dev, int64_t n, int variant,
                                       double *out_host);

/* Host-side dense helpers used by the engines for their O(blocksize^3) pieces (fp64, column-major,
 * n <= 64): eigen!(Hermitian(A)[, Hermitian(B)]) -- eigenvalues ascending in w, eigenvectors in the
 * columns of Z with Z'BZ = I (reference src/lobpcg.jl:615,622 -> LAPACK syevd / sygvd).  B may be NULL.
 * Returns 0; B200_ERR_BREAKDOWN if B is not positive definite or the iteration does not converge.
 * Exposed so that the CPU test-suite can pin them against LAPACK. */
B200_API int b200_dense_sygv_host(int n, const double *A, const double *B, double *w, double *Z);

#ifdef __cplusplus
}
#endif
#endif /* B200KRYLOV_H */
