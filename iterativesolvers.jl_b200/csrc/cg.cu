// cg.cu -- the (P)CG engine: cg!(x, A, b; ...) of reference src/cg.jl:209-242 as fused device kernels.
//
// One CG iteration (reference src/cg.jl:43-66) = three stream-ordered launches, no host round trip:
//   K1  x += alpha_prev*u ; u = r + beta*u     (src/cg.jl:58 of the previous step, :50-51; 5 vector passes)
//   K2  c = A*u  fused with  dot(u,c), alpha   (src/cg.jl:54-55)     <- the HBM-dominant kernel
//   K3  r -= alpha*c ; ||r||^2                 (src/cg.jl:59-62; 3 vector passes)
// (the x update rides in the next K1 because that kernel streams u anyway: 10 vector passes + A per
// iteration instead of the 11 of the algorithmic accounting below; values are identical to the reference
// order of operations, x is just completed one launch later -- k_cg_flush_x closes the last step)
// All scalars (residual, prev_residual, alpha, beta, tol, iteration, done) live in device memory
// (struct CgScal); the reductions finish on the device (last-block ticket) and the same block does
// the scalar bookkeeping, including the reference's termination test (src/cg.jl:36).  Kernels of
// iterations enqueued after `done` return immediately, so the host only polls the flag every
// `check_every` iterations and results do not depend on that period.
// Algorithmic bytes per iteration (SURVEY.md section 8d): nnz*(V+4) + (n+1)*4 + 11*n*V.
//
// Multi-GPU (row slabs, one process per GPU), two interchangeable transports (option "comm"):
//   * peer memory (default when the IPC mapping succeeded, peer.cuh): K3 is followed by k_halo_push of r's
//     boundary values (stored straight into the neighbours' halo segments over NVLink), the next K1 forms the
//     halo part of u locally from them (so K2 never waits; PCG keeps the push of u after K1 and the wait in
//     K2), and the block that finishes a reduction performs the one-shot all-to-all allreduce itself --
//     4 launches per iteration, no NCCL call, no scalar kernel;
//   * NCCL: halo = pack kernel + grouped ncclSend/ncclRecv, each sum = ncclAllReduce of one double followed
//     by a 1-thread bookkeeping kernel.
#include <cooperative_groups.h>

#include "blas1.cuh"
#include "spmv_dia.cuh"
#include "linop.cuh"

using namespace b200;

namespace {

constexpr int kThreads = 256;

struct CgScal {
  double residual;       // it.residual
  double prev_residual;  // it.prev_residual (CGIterable)
  double rho;            // it.rho (PCGIterable)
  double rho_prev;
  double tol;
  double sum;            // NCCL path: local/global sum of the reduction in flight
  double alpha;          // alpha of the current iteration (set when dot(u,c) is known)
  double dot_uc;
  double abstol, reltol;
  long long iter;        // iterations completed
  long long maxiter;
  long long hist_cap;
  int done;
  int fixed;             // bench: ignore convergence
  int breakdown;
  int comm_error;
  int pcg;               // PCGIterable (Jacobi Pl) instead of CGIterable
  int pad;
};

// how the grid-wide sum of one GPU becomes the global sum
enum { COMM_SINGLE = 0, COMM_NCCL = 1, COMM_PEER = 2 };
struct Comm {
  int mode;
  unsigned long long seq;        // allreduce sequence number (COMM_PEER)
  unsigned long long halo_seq;   // halo sequence to wait for before the first gather (COMM_PEER, K2 only)
  unsigned int halo_mask;        // ranks this GPU receives halo values from
  int rev;                       // sweep the rows from the end (consecutive kernels alternate: L2 reuse)
  PeerView pv;
};

// Peer path, CG with Identity: the boundary rows of the new r go to the neighbours from INSIDE K3 (the rows every rank sends
// are one contiguous range per neighbour for slabs of banded operators), and the block that finishes the grid reduction
// raises the halo flags -- one launch (k_halo_push) less per iteration.
struct PushRanges {
  int n;                         // 0: nothing to push from this kernel
  int rank;
  unsigned int send_mask;
  unsigned long long seq;        // halo sequence the flags announce
  long long lo[2], cnt[2];       // local row ranges
  void *dst[2];                  // their place in the neighbour's halo segment (mapped peer memory)
};

// bookkeeping after ||r||^2 is known (src/cg.jl:61-62 + done() :36); single thread
__device__ __forceinline__ void cg_after_norm(CgScal *s, double rr, double *hist, bool pcg) {
  if (!pcg) s->prev_residual = s->residual;
  const double res = sqrt(rr);
  s->residual = res;
  if (hist && s->iter < s->hist_cap) hist[s->iter] = res;
  s->iter += 1;
  if (!(res == res)) s->breakdown = 1;
  const bool conv = !s->fixed && (res <= s->tol);
  s->done = (s->iter >= s->maxiter) || conv || (!s->fixed && s->breakdown);
}

// initial residual norm known (src/cg.jl:140-141)
__device__ __forceinline__ void cg_after_init_norm(CgScal *s, double rr) {
  const double res = sqrt(rr);
  s->residual = res;
  s->prev_residual = 1.0;
  s->rho = 1.0;
  s->rho_prev = 1.0;
  s->tol = fmax(s->reltol * res, s->abstol);
  s->iter = 0;
  s->breakdown = !(res == res);
  const bool conv = !s->fixed && (res <= s->tol);
  s->done = (0 >= s->maxiter) || conv || (!s->fixed && s->breakdown);   // NaN ends the solve: see b200_result.status
}

enum { FIN_NONE = 0, FIN_INIT = 1, FIN_DOT = 2, FIN_NORM = 3, FIN_NORM_PCG = 4, FIN_RHO = 5 };

__device__ __forceinline__ void cg_apply(int kind, CgScal *s, double total, double *hist) {
  switch (kind) {
    case FIN_INIT: cg_after_init_norm(s, total); break;
    case FIN_DOT:                                    // alpha = residual^2 / dot(u,c)  (src/cg.jl:55; PCG :90)
      s->dot_uc = total;
      s->alpha = s->pcg ? s->rho / total : (s->residual * s->residual) / total;
      break;
    case FIN_NORM: cg_after_norm(s, total, hist, false); break;
    case FIN_NORM_PCG: cg_after_norm(s, total, hist, true); break;
    case FIN_RHO: s->rho_prev = s->rho; s->rho = total; break;
    default: break;
  }
}

// called by the FIRST WARP of the block that holds the grid-wide sum of this GPU (lane 0 has it in `total`)
__device__ __forceinline__ void cg_finish(int kind, CgScal *s, double total, double *hist, const Comm &cm) {
  if (cm.mode == COMM_PEER) total = peer_allreduce_sum_warp(cm.pv, total, cm.seq);   // lane q <-> rank q
  if ((threadIdx.x & 31u) != 0) return;
  if (cm.mode == COMM_NCCL) {   // the host enqueues ncclAllReduce(&s->sum) + k_cg_scalar next
    s->sum = total;
    return;
  }
  if (cm.mode == COMM_PEER && cm.pv.hdr[cm.pv.rank]->error) s->comm_error = 1;
  cg_apply(kind, s, total, hist);
}

__global__ void k_cg_scalar(int kind, CgScal *s, double *hist) {
  if (kind != FIN_INIT && s->done) return;  // kernels of iterations past `done` did not produce a sum
  cg_apply(kind, s, s->sum, hist);
}

// r = b - c (c = A*x) or r = b; u = 0; ||r||^2     (src/cg.jl:129-140)
template <typename T>
__global__ void __launch_bounds__(kThreads) k_cg_init(const T *__restrict__ b, const T *__restrict__ c, int has_c,
                                                      T *__restrict__ r, T *__restrict__ u, int64_t n, CgScal *s,
                                                      double *partials, unsigned int *ticket, Comm cm) {
  __shared__ double smem[kThreads / 32];
  double acc = 0.0;
  for (int64_t i = blockIdx.x * (int64_t)kThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kThreads) {
    T ri = b[i];
    if (has_c) ri = ri - c[i];
    r[i] = ri;
    u[i] = (T)0;
    acc += (double)ri * (double)ri;
  }
  acc = block_sum<kThreads>(acc, smem);
  double total;
  if (grid_reduce_finish<kThreads>(acc, partials, ticket, smem, &total) && threadIdx.x < 32)
    cg_finish(FIN_INIT, s, total, nullptr, cm);
}

// every CTA makes sure the neighbours' halo values of this iteration have landed (peer path)
__device__ __forceinline__ void wait_halo(const Comm &cm) {
  if (cm.mode == COMM_PEER && cm.halo_mask) {
    if (threadIdx.x == 0) peer_wait_halo(cm.pv, cm.halo_mask, cm.halo_seq);
    __syncthreads();
  }
}

// K1: x += alpha_prev*u (the x update of the PREVIOUS iteration, src/cg.jl:58) ; u = r + beta*u (src/cg.jl:51)
//     (CG: beta = residual^2/prev_residual^2 ; PCG: u = c + (rho/rho_prev)*u)
// The x update is deferred by one kernel so that u is streamed once for both updates (10 instead of 11
// vector passes per iteration); x_k is formed from the same operands as in the reference, one launch later,
// and k_cg_flush_x applies the last one when the loop ends.
template <typename T>
__global__ void __launch_bounds__(kThreads) k_cg_update_u(const T *__restrict__ r, T *__restrict__ u,
                                                          T *__restrict__ x, int64_t n,
                                                          const CgScal *__restrict__ s, int pcg, int rev,
                                                          const T *r_halo, T *__restrict__ u_halo, int n_halo,
                                                          Comm cm) {
  pdl_wait();
  if (s->done) return;
  const double beta_d = pcg ? s->rho / s->rho_prev
                            : (s->residual * s->residual) / (s->prev_residual * s->prev_residual);
  const T beta = (T)beta_d;
  const T alpha = (T)s->alpha;
  const bool upd_x = s->iter > 0;
  for (int64_t j = blockIdx.x * (int64_t)kThreads + threadIdx.x; j < n; j += (int64_t)gridDim.x * kThreads) {
    const int64_t i = rev ? n - 1 - j : j;
    const T ui = u[i];
    // x .+= alpha .* u ; r .+ beta .* u  -- no FMA contraction, as the reference's broadcasts compute them
    if constexpr (sizeof(T) == 8) {
      if (upd_x) x[i] = __dadd_rn(x[i], __dmul_rn(alpha, ui));
      u[i] = __dadd_rn(r[i], __dmul_rn(beta, ui));
    } else {
      if (upd_x) x[i] = __fadd_rn(x[i], __fmul_rn(alpha, ui));
      u[i] = __fadd_rn(r[i], __fmul_rn(beta, ui));
    }
  }
  pdl_launch_dependents();   // the bulk of this CTA's work is done: let the next kernel's blocks become resident
  // Peer-memory path (CG, Identity): the neighbours pushed the boundary values of r right after their K3 -- one
  // kernel earlier than u exists -- and every GPU forms the halo part of u itself from the same operands
  // (r_halo, beta, previous u_halo): bit-identical to the owner's values, and the NVLink latency of the push is
  // hidden behind this kernel instead of stalling the first gathers of K2.
  if (r_halo && (int64_t)blockIdx.x * kThreads < n_halo) {
    wait_halo(cm);
    for (int64_t h = blockIdx.x * (int64_t)kThreads + threadIdx.x; h < n_halo; h += (int64_t)gridDim.x * kThreads) {
      const T rh = __ldcg(r_halo + h);
      if constexpr (sizeof(T) == 8) u_halo[h] = __dadd_rn(rh, __dmul_rn(beta, u_halo[h]));
      else u_halo[h] = __fadd_rn(rh, __fmul_rn(beta, u_halo[h]));
    }
  }
}

// the deferred x update of the last completed iteration
template <typename T>
__global__ void __launch_bounds__(kThreads) k_cg_flush_x(const T *__restrict__ u, T *__restrict__ x, int64_t n,
                                                         const CgScal *__restrict__ s) {
  if (s->iter <= 0) return;
  const T alpha = (T)s->alpha;
  for (int64_t i = blockIdx.x * (int64_t)kThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kThreads) {
    if constexpr (sizeof(T) == 8) x[i] = __dadd_rn(x[i], __dmul_rn(alpha, u[i]));
    else x[i] = __fadd_rn(x[i], __fmul_rn(alpha, u[i]));
  }
}


// K2 (sub-warp-per-row fallback): c = A*u ; sum u.*c
template <typename T, int LPR>
__global__ void __launch_bounds__(kThreads) k_cg_spmv_dot(const int *__restrict__ rowptr,
                                                          const int *__restrict__ colind,
                                                          const T *__restrict__ vals, XView<T> xv, int64_t m,
                                                          T *__restrict__ c, CgScal *s, double *partials,
                                                          unsigned int *ticket, Comm cm) {
  pdl_wait();
  if (s->done) return;
  __shared__ double smem[kThreads / 32];
  wait_halo(cm);
  constexpr int ROWS = kThreads / LPR;
  const int sub = threadIdx.x % LPR;
  const int rib = threadIdx.x / LPR;
  double acc = 0.0;
  for (int64_t base = (int64_t)blockIdx.x * ROWS; base < m; base += (int64_t)gridDim.x * ROWS) {
    const int64_t row = base + rib;
    const bool valid = row < m;
    const T ci = row_dot<T, LPR>(rowptr, colind, vals, xv, valid ? row : (m - 1), sub);
    if (valid && sub == 0) {
      c[row] = ci;
      acc += (double)xv.x[row] * (double)ci;
    }
  }
  pdl_launch_dependents();
  acc = block_sum<kThreads>(acc, smem);
  double total;
  if (grid_reduce_finish<kThreads>(acc, partials, ticket, smem, &total) && threadIdx.x < 32)
    cg_finish(FIN_DOT, s, total, nullptr, cm);
}

// K2, TMA-streamed form (spmv_stream.cuh): same result contract as k_cg_spmv_dot
template <typename T>
struct CgDotEpi {
  T *__restrict__ c;
  const T *__restrict__ u;
  double acc;
  __device__ __forceinline__ T pre(int64_t row) const { return u[row]; }
  __device__ __forceinline__ void operator()(int64_t row, T v, T ur) {
    c[row] = v;
    acc += (double)ur * (double)v;
  }
};
template <typename T, int LPR>
__global__ void __launch_bounds__(kStreamThreads, kStreamCtasPerSm)
    k_cg_spmv_dot_stream(const int *__restrict__ rowptr, const int *__restrict__ colind, const T *__restrict__ vals,
                         XView<T> xv, int64_t m, T *__restrict__ c, CgScal *s, double *partials,
                         unsigned int *ticket, Comm cm) {
  pdl_wait();
  if (s->done) return;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ double red[kStreamThreads / 32];
  wait_halo(cm);
  CgDotEpi<T> epi{c, xv.x, 0.0};
  spmv_stream_tiles<T, LPR>(rowptr, colind, vals, xv, m, epi, reinterpret_cast<StreamSmem<T> *>(smem_raw), cm.rev != 0);
  pdl_launch_dependents();
  const double acc = block_sum<kStreamThreads>(epi.acc, red);
  double total;
  if (grid_reduce_finish<kStreamThreads>(acc, partials, ticket, red, &total) && threadIdx.x < 32)
    cg_finish(FIN_DOT, s, total, nullptr, cm);
}

// K2 on the DIA copy (spmv_dia.cuh): same row -> thread -> CTA mapping and row sums as the CSR stream, so c and <u,c>
// are bitwise the same
template <typename T>
__global__ void __launch_bounds__(kStreamThreads, kStreamCtasPerSm)
    k_cg_spmv_dot_dia(DiaView<T> dv, XView<T> xv, int64_t m, T *__restrict__ c, CgScal *s, double *partials,
                      unsigned int *ticket, Comm cm) {
  pdl_wait();
  if (s->done) return;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ double red[kStreamThreads / 32];
  CgDotEpi<T> epi{c, xv.x, 0.0};
  spmv_dia_tiles<T>(dv, xv, m, epi, reinterpret_cast<DiaSmem<T> *>(smem_raw), cm.rev != 0);
  pdl_launch_dependents();
  const double acc = block_sum<kStreamThreads>(epi.acc, red);
  double total;
  if (grid_reduce_finish<kStreamThreads>(acc, partials, ticket, red, &total) && threadIdx.x < 32)
    cg_finish(FIN_DOT, s, total, nullptr, cm);
}

// K3: r -= alpha*c ; ||r||^2   (x += alpha*u is applied by the next K1 / k_cg_flush_x)
template <typename T>
__global__ void __launch_bounds__(kThreads) k_cg_update_r(T *__restrict__ r, const T *__restrict__ c, int64_t n,
                                                          CgScal *s, double *hist, double *partials,
                                                          unsigned int *ticket, int pcg, Comm cm, PushRanges pr) {
  pdl_wait();
  if (s->done) return;
  __shared__ double smem[kThreads / 32];
  const T alpha = (T)s->alpha;
  double acc = 0.0;
  for (int64_t j = blockIdx.x * (int64_t)kThreads + threadIdx.x; j < n; j += (int64_t)gridDim.x * kThreads) {
    const int64_t i = cm.rev ? n - 1 - j : j;
    T ri;
    if constexpr (sizeof(T) == 8) ri = __dsub_rn(r[i], __dmul_rn(alpha, c[i]));
    else ri = __fsub_rn(r[i], __fmul_rn(alpha, c[i]));
    r[i] = ri;
    acc += (double)ri * (double)ri;
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const long long k = (long long)i - pr.lo[q];
      if (q < pr.n && k >= 0 && k < pr.cnt[q]) ((T *)pr.dst[q])[k] = ri;   // store to the neighbour's halo segment (NVLink)
    }
  }
  pdl_launch_dependents();
  acc = block_sum<kThreads>(acc, smem);
  double total;
  if (grid_reduce_finish<kThreads>(acc, partials, ticket, smem, &total, pr.n > 0)) {
    if (pr.n > 0 && threadIdx.x == 0) {
      // every block fenced its boundary stores at system scope before taking its ticket: the flags may go out (before this
      // GPU starts waiting for the other ranks' partial sums)
      __threadfence_system();
      for (int p = 0; p < cm.pv.world; ++p)
        if ((pr.send_mask >> p) & 1u) st_release_sys(&cm.pv.hdr[p]->halo_flag[pr.rank], pr.seq);
    }
    if (threadIdx.x < 32) cg_finish(pcg ? FIN_NORM_PCG : FIN_NORM, s, total, hist, cm);
  }
}

// PCG: c = r ./ d ; rho = dot(c, r)    (src/cg.jl:79-82, Jacobi ldiv!)
template <typename T>
__global__ void __launch_bounds__(kThreads) k_pcg_precond(const T *__restrict__ d, const T *__restrict__ r,
                                                          T *__restrict__ c, int64_t n, CgScal *s, double *partials,
                                                          unsigned int *ticket, Comm cm) {
  pdl_wait();
  if (s->done) return;
  __shared__ double smem[kThreads / 32];
  double acc = 0.0;
  for (int64_t i = blockIdx.x * (int64_t)kThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kThreads) {
    const T ri = r[i];
    const T ci = ri / d[i];
    c[i] = ci;
    acc += (double)ci * (double)ri;
  }
  pdl_launch_dependents();
  acc = block_sum<kThreads>(acc, smem);
  double total;
  if (grid_reduce_finish<kThreads>(acc, partials, ticket, smem, &total) && threadIdx.x < 32)
    cg_finish(FIN_RHO, s, total, nullptr, cm);
}


// ------------------------------------------------------------------------------------------------
// Small operators: the whole CG loop in ONE persistent cooperative kernel (single GPU, Identity / Jacobi).
// At config-#1 size (5-point Poisson 128^2, n = 16 384) an iteration is a few microseconds of work and the three launches of
// the streaming path are the cost; here the phases of an iteration are separated by grid-wide barriers instead:
//   [PCG: c = r ./ d, rho]  ->  x += alpha_prev u ; u = r + beta u  -> sync ->  c = A u, <u,c>  -> sync ->
//   r -= alpha c, ||r||^2  -> sync
// Every block sums the per-block partials itself, in the same order, so all blocks hold identical scalars (alpha, beta,
// residual, done) without a broadcast; the reference's operation order and the unfused multiply / add of its broadcasts are
// kept (src/cg.jl:43-66, :72-100), the x update rides one phase behind as in the streaming kernels.
// ------------------------------------------------------------------------------------------------
namespace cgx = cooperative_groups;
constexpr int64_t kPersistMaxRows = 1 << 18;      // above this the TMA-streamed kernels win (vectors no longer L2-resident)

template <int THREADS>
__device__ __forceinline__ double all_blocks_sum(const double *slots, unsigned int nslots, double *smem, double *bcast) {
  double a = 0.0;
  for (unsigned int i = threadIdx.x; i < nslots; i += THREADS) a += __ldcg(&slots[i]);   // same scheme as grid_reduce_finish
  a = block_sum<THREADS>(a, smem);
  if (threadIdx.x == 0) *bcast = a;
  __syncthreads();
  const double t = *bcast;
  __syncthreads();
  return t;
}

template <typename T, int LPR>
__global__ void __launch_bounds__(kThreads) k_cg_persistent(const int *__restrict__ rowptr, const int *__restrict__ colind,
                                                            const T *__restrict__ vals, const T *__restrict__ jac, T *x, T *r,
                                                            T *u, T *c, int64_t n, CgScal *s, double *hist, double *partials,
                                                            long long iters) {
  cgx::grid_group grid = cgx::this_grid();
  __shared__ double smem[kThreads / 32];
  __shared__ double bcast;
  double *pa = partials, *pb = partials + kMaxPartials, *pc = partials + 2 * kMaxPartials;
  // every block keeps its own copy of the scalars; they evolve identically
  double residual = s->residual, prev_residual = s->prev_residual, alpha = s->alpha, rho = s->rho, rho_prev = s->rho_prev;
  const double tol = s->tol;
  long long iter = s->iter;
  const long long maxiter = s->maxiter, hist_cap = s->hist_cap;
  const int fixed = s->fixed, pcg = s->pcg;
  int done = s->done, breakdown = s->breakdown;
  double dot_uc = s->dot_uc;
  const int64_t gstride = (int64_t)gridDim.x * kThreads;
  constexpr int ROWS = kThreads / LPR;
  const int sub = threadIdx.x % LPR, rib = threadIdx.x / LPR;
  XView<T> xv;
  xv.x = u;
  xv.halo = u;
  xv.m = (int)n;
  for (long long it = 0; it < iters && !done; ++it) {
    if (pcg) {                                            // c = Pl \ r ; rho = <c, r>   (:79-82)
      double acc = 0.0;
      for (int64_t i = blockIdx.x * (int64_t)kThreads + threadIdx.x; i < n; i += gstride) {
        const T ri = r[i];
        const T ci = ri / jac[i];
        c[i] = ci;
        acc += (double)ci * (double)ri;
      }
      acc = block_sum<kThreads>(acc, smem);
      if (threadIdx.x == 0) pc[blockIdx.x] = acc;
      __threadfence();
      grid.sync();
      rho_prev = rho;
      rho = all_blocks_sum<kThreads>(pc, gridDim.x, smem, &bcast);
    }
    // x += alpha_prev u (deferred :58) ; u = r + beta u (:50-51 / :85-86)
    const T beta = (T)(pcg ? rho / rho_prev : (residual * residual) / (prev_residual * prev_residual));
    const T al = (T)alpha;
    const bool upd_x = iter > 0;
    const T *src = pcg ? c : r;
    for (int64_t i = blockIdx.x * (int64_t)kThreads + threadIdx.x; i < n; i += gstride) {
      const T ui = u[i];
      if constexpr (sizeof(T) == 8) {
        if (upd_x) x[i] = __dadd_rn(x[i], __dmul_rn(al, ui));
        u[i] = __dadd_rn(src[i], __dmul_rn(beta, ui));
      } else {
        if (upd_x) x[i] = __fadd_rn(x[i], __fmul_rn(al, ui));
        u[i] = __fadd_rn(src[i], __fmul_rn(beta, ui));
      }
    }
    __threadfence();
    grid.sync();
    // c = A u ; <u, c>   (:54-55)
    {
      double acc = 0.0;
      for (int64_t base = (int64_t)blockIdx.x * ROWS; base < n; base += (int64_t)gridDim.x * ROWS) {
        const int64_t row = base + rib;
        const bool valid = row < n;
        const T ci = row_dot<T, LPR>(rowptr, colind, vals, xv, valid ? row : (n - 1), sub);
        if (valid && sub == 0) {
          c[row] = ci;
          acc += (double)u[row] * (double)ci;
        }
      }
      acc = block_sum<kThreads>(acc, smem);
      if (threadIdx.x == 0) pa[blockIdx.x] = acc;
    }
    __threadfence();
    grid.sync();
    dot_uc = all_blocks_sum<kThreads>(pa, gridDim.x, smem, &bcast);
    alpha = pcg ? rho / dot_uc : (residual * residual) / dot_uc;
    // r -= alpha c ; ||r||   (:59-62 / :94-96)
    {
      const T a2 = (T)alpha;
      double acc = 0.0;
      for (int64_t i = blockIdx.x * (int64_t)kThreads + threadIdx.x; i < n; i += gstride) {
        T ri;
        if constexpr (sizeof(T) == 8) ri = __dsub_rn(r[i], __dmul_rn(a2, c[i]));
        else ri = __fsub_rn(r[i], __fmul_rn(a2, c[i]));
        r[i] = ri;
        acc += (double)ri * (double)ri;
      }
      acc = block_sum<kThreads>(acc, smem);
      if (threadIdx.x == 0) pb[blockIdx.x] = acc;
    }
    __threadfence();
    grid.sync();
    const double rr = all_blocks_sum<kThreads>(pb, gridDim.x, smem, &bcast);
    if (!pcg) prev_residual = residual;                   // cg_after_norm
    residual = sqrt(rr);
    if (blockIdx.x == 0 && threadIdx.x == 0 && hist && iter < hist_cap) hist[iter] = residual;
    iter += 1;
    if (!(residual == residual)) breakdown = 1;
    const bool conv = !fixed && (residual <= tol);
    done = (iter >= maxiter) || conv || (!fixed && breakdown);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    s->residual = residual;
    s->prev_residual = prev_residual;
    s->alpha = alpha;
    s->dot_uc = dot_uc;
    s->rho = rho;
    s->rho_prev = rho_prev;
    s->iter = iter;
    s->done = done;
    s->breakdown = breakdown;
  }
}

template <typename T>
struct CgEngine {
  b200_ctx *ctx;
  const b200_csr *A;
  int64_t n;
  T *x, *r, *u, *c;
  const T *b;
  const T *jac;  // NULL => Identity
  CgScal *s;
  double *hist;
  int mode;      // COMM_*
  int lpr, grid_vec, grid_spmv;
  int sweep = 0;   // direction of the next hot kernel (toggled per launch when ctx->opt_snake)
  bool fold_halo = false;   // peer path, Identity: r's boundary is pushed after K3 and K1 forms u's halo locally
  bool fold_push = false;   // ... and K3 itself stores the boundary rows to the neighbours (contiguous send ranges)
  bool persistent = false;  // small single-GPU operator: the whole loop runs in k_cg_persistent
  int grid_persist = 0;

  int next_sweep() {
    const int d = ctx->opt_snake ? sweep : 0;
    sweep ^= 1;
    return d;
  }

  // Comm descriptor for the next reduction (peer path: consumes one sequence number on every rank)
  Comm comm(bool with_halo = false, int rev = 0) {
    Comm cm;
    cm.mode = mode;
    cm.seq = 0;
    cm.halo_seq = 0;
    cm.halo_mask = 0;
    cm.rev = rev;
    if (mode == COMM_PEER) {
      cm.pv = ctx->peer_view;
      cm.seq = ++ctx->ar_seq;
      if (with_halo) {
        cm.halo_seq = ctx->halo_seq;
        cm.halo_mask = A->recv_mask;
      }
    }
    return cm;
  }

  int after_reduce(int kind) {
    if (mode != COMM_NCCL) return B200_OK;
    B200_TRY(allreduce_sum_dev(ctx, &s->sum, 1));
    k_cg_scalar<<<1, 1, 0, ctx->stream>>>(kind, s, hist);
    B200_LAUNCH_CHECK(ctx);
    return B200_OK;
  }

  int spmv_dot() {
    const bool peer = mode == COMM_PEER;
    if (fold_halo) {
      // u's halo was formed by K1 in A->halo: nothing to exchange, nothing to wait for
    } else if (peer) {
      ctx->halo_seq += 1;
      B200_TRY(halo_push(ctx, A, u, ctx->halo_seq, &s->done));
    } else {
      B200_TRY(halo_exchange(ctx, A, u));
    }
    XView<T> xv = make_xview<T>(A, u, peer && !fold_halo);
    const Comm cm = comm(!fold_halo, next_sweep());
    if (use_dia(ctx, A)) {
      const int grid = stream_grid_size(ctx, A);
      const size_t smem = sizeof(DiaSmem<T>);
      ProfScope prof(ctx, 0);
      B200_SMEM_ATTR_ONCE(ctx, smem, k_cg_spmv_dot_dia<T>);
      B200_CUDA(launch_chained(ctx->opt_pdl != 0, k_cg_spmv_dot_dia<T>, dim3(grid), dim3(kStreamThreads), smem,
                               ctx->stream, make_diaview<T>(A), xv, n, c, s, ctx->red.partials, ctx->red.ticket, cm));
    } else if (use_stream(ctx, A)) {
      const int grid = stream_grid_size(ctx, A);
      const size_t smem = sizeof(StreamSmem<T>);
      ProfScope prof(ctx, 0);
#define LAUNCH(L)                                                                                                    \
  do {                                                                                                               \
    B200_SMEM_ATTR_ONCE(ctx, smem, k_cg_spmv_dot_stream<T, L>);                                                      \
    B200_CUDA(launch_chained(ctx->opt_pdl != 0, k_cg_spmv_dot_stream<T, L>, dim3(grid), dim3(kStreamThreads), smem,    \
                             ctx->stream, A->rowptr, A->colind, (const T *)A->vals, xv, n, c, s, ctx->red.partials,  \
                             ctx->red.ticket, cm));                                                                  \
  } while (0)
      switch (A->stream_lpr) {
        case 1: LAUNCH(1); break;
        case 2: LAUNCH(2); break;
        case 4: LAUNCH(4); break;
        case 8: LAUNCH(8); break;
        case 16: LAUNCH(16); break;
        default: LAUNCH(32); break;
      }
#undef LAUNCH
    } else {
      ProfScope prof(ctx, 0);
#define LAUNCH(L)                                                                                               \
  B200_CUDA(launch_chained(ctx->opt_pdl != 0, k_cg_spmv_dot<T, L>, dim3(grid_spmv), dim3(kThreads), 0, ctx->stream, \
                           A->rowptr, A->colind, (const T *)A->vals, xv, n, c, s, ctx->red.partials,             \
                           ctx->red.ticket, cm))
      switch (lpr) {
        case 2: LAUNCH(2); break;
        case 4: LAUNCH(4); break;
        case 8: LAUNCH(8); break;
        case 16: LAUNCH(16); break;
        default: LAUNCH(32); break;
      }
#undef LAUNCH
    }
    B200_LAUNCH_CHECK(ctx);
    return after_reduce(FIN_DOT);
  }

  int iterate() {
    cudaStream_t st = ctx->stream;
    const int pcg = jac != nullptr;
    if (pcg) {
      B200_CUDA(launch_chained(ctx->opt_pdl != 0, k_pcg_precond<T>, dim3(grid_vec), dim3(kThreads), 0, st, jac, r, c, n, s,
                               ctx->red.partials, ctx->red.ticket, comm()));
      B200_LAUNCH_CHECK(ctx);
      B200_TRY(after_reduce(FIN_RHO));
    }
    {
      ProfScope prof(ctx, 2);
      Comm hc;
      hc.mode = mode;
      hc.seq = 0;
      hc.halo_seq = ctx->halo_seq;
      hc.halo_mask = fold_halo ? A->recv_mask : 0;
      hc.rev = 0;
      if (mode == COMM_PEER) hc.pv = ctx->peer_view;
      B200_CUDA(launch_chained(ctx->opt_pdl != 0, k_cg_update_u<T>, dim3(grid_vec), dim3(kThreads), 0, st,
                               (const T *)(pcg ? c : r), u, x, n, (const CgScal *)s, pcg, next_sweep(),
                               fold_halo ? (const T *)A->halo_peer : (const T *)nullptr,
                               fold_halo ? (T *)A->halo : (T *)nullptr, fold_halo ? (int)A->n_halo : 0, hc));
    }
    B200_LAUNCH_CHECK(ctx);
    B200_TRY(spmv_dot());
    PushRanges pr;
    memset(&pr, 0, sizeof(pr));
    if (fold_push) {
      ctx->halo_seq += 1;
      pr.rank = ctx->rank;
      pr.send_mask = A->send_mask;
      pr.seq = ctx->halo_seq;
      const size_t vs = sizeof(T);
      for (int p = 0; p < ctx->world; ++p)
        if (A->send_count[p] > 0) {
          pr.lo[pr.n] = A->send_range_lo[p];
          pr.cnt[pr.n] = A->send_count[p];
          pr.dst[pr.n] = (char *)ctx->peer_ptr[p] + kPeerHeaderBytes + vs * (size_t)A->peer_dst_offset[p];
          pr.n += 1;
        }
    }
    {
      ProfScope prof(ctx, 1);
      B200_CUDA(launch_chained(ctx->opt_pdl != 0, k_cg_update_r<T>, dim3(grid_vec), dim3(kThreads), 0, st, r, (const T *)c, n,
                               s, hist, ctx->red.partials, ctx->red.ticket, pcg, comm(false, next_sweep()), pr));
    }
    B200_LAUNCH_CHECK(ctx);
    B200_TRY(after_reduce(pcg ? FIN_NORM_PCG : FIN_NORM));
    return fold_push ? B200_OK : push_r_halo();
  }

  // k iterations (fewer if done() comes first): one cooperative launch for small operators, k x iterate() otherwise
  int iterate_many(int64_t k) {
    if (!persistent) {
      for (int64_t i = 0; i < k; ++i) B200_TRY(iterate());
      return B200_OK;
    }
    if (k <= 0) return B200_OK;
    const int *rp = A->rowptr, *ci = A->colind;
    const T *va = (const T *)A->vals, *jc = jac;
    T *x_ = x, *r_ = r, *u_ = u, *c_ = c;
    int64_t n_ = n;
    CgScal *s_ = s;
    double *h_ = hist, *pt = ctx->red.partials;
    long long kk = k;
    void *args[] = {(void *)&rp, (void *)&ci, (void *)&va, (void *)&jc, (void *)&x_, (void *)&r_, (void *)&u_, (void *)&c_,
                    (void *)&n_, (void *)&s_, (void *)&h_, (void *)&pt, (void *)&kk};
    const void *kern = nullptr;
    switch (lpr) {
      case 2: kern = (const void *)k_cg_persistent<T, 2>; break;
      case 4: kern = (const void *)k_cg_persistent<T, 4>; break;
      case 8: kern = (const void *)k_cg_persistent<T, 8>; break;
      case 16: kern = (const void *)k_cg_persistent<T, 16>; break;
      default: kern = (const void *)k_cg_persistent<T, 32>; break;
    }
    ProfScope prof(ctx, 0);
    B200_CUDA(cudaLaunchCooperativeKernel(kern, dim3(grid_persist), dim3(kThreads), args, 0, ctx->stream));
    ctx->launches++;
    return B200_OK;
  }

  // boundary values of the new r go to the neighbours now; they are consumed by the next K1
  int push_r_halo() {
    if (!fold_halo) return B200_OK;
    ctx->halo_seq += 1;
    return halo_push(ctx, A, r, ctx->halo_seq, &s->done);
  }
};

// cg_iterator! (src/cg.jl:120-155): fills the engine, uploads the scalars, forms r = b - A x (unless
// initially_zero), u = 0, ||r||, tol.  u/r/c/scal/hist are provided by the caller (solve: context arena;
// iterator: its own buffers or the user's CGStateVariables).
template <typename T>
int cg_setup(CgEngine<T> &e, b200_ctx *ctx, const b200_csr *A, T *x, const T *b, const b200_cg_opts *o, T *u, T *r,
             T *c, CgScal *scal, double *hist, int64_t hist_cap, int64_t *mv_products) {
  cudaStream_t st = ctx->stream;
  const int64_t n = A->m_local;
  const double eps = sizeof(T) == 8 ? 2.220446049250313e-16 : 1.1920928955078125e-07;
  const double reltol = o->reltol < 0 ? sqrt(eps) : o->reltol;
  const int64_t maxiter = o->maxiter < 0 ? A->n_global : o->maxiter;
  e.ctx = ctx;
  e.A = A;
  e.n = n;
  e.x = x;
  e.b = b;
  e.u = u;
  e.r = r;
  e.c = c;
  e.s = scal;
  static_assert(sizeof(CgScal) <= 256, "CgScal too large");
  e.hist = hist_cap ? hist : nullptr;
  e.jac = o->Pl.kind == B200_PREC_JACOBI ? (const T *)o->Pl.diag : nullptr;
  e.mode = ctx->world == 1 ? COMM_SINGLE : (use_peer(ctx, A) ? COMM_PEER : COMM_NCCL);
  e.lpr = pick_lpr(A->avg_row_nnz);
  e.grid_vec = stream_grid(ctx, n, kThreads * 2, 8);
  e.grid_spmv = stream_grid(ctx, n, kThreads / e.lpr, 8);
  e.fold_halo = e.mode == COMM_PEER && !e.jac && A->halo && A->halo_peer && A->n_halo > 0;
  if (e.fold_halo) B200_CUDA(cudaMemsetAsync(A->halo, 0, sizeof(T) * (size_t)A->n_halo, st));   // u_0 = 0
  e.persistent = false;
  if (ctx->world == 1 && ctx->opt_cg_persistent != 0 && n > 0 && n <= kPersistMaxRows) {
    int per_sm = 0;
    const void *kern = nullptr;
    switch (e.lpr) {
      case 2: kern = (const void *)k_cg_persistent<T, 2>; break;
      case 4: kern = (const void *)k_cg_persistent<T, 4>; break;
      case 8: kern = (const void *)k_cg_persistent<T, 8>; break;
      case 16: kern = (const void *)k_cg_persistent<T, 16>; break;
      default: kern = (const void *)k_cg_persistent<T, 32>; break;
    }
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kThreads, 0) == cudaSuccess && per_sm >= 1) {
      const int64_t want = (n + (kThreads / e.lpr) - 1) / (kThreads / e.lpr);          // one SpMV row group per block
      const int64_t cap = std::min<int64_t>((int64_t)ctx->sm_count * std::min(per_sm, 2), kMaxPartials);
      e.grid_persist = (int)std::max<int64_t>(1, std::min<int64_t>(want, cap));
      e.persistent = true;
    }
  }
  e.fold_push = false;
  if (e.fold_halo && ctx->opt_fold_push != 0) {      // at most two neighbours, each receiving one contiguous range of rows
    int peers = 0;
    bool ranges = true;
    for (int p = 0; p < ctx->world; ++p)
      if (A->send_count[p] > 0) {
        peers += 1;
        ranges = ranges && (int)A->send_range_lo.size() > p && A->send_range_lo[p] >= 0;
      }
    e.fold_push = ranges && peers >= 1 && peers <= 2;
  }

  CgScal h;
  memset(&h, 0, sizeof(h));
  h.abstol = o->abstol;
  h.reltol = reltol;
  h.maxiter = maxiter;
  h.hist_cap = hist_cap;
  h.fixed = o->fixed_iterations;
  h.pcg = e.jac != nullptr;
  B200_CUDA(cudaMemcpyAsync(e.s, &h, sizeof(h), cudaMemcpyHostToDevice, st));   // pageable source: staged before return

  *mv_products = 0;
  if (!o->initially_zero) {
    *mv_products = 1;
    B200_TRY(spmv(ctx, A, x, e.c));
  }
  k_cg_init<T><<<e.grid_vec, kThreads, 0, st>>>(b, e.c, o->initially_zero ? 0 : 1, e.r, e.u, n, e.s, ctx->red.partials,
                                                 ctx->red.ticket, e.comm());
  B200_LAUNCH_CHECK(ctx);
  B200_TRY(e.after_reduce(FIN_INIT));
  return e.push_r_halo();
}

template <typename T>
int cg_solve_impl(b200_ctx *ctx, const b200_csr *A, T *x, const T *b, const b200_cg_opts *o, b200_result *res,
                  double *resnorm_host, int64_t resnorm_cap) {
  cudaStream_t st = ctx->stream;
  const int64_t n = A->m_local;
  const int64_t maxiter = o->maxiter < 0 ? A->n_global : o->maxiter;
  const int check_every = o->check_every > 0 ? o->check_every : 32;
  const int64_t hist_cap = resnorm_host ? std::min<int64_t>(resnorm_cap, maxiter) : 0;

  // workspace: u, r, c, scalars, history
  const size_t vec_bytes = align_up(sizeof(T) * (size_t)std::max<int64_t>(n, 1), 256);
  const size_t hist_bytes = align_up(sizeof(double) * (size_t)std::max<int64_t>(hist_cap, 1), 256);
  void *ws = nullptr;
  B200_TRY(ws_get(ctx, 3 * vec_bytes + 256 + hist_bytes, &ws));
  char *p = (char *)ws;
  CgEngine<T> e;
  int64_t mv_products = 0;
  B200_TRY(cg_setup<T>(e, ctx, A, x, b, o, (T *)p, (T *)(p + vec_bytes), (T *)(p + 2 * vec_bytes),
                       (CgScal *)(p + 3 * vec_bytes), (double *)(p + 3 * vec_bytes + 256), hist_cap, &mv_products));

  // the hot loop (src/cg.jl:229): enqueue check_every iterations, poll the device flag
  int64_t enqueued = 0;
  int *h_done = ctx->h_flags;
  for (;;) {
    B200_CUDA(cudaMemcpyAsync(h_done, &e.s->done, sizeof(int), cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));
    if (*h_done || enqueued >= maxiter) break;
    // persistent kernel: a launch runs until done() or its iteration budget, so the budget per host check can be large
    const int64_t batch = std::min<int64_t>(e.persistent ? std::max<int64_t>(check_every, 1024) : check_every, maxiter - enqueued);
    B200_TRY(e.iterate_many(batch));
    enqueued += batch;
  }
  k_cg_flush_x<T><<<e.grid_vec, kThreads, 0, st>>>(e.u, x, n, e.s);   // x += alpha*u of the last iteration
  B200_LAUNCH_CHECK(ctx);
  CgScal h;
  B200_CUDA(cudaMemcpyAsync(&h, e.s, sizeof(h), cudaMemcpyDeviceToHost, st));
  B200_CUDA(cudaStreamSynchronize(st));
  if (h.comm_error) {
    set_error("peer-memory collective timed out (a rank did not reach the same point of the CG loop)");
    return B200_ERR_NCCL;
  }
  if (res) {
    res->iters = h.iter;
    res->mvps = mv_products + h.iter;  // history.mvps (src/cg.jl:226-231)
    res->isconverged = h.residual <= h.tol;
    res->status = h.breakdown ? B200_ERR_BREAKDOWN : 0;
    res->tol = h.tol;
    res->residual = h.residual;
    res->n_resnorm = std::min<int64_t>(h.iter, hist_cap);
  }
  if (hist_cap && h.iter > 0) {
    B200_CUDA(cudaMemcpyAsync(resnorm_host, e.hist, sizeof(double) * std::min<int64_t>(h.iter, hist_cap),
                              cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));
  }
  return B200_OK;
}

// per-call control of an iterator: history window for the coming batch; alpha = 0 after x was completed, so that
// the deferred `x += alpha*u` of the next K1 adds exactly nothing
__global__ void k_cg_iter_ctl(CgScal *s, long long hist_cap, int zero_alpha) {
  if (hist_cap >= 0) s->hist_cap = hist_cap;
  if (zero_alpha) s->alpha = 0.0;
}

constexpr int64_t kIterHistWindow = 4096;   // residuals recorded per b200_cg_iter_next call

template <typename T>
struct CgIterState {
  CgEngine<T> e;
  DevBuf own_vec[3], scal, hist;
  int64_t mv_products = 0, maxiter = 0;
};

template <typename T>
int cg_iter_create_impl(b200_ctx *ctx, const b200_csr *A, T *x, const T *b, const b200_cg_opts *o, T *u, T *r, T *c,
                        CgIterState<T> *it) {
  const size_t vec_bytes = sizeof(T) * (size_t)std::max<int64_t>(A->m_local, 1);
  T *v[3] = {u, r, c};
  for (int k = 0; k < 3; ++k)
    if (!v[k]) {
      B200_TRY(it->own_vec[k].alloc(vec_bytes));
      v[k] = (T *)it->own_vec[k].p;
    }
  B200_TRY(it->scal.alloc(256));
  B200_TRY(it->hist.alloc(sizeof(double) * kIterHistWindow));
  it->maxiter = o->maxiter < 0 ? A->n_global : o->maxiter;
  return cg_setup<T>(it->e, ctx, A, x, b, o, v[0], v[1], v[2], (CgScal *)it->scal.p, (double *)it->hist.p, 0,
                     &it->mv_products);
}

template <typename T>
int cg_iter_next_impl(CgIterState<T> *it, int64_t k, b200_result *res, double *resnorm_host, int64_t cap) {
  CgEngine<T> &e = it->e;
  b200_ctx *ctx = e.ctx;
  cudaStream_t st = ctx->stream;
  CgScal h;
  B200_CUDA(cudaMemcpyAsync(&h, e.s, sizeof(h), cudaMemcpyDeviceToHost, st));
  B200_CUDA(cudaStreamSynchronize(st));
  const int64_t start = h.iter;
  k = std::max<int64_t>(0, std::min<int64_t>(k, it->maxiter - start));
  const int64_t window = resnorm_host ? std::min<int64_t>(std::min<int64_t>(cap, k), kIterHistWindow) : 0;
  // history slots of this batch: hist[iter] lands in the window for iter in [start, start + window)
  e.hist = window ? (double *)it->hist.p - start : nullptr;
  k_cg_iter_ctl<<<1, 1, 0, st>>>(e.s, start + window, 0);
  B200_LAUNCH_CHECK(ctx);
  if (!h.done) B200_TRY(e.iterate_many(k));                         // iterate(it) x k  (src/cg.jl:43-66 / :72-100)
  k_cg_flush_x<T><<<e.grid_vec, kThreads, 0, st>>>(e.u, e.x, e.n, e.s);
  B200_LAUNCH_CHECK(ctx);
  k_cg_iter_ctl<<<1, 1, 0, st>>>(e.s, -1, 1);
  B200_LAUNCH_CHECK(ctx);
  B200_CUDA(cudaMemcpyAsync(&h, e.s, sizeof(h), cudaMemcpyDeviceToHost, st));
  B200_CUDA(cudaStreamSynchronize(st));
  if (h.comm_error) {
    set_error("peer-memory collective timed out (a rank did not reach the same point of the CG loop)");
    return B200_ERR_NCCL;
  }
  const int64_t performed = h.iter - start;
  if (res) {
    res->iters = h.iter;
    res->mvps = it->mv_products + h.iter;
    res->isconverged = h.residual <= h.tol;
    res->status = h.breakdown ? B200_ERR_BREAKDOWN : (h.done ? 1 : 0);   // 1: done() is true (src/cg.jl:36)
    res->tol = h.tol;
    res->residual = h.residual;
    res->n_resnorm = std::min<int64_t>(performed, window);
  }
  if (window && performed > 0) {
    B200_CUDA(cudaMemcpyAsync(resnorm_host, it->hist.p, sizeof(double) * std::min<int64_t>(performed, window),
                              cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));
  }
  return B200_OK;
}

int check_cg_args(b200_ctx *ctx, const b200_csr *A, const void *x, const void *b, const b200_cg_opts *o) {
  B200_REQUIRE(ctx && A && x && b && o, "NULL argument");
  B200_REQUIRE(A->ctx == ctx, "operator belongs to another context");
  B200_REQUIRE(is_square(A), "this solver needs a square operator (got %lld x %lld)", (long long)A->m_global,
               (long long)A->n_global);
  B200_REQUIRE(o->Pl.kind == B200_PREC_IDENTITY || (o->Pl.kind == B200_PREC_JACOBI && o->Pl.diag),
               "unsupported preconditioner");
  return B200_OK;
}

}  // namespace

extern "C" {

int b200_cg_solve(b200_ctx *ctx, const b200_csr *A, void *x_dev, const void *b_dev, const b200_cg_opts *opts,
                  b200_result *res, double *resnorm_host, int64_t resnorm_cap) {
  if (ctx && A && x_dev && b_dev && opts && opts->Pl.kind == B200_PREC_CALLBACK) {   // ldiv! by callback: the general engine
    B200_REQUIRE(A->ctx == ctx, "operator belongs to another context");
    B200_REQUIRE(is_square(A), "this solver needs a square operator");
    return cg_general(ctx, CudaOp{A, nullptr}, A->dtype, A->m_local, A->n_global, nullptr, x_dev, b_dev, opts, res,
                      resnorm_host, resnorm_cap);
  }
  B200_TRY(check_cg_args(ctx, A, x_dev, b_dev, opts));
  B200_CUDA(cudaSetDevice(ctx->device));
  return A->dtype == B200_F64
             ? cg_solve_impl<double>(ctx, A, (double *)x_dev, (const double *)b_dev, opts, res, resnorm_host, resnorm_cap)
             : cg_solve_impl<float>(ctx, A, (float *)x_dev, (const float *)b_dev, opts, res, resnorm_host, resnorm_cap);
}

int b200_cg_solve_host(b200_ctx *ctx, const b200_csr *A, void *x_host, const void *b_host, const b200_cg_opts *opts,
                       b200_result *res, double *resnorm_host, int64_t resnorm_cap) {
  B200_TRY(check_cg_args(ctx, A, x_host, b_host, opts));
  B200_CUDA(cudaSetDevice(ctx->device));
  const size_t bytes = dtype_size(A->dtype) * (size_t)A->m_local;
  struct { void *p; } dx, db;
  B200_TRY(stage_get(ctx, 0, bytes ? bytes : 16, &dx.p));
  B200_TRY(stage_get(ctx, 1, bytes ? bytes : 16, &db.p));
  B200_CUDA(cudaMemcpyAsync(db.p, b_host, bytes, cudaMemcpyHostToDevice, ctx->stream));
  B200_CUDA(cudaMemcpyAsync(dx.p, x_host, bytes, cudaMemcpyHostToDevice, ctx->stream));
  int s = b200_cg_solve(ctx, A, dx.p, db.p, opts, res, resnorm_host, resnorm_cap);
  if (s != B200_OK) return s;
  B200_CUDA(cudaMemcpyAsync(x_host, dx.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  B200_CUDA(cudaStreamSynchronize(ctx->stream));
  return B200_OK;
}

struct b200_cg_iter {
  int dtype;
  CgIterState<double> d;
  CgIterState<float> f;
};

int b200_cg_iter_create(b200_ctx *ctx, const b200_csr *A, void *x_dev, const void *b_dev, const b200_cg_opts *opts,
                        void *u_dev, void *r_dev, void *c_dev, b200_cg_iter **out) {
  B200_TRY(check_cg_args(ctx, A, x_dev, b_dev, opts));
  B200_REQUIRE(out, "NULL argument");
  B200_CUDA(cudaSetDevice(ctx->device));
  b200_cg_iter *it = new b200_cg_iter();
  it->dtype = A->dtype;
  const int st = A->dtype == B200_F64
                     ? cg_iter_create_impl<double>(ctx, A, (double *)x_dev, (const double *)b_dev, opts, (double *)u_dev,
                                                   (double *)r_dev, (double *)c_dev, &it->d)
                     : cg_iter_create_impl<float>(ctx, A, (float *)x_dev, (const float *)b_dev, opts, (float *)u_dev,
                                                  (float *)r_dev, (float *)c_dev, &it->f);
  if (st != B200_OK) {
    delete it;
    return st;
  }
  *out = it;
  return B200_OK;
}

int b200_cg_iter_next(b200_cg_iter *it, int64_t k, b200_result *res, double *resnorm_host, int64_t resnorm_cap) {
  B200_REQUIRE(it, "NULL argument");
  b200_ctx *ctx = it->dtype == B200_F64 ? it->d.e.ctx : it->f.e.ctx;
  B200_CUDA(cudaSetDevice(ctx->device));
  return it->dtype == B200_F64 ? cg_iter_next_impl<double>(&it->d, k, res, resnorm_host, resnorm_cap)
                               : cg_iter_next_impl<float>(&it->f, k, res, resnorm_host, resnorm_cap);
}

int b200_cg_iter_destroy(b200_cg_iter *it) {
  if (!it) return B200_OK;
  b200_ctx *ctx = it->dtype == B200_F64 ? it->d.e.ctx : it->f.e.ctx;
  if (ctx) cudaStreamSynchronize(ctx->stream);
  delete it;
  return B200_OK;
}

}  // extern "C"
