// common.cuh -- shared plumbing of libb200krylov: context, error handling, device helpers.
// sm_100a only (B200).  No CPU fallback anywhere in this library.
#pragma once

#include <cuda_runtime.h>
#include <nccl.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <atomic>
#include <string>
#include <vector>

#include "../../include/b200krylov.h"
#include "peer.cuh"

namespace b200 {

void set_error(const char *fmt, ...);

#define B200_CUDA(call)                                                                          \
  do {                                                                                           \
    cudaError_t _e = (call);                                                                     \
    if (_e != cudaSuccess) {                                                                     \
      b200::set_error("%s:%d CUDA error %s (%s) in `%s`", __FILE__, __LINE__, cudaGetErrorName(_e), \
                      cudaGetErrorString(_e), #call);                                            \
      return B200_ERR_CUDA;                                                                      \
    }                                                                                            \
  } while (0)

// cudaFuncAttributeMaxDynamicSharedMemorySize is a PER-DEVICE attribute of a kernel: raise it once per (kernel
// instantiation, device) -- a process may hold contexts on several devices (b200_ctx_create(device)); thread-safe.
#define B200_SMEM_ATTR_ONCE(ctx, bytes, ...)                                                                      \
  do {                                                                                                            \
    static std::atomic<unsigned long long> b200_attr_done_{0ull};                                                 \
    const unsigned long long b200_bit_ = 1ull << ((ctx)->device & 63);                                            \
    if (!(b200_attr_done_.load(std::memory_order_acquire) & b200_bit_)) {                                         \
      B200_CUDA(cudaFuncSetAttribute(__VA_ARGS__, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes)));    \
      b200_attr_done_.fetch_or(b200_bit_, std::memory_order_release);                                             \
    }                                                                                                             \
  } while (0)

#define B200_NCCL(call)                                                                          \
  do {                                                                                           \
    ncclResult_t _r = (call);                                                                    \
    if (_r != ncclSuccess) {                                                                     \
      b200::set_error("%s:%d NCCL error %s in `%s`", __FILE__, __LINE__, ncclGetErrorString(_r), #call); \
      return B200_ERR_NCCL;                                                                      \
    }                                                                                            \
  } while (0)

#define B200_TRY(call)          \
  do {                          \
    int _s = (call);            \
    if (_s != B200_OK) return _s; \
  } while (0)

#define B200_REQUIRE(cond, ...)          \
  do {                                   \
    if (!(cond)) {                       \
      b200::set_error(__VA_ARGS__);      \
      return B200_ERR_INVALID;           \
    }                                    \
  } while (0)

// launch-error check after every kernel launch (cheap: cudaPeekAtLastError does not synchronise)
#define B200_LAUNCH_CHECK(ctx)                     \
  do {                                             \
    (ctx)->launches++;                             \
    B200_CUDA(cudaPeekAtLastError());              \
  } while (0)

constexpr int kMaxPartials = 4096;  // upper bound on blocks that contribute to one reduction

}  // namespace b200

// Scratch for deterministic grid-wide reductions: per-block partials in a fixed slot order, a ticket
// counter so that the last block to finish reduces the slots in index order (run-to-run reproducible).
struct b200_reduce_ws {
  double *partials;    // [kMaxPartials * kMaxReduceWidth]
  unsigned int *ticket;
};

struct b200_ctx {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  bool own_stream = true;
  cudaStream_t comm_stream = nullptr;  // halo exchange
  cudaEvent_t ev_a = nullptr, ev_b = nullptr, ev_timer0 = nullptr, ev_timer1 = nullptr;
  int rank = 0, world = 1;
  ncclComm_t comm = nullptr;
  int64_t launches = 0;
  b200_reduce_ws red;       // reduction workspace (device)
  double *d_scalars = nullptr;   // small device scratch for scalar results (64 doubles)
  double *h_scalars = nullptr;   // pinned host mirror (64 doubles)
  int *h_flags = nullptr;        // pinned host flags (16 ints)
  int opt_spmv_kernel = 0;       // b200_ctx_set_option("spmv_kernel"): 0 auto, 1 sub-warp per row, 2 TMA stream
  int opt_spmv_format = 0;       // b200_ctx_set_option("spmv_format"): 0 auto (the DIA copy when the operator has one), 1 CSR
  int opt_comm = 0;              // b200_ctx_set_option("comm"): 0 auto (peer memory if mapped), 1 NCCL, 2 peer memory
  int opt_lobpcg_mma = 1;        // b200_ctx_set_option("lobpcg_mma"): fp32 LOBPCG blocks on the tensor cores (3xTF32): 1 = Rayleigh-Ritz Gram on
                                 // tcgen05 (TMEM accumulators), 2 = legacy mma.sync Gram, 0 = SIMT kernels
  int opt_orth_fused = 1;        // b200_ctx_set_option("orth_fused"): 1 = one cooperative launch per CGS/DGKS orthogonalisation and a
                                 // device-resident GMRES cycle (single GPU); 0 = the three-kernel path with host-side recurrences
  int opt_cg_persistent = 1;     // b200_ctx_set_option("cg_persistent"): operators of <= 2^18 rows run the whole cg! loop in one cooperative kernel
  int opt_fold_push = 1;         // b200_ctx_set_option("fold_push"): peer path, cg! with Identity: K3 stores r's boundary rows to the neighbours itself
  int opt_pdl = 0;               // b200_ctx_set_option("pdl"): chain the kernels of a CG iteration with programmatic dependent launch
                                 // (off by default: measured SLOWER, 520 vs 560 it/s at 512^3 on 2 GPUs -- profiles/r2_summary.md)
  int opt_snake = 1;            // b200_ctx_set_option("snake"): consecutive hot kernels sweep the rows in alternating directions
  // peer-memory collectives (peer.cuh), multi-GPU contexts only
  bool peer_ok = false;
  void *peer_local = nullptr;                          // this rank's comm buffer
  void *peer_ptr[b200::kPeerMaxWorld] = {nullptr};     // all ranks' buffers mapped here (peer_ptr[rank] == peer_local)
  b200::PeerView peer_view;
  unsigned long long ar_seq = 0, halo_seq = 0;         // sequence numbers (identical on all ranks)
  // optional per-kernel-class event timing (b200_ctx_profile_*)
  bool prof_on = false;
  std::vector<cudaEvent_t> prof_ev;     // pool of event pairs
  std::vector<int> prof_slot;           // slot of each recorded pair
  size_t prof_used = 0;
  double prof_ms[4] = {0, 0, 0, 0};
  int64_t prof_n[4] = {0, 0, 0, 0};
  void *ws = nullptr;            // grow-only solver workspace (reused across solves: no malloc in the timed path)
  size_t ws_bytes = 0;
  void *stage[2] = {nullptr, nullptr};   // grow-only device staging of the host-buffer entry points (x, b): no cudaMalloc / cudaFree per solve
  size_t stage_bytes[2] = {0, 0};
  void *orth_scal = nullptr;     // device GmScal of the op-level orthogonalize_and_normalize! (gmres.cu), allocated on first use
  int in_callback = 0;           // > 0 while an operator / preconditioner callback runs: the workspace belongs to the caller
};

namespace b200 {

constexpr int kMaxReduceWidth = 64;  // simultaneous sums per reduction (block of dots in CGS)

template <typename T>
struct dtype_of;
template <>
struct dtype_of<double> {
  static constexpr int value = B200_F64;
};
template <>
struct dtype_of<float> {
  static constexpr int value = B200_F32;
};

inline size_t dtype_size(int dtype) { return dtype == B200_F64 ? 8 : 4; }

// ---------------------------------------------------------------- device helpers
#ifdef __CUDACC__

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum of one double per thread; result valid in thread 0.  Fixed tree => deterministic.
template <int THREADS>
__device__ __forceinline__ double block_sum(double v, double *smem /* >= THREADS/32 doubles */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  v = warp_sum(v);
  if (lane == 0) smem[warp] = v;
  __syncthreads();
  double r = 0.0;
  if (warp == 0) {
    r = (lane < THREADS / 32) ? smem[lane] : 0.0;
    r = warp_sum(r);
  }
  __syncthreads();
  return r;
}

// Grid-wide deterministic reduction finish: every block calls with its partial (thread 0 holds it).
// Returns true in ALL threads of exactly one block (the last one to arrive); that block's thread 0
// receives the total in *total (sum over block slots in index order).
template <int THREADS>
__device__ __forceinline__ bool grid_reduce_finish(double block_partial, double *partials, unsigned int *ticket,
                                                   double *smem, double *total, bool system_scope = false) {
  __shared__ bool is_last;
  if (threadIdx.x == 0) {
    partials[blockIdx.x] = block_partial;
    // system_scope: the block also stored to mapped peer memory (boundary values for the neighbours); the barrier inside
    // block_sum ordered those stores before this fence, which makes them visible to the peers before the ticket is taken
    if (system_scope) __threadfence_system();
    else __threadfence();
    const unsigned int t = atomicAdd(ticket, 1u);
    is_last = (t == gridDim.x - 1);
  }
  __syncthreads();
  if (!is_last) return false;
  __threadfence();
  // fixed-order: thread t sums slots t, t+THREADS, ... then the fixed block tree
  double acc = 0.0;
  for (unsigned int i = threadIdx.x; i < gridDim.x; i += THREADS) acc += __ldcg(&partials[i]);
  acc = block_sum<THREADS>(acc, smem);
  if (threadIdx.x == 0) {
    *total = acc;
    *ticket = 0u;  // re-arm for the next reduction on this stream
  }
  return true;
}

// Streaming (read-once) loads: bypass L1 allocation and carry an L2 evict-first policy so that the
// matrix stream does not push the gathered x planes out of L2.  (On sm_100a the direct
// `.L2::evict_first` qualifier exists only for 256-bit loads; narrower loads take a cache-policy.)
__device__ __forceinline__ uint64_t policy_evict_first() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ uint64_t policy_evict_last() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
template <typename T>
__device__ __forceinline__ T ld_stream(const T *p, uint64_t pol);
template <>
__device__ __forceinline__ double ld_stream<double>(const double *p, uint64_t pol) {
  double r;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(r) : "l"(p), "l"(pol));
  return r;
}
template <>
__device__ __forceinline__ float ld_stream<float>(const float *p, uint64_t pol) {
  float r;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(r) : "l"(p), "l"(pol));
  return r;
}
template <>
__device__ __forceinline__ int ld_stream<int>(const int *p, uint64_t pol) {
  int r;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.s32 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(pol));
  return r;
}

// Programmatic dependent launch (PDL): consecutive kernels of an iteration are chained so that the blocks of kernel k+1 are
// already resident (launch latency, prologue) when kernel k ends.  A chained kernel starts with pdl_wait() -- it returns once
// the preceding grid has completed and flushed -- and lets ITS successor be scheduled with pdl_launch_dependents() when its
// row loop is done, i.e. while the grid reduction / the allreduce wait of the last block is still in flight (triggering at
// the start kept the next kernel's blocks resident for the whole kernel and cost 5 % at N = 2).  Both are no-ops for
// launches without the attribute.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_chained(bool chained, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                  Args &&...args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = chained ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
#endif  // __CUDACC__

// profiling scope: records an event pair around a launch when the context's profiler is on
int prof_flush(b200_ctx *ctx);
struct ProfScope {
  b200_ctx *ctx;
  size_t idx = 0;
  bool active = false;
  ProfScope(b200_ctx *c, int slot) : ctx(c) {
    if (!c->prof_on) return;
    if (c->prof_used + 2 > c->prof_ev.size()) {
      if (c->prof_ev.size() >= 8192) prof_flush(c);
      else {
        for (int i = 0; i < 512; ++i) {
          cudaEvent_t e;
          cudaEventCreate(&e);
          c->prof_ev.push_back(e);
        }
      }
    }
    idx = c->prof_used;
    c->prof_used += 2;
    c->prof_slot.resize(c->prof_ev.size() / 2 + 1);
    c->prof_slot[idx / 2] = slot;
    cudaEventRecord(c->prof_ev[idx], c->stream);
    active = true;
  }
  ~ProfScope() {
    if (active) cudaEventRecord(ctx->prof_ev[idx + 1], ctx->stream);
  }
};

// grow-only workspace; contents are scratch (valid until the next ws_get on this context)
inline int ws_get(b200_ctx *ctx, size_t bytes, void **out) {
  if (ctx->in_callback) {
    set_error("a solver was started on this context from inside an operator / preconditioner callback: the context's "
              "workspace is in use by the outer solve (use a second context for nested solves)");
    return B200_ERR_INVALID;
  }
  if (bytes > ctx->ws_bytes) {
    cudaStreamSynchronize(ctx->stream);
    if (ctx->ws) cudaFree(ctx->ws);
    ctx->ws = nullptr;
    ctx->ws_bytes = 0;
    cudaError_t e = cudaMalloc(&ctx->ws, bytes);
    if (e != cudaSuccess) {
      set_error("workspace cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
      return B200_ERR_ALLOC;
    }
    ctx->ws_bytes = bytes;
  }
  *out = ctx->ws;
  return B200_OK;
}
inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// grow-only staging buffer `which` (0 / 1) of the context; contents are scratch.  cudaMalloc / cudaFree per call are not an
// option on multi-GPU contexts: with CUDA-IPC peer mappings each costs tens of milliseconds (profiles/r2_summary.md section 8)
inline int stage_get(b200_ctx *ctx, int which, size_t bytes, void **out) {
  if (bytes > ctx->stage_bytes[which]) {
    cudaStreamSynchronize(ctx->stream);
    if (ctx->stage[which]) cudaFree(ctx->stage[which]);
    ctx->stage[which] = nullptr;
    ctx->stage_bytes[which] = 0;
    cudaError_t e = cudaMalloc(&ctx->stage[which], bytes);
    if (e != cudaSuccess) {
      set_error("staging cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
      return B200_ERR_ALLOC;
    }
    ctx->stage_bytes[which] = bytes;
  }
  *out = ctx->stage[which];
  return B200_OK;
}

// grid size for streaming kernels: a multiple of the SM count (148 on B200), capped by the work
inline int stream_grid(const b200_ctx *ctx, int64_t work_items, int items_per_block, int blocks_per_sm) {
  int64_t need = (work_items + items_per_block - 1) / items_per_block;
  int64_t cap = (int64_t)ctx->sm_count * blocks_per_sm;
  if (need < 1) need = 1;
  int64_t g = need < cap ? need : cap;
  if (g > kMaxPartials) g = kMaxPartials;
  return (int)g;
}

}  // namespace b200
