// spmv.cu -- mul!(y, A, x) and mul!(Y, A, X) (block SpMM) on the device CSR.
#include "spmv_dia.cuh"

using namespace b200;

namespace {

constexpr int kThreads = 256;

// y = A x.  Sub-warp (LPR lanes) per row; blocks stride the rows in interleaved chunks so that all
// resident blocks work on neighbouring rows (keeps the x planes of a stencil matrix in L2).
template <typename T, int LPR>
__global__ void __launch_bounds__(kThreads) k_spmv(const int *__restrict__ rowptr, const int *__restrict__ colind,
                                                   const T *__restrict__ vals, XView<T> xv, int64_t m,
                                                   T *__restrict__ y, const int *__restrict__ gate, int gate_mask) {
  if (gate && (*gate & gate_mask)) return;   // speculatively enqueued launch whose solver has already stopped
  constexpr int ROWS = kThreads / LPR;
  const int sub = threadIdx.x % LPR;
  const int rib = threadIdx.x / LPR;
  for (int64_t base = (int64_t)blockIdx.x * ROWS; base < m; base += (int64_t)gridDim.x * ROWS) {
    const int64_t row = base + rib;
    const bool valid = row < m;
    T s = row_dot<T, LPR>(rowptr, colind, vals, xv, valid ? row : (m - 1), sub);
    if (valid && sub == 0) y[row] = s;
  }
}

// Y = A X for a column-major block of BS vectors: each sub-warp handles one row and keeps BS
// accumulators, so A is streamed ONCE for the whole block (the CPU reference re-streams it per column).
template <typename T, int LPR, int BS>
__global__ void __launch_bounds__(kThreads) k_spmm(const int *__restrict__ rowptr, const int *__restrict__ colind,
                                                   const T *__restrict__ vals, const T *__restrict__ X, int64_t ldx,
                                                   const T *__restrict__ halo, int64_t ldh, int m_own, int64_t m,
                                                   T *__restrict__ Y, int64_t ldy) {
  constexpr int ROWS = kThreads / LPR;
  const int sub = threadIdx.x % LPR;
  const int rib = threadIdx.x / LPR;
  for (int64_t base = (int64_t)blockIdx.x * ROWS; base < m; base += (int64_t)gridDim.x * ROWS) {
    const int64_t row = base + rib;
    const bool valid = row < m;
    const int64_t r = valid ? row : (m - 1);
    const int b = __ldg(rowptr + r), e = __ldg(rowptr + r + 1);
    const uint64_t pol = policy_evict_first();
    T acc[BS];
#pragma unroll
    for (int j = 0; j < BS; ++j) acc[j] = (T)0;
    for (int k = b + sub; k < e; k += LPR) {
      const int c = ld_stream<int>(colind + k, pol);
      const T a = ld_stream<T>(vals + k, pol);
      const T *src = c < m_own ? X + c : halo + (c - m_own);
      const int64_t ld = c < m_own ? ldx : ldh;
#pragma unroll
      for (int j = 0; j < BS; ++j) acc[j] += a * __ldg(src + j * ld);
    }
#pragma unroll
    for (int j = 0; j < BS; ++j) {
#pragma unroll
      for (int o = LPR >> 1; o > 0; o >>= 1) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], o, LPR);
    }
    if (valid && sub == 0) {
#pragma unroll
      for (int j = 0; j < BS; ++j) Y[row + j * ldy] = acc[j];
    }
  }
}

// TMA-streamed y = A x (spmv_stream.cuh)
template <typename T>
struct StoreEpi {
  T *__restrict__ y;
  __device__ __forceinline__ T pre(int64_t) const { return (T)0; }
  __device__ __forceinline__ void operator()(int64_t row, T v, T) { y[row] = v; }
};
template <typename T, int LPR>
__global__ void __launch_bounds__(kStreamThreads, kStreamCtasPerSm)
    k_spmv_stream(const int *__restrict__ rowptr, const int *__restrict__ colind, const T *__restrict__ vals,
                  XView<T> xv, int64_t m, T *__restrict__ y, const int *__restrict__ gate, int gate_mask) {
  if (gate && (*gate & gate_mask)) return;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  StoreEpi<T> epi{y};
  spmv_stream_tiles<T, LPR>(rowptr, colind, vals, xv, m, epi, reinterpret_cast<StreamSmem<T> *>(smem_raw));
}

// the same on the DIA copy (spmv_dia.cuh)
template <typename T>
__global__ void __launch_bounds__(kStreamThreads, kStreamCtasPerSm)
    k_spmv_dia(DiaView<T> dv, XView<T> xv, int64_t m, T *__restrict__ y, const int *__restrict__ gate, int gate_mask) {
  if (gate && (*gate & gate_mask)) return;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  StoreEpi<T> epi{y};
  spmv_dia_tiles<T>(dv, xv, m, epi, reinterpret_cast<DiaSmem<T> *>(smem_raw));
}

template <typename T>
int launch_spmv_dia(b200_ctx *ctx, const b200_csr *A, const void *x, void *y, const int *gate, int gate_mask) {
  const int grid = stream_grid_size(ctx, A);
  const size_t smem = sizeof(DiaSmem<T>);
  B200_SMEM_ATTR_ONCE(ctx, smem, k_spmv_dia<T>);
  k_spmv_dia<T><<<grid, kStreamThreads, smem, ctx->stream>>>(make_diaview<T>(A), make_xview<T>(A, x), A->m_local,
                                                             (T *)y, gate, gate_mask);
  B200_LAUNCH_CHECK(ctx);
  return B200_OK;
}

template <typename T>
int launch_spmv_stream(b200_ctx *ctx, const b200_csr *A, const void *x, void *y, const int *gate, int gate_mask) {
  XView<T> xv = make_xview<T>(A, x);
  const int grid = stream_grid_size(ctx, A);
  const size_t smem = sizeof(StreamSmem<T>);
#define LAUNCH(L)                                                                                                 \
  do {                                                                                                            \
    B200_SMEM_ATTR_ONCE(ctx, smem, k_spmv_stream<T, L>);                                                          \
    k_spmv_stream<T, L><<<grid, kStreamThreads, smem, ctx->stream>>>(A->rowptr, A->colind, (const T *)A->vals,   \
                                                                     xv, A->m_local, (T *)y, gate, gate_mask);  \
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
  B200_LAUNCH_CHECK(ctx);
  return B200_OK;
}

template <typename T>
int launch_spmv(b200_ctx *ctx, const b200_csr *A, const void *x, void *y, const int *gate = nullptr, int gate_mask = 0) {
  if (A->m_local == 0) return B200_OK;
  if (use_dia(ctx, A)) return launch_spmv_dia<T>(ctx, A, x, y, gate, gate_mask);
  if (use_stream(ctx, A)) return launch_spmv_stream<T>(ctx, A, x, y, gate, gate_mask);
  XView<T> xv = make_xview<T>(A, x);
  const int lpr = pick_lpr(A->avg_row_nnz);
  const int rows = kThreads / lpr;
  const int grid = stream_grid(ctx, A->m_local, rows, 8);
#define LAUNCH(L)                                                                                             \
  k_spmv<T, L><<<grid, kThreads, 0, ctx->stream>>>(A->rowptr, A->colind, (const T *)A->vals, xv, A->m_local, \
                                                   (T *)y, gate, gate_mask)
  switch (lpr) {
    case 2: LAUNCH(2); break;
    case 4: LAUNCH(4); break;
    case 8: LAUNCH(8); break;
    case 16: LAUNCH(16); break;
    default: LAUNCH(32); break;
  }
#undef LAUNCH
  B200_LAUNCH_CHECK(ctx);
  return B200_OK;
}

template <typename T, int BS>
int launch_spmm_bs(b200_ctx *ctx, const b200_csr *A, const T *X, int64_t ldx, T *Y, int64_t ldy) {
  const int lpr = pick_lpr(A->avg_row_nnz);
  const int grid = stream_grid(ctx, A->m_local, kThreads / lpr, 4);
  // no halo buffer (single GPU): column indices >= m_local of a wide operator (n > m, lsqr!/lsmr!/svdl) address the rows
  // of X behind the first m_local ones -- the same aliasing make_xview does for the vector kernels
  const T *halo = A->halo ? (const T *)A->halo : X + A->m_local;
  const int64_t ldh = A->halo ? A->n_halo : ldx;
#define LAUNCH(L)                                                                                                   \
  k_spmm<T, L, BS><<<grid, kThreads, 0, ctx->stream>>>(A->rowptr, A->colind, (const T *)A->vals, X, ldx, halo, ldh, \
                                                       (int)A->m_local, A->m_local, Y, ldy)
  switch (lpr) {
    case 2: LAUNCH(2); break;
    case 4: LAUNCH(4); break;
    case 8: LAUNCH(8); break;
    case 16: LAUNCH(16); break;
    default: LAUNCH(32); break;
  }
#undef LAUNCH
  B200_LAUNCH_CHECK(ctx);
  return B200_OK;
}

template <typename T>
int launch_spmm(b200_ctx *ctx, const b200_csr *A, const T *X, int64_t ldx, T *Y, int64_t ldy, int bs) {
  // blocks of up to 16 columns per pass over A
  int done = 0;
  while (done < bs) {
    const int rem = bs - done;
    const T *Xj = X + (int64_t)done * ldx;
    T *Yj = Y + (int64_t)done * ldy;
    if (rem >= 16) { B200_TRY((launch_spmm_bs<T, 16>(ctx, A, Xj, ldx, Yj, ldy))); done += 16; }
    else if (rem >= 8) { B200_TRY((launch_spmm_bs<T, 8>(ctx, A, Xj, ldx, Yj, ldy))); done += 8; }
    else if (rem >= 4) { B200_TRY((launch_spmm_bs<T, 4>(ctx, A, Xj, ldx, Yj, ldy))); done += 4; }
    else if (rem >= 2) { B200_TRY((launch_spmm_bs<T, 2>(ctx, A, Xj, ldx, Yj, ldy))); done += 2; }
    else { B200_TRY((launch_spmm_bs<T, 1>(ctx, A, Xj, ldx, Yj, ldy))); done += 1; }
  }
  return B200_OK;
}

}  // namespace

namespace b200 {
// internal entry used by the solvers (no argument checks)
int spmv(b200_ctx *ctx, const b200_csr *A, const void *x, void *y) {
  B200_TRY(halo_exchange(ctx, A, x));
  return A->dtype == B200_F64 ? launch_spmv<double>(ctx, A, x, y) : launch_spmv<float>(ctx, A, x, y);
}
// single-GPU only: y = A x unless (*gate & gate_mask) != 0 on the device when the kernel starts (launches that a solver
// enqueues ahead of its own device-side stopping test)
int spmv_gated(b200_ctx *ctx, const b200_csr *A, const void *x, void *y, const int *gate, int gate_mask) {
  return A->dtype == B200_F64 ? launch_spmv<double>(ctx, A, x, y, gate, gate_mask)
                              : launch_spmv<float>(ctx, A, x, y, gate, gate_mask);
}
}  // namespace b200

extern "C" {

int b200_spmv(b200_ctx *ctx, const b200_csr *A, const void *x_dev, void *y_dev) {
  B200_REQUIRE(ctx && A && x_dev && y_dev, "NULL argument");
  B200_REQUIRE(x_dev != y_dev, "mul!(y, A, x): y must not alias x");
  return b200::spmv(ctx, A, x_dev, y_dev);
}

int b200_spmm(b200_ctx *ctx, const b200_csr *A, const void *X_dev, int64_t ldx, void *Y_dev, int64_t ldy, int bs) {
  B200_REQUIRE(ctx && A && X_dev && Y_dev && bs >= 1, "bad arguments");
  B200_REQUIRE(ctx->world == 1, "block SpMM is single-GPU in this version");
  B200_REQUIRE(ldx >= A->n_global && ldy >= A->m_local, "leading dimensions too small: X has size(A,2) rows, Y size(A,1)");
  B200_REQUIRE(X_dev != Y_dev, "mul!(Y, A, X): Y must not alias X");
  if (A->m_local == 0) return B200_OK;
  return A->dtype == B200_F64 ? launch_spmm<double>(ctx, A, (const double *)X_dev, ldx, (double *)Y_dev, ldy, bs)
                              : launch_spmm<float>(ctx, A, (const float *)X_dev, ldx, (float *)Y_dev, ldy, bs);
}

}  // extern "C"
