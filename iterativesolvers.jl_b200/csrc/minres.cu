// minres.cu -- minres!(x, A, b; ...) of reference src/minres.jl:200-237 (iterate :97-159) as three
// fused launches per iteration; every scalar (Lanczos coefficients, the two Givens rotations, the
// right-hand side pair, the residual and the done flag) stays in device memory (struct MrScal).
//   Ka  v_next = A v_curr - H[2] v_prev ; proj = dot(v_curr, v_next)        (:104-109)
//   Kb  v_next -= proj v_curr ; H[4] = ||v_next||  -> scalar section (:110-135,147-156) in the
//       last block: rotations, rhs update, residual, iteration counter, done flag
//   Kc  v_next *= 1/H[4] ; w_next = (v_curr - H[2] w_curr - H[1] w_prev)/H[3] ; x += rhs[1] w_next (:115,138-144)
// The vector "rotation" of :147-148 is a pointer swap done by the host (it is unconditional).
// Algorithmic bytes per iteration: nnz*(V+4) + (n+1)*4 + 14*n*V.
#include "blas1.cuh"
#include "spmv_dia.cuh"

using namespace b200;

namespace {

constexpr int kThreads = 256;

struct MrScal {
  double H[4];               // m.H (1-based H[1..4] -> H[0..3])
  double rhs[2];
  double c_prev, s_prev, c_curr, s_curr;
  double resnorm, tol, abstol, reltol;
  double sum;                // reduction in flight
  // coefficients handed to Kc (computed by the scalar section)
  double inv_h4, w_h2, w_h1, inv_h3, x_coef;
  long long iteration;       // reference counter, starts at 1 (:93)
  long long maxiter, hist_cap, n_hist;
  int done, skew, breakdown, pad;
};

__device__ __forceinline__ void givens(double f, double g, double &c, double &s, double &r) {
  if (g == 0.0) { c = 1.0; s = 0.0; r = f; return; }
  if (f == 0.0) { c = 0.0; s = 1.0; r = g; return; }
  r = hypot(f, g);
  c = f / r;
  s = g / r;
  if (fabs(f) > fabs(g) && c < 0.0) { c = -c; s = -s; r = -r; }
}

__device__ __forceinline__ void mr_after_init(MrScal *m, double rr) {          // :65-78
  const double res = sqrt(rr);
  m->resnorm = res;
  m->tol = fmax(m->reltol * res, m->abstol);
  m->H[0] = m->H[1] = m->H[2] = m->H[3] = 0.0;
  m->rhs[0] = res;
  m->rhs[1] = 0.0;
  m->c_prev = 1.0; m->s_prev = 0.0; m->c_curr = 1.0; m->s_curr = 0.0;
  m->iteration = 1;
  m->n_hist = 0;
  m->breakdown = !(res == res);
  m->done = (1 > m->maxiter) || (res <= m->tol);
  m->inv_h4 = 1.0 / res;                                                       // rmul!(v_curr, inv(resnorm)) :74
}

__device__ __forceinline__ void mr_after_proj(MrScal *m, double proj) {        // :109-110
  m->sum = proj;        // Kb reads proj from here
  m->H[2] = proj;       // real(proj) (or proj itself when skew-Hermitian and real => same)
}

// everything between the norm (:114) and the end of iterate (:156)
__device__ __forceinline__ void mr_after_norm(MrScal *m, double nn, double *hist) {
  const long long it = m->iteration;
  m->H[3] = sqrt(nn);                                                          // :114
  m->inv_h4 = 1.0 / m->H[3];                                                   // :115
  if (it > 2) {                                                                // :118-121
    m->H[0] = m->s_prev * m->H[1];
    m->H[1] = m->c_prev * m->H[1];
  }
  if (it > 1) {                                                                // :124-128
    const double tmp = -m->s_curr * m->H[1] + m->c_curr * m->H[2];
    m->H[1] = m->c_curr * m->H[1] + m->s_curr * m->H[2];
    m->H[2] = tmp;
  }
  double c, s, r;
  givens(m->H[2], m->H[3], c, s, r);                                           // :131
  m->H[2] = r;
  m->rhs[1] = -s * m->rhs[0];                                                  // :134
  m->rhs[0] = c * m->rhs[0];                                                   // :135
  m->w_h2 = (it > 1) ? m->H[1] : 0.0;                                          // :139
  m->w_h1 = (it > 2) ? m->H[0] : 0.0;                                          // :140
  m->inv_h3 = 1.0 / m->H[2];                                                   // :141
  m->x_coef = m->rhs[0];                                                       // :144
  m->c_prev = m->c_curr; m->s_prev = m->s_curr; m->c_curr = c; m->s_curr = s;  // :149
  m->rhs[0] = m->rhs[1];                                                       // :150
  m->H[1] = m->skew ? -m->H[3] : m->H[3];                                      // :153
  m->resnorm = fabs(m->rhs[1]);                                                // :156
  if (!(m->resnorm == m->resnorm)) m->breakdown = 1;
  if (hist && m->n_hist < m->hist_cap) hist[m->n_hist] = m->resnorm;
  m->n_hist += 1;
  m->iteration = it + 1;
  // Kc of THIS iteration must still run: `done` is published by k_mr_finish after Kc
}

enum { MR_INIT = 1, MR_PROJ = 2, MR_NORM = 3 };

__device__ __forceinline__ void mr_finish(int kind, MrScal *m, double total, double *hist, bool single) {
  if (!single) {
    m->sum = total;
    return;
  }
  if (kind == MR_INIT) mr_after_init(m, total);
  else if (kind == MR_PROJ) mr_after_proj(m, total);
  else mr_after_norm(m, total, hist);
}
__global__ void k_mr_scalar(int kind, MrScal *m, double *hist) {
  if (kind != MR_INIT && m->done) return;  // kernels of iterations past `done` did not produce a sum
  mr_finish(kind, m, m->sum, hist, true);
}

// v_curr = b - c (or b); ||v_curr||^2
template <typename T>
__global__ void __launch_bounds__(kThreads) k_mr_init(const T *__restrict__ b, const T *__restrict__ c, int has_c,
                                                      T *__restrict__ v, int64_t n, MrScal *m, double *partials,
                                                      unsigned int *ticket, int single) {
  __shared__ double smem[kThreads / 32];
  double acc = 0.0;
  for (int64_t i = blockIdx.x * (int64_t)kThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kThreads) {
    T vi = b[i];
    if (has_c) vi = vi - c[i];
    v[i] = vi;
    acc += (double)vi * (double)vi;
  }
  acc = block_sum<kThreads>(acc, smem);
  double total;
  if (grid_reduce_finish<kThreads>(acc, partials, ticket, smem, &total) && threadIdx.x == 0)
    mr_finish(MR_INIT, m, total, nullptr, single);
}

template <typename T>
__global__ void __launch_bounds__(kThreads) k_mr_scale(T *__restrict__ v, int64_t n, const MrScal *__restrict__ m) {
  const T inv = (T)m->inv_h4;
  for (int64_t i = blockIdx.x * (int64_t)kThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kThreads)
    v[i] = v[i] * inv;
}

// Ka
template <typename T, int LPR>
__global__ void __launch_bounds__(kThreads) k_mr_spmv(const int *__restrict__ rowptr, const int *__restrict__ colind,
                                                      const T *__restrict__ vals, XView<T> xv,
                                                      const T *__restrict__ v_prev, T *__restrict__ v_next,
                                                      int64_t n, MrScal *m, double *partials, unsigned int *ticket,
                                                      int single) {
  if (m->done) return;
  __shared__ double smem[kThreads / 32];
  constexpr int ROWS = kThreads / LPR;
  const int sub = threadIdx.x % LPR, rib = threadIdx.x / LPR;
  const bool use_prev = m->iteration > 1;
  const T h2 = (T)m->H[1];
  double acc = 0.0;
  for (int64_t base = (int64_t)blockIdx.x * ROWS; base < n; base += (int64_t)gridDim.x * ROWS) {
    const int64_t row = base + rib;
    const bool valid = row < n;
    T t = row_dot<T, LPR>(rowptr, colind, vals, xv, valid ? row : (n - 1), sub);
    if (valid && sub == 0) {
      if (use_prev) t = t - h2 * v_prev[row];                                   // axpy!(-H[2], v_prev, v_next) :106
      v_next[row] = t;
      acc += (double)xv.x[row] * (double)t;                                     // dot(v_curr, v_next) :109
    }
  }
  acc = block_sum<kThreads>(acc, smem);
  double total;
  if (grid_reduce_finish<kThreads>(acc, partials, ticket, smem, &total) && threadIdx.x == 0)
    mr_finish(MR_PROJ, m, total, nullptr, single);
}

// Ka, TMA-streamed form (spmv_stream.cuh)
template <typename T>
struct MrEpi {
  T *__restrict__ v_next;
  const T *__restrict__ v_prev;
  const T *__restrict__ v_curr;
  T h2;
  bool use_prev;
  double acc;
  __device__ __forceinline__ T pre(int64_t row) const { return use_prev ? v_prev[row] : (T)0; }
  __device__ __forceinline__ void operator()(int64_t row, T t, T vp) {
    if (use_prev) t = t - h2 * vp;
    v_next[row] = t;
    acc += (double)v_curr[row] * (double)t;
  }
};
template <typename T, int LPR>
__global__ void __launch_bounds__(kStreamThreads, kStreamCtasPerSm)
    k_mr_spmv_stream(const int *__restrict__ rowptr, const int *__restrict__ colind, const T *__restrict__ vals,
                     XView<T> xv, const T *__restrict__ v_prev, T *__restrict__ v_next, int64_t n, MrScal *m,
                     double *partials, unsigned int *ticket, int single) {
  if (m->done) return;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ double red[kStreamThreads / 32];
  MrEpi<T> epi{v_next, v_prev, xv.x, (T)m->H[1], m->iteration > 1, 0.0};
  spmv_stream_tiles<T, LPR>(rowptr, colind, vals, xv, n, epi, reinterpret_cast<StreamSmem<T> *>(smem_raw));
  const double acc = block_sum<kStreamThreads>(epi.acc, red);
  double total;
  if (grid_reduce_finish<kStreamThreads>(acc, partials, ticket, red, &total) && threadIdx.x == 0)
    mr_finish(MR_PROJ, m, total, nullptr, single);
}

// Ka on the DIA copy (spmv_dia.cuh): bitwise the result of k_mr_spmv_stream<T, 1>
template <typename T>
__global__ void __launch_bounds__(kStreamThreads, kStreamCtasPerSm)
    k_mr_spmv_dia(DiaView<T> dv, XView<T> xv, const T *__restrict__ v_prev, T *__restrict__ v_next, int64_t n,
                  MrScal *m, double *partials, unsigned int *ticket, int single) {
  if (m->done) return;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ double red[kStreamThreads / 32];
  MrEpi<T> epi{v_next, v_prev, xv.x, (T)m->H[1], m->iteration > 1, 0.0};
  spmv_dia_tiles<T>(dv, xv, n, epi, reinterpret_cast<DiaSmem<T> *>(smem_raw));
  const double acc = block_sum<kStreamThreads>(epi.acc, red);
  double total;
  if (grid_reduce_finish<kStreamThreads>(acc, partials, ticket, red, &total) && threadIdx.x == 0)
    mr_finish(MR_PROJ, m, total, nullptr, single);
}

// Kb
template <typename T>
__global__ void __launch_bounds__(kThreads) k_mr_orth(const T *__restrict__ v_curr, T *__restrict__ v_next, int64_t n,
                                                      MrScal *m, double *hist, double *partials, unsigned int *ticket,
                                                      int single) {
  if (m->done) return;
  __shared__ double smem[kThreads / 32];
  const T proj = (T)m->sum;
  double acc = 0.0;
  for (int64_t i = blockIdx.x * (int64_t)kThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kThreads) {
    const T t = v_next[i] - proj * v_curr[i];                                   // axpy!(-proj, v_curr, v_next) :111
    v_next[i] = t;
    acc += (double)t * (double)t;
  }
  acc = block_sum<kThreads>(acc, smem);
  double total;
  if (grid_reduce_finish<kThreads>(acc, partials, ticket, smem, &total) && threadIdx.x == 0)
    mr_finish(MR_NORM, m, total, hist, single);
}

// Kc
template <typename T>
__global__ void __launch_bounds__(kThreads) k_mr_update(T *__restrict__ v_next, const T *__restrict__ v_curr,
                                                        const T *__restrict__ w_curr, const T *__restrict__ w_prev,
                                                        T *__restrict__ w_next, T *__restrict__ x, int64_t n,
                                                        const MrScal *__restrict__ m) {
  if (m->done) return;
  const T inv4 = (T)m->inv_h4, h2 = (T)m->w_h2, h1 = (T)m->w_h1, inv3 = (T)m->inv_h3, xc = (T)m->x_coef;
  const bool u2 = m->iteration > 2, u3 = m->iteration > 3;   // iteration was already incremented by the scalar section
  for (int64_t i = blockIdx.x * (int64_t)kThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kThreads) {
    v_next[i] = v_next[i] * inv4;                                               // :115
    T w = v_curr[i];                                                            // copyto!(w_next, v_curr) :138
    if (u2) w = w - h2 * w_curr[i];                                             // :139
    if (u3) w = w - h1 * w_prev[i];                                             // :140
    w = w * inv3;                                                               // :141
    w_next[i] = w;
    x[i] = x[i] + xc * w;                                                       // :144
  }
}

// publishes `done` for the NEXT iteration (reference checks done() at the top of iterate, :99)
__global__ void k_mr_done(MrScal *m) {
  if (m->done) return;
  m->done = (m->iteration > m->maxiter) || (m->resnorm <= m->tol) || m->breakdown;
}

template <typename T>
int minres_impl(b200_ctx *ctx, const b200_csr *A, T *x, const T *b, const b200_minres_opts *o, b200_result *res,
                double *resnorm_host, int64_t resnorm_cap) {
  cudaStream_t st = ctx->stream;
  const int64_t n = A->m_local;
  const double eps = sizeof(T) == 8 ? 2.220446049250313e-16 : 1.1920928955078125e-07;
  const double reltol = o->reltol < 0 ? sqrt(eps) : o->reltol;
  const int64_t maxiter = o->maxiter < 0 ? A->n_global : o->maxiter;
  const int64_t hist_cap = resnorm_host ? std::min<int64_t>(resnorm_cap, maxiter) : 0;
  const int single = ctx->world == 1;
  const int dt = dtype_of<T>::value;

  const size_t vec_bytes = align_up(sizeof(T) * (size_t)std::max<int64_t>(n, 1), 256);
  const size_t hist_bytes = align_up(sizeof(double) * (size_t)std::max<int64_t>(hist_cap, 1), 256);
  void *ws = nullptr;
  B200_TRY(ws_get(ctx, 6 * vec_bytes + 512 + hist_bytes, &ws));
  char *p = (char *)ws;
  T *v[3], *w[3];
  for (int i = 0; i < 3; ++i) { v[i] = (T *)p; p += vec_bytes; }
  for (int i = 0; i < 3; ++i) { w[i] = (T *)p; p += vec_bytes; }
  MrScal *m = (MrScal *)p; p += 512;
  double *hist = hist_cap ? (double *)p : nullptr;
  T *v_prev = v[0], *v_curr = v[1], *v_next = v[2];
  T *w_prev = w[0], *w_curr = w[1], *w_next = w[2];

  MrScal h;
  memset(&h, 0, sizeof(h));
  h.abstol = o->abstol;
  h.reltol = reltol;
  h.maxiter = maxiter;
  h.hist_cap = hist_cap;
  h.skew = o->skew_hermitian;
  B200_CUDA(cudaMemcpyAsync(m, &h, sizeof(h), cudaMemcpyHostToDevice, st));
  const int gv = stream_grid(ctx, n, kThreads * 2, 8);
  const int lpr = pick_lpr(A->avg_row_nnz);
  const int gs = stream_grid(ctx, n, kThreads / lpr, 8);

  auto after = [&](int kind) -> int {
    if (single) return B200_OK;
    B200_TRY(allreduce_sum_dev(ctx, &m->sum, 1));
    k_mr_scalar<<<1, 1, 0, st>>>(kind, m, hist);
    B200_LAUNCH_CHECK(ctx);
    return B200_OK;
  };

  // minres_iterable! (:39-89)
  int64_t mv_products = 0;
  if (!o->initially_zero) {                                                      // :58-63
    B200_TRY(spmv(ctx, A, x, v_next));
    mv_products = 1;
  }
  k_mr_init<T><<<gv, kThreads, 0, st>>>(b, v_next, o->initially_zero ? 0 : 1, v_curr, n, m, ctx->red.partials,
                                         ctx->red.ticket, single);
  B200_LAUNCH_CHECK(ctx);
  B200_TRY(after(MR_INIT));
  k_mr_scale<T><<<gv, kThreads, 0, st>>>(v_curr, n, m);                           // :74
  B200_LAUNCH_CHECK(ctx);
  B200_TRY(fill(ctx, n, 0.0, w_prev, dt));
  B200_TRY(fill(ctx, n, 0.0, w_curr, dt));

  int64_t enqueued = 0;
  const int check_every = 16;
  int *h_done = ctx->h_flags;
  for (;;) {
    B200_CUDA(cudaMemcpyAsync(h_done, &m->done, sizeof(int), cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));
    if (*h_done || enqueued >= maxiter) break;
    const int64_t batch = std::min<int64_t>(check_every, maxiter - enqueued);
    for (int64_t it = 0; it < batch; ++it) {
      B200_TRY(halo_exchange(ctx, A, v_curr));
      XView<T> xv = make_xview<T>(A, v_curr);
      if (use_dia(ctx, A)) {
        const int grid = stream_grid_size(ctx, A);
        const size_t smem = sizeof(DiaSmem<T>);
        ProfScope prof(ctx, 0);
        B200_SMEM_ATTR_ONCE(ctx, smem, k_mr_spmv_dia<T>);
        k_mr_spmv_dia<T><<<grid, kStreamThreads, smem, st>>>(make_diaview<T>(A), xv, v_prev, v_next, n, m,
                                                             ctx->red.partials, ctx->red.ticket, single);
      } else if (use_stream(ctx, A)) {
        const int grid = stream_grid_size(ctx, A);
        const size_t smem = sizeof(StreamSmem<T>);
        ProfScope prof(ctx, 0);
#define LAUNCH(L)                                                                                                  \
  do {                                                                                                             \
    B200_SMEM_ATTR_ONCE(ctx, smem, k_mr_spmv_stream<T, L>);                                                        \
    k_mr_spmv_stream<T, L><<<grid, kStreamThreads, smem, st>>>(A->rowptr, A->colind, (const T *)A->vals, xv,       \
                                                                v_prev, v_next, n, m, ctx->red.partials,           \
                                                                ctx->red.ticket, single);                          \
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
#define LAUNCH(L)                                                                                            \
  k_mr_spmv<T, L><<<gs, kThreads, 0, st>>>(A->rowptr, A->colind, (const T *)A->vals, xv, v_prev, v_next, n, m, \
                                           ctx->red.partials, ctx->red.ticket, single)
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
      B200_TRY(after(MR_PROJ));
      {
        ProfScope prof(ctx, 1);
        k_mr_orth<T><<<gv, kThreads, 0, st>>>(v_curr, v_next, n, m, hist, ctx->red.partials, ctx->red.ticket, single);
      }
      B200_LAUNCH_CHECK(ctx);
      B200_TRY(after(MR_NORM));
      {
        ProfScope prof(ctx, 2);
        k_mr_update<T><<<gv, kThreads, 0, st>>>(v_next, v_curr, w_curr, w_prev, w_next, x, n, m);
      }
      B200_LAUNCH_CHECK(ctx);
      k_mr_done<<<1, 1, 0, st>>>(m);
      B200_LAUNCH_CHECK(ctx);
      // :147-148  (unconditional pointer rotation; harmless after `done`)
      T *t = v_prev; v_prev = v_curr; v_curr = v_next; v_next = t;
      t = w_prev; w_prev = w_curr; w_curr = w_next; w_next = t;
    }
    enqueued += batch;
  }
  B200_CUDA(cudaMemcpyAsync(&h, m, sizeof(h), cudaMemcpyDeviceToHost, st));
  B200_CUDA(cudaStreamSynchronize(st));
  const int64_t iters = h.iteration - 1;
  if (res) {
    res->iters = iters;
    res->mvps = mv_products + iters;
    res->isconverged = h.resnorm <= h.tol;
    res->status = h.breakdown ? B200_ERR_BREAKDOWN : 0;
    res->tol = h.tol;
    res->residual = h.resnorm;
    res->n_resnorm = std::min<int64_t>(iters, hist_cap);
  }
  if (hist_cap && iters > 0) {
    B200_CUDA(cudaMemcpyAsync(resnorm_host, hist, sizeof(double) * std::min<int64_t>(iters, hist_cap),
                              cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));
  }
  return B200_OK;
}

}  // namespace

extern "C" {

int b200_minres_solve(b200_ctx *ctx, const b200_csr *A, void *x_dev, const void *b_dev, const b200_minres_opts *opts,
                      b200_result *res, double *resnorm_host, int64_t resnorm_cap) {
  B200_REQUIRE(ctx && A && x_dev && b_dev && opts, "NULL argument");
  B200_REQUIRE(A->ctx == ctx, "operator belongs to another context");
  B200_REQUIRE(is_square(A), "this solver needs a square operator (got %lld x %lld)", (long long)A->m_global,
               (long long)A->n_global);
  B200_CUDA(cudaSetDevice(ctx->device));
  return A->dtype == B200_F64
             ? minres_impl<double>(ctx, A, (double *)x_dev, (const double *)b_dev, opts, res, resnorm_host, resnorm_cap)
             : minres_impl<float>(ctx, A, (float *)x_dev, (const float *)b_dev, opts, res, resnorm_host, resnorm_cap);
}

}  // extern "C"
