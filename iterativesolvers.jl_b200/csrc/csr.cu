// csr.cu -- building the device operator: SparseMatrixCSC -> CSR int32 (device transpose),
// CSR row slabs, the on-device laplace_matrix generator, halo plans and the halo exchange.
#include <algorithm>
#include <climits>
#include <cub/cub.cuh>

#include "csr.cuh"

using namespace b200;

// ------------------------------------------------------------------------------------------
// halo plan (pure host code)
// ------------------------------------------------------------------------------------------
void b200_halo_plan::rebuild_concat() {
  halo_sorted.clear();
  recv_offset.assign(world + 1, 0);
  for (int o = 0; o < world; ++o) {
    recv_offset[o] = (int64_t)halo_sorted.size();
    halo_sorted.insert(halo_sorted.end(), recv_cols[o].begin(), recv_cols[o].end());
  }
  recv_offset[world] = (int64_t)halo_sorted.size();
}

static int plan_owner(const b200_halo_plan *p, int64_t col) {
  // row_offsets ascending; owner = last r with row_offsets[r] <= col
  auto it = std::upper_bound(p->row_offsets.begin(), p->row_offsets.end(), col);
  return (int)(it - p->row_offsets.begin()) - 1;
}

static void plan_finish_scan(b200_halo_plan *p, std::vector<int64_t> &cols) {
  std::sort(cols.begin(), cols.end());
  cols.erase(std::unique(cols.begin(), cols.end()), cols.end());
  for (auto &v : p->recv_cols) v.clear();
  for (int64_t c : cols) p->recv_cols[plan_owner(p, c)].push_back(c);
  p->rebuild_concat();
}

extern "C" {

int b200_halo_plan_create(int rank, int world, const int64_t *row_offsets, b200_halo_plan **out) {
  B200_REQUIRE(out && row_offsets && world >= 1 && rank >= 0 && rank < world, "bad arguments");
  for (int r = 0; r < world; ++r)
    B200_REQUIRE(row_offsets[r] <= row_offsets[r + 1], "row_offsets must be non-decreasing");
  auto *p = new b200_halo_plan();
  p->rank = rank;
  p->world = world;
  p->row_offsets.assign(row_offsets, row_offsets + world + 1);
  p->recv_cols.resize(world);
  p->send_cols.resize(world);
  p->rebuild_concat();
  *out = p;
  return B200_OK;
}

int b200_halo_plan_scan(b200_halo_plan *p, int64_t m_local, const void *rowptr, const void *colind, int idx_bytes,
                        int base) {
  B200_REQUIRE(p && rowptr && (idx_bytes == 4 || idx_bytes == 8), "bad arguments");
  const int64_t lo = p->row_offsets[p->rank], hi = p->row_offsets[p->rank + 1];
  B200_REQUIRE(hi - lo == m_local, "m_local does not match the plan's slab");
  const int64_t n_global = p->row_offsets[p->world];
  int64_t nnz = idx_bytes == 8 ? ((const int64_t *)rowptr)[m_local] - ((const int64_t *)rowptr)[0]
                               : (int64_t)((const int32_t *)rowptr)[m_local] - ((const int32_t *)rowptr)[0];
  std::vector<int64_t> cols;
  for (int64_t k = 0; k < nnz; ++k) {
    int64_t c = (idx_bytes == 8 ? ((const int64_t *)colind)[k] : (int64_t)((const int32_t *)colind)[k]) - base;
    B200_REQUIRE(c >= 0 && c < n_global, "column index %lld out of range", (long long)c);
    if (c < lo || c >= hi) {
      // cheap de-dup of runs; full de-dup after the sort
      if (cols.empty() || cols.back() != c) cols.push_back(c);
    }
  }
  plan_finish_scan(p, cols);
  return B200_OK;
}

int b200_halo_plan_scan_laplacian(b200_halo_plan *p, int64_t N, int dims) {
  B200_REQUIRE(p && N >= 1 && dims >= 1 && dims <= 6, "bad arguments");
  int64_t n = 1, stride[8];
  for (int d = 0; d < dims; ++d) {
    stride[d] = n;
    n *= N;
  }
  B200_REQUIRE(n == p->row_offsets[p->world], "N^dims != n_global of the plan");
  const int64_t lo = p->row_offsets[p->rank], hi = p->row_offsets[p->rank + 1];
  std::vector<int64_t> cols;
  for (int d = 0; d < dims; ++d) {
    const int64_t s = stride[d];
    // rows whose -s neighbour falls below the slab: r in [lo, min(lo+s, hi)); +s above: r in [max(hi-s,lo), hi)
    for (int64_t r = lo; r < std::min(lo + s, hi); ++r)
      if ((r / s) % N > 0 && r - s < lo) cols.push_back(r - s);
    for (int64_t r = std::max(hi - s, lo); r < hi; ++r)
      if ((r / s) % N < N - 1 && r + s >= hi) cols.push_back(r + s);
  }
  plan_finish_scan(p, cols);
  return B200_OK;
}

int64_t b200_halo_plan_recv_count(const b200_halo_plan *p, int owner) {
  if (!p || owner < 0 || owner >= p->world) return -1;
  return (int64_t)p->recv_cols[owner].size();
}
int b200_halo_plan_recv_cols(const b200_halo_plan *p, int owner, int64_t *cols_out) {
  B200_REQUIRE(p && owner >= 0 && owner < p->world, "bad arguments");
  if (!p->recv_cols[owner].empty()) {
    B200_REQUIRE(cols_out, "cols_out is NULL");
    memcpy(cols_out, p->recv_cols[owner].data(), sizeof(int64_t) * p->recv_cols[owner].size());
  }
  return B200_OK;
}
int b200_halo_plan_set_send(b200_halo_plan *p, int peer, const int64_t *cols, int64_t count) {
  B200_REQUIRE(p && peer >= 0 && peer < p->world && count >= 0 && (count == 0 || cols), "bad arguments");
  const int64_t lo = p->row_offsets[p->rank], hi = p->row_offsets[p->rank + 1];
  for (int64_t i = 0; i < count; ++i)
    B200_REQUIRE(cols[i] >= lo && cols[i] < hi, "peer %d asks for row %lld that rank %d does not own", peer,
                 (long long)cols[i], p->rank);
  p->send_cols[peer].assign(cols, cols + count);
  return B200_OK;
}
int64_t b200_halo_plan_send_count(const b200_halo_plan *p, int peer) {
  if (!p || peer < 0 || peer >= p->world) return -1;
  return (int64_t)p->send_cols[peer].size();
}
int b200_halo_plan_send_range(const b200_halo_plan *p, int peer, int64_t *lo_local) {
  if (!p || peer < 0 || peer >= p->world) return -1;
  const std::vector<int64_t> &c = p->send_cols[peer];
  if (c.empty()) return 0;
  for (size_t k = 1; k < c.size(); ++k)
    if (c[k] != c[0] + (int64_t)k) return 0;
  if (lo_local) *lo_local = c[0] - p->row_offsets[p->rank];
  return 1;
}
int64_t b200_halo_plan_n_halo(const b200_halo_plan *p) { return p ? (int64_t)p->halo_sorted.size() : -1; }
int64_t b200_halo_plan_local_index(const b200_halo_plan *p, int64_t c) {
  if (!p) return -1;
  const int64_t lo = p->row_offsets[p->rank], hi = p->row_offsets[p->rank + 1];
  if (c >= lo && c < hi) return c - lo;
  auto it = std::lower_bound(p->halo_sorted.begin(), p->halo_sorted.end(), c);
  if (it == p->halo_sorted.end() || *it != c) return -1;
  return (hi - lo) + (int64_t)(it - p->halo_sorted.begin());
}
int b200_halo_plan_destroy(b200_halo_plan *p) {
  delete p;
  return B200_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------
// device kernels for construction
// ------------------------------------------------------------------------------------------
namespace {

template <typename I>
__global__ void k_count_rows(const I *__restrict__ rowval, int64_t nnz, int base, int64_t m, int *__restrict__ cnt,
                             int *__restrict__ err) {
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < nnz; k += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = (int64_t)rowval[k] - base;
    if (r < 0 || r >= m) {
      *err = 1;
      continue;
    }
    atomicAdd(&cnt[r], 1);
  }
}

// expand colptr into a per-nonzero column id and the row key used by the stable sort
template <typename I>
__global__ void k_expand_cols(const I *__restrict__ colptr, int64_t n, int base, const I *__restrict__ rowval,
                              unsigned int *__restrict__ key_row, int *__restrict__ col_of) {
  // one warp per column (columns are short); lanes stride the column's entries
  const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t j = warp; j < n; j += nwarps) {
    const int64_t b = (int64_t)colptr[j] - base, e = (int64_t)colptr[j + 1] - base;
    for (int64_t k = b + lane; k < e; k += 32) {
      col_of[k] = (int)j;
      key_row[k] = (unsigned int)((int64_t)rowval[k] - base);
    }
  }
}

template <typename T, typename TI>
__global__ void k_gather_vals(const int *__restrict__ perm, const TI *__restrict__ nz_in, int64_t nnz,
                              T *__restrict__ vals) {
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < nnz; k += (int64_t)gridDim.x * blockDim.x)
    vals[k] = (T)nz_in[perm[k]];
}
__global__ void k_gather_int(const int *__restrict__ perm, const int *__restrict__ in, int64_t nnz,
                             int *__restrict__ out) {
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < nnz; k += (int64_t)gridDim.x * blockDim.x)
    out[k] = in[perm[k]];
}
__global__ void k_iota(int *p, int64_t n) {
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x)
    p[k] = (int)k;
}

// CSR slab: global column -> local extended index (binary search of the sorted halo list)
template <typename I>
__global__ void k_remap_cols(const I *__restrict__ col_in, int64_t nnz, int base, int64_t lo, int64_t hi,
                             const int64_t *__restrict__ halo_sorted, int64_t n_halo, int *__restrict__ col_out,
                             int *__restrict__ err) {
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < nnz; k += (int64_t)gridDim.x * blockDim.x) {
    const int64_t c = (int64_t)col_in[k] - base;
    if (c >= lo && c < hi) {
      col_out[k] = (int)(c - lo);
    } else {
      int64_t a = 0, b = n_halo;
      while (a < b) {
        const int64_t mid = (a + b) >> 1;
        if (halo_sorted[mid] < c) a = mid + 1; else b = mid;
      }
      if (a >= n_halo || halo_sorted[a] != c) {
        *err = 2;
        col_out[k] = 0;
      } else {
        col_out[k] = (int)((hi - lo) + a);
      }
    }
  }
}

template <typename I>
__global__ void k_rowptr_convert(const I *__restrict__ in, int64_t m, int *__restrict__ out) {
  const I first = in[0];
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k <= m; k += (int64_t)gridDim.x * blockDim.x)
    out[k] = (int)(in[k] - first);
}

template <typename T, typename TI>
__global__ void k_convert_vals(const TI *__restrict__ in, int64_t nnz, T *__restrict__ out) {
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < nnz; k += (int64_t)gridDim.x * blockDim.x)
    out[k] = (T)in[k];
}

// laplace_matrix(T,N,dims) on device: count pass and fill pass, one thread per local row
struct LapGeom {
  int64_t N;
  int dims;
  int64_t stride[6];
};
__global__ void k_lap_count(LapGeom g, int64_t row_begin, int64_t m, int *__restrict__ cnt) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    int64_t q = row_begin + i, rem = q;
    int c = 1;
    for (int d = 0; d < g.dims; ++d) {
      const int64_t x = rem % g.N;
      rem /= g.N;
      c += (x > 0) + (x < g.N - 1);
    }
    cnt[i] = c;
  }
}
template <typename T>
__global__ void k_lap_fill(LapGeom g, int64_t row_begin, int64_t m, const int *__restrict__ rowptr,
                           const int64_t *__restrict__ halo_sorted, int64_t n_halo, int *__restrict__ colind,
                           T *__restrict__ vals) {
  const int64_t lo = row_begin, hi = row_begin + m;
  auto local = [&](int64_t c) -> int {
    if (c >= lo && c < hi) return (int)(c - lo);
    int64_t a = 0, b = n_halo;
    while (a < b) {
      const int64_t mid = (a + b) >> 1;
      if (halo_sorted[mid] < c) a = mid + 1; else b = mid;
    }
    return (int)(m + a);
  };
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t q = row_begin + i;
    int64_t coord[6], rem = q;
    for (int d = 0; d < g.dims; ++d) {
      coord[d] = rem % g.N;
      rem /= g.N;
    }
    int k = rowptr[i];
    for (int d = g.dims - 1; d >= 0; --d)
      if (coord[d] > 0) {
        colind[k] = local(q - g.stride[d]);
        vals[k] = (T)-1;
        ++k;
      }
    colind[k] = (int)i;
    vals[k] = (T)(2 * g.dims);
    ++k;
    for (int d = 0; d < g.dims; ++d)
      if (coord[d] < g.N - 1) {
        colind[k] = local(q + g.stride[d]);
        vals[k] = (T)-1;
        ++k;
      }
  }
}

template <typename T>
__global__ void k_diag(const int *__restrict__ rowptr, const int *__restrict__ colind, const T *__restrict__ vals,
                       int64_t m, T *__restrict__ diag) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    T d = (T)0;
    for (int k = rowptr[i]; k < rowptr[i + 1]; ++k)
      if (colind[k] == (int)i) d += vals[k];
    diag[i] = d;
  }
}

__global__ void k_row_stats(const int *__restrict__ rowptr, int64_t m, int *__restrict__ max_len) {
  int local = 0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x)
    local = max(local, rowptr[i + 1] - rowptr[i]);
  for (int o = 16; o > 0; o >>= 1) local = max(local, __shfl_xor_sync(0xffffffffu, local, o));
  if ((threadIdx.x & 31) == 0) atomicMax(max_len, local);
}

// max over uniform tiles of R rows of the tile's nonzero count
__global__ void k_tile_max(const int *__restrict__ rowptr, int64_t m, int R, int *__restrict__ out) {
  const int64_t ntiles = (m + R - 1) / R;
  int local = 0;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < ntiles; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r0 = t * R, r1 = (r0 + R < m) ? r0 + R : m;
    local = max(local, rowptr[r1] - rowptr[r0]);
  }
  for (int o = 16; o > 0; o >>= 1) local = max(local, __shfl_xor_sync(0xffffffffu, local, o));
  if ((threadIdx.x & 31) == 0) atomicMax(out, local);
}

// DIA detection, pass 1 (one read of rowptr/colind): the set of distinct col - row offsets, at most kDiaMaxDiags of
// them, and whether every row's columns are strictly ascending.  Each block collects its offsets in a shared set
// (insertion by CAS into the first free slot: no value lands in two slots) and merges it into the global set the same
// way.  flags[0]: more than kDiaMaxDiags offsets; flags[1]: a row with unsorted or repeated columns.
constexpr int kDiaEmpty = INT_MIN;   // col - row of two int32 indices in [0, 2^31) is > INT_MIN
__device__ __forceinline__ bool dia_set_insert(int *set, int v) {
  for (int s = 0; s < kDiaMaxDiags; ++s) {
    const int cur = *(volatile int *)&set[s];
    if (cur == v) return true;
    if (cur == kDiaEmpty) {
      const int old = atomicCAS(&set[s], kDiaEmpty, v);
      if (old == kDiaEmpty || old == v) return true;
    }
  }
  return false;
}
__global__ void k_dia_scan(const int *__restrict__ rowptr, const int *__restrict__ colind, int64_t m,
                           int *__restrict__ gset, int *__restrict__ flags) {
  __shared__ int set[kDiaMaxDiags];
  __shared__ int bad[2];
  if (threadIdx.x < kDiaMaxDiags) set[threadIdx.x] = kDiaEmpty;
  if (threadIdx.x < 2) bad[threadIdx.x] = 0;
  __syncthreads();
  int last = kDiaEmpty;   // this thread's last inserted offset (rows of a stencil repeat the same few)
  bool over = false, unsorted = false;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < m && !over; i += (int64_t)gridDim.x * blockDim.x) {
    const int b = rowptr[i], e = rowptr[i + 1];
    int prev = -1;
    for (int k = b; k < e; ++k) {
      const int c = colind[k];
      unsorted |= c <= prev;
      prev = c;
      const int v = c - (int)i;
      if (v != last && !dia_set_insert(set, v)) {
        over = true;
        break;
      }
      last = v;
    }
  }
  if (over) bad[0] = 1;
  if (unsorted) bad[1] = 1;
  __syncthreads();
  if (threadIdx.x < kDiaMaxDiags && set[threadIdx.x] != kDiaEmpty && !dia_set_insert(gset, set[threadIdx.x]))
    flags[0] = 1;
  if (threadIdx.x < 2 && bad[threadIdx.x]) flags[threadIdx.x] = 1;
}

// DIA pass 2 (one read of the CSR): scatter the values, set the presence bits.  flags[2]: an offset outside the set
// or a bit set twice (cannot happen after a clean pass 1; checked so that a DIA copy is never wrong).
struct DiaOffsets {
  int off[kDiaMaxDiags];
  int ndiag;
};
template <typename T>
__global__ void k_dia_fill(const int *__restrict__ rowptr, const int *__restrict__ colind, const T *__restrict__ vals,
                           int64_t m, DiaOffsets o, int64_t ld, T *__restrict__ dvals, uint8_t *__restrict__ dmask,
                           int *__restrict__ flags) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < m; i += (int64_t)gridDim.x * blockDim.x) {
    unsigned int bits = 0;
    for (int k = rowptr[i]; k < rowptr[i + 1]; ++k) {
      const int v = colind[k] - (int)i;
      int d = 0;
      while (d < o.ndiag && o.off[d] != v) ++d;
      if (d == o.ndiag || ((bits >> d) & 1u)) {
        flags[2] = 1;
        continue;
      }
      bits |= 1u << d;
      dvals[d * ld + i] = vals[k];
    }
    dmask[i] = (uint8_t)bits;
  }
}

template <typename T>
__global__ void k_pack(const int *__restrict__ idx, const T *__restrict__ x, int64_t n, T *__restrict__ out) {
  for (int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x)
    out[k] = x[idx[k]];
}

int grid_for(const b200_ctx *ctx, int64_t n, int threads = 256) {
  int64_t g = (n + threads - 1) / threads;
  int64_t cap = (int64_t)ctx->sm_count * 8;
  if (g < 1) g = 1;
  return (int)(g < cap ? g : cap);
}

void free_dia(b200_csr *A) {
  cudaFree(A->dia_vals);
  cudaFree(A->dia_mask);
  A->dia_vals = nullptr;
  A->dia_mask = nullptr;
  A->dia_ndiag = 0;
  A->dia_m_pad = 0;
}

// Builds the DIA copy of a square single-GPU operator whose nonzeros lie on at most kDiaMaxDiags diagonals, when that
// copy is at most 0.8x the CSR bytes.  Not building it is never an error: a failed allocation leaves the CSR alone.
int build_dia(b200_ctx *ctx, b200_csr *A) {
  const int64_t m = A->m_local;
  if (ctx->world != 1 || A->n_halo != 0 || !is_square(A) || m == 0 || A->nnz == 0 || A->stream_lpr != 1) return B200_OK;
  cudaStream_t st = ctx->stream;
  int *d_buf = nullptr;   // [0, 8): offset set, [8, 11): flags
  B200_CUDA(cudaMalloc(&d_buf, sizeof(int) * 16));
  std::vector<int> h_init(16, 0);
  for (int s = 0; s < kDiaMaxDiags; ++s) h_init[s] = kDiaEmpty;
  auto done = [&](int s) {
    cudaFree(d_buf);
    return s;
  };
#define CK(call)                                                                        \
  do {                                                                                  \
    cudaError_t _e = (call);                                                            \
    if (_e != cudaSuccess) {                                                            \
      set_error("%s:%d %s in `%s`", __FILE__, __LINE__, cudaGetErrorString(_e), #call); \
      free_dia(A);                                                                      \
      return done(B200_ERR_CUDA);                                                       \
    }                                                                                   \
  } while (0)
  CK(cudaMemcpyAsync(d_buf, h_init.data(), sizeof(int) * 16, cudaMemcpyHostToDevice, st));
  k_dia_scan<<<grid_for(ctx, m), 256, 0, st>>>(A->rowptr, A->colind, m, d_buf, d_buf + kDiaMaxDiags);
  ctx->launches++;
  CK(cudaMemcpyAsync(ctx->h_flags, d_buf, sizeof(int) * 16, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  CK(cudaGetLastError());
  if (ctx->h_flags[kDiaMaxDiags] || ctx->h_flags[kDiaMaxDiags + 1]) return done(B200_OK);
  std::vector<int> offs;
  for (int s = 0; s < kDiaMaxDiags; ++s)
    if (ctx->h_flags[s] != kDiaEmpty) offs.push_back(ctx->h_flags[s]);
  std::sort(offs.begin(), offs.end());
  const int nd = (int)offs.size();
  const size_t vs = dtype_size(A->dtype);
  const double dia_bytes = (double)nd * (double)m * (double)vs + (double)m;
  const double csr_bytes = (double)A->nnz * (double)(vs + 4) + 4.0 * (double)(m + 1);
  if (nd == 0 || dia_bytes > 0.8 * csr_bytes) return done(B200_OK);
  const int64_t m_pad = (m + kDiaRowAlign - 1) / kDiaRowAlign * kDiaRowAlign;
  if (cudaMalloc(&A->dia_vals, vs * nd * m_pad) != cudaSuccess || cudaMalloc(&A->dia_mask, m_pad) != cudaSuccess) {
    cudaGetLastError();   // out of memory is not sticky: clear it and keep serving the CSR
    free_dia(A);
    return done(B200_OK);
  }
  CK(cudaMemsetAsync(A->dia_vals, 0, vs * nd * m_pad, st));
  CK(cudaMemsetAsync(A->dia_mask, 0, m_pad, st));
  DiaOffsets o;
  o.ndiag = nd;
  for (int d = 0; d < kDiaMaxDiags; ++d) o.off[d] = d < nd ? offs[d] : 0;
  if (A->dtype == B200_F64)
    k_dia_fill<double><<<grid_for(ctx, m), 256, 0, st>>>(A->rowptr, A->colind, (const double *)A->vals, m, o, m_pad,
                                                          (double *)A->dia_vals, A->dia_mask, d_buf + kDiaMaxDiags);
  else
    k_dia_fill<float><<<grid_for(ctx, m), 256, 0, st>>>(A->rowptr, A->colind, (const float *)A->vals, m, o, m_pad,
                                                         (float *)A->dia_vals, A->dia_mask, d_buf + kDiaMaxDiags);
  ctx->launches++;
  CK(cudaMemcpyAsync(ctx->h_flags, d_buf + kDiaMaxDiags, sizeof(int) * 3, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  CK(cudaGetLastError());
#undef CK
  if (ctx->h_flags[2]) {
    free_dia(A);
    return done(B200_OK);
  }
  A->dia_ndiag = nd;
  A->dia_m_pad = m_pad;
  for (int d = 0; d < kDiaMaxDiags; ++d) A->dia_off[d] = d < nd ? offs[d] : 0;
  return done(B200_OK);
}

int finish_operator(b200_ctx *ctx, b200_csr *A, const b200_halo_plan *plan) {
  // row statistics for kernel selection
  int *d_max = (int *)ctx->d_scalars;  // reuse scratch (int view)
  B200_CUDA(cudaMemsetAsync(d_max, 0, sizeof(int), ctx->stream));
  if (A->m_local > 0) {
    k_row_stats<<<grid_for(ctx, A->m_local), 256, 0, ctx->stream>>>(A->rowptr, A->m_local, d_max);
    B200_LAUNCH_CHECK(ctx);
  }
  B200_CUDA(cudaMemcpyAsync(ctx->h_flags, d_max, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  B200_CUDA(cudaStreamSynchronize(ctx->stream));
  A->max_row_nnz = ctx->h_flags[0];
  A->avg_row_nnz = A->m_local ? (double)A->nnz / (double)A->m_local : 0.0;
  // TMA-streamed kernel (spmv_stream.cuh): smallest lanes-per-row whose 512/LPR-row tiles hold <= 4096 nonzeros
  A->stream_lpr = 0;
  if (A->m_local > 0) {
    for (int l = 0; l < 6; ++l) {
      B200_CUDA(cudaMemsetAsync(d_max + 1 + l, 0, sizeof(int), ctx->stream));
      k_tile_max<<<grid_for(ctx, (A->m_local + 15) / 16), 256, 0, ctx->stream>>>(A->rowptr, A->m_local, 512 >> l, d_max + 1 + l);
      B200_LAUNCH_CHECK(ctx);
    }
    B200_CUDA(cudaMemcpyAsync(ctx->h_flags, d_max + 1, sizeof(int) * 6, cudaMemcpyDeviceToHost, ctx->stream));
    B200_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int l = 0; l < 6; ++l)
      if (ctx->h_flags[l] <= 4096) {
        A->stream_lpr = 1 << l;
        break;
      }
  }
  B200_TRY(build_dia(ctx, A));
  B200_CUDA(cudaMemsetAsync(d_max, 0, sizeof(double) * 8, ctx->stream));
  // halo exchange lists
  const int W = ctx->world;
  A->send_count.assign(W, 0);
  A->send_offset.assign(W + 1, 0);
  A->recv_count.assign(W, 0);
  A->recv_offset.assign(W + 1, 0);
  if (plan && W > 1) {
    std::vector<int> send_idx;
    for (int p = 0; p < W; ++p) {
      A->send_offset[p] = (int64_t)send_idx.size();
      A->send_count[p] = (int64_t)plan->send_cols[p].size();
      for (int64_t c : plan->send_cols[p]) send_idx.push_back((int)(c - A->row_begin));
      A->recv_count[p] = (int64_t)plan->recv_cols[p].size();
      A->recv_offset[p] = plan->recv_offset[p];
    }
    A->send_offset[W] = (int64_t)send_idx.size();
    A->recv_offset[W] = plan->recv_offset[W];
    A->send_range_lo.assign(W, -1);
    for (int p = 0; p < W; ++p) {
      if (b200_halo_plan_send_range(plan, p, nullptr) == 1) A->send_range_lo[p] = plan->send_cols[p][0] - A->row_begin;
    }
    A->n_send = (int64_t)send_idx.size();
    const size_t vs = dtype_size(A->dtype);
    if (A->n_send) {
      B200_CUDA(cudaMalloc(&A->send_idx, sizeof(int) * A->n_send));
      B200_CUDA(cudaMemcpyAsync(A->send_idx, send_idx.data(), sizeof(int) * A->n_send, cudaMemcpyHostToDevice,
                                ctx->stream));
      B200_CUDA(cudaMalloc(&A->send_buf, vs * A->n_send));
    }
    if (A->n_halo) B200_CUDA(cudaMalloc(&A->halo, vs * A->n_halo));
    B200_CUDA(cudaStreamSynchronize(ctx->stream));
    // peer-memory path: my halo segment lives in my comm buffer; learn where my values go in each peer's segment
    A->peer_halo = false;
    A->peer_dst_offset.assign(W, 0);
    {
      std::vector<long long> mine(W + 1), all((size_t)W * (W + 1));
      for (int p = 0; p <= W; ++p) mine[p] = A->recv_offset[p];
      long long *d_all = nullptr;
      B200_CUDA(cudaMalloc(&d_all, sizeof(long long) * all.size()));
      B200_CUDA(cudaMemcpy(d_all + (size_t)ctx->rank * (W + 1), mine.data(), sizeof(long long) * (W + 1), cudaMemcpyHostToDevice));
      B200_NCCL(ncclAllGather(d_all + (size_t)ctx->rank * (W + 1), d_all, W + 1, ncclInt64, ctx->comm, ctx->stream));
      B200_CUDA(cudaStreamSynchronize(ctx->stream));
      B200_CUDA(cudaMemcpy(all.data(), d_all, sizeof(long long) * all.size(), cudaMemcpyDeviceToHost));
      cudaFree(d_all);
      bool fits = true;
      for (int p = 0; p < W; ++p) {
        A->peer_dst_offset[p] = all[(size_t)p * (W + 1) + ctx->rank];          // peer p's recv_offset[me]
        fits = fits && (size_t)all[(size_t)p * (W + 1) + W] * vs + kPeerHeaderBytes <= kPeerBufferBytes;
      }
      A->recv_mask = A->send_mask = 0;
      for (int p = 0; p < W; ++p) {
        if (A->recv_count[p]) A->recv_mask |= 1u << p;
        if (A->send_count[p]) A->send_mask |= 1u << p;
      }
      if (ctx->peer_ok && fits) {
        A->peer_halo = true;
        A->halo_peer = (char *)ctx->peer_local + kPeerHeaderBytes;
      }
    }
  }
  return B200_OK;
}

int check_dist_args(b200_ctx *ctx, int64_t n_global, int64_t row_begin, int64_t m_local, const b200_halo_plan *plan) {
  B200_REQUIRE(ctx, "ctx is NULL");
  B200_REQUIRE(m_local >= 0 && row_begin >= 0 && row_begin + m_local <= n_global, "bad slab");
  if (ctx->world > 1) {
    B200_REQUIRE(plan, "multi-GPU context needs a halo plan");
    B200_REQUIRE(plan->world == ctx->world && plan->rank == ctx->rank, "plan/context rank mismatch");
    B200_REQUIRE(plan->row_offsets[ctx->rank] == row_begin && plan->row_offsets[ctx->rank + 1] == row_begin + m_local,
                 "slab does not match the plan");
  } else {
    B200_REQUIRE(row_begin == 0 && m_local == n_global, "single-GPU operator must own all rows");
  }
  B200_REQUIRE(m_local + (plan ? (int64_t)plan->halo_sorted.size() : 0) < (int64_t)INT32_MAX,
               "local rows + halo must fit int32");
  return B200_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------
// C ABI: operator construction
// ------------------------------------------------------------------------------------------
template <typename I, typename TI, typename T>
static int csr_from_csc_impl(b200_ctx *ctx, int64_t m, int64_t n, const I *colptr, const I *rowval, const TI *nzval,
                             int base, int64_t nnz, cudaMemcpyKind src_kind, b200_csr *A) {
  // colptr/rowval/nzval: host arrays (src_kind = cudaMemcpyHostToDevice; nnz = colptr[n] - base read by the caller)
  // or device arrays (cudaMemcpyDeviceToDevice: b200_csr_transpose feeds the CSR arrays of A as the CSC of A')
  cudaStream_t st = ctx->stream;
  B200_REQUIRE(nnz >= 0 && nnz < (int64_t)INT32_MAX, "nnz=%lld does not fit int32 CSR", (long long)nnz);
  A->nnz = nnz;
  I *d_colptr = nullptr, *d_rowval = nullptr;
  TI *d_nz = nullptr;
  unsigned int *key_in = nullptr, *key_out = nullptr;
  int *col_of = nullptr, *perm_in = nullptr, *perm_out = nullptr, *d_err = nullptr;
  void *d_tmp = nullptr;
  size_t tmp_bytes = 0, tmp2 = 0;
  int status = B200_OK;
  auto cleanup = [&]() {
    cudaFree(d_colptr); cudaFree(d_rowval); cudaFree(d_nz); cudaFree(key_in); cudaFree(key_out);
    cudaFree(col_of); cudaFree(perm_in); cudaFree(perm_out); cudaFree(d_err); cudaFree(d_tmp);
  };
#define CK(call)                          \
  do {                                    \
    cudaError_t _e = (call);              \
    if (_e != cudaSuccess) {              \
      set_error("%s:%d %s in `%s`", __FILE__, __LINE__, cudaGetErrorString(_e), #call); \
      cleanup();                          \
      return B200_ERR_CUDA;               \
    }                                     \
  } while (0)
  CK(cudaMalloc(&d_colptr, sizeof(I) * (n + 1)));
  CK(cudaMalloc(&d_rowval, sizeof(I) * (nnz ? nnz : 1)));
  CK(cudaMalloc(&d_nz, sizeof(TI) * (nnz ? nnz : 1)));
  CK(cudaMalloc(&d_err, sizeof(int)));
  CK(cudaMemsetAsync(d_err, 0, sizeof(int), st));
  CK(cudaMemcpyAsync(d_colptr, colptr, sizeof(I) * (n + 1), src_kind, st));
  CK(cudaMemcpyAsync(d_rowval, rowval, sizeof(I) * nnz, src_kind, st));
  CK(cudaMemcpyAsync(d_nz, nzval, sizeof(TI) * nnz, src_kind, st));
  CK(cudaMalloc(&A->rowptr, sizeof(int) * (m + kRowptrPad)));
  CK(cudaMalloc(&A->colind, sizeof(int) * (nnz + kNnzPad)));
  CK(cudaMalloc(&A->vals, sizeof(T) * (nnz + kNnzPad)));
  // rowptr: histogram of row ids, exclusive scan
  CK(cudaMemsetAsync(A->rowptr, 0, sizeof(int) * (m + kRowptrPad), st));
  if (nnz) {
    k_count_rows<I><<<grid_for(ctx, nnz), 256, 0, st>>>(d_rowval, nnz, base, m, A->rowptr, d_err);
    ctx->launches++;
  }
  CK(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, A->rowptr, A->rowptr, (int)(m + 1), st));
  // stable radix sort of (row key, original position): orders by (row, column) because the CSC
  // arrays are column-major with ascending rows inside a column
  int end_bit = 1;
  while (end_bit < 32 && (1ull << end_bit) < (unsigned long long)(m > 1 ? m : 2)) ++end_bit;
  CK(cudaMalloc(&key_in, sizeof(unsigned int) * (nnz ? nnz : 1)));
  CK(cudaMalloc(&key_out, sizeof(unsigned int) * (nnz ? nnz : 1)));
  CK(cudaMalloc(&col_of, sizeof(int) * (nnz + kNnzPad)));
  CK(cudaMalloc(&perm_in, sizeof(int) * (nnz + kNnzPad)));
  CK(cudaMalloc(&perm_out, sizeof(int) * (nnz + kNnzPad)));
  CK(cub::DeviceRadixSort::SortPairs(nullptr, tmp2, key_in, key_out, perm_in, perm_out, (int)nnz, 0, end_bit, st));
  tmp_bytes = std::max(tmp_bytes, tmp2);
  CK(cudaMalloc(&d_tmp, tmp_bytes ? tmp_bytes : 16));
  CK(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, A->rowptr, A->rowptr, (int)(m + 1), st));
  ctx->launches++;
  if (nnz) {
    k_expand_cols<I><<<grid_for(ctx, n * 32), 256, 0, st>>>(d_colptr, n, base, d_rowval, key_in, col_of);
    k_iota<<<grid_for(ctx, nnz), 256, 0, st>>>(perm_in, nnz);
    CK(cub::DeviceRadixSort::SortPairs(d_tmp, tmp_bytes, key_in, key_out, perm_in, perm_out, (int)nnz, 0, end_bit, st));
    k_gather_int<<<grid_for(ctx, nnz), 256, 0, st>>>(perm_out, col_of, nnz, A->colind);
    k_gather_vals<T, TI><<<grid_for(ctx, nnz), 256, 0, st>>>(perm_out, d_nz, nnz, (T *)A->vals);
    ctx->launches += 5;
  }
  CK(cudaMemcpyAsync(ctx->h_flags, d_err, sizeof(int), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  CK(cudaGetLastError());
  if (ctx->h_flags[0]) {
    set_error("row index out of range in SparseMatrixCSC arrays");
    status = B200_ERR_INVALID;
  }
#undef CK
  cleanup();
  return status;
}

extern "C" {

int b200_csr_from_csc(b200_ctx *ctx, int64_t m, int64_t n, const void *colptr, const void *rowval, const void *nzval,
                      int idx_bytes, int dtype, int base, b200_csr **out) {
  B200_REQUIRE(ctx && out && colptr && (idx_bytes == 4 || idx_bytes == 8), "bad arguments");
  B200_REQUIRE(dtype == B200_F64 || dtype == B200_F32, "bad dtype");
  B200_REQUIRE(ctx->world == 1, "b200_csr_from_csc is single-GPU; use b200_csr_from_csr_slab on multi-GPU contexts");
  B200_REQUIRE(m >= 0 && n >= 0 && m < INT32_MAX && n < INT32_MAX, "dimensions must fit int32");
  // rectangular operators are accepted (lsqr!/lsmr!); the square-system solvers check is_square(A) themselves
  B200_CUDA(cudaSetDevice(ctx->device));
  auto *A = new b200_csr();
  A->ctx = ctx;
  A->dtype = dtype;
  A->m_local = m;
  A->m_global = m;
  A->n_global = n;
  const int64_t nnz = (idx_bytes == 8 ? (int64_t)((const int64_t *)colptr)[n] : (int64_t)((const int32_t *)colptr)[n]) - base;
  const cudaMemcpyKind h2d = cudaMemcpyHostToDevice;
  int s;
  if (idx_bytes == 8) {
    s = dtype == B200_F64 ? csr_from_csc_impl<int64_t, double, double>(ctx, m, n, (const int64_t *)colptr, (const int64_t *)rowval, (const double *)nzval, base, nnz, h2d, A)
                          : csr_from_csc_impl<int64_t, float, float>(ctx, m, n, (const int64_t *)colptr, (const int64_t *)rowval, (const float *)nzval, base, nnz, h2d, A);
  } else {
    s = dtype == B200_F64 ? csr_from_csc_impl<int32_t, double, double>(ctx, m, n, (const int32_t *)colptr, (const int32_t *)rowval, (const double *)nzval, base, nnz, h2d, A)
                          : csr_from_csc_impl<int32_t, float, float>(ctx, m, n, (const int32_t *)colptr, (const int32_t *)rowval, (const float *)nzval, base, nnz, h2d, A);
  }
  if (s == B200_OK) s = finish_operator(ctx, A, nullptr);
  if (s != B200_OK) {
    b200_csr_destroy(A);
    return s;
  }
  *out = A;
  return B200_OK;
}

/* adjoint(A) as an operator of its own (reference: LanczosDecomp stores `adjoint(A)`, src/qmr.jl:54; lsqr src/lsqr.jl:128,
 * lsmr src/lsmr.jl:117): the device CSR arrays of A are the CSC arrays of A', so the CSC->CSR conversion above builds
 * the CSR of A' without leaving the GPU.  Real element types: adjoint == transpose. */
int b200_csr_transpose(b200_ctx *ctx, const b200_csr *A, b200_csr **out) {
  B200_REQUIRE(ctx && A && out, "NULL argument");
  B200_REQUIRE(A->ctx == ctx, "operator belongs to another context");
  B200_REQUIRE(ctx->world == 1, "b200_csr_transpose is single-GPU; on multi-GPU contexts build the adjoint from its own "
                                "row slabs with b200_csr_from_csr_slab");
  B200_CUDA(cudaSetDevice(ctx->device));
  auto *At = new b200_csr();
  At->ctx = ctx;
  At->dtype = A->dtype;
  At->m_local = A->n_global;
  At->m_global = A->n_global;
  At->n_global = A->m_local;
  const cudaMemcpyKind d2d = cudaMemcpyDeviceToDevice;
  int s = A->dtype == B200_F64
              ? csr_from_csc_impl<int32_t, double, double>(ctx, At->m_local, At->n_global, A->rowptr, A->colind,
                                                           (const double *)A->vals, 0, A->nnz, d2d, At)
              : csr_from_csc_impl<int32_t, float, float>(ctx, At->m_local, At->n_global, A->rowptr, A->colind,
                                                         (const float *)A->vals, 0, A->nnz, d2d, At);
  if (s == B200_OK) s = finish_operator(ctx, At, nullptr);
  if (s != B200_OK) {
    b200_csr_destroy(At);
    return s;
  }
  *out = At;
  return B200_OK;
}

int b200_csr_from_csr_slab(b200_ctx *ctx, int64_t n_global, int64_t row_begin, int64_t m_local, const void *rowptr,
                           const void *colind, const void *vals, int idx_bytes, int dtype, int base,
                           const b200_halo_plan *plan, b200_csr **out) {
  B200_REQUIRE(out && rowptr && (idx_bytes == 4 || idx_bytes == 8), "bad arguments");
  B200_REQUIRE(dtype == B200_F64 || dtype == B200_F32, "bad dtype");
  B200_TRY(check_dist_args(ctx, n_global, row_begin, m_local, plan));
  B200_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const int64_t nnz = idx_bytes == 8 ? ((const int64_t *)rowptr)[m_local] - ((const int64_t *)rowptr)[0]
                                     : (int64_t)((const int32_t *)rowptr)[m_local] - ((const int32_t *)rowptr)[0];
  B200_REQUIRE(nnz >= 0 && nnz < (int64_t)INT32_MAX, "local nnz must fit int32");
  auto *A = new b200_csr();
  A->ctx = ctx;
  A->dtype = dtype;
  A->m_local = m_local;
  A->m_global = n_global;   // row-partitioned operators are square
  A->n_global = n_global;
  A->row_begin = row_begin;
  A->nnz = nnz;
  A->n_halo = plan ? (int64_t)plan->halo_sorted.size() : 0;
  const size_t vs = dtype_size(dtype);
  void *d_rp = nullptr, *d_ci = nullptr;
  int64_t *d_halo = nullptr;
  int *d_err = nullptr;
  int status = B200_OK;
  auto fail = [&](int s) {
    cudaFree(d_rp); cudaFree(d_ci); cudaFree(d_halo); cudaFree(d_err);
    b200_csr_destroy(A);
    return s;
  };
#define CK(call)                                                                        \
  do {                                                                                  \
    cudaError_t _e = (call);                                                            \
    if (_e != cudaSuccess) {                                                            \
      set_error("%s:%d %s in `%s`", __FILE__, __LINE__, cudaGetErrorString(_e), #call); \
      return fail(B200_ERR_CUDA);                                                       \
    }                                                                                   \
  } while (0)
  CK(cudaMalloc(&A->rowptr, sizeof(int) * (m_local + kRowptrPad)));
  CK(cudaMemsetAsync(A->rowptr, 0, sizeof(int) * (m_local + kRowptrPad), st));
  CK(cudaMalloc(&A->colind, sizeof(int) * (nnz + kNnzPad)));
  CK(cudaMalloc(&A->vals, vs * (nnz + kNnzPad)));
  CK(cudaMalloc(&d_rp, (size_t)idx_bytes * (m_local + 1)));
  CK(cudaMalloc(&d_ci, (size_t)idx_bytes * (nnz ? nnz : 1)));
  CK(cudaMalloc(&d_halo, sizeof(int64_t) * (A->n_halo ? A->n_halo : 1)));
  CK(cudaMalloc(&d_err, sizeof(int)));
  CK(cudaMemsetAsync(d_err, 0, sizeof(int), st));
  CK(cudaMemcpyAsync(d_rp, rowptr, (size_t)idx_bytes * (m_local + 1), cudaMemcpyHostToDevice, st));
  if (nnz) {
    CK(cudaMemcpyAsync(d_ci, colind, (size_t)idx_bytes * nnz, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(A->vals, vals, vs * nnz, cudaMemcpyHostToDevice, st));
  }
  if (A->n_halo)
    CK(cudaMemcpyAsync(d_halo, plan->halo_sorted.data(), sizeof(int64_t) * A->n_halo, cudaMemcpyHostToDevice, st));
  const int64_t lo = row_begin, hi = row_begin + m_local;
  if (idx_bytes == 8) {
    k_rowptr_convert<int64_t><<<grid_for(ctx, m_local + 1), 256, 0, st>>>((const int64_t *)d_rp, m_local, A->rowptr);
    if (nnz) k_remap_cols<int64_t><<<grid_for(ctx, nnz), 256, 0, st>>>((const int64_t *)d_ci, nnz, base, lo, hi, d_halo, A->n_halo, A->colind, d_err);
  } else {
    k_rowptr_convert<int32_t><<<grid_for(ctx, m_local + 1), 256, 0, st>>>((const int32_t *)d_rp, m_local, A->rowptr);
    if (nnz) k_remap_cols<int32_t><<<grid_for(ctx, nnz), 256, 0, st>>>((const int32_t *)d_ci, nnz, base, lo, hi, d_halo, A->n_halo, A->colind, d_err);
  }
  ctx->launches += 2;
  CK(cudaMemcpyAsync(ctx->h_flags, d_err, sizeof(int), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  CK(cudaGetLastError());
#undef CK
  if (ctx->h_flags[0]) {
    set_error("column index not owned and not in the halo plan");
    return fail(B200_ERR_INVALID);
  }
  cudaFree(d_rp); cudaFree(d_ci); cudaFree(d_halo); cudaFree(d_err);
  status = finish_operator(ctx, A, plan);
  if (status != B200_OK) {
    b200_csr_destroy(A);
    return status;
  }
  *out = A;
  return B200_OK;
}

int b200_csr_laplacian(b200_ctx *ctx, int64_t N, int dims, int dtype, int64_t row_begin, int64_t m_local,
                       const b200_halo_plan *plan, b200_csr **out) {
  B200_REQUIRE(out && N >= 1 && dims >= 1 && dims <= 6, "bad arguments");
  B200_REQUIRE(dtype == B200_F64 || dtype == B200_F32, "bad dtype");
  LapGeom g;
  g.N = N;
  g.dims = dims;
  int64_t n = 1;
  for (int d = 0; d < dims; ++d) {
    g.stride[d] = n;
    n *= N;
  }
  B200_TRY(check_dist_args(ctx, n, row_begin, m_local, plan));
  B200_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  auto *A = new b200_csr();
  A->ctx = ctx;
  A->dtype = dtype;
  A->m_local = m_local;
  A->m_global = n;
  A->n_global = n;
  A->row_begin = row_begin;
  A->n_halo = plan ? (int64_t)plan->halo_sorted.size() : 0;
  int64_t *d_halo = nullptr;
  void *d_tmp = nullptr;
  size_t tmp_bytes = 0;
  auto fail = [&](int s) {
    cudaFree(d_halo); cudaFree(d_tmp);
    b200_csr_destroy(A);
    return s;
  };
#define CK(call)                                                                        \
  do {                                                                                  \
    cudaError_t _e = (call);                                                            \
    if (_e != cudaSuccess) {                                                            \
      set_error("%s:%d %s in `%s`", __FILE__, __LINE__, cudaGetErrorString(_e), #call); \
      return fail(B200_ERR_CUDA);                                                       \
    }                                                                                   \
  } while (0)
  CK(cudaMalloc(&A->rowptr, sizeof(int) * (m_local + kRowptrPad)));
  CK(cudaMemsetAsync(A->rowptr, 0, sizeof(int) * (m_local + kRowptrPad), st));
  CK(cudaMalloc(&d_halo, sizeof(int64_t) * (A->n_halo ? A->n_halo : 1)));
  if (A->n_halo)
    CK(cudaMemcpyAsync(d_halo, plan->halo_sorted.data(), sizeof(int64_t) * A->n_halo, cudaMemcpyHostToDevice, st));
  if (m_local) k_lap_count<<<grid_for(ctx, m_local), 256, 0, st>>>(g, row_begin, m_local, A->rowptr);
  CK(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, A->rowptr, A->rowptr, (int)(m_local + 1), st));
  CK(cudaMalloc(&d_tmp, tmp_bytes ? tmp_bytes : 16));
  CK(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, A->rowptr, A->rowptr, (int)(m_local + 1), st));
  int nnz32 = 0;
  CK(cudaMemcpyAsync(&nnz32, A->rowptr + m_local, sizeof(int), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  A->nnz = nnz32;
  const size_t vs = dtype_size(dtype);
  CK(cudaMalloc(&A->colind, sizeof(int) * (A->nnz + kNnzPad)));
  CK(cudaMalloc(&A->vals, vs * (A->nnz + kNnzPad)));
  if (m_local) {
    if (dtype == B200_F64)
      k_lap_fill<double><<<grid_for(ctx, m_local), 256, 0, st>>>(g, row_begin, m_local, A->rowptr, d_halo, A->n_halo, A->colind, (double *)A->vals);
    else
      k_lap_fill<float><<<grid_for(ctx, m_local), 256, 0, st>>>(g, row_begin, m_local, A->rowptr, d_halo, A->n_halo, A->colind, (float *)A->vals);
  }
  ctx->launches += 3;
  CK(cudaStreamSynchronize(st));
  CK(cudaGetLastError());
#undef CK
  cudaFree(d_halo); cudaFree(d_tmp);
  int status = finish_operator(ctx, A, plan);
  if (status != B200_OK) {
    b200_csr_destroy(A);
    return status;
  }
  *out = A;
  return B200_OK;
}

int b200_csr_destroy(b200_csr *A) {
  if (!A) return B200_OK;
  if (A->ctx) {
    cudaSetDevice(A->ctx->device);
    cudaStreamSynchronize(A->ctx->stream);
  }
  cudaFree(A->rowptr);
  cudaFree(A->colind);
  cudaFree(A->vals);
  cudaFree(A->send_idx);
  cudaFree(A->send_buf);
  cudaFree(A->halo);
  cudaFree(A->dia_vals);
  cudaFree(A->dia_mask);
  if (A->st_plan && A->st_plan_free) A->st_plan_free(A->st_plan);
  delete A;
  return B200_OK;
}

int b200_csr_info(const b200_csr *A, int64_t *m_local, int64_t *n_global, int64_t *nnz_local, int *dtype,
                  int64_t *row_begin, int64_t *n_halo) {
  B200_REQUIRE(A, "A is NULL");
  if (m_local) *m_local = A->m_local;
  if (n_global) *n_global = A->n_global;
  if (nnz_local) *nnz_local = A->nnz;
  if (dtype) *dtype = A->dtype;
  if (row_begin) *row_begin = A->row_begin;
  if (n_halo) *n_halo = A->n_halo;
  return B200_OK;
}

int b200_csr_format(const b200_csr *A, int *format, int *ndiag, int64_t *offsets) {
  B200_REQUIRE(A, "A is NULL");
  if (format) *format = A->dia_ndiag > 0 ? B200_FORMAT_DIA : B200_FORMAT_CSR;
  if (ndiag) *ndiag = A->dia_ndiag;
  if (offsets)
    for (int d = 0; d < A->dia_ndiag; ++d) offsets[d] = A->dia_off[d];
  return B200_OK;
}

int b200_csr_diag(b200_ctx *ctx, const b200_csr *A, void *diag_dev) {
  B200_REQUIRE(ctx && A && diag_dev, "NULL argument");
  if (A->m_local == 0) return B200_OK;
  if (A->dtype == B200_F64)
    k_diag<double><<<grid_for(ctx, A->m_local), 256, 0, ctx->stream>>>(A->rowptr, A->colind, (const double *)A->vals, A->m_local, (double *)diag_dev);
  else
    k_diag<float><<<grid_for(ctx, A->m_local), 256, 0, ctx->stream>>>(A->rowptr, A->colind, (const float *)A->vals, A->m_local, (float *)diag_dev);
  B200_LAUNCH_CHECK(ctx);
  return B200_OK;
}

int b200_csr_download(b200_ctx *ctx, const b200_csr *A, int32_t *rowptr, int32_t *colind, void *vals) {
  B200_REQUIRE(ctx && A, "NULL argument");
  if (rowptr) B200_CUDA(cudaMemcpyAsync(rowptr, A->rowptr, sizeof(int) * (A->m_local + 1), cudaMemcpyDeviceToHost, ctx->stream));
  if (colind && A->nnz) B200_CUDA(cudaMemcpyAsync(colind, A->colind, sizeof(int) * A->nnz, cudaMemcpyDeviceToHost, ctx->stream));
  if (vals && A->nnz) B200_CUDA(cudaMemcpyAsync(vals, A->vals, dtype_size(A->dtype) * A->nnz, cudaMemcpyDeviceToHost, ctx->stream));
  B200_CUDA(cudaStreamSynchronize(ctx->stream));
  return B200_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------
// halo push over NVLink peer memory (peer.cuh): x[send_idx[k]] -> the peer's halo segment, then flags
// ------------------------------------------------------------------------------------------
namespace {
struct PushArgs {
  int world, rank;
  long long start[kPeerMaxWorld + 1];   // send_offset per peer
  void *dst[kPeerMaxWorld];             // peer halo segment + my offset inside it
  unsigned int send_mask;
};
template <typename T>
__global__ void __launch_bounds__(256) k_halo_push(PushArgs a, const int *__restrict__ idx, const T *__restrict__ x,
                                                   PeerView pv, unsigned long long seq, unsigned int *ticket,
                                                   const int *__restrict__ done_flag) {
  pdl_wait();
  if (done_flag && *done_flag) return;
  const long long n = a.start[a.world];
  for (long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x; k < n; k += (long long)gridDim.x * blockDim.x) {
    int p = 0;
    while (k >= a.start[p + 1]) ++p;
    ((T *)a.dst[p])[k - a.start[p]] = x[idx[k]];      // store to mapped peer memory (NVLink)
  }
  pdl_launch_dependents();
  __threadfence_system();
  __shared__ bool is_last;
  __syncthreads();
  if (threadIdx.x == 0) is_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!is_last) return;
  if (threadIdx.x == 0) {
    __threadfence_system();
    for (int p = 0; p < a.world; ++p)
      if ((a.send_mask >> p) & 1u) st_release_sys(&pv.hdr[p]->halo_flag[a.rank], seq);
    *ticket = 0u;
  }
}
}  // namespace

int b200::halo_push(b200_ctx *ctx, const b200_csr *A, const void *x_dev, unsigned long long seq,
                    const int *done_flag) {
  if (A->send_mask == 0) return B200_OK;
  PushArgs a;
  a.world = ctx->world;
  a.rank = ctx->rank;
  a.send_mask = A->send_mask;
  const size_t vs = dtype_size(A->dtype);
  for (int p = 0; p <= ctx->world; ++p) a.start[p] = A->send_offset[p];
  for (int p = 0; p < ctx->world; ++p)
    a.dst[p] = (char *)ctx->peer_ptr[p] + kPeerHeaderBytes + vs * (size_t)A->peer_dst_offset[p];
  const int grid = std::max(1, std::min(ctx->sm_count, (int)((A->n_send + 1023) / 1024)));
  unsigned int *ticket = ctx->red.ticket + 1;   // own counter: must not interfere with a reduction in flight
  if (A->dtype == B200_F64)
    B200_CUDA(launch_chained(ctx->opt_pdl != 0, k_halo_push<double>, dim3(grid), dim3(256), 0, ctx->stream, a,
                             (const int *)A->send_idx, (const double *)x_dev, ctx->peer_view, seq, ticket, done_flag));
  else
    B200_CUDA(launch_chained(ctx->opt_pdl != 0, k_halo_push<float>, dim3(grid), dim3(256), 0, ctx->stream, a,
                             (const int *)A->send_idx, (const float *)x_dev, ctx->peer_view, seq, ticket, done_flag));
  B200_LAUNCH_CHECK(ctx);
  return B200_OK;
}

// ------------------------------------------------------------------------------------------
// halo exchange: pack boundary values, grouped ncclSend/ncclRecv with every peer that shares rows
// ------------------------------------------------------------------------------------------
int b200::halo_exchange(b200_ctx *ctx, const b200_csr *A, const void *x_dev) {
  if (ctx->world == 1 || (A->n_send == 0 && A->n_halo == 0)) return B200_OK;
  cudaStream_t st = ctx->stream;
  const size_t vs = dtype_size(A->dtype);
  if (A->n_send) {
    if (A->dtype == B200_F64)
      k_pack<double><<<grid_for(ctx, A->n_send), 256, 0, st>>>(A->send_idx, (const double *)x_dev, A->n_send, (double *)A->send_buf);
    else
      k_pack<float><<<grid_for(ctx, A->n_send), 256, 0, st>>>(A->send_idx, (const float *)x_dev, A->n_send, (float *)A->send_buf);
    B200_LAUNCH_CHECK(ctx);
  }
  const ncclDataType_t nt = A->dtype == B200_F64 ? ncclDouble : ncclFloat;
  B200_NCCL(ncclGroupStart());
  for (int p = 0; p < ctx->world; ++p) {
    if (p == ctx->rank) continue;
    if (A->send_count[p])
      B200_NCCL(ncclSend((const char *)A->send_buf + vs * A->send_offset[p], (size_t)A->send_count[p], nt, p, ctx->comm, st));
    if (A->recv_count[p])
      B200_NCCL(ncclRecv((char *)A->halo + vs * A->recv_offset[p], (size_t)A->recv_count[p], nt, p, ctx->comm, st));
  }
  B200_NCCL(ncclGroupEnd());
  return B200_OK;
}
