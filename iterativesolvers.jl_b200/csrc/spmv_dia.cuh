// spmv_dia.cuh -- the TMA-streamed SpMV body for operators stored as offset diagonals (csr.cuh: dia_*).
//
// Why: for a structured-grid operator (the 7-point Laplacian: offsets -N^2, -N, -1, 0, 1, N, N^2) the CSR column
// indices and row pointers describe the same pattern on every row, yet they are 4.29 of the 13.94 GB that one fp64
// SpMV at 512^3 streams.  Here the matrix is one value array per diagonal plus a 1-byte presence mask per row:
// ndiag*V + 1 bytes per row (57 in fp64) instead of nnz/row*(V+4) + 4 (88).
//
// The tile body is spmv_stream_tiles' (spmv_stream.cuh) with other stage contents: the same producer warp,
// mbarrier ring, 512-row tiles, two consumer groups on alternate tiles, rows slot and slot+256 per thread, grid and
// `rev` sweep.  Per tile the producer bulk-copies the mask range and one value range per diagonal; consumers gather
// x[row + off[d]] for the set bits of their rows.  Offsets are ascending (column order) and each row is summed over
// exactly the entries its CSR row stores, left to right with unfused multiply and add, so the result is bitwise the
// one of the CSR stream kernel at LPR == 1 -- for any x, Inf and NaN included (clear bits are never gathered).
#pragma once
#include "spmv_stream.cuh"

namespace b200 {

template <typename T>
struct alignas(128) DiaStage {
  T val[kDiaMaxDiags][kStreamTileRows];
  uint8_t mask[kStreamTileRows];
};
template <typename T>
struct DiaSmem {
  DiaStage<T> stage[kStreamStages];
  alignas(8) unsigned long long full[kStreamStages];
  alignas(8) unsigned long long empty[kStreamStages];
};

// kernel argument (by value): the DIA arrays of an operator
template <typename T>
struct DiaView {
  const T *__restrict__ vals;        // ndiag * ld, diagonal-major
  const uint8_t *__restrict__ mask;  // ld bytes
  int64_t ld;                        // padded row count (multiple of the tile)
  int64_t off[kDiaMaxDiags];         // ascending; unused entries 0 (their mask bits are clear)
  int ndiag;
};
template <typename T>
inline DiaView<T> make_diaview(const b200_csr *A) {
  DiaView<T> v;
  v.vals = (const T *)A->dia_vals;
  v.mask = A->dia_mask;
  v.ld = A->dia_m_pad;
  for (int d = 0; d < kDiaMaxDiags; ++d) v.off[d] = d < A->dia_ndiag ? A->dia_off[d] : 0;
  v.ndiag = A->dia_ndiag;
  return v;
}

#ifdef __CUDACC__

// Runs over all tiles of this CTA; same contract as spmv_stream_tiles (epi.pre(row), epi(row, value, pre)).
template <typename T, typename XV, typename Epi>
__device__ __forceinline__ void spmv_dia_tiles(const DiaView<T> &dv, const XV &xv, int64_t m, Epi &epi,
                                               DiaSmem<T> *sm, bool rev = false) {
  constexpr int R = kStreamTileRows;
  constexpr int SLOTS = kStreamGroupThreads;
  const int tid = threadIdx.x;
  const int64_t ntiles = (m + R - 1) / R;
  auto phys = [&](int64_t seq) -> int64_t { return rev ? ntiles - 1 - seq : seq; };
  if (tid == 0) {
    for (int s = 0; s < kStreamStages; ++s) {
      mbar_init(&sm->full[s], 1);
      mbar_init(&sm->empty[s], kStreamGroupThreads / 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  if (tid >= kStreamConsumers) {
    // ------------------------------------------------------------ producer warp
    if (tid == kStreamConsumers) {
      const uint64_t pol_stream = policy_evict_first();
      const uint32_t b_val = (uint32_t)(R * sizeof(T));
      const uint32_t bytes = (uint32_t)dv.ndiag * b_val + (uint32_t)R;
      int it = 0;
      for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, ++it) {
        const int s = it % kStreamStages;
        const uint32_t ph = (uint32_t)((it / kStreamStages) & 1);
        const int64_t r0 = phys(t) * R;
        mbar_wait(&sm->empty[s], ph ^ 1u);
        DiaStage<T> *st = &sm->stage[s];
        mbar_expect_tx(&sm->full[s], bytes);
        bulk_g2s(st->mask, dv.mask + r0, (uint32_t)R, &sm->full[s], pol_stream);
        for (int d = 0; d < dv.ndiag; ++d) bulk_g2s(st->val[d], dv.vals + d * dv.ld + r0, b_val, &sm->full[s], pol_stream);
      }
    }
  } else {
    // ------------------------------------------------------------ consumers: group g takes tiles k = g, g+2, ...
    const int grp = tid / kStreamGroupThreads;
    const int slot = tid % kStreamGroupThreads;
    for (int64_t k = grp;; k += kStreamGroups) {
      const int64_t t = (int64_t)blockIdx.x + k * gridDim.x;
      if (t >= ntiles) break;
      const int s = (int)(k % kStreamStages);
      const uint32_t ph = (uint32_t)((k / kStreamStages) & 1);
      const int64_t r0 = phys(t) * R;
      mbar_wait(&sm->full[s], ph);
      const DiaStage<T> *st = &sm->stage[s];
      bool valid[2];
      unsigned int mk[2];
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const int rib = slot + q * SLOTS;
        valid[q] = r0 + rib < m;
        mk[q] = valid[q] ? st->mask[rib] : 0u;
      }
      // the epilogue's per-row operand is requested before the gathers (see spmv_stream_tiles)
      T pre[2] = {(T)0, (T)0};
      if (valid[0]) pre[0] = epi.pre(r0 + slot);
      if (valid[1]) pre[1] = epi.pre(r0 + slot + SLOTS);
      // 2 rows x up to 8 gathers in flight; left-to-right over the set bits, unfused multiply-add
      T xa[2][kDiaMaxDiags];
#pragma unroll
      for (int d = 0; d < kDiaMaxDiags; ++d) {
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const bool on = (mk[q] >> d) & 1u;
          xa[q][d] = on ? xv((int)(r0 + slot + q * SLOTS + dv.off[d])) : (T)0;
        }
      }
      T acc[2] = {(T)0, (T)0};
#pragma unroll
      for (int d = 0; d < kDiaMaxDiags; ++d) {
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          if ((mk[q] >> d) & 1u) {
            const T a = st->val[d][slot + q * SLOTS];
            if constexpr (sizeof(T) == 8) acc[q] = __dadd_rn(acc[q], __dmul_rn(a, xa[q][d]));
            else acc[q] = __fadd_rn(acc[q], __fmul_rn(a, xa[q][d]));
          }
        }
      }
      if (valid[0]) epi(r0 + slot, acc[0], pre[0]);
      if (valid[1]) epi(r0 + slot + SLOTS, acc[1], pre[1]);
      __syncwarp();
      if ((tid & 31) == 0) mbar_arrive(&sm->empty[s]);
    }
  }
}

#endif  // __CUDACC__

// true if the DIA body serves this operator: it has a DIA copy, the format is not forced to CSR and the SpMV is not
// forced to the sub-warp CSR kernel.  The DIA copy exists only for operators whose CSR tiles stream at LPR == 1, so
// the grid is stream_grid_size's.
inline bool use_dia(const b200_ctx *ctx, const b200_csr *A) {
  return A->dia_ndiag > 0 && A->stream_lpr == 1 && ctx->opt_spmv_format == 0 && ctx->opt_spmv_kernel != 1;
}

}  // namespace b200
