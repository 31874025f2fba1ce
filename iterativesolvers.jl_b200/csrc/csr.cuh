// csr.cuh -- the device operator (CSR int32, row slab) and the host halo plan.
#pragma once
#include "common.cuh"

struct b200_halo_plan {
  int rank = 0, world = 1;
  std::vector<int64_t> row_offsets;                // world+1
  std::vector<std::vector<int64_t>> recv_cols;     // [owner] -> sorted global columns needed from owner
  std::vector<std::vector<int64_t>> send_cols;     // [peer]  -> my global rows the peer needs
  std::vector<int64_t> halo_sorted;                // concatenation of recv_cols (globally ascending)
  std::vector<int64_t> recv_offset;                // world+1 prefix over owners into halo_sorted
  void rebuild_concat();
};

namespace b200 {
// slack behind the CSR arrays so that the 16-byte-granular TMA bulk copies of the last tile stay
// inside the allocations (spmv_stream.cuh)
constexpr int64_t kRowptrPad = 520;
constexpr int64_t kNnzPad = 16;
// offset-diagonal (DIA) copy of a square single-GPU operator whose nonzeros lie on at most this many diagonals
// (spmv_dia.cuh); rows are padded to whole 512-row tiles so that every bulk copy of a tile stays in bounds
constexpr int kDiaMaxDiags = 8;
constexpr int64_t kDiaRowAlign = 512;
}  // namespace b200
using b200::kNnzPad;
using b200::kRowptrPad;

struct b200_csr {
  b200_ctx *ctx = nullptr;
  int stream_lpr = 0;      // lanes per row of the TMA-streamed kernel; 0 = tiles do not fit, use the sub-warp kernel
  int dtype = B200_F64;
  int64_t m_local = 0, n_global = 0, row_begin = 0, nnz = 0, n_halo = 0;
  int64_t m_global = 0;    // size(A,1); != n_global only for single-GPU rectangular operators (lsqr!/lsmr!)
  int *rowptr = nullptr;   // m_local+1
  int *colind = nullptr;   // nnz; local extended index: [0,m_local) own, [m_local,m_local+n_halo) halo
  void *vals = nullptr;    // nnz
  int max_row_nnz = 0;
  double avg_row_nnz = 0.0;
  // DIA copy (spmv_dia.cuh), built next to the CSR when the operator has few distinct col - row offsets:
  // dia_vals[d * dia_m_pad + row] = A[row, row + dia_off[d]], bit d of dia_mask[row] set iff the CSR row stores that
  // entry (explicit zeros included).  Offsets ascending = column order.  dia_ndiag == 0: no DIA copy.
  int dia_ndiag = 0;
  int64_t dia_off[b200::kDiaMaxDiags] = {0};
  int64_t dia_m_pad = 0;       // m_local rounded up to kDiaRowAlign
  void *dia_vals = nullptr;    // dia_ndiag * dia_m_pad values, diagonal-major
  uint8_t *dia_mask = nullptr; // dia_m_pad bytes (zero in the padding rows)
  // halo exchange state (world > 1)
  std::vector<int64_t> send_count, send_offset, recv_count, recv_offset;  // per peer
  int64_t n_send = 0;
  int *send_idx = nullptr;   // device: local row index to pack, grouped by peer
  void *send_buf = nullptr;  // device: n_send values
  void *halo = nullptr;      // device: n_halo values (recv buffer == halo part of the extended vector), NCCL path
  // peer-memory path (peer.cuh): the halo segment lives in this rank's comm buffer, neighbours store into it
  bool peer_halo = false;
  void *halo_peer = nullptr;               // = ctx->peer_local + kPeerHeaderBytes
  std::vector<int64_t> peer_dst_offset;    // [peer] element offset of MY values inside the peer's halo segment
  std::vector<int64_t> send_range_lo;      // [peer] first local row when the rows sent to `peer` are ONE ascending contiguous range
                                           // (slabs of banded operators), -1 otherwise
  unsigned int recv_mask = 0, send_mask = 0;
  // lazily built analysis of the stationary sweeps (stationary.cu): diagonal positions and dependency levels; the
  // operator is immutable, so the plan stays valid for its lifetime
  mutable void *st_plan = nullptr;
  mutable void (*st_plan_free)(void *) = nullptr;
};

namespace b200 {
// packs x[send_idx] and exchanges with the peers; after return (stream-ordered) A->halo is valid
int halo_exchange(b200_ctx *ctx, const b200_csr *A, const void *x_dev);
// peer-memory variant: stores x[send_idx] into the neighbours' halo segments and raises halo flag `seq`
// (skipped on the device when *done_flag != 0); consumers wait with peer_wait_halo(.., A->recv_mask, seq)
int halo_push(b200_ctx *ctx, const b200_csr *A, const void *x_dev, unsigned long long seq, const int *done_flag);
inline bool is_square(const b200_csr *A) { return A->m_global == A->n_global; }
inline bool use_peer(const b200_ctx *ctx, const b200_csr *A) {
  return ctx->world > 1 && ctx->peer_ok && A->peer_halo && ctx->opt_comm != 1;
}
}  // namespace b200
