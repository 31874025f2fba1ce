// ctx.cu -- context, memory, NCCL bootstrap, timers.
#include <stdarg.h>

#include "common.cuh"

namespace b200 {
static thread_local char g_err[1024] = "";
void set_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
}  // namespace b200

using namespace b200;

int b200::prof_flush(b200_ctx *c) {
  if (c->prof_used == 0) return B200_OK;
  B200_CUDA(cudaStreamSynchronize(c->stream));
  for (size_t i = 0; i + 1 < c->prof_used; i += 2) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, c->prof_ev[i], c->prof_ev[i + 1]) == cudaSuccess) {
      const int slot = c->prof_slot[i / 2];
      c->prof_ms[slot] += ms;
      c->prof_n[slot] += 1;
    }
  }
  c->prof_used = 0;
  return B200_OK;
}

extern "C" {

int b200_version(void) { return 100; }
const char *b200_last_error(void) { return b200::g_err; }

int b200_device_count(int *count) {
  B200_REQUIRE(count, "count is NULL");
  *count = 0;
  B200_CUDA(cudaGetDeviceCount(count));
  return B200_OK;
}

static int ctx_init_common(b200_ctx *c) {
  B200_CUDA(cudaSetDevice(c->device));
  cudaDeviceProp prop;
  B200_CUDA(cudaGetDeviceProperties(&prop, c->device));
  c->sm_count = prop.multiProcessorCount;
  if (prop.major != 10) {
    set_error("libb200krylov is built for sm_100a only; device %d is sm_%d%d", c->device, prop.major, prop.minor);
    return B200_ERR_UNSUPPORTED;
  }
  B200_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  c->own_stream = true;
  B200_CUDA(cudaStreamCreateWithFlags(&c->comm_stream, cudaStreamNonBlocking));
  B200_CUDA(cudaEventCreateWithFlags(&c->ev_a, cudaEventDisableTiming));
  B200_CUDA(cudaEventCreateWithFlags(&c->ev_b, cudaEventDisableTiming));
  B200_CUDA(cudaEventCreate(&c->ev_timer0));
  B200_CUDA(cudaEventCreate(&c->ev_timer1));
  B200_CUDA(cudaMalloc(&c->red.partials, sizeof(double) * kMaxPartials * kMaxReduceWidth));
  B200_CUDA(cudaMalloc(&c->red.ticket, sizeof(unsigned int) * 4));
  B200_CUDA(cudaMemset(c->red.ticket, 0, sizeof(unsigned int) * 4));
  B200_CUDA(cudaMalloc(&c->d_scalars, sizeof(double) * 256));
  B200_CUDA(cudaMemset(c->d_scalars, 0, sizeof(double) * 256));
  B200_CUDA(cudaMallocHost(&c->h_scalars, sizeof(double) * 256));
  B200_CUDA(cudaMallocHost(&c->h_flags, sizeof(int) * 16));
  return B200_OK;
}

// Map every rank's comm buffer into this process (CUDA IPC; handles all-gathered over NCCL).  If the
// platform refuses (no P2P between the two devices, IPC disabled), peer_ok stays false and the engines
// keep using NCCL for the collectives.
static int peer_setup(b200_ctx *c) {
  c->peer_ok = false;
  if (c->world > kPeerMaxWorld) return B200_OK;
  B200_CUDA(cudaMalloc(&c->peer_local, kPeerBufferBytes));
  B200_CUDA(cudaMemset(c->peer_local, 0, kPeerBufferBytes));
  cudaIpcMemHandle_t mine;
  cudaError_t e = cudaIpcGetMemHandle(&mine, c->peer_local);
  int ok = (e == cudaSuccess);
  if (!ok) cudaGetLastError();
  // all-gather {ok flag, handle} through NCCL (device staging in the comm buffer's tail is not needed: d_scalars is 2 KB)
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  unsigned char *d_stage = nullptr;
  const size_t rec = 128;
  B200_CUDA(cudaMalloc(&d_stage, rec * c->world));
  unsigned char h_rec[128];
  memset(h_rec, 0, sizeof(h_rec));
  h_rec[0] = (unsigned char)ok;
  memcpy(h_rec + 64, &mine, 64);
  B200_CUDA(cudaMemcpy(d_stage + rec * c->rank, h_rec, rec, cudaMemcpyHostToDevice));
  B200_NCCL(ncclAllGather(d_stage + rec * c->rank, d_stage, rec, ncclChar, c->comm, c->stream));
  B200_CUDA(cudaStreamSynchronize(c->stream));
  std::vector<unsigned char> all(rec * c->world);
  B200_CUDA(cudaMemcpy(all.data(), d_stage, all.size(), cudaMemcpyDeviceToHost));
  cudaFree(d_stage);
  for (int r = 0; r < c->world && ok; ++r) ok = ok && all[rec * r] == 1;
  for (int r = 0; r < c->world && ok; ++r) {
    if (r == c->rank) {
      c->peer_ptr[r] = c->peer_local;
      continue;
    }
    cudaIpcMemHandle_t h;
    memcpy(&h, all.data() + rec * r + 64, 64);
    e = cudaIpcOpenMemHandle(&c->peer_ptr[r], h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      cudaGetLastError();
      ok = 0;
    }
  }
  // every rank must agree, otherwise nobody uses the peer path
  double flag = ok ? 0.0 : 1.0;
  double *d = c->d_scalars + 128;
  B200_CUDA(cudaMemcpy(d, &flag, sizeof(double), cudaMemcpyHostToDevice));
  B200_NCCL(ncclAllReduce(d, d, 1, ncclDouble, ncclSum, c->comm, c->stream));
  B200_CUDA(cudaMemcpyAsync(&flag, d, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  B200_CUDA(cudaStreamSynchronize(c->stream));
  c->peer_ok = (flag == 0.0);
  c->peer_view.world = c->world;
  c->peer_view.rank = c->rank;
  for (int r = 0; r < c->world; ++r) c->peer_view.hdr[r] = c->peer_ok ? (PeerHeader *)c->peer_ptr[r] : nullptr;
  return B200_OK;
}

int b200_ctx_create(int device, b200_ctx **out) {
  B200_REQUIRE(out, "out is NULL");
  b200_ctx *c = new b200_ctx();
  c->device = device;
  int s = ctx_init_common(c);
  if (s != B200_OK) {
    delete c;
    return s;
  }
  *out = c;
  return B200_OK;
}

int b200_nccl_unique_id(void *out128) {
  B200_REQUIRE(out128, "out128 is NULL");
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId size");
  ncclUniqueId id;
  B200_NCCL(ncclGetUniqueId(&id));
  memcpy(out128, &id, sizeof(id));
  return B200_OK;
}

int b200_ctx_create_dist(int device, int rank, int world, const void *nccl_id128, b200_ctx **out) {
  B200_REQUIRE(out && world >= 1 && rank >= 0 && rank < world, "bad rank/world");
  b200_ctx *c = new b200_ctx();
  c->device = device;
  c->rank = rank;
  c->world = world;
  int s = ctx_init_common(c);
  if (s != B200_OK) {
    delete c;
    return s;
  }
  if (world > 1) {
    B200_REQUIRE(nccl_id128, "nccl_id128 is NULL");
    ncclUniqueId id;
    memcpy(&id, nccl_id128, sizeof(id));
    B200_NCCL(ncclCommInitRank(&c->comm, world, id, rank));
    int s2 = peer_setup(c);
    if (s2 != B200_OK) {
      delete c;
      return s2;
    }
  }
  *out = c;
  return B200_OK;
}

int b200_ctx_destroy(b200_ctx *c) {
  if (!c) return B200_OK;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  for (int r = 0; r < c->world && r < kPeerMaxWorld; ++r)
    if (r != c->rank && c->peer_ptr[r]) cudaIpcCloseMemHandle(c->peer_ptr[r]);
  if (c->peer_local) cudaFree(c->peer_local);
  if (c->comm) ncclCommDestroy(c->comm);
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  if (c->comm_stream) cudaStreamDestroy(c->comm_stream);
  cudaEventDestroy(c->ev_a);
  cudaEventDestroy(c->ev_b);
  cudaEventDestroy(c->ev_timer0);
  cudaEventDestroy(c->ev_timer1);
  cudaFree(c->red.partials);
  cudaFree(c->red.ticket);
  cudaFree(c->d_scalars);
  if (c->ws) cudaFree(c->ws);
  if (c->orth_scal) cudaFree(c->orth_scal);
  for (int k = 0; k < 2; ++k)
    if (c->stage[k]) cudaFree(c->stage[k]);
  for (auto e : c->prof_ev) cudaEventDestroy(e);
  cudaFreeHost(c->h_scalars);
  cudaFreeHost(c->h_flags);
  delete c;
  return B200_OK;
}

int b200_ctx_set_stream(b200_ctx *c, void *cuda_stream) {
  B200_REQUIRE(c, "ctx is NULL");
  B200_CUDA(cudaStreamSynchronize(c->stream));
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  c->stream = (cudaStream_t)cuda_stream;
  c->own_stream = false;
  return B200_OK;
}

int b200_ctx_sync(b200_ctx *c) {
  B200_REQUIRE(c, "ctx is NULL");
  B200_CUDA(cudaStreamSynchronize(c->stream));
  return B200_OK;
}

int b200_ctx_info(const b200_ctx *c, int *device, int *rank, int *world, int *sm_count) {
  B200_REQUIRE(c, "ctx is NULL");
  if (device) *device = c->device;
  if (rank) *rank = c->rank;
  if (world) *world = c->world;
  if (sm_count) *sm_count = c->sm_count;
  return B200_OK;
}

int64_t b200_ctx_launch_count(const b200_ctx *c) { return c ? c->launches : -1; }

int b200_ctx_timer_start(b200_ctx *c) {
  B200_REQUIRE(c, "ctx is NULL");
  B200_CUDA(cudaEventRecord(c->ev_timer0, c->stream));
  return B200_OK;
}
int b200_ctx_timer_stop(b200_ctx *c, float *ms) {
  B200_REQUIRE(c && ms, "NULL argument");
  B200_CUDA(cudaEventRecord(c->ev_timer1, c->stream));
  B200_CUDA(cudaEventSynchronize(c->ev_timer1));
  B200_CUDA(cudaEventElapsedTime(ms, c->ev_timer0, c->ev_timer1));
  return B200_OK;
}

int b200_ctx_set_option(b200_ctx *c, const char *name, int64_t value) {
  B200_REQUIRE(c && name, "NULL argument");
  if (strcmp(name, "spmv_kernel") == 0) {
    B200_REQUIRE(value >= 0 && value <= 2, "spmv_kernel must be 0, 1 or 2");
    c->opt_spmv_kernel = (int)value;
    return B200_OK;
  }
  if (strcmp(name, "spmv_format") == 0) {
    B200_REQUIRE(value == 0 || value == 1, "spmv_format must be 0 (auto) or 1 (CSR)");
    c->opt_spmv_format = (int)value;
    return B200_OK;
  }
  if (strcmp(name, "snake") == 0) {
    c->opt_snake = value != 0;
    return B200_OK;
  }
  if (strcmp(name, "cg_persistent") == 0) {
    c->opt_cg_persistent = value != 0;
    return B200_OK;
  }
  if (strcmp(name, "fold_push") == 0) {
    c->opt_fold_push = value != 0;
    return B200_OK;
  }
  if (strcmp(name, "pdl") == 0) {
    c->opt_pdl = value != 0;
    return B200_OK;
  }
  if (strcmp(name, "orth_fused") == 0) {
    c->opt_orth_fused = value != 0;
    return B200_OK;
  }
  if (strcmp(name, "lobpcg_mma") == 0) {
    c->opt_lobpcg_mma = (int)(value < 0 ? 0 : (value > 2 ? 2 : value));
    return B200_OK;
  }
  if (strcmp(name, "comm") == 0) {
    B200_REQUIRE(value >= 0 && value <= 2, "comm must be 0 (auto), 1 (NCCL) or 2 (peer memory)");
    B200_REQUIRE(value != 2 || c->peer_ok || c->world == 1, "peer-memory collectives are not available on this context");
    c->opt_comm = (int)value;
    return B200_OK;
  }
  set_error("unknown option `%s`", name);
  return B200_ERR_INVALID;
}

int b200_ctx_get_option(const b200_ctx *c, const char *name, int64_t *value) {
  B200_REQUIRE(c && name && value, "NULL argument");
  if (strcmp(name, "spmv_kernel") == 0) *value = c->opt_spmv_kernel;
  else if (strcmp(name, "spmv_format") == 0) *value = c->opt_spmv_format;
  else if (strcmp(name, "comm") == 0) *value = c->opt_comm;
  else if (strcmp(name, "lobpcg_mma") == 0) *value = c->opt_lobpcg_mma;
  else if (strcmp(name, "snake") == 0) *value = c->opt_snake;
  else if (strcmp(name, "orth_fused") == 0) *value = c->opt_orth_fused;
  else if (strcmp(name, "pdl") == 0) *value = c->opt_pdl;
  else if (strcmp(name, "fold_push") == 0) *value = c->opt_fold_push;
  else if (strcmp(name, "cg_persistent") == 0) *value = c->opt_cg_persistent;
  else if (strcmp(name, "peer_ok") == 0) *value = c->peer_ok ? 1 : 0;
  else {
    set_error("unknown option `%s`", name);
    return B200_ERR_INVALID;
  }
  return B200_OK;
}

int b200_ctx_profile_enable(b200_ctx *c, int on) {
  B200_REQUIRE(c, "ctx is NULL");
  if (!on && c->prof_on) prof_flush(c);
  c->prof_on = on != 0;
  return B200_OK;
}
int b200_ctx_profile_read(b200_ctx *c, int slot, double *total_ms, int64_t *launches, int reset) {
  B200_REQUIRE(c && slot >= 0 && slot < 4, "bad arguments");
  B200_TRY(prof_flush(c));
  if (total_ms) *total_ms = c->prof_ms[slot];
  if (launches) *launches = c->prof_n[slot];
  if (reset) {
    c->prof_ms[slot] = 0;
    c->prof_n[slot] = 0;
  }
  return B200_OK;
}

int b200_ctx_allreduce_f64(b200_ctx *c, double *host_inout, int count, int op_max) {
  B200_REQUIRE(c && host_inout && count > 0 && count <= 128, "bad arguments");
  if (c->world == 1) return B200_OK;
  double *d = c->d_scalars + 128;
  B200_CUDA(cudaMemcpyAsync(d, host_inout, sizeof(double) * count, cudaMemcpyHostToDevice, c->stream));
  B200_NCCL(ncclAllReduce(d, d, count, ncclDouble, op_max ? ncclMax : ncclSum, c->comm, c->stream));
  B200_CUDA(cudaMemcpyAsync(host_inout, d, sizeof(double) * count, cudaMemcpyDeviceToHost, c->stream));
  B200_CUDA(cudaStreamSynchronize(c->stream));
  return B200_OK;
}

int b200_ctx_barrier(b200_ctx *c) {
  B200_REQUIRE(c, "ctx is NULL");
  double z = 0.0;
  B200_TRY(b200_ctx_allreduce_f64(c, &z, 1, 0));
  B200_CUDA(cudaStreamSynchronize(c->stream));
  return B200_OK;
}

int b200_malloc(b200_ctx *c, size_t bytes, void **dptr) {
  B200_REQUIRE(c && dptr, "NULL argument");
  B200_CUDA(cudaSetDevice(c->device));
  cudaError_t e = cudaMalloc(dptr, bytes ? bytes : 16);
  if (e != cudaSuccess) {
    set_error("cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
    return B200_ERR_ALLOC;
  }
  return B200_OK;
}
int b200_free(b200_ctx *c, void *dptr) {
  B200_REQUIRE(c, "ctx is NULL");
  if (dptr) {
    B200_CUDA(cudaStreamSynchronize(c->stream));
    B200_CUDA(cudaFree(dptr));
  }
  return B200_OK;
}
int b200_upload(b200_ctx *c, void *dst_dev, const void *src_host, size_t bytes) {
  B200_REQUIRE(c && (bytes == 0 || (dst_dev && src_host)), "NULL argument");
  if (bytes) B200_CUDA(cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, c->stream));
  B200_CUDA(cudaStreamSynchronize(c->stream));
  return B200_OK;
}
int b200_download(b200_ctx *c, void *dst_host, const void *src_dev, size_t bytes) {
  B200_REQUIRE(c && (bytes == 0 || (dst_host && src_dev)), "NULL argument");
  if (bytes) B200_CUDA(cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, c->stream));
  B200_CUDA(cudaStreamSynchronize(c->stream));
  return B200_OK;
}
int b200_host_alloc_pinned(size_t bytes, void **hptr) {
  B200_REQUIRE(hptr, "NULL argument");
  B200_CUDA(cudaMallocHost(hptr, bytes ? bytes : 16));
  return B200_OK;
}
int b200_host_free_pinned(void *hptr) {
  if (hptr) B200_CUDA(cudaFreeHost(hptr));
  return B200_OK;
}

}  // extern "C"
