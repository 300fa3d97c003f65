// ctx.cu — context lifetime, NCCL communicator plumbing, library self-description.
#include <utility>

#include "lld_ctx.h"

#ifdef LLD_WITH_NCCL
#include <nccl.h>
#endif

struct BaState;
void lld_ba_state_free(BaState*);
void lld_ba_host_free(void*);

std::mutex& lld_capture_mutex() {
  static std::mutex m;
  return m;
}

// cudaFuncSetAttribute applies to the CURRENT device only: the cache of what has been raised is keyed by (device, kernel),
// so a second context on another GPU of the same process sets the attribute on its own device too.
cudaError_t lld_raise_dyn_smem(const void* func, int bytes) {
  struct Seen { int device; const void* func; int bytes; };
  static std::mutex mu;
  static std::vector<Seen> seen;
  int dev = 0;
  cudaError_t r = cudaGetDevice(&dev);
  if (r != cudaSuccess) return r;
  std::lock_guard<std::mutex> lk(mu);
  for (auto& e : seen)
    if (e.device == dev && e.func == func) {
      if (bytes <= e.bytes) return cudaSuccess;
      r = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
      if (r == cudaSuccess) e.bytes = bytes;
      return r;
    }
  r = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (r == cudaSuccess) seen.push_back({dev, func, bytes});
  return r;
}

int lld_call_begin(LldCtx* c, bool full) {
  LLD_CUDA(c, cudaSetDevice(c->device));
  if (full) c->launches = 0;
  c->pool_reset();
  LLD_CUDA(c, cudaEventRecord(c->ev[0], c->stream));
  return LLD_OK;
}

int lld_call_end(LldCtx* c) {
  LLD_CUDA(c, cudaEventRecord(c->ev[3], c->stream));
  LLD_CUDA(c, cudaStreamSynchronize(c->stream));
  cudaEventElapsedTime(&c->ms_h2d, c->ev[0], c->ev[1]);
  cudaEventElapsedTime(&c->ms_compute, c->ev[1], c->ev[2]);
  cudaEventElapsedTime(&c->ms_d2h, c->ev[2], c->ev[3]);
  return LLD_OK;
}

extern "C" const char* lld_version(void) { return "lldba 0.1 (sm_100a)"; }

extern "C" int lld_ctx_create(int device, void** out) {
  if (!out) return LLD_ERR_ARG;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) return LLD_ERR_CUDA;
  if (cudaSetDevice(device) != cudaSuccess) return LLD_ERR_CUDA;
  LldCtx* c = new LldCtx();
  c->device = device;
  if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return LLD_ERR_CUDA; }
  for (int i = 0; i < 4; i++)
    if (cudaEventCreate(&c->ev[i]) != cudaSuccess) { delete c; return LLD_ERR_CUDA; }
  for (int i = 0; i < 2; i++)
    if (cudaEventCreate(&c->ev_user[i]) != cudaSuccess) { delete c; return LLD_ERR_CUDA; }
  for (int i = 0; i < 2; i++) {
    if (cudaStreamCreateWithFlags(&c->side[i], cudaStreamNonBlocking) != cudaSuccess) { delete c; return LLD_ERR_CUDA; }
    if (cudaEventCreateWithFlags(&c->ev_join[i], cudaEventDisableTiming) != cudaSuccess) { delete c; return LLD_ERR_CUDA; }
  }
  if (cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming) != cudaSuccess) { delete c; return LLD_ERR_CUDA; }
  for (int i = 0; i < 2; i++)
    if (cudaEventCreateWithFlags(&c->ev_grp[i], cudaEventDisableTiming) != cudaSuccess) { delete c; return LLD_ERR_CUDA; }
  cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device);
  c->pinned_cap = 1 << 16;
  if (cudaMallocHost(&c->pinned, c->pinned_cap) != cudaSuccess) { delete c; return LLD_ERR_CUDA; }
  *out = c;
  return LLD_OK;
}

extern "C" void lld_ctx_destroy(void* ctx) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c) return;
  for (int i = 0; i < 2; i++)
    if (c->child[i]) { lld_ctx_destroy(c->child[i]); c->child[i] = nullptr; }
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
#ifdef LLD_WITH_NCCL
  if (c->comm) ncclCommDestroy(reinterpret_cast<ncclComm_t>(c->comm));
#endif
  for (auto& b : c->pool) b.release();
  for (auto e : c->ev_pool) cudaEventDestroy(e);
  if (c->pinned) cudaFreeHost(c->pinned);
  for (int i = 0; i < 4; i++)
    if (c->ev[i]) cudaEventDestroy(c->ev[i]);
  lld_ba_state_free(c->ba);  // graphs first: they reference the streams
  for (int i = 0; i < 2; i++)
    if (c->resident[i] && c->resident_free[i]) c->resident_free[i](c->resident[i]);
  lld_ba_host_free(c->ba_host);
  for (int i = 0; i < 2; i++) {
    if (c->side[i]) cudaStreamDestroy(c->side[i]);
    if (c->ev_join[i]) cudaEventDestroy(c->ev_join[i]);
  }
  for (int r = 0; r < 2; r++)
    for (int k = 0; k < 2; k++)
      if (c->ba_graph[r][k]) cudaGraphExecDestroy(c->ba_graph[r][k]);
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  for (int i = 0; i < 2; i++) if (c->ev_grp[i]) cudaEventDestroy(c->ev_grp[i]);
  for (int i = 0; i < 2; i++)
    if (c->ev_user[i]) cudaEventDestroy(c->ev_user[i]);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

extern "C" const char* lld_ctx_last_error(void* ctx) {
  LldCtx* c = lld_ctx_cast(ctx);
  return c ? c->err : "null context";
}
extern "C" int64_t lld_ctx_launch_count(void* ctx) {
  LldCtx* c = lld_ctx_cast(ctx);
  return c ? c->launches : 0;
}
// BA topology cache of this context (and of its pipeline workers): 1 = on, 0 = off, -1 = default
extern "C" void lld_ctx_set_topo_cache(void* ctx, int on) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (c) c->topo_cache = on;
}
// global BA across loop closures: 1 = a reduced system too wide for the on-chip solvers is solved by block elimination
// over its super-block graph (sp_solver.cuh), 0 = it is rejected with LLD_ERR_UNSUPPORTED
extern "C" void lld_ctx_set_gba_sparse(void* ctx, int on) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (c) c->gba_sparse = on != 0;
}
// collectives issued and bytes all-reduced (per rank) since the last lld_ba_global / lld_ba_upload on this context
extern "C" void lld_ctx_nccl_stats(void* ctx, int64_t* calls, int64_t* bytes) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (calls) *calls = c ? c->nccl_calls : 0;
  if (bytes) *bytes = c ? c->nccl_bytes : 0;
}
extern "C" void lld_ctx_last_timing(void* ctx, float* a, float* b, float* d) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c) return;
  if (a) *a = c->ms_h2d;
  if (b) *b = c->ms_compute;
  if (d) *d = c->ms_d2h;
}
// per-kernel CUDA-event profile: enable, run, then read a JSON report {"kernel": {"ms": total, "n": launches}, ...}
extern "C" void lld_ctx_profile(void* ctx, int on) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c) return;
  c->prof_on = on != 0;
  c->prof.clear();
  c->ev_next = 0;
}
extern "C" int lld_ctx_profile_report(void* ctx, char* buf, int cap) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !buf || cap < 8) return LLD_ERR_ARG;
  cudaStreamSynchronize(c->stream);
  struct Acc { const char* name; double ms; long n; };
  std::vector<Acc> acc;
  for (auto& r : c->prof) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, r.a, r.b) != cudaSuccess) continue;
    Acc* f = nullptr;
    for (auto& a : acc)
      if (a.name == r.name || !strcmp(a.name, r.name)) { f = &a; break; }
    if (!f) { acc.push_back({r.name, 0.0, 0}); f = &acc.back(); }
    f->ms += ms;
    f->n++;
  }
  int off = snprintf(buf, cap, "{");
  for (size_t i = 0; i < acc.size() && off < cap - 96; i++)
    off += snprintf(buf + off, cap - off, "%s\"%s\": {\"ms\": %.6f, \"n\": %ld}", i ? ", " : "", acc[i].name, acc[i].ms, acc[i].n);
  snprintf(buf + off, cap - off, "}");
  return LLD_OK;
}
extern "C" void lld_ctx_last_bytes(void* ctx, int64_t* h2d, int64_t* d2h) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c) return;
  if (h2d) *h2d = (int64_t)c->last_h2d_bytes;
  if (d2h) *d2h = (int64_t)c->last_d2h_bytes;
}

// CUDA-event timing on the context's stream (torch.cuda.Event only sees torch's stream)
extern "C" int lld_ctx_event_record(void* ctx, int which) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || which < 0 || which > 1) return LLD_ERR_ARG;
  LLD_CUDA(c, cudaEventRecord(c->ev_user[which], c->stream));
  return LLD_OK;
}
extern "C" float lld_ctx_event_elapsed_ms(void* ctx) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c) return -1.f;
  cudaEventSynchronize(c->ev_user[1]);
  float ms = -1.f;
  cudaEventElapsedTime(&ms, c->ev_user[0], c->ev_user[1]);
  return ms;
}

extern "C" void* lld_ctx_stream(void* ctx) {
  LldCtx* c = lld_ctx_cast(ctx);
  return c ? (void*)c->stream : nullptr;
}

extern "C" int lld_comm_unique_id(uint8_t id_out[128]) {
#ifdef LLD_WITH_NCCL
  ncclUniqueId id;
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId size");
  if (ncclGetUniqueId(&id) != ncclSuccess) return LLD_ERR_NCCL;
  memcpy(id_out, &id, 128);
  return LLD_OK;
#else
  (void)id_out;
  return LLD_ERR_UNSUPPORTED;
#endif
}

extern "C" int lld_comm_init(void* ctx, int n_ranks, int rank, const uint8_t unique_id[128]) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c) return LLD_ERR_ARG;
#ifdef LLD_WITH_NCCL
  LLD_CUDA(c, cudaSetDevice(c->device));
  ncclUniqueId id;
  memcpy(&id, unique_id, 128);
  ncclComm_t comm;
  ncclResult_t r = ncclCommInitRank(&comm, n_ranks, id, rank);
  if (r != ncclSuccess) {
    snprintf(c->err, sizeof(c->err), "ncclCommInitRank: %s", ncclGetErrorString(r));
    return LLD_ERR_NCCL;
  }
  c->comm = reinterpret_cast<ncclComm*>(comm);
  c->n_ranks = n_ranks;
  c->rank = rank;
  return LLD_OK;
#else
  (void)n_ranks; (void)rank; (void)unique_id;
  return LLD_ERR_UNSUPPORTED;
#endif
}
