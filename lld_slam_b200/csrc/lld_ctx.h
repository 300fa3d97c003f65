// lld_ctx.h — per-thread context (stream, workspace, timing) shared by the C-ABI translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <mutex>
#include <type_traits>
#include <vector>

#include "../../include/lldba.h"

// Device / pinned allocations (implicit device-wide synchronisation) must not run while another host thread of this
// library captures a CUDA graph: both sides take this mutex (ctx.cu).
std::mutex& lld_capture_mutex();
// cudaFuncAttributeMaxDynamicSharedMemorySize is per function and process-wide, while contexts of several host threads
// launch the same kernels with different sizes: keep it monotone (never lower it under another thread's launch).
cudaError_t lld_raise_dyn_smem(const void* func, int bytes);
template <typename F>
inline cudaError_t lld_raise_dyn_smem(F* func, size_t bytes) { return lld_raise_dyn_smem(reinterpret_cast<const void*>(func), (int)bytes); }

struct BaState;      // ba.cu
struct ncclComm;

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  // grow-only device allocation; contents are NOT preserved on growth
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    std::lock_guard<std::mutex> lk(lld_capture_mutex());
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
};

struct LldCtx {
  int device = 0;
  cudaStream_t stream = nullptr;
  // side streams + fork/join events: independent kernels of one LM step (point / line / pose passes) run concurrently
  cudaStream_t side[2] = {nullptr, nullptr};
  cudaEvent_t ev_fork = nullptr, ev_join[2] = {nullptr, nullptr};
  cudaEvent_t ev_grp[2] = {nullptr, nullptr};   // completion of the LM step groups in flight (ba_run_round)
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t ev_user[2] = {nullptr, nullptr};  // bench.py timing on this context's stream
  char err[512] = {0};
  int64_t launches = 0;
  int64_t nccl_calls = 0;      // collectives issued / bytes all-reduced by the last multi-rank call (bench reporting)
  int64_t nccl_bytes = 0;
  float ms_h2d = 0, ms_compute = 0, ms_d2h = 0;
  int sm_count = 148;
  bool host_only = false;  // no device work in the upload helpers (host-stage timing hook)
  // NCCL (global BA)
  ncclComm* comm = nullptr;
  int n_ranks = 1, rank = 0;
  // pooled device buffers, reused across calls (index = allocation order inside one call)
  std::vector<DevBuf> pool;
  size_t pool_next = 0;
  // pinned host scratch for small read-backs
  void* pinned = nullptr;
  size_t pinned_cap = 0;
  BaState* ba = nullptr;
  // resident-mode problem views of the matcher / pose kernels (bench entry points lld_sbp_frame_upload / lld_pose_upload): owned by
  // the context (slot 0: match.cu, slot 1: pose.cu), valid while the pool generation they were uploaded under is current
  void* resident[2] = {nullptr, nullptr};
  void (*resident_free[2])(void*) = {nullptr, nullptr};
  unsigned long long resident_gen[2] = {0, 0};
  void* ba_host = nullptr;                // BaHost: persistent host scratch + worker threads of the indexing stage (ba.cu)
  LldCtx* child[2] = {nullptr, nullptr};  // worker contexts of the pipelined batched local BA (ba.cu)
  size_t last_h2d_bytes = 0, last_d2h_bytes = 0;
  // optional per-launch CUDA-event profiling (bench.py roofline): one event pair around every kernel launch
  struct ProfRec { const char* name; cudaEvent_t a, b; };
  bool prof_on = false;
  std::vector<ProfRec> prof;
  std::vector<cudaEvent_t> ev_pool;
  size_t ev_next = 0;
  cudaEvent_t prof_event() {
    if (ev_next >= ev_pool.size()) {
      cudaEvent_t e;
      cudaEventCreate(&e);
      ev_pool.push_back(e);
    }
    return ev_pool[ev_next++];
  }

  // every entry point that (re)uses the pooled buffers bumps the generation: state that lives in them (the uploaded BA
  // problem and its captured graphs, the resident matcher / pose inputs) is valid only while the generation is unchanged
  uint64_t pool_gen = 0;
  // executable graphs of one LM step [round][first / later step], kept across uploads: a new problem re-captures the step
  // and updates the executable in place (cudaGraphExecUpdate) instead of instantiating a new one
  cudaGraphExec_t ba_graph[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};
  int ba_graph_kernels[2][2] = {{0, 0}, {0, 0}};
  int topo_cache = -1;   // BA topology cache: -1 = default (on unless LLD_BA_TOPO_CACHE=0), 0 = off, 1 = on (lld_ctx_set_topo_cache)
  int gba_sparse = 0;    // global BA whose envelope is too wide for the on-chip solvers: 1 = plan-driven block elimination (lld_ctx_set_gba_sparse)
  void pool_reset() { pool_next = 0; pool_gen++; }
  template <typename T>
  T* alloc(size_t n, cudaError_t* e) {
    if (pool_next >= pool.size()) pool.emplace_back();
    DevBuf& b = pool[pool_next++];
    cudaError_t r = b.reserve(n * sizeof(T) + 16);
    if (r != cudaSuccess) {
      *e = r;
      return nullptr;
    }
    return reinterpret_cast<T*>(b.p);
  }
};

#define LLD_CUDA(ctx, call)                                                                            \
  do {                                                                                                 \
    cudaError_t _e = (call);                                                                           \
    if (_e != cudaSuccess) {                                                                           \
      snprintf((ctx)->err, sizeof((ctx)->err), "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e)); \
      return LLD_ERR_CUDA;                                                                             \
    }                                                                                                  \
  } while (0)

#define LLD_ARG(ctx, cond)                                                                     \
  do {                                                                                         \
    if (!(cond)) {                                                                             \
      snprintf((ctx)->err, sizeof((ctx)->err), "%s:%d bad argument: %s", __FILE__, __LINE__, #cond); \
      return LLD_ERR_ARG;                                                                      \
    }                                                                                          \
  } while (0)

// kernel launch with bookkeeping (the launch count feeds bench.py's gpu_launches)
#define LLD_LAUNCH_S(ctx, strm, kernel, grid, block, smem, ...)                 \
  do {                                                                          \
    cudaEvent_t _pa = nullptr, _pb = nullptr;                                   \
    if ((ctx)->prof_on) {                                                       \
      _pa = (ctx)->prof_event();                                                \
      cudaEventRecord(_pa, (strm));                                             \
    }                                                                           \
    kernel<<<(grid), (block), (smem), (strm)>>>(__VA_ARGS__);                   \
    if ((ctx)->prof_on) {                                                       \
      _pb = (ctx)->prof_event();                                                \
      cudaEventRecord(_pb, (strm));                                             \
      (ctx)->prof.push_back({#kernel, _pa, _pb});                               \
    }                                                                           \
    (ctx)->launches++;                                                          \
  } while (0)
#define LLD_LAUNCH(ctx, kernel, grid, block, smem, ...) LLD_LAUNCH_S(ctx, (ctx)->stream, kernel, grid, block, smem, __VA_ARGS__)

// ---- one C-ABI call: ev[0] .. ev[1] upload, ev[1] .. ev[2] compute, ev[2] .. ev[3] download (lld_ctx_last_timing) ----
// Each entry point records ev[1] and ev[2] itself, at its own phase boundaries.

// Opens a call: current device, launch count (full: the resident-mode uploads keep it), a fresh device pool, ev[0].
int lld_call_begin(LldCtx* c, bool full);
// Closes a call: ev[3], waits for the stream and fills ms_h2d / ms_compute / ms_d2h.
int lld_call_end(LldCtx* c);

// Takes the next pool buffer, max(n, 1) elements of T, and copies n elements from src into it when n && src (no source:
// device-only scratch).  T comes from the destination alone, so a const T* field of a copied problem struct takes it as is.
template <typename T>
inline int lld_up(LldCtx* c, T*& dst, const std::remove_const_t<T>* src, size_t n) {
  cudaError_t e = cudaSuccess;
  std::remove_const_t<T>* d = c->alloc<std::remove_const_t<T>>(n ? n : 1, &e);
  if (e != cudaSuccess) {
    snprintf(c->err, sizeof(c->err), "cudaMalloc(%zu bytes): %s", n * sizeof(T), cudaGetErrorString(e));
    return LLD_ERR_CUDA;
  }
  if (n && src) {
    e = cudaMemcpyAsync(d, src, n * sizeof(T), cudaMemcpyHostToDevice, c->stream);
    if (e != cudaSuccess) {
      snprintf(c->err, sizeof(c->err), "cudaMemcpyAsync H2D: %s", cudaGetErrorString(e));
      return LLD_ERR_CUDA;
    }
  }
  dst = d;
  return LLD_OK;
}
// Copies n elements device-to-host when n && dst (an output the caller did not ask for is skipped).
template <typename T>
inline int lld_down(LldCtx* c, T* dst, const T* src, size_t n) {
  if (!n || !dst) return LLD_OK;
  cudaError_t e = cudaMemcpyAsync(dst, src, n * sizeof(T), cudaMemcpyDeviceToHost, c->stream);
  if (e != cudaSuccess) {
    snprintf(c->err, sizeof(c->err), "cudaMemcpyAsync D2H: %s", cudaGetErrorString(e));
    return LLD_ERR_CUDA;
  }
  return LLD_OK;
}
#define LLD_UP(ctx, dst, src, n)                               \
  do {                                                         \
    int _r = lld_up((ctx), (dst), (src), (size_t)(n));         \
    if (_r) return _r;                                         \
  } while (0)
#define LLD_DEV(ctx, dst, n) LLD_UP(ctx, dst, nullptr, n)
#define LLD_DOWN(ctx, dst, src, n)                             \
  do {                                                         \
    int _r = lld_down((ctx), (dst), (src), (size_t)(n));       \
    if (_r) return _r;                                         \
  } while (0)

static inline LldCtx* lld_ctx_cast(void* p) { return reinterpret_cast<LldCtx*>(p); }
