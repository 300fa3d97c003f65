// ba.cu — host driver of the batched point+line bundle adjustment and the lld_ba_* C-ABI entry points.
//
// Replaces the bodies of Optimizer::LocalBundleAdjustment (src/Optimizer.cc:1019-1386) and
// Optimizer::BundleAdjustment (src/Optimizer.cc:321-559): the g2o graph + BlockSolver + Levenberg loop become
// the kernel sequence of ba_kernels.cuh; LM control runs on the device, the host only enqueues steps and polls
// one counter.  No CPU fallback: every path below ends in kernel launches on the context's stream.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <cstdlib>
#include <cstring>
#ifdef __linux__
#include <sched.h>
#endif
#include <numeric>
#include <vector>

#include "ba_kernels.cuh"
#include "cr_solver.cuh"
#include "sp_solver.cuh"
#include "lld_ctx.h"

#include <array>
#include <map>
#include <string>

#ifdef LLD_WITH_NCCL
#include <nccl.h>
#endif

using namespace lld;

static const int CHUNK_DENSE = 512;
static const int CHUNK = 256;          // edge-list entries per chunk (k_lin_poses / k_schur_rows CTA)
static const int SMEM_SOLVE_MAX_N = 156;  // dense LDL^T in shared memory up to this dimension (26 free KFs)

void lld_ba_state_free(struct BaState* s);

struct BaState {
  BaView v{};
  // host copies needed after upload
  int n_win = 0;
  int max_n = 0;       // largest reduced system dimension over the windows
  int max_nnb = 0;
  size_t n_nb_total = 0;
  bool gather_long = false;   // dense mode: average S-block gather list longer than a warp -> k_reduce_piece_warp
  size_t env_smem = 0;
  bool use_cr = false;     // global BA: block cyclic reduction of the reduced camera system (cr_solver.cuh)
  CrView cr{};
  bool use_sp = false;     // global BA across loop closures: plan-driven block elimination (sp_solver.cuh)
  SpView sp{};
  struct SpLevel { int p0, n_el, ntile, u0, n_blk, n_rhs; };
  std::vector<SpLevel> sp_levels;
  long long sp_z_total = 0, sp_n_slot = 0;
  std::string sp_report;   // JSON of the plan (host-only runs: lld_gba_sparse_plan_report)
  bool global_mode = false;
  bool forked = false;     // dense single-rank batch small enough that concurrent passes shorten the critical path
  bool use_graph = false;  // replay one captured LM step instead of re-launching its kernels
  const double* d_kf_Tcw_in = nullptr;
  const double* d_pt_in = nullptr;
  const double* d_ln_in = nullptr;
  size_t h2d_bytes = 0;
  // output staging on device
  double* d_out_kf = nullptr;
  double* d_out_pt = nullptr;
  double* d_out_ln = nullptr;
  uint8_t* d_pt_bad = nullptr;
  uint8_t* d_ln_bad = nullptr;
  // one LM step captured as a CUDA graph per round (kernel arguments differ: round, robust flags)
  // topology cache: a repeated call with the same structure (same windows, observations lists and fixed flags — a
  // re-optimisation, or the bench's steady state) skips the host indexing stage and only refreshes the value arrays
  bool topo_ok = false;
  uint64_t topo_hash = 0, pool_gen = 0;
  int topo_log_stride = 0;
  bool lean = false;       // dense single-rank: steps after the first of a round run ba_step_lean
  // [round][0: first step of the round (separate kernels, lambda_0), 1: later step]: the context's executable graph
  // (LldCtx::ba_graph) matches this problem
  bool graph_fresh[2][2] = {{false, false}, {false, false}};
  void drop_graphs() {
    for (int r = 0; r < 2; r++)
      for (int k = 0; k < 2; k++) graph_fresh[r][k] = false;
  }
};

// Host-side scratch of the flattening / indexing stage, kept in the context across calls: fresh allocations of this size
// cost more in page faults and zero fill than the indexing itself.
// page-locked storage for the index tables (asynchronous DMA instead of staged copies); plain malloc without a device
template <typename T>
struct PinnedAlloc {
  using value_type = T;
  PinnedAlloc() = default;
  template <class U>
  PinnedAlloc(const PinnedAlloc<U>&) {}
  T* allocate(size_t n) {
    void* p = nullptr;
    const size_t bytes = n * sizeof(T) + 16;
    std::lock_guard<std::mutex> lk(lld_capture_mutex());
    if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) == cudaSuccess) {
      *reinterpret_cast<uint64_t*>(p) = 1;
    } else {
      cudaGetLastError();
      p = malloc(bytes);
      if (!p) throw std::bad_alloc();
      *reinterpret_cast<uint64_t*>(p) = 0;
    }
    return reinterpret_cast<T*>(reinterpret_cast<char*>(p) + 16);
  }
  void deallocate(T* q, size_t) {
    void* p = reinterpret_cast<char*>(q) - 16;
    std::lock_guard<std::mutex> lk(lld_capture_mutex());
    if (*reinterpret_cast<uint64_t*>(p)) cudaFreeHost(p);
    else free(p);
  }
  template <class U>
  bool operator==(const PinnedAlloc<U>&) const { return true; }
  template <class U>
  bool operator!=(const PinnedAlloc<U>&) const { return false; }
};
template <typename T>
using pvec = std::vector<T, PinnedAlloc<T>>;

struct BaDenseJob {
  std::vector<int> pb, pe, pn, itp, itt;
  std::vector<long long> pout;
  std::vector<std::pair<int, long long>> gb, gv;
  long long dsize = 0;
  void clear() { pb.clear(); pe.clear(); pn.clear(); itp.clear(); itt.clear(); pout.clear(); gb.clear(); gv.clear(); dsize = 0; }
};
struct BaHost {
  pvec<int> kf_win, kf_g, w_g0, g_kf;
  pvec<int> pe_kf, pe_pt, lc_kf, lc_ln;
  pvec<int> pt_order, ln_order;
  std::vector<uint64_t> pt_key, ln_key;
  pvec<int> pl_off, pl_edge, pe_pos, ll_off, ll_cell, lc_pos;
  pvec<int> pt_spos, ln_spos, pts_w0, lns_w0;
  pvec<uint32_t> pts_mask, lns_mask;
  pvec<int> gb_off, gv_off;
  pvec<SchurItem> it_rec, it_tmp;
  std::vector<uint64_t> it_keys;
  pvec<long long> gb_src, gv_src;
  std::vector<BaDenseJob> jobs;
  pvec<int> ch_g, ch_begin, ch_end, ch_seg0, seg_begin, seg_end, g_chp0, g_chl0;
  pvec<long long> ch_S_off;
  pvec<int> pl_tab, ll_tab;   // sparse-mode position tables (hundreds of MB in global BA: kept page-locked across calls)
  // persistent worker threads for the per-window loops
  std::vector<std::thread> workers;
  std::mutex mu;
  std::condition_variable cv_go, cv_done;
  std::function<void(int)> job;
  std::atomic<int> next{0};
  int job_n = 0, generation = 0, running = 0;
  bool quit = false;
  void worker_loop() {
    int seen = 0;
    for (;;) {
      {
        std::unique_lock<std::mutex> lk(mu);
        cv_go.wait(lk, [&] { return quit || generation != seen; });
        if (quit) return;
        seen = generation;
      }
      for (;;) {
        const int i = next.fetch_add(1);
        if (i >= job_n) break;
        job(i);
      }
      {
        std::lock_guard<std::mutex> lk(mu);
        if (--running == 0) cv_done.notify_one();
      }
    }
  }
  template <class F>
  void par_for(int n, F f) {
    if (n < 4) {
      for (int i = 0; i < n; i++) f(i);
      return;
    }
    if (workers.empty()) {
      // the cores this process may use (affinity mask), shared fairly between the processes of one node: torchrun
      // exports LOCAL_WORLD_SIZE; LLD_HOST_THREADS overrides.  An oversubscribed pool (8 ranks x 16 threads on 32 cores)
      // is what made the end-to-end path scale worse than the device path.
      unsigned cores = std::max(1u, std::thread::hardware_concurrency());
#ifdef __linux__
      {
        cpu_set_t set;
        if (sched_getaffinity(0, sizeof(set), &set) == 0) cores = std::max(1, CPU_COUNT(&set));
      }
#endif
      unsigned share = 1;
      if (const char* e = getenv("LOCAL_WORLD_SIZE")) share = std::max(1, atoi(e));
      unsigned want = std::min<unsigned>(std::max(2u, cores / share), 16u);
      if (const char* e = getenv("LLD_HOST_THREADS")) want = std::max(1, atoi(e));
      const unsigned nt = std::max(1u, want - 1);
      for (unsigned t = 0; t < nt; t++) workers.emplace_back([this] { worker_loop(); });
    }
    {
      std::lock_guard<std::mutex> lk(mu);
      job = f;
      job_n = n;
      next.store(0);
      running = (int)workers.size();
      generation++;
    }
    cv_go.notify_all();
    for (;;) {
      const int i = next.fetch_add(1);
      if (i >= n) break;
      f(i);
    }
    std::unique_lock<std::mutex> lk(mu);
    cv_done.wait(lk, [&] { return running == 0; });
  }
  ~BaHost() {
    {
      std::lock_guard<std::mutex> lk(mu);
      quit = true;
    }
    cv_go.notify_all();
    for (auto& t : workers) t.join();
  }
};
void lld_ba_host_free(void* h) { delete reinterpret_cast<BaHost*>(h); }

namespace {

// LLD_UP_TRACE: FNV-1a of an uploaded array (host-stage refactors are checked to produce identical index arrays)
static unsigned long long up_trace_hash(const void* p, size_t bytes) {
  unsigned long long h = 1469598103934665603ull;
  const unsigned char* b = static_cast<const unsigned char*>(p);
  for (size_t i = 0; p && i < bytes; i++) { h ^= b[i]; h *= 1099511628211ull; }
  return h;
}

template <typename T>
int up(LldCtx* c, T** dst, const T* src, size_t n, size_t* bytes) {
  if (c->host_only) {  // lld_ba_index_only: time / test the host stage without a device
    *dst = nullptr;
    return LLD_OK;
  }
  cudaError_t e = cudaSuccess;
  T* d = c->alloc<T>(n ? n : 1, &e);
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
    if (bytes) *bytes += n * sizeof(T);
  }
  *dst = d;
  return LLD_OK;
}
#define UP(dst, src, n)                                                     \
  do {                                                                      \
    if (getenv("LLD_UP_TRACE")) fprintf(stderr, "[up] %-28s %10.3f MB  fnv %016llx\n", #src, (double)(n) * sizeof(*(dst)) / 1e6, \
                                        up_trace_hash((src), (size_t)(n) * sizeof(*(dst))));                \
    int _r = up(c, &(dst), (src), (size_t)(n), &S->h2d_bytes);              \
    if (_r != LLD_OK) return _r;                                            \
  } while (0)
#define DEV(dst, T, n)                                                      \
  do {                                                                      \
    T* _p = nullptr;                                                        \
    int _r = up<T>(c, &_p, nullptr, (size_t)(n), nullptr);                  \
    if (_r != LLD_OK) return _r;                                            \
    (dst) = _p;                                                             \
  } while (0)

}  // namespace

// 64-bit hash of an array, 8 bytes per step (structure hash of the topology cache)
static uint64_t hash_words(const void* data, size_t bytes, uint64_t h) {
  const uint64_t* w = static_cast<const uint64_t*>(data);
  const size_t n = bytes / 8;
  for (size_t i = 0; i < n; i++) {
    h ^= w[i];
    h *= 0x9E3779B97F4A7C15ull;
    h ^= h >> 29;
  }
  const unsigned char* b = static_cast<const unsigned char*>(data) + 8 * n;
  for (size_t i = 0; i < bytes - 8 * n; i++) { h ^= b[i]; h *= 0x100000001B3ull; }
  return h;
}

// everything the index tables depend on: window / landmark / observation offsets, observing keyframes, fixed flags
static uint64_t ba_topology_hash(BaHost& H, const lld_ba_problem* p, bool global_mode, int log_stride, const lld_ba_problem* full, int n_ranks, int rank,
                                 int gba_sparse) {
  const int nw = p->n_win;
  const int n_kf = p->kf_off[nw], n_pt = p->pt_off[nw], n_ln = p->ln_off[nw];
  const int n_pe = p->pt_obs_off[n_pt], n_lc = p->ln_obs_off[n_ln];
  struct Part { const void* d; size_t bytes; };
  std::vector<Part> parts = {{p->kf_off, 4 * (size_t)(nw + 1)}, {p->pt_off, 4 * (size_t)(nw + 1)}, {p->ln_off, 4 * (size_t)(nw + 1)},
                             {p->kf_fixed, (size_t)n_kf}, {p->pt_obs_off, 4 * (size_t)(n_pt + 1)}, {p->ln_obs_off, 4 * (size_t)(n_ln + 1)}};
  // the two long arrays in slices, hashed in parallel
  const int slices = 16;
  for (int k = 0; k < slices; k++) {
    const size_t a = (size_t)n_pe * k / slices, b = (size_t)n_pe * (k + 1) / slices;
    parts.push_back({p->pt_obs_kf + a, 4 * (b - a)});
  }
  for (int k = 0; k < slices; k++) {
    const size_t a = (size_t)n_lc * k / slices, b = (size_t)n_lc * (k + 1) / slices;
    parts.push_back({p->ln_obs_kf + a, 4 * (b - a)});
  }
  std::vector<uint64_t> hs(parts.size());
  H.par_for((int)parts.size(), [&](int i) { hs[(size_t)i] = hash_words(parts[(size_t)i].d, parts[(size_t)i].bytes, 0xCBF29CE484222325ull + (uint64_t)i); });
  uint64_t h = 0x84222325CBF29CE4ull;
  const uint64_t meta[9] = {(uint64_t)nw, (uint64_t)global_mode, (uint64_t)log_stride, (uint64_t)n_ranks, (uint64_t)rank, (uint64_t)(full != nullptr),
                            (uint64_t)n_pe, (uint64_t)n_lc, (uint64_t)gba_sparse};
  h = hash_words(meta, sizeof(meta), h);
  h = hash_words(hs.data(), 8 * hs.size(), h);
  return h;
}

static void ba_set_params(BaView& v, const lld_ba_problem* p) {
  v.prm.robust_pt = p->robust_points;
  v.prm.robust_ln = 1;
  v.prm.delta_pt_mono = p->delta_pt_mono; v.prm.delta_pt_stereo = p->delta_pt_stereo;
  v.prm.delta_ln_mono = p->delta_ln_mono; v.prm.delta_ln_stereo = p->delta_ln_stereo;
  v.prm.chi2_pt_mono = p->chi2_pt_mono; v.prm.chi2_pt_stereo = p->chi2_pt_stereo;
  v.prm.ln_norm = p->ln_endpoints_normalized;
  v.prm.ln_filter = p->ln_filter;
}

// Symbolic plan of the block elimination of sp_solver.cuh, from the keyframe block pattern (nb lists) alone.
// Super-blocks of mb consecutive free keyframes, mb = the largest distance <= 26 between two covisible free keyframes
// (6 mb <= CR_MAX_M); longer distances become edges of the super-block graph.  Levels: a maximal independent set of the
// remaining nodes, scanned in ascending (degree, index) order, is eliminated, and the remaining neighbours of each
// eliminated node are joined pairwise (fill).  On a chain this is odd / even cyclic reduction; a ring takes ~log2 N levels.
static const int SP_MAX_MB = CR_MAX_M / 6;
static const long long SP_MAX_BYTES = 2LL << 30;   // device storage of one plan (include/lldba.h, capacity limits)

struct SpPlan {
  int mb = 1, N = 0, m = 6, n_orig = 0;
  std::vector<std::pair<int, int>> blocks;   // off-diagonal slots N, N + 1, ...: (I, J), I < J, fill included
  std::vector<int> q_slot, el_node, el_nb_off, nb_node, nb_slot2, up_out, up_c_off, c_slot2, c_pos, c_col;
  std::vector<long long> z_off;
  std::vector<BaState::SpLevel> levels;
  long long z_total = 0, bytes = 0;
};

static void sp_plan_build(int nG, const std::vector<int>& nb_off, const std::vector<int>& nb_g, SpPlan& P) {
  int mb = 1;
  for (int a = 0; a < nG; a++)
    for (int q = nb_off[a]; q < nb_off[a + 1]; q++)
      if (nb_g[q] - a <= SP_MAX_MB) mb = std::max(mb, nb_g[q] - a);
  const int N = (nG + mb - 1) / mb, m = 6 * mb;
  P.mb = mb; P.N = N; P.m = m;
  std::vector<std::vector<int>> adj((size_t)N);   // sorted, both directions
  auto link = [&](int I, int J) {
    auto& A = adj[(size_t)I];
    auto it = std::lower_bound(A.begin(), A.end(), J);
    if (it == A.end() || *it != J) A.insert(it, J);
  };
  for (int a = 0; a < nG; a++)
    for (int q = nb_off[a]; q < nb_off[a + 1]; q++) {
      const int I = a / mb, J = nb_g[q] / mb;
      if (I != J) { link(I, J); link(J, I); }
    }
  for (auto& A : adj) P.n_orig += (int)A.size();
  P.n_orig /= 2;
  // levels
  std::vector<char> alive((size_t)N, 1), blocked((size_t)N);
  std::vector<std::vector<int>> lv_nodes, lv_nbrs;   // per position: its remaining neighbours
  int n_alive = N;
  while (n_alive > 0) {
    std::vector<std::pair<int, int>> order;
    for (int i = 0; i < N; i++)
      if (alive[(size_t)i]) {
        int d = 0;
        for (int j : adj[(size_t)i]) d += alive[(size_t)j];
        order.push_back({d, i});
      }
    std::sort(order.begin(), order.end());
    std::fill(blocked.begin(), blocked.end(), 0);
    std::vector<int> E;
    for (auto& o : order) {
      const int i = o.second;
      if (blocked[(size_t)i]) continue;
      E.push_back(i);
      blocked[(size_t)i] = 1;
      for (int j : adj[(size_t)i]) blocked[(size_t)j] = 1;
    }
    std::sort(E.begin(), E.end());
    for (int i : E) {
      std::vector<int> nb;
      for (int j : adj[(size_t)i])
        if (alive[(size_t)j]) nb.push_back(j);
      lv_nbrs.push_back(nb);
    }
    for (size_t e = 0; e < E.size(); e++) {
      const auto& nb = lv_nbrs[lv_nbrs.size() - E.size() + e];
      for (size_t x = 0; x < nb.size(); x++)
        for (size_t y = x + 1; y < nb.size(); y++) { link(nb[x], nb[y]); link(nb[y], nb[x]); }
    }
    for (int i : E) alive[(size_t)i] = 0;
    n_alive -= (int)E.size();
    lv_nodes.push_back(E);
  }
  // slots: diagonal I, then every off-diagonal block of the filled pattern in (I, J) order
  std::map<std::pair<int, int>, int> slot;
  for (int I = 0; I < N; I++)
    for (int J : adj[(size_t)I])
      if (J > I) { slot[{I, J}] = N + (int)P.blocks.size(); P.blocks.push_back({I, J}); }
  auto slot2 = [&](int i, int j) { return i < j ? 2 * slot[{i, j}] : 2 * slot[{j, i}] + 1; };   // U_ij, transposed when stored as (j, i)
  P.q_slot.resize(nb_g.size());
  for (int a = 0; a < nG; a++)
    for (int q = nb_off[a]; q < nb_off[a + 1]; q++) {
      const int I = a / mb, J = nb_g[q] / mb;
      P.q_slot[(size_t)q] = I == J ? I : slot[{I, J}];
    }
  // positions, neighbour lists, Z offsets, update items (blocks in (j, k) order, then right-hand sides in j order; the
  // contributions of each in ascending i)
  P.el_nb_off.push_back(0);
  P.up_c_off.push_back(0);
  int pos = 0;
  for (const auto& E : lv_nodes) {
    BaState::SpLevel L{pos, (int)E.size(), 0, (int)P.up_out.size(), 0, 0};
    std::map<std::pair<int, int>, std::vector<std::array<int, 3>>> blk;
    std::map<int, std::vector<std::array<int, 3>>> rhs;
    for (int i : E) {
      const auto& nb = lv_nbrs[(size_t)pos];
      P.el_node.push_back(i);
      P.z_off.push_back(P.z_total);
      P.z_total += (long long)m * m * (long long)nb.size();
      for (int j : nb) { P.nb_node.push_back(j); P.nb_slot2.push_back(slot2(i, j)); }
      P.el_nb_off.push_back((int)P.nb_node.size());
      L.ntile = std::max(L.ntile, (m * (int)nb.size() + CR_TC - 1) / CR_TC);
      for (size_t x = 0; x < nb.size(); x++) {
        rhs[nb[x]].push_back({slot2(i, nb[x]), pos, (int)x});
        for (size_t y = x; y < nb.size(); y++) blk[{nb[x], nb[y]}].push_back({slot2(i, nb[x]), pos, (int)y});
      }
      pos++;
    }
    auto put = [&](int out, const std::vector<std::array<int, 3>>& cs) {
      P.up_out.push_back(out);
      for (auto& cc : cs) { P.c_slot2.push_back(cc[0]); P.c_pos.push_back(cc[1]); P.c_col.push_back(cc[2]); }
      P.up_c_off.push_back((int)P.c_slot2.size());
    };
    for (auto& kv : blk) put(kv.first.first == kv.first.second ? kv.first.first : slot[kv.first], kv.second);
    for (auto& kv : rhs) put(kv.first, kv.second);
    L.n_blk = (int)blk.size(); L.n_rhs = (int)rhs.size();
    P.levels.push_back(L);
  }
  const long long mm = (long long)m * m, n_slot = N + (long long)P.blocks.size();
  P.bytes = 8 * (n_slot * mm + N * mm + P.z_total + 3LL * N * m + (long long)P.z_off.size()) +
            4 * (long long)(P.q_slot.size() + P.el_node.size() + P.el_nb_off.size() + P.nb_node.size() + P.nb_slot2.size() +
                            P.up_out.size() + P.up_c_off.size() + P.c_slot2.size() + P.c_pos.size() + P.c_col.size());
}

static std::string sp_plan_json(const SpPlan& P) {
  std::string s;
  char tmp[96];
  auto num = [&](long long x) { snprintf(tmp, sizeof(tmp), "%lld", x); s += tmp; };
  auto list = [&](const int* a, int n) {
    s += "[";
    for (int k = 0; k < n; k++) { if (k) s += ","; num(a[k]); }
    s += "]";
  };
  s += "{\"solver\":\"sparse\",\"mb\":"; num(P.mb); s += ",\"N\":"; num(P.N); s += ",\"m\":"; num(P.m);
  s += ",\"n_orig_blocks\":"; num(P.n_orig); s += ",\"bytes\":"; num(P.bytes); s += ",\"limit\":"; num(SP_MAX_BYTES);
  s += ",\"blocks\":[";
  for (size_t k = 0; k < P.blocks.size(); k++) { s += k ? ",[" : "["; num(P.blocks[k].first); s += ","; num(P.blocks[k].second); s += "]"; }
  s += "],\"levels\":[";
  for (size_t l = 0; l < P.levels.size(); l++) {
    const auto& L = P.levels[l];
    s += l ? ",{" : "{";
    s += "\"nodes\":"; list(P.el_node.data() + L.p0, L.n_el);
    s += ",\"nbrs\":[";
    for (int p = L.p0; p < L.p0 + L.n_el; p++) { if (p > L.p0) s += ","; list(P.nb_node.data() + P.el_nb_off[(size_t)p], P.el_nb_off[(size_t)p + 1] - P.el_nb_off[(size_t)p]); }
    s += "],\"z_off\":[";
    for (int p = L.p0; p < L.p0 + L.n_el; p++) { if (p > L.p0) s += ","; num(P.z_off[(size_t)p]); }
    // update items: [output slot or node, [[i, slot(i, j), transposed, column block of k], ...]]
    s += "],\"items\":[";
    for (int it = L.u0; it < L.u0 + L.n_blk + L.n_rhs; it++) {
      s += it > L.u0 ? ",[" : "[";
      num(P.up_out[(size_t)it]); s += ",[";
      for (int q = P.up_c_off[(size_t)it]; q < P.up_c_off[(size_t)it + 1]; q++) {
        s += q > P.up_c_off[(size_t)it] ? ",[" : "[";
        num(P.el_node[(size_t)P.c_pos[(size_t)q]]); s += ","; num(P.c_slot2[(size_t)q] >> 1); s += ","; num(P.c_slot2[(size_t)q] & 1);
        s += ","; num(P.c_col[(size_t)q]); s += "]";
      }
      s += "]]";
    }
    s += "],\"n_blk\":"; num(L.n_blk); s += "}";
  }
  s += "]}";
  return s;
}

// Flatten + index the problem on the host, upload, initialise device state.
static int ba_upload(LldCtx* c, const lld_ba_problem* p, bool global_mode, int log_stride,
                     const lld_ba_problem* full = nullptr /* multi-rank: whole problem, for the rank-invariant structure */) {
  if (!c->ba) c->ba = new BaState();
  BaState* S = c->ba;
  LLD_ARG(c, p->n_win >= 1);
  if (!c->ba_host) c->ba_host = new BaHost();
  static const bool topo_env = !(getenv("LLD_BA_TOPO_CACHE") && getenv("LLD_BA_TOPO_CACHE")[0] == '0');
  const bool topo_cache = c->topo_cache < 0 ? topo_env : c->topo_cache != 0;
  uint64_t th = 0;
  if (topo_cache && !c->host_only) {
    th = ba_topology_hash(*reinterpret_cast<BaHost*>(c->ba_host), p, global_mode, log_stride, full, c->n_ranks, c->rank, c->gba_sparse);
    if (S->topo_ok && S->topo_hash == th && S->pool_gen == c->pool_gen && S->global_mode == global_mode && S->topo_log_stride == log_stride) {
      // same structure as the problem already indexed on the device: refresh the values only
      BaView& v = S->v;
      const size_t n_kf = (size_t)v.n_kf, n_pt = (size_t)v.n_pt, n_ln = (size_t)v.n_ln, n_pe = (size_t)v.n_pe, n_lc = (size_t)v.n_lc;
      size_t bytes = 0;
      auto put = [&](const void* dst, const void* src, size_t nb) -> cudaError_t {
        bytes += nb;
        return nb ? cudaMemcpyAsync(const_cast<void*>(dst), src, nb, cudaMemcpyHostToDevice, c->stream) : cudaSuccess;
      };
      LLD_CUDA(c, put(v.kf_intr, p->kf_intr, 40 * n_kf));
      LLD_CUDA(c, put(v.kf_lcam, p->kf_line_cam, 32 * n_kf));
      LLD_CUDA(c, put(v.pe_uvr, p->pt_obs_uvr, 12 * n_pe));
      LLD_CUDA(c, put(v.pe_info, p->pt_obs_info, 4 * n_pe));
      LLD_CUDA(c, put(v.lc_left, p->ln_obs_left, 16 * n_lc));
      LLD_CUDA(c, put(v.lc_right, p->ln_obs_right, 16 * n_lc));
      LLD_CUDA(c, put(v.lc_info, p->ln_obs_info, 16 * n_lc));
      LLD_CUDA(c, put(v.lc_stereo, p->ln_obs_stereo, n_lc));
      LLD_CUDA(c, put(S->d_kf_Tcw_in, p->kf_Tcw, 96 * n_kf));
      LLD_CUDA(c, put(S->d_pt_in, p->pt_xyz, 24 * n_pt));
      LLD_CUDA(c, put(S->d_ln_in, p->ln_x0_dir, 48 * n_ln));
      const BaParams old = v.prm;
      ba_set_params(v, p);
      if (memcmp(&old, &v.prm, sizeof(BaParams)) != 0) S->drop_graphs();   // the captured steps carry the parameters by value
      LLD_CUDA(c, cudaMemsetAsync(v.chi2_log, 0, sizeof(double) * (size_t)v.n_win * log_stride, c->stream));
      LLD_CUDA(c, cudaMemsetAsync(v.lambda_log, 0, sizeof(double) * (size_t)v.n_win * log_stride, c->stream));
      LLD_CUDA(c, cudaMemsetAsync(v.trials_log, 0, sizeof(int) * (size_t)v.n_win * log_stride, c->stream));
      LLD_CUDA(c, cudaMemsetAsync(S->d_pt_bad, 0, n_pe ? n_pe : 1, c->stream));
      LLD_CUDA(c, cudaMemsetAsync(S->d_ln_bad, 0, n_lc ? 2 * n_lc : 1, c->stream));
      S->h2d_bytes = bytes;
      c->last_h2d_bytes = bytes;
      return LLD_OK;
    }
  }
  S->drop_graphs();
  *S = BaState();
  S->global_mode = global_mode;
  c->pool_reset();
  S->pool_gen = c->pool_gen;
  S->topo_hash = th; S->topo_log_stride = log_stride;
  BaView& v = S->v;
  const int nw = p->n_win;
  LLD_ARG(c, nw >= 1);
  const int n_kf = p->kf_off[nw], n_pt = p->pt_off[nw], n_ln = p->ln_off[nw];
  const int n_pe = p->pt_obs_off[n_pt], n_lc = p->ln_obs_off[n_ln];
  v.n_win = nw; v.n_kf = n_kf; v.n_pt = n_pt; v.n_ln = n_ln; v.n_pe = n_pe; v.n_lc = n_lc;
  S->n_win = nw;

  // ---- caller-owned arrays first: with pinned host memory these DMA transfers run while the host builds the index tables ----
  int* tmp_i;
  double* tmp_d;
  float* tmp_f;
  uint8_t* tmp_u;
  UP(tmp_i, p->kf_off, nw + 1); v.kf_off = tmp_i;
  UP(tmp_i, p->pt_off, nw + 1); v.pt_off = tmp_i;
  UP(tmp_i, p->ln_off, nw + 1); v.ln_off = tmp_i;
  UP(tmp_d, p->kf_intr, 5 * (size_t)n_kf); v.kf_intr = tmp_d;
  UP(tmp_d, p->kf_line_cam, 4 * (size_t)n_kf); v.kf_lcam = tmp_d;
  UP(tmp_i, p->pt_obs_off, n_pt + 1); v.pt_obs_off = tmp_i;
  UP(tmp_f, p->pt_obs_uvr, 3 * (size_t)n_pe); v.pe_uvr = tmp_f;
  UP(tmp_f, p->pt_obs_info, n_pe); v.pe_info = tmp_f;
  UP(tmp_i, p->ln_obs_off, n_ln + 1); v.ln_obs_off = tmp_i;
  UP(tmp_f, p->ln_obs_left, 4 * (size_t)n_lc); v.lc_left = tmp_f;
  UP(tmp_f, p->ln_obs_right, 4 * (size_t)n_lc); v.lc_right = tmp_f;
  UP(tmp_d, p->ln_obs_info, 2 * (size_t)n_lc); v.lc_info = tmp_d;
  UP(tmp_u, p->ln_obs_stereo, n_lc); v.lc_stereo = tmp_u;
  {
    double *d_T, *d_P, *d_L;
    UP(d_T, p->kf_Tcw, 12 * (size_t)n_kf);
    UP(d_P, p->pt_xyz, 3 * (size_t)n_pt);
    UP(d_L, p->ln_x0_dir, 6 * (size_t)n_ln);
    S->d_kf_Tcw_in = d_T; S->d_pt_in = d_P; S->d_ln_in = d_L;
  }

  // ---- host indexing ----
  const bool timing = getenv("LLD_TIMING") != nullptr;
  auto t_prev = std::chrono::steady_clock::now();
  auto stage = [&](const char* name) {
    if (!timing) return;
    auto now = std::chrono::steady_clock::now();
    fprintf(stderr, "[lld_ba_upload] %-28s %8.3f ms\n", name, std::chrono::duration<double, std::milli>(now - t_prev).count());
    t_prev = now;
  };
  if (!c->ba_host) c->ba_host = new BaHost();
  BaHost& H = *reinterpret_cast<BaHost*>(c->ba_host);
  auto par_for = [&](int n, auto f) { H.par_for(n, f); };
  auto& kf_win = H.kf_win; auto& kf_g = H.kf_g; auto& w_g0 = H.w_g0;
  auto& g_kf = H.g_kf;
  kf_win.resize(n_kf); kf_g.assign(n_kf, -1); w_g0.assign(nw + 1, 0);   // (landmark -> window owners: device only)
  g_kf.clear();
  for (int w = 0; w < nw; w++) {
    w_g0[w] = (int)g_kf.size();
    for (int k = p->kf_off[w]; k < p->kf_off[w + 1]; k++) {
      kf_win[k] = w;
      if (!p->kf_fixed[k]) {
        kf_g[k] = (int)g_kf.size();
        g_kf.push_back(k);
      }
    }
    S->max_n = std::max(S->max_n, 6 * ((int)g_kf.size() - w_g0[w]));
  }
  w_g0[nw] = (int)g_kf.size();
  const int nG = (int)g_kf.size();
  v.n_free_total = nG;

  auto& pe_kf = H.pe_kf; auto& pe_pt = H.pe_pt; auto& lc_kf = H.lc_kf; auto& lc_ln = H.lc_ln;
  pe_kf.resize(n_pe); pe_pt.resize(n_pe); lc_kf.resize(n_lc); lc_ln.resize(n_lc);
  std::atomic<int> bad_arg{0};
  // Three per-window passes, run back to back by the same worker while the window's edges are in its cache:
  //   (1) global keyframe / landmark ids of every edge (+ argument checks),
  //   (2) co-visibility signature of every landmark (set of free blocks observing it) and the stable signature order:
  //       landmarks with the same signature are adjacent in every keyframe's list, so k_schur_rows tests "does neighbour j
  //       see these landmarks" once per segment, and dense mode cuts the order into pieces,
  //   (3) lengths of the per-free-keyframe edge lists.
  auto ids_window = [&](int w) -> bool {
    bool ok = true;
    const int k0 = p->kf_off[w], nk = p->kf_off[w + 1] - k0;
    for (int i = p->pt_off[w]; i < p->pt_off[w + 1]; i++) {
      if (p->pt_obs_off[i + 1] - p->pt_obs_off[i] > 254) ok = false;
      for (int e = p->pt_obs_off[i]; e < p->pt_obs_off[i + 1]; e++) {
        if (p->pt_obs_kf[e] < 0 || p->pt_obs_kf[e] >= nk) { ok = false; continue; }
        pe_kf[e] = k0 + p->pt_obs_kf[e];
      }
    }
    for (int i = p->ln_off[w]; i < p->ln_off[w + 1]; i++) {
      if (p->ln_obs_off[i + 1] - p->ln_obs_off[i] > 254) ok = false;
      for (int e = p->ln_obs_off[i]; e < p->ln_obs_off[i + 1]; e++) {
        if (p->ln_obs_kf[e] < 0 || p->ln_obs_kf[e] >= nk) { ok = false; continue; }
        lc_kf[e] = k0 + p->ln_obs_kf[e];
      }
    }
    if (!ok) bad_arg = 1;
    return ok;
  };
  std::atomic<int> dup_free{0};   // a landmark observed twice by the same free keyframe (never happens in the reference)
  auto signature = [&](const int* off, const pvec<int>& ekf, int i, int g0, int nf) -> uint64_t {
    uint64_t key = 0;
    if (nf <= 64) {
      for (int e = off[i]; e < off[i + 1]; e++) {
        const int g = kf_g[ekf[e]];
        if (g >= 0) {
          if (key & (1ull << (g - g0))) dup_free = 1;
          key |= 1ull << (g - g0);
        }
      }
    } else {  // FNV-1a over the sorted block list; segments are verified exactly below, the key only orders
      static thread_local std::vector<int> gs;   // (one allocation per worker thread, not one per landmark)
      gs.clear();
      for (int e = off[i]; e < off[i + 1]; e++)
        if (kf_g[ekf[e]] >= 0) gs.push_back(kf_g[ekf[e]]);
      std::sort(gs.begin(), gs.end());
      if (std::adjacent_find(gs.begin(), gs.end()) != gs.end()) dup_free = 1;
      key = 1469598103934665603ull;
      for (int g : gs) { key ^= (uint64_t)(g + 1); key *= 1099511628211ull; }
    }
    return key;
  };
  auto& pt_order = H.pt_order; auto& ln_order = H.ln_order; auto& pt_key = H.pt_key; auto& ln_key = H.ln_key;
  pt_order.resize(n_pt); ln_order.resize(n_ln); pt_key.resize(n_pt); ln_key.resize(n_ln);
  bool keys_ready = false;   // single large window (global BA): ids and signatures are computed by landmark ranges in parallel
  auto sort_window = [&](int w) {
    const int g0 = w_g0[w], nf = w_g0[w + 1] - g0;
    // stable order by signature; with <= 32 free keyframes the key and the landmark's window-local index fit one 64-bit word
    auto sort_by_key = [&](const int* lm_off, const int* off, const pvec<int>& ekf, std::vector<uint64_t>& key, pvec<int>& order) {
      const int b = lm_off[w], e = lm_off[w + 1];
      if (!keys_ready)
        for (int i = b; i < e; i++) key[i] = signature(off, ekf, i, g0, nf);
      if (nf <= 32) {
        // LSD radix sort on the nf mask bits, 11 bits per pass; the low word (window-local index) starts ascending and
        // the passes are stable, so equal signatures keep the reference's insertion order
        const int m = e - b;
        static thread_local std::vector<uint64_t> packed, tmp;   // per worker thread, reused across windows and calls
        if ((int)packed.size() < m) { packed.resize((size_t)m); tmp.resize((size_t)m); }
        for (int i = b; i < e; i++) packed[i - b] = (key[i] << 32) | (uint32_t)(i - b);
        uint64_t* src = packed.data();
        uint64_t* dst = tmp.data();
        const int RB = 11;   // bits per pass: 19-20 free keyframes (the usual local window) sort in two passes
        for (int sh = 32; sh < 32 + nf; sh += RB) {
          int cnt[(1 << RB) + 1] = {0};
          for (int i = 0; i < m; i++) cnt[((src[i] >> sh) & ((1u << RB) - 1)) + 1]++;
          for (int q = 0; q < (1 << RB); q++) cnt[q + 1] += cnt[q];
          for (int i = 0; i < m; i++) dst[cnt[(src[i] >> sh) & ((1u << RB) - 1)]++] = src[i];
          std::swap(src, dst);
        }
        for (int i = b; i < e; i++) order[i] = b + (int)(src[i - b] & 0xffffffffu);
      } else {
        // 64-bit keys (hash of the block list): stable LSD radix sort of (key, index) pairs, 11 bits per pass -- the same
        // order as a stable sort by key, several times faster on the 300 k landmarks of a global problem
        const int m = e - b;
        static thread_local std::vector<uint64_t> kk, kt;
        static thread_local std::vector<int> ii, it;
        if ((int)kk.size() < m) { kk.resize((size_t)m); kt.resize((size_t)m); ii.resize((size_t)m); it.resize((size_t)m); }
        for (int i = 0; i < m; i++) { kk[i] = key[b + i]; ii[i] = b + i; }
        uint64_t* ks = kk.data(); uint64_t* kd = kt.data();
        int* is = ii.data(); int* id = it.data();
        const int RB = 11;
        for (int sh = 0; sh < 64; sh += RB) {
          std::vector<int> cnt((1 << RB) + 1, 0);
          for (int i = 0; i < m; i++) cnt[((ks[i] >> sh) & ((1u << RB) - 1)) + 1]++;
          if (cnt[1] == m) continue;   // every key has a zero digit here
          for (int q = 0; q < (1 << RB); q++) cnt[q + 1] += cnt[q];
          for (int i = 0; i < m; i++) {
            const int pos = cnt[(ks[i] >> sh) & ((1u << RB) - 1)]++;
            kd[pos] = ks[i]; id[pos] = is[i];
          }
          std::swap(ks, kd); std::swap(is, id);
        }
        for (int i = 0; i < m; i++) order[b + i] = is[i];
      }
    };
    sort_by_key(p->pt_off, p->pt_obs_off, pe_kf, pt_key, pt_order);
    sort_by_key(p->ln_off, p->ln_obs_off, lc_kf, ln_key, ln_order);
  };
  // per-free-keyframe lists (counting sort in signature order), separately for point edges and line cells.  A window's
  // edges only touch the window's own free blocks; the counters of neighbouring windows share cache lines (19 ints per
  // window), so every worker counts in a private array and touches the shared one once per block.
  auto& pl_off = H.pl_off; auto& pl_edge = H.pl_edge; auto& pe_pos = H.pe_pos;
  auto& ll_off = H.ll_off; auto& ll_cell = H.ll_cell; auto& lc_pos = H.lc_pos;
  pl_off.assign(nG + 1, 0); ll_off.assign(nG + 1, 0);
  auto count_window = [&](int w, const int* lm_off, const int* off, const pvec<int>& ekf, pvec<int>& l_off) {
    const int g0 = w_g0[w], nf = w_g0[w + 1] - g0;
    std::vector<int> cnt((size_t)nf, 0);
    for (int e = off[lm_off[w]]; e < off[lm_off[w + 1]]; e++)
      if (kf_g[ekf[e]] >= 0) cnt[kf_g[ekf[e]] - g0]++;
    for (int j = 0; j < nf; j++) l_off[g0 + j + 1] = cnt[j];
  };
  auto fill_window = [&](int w, const int* lm_off, const int* off, const pvec<int>& ekf, const pvec<int>& order,
                         const pvec<int>& l_off, pvec<int>& l_ref, pvec<int>& e_pos) {
    const int g0 = w_g0[w], nf = w_g0[w + 1] - g0;
    std::vector<int> cur(l_off.begin() + g0, l_off.begin() + g0 + nf);
    for (int oi = lm_off[w]; oi < lm_off[w + 1]; oi++) {
      const int i = order[oi];
      for (int e = off[i]; e < off[i + 1]; e++) {
        const int g = kf_g[ekf[e]];
        if (g < 0) { e_pos[e] = -1; continue; }
        e_pos[e] = cur[g - g0];
        l_ref[cur[g - g0]++] = e;
      }
    }
  };
  if (nw == 1 && n_pt + n_ln >= 65536) {
    const int nk = p->kf_off[1] - p->kf_off[0], g0 = w_g0[0], nf = w_g0[1] - g0, parts = 64;
    par_for(parts, [&](int part) {
      bool ok = true;
      auto range = [&](int n_lm, const int32_t* off, const int32_t* okf, pvec<int>& ekf, std::vector<uint64_t>& key) {
        const int i0 = (int)((long long)n_lm * part / parts), i1 = (int)((long long)n_lm * (part + 1) / parts);
        for (int i = i0; i < i1; i++) {
          if (off[i + 1] - off[i] > 254) ok = false;
          for (int e = off[i]; e < off[i + 1]; e++) {
            if (okf[e] < 0 || okf[e] >= nk) { ok = false; ekf[e] = p->kf_off[0]; continue; }
            ekf[e] = p->kf_off[0] + okf[e];
          }
        }
        if (ok)
          for (int i = i0; i < i1; i++) key[i] = signature(off, ekf, i, g0, nf);
      };
      range(n_pt, p->pt_obs_off, p->pt_obs_kf, pe_kf, pt_key);
      range(n_ln, p->ln_obs_off, p->ln_obs_kf, lc_kf, ln_key);
      if (!ok) bad_arg = 1;
    });
    if (bad_arg.load()) {
      snprintf(c->err, sizeof(c->err), "malformed problem: an observation names a keyframe outside the window, or a landmark has more than 254 observations (include/lldba.h, capacity limits)");
      return LLD_ERR_ARG;
    }
    keys_ready = true;
  }
  // single large window: the two signature sorts run side by side, and the keyframe lists are a parallel counting sort over
  // ranges of the signature order (per-range counters, prefix over the ranges, private cursors: the same lists as the serial fill)
  const bool big_single = keys_ready;
  const int LP = 64;   // ranges
  std::vector<int> cnt_pt, cnt_ln;
  auto count_ranges = [&](int n_lm, const int* off, const pvec<int>& ekf, const pvec<int>& order, std::vector<int>& cntp) {
    const int g0 = w_g0[0], nf = w_g0[1] - g0;
    cntp.assign((size_t)LP * nf, 0);
    par_for(LP, [&](int part) {
      int* cn = cntp.data() + (size_t)part * nf;
      for (int oi = (int)((long long)n_lm * part / LP); oi < (int)((long long)n_lm * (part + 1) / LP); oi++) {
        const int i = order[oi];
        for (int e = off[i]; e < off[i + 1]; e++)
          if (kf_g[ekf[e]] >= 0) cn[kf_g[ekf[e]] - g0]++;
      }
    });
  };
  if (big_single) {
    sort_window(0);
    count_ranges(n_pt, p->pt_obs_off, pe_kf, pt_order, cnt_pt);
    count_ranges(n_ln, p->ln_obs_off, lc_kf, ln_order, cnt_ln);
    const int g0 = w_g0[0], nf = w_g0[1] - g0;
    for (int j = 0; j < nf; j++) {
      int sp = 0, sl = 0;
      for (int part = 0; part < LP; part++) { sp += cnt_pt[(size_t)part * nf + j]; sl += cnt_ln[(size_t)part * nf + j]; }
      pl_off[g0 + j + 1] = sp; ll_off[g0 + j + 1] = sl;
    }
  } else {
    par_for(nw, [&](int w) {
      if (!keys_ready && !ids_window(w)) return;   // malformed window: rejected below, nothing else may index with its ids
      sort_window(w);
      count_window(w, p->pt_off, p->pt_obs_off, pe_kf, pl_off);
      count_window(w, p->ln_off, p->ln_obs_off, lc_kf, ll_off);
    });
  }
  if (bad_arg.load()) {
    snprintf(c->err, sizeof(c->err), "malformed problem: an observation names a keyframe outside the window, or a landmark has more than 254 observations (include/lldba.h, capacity limits)");
    return LLD_ERR_ARG;
  }
  // arrays that are final from here on go to the device now: their DMA (queued behind the caller's raw arrays on the
  // same stream) runs under the rest of the indexing instead of after it
  UP(tmp_i, pe_kf.data(), n_pe); v.pe_kf = tmp_i;
  UP(tmp_i, lc_kf.data(), n_lc); v.lc_kf = tmp_i;
  UP(tmp_i, pt_order.data(), n_pt); v.pt_sorted = tmp_i;
  UP(tmp_i, ln_order.data(), n_ln); v.ln_sorted = tmp_i;
  stage("ids + signature order + list counts");
  // dense mode: every window small enough to keep its whole S in registers / one edge per (landmark, free KF)
  const bool dense = !global_mode && S->max_n <= 6 * 32 && dup_free.load() == 0;
  LLD_ARG(c, dup_free.load() == 0 || !global_mode);
  v.dense_mode = dense ? 1 : 0;
  for (int g = 0; g < nG; g++) { pl_off[g + 1] += pl_off[g]; ll_off[g + 1] += ll_off[g]; }
  pl_edge.resize(std::max(pl_off[nG], 1)); ll_cell.resize(std::max(ll_off[nG], 1));
  pe_pos.resize(std::max(n_pe, 1)); lc_pos.resize(std::max(n_lc, 1));
  auto fill_ranges = [&](int n_lm, const int* off, const pvec<int>& ekf, const pvec<int>& order, std::vector<int>& cntp,
                         const pvec<int>& l_off, pvec<int>& l_ref, pvec<int>& e_pos) {
    const int g0 = w_g0[0], nf = w_g0[1] - g0;
    for (int j = 0; j < nf; j++) {   // counters -> first list position of every (range, keyframe)
      int run = l_off[g0 + j];
      for (int part = 0; part < LP; part++) { const int c2 = cntp[(size_t)part * nf + j]; cntp[(size_t)part * nf + j] = run; run += c2; }
    }
    par_for(LP, [&](int part) {
      int* cur = cntp.data() + (size_t)part * nf;
      for (int oi = (int)((long long)n_lm * part / LP); oi < (int)((long long)n_lm * (part + 1) / LP); oi++) {
        const int i = order[oi];
        for (int e = off[i]; e < off[i + 1]; e++) {
          const int g = kf_g[ekf[e]];
          if (g < 0) { e_pos[e] = -1; continue; }
          e_pos[e] = cur[g - g0];
          l_ref[cur[g - g0]++] = e;
        }
      }
    });
  };
  if (big_single) {
    fill_ranges(n_pt, p->pt_obs_off, pe_kf, pt_order, cnt_pt, pl_off, pl_edge, pe_pos);
    fill_ranges(n_ln, p->ln_obs_off, lc_kf, ln_order, cnt_ln, ll_off, ll_cell, lc_pos);
  } else {
    par_for(nw, [&](int w) {
      fill_window(w, p->pt_off, p->pt_obs_off, pe_kf, pt_order, pl_off, pl_edge, pe_pos);
      fill_window(w, p->ln_off, p->ln_obs_off, lc_kf, ln_order, ll_off, ll_cell, lc_pos);
    });
  }
  // sparse mode, a landmark seen more than once by one free keyframe: per (landmark, keyframe) the list position the position
  // tables name (the last such edge) and the positions whose W records k_fold_dup adds into it
  std::vector<int> fold_off(1, 0), fold_dst, fold_src;
  int n_fold_pt = 0;
  if (!dense && dup_free.load()) {
    auto fold_groups = [&](int n_lm, const int* off, const pvec<int>& ekf, const pvec<int>& e_pos) {
      std::vector<std::pair<int, int>> gs;   // (free block, edge) of one landmark, sorted: edges of a block in list order
      for (int i = 0; i < n_lm; i++) {
        gs.clear();
        for (int e = off[i]; e < off[i + 1]; e++)
          if (kf_g[ekf[e]] >= 0) gs.push_back({kf_g[ekf[e]], e});
        std::sort(gs.begin(), gs.end());
        for (size_t a = 0; a < gs.size();) {
          size_t b = a + 1;
          while (b < gs.size() && gs[b].first == gs[a].first) b++;
          if (b - a > 1) {
            fold_dst.push_back(e_pos[gs[b - 1].second]);
            for (size_t k = a; k + 1 < b; k++) fold_src.push_back(e_pos[gs[k].second]);
            fold_off.push_back((int)fold_src.size());
          }
          a = b;
        }
      }
    };
    fold_groups(n_pt, p->pt_obs_off, pe_kf, pe_pos);
    n_fold_pt = (int)fold_dst.size();
    fold_groups(n_ln, p->ln_obs_off, lc_kf, lc_pos);
  }
  v.n_fold = (int)fold_dst.size(); v.n_fold_pt = n_fold_pt;
  UP(tmp_i, fold_off.data(), fold_off.size()); v.fold_off = tmp_i;
  UP(tmp_i, fold_dst.data(), fold_dst.size()); v.fold_dst = tmp_i;
  UP(tmp_i, fold_src.data(), fold_src.size()); v.fold_src = tmp_i;
  const int n_plist = pl_off[nG], n_llist = ll_off[nG];
  UP(tmp_i, pl_off.data(), nG + 1); v.pl_off = tmp_i;
  UP(tmp_i, pl_edge.data(), n_plist); v.pl_edge = tmp_i;
  UP(tmp_i, ll_off.data(), nG + 1); v.ll_off = tmp_i;
  UP(tmp_i, ll_cell.data(), n_llist); v.ll_cell = tmp_i;
  stage("kf lists");
  // neighbour lists (block columns >= own row)
  std::vector<int> nb_off(nG + 1, 0), nb_g;
  if (!global_mode) {
    for (int w = 0; w < nw; w++)
      for (int g = w_g0[w]; g < w_g0[w + 1]; g++) {
        nb_off[g] = (int)nb_g.size();
        for (int b = g; b < w_g0[w + 1]; b++) nb_g.push_back(b);
      }
    nb_off[nG] = (int)nb_g.size();
  } else {
    // covisibility: blocks sharing at least one landmark.  One bit per (row block a, column block b >= a); every worker
    // marks the pairs of its landmark range in a private nG x nG bitmap (280 KB at 1.5k keyframes: cache resident), the
    // bitmaps are OR-ed row by row when the lists are extracted.
    // every rank derives the block pattern from the WHOLE problem (single window: kf index == local index)
    const lld_ba_problem* sp = full ? full : p;
    const int sn_pt = sp->pt_off[1], sn_ln = sp->ln_off[1];
    const size_t row_w = ((size_t)nG + 63) / 64;
    const int n_part = std::max(1, std::min<int>(16, (sn_pt + sn_ln) / 4096));
    std::vector<std::vector<uint64_t>> bm((size_t)n_part);
    par_for(n_part, [&](int part) {
      auto& B = bm[(size_t)part];
      B.assign(row_w * (size_t)nG, 0);
      std::vector<int> gs;
      auto mark = [&](const int32_t* off, const int32_t* okf, int i) {
        gs.clear();
        for (int e = off[i]; e < off[i + 1]; e++)
          if (kf_g[okf[e]] >= 0) gs.push_back(kf_g[okf[e]]);
        std::sort(gs.begin(), gs.end());
        for (size_t a = 0; a < gs.size(); a++)
          for (size_t b = a; b < gs.size(); b++) B[row_w * (size_t)gs[a] + ((size_t)gs[b] >> 6)] |= 1ull << (gs[b] & 63);
      };
      for (int i = (int)((long long)sn_pt * part / n_part); i < (int)((long long)sn_pt * (part + 1) / n_part); i++) mark(sp->pt_obs_off, sp->pt_obs_kf, i);
      for (int i = (int)((long long)sn_ln * part / n_part); i < (int)((long long)sn_ln * (part + 1) / n_part); i++) mark(sp->ln_obs_off, sp->ln_obs_kf, i);
    });
    for (int g = 0; g < nG; g++) {
      nb_off[g] = (int)nb_g.size();
      for (size_t wd = (size_t)g >> 6; wd < row_w; wd++) {
        uint64_t bits = 0;
        for (int part = 0; part < n_part; part++) bits |= bm[(size_t)part][row_w * (size_t)g + wd];
        if (wd == ((size_t)g >> 6)) bits |= 1ull << (g & 63);   // the diagonal block always exists
        while (bits) {
          const int b = (int)(wd * 64) + __builtin_ctzll(bits);
          bits &= bits - 1;
          nb_g.push_back(b);
        }
      }
    }
    nb_off[nG] = (int)nb_g.size();
  }
  for (int g = 0; g < nG; g++) S->max_nnb = std::max(S->max_nnb, nb_off[g + 1] - nb_off[g]);
  S->n_nb_total = nb_g.size();
  if (6 * S->max_nnb > 1024) {
    snprintf(c->err, sizeof(c->err), "a keyframe is covisible with %d free keyframes; this implementation supports at most 170 (include/lldba.h, capacity limits)", S->max_nnb);
    return LLD_ERR_UNSUPPORTED;
  }
  stage("neighbours");
  // position tables: per list entry and neighbour, the list position of the co-edge (or -1)
  // The tables themselves (hundreds of MB in global BA) are filled on the DEVICE from arrays it has anyway (k_build_tab):
  // the host only lays them out.  LLD_TAB_CHECK=1 also builds them here and compares after the device pass.
  static const bool tab_check = getenv("LLD_TAB_CHECK") != nullptr;
  auto build_tab = [&](const pvec<int>& l_off, const pvec<int>& l_ref, const int* off, const pvec<int>& e_lm,
                       const pvec<int>& ekf, const pvec<int>& e_pos, std::vector<long long>& t_off, pvec<int>& tab, long long* tot_out) {
    t_off.assign(std::max(nG, 1), 0);
    long long tot = 0;
    for (int g = 0; g < nG; g++) {
      t_off[g] = tot;
      tot += (long long)(l_off[g + 1] - l_off[g]) * (nb_off[g + 1] - nb_off[g]);
    }
    *tot_out = tot;
    if (!tab_check) return;
    tab.resize((size_t)std::max(tot, 1LL));   // (no fill here: every worker initialises the rows it owns)
    if (tot == 0) tab[0] = -1;
    par_for(nG, [&](int g) {
      const int nnb = nb_off[g + 1] - nb_off[g];
      const int* nbl = nb_g.data() + nb_off[g];
      std::fill(tab.data() + t_off[g], tab.data() + t_off[g] + (long long)(l_off[g + 1] - l_off[g]) * nnb, -1);
      for (int i = l_off[g]; i < l_off[g + 1]; i++) {
        int* row = tab.data() + t_off[g] + (long long)(i - l_off[g]) * nnb;
        const int lm = e_lm[l_ref[i]];
        for (int e2 = off[lm]; e2 < off[lm + 1]; e2++) {
          const int b = kf_g[ekf[e2]];
          if (b < g) continue;
          const int j = global_mode ? (int)(std::lower_bound(nbl, nbl + nnb, b) - nbl) : b - g;
          row[j] = e_pos[e2];
        }
      }
    });
  };
  std::vector<long long> pl_tab_off(std::max(nG, 1), 0), ll_tab_off(std::max(nG, 1), 0);
  auto& pl_tab = H.pl_tab; auto& ll_tab = H.ll_tab;
  long long pl_tab_total = 0, ll_tab_total = 0;
  if (dense) { pl_tab.resize(1); ll_tab.resize(1); pl_tab[0] = -1; ll_tab[0] = -1; }
  if (!dense) {
    // edge -> landmark owners: only these sparse-mode tables read them on the host (the device derives its own copy)
    par_for(nw, [&](int w) {
      for (int i = p->pt_off[w]; i < p->pt_off[w + 1]; i++)
        for (int e = p->pt_obs_off[i]; e < p->pt_obs_off[i + 1]; e++) pe_pt[e] = i;
      for (int i = p->ln_off[w]; i < p->ln_off[w + 1]; i++)
        for (int e = p->ln_obs_off[i]; e < p->ln_obs_off[i + 1]; e++) lc_ln[e] = i;
    });
    build_tab(pl_off, pl_edge, p->pt_obs_off, pe_pt, pe_kf, pe_pos, pl_tab_off, pl_tab, &pl_tab_total);
    build_tab(ll_off, ll_cell, p->ln_obs_off, lc_ln, lc_kf, lc_pos, ll_tab_off, ll_tab, &ll_tab_total);
  }
  stage("position tables");
  // dense-mode structures
  auto& pt_spos = H.pt_spos; auto& ln_spos = H.ln_spos; auto& pts_w0 = H.pts_w0; auto& lns_w0 = H.lns_w0;
  auto& pts_mask = H.pts_mask; auto& lns_mask = H.lns_mask;
  auto& gb_off = H.gb_off; auto& gv_off = H.gv_off; auto& gb_src = H.gb_src; auto& gv_src = H.gv_src;
  pt_spos.resize(std::max(n_pt, 1)); ln_spos.resize(std::max(n_ln, 1)); pts_w0.resize(n_pt + 1); lns_w0.resize(n_ln + 1);
  pts_w0[0] = 0; lns_w0[0] = 0;
  pts_mask.resize(std::max(n_pt, 1)); lns_mask.resize(std::max(n_ln, 1));
  gb_off.assign(1, 0); gv_off.assign(1, 0); gb_src.assign(1, 0); gv_src.assign(1, 0);
  long long dpart_total = 0;
  int n_items_pt = 0, n_items_all = 0;
  size_t n_pw = 0, n_lw = 0;
  if (dense) {
    // W slots: landmarks in signature order, each landmark's free edges sorted by keyframe
    // (the W slot of an edge = w0 of its landmark + rank of its keyframe in the mask is derived on the device: k_dense_wpos)
    // a landmark owns one W slot per free keyframe that sees it = one entry in one keyframe list, so the first slot of a
    // window is the first list position of its first free block: every window writes its own absolute prefix in parallel
    auto slots = [&](const int* lm_off, const pvec<int>& order, const std::vector<uint64_t>& key, pvec<int>& spos,
                     pvec<uint32_t>& mask, pvec<int>& w0, const pvec<int>& l_off) {
      par_for(nw, [&](int w) {
        int run = l_off[w_g0[w]];
        for (int oi = lm_off[w]; oi < lm_off[w + 1]; oi++) {
          const int i = order[oi];
          spos[i] = oi;
          mask[oi] = (uint32_t)key[i];
          run += __builtin_popcountll(key[i]);
          w0[oi + 1] = run;
        }
      });
    };
    slots(p->pt_off, pt_order, pt_key, pt_spos, pts_mask, pts_w0, pl_off);
    slots(p->ln_off, ln_order, ln_key, ln_spos, lns_mask, lns_w0, ll_off);
    n_pw = (size_t)pts_w0[n_pt]; n_lw = (size_t)lns_w0[n_ln];
    stage("dense: W slots");
    int PIECE_CAP = 128;  // shorter pieces when the batch is small, so that every SM gets warps
    while (PIECE_CAP > 8 && (long long)(n_pt + n_ln) * 5 / (2 * PIECE_CAP) < 16LL * c->sm_count) PIECE_CAP >>= 1;
    // pieces / items / gather entries: built per (kind, window) with local offsets, merged in order afterwards
    using Job = BaDenseJob;
    auto& jobs = H.jobs;
    if (jobs.size() < 2 * (size_t)nw) jobs.resize(2 * (size_t)nw);
    for (size_t j = 0; j < 2 * (size_t)nw; j++) jobs[j].clear();
    const size_t n_jobs = 2 * (size_t)nw;
    par_for(2 * nw, [&](int jid) {
      const int kind = jid / nw, w = jid % nw;
      Job& J = jobs[jid];
      const int* loff = kind == 0 ? p->pt_off : p->ln_off;
      const pvec<uint32_t>& mask = kind == 0 ? pts_mask : lns_mask;
      const int g0 = w_g0[w];
      int b = loff[w];
      while (b < loff[w + 1]) {
        int e = b + 1;
        while (e < loff[w + 1] && mask[e] == mask[b] && e - b < PIECE_CAP) e++;
        const uint32_t m = mask[b];
        const int n = __builtin_popcount(m);
        if (n > 0) {   // landmarks seen by fixed keyframes only have no Schur tasks
          const int pc = (int)J.pb.size();
          J.pb.push_back(b); J.pe.push_back(e); J.pn.push_back(n); J.pout.push_back(J.dsize);
          const int npair = n * (n + 1) / 2, ntask = 6 * npair + n;
          int hl[32], k = 0;
          for (int h = 0; h < 32; h++)
            if ((m >> h) & 1u) hl[k++] = h;
          int pr = 0;
          for (int ia = 0; ia < n; ia++)
            for (int ib = ia; ib < n; ib++, pr++) J.gb.push_back({nb_off[g0 + hl[ia]] + (hl[ib] - hl[ia]), J.dsize + 36LL * pr});
          for (int ia = 0; ia < n; ia++) J.gv.push_back({g0 + hl[ia], J.dsize + 36LL * npair + (long long)SCHUR_KS * ia});
          for (int t0 = 0; t0 < 2 * npair + n; t0 += SP_TPB) { J.itp.push_back(pc); J.itt.push_back(t0); }
          J.dsize += 36LL * npair + (long long)SCHUR_KS * n;
        }
        b = e;
      }
    });
    stage("dense: pieces");
    // merge the per-(kind, window) jobs: serial prefix over the job sizes, everything else per job / per window in parallel
    std::vector<long long> jd(n_jobs + 1, 0);
    std::vector<int> ji(n_jobs + 1, 0);
    for (size_t jid = 0; jid < n_jobs; jid++) {
      jd[jid + 1] = jd[jid] + jobs[jid].dsize;
      ji[jid + 1] = ji[jid] + (int)jobs[jid].itp.size();
    }
    dpart_total = jd[n_jobs];
    n_items_pt = ji[std::min<size_t>((size_t)nw, n_jobs)];
    n_items_all = ji[n_jobs];
    H.it_rec.resize(std::max(ji[n_jobs], 1));
    gb_off.assign(nb_g.size() + 1, 0);
    gv_off.assign(nG + 1, 0);
    par_for((int)n_jobs, [&](int jid) {
      Job& J = jobs[jid];
      const int ibase = ji[jid];
      const int kind = jid / nw, jw = jid % nw;
      for (size_t k = 0; k < J.itp.size(); k++) {
        const int q = J.itp[k];
        SchurItem& R = H.it_rec[ibase + k];
        R.l0 = J.pb[q]; R.nl = J.pe[q] - J.pb[q]; R.n = J.pn[q]; R.t0 = J.itt[k];
        R.w = jw; R.w0 = (kind == 0 ? pts_w0 : lns_w0)[J.pb[q]]; R.out = J.pout[q] + jd[jid];
        schur_item_shape(kind == 0 ? 3 : 4, R.n, R.nl, R.t0, &R.lc, &R.S, &R.nchunk);
      }
    });
    stage("dense: item records");
    {
      // k_schur_tile's CTAs take items b, b + G, ... : order each kind by decreasing cost and deal the rows in snake
      // order, so that every CTA gets about the same landmark x task volume
      auto& tmp = H.it_tmp; auto& keys = H.it_keys;
      tmp.resize(H.it_rec.size()); keys.resize(H.it_rec.size());
      auto item_order = [&](int kind) {
        const int i0 = kind == 0 ? 0 : n_items_pt, i1 = kind == 0 ? n_items_pt : ji[n_jobs];
        const int cntk = i1 - i0;
        if (cntk <= 0) return;
        const int G = std::min(cntk, 4 * c->sm_count);
        // counting sort by quantised cost (descending; 1024 buckets of 32 cost units, equal buckets keep their order)
        constexpr int NB = 1024;
        std::vector<int> cnt(NB + 1, 0);
        for (int i = i0; i < i1; i++) {
          const SchurItem& R = H.it_rec[i];
          const int ntask = R.n * (R.n + 1) + R.n;
          const uint64_t cost = 64 + (uint64_t)R.nl * (uint64_t)(std::min(ntask - R.t0, (int)SP_TPB) + R.n + 1);
          const int bkt = NB - 1 - (int)std::min<uint64_t>(cost >> 5, NB - 1);
          keys[i] = (uint64_t)bkt;
          cnt[bkt + 1]++;
          tmp[i] = R;
        }
        for (int q = 0; q < NB; q++) cnt[q + 1] += cnt[q];
        for (int i = i0; i < i1; i++) {
          const int k = cnt[(int)keys[i]]++;   // rank in cost order
          const int r = k / G, j = k - r * G, len = std::min(G, cntk - r * G);
          const int pos = (r & 1) ? len - 1 - j : j;
          H.it_rec[i0 + r * G + pos] = tmp[i];
        }
      };
      // a block / keyframe belongs to one window: its contributions come from that window's point job, then its line job.
      // The two item-order tasks (serial each) run in the same parallel region as the per-window gather counts.
      par_for(nw + 2, [&](int t) {
        if (t < 2) { item_order(t); return; }
        const int w = t - 2;
        for (int kind = 0; kind < 2; kind++) {
          Job& J = jobs[(size_t)kind * nw + w];
          for (auto& x : J.gb) gb_off[x.first + 1]++;
          for (auto& x : J.gv) gv_off[x.first + 1]++;
        }
      });
    }
    stage("dense: item order + gather counts");
    for (size_t i = 0; i < nb_g.size(); i++) gb_off[i + 1] += gb_off[i];
    for (int i = 0; i < nG; i++) gv_off[i + 1] += gv_off[i];
    gb_src.resize(std::max<size_t>((size_t)gb_off[nb_g.size()], 1));
    gv_src.resize(std::max<size_t>((size_t)gv_off[nG], 1));
    {
      std::vector<int> curb(gb_off.begin(), gb_off.end() - 1), curv(gv_off.begin(), gv_off.end() - 1);
      par_for(nw, [&](int w) {
        for (int kind = 0; kind < 2; kind++) {
          const size_t jid = (size_t)kind * nw + w;
          Job& J = jobs[jid];
          for (auto& x : J.gb) gb_src[curb[x.first]++] = x.second + jd[jid];
          for (auto& x : J.gv) gv_src[curv[x.first]++] = x.second + jd[jid];
        }
      });
    }
  }
  S->gather_long = dense && gb_src.size() > 32 * std::max<size_t>(nb_g.size(), 1);
  v.n_items = n_items_all;
  v.n_items_pt = dense ? n_items_pt : 0;

  stage("dense: gather lists");
  // chunks + segments (runs of entries whose table rows have the same -1 pattern)
  const long long n_list_total = (long long)n_plist + n_llist;
  int CH = dense ? CHUNK_DENSE : CHUNK;   // dense mode: the chunk is only the pose pass's reduction unit, longer amortises the CTA sum
  while (CH > 32 && n_list_total / CH < 2 * (long long)c->sm_count) CH >>= 1;
  auto& ch_g = H.ch_g; auto& ch_begin = H.ch_begin; auto& ch_end = H.ch_end; auto& ch_seg0 = H.ch_seg0;
  auto& seg_begin = H.seg_begin; auto& seg_end = H.seg_end; auto& g_chp0 = H.g_chp0; auto& g_chl0 = H.g_chl0;
  ch_g.clear(); ch_begin.clear(); ch_end.clear(); ch_seg0.clear(); seg_begin.clear(); seg_end.clear();
  g_chp0.assign(nG + 1, 0); g_chl0.assign(nG + 1, 0);
  auto build_chunks = [&](const pvec<int>& l_off, const pvec<int>& l_ref, const int* off, const pvec<int>& e_lm,
                          const pvec<int>& ekf, pvec<int>& g_c0) {
    // A segment is a run of list entries whose table rows have the same -1 pattern, i.e. whose landmarks are seen by the same
    // set of free blocks b >= g.  The sets are compared directly (a handful of ints per landmark), by the worker pool; the
    // lists below are then appended in keyframe order.
    std::vector<std::vector<int>> cuts;   // per keyframe: list positions i where a new segment starts
    if (!dense) {
      cuts.resize((size_t)nG);
      par_for(nG, [&](int g) {
        auto& cg = cuts[(size_t)g];
        int sa[256], sb[256];
        int na = 0;
        auto collect = [&](int i, int* out) {
          const int lm = e_lm[l_ref[i]];
          int n = 0;
          for (int e = off[lm]; e < off[lm + 1]; e++) {
            const int b = kf_g[ekf[e]];
            if (b >= g) out[n++] = b;
          }
          std::sort(out, out + n);
          return n;
        };
        int* pa = sa;
        int* pb = sb;
        bool have_a = false;
        for (int i = l_off[g] + 1; i < l_off[g + 1]; i++) {
          // entries are in signature order: most neighbours observe the same keyframes in the same order -- then the sets
          // are equal and nothing needs to be collected
          const int la = e_lm[l_ref[i - 1]], lb = e_lm[l_ref[i]];
          const int ea = off[la], eb = off[lb], n_e = off[la + 1] - ea;
          if (n_e == off[lb + 1] - eb && std::equal(ekf.data() + ea, ekf.data() + ea + n_e, ekf.data() + eb)) continue;   // pa stays valid for la's set == lb's set
          if (!have_a) na = collect(i - 1, pa);
          const int nb2 = collect(i, pb);
          if (nb2 != na || !std::equal(pa, pa + na, pb)) cg.push_back(i);
          std::swap(pa, pb);
          na = nb2;
          have_a = true;
        }
      });
    }
    for (int g = 0; g < nG; g++) {
      g_c0[g] = (int)ch_g.size();
      size_t ci = 0;
      for (int b = l_off[g]; b < l_off[g + 1]; b += CH) {
        const int e = std::min(b + CH, l_off[g + 1]);
        ch_g.push_back(g); ch_begin.push_back(b); ch_end.push_back(e);
        ch_seg0.push_back((int)seg_begin.size());
        int s0 = b;
        if (dense) { seg_begin.push_back(b); seg_end.push_back(e); }
        else {
          const auto& cg = cuts[(size_t)g];
          while (ci < cg.size() && cg[ci] <= b) ci++;          // a cut at the chunk start is the chunk boundary itself
          for (; ci < cg.size() && cg[ci] < e; ci++) { seg_begin.push_back(s0); seg_end.push_back(cg[ci]); s0 = cg[ci]; }
          seg_begin.push_back(s0); seg_end.push_back(e);
        }
      }
    }
    g_c0[nG] = (int)ch_g.size();
  };
  build_chunks(pl_off, pl_edge, p->pt_obs_off, pe_pt, pe_kf, g_chp0);
  const int n_chp = (int)ch_g.size();
  build_chunks(ll_off, ll_cell, p->ln_obs_off, lc_ln, lc_kf, g_chl0);
  const int n_ch = (int)ch_g.size();
  ch_seg0.push_back((int)seg_begin.size());
  v.n_chunks = n_ch;
  v.n_chunks_pt = n_chp;
  auto& ch_S_off = H.ch_S_off;
  ch_S_off.assign(std::max(n_ch, 1), 0);
  long long chS_total = 0;
  for (int ch = 0; ch < n_ch; ch++) {
    ch_S_off[ch] = chS_total;
    const int nnb = nb_off[ch_g[ch] + 1] - nb_off[ch_g[ch]];
    chS_total += 36LL * nnb + 6;
  }
  // envelope of the reduced camera system (global BA with a system too large for the dense solvers)
  std::vector<int> env_first(1, 0), env_blk_last(1, 0);
  std::vector<long long> env_rowptr(2, 0);
  v.env_mode = 0;
  if (global_mode && S->max_n > SMEM_SOLVE_MAX_N) {
    std::vector<int> fb(nG);
    for (int g = 0; g < nG; g++) fb[g] = g;
    for (int a = 0; a < nG; a++)
      for (int q = nb_off[a]; q < nb_off[a + 1]; q++) fb[nb_g[q]] = std::min(fb[nb_g[q]], a);
    const int n = 6 * nG;
    env_first.assign(n, 0); env_rowptr.assign(n + 1, 0); env_blk_last.assign(nG, 0);
    int maxlen = 1, ph = 6;
    for (int i = 0; i < n; i++) {
      env_first[i] = 6 * fb[i / 6];
      env_rowptr[i + 1] = env_rowptr[i] + (i - env_first[i] + 1);
      maxlen = std::max(maxlen, i - env_first[i] + 1);
    }
    for (int g = 0; g < nG; g++) env_blk_last[g] = g;
    for (int b = 0; b < nG; b++)
      for (int k = fb[b]; k <= b; k++) env_blk_last[k] = std::max(env_blk_last[k], b);
    for (int k = 0; k < nG; k++) ph = std::max(ph, 6 * (env_blk_last[k] - k));
    v.env_mode = 1; v.env_panel_h = ph; v.env_maxlen = maxlen;
    // block half-bandwidth: the longest free-keyframe span of one landmark
    int B = 1;
    for (int g = 0; g < nG; g++) B = std::max(B, g - fb[g]);
    S->env_smem = sizeof(double) * (6 * (size_t)ph + 8 + 32 * (size_t)maxlen + (size_t)n) + 64;
    // cyclic reduction over super-blocks of B keyframes whenever a dense super-block fits one SM's shared memory
    S->use_cr = 6 * B <= CR_MAX_M;
    if (S->use_cr) { S->cr.mb = B; S->cr.m = 6 * B; S->cr.N = (nG + B - 1) / B; S->cr.zs = 12 * B; }
    if (!S->use_cr && S->env_smem > 220 * 1024 && c->gba_sparse) {
      // loop closures: block elimination over the super-block graph (sp_solver.cuh)
      SpPlan P;
      sp_plan_build(nG, nb_off, nb_g, P);
      if (P.bytes > SP_MAX_BYTES) {
        snprintf(c->err, sizeof(c->err),
                 "global BA: the block-elimination plan of the reduced system needs %lld bytes of device memory (%d super-blocks "
                 "of %d keyframes, %zu off-diagonal blocks with fill), the limit is %lld (include/lldba.h, capacity limits)",
                 P.bytes, P.N, P.mb, P.blocks.size(), SP_MAX_BYTES);
        return LLD_ERR_UNSUPPORTED;
      }
      S->use_sp = true;
      S->sp.N = P.N; S->sp.m = P.m; S->sp.mb = P.mb;
      S->sp_levels = P.levels;
      if (c->host_only) S->sp_report = sp_plan_json(P);
      UP(tmp_i, P.q_slot.data(), P.q_slot.size()); S->sp.q_slot = tmp_i;
      UP(tmp_i, P.el_node.data(), P.el_node.size()); S->sp.el_node = tmp_i;
      UP(tmp_i, P.el_nb_off.data(), P.el_nb_off.size()); S->sp.el_nb_off = tmp_i;
      { long long* tmp_z; UP(tmp_z, P.z_off.data(), P.z_off.size()); S->sp.z_off = tmp_z; }
      UP(tmp_i, P.nb_node.data(), P.nb_node.size()); S->sp.nb_node = tmp_i;
      UP(tmp_i, P.nb_slot2.data(), P.nb_slot2.size()); S->sp.nb_slot2 = tmp_i;
      UP(tmp_i, P.up_out.data(), P.up_out.size()); S->sp.up_out = tmp_i;
      UP(tmp_i, P.up_c_off.data(), P.up_c_off.size()); S->sp.up_c_off = tmp_i;
      UP(tmp_i, P.c_slot2.data(), P.c_slot2.size()); S->sp.c_slot2 = tmp_i;
      UP(tmp_i, P.c_pos.data(), P.c_pos.size()); S->sp.c_pos = tmp_i;
      UP(tmp_i, P.c_col.data(), P.c_col.size()); S->sp.c_col = tmp_i;
      S->sp_z_total = P.z_total; S->sp_n_slot = P.N + (long long)P.blocks.size();
    } else if (!S->use_cr && S->env_smem > 220 * 1024) {
      snprintf(c->err, sizeof(c->err),
               "global BA: envelope of the reduced system too wide for the on-chip solver: a landmark spans %d free keyframes "
               "(panel %d rows, row %d, n %d) and needs %zu bytes of shared memory, the limit is %d (include/lldba.h, capacity limits)",
               B + 1, ph, maxlen, n, S->env_smem, 220 * 1024);
      return LLD_ERR_UNSUPPORTED;
    }
  }
  // global-memory solve scratch for windows too large for shared memory
  std::vector<long long> w_scr(nw, 0);
  long long scr_total = 0;
  for (int w = 0; w < nw; w++) {
    const long long n = 6LL * (w_g0[w + 1] - w_g0[w]);
    w_scr[w] = scr_total;
    if (S->max_n > SMEM_SOLVE_MAX_N && !v.env_mode) scr_total += n * n + 8 * n + 40;
  }

  stage("chunks");
  // ---- upload (timed as h2d) ----
  UP(tmp_i, kf_win.data(), n_kf); v.kf_win = tmp_i;
  // owner arrays (landmark -> window, edge -> landmark) and W slots are derived on the device from the offsets / masks
  int *d_pt_win, *d_ln_win, *d_pe_pt, *d_lc_ln, *d_pe_wpos, *d_lc_wpos;
  DEV(d_pt_win, int, n_pt); v.pt_win = d_pt_win;
  DEV(d_ln_win, int, n_ln); v.ln_win = d_ln_win;
  UP(tmp_i, kf_g.data(), n_kf); v.kf_g = tmp_i;
  UP(tmp_i, g_kf.data(), nG); v.g_kf = tmp_i;
  UP(tmp_i, w_g0.data(), nw + 1); v.w_g0 = tmp_i;
  DEV(d_pe_pt, int, n_pe); v.pe_pt = d_pe_pt;
  DEV(d_lc_ln, int, n_lc); v.lc_ln = d_lc_ln;
  UP(tmp_i, pe_pos.data(), dense ? 0 : n_pe); v.pe_pos = tmp_i;   // list positions are only read outside dense mode
  UP(tmp_i, lc_pos.data(), dense ? 0 : n_lc); v.lc_pos = tmp_i;
  UP(tmp_i, ch_g.data(), n_ch); v.ch_g = tmp_i;
  UP(tmp_i, ch_begin.data(), n_ch); v.ch_begin = tmp_i;
  UP(tmp_i, ch_end.data(), n_ch); v.ch_end = tmp_i;
  UP(tmp_i, ch_seg0.data(), ch_seg0.size()); v.ch_seg0 = tmp_i;
  UP(tmp_i, seg_begin.data(), seg_begin.size()); v.seg_begin = tmp_i;
  UP(tmp_i, seg_end.data(), seg_end.size()); v.seg_end = tmp_i;
  UP(tmp_i, g_chp0.data(), nG + 1); v.g_chp0 = tmp_i;
  UP(tmp_i, g_chl0.data(), nG + 1); v.g_chl0 = tmp_i;
  UP(tmp_i, nb_off.data(), nG + 1); v.nb_off = tmp_i;
  UP(tmp_i, nb_g.data(), nb_g.size()); v.nb_g = tmp_i;
  int *d_pl_tab = nullptr, *d_ll_tab = nullptr;
  DEV(d_pl_tab, int, std::max(pl_tab_total, 1LL)); v.pl_tab = d_pl_tab;
  DEV(d_ll_tab, int, std::max(ll_tab_total, 1LL)); v.ll_tab = d_ll_tab;
  long long* tmp_l;
  UP(tmp_l, pl_tab_off.data(), nG); v.pl_tab_off = tmp_l;
  UP(tmp_l, ll_tab_off.data(), nG); v.ll_tab_off = tmp_l;
  UP(tmp_l, ch_S_off.data(), n_ch); v.ch_S_off = tmp_l;
  UP(tmp_i, pt_spos.data(), n_pt); v.pt_spos = tmp_i;
  UP(tmp_i, ln_spos.data(), n_ln); v.ln_spos = tmp_i;
  UP(tmp_i, pts_w0.data(), n_pt + 1); v.pts_w0 = tmp_i;
  UP(tmp_i, lns_w0.data(), n_ln + 1); v.lns_w0 = tmp_i;
  DEV(d_pe_wpos, int, n_pe); v.pe_wpos = d_pe_wpos;
  DEV(d_lc_wpos, int, n_lc); v.lc_wpos = d_lc_wpos;
  { SchurItem* tmp_r; UP(tmp_r, H.it_rec.data(), (size_t)n_items_all); v.it_rec = tmp_r; }
  UP(tmp_i, gb_off.data(), gb_off.size()); v.gb_off = tmp_i;
  UP(tmp_l, gb_src.data(), gb_src.size()); v.gb_src = tmp_l;
  UP(tmp_i, gv_off.data(), gv_off.size()); v.gv_off = tmp_i;
  UP(tmp_l, gv_src.data(), gv_src.size()); v.gv_src = tmp_l;
  {
    uint32_t* tmp_m;
    UP(tmp_m, pts_mask.data(), n_pt); v.pts_mask = tmp_m;
    UP(tmp_m, lns_mask.data(), n_ln); v.lns_mask = tmp_m;
  }
  UP(tmp_l, w_scr.data(), nw); v.w_scratch_off = tmp_l;
  UP(tmp_i, env_first.data(), env_first.size()); v.env_first = tmp_i;
  UP(tmp_i, env_blk_last.data(), env_blk_last.size()); v.env_blk_last = tmp_i;
  UP(tmp_l, env_rowptr.data(), env_rowptr.size()); v.env_rowptr = tmp_l;

  stage("H2D enqueue");
  if (c->host_only) return LLD_OK;  // lld_ba_index_only: the host stage is complete
  // ---- device-only buffers ----
  for (int b = 0; b < 2; b++) {
    DEV(v.pose_qt[b], double, 7 * (size_t)n_kf);
    DEV(v.pose_Rt[b], double, 12 * (size_t)n_kf);
    DEV(v.pt_xyz[b], double, 3 * (size_t)n_pt);
    DEV(v.ln_st[b], double, 5 * (size_t)n_ln);
  }
  DEV(v.pe_level, uint8_t, n_pe); DEV(v.lc_level, uint8_t, 2 * (size_t)n_lc); DEV(v.ln_removed, uint8_t, n_ln);
  DEV(v.pe_chi2, double, n_pe); DEV(v.lc_chi2, double, 2 * (size_t)n_lc);
  DEV(v.pt_H, double, 9 * (size_t)n_pt); DEV(v.ln_H, double, 14 * (size_t)n_ln);
  DEV(v.P_rec, double, dense ? 1 : 27 * (size_t)n_plist); DEV(v.L_rec, double, dense ? 1 : 38 * (size_t)n_llist);
  DEV(v.pe_Wl, double, 18 * n_pw); DEV(v.lc_Wl, double, 24 * n_lw);
  DEV(v.pts_D, double, dense ? 10 * (size_t)n_pt : 1); DEV(v.lns_D, double, dense ? 14 * (size_t)n_ln : 1);
  DEV(v.dpart, double, (size_t)dpart_total);
  DEV(v.ch_pose, double, 28 * (size_t)n_ch);
  // [g_bp | w_red_sum | g_Hpp] and [S_blk | g_bs] are contiguous: the multi-rank global BA all-reduces each group in one call
  DEV(v.g_bp, double, 6 * (size_t)nG + 4 * (size_t)nw + 21 * (size_t)nG);
  v.w_red_sum = v.g_bp + 6 * (size_t)nG; v.g_Hpp = v.w_red_sum + 4 * (size_t)nw;
  DEV(v.g_nact, int, nG);
  DEV(v.lm_chi2lin, double, n_pt + n_ln); DEV(v.lm_maxdiag, double, n_pt + n_ln); DEV(v.lm_active, uint8_t, n_pt + n_ln);
  DEV(v.ch_S, double, (size_t)chS_total);
  DEV(v.S_blk, double, 36 * nb_g.size() + 6 * (size_t)nG);
  v.g_bs = v.S_blk + 36 * nb_g.size(); DEV(v.g_x, double, 6 * (size_t)nG);
  DEV(v.pt_D, double, 9 * (size_t)n_pt); DEV(v.ln_D, double, 14 * (size_t)n_ln);
  DEV(v.pt_xl, double, 3 * (size_t)n_pt); DEV(v.ln_xl, double, 4 * (size_t)n_ln);
  DEV(v.lm_chi2, double, n_pt + n_ln); DEV(v.lm_scale, double, n_pt + n_ln);
  DEV(v.w_phase, int, nw); DEV(v.w_sel, int, nw); DEV(v.w_iter, int, nw); DEV(v.w_trials, int, nw);
  DEV(v.w_maxit, int, nw); DEV(v.w_nbad, int, nw); DEV(v.w_ok, int, nw); DEV(v.w_nlog, int, nw);
  DEV(v.w_lambda, double, nw); DEV(v.w_ni, double, nw); DEV(v.w_curchi, double, nw); DEV(v.w_inichi, double, nw);
  DEV(v.w_scale_p, double, nw); DEV(v.w_red_max, double, nw);
  {
    int max_lm = 0;
    for (int w = 0; w < nw; w++) max_lm = std::max(max_lm, (p->pt_off[w + 1] - p->pt_off[w]) + (p->ln_off[w + 1] - p->ln_off[w]));
    v.n_slices = std::max(1, std::min(128, max_lm / 16384));
  }
  DEV(v.w_part, double, 4 * (size_t)nw * v.n_slices);
  DEV(v.n_active_win, int, 2);   // [0] windows still running, [1] multi-rank stop agreement word
  v.log_stride = log_stride;
  DEV(v.chi2_log, double, (size_t)nw * log_stride); DEV(v.lambda_log, double, (size_t)nw * log_stride);
  DEV(v.trials_log, int, (size_t)nw * log_stride); DEV(v.iter_done, int, 2 * (size_t)nw);
  DEV(v.solve_scratch, double, (size_t)scr_total);
  DEV(v.env_A, double, (S->use_cr || S->use_sp) ? 1 : (size_t)env_rowptr.back());
  if (S->use_cr) {
    CrView& cr = S->cr;
    const size_t mm = (size_t)cr.m * cr.m, N = (size_t)cr.N;
    // D and U[0] are zero-filled together before every assembly: one allocation
    DEV(cr.D, double, 2 * N * mm); cr.U[0] = cr.D + N * mm;
    DEV(cr.U[1], double, N * mm); DEV(cr.L, double, N * mm); DEV(cr.Z, double, N * cr.m * cr.zs);
    DEV(cr.b, double, N * cr.m); DEV(cr.zc, double, N * cr.m); DEV(cr.x, double, N * cr.m);
    DEV(cr.ok, int, 1);
  }
  if (S->use_sp) {
    SpView& sp = S->sp;
    const size_t mm = (size_t)sp.m * sp.m, N = (size_t)sp.N;
    DEV(sp.W, double, (size_t)S->sp_n_slot * mm); DEV(sp.L, double, N * mm); DEV(sp.Z, double, std::max(S->sp_z_total, 1LL));
    DEV(sp.b, double, N * sp.m); DEV(sp.zc, double, N * sp.m); DEV(sp.x, double, N * sp.m);
    DEV(sp.ok, int, 1);
  }
  DEV(S->d_out_kf, double, 12 * (size_t)n_kf); DEV(S->d_out_pt, double, 3 * (size_t)n_pt);
  DEV(S->d_out_ln, double, 6 * (size_t)n_ln);
  DEV(S->d_pt_bad, uint8_t, n_pe); DEV(S->d_ln_bad, uint8_t, 2 * (size_t)n_lc);
  LLD_CUDA(c, cudaMemsetAsync(v.chi2_log, 0, sizeof(double) * (size_t)nw * log_stride, c->stream));
  LLD_CUDA(c, cudaMemsetAsync(v.lambda_log, 0, sizeof(double) * (size_t)nw * log_stride, c->stream));
  LLD_CUDA(c, cudaMemsetAsync(v.trials_log, 0, sizeof(int) * (size_t)nw * log_stride, c->stream));
  LLD_CUDA(c, cudaMemsetAsync(S->d_pt_bad, 0, n_pe ? n_pe : 1, c->stream));
  LLD_CUDA(c, cudaMemsetAsync(S->d_ln_bad, 0, n_lc ? 2 * (size_t)n_lc : 1, c->stream));

  ba_set_params(v, p);
  stage("device buffers");
  c->last_h2d_bytes = S->h2d_bytes;
  {
    const char* e = getenv("LLD_BA_GRAPH");
    const bool allow = !(e && e[0] == '0');
    const bool dense_single = v.dense_mode && !(global_mode && c->n_ranks > 1) && v.n_slices == 1 && S->max_n <= SMEM_SOLVE_MAX_N && !v.env_mode;
    S->forked = allow && dense_single;
    S->use_graph = allow && dense_single;
    S->lean = dense_single;
  }
  // derived index arrays (stream-ordered after the uploads, before any consumer)
  {
    auto grid = [](int n) { return (n + 255) / 256; };
    if (n_pt) LLD_LAUNCH(c, k_expand_owner, grid(n_pt), 256, 0, n_pt, nw, v.pt_off, d_pt_win);
    if (n_ln) LLD_LAUNCH(c, k_expand_owner, grid(n_ln), 256, 0, n_ln, nw, v.ln_off, d_ln_win);
    if (n_pe) LLD_LAUNCH(c, k_expand_owner, grid(n_pe), 256, 0, n_pe, n_pt, v.pt_obs_off, d_pe_pt);
    if (n_lc) LLD_LAUNCH(c, k_expand_owner, grid(n_lc), 256, 0, n_lc, n_ln, v.ln_obs_off, d_lc_ln);
    if (!v.dense_mode) {   // sparse-mode position tables (k_build_tab)
      LLD_CUDA(c, cudaMemsetAsync(d_pl_tab, 0xFF, sizeof(int) * (size_t)std::max(pl_tab_total, 1LL), c->stream));
      LLD_CUDA(c, cudaMemsetAsync(d_ll_tab, 0xFF, sizeof(int) * (size_t)std::max(ll_tab_total, 1LL), c->stream));
      if (n_plist) LLD_LAUNCH(c, k_build_tab, grid(n_plist), 256, 0, n_plist, nG, v.pl_off, v.pl_edge, v.pt_obs_off, v.pe_pt, v.pe_kf, v.kf_g,
                              v.pe_pos, v.nb_off, v.nb_g, v.pl_tab_off, d_pl_tab);
      if (n_llist) LLD_LAUNCH(c, k_build_tab, grid(n_llist), 256, 0, n_llist, nG, v.ll_off, v.ll_cell, v.ln_obs_off, v.lc_ln, v.lc_kf, v.kf_g,
                              v.lc_pos, v.nb_off, v.nb_g, v.ll_tab_off, d_ll_tab);
      if (tab_check) {
        std::vector<int> back((size_t)std::max(std::max(pl_tab_total, ll_tab_total), 1LL));
        for (int which = 0; which < 2; which++) {
          const long long tot = which ? ll_tab_total : pl_tab_total;
          LLD_CUDA(c, cudaMemcpyAsync(back.data(), which ? d_ll_tab : d_pl_tab, sizeof(int) * (size_t)tot, cudaMemcpyDeviceToHost, c->stream));
          LLD_CUDA(c, cudaStreamSynchronize(c->stream));
          const pvec<int>& ref = which ? ll_tab : pl_tab;
          long long bad = 0;
          for (long long k = 0; k < tot; k++) bad += back[(size_t)k] != ref[(size_t)k];
          fprintf(stderr, "[lld_ba_upload] LLD_TAB_CHECK %s table: %lld entries, %lld differ from the host build\n", which ? "line" : "point", tot, bad);
          if (bad) { snprintf(c->err, sizeof(c->err), "device-built position table differs from the host build"); return LLD_ERR_CUDA; }
        }
      }
    }
    if (v.dense_mode) {
      if (n_pe) LLD_LAUNCH(c, k_dense_wpos, grid(n_pe), 256, 0, n_pe, v.pe_pt, v.pe_kf, v.kf_g, v.pt_win, v.w_g0, v.pt_spos, v.pts_mask, v.pts_w0, d_pe_wpos);
      if (n_lc) LLD_LAUNCH(c, k_dense_wpos, grid(n_lc), 256, 0, n_lc, v.lc_ln, v.lc_kf, v.kf_g, v.ln_win, v.w_g0, v.ln_spos, v.lns_mask, v.lns_w0, d_lc_wpos);
    }
    LLD_CUDA(c, cudaGetLastError());
  }
  // dynamic shared memory opt-in of the solvers (once per upload, outside any stream capture)
  if (v.dense_mode) {
    LLD_CUDA(c, lld_raise_dyn_smem(k_schur_tile<3>, (size_t)SP_SMEM_BYTES));
    LLD_CUDA(c, lld_raise_dyn_smem(k_schur_tile<4>, (size_t)SP_SMEM_BYTES));
  }
  if (v.env_mode && S->use_cr) {
    LLD_CUDA(c, lld_raise_dyn_smem(k_cr_factor, sizeof(double) * ((size_t)S->cr.m * S->cr.m + 8 * (size_t)S->cr.m + 40)));
    LLD_CUDA(c, lld_raise_dyn_smem(k_cr_solve<15>, sizeof(double) * ((size_t)S->cr.m * S->cr.m + CR_RPT * CR_TC)));
    LLD_CUDA(c, lld_raise_dyn_smem(k_cr_solve<20>, sizeof(double) * ((size_t)S->cr.m * S->cr.m + CR_RPT * CR_TC)));
  } else if (v.env_mode && S->use_sp) {
    LLD_CUDA(c, lld_raise_dyn_smem(k_sp_factor, sizeof(double) * ((size_t)S->sp.m * S->sp.m + 8 * (size_t)S->sp.m + 40)));
    LLD_CUDA(c, lld_raise_dyn_smem(k_sp_solve<15>, sizeof(double) * ((size_t)S->sp.m * S->sp.m + CR_RPT * CR_TC)));
    LLD_CUDA(c, lld_raise_dyn_smem(k_sp_solve<20>, sizeof(double) * ((size_t)S->sp.m * S->sp.m + CR_RPT * CR_TC)));
  } else if (v.env_mode) LLD_CUDA(c, lld_raise_dyn_smem(k_solve_env, (size_t)(int)S->env_smem));
  else if (S->max_n <= SMEM_SOLVE_MAX_N)
    LLD_CUDA(c, lld_raise_dyn_smem(k_solve<true>, (size_t)(int)(sizeof(double) * ((size_t)S->max_n * S->max_n + 8 * (size_t)S->max_n + 40))));
  S->topo_ok = topo_cache && th != 0;
  return LLD_OK;
}

static inline int cdiv(int a, int b) { return (a + b - 1) / b; }

static int ba_init_state(LldCtx* c) {
  BaState* S = c->ba;
  BaView& v = S->v;
  const int n = std::max({v.n_kf, v.n_pt, v.n_ln, v.n_pe, v.n_lc, v.n_free_total, 1});
  LLD_LAUNCH(c, k_init_state, cdiv(n, 256), 256, 0, v, S->d_kf_Tcw_in, S->d_pt_in, S->d_ln_in, v.lc_right);
  LLD_CUDA(c, cudaGetLastError());
  return LLD_OK;
}

#ifdef LLD_WITH_NCCL
#define LLD_NCCL(ctx, call)                                                                              \
  do {                                                                                                   \
    ncclResult_t _r = (call);                                                                            \
    if (_r != ncclSuccess) {                                                                             \
      snprintf((ctx)->err, sizeof((ctx)->err), "%s:%d %s: %s", __FILE__, __LINE__, #call, ncclGetErrorString(_r)); \
      return LLD_ERR_NCCL;                                                                               \
    }                                                                                                    \
  } while (0)
#endif

// all-reduce hooks of the global BA (no-ops on one rank)
static int ba_allreduce_lin(LldCtx* c) {
#ifdef LLD_WITH_NCCL
  if (c->n_ranks > 1) {
    BaView& v = c->ba->v;
    ncclComm_t comm = reinterpret_cast<ncclComm_t>(c->comm);
    // one packed sum [g_bp | w_red_sum | g_Hpp] (contiguous by construction), the active-edge counts, the lambda_0 maximum
    LLD_NCCL(c, ncclAllReduce(v.g_bp, v.g_bp, 27 * (size_t)v.n_free_total + 4 * (size_t)v.n_win, ncclDouble, ncclSum, comm, c->stream));
    LLD_NCCL(c, ncclAllReduce(v.g_nact, v.g_nact, (size_t)v.n_free_total, ncclInt, ncclSum, comm, c->stream));
    LLD_NCCL(c, ncclAllReduce(v.w_red_max, v.w_red_max, (size_t)v.n_win, ncclDouble, ncclMax, comm, c->stream));
    c->nccl_calls += 3; c->nccl_bytes += 8 * (27 * (size_t)v.n_free_total + 5 * (size_t)v.n_win) + 4 * (size_t)v.n_free_total;
  }
#endif
  return LLD_OK;
}
static int ba_allreduce_trial(LldCtx* c) {
#ifdef LLD_WITH_NCCL
  if (c->n_ranks > 1) {
    BaView& v = c->ba->v;
    ncclComm_t comm = reinterpret_cast<ncclComm_t>(c->comm);
    LLD_NCCL(c, ncclAllReduce(v.w_red_sum, v.w_red_sum, 4 * (size_t)v.n_win, ncclDouble, ncclSum, comm, c->stream));
    c->nccl_calls += 1; c->nccl_bytes += 32 * (size_t)v.n_win;
  }
#endif
  return LLD_OK;
}

// multi-GPU: every rank holds the Schur contributions of its own landmarks; rank 0 alone carries Hpp + lambda I and bp
static int ba_allreduce_rows(LldCtx* c) {
#ifdef LLD_WITH_NCCL
  if (c->n_ranks > 1) {
    BaState* S = c->ba;
    BaView& v = S->v;
    ncclComm_t comm = reinterpret_cast<ncclComm_t>(c->comm);
    // S blocks and b_schur in one buffer: one all-reduce per LM trial carries the whole reduced camera system
    LLD_NCCL(c, ncclAllReduce(v.S_blk, v.S_blk, 36 * S->n_nb_total + 6 * (size_t)v.n_free_total, ncclDouble, ncclSum, comm, c->stream));
    c->nccl_calls += 1; c->nccl_bytes += 8 * (36 * S->n_nb_total + 6 * (size_t)v.n_free_total);
  }
#endif
  return LLD_OK;
}

// global BA: reduced camera system by block cyclic reduction (cr_solver.cuh); every kernel returns early when the window
// is done or an earlier factorisation failed
static int ba_solve_cr(LldCtx* c) {
  BaState* S = c->ba;
  BaView& v = S->v;
  const CrView& cr = S->cr;
  const int N = cr.N, m = cr.m;
  const size_t mm = (size_t)m * m;
  LLD_CUDA(c, cudaMemsetAsync(cr.D, 0, sizeof(double) * 2 * (size_t)N * mm, c->stream));
  const int nblk = (int)S->n_nb_total;
  LLD_LAUNCH(c, k_cr_assemble, (nblk * 36 + N * m + 255) / 256, 256, 0, v, cr, nblk);
  const size_t smem_f = sizeof(double) * (mm + 8 * (size_t)m + 40), smem_s = sizeof(double) * (mm + CR_RPT * CR_TC);
  const int ntile = (2 * m + CR_TC - 1) / CR_TC, T = (m + CR_TILE - 1) / CR_TILE, per = 2 * T * T + 1;
  int cur = 0, s = 1;
  for (; s < N; s *= 2, cur ^= 1) {
    const int n_el = ((N - 1) / s + 1) / 2, n_sv = (N - 1) / (2 * s) + 1;
    LLD_LAUNCH(c, k_cr_factor, n_el, 512, smem_f, v, cr, s);
    if (m <= 15 * CR_RG) LLD_LAUNCH(c, k_cr_solve<15>, n_el * ntile, CR_TC / 2 * CR_RG, smem_s, v, cr, s, cur);
    else LLD_LAUNCH(c, k_cr_solve<20>, n_el * ntile, CR_TC / 2 * CR_RG, smem_s, v, cr, s, cur);
    LLD_LAUNCH(c, k_cr_update, n_sv * per, 256, 0, v, cr, s, cur);
  }
  LLD_LAUNCH(c, k_cr_factor, 1, 512, smem_f, v, cr, 0);
  const int per_b = (m + 7) / 8;
  for (s >>= 1; s >= 1; s >>= 1) {
    const int n_el = ((N - 1) / s + 1) / 2;
    LLD_LAUNCH(c, k_cr_backsub, n_el * per_b, 256, 0, v, cr, s);
  }
  LLD_LAUNCH(c, k_cr_finish, 1, 1024, 0, v, cr);
  return LLD_OK;
}

// global BA across loop closures: the plan's levels (sp_solver.cuh); every kernel returns early when the window is done or
// an earlier factorisation failed
static int ba_solve_sp(LldCtx* c) {
  BaState* S = c->ba;
  BaView& v = S->v;
  const SpView& sp = S->sp;
  const int N = sp.N, m = sp.m;
  const size_t mm = (size_t)m * m;
  LLD_CUDA(c, cudaMemsetAsync(sp.W, 0, sizeof(double) * (size_t)S->sp_n_slot * mm, c->stream));
  const int nblk = (int)S->n_nb_total;
  LLD_LAUNCH(c, k_sp_assemble, (nblk * 36 + N * m + 255) / 256, 256, 0, v, sp, nblk);
  const size_t smem_f = sizeof(double) * (mm + 8 * (size_t)m + 40), smem_s = sizeof(double) * (mm + CR_RPT * CR_TC);
  const int T = (m + CR_TILE - 1) / CR_TILE;
  for (const auto& L : S->sp_levels) {
    LLD_LAUNCH(c, k_sp_factor, L.n_el, 512, smem_f, v, sp, L.p0);
    if (L.ntile == 0) continue;   // no remaining neighbours: nothing to eliminate into
    if (m <= 15 * CR_RG) LLD_LAUNCH(c, k_sp_solve<15>, L.n_el * L.ntile, CR_TC / 2 * CR_RG, smem_s, v, sp, L.p0, L.ntile);
    else LLD_LAUNCH(c, k_sp_solve<20>, L.n_el * L.ntile, CR_TC / 2 * CR_RG, smem_s, v, sp, L.p0, L.ntile);
    LLD_LAUNCH(c, k_sp_update, L.n_blk * T * T + L.n_rhs, 256, 0, v, sp, L.u0, L.n_blk);
  }
  const int per_b = (m + 7) / 8;
  for (auto it = S->sp_levels.rbegin(); it != S->sp_levels.rend(); ++it) LLD_LAUNCH(c, k_sp_backsub, it->n_el * per_b, 256, 0, v, sp, it->p0);
  CrView out{};   // k_cr_finish reads the solution and the ok flag only
  out.x = sp.x; out.ok = sp.ok;
  LLD_LAUNCH(c, k_cr_finish, 1, 1024, 0, v, out);
  return LLD_OK;
}

template <bool SMEM>
static int launch_solve(LldCtx* c, BaView& v, int max_n) {
  size_t smem = SMEM ? sizeof(double) * ((size_t)max_n * max_n + 8 * (size_t)max_n + 40) : 0;
  LLD_LAUNCH(c, k_solve<SMEM>, v.n_win, 512, smem, v);
  return LLD_OK;
}

// up to this many map lines the line kernels run eight lanes per line (single windows); one lane per line above
constexpr int LN_WIDE_MAX = 8192;
// same for map points, four lanes per point
constexpr int PT_WIDE_MAX = 32768;

// lanes per map line in k_lin_lines / k_backsub_lines: enough threads to fill the SMs, no more (idle lanes still shuffle)
static int lanes_per_line(const LldCtx* c, int n_ln) {
  static const int forced = getenv("LLD_LN_G") ? atoi(getenv("LLD_LN_G")) : 0;
  if (forced == 1 || forced == 2 || forced == 4 || forced == 8) return forced;
  if (n_ln <= LN_WIDE_MAX) return 8;
  return n_ln <= 1024 * c->sm_count ? 2 : 1;
}
static int launch_line_kernel(LldCtx* c, cudaStream_t strm, const BaView& v, bool lin, bool with_d = false) {
  if (!v.n_ln) return LLD_OK;
  const int g = lanes_per_line(c, v.n_ln);
  const int grid = cdiv(v.n_ln * g, LM_TPB);
#define LLD_LINE_CASE(G)                                                                   \
  case G:                                                                                  \
    if (lin && with_d) LLD_LAUNCH_S(c, strm, (k_lin_lines<G, true>), grid, LM_TPB, 0, v);  \
    else if (lin) LLD_LAUNCH_S(c, strm, (k_lin_lines<G, false>), grid, LM_TPB, 0, v);      \
    else LLD_LAUNCH_S(c, strm, k_backsub_lines<G>, grid, LM_TPB, 0, v);                    \
    break;
  switch (g) {
    LLD_LINE_CASE(1)
    LLD_LINE_CASE(2)
    LLD_LINE_CASE(4)
    LLD_LINE_CASE(8)
  }
#undef LLD_LINE_CASE
  return LLD_OK;
}

// Lean LM step (dense mode, every step of a round but the first; lambda is known when the step starts): 11 launches on three
// streams, critical path lin_points -> schur_tile<3> -> reduce -> solve -> backsub -> decide
//   s0: k_lin_points<G, D> -> k_schur_tile<3> |
//   s1: k_lin_lines<G, D>  -> k_schur_tile<4> |-> k_reduce_piece -> k_solve -> [k_backsub_points | k_backsub_lines] -> k_decide_carry
//   s2: k_lin_poses -> k_pose_sum             |
// against the first step: no k_begin_fused (chi2 is carried over from the accepted trial, lambda_0 is not needed), no
// k_schur_points / k_schur_lines (the linearisation kernels form D^-1 themselves), the pose sums leave the critical path.
static int ba_step_lean(LldCtx* c, int round, int stop_now) {
  BaState* S = c->ba;
  BaView& v = S->v;
  const int gp = cdiv(std::max(v.n_pt, 1), LM_TPB);
  const bool par = S->forked && !c->prof_on;
  cudaStream_t s0 = c->stream, s1 = par ? c->side[0] : c->stream, s2 = par ? c->side[1] : c->stream;
  auto fork = [&](cudaStream_t t) -> cudaError_t { return par ? cudaStreamWaitEvent(t, c->ev_fork, 0) : cudaSuccess; };
  auto join = [&](int i) -> cudaError_t {
    if (!par) return cudaSuccess;
    cudaError_t e = cudaEventRecord(c->ev_join[i], c->side[i]);
    return e != cudaSuccess ? e : cudaStreamWaitEvent(s0, c->ev_join[i], 0);
  };
  if (par) LLD_CUDA(c, cudaEventRecord(c->ev_fork, s0));
  LLD_CUDA(c, fork(s1));
  LLD_CUDA(c, fork(s2));
  const int nip = v.n_items_pt, nil = v.n_items - v.n_items_pt;
  if (v.n_pt && v.n_pt <= PT_WIDE_MAX) LLD_LAUNCH_S(c, s0, (k_lin_points<4, true>), cdiv(v.n_pt * 4, LM_TPB), LM_TPB, 0, v);
  else if (v.n_pt) LLD_LAUNCH_S(c, s0, (k_lin_points<1, true>), gp, LM_TPB, 0, v);
  if (nip) LLD_LAUNCH_S(c, s0, k_schur_tile<3>, std::min(nip, 4 * c->sm_count), SP_TPB, SP_SMEM_BYTES, v, 0, nip);
  { int r = launch_line_kernel(c, s1, v, true, true); if (r) return r; }
  if (nil) LLD_LAUNCH_S(c, s1, k_schur_tile<4>, std::min(nil, 4 * c->sm_count), SP_TPB, SP_SMEM_BYTES, v, nip, nil);
  if (v.n_chunks) LLD_LAUNCH_S(c, s2, k_lin_poses, v.n_chunks, LM_TPB, 0, v);
  if (v.n_free_total) LLD_LAUNCH_S(c, s2, k_pose_sum, cdiv(28 * v.n_free_total, 128), 128, 0, v);
  LLD_CUDA(c, join(0));
  LLD_CUDA(c, join(1));
  const int nblk = (int)S->n_nb_total;
  if (S->gather_long) LLD_LAUNCH_S(c, s0, k_reduce_piece_warp, cdiv(nblk * 6 + v.n_free_total, 8), 256, 0, v, nblk);
  else LLD_LAUNCH_S(c, s0, k_reduce_piece, cdiv(nblk * 36 + 6 * v.n_free_total, 256), 256, 0, v, nblk);
  { int r = launch_solve<true>(c, v, S->max_n); if (r) return r; }
  if (par) LLD_CUDA(c, cudaEventRecord(c->ev_fork, s0));
  LLD_CUDA(c, fork(s1));
  if (v.n_pt && v.n_pt <= PT_WIDE_MAX) LLD_LAUNCH_S(c, s0, k_backsub_points<4>, cdiv(v.n_pt * 4, LM_TPB), LM_TPB, 0, v);
  else if (v.n_pt) LLD_LAUNCH_S(c, s0, k_backsub_points<1>, gp, LM_TPB, 0, v);
  { int r = launch_line_kernel(c, s1, v, false); if (r) return r; }
  LLD_CUDA(c, join(0));
  LLD_LAUNCH_S(c, s0, k_decide_carry, v.n_win, FUSED_RED_TPB, 0, v, round, stop_now);
  LLD_CUDA(c, cudaGetLastError());
  return LLD_OK;
}

// one LM step of every window still running; first = first step of the round (every window at iteration 0).
// A dense single-rank batch (S->forked) runs the independent passes of the step on concurrent streams:
//   [lin_points | lin_lines | lin_poses] -> begin -> [schur_points -> schur_tile<3> | schur_lines -> schur_tile<4>] ->
//   reduce -> solve -> [backsub_points | backsub_lines] -> decide
// (a small batch does not fill the GPU with any single pass; the critical path is what counts).  Works eagerly and
// under stream capture (the side streams join the capture through the fork event).  Otherwise, and in profiled runs, the
// same launches go in the same order on one stream.
static int ba_step(LldCtx* c, int round, int stop_now, bool first = true) {
  BaState* S = c->ba;
  BaView& v = S->v;
  if (S->lean && !first) return ba_step_lean(c, round, stop_now);
  const int gp = cdiv(std::max(v.n_pt, 1), LM_TPB), gl = cdiv(std::max(v.n_ln, 1), LM_TPB);
  const bool par = S->forked && !c->prof_on;
  cudaStream_t s0 = c->stream, s1 = par ? c->side[0] : c->stream, s2 = par ? c->side[1] : c->stream;
  auto fork = [&](cudaStream_t t) -> cudaError_t { return par ? cudaStreamWaitEvent(t, c->ev_fork, 0) : cudaSuccess; };
  auto join = [&](int i) -> cudaError_t {
    if (!par) return cudaSuccess;
    cudaError_t e = cudaEventRecord(c->ev_join[i], c->side[i]);
    return e != cudaSuccess ? e : cudaStreamWaitEvent(s0, c->ev_join[i], 0);
  };
  if (par) LLD_CUDA(c, cudaEventRecord(c->ev_fork, s0));
  LLD_CUDA(c, fork(s1));
  LLD_CUDA(c, fork(s2));
  if (v.n_pt && v.n_pt <= PT_WIDE_MAX) LLD_LAUNCH_S(c, s0, k_lin_points<4>, cdiv(v.n_pt * 4, LM_TPB), LM_TPB, 0, v);
  else if (v.n_pt) LLD_LAUNCH_S(c, s0, k_lin_points<1>, gp, LM_TPB, 0, v);
  { int r = launch_line_kernel(c, s1, v, true); if (r) return r; }
  if (v.n_chunks) LLD_LAUNCH_S(c, s2, k_lin_poses, v.n_chunks, LM_TPB, 0, v);
  LLD_CUDA(c, join(0));
  LLD_CUDA(c, join(1));
  const bool multi = S->global_mode && c->n_ranks > 1;
  const bool fused = !multi && v.n_slices == 1;
  if (fused) {
    LLD_LAUNCH(c, k_begin_fused, v.n_win, FUSED_RED_TPB, 0, v);
  } else {
    if (v.n_free_total) LLD_LAUNCH(c, k_reduce_pose, cdiv(v.n_free_total * 28, 128), 128, 0, v);
    LLD_LAUNCH(c, k_reduce_lin, v.n_win * v.n_slices, 256, 0, v);
    LLD_LAUNCH(c, k_sum_lin, cdiv(v.n_win, 64), 64, 0, v);
    if (multi) { int r = ba_allreduce_lin(c); if (r) return r; }
    LLD_LAUNCH(c, k_begin, cdiv(v.n_win, 64), 64, 0, v);
  }
  const int nip = v.n_items_pt, nil = v.n_items - v.n_items_pt;   // dense-mode work items (none in sparse mode)
  if (par) LLD_CUDA(c, cudaEventRecord(c->ev_fork, s0));
  LLD_CUDA(c, fork(s1));
  if (v.n_pt) LLD_LAUNCH_S(c, s0, k_schur_points, gp, LM_TPB, 0, v);
  if (nip) LLD_LAUNCH_S(c, s0, k_schur_tile<3>, std::min(nip, 4 * c->sm_count), SP_TPB, SP_SMEM_BYTES, v, 0, nip);
  if (v.n_ln) LLD_LAUNCH_S(c, s1, k_schur_lines, gl, LM_TPB, 0, v);
  if (nil) LLD_LAUNCH_S(c, s1, k_schur_tile<4>, std::min(nil, 4 * c->sm_count), SP_TPB, SP_SMEM_BYTES, v, nip, nil);
  LLD_CUDA(c, join(0));
  if (v.dense_mode) {
    const int nblk = (int)S->n_nb_total;
    if (S->gather_long) LLD_LAUNCH(c, k_reduce_piece_warp, cdiv(nblk * 6 + v.n_free_total, 8), 256, 0, v, nblk);
    else LLD_LAUNCH(c, k_reduce_piece, cdiv(nblk * 36 + 6 * v.n_free_total, 256), 256, 0, v, nblk);
  } else {
    if (v.n_fold) LLD_LAUNCH(c, k_fold_dup, cdiv(v.n_fold, 128), 128, 0, v);
    const int tpb = 32 * cdiv(6 * S->max_nnb, 32);
    const int nl = v.n_chunks - v.n_chunks_pt;
    if (tpb <= 256) {
      if (v.n_chunks_pt) LLD_LAUNCH(c, (k_schur_rows<3, 256>), v.n_chunks_pt, tpb, 0, v, 0);
      if (nl) LLD_LAUNCH(c, (k_schur_rows<4, 256>), nl, tpb, 0, v, v.n_chunks_pt);
    } else {
      if (v.n_chunks_pt) LLD_LAUNCH(c, (k_schur_rows<3, 1024>), v.n_chunks_pt, tpb, 0, v, 0);
      if (nl) LLD_LAUNCH(c, (k_schur_rows<4, 1024>), nl, tpb, 0, v, v.n_chunks_pt);
    }
    if (v.n_free_total) {
      const int tpb2 = std::min(256, 32 * cdiv(6 * S->max_nnb, 32));
      LLD_LAUNCH(c, k_reduce_rows, v.n_free_total, tpb2, 0, v, (S->global_mode && c->n_ranks > 1 && c->rank != 0) ? 0 : 1);
    }
  }
  if (S->global_mode) { int r = ba_allreduce_rows(c); if (r) return r; }
  if (v.env_mode && S->use_cr) {
    int r = ba_solve_cr(c);
    if (r) return r;
  } else if (v.env_mode && S->use_sp) {
    int r = ba_solve_sp(c);
    if (r) return r;
  } else if (v.env_mode) {
    LLD_LAUNCH(c, k_solve_env, 1, 1024, S->env_smem, v);
  } else if (S->max_n <= SMEM_SOLVE_MAX_N) { int r = launch_solve<true>(c, v, S->max_n); if (r) return r; }
  else { int r = launch_solve<false>(c, v, S->max_n); if (r) return r; }
  if (par) LLD_CUDA(c, cudaEventRecord(c->ev_fork, s0));
  LLD_CUDA(c, fork(s1));
  if (v.n_pt && v.n_pt <= PT_WIDE_MAX) LLD_LAUNCH_S(c, s0, k_backsub_points<4>, cdiv(v.n_pt * 4, LM_TPB), LM_TPB, 0, v);
  else if (v.n_pt) LLD_LAUNCH_S(c, s0, k_backsub_points<1>, gp, LM_TPB, 0, v);
  { int r = launch_line_kernel(c, s1, v, false); if (r) return r; }
  LLD_CUDA(c, join(0));
  if (fused) {
    LLD_LAUNCH(c, k_decide_fused, v.n_win, FUSED_RED_TPB, 0, v, round, stop_now);
  } else {
    LLD_LAUNCH(c, k_reduce_trial, v.n_win * v.n_slices, 256, 0, v);
    LLD_LAUNCH(c, k_sum_trial, cdiv(v.n_win, 64), 64, 0, v);
    if (multi) { int r = ba_allreduce_trial(c); if (r) return r; }
    LLD_LAUNCH(c, k_decide, cdiv(v.n_win, 64), 64, 0, v, round, stop_now);
  }
  LLD_CUDA(c, cudaGetLastError());
  return LLD_OK;
}

// optimize(maxit) for the whole batch (SparseOptimizer::optimize, sparse_optimizer.cpp:354-419).
// LM steps are enqueued in groups of two with at most two groups in flight: before group k + 2 is enqueued the host waits
// for group k, reads the number of windows still running and polls pbStopFlag — the reference polls it between LM
// iterations and trials (sparse_optimizer.cpp:376, optimization_algorithm_levenberg.cpp:149); here a flag set mid-run is
// seen within two groups.  A set flag enqueues one last step with stop_now (every window finishes its current iteration
// and terminates).  Multi-rank: the ranks agree on the flag through an all-reduce(max), so that all of them issue the same
// collectives.
static int ba_run_round(LldCtx* c, int maxit, int round, const volatile uint8_t* stop) {
  BaState* S = c->ba;
  BaView& v = S->v;
  LLD_LAUNCH(c, k_round_init, cdiv(v.n_win, 64), 64, 0, v, maxit, round);
  if (maxit <= 0) return LLD_OK;
  int* h_active = reinterpret_cast<int*>(c->pinned);        // [2] one per group slot, [2] = stop agreement word
  const bool multi = S->global_mode && c->n_ranks > 1;
  const int hard_cap = maxit * 10 + 4;
  static const int group_len = getenv("LLD_BA_GROUP") ? std::max(1, atoi(getenv("LLD_BA_GROUP"))) : 2;
  int launched = 0;
  auto one_step = [&](int stop_now) -> int {
    const bool first = launched == 0;
    const int kind = (S->lean && !first) ? 1 : 0;
    if (S->use_graph && !c->prof_on && !stop_now && round < 2) {
      if (!S->graph_fresh[round][kind]) {  // capture one LM step (fork / join over the side streams included)
        const int64_t l0 = c->launches;
        cudaGraph_t g = nullptr;
        std::lock_guard<std::mutex> lk(lld_capture_mutex());  // no allocation in any thread while this one captures
        LLD_CUDA(c, cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
        int r = ba_step(c, round, 0, first);
        cudaError_t e = cudaStreamEndCapture(c->stream, &g);
        if (r) { if (g) cudaGraphDestroy(g); return r; }
        LLD_CUDA(c, e);
        // a new problem on a context that already ran one: same node topology, new kernel arguments -> update in place
        bool updated = false;
        if (c->ba_graph[round][kind]) {
          cudaGraphExecUpdateResultInfo info;
          if (cudaGraphExecUpdate(c->ba_graph[round][kind], g, &info) == cudaSuccess) updated = true;
          else {
            cudaGetLastError();
            cudaGraphExecDestroy(c->ba_graph[round][kind]);
            c->ba_graph[round][kind] = nullptr;
          }
        }
        if (!updated) e = cudaGraphInstantiate(&c->ba_graph[round][kind], g, 0);
        cudaGraphDestroy(g);
        LLD_CUDA(c, e);
        c->ba_graph_kernels[round][kind] = (int)(c->launches - l0);
        c->launches = l0;
        S->graph_fresh[round][kind] = true;
      }
      {
        std::lock_guard<std::mutex> lk(lld_capture_mutex());  // graph launches and captures of other threads do not interleave
        LLD_CUDA(c, cudaGraphLaunch(c->ba_graph[round][kind], c->stream));
      }
      c->launches += c->ba_graph_kernels[round][kind];
      return LLD_OK;
    }
    return ba_step(c, round, stop_now, first);
  };
  for (int k = 0;; k++) {
    const int slot = k & 1;
    if (k >= 2) {   // group k - 2 has finished: anything left to do?
      LLD_CUDA(c, cudaEventSynchronize(c->ev_grp[slot]));
      if (h_active[slot] <= 0) break;
    }
    int stop_now = (stop && *stop) ? 1 : 0;
#ifdef LLD_WITH_NCCL
    if (multi && stop) {   // collective decision (device word, max over ranks)
      h_active[2] = stop_now;
      LLD_CUDA(c, cudaMemcpyAsync(v.n_active_win + 1, &h_active[2], sizeof(int), cudaMemcpyHostToDevice, c->stream));
      LLD_NCCL(c, ncclAllReduce(v.n_active_win + 1, v.n_active_win + 1, 1, ncclInt, ncclMax, reinterpret_cast<ncclComm_t>(c->comm), c->stream));
      LLD_CUDA(c, cudaMemcpyAsync(&h_active[2], v.n_active_win + 1, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
      LLD_CUDA(c, cudaStreamSynchronize(c->stream));
      stop_now = h_active[2];
    }
#endif
    const int n = stop_now ? 1 : group_len;
    for (int s2 = 0; s2 < n; s2++) {
      int r = one_step(stop_now);
      if (r) return r;
      launched++;
    }
    LLD_CUDA(c, cudaMemcpyAsync(&h_active[slot], v.n_active_win, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    LLD_CUDA(c, cudaEventRecord(c->ev_grp[slot], c->stream));
    if (stop_now) break;
    if (launched >= hard_cap + 2 * group_len) {
      LLD_CUDA(c, cudaStreamSynchronize(c->stream));
      snprintf(c->err, sizeof(c->err), "LM step budget exhausted (%d steps, %d windows still active)", launched, h_active[slot]);
      return LLD_ERR_CUDA;
    }
  }
  LLD_CUDA(c, cudaStreamSynchronize(c->stream));
  return LLD_OK;
}

static int ba_download(LldCtx* c, const lld_ba_problem* p, lld_ba_result* out, bool local) {
  BaState* S = c->ba;
  BaView& v = S->v;
  const int n = std::max({v.n_kf, v.n_pt, v.n_ln, 1});
  if (local) {
    if (v.n_pe) LLD_LAUNCH(c, k_flag_points, cdiv(v.n_pe, 256), 256, 0, v, S->d_pt_bad);
    if (v.n_ln) LLD_LAUNCH(c, k_final_lines, cdiv(v.n_ln, 128), 128, 0, v, S->d_ln_bad);
  }
  LLD_LAUNCH(c, k_export, cdiv(n, 256), 256, 0, v, S->d_out_kf, S->d_out_pt, S->d_out_ln, S->d_ln_in);
  LLD_CUDA(c, cudaGetLastError());
  LLD_CUDA(c, cudaEventRecord(c->ev[2], c->stream));
  auto D2H = [&](void* dst, const void* src, size_t bytes) -> cudaError_t {
    if (!dst || !bytes) return cudaSuccess;
    return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream);
  };
  LLD_CUDA(c, D2H(out->kf_Tcw, S->d_out_kf, sizeof(double) * 12 * (size_t)v.n_kf));
  LLD_CUDA(c, D2H(out->pt_xyz, S->d_out_pt, sizeof(double) * 3 * (size_t)v.n_pt));
  LLD_CUDA(c, D2H(out->ln_x0_dir, S->d_out_ln, sizeof(double) * 6 * (size_t)v.n_ln));
  LLD_CUDA(c, D2H(out->pt_obs_bad, S->d_pt_bad, (size_t)v.n_pe));
  LLD_CUDA(c, D2H(out->ln_obs_bad, S->d_ln_bad, 2 * (size_t)v.n_lc));
  LLD_CUDA(c, D2H(out->ln_removed, v.ln_removed, (size_t)v.n_ln));
  const int ls = std::min(out->log_stride, v.log_stride);
  if (out->log_stride == v.log_stride) {
    LLD_CUDA(c, D2H(out->chi2_log, v.chi2_log, sizeof(double) * (size_t)v.n_win * ls));
    LLD_CUDA(c, D2H(out->lambda_log, v.lambda_log, sizeof(double) * (size_t)v.n_win * ls));
    LLD_CUDA(c, D2H(out->trials_log, v.trials_log, sizeof(int) * (size_t)v.n_win * ls));
  }
  LLD_CUDA(c, D2H(out->n_iter_done, v.iter_done, sizeof(int) * 2 * (size_t)v.n_win));
  LLD_CUDA(c, cudaEventRecord(c->ev[3], c->stream));
  LLD_CUDA(c, cudaStreamSynchronize(c->stream));
  cudaEventElapsedTime(&c->ms_h2d, c->ev[0], c->ev[1]);
  cudaEventElapsedTime(&c->ms_compute, c->ev[1], c->ev[2]);
  cudaEventElapsedTime(&c->ms_d2h, c->ev[2], c->ev[3]);
  c->last_d2h_bytes = sizeof(double) * (12 * (size_t)v.n_kf + 3 * (size_t)v.n_pt + 6 * (size_t)v.n_ln) + (size_t)v.n_pe +
                      2 * (size_t)v.n_lc + (size_t)v.n_ln + (sizeof(double) * 2 + sizeof(int)) * (size_t)v.n_win * ls +
                      sizeof(int) * 2 * (size_t)v.n_win;
  (void)p;
  return LLD_OK;
}

// ---- resident-mode entry points (bench: inputs already in HBM) ---------------------------------------------
extern "C" int lld_ba_upload(void* ctx, const lld_ba_problem* p, int global_mode, int log_stride) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !p) return LLD_ERR_ARG;
  LLD_CUDA(c, cudaSetDevice(c->device));
  LLD_CUDA(c, cudaEventRecord(c->ev[0], c->stream));
  int r = ba_upload(c, p, global_mode != 0, log_stride);
  if (r) return r;
  LLD_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
  LLD_CUDA(c, cudaStreamSynchronize(c->stream));
  return LLD_OK;
}

// (re)initialise the device state from the uploaded inputs and run; round-2 parameters as in lld_ba_local.
// the uploaded problem lives in the context's pooled buffers: any other entry point on the same context recycles them
static int ba_state_valid(LldCtx* c) {
  if (c->ba->pool_gen != c->pool_gen) {
    snprintf(c->err, sizeof(c->err), "the uploaded BA problem was invalidated by another call on this context (upload again)");
    return LLD_ERR_ARG;
  }
  return LLD_OK;
}

extern "C" int lld_ba_run_local(void* ctx, int its1, int its2, const volatile uint8_t* stop) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !c->ba) return LLD_ERR_ARG;
  { int r0 = ba_state_valid(c); if (r0) return r0; }
  LLD_CUDA(c, cudaSetDevice(c->device));
  BaState* S = c->ba;
  BaView& v = S->v;
  int r = ba_init_state(c);
  if (r) return r;
  if (stop && *stop) {  // src/Optimizer.cc:1220-1222
    LLD_LAUNCH(c, k_round_init, cdiv(v.n_win, 64), 64, 0, v, 0, 0);
    return LLD_OK;
  }
  const int rp = v.prm.robust_pt;
  v.prm.robust_ln = 1;
  r = ba_run_round(c, its1, 0, stop);
  if (r) return r;
  if (!(stop && *stop)) {  // bDoMore, src/Optimizer.cc:1230-1236
    if (v.n_pe) LLD_LAUNCH(c, k_flag_points, cdiv(v.n_pe, 256), 256, 0, v, (uint8_t*)nullptr);
    if (v.n_ln) LLD_LAUNCH(c, k_flag_lines, cdiv(v.n_ln, 128), 128, 0, v);
    v.prm.robust_pt = 0;
    v.prm.robust_ln = 0;
    r = ba_run_round(c, its2, 1, stop);
    v.prm.robust_pt = rp;
    v.prm.robust_ln = 1;
    if (r) return r;
  }
  return LLD_OK;
}

extern "C" int lld_ba_run_global(void* ctx, int n_iter, const volatile uint8_t* stop) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !c->ba) return LLD_ERR_ARG;
  { int r0 = ba_state_valid(c); if (r0) return r0; }
  LLD_CUDA(c, cudaSetDevice(c->device));
  c->nccl_calls = 0; c->nccl_bytes = 0;
  int r = ba_init_state(c);
  if (r) return r;
  c->ba->v.prm.robust_ln = 1;
  return ba_run_round(c, n_iter, 0, stop);
}

extern "C" int lld_ba_sync(void* ctx) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c) return LLD_ERR_ARG;
  LLD_CUDA(c, cudaStreamSynchronize(c->stream));
  return LLD_OK;
}

extern "C" int lld_ba_download(void* ctx, const lld_ba_problem* p, lld_ba_result* out, int local) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !c->ba || !out) return LLD_ERR_ARG;
  { int r0 = ba_state_valid(c); if (r0) return r0; }
  return ba_download(c, p, out, local != 0);
}

// ---- reference-shaped entry points -------------------------------------------------------------------------
static int ba_local_single(LldCtx* c, const lld_ba_problem* p, int its1, int its2, const volatile uint8_t* stop, lld_ba_result* out) {
  c->launches = 0;
  int r = lld_ba_upload(c, p, 0, its1 + its2 + 2);
  if (r) return r;
  LLD_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
  r = lld_ba_run_local(c, its1, its2, stop);
  if (r) return r;
  return ba_download(c, p, out, true);
}

// Windows are independent, so a large batch is cut into sub-batches that two worker threads (each with its own child
// context = stream + workspace) push through index -> upload -> LM -> download out of phase: while the GPU runs the LM
// steps of one sub-batch the host builds the index tables of the next.  Results are written into disjoint slices of
// the caller's arrays; every window computes exactly what it computes alone.
static int ba_local_pipelined(LldCtx* c, const lld_ba_problem* p, int its1, int its2, const volatile uint8_t* stop,
                              lld_ba_result* out, int n_sub) {
  const int nw = p->n_win, W = 2;
  for (int i = 0; i < W; i++)
    if (!c->child[i]) {
      void* h = nullptr;
      int r = lld_ctx_create(c->device, &h);
      if (r) { snprintf(c->err, sizeof(c->err), "pipelined local BA: child context %d failed", i); return r; }
      c->child[i] = lld_ctx_cast(h);
    }
  std::atomic<int> next{0}, rc{0};
  std::atomic<long long> launches{0}, h2d{0}, d2h{0};
  auto t0 = std::chrono::steady_clock::now();
  static const bool timing = getenv("LLD_TIMING") != nullptr;
  auto worker = [&](int wi) {
    LldCtx* cc = c->child[wi];
    cc->prof_on = false;
    cc->topo_cache = c->topo_cache;
    for (;;) {
      const int k = next.fetch_add(1);
      if (k >= n_sub || rc.load() != 0) break;
      const int w0 = (int)((long long)nw * k / n_sub), w1 = (int)((long long)nw * (k + 1) / n_sub), m = w1 - w0;
      if (m <= 0) continue;
      const int k0 = p->kf_off[w0], p0 = p->pt_off[w0], l0 = p->ln_off[w0];
      const int e0 = p->pt_obs_off[p0], c0 = p->ln_obs_off[l0];
      const int npt = p->pt_off[w1] - p0, nln = p->ln_off[w1] - l0;
      std::vector<int32_t> kfo(m + 1), pto(m + 1), lno(m + 1), peo(npt + 1), lco(nln + 1);
      for (int i = 0; i <= m; i++) { kfo[i] = p->kf_off[w0 + i] - k0; pto[i] = p->pt_off[w0 + i] - p0; lno[i] = p->ln_off[w0 + i] - l0; }
      for (int i = 0; i <= npt; i++) peo[i] = p->pt_obs_off[p0 + i] - e0;
      for (int i = 0; i <= nln; i++) lco[i] = p->ln_obs_off[l0 + i] - c0;
      lld_ba_problem sp = *p;
      sp.n_win = m; sp.kf_off = kfo.data(); sp.pt_off = pto.data(); sp.ln_off = lno.data();
      sp.kf_Tcw = p->kf_Tcw + 12 * (size_t)k0; sp.kf_fixed = p->kf_fixed + k0; sp.kf_intr = p->kf_intr + 5 * (size_t)k0;
      sp.kf_line_cam = p->kf_line_cam + 4 * (size_t)k0;
      sp.pt_xyz = p->pt_xyz + 3 * (size_t)p0; sp.pt_obs_off = peo.data(); sp.pt_obs_kf = p->pt_obs_kf + e0;
      sp.pt_obs_uvr = p->pt_obs_uvr + 3 * (size_t)e0; sp.pt_obs_info = p->pt_obs_info + e0;
      sp.ln_x0_dir = p->ln_x0_dir + 6 * (size_t)l0; sp.ln_obs_off = lco.data(); sp.ln_obs_kf = p->ln_obs_kf + c0;
      sp.ln_obs_left = p->ln_obs_left + 4 * (size_t)c0; sp.ln_obs_right = p->ln_obs_right + 4 * (size_t)c0;
      sp.ln_obs_info = p->ln_obs_info + 2 * (size_t)c0; sp.ln_obs_stereo = p->ln_obs_stereo + c0;
      lld_ba_result so = *out;
      so.kf_Tcw = out->kf_Tcw + 12 * (size_t)k0; so.pt_xyz = out->pt_xyz + 3 * (size_t)p0; so.ln_x0_dir = out->ln_x0_dir + 6 * (size_t)l0;
      so.pt_obs_bad = out->pt_obs_bad + e0; so.ln_obs_bad = out->ln_obs_bad + 2 * (size_t)c0; so.ln_removed = out->ln_removed + l0;
      const size_t ls = (size_t)out->log_stride;
      so.chi2_log = out->chi2_log ? out->chi2_log + ls * w0 : nullptr;
      so.lambda_log = out->lambda_log ? out->lambda_log + ls * w0 : nullptr;
      so.trials_log = out->trials_log ? out->trials_log + ls * w0 : nullptr;
      so.n_iter_done = out->n_iter_done ? out->n_iter_done + 2 * (size_t)w0 : nullptr;
      int r;
      if (timing) {  // LLD_TIMING: wall-clock timeline of the sub-batch relative to the call
        auto ms = [&]() { return std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count(); };
        const float ta = ms();
        cc->launches = 0;
        r = lld_ba_upload(cc, &sp, 0, its1 + its2 + 2);
        const float tb = ms();
        if (!r) r = cudaEventRecord(cc->ev[1], cc->stream) == cudaSuccess ? LLD_OK : LLD_ERR_CUDA;
        if (!r) r = lld_ba_run_local(cc, its1, its2, stop);
        const float tc = ms();
        if (!r) r = ba_download(cc, &sp, &so, true);
        const float td = ms();
        fprintf(stderr, "[lld_ba_local] worker %d sub-batch %d (%d windows): start %.2f  indexed+uploaded %.2f  LM done %.2f  downloaded %.2f ms\n",
                wi, k, m, ta, tb, tc, td);
      } else {
        r = ba_local_single(cc, &sp, its1, its2, stop, &so);
      }
      if (r) {
        int z = 0;
        if (rc.compare_exchange_strong(z, r)) snprintf(c->err, sizeof(c->err), "%s", cc->err);
        break;
      }
      launches += cc->launches;
      h2d += (long long)cc->last_h2d_bytes;
      d2h += (long long)cc->last_d2h_bytes;
    }
  };
  std::thread th(worker, 1);
  worker(0);
  th.join();
  c->launches = launches.load();
  c->last_h2d_bytes = (size_t)h2d.load();
  c->last_d2h_bytes = (size_t)d2h.load();
  c->ms_h2d = 0.f;
  c->ms_compute = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();  // wall: phases overlap
  c->ms_d2h = 0.f;
  return rc.load();
}

extern "C" int lld_ba_local(void* ctx, const lld_ba_problem* p, int its1, int its2, const volatile uint8_t* stop,
                            lld_ba_result* out) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !p || !out) return LLD_ERR_ARG;
  LLD_ARG(c, p->n_win >= 1);
  // two sub-batches from 16 windows up (measured: more sub-batches lose more GPU efficiency than the overlap wins);
  // LLD_BA_PIPE=<n> overrides, 0/1 disables
  int n_sub = p->n_win >= 16 ? 2 : 1;
  if (const char* e = getenv("LLD_BA_PIPE")) n_sub = std::min(atoi(e), p->n_win);
  if (n_sub >= 2 && !c->prof_on) return ba_local_pipelined(c, p, its1, its2, stop, out, n_sub);
  return ba_local_single(c, p, its1, its2, stop, out);
}

// host-side indexing only (no device needed): used to time / test the flattening stage on a CPU-only box.
// Returns LLD_ERR_CUDA when it reaches the first device allocation, which is the expected outcome without a GPU.
extern "C" int lld_ba_index_only(const lld_ba_problem* p, int global_mode) {
  static LldCtx c;  // keeps the host scratch across calls, like a real context (single-threaded helper)
  c.host_only = true;
  return ba_upload(&c, p, global_mode != 0, 8);
}

// the block-elimination plan lld_ba_global would run for p on a context with lld_ctx_set_gba_sparse(ctx, 1), as JSON
// (host arithmetic only, no device needed: used by the CPU-side tests).  A problem that another solver takes writes
// {"solver": "other"}; an error writes its message.
extern "C" int lld_gba_sparse_plan_report(const lld_ba_problem* p, char* buf, int len) {
  if (!p || !buf || len < 64) return LLD_ERR_ARG;
  LldCtx c;
  c.host_only = true;
  c.gba_sparse = 1;
  int r = ba_upload(&c, p, true, 8);
  std::string s = r ? std::string(c.err) : c.ba->use_sp ? c.ba->sp_report : std::string("{\"solver\":\"other\"}");
  lld_ba_state_free(c.ba);
  lld_ba_host_free(c.ba_host);
  c.ba = nullptr; c.ba_host = nullptr;
  if ((int)s.size() >= len) {
    snprintf(buf, (size_t)len, "report needs %zu bytes", s.size() + 1);
    return LLD_ERR_ARG;
  }
  memcpy(buf, s.c_str(), s.size() + 1);
  return r;
}

// landmark block partition of the multi-rank global BA (host arithmetic only; also used by the CPU-side tests)
extern "C" void lld_ba_shard_bounds(int32_t n_pt, int32_t n_ln, int32_t rank, int32_t n_ranks, int32_t out[4]) {
  out[0] = (int32_t)((long long)n_pt * rank / n_ranks);
  out[1] = (int32_t)((long long)n_pt * (rank + 1) / n_ranks);
  out[2] = (int32_t)((long long)n_ln * rank / n_ranks);
  out[3] = (int32_t)((long long)n_ln * (rank + 1) / n_ranks);
}

// Multi-rank global BA: the view of the caller's arrays that holds this rank's contiguous landmark block (re-based CSR
// offsets in poff / loff, which must outlive the upload) and the matching slices of the result arrays.
struct GbaShard {
  std::vector<int32_t> poff, loff;
  int32_t pto[2], lno[2];
  lld_ba_problem sh;
  lld_ba_result so;
  void make(const lld_ba_problem* p, const lld_ba_result* out, int rk, int R) {
    int32_t sb[4];
    lld_ba_shard_bounds(p->pt_off[1], p->ln_off[1], rk, R, sb);
    const int plo = sb[0], phi = sb[1], llo = sb[2], lhi = sb[3];
    const int pe0 = p->pt_obs_off[plo], lc0 = p->ln_obs_off[llo];
    poff.resize(phi - plo + 1); loff.resize(lhi - llo + 1);
    for (int i = 0; i <= phi - plo; i++) poff[i] = p->pt_obs_off[plo + i] - pe0;
    for (int i = 0; i <= lhi - llo; i++) loff[i] = p->ln_obs_off[llo + i] - lc0;
    pto[0] = 0; pto[1] = phi - plo; lno[0] = 0; lno[1] = lhi - llo;
    sh = *p;
    sh.pt_off = pto; sh.ln_off = lno;
    sh.pt_xyz = p->pt_xyz + 3 * (size_t)plo; sh.pt_obs_off = poff.data();
    sh.pt_obs_kf = p->pt_obs_kf + pe0; sh.pt_obs_uvr = p->pt_obs_uvr + 3 * (size_t)pe0; sh.pt_obs_info = p->pt_obs_info + pe0;
    sh.ln_x0_dir = p->ln_x0_dir + 6 * (size_t)llo; sh.ln_obs_off = loff.data();
    sh.ln_obs_kf = p->ln_obs_kf + lc0; sh.ln_obs_left = p->ln_obs_left + 4 * (size_t)lc0; sh.ln_obs_right = p->ln_obs_right + 4 * (size_t)lc0;
    sh.ln_obs_info = p->ln_obs_info + 2 * (size_t)lc0; sh.ln_obs_stereo = p->ln_obs_stereo + lc0;
    if (out) {
      so = *out;
      so.pt_xyz = out->pt_xyz + 3 * (size_t)plo; so.ln_x0_dir = out->ln_x0_dir + 6 * (size_t)llo;
      so.pt_obs_bad = out->pt_obs_bad + pe0; so.ln_obs_bad = out->ln_obs_bad + 2 * (size_t)lc0; so.ln_removed = out->ln_removed + llo;
    }
  }
};

// resident-mode upload of a global BA (bench: inputs already in HBM): single rank = lld_ba_upload(global_mode = 1); with a
// communicator every rank passes the whole problem and keeps its landmark block, exactly as lld_ba_global does
extern "C" int lld_ba_upload_global(void* ctx, const lld_ba_problem* p, int log_stride) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !p) return LLD_ERR_ARG;
  LLD_ARG(c, p->n_win == 1);
  LLD_CUDA(c, cudaSetDevice(c->device));
  c->nccl_calls = 0; c->nccl_bytes = 0;
  LLD_CUDA(c, cudaEventRecord(c->ev[0], c->stream));
  int r;
  if (c->n_ranks <= 1) {
    r = ba_upload(c, p, true, log_stride);
  } else {
    GbaShard G;
    G.make(p, nullptr, c->rank, c->n_ranks);
    r = ba_upload(c, &G.sh, true, log_stride, p);
    if (!r) LLD_CUDA(c, cudaStreamSynchronize(c->stream));   // the shard's offset arrays die with G
  }
  if (r) return r;
  LLD_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
  LLD_CUDA(c, cudaStreamSynchronize(c->stream));
  return LLD_OK;
}

extern "C" int lld_ba_global(void* ctx, const lld_ba_problem* p, int n_iter, const volatile uint8_t* stop,
                             lld_ba_result* out) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !p || !out) return LLD_ERR_ARG;
  LLD_ARG(c, p->n_win == 1);
  LLD_CUDA(c, cudaSetDevice(c->device));
  c->launches = 0;
  c->nccl_calls = 0; c->nccl_bytes = 0;
  const int R = c->n_ranks, rk = c->rank;
  if (R <= 1) {
    LLD_CUDA(c, cudaEventRecord(c->ev[0], c->stream));
    int r = ba_upload(c, p, true, n_iter + 2);
    if (r) return r;
    LLD_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
    r = lld_ba_run_global(ctx, n_iter, stop);
    if (r) return r;
    return ba_download(c, p, out, false);
  }
  // multi-rank: every rank receives the whole problem and keeps a contiguous block of the landmarks; keyframes are
  // replicated.  The shard is a view on the caller's arrays with re-based CSR offsets.
  GbaShard G;
  G.make(p, out, rk, R);
  LLD_CUDA(c, cudaEventRecord(c->ev[0], c->stream));
  int r = ba_upload(c, &G.sh, true, n_iter + 2, p);
  if (r) return r;
  LLD_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
  r = lld_ba_run_global(ctx, n_iter, stop);
  if (r) return r;
  return ba_download(c, &G.sh, &G.so, false);
}

void lld_ba_state_free(BaState* s) {
  if (s) s->drop_graphs();
  delete s;
}
