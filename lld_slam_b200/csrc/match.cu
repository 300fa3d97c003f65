// match.cu — 256-bit ORB Hamming matching: both Frame-level ORBmatcher::SearchByProjection variants, the keyframe searches
// (Fuse, SearchByProjection with Sim3) and ORBmatcher::SearchForInitialization (section at the end of the kernels).
//
// Reference: src/ORBmatcher.cc:45-129 (map points -> frame), :1328-1470 (last frame -> current frame),
// Frame::GetFeaturesInArea / AssignFeaturesToGrid (src/Frame.cc:294-309,391-456), DescriptorDistance (:1647-1663).
//
// Device plan per frame pair:
//   k_cell_count  : PosInGrid cell of every current keypoint, per-cell counts (integer atomics)
//   k_cell_scan   : exclusive scan of the 64x48 cell counts (one CTA per pair)
//   k_cell_fill   : keypoints re-ordered by cell into a packed, coalesced copy (xy, octave, uRight, descriptor)
//   k_match       : 8 lanes per query; the window's cell columns are contiguous ranges of the packed copy;
//                   uint4 descriptor loads + __popc; lexicographic (distance, grid order) top-2 so that ties
//                   resolve exactly like the reference's sequential scan (cell x outer, y inner, insertion order)
//   k_claim / k_match again: the reference lets an accepted match "claim" its keypoint for later queries
//                   (src/ORBmatcher.cc:87-89,1403-1405); we iterate the parallel matcher to the fixed point of that
//                   sequential rule (query i ignores keypoints owned by an accepted query j < i).
//   k_finalize    : rotation histogram + ComputeThreeMaxima (src/ORBmatcher.cc:1431-1466,1601-1642), match table.
// Float arithmetic is kept in float with explicit round-to-nearest intrinsics (no FMA contraction) wherever the
// reference computes in float; compile this unit with --fmad=false.
#include <algorithm>
#include <climits>
#include <cstdlib>

#include "lld_ctx.h"
#include "orb_common.cuh"

namespace {

constexpr int GRID_COLS = 64, GRID_ROWS = 48, N_CELLS = GRID_COLS * GRID_ROWS;
constexpr int TH_HIGH = 100, TH_LOW = 50;

struct MatchView {
  int n_pairs, n_cur, n_q;
  int variant;  // 0: frame-frame (best only), 1: map points (best / second best + ratio), 2: map points -> keyframe (Fuse / Sim3 search)
  // geometry
  float fx, fy, cx, cy, bf, b;
  float min_x, max_x, min_y, max_y, winv, hinv;
  int n_levels;
  const float* scale;
  float th, nn_ratio;
  int mono, check_ori;
  // current keypoints (input order)
  const int* cur_off;
  const float* cur_xy;
  const uint8_t* cur_octave;
  const float* cur_angle;
  const float* cur_uright;
  const uint8_t* cur_desc;
  const uint8_t* cur_claimed;
  // packed by cell
  int* cell_count;  // [n_pairs][N_CELLS+1] -> start offsets after the scan
  int* cell_fill;   // [n_pairs][N_CELLS]
  int* kp_cell;     // [n_cur] cell of each keypoint or -1
  uint4* s_rec;     // packed by cell, 48 B per keypoint: {x, y, uRight, meta} + 32 B descriptor, 16-byte aligned
                    // meta = idx (16) | cell (12) << 16 | octave (3) << 28 | claimed-on-entry << 31
  // queries
  const int* q_off;
  const uint8_t* q_valid;
  const float* q_xw;       // v0: world point ; v1: proj (u, v, uR)
  const uint8_t* q_octave; // v0
  const int* q_level;      // v1
  const float* q_viewcos;  // v1
  const float* q_angle;    // v0
  const uint8_t* q_desc;
  const uint8_t* q_has_obs;
  const float* cur_Tcw;    // v0 [n_pairs][12]
  const float* last_Tcw;
  // results / iteration state
  int* owner;      // [n_cur] smallest accepted query (with observations) that matched the keypoint; -1 = claimed on entry
  int* q_best;     // [n_q] matched keypoint (pair-local, original index) or -1
  int* q_dist;
  int* changed;    // [1]
  int* q_pair;     // [n_q] pair of the query
  int* pair_mode;  // [n_pairs] v0: 0 = levels [oct-1, oct+1], 1 = forward, 2 = backward
  unsigned long long* q_top;  // [n_q][4] four best candidates, packed (dist | cell | idx | octave), ascending
  int* q_ncand;    // [n_q] number of admissible candidates seen by the scan
  int* match;      // [n_cur]
  int* n_matches;  // [n_pairs]
  int th_high;         // acceptance threshold on the best distance (TH_HIGH, or ORBdist of the relocalisation variant)
  int allow_neg_z;     // no invzc < 0 rejection (relocalisation variant)
  int chi2_gate;       // variant 2: Fuse's reprojection gate (src/ORBmatcher.cc:905-925)
  float inv_sigma2[8]; // variant 2: mvInvLevelSigma2
  int max_cur, max_q;  // largest pair (host side dispatch)
  int fused_ok;
};

__device__ __forceinline__ int find_pair(const int* off, int n_pairs, int i) {
  int lo = 0, hi = n_pairs;  // largest p with off[p] <= i
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (off[mid] <= i) lo = mid;
    else hi = mid;
  }
  return lo;
}

// Frame::GetFeaturesInArea cell window  src/Frame.cc:396-410: columns [x0, x1], rows [y0, y1]; false when it misses the grid
struct CellWin { int x0, x1, y0, y1; };
__device__ __forceinline__ bool area_cells(const MatchView& v, float x, float y, float r, CellWin& c) {
  c.x0 = max(0, (int)floorf(__fmul_rn(__fsub_rn(__fsub_rn(x, v.min_x), r), v.winv)));
  c.x1 = min(GRID_COLS - 1, (int)ceilf(__fmul_rn(__fadd_rn(__fsub_rn(x, v.min_x), r), v.winv)));
  c.y0 = max(0, (int)floorf(__fmul_rn(__fsub_rn(__fsub_rn(y, v.min_y), r), v.hinv)));
  c.y1 = min(GRID_ROWS - 1, (int)ceilf(__fmul_rn(__fadd_rn(__fsub_rn(y, v.min_y), r), v.hinv)));
  return c.x0 < GRID_COLS && c.x1 >= 0 && c.y0 < GRID_ROWS && c.y1 >= 0;
}

__global__ void k_cell_count(MatchView v) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= v.n_cur) return;
  const int p = find_pair(v.cur_off, v.n_pairs, i);
  // Frame::PosInGrid  src/Frame.cc:446-456
  const float x = v.cur_xy[2 * (size_t)i], y = v.cur_xy[2 * (size_t)i + 1];
  const int px = (int)roundf(__fmul_rn(__fsub_rn(x, v.min_x), v.winv));
  const int py = (int)roundf(__fmul_rn(__fsub_rn(y, v.min_y), v.hinv));
  int cell = -1;
  if (!(px < 0 || px >= GRID_COLS || py < 0 || py >= GRID_ROWS)) {
    cell = px * GRID_ROWS + py;
    atomicAdd(&v.cell_count[(size_t)p * (N_CELLS + 1) + cell], 1);
  }
  v.kp_cell[i] = cell;
  v.owner[i] = v.cur_claimed[i] ? -1 : INT_MAX;
  v.match[i] = -1;
}

__global__ void __launch_bounds__(1024) k_cell_scan(MatchView v) {
  const int p = blockIdx.x;
  int* cnt = v.cell_count + (size_t)p * (N_CELLS + 1);
  __shared__ int part[1024];
  const int t = threadIdx.x;
  // 3 cells per thread
  const int c0 = cnt[3 * t], c1 = cnt[3 * t + 1], c2 = cnt[3 * t + 2];
  part[t] = c0 + c1 + c2;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {
    const int x = (t >= o) ? part[t - o] : 0;
    __syncthreads();
    part[t] += x;
    __syncthreads();
  }
  const int base = part[t] - (c0 + c1 + c2);
  cnt[3 * t] = base;
  cnt[3 * t + 1] = base + c0;
  cnt[3 * t + 2] = base + c0 + c1;
  if (t == 1023) cnt[N_CELLS] = part[t];
  v.cell_fill[(size_t)p * N_CELLS + 3 * t] = 0;
  v.cell_fill[(size_t)p * N_CELLS + 3 * t + 1] = 0;
  v.cell_fill[(size_t)p * N_CELLS + 3 * t + 2] = 0;
}

__global__ void k_cell_fill(MatchView v) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= v.n_cur) return;
  const int cell = v.kp_cell[i];
  if (cell < 0) return;
  const int p = find_pair(v.cur_off, v.n_pairs, i);
  const int slot = atomicAdd(&v.cell_fill[(size_t)p * N_CELLS + cell], 1);
  const size_t d = (size_t)v.cur_off[p] + v.cell_count[(size_t)p * (N_CELLS + 1) + cell] + slot;
  const unsigned meta = (unsigned)(i - v.cur_off[p]) | ((unsigned)cell << 16) | ((unsigned)(v.cur_octave[i] & 7) << 28) |
                        (v.cur_claimed[i] ? 0x80000000u : 0u);
  uint4 h;
  h.x = __float_as_uint(v.cur_xy[2 * (size_t)i]);
  h.y = __float_as_uint(v.cur_xy[2 * (size_t)i + 1]);
  h.z = __float_as_uint(v.cur_uright[i]);
  h.w = meta;
  const uint4* src = reinterpret_cast<const uint4*>(v.cur_desc + 32 * (size_t)i);
  v.s_rec[3 * d] = h;
  v.s_rec[3 * d + 1] = src[0];
  v.s_rec[3 * d + 2] = src[1];
}

// packed candidate key: lexicographic (distance, grid traversal order) == integer order
//   [dist:9 | cell:12 | idx:16 | octave:3]   (cell = ix*48+iy : x outer, y inner; idx = insertion order inside a cell)
constexpr unsigned long long EMPTY_KEY = ~0ull;
__device__ __forceinline__ unsigned long long pack_key(int d, int cell, int idx, int oct) {
  return ((unsigned long long)d << 31) | ((unsigned long long)cell << 19) | ((unsigned long long)idx << 3) | (unsigned long long)oct;
}
__device__ __forceinline__ int key_dist(unsigned long long k) { return (int)(k >> 31); }
__device__ __forceinline__ int key_idx(unsigned long long k) { return (int)((k >> 3) & 0xFFFFull); }
__device__ __forceinline__ int key_oct(unsigned long long k) { return (int)(k & 7ull); }

// cv::Mat (CV_32F) row of R*x + t : double accumulation, one rounding
__device__ __forceinline__ float gemm_row(const float* R, const float* x, float t) {
  const double s = __dadd_rn(__dadd_rn(__dmul_rn((double)R[0], (double)x[0]), __dmul_rn((double)R[1], (double)x[1])),
                             __dmul_rn((double)R[2], (double)x[2]));
  return (float)__dadd_rn(s, (double)t);
}

// per pair: forward / backward decision of the frame-to-frame variant (src/ORBmatcher.cc:1340-1350)
__device__ __forceinline__ int pair_mode_of(const MatchView& v, int p) {
  int mode = 0;
  {
    const float* Tc = v.cur_Tcw + 12 * (size_t)p;
    const float* Tl = v.last_Tcw + 12 * (size_t)p;
    float twc[3];
#pragma unroll
    for (int i = 0; i < 3; i++) {
      const double s = __dadd_rn(__dadd_rn(__dmul_rn((double)Tc[i], (double)Tc[9]), __dmul_rn((double)Tc[3 + i], (double)Tc[10])),
                                 __dmul_rn((double)Tc[6 + i], (double)Tc[11]));
      twc[i] = (float)(-s);
    }
    const float tlc2 = gemm_row(Tl + 6, twc, Tl[11]);
    const bool fwd = tlc2 > v.b && !v.mono;
    const bool bwd = -tlc2 > v.b && !v.mono;
    mode = fwd ? 1 : (bwd ? 2 : 0);
  }
  return mode;
}
__global__ void k_pair_prep(MatchView v) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= v.n_pairs) return;
  v.pair_mode[p] = v.variant == 0 ? pair_mode_of(v, p) : 0;
}
__global__ void k_query_pair(MatchView v) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= v.n_q) return;
  v.q_pair[q] = find_pair(v.q_off, v.n_pairs, q);
}

struct QueryWin {
  bool valid;
  float x, y, r, urq;
  int minLevel, maxLevel;
};
__device__ __forceinline__ QueryWin query_window(const MatchView& v, int q, int p, int mode) {
  QueryWin w;
  w.valid = v.q_valid[q] != 0;
  w.x = w.y = w.r = w.urq = 0.f;
  w.minLevel = w.maxLevel = -1;
  if (!w.valid) return w;
  if (v.variant == 0) {
    const float* Tc = v.cur_Tcw + 12 * (size_t)p;
    const float* Xw = v.q_xw + 3 * (size_t)q;
    const float xc = gemm_row(Tc, Xw, Tc[9]);
    const float yc = gemm_row(Tc + 3, Xw, Tc[10]);
    const float zc = gemm_row(Tc + 6, Xw, Tc[11]);
    const float invzc = (float)(1.0 / (double)zc);
    if (invzc < 0 && !v.allow_neg_z) w.valid = false;
    w.x = __fadd_rn(__fmul_rn(__fmul_rn(v.fx, xc), invzc), v.cx);
    w.y = __fadd_rn(__fmul_rn(__fmul_rn(v.fy, yc), invzc), v.cy);
    if (w.x < v.min_x || w.x > v.max_x) w.valid = false;
    if (w.y < v.min_y || w.y > v.max_y) w.valid = false;
    const int oct = v.q_octave[q];
    w.r = __fmul_rn(v.th, v.scale[oct]);
    w.urq = __fsub_rn(w.x, __fmul_rn(v.bf, invzc));
    if (mode == 1) { w.minLevel = oct; w.maxLevel = -1; }
    else if (mode == 2) { w.minLevel = 0; w.maxLevel = oct; }
    else { w.minLevel = oct - 1; w.maxLevel = oct + 1; }
  } else if (v.variant == 2) {   // Fuse / SearchByProjection(KeyFrame*, Scw, ...): radius = th * mvScaleFactors[nPredictedLevel]
    const float* pj = v.q_xw + 3 * (size_t)q;
    w.x = pj[0]; w.y = pj[1]; w.urq = pj[2];
    const int lvl = v.q_level[q];
    w.r = __fmul_rn(v.th, v.scale[lvl]);
    w.minLevel = lvl - 1; w.maxLevel = lvl;
  } else {
    const float* pj = v.q_xw + 3 * (size_t)q;
    w.x = pj[0]; w.y = pj[1]; w.urq = pj[2];
    const int lvl = v.q_level[q];
    float rr = ((double)v.q_viewcos[q] > 0.998) ? 2.5f : 4.0f;  // RadiusByViewingCos :131-137
    if (v.th != 1.0f) rr = __fmul_rn(rr, v.th);
    w.r = __fmul_rn(rr, v.scale[lvl]);
    w.minLevel = lvl - 1; w.maxLevel = lvl;
  }
  return w;
}

// Per-candidate test after the window test: stereo consistency of the Frame-level searches (|ur_q - ur| <= r when the keypoint
// has a right coordinate; src/ORBmatcher.cc:91-96,1407-1413), or, for the keyframe searches, Fuse's reprojection gate
// e2 * mvInvLevelSigma2[kpLevel] > 7.8 (mvuRight >= 0) / 5.99 (:905-925) -- float products, compared in double like the reference
template <int VARIANT = -1>   // -1: read the variant from the view (multi-kernel path)
__device__ __forceinline__ bool candidate_gate(const MatchView& v, const QueryWin& w, float dx, float dy, float ur, int oct) {
  if ((VARIANT >= 0 ? VARIANT : v.variant) != 2) return !(ur > 0 && fabsf(__fsub_rn(w.urq, ur)) > w.r);
  if (!v.chi2_gate) return true;
  const float exy = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
  if (ur >= 0) {
    const float er = __fsub_rn(w.urq, ur);
    return !((double)__fmul_rn(__fadd_rn(exy, __fmul_rn(er, er)), v.inv_sigma2[oct]) > 7.8);
  }
  return !((double)__fmul_rn(exy, v.inv_sigma2[oct]) > 5.99);
}

// Scan the window of one query (one thread).  excl_below >= 0: skip keypoints owned by a query < excl_below.
// Keeps the four smallest keys in t[0..3]; returns the number of admissible candidates.
__device__ __forceinline__ int scan_window(const MatchView& v, int q, int p, const QueryWin& w, int excl_below,
                                           unsigned long long* t) {
  t[0] = t[1] = t[2] = t[3] = EMPTY_KEY;
  if (!w.valid) return 0;
  CellWin cw;
  if (!area_cells(v, w.x, w.y, w.r, cw)) return 0;
  const int x0 = cw.x0, x1 = cw.x1, y0 = cw.y0, y1 = cw.y1;
  const bool check_levels = (w.minLevel > 0) || (w.maxLevel >= 0);
  const uint4* qd = reinterpret_cast<const uint4*>(v.q_desc + 32 * (size_t)q);
  const uint4 a0 = qd[0], a1 = qd[1];
  const int* cstart = v.cell_count + (size_t)p * (N_CELLS + 1);
  const size_t base = (size_t)v.cur_off[p];
  const int* own = v.owner + base;
  int ncand = 0;
  const uint4* rec = v.s_rec + 3 * base;
  for (int ix = x0; ix <= x1; ix++) {
    const int s0 = cstart[ix * GRID_ROWS + y0], s1 = cstart[ix * GRID_ROWS + y1 + 1];
#pragma unroll 2
    for (int s = s0; s < s1; s++) {
      const uint4 h = rec[3 * (size_t)s];
      const uint4 b0 = rec[3 * (size_t)s + 1], b1 = rec[3 * (size_t)s + 2];
      const unsigned meta = h.w;
      if (meta & 0x80000000u) continue;  // claimed on entry
      const int oct = (meta >> 28) & 7;
      if (check_levels) {
        if (oct < w.minLevel) continue;
        if (w.maxLevel >= 0 && oct > w.maxLevel) continue;
      }
      const float dx = __fsub_rn(__uint_as_float(h.x), w.x), dy = __fsub_rn(__uint_as_float(h.y), w.y);
      if (!(fabsf(dx) < w.r && fabsf(dy) < w.r)) continue;
      const int idx = meta & 0xFFFF;
      if (excl_below >= 0 && own[idx] < excl_below) continue;  // owned by an earlier accepted query
      const float ur = __uint_as_float(h.z);
      if (!candidate_gate(v, w, dx, dy, ur, oct)) continue;
      const int d = popc256(a0, a1, b0, b1);
      ncand++;
      unsigned long long k = pack_key(d, (meta >> 16) & 0xFFF, idx, oct);
      if (k < t[3]) {
        t[3] = k;
        if (t[3] < t[2]) { const unsigned long long u = t[2]; t[2] = t[3]; t[3] = u; }
        if (t[2] < t[1]) { const unsigned long long u = t[1]; t[1] = t[2]; t[2] = u; }
        if (t[1] < t[0]) { const unsigned long long u = t[0]; t[0] = t[1]; t[1] = u; }
      }
    }
  }
  return ncand;
}

// pass 0: one thread per query scans its window once and caches the four best candidates
__global__ void __launch_bounds__(128) k_match_scan(MatchView v) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= v.n_q) return;
  const int p = v.q_pair[q];
  const QueryWin w = query_window(v, q, p, v.variant == 0 ? v.pair_mode[p] : 0);
  unsigned long long t[4];
  const int n = scan_window(v, q, p, w, -1, t);
  ulonglong2* dst = reinterpret_cast<ulonglong2*>(v.q_top + 4 * (size_t)q);
  dst[0] = make_ulonglong2(t[0], t[1]);
  dst[1] = make_ulonglong2(t[2], t[3]);
  v.q_ncand[q] = n;
}

// resolution pass: best (and second best) candidate not owned by an earlier accepted query, from the cached top-4;
// a rescan is only needed when the cache is exhausted although more candidates exist
__global__ void __launch_bounds__(128) k_match_resolve(MatchView v, int pass) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= v.n_q) return;
  const int p = v.q_pair[q];
  const int qi = q - v.q_off[p];
  const int* own = v.owner + (size_t)v.cur_off[p];
  const ulonglong2* src = reinterpret_cast<const ulonglong2*>(v.q_top + 4 * (size_t)q);
  const ulonglong2 ta = src[0], tb = src[1];
  unsigned long long t[4] = {ta.x, ta.y, tb.x, tb.y};
  const int need = v.variant == 1 ? 2 : 1;
  unsigned long long k1 = EMPTY_KEY, k2 = EMPTY_KEY;
  int found = 0;
#pragma unroll
  for (int j = 0; j < 4; j++) {
    if (t[j] == EMPTY_KEY || found >= need) continue;
    if (own[key_idx(t[j])] < qi) continue;
    if (found == 0) k1 = t[j];
    else k2 = t[j];
    found++;
  }
  if (found < need && v.q_ncand[q] > 4) {  // cache exhausted: scan again with the exclusion applied
    const QueryWin w = query_window(v, q, p, v.variant == 0 ? v.pair_mode[p] : 0);
    scan_window(v, q, p, w, qi, t);
    k1 = t[0];
    k2 = t[1];
  }
  int best = -1, bdist = 256;
  if (k1 != EMPTY_KEY && key_dist(k1) <= v.th_high) {
    bool ok = true;
    if (v.variant == 1) {
      // ratio test only when best and second best share the level  (src/ORBmatcher.cc:118-121)
      const int d2 = k2 != EMPTY_KEY ? key_dist(k2) : 256;
      const int l2 = k2 != EMPTY_KEY ? key_oct(k2) : -1;
      if (key_oct(k1) == l2 && (float)key_dist(k1) > __fmul_rn(v.nn_ratio, (float)d2)) ok = false;
    }
    if (ok) { best = key_idx(k1); bdist = key_dist(k1); }
  }
  if (pass > 0 && v.q_best[q] != best) atomicOr(v.changed, 1);
  v.q_best[q] = best;
  v.q_dist[q] = bdist;
}

__global__ void k_owner_reset(MatchView v) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= v.n_cur) return;
  v.owner[i] = v.cur_claimed[i] ? -1 : INT_MAX;
  if (i == 0) *v.changed = 0;
}
__global__ void k_claim(MatchView v) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= v.n_q) return;
  const int b = v.q_best[q];
  if (b < 0 || !v.q_has_obs[q]) return;
  const int p = v.q_pair[q];
  atomicMin(&v.owner[(size_t)v.cur_off[p] + b], q - v.q_off[p]);
}

// per pair: match table, rotation-consistency filter, counts
__global__ void __launch_bounds__(256) k_finalize(MatchView v) {
  const int p = blockIdx.x;
  __shared__ int hist[HISTO_LENGTH];
  __shared__ int keep[3];
  __shared__ int cnt_acc, cnt_rej;
  const int q0 = v.q_off[p], q1 = v.q_off[p + 1];
  const size_t base = (size_t)v.cur_off[p];
  if (threadIdx.x < HISTO_LENGTH) hist[threadIdx.x] = 0;
  if (threadIdx.x == 0) { cnt_acc = 0; cnt_rej = 0; keep[0] = keep[1] = keep[2] = -1; }
  __syncthreads();
  const bool ori = v.variant == 0 && v.check_ori;
  for (int q = q0 + threadIdx.x; q < q1; q += blockDim.x) {
    const int b = v.q_best[q];
    if (b < 0) continue;
    atomicAdd(&cnt_acc, 1);
    atomicMax(&v.match[base + b], q - q0);
    if (ori) atomicAdd(&hist[rot_bin(v.q_angle[q], v.cur_angle[base + b])], 1);
  }
  __syncthreads();
  if (ori) {
    if (threadIdx.x == 0) three_maxima(hist, keep);
    __syncthreads();
    for (int q = q0 + threadIdx.x; q < q1; q += blockDim.x) {
      const int b = v.q_best[q];
      if (b < 0) continue;
      const int bin = rot_bin(v.q_angle[q], v.cur_angle[base + b]);
      if (bin != keep[0] && bin != keep[1] && bin != keep[2]) {
        v.match[base + b] = -1;  // runs after every atomicMax above (barrier) -> NULL wins, as in the reference
        atomicAdd(&cnt_rej, 1);
      }
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) v.n_matches[p] = cnt_acc - cnt_rej;
}


// ------------------------------------------------------------------------------------------------
// Fused matcher: ONE CTA per frame pair, the whole pair resident in shared memory.
//   build : PosInGrid counting sort of the current keypoints (smem integer atomics), slots inside a cell ordered by
//           keypoint index, so "slot order" == the reference's candidate traversal order (cell x outer, y inner,
//           insertion order); 16 B headers {x, y, uRight, owner:16 | octave | claimed} + 32 B descriptors in smem
//   scan  : one thread per query (<= FUSED_QPT queries per thread), candidates read from shared memory; the four best
//           candidates are kept in registers as 32-bit keys (distance << 16 | slot)
//   claim : the sequential "claimed keypoint" rule (src/ORBmatcher.cc:87-89,1403-1405) as a fixed point iterated inside
//           the CTA (owner = 16 high bits of the header word, smem atomicMin), no host round trips
//   final : rotation histogram + ComputeThreeMaxima, match table, counts
// HBM traffic = the pair's inputs once + the outputs: the SURVEY §8(d) algorithmic bytes.  Used when every pair fits
// (keypoints <= smem capacity, queries <= FUSED_QPT * FUSED_NT); larger frames take the multi-kernel path above.
// ------------------------------------------------------------------------------------------------
#ifndef LLD_MATCH_DBG
#define LLD_MATCH_DBG 0
#endif
constexpr int FUSED_NT = 512, FUSED_QPT = 4, FUSED_KPT = 4;  // <= 2048 queries and 2048 keypoints per pair
constexpr unsigned EMPTY32 = 0xFFFFFFFFu;

struct FusedLayout {
  int ncap;        // keypoint capacity (multiple of 8)
  int off_desc;    // byte offsets into dynamic shared memory
  int off_cstart;
  int off_sidx;
  int off_perm;
  int total;
};
static FusedLayout fused_layout(int max_cur) {
  FusedLayout L;
  L.ncap = std::max(8, (max_cur + 7) & ~7);
  L.off_desc = 16 * L.ncap;
  const int desc_bytes = std::max(32 * L.ncap, 4 * N_CELLS);   // the cell counters alias the descriptor area during the build
  L.off_cstart = L.off_desc + desc_bytes;
  L.off_sidx = L.off_cstart + ((2 * (N_CELLS + 2) + 15) & ~15);
  L.off_perm = L.off_sidx + ((2 * L.ncap + 15) & ~15);
  L.total = L.off_perm + 2 * FUSED_QPT * FUSED_NT;   // query permutation (sorted by octave), 16-bit
  return L;
}

// Scan the window of one query against the smem-resident pair; top-4 32-bit keys in t, #admissible candidates returned.
// The walk covers the cells of Frame::GetFeaturesInArea (src/Frame.cc:396-410) that can hold an admissible keypoint:
// PosInGrid (:446-456) is monotone in the coordinate, so the cells of (x -+ (r + margin)) bound every keypoint passing
// |dx| < r; this drops the outermost column / row that floor / ceil add (none of their keypoints can pass the test).
// The admission test is branch-free on one 16 B header; admitted slots go to a 4-deep pending list that is drained
// through the 256-bit popcount + top-4 insertion when full and once after the walk, where the lanes have reconverged.
template <int VARIANT>
__device__ __forceinline__ int fused_scan(const MatchView& v, const QueryWin& w, const uint4& a0, const uint4& a1,
                                          const uint4* __restrict__ hdr, const uint4* __restrict__ dsc,
                                          const unsigned short* __restrict__ cstart, int excl_below, unsigned* t) {
  t[0] = t[1] = t[2] = t[3] = EMPTY32;
  if (!w.valid) return 0;
  CellWin cw;
  if (!area_cells(v, w.x, w.y, w.r, cw)) return 0;
  int x0 = cw.x0, x1 = cw.x1, y0 = cw.y0, y1 = cw.y1;
  {
    const float m = w.r + 0.0625f;  // far above the rounding of the float subtraction in the admission test
    x0 = max(x0, (int)roundf(__fmul_rn(__fsub_rn(w.x - m, v.min_x), v.winv)));
    x1 = min(x1, (int)roundf(__fmul_rn(__fsub_rn(w.x + m, v.min_x), v.winv)));
    y0 = max(y0, (int)roundf(__fmul_rn(__fsub_rn(w.y - m, v.min_y), v.hinv)));
    y1 = min(y1, (int)roundf(__fmul_rn(__fsub_rn(w.y + m, v.min_y), v.hinv)));
  }
  const bool check_levels = (w.minLevel > 0) || (w.maxLevel >= 0);
  const int lvl_lo = check_levels ? w.minLevel : -1;
  const int lvl_hi = (check_levels && w.maxLevel >= 0) ? w.maxLevel : 8;
  const int excl = excl_below >= 0 ? excl_below : 0;  // owners are >= 0, so 0 excludes nothing
  unsigned long long pend = 0;
  int np = 0, ncand = 0;
  auto drain = [&]() {
#pragma unroll
    for (int j = 0; j < 4; j++) {
      if (j < np) {
        const int sl = (int)((pend >> (16 * j)) & 0xFFFFull);
        const int d = popc256(a0, a1, dsc[2 * sl], dsc[2 * sl + 1]);
        const unsigned k = ((unsigned)d << 16) | (unsigned)sl;
        if (k < t[3]) {
          t[3] = k;
          if (t[3] < t[2]) { const unsigned u = t[2]; t[2] = t[3]; t[3] = u; }
          if (t[2] < t[1]) { const unsigned u = t[1]; t[1] = t[2]; t[2] = u; }
          if (t[1] < t[0]) { const unsigned u = t[0]; t[0] = t[1]; t[1] = u; }
        }
      }
    }
    ncand += np;
    np = 0;
  };
  for (int ix = x0; ix <= x1; ix++) {
    const int s0 = cstart[ix * GRID_ROWS + y0], s1 = y1 >= y0 ? cstart[ix * GRID_ROWS + y1 + 1] : s0;
    for (int s = s0; s < s1; s++) {
      const uint4 h = hdr[s];
      const unsigned meta = h.w;
      const int oct = (meta >> 1) & 7;
      const float dx = __fsub_rn(__uint_as_float(h.x), w.x), dy = __fsub_rn(__uint_as_float(h.y), w.y);
      const float ur = __uint_as_float(h.z);
      bool ok = !(meta & 1u);                          // not claimed on entry
      ok = ok && oct >= lvl_lo && oct <= lvl_hi;       // level range (Frame::GetFeaturesInArea)
      ok = ok && fabsf(dx) < w.r && fabsf(dy) < w.r;
      ok = ok && (int)(meta >> 16) >= excl;            // not owned by an earlier accepted query
      ok = ok && candidate_gate<VARIANT>(v, w, dx, dy, ur, oct);   // stereo consistency / Fuse's reprojection gate
      if (ok) {
        if (np == 4) drain();
        pend = (pend << 16) | (unsigned long long)s;
        np++;
      }
    }
  }
  drain();
  return ncand;
}

template <int VARIANT>
__global__ void __launch_bounds__(FUSED_NT, 2) k_match_fused(MatchView v, FusedLayout L) {
  extern __shared__ uint4 fsm[];
  __shared__ int s_warp[FUSED_NT / 32];
  __shared__ int s_hist[HISTO_LENGTH];
  __shared__ int s_keep[3];
  __shared__ int s_acc, s_rej, s_mode;
  const int p = blockIdx.x, tid = threadIdx.x;
  const int c0 = v.cur_off[p], nc = v.cur_off[p + 1] - c0;
  const int q0 = v.q_off[p], nq = v.q_off[p + 1] - q0;
  uint4* hdr = fsm;
  uint4* dsc = reinterpret_cast<uint4*>(reinterpret_cast<char*>(fsm) + L.off_desc);
  int* cnt = reinterpret_cast<int*>(dsc);  // aliases the descriptor area until the records are loaded
  unsigned short* cstart = reinterpret_cast<unsigned short*>(reinterpret_cast<char*>(fsm) + L.off_cstart);
  unsigned short* sidx = reinterpret_cast<unsigned short*>(reinterpret_cast<char*>(fsm) + L.off_sidx);
  unsigned short* perm = reinterpret_cast<unsigned short*>(reinterpret_cast<char*>(fsm) + L.off_perm);
  unsigned* hdr_w = reinterpret_cast<unsigned*>(hdr);  // word 4*s+3 = meta of slot s
  const int lane = tid & 31, wid = tid >> 5;
  constexpr int NW = FUSED_NT / 32;

  // ---- issue the global loads of this CTA's keypoints (thread tid owns keypoints tid + u * FUSED_NT) and of the query
  // sort keys up front, so that their latency overlaps the ballot sort below
  float kx[FUSED_KPT], ky[FUSED_KPT], kur[FUSED_KPT];
  unsigned kmeta[FUSED_KPT];
#pragma unroll
  for (int u = 0; u < FUSED_KPT; u++) {
    const int i = tid + u * FUSED_NT;
    kx[u] = ky[u] = kur[u] = 0.f;
    kmeta[u] = 0;
    if (i < nc) {
      const size_t gi = (size_t)c0 + i;
      const float2 xy = reinterpret_cast<const float2*>(v.cur_xy)[gi];
      kx[u] = xy.x;
      ky[u] = xy.y;
      kur[u] = v.cur_uright[gi];
      kmeta[u] = 0xFFFF0000u | ((unsigned)(v.cur_octave[gi] & 7) << 1) | (v.cur_claimed[gi] ? 1u : 0u);
    }
  }
  int key[FUSED_QPT];
#pragma unroll
  for (int u = 0; u < FUSED_QPT; u++) {
    const int qi = tid + u * FUSED_NT;
    key[u] = 9;
    if (qi < nq) {
      const int q = q0 + qi;
      const int lv = VARIANT == 0 ? min((int)v.q_octave[q], 7) : min(max(v.q_level[q], 0), 7);
      key[u] = v.q_valid[q] ? lv : 8;
    }
  }
  if (tid < HISTO_LENGTH) s_hist[tid] = 0;
  if (tid == 0) {
    s_acc = 0; s_rej = 0;
    s_keep[0] = s_keep[1] = s_keep[2] = -1;
    s_mode = VARIANT == 0 ? pair_mode_of(v, p) : 0;
  }

  // ---- queries sorted by octave: the window radius is th * scale[octave], so the lanes of a warp then walk windows of
  // similar size (the claim order still uses the original query index).  Ballot counting sort, 9 buckets (8 = invalid).
  {
    int* wcnt = cnt;  // [9][FUSED_QPT * NW], scratch in the (still unused) descriptor area
    int rnk[FUSED_QPT];
#pragma unroll
    for (int u = 0; u < FUSED_QPT; u++) {
      rnk[u] = 0;
#pragma unroll
      for (int b = 0; b < 9; b++) {
        const unsigned m = __ballot_sync(0xffffffffu, key[u] == b);
        if (key[u] == b) rnk[u] = __popc(m & ((1u << lane) - 1u));
        if (lane == 0) wcnt[b * (FUSED_QPT * NW) + u * NW + wid] = __popc(m);
      }
    }
    __syncthreads();
    if (wid == 0) {  // exclusive prefix over the 9 * 64 (bucket-major) group counts
      constexpr int TOT = 9 * FUSED_QPT * NW, PER = TOT / 32;
      static_assert(PER * 32 == TOT, "group counts must divide over one warp");
      int loc[PER], sum = 0;
#pragma unroll
      for (int k = 0; k < PER; k++) { loc[k] = wcnt[PER * lane + k]; sum += loc[k]; }
      int incl = sum;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int x = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += x;
      }
      int base = incl - sum;
#pragma unroll
      for (int k = 0; k < PER; k++) { wcnt[PER * lane + k] = base; base += loc[k]; }
    }
    __syncthreads();
#pragma unroll
    for (int u = 0; u < FUSED_QPT; u++)
      if (key[u] <= 8) perm[wcnt[key[u] * (FUSED_QPT * NW) + u * NW + wid] + rnk[u]] = (unsigned short)(tid + u * FUSED_NT);
    __syncthreads();
  }

  // ---- build: count -> scan -> fill -> order inside cells -> inverse -> records written by the owning threads
  for (int i = tid; i < N_CELLS; i += FUSED_NT) cnt[i] = 0;
  __syncthreads();
  int kcell[FUSED_KPT];
#pragma unroll
  for (int u = 0; u < FUSED_KPT; u++) {
    const int i = tid + u * FUSED_NT;
    kcell[u] = -1;
    if (i < nc) {  // Frame::PosInGrid  src/Frame.cc:446-456
      const int px = (int)roundf(__fmul_rn(__fsub_rn(kx[u], v.min_x), v.winv));
      const int py = (int)roundf(__fmul_rn(__fsub_rn(ky[u], v.min_y), v.hinv));
      if (!(px < 0 || px >= GRID_COLS || py < 0 || py >= GRID_ROWS)) kcell[u] = px * GRID_ROWS + py;
      if (kcell[u] >= 0) atomicAdd(&cnt[kcell[u]], 1);
      v.match[(size_t)c0 + i] = -1;
    }
  }
  __syncthreads();
  {
    constexpr int PER = N_CELLS / FUSED_NT;  // 6 consecutive cells per thread
    static_assert(PER * FUSED_NT == N_CELLS, "cells must divide over the CTA");
    int loc[PER], sum = 0;
#pragma unroll
    for (int k = 0; k < PER; k++) { loc[k] = cnt[PER * tid + k]; sum += loc[k]; }
    int incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int x = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += x;
    }
    if (lane == 31) s_warp[wid] = incl;
    __syncthreads();
    if (wid == 0) {
      int x = lane < FUSED_NT / 32 ? s_warp[lane] : 0;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
      }
      if (lane < FUSED_NT / 32) s_warp[lane] = x;  // inclusive over warps
    }
    __syncthreads();
    int base = incl - sum + (wid ? s_warp[wid - 1] : 0);
#pragma unroll
    for (int k = 0; k < PER; k++) {
      cstart[PER * tid + k] = (unsigned short)base;
      cnt[PER * tid + k] = base;  // fill cursor
      base += loc[k];
    }
    if (tid == FUSED_NT - 1) cstart[N_CELLS] = (unsigned short)base;
  }
  __syncthreads();
#pragma unroll
  for (int u = 0; u < FUSED_KPT; u++)
    if (kcell[u] >= 0) sidx[atomicAdd(&cnt[kcell[u]], 1)] = (unsigned short)(tid + u * FUSED_NT);
  __syncthreads();
  for (int c = tid; c < N_CELLS; c += FUSED_NT) {  // insertion order inside a cell (cells hold ~1 keypoint)
    const int b = cstart[c], e = cstart[c + 1];
    for (int i = b + 1; i < e; i++) {
      const unsigned short x = sidx[i];
      int j = i - 1;
      while (j >= b && sidx[j] > x) { sidx[j + 1] = sidx[j]; j--; }
      sidx[j + 1] = x;
    }
  }
  __syncthreads();
  const int ntot = cstart[N_CELLS];
  {
    unsigned short* inv = reinterpret_cast<unsigned short*>(hdr);  // keypoint -> slot, consumed before the headers land
    for (int s2 = tid; s2 < ntot; s2 += FUSED_NT) inv[sidx[s2]] = (unsigned short)s2;
    __syncthreads();
    int kslot[FUSED_KPT];
#pragma unroll
    for (int u = 0; u < FUSED_KPT; u++) kslot[u] = kcell[u] >= 0 ? (int)inv[tid + u * FUSED_NT] : -1;
    __syncthreads();
#pragma unroll
    for (int u = 0; u < FUSED_KPT; u++) {
      if (kslot[u] < 0) continue;
      const uint4* src = reinterpret_cast<const uint4*>(v.cur_desc + 32 * ((size_t)c0 + tid + u * FUSED_NT));
      const uint4 d0 = src[0], d1 = src[1];
      hdr[kslot[u]] = make_uint4(__float_as_uint(kx[u]), __float_as_uint(ky[u]), __float_as_uint(kur[u]), kmeta[u]);
      dsc[2 * kslot[u]] = d0;
      dsc[2 * kslot[u] + 1] = d1;
    }
  }
  __syncthreads();

#if LLD_MATCH_DBG == 1   // timing experiment: loads, query sort and grid build only
  if (tid == 0) v.n_matches[p] = ntot;
  return;
#endif
  // ---- scan: top-4 per query in registers (thread tid, round u <-> sorted position tid + u * FUSED_NT)
  unsigned t[FUSED_QPT][4];
  unsigned many = 0, hasobs = 0;
  const int mode = s_mode;
#pragma unroll
  for (int u = 0; u < FUSED_QPT; u++) {
    const int sp = tid + u * FUSED_NT;
    QueryWin w;
    w.valid = false;
    w.x = w.y = w.r = w.urq = 0.f;
    w.minLevel = w.maxLevel = -1;
    uint4 a0 = make_uint4(0, 0, 0, 0), a1 = a0;
    if (sp < nq) {
      const int q = q0 + perm[sp];
      w = query_window(v, q, p, mode);
      const uint4* qd = reinterpret_cast<const uint4*>(v.q_desc + 32 * (size_t)q);
      a0 = qd[0];
      a1 = qd[1];
      if (v.q_has_obs[q]) hasobs |= 1u << u;
    }
    const int n = fused_scan<VARIANT>(v, w, a0, a1, hdr, dsc, cstart, -1, t[u]);
    if (n > 4) many |= 1u << u;
  }

#if LLD_MATCH_DBG == 2   // timing experiment: build + one scan of every window, no claim passes
  {
    unsigned acc = 0;
#pragma unroll
    for (int u = 0; u < FUSED_QPT; u++) acc += t[u][0] + t[u][1];
    if (acc == 0x12345678u) v.n_matches[p] = (int)acc;
    return;
  }
#endif
  // ---- claim fixed point
  unsigned bestkey[FUSED_QPT];
#pragma unroll
  for (int u = 0; u < FUSED_QPT; u++) bestkey[u] = EMPTY32;
  constexpr int need = VARIANT == 1 ? 2 : 1;
  auto decide = [&](unsigned k1, unsigned k2) -> unsigned {
    if (k1 == EMPTY32 || (int)(k1 >> 16) > v.th_high) return EMPTY32;
    if (VARIANT == 1) {  // ratio test only when best and second best share the level  (src/ORBmatcher.cc:118-121)
      const int d2 = k2 != EMPTY32 ? (int)(k2 >> 16) : 256;
      const int l1 = (hdr_w[4 * (k1 & 0xFFFFu) + 3] >> 1) & 7;
      const int l2 = k2 != EMPTY32 ? (int)((hdr_w[4 * (k2 & 0xFFFFu) + 3] >> 1) & 7) : -1;
      if (l1 == l2 && (float)(k1 >> 16) > __fmul_rn(v.nn_ratio, (float)d2)) return EMPTY32;
    }
    return k1;
  };
  for (int pass = 0;; pass++) {
    unsigned newkey[FUSED_QPT];
    unsigned resc = 0;
#pragma unroll
    for (int u = 0; u < FUSED_QPT; u++) {
      const int sp = tid + u * FUSED_NT;
      const int qi = sp < nq ? (int)perm[sp] : -1;
      unsigned k1 = EMPTY32, k2 = EMPTY32;
      int found = 0;
#pragma unroll
      for (int j = 0; j < 4; j++) {
        const unsigned k = t[u][j];
        if (qi < 0 || k == EMPTY32 || found >= need) continue;
        if ((int)(hdr_w[4 * (k & 0xFFFFu) + 3] >> 16) < qi) continue;
        if (found == 0) k1 = k;
        else k2 = k;
        found++;
      }
      newkey[u] = EMPTY32;
      if (qi >= 0 && found < need && ((many >> u) & 1u)) resc |= 1u << u;  // cache exhausted, more candidates exist
      else if (qi >= 0) newkey[u] = decide(k1, k2);
    }
    // rescans with the exclusion applied: warp-uniform calls, every lane works on its own pending query (if any)
    while (__any_sync(0xffffffffu, resc != 0)) {
      const int u = resc ? __ffs(resc) - 1 : -1;
      QueryWin w;
      w.valid = false;
      w.x = w.y = w.r = w.urq = 0.f;
      w.minLevel = w.maxLevel = -1;
      uint4 a0 = make_uint4(0, 0, 0, 0), a1 = a0;
      int qi = -1;
      if (u >= 0) {
        qi = perm[tid + u * FUSED_NT];
        const int q = q0 + qi;
        w = query_window(v, q, p, mode);
        const uint4* qd = reinterpret_cast<const uint4*>(v.q_desc + 32 * (size_t)q);
        a0 = qd[0];
        a1 = qd[1];
      }
      unsigned tt[4];
      fused_scan<VARIANT>(v, w, a0, a1, hdr, dsc, cstart, qi, tt);
      if (u >= 0) {
        const unsigned acc = decide(tt[0], tt[1]);
#pragma unroll
        for (int uu = 0; uu < FUSED_QPT; uu++)
          if (uu == u) newkey[uu] = acc;
        resc &= resc - 1;
      }
    }
    int changed = 0;
#pragma unroll
    for (int u = 0; u < FUSED_QPT; u++) {
      if (newkey[u] != bestkey[u]) changed = 1;
      bestkey[u] = newkey[u];
    }
    const int any = __syncthreads_or(changed);
    if (pass > 0 && !any) break;
    if (pass >= 64) {
      if (tid == 0) atomicOr(v.changed, 2);  // did not converge: reported by the host after the run
      break;
    }
    for (int s = tid; s < ntot; s += FUSED_NT) hdr_w[4 * s + 3] |= 0xFFFF0000u;
    __syncthreads();
#pragma unroll
    for (int u = 0; u < FUSED_QPT; u++) {
      const int sp = tid + u * FUSED_NT;
      if (sp < nq && bestkey[u] != EMPTY32 && ((hasobs >> u) & 1u)) {
        unsigned* wp = hdr_w + 4 * (bestkey[u] & 0xFFFFu) + 3;
        atomicMin(wp, ((unsigned)perm[sp] << 16) | (*wp & 0xFFFFu));
      }
    }
    __syncthreads();
  }

  // ---- results: per-query best, match table (last accepted query of a keypoint wins), rotation consistency
  const bool ori = VARIANT == 0 && v.check_ori;
  int bins[FUSED_QPT];
#pragma unroll
  for (int u = 0; u < FUSED_QPT; u++) {
    const int sp = tid + u * FUSED_NT;
    bins[u] = -1;
    if (sp >= nq) continue;
    const int qi = perm[sp];
    const int q = q0 + qi;
    int best = -1, bd = 256;
    if (bestkey[u] != EMPTY32) {
      best = sidx[bestkey[u] & 0xFFFFu];
      bd = (int)(bestkey[u] >> 16);
      atomicAdd(&s_acc, 1);
      atomicMax(&v.match[(size_t)c0 + best], qi);
      if (ori) {
        bins[u] = rot_bin(v.q_angle[q], v.cur_angle[(size_t)c0 + best]);
        atomicAdd(&s_hist[bins[u]], 1);
      }
    }
    v.q_best[q] = best;
    v.q_dist[q] = bd;
  }
  __syncthreads();
  if (ori) {
    if (tid == 0) three_maxima(s_hist, s_keep);
    __syncthreads();
#pragma unroll
    for (int u = 0; u < FUSED_QPT; u++) {
      if (bins[u] < 0) continue;
      if (bins[u] != s_keep[0] && bins[u] != s_keep[1] && bins[u] != s_keep[2]) {
        v.match[(size_t)c0 + sidx[bestkey[u] & 0xFFFFu]] = -1;  // after every atomicMax (barrier): NULL wins, as in the reference
        atomicAdd(&s_rej, 1);
      }
    }
    __syncthreads();
  }
  if (tid == 0) v.n_matches[p] = s_acc - s_rej;
}

// ------------------------------------------------------------------------------------------------
// ORBmatcher::SearchForInitialization (src/ORBmatcher.cc:405), batched over frame pairs (F1 = the initial frame,
// F2 = the current one).  F2's grid is built by k_cell_count / k_cell_scan / k_cell_fill above.
//   k_init_count    : one thread per level-0 F1 keypoint: the candidates of GetFeaturesInArea(vbPrevMatched[i1],
//                     windowSize, 0, 0) with dist <= keep_max, counted
//   k_init_scan     : per pair, exclusive scan of the counts -> CSR offsets of the candidate lists
//   k_init_fill     : the same walk again, packed keys (dist, cell, idx) written and sorted ascending per query
//   k_init_resolve_smem / k_init_resolve_global : one warp per pair walks the queries in index order (the reference's
//                     sequential loop); vMatchedDistance / vnMatches21 of F2 live in shared memory when the largest F2
//                     fits, else in global memory (owner / match of k_cell_count, initialised to INT_MAX / -1)
//   k_init_finalize : rotation histogram over every accepted match (displaced ones included), ComputeThreeMaxima,
//                     match counts and vbPrevMatched
// The sorted list makes the sequential rule cheap: the reference's best is the first candidate with
// vMatchedDistance[i2] > dist in (dist, traversal order) -- strict-< first minimum -- and bestDist2 is the distance of the
// next such candidate.  Candidates above keep_max never change the outcome: when the best is <= TH_LOW every bestDist2
// > keep_max passes the ratio test (host: smallest such bound), and a best above keep_max is above TH_LOW.
// ------------------------------------------------------------------------------------------------
constexpr int INIT_KBUF = 512;  // candidate keys of 32 queries staged in shared memory by the resolve warp

struct InitView {
  int n_pairs, n1;
  float window;    // (float)windowSize
  float nn_ratio;
  int keep_max;
  int check_ori;
  const int* kp1_off;
  const uint8_t* kp1_octave;
  const float* kp1_angle;
  const uint8_t* kp1_desc;
  float* prev;                // [n1][2] vbPrevMatched: read by the scans, rewritten by k_init_finalize
  const float* kp2_angle;
  int* cnt;                   // [n1] candidate counts -> pair-local exclusive offsets
  int* pair_total;            // [n_pairs] candidates of the pair
  const int* pair_base;       // [n_pairs] first candidate of the pair in keys
  unsigned long long* keys;   // pack_key(dist, cell, idx, 0)
  int* m12;                   // [n1] vnMatches12
  int* b2;                    // [n1] bestIdx2 of every accepted query (the rotHist entries), -1 otherwise
  int* n_matches;             // [n_pairs]
};

// walk the window of F1 keypoint i (pair p); WRITE = false counts, WRITE = true also stores the keys
template <bool WRITE>
__device__ __forceinline__ int init_scan(const MatchView& v, const InitView& w, int i, int p, unsigned long long* out) {
  const float x = w.prev[2 * (size_t)i], y = w.prev[2 * (size_t)i + 1], r = w.window;
  CellWin cw;
  if (!area_cells(v, x, y, r, cw)) return 0;
  const uint4* qd = reinterpret_cast<const uint4*>(w.kp1_desc + 32 * (size_t)i);
  const uint4 a0 = qd[0], a1 = qd[1];
  const int* cstart = v.cell_count + (size_t)p * (N_CELLS + 1);
  const uint4* rec = v.s_rec + 3 * (size_t)v.cur_off[p];
  int n = 0;
  for (int ix = cw.x0; ix <= cw.x1; ix++) {
    const int s0 = cstart[ix * GRID_ROWS + cw.y0], s1 = cstart[ix * GRID_ROWS + cw.y1 + 1];
    for (int s = s0; s < s1; s++) {
      const uint4 h = rec[3 * (size_t)s];
      const unsigned meta = h.w;
      if ((meta >> 28) & 7) continue;  // minLevel = maxLevel = 0
      const float dx = __fsub_rn(__uint_as_float(h.x), x), dy = __fsub_rn(__uint_as_float(h.y), y);
      if (!(fabsf(dx) < r && fabsf(dy) < r)) continue;
      const int d = popc256(a0, a1, rec[3 * (size_t)s + 1], rec[3 * (size_t)s + 2]);
      if (d > w.keep_max) continue;
      if (WRITE) out[n] = pack_key(d, (meta >> 16) & 0xFFF, meta & 0xFFFF, 0);
      n++;
    }
  }
  return n;
}

__global__ void __launch_bounds__(128) k_init_count(MatchView v, InitView w) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= w.n1) return;
  w.m12[i] = -1;
  w.b2[i] = -1;
  const int p = find_pair(w.kp1_off, w.n_pairs, i);
  w.cnt[i] = w.kp1_octave[i] == 0 ? init_scan<false>(v, w, i, p, nullptr) : 0;
}

__global__ void __launch_bounds__(1024) k_init_scan(InitView w) {
  __shared__ int s_warp[32];
  __shared__ int s_carry;
  const int p = blockIdx.x, t = threadIdx.x, lane = t & 31, wid = t >> 5;
  const int a0 = w.kp1_off[p], n = w.kp1_off[p + 1] - a0;
  if (t == 0) s_carry = 0;
  __syncthreads();
  for (int b = 0; b < n; b += 1024) {
    const int x = b + t < n ? w.cnt[a0 + b + t] : 0;
    int incl = x;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += y;
    }
    if (lane == 31) s_warp[wid] = incl;
    __syncthreads();
    if (wid == 0) {
      int z = s_warp[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, z, o);
        if (lane >= o) z += y;
      }
      s_warp[lane] = z;
    }
    __syncthreads();
    const int carry = s_carry;
    if (b + t < n) w.cnt[a0 + b + t] = carry + incl - x + (wid ? s_warp[wid - 1] : 0);
    __syncthreads();
    if (t == 0) s_carry = carry + s_warp[31];
    __syncthreads();
  }
  if (t == 0) w.pair_total[p] = s_carry;
}

__global__ void __launch_bounds__(128) k_init_fill(MatchView v, InitView w) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= w.n1 || w.kp1_octave[i] != 0) return;
  const int p = find_pair(w.kp1_off, w.n_pairs, i);
  unsigned long long* out = w.keys + (size_t)w.pair_base[p] + w.cnt[i];
  const int n = init_scan<true>(v, w, i, p, out);
  for (int a = 1; a < n; a++) {  // insertion sort: the lists hold the few candidates within keep_max
    const unsigned long long k = out[a];
    int b = a - 1;
    while (b >= 0 && out[b] > k) { out[b + 1] = out[b]; b--; }
    out[b + 1] = k;
  }
}

// SMEM: state word per F2 keypoint = vMatchedDistance (16 high bits, 0xFFFF = INT_MAX: distances are <= 256) |
// vnMatches21 (16 low bits, 0xFFFF = -1); else v.owner / v.match in global memory
template <bool SMEM>
__device__ __forceinline__ void init_resolve(const MatchView& v, const InitView& w, unsigned* st) {
  __shared__ unsigned long long kbuf[INIT_KBUF];
  constexpr unsigned FULL = 0xffffffffu;
  const int p = blockIdx.x, lane = threadIdx.x;
  const int a0 = w.kp1_off[p], n1 = w.kp1_off[p + 1] - a0;
  const int c0 = v.cur_off[p], n2 = v.cur_off[p + 1] - c0;
  const unsigned long long* keys = w.keys + (size_t)w.pair_base[p];
  const int ktot = w.pair_total[p];
  const int* off = w.cnt + a0;
  int* md_g = v.owner + c0;
  int* m21_g = v.match + c0;
  if (SMEM) {
    for (int j = lane; j < n2; j += 32) st[j] = 0xFFFFFFFFu;
    __syncwarp();
  }
  for (int qb = 0; qb < n1; qb += 32) {
    const int qn = min(32, n1 - qb), q = qb + lane;
    const int lo = q < n1 ? off[q] : ktot, hi = q + 1 < n1 ? off[q + 1] : ktot;  // lane's query: keys [lo, hi)
    const int blo = __shfl_sync(FULL, lo, 0), bhi = __shfl_sync(FULL, hi, qn - 1);
    const bool staged = bhi - blo <= INIT_KBUF;
    if (staged)
      for (int k = blo + lane; k < bhi; k += 32) kbuf[k - blo] = keys[k];
    __syncwarp();
    for (int j = 0; j < qn; j++) {
      const int qlo = __shfl_sync(FULL, lo, j), qhi = __shfl_sync(FULL, hi, j);
      int found = 0, d1 = INT_MAX, d2 = INT_MAX, best = -1;
      for (int c = qlo; c < qhi && found < 2; c += 32) {
        const int k = c + lane;
        unsigned long long key = 0;
        bool elig = false;
        if (k < qhi) {
          key = staged ? kbuf[k - blo] : keys[k];
          const int idx = key_idx(key);
          const int md = SMEM ? (int)(st[idx] >> 16) : md_g[idx];
          elig = md > key_dist(key);  // the reference skips vMatchedDistance[i2] <= dist
        }
        unsigned m = __ballot_sync(FULL, elig);
        while (m && found < 2) {
          const unsigned long long kk = __shfl_sync(FULL, key, __ffs(m) - 1);
          m &= m - 1;
          if (found == 0) { d1 = key_dist(kk); best = key_idx(kk); }
          else d2 = key_dist(kk);
          found++;
        }
      }
      // bestDist <= TH_LOW && bestDist < (float)bestDist2 * mfNNratio
      if (d1 <= TH_LOW && (float)d1 < __fmul_rn((float)d2, w.nn_ratio)) {
        if (lane == 0) {
          const int i1 = qb + j;
          int prev;
          if (SMEM) {
            prev = (int)(st[best] & 0xFFFFu);
            if (prev == 0xFFFF) prev = -1;
            st[best] = ((unsigned)d1 << 16) | (unsigned)i1;
          } else {
            prev = m21_g[best];
            m21_g[best] = i1;
            md_g[best] = d1;
          }
          if (prev >= 0) w.m12[a0 + prev] = -1;  // the earlier query loses its match
          w.m12[a0 + i1] = best;
          w.b2[a0 + i1] = best;
        }
        __syncwarp();
      }
    }
    __syncwarp();
  }
}

__global__ void __launch_bounds__(32) k_init_resolve_smem(MatchView v, InitView w) {
  extern __shared__ unsigned init_state[];
  init_resolve<true>(v, w, init_state);
}
__global__ void __launch_bounds__(32) k_init_resolve_global(MatchView v, InitView w) { init_resolve<false>(v, w, nullptr); }

__global__ void __launch_bounds__(256) k_init_finalize(MatchView v, InitView w) {
  __shared__ int s_hist[HISTO_LENGTH];
  __shared__ int s_keep[3];
  __shared__ int s_n;
  const int p = blockIdx.x, tid = threadIdx.x;
  const int a0 = w.kp1_off[p], n1 = w.kp1_off[p + 1] - a0;
  const int c0 = v.cur_off[p];
  if (tid < HISTO_LENGTH) s_hist[tid] = 0;
  if (tid == 0) s_n = 0;
  __syncthreads();
  if (w.check_ori) {
    for (int i = tid; i < n1; i += blockDim.x) {
      const int b = w.b2[a0 + i];
      if (b >= 0) atomicAdd(&s_hist[rot_bin(w.kp1_angle[a0 + i], w.kp2_angle[c0 + b])], 1);
    }
    __syncthreads();
    if (tid == 0) three_maxima(s_hist, s_keep);
    __syncthreads();
  }
  int n = 0;
  for (int i = tid; i < n1; i += blockDim.x) {
    int m = w.m12[a0 + i];
    if (m >= 0 && w.check_ori) {  // a live match is its query's rotHist entry
      const int bin = rot_bin(w.kp1_angle[a0 + i], w.kp2_angle[c0 + m]);
      if (bin != s_keep[0] && bin != s_keep[1] && bin != s_keep[2]) {
        m = -1;
        w.m12[a0 + i] = -1;
      }
    }
    if (m >= 0) {
      n++;
      const float2 xy = reinterpret_cast<const float2*>(v.cur_xy)[c0 + m];
      reinterpret_cast<float2*>(w.prev)[a0 + i] = xy;
    }
  }
  atomicAdd(&s_n, n);
  __syncthreads();
  if (tid == 0) w.n_matches[p] = s_n;
}

inline int cdiv(int a, int b) { return (a + b - 1) / b; }

struct MatchState {
  MatchView v{};
};

}  // namespace

// device pipeline shared by both variants; everything already uploaded into v
static int match_run(LldCtx* c, MatchView& v, int* passes_out) {
  if (v.fused_ok) {  // every pair fits one CTA's shared memory: single launch, no host round trips
    const FusedLayout L = fused_layout(v.max_cur);
    if (v.variant == 0) {
      LLD_CUDA(c, lld_raise_dyn_smem(k_match_fused<0>, (size_t)L.total));
      LLD_LAUNCH(c, k_match_fused<0>, v.n_pairs, FUSED_NT, L.total, v, L);
    } else if (v.variant == 1) {
      LLD_CUDA(c, lld_raise_dyn_smem(k_match_fused<1>, (size_t)L.total));
      LLD_LAUNCH(c, k_match_fused<1>, v.n_pairs, FUSED_NT, L.total, v, L);
    } else {
      LLD_CUDA(c, lld_raise_dyn_smem(k_match_fused<2>, (size_t)L.total));
      LLD_LAUNCH(c, k_match_fused<2>, v.n_pairs, FUSED_NT, L.total, v, L);
    }
    LLD_CUDA(c, cudaGetLastError());
    if (passes_out) *passes_out = 0;
    return LLD_OK;
  }
  LLD_CUDA(c, cudaMemsetAsync(v.cell_count, 0, sizeof(int) * (size_t)v.n_pairs * (N_CELLS + 1), c->stream));
  if (v.n_cur) LLD_LAUNCH(c, k_cell_count, cdiv(v.n_cur, 256), 256, 0, v);
  LLD_LAUNCH(c, k_cell_scan, v.n_pairs, 1024, 0, v);
  if (v.n_cur) LLD_LAUNCH(c, k_cell_fill, cdiv(v.n_cur, 256), 256, 0, v);
  int* h_changed = reinterpret_cast<int*>(c->pinned);
  int pass = 0;
  const int max_pass = 64;
  if (v.n_q) {
    LLD_LAUNCH(c, k_pair_prep, cdiv(v.n_pairs, 128), 128, 0, v);
    LLD_LAUNCH(c, k_query_pair, cdiv(v.n_q, 256), 256, 0, v);
    LLD_LAUNCH(c, k_match_scan, cdiv(v.n_q, 128), 128, 0, v);
    while (true) {
      LLD_LAUNCH(c, k_match_resolve, cdiv(v.n_q, 128), 128, 0, v, pass);
      if (pass > 0) {
        LLD_DOWN(c, h_changed, v.changed, 1);
        LLD_CUDA(c, cudaStreamSynchronize(c->stream));
        if (!*h_changed) break;
      }
      if (pass >= max_pass) {
        snprintf(c->err, sizeof(c->err), "claim resolution did not converge in %d passes", max_pass);
        return LLD_ERR_CUDA;
      }
      if (v.n_cur) LLD_LAUNCH(c, k_owner_reset, cdiv(v.n_cur, 256), 256, 0, v);
      LLD_LAUNCH(c, k_claim, cdiv(v.n_q, 256), 256, 0, v);
      pass++;
    }
  }
  LLD_LAUNCH(c, k_finalize, v.n_pairs, 256, 0, v);
  LLD_CUDA(c, cudaGetLastError());
  if (passes_out) *passes_out = pass + 1;
  return LLD_OK;
}

static int match_alloc_common(LldCtx* c, MatchView& v) {
  LLD_DEV(c, v.cell_count, (size_t)v.n_pairs * (N_CELLS + 1));
  LLD_DEV(c, v.cell_fill, (size_t)v.n_pairs * N_CELLS);
  LLD_DEV(c, v.kp_cell, v.n_cur);
  LLD_DEV(c, v.s_rec, 3 * (size_t)v.n_cur);
  LLD_DEV(c, v.owner, v.n_cur);
  LLD_DEV(c, v.q_best, v.n_q);
  LLD_DEV(c, v.q_dist, v.n_q);
  LLD_DEV(c, v.changed, 1);
  LLD_DEV(c, v.q_pair, v.n_q);
  LLD_DEV(c, v.pair_mode, v.n_pairs);
  LLD_DEV(c, v.q_top, 4 * (size_t)v.n_q);
  LLD_DEV(c, v.q_ncand, v.n_q);
  LLD_DEV(c, v.match, v.n_cur);
  LLD_DEV(c, v.n_matches, v.n_pairs);
  LLD_CUDA(c, cudaMemsetAsync(v.changed, 0, sizeof(int), c->stream));
  return LLD_OK;
}

// fused single-CTA path when the largest pair fits shared memory (LLD_MATCH_FUSED=0 forces the multi-kernel path)
static void set_dispatch(MatchView& v, const int32_t* cur_off, const int32_t* q_off) {
  v.max_cur = 0; v.max_q = 0;
  for (int i = 0; i < v.n_pairs; i++) {
    v.max_cur = std::max(v.max_cur, cur_off[i + 1] - cur_off[i]);
    v.max_q = std::max(v.max_q, q_off[i + 1] - q_off[i]);
  }
  const char* e = getenv("LLD_MATCH_FUSED");
  const bool allow = !(e && e[0] == '0');
  v.fused_ok = allow && fused_layout(v.max_cur).total <= 227 * 1024 && v.max_q <= FUSED_QPT * FUSED_NT && v.max_cur <= FUSED_KPT * FUSED_NT;
}

static void set_geom(MatchView& v, const lld_frame_geom& g) {
  v.fx = g.fx; v.fy = g.fy; v.cx = g.cx; v.cy = g.cy; v.bf = g.bf; v.b = g.b;
  v.min_x = g.min_x; v.max_x = g.max_x; v.min_y = g.min_y; v.max_y = g.max_y;
  v.winv = static_cast<float>(GRID_COLS) / (g.max_x - g.min_x);   // src/Frame.cc:143-144
  v.hinv = static_cast<float>(GRID_ROWS) / (g.max_y - g.min_y);
  v.n_levels = g.n_levels;
}

static int match_download(LldCtx* c, MatchView& v, lld_sbp_result* out) {
  LLD_CUDA(c, cudaEventRecord(c->ev[2], c->stream));
  int* h_flag = reinterpret_cast<int*>(c->pinned);
  LLD_DOWN(c, h_flag, v.changed, 1);
  LLD_DOWN(c, out->match, v.match, v.n_cur);
  LLD_DOWN(c, out->n_matches, v.n_matches, v.n_pairs);
  LLD_DOWN(c, out->best_idx, v.q_best, v.n_q);
  LLD_DOWN(c, out->best_dist, v.q_dist, v.n_q);
  if (int r = lld_call_end(c)) return r;
  if (*h_flag & 2) {
    snprintf(c->err, sizeof(c->err), "claim resolution did not converge in 64 passes");
    return LLD_ERR_CUDA;
  }
  return LLD_OK;
}

// resident-mode view (bench): uploaded once, run many times; owned by the context, invalid as soon as another entry point of the
// same context recycles the device pool
static MatchView* resident_view(LldCtx* c, bool create) {
  if (!c->resident[0] && create) {
    c->resident[0] = new MatchView();
    c->resident_free[0] = [](void* p) { delete static_cast<MatchView*>(p); };
  }
  return static_cast<MatchView*>(c->resident[0]);
}
static bool resident_valid(LldCtx* c) {
  if (c->resident[0] && c->resident_gen[0] == c->pool_gen) return true;
  snprintf(c->err, sizeof(c->err), "no resident matcher problem (not uploaded, or another call on this context recycled the device pool)");
  return false;
}

static int sbp_frame_upload(LldCtx* c, const lld_sbp_frame_problem* p, MatchView& v) {
  v = MatchView();
  v.n_pairs = p->n_pairs;
  LLD_ARG(c, p->n_pairs >= 1);
  v.n_cur = p->cur_off[p->n_pairs];
  v.n_q = p->last_off[p->n_pairs];
  LLD_ARG(c, p->geom.n_levels >= 1 && p->geom.n_levels <= 8);  // octave is packed into 3 bits of the candidate key
  for (int i = 0; i < p->n_pairs; i++) LLD_ARG(c, p->cur_off[i + 1] - p->cur_off[i] <= 65535);
  set_dispatch(v, p->cur_off, p->last_off);
  v.variant = 0;
  set_geom(v, p->geom);
  v.th = p->th; v.nn_ratio = 0; v.mono = p->mono; v.check_ori = p->check_orientation;
  v.th_high = p->th_high > 0 ? p->th_high : TH_HIGH; v.allow_neg_z = p->allow_negative_depth != 0;
  LLD_UP(c, v.scale, p->geom.scale_factors, p->geom.n_levels);
  LLD_UP(c, v.cur_off, p->cur_off, p->n_pairs + 1);
  LLD_UP(c, v.cur_xy, p->cur_xy, 2 * (size_t)v.n_cur);
  LLD_UP(c, v.cur_octave, p->cur_octave, v.n_cur);
  LLD_UP(c, v.cur_angle, p->cur_angle, v.n_cur);
  LLD_UP(c, v.cur_uright, p->cur_uright, v.n_cur);
  LLD_UP(c, v.cur_desc, p->cur_desc, 32 * (size_t)v.n_cur);
  LLD_UP(c, v.cur_claimed, p->cur_claimed, v.n_cur);
  LLD_UP(c, v.cur_Tcw, p->cur_Tcw, 12 * (size_t)p->n_pairs);
  LLD_UP(c, v.last_Tcw, p->last_Tcw, 12 * (size_t)p->n_pairs);
  LLD_UP(c, v.q_off, p->last_off, p->n_pairs + 1);
  LLD_UP(c, v.q_valid, p->last_valid, v.n_q);
  LLD_UP(c, v.q_xw, p->last_xw, 3 * (size_t)v.n_q);
  LLD_UP(c, v.q_octave, p->last_octave, v.n_q);
  LLD_UP(c, v.q_angle, p->last_angle, v.n_q);
  LLD_UP(c, v.q_desc, p->last_desc, 32 * (size_t)v.n_q);
  LLD_UP(c, v.q_has_obs, p->last_has_obs, v.n_q);
  return match_alloc_common(c, v);
}

static int sbp_mp_upload(LldCtx* c, const lld_sbp_mp_problem* p, MatchView& v) {
  v = MatchView();
  v.n_pairs = p->n_pairs;
  LLD_ARG(c, p->n_pairs >= 1);
  v.n_cur = p->cur_off[p->n_pairs];
  v.n_q = p->mp_off[p->n_pairs];
  LLD_ARG(c, p->geom.n_levels >= 1 && p->geom.n_levels <= 8);
  for (int i = 0; i < p->n_pairs; i++) LLD_ARG(c, p->cur_off[i + 1] - p->cur_off[i] <= 65535);
  set_dispatch(v, p->cur_off, p->mp_off);
  v.variant = 1;
  set_geom(v, p->geom);
  v.th = p->th; v.nn_ratio = p->nn_ratio; v.mono = 0; v.check_ori = 0;
  v.th_high = TH_HIGH; v.allow_neg_z = 0;
  LLD_UP(c, v.scale, p->geom.scale_factors, p->geom.n_levels);
  LLD_UP(c, v.cur_off, p->cur_off, p->n_pairs + 1);
  LLD_UP(c, v.cur_xy, p->cur_xy, 2 * (size_t)v.n_cur);
  LLD_UP(c, v.cur_octave, p->cur_octave, v.n_cur);
  LLD_UP(c, v.cur_uright, p->cur_uright, v.n_cur);
  LLD_UP(c, v.cur_desc, p->cur_desc, 32 * (size_t)v.n_cur);
  LLD_UP(c, v.cur_claimed, p->cur_claimed, v.n_cur);
  v.cur_angle = nullptr;
  LLD_UP(c, v.q_off, p->mp_off, p->n_pairs + 1);
  LLD_UP(c, v.q_valid, p->mp_valid, v.n_q);
  LLD_UP(c, v.q_xw, p->mp_proj, 3 * (size_t)v.n_q);
  LLD_UP(c, v.q_level, p->mp_level, v.n_q);
  LLD_UP(c, v.q_viewcos, p->mp_viewcos, v.n_q);
  LLD_UP(c, v.q_desc, p->mp_desc, 32 * (size_t)v.n_q);
  LLD_UP(c, v.q_has_obs, p->mp_has_obs, v.n_q);
  return match_alloc_common(c, v);
}

// keyframe searches (Fuse, Fuse with Sim3, SearchByProjection with Sim3): variant 2
static int kf_search_upload(LldCtx* c, const lld_kf_search_problem* p, MatchView& v) {
  v = MatchView();
  v.n_pairs = p->n_pairs;
  LLD_ARG(c, p->n_pairs >= 1);
  v.n_cur = p->kp_off[p->n_pairs];
  v.n_q = p->mp_off[p->n_pairs];
  LLD_ARG(c, p->geom.n_levels >= 1 && p->geom.n_levels <= 8);
  for (int i = 0; i < p->n_pairs; i++) LLD_ARG(c, p->kp_off[i + 1] - p->kp_off[i] <= 65535);
  set_dispatch(v, p->kp_off, p->mp_off);
  v.variant = 2;
  set_geom(v, p->geom);
  v.th = p->th; v.nn_ratio = 0.f; v.mono = 0; v.check_ori = 0;
  v.th_high = p->th_low; v.allow_neg_z = 0;
  v.chi2_gate = p->chi2_gate != 0;
  for (int i = 0; i < 8; i++) v.inv_sigma2[i] = p->inv_level_sigma2[i];
  LLD_UP(c, v.scale, p->geom.scale_factors, p->geom.n_levels);
  LLD_UP(c, v.cur_off, p->kp_off, p->n_pairs + 1);
  LLD_UP(c, v.cur_xy, p->kp_xy, 2 * (size_t)v.n_cur);
  LLD_UP(c, v.cur_octave, p->kp_octave, v.n_cur);
  LLD_UP(c, v.cur_uright, p->kp_uright, v.n_cur);
  LLD_UP(c, v.cur_desc, p->kp_desc, 32 * (size_t)v.n_cur);
  LLD_UP(c, v.cur_claimed, p->kp_claimed, v.n_cur);
  v.cur_angle = nullptr;
  LLD_UP(c, v.q_off, p->mp_off, p->n_pairs + 1);
  LLD_UP(c, v.q_valid, p->mp_valid, v.n_q);
  LLD_UP(c, v.q_xw, p->mp_proj, 3 * (size_t)v.n_q);
  LLD_UP(c, v.q_level, p->mp_level, v.n_q);
  v.q_viewcos = nullptr;
  LLD_UP(c, v.q_desc, p->mp_desc, 32 * (size_t)v.n_q);
  // every accepted point claims its keypoint (vpMatched[bestIdx] = pMP) or none does (Fuse)
  uint8_t* has = nullptr;
  LLD_DEV(c, has, v.n_q);
  LLD_CUDA(c, cudaMemsetAsync(has, p->sequential_claims ? 1 : 0, v.n_q ? v.n_q : 1, c->stream));
  v.q_has_obs = has;
  return match_alloc_common(c, v);
}

extern "C" int lld_kf_search(void* ctx, const lld_kf_search_problem* p, lld_sbp_result* out) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !p || !out) return LLD_ERR_ARG;
  if (int r = lld_call_begin(c, true)) return r;
  MatchView v;
  int r = kf_search_upload(c, p, v);
  if (r) return r;
  LLD_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
  r = match_run(c, v, nullptr);
  if (r) return r;
  return match_download(c, v, out);
}

// smallest candidate distance bound above which the outcome of a query cannot change: for a best distance <= TH_LOW, every
// bestDist2 > keep_max passes bestDist < (float)bestDist2 * nn_ratio (IEEE multiplication is monotone); 256 keeps everything
static int init_keep_max(float nn_ratio) {
  for (int d = TH_LOW; d < 256; d++)
    if ((float)TH_LOW < (float)(d + 1) * nn_ratio) return d;
  return 256;
}

// largest F2 (keypoints) whose resolve state fits shared memory next to the staged keys
static constexpr int INIT_SMEM_MAX_KP = (227 * 1024 - 8 * INIT_KBUF) / 4;

extern "C" int lld_init_search(void* ctx, const lld_init_search_problem* p, lld_init_search_result* out) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !p || !out) return LLD_ERR_ARG;
  LLD_ARG(c, p->n_pairs >= 1);
  const int P = p->n_pairs, n1 = p->kp1_off[P], n2 = p->kp2_off[P];
  int max2 = 0;
  for (int i = 0; i < P; i++) {
    const int a = p->kp1_off[i + 1] - p->kp1_off[i], b = p->kp2_off[i + 1] - p->kp2_off[i];
    LLD_ARG(c, a >= 0 && a <= 65535 && b >= 0 && b <= 65535);
    max2 = std::max(max2, b);
  }
  for (int i = 0; i < n2; i++) LLD_ARG(c, p->kp2_octave[i] < 8);   // 3 bits of the grid record
  if (p->check_orientation) {   // keeps every rotation bin in [0, HISTO_LENGTH]
    for (int i = 0; i < n1; i++) LLD_ARG(c, p->kp1_angle[i] >= 0.f && p->kp1_angle[i] < 900.f);
    for (int i = 0; i < n2; i++) LLD_ARG(c, p->kp2_angle[i] >= 0.f && p->kp2_angle[i] < 360.f);
  }
  if (int r = lld_call_begin(c, true)) return r;
  MatchView v{};
  v.n_pairs = P;
  v.n_cur = n2;
  set_geom(v, p->geom);
  LLD_UP(c, v.cur_off, p->kp2_off, P + 1);
  LLD_UP(c, v.cur_xy, p->kp2_xy, 2 * (size_t)n2);
  LLD_UP(c, v.cur_octave, p->kp2_octave, n2);
  LLD_UP(c, v.cur_desc, p->kp2_desc, 32 * (size_t)n2);
  float* uright = nullptr;   // the grid record's stereo and claim fields are not used by this search
  uint8_t* claimed = nullptr;
  LLD_DEV(c, uright, n2);
  LLD_DEV(c, claimed, n2);
  LLD_CUDA(c, cudaMemsetAsync(uright, 0, sizeof(float) * (size_t)std::max(n2, 1), c->stream));
  LLD_CUDA(c, cudaMemsetAsync(claimed, 0, (size_t)std::max(n2, 1), c->stream));
  v.cur_uright = uright;
  v.cur_claimed = claimed;
  LLD_DEV(c, v.cell_count, (size_t)P * (N_CELLS + 1));
  LLD_DEV(c, v.cell_fill, (size_t)P * N_CELLS);
  LLD_DEV(c, v.kp_cell, n2);
  LLD_DEV(c, v.s_rec, 3 * (size_t)n2);
  LLD_DEV(c, v.owner, n2);
  LLD_DEV(c, v.match, n2);
  InitView w{};
  w.n_pairs = P;
  w.n1 = n1;
  w.window = (float)p->window_size;
  w.nn_ratio = p->nn_ratio;
  w.keep_max = init_keep_max(p->nn_ratio);
  w.check_ori = p->check_orientation != 0;
  LLD_UP(c, w.kp1_off, p->kp1_off, P + 1);
  LLD_UP(c, w.kp1_octave, p->kp1_octave, n1);
  LLD_UP(c, w.kp1_angle, p->kp1_angle, n1);
  LLD_UP(c, w.kp1_desc, p->kp1_desc, 32 * (size_t)n1);
  LLD_UP(c, w.prev, p->prev_matched, 2 * (size_t)n1);
  LLD_UP(c, w.kp2_angle, p->kp2_angle, n2);
  LLD_DEV(c, w.cnt, n1);
  LLD_DEV(c, w.pair_total, P);
  LLD_DEV(c, w.m12, n1);
  LLD_DEV(c, w.b2, n1);
  LLD_DEV(c, w.n_matches, P);
  int* pair_base = nullptr;
  LLD_DEV(c, pair_base, P);
  w.pair_base = pair_base;
  LLD_CUDA(c, cudaEventRecord(c->ev[1], c->stream));

  LLD_CUDA(c, cudaMemsetAsync(v.cell_count, 0, sizeof(int) * (size_t)P * (N_CELLS + 1), c->stream));
  if (n2) LLD_LAUNCH(c, k_cell_count, cdiv(n2, 256), 256, 0, v);
  LLD_LAUNCH(c, k_cell_scan, P, 1024, 0, v);
  if (n2) LLD_LAUNCH(c, k_cell_fill, cdiv(n2, 256), 256, 0, v);
  if (n1) LLD_LAUNCH(c, k_init_count, cdiv(n1, 128), 128, 0, v, w);
  LLD_LAUNCH(c, k_init_scan, P, 1024, 0, w);
  // the candidate buffer is sized from the counts: one read-back of the pair totals
  std::vector<int> total((size_t)P), base((size_t)P);
  LLD_DOWN(c, total.data(), w.pair_total, P);
  LLD_CUDA(c, cudaStreamSynchronize(c->stream));
  long long sum = 0;
  for (int i = 0; i < P; i++) {
    base[(size_t)i] = (int)sum;
    sum += total[(size_t)i];
    if (sum > INT_MAX) {
      snprintf(c->err, sizeof(c->err), "lld_init_search: more than 2^31 - 1 candidates in one batch; split the batch");
      return LLD_ERR_UNSUPPORTED;
    }
  }
  LLD_CUDA(c, cudaMemcpyAsync(pair_base, base.data(), sizeof(int) * (size_t)P, cudaMemcpyHostToDevice, c->stream));
  LLD_DEV(c, w.keys, (size_t)sum);
  if (n1) LLD_LAUNCH(c, k_init_fill, cdiv(n1, 128), 128, 0, v, w);
  if (max2 <= INIT_SMEM_MAX_KP) {
    const int smem = 4 * std::max(max2, 1);
    LLD_CUDA(c, lld_raise_dyn_smem(k_init_resolve_smem, (size_t)smem));
    LLD_LAUNCH(c, k_init_resolve_smem, P, 32, smem, v, w);
  } else {
    LLD_LAUNCH(c, k_init_resolve_global, P, 32, 0, v, w);
  }
  LLD_LAUNCH(c, k_init_finalize, P, 256, 0, v, w);
  LLD_CUDA(c, cudaGetLastError());
  LLD_CUDA(c, cudaEventRecord(c->ev[2], c->stream));
  LLD_DOWN(c, out->match12, w.m12, n1);
  LLD_DOWN(c, out->prev_matched, w.prev, 2 * (size_t)n1);
  LLD_DOWN(c, out->n_matches, w.n_matches, P);
  return lld_call_end(c);
}

extern "C" int lld_sbp_frame(void* ctx, const lld_sbp_frame_problem* p, lld_sbp_result* out) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !p || !out) return LLD_ERR_ARG;
  if (int r = lld_call_begin(c, true)) return r;
  MatchView v;
  int r = sbp_frame_upload(c, p, v);
  if (r) return r;
  LLD_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
  r = match_run(c, v, nullptr);
  if (r) return r;
  return match_download(c, v, out);
}

extern "C" int lld_sbp_mappoints(void* ctx, const lld_sbp_mp_problem* p, lld_sbp_result* out) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !p || !out) return LLD_ERR_ARG;
  if (int r = lld_call_begin(c, true)) return r;
  MatchView v;
  int r = sbp_mp_upload(c, p, v);
  if (r) return r;
  LLD_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
  r = match_run(c, v, nullptr);
  if (r) return r;
  return match_download(c, v, out);
}

// resident mode for the bench: upload once, run repeatedly with inputs in HBM
extern "C" int lld_sbp_frame_upload(void* ctx, const lld_sbp_frame_problem* p) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !p) return LLD_ERR_ARG;
  if (int r = lld_call_begin(c, false)) return r;
  int r = sbp_frame_upload(c, p, *resident_view(c, true));
  c->resident_gen[0] = r ? 0 : c->pool_gen;
  if (r) return r;
  LLD_CUDA(c, cudaStreamSynchronize(c->stream));
  return LLD_OK;
}
extern "C" int lld_sbp_run(void* ctx, int* passes) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !resident_valid(c)) return LLD_ERR_ARG;
  LLD_CUDA(c, cudaSetDevice(c->device));
  return match_run(c, *resident_view(c, false), passes);
}
extern "C" int lld_sbp_download(void* ctx, lld_sbp_result* out) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !out || !resident_valid(c)) return LLD_ERR_ARG;
  LLD_CUDA(c, cudaEventRecord(c->ev[0], c->stream));
  LLD_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
  return match_download(c, *resident_view(c, false), out);
}

// host inline popcount distance (ORBmatcher::DescriptorDistance): API completeness, no device involved
extern "C" int lld_descriptor_distance(const uint8_t a[32], const uint8_t b[32]) {
  int dist = 0;
  for (int i = 0; i < 8; i++) {
    uint32_t pa, pb;
    memcpy(&pa, a + 4 * i, 4);
    memcpy(&pb, b + 4 * i, 4);
    dist += __builtin_popcount(pa ^ pb);
  }
  return dist;
}
