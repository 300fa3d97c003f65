// stereo.cu — Frame::ComputeStereoMatches (src/Frame.cc:530-704) for a batch of stereo frames.
//
// One CTA per frame:
//   A  row bands: thread = image row; it walks the right keypoints in index order and lists those whose band
//      [floor(y - r), ceil(y + r)], r = 2 scale[octave], contains the row (vRowIndices, :539-556).  Index order inside a
//      row is the reference's push_back order, which decides ties of the Hamming distance; no atomics, no sort.
//   B  thread = left keypoint: candidates of row (int)vL, octave +-1, disparity window [uL - maxD, uL], best 256-bit Hamming
//      distance (strict <: first candidate wins a tie), accepted below (TH_HIGH + TH_LOW) / 2 (:565-613).
//   C  warp = accepted keypoint: 11x11 SAD of the left patch against the right patch slid over -5..+5 pixels at the
//      keypoint's pyramid level.  The reference subtracts the centre pixel as float and takes cv::norm(NORM_L1); both
//      patches hold small integers, so integer arithmetic gives the same sums exactly.  Parabola fit, disparity / depth in
//      float with the reference's operation order (this file is compiled with --fmad=false) (:615-688).
//   D  median gate: k-th order statistic of the SAD distances by two 8-bit histogram passes (the reference sorts
//      (distance, index) pairs; only the distance of the middle element is used), reject distance >= 1.5 * 1.4 * median
//      (:692-703).
// Undefined behaviour of the reference (unchecked row index, patches leaving the pyramid image, median of an empty list)
// is resolved as DESIGN.md documents (and as the test oracle does): the point gets no stereo match.
#include <algorithm>
#include <cfloat>
#include <climits>
#include <cmath>

#include "lld_ctx.h"

namespace {

constexpr int ST_NT = 512;
constexpr int TH_HIGH_S = 100, TH_LOW_S = 50;

struct StereoView {
  int n_frames;
  const int* l_off;
  const int* r_off;
  const float* l_xy;
  const uint8_t* l_oct;
  const uint8_t* l_desc;
  const float* r_xy;
  const uint8_t* r_oct;
  const uint8_t* r_desc;
  int n_levels;
  float scale[8], inv_scale[8];
  int rows[8], cols[8], stride[8];
  const uint8_t* pyr;
  const long long* pyr_off;   // [n_frames][2][n_levels]
  float mb, mbf;
  // per-frame scratch in global memory
  int* row_start;      // [n_frames][rows0 + 1]
  unsigned short* row_list;  // [n_frames][list_cap]
  int list_cap;
  int* best_r;         // [n_left] matched right keypoint or -1
  int* sad;            // [n_left] best SAD distance of an accepted match, -1 otherwise
  float* uright;
  float* depth;
  int* n_matched;
  int* overflow;
};

__device__ __forceinline__ int popc256s(const uint4& a0, const uint4& a1, const uint4& b0, const uint4& b1) {
  return __popc(a0.x ^ b0.x) + __popc(a0.y ^ b0.y) + __popc(a0.z ^ b0.z) + __popc(a0.w ^ b0.w) + __popc(a1.x ^ b1.x) +
         __popc(a1.y ^ b1.y) + __popc(a1.z ^ b1.z) + __popc(a1.w ^ b1.w);
}

__global__ void __launch_bounds__(ST_NT) k_stereo(StereoView v) {
  const int f = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int l0 = v.l_off[f], nl = v.l_off[f + 1] - l0;
  const int r0g = v.r_off[f], nr = v.r_off[f + 1] - r0g;
  const int nRows = v.rows[0];
  int* rstart = v.row_start + (size_t)f * (nRows + 1);
  unsigned short* rlist = v.row_list + (size_t)f * v.list_cap;
  __shared__ int s_cnt[ST_NT];
  __shared__ int s_hist[256];
  __shared__ int s_misc[4];
  // ---- A: row bands.  pass 1 counts, pass 2 fills (thread = row, right keypoints in index order) ----
  for (int pass = 0; pass < 2; pass++) {
    for (int base = 0; base < nRows; base += ST_NT) {
      const int yi = base + tid;
      int cnt = 0;
      const int dst = (pass == 1 && yi < nRows) ? rstart[yi] : 0;
      if (yi < nRows) {
        for (int i = 0; i < nr; i++) {
          const float ky = v.r_xy[2 * (size_t)(r0g + i) + 1];
          const float r = 2.0f * v.scale[v.r_oct[r0g + i]];
          const int maxr = (int)ceilf(ky + r), minr = (int)floorf(ky - r);
          if (yi >= minr && yi <= maxr) {
            if (pass == 1 && dst + cnt < v.list_cap) rlist[dst + cnt] = (unsigned short)i;
            cnt++;
          }
        }
      }
      if (pass == 0 && yi < nRows) rstart[yi] = cnt;   // counts first, turned into offsets below
    }
    __syncthreads();
    if (pass == 0) {
      if (tid == 0) {   // exclusive prefix over <= a few hundred rows
        int run = 0;
        for (int y = 0; y < nRows; y++) { const int c = rstart[y]; rstart[y] = run; run += c; }
        rstart[nRows] = run;
        if (run > v.list_cap) atomicOr(v.overflow, 1);
      }
      __syncthreads();
    }
  }
  __syncthreads();
  // ---- B: best Hamming candidate per left keypoint ----
  const float maxD = v.mbf / v.mb;
  const int thOrbDist = (TH_HIGH_S + TH_LOW_S) / 2;
  for (int i = tid; i < nl; i += ST_NT) {
    const size_t gi = (size_t)(l0 + i);
    v.uright[gi] = -1.0f; v.depth[gi] = -1.0f; v.sad[gi] = -1;
    int best_r = -1;
    const float uL = v.l_xy[2 * gi], vL = v.l_xy[2 * gi + 1];
    const int levelL = v.l_oct[gi];
    if (vL >= 0.0f && (int)vL < nRows) {
      const int row = (int)vL;
      const int c0 = rstart[row], c1 = min(rstart[row + 1], v.list_cap);
      const float minU = uL - maxD, maxU = uL;
      if (c1 > c0 && !(maxU < 0)) {
        const uint4* dl = reinterpret_cast<const uint4*>(v.l_desc + 32 * gi);
        const uint4 a0 = dl[0], a1 = dl[1];
        int bestDist = TH_HIGH_S;
        for (int c = c0; c < c1; c++) {
          const int ir = rlist[c];
          const int oc = v.r_oct[r0g + ir];
          if (oc < levelL - 1 || oc > levelL + 1) continue;
          const float uR = v.r_xy[2 * (size_t)(r0g + ir)];
          if (uR >= minU && uR <= maxU) {
            const uint4* dr = reinterpret_cast<const uint4*>(v.r_desc + 32 * (size_t)(r0g + ir));
            const int dist = popc256s(a0, a1, dr[0], dr[1]);
            if (dist < bestDist) { bestDist = dist; best_r = ir; }
          }
        }
        if (!(bestDist < thOrbDist)) best_r = -1;
      }
    }
    v.best_r[gi] = best_r;
  }
  __syncthreads();
  // ---- C: SAD refinement, one warp per accepted keypoint ----
  const int nw = ST_NT / 32;
  for (int i = wid; i < nl; i += nw) {
    const size_t gi = (size_t)(l0 + i);
    const int ir = v.best_r[gi];
    if (ir < 0) continue;                          // warp-uniform
    const float uL = v.l_xy[2 * gi], vL = v.l_xy[2 * gi + 1];
    const int lvl = v.l_oct[gi];
    const float uR0 = v.r_xy[2 * (size_t)(r0g + ir)];
    const float sfac = v.inv_scale[lvl];
    const float scaleduL = roundf(uL * sfac), scaledvL = roundf(vL * sfac), scaleduR0 = roundf(uR0 * sfac);
    const int w = 5, L = 5;
    const int rows = v.rows[lvl], cols = v.cols[lvl], stride = v.stride[lvl];
    const int pr0 = (int)(scaledvL - w), c0L = (int)(scaleduL - w);
    if (pr0 < 0 || pr0 + 2 * w + 1 > rows || c0L < 0 || c0L + 2 * w + 1 > cols) continue;
    const float iniu = scaleduR0 + L - w, endu = scaleduR0 + L + w + 1;
    if (iniu < 0 || endu >= (float)cols) continue;
    const int cR = (int)(scaleduR0 - L - w);       // first column of the strip: c0R at incR = -L
    // (int)(scaleduR0 + incR - w) = (int)scaleduR0 + incR - w for the integral-valued scaleduR0 >= 0 checked above
    if (cR < 0 || cR + 2 * L + 2 * w + 1 > cols) continue;
    const uint8_t* imL = v.pyr + v.pyr_off[((size_t)f * 2 + 0) * v.n_levels + lvl];
    const uint8_t* imR = v.pyr + v.pyr_off[((size_t)f * 2 + 1) * v.n_levels + lvl];
    const int cenL = imL[(size_t)(pr0 + w) * stride + c0L + w];
    int acc[11];
#pragma unroll
    for (int k = 0; k < 11; k++) acc[k] = 0;
    // centre pixels of the 11 right patches: row pr0 + w, columns cR + w + k
    int cenR[11];
#pragma unroll
    for (int k = 0; k < 11; k++) cenR[k] = imR[(size_t)(pr0 + w) * stride + cR + w + k];
    for (int px = lane; px < 121; px += 32) {
      const int y = px / 11, x = px - 11 * y;
      const int dlv = (int)imL[(size_t)(pr0 + y) * stride + c0L + x] - cenL;
      const uint8_t* rr = imR + (size_t)(pr0 + y) * stride + cR + x;
#pragma unroll
      for (int k = 0; k < 11; k++) acc[k] += abs(dlv - ((int)rr[k] - cenR[k]));
    }
#pragma unroll
    for (int k = 0; k < 11; k++)
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
    if (lane == 0) {
      int bestDistS = INT_MAX, bestinc = 0;
#pragma unroll
      for (int k = 0; k < 11; k++) {
        const float dist = (float)acc[k];
        if (dist < (float)bestDistS) { bestDistS = (int)dist; bestinc = k - L; }
      }
      if (bestinc != -L && bestinc != L) {
        float d1 = 0.f, d2 = 0.f, d3 = 0.f;
#pragma unroll
        for (int k = 1; k < 10; k++)
          if (k - L == bestinc) { d1 = (float)acc[k - 1]; d2 = (float)acc[k]; d3 = (float)acc[k + 1]; }
        const float deltaR = (d1 - d3) / (2.0f * (d1 + d3 - 2.0f * d2));
        if (!(deltaR < -1 || deltaR > 1)) {
          float bestuR = v.scale[lvl] * ((float)scaleduR0 + (float)bestinc + deltaR);
          float disparity = uL - bestuR;
          if (disparity >= 0 && disparity < maxD) {
            if (disparity <= 0) {
              disparity = 0.01;
              bestuR = uL - 0.01;          // float - double, narrowed: as the reference
            }
            v.depth[gi] = v.mbf / disparity;
            v.uright[gi] = bestuR;
            v.sad[gi] = bestDistS;
          }
        }
      }
    }
  }
  __syncthreads();
  // ---- D: median gate.  k = count / 2-th smallest SAD (0-based), by two 8-bit histogram levels (distances < 2^16) ----
  int cnt_local = 0;
  for (int i = tid; i < nl; i += ST_NT) cnt_local += v.sad[l0 + i] >= 0;
  s_cnt[tid] = cnt_local;
  __syncthreads();
  if (tid == 0) {
    int tot = 0;
    for (int t = 0; t < ST_NT; t++) tot += s_cnt[t];
    s_misc[0] = tot;
  }
  __syncthreads();
  const int total = s_misc[0];
  if (total == 0) {
    if (tid == 0) v.n_matched[f] = 0;
    return;
  }
  int k = total / 2, prefix = 0;
  for (int level = 0; level < 2; level++) {
    for (int b = tid; b < 256; b += ST_NT) s_hist[b] = 0;
    __syncthreads();
    for (int i = tid; i < nl; i += ST_NT) {
      const int s = v.sad[l0 + i];
      if (s < 0) continue;
      const int sc = min(s, 65535);
      if (level == 0) atomicAdd(&s_hist[sc >> 8], 1);
      else if ((sc >> 8) == prefix) atomicAdd(&s_hist[sc & 255], 1);
    }
    __syncthreads();
    if (tid == 0) {
      int run = 0, b = 0;
      for (; b < 256; b++) {
        if (run + s_hist[b] > k) break;
        run += s_hist[b];
      }
      s_misc[1] = b;
      s_misc[2] = k - run;
    }
    __syncthreads();
    if (level == 0) prefix = s_misc[1];
    else prefix = (prefix << 8) | s_misc[1];
    k = s_misc[2];
    __syncthreads();
  }
  const float median = (float)prefix;
  const float thDist = 1.5f * 1.4f * median;
  int kept = 0;
  for (int i = tid; i < nl; i += ST_NT) {
    const size_t gi = (size_t)(l0 + i);
    const int s = v.sad[gi];
    if (s < 0) continue;
    if ((float)s < thDist) kept++;
    else { v.uright[gi] = -1.0f; v.depth[gi] = -1.0f; }
  }
  s_cnt[tid] = kept;
  __syncthreads();
  if (tid == 0) {
    int tot = 0;
    for (int t = 0; t < ST_NT; t++) tot += s_cnt[t];
    v.n_matched[f] = tot;
  }
}

}  // namespace

// Frame::ComputeStereoMatches for a batch of frames (include/lldba.h)
extern "C" int lld_stereo_matches(void* ctx, const lld_stereo_problem* p, lld_stereo_result* out) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !p || !out) return LLD_ERR_ARG;
  c->launches = 0;   // a rejected call reports no launches
  LLD_ARG(c, p->n_frames >= 1 && p->n_levels >= 1 && p->n_levels <= 8);
  const int F = p->n_frames, n_l = p->left_off[F], n_r = p->right_off[F];
  int max_r = 0;
  for (int f = 0; f < F; f++) max_r = std::max(max_r, p->right_off[f + 1] - p->right_off[f]);
  LLD_ARG(c, max_r <= 65535);
  // octaves index scale / rows / cols / stride and pyr_off on the device
  for (int i = 0; i < n_l; i++) LLD_ARG(c, p->left_octave[i] < p->n_levels);
  for (int i = 0; i < n_r; i++) LLD_ARG(c, p->right_octave[i] < p->n_levels);
  if (int r = lld_call_begin(c, true)) return r;
  StereoView v{};
  v.n_frames = F; v.n_levels = p->n_levels; v.mb = p->mb; v.mbf = p->mbf;
  for (int l = 0; l < p->n_levels; l++) {
    v.scale[l] = p->scale_factors[l]; v.inv_scale[l] = p->inv_scale_factors[l];
    v.rows[l] = p->pyr_rows[l]; v.cols[l] = p->pyr_cols[l]; v.stride[l] = p->pyr_stride[l];
  }
  // row-band lists: a keypoint covers at most 2 * ceil(2 * scale_max) + 2 rows
  float smax = 1.f;
  for (int l = 0; l < p->n_levels; l++) smax = std::max(smax, p->scale_factors[l]);
  v.list_cap = std::max(1, max_r) * (2 * (int)std::ceil(2.0f * smax) + 3);
  LLD_UP(c, v.l_off, p->left_off, F + 1);
  LLD_UP(c, v.r_off, p->right_off, F + 1);
  LLD_UP(c, v.l_xy, p->left_xy, 2 * (size_t)n_l);
  LLD_UP(c, v.l_oct, p->left_octave, n_l);
  LLD_UP(c, v.l_desc, p->left_desc, 32 * (size_t)n_l);
  LLD_UP(c, v.r_xy, p->right_xy, 2 * (size_t)n_r);
  LLD_UP(c, v.r_oct, p->right_octave, n_r);
  LLD_UP(c, v.r_desc, p->right_desc, 32 * (size_t)n_r);
  LLD_UP(c, v.pyr, p->pyr, (size_t)p->pyr_bytes);
  LLD_UP(c, v.pyr_off, reinterpret_cast<const long long*>(p->pyr_off), (size_t)F * 2 * p->n_levels);
  LLD_DEV(c, v.row_start, (size_t)F * (v.rows[0] + 1));
  LLD_DEV(c, v.row_list, (size_t)F * v.list_cap);
  LLD_DEV(c, v.best_r, n_l);
  LLD_DEV(c, v.sad, n_l);
  LLD_DEV(c, v.uright, n_l);
  LLD_DEV(c, v.depth, n_l);
  LLD_DEV(c, v.n_matched, F);
  LLD_DEV(c, v.overflow, 1);
  LLD_CUDA(c, cudaMemsetAsync(v.overflow, 0, 4, c->stream));
  LLD_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
  LLD_LAUNCH(c, k_stereo, F, ST_NT, 0, v);
  LLD_CUDA(c, cudaGetLastError());
  LLD_CUDA(c, cudaEventRecord(c->ev[2], c->stream));
  int* h_over = reinterpret_cast<int*>(c->pinned);
  LLD_DOWN(c, out->uright, v.uright, n_l);
  LLD_DOWN(c, out->depth, v.depth, n_l);
  LLD_DOWN(c, out->n_matched, v.n_matched, F);
  LLD_DOWN(c, h_over, v.overflow, 1);
  if (int r = lld_call_end(c)) return r;
  if (*h_over) {
    snprintf(c->err, sizeof(c->err), "stereo matching: row-band list capacity exceeded");
    return LLD_ERR_UNSUPPORTED;
  }
  return LLD_OK;
}
