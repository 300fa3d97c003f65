// medoid.cu — distinctive (medoid) descriptor of map points / map lines for a batch of landmarks.
//
// MapPoint::ComputeDistinctiveDescriptors (src/MapPoint.cc:242-307): all-pairs 256-bit Hamming distances of the landmark's
// observed ORB descriptors, per descriptor the median distance to the others (element (int)(0.5 (N-1)) of the sorted row),
// the descriptor with the least median wins (strict <: the first one on a tie).
// MapLine::ComputeDistinctiveDescriptors (src/MapLine.cc:133-201): the same with float descriptors and the L2 norm
// cv::norm(a - b) (float difference, squares summed in double), the distance stored as float and the median TRUNCATED to
// int before the comparison (`int median = vDists[...]`).
// One warp per landmark.  Row i: lane j holds d(i, j), j = lane, lane + 32, ...; the k-th order statistic of the row is
// found by bisection on the value with ballot-free warp counts (distances are small non-negative integers after the
// reference's truncation; truncation is monotone, so the k-th smallest truncated value is the truncated k-th smallest).
#include <climits>

#include "lld_ctx.h"

namespace {

constexpr int MD_MAXC = 8;   // descriptors per lane: landmarks with up to 256 observations

__device__ __forceinline__ int warp_sum_i(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ int warp_max_i(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// k-th smallest (0-based) of the N values held as val[c] for element lane + 32 c
__device__ __forceinline__ int warp_select(const int* val, int N, int k, int lane) {
  int hi = 0;
#pragma unroll
  for (int c = 0; c < MD_MAXC; c++)
    if (lane + 32 * c < N) hi = max(hi, val[c]);
  hi = warp_max_i(hi);
  int lo = 0;   // smallest v with #{x <= v} >= k + 1
  while (lo < hi) {
    const int mid = lo + (hi - lo) / 2;
    int cnt = 0;
#pragma unroll
    for (int c = 0; c < MD_MAXC; c++)
      if (lane + 32 * c < N && val[c] <= mid) cnt++;
    cnt = warp_sum_i(cnt);
    if (cnt >= k + 1) hi = mid;
    else lo = mid + 1;
  }
  return lo;
}

__global__ void __launch_bounds__(256) k_medoid_orb(int n_lm, const int* __restrict__ off, const uint8_t* __restrict__ desc, int* __restrict__ best) {
  const int l = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (l >= n_lm) return;
  const int o0 = off[l], N = off[l + 1] - o0;
  if (N <= 0) {
    if (lane == 0) best[l] = -1;
    return;
  }
  const int k = (int)(0.5 * (N - 1));
  uint4 mine[MD_MAXC][2];
#pragma unroll
  for (int c = 0; c < MD_MAXC; c++) {
    const int j = lane + 32 * c;
    if (j < N) {
      const uint4* p = reinterpret_cast<const uint4*>(desc + 32 * (size_t)(o0 + j));
      mine[c][0] = p[0]; mine[c][1] = p[1];
    } else {
      mine[c][0] = mine[c][1] = make_uint4(0, 0, 0, 0);
    }
  }
  int bestMedian = INT_MAX, bestIdx = 0;
  for (int i = 0; i < N; i++) {
    const uint4* p = reinterpret_cast<const uint4*>(desc + 32 * (size_t)(o0 + i));
    const uint4 a0 = p[0], a1 = p[1];
    int val[MD_MAXC];
#pragma unroll
    for (int c = 0; c < MD_MAXC; c++)
      val[c] = __popc(a0.x ^ mine[c][0].x) + __popc(a0.y ^ mine[c][0].y) + __popc(a0.z ^ mine[c][0].z) + __popc(a0.w ^ mine[c][0].w) +
               __popc(a1.x ^ mine[c][1].x) + __popc(a1.y ^ mine[c][1].y) + __popc(a1.z ^ mine[c][1].z) + __popc(a1.w ^ mine[c][1].w);
    const int median = warp_select(val, N, k, lane);
    if (median < bestMedian) { bestMedian = median; bestIdx = i; }
  }
  if (lane == 0) best[l] = bestIdx;
}

__global__ void __launch_bounds__(256) k_medoid_float(int n_lm, const int* __restrict__ off, int D, const float* __restrict__ desc,
                                                        int* __restrict__ best) {
  const int l = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (l >= n_lm) return;
  const int o0 = off[l], N = off[l + 1] - o0;
  if (N <= 0) {
    if (lane == 0) best[l] = -1;
    return;
  }
  const int k = (int)(0.5 * (N - 1));
  int bestMedian = INT_MAX, bestIdx = 0;
  for (int i = 0; i < N; i++) {
    const float* a = desc + (size_t)D * (o0 + i);
    int val[MD_MAXC];
#pragma unroll
    for (int c = 0; c < MD_MAXC; c++) {
      const int j = lane + 32 * c;
      val[c] = 0;
      if (j < N && j != i) {
        const float* b = desc + (size_t)D * (o0 + j);
        double s = 0;
        for (int q = 0; q < D; q++) {
          const float df = __fsub_rn(a[q], b[q]);
          s = __dadd_rn(s, __dmul_rn((double)df, (double)df));   // the reference's summation order, no contraction
        }
        val[c] = (int)(float)sqrt(s);
      }
    }
    const int median = warp_select(val, N, k, lane);
    if (median < bestMedian) { bestMedian = median; bestIdx = i; }
  }
  if (lane == 0) best[l] = bestIdx;
}

}  // namespace

static int medoid_common(LldCtx* c, int n_lm, const int32_t* off, const void* desc, size_t row_bytes, int D, int32_t* best) {
  LLD_ARG(c, n_lm >= 1 && off && best);
  if (int r = lld_call_begin(c, true)) return r;
  const int n = off[n_lm];
  for (int l = 0; l < n_lm; l++)
    if (off[l + 1] - off[l] > 32 * MD_MAXC) {
      snprintf(c->err, sizeof(c->err), "medoid descriptor: a landmark has %d observations, at most %d are supported", off[l + 1] - off[l], 32 * MD_MAXC);
      return LLD_ERR_UNSUPPORTED;
    }
  const int* d_off;
  const uint8_t* d_desc;
  int* d_best;
  LLD_UP(c, d_off, off, n_lm + 1);
  LLD_UP(c, d_desc, static_cast<const uint8_t*>(desc), row_bytes * (size_t)n);
  LLD_DEV(c, d_best, n_lm);
  LLD_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
  const int grid = (n_lm + 7) / 8;
  if (D == 0) LLD_LAUNCH(c, k_medoid_orb, grid, 256, 0, n_lm, d_off, d_desc, d_best);
  else LLD_LAUNCH(c, k_medoid_float, grid, 256, 0, n_lm, d_off, D, reinterpret_cast<const float*>(d_desc), d_best);
  LLD_CUDA(c, cudaGetLastError());
  LLD_CUDA(c, cudaEventRecord(c->ev[2], c->stream));
  LLD_DOWN(c, best, d_best, n_lm);
  return lld_call_end(c);
}

extern "C" int lld_medoid_orb(void* ctx, int32_t n_lm, const int32_t* off, const uint8_t* desc, int32_t* best) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c) return LLD_ERR_ARG;
  return medoid_common(c, n_lm, off, desc, 32, 0, best);
}

extern "C" int lld_medoid_float(void* ctx, int32_t n_lm, const int32_t* off, int32_t D, const float* desc, int32_t* best) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c) return LLD_ERR_ARG;
  LLD_ARG(c, D >= 1);
  return medoid_common(c, n_lm, off, desc, 4 * (size_t)D, D, best);
}
