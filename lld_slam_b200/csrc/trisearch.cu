// trisearch.cu — ORBmatcher::SearchForTriangulation (src/ORBmatcher.cc:657-823) with CheckDistEpipolarLine (:140-157), batched
// over keyframe pairs.
//
// The reference walks the two DBoW2 feature vectors in step and compares the keypoints of a common vocabulary node all against
// all.  It never sets vbMatched2, so the keypoints of keyframe 1 are independent of each other: one thread per feature-vector entry
// of keyframe 1 finds the node in keyframe 2's (sorted) node list by bisection and scans that bucket in order with the
// reference's rules -- candidates with a map point or (bOnlyStereo) without a right coordinate are skipped, dist <= TH_LOW and
// dist <= best so far (so the LAST of equal distances wins), the epipole-distance test for monocular pairs and the epipolar-line
// test decide -- then the CTA applies the rotation-histogram filter (ComputeThreeMaxima, :1601-1642).  One CTA per keyframe pair.
// Float arithmetic in the reference's operation order, no FMA contraction (--fmad=false), comparisons against double products
// where the reference has them: vMatches12 is bit-exact against the CPU path.
#include <algorithm>

#include "lld_ctx.h"
#include "orb_common.cuh"

namespace {

constexpr int TH_LOW = 50, TS_NT = 256;

struct TriView {
  lld_tri_search_problem p;   // device pointers
  int* match12;
  int* n_matches;
};

__global__ void __launch_bounds__(TS_NT) k_tri_search(TriView v) {
  __shared__ int s_hist[HISTO_LENGTH];
  __shared__ int s_keep[3];
  __shared__ int s_n;
  const lld_tri_search_problem& p = v.p;
  const int pr = blockIdx.x, tid = threadIdx.x;
  const int a0 = p.kp1_off[pr], n1 = p.kp1_off[pr + 1] - a0;
  const int b0 = p.kp2_off[pr];
  const int f1b = p.fv1_node_off[pr], f1e = p.fv1_node_off[pr + 1];
  const int f2b = p.fv2_node_off[pr], f2e = p.fv2_node_off[pr + 1];
  const float* F12 = p.F12 + 9 * (size_t)pr;
  const float ex = p.epipole[2 * pr], ey = p.epipole[2 * pr + 1];
  if (tid < HISTO_LENGTH) s_hist[tid] = 0;
  if (tid == 0) s_n = 0;
  for (int i = tid; i < n1; i += TS_NT) v.match12[a0 + i] = -1;
  __syncthreads();
  // entries of keyframe 1's feature vector: [fv1_idx_off[f1b], fv1_idx_off[f1e])
  const int e_begin = f1b < f1e ? p.fv1_idx_off[f1b] : 0, e_end = f1b < f1e ? p.fv1_idx_off[f1e] : 0;
  for (int e = e_begin + tid; e < e_end; e += TS_NT) {
    const int idx1 = p.fv1_idx[e];
    if (p.kp1_has_mp[a0 + idx1]) continue;
    const bool bStereo1 = p.kp1_uright[a0 + idx1] >= 0;
    if (p.only_stereo && !bStereo1) continue;
    // node of this entry: last f with fv1_idx_off[f] <= e
    int lo = f1b, hi = f1e;
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (p.fv1_idx_off[mid] <= e) lo = mid;
      else hi = mid;
    }
    const int node = p.fv1_node[lo];
    // the same node in keyframe 2 (node ids ascending)
    int l2 = f2b, h2 = f2e;
    while (l2 < h2) {
      const int mid = (l2 + h2) >> 1;
      if (p.fv2_node[mid] < node) l2 = mid + 1;
      else h2 = mid;
    }
    if (l2 >= f2e || p.fv2_node[l2] != node) continue;
    const float k1x = p.kp1_xy[2 * (size_t)(a0 + idx1)], k1y = p.kp1_xy[2 * (size_t)(a0 + idx1) + 1];
    // epipolar line in the second image l = x1' F12 = [a b c]   (:143-145)
    const float a = __fadd_rn(__fadd_rn(__fmul_rn(k1x, F12[0]), __fmul_rn(k1y, F12[3])), F12[6]);
    const float b = __fadd_rn(__fadd_rn(__fmul_rn(k1x, F12[1]), __fmul_rn(k1y, F12[4])), F12[7]);
    const float c = __fadd_rn(__fadd_rn(__fmul_rn(k1x, F12[2]), __fmul_rn(k1y, F12[5])), F12[8]);
    const float den = __fadd_rn(__fmul_rn(a, a), __fmul_rn(b, b));
    const uint4* d1 = reinterpret_cast<const uint4*>(p.kp1_desc + 32 * (size_t)(a0 + idx1));
    const uint4 q0 = d1[0], q1 = d1[1];
    int bestDist = TH_LOW, bestIdx2 = -1;
    for (int i2 = p.fv2_idx_off[l2]; i2 < p.fv2_idx_off[l2 + 1]; i2++) {
      const int idx2 = p.fv2_idx[i2];
      if (p.kp2_has_mp[b0 + idx2]) continue;
      const bool bStereo2 = p.kp2_uright[b0 + idx2] >= 0;
      if (p.only_stereo && !bStereo2) continue;
      const uint4* d2 = reinterpret_cast<const uint4*>(p.kp2_desc + 32 * (size_t)(b0 + idx2));
      const int dist = popc256(q0, q1, d2[0], d2[1]);
      if (dist > TH_LOW || dist > bestDist) continue;
      const float k2x = p.kp2_xy[2 * (size_t)(b0 + idx2)], k2y = p.kp2_xy[2 * (size_t)(b0 + idx2) + 1];
      const int oct2 = p.kp2_octave[b0 + idx2];
      if (!bStereo1 && !bStereo2) {
        const float distex = __fsub_rn(ex, k2x), distey = __fsub_rn(ey, k2y);
        if (__fadd_rn(__fmul_rn(distex, distex), __fmul_rn(distey, distey)) < __fmul_rn(100.f, p.scale_factors[oct2])) continue;
      }
      const float num = __fadd_rn(__fadd_rn(__fmul_rn(a, k2x), __fmul_rn(b, k2y)), c);
      if (den == 0) continue;
      const float dsqr = __fdiv_rn(__fmul_rn(num, num), den);
      if ((double)dsqr < 3.84 * (double)p.level_sigma2[oct2]) { bestIdx2 = idx2; bestDist = dist; }
    }
    if (bestIdx2 >= 0) {
      v.match12[a0 + idx1] = bestIdx2;
      atomicAdd(&s_n, 1);
      if (p.check_orientation) {
        const int bin = rot_bin(p.kp1_angle[a0 + idx1], p.kp2_angle[b0 + bestIdx2]);
        atomicAdd(&s_hist[bin], 1);
      }
    }
  }
  __syncthreads();
  if (p.check_orientation) {
    if (tid == 0) three_maxima(s_hist, s_keep);
    __syncthreads();
    for (int i = tid; i < n1; i += TS_NT) {
      const int m = v.match12[a0 + i];
      if (m < 0) continue;
      const int bin = rot_bin(p.kp1_angle[a0 + i], p.kp2_angle[b0 + m]);
      if (bin != s_keep[0] && bin != s_keep[1] && bin != s_keep[2]) {
        v.match12[a0 + i] = -1;
        atomicSub(&s_n, 1);
      }
    }
    __syncthreads();
  }
  if (tid == 0) v.n_matches[pr] = s_n;
}

// ORBmatcher::SearchByBoW (src/ORBmatcher.cc:159-288, :522-655): one thread per vocabulary node of side 1.  The claims
// (vpMapPointMatches[realIdxF] / vbMatched2[idx2]) only ever concern keypoints of the same node -- a keypoint belongs to exactly
// one node -- so a thread that walks its node's side-1 entries in order, each against the node's side-2 bucket in order, reproduces
// the reference's sequential result without any exchange between threads.
struct BowView {
  lld_bow_search_problem p;   // device pointers
  int* match12;
  int* n_matches;
  uint8_t* matched2;          // [n2] zeroed
};

__global__ void __launch_bounds__(TS_NT) k_bow_search(BowView v) {
  __shared__ int s_hist[HISTO_LENGTH];
  __shared__ int s_keep[3];
  __shared__ int s_n;
  const lld_bow_search_problem& p = v.p;
  const int pr = blockIdx.x, tid = threadIdx.x;
  const int a0 = p.kp1_off[pr], n1 = p.kp1_off[pr + 1] - a0;
  const int b0 = p.kp2_off[pr];
  const int f1b = p.fv1_node_off[pr], f1e = p.fv1_node_off[pr + 1];
  const int f2b = p.fv2_node_off[pr], f2e = p.fv2_node_off[pr + 1];
  if (tid < HISTO_LENGTH) s_hist[tid] = 0;
  if (tid == 0) s_n = 0;
  for (int i = tid; i < n1; i += TS_NT) v.match12[a0 + i] = -1;
  __syncthreads();
  for (int f1 = f1b + tid; f1 < f1e; f1 += TS_NT) {
    const int node = p.fv1_node[f1];
    int l2 = f2b, h2 = f2e;
    while (l2 < h2) {
      const int mid = (l2 + h2) >> 1;
      if (p.fv2_node[mid] < node) l2 = mid + 1;
      else h2 = mid;
    }
    if (l2 >= f2e || p.fv2_node[l2] != node) continue;
    const int s2b = p.fv2_idx_off[l2], s2e = p.fv2_idx_off[l2 + 1];
    for (int i1 = p.fv1_idx_off[f1]; i1 < p.fv1_idx_off[f1 + 1]; i1++) {
      const int idx1 = p.fv1_idx[i1];
      if (!p.kp1_valid[a0 + idx1]) continue;
      const uint4* d1 = reinterpret_cast<const uint4*>(p.kp1_desc + 32 * (size_t)(a0 + idx1));
      const uint4 q0 = d1[0], q1 = d1[1];
      int bestDist1 = 256, bestIdx2 = -1, bestDist2 = 256;
      for (int i2 = s2b; i2 < s2e; i2++) {
        const int idx2 = p.fv2_idx[i2];
        if (v.matched2[b0 + idx2] || !p.kp2_valid[b0 + idx2]) continue;
        const uint4* d2 = reinterpret_cast<const uint4*>(p.kp2_desc + 32 * (size_t)(b0 + idx2));
        const int dist = popc256(q0, q1, d2[0], d2[1]);
        if (dist < bestDist1) { bestDist2 = bestDist1; bestDist1 = dist; bestIdx2 = idx2; }
        else if (dist < bestDist2) bestDist2 = dist;
      }
      if (!(p.strict_th ? bestDist1 < TH_LOW : bestDist1 <= TH_LOW)) continue;
      if (!((float)bestDist1 < __fmul_rn(p.nn_ratio, (float)bestDist2))) continue;
      v.match12[a0 + idx1] = bestIdx2;
      v.matched2[b0 + bestIdx2] = 1;          // read again only by this thread (same node)
      atomicAdd(&s_n, 1);
      if (p.check_orientation) {
        const int bin = rot_bin(p.kp1_angle[a0 + idx1], p.kp2_angle[b0 + bestIdx2]);
        atomicAdd(&s_hist[bin], 1);
      }
    }
  }
  __syncthreads();
  if (p.check_orientation) {
    if (tid == 0) three_maxima(s_hist, s_keep);
    __syncthreads();
    for (int i = tid; i < n1; i += TS_NT) {
      const int m = v.match12[a0 + i];
      if (m < 0) continue;
      const int bin = rot_bin(p.kp1_angle[a0 + i], p.kp2_angle[b0 + m]);
      if (bin != s_keep[0] && bin != s_keep[1] && bin != s_keep[2]) {
        v.match12[a0 + i] = -1;
        atomicSub(&s_n, 1);
      }
    }
    __syncthreads();
  }
  if (tid == 0) v.n_matches[pr] = s_n;
}

}  // namespace

extern "C" int lld_bow_search(void* ctx, const lld_bow_search_problem* p, lld_tri_search_result* out) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !p || !out) return LLD_ERR_ARG;
  LLD_ARG(c, p->n_pairs >= 1);
  LLD_CUDA(c, cudaSetDevice(c->device));
  c->launches = 0;
  c->pool_reset();
  const int P = p->n_pairs, n1 = p->kp1_off[P], n2 = p->kp2_off[P];
  const int nn1 = p->fv1_node_off[P], nn2 = p->fv2_node_off[P];
  const int ne1 = nn1 ? p->fv1_idx_off[nn1] : 0, ne2 = nn2 ? p->fv2_idx_off[nn2] : 0;
  cudaError_t e = cudaSuccess;
  auto up = [&](const void* src, size_t bytes) -> void* {
    if (e != cudaSuccess) return nullptr;
    uint8_t* d = c->alloc<uint8_t>(bytes ? bytes : 1, &e);
    if (e == cudaSuccess && bytes) e = cudaMemcpyAsync(d, src, bytes, cudaMemcpyHostToDevice, c->stream);
    return d;
  };
  BowView v{};
  v.p = *p;
  LLD_CUDA(c, cudaEventRecord(c->ev[0], c->stream));
  v.p.kp1_off = (const int32_t*)up(p->kp1_off, 4 * (size_t)(P + 1));
  v.p.kp1_angle = (const float*)up(p->kp1_angle, 4 * (size_t)n1);
  v.p.kp1_valid = (const uint8_t*)up(p->kp1_valid, (size_t)n1);
  v.p.kp1_desc = (const uint8_t*)up(p->kp1_desc, 32 * (size_t)n1);
  v.p.kp2_off = (const int32_t*)up(p->kp2_off, 4 * (size_t)(P + 1));
  v.p.kp2_angle = (const float*)up(p->kp2_angle, 4 * (size_t)n2);
  v.p.kp2_valid = (const uint8_t*)up(p->kp2_valid, (size_t)n2);
  v.p.kp2_desc = (const uint8_t*)up(p->kp2_desc, 32 * (size_t)n2);
  v.p.fv1_node_off = (const int32_t*)up(p->fv1_node_off, 4 * (size_t)(P + 1));
  v.p.fv1_node = (const int32_t*)up(p->fv1_node, 4 * (size_t)nn1);
  v.p.fv1_idx_off = (const int32_t*)up(p->fv1_idx_off, 4 * (size_t)(nn1 + 1));
  v.p.fv1_idx = (const int32_t*)up(p->fv1_idx, 4 * (size_t)ne1);
  v.p.fv2_node_off = (const int32_t*)up(p->fv2_node_off, 4 * (size_t)(P + 1));
  v.p.fv2_node = (const int32_t*)up(p->fv2_node, 4 * (size_t)nn2);
  v.p.fv2_idx_off = (const int32_t*)up(p->fv2_idx_off, 4 * (size_t)(nn2 + 1));
  v.p.fv2_idx = (const int32_t*)up(p->fv2_idx, 4 * (size_t)ne2);
  if (e == cudaSuccess) v.match12 = c->alloc<int>((size_t)std::max(n1, 1), &e);
  if (e == cudaSuccess) v.n_matches = c->alloc<int>((size_t)P, &e);
  if (e == cudaSuccess) v.matched2 = c->alloc<uint8_t>((size_t)std::max(n2, 1), &e);
  LLD_CUDA(c, e);
  LLD_CUDA(c, cudaMemsetAsync(v.matched2, 0, (size_t)std::max(n2, 1), c->stream));
  LLD_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
  LLD_LAUNCH(c, k_bow_search, P, TS_NT, 0, v);
  LLD_CUDA(c, cudaGetLastError());
  LLD_CUDA(c, cudaEventRecord(c->ev[2], c->stream));
  if (n1) LLD_CUDA(c, cudaMemcpyAsync(out->match12, v.match12, 4 * (size_t)n1, cudaMemcpyDeviceToHost, c->stream));
  LLD_CUDA(c, cudaMemcpyAsync(out->n_matches, v.n_matches, 4 * (size_t)P, cudaMemcpyDeviceToHost, c->stream));
  LLD_CUDA(c, cudaEventRecord(c->ev[3], c->stream));
  LLD_CUDA(c, cudaStreamSynchronize(c->stream));
  cudaEventElapsedTime(&c->ms_h2d, c->ev[0], c->ev[1]);
  cudaEventElapsedTime(&c->ms_compute, c->ev[1], c->ev[2]);
  cudaEventElapsedTime(&c->ms_d2h, c->ev[2], c->ev[3]);
  return LLD_OK;
}

extern "C" int lld_tri_search(void* ctx, const lld_tri_search_problem* p, lld_tri_search_result* out) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !p || !out) return LLD_ERR_ARG;
  LLD_ARG(c, p->n_pairs >= 1 && p->n_levels >= 1 && p->n_levels <= 8);
  LLD_CUDA(c, cudaSetDevice(c->device));
  c->launches = 0;
  c->pool_reset();
  const int P = p->n_pairs, n1 = p->kp1_off[P], n2 = p->kp2_off[P];
  const int nn1 = p->fv1_node_off[P], nn2 = p->fv2_node_off[P];
  const int ne1 = nn1 ? p->fv1_idx_off[nn1] : 0, ne2 = nn2 ? p->fv2_idx_off[nn2] : 0;
  cudaError_t e = cudaSuccess;
  auto up = [&](const void* src, size_t bytes) -> void* {
    if (e != cudaSuccess) return nullptr;
    uint8_t* d = c->alloc<uint8_t>(bytes ? bytes : 1, &e);
    if (e == cudaSuccess && bytes) e = cudaMemcpyAsync(d, src, bytes, cudaMemcpyHostToDevice, c->stream);
    return d;
  };
  TriView v{};
  v.p = *p;
  LLD_CUDA(c, cudaEventRecord(c->ev[0], c->stream));
  v.p.F12 = (const float*)up(p->F12, 36 * (size_t)P);
  v.p.epipole = (const float*)up(p->epipole, 8 * (size_t)P);
  v.p.kp1_off = (const int32_t*)up(p->kp1_off, 4 * (size_t)(P + 1));
  v.p.kp1_xy = (const float*)up(p->kp1_xy, 8 * (size_t)n1);
  v.p.kp1_angle = (const float*)up(p->kp1_angle, 4 * (size_t)n1);
  v.p.kp1_uright = (const float*)up(p->kp1_uright, 4 * (size_t)n1);
  v.p.kp1_has_mp = (const uint8_t*)up(p->kp1_has_mp, (size_t)n1);
  v.p.kp1_desc = (const uint8_t*)up(p->kp1_desc, 32 * (size_t)n1);
  v.p.kp2_off = (const int32_t*)up(p->kp2_off, 4 * (size_t)(P + 1));
  v.p.kp2_xy = (const float*)up(p->kp2_xy, 8 * (size_t)n2);
  v.p.kp2_octave = (const uint8_t*)up(p->kp2_octave, (size_t)n2);
  v.p.kp2_angle = (const float*)up(p->kp2_angle, 4 * (size_t)n2);
  v.p.kp2_uright = (const float*)up(p->kp2_uright, 4 * (size_t)n2);
  v.p.kp2_has_mp = (const uint8_t*)up(p->kp2_has_mp, (size_t)n2);
  v.p.kp2_desc = (const uint8_t*)up(p->kp2_desc, 32 * (size_t)n2);
  v.p.fv1_node_off = (const int32_t*)up(p->fv1_node_off, 4 * (size_t)(P + 1));
  v.p.fv1_node = (const int32_t*)up(p->fv1_node, 4 * (size_t)nn1);
  v.p.fv1_idx_off = (const int32_t*)up(p->fv1_idx_off, 4 * (size_t)(nn1 + 1));
  v.p.fv1_idx = (const int32_t*)up(p->fv1_idx, 4 * (size_t)ne1);
  v.p.fv2_node_off = (const int32_t*)up(p->fv2_node_off, 4 * (size_t)(P + 1));
  v.p.fv2_node = (const int32_t*)up(p->fv2_node, 4 * (size_t)nn2);
  v.p.fv2_idx_off = (const int32_t*)up(p->fv2_idx_off, 4 * (size_t)(nn2 + 1));
  v.p.fv2_idx = (const int32_t*)up(p->fv2_idx, 4 * (size_t)ne2);
  if (e == cudaSuccess) v.match12 = c->alloc<int>((size_t)std::max(n1, 1), &e);
  if (e == cudaSuccess) v.n_matches = c->alloc<int>((size_t)P, &e);
  LLD_CUDA(c, e);
  LLD_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
  LLD_LAUNCH(c, k_tri_search, P, TS_NT, 0, v);
  LLD_CUDA(c, cudaGetLastError());
  LLD_CUDA(c, cudaEventRecord(c->ev[2], c->stream));
  if (n1) LLD_CUDA(c, cudaMemcpyAsync(out->match12, v.match12, 4 * (size_t)n1, cudaMemcpyDeviceToHost, c->stream));
  LLD_CUDA(c, cudaMemcpyAsync(out->n_matches, v.n_matches, 4 * (size_t)P, cudaMemcpyDeviceToHost, c->stream));
  LLD_CUDA(c, cudaEventRecord(c->ev[3], c->stream));
  LLD_CUDA(c, cudaStreamSynchronize(c->stream));
  cudaEventElapsedTime(&c->ms_h2d, c->ev[0], c->ev[1]);
  cudaEventElapsedTime(&c->ms_compute, c->ev[1], c->ev[2]);
  cudaEventElapsedTime(&c->ms_d2h, c->ev[2], c->ev[3]);
  return LLD_OK;
}
