// orb_common.cuh — device pieces every ORBmatcher search shares: DescriptorDistance on 256-bit descriptors, the rotation
// histogram bin and ORBmatcher::ComputeThreeMaxima (src/ORBmatcher.cc:1601-1642).  Float arithmetic with explicit
// round-to-nearest intrinsics; the including units compile with --fmad=false.
#pragma once
#include <cuda_runtime.h>

constexpr int HISTO_LENGTH = 30;

__device__ __forceinline__ int popc256(const uint4& a0, const uint4& a1, const uint4& b0, const uint4& b1) {
  return __popc(a0.x ^ b0.x) + __popc(a0.y ^ b0.y) + __popc(a0.z ^ b0.z) + __popc(a0.w ^ b0.w) + __popc(a1.x ^ b1.x) +
         __popc(a1.y ^ b1.y) + __popc(a1.z ^ b1.z) + __popc(a1.w ^ b1.w);
}

// rot = angle1 - angle2 (+360 when negative); bin = round(rot * (1/HISTO_LENGTH)), HISTO_LENGTH wraps to 0
__device__ __forceinline__ int rot_bin(float angle1, float angle2) {
  float rot = __fsub_rn(angle1, angle2);
  if (rot < 0.0f) rot = __fadd_rn(rot, 360.0f);
  int bin = (int)roundf(__fmul_rn(rot, 1.0f / HISTO_LENGTH));
  if (bin == HISTO_LENGTH) bin = 0;
  return bin;
}

// ORBmatcher::ComputeThreeMaxima over hist[HISTO_LENGTH]: keep[0..2] = the bins that survive (-1 = none)
__device__ __forceinline__ void three_maxima(const int* hist, int* keep) {
  int max1 = 0, max2 = 0, max3 = 0, ind1 = -1, ind2 = -1, ind3 = -1;
  for (int i = 0; i < HISTO_LENGTH; i++) {
    const int s = hist[i];
    if (s > max1) { max3 = max2; max2 = max1; max1 = s; ind3 = ind2; ind2 = ind1; ind1 = i; }
    else if (s > max2) { max3 = max2; max2 = s; ind3 = ind2; ind2 = i; }
    else if (s > max3) { max3 = s; ind3 = i; }
  }
  if ((float)max2 < 0.1f * (float)max1) { ind2 = -1; ind3 = -1; }
  else if ((float)max3 < 0.1f * (float)max1) { ind3 = -1; }
  keep[0] = ind1; keep[1] = ind2; keep[2] = ind3;
}
