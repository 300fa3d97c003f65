// linematch.cu — stereo line matching with float line descriptors (TwoFrameLineMatcher::MatchLines).
//
// Reference: src/TwoFrameLineMatcher.cc:26-124 with vgl::TriangulateLine (src/vgl.cc:78-108),
// ReprojectKeyLineTo3D (src/LineMatching.cc:277-291), NormalizedLineEquation (src/vgl.cc:578-585).
// The descriptor distance LineMatcher::MatchLineDescriptors lives in the un-vendored LBDMOD library
// (un-vendored and unpinned, so parity is unpinned): defined here as the L2 norm of the float rows.
//
// Two device plans per batch: the tensor-core path further down (tcgen05, default: D multiple of 8 up to 72 floats and
// <= 512 lines per side of a pair) and the FP32 tile path for everything else:
//   k_line_prep   : per line, K^T-normalised image line equation, unit plane normal and pixel length
//   k_line_dist   : 32x32 tiles of the (left x right) pair matrix; descriptors staged in shared memory, dense
//                   ||a-b||^2 contraction in FP32, fused epilogue = the geometric gates of CheckLinePair
//                   (octave, length, triangulation angle, |X0|, endpoint depths) and the tau threshold;
//                   writes the masked distance matrix
//   k_line_greedy : one warp per pair replays the reference's sequential greedy assignment (left lines in index
//                   order, first minimum wins, matched right lines are removed)
// Tolerance (stated, because LBDMOD is unpinned): |d_gpu - d_oracle| <= 1e-5 * max(1, d); identical matches unless
// the two best candidates of a row are closer than that.  (The tensor-core path ranks by 3xTF32 distances, |error| ~ 1e-6
// in d^2, and reports exact FP32 distances.)
#include <cfloat>
#include <cstdlib>
#include <vector>
#include <algorithm>

#include "lld_ctx.h"
#include "lld_math.cuh"

using namespace lld;

namespace {

struct LineMatchView {
  int n_pairs, D;
  const int* left_off;
  const int* right_off;
  const float* left_seg;
  const int* left_oct;
  const float* right_seg;
  const int* right_oct;
  const float* left_desc;
  const float* right_desc;
  double K[9];
  double baseline, tau;
  int min_len;
  double* left_leq;   // [n_left][3]
  double* right_leq;
  double* left_len;
  double* right_len;
  double* left_un;    // [n_left][3] unit normal of the back-projection plane (leq / |leq|)
  double* right_un;
  const long long* mat_off;  // [n_pairs] offset of the pair's nl x nr matrix
  float* dist;        // masked distance matrix, +inf where a gate fails
  int* match;
  float* mdist;
};

// FP32 records of the second-generation tensor-core path (formed here, where the FP64 values are in registers)
struct LineRecs {
  float4* lrec;    // [n_left]  {|a|^2 (filled by k_line_prep2), unit plane normal}
  float4* rrec;    // [n_right] {|b|^2 (filled by k_line_prep2), unit plane normal}
  float* rh;       // [n_right] |X0| >= 1/2  <=>  parallax cosine >= rh
  int8_t* loct;    // [n_left]  octave, -2 when the line is too short
  int8_t* roct;    // [n_right] octave, -1 when the line is too short
  float4* rleq;    // [n_right] {K^T l normalised, beta = l_x * baseline}
  float4* lgeo;    // [n_left][7] {l1, |l1|^2}, {-, |a0|^2, |a1|^2, -}, M0 | M1 with M = [a]_x K per endpoint a
};
template <bool WITH_RECS>
__global__ void k_line_prep(LineMatchView v, LineRecs t, int n_left, int n_right) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  for (int side = 0; side < 2; side++) {
    const int n = side ? n_right : n_left;
    if (i >= n) continue;
    const float* s = (side ? v.right_seg : v.left_seg) + 4 * (size_t)i;
    const double Xs[3] = {s[0], s[1], 1.0}, Xe[3] = {s[2], s[3], 1.0};
    double li[3], leq[3];
    cross3(Xs, Xe, li);
#pragma unroll
    for (int k = 0; k < 3; k++) leq[k] = v.K[k] * li[0] + v.K[3 + k] * li[1] + v.K[6 + k] * li[2];  // K^T l
    const double n2 = sqrt(leq[0] * leq[0] + leq[1] * leq[1]);
    double* o = (side ? v.right_leq : v.left_leq) + 3 * (size_t)i;
    o[0] = leq[0] / n2; o[1] = leq[1] / n2; o[2] = leq[2] / n2;
    const double n3 = sqrt(o[0] * o[0] + o[1] * o[1] + o[2] * o[2]);
    double* u = (side ? v.right_un : v.left_un) + 3 * (size_t)i;
    u[0] = o[0] / n3; u[1] = o[1] / n3; u[2] = o[2] / n3;
    const double dx = (double)s[0] - (double)s[2], dy = (double)s[1] - (double)s[3];
    const double len = sqrt(dx * dx + dy * dy);
    (side ? v.right_len : v.left_len)[i] = len;
    if (WITH_RECS) {
      const bool too_short = len < (double)v.min_len;
      const int oct = min(max((side ? v.right_oct : v.left_oct)[i], 0), 127);
      const double l1sq = o[0] * o[0] + o[1] * o[1] + o[2] * o[2];
      if (side) {
        // |X0|^2 = beta^2 |l1|^2 / |l1 x l2|^2 and |l1 x l2|^2 = |l1|^2 |l2|^2 (1 - cs^2) with cs the cosine between the
        // unit normals: |X0| >= 1/2  <=>  cs^2 >= 1 - 4 beta^2 / |l2|^2, a per-right-line bound the selectors test for free
        const double beta = o[0] * v.baseline;
        float* rr = reinterpret_cast<float*>(t.rrec + i);
        rr[1] = (float)u[0]; rr[2] = (float)u[1]; rr[3] = (float)u[2];
        t.rh[i] = (float)sqrt(fmax(0.0, 1.0 - 4.0 * beta * beta / l1sq));
        t.roct[i] = (int8_t)(too_short ? -1 : oct);
        t.rleq[i] = make_float4((float)o[0], (float)o[1], (float)o[2], (float)beta);
      } else {
        float* lr = reinterpret_cast<float*>(t.lrec + i);
        lr[1] = (float)u[0]; lr[2] = (float)u[1]; lr[3] = (float)u[2];
        t.loct[i] = (int8_t)(too_short ? -2 : oct);
        float m[20], aa[2];
#pragma unroll
        for (int e = 0; e < 2; e++) {
          const double a[3] = {s[2 * e], s[2 * e + 1], 1.0};
          const double* K = v.K;
#pragma unroll
          for (int cc = 0; cc < 3; cc++) {   // [a]_x K, column cc
            m[9 * e + 0 + cc] = (float)(-a[2] * K[3 + cc] + a[1] * K[6 + cc]);
            m[9 * e + 3 + cc] = (float)(a[2] * K[cc] - a[0] * K[6 + cc]);
            m[9 * e + 6 + cc] = (float)(-a[1] * K[cc] + a[0] * K[3 + cc]);
          }
          aa[e] = (float)(a[0] * a[0] + a[1] * a[1] + 1.0);
        }
        m[18] = m[19] = 0.f;
        float4* g = t.lgeo + 7 * (size_t)i;
        g[0] = make_float4((float)o[0], (float)o[1], (float)o[2], (float)l1sq);
        g[1] = make_float4(0.f, aa[0], aa[1], 0.f);
#pragma unroll
        for (int k = 0; k < 5; k++) g[2 + k] = make_float4(m[4 * k], m[4 * k + 1], m[4 * k + 2], m[4 * k + 3]);
      }
    }
  }
}

// least squares [ (px,py,1) | -K d ] (depth, s) = K X0 -> s   (vgl::ReprojectLinePointTo3D)
__device__ __forceinline__ double reproject_param(const double* y, const double* c, double px, double py) {
  const double a[3] = {px, py, 1.0};
  const double aa = dot3(a, a), ac = dot3(a, c), cc = dot3(c, c), ay = dot3(a, y), cy = dot3(c, y);
  const double det = aa * cc - ac * ac;
  return (aa * cy - ac * ay) / det;
}

__device__ __forceinline__ bool line_pair_gate(const LineMatchView& v, const float* s1, const double* l1, const double* l2) {
  // vgl::TriangulateLine with T1 = [I|0], T2 = [I|(b,0,0)]
  const double n1n = sqrt(dot3(l1, l1)), n2n = sqrt(dot3(l2, l2));
  if (fabs(dot3(l1, l2)) / n1n / n2n > 0.975) return false;
  double dir[3];
  cross3(l1, l2, dir);
  const double dn = sqrt(dot3(dir, dir));
  dir[0] /= dn; dir[1] /= dn; dir[2] /= dn;
  // rows (n1, n2, dir), rhs (0, n2.t2, 0):  X0 = beta (dir x n1) / (n1 . (n2 x dir))
  const double beta = l2[0] * v.baseline;
  double c1[3], c2[3];
  cross3(dir, l1, c1);
  cross3(l2, dir, c2);
  const double det = dot3(l1, c2);
  if (!(fabs(det) > 0.0)) return false;
  const double X0[3] = {beta * c1[0] / det, beta * c1[1] / det, beta * c1[2] / det};
  if (sqrt(dot3(X0, X0)) < 0.5) return false;
  // ReprojectKeyLineTo3D with T = I: both endpoints must land at z >= 0
  const double* K = v.K;
  const double y[3] = {K[0] * X0[0] + K[1] * X0[1] + K[2] * X0[2], K[3] * X0[0] + K[4] * X0[1] + K[5] * X0[2],
                       K[6] * X0[0] + K[7] * X0[1] + K[8] * X0[2]};
  const double c[3] = {-(K[0] * dir[0] + K[1] * dir[1] + K[2] * dir[2]), -(K[3] * dir[0] + K[4] * dir[1] + K[5] * dir[2]),
                       -(K[6] * dir[0] + K[7] * dir[1] + K[8] * dir[2])};
  const double pa = reproject_param(y, c, s1[0], s1[1]);
  const double pb = reproject_param(y, c, s1[2], s1[3]);
  if (X0[2] + pa * dir[2] < 0 || X0[2] + pb * dir[2] < 0) return false;
  return true;
}

// The same gates for a pair that already passed the parallax test, without the normalisations that cancel out
// algebraically (X0 and the endpoint depths are homogeneous of degree 0 in |dir|; |X0| < 0.5 is tested squared):
// three FP64 divisions and no square root on the latency path of the sequential greedy.  Differs from
// line_pair_gate only in the last bits of the compared quantities.
__device__ __forceinline__ bool line_pair_gate_fast(const LineMatchView& v, const float* s1, const double* l1, const double* l2) {
  double dir[3];
  cross3(l1, l2, dir);
  const double beta = l2[0] * v.baseline;
  double c1[3], c2[3];
  cross3(dir, l1, c1);
  cross3(l2, dir, c2);
  const double det = dot3(l1, c2);
  if (!(fabs(det) > 0.0)) return false;
  const double f = beta / det;
  const double X0[3] = {f * c1[0], f * c1[1], f * c1[2]};
  if (dot3(X0, X0) < 0.25) return false;
  const double* K = v.K;
  const double y[3] = {K[0] * X0[0] + K[1] * X0[1] + K[2] * X0[2], K[3] * X0[0] + K[4] * X0[1] + K[5] * X0[2],
                       K[6] * X0[0] + K[7] * X0[1] + K[8] * X0[2]};
  const double c[3] = {-(K[0] * dir[0] + K[1] * dir[1] + K[2] * dir[2]), -(K[3] * dir[0] + K[4] * dir[1] + K[5] * dir[2]),
                       -(K[6] * dir[0] + K[7] * dir[1] + K[8] * dir[2])};
  const double pa = reproject_param(y, c, s1[0], s1[1]);
  const double pb = reproject_param(y, c, s1[2], s1[3]);
  if (X0[2] + pa * dir[2] < 0 || X0[2] + pb * dir[2] < 0) return false;
  return true;
}

constexpr int LT = 32;  // tile edge

// grid: (tiles_x * tiles_y summed over pairs) flattened through tile_pair / tile_row / tile_col tables
__global__ void __launch_bounds__(256) k_line_dist(LineMatchView v, const int* __restrict__ tile_pair,
                                                   const int* __restrict__ tile_r, const int* __restrict__ tile_c) {
  extern __shared__ float sm[];
  const int p = tile_pair[blockIdx.x];
  const int a0 = v.left_off[p], na = v.left_off[p + 1] - a0;
  const int b0 = v.right_off[p], nb = v.right_off[p + 1] - b0;
  const int r0 = tile_r[blockIdx.x] * LT, c0 = tile_c[blockIdx.x] * LT;
  const int D = v.D, ld = D + 1;
  float* sa = sm;
  float* sb = sm + LT * ld;
  for (int i = threadIdx.x; i < LT * D; i += blockDim.x) {
    const int r = i / D, k = i - r * D;
    sa[r * ld + k] = (r0 + r < na) ? v.left_desc[(size_t)(a0 + r0 + r) * D + k] : 0.f;
    sb[r * ld + k] = (c0 + r < nb) ? v.right_desc[(size_t)(b0 + c0 + r) * D + k] : 0.f;
  }
  __syncthreads();
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;  // 16 x 16 threads, 2 x 2 micro tile
  float acc[2][2] = {{0, 0}, {0, 0}};
  for (int k = 0; k < D; k++) {
    const float x0 = sa[(2 * ty) * ld + k], x1 = sa[(2 * ty + 1) * ld + k];
    const float y0 = sb[(2 * tx) * ld + k], y1 = sb[(2 * tx + 1) * ld + k];
    float d;
    d = x0 - y0; acc[0][0] = fmaf(d, d, acc[0][0]);
    d = x0 - y1; acc[0][1] = fmaf(d, d, acc[0][1]);
    d = x1 - y0; acc[1][0] = fmaf(d, d, acc[1][0]);
    d = x1 - y1; acc[1][1] = fmaf(d, d, acc[1][1]);
  }
  float* M = v.dist + v.mat_off[p];
#pragma unroll
  for (int i = 0; i < 2; i++)
#pragma unroll
    for (int j = 0; j < 2; j++) {
      const int r = r0 + 2 * ty + i, c = c0 + 2 * tx + j;
      if (r >= na || c >= nb) continue;
      float out = INFINITY;
      const float d = sqrtf(acc[i][j]);
      if (v.left_oct[a0 + r] == v.right_oct[b0 + c] && !(v.left_len[a0 + r] < (double)v.min_len) &&
          !(v.right_len[b0 + c] < (double)v.min_len) && (double)d < v.tau) {
        if (line_pair_gate(v, v.left_seg + 4 * (size_t)(a0 + r), v.left_leq + 3 * (size_t)(a0 + r),
                           v.right_leq + 3 * (size_t)(b0 + c)))
          out = d;
      }
      M[(size_t)r * nb + c] = out;
    }
}

// one warp per pair: sequential greedy over the left lines
__global__ void __launch_bounds__(32) k_line_greedy(LineMatchView v, int* taken_all, const long long* taken_off) {
  const int p = blockIdx.x;
  const int lane = threadIdx.x;
  const int a0 = v.left_off[p], na = v.left_off[p + 1] - a0;
  const int b0 = v.right_off[p], nb = v.right_off[p + 1] - b0;
  const float* M = v.dist + v.mat_off[p];
  int* taken = taken_all + taken_off[p];
  for (int c = lane; c < nb; c += 32) taken[c] = 0;
  __syncwarp();
  for (int j = 0; j < na; j++) {
    float best = INFINITY;
    int bi = -1;
    for (int c = lane; c < nb; c += 32) {
      const float d = M[(size_t)j * nb + c];
      if (d < best && !taken[c]) { best = d; bi = c; }  // strict <: first minimum within the lane's stride
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float od = __shfl_xor_sync(0xffffffffu, best, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (oi >= 0 && (od < best || (od == best && (bi < 0 || oi < bi)))) { best = od; bi = oi; }
    }
    if (lane == 0) {
      v.match[a0 + j] = bi;
      v.mdist[a0 + j] = bi >= 0 ? best : INFINITY;
      if (bi >= 0) taken[bi] = 1;
    }
    __syncwarp();
  }
}


// ---- tcgen05 / TMEM / mbarrier helpers of the tensor-core path
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
// UMMA shared-memory descriptor, K-major, no swizzle: 8 x 16 B core matrices; LBO = byte distance between the two
// 16 B K-chunks of one MMA, SBO = byte distance between 8-row groups (cute::UMMA::SmemDescriptor, version 1)
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) | (1ull << 46);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(0), "r"(0), "r"(0), "r"(0)
      : "memory");
}
// bounded wait: a tensor-core completion that never arrives is reported (err_flag) instead of hanging the device
__device__ __forceinline__ bool mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  for (int spin = 0; spin < (1 << 22); spin++) {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                 : "=r"(ok)
                 : "r"(bar), "r"(parity)
                 : "memory");
    if (ok) return true;
  }
  return false;
}
#define TMEM_LD32(r, taddr)                                                                                              \
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, " \
               "%15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"            \
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),          \
                 "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),    \
                 "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),  \
                 "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])   \
               : "r"(taddr))

// exact squared distance of one (left, right) pair by a warp (FP32, difference form)
__device__ __forceinline__ float warp_exact_d2(const float* a, const float* b, int D, int lane) {
  float s2 = 0.f;
  for (int k = lane; k < D; k += 32) {
    const float d = a[k] - b[k];
    s2 = fmaf(d, d, s2);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s2 += __shfl_xor_sync(0xffffffffu, s2, o);
  return s2;
}

// ================================================================================================
// Tensor-core path (sm_100a tcgen05, default): the left x right descriptor contraction as 3xTF32 UMMAs (a = a_hi + a_lo,
// a.b ~ a_hi.b_hi + a_hi.b_lo + a_lo.b_hi, fp32 accumulation in TMEM; |error| ~ 1e-6 in d^2) with the candidate
// selection fused into the TMEM epilogue.  One persistent CTA per SM walks over stereo pairs; inside it the work
// is split by warp role so that staging, tensor-core contraction and candidate selection of consecutive steps overlap:
//   producers (4 warps) : split the descriptors into TF32 hi / lo parts while staging them into the canonical K-major
//                         UMMA layout; one elected thread issues the 3xTF32 tcgen05.mma sequence of a step
//   selectors (16 warps): read the finished accumulator from TMEM and compact the survivors of the cheap gates
//   step = (chunk of NL left lines) x (block of 128 right lines); the accumulator is TRANSPOSED: TMEM lane = right line,
//   TMEM column = left line.  A selector thread therefore owns one right line (its |b|^2, unit normal, octave and |X0|
//   bound live in registers), a warp looks at 32 consecutive right lines of ONE left line at a time, and the survivors
//   of that left line are appended with a ballot + one shared-memory atomic per 32 lines: the stores of a warp land in
//   one or two 32 B sectors (a row-per-thread epilogue scatters 4-byte stores over 32 sectors and is bound by them).
//   Two accumulators (2 x 256 TMEM columns) are in flight.
//   k_line_prep2  : per line |d|^2 and FP32 copies of the geometry the selection and the gates read
//   k_line_tc2    : as above; candidate list per left line = (3xTF32 d^2, right line), any order
//   k_line_gate32 : the remaining gates of CheckLinePair over the lists.  Decided in FP32 with a running error bound;
//                   an entry closer to a threshold than the bound is decided by the FP64 formulas the FP32 tile path uses
//                   (LLD_LINE_CHECK=1 evaluates both for every entry and fails the call on a disagreement)
//   k_line_greedy2: one warp per pair, sequential over the left lines: smallest (d^2, right line) among the admissible
//                   untaken entries -- two warp reductions per line
//   k_line_exact2 : exact FP32 distance of each match
// ================================================================================================
constexpr int T2_M = 128;                 // right lines per block = TMEM lanes
constexpr int T2_ROWS = 512;              // lines per side of a pair at most
constexpr int T2_CAP = 256;               // candidate slots per left line
constexpr int T2_SEL_WARPS = 16, T2_PROD_WARPS = 4;
constexpr int T2_SEL = 32 * T2_SEL_WARPS, T2_PROD = 32 * T2_PROD_WARPS, T2_NT = T2_SEL + T2_PROD;

struct LineTc2View {
  LineMatchView v;
  int nl_chunk;             // left lines per step (256, or 128 for wide descriptors)
  LineRecs rc;              // FP32 geometry records (k_line_prep)
  uint2* cand;              // [n_left][T2_CAP] {float bits of the 3xTF32 d^2 (0xFFFFFFFF: dead), right line}
  uint16_t* cand_cnt;       // [n_left] listed candidates (> T2_CAP: overflow)
  int* err_flag;            // 0: barrier time-out; 1: overflow rows; 2: listed; 4: decided in FP64; 5: FP32 / FP64 disagreements;
                            // 6: float bits of the largest observed |T_fp32 - T_fp64| / bound (check runs)
};

// squared descriptor norms, 8 lanes per line
__global__ void __launch_bounds__(256) k_line_prep2(LineTc2View t, int n_left, int n_right) {
  const LineMatchView& v = t.v;
  const int gl = (blockIdx.x * blockDim.x + threadIdx.x) >> 3, sub = threadIdx.x & 7;
  const int side = gl >= n_left;
  const int i = side ? gl - n_left : gl;
  const bool live = gl < n_left + n_right;   // (no early return: the shuffles below are full-warp)
  float s2 = 0.f;
  if (live) {
    const float* g = (side ? v.right_desc : v.left_desc) + (size_t)i * v.D;
    for (int k = 4 * sub; k < v.D; k += 32) {
      const float4 x = *reinterpret_cast<const float4*>(g + k);
      s2 = fmaf(x.x, x.x, s2); s2 = fmaf(x.y, x.y, s2); s2 = fmaf(x.z, x.z, s2); s2 = fmaf(x.w, x.w, s2);
    }
  }
  s2 += __shfl_xor_sync(0xffffffffu, s2, 1);
  s2 += __shfl_xor_sync(0xffffffffu, s2, 2);
  s2 += __shfl_xor_sync(0xffffffffu, s2, 4);
  if (live && sub == 0) reinterpret_cast<float*>((side ? t.rc.rrec : t.rc.lrec) + i)[0] = s2;
}

__device__ __forceinline__ void named_bar(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }

// stage `rows` descriptors (global row-major fp32, D multiple of 8) as TF32 hi / lo parts into the UMMA K-major layout:
// element (r, k) at (r/8) * sbo + (k/4) * 128 + (r%8) * 16 + (k%4) * 4 ; a warp writes 512 contiguous bytes per step;
// warp w of nw, two row groups in flight
__device__ __forceinline__ void stage_split2(const float* __restrict__ g, int n_valid, int rows, int D, uint8_t* hi, uint8_t* lo,
                                             int w, int nw, int lane) {
  const int chunks = D >> 2, sbo = chunks * 128;
  const int r_in = lane & 7, c_in = lane >> 3;
  const int n_groups = rows >> 3;
  constexpr int U = 5;  // chunks <= 18 -> at most 5 chunks per lane and row
  for (int rg0 = w; rg0 < n_groups; rg0 += 2 * nw) {
    float4 x[2][U];
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const int rg = rg0 + h * nw;
      const int r = rg * 8 + r_in;
      const bool rv = rg < n_groups && r < n_valid;
      const float* grow = g + (size_t)r * D;
#pragma unroll
      for (int u = 0; u < U; u++) {
        const int kc = c_in + 4 * u;
        x[h][u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (rv && kc < chunks) x[h][u] = __ldg(reinterpret_cast<const float4*>(grow + 4 * kc));
      }
    }
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const int rg = rg0 + h * nw;
      if (rg >= n_groups) continue;
#pragma unroll
      for (int u = 0; u < U; u++) {
        const int kc = c_in + 4 * u;
        if (kc >= chunks) continue;
        const float4 q = x[h][u];
        uint4 hh, ll;
        hh.x = to_tf32(q.x); hh.y = to_tf32(q.y); hh.z = to_tf32(q.z); hh.w = to_tf32(q.w);
        ll.x = to_tf32(q.x - __uint_as_float(hh.x)); ll.y = to_tf32(q.y - __uint_as_float(hh.y));
        ll.z = to_tf32(q.z - __uint_as_float(hh.z)); ll.w = to_tf32(q.w - __uint_as_float(hh.w));
        const int off = rg * sbo + kc * 128 + r_in * 16;
        *reinterpret_cast<uint4*>(hi + off) = hh;
        *reinterpret_cast<uint4*>(lo + off) = ll;
      }
    }
  }
}

__global__ void __launch_bounds__(T2_NT, 1) k_line_tc2(LineTc2View t) {
  extern __shared__ __align__(1024) uint8_t tsm[];
  const LineMatchView& v = t.v;
  const int D = v.D, NL = t.nl_chunk;
  const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31;
  const uint32_t l_bytes = (uint32_t)NL * D * 4, r_bytes = (uint32_t)T2_M * D * 4;
  uint8_t* L_hi = tsm;
  uint8_t* L_lo = L_hi + l_bytes;
  uint8_t* R_hi = L_lo + l_bytes;
  uint8_t* R_lo = R_hi + r_bytes;
  float4* rowv = reinterpret_cast<float4*>(R_lo + r_bytes);      // [2][T2_ROWS] records of the pair's left lines
  int* s_cnt = reinterpret_cast<int*>(rowv + 2 * T2_ROWS);       // [2][T2_ROWS] list lengths
  int8_t* rowm = reinterpret_cast<int8_t*>(s_cnt + 2 * T2_ROWS); // [2][T2_ROWS] octaves
  uint64_t* bars = reinterpret_cast<uint64_t*>(rowm + 2 * T2_ROWS);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 6);
  // a barrier that never completes is reported instead of hanging the device: the role that timed out raises its flag,
  // keeps walking through its named barriers without waiting any more, and leaves at the next point where all of its
  // threads agree on the flag; the other role runs into its own time-outs in turn
  volatile int* dead_prod = reinterpret_cast<volatile int*>(tmem_slot + 1);
  volatile int* dead_sel = dead_prod + 1;
  const uint32_t bar_mma = smem_u32(bars), bar_free = smem_u32(bars + 2), bar_row = smem_u32(bars + 4);

  if (wid == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  if (tid == 0) {
    for (int b = 0; b < 2; b++) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar_mma + 8 * b), "r"(1));
      asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar_free + 8 * b), "r"(T2_SEL_WARPS));
      asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar_row + 8 * b), "r"(T2_PROD));
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::);
  }
  for (int j = tid; j < 2 * T2_ROWS; j += T2_NT) s_cnt[j] = 0;
  if (tid == 0) { *dead_prod = 0; *dead_sel = 0; }
  asm volatile("tcgen05.fence::before_thread_sync;" ::);
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::);
  const uint32_t tmem = *tmem_slot;
  const uint32_t sbo = (uint32_t)(D >> 2) * 128u;
  // instruction descriptor: D fp32, A / B TF32, both K-major, N = NL, M = 128
  const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(NL >> 3) << 17) | ((uint32_t)(T2_M >> 4) << 24);
  auto wait_or_flag = [&](uint32_t bar, uint32_t parity, volatile int* flag) {
    if (*flag) return;
    if (!mbar_wait(bar, parity)) *flag = 1;
  };

  if (wid >= T2_SEL_WARPS) {
    // ------------------------------------------------------------------ producers
    const int pw = wid - T2_SEL_WARPS, ptid = tid - T2_SEL;
    uint32_t it = 0, freed = 0;     // steps issued; accumulator releases consumed by the issuing thread (in order)
    int end1 = -1, end2 = -1;       // last step of the previous pair / of the pair before it
    int pp = 0;
    auto consume_free = [&](int upto) {   // issuing thread only
      while ((int)freed <= upto) {
        wait_or_flag(bar_free + 8 * (freed & 1), (freed >> 1) & 1, dead_prod);
        freed++;
      }
    };
    bool out = false;
    for (int p = blockIdx.x; p < v.n_pairs && !out; p += gridDim.x) {
      const int a0 = v.left_off[p], na = v.left_off[p + 1] - a0;
      const int b0 = v.right_off[p], nb = v.right_off[p + 1] - b0;
      if (na == 0 || nb == 0) continue;
      // the selectors must be through with the pair that used this half of the row tables
      if (ptid == 0) consume_free(end2);
      named_bar(1, T2_PROD);
      if (*dead_prod) break;
      for (int j = ptid; j < T2_ROWS; j += T2_PROD) {
        rowv[pp * T2_ROWS + j] = j < na ? t.rc.lrec[a0 + j] : make_float4(0.f, 0.f, 0.f, 0.f);
        rowm[pp * T2_ROWS + j] = j < na ? t.rc.loct[a0 + j] : (int8_t)-2;
      }
      mbar_arrive(bar_row + 8 * pp);
      const int n_lc = (na + NL - 1) / NL, n_m = (nb + T2_M - 1) / T2_M;
      for (int lc = 0; lc < n_lc && !out; lc++)
        for (int m = 0; m < n_m; m++) {
          // the MMAs of the previous step have read the R (and L) buffers
          if (it >= 1) wait_or_flag(bar_mma + 8 * ((it - 1) & 1), ((it - 1) >> 1) & 1, dead_prod);
          if (m == 0) stage_split2(v.left_desc + (size_t)(a0 + lc * NL) * D, na - lc * NL, NL, D, L_hi, L_lo, pw, T2_PROD_WARPS, lane);
          stage_split2(v.right_desc + (size_t)(b0 + m * T2_M) * D, nb - m * T2_M, T2_M, D, R_hi, R_lo, pw, T2_PROD_WARPS, lane);
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          named_bar(1, T2_PROD);
          if (*dead_prod) { out = true; break; }
          if (ptid == 0) {
            if (it >= 2) consume_free((int)it - 2);
            asm volatile("tcgen05.fence::after_thread_sync;" ::);
            const uint32_t d_tmem = tmem + (it & 1) * 256u;
            uint32_t acc = 0;
            for (int ks = 0; ks < D / 8; ks++) {
              const uint32_t koff = (uint32_t)ks * 256u;
              const uint64_t rh = umma_desc(smem_u32(R_hi) + koff, 128, sbo), rl = umma_desc(smem_u32(R_lo) + koff, 128, sbo);
              const uint64_t lh = umma_desc(smem_u32(L_hi) + koff, 128, sbo), ll = umma_desc(smem_u32(L_lo) + koff, 128, sbo);
              umma_tf32(d_tmem, rh, lh, idesc, acc);
              umma_tf32(d_tmem, rh, ll, idesc, 1);
              umma_tf32(d_tmem, rl, lh, idesc, 1);
              acc = 1;
            }
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar_mma + 8 * (it & 1)) : "memory");
          }
          it++;
        }
      end2 = end1; end1 = (int)it - 1; pp ^= 1;
    }
    if (*dead_prod && ptid == 0) atomicExch(t.err_flag, 1);
  } else {
    // ------------------------------------------------------------------ selectors
    const int q = wid & 3, part = wid >> 2;            // TMEM lane quarter; share of the accumulator's column groups
    const int n_grp = NL >> 5, gpw = n_grp / (T2_SEL_WARPS / 4);   // 32-column groups per accumulator / per warp
    const float tau2 = (float)(v.tau * v.tau);
    uint32_t it = 0, rows_seen[2] = {0, 0};
    int pp = 0;
    for (int p = blockIdx.x; p < v.n_pairs; p += gridDim.x) {
      const int a0 = v.left_off[p], na = v.left_off[p + 1] - a0;
      const int b0 = v.right_off[p], nb = v.right_off[p + 1] - b0;
      if (na == 0 || nb == 0) continue;
      wait_or_flag(bar_row + 8 * pp, rows_seen[pp] & 1, dead_sel);
      rows_seen[pp]++;
      const float4* rv = rowv + pp * T2_ROWS;
      const int8_t* rm = rowm + pp * T2_ROWS;
      int* cnt = s_cnt + pp * T2_ROWS;
      const int n_lc = (na + NL - 1) / NL, n_m = (nb + T2_M - 1) / T2_M;
      for (int lc = 0; lc < n_lc; lc++)
        for (int m = 0; m < n_m; m++) {
          const int c = m * T2_M + 32 * q + lane;     // this thread's right line
          float4 cv = make_float4(0.f, 0.f, 0.f, 0.f);
          int octc = -1;
          float hc = 0.f;
          if (c < nb) { cv = t.rc.rrec[b0 + c]; octc = t.rc.roct[b0 + c]; hc = t.rc.rh[b0 + c] - 1e-4f; }
          wait_or_flag(bar_mma + 8 * (it & 1), (it >> 1) & 1, dead_sel);
          // (warp-uniform: the flag is only ever raised, and a warp that disagrees on it for one step merely reads an
          //  accumulator that is reported as invalid anyway)
          const bool skip = __any_sync(0xffffffffu, *dead_sel != 0);
          asm volatile("tcgen05.fence::after_thread_sync;" ::);
          for (int gi = 0; gi < gpw && !skip; gi++) {
            const int g = part * gpw + gi;
            const int j0 = lc * NL + 32 * g;
            if (j0 >= na) break;   // warp-uniform
            uint32_t r[32];
            TMEM_LD32(r, tmem + ((uint32_t)(32 * q) << 16) + (it & 1) * 256u + (uint32_t)(32 * g));
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            // pass 1 (branch-free): survivors of the 32 left lines of this group; lane jj keeps the ballot of row j0 + jj.
            // cheap gates of CheckLinePair, the parallax test of vgl::TriangulateLine and a superset of |X0| >= 1/2
            unsigned my_mask = 0;
            bool edge_any = false;
#pragma unroll
            for (int jj = 0; jj < 32; jj++) {
              const int j = j0 + jj;       // rows past the pair carry octave -2 and never pass
              const float4 lv = rv[j];
              const float d2 = fmaxf(lv.x + cv.x - 2.f * __uint_as_float(r[jj]), 0.f);
              const float cs = fabsf(fmaf(lv.y, cv.y, fmaf(lv.z, cv.z, lv.w * cv.w)));
              const bool pass = ((int)rm[j] == octc) & (d2 < tau2) & !(cs > 0.975f + 1e-5f) & (cs >= hc);
              edge_any |= pass & (cs > 0.975f - 1e-5f);
              const unsigned mask = __ballot_sync(0xffffffffu, pass);
              if (lane == jj) my_mask = mask;
            }
            if (__any_sync(0xffffffffu, edge_any)) {
              // some pair of the tile has its parallax cosine within 1e-5 of the threshold (rare): the masks are formed
              // again with those pairs decided in FP64, as the reference computes the test
#pragma unroll 1
              for (int jj = 0; jj < 32; jj++) {
                const int j = j0 + jj;
                const float4 lv = rv[j];
                uint32_t rj;      // column jj of the group, read again from TMEM (no dynamic register indexing)
                asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];\n" : "=r"(rj) : "r"(tmem + ((uint32_t)(32 * q) << 16) + (it & 1) * 256u + (uint32_t)(32 * g + jj)));
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                const float d2 = fmaxf(lv.x + cv.x - 2.f * __uint_as_float(rj), 0.f);
                const float cs = fabsf(fmaf(lv.y, cv.y, fmaf(lv.z, cv.z, lv.w * cv.w)));
                bool pass = ((int)rm[j] == octc) & (d2 < tau2) & !(cs > 0.975f + 1e-5f) & (cs >= hc);
                if (pass && cs > 0.975f - 1e-5f) {
                  const double* ul = v.left_un + 3 * (size_t)(a0 + j);
                  const double* un = v.right_un + 3 * (size_t)(b0 + c);
                  pass = !(fabs(ul[0] * un[0] + ul[1] * un[1] + ul[2] * un[2]) > 0.975);
                }
                const unsigned mask = __ballot_sync(0xffffffffu, pass);
                if (lane == jj) my_mask = mask;
              }
            }
            // one shared-memory atomic per row, all 32 rows at once
            int my_base = 0;
            if (my_mask) my_base = atomicAdd(&cnt[j0 + lane], __popc(my_mask));
            // pass 2 (branch-free): the survivors of a row go to consecutive slots of its list.  The accumulator is read
            // from TMEM a second time: keeping the 32 values of pass 1 alive across both passes costs more registers than
            // the kernel has (it runs at the 96-register limit of a 640-thread CTA) and the compiler spills them
            TMEM_LD32(r, tmem + ((uint32_t)(32 * q) << 16) + (it & 1) * 256u + (uint32_t)(32 * g));
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            const unsigned lt = (1u << lane) - 1u;
            uint2* const out0 = t.cand + (size_t)(a0 + j0) * T2_CAP;
#pragma unroll
            for (int jj = 0; jj < 32; jj++) {
              const unsigned mask = __shfl_sync(0xffffffffu, my_mask, jj);
              const int slot = __shfl_sync(0xffffffffu, my_base, jj) + __popc(mask & lt);
              const float d2 = fmaxf(rv[j0 + jj].x + cv.x - 2.f * __uint_as_float(r[jj]), 0.f);
              if (((mask >> lane) & 1u) && slot < T2_CAP) out0[jj * T2_CAP + slot] = make_uint2(__float_as_uint(d2), (uint32_t)c);
            }
          }
          asm volatile("tcgen05.fence::before_thread_sync;" ::);
          __syncwarp();
          if (lane == 0) mbar_arrive(bar_free + 8 * (it & 1));
          it++;
        }
      named_bar(2, T2_SEL);
      if (*dead_sel) break;
      for (int j = tid; j < na; j += T2_SEL) {
        t.cand_cnt[a0 + j] = (uint16_t)min(cnt[j], T2_CAP + 1);
        cnt[j] = 0;
      }
      pp ^= 1;
    }
    if (*dead_sel && tid == 0) atomicExch(t.err_flag, 1);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::);
  __syncthreads();
  if (wid == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512));
}

// FP32 evaluation of the gates that line_pair_gate_fast applies in FP64, division-free and with a bound on its own
// rounding error: 1 admissible, 0 not admissible, -1 too close to a threshold to tell (the caller decides those in FP64).
// With dir = l1 x l2, c1 = dir x l1, f = beta / |dir|^2 (X0 = f c1), and, per endpoint a = (px, py, 1), u = a x (K dir),
// w = a x (K c1) (both as products with the per-endpoint matrix M = [a]_x K that k_line_prep2 forms in FP64):
//   |X0|^2 >= 1/4            <=>  beta^2 |l1|^2 >= |dir|^2 / 4                  (dir is perpendicular to l1; the selectors
//                                                                                 have applied a superset of this test)
//   endpoint depth >= 0      <=>  beta T >= 0,  T = c1_z |u|^2 - (u.w) dir_z    (Binet-Cauchy: aa cy - ac ay = (a x c).(a x y);
//                                                                                 depth = f T / |u|^2)
// Error model: every computed vector carries an absolute error of k eps times the product of the norms that went into
// it; with E = |K|_F |a| |dir| >= |u| and q = |u| this gives |dT| <= k eps |dir| (q + E) 3 (|l1| q + |w|), tested in the
// square-root-free form T^2 > (k eps)^2 |dir|^2 2 (q^2 + E^2) 9 2 (|l1|^2 q^2 + |w|^2).
struct GateK { float kn2; float c_tol2; };
struct GateL {     // per left line (registers, warp-uniform)
  float l1[3], l1sq, aa[2];
  float M[2][9];
};
__device__ __forceinline__ void cross3f(const float* a, const float* b, float* o) {
  o[0] = a[1] * b[2] - a[2] * b[1]; o[1] = a[2] * b[0] - a[0] * b[2]; o[2] = a[0] * b[1] - a[1] * b[0];
}
__device__ __forceinline__ float dot3f(const float* a, const float* b) { return fmaf(a[0], b[0], fmaf(a[1], b[1], a[2] * b[2])); }
__device__ __forceinline__ void mat3f(const float* M, const float* x, float* o) {
  o[0] = fmaf(M[0], x[0], fmaf(M[1], x[1], M[2] * x[2]));
  o[1] = fmaf(M[3], x[0], fmaf(M[4], x[1], M[5] * x[2]));
  o[2] = fmaf(M[6], x[0], fmaf(M[7], x[1], M[8] * x[2]));
}
__device__ __forceinline__ GateL load_gate_left(const float4* g) {
  GateL L;
  const float4 g0 = g[0], g1 = g[1], g2 = g[2], g3 = g[3], g4 = g[4], g5 = g[5], g6 = g[6];
  L.l1[0] = g0.x; L.l1[1] = g0.y; L.l1[2] = g0.z; L.l1sq = g0.w;
  L.aa[0] = g1.y; L.aa[1] = g1.z;
  const float m[20] = {g2.x, g2.y, g2.z, g2.w, g3.x, g3.y, g3.z, g3.w, g4.x, g4.y, g4.z, g4.w, g5.x, g5.y, g5.z, g5.w, g6.x, g6.y, g6.z, g6.w};
#pragma unroll
  for (int k = 0; k < 9; k++) { L.M[0][k] = m[k]; L.M[1][k] = m[9 + k]; }
  return L;
}
// T and its bound for endpoint e (shared by the decision and by the check statistics)
__device__ __forceinline__ void gate32_endpoint(const GateK& gk, const GateL& L, int e, const float* dir, const float* c1, float dd,
                                                float* T, float* tol2, bool* cond) {
  float u[3], w[3];
  mat3f(L.M[e], dir, u);
  mat3f(L.M[e], c1, w);
  const float det2 = dot3f(u, u), uw = dot3f(u, w), ww = dot3f(w, w);
  *T = c1[2] * det2 - uw * dir[2];
  const float E2 = gk.kn2 * dd * L.aa[e];
  *cond = det2 > 1e-6f * E2;
  *tol2 = gk.c_tol2 * (det2 + E2) * dd * fmaf(L.l1sq, det2, ww);
}
__device__ __forceinline__ int line_gate32(const GateK& gk, const GateL& L, const float* l2, float beta) {
  // straight-line code: every entry runs the same instructions and the verdict is assembled from predicates at the end (the
  // selectors have already removed the entries the early tests would reject, so early exits only cost divergence here)
  float dir[3], c1[3];
  cross3f(L.l1, l2, dir);
  const float dd = dot3f(dir, dir);
  const float lhs = beta * beta * L.l1sq, rhs = 0.25f * dd;
  cross3f(dir, L.l1, c1);
  bool undecided = !(dd > 1e-12f) || (!(lhs < rhs * (1.f - 2e-3f)) && !(lhs > rhs * (1.f + 2e-3f)));
  bool rejected = lhs < rhs * (1.f - 2e-3f);
#pragma unroll
  for (int e = 0; e < 2; e++) {
    float T, tol2;
    bool cond;
    gate32_endpoint(gk, L, e, dir, c1, dd, &T, &tol2, &cond);
    const bool clear = cond && (T * T > tol2);
    undecided |= !clear;
    rejected |= clear && (beta * T < 0.f);     // a clear rejection by one endpoint stands whatever the other one says
  }
  // (a clear |X0| rejection or endpoint rejection wins over "undecided": the FP64 formulas could only confirm it)
  return rejected && (dd > 1e-12f) ? 0 : (undecided ? -1 : 1);
}
// FP64 value of T for the check statistics (same formula from the FP64 line equations)
__device__ __forceinline__ double gate64_T(const LineMatchView& v, const float* s1, const double* l1, const double* l2, int e) {
  double dir[3], c1[3];
  cross3(l1, l2, dir);
  cross3(dir, l1, c1);
  const double* K = v.K;
  const double kd[3] = {K[0] * dir[0] + K[1] * dir[1] + K[2] * dir[2], K[3] * dir[0] + K[4] * dir[1] + K[5] * dir[2], K[6] * dir[0] + K[7] * dir[1] + K[8] * dir[2]};
  const double kc[3] = {K[0] * c1[0] + K[1] * c1[1] + K[2] * c1[2], K[3] * c1[0] + K[4] * c1[1] + K[5] * c1[2], K[6] * c1[0] + K[7] * c1[1] + K[8] * c1[2]};
  const double a[3] = {s1[2 * e], s1[2 * e + 1], 1.0};
  double u[3], w[3];
  cross3(a, kd, u);
  cross3(a, kc, w);
  return c1[2] * dot3(u, u) - dot3(u, w) * dir[2];
}

// The remaining gates of CheckLinePair over the candidate lists, and compaction of each list to its admissible entries
// (in place: the write position never passes the read position).  A warp takes G32_ROWS consecutive left lines of a pair.
// The kernel is latency-bound (two dependent loads per entry and ~150 instructions), so the warp first pulls everything
// it will read from HBM -- the list heads (64 entries per line) and the left-line geometry -- into shared memory with
// one burst of cp.async, and only then walks the lines.  Entries the FP32 evaluation cannot decide stay in the list
// provisionally and are queued (per warp, shared memory); the queue is worked off 32 entries at a time by the FP64
// formulas, so that the FP64 path runs with full warps instead of one or two lanes per list; an entry that fails there
// is overwritten by the dead key.
// grid (row blocks, pairs), or (pairs, row blocks) when there are more than 65535 pairs.
constexpr int G32_ROWS = 8, G32_WARPS = 4, G32_HEAD = 64;
struct GateQ { uint32_t slot_lo; uint32_t slot_hi; int gl; int c; };   // list slot, left line, right line (global indices)
__device__ __forceinline__ void cp_async8(void* smem, const void* g) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(smem)), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async16(void* smem, const void* g) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem)), "l"(g) : "memory");
}
__global__ void __launch_bounds__(32 * G32_WARPS) k_line_gate32(LineTc2View t, GateK gk, int swap_grid, int check) {
  __shared__ __align__(16) uint2 s_ent[G32_WARPS][G32_ROWS][G32_HEAD];
  __shared__ __align__(16) float4 s_geo[G32_WARPS][G32_ROWS][7];
  __shared__ GateQ queue[G32_WARPS][64];
  const LineMatchView& v = t.v;
  const int p = swap_grid ? blockIdx.x : blockIdx.y, jb = swap_grid ? blockIdx.y : blockIdx.x;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int a0 = v.left_off[p], na = v.left_off[p + 1] - a0, b0 = v.right_off[p];
  const int j_begin = (jb * G32_WARPS + wid) * G32_ROWS;
  if (j_begin >= na) return;
  const int n_rows = min(G32_ROWS, na - j_begin);
  // ---- one burst: list lengths, list heads, left-line geometry
  int my_cnt = 0;
  if (lane < n_rows) my_cnt = t.cand_cnt[a0 + j_begin + lane];
  for (int r = 0; r < n_rows; r++) {
    const uint2* src = t.cand + (size_t)(a0 + j_begin + r) * T2_CAP;
    cp_async8(&s_ent[wid][r][lane], src + lane);
    cp_async8(&s_ent[wid][r][lane + 32], src + lane + 32);
  }
  for (int k = lane; k < 7 * n_rows; k += 32) cp_async16(&s_geo[wid][0][0] + k, t.rc.lgeo + 7 * (size_t)(a0 + j_begin) + k);
  asm volatile("cp.async.commit_group;" ::: "memory");
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncwarp();
  GateQ* q = queue[wid];
  int qn = 0;
  int n_listed = 0, n_border = 0, n_bad = 0;
  float worst = 0.f;
  const unsigned lt = (1u << lane) - 1u;
  auto settle = [&](const GateQ& it) {   // FP64 verdict for a queued entry
    if (!line_pair_gate_fast(v, v.left_seg + 4 * (size_t)it.gl, v.left_leq + 3 * (size_t)it.gl, v.right_leq + 3 * (size_t)it.c))
      t.cand[((size_t)it.slot_hi << 32) | it.slot_lo].x = 0xFFFFFFFFu;
  };
  for (int r = 0; r < n_rows; r++) {
    const int gl = a0 + j_begin + r;
    const int cnt_raw = __shfl_sync(0xffffffffu, my_cnt, r), cnt = min(cnt_raw, T2_CAP);
    const GateL L = load_gate_left(s_geo[wid][r]);
    const size_t row = (size_t)gl * T2_CAP;
    int out = 0;
    for (int e0 = 0; e0 < cnt; e0 += 64) {
      // two entries per lane and trip: two independent dependency chains (the kernel is latency-bound)
      bool valid[2];
      uint32_t d2[2] = {0xFFFFFFFFu, 0xFFFFFFFFu};
      int col[2] = {0, 0}, g[2] = {0, 0};
      float4 l2v[2];
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const int e = e0 + 32 * h + lane;
        valid[h] = e < cnt;
        l2v[h] = make_float4(1.f, 0.f, 0.f, 0.f);
        if (valid[h]) {
          const uint2 en = e < G32_HEAD ? s_ent[wid][r][e] : t.cand[row + e];
          d2[h] = en.x;
          col[h] = (int)en.y;
          l2v[h] = t.rc.rleq[b0 + col[h]];
        }
      }
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const float l2[3] = {l2v[h].x, l2v[h].y, l2v[h].z};
        g[h] = valid[h] ? line_gate32(gk, L, l2, l2v[h].w) : 0;
        if (check && valid[h]) {
          const float* s1 = v.left_seg + 4 * (size_t)gl;
          const bool g64 = line_pair_gate_fast(v, s1, v.left_leq + 3 * (size_t)gl, v.right_leq + 3 * (size_t)(b0 + col[h]));
          if (g[h] >= 0 && (g[h] != 0) != g64) n_bad++;
          // observed error of T against its bound (both endpoints), in units of the bound
          float dir[3], c1[3];
          cross3f(L.l1, l2, dir);
          cross3f(dir, L.l1, c1);
          const float dd = dot3f(dir, dir);
          for (int ep = 0; ep < 2; ep++) {
            float T, tol2;
            bool cond;
            gate32_endpoint(gk, L, ep, dir, c1, dd, &T, &tol2, &cond);
            const double T64 = gate64_T(v, s1, v.left_leq + 3 * (size_t)gl, v.right_leq + 3 * (size_t)(b0 + col[h]), ep);
            if (cond && tol2 > 0.f) worst = fmaxf(worst, (float)(fabs((double)T - T64) / sqrt((double)tol2)));
          }
        }
      }
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const bool keep = valid[h] && g[h] != 0, border = valid[h] && g[h] < 0;
        const unsigned km = __ballot_sync(0xffffffffu, keep), bm = __ballot_sync(0xffffffffu, border);
        const int pos = out + __popc(km & lt);
        if (keep) t.cand[row + pos] = make_uint2(d2[h], (uint32_t)col[h]);
        if (border) {
          GateQ it;
          const size_t slot = row + pos;
          it.slot_lo = (uint32_t)slot; it.slot_hi = (uint32_t)(slot >> 32); it.gl = gl; it.c = b0 + col[h];
          q[qn + __popc(bm & lt)] = it;
        }
        out += __popc(km);
        qn += __popc(bm);
        n_border += __popc(bm);
        __syncwarp();
        if (qn >= 32) {
          qn -= 32;
          settle(q[qn + lane]);
          __syncwarp();
        }
      }
    }
    if (lane == 0 && cnt_raw <= T2_CAP) t.cand_cnt[gl] = (uint16_t)out;   // (an overflowed row keeps its marker: exact scan in the greedy)
    n_listed += cnt;
  }
  if (lane < qn) settle(q[lane]);
  if (check) {
    if (lane == 0) { atomicAdd(t.err_flag + 2, n_listed); atomicAdd(t.err_flag + 4, n_border); }
    if (n_bad) atomicAdd(t.err_flag + 5, n_bad);
    atomicMax(reinterpret_cast<unsigned*>(t.err_flag) + 6, __float_as_uint(worst));
  }
}

// One warp per pair replays the sequential greedy over the compacted lists: smallest (d^2, right line) among the
// untaken live entries of the row, two warp reductions per left line.  Nothing on the per-line dependency chain touches
// memory: the "taken" set lives in registers (lane w holds the bits of right lines [32 w, 32 w + 32), looked up by
// shuffle), the first 64 entries of the next G2_PF rows are prefetched into registers (the lists stream from HBM), and
// the matches are collected in shared memory and written out at the end.  Longer lists read their tail on demand.
constexpr int G2_PF = 4;
__global__ void __launch_bounds__(32) k_line_greedy2(LineTc2View t) {
  __shared__ uint16_t s_cnt[T2_ROWS];
  __shared__ int16_t s_match[T2_ROWS];
  const LineMatchView& v = t.v;
  const int lane = threadIdx.x, p = blockIdx.x;
  const int a0 = v.left_off[p], na = v.left_off[p + 1] - a0;
  const int b0 = v.right_off[p], nb = v.right_off[p + 1] - b0;
  if (na == 0) return;
  for (int j = lane; j < na; j += 32) s_cnt[j] = t.cand_cnt[a0 + j];
  __syncwarp();
  uint32_t taken = 0u;   // lane w < 16: right lines [32 w, 32 w + 32)
  uint32_t pd2[G2_PF][2];
  uint32_t pcol[G2_PF][2];
  // both loads of a row are issued unconditionally (every slot of a list exists); the list length masks them at use
  auto fetch = [&](int j, int u) {
    pd2[u][0] = pd2[u][1] = 0xFFFFFFFFu;
    pcol[u][0] = pcol[u][1] = 0;
    if (j < na) {
      const uint2* o = t.cand + (size_t)(a0 + j) * T2_CAP;
      const uint2 e0 = o[lane], e1 = o[lane + 32];
      pd2[u][0] = e0.x; pcol[u][0] = e0.y;
      pd2[u][1] = e1.x; pcol[u][1] = e1.y;
    }
  };
#pragma unroll
  for (int u = 0; u < G2_PF; u++) fetch(u, u);
  for (int jb = 0; jb < na; jb += G2_PF) {
#pragma unroll
    for (int u = 0; u < G2_PF; u++) {
      const int j = jb + u;
      if (j >= na) break;
      const int cnt = s_cnt[j];
      uint32_t bd = 0xFFFFFFFFu, bc = 0xFFFFFFFFu;
      auto offer = [&](bool valid, uint32_t d2, uint32_t c) {   // (the shuffle is executed by every lane)
        const uint32_t w = __shfl_sync(0xffffffffu, taken, (c >> 5) & 31);
        const bool live = valid && d2 != 0xFFFFFFFFu && !((w >> (c & 31)) & 1u);
        if (live && (d2 < bd || (d2 == bd && c < bc))) { bd = d2; bc = c; }
      };
      offer(lane < cnt, pd2[u][0], pcol[u][0]);
      offer(lane + 32 < cnt, pd2[u][1], pcol[u][1]);
      fetch(j + G2_PF, u);
      int bi = -1;
      if (cnt <= T2_CAP) {
        if (cnt > 64) {   // warp-uniform
          const uint2* o = t.cand + (size_t)(a0 + j) * T2_CAP;
          for (int e0 = 64; e0 < cnt; e0 += 32) {
            const int e = e0 + lane;
            uint2 en = make_uint2(0xFFFFFFFFu, 0u);
            if (e < cnt) en = o[e];
            offer(e < cnt, en.x, en.y);
          }
        }
        const uint32_t m = __reduce_min_sync(0xffffffffu, bd);
        if (m != 0xFFFFFFFFu) bi = (int)__reduce_min_sync(0xffffffffu, bd == m ? bc : 0xFFFFFFFFu);
      } else {
        if (lane == 0) atomicAdd(t.err_flag + 1, 1);
        // overflowed list: exact scan of the row.  Pass A: lanes stride over the right lines and apply every gate of
        // CheckLinePair; pass B: exact FP32 distances of the few admissible ones, computed by the whole warp per line.
        const int gl = a0 + j;
        const bool l_ok = !(v.left_len[gl] < (double)v.min_len);
        const double* ul = v.left_un + 3 * (size_t)gl;
        float best = INFINITY;
        for (int cb = 0; cb < nb && l_ok; cb += 32) {
          const int c = cb + lane;
          const uint32_t w = __shfl_sync(0xffffffffu, taken, cb >> 5);
          bool ok = false;
          if (c < nb && !((w >> lane) & 1u)) {
            const int gc = b0 + c;
            if (v.left_oct[gl] == v.right_oct[gc] && !(v.right_len[gc] < (double)v.min_len)) {
              const double* un = v.right_un + 3 * (size_t)gc;
              if (!(fabs(ul[0] * un[0] + ul[1] * un[1] + ul[2] * un[2]) > 0.975))
                ok = line_pair_gate(v, v.left_seg + 4 * (size_t)gl, v.left_leq + 3 * (size_t)gl, v.right_leq + 3 * (size_t)gc);
            }
          }
          unsigned mm = __ballot_sync(0xffffffffu, ok);
          while (mm) {  // ascending column order, strict <: the first minimum wins as in the reference
            const int c2 = cb + __ffs(mm) - 1;
            mm &= mm - 1;
            const float d = sqrtf(warp_exact_d2(v.left_desc + (size_t)gl * v.D, v.right_desc + (size_t)(b0 + c2) * v.D, v.D, lane));
            if ((double)d < v.tau && d < best) { best = d; bi = c2; }
          }
        }
      }
      if (bi >= 0 && lane == (bi >> 5)) taken |= 1u << (bi & 31);
      if (lane == 0) s_match[j] = (int16_t)bi;
    }
  }
  __syncwarp();
  for (int j = lane; j < na; j += 32) v.match[a0 + j] = s_match[j];
}

// exact distance of every match (FP32, difference form): 8 lanes per left line, 32 lines per block
__global__ void __launch_bounds__(256) k_line_exact2(LineTc2View t, int swap_grid) {
  const LineMatchView& v = t.v;
  const int p = swap_grid ? blockIdx.x : blockIdx.y, jb = swap_grid ? blockIdx.y : blockIdx.x;
  const int sub = threadIdx.x & 7, j = jb * 32 + (threadIdx.x >> 3);
  const int a0 = v.left_off[p], na = v.left_off[p + 1] - a0;
  const bool live = j < na;
  const int bi = live ? v.match[a0 + j] : -1;
  float s2 = 0.f;
  if (bi >= 0) {
    const float* a = v.left_desc + (size_t)(a0 + j) * v.D;
    const float* b = v.right_desc + (size_t)(v.right_off[p] + bi) * v.D;
    for (int k = 4 * sub; k < v.D; k += 32) {
      const float4 x = *reinterpret_cast<const float4*>(a + k), y = *reinterpret_cast<const float4*>(b + k);
      float d;
      d = x.x - y.x; s2 = fmaf(d, d, s2);
      d = x.y - y.y; s2 = fmaf(d, d, s2);
      d = x.z - y.z; s2 = fmaf(d, d, s2);
      d = x.w - y.w; s2 = fmaf(d, d, s2);
    }
  }
  s2 += __shfl_xor_sync(0xffffffffu, s2, 1);
  s2 += __shfl_xor_sync(0xffffffffu, s2, 2);
  s2 += __shfl_xor_sync(0xffffffffu, s2, 4);
  if (live && sub == 0) v.mdist[a0 + j] = bi >= 0 ? sqrtf(s2) : INFINITY;
}

inline int cdiv(int a, int b) { return (a + b - 1) / b; }

}  // namespace

extern "C" int lld_line_match(void* ctx, const lld_line_match_problem* p, lld_line_match_result* out) {
  LldCtx* c = lld_ctx_cast(ctx);
  if (!c || !p || !out) return LLD_ERR_ARG;
  if (int r = lld_call_begin(c, true)) return r;
  LLD_ARG(c, p->n_pairs >= 1 && p->desc_dim >= 1 && p->desc_dim <= 512);
  LineMatchView v;
  const int P = p->n_pairs;
  const int n_left = p->left_off[P], n_right = p->right_off[P];
  v.n_pairs = P; v.D = p->desc_dim;
  for (int i = 0; i < 9; i++) v.K[i] = p->K[i];
  v.baseline = p->baseline; v.tau = p->tau; v.min_len = p->min_line_length;
  // tensor-core path: D multiple of 8 up to 72 floats, at most 512 lines per side of a pair (LLD_LINE_TC=0 forces the
  // FP32 tile path, which takes everything else)
  int max_na = 0, max_nb = 0;
  for (int i = 0; i < P; i++) {
    max_na = std::max(max_na, p->left_off[i + 1] - p->left_off[i]);
    max_nb = std::max(max_nb, p->right_off[i + 1] - p->right_off[i]);
  }
  const char* e_tc = getenv("LLD_LINE_TC");
  const bool use_tc = !(e_tc && e_tc[0] == '0') && v.D % 8 == 0 && v.D >= 8 && v.D <= 72 && max_nb <= T2_ROWS && max_na <= T2_ROWS &&
                      max_nb >= 1 && max_na >= 1;
  // tile path: tiles + matrix offsets
  std::vector<long long> mat_off(P), taken_off(P);
  std::vector<int> tp, tr, tc;
  long long tot = 0, ttot = 0;
  for (int i = 0; i < P && !use_tc; i++) {
    const int na = p->left_off[i + 1] - p->left_off[i], nb = p->right_off[i + 1] - p->right_off[i];
    mat_off[i] = tot; tot += (long long)na * nb;
    taken_off[i] = ttot; ttot += nb;
    for (int r = 0; r < cdiv(na, LT); r++)
      for (int cc = 0; cc < cdiv(nb, LT); cc++) { tp.push_back(i); tr.push_back(r); tc.push_back(cc); }
  }
  LLD_UP(c, v.left_off, p->left_off, P + 1);
  LLD_UP(c, v.right_off, p->right_off, P + 1);
  LLD_UP(c, v.left_seg, p->left_seg, 4 * (size_t)n_left);
  LLD_UP(c, v.left_oct, p->left_octave, n_left);
  LLD_UP(c, v.right_seg, p->right_seg, 4 * (size_t)n_right);
  LLD_UP(c, v.right_oct, p->right_octave, n_right);
  LLD_UP(c, v.left_desc, p->left_desc, (size_t)n_left * v.D);
  LLD_UP(c, v.right_desc, p->right_desc, (size_t)n_right * v.D);
  LLD_UP(c, v.mat_off, mat_off.data(), P);
  long long* d_taken_off;
  LLD_UP(c, d_taken_off, taken_off.data(), P);
  int *d_tp, *d_tr, *d_tc;
  LLD_UP(c, d_tp, tp.data(), tp.size());
  LLD_UP(c, d_tr, tr.data(), tr.size());
  LLD_UP(c, d_tc, tc.data(), tc.size());
  LLD_DEV(c, v.left_leq, 3 * (size_t)n_left);
  LLD_DEV(c, v.right_leq, 3 * (size_t)n_right);
  LLD_DEV(c, v.left_len, n_left);
  LLD_DEV(c, v.right_len, n_right);
  LLD_DEV(c, v.left_un, 3 * (size_t)n_left);
  LLD_DEV(c, v.right_un, 3 * (size_t)n_right);
  LLD_DEV(c, v.dist, (size_t)tot);
  LLD_DEV(c, v.match, n_left);
  LLD_DEV(c, v.mdist, n_left);
  int* d_taken;
  LLD_DEV(c, d_taken, (size_t)ttot);
  LLD_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
  const int nmax = std::max(std::max(n_left, n_right), 1);
  int* d_tc_err = nullptr;
  const bool check = getenv("LLD_LINE_CHECK") != nullptr || getenv("LLD_LINE_STATS") != nullptr;
  if (use_tc) {
    LineTc2View t;
    t.v = v;
    t.nl_chunk = v.D <= 64 ? 256 : 128;
    LLD_DEV(c, t.rc.lrec, n_left);
    LLD_DEV(c, t.rc.rrec, n_right);
    LLD_DEV(c, t.rc.rh, n_right);
    LLD_DEV(c, t.rc.loct, n_left);
    LLD_DEV(c, t.rc.roct, n_right);
    LLD_DEV(c, t.rc.lgeo, 7 * (size_t)n_left);
    LLD_DEV(c, t.rc.rleq, n_right);
    LLD_DEV(c, t.cand, (size_t)n_left * T2_CAP);
    LLD_DEV(c, t.cand_cnt, n_left);
    LLD_DEV(c, t.err_flag, 8);
    d_tc_err = t.err_flag;
    LLD_CUDA(c, cudaMemsetAsync(t.err_flag, 0, 8 * sizeof(int), c->stream));
    LLD_CUDA(c, cudaMemsetAsync(t.cand_cnt, 0, sizeof(uint16_t) * (size_t)n_left, c->stream));   // pairs without right lines
    const size_t smem = (size_t)(t.nl_chunk + T2_M) * v.D * 8 + 2 * T2_ROWS * (16 + 4 + 1) + 6 * 8 + 16;
    LLD_CUDA(c, lld_raise_dyn_smem(k_line_tc2, (size_t)(int)smem));
    GateK gk;
    double kn = 0;
    for (int i = 0; i < 9; i++) kn += v.K[i] * v.K[i];
    gk.kn2 = (float)kn;
    double c_tol = 2e-6;   // k eps with k = 32; check runs report the largest observed error in units of the bound (err_flag[6])
    if (const char* e_c = getenv("LLD_LINE_CTOL")) c_tol = atof(e_c);
    gk.c_tol2 = (float)(36.0 * c_tol * c_tol);
    const int swap_grid = P > 65535;
    const int gate_blocks = cdiv(max_na, G32_ROWS * G32_WARPS), exact_blocks = cdiv(max_na, 32);
    const dim3 grid_gate = swap_grid ? dim3(P, gate_blocks) : dim3(gate_blocks, P);
    const dim3 grid_exact = swap_grid ? dim3(P, exact_blocks) : dim3(exact_blocks, P);
    LLD_LAUNCH(c, k_line_prep<true>, cdiv(nmax, 128), 128, 0, v, t.rc, n_left, n_right);
    LLD_LAUNCH(c, k_line_prep2, cdiv(8 * (n_left + n_right), 256), 256, 0, t, n_left, n_right);
    LLD_LAUNCH(c, k_line_tc2, std::min(P, c->sm_count), T2_NT, smem, t);
    LLD_LAUNCH(c, k_line_gate32, grid_gate, 32 * G32_WARPS, 0, t, gk, swap_grid, (int)check);
    LLD_LAUNCH(c, k_line_greedy2, P, 32, 0, t);
    LLD_LAUNCH(c, k_line_exact2, grid_exact, 256, 0, t, swap_grid);
  } else {
    LLD_LAUNCH(c, k_line_prep<false>, cdiv(nmax, 128), 128, 0, v, LineRecs(), n_left, n_right);
    if (!tp.empty()) {
      const size_t smem = sizeof(float) * 2 * LT * (v.D + 1);
      LLD_CUDA(c, lld_raise_dyn_smem(k_line_dist, (size_t)(int)smem));
      LLD_LAUNCH(c, k_line_dist, (int)tp.size(), 256, smem, v, d_tp, d_tr, d_tc);
    }
    LLD_LAUNCH(c, k_line_greedy, P, 32, 0, v, d_taken, d_taken_off);
  }
  LLD_CUDA(c, cudaGetLastError());
  LLD_CUDA(c, cudaEventRecord(c->ev[2], c->stream));
  int* h_err = reinterpret_cast<int*>(c->pinned);
  for (int i = 0; i < 8; i++) h_err[i] = 0;
  if (d_tc_err) LLD_DOWN(c, h_err, d_tc_err, 8);
  LLD_DOWN(c, out->match, v.match, n_left);
  LLD_DOWN(c, out->dist, v.mdist, n_left);
  if (int r = lld_call_end(c)) return r;
  if (getenv("LLD_LINE_STATS") && d_tc_err)
    fprintf(stderr, "[lld_line_match] rows with an overflowed list %d, listed candidates %d, decided in FP64 %d, FP32/FP64 disagreements %d, largest FP32 error / bound %.3g\n",
            h_err[1], h_err[2], h_err[4], h_err[5], (double)*reinterpret_cast<float*>(h_err + 6));
  if (h_err[0]) {
    snprintf(c->err, sizeof(c->err), "line matcher: a tensor-core pipeline barrier timed out");
    return LLD_ERR_CUDA;
  }
  if (check && h_err[5]) {
    snprintf(c->err, sizeof(c->err), "line matcher: %d FP32 gate decisions differ from FP64 (LLD_LINE_CHECK)", h_err[5]);
    return LLD_ERR_CUDA;
  }
  return LLD_OK;
}
