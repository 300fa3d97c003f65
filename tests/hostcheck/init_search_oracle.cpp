// ORACLE — TEST INFRASTRUCTURE ONLY.  CPU restatement of ORBmatcher::SearchForInitialization (src/ORBmatcher.cc:405; the
// ORB-SLAM2 function LLD-SLAM inherits unchanged) under the C-ABI of include/lldba.h with the lldo_ prefix, like the oracle
// library in oracle/.  Built by __graft_entry__.build() into tests/hostcheck/libinit_search_oracle.so with -ffp-contract=off,
// so that the float window and rotation arithmetic rounds where the reference's source rounds.  The product never loads it.
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../include/lldba.h"

namespace {

// ORBmatcher::DescriptorDistance: the SWAR popcount of the reference over eight 32-bit words
int descriptor_distance(const uint8_t* a, const uint8_t* b) {
  int dist = 0;
  for (int i = 0; i < 8; i++) {
    uint32_t pa, pb;
    std::memcpy(&pa, a + 4 * i, 4);
    std::memcpy(&pb, b + 4 * i, 4);
    uint32_t v = pa ^ pb;
    v = v - ((v >> 1) & 0x55555555);
    v = (v & 0x33333333) + ((v >> 2) & 0x33333333);
    dist += (((v + (v >> 4)) & 0xF0F0F0F) * 0x1010101) >> 24;
  }
  return dist;
}

const int GRID_COLS = 64, GRID_ROWS = 48;  // include/Frame.h

// Frame::AssignFeaturesToGrid / PosInGrid and Frame::GetFeaturesInArea over F2's undistorted keypoints
struct Grid {
  float min_x, min_y, winv, hinv;
  std::vector<std::vector<int>> cell;  // [col * ROWS + row], keypoint index order
  void build(const lld_frame_geom& g, const float* xy, int n) {
    min_x = g.min_x; min_y = g.min_y;
    winv = static_cast<float>(GRID_COLS) / (g.max_x - g.min_x);
    hinv = static_cast<float>(GRID_ROWS) / (g.max_y - g.min_y);
    cell.assign(GRID_COLS * GRID_ROWS, {});
    for (int i = 0; i < n; i++) {
      const int px = (int)std::round((xy[2 * i] - min_x) * winv);
      const int py = (int)std::round((xy[2 * i + 1] - min_y) * hinv);
      if (px < 0 || px >= GRID_COLS || py < 0 || py >= GRID_ROWS) continue;
      cell[px * GRID_ROWS + py].push_back(i);
    }
  }
  void features_in_area(float x, float y, float r, int minLevel, int maxLevel, const float* xy, const uint8_t* octave,
                        std::vector<int>& out) const {
    out.clear();
    const int nMinCellX = std::max(0, (int)std::floor((x - min_x - r) * winv));
    if (nMinCellX >= GRID_COLS) return;
    const int nMaxCellX = std::min(GRID_COLS - 1, (int)std::ceil((x - min_x + r) * winv));
    if (nMaxCellX < 0) return;
    const int nMinCellY = std::max(0, (int)std::floor((y - min_y - r) * hinv));
    if (nMinCellY >= GRID_ROWS) return;
    const int nMaxCellY = std::min(GRID_ROWS - 1, (int)std::ceil((y - min_y + r) * hinv));
    if (nMaxCellY < 0) return;
    const bool bCheckLevels = (minLevel > 0) || (maxLevel >= 0);
    for (int ix = nMinCellX; ix <= nMaxCellX; ix++)
      for (int iy = nMinCellY; iy <= nMaxCellY; iy++)
        for (int idx : cell[ix * GRID_ROWS + iy]) {
          if (bCheckLevels) {
            if ((int)octave[idx] < minLevel) continue;
            if (maxLevel >= 0 && (int)octave[idx] > maxLevel) continue;
          }
          const float distx = xy[2 * idx] - x;
          const float disty = xy[2 * idx + 1] - y;
          if (std::fabs(distx) < r && std::fabs(disty) < r) out.push_back(idx);
        }
  }
};

// ORBmatcher::ComputeThreeMaxima
void three_maxima(const std::vector<int>* histo, int L, int& ind1, int& ind2, int& ind3) {
  int max1 = 0, max2 = 0, max3 = 0;
  for (int i = 0; i < L; i++) {
    const int s = (int)histo[i].size();
    if (s > max1) { max3 = max2; max2 = max1; max1 = s; ind3 = ind2; ind2 = ind1; ind1 = i; }
    else if (s > max2) { max3 = max2; max2 = s; ind3 = ind2; ind2 = i; }
    else if (s > max3) { max3 = s; ind3 = i; }
  }
  if (max2 < 0.1f * (float)max1) { ind2 = -1; ind3 = -1; }
  else if (max3 < 0.1f * (float)max1) { ind3 = -1; }
}

}  // namespace

extern "C" int lldo_init_search(void*, const lld_init_search_problem* p, lld_init_search_result* out) {
  const int TH_LOW = 50, HISTO_LENGTH = 30;
  const float factor = 1.0f / HISTO_LENGTH;
  std::vector<int> cand;
  for (int pr = 0; pr < p->n_pairs; pr++) {
    const int a0 = p->kp1_off[pr], n1 = p->kp1_off[pr + 1] - a0;
    const int b0 = p->kp2_off[pr], n2 = p->kp2_off[pr + 1] - b0;
    const float* xy2 = p->kp2_xy + 2 * (size_t)b0;
    Grid G;
    G.build(p->geom, xy2, n2);
    std::vector<int> vnMatches12(n1, -1), vMatchedDistance(n2, INT_MAX), vnMatches21(n2, -1);
    std::vector<int> rotHist[30];
    std::vector<float> prev(p->prev_matched + 2 * (size_t)a0, p->prev_matched + 2 * (size_t)(a0 + n1));
    int nmatches = 0;
    for (int i1 = 0; i1 < n1; i1++) {
      if (p->kp1_octave[a0 + i1] > 0) continue;
      G.features_in_area(prev[2 * i1], prev[2 * i1 + 1], (float)p->window_size, 0, 0, xy2, p->kp2_octave + b0, cand);
      if (cand.empty()) continue;
      const uint8_t* d1 = p->kp1_desc + 32 * (size_t)(a0 + i1);
      int bestDist = INT_MAX, bestDist2 = INT_MAX, bestIdx2 = -1;
      for (int i2 : cand) {
        const int dist = descriptor_distance(d1, p->kp2_desc + 32 * (size_t)(b0 + i2));
        if (vMatchedDistance[i2] <= dist) continue;
        if (dist < bestDist) { bestDist2 = bestDist; bestDist = dist; bestIdx2 = i2; }
        else if (dist < bestDist2) bestDist2 = dist;
      }
      if (bestDist <= TH_LOW && bestDist < (float)bestDist2 * p->nn_ratio) {
        if (vnMatches21[bestIdx2] >= 0) { vnMatches12[vnMatches21[bestIdx2]] = -1; nmatches--; }
        vnMatches12[i1] = bestIdx2;
        vnMatches21[bestIdx2] = i1;
        vMatchedDistance[bestIdx2] = bestDist;
        nmatches++;
        if (p->check_orientation) {
          float rot = p->kp1_angle[a0 + i1] - p->kp2_angle[b0 + bestIdx2];
          if (rot < 0.0) rot += 360.0f;
          int bin = (int)std::round(rot * factor);
          if (bin == HISTO_LENGTH) bin = 0;
          rotHist[bin].push_back(i1);
        }
      }
    }
    if (p->check_orientation) {
      int ind1 = -1, ind2 = -1, ind3 = -1;
      three_maxima(rotHist, HISTO_LENGTH, ind1, ind2, ind3);
      for (int i = 0; i < HISTO_LENGTH; i++) {
        if (i == ind1 || i == ind2 || i == ind3) continue;
        for (int idx1 : rotHist[i])
          if (vnMatches12[idx1] >= 0) { vnMatches12[idx1] = -1; nmatches--; }
      }
    }
    for (int i1 = 0; i1 < n1; i1++) {
      out->match12[a0 + i1] = vnMatches12[i1];
      const int m = vnMatches12[i1];
      out->prev_matched[2 * (size_t)(a0 + i1)] = m >= 0 ? xy2[2 * m] : prev[2 * i1];
      out->prev_matched[2 * (size_t)(a0 + i1) + 1] = m >= 0 ? xy2[2 * m + 1] : prev[2 * i1 + 1];
    }
    out->n_matches[pr] = nmatches;
  }
  return 0;
}
