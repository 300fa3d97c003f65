// lld_shim.h — C++ host shim that keeps the reference's class / method names over the C-ABI (include/lldba.h).
//
// The reference's KeyFrame / MapPoint / MapLine / Frame classes need OpenCV and the rest of the SLAM system; the shim
// works on POD mirrors that carry exactly the fields the hot path reads and writes, under the same names
// (include/KeyFrame.h, include/MapPoint.h, include/MapLine.h, include/Frame.h).  A maintainer dropping this into
// LLD-SLAM replaces the bodies of the corresponding members with the flatten -> lld_* -> write-back code below
// (INTEGRATION.md).  Header-only, C++14, no dependency besides include/lldba.h.
//
//   lld::Optimizer::LocalBundleAdjustment   <- src/Optimizer.cc:936-1388   (graph construction :1037-1218, write-back :1334-1386)
//   lld::Optimizer::BundleAdjustment        <- src/Optimizer.cc:321-559     (+ AddLineMinimalGlobal :149-247)
//   lld::Optimizer::GlobalBundleAdjustemnt  <- src/Optimizer.cc:312-319     (sic, the reference's spelling)
//   lld::Optimizer::PoseOptimization        <- src/Optimizer.cc:653-932
//   lld::LineOptimizer                      <- include/LineOptimizer.h:11-33, src/LineOptimizer.cc:28-201
//   lld::ORBmatcher::SearchByProjection     <- src/ORBmatcher.cc:1328-1470 (frame to frame), :45-129 (frame to map points) and
//                                              :1472-1599 (frame to keyframe, relocalisation)
//   lld::ORBmatcher::SearchForInitialization <- src/ORBmatcher.cc:405
//   lld::Optimizer::OptimizeSim3            <- src/Optimizer.cc:1656-1858
//   lld::TwoFrameLineMatcher::MatchLines    <- src/TwoFrameLineMatcher.cc:26-77
// Every entry point takes the library context as an extra first argument (the reference keeps its g2o optimizer on the
// stack instead); Flatten* expose the flattened problem so that tests can compare it array by array with a reference
// flattening (tests/hostcheck/shim_run.cpp).
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <map>
#include <set>
#include <utility>
#include <vector>

#include "../../include/lldba.h"

namespace lld {

struct KeyPoint { float x, y; int octave; float angle; };
struct Point2f { float x, y; };                  // cv::Point2f
struct Sim3 { double q[4], t[3], s; };           // g2o::Sim3: rotation (x y z w), translation, scale; map(x) = s (q x) + t
struct KeyLine { float startPointX, startPointY, endPointX, endPointY; int octave; };

struct KeyFrame {
  unsigned long mnId = 0;
  float Tcw[12];                       // R row-major + t  (GetPose(), CV_32F)
  float fx, fy, cx, cy, mbf;
  std::vector<float> mvInvLevelSigma2;
  std::vector<KeyPoint> mvKeysUn;
  std::vector<float> mvuRight;
  std::vector<KeyLine> mvLinesLeft, mvLinesRight;
  std::vector<int> line_matches;
  bool bad = false;
  bool isBad() const { return bad; }
  std::vector<struct MapPoint*> mvpMapPoints;   // GetMapPointMatches()
  // what the keyframe-targeted searches read (ORBmatcher::Fuse, SearchByProjection(KeyFrame*, Scw, ...)): include/KeyFrame.h:160-200
  float mnMinX = 0, mnMaxX = 0, mnMinY = 0, mnMaxY = 0;
  std::vector<float> mvScaleFactors;
  float mfLogScaleFactor = 0;
  int mnScaleLevels = 0;
  std::vector<uint8_t> mDescriptors;            // N x 32
  std::map<unsigned, std::vector<unsigned>> mFeatVec;   // DBoW2::FeatureVector: vocabulary node -> keypoint indices
  std::vector<float> mvLevelSigma2;
  bool IsInImage(float x, float y) const { return x >= mnMinX && x < mnMaxX && y >= mnMinY && y < mnMaxY; }   // src/KeyFrame.cc:639-642
  // GBA shadow fields (src/Optimizer.cc:509-512)
  float mTcwGBA[12];
  unsigned long mnBAGlobalForKF = 0;
};
struct MapPoint {
  unsigned long mnId = 0;
  float pos[3];                                      // GetWorldPos(), CV_32F
  std::map<KeyFrame*, size_t> observations;          // GetObservations()
  bool bad = false;
  bool isBad() const { return bad; }
  int Observations() const { return (int)observations.size(); }
  float mPosGBA[3];
  unsigned long mnBAGlobalForKF = 0;
  // Frame::isInFrustum results read by SearchByProjection(Frame&, vector<MapPoint*>&, th)  (include/MapPoint.h:88-95)
  bool mbTrackInView = false;
  float mTrackProjX = 0, mTrackProjY = 0, mTrackProjXR = 0, mTrackViewCos = 0;
  int mnTrackScaleLevel = 0;
  uint8_t mDescriptor[32] = {0};                     // GetDescriptor()
  float mNormalVector[3] = {0, 0, 1};                // GetNormal()
  bool IsInKeyFrame(KeyFrame* pKF) const { return observations.count(pKF) != 0; }
  int GetIndexInKeyFrame(KeyFrame* pKF) const {                 // src/MapPoint.cc
    auto it = observations.find(pKF);
    return it == observations.end() ? -1 : (int)it->second;
  }
  float mfMinDistance = 0, mfMaxDistance = 0;        // scale-invariance range (src/MapPoint.cc:373-383)
  float GetMinDistanceInvariance() const { return 0.8f * mfMinDistance; }
  float GetMaxDistanceInvariance() const { return 1.2f * mfMaxDistance; }
  // int MapPoint::PredictScale(const float&, Frame*)  src/MapPoint.cc:402-417
  int PredictScale(float currentDist, float mfLogScaleFactor, int mnScaleLevels) const {
    const float ratio = mfMaxDistance / currentDist;
    int nScale = (int)std::ceil(std::log(ratio) / mfLogScaleFactor);
    if (nScale < 0) nScale = 0;
    else if (nScale >= mnScaleLevels) nScale = mnScaleLevels - 1;
    return nScale;
  }
};
struct MapLine {
  unsigned long mnId = 0;
  double X0[3], line_dir[3];                         // GetMinimalPos(): doubles (include/MapLine.h:120)
  std::map<KeyFrame*, size_t> observations;
  bool bad = false;
  bool isBad() const { return bad; }
  int Observations() const { return (int)observations.size(); }
};
struct Map {                                          // the three getters GlobalBundleAdjustemnt uses (src/Optimizer.cc:314-317)
  std::vector<KeyFrame*> keyframes;
  std::vector<MapPoint*> points;
  std::vector<MapLine*> lines;
  std::vector<KeyFrame*> GetAllKeyFrames() const { return keyframes; }
  std::vector<MapPoint*> GetAllMapPoints() const { return points; }
  std::vector<MapLine*> GetAllMapLines() const { return lines; }
};
struct Frame {
  float mTcw[12];
  float fx, fy, cx, cy, mbf, mb;
  float mnMinX, mnMaxX, mnMinY, mnMaxY;
  std::vector<float> mvScaleFactors, mvInvLevelSigma2;
  float mfLogScaleFactor = 0;
  int mnScaleLevels = 0;
  int N = 0;
  std::vector<KeyPoint> mvKeys, mvKeysUn;
  std::vector<float> mvuRight;
  std::vector<uint8_t> mDescriptors;                  // N x 32
  std::vector<MapPoint*> mvpMapPoints;
  std::vector<uint8_t> mvpMapPointDesc;               // descriptor of mvpMapPoints[i] (pMP->GetDescriptor()), N x 32
  std::vector<uint8_t> mvpMapPointHasObs;             // pMP->Observations() > 0
  std::vector<bool> mvbOutlier;
  std::vector<KeyLine> mvLinesLeft, mvLinesRight;
  std::vector<int> line_matches;
  std::vector<MapLine*> mvpMapLines;
  std::vector<bool> mvbOutlierLines;
};

// LinePyrFactor = 1.44, GetReprojThrPyramid  (src/LineMatching.cc:27,239-247)
inline double GetReprojThrPyramid(double base, int lev) {
  double t = base;
  for (int i = 0; i < lev; i++) t *= 1.44;
  return t;
}

namespace detail {
inline void widen12(const float* T, std::vector<double>& out) { for (int i = 0; i < 12; i++) out.push_back((double)T[i]); }
}

// The flattened bundle-adjustment problem of ONE window (lld_ba_problem with n_win = 1) plus the owners needed to write
// the result back into the caller's objects.
struct FlatBA {
  std::vector<KeyFrame*> kfs;                    // window-local keyframe index -> object
  std::map<KeyFrame*, int> kf_index;
  std::map<int, int> kf_index_by_id;             // mnId -> window-local index (LineOptimizer::AddLineMinimal is keyed by id)
  std::vector<double> T, intr, lcam, pxyz, lxd, linfo;
  std::vector<uint8_t> fixed, lstereo;
  std::vector<int32_t> poff{0}, pkf, loff{0}, lkf;
  std::vector<float> puvr, pinfo, lleft, lright;
  std::vector<std::pair<KeyFrame*, MapPoint*>> edge_owner;   // one per point observation
  std::vector<MapPoint*> points;                              // one per flattened point
  std::vector<int> line_ids;                                  // one per flattened line (AddLineMinimal's line_id)
  int32_t one_kf[2] = {0, 0}, one_pt[2] = {0, 0}, one_ln[2] = {0, 0};
  lld_ba_problem p;
  // results
  std::vector<double> oT, oP, oL;
  std::vector<uint8_t> pbad, lbad, lrem;
  lld_ba_result r;

  int AddKeyFrame(KeyFrame* k, bool is_fixed, const double line_cam[4]) {
    const int i = (int)kfs.size();
    kfs.push_back(k); kf_index[k] = i; kf_index_by_id[(int)k->mnId] = i;
    for (int c = 0; c < 12; c++) T.push_back((double)k->Tcw[c]);          // Converter::toSE3Quat(pKF->GetPose())
    fixed.push_back(is_fixed);
    const double in[5] = {k->fx, k->fy, k->cx, k->cy, k->mbf};
    intr.insert(intr.end(), in, in + 5);
    lcam.insert(lcam.end(), line_cam, line_cam + 4);
    return i;
  }
  // binds the pointers; call after the last Add*
  void Finish() {
    one_kf[1] = (int32_t)kfs.size(); one_pt[1] = (int32_t)points.size(); one_ln[1] = (int32_t)line_ids.size();
    std::memset(&p, 0, sizeof(p));
    p.n_win = 1; p.kf_off = one_kf; p.pt_off = one_pt; p.ln_off = one_ln;
    p.kf_Tcw = T.data(); p.kf_fixed = fixed.data(); p.kf_intr = intr.data(); p.kf_line_cam = lcam.data();
    p.pt_xyz = pxyz.data(); p.pt_obs_off = poff.data(); p.pt_obs_kf = pkf.data(); p.pt_obs_uvr = puvr.data(); p.pt_obs_info = pinfo.data();
    p.ln_x0_dir = lxd.data(); p.ln_obs_off = loff.data(); p.ln_obs_kf = lkf.data(); p.ln_obs_left = lleft.data();
    p.ln_obs_right = lright.data(); p.ln_obs_info = linfo.data(); p.ln_obs_stereo = lstereo.data();
    oT.assign(T.size(), 0.0); oP.assign(pxyz.size(), 0.0); oL.assign(lxd.size(), 0.0);
    pbad.assign(pkf.size() + 1, 0); lbad.assign(2 * lkf.size() + 2, 0); lrem.assign(line_ids.size() + 1, 0);
    std::memset(&r, 0, sizeof(r));
    r.kf_Tcw = oT.data(); r.pt_xyz = oP.data(); r.ln_x0_dir = oL.data();
    r.pt_obs_bad = pbad.data(); r.ln_obs_bad = lbad.data(); r.ln_removed = lrem.data();
  }
};

// include/LineOptimizer.h:11-33.  The reference class adds VertexSBALine / EdgeSE3ProjectLine objects to a g2o optimizer;
// here it appends the same edges, in the same order, to the flattened problem.  DisableOutliers runs on the device between
// the two rounds of lld_ba_local (k_flag_lines), GetLineData reads the result arrays.
class LineOptimizer {
 public:
  LineOptimizer(FlatBA& flat, int maxPtId, double thHuberLinesStereo, double thHuberLinesMono, double gamma)
      : flat_(flat), maxPtId_(maxPtId), thStereo_(thHuberLinesStereo * gamma), thMono_(thHuberLinesMono * gamma), infoLines_(gamma * gamma) {}
  double thHuberLinesStereo() const { return thStereo_; }
  double thHuberLinesMono() const { return thMono_; }
  // src/LineOptimizer.cc:39-127.  proj_map: keyframe id -> (left KeyLine, right KeyLine with startPointX < 0 when absent).
  // K and stereo_b are per call in the reference but LocalBundleAdjustment passes the current keyframe's for every line
  // (src/Optimizer.cc:1211-1215); they were given to FlatBA::AddKeyFrame as line_cam.
  void AddLineMinimal(int line_id, const double X0[3], const double line_dir[3],
                      const std::map<int, std::pair<KeyLine, KeyLine>>& proj_map) {
    for (int c = 0; c < 3; c++) flat_.lxd.push_back(X0[c]);
    for (int c = 0; c < 3; c++) flat_.lxd.push_back(line_dir[c]);
    line_row_[line_id] = (int)flat_.line_ids.size();
    flat_.line_ids.push_back(line_id);
    for (auto& kv : proj_map) {                       // std::map order = ascending keyframe id (:59)
      const auto it = flat_.kf_index_by_id.find(kv.first);
      if (it == flat_.kf_index_by_id.end()) continue;  // optimizer.vertex(kf_id) would be null in the reference
      const KeyLine& kl = kv.second.first;
      const KeyLine& kr = kv.second.second;
      const bool stereo = !(kr.startPointX < 0);      // :65-68, 83-88
      flat_.lkf.push_back(it->second);
      const float l4[4] = {kl.startPointX, kl.startPointY, kl.endPointX, kl.endPointY};
      flat_.lleft.insert(flat_.lleft.end(), l4, l4 + 4);
      const float r4[4] = {stereo ? kr.startPointX : -1.f, stereo ? kr.startPointY : -1.f, stereo ? kr.endPointX : -1.f, stereo ? kr.endPointY : -1.f};
      flat_.lright.insert(flat_.lright.end(), r4, r4 + 4);
      const double thrL = GetReprojThrPyramid(1.0, kl.octave), thrR = stereo ? GetReprojThrPyramid(1.0, kr.octave) : thrL;
      flat_.linfo.push_back(infoLines_ / (thrL * thrL));   // :97-101
      flat_.linfo.push_back(infoLines_ / (thrR * thrR));
      flat_.lstereo.push_back(stereo);
    }
    flat_.loff.push_back((int32_t)flat_.lkf.size());
  }
  void DisableOutliers() {}   // src/LineOptimizer.cc:129-170: part of lld_ba_local
  // src/LineOptimizer.cc:172-201; valid after the optimisation ran.  false: the line vertex was removed by DisableOutliers.
  bool GetLineData(int line_id, double X0[3], double line_dir[3], std::vector<int>* outlier_projs) const {
    const auto it = line_row_.find(line_id);
    if (it == line_row_.end()) return false;
    const int i = it->second;
    if (flat_.lrem[(size_t)i]) return false;
    for (int c = 0; c < 3; c++) { X0[c] = flat_.oL[6 * (size_t)i + c]; line_dir[c] = flat_.oL[6 * (size_t)i + 3 + c]; }
    for (int c = flat_.loff[(size_t)i]; c < flat_.loff[(size_t)i + 1]; c++)
      for (int s = 0; s < 2; s++)
        if (flat_.lbad[2 * (size_t)c + s]) outlier_projs->push_back((int)flat_.kfs[(size_t)flat_.lkf[(size_t)c]]->mnId);   // one entry per bad edge
    return true;
  }
 private:
  FlatBA& flat_;
  int maxPtId_;
  double thStereo_, thMono_, infoLines_;
  std::map<int, int> line_row_;
};

// The sets LocalBundleAdjustment gathers before building the graph (src/Optimizer.cc:938-1018).
struct LocalWindow {
  KeyFrame* pKF = nullptr;                    // current keyframe (its K and baseline drive every line edge)
  std::vector<KeyFrame*> lLocalKeyFrames;     // optimised (fixed only when mnId==0)
  std::vector<KeyFrame*> lFixedCameras;
  std::vector<MapPoint*> lLocalMapPoints;
  std::vector<MapLine*> lLocalMapLines;       // already filtered by Observations()>=4 (:974)
};
struct LocalBAResult {
  std::vector<std::pair<KeyFrame*, MapPoint*>> vToErase;       // src/Optimizer.cc:1278-1311
  std::vector<std::pair<KeyFrame*, MapLine*>> vToEraseLines;   // :1313-1329
};

class Optimizer {
 public:
  // graph construction of LocalBundleAdjustment, src/Optimizer.cc:1037-1218, as flat arrays
  static void FlattenLocal(const LocalWindow& w, double gamma, FlatBA* F, LineOptimizer** lo_out = nullptr) {
    const float baseline = w.pKF->mbf / w.pKF->fx;   // pKF->mbf / pKF->mK.at<float>(0,0): float division (:1215)
    const double lc[4] = {w.pKF->fx, w.pKF->cx, w.pKF->cy, baseline};  // current KF's K for every line edge (:1211-1215)
    for (KeyFrame* k : w.lLocalKeyFrames) F->AddKeyFrame(k, k->mnId == 0, lc);   // :1043
    for (KeyFrame* k : w.lFixedCameras) F->AddKeyFrame(k, true, lc);             // :1057
    unsigned long maxPtId = 0;
    for (MapPoint* mp : w.lLocalMapPoints) {
      for (int c = 0; c < 3; c++) F->pxyz.push_back((double)mp->pos[c]);
      F->points.push_back(mp);
      if (mp->mnId > maxPtId) maxPtId = mp->mnId;
      for (auto& ob : mp->observations) {          // std::map<KeyFrame*, size_t>: pointer order, as the reference iterates (:1107-1110)
        KeyFrame* k = ob.first;
        if (k->isBad() || !F->kf_index.count(k)) continue;
        const KeyPoint& kp = k->mvKeysUn[ob.second];
        F->pkf.push_back(F->kf_index[k]);
        F->puvr.push_back(kp.x); F->puvr.push_back(kp.y); F->puvr.push_back(k->mvuRight[ob.second]);
        F->pinfo.push_back(k->mvInvLevelSigma2[kp.octave]);
        F->edge_owner.push_back({k, mp});
      }
      F->poff.push_back((int32_t)F->pkf.size());
    }
    const float thHuberMono = (float)std::sqrt(5.991), thHuberStereo = (float)std::sqrt(7.815);   // const float = sqrt(double) (:1088-1089)
    LineOptimizer* lo = new LineOptimizer(*F, (int)maxPtId, thHuberStereo, thHuberMono, gamma);    // :1180-1182
    for (MapLine* ml : w.lLocalMapLines) {
      std::map<int, std::pair<KeyLine, KeyLine>> proj_map;      // keyed by keyframe id (:1189-1209)
      for (auto& ob : ml->observations) {
        KeyFrame* k = ob.first;
        if (k->isBad() || !F->kf_index.count(k)) continue;
        const size_t li = ob.second;
        KeyLine right;
        right.startPointX = -1;                                   // "no right line" marker (:1200-1206)
        right.startPointY = right.endPointX = right.endPointY = -1; right.octave = 0;
        if (k->line_matches[li] >= 0) right = k->mvLinesRight[k->line_matches[li]];
        proj_map[(int)k->mnId] = {k->mvLinesLeft[li], right};
      }
      lo->AddLineMinimal((int)ml->mnId, ml->X0, ml->line_dir, proj_map);
    }
    F->Finish();
    lld_ba_problem& p = F->p;
    p.robust_points = 1;
    p.delta_pt_mono = thHuberMono; p.delta_pt_stereo = thHuberStereo;
    p.delta_ln_mono = lo->thHuberLinesMono(); p.delta_ln_stereo = lo->thHuberLinesStereo();
    p.chi2_pt_mono = 5.991; p.chi2_pt_stereo = 7.815; p.ln_endpoints_normalized = 0; p.ln_filter = 4;
    if (lo_out) *lo_out = lo;
    else delete lo;
  }

  // void static LocalBundleAdjustment(KeyFrame* pKF, bool* pbStopFlag, Map* pMap, double gamma = 1.0)  include/Optimizer.h:49
  static int LocalBundleAdjustment(void* ctx, const LocalWindow& w, bool* pbStopFlag, double gamma, LocalBAResult* res) {
    FlatBA F;
    LineOptimizer* lo = nullptr;
    FlattenLocal(w, gamma, &F, &lo);
    struct Guard { LineOptimizer* p; ~Guard() { delete p; } } guard{lo};
    if (pbStopFlag && *pbStopFlag) return 0;   // :1220-1222 nothing is written back
    // pbStopFlag is a bool written by another thread; bool and uint8_t share their object representation here
    const volatile uint8_t* sp = pbStopFlag ? reinterpret_cast<const volatile uint8_t*>(pbStopFlag) : nullptr;
    const int rc = lld_ba_local(ctx, &F.p, 5, 15, sp, &F.r);
    if (rc) return rc;
    // write-back (under the map mutex in the reference, :1334-1386); float narrowing as Converter::toCvMat
    if (res) {
      for (size_t e = 0; e < F.pkf.size(); e++)
        if (F.pbad[e] && !F.edge_owner[e].second->isBad()) res->vToErase.push_back(F.edge_owner[e]);   // pMP->isBad() is skipped (:1284,1299)
      for (size_t i = 0; i < w.lLocalMapLines.size(); i++) {                                             // :1313-1329
        double X0[3], dir[3];
        std::vector<int> bad_obs;
        if (!lo->GetLineData((int)w.lLocalMapLines[i]->mnId, X0, dir, &bad_obs)) continue;
        for (int id : bad_obs) res->vToEraseLines.push_back({F.kfs[(size_t)F.kf_index_by_id[id]], w.lLocalMapLines[i]});
      }
    }
    for (size_t i = 0; i < w.lLocalKeyFrames.size(); i++)
      for (int c = 0; c < 12; c++) F.kfs[i]->Tcw[c] = (float)F.oT[12 * i + c];
    for (size_t i = 0; i < w.lLocalMapPoints.size(); i++)
      for (int c = 0; c < 3; c++) w.lLocalMapPoints[i]->pos[c] = (float)F.oP[3 * i + c];
    for (size_t i = 0; i < w.lLocalMapLines.size(); i++) {
      double X0[3], dir[3];
      std::vector<int> unused;
      if (!lo->GetLineData((int)w.lLocalMapLines[i]->mnId, X0, dir, &unused)) continue;   // removed: SetMinimalPos is not called
      for (int c = 0; c < 3; c++) { w.lLocalMapLines[i]->X0[c] = X0[c]; w.lLocalMapLines[i]->line_dir[c] = dir[c]; }
    }
    return 0;
  }

  // graph construction of BundleAdjustment, src/Optimizer.cc:341-488 (+ AddLineMinimalGlobal :149-247).
  // included_pt / included_ln: !vbNotIncludedMP / !vbNotIncludedML.
  // Carve-outs of undefined behaviour in the reference, resolved as documented in DESIGN.md: mvInvLevelSigma2[octave*2]
  // (:405,428) reads past the 8-level table for octave >= 4 — the index is clamped to the last level; a line observation
  // without a right match makes AddLineMinimalGlobal read mvLinesRight[-1] (:226-230) — no right edge is created.
  static void FlattenGlobal(const std::vector<KeyFrame*>& vpKFs, const std::vector<MapPoint*>& vpMP, const std::vector<MapLine*>& vpML,
                            bool bRobust, FlatBA* F, std::vector<bool>* included_pt, std::vector<bool>* included_ln) {
    unsigned long maxKFid = 0;
    for (KeyFrame* k : vpKFs) {
      if (k->isBad()) continue;
      const float bl = k->mbf / k->fx;                       // pKFi->mbf / pKFi->mK.at<float>(0,0)  (:207)
      const double lc[4] = {k->fx, k->cx, k->cy, bl};        // each keyframe's own K (:200-202)
      F->AddKeyFrame(k, k->mnId == 0, lc);                   // :348-352
      if (k->mnId > maxKFid) maxKFid = k->mnId;
    }
    included_pt->assign(vpMP.size(), false);
    included_ln->assign(vpML.size(), false);
    for (size_t i = 0; i < vpMP.size(); i++) {
      MapPoint* mp = vpMP[i];
      if (mp->isBad()) continue;
      const size_t e0 = F->pkf.size();
      for (auto& ob : mp->observations) {
        KeyFrame* k = ob.first;
        if (k->isBad() || k->mnId > maxKFid || !F->kf_index.count(k)) continue;   // :393-394
        const KeyPoint& kp = k->mvKeysUn[ob.second];
        F->pkf.push_back(F->kf_index[k]);
        F->puvr.push_back(kp.x); F->puvr.push_back(kp.y); F->puvr.push_back(k->mvuRight[ob.second]);
        const size_t lvl = std::min<size_t>((size_t)kp.octave * 2, k->mvInvLevelSigma2.size() - 1);
        F->pinfo.push_back(k->mvInvLevelSigma2[lvl]);
        F->edge_owner.push_back({k, mp});
      }
      if (F->pkf.size() == e0) continue;                     // nEdges == 0: vertex removed (:456-460)
      (*included_pt)[i] = true;
      for (int c = 0; c < 3; c++) F->pxyz.push_back((double)mp->pos[c]);
      F->points.push_back(mp);
      F->poff.push_back((int32_t)F->pkf.size());
    }
    for (size_t i = 0; i < vpML.size(); i++) {
      MapLine* ml = vpML[i];
      if (!ml || ml->isBad() || ml->Observations() < 4) continue;   // :473
      const size_t c0 = F->lkf.size();
      for (auto& ob : ml->observations) {                    // std::map<KeyFrame*, size_t>: pointer order (:176)
        KeyFrame* k = ob.first;
        if (k->isBad() || !F->kf_index.count(k)) continue;
        const size_t li = ob.second;
        const KeyLine& kl = k->mvLinesLeft[li];
        F->lkf.push_back(F->kf_index[k]);
        const float l4[4] = {kl.startPointX, kl.startPointY, kl.endPointX, kl.endPointY};
        F->lleft.insert(F->lleft.end(), l4, l4 + 4);
        if (k->line_matches[li] >= 0) {
          const KeyLine& kr = k->mvLinesRight[k->line_matches[li]];
          const float r4[4] = {kr.startPointX, kr.startPointY, kr.endPointX, kr.endPointY};
          F->lright.insert(F->lright.end(), r4, r4 + 4);
        } else {
          const float r4[4] = {-1, -1, -1, -1};
          F->lright.insert(F->lright.end(), r4, r4 + 4);
        }
        F->linfo.push_back(1.0); F->linfo.push_back(1.0);    // setInformation(Identity) (:216)
        F->lstereo.push_back(1);                             // one Huber delta for every line edge (:218-220)
      }
      if (F->lkf.size() == c0) continue;                     // edge_cnt == 0 (:242-245)
      (*included_ln)[i] = true;
      for (int c = 0; c < 3; c++) F->lxd.push_back(ml->X0[c]);
      for (int c = 0; c < 3; c++) F->lxd.push_back(ml->line_dir[c]);
      F->line_ids.push_back((int)ml->mnId);
      F->loff.push_back((int32_t)F->lkf.size());
    }
    F->Finish();
    lld_ba_problem& p = F->p;
    const float thHuber2D = (float)std::sqrt(5.99), thHuber3D = (float)std::sqrt(7.815);   // :359-360
    p.robust_points = bRobust ? 1 : 0;
    p.delta_pt_mono = thHuber2D; p.delta_pt_stereo = thHuber3D;
    p.delta_ln_mono = p.delta_ln_stereo = thHuber3D / 2.0;                                  // :361
    p.chi2_pt_mono = 5.991; p.chi2_pt_stereo = 7.815; p.ln_endpoints_normalized = 1; p.ln_filter = 4;
  }

  // void static BundleAdjustment(const vector<KeyFrame*>&, const vector<MapPoint*>&, const vector<MapLine*>&, int nIterations = 5,
  //                              bool* pbStopFlag = NULL, const unsigned long nLoopKF = 0, const bool bRobust = true)   include/Optimizer.h:43-45
  static int BundleAdjustment(void* ctx, const std::vector<KeyFrame*>& vpKFs, const std::vector<MapPoint*>& vpMP,
                              const std::vector<MapLine*>& vpML, int nIterations = 5, bool* pbStopFlag = nullptr,
                              const unsigned long nLoopKF = 0, const bool bRobust = true) {
    FlatBA F;
    std::vector<bool> inc_pt, inc_ln;
    FlattenGlobal(vpKFs, vpMP, vpML, bRobust, &F, &inc_pt, &inc_ln);
    const volatile uint8_t* sp = pbStopFlag ? reinterpret_cast<const volatile uint8_t*>(pbStopFlag) : nullptr;
    const int rc = lld_ba_global(ctx, &F.p, nIterations, sp, &F.r);
    if (rc) return rc;
    // :494-557: live state when nLoopKF == 0, the *GBA shadow fields otherwise
    for (size_t i = 0; i < F.kfs.size(); i++) {
      KeyFrame* k = F.kfs[i];
      float* dst = nLoopKF == 0 ? k->Tcw : k->mTcwGBA;
      for (int c = 0; c < 12; c++) dst[c] = (float)F.oT[12 * i + c];
      if (nLoopKF != 0) k->mnBAGlobalForKF = nLoopKF;
    }
    for (size_t i = 0; i < F.points.size(); i++) {
      MapPoint* mp = F.points[i];
      float* dst = nLoopKF == 0 ? mp->pos : mp->mPosGBA;
      for (int c = 0; c < 3; c++) dst[c] = (float)F.oP[3 * i + c];
      if (nLoopKF != 0) mp->mnBAGlobalForKF = nLoopKF;
    }
    // lines: SetMinimalPos for every included line (the reference tests vbNotIncludedMP[i] here, :542 — a typo that indexes
    // the point flags with a line index; the shim uses the line flags)
    size_t row = 0;
    for (size_t i = 0; i < vpML.size(); i++) {
      if (!inc_ln[i]) continue;
      for (int c = 0; c < 3; c++) { vpML[i]->X0[c] = F.oL[6 * row + c]; vpML[i]->line_dir[c] = F.oL[6 * row + 3 + c]; }
      row++;
    }
    return 0;
  }

  // void static GlobalBundleAdjustemnt(Map* pMap, int nIterations = 5, bool* pbStopFlag = NULL, const unsigned long nLoopKF = 0,
  //                                    const bool bRobust = true)    include/Optimizer.h:46-47, src/Optimizer.cc:312-319
  static int GlobalBundleAdjustemnt(void* ctx, Map* pMap, int nIterations = 5, bool* pbStopFlag = nullptr, const unsigned long nLoopKF = 0,
                                    const bool bRobust = true) {
    return BundleAdjustment(ctx, pMap->GetAllKeyFrames(), pMap->GetAllMapPoints(), pMap->GetAllMapLines(), nIterations, pbStopFlag,
                            nLoopKF, bRobust);
  }

  // int static PoseOptimization(Frame* pFrame, double gamma = 1.0)   include/Optimizer.h:50
  static int PoseOptimization(void* ctx, Frame* F, double gamma = 1.0) {
    std::vector<float> xw, uvr, info, left, right;
    std::vector<double> x0d, linfo;
    std::vector<uint8_t> lst, lgate;
    std::vector<int> pidx, lidx;
    for (int i = 0; i < F->N; i++) {
      MapPoint* mp = F->mvpMapPoints[i];
      if (!mp) continue;
      F->mvbOutlier[i] = false;
      pidx.push_back(i);
      for (int c = 0; c < 3; c++) xw.push_back(mp->pos[c]);
      uvr.push_back(F->mvKeysUn[i].x); uvr.push_back(F->mvKeysUn[i].y); uvr.push_back(F->mvuRight[i]);
      info.push_back(F->mvInvLevelSigma2[F->mvKeysUn[i].octave]);
    }
    std::vector<bool> vnStereoLines;   // one entry per EDGE, indexed by LINE id in the reference (:894-898)
    for (size_t i = 0; i < F->mvpMapLines.size(); i++) {
      MapLine* ml = F->mvpMapLines[i];
      if (!ml) continue;
      lidx.push_back((int)i);
      for (int c = 0; c < 3; c++) x0d.push_back(ml->X0[c]);
      for (int c = 0; c < 3; c++) x0d.push_back(ml->line_dir[c]);
      const KeyLine& kl = F->mvLinesLeft[i];
      const float l4[4] = {kl.startPointX, kl.startPointY, kl.endPointX, kl.endPointY};
      left.insert(left.end(), l4, l4 + 4);
      const bool st = F->line_matches[i] >= 0;
      double tl = GetReprojThrPyramid(1.0, kl.octave), tr = tl;
      if (st) {
        const KeyLine& kr = F->mvLinesRight[F->line_matches[i]];
        const float r4[4] = {kr.startPointX, kr.startPointY, kr.endPointX, kr.endPointY};
        right.insert(right.end(), r4, r4 + 4);
        tr = GetReprojThrPyramid(1.0, kr.octave);
      } else {
        const float r4[4] = {-1, -1, -1, -1};
        right.insert(right.end(), r4, r4 + 4);
      }
      linfo.push_back(gamma * gamma / (tl * tl)); linfo.push_back(gamma * gamma / (tr * tr));
      lst.push_back(st);
      vnStereoLines.push_back(st);
      if (st) vnStereoLines.push_back(st);
    }
    for (size_t j = 0; j < lidx.size(); j++)
      for (int s = 0; s < 2; s++) {
        const size_t idx = (size_t)lidx[j];   // the reference reads vnStereoLines[idx]; out of range -> own flag (carve-out)
        lgate.push_back(idx < vnStereoLines.size() ? (uint8_t)vnStereoLines[idx] : lst[j]);
      }
    std::vector<double> T;
    detail::widen12(F->mTcw, T);
    const double in[5] = {F->fx, F->fy, F->cx, F->cy, F->mbf};
    const float bl = F->mbf / F->fx;
    const double lc[4] = {F->fx, F->cx, F->cy, bl};
    const int32_t po[2] = {0, (int32_t)pidx.size()}, lo[2] = {0, (int32_t)lidx.size()};
    lld_pose_problem p;
    std::memset(&p, 0, sizeof(p));
    p.n_frames = 1; p.Tcw = T.data(); p.intr = in; p.line_cam = lc;
    p.pt_off = po; p.pt_xw = xw.data(); p.pt_uvr = uvr.data(); p.pt_info = info.data();
    p.ln_off = lo; p.ln_x0_dir = x0d.data(); p.ln_left = left.data(); p.ln_right = right.data(); p.ln_info = linfo.data();
    p.ln_stereo = lst.data(); p.ln_gate_stereo = lgate.data();
    const float dM = (float)std::sqrt(5.991), dS = (float)std::sqrt(7.815);
    float dLS = dS, dLM = dM;
    dLS *= gamma; dLM *= gamma;                      // float *= double (:702-703)
    p.delta_mono = dM; p.delta_stereo = dS; p.delta_ln_mono = dLM; p.delta_ln_stereo = dLS;
    p.chi2_mono = 5.991f; p.chi2_stereo = 7.815f;
    p.gate_ln_mono = (double)(dLM * dLM); p.gate_ln_stereo = (double)(dLS * dLS);
    p.n_rounds = 4; p.its = 10;
    std::vector<double> oT(12);
    std::vector<uint8_t> po_(pidx.size() + 1), lo_(lidx.size() + 1);
    int n_inl = 0;
    lld_pose_result r;
    std::memset(&r, 0, sizeof(r));
    r.Tcw = oT.data(); r.pt_outlier = po_.data(); r.ln_outlier = lo_.data(); r.n_inliers = &n_inl;
    const int rc = lld_pose_opt(ctx, &p, &r);
    if (rc) return rc;
    if (pidx.size() < 3) return 0;
    for (size_t j = 0; j < pidx.size(); j++) F->mvbOutlier[pidx[j]] = po_[j] != 0;
    for (size_t j = 0; j < lidx.size(); j++) F->mvbOutlierLines[lidx[j]] = lo_[j] != 0;
    for (int c = 0; c < 12; c++) F->mTcw[c] = (float)oT[c];
    return n_inl;
  }

  // int static OptimizeSim3(KeyFrame* pKF1, KeyFrame* pKF2, vector<MapPoint*>& vpMatches1, g2o::Sim3& g2oS12, const float th2,
  //                         const bool bFixScale)   include/Optimizer.h, src/Optimizer.cc:1656-1858
  // Correspondences without a map point in pKF1, with a bad point or with a point not in pKF2 are skipped and their vpMatches1
  // entries left as they are; P1c / P2c in float (cv::Mat: R * X + t accumulates in double and rounds once) -> lld_sim3_opt ->
  // vpMatches1[i] cleared for the dropped correspondences, g2oS12 written unless fewer than 10 correspondences survived.
  static int OptimizeSim3(void* ctx, KeyFrame* pKF1, KeyFrame* pKF2, std::vector<MapPoint*>& vpMatches1, Sim3& g2oS12, const float th2,
                          const bool bFixScale) {
    const std::vector<MapPoint*>& vpMapPoints1 = pKF1->mvpMapPoints;   // GetMapPointMatches()
    std::vector<float> p1c, p2c, obs1, obs2, info1, info2;
    std::vector<size_t> vnIndexEdge;
    auto cam_frame = [](const KeyFrame* k, const float* X, std::vector<float>& out) {
      const float* T = k->Tcw;
      for (int r = 0; r < 3; r++)
        out.push_back((float)((double)T[3 * r] * X[0] + (double)T[3 * r + 1] * X[1] + (double)T[3 * r + 2] * X[2] + (double)T[9 + r]));
    };
    for (size_t i = 0; i < vpMatches1.size(); i++) {
      if (!vpMatches1[i]) continue;
      MapPoint* pMP1 = vpMapPoints1[i];
      MapPoint* pMP2 = vpMatches1[i];
      const int i2 = pMP2->GetIndexInKeyFrame(pKF2);
      if (!pMP1 || pMP1->isBad() || pMP2->isBad() || i2 < 0) continue;
      cam_frame(pKF1, pMP1->pos, p1c);
      cam_frame(pKF2, pMP2->pos, p2c);
      const KeyPoint& k1 = pKF1->mvKeysUn[i];
      const KeyPoint& k2 = pKF2->mvKeysUn[(size_t)i2];
      obs1.push_back(k1.x); obs1.push_back(k1.y);
      obs2.push_back(k2.x); obs2.push_back(k2.y);
      info1.push_back(pKF1->mvInvLevelSigma2[k1.octave]);
      info2.push_back(pKF2->mvInvLevelSigma2[k2.octave]);
      vnIndexEdge.push_back(i);
    }
    const int m = (int)vnIndexEdge.size();
    double S[8] = {g2oS12.q[0], g2oS12.q[1], g2oS12.q[2], g2oS12.q[3], g2oS12.t[0], g2oS12.t[1], g2oS12.t[2], g2oS12.s};
    const double cam[8] = {pKF1->fx, pKF1->fy, pKF1->cx, pKF1->cy, pKF2->fx, pKF2->fy, pKF2->cx, pKF2->cy};
    const int32_t fix = bFixScale ? 1 : 0, off[2] = {0, m};
    lld_sim3_problem p;
    std::memset(&p, 0, sizeof(p));
    p.n_problems = 1; p.S12 = S; p.cam = cam; p.fix_scale = &fix; p.th2 = &th2; p.off = off;
    p.p1c = p1c.data(); p.p2c = p2c.data(); p.obs1 = obs1.data(); p.obs2 = obs2.data(); p.info1 = info1.data(); p.info2 = info2.data();
    p.its_first = 5; p.its_more_outliers = 10; p.its_more_clean = 5;
    double oS[8];
    std::vector<uint8_t> inl((size_t)m + 1);
    int32_t n_in = 0;
    lld_sim3_result r;
    std::memset(&r, 0, sizeof(r));
    r.S12 = oS; r.inlier = inl.data(); r.n_in = &n_in;
    const int rc = lld_sim3_opt(ctx, &p, &r);
    if (rc) return rc;
    for (int j = 0; j < m; j++)
      if (!inl[j]) vpMatches1[vnIndexEdge[j]] = nullptr;
    for (int k = 0; k < 4; k++) g2oS12.q[k] = oS[k];   // the early return hands the input back: g2oS12 keeps its value
    for (int k = 0; k < 3; k++) g2oS12.t[k] = oS[4 + k];
    g2oS12.s = oS[7];
    return n_in;
  }
};

class ORBmatcher {
 public:
  ORBmatcher(float nnratio = 0.6f, bool checkOri = true) : mfNNratio(nnratio), mbCheckOrientation(checkOri) {}
  static int DescriptorDistance(const uint8_t* a, const uint8_t* b) { return lld_descriptor_distance(a, b); }
  // int SearchByProjection(Frame &CurrentFrame, const Frame &LastFrame, const float th, const bool bMono)  include/ORBmatcher.h:52
  int SearchByProjection(void* ctx, Frame& Cur, const Frame& Last, float th, bool bMono, std::vector<int>* match_out) {
    lld_sbp_frame_problem p;
    std::memset(&p, 0, sizeof(p));
    p.n_pairs = 1;
    p.geom.fx = Cur.fx; p.geom.fy = Cur.fy; p.geom.cx = Cur.cx; p.geom.cy = Cur.cy; p.geom.bf = Cur.mbf; p.geom.b = Cur.mb;
    p.geom.min_x = Cur.mnMinX; p.geom.max_x = Cur.mnMaxX; p.geom.min_y = Cur.mnMinY; p.geom.max_y = Cur.mnMaxY;
    p.geom.n_levels = (int)Cur.mvScaleFactors.size(); p.geom.scale_factors = Cur.mvScaleFactors.data();
    p.th = th; p.mono = bMono; p.check_orientation = mbCheckOrientation;
    std::vector<float> cxy, cang, lxw, lang;
    std::vector<uint8_t> coct, cclaimed, lvalid, loct, lhas, ldesc(32 * (size_t)Last.N, 0);
    for (int i = 0; i < Cur.N; i++) {
      cxy.push_back(Cur.mvKeysUn[i].x); cxy.push_back(Cur.mvKeysUn[i].y);
      coct.push_back((uint8_t)Cur.mvKeysUn[i].octave); cang.push_back(Cur.mvKeysUn[i].angle);
      cclaimed.push_back(Cur.mvpMapPoints[i] && Cur.mvpMapPointHasObs[i]);
    }
    for (int i = 0; i < Last.N; i++) {
      MapPoint* mp = Last.mvpMapPoints[i];
      const bool ok = mp && !Last.mvbOutlier[i];
      lvalid.push_back(ok);
      for (int c = 0; c < 3; c++) lxw.push_back(ok ? mp->pos[c] : 0.f);
      loct.push_back((uint8_t)Last.mvKeys[i].octave); lang.push_back(Last.mvKeysUn[i].angle);
      lhas.push_back(ok && Last.mvpMapPointHasObs[i]);
      if (ok) std::memcpy(&ldesc[32 * (size_t)i], &Last.mvpMapPointDesc[32 * (size_t)i], 32);
    }
    const int32_t co[2] = {0, Cur.N}, lo[2] = {0, Last.N};
    p.cur_off = co; p.cur_xy = cxy.data(); p.cur_octave = coct.data(); p.cur_angle = cang.data(); p.cur_uright = Cur.mvuRight.data();
    p.cur_desc = Cur.mDescriptors.data(); p.cur_claimed = cclaimed.data(); p.cur_Tcw = Cur.mTcw; p.last_Tcw = Last.mTcw;
    p.last_off = lo; p.last_valid = lvalid.data(); p.last_xw = lxw.data(); p.last_octave = loct.data(); p.last_angle = lang.data();
    p.last_desc = ldesc.data(); p.last_has_obs = lhas.data();
    std::vector<int32_t> match(Cur.N, -1);
    int32_t nm = 0;
    lld_sbp_result r;
    std::memset(&r, 0, sizeof(r));
    r.match = match.data(); r.n_matches = &nm;
    const int rc = lld_sbp_frame(ctx, &p, &r);
    if (rc) return rc;
    for (int i = 0; i < Cur.N; i++)
      if (match[i] >= 0) Cur.mvpMapPoints[i] = Last.mvpMapPoints[match[i]];
    if (match_out) match_out->assign(match.begin(), match.end());
    return nm;
  }
  // int SearchByProjection(Frame &CurrentFrame, KeyFrame* pKF, const std::set<MapPoint*> &sAlreadyFound, const float th, const int ORBdist)
  //   include/ORBmatcher.h:56, src/ORBmatcher.cc:1472-1599 (relocalisation).  The per-point tests that need the MapPoint object
  //   (already found, scale-invariance range, PredictScale) run here; projection, window search, claims and the rotation
  //   histogram run in lld_sbp_frame with the relocalisation parameters.
  int SearchByProjection(void* ctx, Frame& Cur, KeyFrame* pKF, const std::set<MapPoint*>& sAlreadyFound, float th, int ORBdist,
                         std::vector<int>* match_out = nullptr) {
    lld_sbp_frame_problem p;
    std::memset(&p, 0, sizeof(p));
    p.n_pairs = 1;
    p.geom.fx = Cur.fx; p.geom.fy = Cur.fy; p.geom.cx = Cur.cx; p.geom.cy = Cur.cy; p.geom.bf = Cur.mbf; p.geom.b = Cur.mb;
    p.geom.min_x = Cur.mnMinX; p.geom.max_x = Cur.mnMaxX; p.geom.min_y = Cur.mnMinY; p.geom.max_y = Cur.mnMaxY;
    p.geom.n_levels = (int)Cur.mvScaleFactors.size(); p.geom.scale_factors = Cur.mvScaleFactors.data();
    p.th = th; p.mono = 1; p.check_orientation = mbCheckOrientation;
    p.th_high = ORBdist; p.allow_negative_depth = 1;
    // Ow = -Rcw^T tcw: cv::Mat float product (double accumulation, one rounding)  :1476-1478
    float Ow[3];
    for (int i = 0; i < 3; i++)
      Ow[i] = (float)(-((double)Cur.mTcw[i] * (double)Cur.mTcw[9] + (double)Cur.mTcw[3 + i] * (double)Cur.mTcw[10] + (double)Cur.mTcw[6 + i] * (double)Cur.mTcw[11]));
    const std::vector<MapPoint*>& vpMPs = pKF->mvpMapPoints;
    const int nq = (int)vpMPs.size();
    std::vector<float> cxy, cang, cur(Cur.N > 0 ? Cur.N : 1, -1.0f), lxw(3 * (size_t)nq, 0.f), lang((size_t)nq, 0.f);
    std::vector<uint8_t> coct, cclaimed, lvalid((size_t)nq, 0), loct((size_t)nq, 0), lhas((size_t)nq, 1), ldesc(32 * (size_t)nq, 0);
    for (int i = 0; i < Cur.N; i++) {
      cxy.push_back(Cur.mvKeysUn[i].x); cxy.push_back(Cur.mvKeysUn[i].y);
      coct.push_back((uint8_t)Cur.mvKeysUn[i].octave); cang.push_back(Cur.mvKeysUn[i].angle);
      cclaimed.push_back(Cur.mvpMapPoints[i] != nullptr);                    // :1534
    }
    for (int i = 0; i < nq; i++) {
      MapPoint* mp = vpMPs[(size_t)i];
      if (!mp || mp->isBad() || sAlreadyFound.count(mp)) continue;           // :1490-1493
      const float PO[3] = {mp->pos[0] - Ow[0], mp->pos[1] - Ow[1], mp->pos[2] - Ow[2]};
      const float dist3D = (float)std::sqrt((double)PO[0] * PO[0] + (double)PO[1] * PO[1] + (double)PO[2] * PO[2]);   // cv::norm :1512
      if (dist3D < mp->GetMinDistanceInvariance() || dist3D > mp->GetMaxDistanceInvariance()) continue;              // :1518
      lvalid[(size_t)i] = 1;
      loct[(size_t)i] = (uint8_t)mp->PredictScale(dist3D, Cur.mfLogScaleFactor, Cur.mnScaleLevels);                   // :1521
      for (int c = 0; c < 3; c++) lxw[3 * (size_t)i + c] = mp->pos[c];
      lang[(size_t)i] = pKF->mvKeysUn[(size_t)i].angle;
      std::memcpy(&ldesc[32 * (size_t)i], mp->mDescriptor, 32);
    }
    const int32_t co[2] = {0, Cur.N}, lo[2] = {0, nq};
    p.cur_off = co; p.cur_xy = cxy.data(); p.cur_octave = coct.data(); p.cur_angle = cang.data(); p.cur_uright = cur.data();
    p.cur_desc = Cur.mDescriptors.data(); p.cur_claimed = cclaimed.data(); p.cur_Tcw = Cur.mTcw; p.last_Tcw = Cur.mTcw;
    p.last_off = lo; p.last_valid = lvalid.data(); p.last_xw = lxw.data(); p.last_octave = loct.data(); p.last_angle = lang.data();
    p.last_desc = ldesc.data(); p.last_has_obs = lhas.data();
    std::vector<int32_t> match((size_t)Cur.N + 1, -1);
    int32_t nm = 0;
    lld_sbp_result r;
    std::memset(&r, 0, sizeof(r));
    r.match = match.data(); r.n_matches = &nm;
    const int rc = lld_sbp_frame(ctx, &p, &r);
    if (rc) return rc;
    for (int i = 0; i < Cur.N; i++)
      if (match[(size_t)i] >= 0) Cur.mvpMapPoints[i] = vpMPs[(size_t)match[(size_t)i]];
    if (match_out) match_out->assign(match.begin(), match.begin() + Cur.N);
    return nm;
  }
  // int SearchByProjection(Frame &F, const std::vector<MapPoint*> &vpMapPoints, const float th = 3)   include/ORBmatcher.h:47
  int SearchByProjection(void* ctx, Frame& F, const std::vector<MapPoint*>& vpMapPoints, float th = 3.f, std::vector<int>* match_out = nullptr) {
    lld_sbp_mp_problem p;
    std::memset(&p, 0, sizeof(p));
    p.n_pairs = 1;
    p.geom.fx = F.fx; p.geom.fy = F.fy; p.geom.cx = F.cx; p.geom.cy = F.cy; p.geom.bf = F.mbf; p.geom.b = F.mb;
    p.geom.min_x = F.mnMinX; p.geom.max_x = F.mnMaxX; p.geom.min_y = F.mnMinY; p.geom.max_y = F.mnMaxY;
    p.geom.n_levels = (int)F.mvScaleFactors.size(); p.geom.scale_factors = F.mvScaleFactors.data();
    p.th = th; p.nn_ratio = mfNNratio;
    std::vector<float> cxy, proj, vcos;
    std::vector<uint8_t> coct, cclaimed, valid, has, desc(32 * vpMapPoints.size(), 0);
    std::vector<int32_t> lvl;
    for (int i = 0; i < F.N; i++) {
      cxy.push_back(F.mvKeysUn[i].x); cxy.push_back(F.mvKeysUn[i].y);
      coct.push_back((uint8_t)F.mvKeysUn[i].octave);
      cclaimed.push_back(F.mvpMapPoints[i] && F.mvpMapPoints[i]->Observations() > 0);   // :87-89
    }
    for (size_t i = 0; i < vpMapPoints.size(); i++) {
      MapPoint* mp = vpMapPoints[i];
      valid.push_back(mp->mbTrackInView && !mp->isBad());                               // :54-58
      proj.push_back(mp->mTrackProjX); proj.push_back(mp->mTrackProjY); proj.push_back(mp->mTrackProjXR);
      lvl.push_back(mp->mnTrackScaleLevel); vcos.push_back(mp->mTrackViewCos);
      has.push_back(mp->Observations() > 0);
      std::memcpy(&desc[32 * i], mp->mDescriptor, 32);
    }
    const int32_t co[2] = {0, F.N}, mo[2] = {0, (int32_t)vpMapPoints.size()};
    p.cur_off = co; p.cur_xy = cxy.data(); p.cur_octave = coct.data(); p.cur_uright = F.mvuRight.data();
    p.cur_desc = F.mDescriptors.data(); p.cur_claimed = cclaimed.data();
    p.mp_off = mo; p.mp_valid = valid.data(); p.mp_proj = proj.data(); p.mp_level = lvl.data(); p.mp_viewcos = vcos.data();
    p.mp_desc = desc.data(); p.mp_has_obs = has.data();
    std::vector<int32_t> match((size_t)F.N + 1, -1);
    int32_t nm = 0;
    lld_sbp_result r;
    std::memset(&r, 0, sizeof(r));
    r.match = match.data(); r.n_matches = &nm;
    const int rc = lld_sbp_mappoints(ctx, &p, &r);
    if (rc) return rc;
    for (int i = 0; i < F.N; i++)
      if (match[(size_t)i] >= 0) F.mvpMapPoints[i] = vpMapPoints[(size_t)match[(size_t)i]];   // F.mvpMapPoints[bestIdx] = pMP (:123)
    if (match_out) match_out->assign(match.begin(), match.begin() + F.N);
    return nm;
  }
  // int SearchForTriangulation(KeyFrame* pKF1, KeyFrame* pKF2, cv::Mat F12, vector<pair<size_t,size_t>>& vMatchedPairs, bool bOnlyStereo)
  // include/ORBmatcher.h:71-72, src/ORBmatcher.cc:657-823.  Host part: the epipole (:665-671) and the flattening of the two feature
  // vectors (std::map iteration order = ascending node id, as the reference's merge walks them).
  int SearchForTriangulation(void* ctx, KeyFrame* pKF1, KeyFrame* pKF2, const float F12[9],
                             std::vector<std::pair<size_t, size_t>>& vMatchedPairs, bool bOnlyStereo, float* epipole_out = nullptr) {
    // Cw = -R1w' t1w (KeyFrame::GetCameraCenter), C2 = R2w Cw + t2w: cv::Mat CV_32F products, double accumulation, one rounding
    const float* T1 = pKF1->Tcw; const float* T2 = pKF2->Tcw;
    float Cw[3], C2[3];
    for (int k = 0; k < 3; k++) Cw[k] = (float)(-((double)T1[k] * T1[9] + (double)T1[3 + k] * T1[10] + (double)T1[6 + k] * T1[11]));
    for (int r = 0; r < 3; r++) C2[r] = (float)((double)T2[3 * r] * Cw[0] + (double)T2[3 * r + 1] * Cw[1] + (double)T2[3 * r + 2] * Cw[2] + (double)T2[9 + r]);
    const float invz = 1.0f / C2[2];
    const float ep[2] = {pKF2->fx * C2[0] * invz + pKF2->cx, pKF2->fy * C2[1] * invz + pKF2->cy};
    if (epipole_out) { epipole_out[0] = ep[0]; epipole_out[1] = ep[1]; }
    lld_tri_search_problem p;
    std::memset(&p, 0, sizeof(p));
    p.n_pairs = 1; p.only_stereo = bOnlyStereo; p.check_orientation = mbCheckOrientation;
    p.n_levels = (int)pKF2->mvScaleFactors.size();
    for (int l = 0; l < p.n_levels && l < 8; l++) { p.scale_factors[l] = pKF2->mvScaleFactors[(size_t)l]; p.level_sigma2[l] = pKF2->mvLevelSigma2[(size_t)l]; }
    p.F12 = F12; p.epipole = ep;
    struct Flat { std::vector<float> xy, ang; std::vector<uint8_t> oct, has; std::vector<int32_t> node, ioff{0}, idx; int32_t koff[2], noff[2]; };
    auto flatten = [](KeyFrame* k, Flat& f) {
      const size_t N = k->mvKeysUn.size();
      for (size_t i = 0; i < N; i++) {
        f.xy.push_back(k->mvKeysUn[i].x); f.xy.push_back(k->mvKeysUn[i].y); f.ang.push_back(k->mvKeysUn[i].angle);
        f.oct.push_back((uint8_t)k->mvKeysUn[i].octave); f.has.push_back(k->mvpMapPoints[i] != nullptr);
      }
      for (auto& kv : k->mFeatVec) {
        f.node.push_back((int32_t)kv.first);
        for (unsigned i : kv.second) f.idx.push_back((int32_t)i);
        f.ioff.push_back((int32_t)f.idx.size());
      }
      f.koff[0] = 0; f.koff[1] = (int32_t)N; f.noff[0] = 0; f.noff[1] = (int32_t)f.node.size();
    };
    Flat a, b;
    flatten(pKF1, a); flatten(pKF2, b);
    p.kp1_off = a.koff; p.kp1_xy = a.xy.data(); p.kp1_angle = a.ang.data(); p.kp1_uright = pKF1->mvuRight.data(); p.kp1_has_mp = a.has.data();
    p.kp1_desc = pKF1->mDescriptors.data();
    p.kp2_off = b.koff; p.kp2_xy = b.xy.data(); p.kp2_octave = b.oct.data(); p.kp2_angle = b.ang.data(); p.kp2_uright = pKF2->mvuRight.data();
    p.kp2_has_mp = b.has.data(); p.kp2_desc = pKF2->mDescriptors.data();
    p.fv1_node_off = a.noff; p.fv1_node = a.node.data(); p.fv1_idx_off = a.ioff.data(); p.fv1_idx = a.idx.data();
    p.fv2_node_off = b.noff; p.fv2_node = b.node.data(); p.fv2_idx_off = b.ioff.data(); p.fv2_idx = b.idx.data();
    std::vector<int32_t> m12(pKF1->mvKeysUn.size() + 1, -1);
    int32_t nm = 0;
    lld_tri_search_result r{m12.data(), &nm};
    const int rc = lld_tri_search(ctx, &p, &r);
    if (rc) return rc;
    vMatchedPairs.clear();
    vMatchedPairs.reserve((size_t)nm);
    for (size_t i = 0; i < pKF1->mvKeysUn.size(); i++)
      if (m12[i] >= 0) vMatchedPairs.push_back(std::make_pair(i, (size_t)m12[i]));   // :813-818
    return nm;
  }
  // int SearchByBoW(KeyFrame* pKF1, KeyFrame* pKF2, vector<MapPoint*>& vpMatches12)   include/ORBmatcher.h:60, src/ORBmatcher.cc:522-655
  // (the KeyFrame -> Frame overload :159-288 flattens the same way with kp2_valid = 1, strict_th = 0 and inverts match12 into
  // vpMapPointMatches[match12[i]] = vpMapPointsKF[i])
  int SearchByBoW(void* ctx, KeyFrame* pKF1, KeyFrame* pKF2, std::vector<MapPoint*>& vpMatches12) {
    lld_bow_search_problem p;
    std::memset(&p, 0, sizeof(p));
    p.n_pairs = 1; p.strict_th = 1; p.check_orientation = mbCheckOrientation; p.nn_ratio = mfNNratio;
    struct Flat { std::vector<float> ang; std::vector<uint8_t> valid; std::vector<int32_t> node, ioff{0}, idx; int32_t koff[2], noff[2]; };
    auto flatten = [](KeyFrame* k, Flat& f) {
      const size_t N = k->mvKeysUn.size();
      for (size_t i = 0; i < N; i++) {
        f.ang.push_back(k->mvKeysUn[i].angle);
        f.valid.push_back(k->mvpMapPoints[i] != nullptr && !k->mvpMapPoints[i]->isBad());     // :552-557, :573-578
      }
      for (auto& kv : k->mFeatVec) {
        f.node.push_back((int32_t)kv.first);
        for (unsigned i : kv.second) f.idx.push_back((int32_t)i);
        f.ioff.push_back((int32_t)f.idx.size());
      }
      f.koff[0] = 0; f.koff[1] = (int32_t)N; f.noff[0] = 0; f.noff[1] = (int32_t)f.node.size();
    };
    Flat a, b;
    flatten(pKF1, a); flatten(pKF2, b);
    p.kp1_off = a.koff; p.kp1_angle = a.ang.data(); p.kp1_valid = a.valid.data(); p.kp1_desc = pKF1->mDescriptors.data();
    p.kp2_off = b.koff; p.kp2_angle = b.ang.data(); p.kp2_valid = b.valid.data(); p.kp2_desc = pKF2->mDescriptors.data();
    p.fv1_node_off = a.noff; p.fv1_node = a.node.data(); p.fv1_idx_off = a.ioff.data(); p.fv1_idx = a.idx.data();
    p.fv2_node_off = b.noff; p.fv2_node = b.node.data(); p.fv2_idx_off = b.ioff.data(); p.fv2_idx = b.idx.data();
    std::vector<int32_t> m12(pKF1->mvKeysUn.size() + 1, -1);
    int32_t nm = 0;
    lld_tri_search_result r{m12.data(), &nm};
    const int rc = lld_bow_search(ctx, &p, &r);
    if (rc) return rc;
    vpMatches12.assign(pKF1->mvKeysUn.size(), nullptr);                                       // :536
    for (size_t i = 0; i < pKF1->mvKeysUn.size(); i++)
      if (m12[i] >= 0) vpMatches12[i] = pKF2->mvpMapPoints[(size_t)m12[i]];                   // :597
    return nm;
  }
  // int SearchForInitialization(Frame &F1, Frame &F2, vector<cv::Point2f> &vbPrevMatched, vector<int> &vnMatches12, int windowSize)
  // src/ORBmatcher.cc:405: both frames flattened as they are (F2's grid comes from its bounds and
  // mvKeysUn) -> lld_init_search -> vnMatches12 and vbPrevMatched
  int SearchForInitialization(void* ctx, Frame& F1, Frame& F2, std::vector<Point2f>& vbPrevMatched, std::vector<int>& vnMatches12,
                              int windowSize = 10) {
    const size_t N1 = F1.mvKeysUn.size(), N2 = F2.mvKeysUn.size();
    lld_init_search_problem p;
    std::memset(&p, 0, sizeof(p));
    p.n_pairs = 1;
    p.geom.min_x = F2.mnMinX; p.geom.max_x = F2.mnMaxX; p.geom.min_y = F2.mnMinY; p.geom.max_y = F2.mnMaxY;
    p.geom.n_levels = (int)F2.mvScaleFactors.size(); p.geom.scale_factors = F2.mvScaleFactors.data();
    p.window_size = windowSize; p.nn_ratio = mfNNratio; p.check_orientation = mbCheckOrientation;
    std::vector<float> ang1, prev, xy2, ang2;
    std::vector<uint8_t> oct1, oct2;
    for (size_t i = 0; i < N1; i++) {
      oct1.push_back((uint8_t)F1.mvKeysUn[i].octave); ang1.push_back(F1.mvKeysUn[i].angle);
      prev.push_back(vbPrevMatched[i].x); prev.push_back(vbPrevMatched[i].y);
    }
    for (size_t i = 0; i < N2; i++) {
      xy2.push_back(F2.mvKeysUn[i].x); xy2.push_back(F2.mvKeysUn[i].y);
      oct2.push_back((uint8_t)F2.mvKeysUn[i].octave); ang2.push_back(F2.mvKeysUn[i].angle);
    }
    const int32_t o1[2] = {0, (int32_t)N1}, o2[2] = {0, (int32_t)N2};
    p.kp1_off = o1; p.kp1_octave = oct1.data(); p.kp1_angle = ang1.data(); p.kp1_desc = F1.mDescriptors.data(); p.prev_matched = prev.data();
    p.kp2_off = o2; p.kp2_xy = xy2.data(); p.kp2_octave = oct2.data(); p.kp2_angle = ang2.data(); p.kp2_desc = F2.mDescriptors.data();
    std::vector<int32_t> m12(N1 + 1, -1);
    int32_t nm = 0;
    lld_init_search_result r{m12.data(), &nm, prev.data()};
    const int rc = lld_init_search(ctx, &p, &r);
    if (rc) return rc;
    vnMatches12.assign(m12.begin(), m12.begin() + N1);
    for (size_t i = 0; i < N1; i++) { vbPrevMatched[i].x = prev[2 * i]; vbPrevMatched[i].y = prev[2 * i + 1]; }
    return nm;
  }
  // What ORBmatcher::Fuse decides for one map point (src/ORBmatcher.cc:949-968); Replace() itself is map bookkeeping and stays
  // with the caller: `survivor` replaces `replaced`; both null = a new observation was added (done here)
  struct FuseAction { MapPoint* pMP; int bestIdx; MapPoint* survivor; MapPoint* replaced; };
  // int Fuse(KeyFrame* pKF, const vector<MapPoint*>& vpMapPoints, const float th = 3.0)   include/ORBmatcher.h:80, src/ORBmatcher.cc:825-975
  // Host part = everything before GetFeaturesInArea, in the reference's float arithmetic (cv::Mat CV_32F products accumulate in
  // double and round once); the windowed search with the reprojection gate is lld_kf_search; the sequential Replace / Add logic
  // runs afterwards over the accepted points in order.
  int Fuse(void* ctx, KeyFrame* pKF, const std::vector<MapPoint*>& vpMapPoints, float th = 3.0f, std::vector<FuseAction>* actions = nullptr) {
    const float* T = pKF->Tcw;
    auto row = [&](int r, const float* x, float t) { return (float)((double)T[3 * r] * x[0] + (double)T[3 * r + 1] * x[1] + (double)T[3 * r + 2] * x[2] + (double)t); };
    float Ow[3];   // KeyFrame::SetPose: Ow = -Rcw.t() * tcw  (src/KeyFrame.cc:75-90)
    for (int k = 0; k < 3; k++) Ow[k] = (float)(-((double)T[k] * T[9] + (double)T[3 + k] * T[10] + (double)T[6 + k] * T[11]));
    const size_t n = vpMapPoints.size(), N = pKF->mvKeysUn.size();
    std::vector<uint8_t> valid(n, 0), desc(32 * n, 0), koct(N), claimed(N, 0);
    std::vector<float> proj(3 * n, 0.f), kxy(2 * N);
    std::vector<int32_t> lvl(n, 0);
    for (size_t i = 0; i < n; i++) {
      MapPoint* pMP = vpMapPoints[i];
      if (!pMP) continue;
      if (pMP->isBad() || pMP->IsInKeyFrame(pKF)) continue;
      const float* Xw = pMP->pos;
      const float xc = row(0, Xw, T[9]), yc = row(1, Xw, T[10]), zc = row(2, Xw, T[11]);
      if (zc < 0.0f) continue;                                          // :851
      const float invz = 1 / zc;
      const float x = xc * invz, y = yc * invz;
      const float u = pKF->fx * x + pKF->cx, v = pKF->fy * y + pKF->cy;
      if (!pKF->IsInImage(u, v)) continue;                              // :862
      const float ur = u - pKF->mbf * invz;
      const float PO[3] = {Xw[0] - Ow[0], Xw[1] - Ow[1], Xw[2] - Ow[2]};
      const float dist3D = (float)std::sqrt((double)PO[0] * PO[0] + (double)PO[1] * PO[1] + (double)PO[2] * PO[2]);   // cv::norm
      if (dist3D < pMP->GetMinDistanceInvariance() || dist3D > pMP->GetMaxDistanceInvariance()) continue;            // :873
      const float* Pn = pMP->mNormalVector;
      if ((double)PO[0] * Pn[0] + (double)PO[1] * Pn[1] + (double)PO[2] * Pn[2] < 0.5 * dist3D) continue;            // :879
      valid[i] = 1;
      proj[3 * i] = u; proj[3 * i + 1] = v; proj[3 * i + 2] = ur;
      lvl[i] = pMP->PredictScale(dist3D, pKF->mfLogScaleFactor, pKF->mnScaleLevels);
      std::memcpy(&desc[32 * i], pMP->mDescriptor, 32);
    }
    for (size_t i = 0; i < N; i++) { kxy[2 * i] = pKF->mvKeysUn[i].x; kxy[2 * i + 1] = pKF->mvKeysUn[i].y; koct[i] = (uint8_t)pKF->mvKeysUn[i].octave; }
    lld_kf_search_problem p;
    std::memset(&p, 0, sizeof(p));
    p.n_pairs = 1;
    p.geom.fx = pKF->fx; p.geom.fy = pKF->fy; p.geom.cx = pKF->cx; p.geom.cy = pKF->cy; p.geom.bf = pKF->mbf;
    p.geom.min_x = pKF->mnMinX; p.geom.max_x = pKF->mnMaxX; p.geom.min_y = pKF->mnMinY; p.geom.max_y = pKF->mnMaxY;
    p.geom.n_levels = (int)pKF->mvScaleFactors.size(); p.geom.scale_factors = pKF->mvScaleFactors.data();
    p.th = th; p.th_low = 50; p.chi2_gate = 1; p.sequential_claims = 0;
    for (size_t l = 0; l < 8 && l < pKF->mvInvLevelSigma2.size(); l++) p.inv_level_sigma2[l] = pKF->mvInvLevelSigma2[l];
    const int32_t ko[2] = {0, (int32_t)N}, mo[2] = {0, (int32_t)n};
    p.kp_off = ko; p.kp_xy = kxy.data(); p.kp_octave = koct.data(); p.kp_uright = pKF->mvuRight.data(); p.kp_desc = pKF->mDescriptors.data();
    p.kp_claimed = claimed.data();
    p.mp_off = mo; p.mp_valid = valid.data(); p.mp_proj = proj.data(); p.mp_level = lvl.data(); p.mp_desc = desc.data();
    std::vector<int32_t> match(N + 1, -1), best(n + 1, -1), bdist(n + 1, 256);
    int32_t nm = 0;
    lld_sbp_result r;
    std::memset(&r, 0, sizeof(r));
    r.match = match.data(); r.n_matches = &nm; r.best_idx = best.data(); r.best_dist = bdist.data();
    const int rc = lld_kf_search(ctx, &p, &r);
    if (rc) return rc;
    int nFused = 0;
    for (size_t i = 0; i < n; i++) {                                    // :949-968, in the order of vpMapPoints
      if (best[i] < 0) continue;
      MapPoint* pMP = vpMapPoints[i];
      MapPoint* pMPinKF = pKF->mvpMapPoints[(size_t)best[i]];
      FuseAction a{pMP, best[i], nullptr, nullptr};
      if (pMPinKF) {
        if (!pMPinKF->isBad()) {
          if (pMPinKF->Observations() > pMP->Observations()) { a.survivor = pMPinKF; a.replaced = pMP; }
          else { a.survivor = pMP; a.replaced = pMPinKF; }
        }
      } else {
        pMP->observations[pKF] = (size_t)best[i];
        pKF->mvpMapPoints[(size_t)best[i]] = pMP;
      }
      if (actions) actions->push_back(a);
      nFused++;
    }
    return nFused;
  }
 private:
  float mfNNratio;
  bool mbCheckOrientation;
};

class TwoFrameLineMatcher {
 public:
  // TwoFrameLineMatcher(const Eigen::Matrix3d& K, double b, double tau, int minLineLength, LineMatcher*)  include/TwoFrameLineMatcher.h:31-37
  TwoFrameLineMatcher(const double K_[9], double b, double tau_, int minLineLength_) : b_(b), tau(tau_), minLineLength(minLineLength_) {
    for (int i = 0; i < 9; i++) K[i] = K_[i];
  }
  // void MatchLines(lines, other_lines, descsLeft, descsRight, std::vector<int>* desc_matches)  :39-40
  int MatchLines(void* ctx, const std::vector<KeyLine>& L, const std::vector<KeyLine>& R, const float* descL, const float* descR,
                 int desc_dim, std::vector<int>* desc_matches) {
    std::vector<float> ls, rs;
    std::vector<int32_t> lo_, ro_;
    for (auto& k : L) { ls.push_back(k.startPointX); ls.push_back(k.startPointY); ls.push_back(k.endPointX); ls.push_back(k.endPointY); lo_.push_back(k.octave); }
    for (auto& k : R) { rs.push_back(k.startPointX); rs.push_back(k.startPointY); rs.push_back(k.endPointX); rs.push_back(k.endPointY); ro_.push_back(k.octave); }
    const int32_t lof[2] = {0, (int32_t)L.size()}, rof[2] = {0, (int32_t)R.size()};
    lld_line_match_problem p;
    std::memset(&p, 0, sizeof(p));
    p.n_pairs = 1; p.desc_dim = desc_dim; p.left_off = lof; p.right_off = rof;
    p.left_seg = ls.data(); p.left_octave = lo_.data(); p.right_seg = rs.data(); p.right_octave = ro_.data();
    p.left_desc = descL; p.right_desc = descR;
    for (int i = 0; i < 9; i++) p.K[i] = K[i];
    p.baseline = b_; p.tau = tau; p.min_line_length = minLineLength;
    std::vector<int32_t> m(L.size() + 1, -1);
    lld_line_match_result r;
    std::memset(&r, 0, sizeof(r));
    r.match = m.data();
    const int rc = lld_line_match(ctx, &p, &r);
    if (rc) return rc;
    desc_matches->assign(m.begin(), m.begin() + L.size());
    return 0;
  }
 private:
  double K[9], b_, tau;
  int minLineLength;
};

}  // namespace lld
