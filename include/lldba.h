/*
 * lldba.h — C-ABI of the B200-native point+line bundle-adjustment and descriptor-matching core.
 *
 * This is the drop-in boundary for the hot path of LLD-SLAM (reference tree paths below are relative
 * to the reference repository root).  The reference has no FFI layer: its callers invoke C++ members
 * directly.  Each entry point here replaces the *body* of one of those members; the thin C++ shim in
 * lld_slam_b200/host/ keeps the reference's class / method names and flattens the caller's objects
 * into the plain arrays declared here.
 *
 *   lld_ba_local           <- Optimizer::LocalBundleAdjustment      include/Optimizer.h:49,  src/Optimizer.cc:936-1388
 *                             + LineOptimizer::{AddLineMinimal,DisableOutliers,GetLineData}  include/LineOptimizer.h:13-20
 *   lld_ba_global          <- Optimizer::BundleAdjustment / GlobalBundleAdjustment           include/Optimizer.h:43-47, src/Optimizer.cc:312-559
 *   lld_pose_opt           <- Optimizer::PoseOptimization            include/Optimizer.h:50,  src/Optimizer.cc:653-932
 *   lld_descriptor_distance<- ORBmatcher::DescriptorDistance         include/ORBmatcher.h:51, src/ORBmatcher.cc:1647-1663
 *   lld_sbp_frame          <- ORBmatcher::SearchByProjection(Frame&,const Frame&,th,bMono)   include/ORBmatcher.h:52, src/ORBmatcher.cc:1328-1470
 *   lld_sbp_mappoints      <- ORBmatcher::SearchByProjection(Frame&,vector<MapPoint*>&,th)   include/ORBmatcher.h:47, src/ORBmatcher.cc:45-129
 *   lld_line_match         <- TwoFrameLineMatcher::MatchLines        include/TwoFrameLineMatcher.h:39, src/TwoFrameLineMatcher.cc:26-124
 *   the callers either side of that path (SURVEY section 8(f)):
 *   lld_stereo_matches     <- Frame::ComputeStereoMatches            src/Frame.cc:530-704
 *   lld_sbp_frame(th_high) <- ORBmatcher::SearchByProjection(Frame&,KeyFrame*,sAlreadyFound,th,ORBdist)  src/ORBmatcher.cc:1472-1599
 *   lld_kf_search          <- ORBmatcher::Fuse x2, SearchByProjection(KeyFrame*,Scw,...)     src/ORBmatcher.cc:825-975, 977-1100, 290-403
 *   lld_tri_search         <- ORBmatcher::SearchForTriangulation     src/ORBmatcher.cc:657-823
 *   lld_bow_search         <- ORBmatcher::SearchByBoW x2             src/ORBmatcher.cc:159-288, 522-655
 *   lld_init_search        <- ORBmatcher::SearchForInitialization    src/ORBmatcher.cc:405
 *   lld_sim3_opt           <- Optimizer::OptimizeSim3                src/Optimizer.cc:1656-1858
 *   lld_sim3_ransac        <- Sim3Solver::iterate / ComputeSim3 / CheckInliers (ORB-SLAM2 src/Sim3Solver.cc)
 *   lld_pnp_ransac         <- PnPsolver::iterate / Refine / CheckInliers / compute_pose (ORB-SLAM2 src/PnPsolver.cc)
 *   lld_line_associate     <- Tracking::AddLinesFrom                 src/Tracking.cc:996-1124
 *   lld_medoid_orb / _float<- MapPoint / MapLine::ComputeDistinctiveDescriptors              src/MapPoint.cc:242-307, src/MapLine.cc:133-201
 *
 * Conventions
 *   - Plain pointers and sizes only.  All arrays are caller-owned HOST memory, contiguous, little endian.
 *   - Every problem struct is *batched*: entity arrays of all independent units (BA windows, frames,
 *     frame pairs) are concatenated and addressed through CSR offset arrays.  A single reference call is
 *     the batch-of-one case.
 *   - Return value: 0 = ok; <0 = error (LLD_ERR_*).  Nothing throws.  On error the outputs are undefined.
 *   - A context owns one CUDA stream plus its device workspace.  Contexts are not shared between threads;
 *     the reference enters this path from three threads concurrently (Tracking, LocalMapping, GBA), so a
 *     caller creates one context per calling thread.
 *   - There is no CPU fallback: every compute entry point fails with LLD_ERR_CUDA when no device is usable.
 *   - Precision contract of the reference (src/Converter.cc:37-47,110-116): map state arrives float-valued,
 *     is widened to double, optimised in double and narrowed by the caller.  Arrays typed `double` below
 *     carry such widened values; arrays typed `float` are values the reference itself keeps as float.
 */
#ifndef LLDBA_H
#define LLDBA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LLD_OK 0
#define LLD_ERR_CUDA (-1)
#define LLD_ERR_ARG (-2)
#define LLD_ERR_NCCL (-3)
#define LLD_ERR_UNSUPPORTED (-4)

/* ------------------------------------------------------------------------------------------------
 * Bundle adjustment (local windows and global map)
 * ---------------------------------------------------------------------------------------------- */

/* Capacity limits of this implementation (the reference has none; a call outside them returns LLD_ERR_ARG /
 * LLD_ERR_UNSUPPORTED and lld_ctx_last_error() names the limit):
 *   - at most 254 observations per landmark;
 *   - a free keyframe may have at most 169 later free neighbours (6 * (neighbours + itself) <= 1024), else LLD_ERR_UNSUPPORTED.
 *     In lld_ba_local every later free keyframe of the window counts as a neighbour, so this is a window of at most 170 free
 *     keyframes; in lld_ba_global a neighbour is a later free keyframe that shares a landmark, and the envelope limit below
 *     is always reached first;
 *   - lld_ba_global: let B be the largest distance, in free-keyframe indices (fixed keyframes are skipped), between two free
 *     keyframes that observe one landmark.  B <= 26 solves by block cyclic reduction over super-blocks of B keyframes
 *     (6B <= 156); B >= 27 takes the single-CTA skyline LDL^T, whose envelope must fit 220 KB of shared memory.  For a
 *     band-shaped envelope over n_free free keyframes that is 228 B + 6 n_free <= 27952: B <= 117 at 200 free keyframes,
 *     B <= 83 at 1500.  A wider envelope (e.g. a loop-closure landmark across the map) returns LLD_ERR_UNSUPPORTED,
 *     unless lld_ctx_set_gba_sparse(ctx, 1) is on: then it is solved by block elimination over super-blocks of mb
 *     keyframes (mb = the largest such distance that is <= 26; longer ones become edges of the super-block graph), whose
 *     plan (blocks with fill, Z factors, solution) must fit 2 GiB of device memory (2147483648 bytes), else
 *     LLD_ERR_UNSUPPORTED with the plan's size in the message;
 *   - lld_ba_global: one free keyframe observing the same landmark twice is LLD_ERR_ARG (lld_ba_local accepts it and takes the
 *     sparse path);
 *   - local windows with more than 32 free keyframes take the general (slower) sparse path;
 *   - lld_sbp_*, lld_kf_search: n_levels <= 8, at most 65535 keypoints per frame; pairs with more than 2048 keypoints or queries
 *     take the multi-kernel path instead of the single-CTA one;
 *   - lld_init_search: at most 65535 keypoints per frame, F2 octaves < 8; with check_orientation, F1 angles in [0, 900) and F2
 *     angles in [0, 360) (ORB angles are in [0, 360)).  The sequential resolve keeps F2's state in shared memory when every F2
 *     of the batch has at most 57088 keypoints (k_init_resolve_smem), else in global memory (k_init_resolve_global);
 *   - lld_sim3_opt: no limit on the correspondences of a problem.  When every problem of the batch has at most 4266 (48 bytes each
 *     within 200 KB) the edge records are staged in shared memory (k_sim3_opt_smem), else read from global memory (k_sim3_opt_global);
 *   - lld_sim3_ransac: no limit on the correspondences or minimal sets of a problem (correspondence data is read from global
 *     memory; one CTA per problem evaluates 8 minimal sets at a time, k_sim3_ransac);
 *   - lld_pnp_ransac: no limit on the correspondences or minimal sets of a problem (one CTA per problem, one warp per minimal
 *     set, 8 at a time, Refine over the whole CTA; correspondence data is read from global memory, k_pnp_ransac);
 *   - lld_line_match: descriptor widths that are a multiple of 8 up to 72 floats and at most 512 lines per side of a pair run on the
 *     tensor cores, everything else on the FP32 tile path (no failure).
 */

/* One batch of independent BA problems ("windows").  Entities of window w live at
 * [kf_off[w], kf_off[w+1]) etc.; KF indices stored in observations are window-local.
 * Observations are grouped by landmark in the reference's insertion order
 * (src/Optimizer.cc:1093-1178 for points, :1182-1218 / src/LineOptimizer.cc:59-125 for lines). */
typedef struct lld_ba_problem {
  int32_t n_win;
  const int32_t* kf_off; /* [n_win+1] */
  const int32_t* pt_off; /* [n_win+1] */
  const int32_t* ln_off; /* [n_win+1] */

  /* keyframes */
  const double* kf_Tcw;     /* [n_kf][12]  R row-major (9) then t (3): world->camera, as Converter::toSE3Quat receives it */
  const uint8_t* kf_fixed;  /* [n_kf]      vSE3->setFixed(...)  src/Optimizer.cc:1043,1057 */
  const double* kf_intr;    /* [n_kf][5]   fx fy cx cy bf used by point edges */
  const double* kf_line_cam;/* [n_kf][4]   f cx cy baseline used by line edges observed from this KF.
                               LocalBA: the *current* KF's values for every KF (src/Optimizer.cc:1211-1215);
                               GBA: each KF's own (src/Optimizer.cc:200-210). */

  /* map points */
  const double* pt_xyz;       /* [n_pt][3] */
  const int32_t* pt_obs_off;  /* [n_pt+1]  CSR into the point observation arrays */
  const int32_t* pt_obs_kf;   /* [n_pt_obs] window-local KF index */
  const float* pt_obs_uvr;    /* [n_pt_obs][3] u v uR ; uR<0 => monocular edge (src/Optimizer.cc:1119) */
  const float* pt_obs_info;   /* [n_pt_obs]  invSigma2 (float in the reference, src/Optimizer.cc:1129) */

  /* map lines, minimal (X0, dir) parametrisation of MapLine::GetMinimalPos */
  const double* ln_x0_dir;    /* [n_ln][6]  X0 (closest point to origin), unit direction */
  const int32_t* ln_obs_off;  /* [n_ln+1]   CSR; one entry per (line, KF) = one proj_map element */
  const int32_t* ln_obs_kf;   /* [n_ln_obs] */
  const float* ln_obs_left;   /* [n_ln_obs][4] xs ys xe ye of the left KeyLine (pixels) */
  const float* ln_obs_right;  /* [n_ln_obs][4] right KeyLine, xs<0 => no right edge (src/LineOptimizer.cc:65-68) */
  const double* ln_obs_info;  /* [n_ln_obs][2] information of the left / right edge (gamma^2 / 1.44^(2*octave); 1 in GBA) */
  const uint8_t* ln_obs_stereo;/* [n_ln_obs] 1: Huber delta / chi2 gate = stereo value, 0: mono value (src/LineOptimizer.cc:83-88) */

  /* constants of the entry point (SURVEY A.6) */
  int32_t robust_points;      /* Huber on point edges (LocalBA: 1; GBA: bRobust) */
  double delta_pt_mono;       /* (double)(float)sqrt(5.991) */
  double delta_pt_stereo;     /* (double)(float)sqrt(7.815) */
  double delta_ln_mono;       /* gamma-scaled, src/LineOptimizer.cc:33-36 */
  double delta_ln_stereo;
  double chi2_pt_mono;        /* 5.991 outlier gate, src/Optimizer.cc:1246 */
  double chi2_pt_stereo;      /* 7.815 */
  int32_t ln_endpoints_normalized; /* 0: pixel endpoints used as homogeneous (x,y,1) (LocalBA, src/LineOptimizer.cc:106-113);
                                      1: K^-1 * (x,y,1) with the KF's fx fy cx cy (GBA, src/Optimizer.cc:234-235) */
  int32_t ln_filter;          /* 4: line dropped after round 1 when 2*(#inlier edges) <= ln_filter (include/LineOptimizer.h:23) */
} lld_ba_problem;

typedef struct lld_ba_result {
  double* kf_Tcw;        /* [n_kf][12]   optimised poses (fixed KFs: re-orthonormalised input, as toCvMat(SE3Quat) gives) */
  double* pt_xyz;        /* [n_pt][3] */
  double* ln_x0_dir;     /* [n_ln][6]    GetLineData / GBA read-back: X0 = alpha*R[:,1], dir = R[:,0] */
  uint8_t* pt_obs_bad;   /* [n_pt_obs]   1 => (KF,point) goes to vToErase (src/Optimizer.cc:1281-1311); zero in GBA */
  uint8_t* ln_obs_bad;   /* [n_ln_obs][2] 1 => GetLineData lists this edge's KF as outlier projection */
  uint8_t* ln_removed;   /* [n_ln]       1 => line vertex removed by DisableOutliers, GetLineData returns false */
  /* LM trace, [n_win][log_stride]: entry 0 = initial robust chi2, entry k = chi2 after outer iteration k.
   * Round 2 of LocalBA is appended after round 1.  n_iter_done[w][r] = outer iterations executed in round r. */
  int32_t log_stride;
  double* chi2_log;      /* may be NULL */
  double* lambda_log;    /* may be NULL */
  int32_t* trials_log;   /* may be NULL */
  int32_t* n_iter_done;  /* [n_win][2], may be NULL */
} lld_ba_result;

int lld_ctx_create(int device, void** ctx);
void lld_ctx_destroy(void* ctx);
/* last CUDA / NCCL error text of this context (static storage inside ctx) */
const char* lld_ctx_last_error(void* ctx);

/* Multi-GPU: join an NCCL communicator created from `unique_id` (128 bytes from lld_comm_unique_id on rank 0,
 * distributed by the caller, e.g. torch.distributed broadcast).  Needed only by lld_ba_global with n_ranks>1. */
int lld_comm_unique_id(uint8_t id_out[128]);
int lld_comm_init(void* ctx, int n_ranks, int rank, const uint8_t unique_id[128]);

/* LocalBundleAdjustment: its_round1 (5) LM iterations with Huber, outlier gating, its_round2 (15) without.
 * stop_flag mirrors pbStopFlag (src/Optimizer.cc:1220-1236): polled on the host between LM steps. */
int lld_ba_local(void* ctx, const lld_ba_problem* p, int its_round1, int its_round2,
                 const volatile uint8_t* stop_flag, lld_ba_result* out);

/* BundleAdjustment: one optimize(n_iter) pass, no outlier round.
 * Multi-rank (a communicator of n_ranks>1 joined with lld_comm_init): EVERY rank passes the SAME, WHOLE problem (all
 * keyframes, all landmarks, identical order).  The library keeps the contiguous landmark block lld_ba_shard_bounds()
 * assigns to the calling rank, indexes and uploads only that block (the block pattern of the reduced camera system is
 * derived from the whole problem, so it is rank-invariant), and all-reduces the reduced camera system (one packed
 * call per LM trial) and the chi2 / scale scalars over NCCL.  Do NOT pre-shard the input.
 * Outputs on n_ranks>1: kf_Tcw and the LM trace are complete and identical on every rank; pt_xyz / ln_x0_dir (and the
 * all-zero flag arrays) are written for the rank's own landmark block only — the caller gathers them (rank r owns
 * points [b[0],b[1]) and lines [b[2],b[3]) of lld_ba_shard_bounds).
 * stop_flag on n_ranks>1: the ranks agree on the flag with an all-reduce(max) before every group of LM steps, so every
 * rank stops at the same step whichever rank saw the flag first. */
int lld_ba_global(void* ctx, const lld_ba_problem* p, int n_iter, const volatile uint8_t* stop_flag,
                  lld_ba_result* out);

/* Global BA after a loop closure: on = 1 lets lld_ba_global solve a reduced camera system whose envelope is too wide
 * for the on-chip solvers (a landmark seen by keyframes at both ends of the map) by block elimination over its
 * super-block graph; on = 0 (the default) rejects it with LLD_ERR_UNSUPPORTED.  Problems that the other solvers take are
 * not affected.  Part of the topology-cache key: a cached structure is indexed again when the switch changes. */
void lld_ctx_set_gba_sparse(void* ctx, int on);

/* The block-elimination plan lld_ba_global would run for p with the switch on, as JSON in buf (host arithmetic only, no
 * device needed; for tests): super-block size mb, count N, the elimination levels with their neighbour lists, the
 * off-diagonal blocks with fill, the Z offsets and the ordered Schur contributions of every output block.  A problem
 * another solver takes gives {"solver":"other"}; an error code comes with its message in buf. */
int lld_gba_sparse_plan_report(const lld_ba_problem* p, char* buf, int len);

/* Landmark partition used by lld_ba_global on n_ranks>1: rank r owns points [out[0], out[1]) and lines
 * [out[2], out[3]) (contiguous blocks; keyframes are replicated).  Host arithmetic only, no device needed.
 * There is no reference counterpart (the reference is single-process); the partitioned loop is the independent
 * per-landmark Schur loop of Thirdparty/g2o/g2o/core/block_solver.hpp:381-432. */
void lld_ba_shard_bounds(int32_t n_pt, int32_t n_ln, int32_t rank, int32_t n_ranks, int32_t out[4]);

/* ------------------------------------------------------------------------------------------------
 * Motion-only pose optimisation (batched frames)
 * ---------------------------------------------------------------------------------------------- */
typedef struct lld_pose_problem {
  int32_t n_frames;
  const double* Tcw;        /* [n_frames][12] initial pose (pFrame->mTcw widened) */
  const double* intr;       /* [n_frames][5]  fx fy cx cy bf */
  const double* line_cam;   /* [n_frames][4]  f(=fx) cx cy baseline(=mbf/fx as float)  src/Optimizer.cc:600-631 */
  const int32_t* pt_off;    /* [n_frames+1] */
  const float* pt_xw;       /* [n_pt][3]  MapPoint world position (float, src/Optimizer.cc:745-748) */
  const float* pt_uvr;      /* [n_pt][3]  uR<0 => mono */
  const float* pt_info;     /* [n_pt] */
  const int32_t* ln_off;    /* [n_frames+1] one entry per frame line with a MapLine */
  const double* ln_x0_dir;  /* [n_ln][6] */
  const float* ln_left;     /* [n_ln][4] */
  const float* ln_right;    /* [n_ln][4] xs<0 => no right edge */
  const double* ln_info;    /* [n_ln][2] */
  const uint8_t* ln_stereo; /* [n_ln]    Huber delta selector (line_matches[i]>=0) */
  const uint8_t* ln_gate_stereo; /* [n_ln][2] chi2-gate selector per edge: the reference indexes vnStereoLines by the
                                    frame line id, not the edge id (src/Optimizer.cc:894-898); the shim reproduces that */
  double delta_mono, delta_stereo;        /* (double)(float)sqrt(5.991|7.815) */
  double delta_ln_mono, delta_ln_stereo;  /* (double)(float)(delta*gamma) */
  float chi2_mono, chi2_stereo;           /* 5.991f 7.815f */
  double gate_ln_mono, gate_ln_stereo;    /* (double)(deltaLines*deltaLines as float) */
  int32_t n_rounds;  /* 4 */
  int32_t its;       /* 10 */
} lld_pose_problem;

typedef struct lld_pose_result {
  double* Tcw;           /* [n_frames][12] */
  uint8_t* pt_outlier;   /* [n_pt]  pFrame->mvbOutlier */
  uint8_t* ln_outlier;   /* [n_ln]  pFrame->mvbOutlierLines (last edge of the line wins, as in the reference) */
  int32_t* n_inliers;    /* [n_frames] return value nInitialCorrespondences - nBad (0 when <3 correspondences) */
  double* chi2_final;    /* [n_frames] robust chi2 after the last LM iteration of the last round; may be NULL */
} lld_pose_result;

int lld_pose_opt(void* ctx, const lld_pose_problem* p, lld_pose_result* out);

/* ------------------------------------------------------------------------------------------------
 * ORB descriptor matching
 * ---------------------------------------------------------------------------------------------- */
/* host inline popcount distance, identical to ORBmatcher::DescriptorDistance */
int lld_descriptor_distance(const uint8_t a[32], const uint8_t b[32]);

/* Frame grid parameters shared by both SearchByProjection variants (src/Frame.cc:391-456, include/Frame.h:43-44) */
typedef struct lld_frame_geom {
  float fx, fy, cx, cy, bf, b; /* b = mb, stereo baseline in metres (forward/backward test) */
  float min_x, max_x, min_y, max_y; /* mnMinX ... image bounds after undistortion */
  int32_t n_levels;
  const float* scale_factors; /* [n_levels] mvScaleFactors */
} lld_frame_geom;

/* SearchByProjection(CurrentFrame, LastFrame, th, bMono), batched over frame pairs. */
typedef struct lld_sbp_frame_problem {
  int32_t n_pairs;
  lld_frame_geom geom;
  float th;
  int32_t mono;              /* bMono */
  int32_t check_orientation; /* mbCheckOrientation */
  /* current frames */
  const int32_t* cur_off;    /* [n_pairs+1] */
  const float* cur_xy;       /* [n_cur][2] mvKeysUn[i].pt */
  const uint8_t* cur_octave; /* [n_cur] */
  const float* cur_angle;    /* [n_cur] */
  const float* cur_uright;   /* [n_cur] */
  const uint8_t* cur_desc;   /* [n_cur][32] */
  const uint8_t* cur_claimed;/* [n_cur] mvpMapPoints[i] && Observations()>0 on entry */
  const float* cur_Tcw;      /* [n_pairs][12] float */
  const float* last_Tcw;     /* [n_pairs][12] float */
  /* last frames */
  const int32_t* last_off;   /* [n_pairs+1] */
  const uint8_t* last_valid; /* [n_last] mvpMapPoints[i] && !mvbOutlier[i] */
  const float* last_xw;      /* [n_last][3] pMP->GetWorldPos() */
  const uint8_t* last_octave;/* [n_last] mvKeys[i].octave */
  const float* last_angle;   /* [n_last] mvKeysUn[i].angle */
  const uint8_t* last_desc;  /* [n_last][32] pMP->GetDescriptor() */
  const uint8_t* last_has_obs;/* [n_last] pMP->Observations()>0 : a kp claimed by this point blocks later points */
  /* The relocalisation variant ORBmatcher::SearchByProjection(Frame&, KeyFrame*, const set<MapPoint*>&, th, ORBdist)
   * (include/ORBmatcher.h:56, src/ORBmatcher.cc:1472-1599) is the same search with: "last" = the keyframe's map points
   * (last_valid = non-null, not bad, not in sAlreadyFound, dist3D inside the scale-invariance range; last_octave = the
   * PredictScale level; last_angle = pKF->mvKeysUn[i].angle; last_has_obs = 1: every accepted match claims its keypoint),
   * mono = 1 (levels [l-1, l+1]), cur_uright = -1 (no stereo test), cur_claimed = mvpMapPoints[i] != NULL, and the two
   * fields below.  Zero (a memset struct) selects the frame-to-frame behaviour. */
  int32_t th_high;              /* accept bestDist <= th_high; 0 = TH_HIGH (100).  Relocalisation: ORBdist */
  int32_t allow_negative_depth; /* 1: no `invzc < 0` rejection (src/ORBmatcher.cc:1497-1502 has none) */
} lld_sbp_frame_problem;

typedef struct lld_sbp_result {
  int32_t* match;      /* [n_cur]  index (pair-local) of the matched last/map point, -1 = none; = CurrentFrame.mvpMapPoints after the call */
  int32_t* n_matches;  /* [n_pairs] return value */
  int32_t* best_idx;   /* [n_last] best current kp found for each query before the orientation filter, -1 = none; may be NULL */
  int32_t* best_dist;  /* [n_last] its Hamming distance (256 when none); may be NULL */
} lld_sbp_result;

int lld_sbp_frame(void* ctx, const lld_sbp_frame_problem* p, lld_sbp_result* out);

/* SearchByProjection(Frame& F, const vector<MapPoint*>&, th), batched over (frame, local-map) pairs. */
typedef struct lld_sbp_mp_problem {
  int32_t n_pairs;
  lld_frame_geom geom;
  float th;
  float nn_ratio;            /* mfNNratio */
  const int32_t* cur_off;    /* frame keypoints, as above */
  const float* cur_xy;
  const uint8_t* cur_octave;
  const float* cur_uright;
  const uint8_t* cur_desc;
  const uint8_t* cur_claimed;
  const int32_t* mp_off;     /* [n_pairs+1] */
  const uint8_t* mp_valid;   /* [n_mp] mbTrackInView && !isBad() */
  const float* mp_proj;      /* [n_mp][3] mTrackProjX, mTrackProjY, mTrackProjXR */
  const int32_t* mp_level;   /* [n_mp] mnTrackScaleLevel */
  const float* mp_viewcos;   /* [n_mp] mTrackViewCos */
  const uint8_t* mp_desc;    /* [n_mp][32] */
  const uint8_t* mp_has_obs; /* [n_mp] */
} lld_sbp_mp_problem;

int lld_sbp_mappoints(void* ctx, const lld_sbp_mp_problem* p, lld_sbp_result* out);

/* Windowed Hamming search of projected map points in a KEYFRAME, batched over (keyframe, point set) pairs:
 *   ORBmatcher::Fuse(KeyFrame*, const vector<MapPoint*>&, th)                      src/ORBmatcher.cc:825-975   chi2_gate = 1, sequential_claims = 0
 *   ORBmatcher::Fuse(KeyFrame*, cv::Mat Scw, const vector<MapPoint*>&, th, ...)   src/ORBmatcher.cc:977-1100  chi2_gate = 0, sequential_claims = 0
 *   ORBmatcher::SearchByProjection(KeyFrame*, cv::Mat Scw, vpPoints, vpMatched, th) src/ORBmatcher.cc:290-403 chi2_gate = 0, sequential_claims = 1,
 *                                                                                   kp_claimed = (vpMatched[idx] != NULL) on entry
 * The caller does what precedes the search in those functions (projection with Rcw / tcw or the decomposed Scw, depth, image bounds,
 * distance-invariance and viewing-angle tests, MapPoint::PredictScale -- its logf stays on the host) and passes u, v, ur and the predicted
 * level; invalid points are flagged in mp_valid.  The library runs KeyFrame::GetFeaturesInArea (radius th * mvScaleFactors[level], same
 * 64 x 48 grid as the Frame), the level window [level - 1, level], the optional reprojection gate of Fuse
 * (e2 * mvInvLevelSigma2[kpLevel] > 7.8 with mvuRight >= 0, > 5.99 otherwise; :905-925), strict-< first-minimum selection, acceptance at
 * bestDist <= th_low, and -- with sequential_claims -- the rule that an accepted match removes its keypoint for the points after it.
 * What follows the search in Fuse (Replace / AddObservation under the map mutex) stays with the caller, fed from best_idx.
 * Result: lld_sbp_result; best_idx / best_dist per map point (-1 / 256 when not accepted), match = last accepted point per keypoint. */
typedef struct lld_kf_search_problem {
  int32_t n_pairs;
  lld_frame_geom geom;
  float th;
  int32_t th_low;             /* TH_LOW = 50 */
  int32_t chi2_gate;
  int32_t sequential_claims;
  float inv_level_sigma2[8];  /* mvInvLevelSigma2 */
  const int32_t* kp_off;      /* [n_pairs+1] keyframe keypoints */
  const float* kp_xy;         /* [n_kp][2] mvKeysUn */
  const uint8_t* kp_octave;
  const float* kp_uright;     /* mvuRight (< 0: monocular keypoint) */
  const uint8_t* kp_desc;     /* [n_kp][32] */
  const uint8_t* kp_claimed;  /* [n_kp] skipped keypoints (vpMatched[idx] on entry); zeros for Fuse */
  const int32_t* mp_off;      /* [n_pairs+1] */
  const uint8_t* mp_valid;    /* [n_mp] passed every test before GetFeaturesInArea */
  const float* mp_proj;       /* [n_mp][3] u, v, ur */
  const int32_t* mp_level;    /* [n_mp] nPredictedLevel */
  const uint8_t* mp_desc;     /* [n_mp][32] */
} lld_kf_search_problem;

int lld_kf_search(void* ctx, const lld_kf_search_problem* p, lld_sbp_result* out);

/* ORBmatcher::SearchForTriangulation(KeyFrame* pKF1, KeyFrame* pKF2, cv::Mat F12, vMatchedPairs, bOnlyStereo)
 * src/ORBmatcher.cc:657-823 with CheckDistEpipolarLine (:140-157), batched over keyframe pairs.
 * Keypoints of the two keyframes that share a vocabulary node (DBoW2::FeatureVector: node id -> keypoint indices; passed as CSR
 * lists sorted by node id, the order std::map iterates in) are compared all against all; per keypoint of KF1 without a map point the
 * LAST keypoint of KF2's bucket (bucket order) with dist <= TH_LOW and dist <= the best so far that has no map point, is not
 * within 10 sqrt(scale) px of the epipole (both monocular) and lies within 3.84 sigma^2 of the epipolar line wins; then the
 * rotation-histogram filter.  (vbMatched2 is never set by the reference, so the keypoints of KF1 are independent.)
 * The caller computes the epipole (ex, ey) (:665-671). */
typedef struct lld_tri_search_problem {
  int32_t n_pairs;
  int32_t only_stereo;          /* bOnlyStereo */
  int32_t check_orientation;    /* mbCheckOrientation */
  int32_t n_levels;
  float scale_factors[8];       /* pKF2->mvScaleFactors */
  float level_sigma2[8];        /* pKF2->mvLevelSigma2 */
  const float* F12;             /* [n_pairs][9] row-major */
  const float* epipole;         /* [n_pairs][2] ex, ey */
  /* keyframe 1 / keyframe 2 keypoints, CSR over pairs */
  const int32_t* kp1_off;       /* [n_pairs+1] */
  const float* kp1_xy;          /* [n1][2] mvKeysUn */
  const float* kp1_angle;       /* [n1] */
  const float* kp1_uright;      /* [n1] mvuRight */
  const uint8_t* kp1_has_mp;    /* [n1] GetMapPoint(idx) != NULL */
  const uint8_t* kp1_desc;      /* [n1][32] */
  const int32_t* kp2_off;
  const float* kp2_xy;
  const uint8_t* kp2_octave;
  const float* kp2_angle;
  const float* kp2_uright;
  const uint8_t* kp2_has_mp;
  const uint8_t* kp2_desc;
  /* feature vectors: per pair a run of nodes (ascending node id), per node a run of pair-local keypoint indices */
  const int32_t* fv1_node_off;  /* [n_pairs+1] into fv1_node / fv1_idx_off */
  const int32_t* fv1_node;      /* [n_nodes1] node ids */
  const int32_t* fv1_idx_off;   /* [n_nodes1+1] into fv1_idx */
  const int32_t* fv1_idx;       /* keypoint indices (pair-local) */
  const int32_t* fv2_node_off;
  const int32_t* fv2_node;
  const int32_t* fv2_idx_off;
  const int32_t* fv2_idx;
} lld_tri_search_problem;

typedef struct lld_tri_search_result {
  int32_t* match12;    /* [n1] vMatches12: pair-local index in keyframe 2 or -1 (after the rotation filter) */
  int32_t* n_matches;  /* [n_pairs] */
} lld_tri_search_result;

int lld_tri_search(void* ctx, const lld_tri_search_problem* p, lld_tri_search_result* out);

/* ORBmatcher::SearchByBoW(KeyFrame* pKF, Frame& F, vpMapPointMatches)        src/ORBmatcher.cc:159-288   strict_th = 0, kp2_valid = all ones
 * ORBmatcher::SearchByBoW(KeyFrame* pKF1, KeyFrame* pKF2, vpMatches12)         src/ORBmatcher.cc:522-655   strict_th = 1, kp2_valid = good map point
 * batched over pairs.  Keypoints of side 1 that carry a good map point (kp1_valid) are matched against the keypoints of side 2 in the
 * same vocabulary node: best and second best Hamming distance over the bucket (strict <, bucket order), acceptance at
 * bestDist1 <= TH_LOW (< TH_LOW when strict_th) and bestDist1 < nn_ratio * bestDist2 (float), an accepted match removes its side-2
 * keypoint for the entries after it (vpMapPointMatches[realIdxF] / vbMatched2[idx2]; only entries of the same node can compete for
 * it), then the rotation-histogram filter.  match12[i] = matched side-2 keypoint of side-1 keypoint i (each side-2 keypoint at most
 * once, so the first overload's vpMapPointMatches[match12[i]] = pMP_i is the inverse map). */
typedef struct lld_bow_search_problem {
  int32_t n_pairs;
  int32_t strict_th;
  int32_t check_orientation;
  float nn_ratio;
  const int32_t* kp1_off;       /* [n_pairs+1] */
  const float* kp1_angle;       /* [n1] mvKeysUn[i].angle */
  const uint8_t* kp1_valid;     /* [n1] map point present and not bad */
  const uint8_t* kp1_desc;      /* [n1][32] */
  const int32_t* kp2_off;
  const float* kp2_angle;       /* F.mvKeys[i].angle / mvKeysUn[i].angle */
  const uint8_t* kp2_valid;
  const uint8_t* kp2_desc;
  const int32_t* fv1_node_off;  /* feature vectors as in lld_tri_search_problem */
  const int32_t* fv1_node;
  const int32_t* fv1_idx_off;
  const int32_t* fv1_idx;
  const int32_t* fv2_node_off;
  const int32_t* fv2_node;
  const int32_t* fv2_idx_off;
  const int32_t* fv2_idx;
} lld_bow_search_problem;

int lld_bow_search(void* ctx, const lld_bow_search_problem* p, lld_tri_search_result* out);

/* ORBmatcher::SearchForInitialization(Frame& F1, Frame& F2, vector<cv::Point2f>& vbPrevMatched, vector<int>& vnMatches12,
 * int windowSize)  src/ORBmatcher.cc:405, batched over frame pairs (Tracking::MonocularInitialization: ORBmatcher(0.9, true),
 * windowSize = 100, vbPrevMatched carried from one call to the next).
 * For every F1 keypoint of octave 0, in index order: the level-0 F2 keypoints of F2.GetFeaturesInArea(vbPrevMatched[i1],
 * windowSize) (F2's 64 x 48 grid over mvKeysUn, cells x outer / y inner, insertion order) whose vMatchedDistance is above the
 * distance are compared; best / second best with strict <; accepted at bestDist <= TH_LOW (50) and
 * bestDist < (float)bestDist2 * nn_ratio.  An accepted match takes its F2 keypoint away from an earlier query (which becomes -1).
 * Then the rotation-histogram filter over every accepted match, displaced ones included (ComputeThreeMaxima), and
 * vbPrevMatched[i1] = F2.mvKeysUn[vnMatches12[i1]].pt for the matched i1. */
typedef struct lld_init_search_problem {
  int32_t n_pairs;
  lld_frame_geom geom;          /* F2's grid: only min_x, max_x, min_y, max_y are read */
  int32_t window_size;          /* windowSize */
  float nn_ratio;               /* mfNNratio */
  int32_t check_orientation;    /* mbCheckOrientation */
  const int32_t* kp1_off;       /* [n_pairs+1] F1 keypoints */
  const uint8_t* kp1_octave;    /* [n1] F1.mvKeysUn[i].octave */
  const float* kp1_angle;       /* [n1] F1.mvKeysUn[i].angle */
  const uint8_t* kp1_desc;      /* [n1][32] F1.mDescriptors */
  const float* prev_matched;    /* [n1][2] vbPrevMatched on entry */
  const int32_t* kp2_off;       /* [n_pairs+1] F2 keypoints */
  const float* kp2_xy;          /* [n2][2] F2.mvKeysUn[i].pt */
  const uint8_t* kp2_octave;    /* [n2] */
  const float* kp2_angle;       /* [n2] */
  const uint8_t* kp2_desc;      /* [n2][32] */
} lld_init_search_problem;

typedef struct lld_init_search_result {
  int32_t* match12;       /* [n1] vnMatches12: pair-local F2 index or -1 */
  int32_t* n_matches;     /* [n_pairs] return value */
  float* prev_matched;    /* [n1][2] vbPrevMatched after the call; may be the problem's prev_matched array */
} lld_init_search_result;

int lld_init_search(void* ctx, const lld_init_search_problem* p, lld_init_search_result* out);

/* ------------------------------------------------------------------------------------------------
 * Loop-candidate Sim3 optimisation: Optimizer::OptimizeSim3(pKF1, pKF2, vpMatches1, g2oS12, th2, bFixScale)
 * src/Optimizer.cc:1656-1858, batched over loop candidates (LoopClosing::ComputeSim3 calls it with th2 = 10 and mbFixScale).
 * One VertexSim3Expmap (estimate g2oS12, _fix_scale, K1 / K2) and, per correspondence i in vpMatches1 order, the fixed
 * camera-frame points P1c = R1w X1w + t1w, P2c = R2w X2w + t2w and two edges in this order:
 *   e12 = obs1 - cam_map1(project(S12.map(P2c))),  e21 = obs2 - cam_map2(project(S12.inverse().map(P1c))),
 * information invSigma2 I2 of the keypoint's own keyframe, Huber delta = sqrtf(th2).  The edges are differentiated
 * numerically as g2o does (central differences at 1e-9; with a fixed scale the scale column is 0).  Levenberg-Marquardt
 * with a dense 7x7 LDL^T: optimize(its_first); a correspondence whose e12 or e21 chi2 (of the last evaluated error, also
 * when that LM trial was rejected) exceeds th2 is dropped (inlier = 0); fewer than 10 left: n_in = 0 and S12 = the input
 * (the drops stay); else optimize(its_more_outliers if any was dropped, its_more_clean otherwise) from the state reached,
 * the same test again, n_in = the correspondences that pass it.  Correspondences the reference skips (no map point in
 * pKF1, a bad point, i2 < 0) are not passed; the caller leaves their vpMatches1 entries as they are.
 * ---------------------------------------------------------------------------------------------- */
typedef struct lld_sim3_problem {
  int32_t n_problems;
  const double* S12;          /* [n][8] g2o::Sim3: qx qy qz qw, tx ty tz, s */
  const double* cam;          /* [n][8] fx1 fy1 cx1 cy1 fx2 fy2 cx2 cy2: pKF1->mK, pKF2->mK (float values, widened) */
  const int32_t* fix_scale;   /* [n] bFixScale: 0 or 1 */
  const float* th2;           /* [n] th2 > 0 */
  const int32_t* off;         /* [n+1] CSR over correspondences, off[0] = 0 */
  const float* p1c;           /* [m][3] P1c, computed in float as the reference does (cv::Mat) */
  const float* p2c;           /* [m][3] P2c */
  const float* obs1;          /* [m][2] pKF1->mvKeysUn[i].pt */
  const float* obs2;          /* [m][2] pKF2->mvKeysUn[i2].pt */
  const float* info1;         /* [m] pKF1->mvInvLevelSigma2[octave of kpUn1] */
  const float* info2;         /* [m] pKF2->mvInvLevelSigma2[octave of kpUn2] */
  int32_t its_first;          /* 5 */
  int32_t its_more_outliers;  /* 10 */
  int32_t its_more_clean;     /* 5 */
} lld_sim3_problem;

typedef struct lld_sim3_result {
  double* S12;          /* [n][8] g2oS12 after the call */
  uint8_t* inlier;      /* [m] 1 = vpMatches1[i] kept, 0 = cleared */
  int32_t* n_in;        /* [n] return value */
  /* LM trace, [n][log_stride] (log_stride >= its_first + max(its_more_*) + 2 when a log is given): round 1 at entry 0, round 2
   * at entry its_first + 1; in each round entry 0 = robust chi2 at the start, entry k = chi2 / lambda / trials after LM
   * iteration k; the rest is 0.  n_iter_done[n][2] = iterations run per round (0 for a round that did not run). */
  int32_t log_stride;
  double* chi2_log;     /* may be NULL */
  double* lambda_log;   /* may be NULL */
  int32_t* trials_log;  /* may be NULL */
  int32_t* n_iter_done; /* may be NULL */
} lld_sim3_result;

int lld_sim3_opt(void* ctx, const lld_sim3_problem* p, lld_sim3_result* out);

/* ------------------------------------------------------------------------------------------------
 * Loop-candidate Sim3 RANSAC: Sim3Solver (ORB-SLAM2 src/Sim3Solver.cc, inherited unchanged by LLD-SLAM), batched over loop
 * candidates (LoopClosing::ComputeSim3 calls SetRansacParameters(0.99, 20, 300) and iterate(5, ...) per candidate per round).
 * Correspondences are the ones the constructor keeps (vpMatched12[i1] and pKF1's map point i1 both present and good, and both
 * points' GetIndexInKeyFrame >= 0), in vpMatched12 order; x1c / x2c are their camera-frame points mvX3Dc1 / mvX3Dc2 as the
 * caller computed them, sigma2_1 / sigma2_2 the mvLevelSigma2 of their keypoints' octaves.  The library forms everything else
 * as the reference does:
 *   - thresholds mvnMaxError = 9.210 * sigma2 stored in a size_t, i.e. truncated to an integer (9 at octave 0);
 *   - mvP1im1 / mvP2im2: the points' own camera coordinates projected with K1 / K2 (float invz, no depth test);
 *   - ComputeSim3 (Horn 1987) in CV_32F: centroids (cv::reduce, then / 3), M = Pr2 Pr1^T, the symmetric 4x4 N, the eigenvector
 *     of its largest eigenvalue as the quaternion (w first), ang = atan2(|v|, w) and v = 2 ang v / |v| in double,
 *     cv::Rodrigues, s = Pr1 . (R Pr2) / sum (R Pr2)^2 (nom, den in double; s = 1 with fix_scale), t = O1 - s R O2,
 *     T12 = [sR | t], T21 = [(1/s) R^T | -(1/s) R^T t];
 *   - CheckInliers: x2c projected with T12 / K1 against mvP1im1 and x1c with T21 / K2 against mvP2im2, err = dist . dist
 *     (float); inlier iff err1 < maxErr1 && err2 < maxErr2 (a NaN from a degenerate minimal set is an outlier).
 * Products of small CV_32F matrices follow cv::gemm: a 3-long product without transposition sums float products in float,
 * M = Pr2 Pr1^T sums in double; both round once to float.  The eigen solver is a cyclic Jacobi in double on the float N, not
 * OpenCV's: its eigenvector may differ in the last bits, and the sign of the eigenvector cancels in the atan2 form.
 *
 * iterate(nIterations): with N = off[p+1] - off[p] < min_inliers nothing is drawn, no_more = 1.  Otherwise minimal sets are
 * evaluated in order while its_done < max_its and fewer than n_iterations were evaluated in this call: a set whose inlier
 * count reaches best_inliers (>=) becomes the best; if its count also exceeds min_inliers (strictly: 20 is not enough, 21 is)
 * the call stops with found = 1 and that estimate.  Afterwards (no success) no_more = its_done >= max_its; a success on the
 * last allowed set returns no_more = 0 and the next call evaluates nothing and sets it.  its_done and best_inliers are the
 * solver's mnIterations and mnBestInliers: the caller passes them back in the next round (a candidate whose OptimizeSim3
 * failed is iterated again and a new set must reach the carried best).
 *
 * Random draws: the reference draws each set with DUtils::Random::RandomInt(0, size - 1) on rand() by swap-with-back from a
 * fresh copy of 0..N-1.  rand() is one stream for the whole process (relocalisation's PnPsolver draws from it on another
 * thread), so the global sequence is not a contract.  The contract is: given the same minimal sets, this computes what
 * iterate() computes.  The caller draws the sets: problem p receives exactly
 *   B = N < min_inliers ? 0 : min(n_iterations, max(0, max_its - its_done))
 * sets (hyp_off[p+1] - hyp_off[p] == B).  Drawing a whole round up front consumes draws from rand() after an early success,
 * which the reference would not consume.
 * ---------------------------------------------------------------------------------------------- */
typedef struct lld_sim3_ransac_problem {
  int32_t n_problems;
  const float* cam;            /* [n][8] fx1 fy1 cx1 cy1 fx2 fy2 cx2 cy2: pKF1->mK, pKF2->mK */
  const int32_t* fix_scale;    /* [n] mbFixScale: 0 or 1 */
  const int32_t* off;          /* [n+1] CSR over correspondences, off[0] = 0 */
  const float* x1c;            /* [m][3] mvX3Dc1 */
  const float* x2c;            /* [m][3] mvX3Dc2 */
  const float* sigma2_1;       /* [m] pKF1->mvLevelSigma2[octave] */
  const float* sigma2_2;       /* [m] pKF2->mvLevelSigma2[octave] */
  int32_t min_inliers;         /* mRansacMinInliers (20) */
  const int32_t* max_its;      /* [n] mRansacMaxIts after SetRansacParameters (lld_sim3_ransac_max_its), >= 1 */
  const int32_t* its_done;     /* [n] mnIterations before the call */
  const int32_t* best_inliers; /* [n] mnBestInliers before the call */
  int32_t n_iterations;        /* iterate(nIterations): 5 in LoopClosing::ComputeSim3 */
  const int32_t* hyp_off;      /* [n+1] CSR over minimal sets, hyp_off[0] = 0, B sets per problem (above) */
  const int32_t* hyp_idx;      /* [h][3] problem-local correspondence indices of each set, in draw order, distinct */
} lld_sim3_ransac_problem;

typedef struct lld_sim3_ransac_result {
  uint8_t* found;          /* [n] iterate() returned an estimate */
  uint8_t* no_more;        /* [n] bNoMore */
  int32_t* n_inliers;      /* [n] nInliers (0 unless found) */
  float* T12;              /* [n][13] GetEstimatedRotation (R, row-major, unscaled), GetEstimatedTranslation, GetEstimatedScale;
                              written where found, zero elsewhere */
  uint8_t* inlier;         /* [m] vbInliers in CSR order (all 0 unless found) */
  int32_t* its_done;       /* [n] mnIterations after the call (may alias the input) */
  int32_t* best_inliers;   /* [n] mnBestInliers after the call (may alias the input) */
  int32_t* hyp_inliers;    /* [h] mnInliersi of each set, -1 where the set was not evaluated; may be NULL */
} lld_sim3_ransac_result;

/* SetRansacParameters(probability, minInliers, maxIterations) for N = n_corr correspondences, host arithmetic:
 * epsilon = (float)minInliers / N; nIterations = minInliers == N ? 1 : ceil(log(1 - p) / log(1 - pow(epsilon, 3)));
 * returns max(1, min(nIterations, maxIterations)).  Defined for n_corr >= min_inliers; below, iterate() draws nothing and the
 * function returns 1. */
int32_t lld_sim3_ransac_max_its(int32_t n_corr, double probability, int32_t min_inliers, int32_t max_iterations);

int lld_sim3_ransac(void* ctx, const lld_sim3_ransac_problem* p, lld_sim3_ransac_result* out);

/* ------------------------------------------------------------------------------------------------
 * Relocalisation EPnP RANSAC: PnPsolver (ORB-SLAM2 src/PnPsolver.cc, inherited unchanged by LLD-SLAM), batched over
 * relocalisation candidates (Tracking::Relocalization calls SetRansacParameters(0.99, 10, 300, 4, 0.5, 5.991) and
 * iterate(5, ...) per candidate per round).  The reference source is not at hand: the rules below are transcribed from
 * ORB-SLAM2's PnPsolver.cc as recalled, and they are the contract.
 *   - Constructor PnPsolver(F, vpMapPointMatches): every i whose map point is present and not bad, in index order; p2d =
 *     F.mvKeysUn[i].pt, p3dw = GetWorldPos() (float), sigma2 = F.mvLevelSigma2[octave]; fu fv uc vc = F.fx fy cx cy.
 *   - max_err[i] = mvMaxError[i] = sigma2 * th2 in float, formed by the caller.
 *   - iterate(nIterations): with N < min_inliers nothing is drawn and no_more = 1.  Otherwise minimal sets of 4 are evaluated
 *     while (its_done < max_its || evaluated in this call < n_iterations) (an ||, where Sim3Solver has &&).  Per set: EPnP,
 *     CheckInliers; if its count reaches min_inliers (>=): when it beats best_inliers (strictly) its mask, count and pose become
 *     the best, and then Refine runs on the best mask (possibly carried from an earlier set or call): EPnP over every best
 *     inlier, CheckInliers; it succeeds iff the refined count exceeds min_inliers (strictly), and the call returns the refined
 *     pose, count and mask with found = 1, no_more = 0.  After the loop no_more = 1 and, if best_inliers >= min_inliers, the call
 *     returns the best pose, count and mask (found = 1).  A call that does not succeed always ends with no_more = 1.
 *   - CheckInliers: Xc, Yc, invZc = 1 / (...) computed in double (double R, t times the float point) and stored to float;
 *     ue = uc + fu * Xc * invZc in double; distX = u - ue stored to float; error2 = distX^2 + distY^2 in float; inlier iff
 *     error2 < max_err (a NaN is an outlier; there is no depth test).
 *   - EPnP (compute_pose) is Lepetit's epnp.cpp: control points (centroid, principal axes of PW0^T PW0 scaled by sqrt(d / n)),
 *     barycentric coordinates through CC^-1 (the SVD pseudo-inverse), M^T M, the eigenvectors of its four smallest eigenvalues, L_6x10 and rho,
 *     find_betas_approx_1 / 2 / 3 (L columns {0,1,3,6} / {0,1,2} / {0,1,2,3,4}, least squares through the SVD, their sign and
 *     sqrt rules; as in OpenCV's back-substitution, the SVD solves and CC^-1 skip singular values at or below
 *     2 DBL_EPSILON times their sum, so coplanar world points drop the vanishing control axis; for
 *     them the third left singular vector of ABt, which OpenCV draws from its RNG, is the cross product of the other two), each followed by 5 Gauss-Newton steps (unpivoted Householder QR of the 6x4 system; a singular system adds
 *     nothing), compute_R_and_t (ccs from ut rows 11 - i, pcs, the sign flip on the first point's depth, R = U V^T of the SVD
 *     of ABt with row 2 negated when det < 0, the mean of the sqrt reprojection distances).  Solution 1 is kept, replaced by 2
 *     if its error is smaller, then by 3 if smaller than the kept one.  The SVDs and the eigen decomposition are cyclic
 *     Jacobi in double (two-sided on the symmetric PW0^T PW0 and M^T M, one-sided on CC, ABt and the L systems), not OpenCV's:
 *     singular vectors differ in sign and, in a repeated null space (four points), in basis, which the betas absorb.
 *     Every sum over correspondences runs serially in correspondence order.
 * Random draws: as lld_sim3_ransac, the caller draws the sets (DUtils::Random::RandomInt on rand(), swap-with-back from a fresh
 * 0..N-1); given the same sets this computes what iterate() computes.  Problem p receives exactly
 *   B = N < min_inliers ? 0 : max(n_iterations, max_its - its_done)
 * sets.  The state the reference keeps between calls (mnIterations, mnBestInliers, mvbBestInliers, mBestTcw) is passed in and
 * out.  The minimal set size is 4 (SetRansacParameters' minSet only enters the min_inliers floor).
 * ---------------------------------------------------------------------------------------------- */
typedef struct lld_pnp_ransac_problem {
  int32_t n_problems;
  const float* cam;            /* [n][4] fx fy cx cy (widened to double as fu fv uc vc) */
  const int32_t* min_inliers;  /* [n] mRansacMinInliers after SetRansacParameters (lld_pnp_ransac_params), >= 4 */
  const int32_t* max_its;      /* [n] mRansacMaxIts after SetRansacParameters, >= 1 */
  const int32_t* its_done;     /* [n] mnIterations before the call */
  const int32_t* best_inliers; /* [n] mnBestInliers before the call */
  const int32_t* off;          /* [n+1] CSR over correspondences, off[0] = 0 */
  const float* p2d;            /* [m][2] mvP2D */
  const float* p3dw;           /* [m][3] mvP3Dw */
  const float* max_err;        /* [m] mvMaxError = mvSigma2 * th2 (float) */
  const uint8_t* best_mask;    /* [m] mvbBestInliers before the call (read where best_inliers >= min_inliers) */
  const float* best_Tcw;       /* [n][12] mBestTcw before the call: R row-major, t */
  int32_t n_iterations;        /* iterate(nIterations): 5 in Tracking::Relocalization */
  const int32_t* hyp_off;      /* [n+1] CSR over minimal sets, hyp_off[0] = 0, B sets per problem (above) */
  const int32_t* hyp_idx;      /* [h][4] problem-local correspondence indices of each set, in draw order, distinct */
} lld_pnp_ransac_problem;

typedef struct lld_pnp_ransac_result {
  uint8_t* found;          /* [n] iterate() returned a pose */
  uint8_t* no_more;        /* [n] bNoMore */
  int32_t* n_inliers;      /* [n] nInliers (0 unless found) */
  float* Tcw;              /* [n][12] the returned pose, R row-major then t (float); zero where not found */
  uint8_t* inlier;         /* [m] vbInliers in CSR order (all 0 unless found) */
  int32_t* its_done;       /* [n] mnIterations after the call (may alias the input) */
  int32_t* best_inliers;   /* [n] mnBestInliers after the call (may alias the input) */
  uint8_t* best_mask;      /* [m] mvbBestInliers after the call (may alias the input) */
  float* best_Tcw;         /* [n][12] mBestTcw after the call (may alias the input) */
  int32_t* hyp_inliers;    /* [h] mnInliersi of each set, -1 where the set was not evaluated; may be NULL */
} lld_pnp_ransac_result;

/* SetRansacParameters(probability, minInliers, maxIterations, minSet, epsilon, th2) for N = n_corr, host arithmetic:
 * nMinInliers = (int)(N * epsilon) (float product), raised to minInliers, then to minSet; epsilon raised to
 * (float)nMinInliers / N; nIterations = nMinInliers == N ? 1 : ceil(log(1 - p) / log(1 - pow(epsilon, 3))); out[0] = nMinInliers,
 * out[1] = max(1, min(nIterations, maxIterations)) (1 where the logarithm is undefined, N < nMinInliers).  Returns LLD_ERR_ARG
 * for n_corr < 0 or a NULL out. */
int lld_pnp_ransac_params(int32_t n_corr, double probability, int32_t min_inliers, int32_t max_iterations, int32_t min_set,
                          float epsilon, int32_t out[2]);

int lld_pnp_ransac(void* ctx, const lld_pnp_ransac_problem* p, lld_pnp_ransac_result* out);

/* ------------------------------------------------------------------------------------------------
 * Stereo line matching (float line descriptors)
 * ---------------------------------------------------------------------------------------------- */
typedef struct lld_line_match_problem {
  int32_t n_pairs;
  int32_t desc_dim;         /* D floats per descriptor row */
  const int32_t* left_off;  /* [n_pairs+1] */
  const int32_t* right_off; /* [n_pairs+1] */
  const float* left_seg;    /* [n_left][4] startPointX startPointY endPointX endPointY */
  const int32_t* left_octave;
  const float* right_seg;
  const int32_t* right_octave;
  const float* left_desc;   /* [n_left][D] */
  const float* right_desc;  /* [n_right][D] */
  double K[9];              /* row-major */
  double baseline;          /* b of TwoFrameLineMatcher(K,b,tau,minLineLength,matcher) */
  double tau;
  int32_t min_line_length;
} lld_line_match_problem;

typedef struct lld_line_match_result {
  int32_t* match;  /* [n_left] pair-local right index or -1 */
  float* dist;     /* [n_left] descriptor distance of the match (inf when none); may be NULL */
} lld_line_match_result;

int lld_line_match(void* ctx, const lld_line_match_problem* p, lld_line_match_result* out);

/* ------------------------------------------------------------------------------------------------
 * Stereo keypoint matching of a frame: Frame::ComputeStereoMatches  include/Frame.h:86, src/Frame.cc:530-704
 * (row-banded Hamming candidates, 11x11 SAD slide at the keypoint's pyramid level, parabola fit, median gate).
 * Batched over frames; every frame brings its own left / right image pyramids (ORBextractor::mvImagePyramid).
 * ---------------------------------------------------------------------------------------------- */
typedef struct lld_stereo_problem {
  int32_t n_frames;
  const int32_t* left_off;     /* [n_frames+1] */
  const int32_t* right_off;    /* [n_frames+1]; at most 65535 right keypoints per frame */
  const float* left_xy;        /* [n_left][2]  mvKeys[i].pt (level-0 pixel coordinates) */
  const uint8_t* left_octave;  /* [n_left]     mvKeys[i].octave, < n_levels (both sides) */
  const uint8_t* left_desc;    /* [n_left][32] mDescriptors */
  const float* right_xy;       /* mvKeysRight, mDescriptorsRight */
  const uint8_t* right_octave;
  const uint8_t* right_desc;
  int32_t n_levels;            /* <= 8 */
  const float* scale_factors;      /* [n_levels] mvScaleFactors */
  const float* inv_scale_factors;  /* [n_levels] mvInvScaleFactors */
  const uint8_t* pyr;          /* all pyramid images of the batch, 8-bit, concatenated */
  int64_t pyr_bytes;
  const int64_t* pyr_off;      /* [n_frames][2][n_levels] byte offset of image (frame, 0 = left / 1 = right, level) in pyr */
  const int32_t* pyr_rows;     /* [n_levels] the same geometry for every frame */
  const int32_t* pyr_cols;
  const int32_t* pyr_stride;   /* row stride in bytes */
  float mb, mbf;               /* baseline in metres, baseline * fx */
} lld_stereo_problem;

typedef struct lld_stereo_result {
  float* uright;       /* [n_left] mvuRight, -1 = no stereo match */
  float* depth;        /* [n_left] mvDepth,  -1 = no stereo match */
  int32_t* n_matched;  /* [n_frames] may be NULL */
} lld_stereo_result;

int lld_stereo_matches(void* ctx, const lld_stereo_problem* p, lld_stereo_result* out);

/* ------------------------------------------------------------------------------------------------
 * Distinctive (medoid) descriptors: MapPoint::ComputeDistinctiveDescriptors  include/MapPoint.h:62, src/MapPoint.cc:242-307
 *                                   MapLine::ComputeDistinctiveDescriptors   include/MapLine.h:66,  src/MapLine.cc:133-201
 * Batched over landmarks: landmark l owns descriptors [off[l], off[l+1]) — the rows of its observations in non-bad
 * keyframes, in std::map<KeyFrame*, size_t> order.  best[l] = landmark-local index of the descriptor with the least median
 * distance to the others (the first one on ties), -1 for a landmark without descriptors.  At most 256 per landmark.
 * ---------------------------------------------------------------------------------------------- */
int lld_medoid_orb(void* ctx, int32_t n_lm, const int32_t* off, const uint8_t* desc /*[n][32]*/, int32_t* best);
int lld_medoid_float(void* ctx, int32_t n_lm, const int32_t* off, int32_t desc_dim, const float* desc /*[n][desc_dim]*/, int32_t* best);

/* ------------------------------------------------------------------------------------------------
 * Temporal line association: Tracking::AddLinesFrom  include/Tracking.h, src/Tracking.cc:996-1124
 * (reprojection gate vgl::LineReprojErrorL1 src/vgl.cc:548-559 in the left and the right image, octave-scaled threshold
 * GetReprojThrPyramid src/LineMatching.cc:239-247, smallest descriptor distance, sequential claim of current lines).
 * Batched over frames.  The candidate lists are an input: the reference takes them from Frame::lines_grid through
 * SubselectWithGrid, but the release never fills that grid; the caller decides which current lines a map line sees.
 * ---------------------------------------------------------------------------------------------- */
typedef struct lld_line_assoc_problem {
  int32_t n_frames;
  const int32_t* ml_off;         /* [n_frames+1] map lines offered to the frame (lines_last), in call order */
  const uint8_t* ml_valid;       /* [n_ml] pML && pML->tracked_last_id != frame id && !pML->isBad() */
  const double* ml_x0_dir;       /* [n_ml][6] GetMinimalPos */
  const double* ml_x1x2;         /* [n_ml][6] GetMainPoints3D */
  const float* ml_desc;          /* [n_ml][desc_dim] descs[i] / mLastFrame.mDescriptorsLines.row(i) */
  const int32_t* cand_off;       /* [n_ml+1] */
  const int32_t* cand_idx;       /* sub_inds: frame-local indices of current left lines, in SubselectWithGrid order;
                                    in [0, the frame's current lines) */
  const int32_t* cur_off;        /* [n_frames+1] current frame left lines */
  const float* cur_left;         /* [n_cur][4] mvLinesLeft start / end point */
  const int32_t* cur_octave;     /* [n_cur] mvLinesLeft[si].octave */
  const int32_t* cur_line_match; /* [n_cur] line_matches[si]: frame-local right line (< the frame's right lines) or -1 */
  const uint8_t* cur_taken;      /* [n_cur] mvpMapLines[si] != NULL on entry */
  const float* cur_desc;         /* [n_cur][desc_dim] mDescriptorsLines */
  const int32_t* right_off;      /* [n_frames+1] */
  const float* cur_right;        /* [n_right][4] mvLinesRight */
  int32_t desc_dim;
  const double* T_curr;          /* [n_frames][16] row-major 4x4, the convention of vgl::MapPoint: R^T (X - c) */
  const double* T_right;         /* [n_frames][16] GetTForRight(T_curr, mb) */
  double K[9];
  double thr_reproj_base;        /* thrReprojLineBase */
  double md_thr;                 /* mdThr */
  int32_t monocular;             /* mSensor == System::MONOCULAR */
} lld_line_assoc_problem;

typedef struct lld_line_assoc_result {
  int32_t* cur_assoc;  /* [n_cur] frame-local index of the map line newly associated with the current line, -1 = none */
  int32_t* n_added;    /* [n_frames] cnt_added; may be NULL */
} lld_line_assoc_result;

int lld_line_associate(void* ctx, const lld_line_assoc_problem* p, lld_line_assoc_result* out);

/* Library self-description (for tests and the bench): version string, number of kernels launched by the
 * last call on this context, device-side duration of the last call measured with CUDA events on the
 * context's stream (milliseconds; h2d/compute/d2h). */
const char* lld_version(void);
int64_t lld_ctx_launch_count(void* ctx);
/* lld_ba_local / lld_ba_global keep the index tables of the last problem on the device; a call whose STRUCTURE (windows,
 * observation lists, fixed flags: a 64-bit hash of those arrays) equals the previous one's skips the host indexing stage
 * and only uploads the value arrays.  on = 1 / 0 switches this per context, -1 restores the default (on; the environment
 * variable LLD_BA_TOPO_CACHE=0 turns the default off). */
void lld_ctx_set_topo_cache(void* ctx, int on);
/* NCCL collectives issued / bytes all-reduced per rank by the last lld_ba_global call on this context */
void lld_ctx_nccl_stats(void* ctx, int64_t* calls, int64_t* bytes);
void lld_ctx_last_timing(void* ctx, float* ms_h2d, float* ms_compute, float* ms_d2h);

#ifdef __cplusplus
}
#endif
#endif /* LLDBA_H */
