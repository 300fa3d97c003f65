// ba.cuh — device-side view of one batched bundle-adjustment problem and the per-window LM state.
//
// Data layout in HBM (all SoA, one contiguous array per field over the whole batch):
//   keyframes   : pose_qt[2][n_kf][7]  (double buffer selected per window by w_sel), pose_Rt[2][n_kf][12] derived,
//                 kf_intr[n_kf][5], kf_lcam[n_kf][4], kf_g[n_kf] (global free-pose block index or -1)
//   map points  : pt_xyz[2][n_pt][3]; CSR pt_obs_off; per edge pe_kf (global kf id), pe_uvr (3 x f32), pe_info (f32)
//   map lines   : ln_st[2][n_ln][5] (q, alpha); CSR ln_obs_off over cells; per cell lc_kf, lc_left/right (4 x f32),
//                 lc_info (2 x f64), lc_stereo
//   edges are grouped by landmark (the reference's insertion order), so one thread owns one landmark's edges;
//   a second index (kfl_*) lists, per free keyframe, the edges that touch it, cut into fixed-size chunks.
#pragma once
#include <stdint.h>

namespace lld {

enum : int { PH_LIN = 0, PH_RETRY = 1, PH_DONE = 2 };

// dense mode, per keyframe slot of a piece in the partial-sum scratch (dpart): the keyframe's b_schur part (6), written by
// k_schur_tile
constexpr int SCHUR_KS = 6;

struct BaParams {
  int robust_pt, robust_ln;
  double delta_pt_mono, delta_pt_stereo, delta_ln_mono, delta_ln_stereo;
  double chi2_pt_mono, chi2_pt_stereo;
  int ln_norm;  // endpoints K^-1-normalised
  int ln_filter;
};

// one work item of k_schur_tile: a block of tasks of one piece, with everything the kernel needs in three 16-byte loads
struct __align__(16) SchurItem {
  int l0, nl, n, t0;   // first landmark (sorted position), landmarks, free keyframes per landmark, first task
  int w, lc;           // window, landmarks per shared-memory chunk
  long long w0;        // first W block of the piece
  long long out;       // scratch offset of the piece's outputs
  int S, nchunk;       // landmark slices per task, chunks of the piece
};

struct BaView {
  int n_win, n_kf, n_pt, n_ln, n_pe, n_lc;
  int n_free_total;  // sum of free poses over the batch
  int n_chunks;
  // static topology
  const int *kf_off, *pt_off, *ln_off;
  const int *kf_win, *pt_win, *ln_win;
  const int* kf_g;       // [n_kf] global free block index or -1
  const int* g_kf;       // [n_free_total] inverse map
  const int* w_g0;       // [n_win+1] first global free block of window
  const double* kf_intr;
  const double* kf_lcam;
  const int* pt_obs_off;
  const int* pe_kf;
  const int* pe_pt;
  const float* pe_uvr;
  const float* pe_info;
  const int* ln_obs_off;
  const int* lc_kf;
  const int* lc_ln;
  const float* lc_left;
  const float* lc_right;
  const double* lc_info;
  const uint8_t* lc_stereo;
  // per-free-KF edge lists ("rows"): points and line cells separately, entries grouped by co-visibility signature,
  // cut into chunks; chunk ids [0, n_chunks_pt) are point chunks, [n_chunks_pt, n_chunks) line chunks
  int n_chunks_pt;
  const int* pl_off;     // [n_free_total+1] point-list offsets
  const int* pl_edge;    // [n_plist] point edge id of the list entry
  const int* pe_pos;     // [n_pe] list position of the edge or -1 (fixed keyframe)
  const int* ll_off;     // [n_free_total+1] line-list offsets
  const int* ll_cell;    // [n_llist] line cell id
  const int* lc_pos;     // [n_lc]
  const int* ch_g;       // [n_chunks] free block of the chunk
  const int* ch_begin;   // [n_chunks] list range of the chunk
  const int* ch_end;
  const int* ch_seg0;    // [n_chunks+1] first segment of the chunk
  const int* seg_begin;  // segments: runs of list entries with the same set of co-observing keyframes
  const int* seg_end;
  const int* g_chp0;     // [n_free_total+1] first point chunk of each free block
  const int* g_chl0;     // [n_free_total+1] first line chunk (absolute chunk id)
  // Schur row structure
  const int* nb_off;     // [n_free_total+1] neighbour list (block columns >= own) per free block, in blocks
  const int* nb_g;       // neighbour global block ids, ascending, first = self
  const int* pl_tab;     // per point-list entry: nnb(a) ints, list position of the co-edge on neighbour j or -1
  const long long* pl_tab_off;  // [n_free_total] offset of block a's first entry row
  const int* ll_tab;
  const long long* ll_tab_off;
  // sparse mode, landmarks seen more than once by one free keyframe: fold group i adds the W records at list positions
  // fold_src[fold_off[i] .. fold_off[i+1]) into the one at fold_dst[i] (the co-edge the tables name) and zeroes them;
  // groups [0, n_fold_pt) are point records, the rest line records (k_fold_dup)
  int n_fold, n_fold_pt;
  const int* fold_off;
  const int* fold_dst;
  const int* fold_src;
  // dense mode (every window has <= 32 free keyframes): landmarks in co-visibility-signature order, W stored per
  // landmark with its free edges sorted by keyframe; k_schur_dense keeps a window's whole S in registers
  int dense_mode;
  const int* pt_sorted;    // [n_pt] landmark at each sorted position
  const int* ln_sorted;
  const int* pt_spos;      // [n_pt] position of the point in signature order (window-contiguous)
  const int* ln_spos;      // [n_ln]
  const uint32_t* pts_mask;  // [n_pt] by sorted position: bit h set when free keyframe h (window-local) observes it
  const uint32_t* lns_mask;  // [n_ln]
  const int* pts_w0;       // [n_pt+1] by sorted position: first W slot of the landmark (free edges, ascending keyframe)
  const int* lns_w0;       // [n_ln+1]
  const int* pe_wpos;      // [n_pe] W slot of the edge or -1
  const int* lc_wpos;      // [n_lc]
  // dense-mode work decomposition: a "piece" is a run of <= 128 landmarks (sorted positions) with the same mask;
  // its tasks are (pair of its keyframes, column c) plus one b_schur task per keyframe; 32 tasks = one warp item
  int n_items;             // warp work items (points first, then lines)
  int n_items_pt;
  const SchurItem* it_rec; // [n_items] self-contained item records (k_schur_tile)
  // gather lists for the reduction: per unit (window, block (a,b)) the contributing (piece, pair) outputs
  const int* gb_off;       // [n_blocks_total+1]   blocks in nb order (same indexing as S_blk)
  const long long* gb_src; // dpart offsets of the pair's first task (6 columns x 6 doubles contiguous)
  const int* gv_off;       // [n_free_total+1]     per free keyframe: b_schur task outputs
  const long long* gv_src;
  double* pe_Wl;           // [n_pwslots][18]
  double* lc_Wl;           // [n_lwslots][24]
  double* pts_D;           // [n_pt][10] by sorted position: inverse packed (6) + D^-1 b_l (3) + pad
  double* lns_D;           // [n_ln][14]
  double* dpart;           // per-task partial sums (6 doubles per task)
  // dynamic state
  double* pose_qt[2];
  double* pose_Rt[2];
  double* pt_xyz[2];
  double* ln_st[2];
  uint8_t* pe_level;
  uint8_t* lc_level;   // [n_lc][2]
  uint8_t* ln_removed;
  double* pe_chi2;
  double* lc_chi2;     // [n_lc][2]
  // linearisation
  double* pt_H;   // [n_pt][9]  Hll (00 01 02 11 12 22) + bl (3)
  double* ln_H;   // [n_ln][14] Hll upper (10) + bl (4)
  double* P_rec;  // [n_plist][27] per point-list entry: W (6x3), (Hll+lambda I)^-1 packed (6), D^-1 b_l (3)
  double* L_rec;  // [n_llist][38] per line-list entry:  W (6x4), inverse packed (10), D^-1 b_l (4)
  double* ch_pose;  // [n_chunks][28] partial Hpp (21 upper) + bp (6) + n_active
  double* g_Hpp;    // [n_free_total][21]
  double* g_bp;     // [n_free_total][6]
  int* g_nact;      // [n_free_total]
  double* lm_chi2lin;  // [n_pt+n_ln]
  double* lm_maxdiag;  // [n_pt+n_ln]
  uint8_t* lm_active;  // [n_pt+n_ln]
  // trial
  double* ch_S;   // chunk partial rows: at ch_S_off[chunk], 6 x (6*nnb) doubles + 6 (b part)
  const long long* ch_S_off;
  double* S_blk;  // [n_nb_total][36]
  double* g_bs;   // [n_free_total][6] bschur
  double* g_x;    // [n_free_total][6] pose solution (kept on failure)
  double* pt_xl;  // [n_pt][3] landmark solution of the last successful solve (applied again when a solve fails, as g2o does)
  double* ln_xl;  // [n_ln][4]
  double* pt_D;   // [n_pt][9]  (Hll+lambda I)^-1 packed (6) + D^-1 b_l (3)
  double* ln_D;   // [n_ln][14] inverse packed (10) + D^-1 b_l (4)
  double* lm_chi2;
  double* lm_scale;
  // per-window LM state
  int* w_phase;
  int* w_sel;
  int* w_iter;
  int* w_trials;
  int* w_maxit;
  int* w_nbad;
  int* w_ok;
  int* w_nlog;
  double* w_lambda;
  double* w_ni;
  double* w_curchi;
  double* w_inichi;
  double* w_scale_p;
  double* w_red_sum;  // [n_win][4] reduced scalars (chi2, scale_l, n_active_landmarks, spare) — NCCL sum in multi-GPU
  double* w_red_max;  // [n_win]    max |diag Hll| — NCCL max in multi-GPU
  int n_slices;       // CTAs per window in the two-level landmark reductions (large problems / multi-rank)
  double* w_part;     // [n_win][n_slices][4]
  int* n_active_win;  // [1]
  // logs
  int log_stride;
  double* chi2_log;
  double* lambda_log;
  int* trials_log;
  int* iter_done;  // [n_win][2]
  // dense solve scratch (global-memory path) per window
  double* solve_scratch;
  const long long* w_scratch_off;
  // envelope (profile) storage of the reduced camera system for large single problems (global BA):
  // scalar row i holds columns [env_first[i], i] at env_A + env_rowptr[i]
  int env_mode;
  int env_panel_h;            // max number of scalar rows below a pivot block that touch it
  int env_maxlen;             // longest row
  const int* env_first;       // [n]
  const long long* env_rowptr;// [n+1]
  const int* env_blk_last;    // [n/6] last block row whose envelope reaches block column k
  double* env_A;
  BaParams prm;
};

}  // namespace lld
