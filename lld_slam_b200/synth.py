"""Seeded synthetic KITTI-like inputs for the BASELINE.json configs (SURVEY.md §8(d)).

Everything is emitted directly in the flattened layout of include/lldba.h.  Values the reference keeps as
CV_32F (poses, map points, keypoints, info weights) are rounded to float32 before being widened, as
src/Converter.cc:37-47,110-116 does.  Camera and thresholds: Examples/Stereo/KITTI04-12_LBD.yaml.
"""
from __future__ import annotations

import numpy as np

# Examples/Stereo/KITTI04-12_LBD.yaml:8-25
FX = 707.0912
FY = 707.0912
CX = 601.8873
CY = 183.1104
BF = 379.8145
IMG_W = 1241.0
IMG_H = 376.0
TH_DEPTH = 40.0
N_LEVELS = 8
SCALE = 1.2
LINE_PYR = 1.44  # src/LineMatching.cc:27


def f32(x):
    return np.asarray(x, dtype=np.float32)


def inv_level_sigma2():
    """mvInvLevelSigma2 of the ORB pyramid (src/ORBextractor.cc:415-430): float 1 / 1.2^(2 level)"""
    return f32(1.0 / (f32(SCALE) ** (2 * np.arange(N_LEVELS))).astype(np.float32))


def seed_for(config_index: int) -> int:
    return 0x11D51A00 + config_index


def _rot_y(a):
    c, s = np.cos(a), np.sin(a)
    R = np.zeros(a.shape + (3, 3))
    R[..., 0, 0] = c; R[..., 0, 2] = s; R[..., 1, 1] = 1; R[..., 2, 0] = -s; R[..., 2, 2] = c
    return R


def _rodrigues(w):
    """rotation matrices from rotation vectors [...,3]"""
    th = np.linalg.norm(w, axis=-1, keepdims=True)
    th = np.maximum(th, 1e-12)
    k = w / th
    K = np.zeros(w.shape[:-1] + (3, 3))
    K[..., 0, 1] = -k[..., 2]; K[..., 0, 2] = k[..., 1]
    K[..., 1, 0] = k[..., 2]; K[..., 1, 2] = -k[..., 0]
    K[..., 2, 0] = -k[..., 1]; K[..., 2, 1] = k[..., 0]
    s = np.sin(th)[..., None]; c = np.cos(th)[..., None]
    return np.eye(3) + s * K + (1 - c) * (K @ K)


def trajectory(n_kf: int, rng, start: int = 0):
    """KFs 1.0 m apart along +z, yaw 2deg*sin(0.3k), y jitter N(0,2cm).  Returns Rwc [n,3,3], twc [n,3]."""
    k = np.arange(start, start + n_kf, dtype=np.float64)
    yaw = np.deg2rad(2.0) * np.sin(0.3 * k)
    Rwc = _rot_y(yaw)
    twc = np.stack([np.zeros(n_kf), rng.normal(0, 0.02, n_kf), 1.0 * k], axis=1)
    return Rwc, twc


def _tcw(Rwc, twc):
    Rcw = np.swapaxes(Rwc, -1, -2)
    tcw = -(Rcw @ twc[..., None])[..., 0]
    return Rcw, tcw


def _pack_T(Rcw, tcw):
    return np.concatenate([Rcw.reshape(-1, 9), tcw.reshape(-1, 3)], axis=1)


def _csr(counts):
    off = np.zeros(len(counts) + 1, dtype=np.int32)
    np.cumsum(counts, out=off[1:])
    return off


def _project(Rcw, tcw, X):
    Xc = (Rcw @ X[..., None])[..., 0] + tcw
    z = Xc[..., 2]
    u = FX * Xc[..., 0] / z + CX
    v = FY * Xc[..., 1] / z + CY
    return u, v, z, Xc


def make_ba_window(n_kf, n_pt, n_ln, rng, *, mean_track=5.0, track_mode="normal", n_fixed_extra=0,
                   outlier_frac=0.05, gamma=1.0, perturb=True, global_mode=False, kf_start=0):
    """One BA problem (window).  Returns a dict of arrays for a single window (kf indices window-local)."""
    n_all = n_kf + n_fixed_extra
    Rwc, twc = trajectory(n_all, rng, kf_start)
    Rcw, tcw = _tcw(Rwc, twc)
    baseline = np.float32(BF) / np.float32(FX)  # mbf / mK(0,0), float as in the reference

    # ---- points: anchored at a random KF, local box in that KF's camera frame ----
    anchor = rng.integers(0, n_all, n_pt)
    Xl = np.stack([rng.uniform(-15, 15, n_pt), rng.uniform(-2, 3, n_pt), rng.uniform(4, 60, n_pt)], axis=1)
    Xw = (Rwc[anchor] @ Xl[..., None])[..., 0] + twc[anchor]
    if track_mode == "geometric":
        L = np.clip(rng.geometric(1.0 / mean_track, n_pt), 2, 20)
    else:
        L = np.clip(np.rint(rng.normal(mean_track, 1.5, n_pt)), 2, n_all).astype(np.int64)
    Lmax = int(L.max()) if n_pt else 1
    start = anchor - L + 1 + rng.integers(0, 3, n_pt)
    cand = start[:, None] + np.arange(Lmax)[None, :]
    ok = (np.arange(Lmax)[None, :] < L[:, None]) & (cand >= 0) & (cand < n_all)
    candc = np.clip(cand, 0, n_all - 1)
    u, v, z, _ = _project(Rcw[candc], tcw[candc], np.broadcast_to(Xw[:, None, :], candc.shape + (3,)))
    ok &= (z > 0.5) & (u >= 0) & (u < IMG_W) & (v >= 0) & (v < IMG_H)
    # guarantee at least one observation: fall back to the anchor
    none = ~ok.any(axis=1)
    if none.any():
        ok[none, 0] = True
        candc[none, 0] = anchor[none]
        uu, vv, zz, _ = _project(Rcw[anchor[none]], tcw[anchor[none]], Xw[none])
        u[none, 0] = uu; v[none, 0] = vv; z[none, 0] = zz
    cnt = ok.sum(axis=1)
    pt_obs_off = _csr(cnt)
    sel = np.nonzero(ok)
    okf = candc[sel].astype(np.int32)
    ou, ov, oz = u[sel], v[sel], z[sel]
    n_obs = okf.shape[0]
    octave = rng.integers(0, N_LEVELS, n_obs)
    sig = SCALE ** octave
    ou = ou + rng.normal(0, 1, n_obs) * sig
    ov = ov + rng.normal(0, 1, n_obs) * sig
    our = np.where(oz < TH_DEPTH * float(baseline), ou - BF / oz + rng.normal(0, 1, n_obs) * sig, -1.0)
    out_mask = rng.random(n_obs) < outlier_frac
    ou = ou + out_mask * rng.uniform(10, 50, n_obs) * rng.choice([-1.0, 1.0], n_obs)
    # keep uR>=0 semantics: stereo obs must not go negative
    our = np.where((our >= 0) | (our == -1.0), our, 0.0)
    pt_obs_uvr = f32(np.stack([ou, ov, our], axis=1))
    inv_sigma2 = inv_level_sigma2()
    if global_mode:
        # reference quirk (src/Optimizer.cc:407,435): mvInvLevelSigma2[octave*2]; the shim resolves the index,
        # octaves >= 4 would read out of range, so the synthetic GBA keeps octaves in {0..3}
        octave = octave % 4
        pt_obs_info = inv_sigma2[octave * 2]
    else:
        pt_obs_info = inv_sigma2[octave]

    # ---- lines: anchored the same way; minimal (X0, dir) with dir ⟂ X0 in WORLD coordinates ----
    anchor_l = rng.integers(0, n_all, n_ln)
    Pl = np.stack([rng.uniform(-12, 12, n_ln), rng.uniform(-2, 3, n_ln), rng.uniform(5, 40, n_ln)], axis=1)
    Pw = (Rwc[anchor_l] @ Pl[..., None])[..., 0] + twc[anchor_l]
    d = rng.normal(0, 1, (n_ln, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    X0 = Pw - (Pw * d).sum(1, keepdims=True) * d            # closest point of the line to the origin
    small = np.linalg.norm(X0, axis=1) < 1.0                  # keep alpha away from 0
    X0[small] += np.cross(d[small], np.array([0.3, 1.0, 0.2])) * 2.0
    X0 = X0 - (X0 * d).sum(1, keepdims=True) * d
    half = rng.uniform(1, 4, n_ln)
    s_mid = (Pw * d).sum(1)
    E1 = X0 + (s_mid - half)[:, None] * d
    E2 = X0 + (s_mid + half)[:, None] * d
    Ll = np.clip(np.rint(rng.normal(mean_track, 1.5, n_ln)), 3, n_all).astype(np.int64)
    Lmaxl = int(Ll.max()) if n_ln else 1
    startl = anchor_l - Ll + 1 + rng.integers(0, 3, n_ln)
    candl = startl[:, None] + np.arange(Lmaxl)[None, :]
    okl = (np.arange(Lmaxl)[None, :] < Ll[:, None]) & (candl >= 0) & (candl < n_all)
    candlc = np.clip(candl, 0, n_all - 1)
    sh = candlc.shape + (3,)
    u1, v1, z1, _ = _project(Rcw[candlc], tcw[candlc], np.broadcast_to(E1[:, None, :], sh))
    u2, v2, z2, _ = _project(Rcw[candlc], tcw[candlc], np.broadcast_to(E2[:, None, :], sh))
    okl &= (z1 > 1.0) & (z2 > 1.0) & (u1 > -200) & (u1 < IMG_W + 200) & (u2 > -200) & (u2 < IMG_W + 200)
    okl &= (np.hypot(u1 - u2, v1 - v2) > 8.0)
    cntl = okl.sum(axis=1)
    ln_obs_off = _csr(cntl)
    sell = np.nonzero(okl)
    lkf = candlc[sell].astype(np.int32)
    n_lobs = lkf.shape[0]
    lid = sell[0]
    loct = rng.integers(0, 3, n_lobs)

    def _noisy_segment(ua, va, ub, vb, sig):
        tx, ty = ub - ua, vb - va
        ln = np.hypot(tx, ty)
        tx, ty = tx / ln, ty / ln
        nx, ny = -ty, tx
        ja, jb = rng.uniform(-10, 10, n_lobs), rng.uniform(-10, 10, n_lobs)
        ca, cb = rng.normal(0, 1, n_lobs) * sig, rng.normal(0, 1, n_lobs) * sig
        return (ua + ja * tx + ca * nx, va + ja * ty + ca * ny, ub + jb * tx + cb * nx, vb + jb * ty + cb * ny)

    sigl = LINE_PYR ** loct
    la = _noisy_segment(u1[sell], v1[sell], u2[sell], v2[sell], sigl)
    # right image: camera centre shifted by +baseline along camera x  (edge model: K (T.map(X) + (-baseline,0,0)))
    bl = float(baseline)
    Xc1 = (Rcw[lkf] @ E1[lid][..., None])[..., 0] + tcw[lkf]
    Xc2 = (Rcw[lkf] @ E2[lid][..., None])[..., 0] + tcw[lkf]
    ur1 = FX * (Xc1[:, 0] - bl) / Xc1[:, 2] + CX; vr1 = FY * Xc1[:, 1] / Xc1[:, 2] + CY
    ur2 = FX * (Xc2[:, 0] - bl) / Xc2[:, 2] + CX; vr2 = FY * Xc2[:, 1] / Xc2[:, 2] + CY
    ra = _noisy_segment(ur1, vr1, ur2, vr2, sigl)
    has_right = rng.random(n_lobs) < 0.8
    if global_mode:
        has_right[:] = True  # GBA adds both edges unconditionally (src/Optimizer.cc:196)
    lout = rng.random(n_lobs) < outlier_frac
    off = lout * rng.uniform(10, 50, n_lobs)
    left = np.stack([la[0], la[1] + off, la[2], la[3] + off], axis=1)
    right = np.stack([ra[0], ra[1], ra[2], ra[3]], axis=1)
    right[~has_right] = -1.0
    right[has_right, 0] = np.maximum(right[has_right, 0], 0.0)  # xs<0 is the "no right line" marker
    ln_obs_left = f32(left)
    ln_obs_right = f32(right)
    if global_mode:
        ln_obs_info = np.ones((n_lobs, 2))
    else:
        # GetReprojThrPyramid(1.0, octave): repeated multiplication by 1.44, src/LineMatching.cc:239-247
        thr = np.array([1.0, LINE_PYR, LINE_PYR * LINE_PYR])[loct]
        info = (1.0 * gamma * gamma) / (thr * thr)
        ln_obs_info = np.stack([info, info], axis=1)
    ln_obs_stereo = has_right.astype(np.uint8)

    # ---- initial estimates: perturb, then quantise what the reference stores as float ----
    Rcw_i, tcw_i = Rcw.copy(), tcw.copy()
    Xw_i = Xw.copy()
    X0_i, d_i = X0.copy(), d.copy()
    if perturb:
        dr = _rodrigues(rng.normal(0, np.deg2rad(0.5) / np.sqrt(3), (n_all, 3)))
        dt = rng.normal(0, 0.05 / np.sqrt(3), (n_all, 3))
        dr[0] = np.eye(3); dt[0] = 0
        Rcw_i = dr @ Rcw
        tcw_i = (dr @ tcw[..., None])[..., 0] + dt
        depth = np.maximum(Xl[:, 2], 1.0)
        Xw_i = Xw + rng.normal(0, 1, (n_pt, 3)) * (0.05 * depth / 10.0)[:, None]
        rl = _rodrigues(rng.normal(0, np.deg2rad(1.0) / np.sqrt(3), (n_ln, 3)))
        d_i = (rl @ d[..., None])[..., 0]
        P_i = Pw + rng.normal(0, 0.05 / np.sqrt(3), (n_ln, 3))
        X0_i = P_i - (P_i * d_i).sum(1, keepdims=True) * d_i
    kf_Tcw = _pack_T(Rcw_i, tcw_i).astype(np.float32).astype(np.float64)
    pt_xyz = Xw_i.astype(np.float32).astype(np.float64)
    ln_x0_dir = np.concatenate([X0_i, d_i], axis=1)  # MapLine keeps doubles (include/MapLine.h:120)

    kf_fixed = np.zeros(n_all, dtype=np.uint8)
    kf_fixed[0] = 1
    if n_fixed_extra:
        kf_fixed[n_kf:] = 1
    intr = np.array([f32(FX), f32(FY), f32(CX), f32(CY), f32(BF)], dtype=np.float64)
    kf_intr = np.tile(intr, (n_all, 1))
    kf_line_cam = np.tile(np.array([intr[0], intr[2], intr[3], float(baseline)]), (n_all, 1))

    return dict(
        n_kf=n_all, n_pt=n_pt, n_ln=n_ln,
        kf_Tcw=kf_Tcw, kf_fixed=kf_fixed, kf_intr=kf_intr, kf_line_cam=kf_line_cam,
        pt_xyz=pt_xyz, pt_obs_off=pt_obs_off, pt_obs_kf=okf, pt_obs_uvr=pt_obs_uvr, pt_obs_info=f32(pt_obs_info),
        ln_x0_dir=ln_x0_dir, ln_obs_off=ln_obs_off, ln_obs_kf=lkf, ln_obs_left=ln_obs_left, ln_obs_right=ln_obs_right,
        ln_obs_info=np.ascontiguousarray(ln_obs_info, dtype=np.float64), ln_obs_stereo=ln_obs_stereo,
        truth=dict(kf_Tcw=_pack_T(Rcw, tcw), pt_xyz=Xw, ln_x0_dir=np.concatenate([X0, d], axis=1)),
    )


def ba_constants(mode: str, gamma: float = 1.0, robust_points: bool = True):
    """Entry-point constants (SURVEY.md A.6)."""
    if mode == "local":  # src/Optimizer.cc:1088-1089,1180-1182 ; src/LineOptimizer.cc:33-36
        d_mono = float(np.float32(np.sqrt(5.991)))
        d_stereo = float(np.float32(np.sqrt(7.815)))
        return dict(robust_points=1, delta_pt_mono=d_mono, delta_pt_stereo=d_stereo,
                    delta_ln_mono=d_mono * gamma, delta_ln_stereo=d_stereo * gamma,
                    chi2_pt_mono=5.991, chi2_pt_stereo=7.815, ln_endpoints_normalized=0, ln_filter=4)
    if mode == "global":  # src/Optimizer.cc:359-361
        d2 = float(np.float32(np.sqrt(5.99)))
        d3 = float(np.float32(np.sqrt(7.815)))
        dl = float(np.float32(np.sqrt(7.815))) / 2.0
        return dict(robust_points=int(robust_points), delta_pt_mono=d2, delta_pt_stereo=d3,
                    delta_ln_mono=dl, delta_ln_stereo=dl,
                    chi2_pt_mono=5.991, chi2_pt_stereo=7.815, ln_endpoints_normalized=1, ln_filter=4)
    raise ValueError(mode)


_BA_CAT = ["kf_Tcw", "kf_fixed", "kf_intr", "kf_line_cam", "pt_xyz", "pt_obs_kf", "pt_obs_uvr", "pt_obs_info",
           "ln_x0_dir", "ln_obs_kf", "ln_obs_left", "ln_obs_right", "ln_obs_info", "ln_obs_stereo"]


def batch_ba(windows, mode="local", gamma=1.0, robust_points=True):
    """Concatenate single-window dicts into one batched lld_ba_problem field dict."""
    out = {k: np.ascontiguousarray(np.concatenate([w[k] for w in windows], axis=0)) for k in _BA_CAT}
    out["n_win"] = len(windows)
    out["kf_off"] = _csr([w["n_kf"] for w in windows])
    out["pt_off"] = _csr([w["n_pt"] for w in windows])
    out["ln_off"] = _csr([w["n_ln"] for w in windows])
    po, lo = [np.zeros(1, np.int32)], [np.zeros(1, np.int32)]
    pb = lb = 0
    for w in windows:
        po.append(w["pt_obs_off"][1:] + pb); pb += int(w["pt_obs_off"][-1])
        lo.append(w["ln_obs_off"][1:] + lb); lb += int(w["ln_obs_off"][-1])
    out["pt_obs_off"] = np.concatenate(po).astype(np.int32)
    out["ln_obs_off"] = np.concatenate(lo).astype(np.int32)
    out.update(ba_constants(mode, gamma, robust_points))
    return out


def make_local_ba_batch(n_win, n_kf, n_pt, n_ln, seed, **kw):
    rng = np.random.default_rng(seed)
    return batch_ba([make_ba_window(n_kf, n_pt, n_ln, rng, **kw) for _ in range(n_win)], "local", kw.get("gamma", 1.0))


def make_global_ba(n_kf, n_pt, n_ln, seed, robust_points=False, **kw):
    rng = np.random.default_rng(seed)
    w = make_ba_window(n_kf, n_pt, n_ln, rng, mean_track=6.0, track_mode="geometric", global_mode=True, **kw)
    return batch_ba([w], "global", 1.0, robust_points)


def shard_ba_landmarks(p, rank, n_ranks):
    """Block-partition the landmarks (points and lines) of a single-window problem over ranks; KFs replicated."""
    assert p["n_win"] == 1
    out = dict(p)
    n_pt, n_ln = int(p["pt_off"][1]), int(p["ln_off"][1])

    def rng_(n):
        return (n * rank) // n_ranks, (n * (rank + 1)) // n_ranks

    a, b = rng_(n_pt)
    e0, e1 = int(p["pt_obs_off"][a]), int(p["pt_obs_off"][b])
    out["pt_xyz"] = np.ascontiguousarray(p["pt_xyz"][a:b])
    out["pt_obs_off"] = np.ascontiguousarray(p["pt_obs_off"][a:b + 1] - e0).astype(np.int32)
    for k in ("pt_obs_kf", "pt_obs_uvr", "pt_obs_info"):
        out[k] = np.ascontiguousarray(p[k][e0:e1])
    out["pt_off"] = np.array([0, b - a], np.int32)
    a, b = rng_(n_ln)
    e0, e1 = int(p["ln_obs_off"][a]), int(p["ln_obs_off"][b])
    out["ln_x0_dir"] = np.ascontiguousarray(p["ln_x0_dir"][a:b])
    out["ln_obs_off"] = np.ascontiguousarray(p["ln_obs_off"][a:b + 1] - e0).astype(np.int32)
    for k in ("ln_obs_kf", "ln_obs_left", "ln_obs_right", "ln_obs_info", "ln_obs_stereo"):
        out[k] = np.ascontiguousarray(p[k][e0:e1])
    out["ln_off"] = np.array([0, b - a], np.int32)
    return out


# ---------------------------------------------------------------------------------------------
# PoseOptimization batch (cfg 3)
# ---------------------------------------------------------------------------------------------
def make_pose_batch(n_frames, n_pt, n_ln, seed, gamma=0.5, outlier_frac=0.08, stereo_frac=0.7, right_frac=0.8):
    rng = np.random.default_rng(seed)
    baseline = float(np.float32(BF) / np.float32(FX))
    F = n_frames
    yaw = rng.normal(0, np.deg2rad(3), F)
    Rwc = _rot_y(yaw)
    twc = np.stack([rng.normal(0, 0.3, F), rng.normal(0, 0.05, F), rng.uniform(0, 100, F)], axis=1)
    Rcw, tcw = _tcw(Rwc, twc)
    # points in the camera frame, visible by construction
    z = rng.uniform(4, 60, (F, n_pt))
    u = rng.uniform(20, IMG_W - 20, (F, n_pt))
    v = rng.uniform(20, IMG_H - 20, (F, n_pt))
    Xc = np.stack([(u - CX) / FX * z, (v - CY) / FY * z, z], axis=-1)
    Xw = (Rwc[:, None] @ Xc[..., None])[..., 0] + twc[:, None]
    octv = rng.integers(0, N_LEVELS, (F, n_pt))
    sig = SCALE ** octv
    un = u + rng.normal(0, 1, u.shape) * sig
    vn = v + rng.normal(0, 1, u.shape) * sig
    stereo = rng.random((F, n_pt)) < stereo_frac
    ur = np.where(stereo, un - BF / z + rng.normal(0, 1, u.shape) * sig, -1.0)
    ur = np.where(stereo, np.maximum(ur, 0.0), -1.0)
    outl = rng.random((F, n_pt)) < outlier_frac
    un = un + outl * rng.uniform(10, 50, u.shape) * rng.choice([-1.0, 1.0], u.shape)
    inv_sigma2 = inv_level_sigma2()
    # lines
    P = np.stack([rng.uniform(-12, 12, (F, n_ln)), rng.uniform(-2, 3, (F, n_ln)), rng.uniform(5, 40, (F, n_ln))], axis=-1)
    dc = rng.normal(0, 1, (F, n_ln, 3))
    dc /= np.linalg.norm(dc, axis=-1, keepdims=True)
    half = rng.uniform(1, 4, (F, n_ln))
    E1c = P - half[..., None] * dc
    E2c = P + half[..., None] * dc
    E1c[..., 2] = np.maximum(E1c[..., 2], 1.5); E2c[..., 2] = np.maximum(E2c[..., 2], 1.5)
    dc = E2c - E1c
    dc /= np.linalg.norm(dc, axis=-1, keepdims=True)
    Pw = (Rwc[:, None] @ E1c[..., None])[..., 0] + twc[:, None]
    dw = (Rwc[:, None] @ dc[..., None])[..., 0]
    X0 = Pw - (Pw * dw).sum(-1, keepdims=True) * dw
    loct = rng.integers(0, 3, (F, n_ln))
    sl = LINE_PYR ** loct

    def seg(E1, E2, shift):
        a = np.stack([FX * (E1[..., 0] - shift) / E1[..., 2] + CX, FY * E1[..., 1] / E1[..., 2] + CY], -1)
        b = np.stack([FX * (E2[..., 0] - shift) / E2[..., 2] + CX, FY * E2[..., 1] / E2[..., 2] + CY], -1)
        t = b - a
        t /= np.maximum(np.linalg.norm(t, axis=-1, keepdims=True), 1e-9)
        n = np.stack([-t[..., 1], t[..., 0]], -1)
        a = a + rng.uniform(-10, 10, a.shape[:-1])[..., None] * t + (rng.normal(0, 1, a.shape[:-1]) * sl)[..., None] * n
        b = b + rng.uniform(-10, 10, a.shape[:-1])[..., None] * t + (rng.normal(0, 1, a.shape[:-1]) * sl)[..., None] * n
        return np.concatenate([a, b], -1)

    left = seg(E1c, E2c, 0.0)
    right = seg(E1c, E2c, baseline)
    has_r = rng.random((F, n_ln)) < right_frac
    lout = rng.random((F, n_ln)) < outlier_frac
    left[..., 1] += lout * rng.uniform(10, 50, lout.shape)
    left[..., 3] += lout * rng.uniform(10, 50, lout.shape)
    right[~has_r] = -1.0
    right[..., 0] = np.where(has_r, np.maximum(right[..., 0], 0.0), -1.0)
    thr = np.array([1.0, LINE_PYR, LINE_PYR * LINE_PYR])[loct]
    info = (1.0 * gamma * gamma) / (thr * thr)
    # initial pose: truth perturbed (motion-model error), float-quantised
    dr = _rodrigues(rng.normal(0, np.deg2rad(1.0) / np.sqrt(3), (F, 3)))
    dt = rng.normal(0, 0.10 / np.sqrt(3), (F, 3))
    Ri = dr @ Rcw
    ti = (dr @ tcw[..., None])[..., 0] + dt
    intr = np.array([f32(FX), f32(FY), f32(CX), f32(CY), f32(BF)], dtype=np.float64)
    d_mono = np.float32(np.sqrt(5.991)); d_stereo = np.float32(np.sqrt(7.815))
    dls = np.float32(np.float64(d_stereo) * gamma); dlm = np.float32(np.float64(d_mono) * gamma)
    st = has_r.reshape(-1).astype(np.uint8)
    return dict(
        n_frames=F,
        Tcw=_pack_T(Ri, ti).astype(np.float32).astype(np.float64),
        intr=np.tile(intr, (F, 1)),
        line_cam=np.tile(np.array([intr[0], intr[2], intr[3], baseline]), (F, 1)),
        pt_off=(np.arange(F + 1) * n_pt).astype(np.int32),
        pt_xw=f32(Xw.reshape(-1, 3)), pt_uvr=f32(np.stack([un, vn, ur], -1).reshape(-1, 3)),
        pt_info=np.ascontiguousarray(inv_sigma2[octv.reshape(-1)]),
        ln_off=(np.arange(F + 1) * n_ln).astype(np.int32),
        ln_x0_dir=np.ascontiguousarray(np.concatenate([X0, dw], -1).reshape(-1, 6)),
        ln_left=f32(left.reshape(-1, 4)), ln_right=f32(right.reshape(-1, 4)),
        ln_info=np.ascontiguousarray(np.stack([info, info], -1).reshape(-1, 2)),
        ln_stereo=st, ln_gate_stereo=np.ascontiguousarray(np.stack([st, st], -1)),
        delta_mono=float(d_mono), delta_stereo=float(d_stereo),
        delta_ln_mono=float(dlm), delta_ln_stereo=float(dls),
        chi2_mono=float(np.float32(5.991)), chi2_stereo=float(np.float32(7.815)),
        gate_ln_mono=float(np.float32(dlm * dlm)), gate_ln_stereo=float(np.float32(dls * dls)),
        n_rounds=4, its=10,
        truth=dict(Tcw=_pack_T(Rcw, tcw)),
    )


# ---------------------------------------------------------------------------------------------
# Stereo frame-pair matching (cfg 2): ORB SearchByProjection + float line descriptors
# ---------------------------------------------------------------------------------------------
def frame_geom():
    sf = f32(f32(SCALE) ** np.arange(N_LEVELS))
    return dict(fx=float(f32(FX)), fy=float(f32(FY)), cx=float(f32(CX)), cy=float(f32(CY)), bf=float(f32(BF)),
                b=float(np.float32(BF) / np.float32(FX)), min_x=0.0, max_x=IMG_W, min_y=0.0, max_y=IMG_H,
                scale_factors=sf)


def _flip_bits(desc, p, rng):
    bits = np.unpackbits(desc, axis=-1)
    flip = rng.random(bits.shape) < p
    return np.packbits(bits ^ flip.astype(np.uint8), axis=-1)


def make_sbp_frame_batch(n_pairs, n_kp, seed, th=7.0, unrelated_frac=0.3, flip_p=0.08):
    rng = np.random.default_rng(seed)
    P, N = n_pairs, n_kp
    baseline = float(np.float32(BF) / np.float32(FX))
    # last frame at identity-ish pose, current frame moved ~1 m forward with small rotation
    yaw_l = rng.normal(0, np.deg2rad(1), P)
    Rwl = _rot_y(yaw_l); twl = np.stack([rng.normal(0, 0.1, P), rng.normal(0, 0.02, P), rng.uniform(0, 50, P)], 1)
    fwd = rng.choice([1.0, 1.0, 1.0, -1.0, 0.2], P)  # forward / backward / nearly static -> all three level modes
    yaw_c = yaw_l + rng.normal(0, np.deg2rad(1), P)
    Rwc = _rot_y(yaw_c); twc = twl + np.stack([rng.normal(0, 0.05, P), rng.normal(0, 0.02, P), fwd * rng.uniform(0.6, 1.2, P)], 1)
    Rlw, tlw = _tcw(Rwl, twl)
    Rcw, tcw = _tcw(Rwc, twc)
    # last-frame keypoints with map points
    ul = rng.uniform(10, IMG_W - 10, (P, N)); vl = rng.uniform(10, IMG_H - 10, (P, N)); zl = rng.uniform(4, 60, (P, N))
    Xl = np.stack([(ul - CX) / FX * zl, (vl - CY) / FY * zl, zl], -1)
    Xw = (Rwl[:, None] @ Xl[..., None])[..., 0] + twl[:, None]
    Xw32 = f32(Xw)
    last_oct = rng.integers(0, N_LEVELS, (P, N)).astype(np.uint8)
    last_ang = f32(rng.uniform(0, 360, (P, N)))
    last_desc = rng.integers(0, 256, (P, N, 32), dtype=np.uint8)
    last_valid = (rng.random((P, N)) < 0.9).astype(np.uint8)
    last_has_obs = (rng.random((P, N)) < 0.95).astype(np.uint8)
    # current frame: related keypoints = projections + N(0,3px); unrelated = random
    uc, vc, zc, _ = _project(Rcw[:, None], tcw[:, None], Xw32.astype(np.float64))
    related = rng.random((P, N)) >= unrelated_frac
    cu = np.where(related, uc + rng.normal(0, 3, uc.shape), rng.uniform(0, IMG_W, uc.shape))
    cv_ = np.where(related, vc + rng.normal(0, 3, uc.shape), rng.uniform(0, IMG_H, uc.shape))
    cur_desc = np.where(related[..., None], _flip_bits(last_desc, flip_p, rng), rng.integers(0, 256, (P, N, 32), dtype=np.uint8)).astype(np.uint8)
    doct = rng.choice([0, 0, 0, 1, -1], (P, N))
    cur_oct = np.clip(last_oct.astype(np.int64) + doct, 0, N_LEVELS - 1).astype(np.uint8)
    cur_ang = f32(np.mod(np.where(related & (rng.random((P, N)) < 0.9), last_ang + rng.normal(5, 3, (P, N)), rng.uniform(0, 360, (P, N))), 360.0))
    zc_safe = np.where(zc > 0.5, zc, 10.0)
    cur_ur = np.where(rng.random((P, N)) < 0.7, cu - BF / zc_safe + rng.normal(0, 2, uc.shape), -1.0)
    # shuffle the current keypoints so indices do not line up with the last frame
    perm = np.argsort(rng.random((P, N)), axis=1)
    take = lambda a: np.take_along_axis(a, perm if a.ndim == 2 else perm[..., None], axis=1)
    cu, cv_, cur_oct, cur_ang, cur_ur, cur_desc = take(cu), take(cv_), take(cur_oct), take(cur_ang), take(cur_ur), take(cur_desc)
    cur_claimed = (rng.random((P, N)) < 0.03).astype(np.uint8)
    g = frame_geom()
    return dict(
        n_pairs=P, geom=g, th=float(th), mono=0, check_orientation=1,
        cur_off=(np.arange(P + 1) * N).astype(np.int32),
        cur_xy=f32(np.stack([cu, cv_], -1).reshape(-1, 2)), cur_octave=np.ascontiguousarray(cur_oct.reshape(-1)),
        cur_angle=np.ascontiguousarray(cur_ang.reshape(-1)), cur_uright=f32(cur_ur.reshape(-1)),
        cur_desc=np.ascontiguousarray(cur_desc.reshape(-1, 32)), cur_claimed=np.ascontiguousarray(cur_claimed.reshape(-1)),
        cur_Tcw=f32(_pack_T(Rcw, tcw)), last_Tcw=f32(_pack_T(Rlw, tlw)),
        last_off=(np.arange(P + 1) * N).astype(np.int32),
        last_valid=np.ascontiguousarray(last_valid.reshape(-1)), last_xw=np.ascontiguousarray(Xw32.reshape(-1, 3)),
        last_octave=np.ascontiguousarray(last_oct.reshape(-1)), last_angle=np.ascontiguousarray(last_ang.reshape(-1)),
        last_desc=np.ascontiguousarray(last_desc.reshape(-1, 32)), last_has_obs=np.ascontiguousarray(last_has_obs.reshape(-1)),
    )


def concat_sbp_frame(parts):
    """concatenate frame-pair batches of different sizes into one ragged batch (same geometry / thresholds)"""
    out = dict(parts[0])
    out["n_pairs"] = int(sum(p["n_pairs"] for p in parts))
    for off_key, keys in (("cur_off", ("cur_xy", "cur_octave", "cur_angle", "cur_uright", "cur_desc", "cur_claimed")),
                          ("last_off", ("last_valid", "last_xw", "last_octave", "last_angle", "last_desc", "last_has_obs"))):
        offs, base = [np.zeros(1, np.int32)], 0
        for p in parts:
            offs.append((p[off_key][1:] + base).astype(np.int32))
            base += int(p[off_key][-1])
        out[off_key] = np.concatenate(offs)
        for k in keys:
            out[k] = np.ascontiguousarray(np.concatenate([p[k] for p in parts], 0))
    for k in ("cur_Tcw", "last_Tcw"):
        out[k] = np.ascontiguousarray(np.concatenate([p[k] for p in parts], 0))
    return out


def make_sbp_mp_batch(n_pairs, n_kp, n_mp, seed, th=3.0, nn_ratio=0.8):
    """SearchByProjection(F, local map points): map points pre-projected (isInFrustum fields)."""
    rng = np.random.default_rng(seed)
    P, N, M = n_pairs, n_kp, n_mp
    cu = rng.uniform(0, IMG_W, (P, N)); cv_ = rng.uniform(0, IMG_H, (P, N))
    cur_oct = rng.integers(0, N_LEVELS, (P, N)).astype(np.uint8)
    cur_desc = rng.integers(0, 256, (P, N, 32), dtype=np.uint8)
    cur_ur = np.where(rng.random((P, N)) < 0.7, cu - rng.uniform(5, 90, (P, N)), -1.0)
    # each map point is tied to a random keypoint (70 %) or unrelated
    src = rng.integers(0, N, (P, M))
    rel = rng.random((P, M)) < 0.7
    g_u = np.take_along_axis(cu, src, 1); g_v = np.take_along_axis(cv_, src, 1)
    g_ur = np.take_along_axis(cur_ur, src, 1); g_oct = np.take_along_axis(cur_oct, src, 1)
    g_desc = np.take_along_axis(cur_desc, src[..., None], 1)
    pu = np.where(rel, g_u + rng.normal(0, 2, (P, M)), rng.uniform(0, IMG_W, (P, M)))
    pv = np.where(rel, g_v + rng.normal(0, 2, (P, M)), rng.uniform(0, IMG_H, (P, M)))
    pur = np.where(rel & (g_ur > 0), g_ur + rng.normal(0, 2, (P, M)), pu - rng.uniform(5, 90, (P, M)))
    lvl = np.clip(g_oct.astype(np.int64) + rng.choice([0, 0, 1], (P, M)), 0, N_LEVELS - 1).astype(np.int32)
    mp_desc = np.where(rel[..., None], _flip_bits(g_desc, 0.1, rng), rng.integers(0, 256, (P, M, 32), dtype=np.uint8)).astype(np.uint8)
    g = frame_geom()
    return dict(
        n_pairs=P, geom=g, th=float(th), nn_ratio=float(nn_ratio),
        cur_off=(np.arange(P + 1) * N).astype(np.int32),
        cur_xy=f32(np.stack([cu, cv_], -1).reshape(-1, 2)), cur_octave=np.ascontiguousarray(cur_oct.reshape(-1)),
        cur_uright=f32(cur_ur.reshape(-1)), cur_desc=np.ascontiguousarray(cur_desc.reshape(-1, 32)),
        cur_claimed=np.ascontiguousarray((rng.random((P, N)) < 0.05).astype(np.uint8).reshape(-1)),
        mp_off=(np.arange(P + 1) * M).astype(np.int32),
        mp_valid=np.ascontiguousarray((rng.random((P, M)) < 0.9).astype(np.uint8).reshape(-1)),
        mp_proj=f32(np.stack([pu, pv, pur], -1).reshape(-1, 3)), mp_level=np.ascontiguousarray(lvl.reshape(-1)),
        mp_viewcos=f32(rng.uniform(0.99, 1.0, (P, M)).reshape(-1)), mp_desc=np.ascontiguousarray(mp_desc.reshape(-1, 32)),
        mp_has_obs=np.ascontiguousarray((rng.random((P, M)) < 0.95).astype(np.uint8).reshape(-1)),
    )


def make_kf_search_batch(n_pairs, n_kp, n_mp, seed, th=3.0, th_low=50, chi2_gate=1, sequential_claims=0):
    """Fuse / SearchByProjection(KeyFrame*, Scw, ...): map points already projected into the keyframes (u, v, ur, predicted level);
    most of them sit within a few pixels of a keypoint whose descriptor they share up to a few bits, so that the reprojection gate
    and TH_LOW both cut; several points per keypoint, so that the sequential claims matter"""
    m = make_sbp_mp_batch(n_pairs, n_kp, n_mp, seed, th=th)
    rng = np.random.default_rng(seed + 17)
    ur = m["cur_uright"].copy()
    ur[ur < 0] = -1.0
    return dict(
        n_pairs=n_pairs, geom=m["geom"], th=float(th), th_low=int(th_low), chi2_gate=int(chi2_gate), sequential_claims=int(sequential_claims),
        inv_level_sigma2=np.pad(inv_level_sigma2(), (0, max(0, 8 - N_LEVELS)))[:8],
        kp_off=m["cur_off"], kp_xy=m["cur_xy"], kp_octave=m["cur_octave"], kp_uright=ur, kp_desc=m["cur_desc"],
        kp_claimed=m["cur_claimed"] if sequential_claims else np.zeros_like(m["cur_claimed"]),
        mp_off=m["mp_off"], mp_valid=m["mp_valid"], mp_proj=m["mp_proj"], mp_level=m["mp_level"], mp_desc=m["mp_desc"],
    )


def make_tri_search_batch(n_pairs, n_kp, seed, n_nodes=300, only_stereo=0, check_orientation=1):
    """SearchForTriangulation: two keyframes a small baseline apart looking at the same random 3D points; a keypoint and its
    counterpart share a vocabulary node (most of the time) and a descriptor up to a few bits; F12 from the relative pose;
    30 % of the keypoints already carry a map point, 60 % have a right coordinate."""
    rng = np.random.default_rng(seed)
    g = frame_geom()
    K = np.array([[g["fx"], 0, g["cx"]], [0, g["fy"], g["cy"]], [0, 0, 1.0]])
    Ki = np.linalg.inv(K)
    sf = np.asarray(g["scale_factors"], np.float32)
    nl = len(sf)
    out = dict(n_pairs=n_pairs, only_stereo=int(only_stereo), check_orientation=int(check_orientation), n_levels=nl,
               scale_factors=np.pad(sf, (0, 8 - nl)), level_sigma2=np.pad((sf * sf).astype(np.float32), (0, 8 - nl)))
    F12s, epis = [], []
    acc = {k: [] for k in ("kp1_xy", "kp1_angle", "kp1_uright", "kp1_has_mp", "kp1_desc", "kp2_xy", "kp2_octave", "kp2_angle", "kp2_uright",
                           "kp2_has_mp", "kp2_desc", "fv1_node", "fv1_idx", "fv2_node", "fv2_idx")}
    kp1_off, kp2_off, n1o, n2o = [0], [0], [0], [0]

    def fv(nodes):
        order = np.argsort(nodes, kind="stable")          # DBoW2 pushes the indices of a node in keypoint order
        ids, cnt = np.unique(nodes, return_counts=True)
        return ids.astype(np.int32), np.cumsum(cnt), order.astype(np.int32)

    for pr in range(n_pairs):
        N = int(n_kp[pr]) if np.ndim(n_kp) else n_kp          # a list gives ragged pairs (0 = a pair without keypoints)
        X = np.stack([rng.uniform(-10, 10, N), rng.uniform(-3, 3, N), rng.uniform(5, 40, N)], 1)
        yaw = rng.normal(0, 0.03)
        R21 = _rot_y(np.array(yaw))                          # camera 1 -> camera 2
        t21 = np.array([rng.uniform(0.5, 1.5), rng.normal(0, 0.05), rng.normal(0, 0.2)])
        X2 = (R21 @ X.T).T + t21

        def proj(Xc):
            return np.stack([g["fx"] * Xc[:, 0] / Xc[:, 2] + g["cx"], g["fy"] * Xc[:, 1] / Xc[:, 2] + g["cy"]], 1)
        p1 = proj(X) + rng.normal(0, 0.4, (N, 2))
        p2 = proj(X2) + rng.normal(0, 0.4, (N, 2))
        unrel = rng.random(N) < 0.15
        p2[unrel] = np.stack([rng.uniform(0, IMG_W, unrel.sum()), rng.uniform(0, IMG_H, unrel.sum())], 1).reshape(-1, 2)
        perm = rng.permutation(N)                            # keyframe 2 stores its keypoints in another order
        tx = np.array([[0, -t21[2], t21[1]], [t21[2], 0, -t21[0]], [-t21[1], t21[0], 0]])
        F12 = (Ki.T @ (tx @ R21).T @ Ki)                     # x1' F12 x2 = 0
        F12s.append(F12.reshape(-1))
        C2 = t21                                             # camera centre of keyframe 1 in camera 2
        epis.append([g["fx"] * C2[0] / C2[2] + g["cx"], g["fy"] * C2[1] / C2[2] + g["cy"]])
        d1 = rng.integers(0, 256, (N, 32), dtype=np.uint8)
        d2 = (np.where(unrel[:, None], rng.integers(0, 256, (N, 32), dtype=np.uint8), _flip_bits(d1[None], 0.06, rng)[0]).astype(np.uint8)
              if N else d1.copy())
        node1 = rng.integers(0, n_nodes, N)
        node2 = np.where(rng.random(N) < 0.9, node1, rng.integers(0, n_nodes, N))
        ang1 = rng.uniform(0, 360, N); ang2 = (ang1 + rng.normal(3, 4, N) + np.where(rng.random(N) < 0.1, rng.uniform(0, 360, N), 0)) % 360
        ur1 = np.where(rng.random(N) < 0.6, p1[:, 0] - g["bf"] / X[:, 2], -1.0)
        ur2 = np.where(rng.random(N) < 0.6, p2[:, 0] - g["bf"] / np.maximum(X2[:, 2], 1.0), -1.0)
        acc["kp1_xy"].append(p1); acc["kp1_angle"].append(ang1); acc["kp1_uright"].append(ur1)
        acc["kp1_has_mp"].append(rng.random(N) < 0.3); acc["kp1_desc"].append(d1)
        acc["kp2_xy"].append(p2[perm]); acc["kp2_octave"].append(rng.integers(0, nl, N)); acc["kp2_angle"].append(ang2[perm])
        acc["kp2_uright"].append(ur2[perm]); acc["kp2_has_mp"].append(rng.random(N) < 0.3); acc["kp2_desc"].append(d2[perm])
        ids, ends, order = fv(node1)
        acc["fv1_node"].append(ids); acc["fv1_idx"].append(order); n1o.append(n1o[-1] + len(ids))
        f1_ends = ends
        ids2, ends2, order2 = fv(node2[perm])
        acc["fv2_node"].append(ids2); acc["fv2_idx"].append(order2); n2o.append(n2o[-1] + len(ids2))
        out.setdefault("_e1", []).append(f1_ends); out.setdefault("_e2", []).append(ends2)
        kp1_off.append(kp1_off[-1] + N); kp2_off.append(kp2_off[-1] + N)
    # global CSR of the feature-vector entries
    def idx_off(ends_list):
        off, base = [0], 0
        for e in ends_list:
            off += list(base + e); base += int(e[-1]) if len(e) else 0
        return np.asarray(off, np.int32)
    out["fv1_idx_off"] = idx_off(out.pop("_e1")); out["fv2_idx_off"] = idx_off(out.pop("_e2"))
    out["F12"] = f32(np.stack(F12s)); out["epipole"] = f32(np.asarray(epis))
    out["kp1_off"] = np.asarray(kp1_off, np.int32); out["kp2_off"] = np.asarray(kp2_off, np.int32)
    out["fv1_node_off"] = np.asarray(n1o, np.int32); out["fv2_node_off"] = np.asarray(n2o, np.int32)
    for k, v in acc.items():
        a = np.concatenate(v)
        if k.endswith("_xy") or k.endswith("_angle") or k.endswith("_uright"):
            a = f32(a)
        elif k.endswith("_has_mp") or k.endswith("_octave") or k.endswith("_desc"):
            a = a.astype(np.uint8)
        else:
            a = a.astype(np.int32)
        out[k] = np.ascontiguousarray(a)
    return out


def make_bow_search_batch(n_pairs, n_kp, seed, n_nodes=150, strict_th=0, nn_ratio=0.7, check_orientation=1):
    """SearchByBoW: the keyframe pairs of make_tri_search_batch with fewer vocabulary nodes (larger buckets, so that second-best
    distances, the ratio test and the claims inside a bucket all matter); side 1 keypoints carry a good map point with
    probability 0.7, side 2 keypoints are all valid (frame) or carry one with probability 0.8 (keyframe, strict_th)"""
    t = make_tri_search_batch(n_pairs, n_kp, seed, n_nodes=n_nodes)
    rng = np.random.default_rng(seed + 5)
    n1, n2 = int(t["kp1_off"][-1]), int(t["kp2_off"][-1])
    out = dict(n_pairs=n_pairs, strict_th=int(strict_th), check_orientation=int(check_orientation), nn_ratio=float(nn_ratio),
               kp1_off=t["kp1_off"], kp1_angle=t["kp1_angle"], kp1_valid=(rng.random(n1) < 0.7).astype(np.uint8), kp1_desc=t["kp1_desc"],
               kp2_off=t["kp2_off"], kp2_angle=t["kp2_angle"],
               kp2_valid=(rng.random(n2) < 0.8).astype(np.uint8) if strict_th else np.ones(n2, np.uint8), kp2_desc=t["kp2_desc"])
    for k in ("fv1_node_off", "fv1_node", "fv1_idx_off", "fv1_idx", "fv2_node_off", "fv2_node", "fv2_idx_off", "fv2_idx"):
        out[k] = t[k]
    return out


def make_init_search_batch(n_pairs, n_kp, seed, window_size=100, nn_ratio=0.9, check_orientation=1, n_kp2=None, flow=20.0,
                           unrelated_frac=0.3, flip_p=0.06, rotated_frac=0.15, dup_frac=0.05):
    """SearchForInitialization (Tracking::MonocularInitialization): F1 = the initial frame, vbPrevMatched = its keypoints; F2 = F1
    moved by a per-pair flow (up to `flow` px) plus 1.5 px noise, shuffled, with a share of unrelated keypoints mixed in.
    Related descriptors differ by a few bit flips; angles follow F1 up to a small rotation except for a share of rotated
    outliers, which the histogram filter removes.  A share of F1 keypoints repeats another one's texture nearby, so that later
    queries take F2 keypoints away from earlier ones.  n_kp / n_kp2 may be lists (ragged pairs, 0 allowed); n_kp2 defaults to n_kp."""
    rng = np.random.default_rng(seed)
    g = frame_geom()
    lvl_p = np.asarray([SCALE ** (-2.0 * l) for l in range(N_LEVELS)]); lvl_p /= lvl_p.sum()   # ORB's per-level feature share
    acc = {k: [] for k in ("kp1_octave", "kp1_angle", "kp1_desc", "prev_matched", "kp2_xy", "kp2_octave", "kp2_angle", "kp2_desc")}
    kp1_off, kp2_off = [0], [0]
    for pr in range(n_pairs):
        N1 = int(n_kp[pr]) if np.ndim(n_kp) else int(n_kp)
        N2 = N1 if n_kp2 is None else (int(n_kp2[pr]) if np.ndim(n_kp2) else int(n_kp2))
        xy1 = np.stack([rng.uniform(0, IMG_W, N1), rng.uniform(0, IMG_H, N1)], 1)
        oct1 = rng.choice(N_LEVELS, N1, p=lvl_p)
        ang1 = rng.uniform(0, 360, N1)
        d1 = rng.integers(0, 256, (N1, 32), dtype=np.uint8)
        # repeated texture: near-duplicate level-0 F1 keypoints a few pixels apart compete for the same F2 keypoint
        n_dup = int(N1 * dup_frac) if N1 >= 2 else 0
        dst, srcd = rng.choice(N1, n_dup, replace=False), rng.integers(0, N1, n_dup)
        ok = dst != srcd
        dst, srcd = dst[ok], srcd[ok]
        d1[dst] = _flip_bits(d1[srcd], flip_p, rng)
        xy1[dst] = np.clip(xy1[srcd] + rng.normal(0, 10, (len(dst), 2)), 0, [IMG_W - 1e-3, IMG_H - 1e-3])
        oct1[dst] = 0; oct1[srcd] = 0
        # F2: the first min(N1, N2) * (1 - unrelated_frac) keypoints follow F1, the rest are unrelated
        n_rel = int(min(N1, N2) * (1.0 - unrelated_frac))
        src = rng.permutation(N1)[:n_rel]
        f = rng.uniform(-flow, flow, 2)
        xy2 = np.concatenate([xy1[src] + f + rng.normal(0, 1.5, (n_rel, 2)),
                              np.stack([rng.uniform(0, IMG_W, N2 - n_rel), rng.uniform(0, IMG_H, N2 - n_rel)], 1)])
        oct2 = np.concatenate([np.where(rng.random(n_rel) < 0.9, oct1[src], rng.choice(N_LEVELS, n_rel, p=lvl_p)),
                               rng.choice(N_LEVELS, N2 - n_rel, p=lvl_p)])
        rot = np.where(rng.random(n_rel) < rotated_frac, rng.uniform(0, 360, n_rel), rng.normal(4, 3, n_rel))
        ang2 = np.concatenate([np.mod(ang1[src] + rot, 360.0), rng.uniform(0, 360, N2 - n_rel)])
        d2 = np.concatenate([_flip_bits(d1[src], flip_p, rng) if n_rel else d1[:0],
                             rng.integers(0, 256, (N2 - n_rel, 32), dtype=np.uint8)])
        perm = rng.permutation(N2)
        acc["kp1_octave"].append(oct1); acc["kp1_angle"].append(ang1); acc["kp1_desc"].append(d1); acc["prev_matched"].append(xy1)
        acc["kp2_xy"].append(xy2[perm]); acc["kp2_octave"].append(oct2[perm]); acc["kp2_angle"].append(ang2[perm])
        acc["kp2_desc"].append(d2[perm])
        kp1_off.append(kp1_off[-1] + N1); kp2_off.append(kp2_off[-1] + N2)
    out = dict(n_pairs=n_pairs, geom=g, window_size=int(window_size), nn_ratio=float(nn_ratio), check_orientation=int(check_orientation),
               kp1_off=np.asarray(kp1_off, np.int32), kp2_off=np.asarray(kp2_off, np.int32))
    for k, v in acc.items():
        a = np.concatenate(v)
        if k.endswith("_octave") or k.endswith("_desc"):
            a = a.astype(np.uint8)
        else:
            a = f32(a)
            if k.endswith("_angle"):
                a = np.mod(a, f32(360.0))
                a[a >= 360.0] = 0.0   # float32 rounding of a tiny negative angle + 360
        out[k] = np.ascontiguousarray(a.reshape(-1, 32) if k.endswith("_desc") else a)
    return out


def _quat_xyzw(R):
    """unit quaternion (x y z w, w >= 0) of a rotation matrix"""
    w = np.sqrt(max(0.0, 1.0 + R[0, 0] + R[1, 1] + R[2, 2])) / 2.0
    x = np.copysign(np.sqrt(max(0.0, 1.0 + R[0, 0] - R[1, 1] - R[2, 2])) / 2.0, R[2, 1] - R[1, 2])
    y = np.copysign(np.sqrt(max(0.0, 1.0 - R[0, 0] + R[1, 1] - R[2, 2])) / 2.0, R[0, 2] - R[2, 0])
    z = np.copysign(np.sqrt(max(0.0, 1.0 - R[0, 0] - R[1, 1] + R[2, 2])) / 2.0, R[1, 0] - R[0, 1])
    q = np.array([x, y, z, w])
    return q / np.linalg.norm(q)


def make_sim3_batch(n_problems, n_corr, seed, fix_scale=1, outlier_frac=0.1, th2=10.0, rot_deg=3.0, trans_m=0.3, scale_pct=3.0):
    """Optimizer::OptimizeSim3 as LoopClosing::ComputeSim3 calls it (th2 = 10, 5 / 10 / 5 iterations): per loop candidate two
    KITTI-camera keyframes related by a Sim3 S12 (P1c = s R P2c + t; s = 1 with fix_scale, s in [0.5, 2] otherwise), points 4-40 m
    in front of keyframe 1 and visible from both, keypoints at ORB octaves 0-7 with 1.2^octave px noise, a share of gross outliers
    (one of the two keypoints replaced by an unrelated one), and an initial S12 off by a few degrees, decimetres and (free
    scale) percent.  n_corr may be a list (ragged problems, 0 allowed)."""
    rng = np.random.default_rng(seed)
    lvl_p = np.asarray([SCALE ** (-2.0 * l) for l in range(N_LEVELS)]); lvl_p /= lvl_p.sum()
    isig = inv_level_sigma2()
    K = np.array([FX, FY, CX, CY], np.float32).astype(np.float64)
    acc = {k: [] for k in ("p1c", "p2c", "obs1", "obs2", "info1", "info2")}
    S12, cams, off = [], [], [0]
    for pb in range(n_problems):
        m = int(n_corr[pb]) if np.ndim(n_corr) else int(n_corr)
        R = _rodrigues(rng.normal(0, 1, 3) * np.deg2rad(4.0) / np.sqrt(3))
        t = np.array([rng.uniform(-1, 1), rng.uniform(-0.2, 0.2), rng.uniform(-2, 2)])
        s = 1.0 if fix_scale else float(np.exp(rng.uniform(np.log(0.5), np.log(2.0))))
        # points in keyframe 1: inside its image, visible from keyframe 2
        X1 = np.zeros((0, 3))
        while len(X1) < m:
            z = rng.uniform(4.0, 40.0, 2 * m + 8)
            u, v = rng.uniform(20, IMG_W - 20, z.size), rng.uniform(20, IMG_H - 20, z.size)
            X = np.stack([(u - CX) / FX * z, (v - CY) / FY * z, z], 1)
            X2 = ((X - t) @ R) / s                         # S12^-1
            u2 = FX * X2[:, 0] / X2[:, 2] + CX; v2 = FY * X2[:, 1] / X2[:, 2] + CY
            ok = (X2[:, 2] > 1.0) & (u2 > 0) & (u2 < IMG_W) & (v2 > 0) & (v2 < IMG_H)
            X1 = np.concatenate([X1, X[ok]])[:m]
        X2 = ((X1 - t) @ R) / s
        oct1, oct2 = rng.choice(N_LEVELS, m, p=lvl_p), rng.choice(N_LEVELS, m, p=lvl_p)
        def obs(X, o):
            return np.stack([FX * X[:, 0] / X[:, 2] + CX, FY * X[:, 1] / X[:, 2] + CY], 1) + rng.normal(0, 1, (len(X), 2)) * (SCALE ** o)[:, None]
        o1, o2 = obs(X1, oct1), obs(X2, oct2)
        bad = rng.random(m) < outlier_frac
        side = rng.random(m) < 0.5
        junk = np.stack([rng.uniform(0, IMG_W, m), rng.uniform(0, IMG_H, m)], 1)
        o1[bad & side] = junk[bad & side]; o2[bad & ~side] = junk[bad & ~side]
        # map point positions carry their own small errors (5 mm at 10 m, growing with depth)
        P1 = X1 + rng.normal(0, 1, X1.shape) * 0.0005 * X1[:, 2:3]
        P2 = X2 + rng.normal(0, 1, X2.shape) * 0.0005 * X2[:, 2:3]
        acc["p1c"].append(P1); acc["p2c"].append(P2); acc["obs1"].append(o1); acc["obs2"].append(o2)
        acc["info1"].append(isig[oct1]); acc["info2"].append(isig[oct2])
        # initial estimate: the truth off by a few degrees, decimetres and percent
        dR = _rodrigues(rng.normal(0, 1, 3) * np.deg2rad(rot_deg) / np.sqrt(3))
        s0 = s if fix_scale else s * (1.0 + rng.uniform(-1, 1) * scale_pct / 100.0)
        S12.append(np.concatenate([_quat_xyzw(dR @ R), t + rng.normal(0, 1, 3) * trans_m / np.sqrt(3), [s0]]))
        cams.append(np.concatenate([K, K]))
        off.append(off[-1] + m)
    out = dict(n_problems=n_problems, S12=np.ascontiguousarray(np.asarray(S12, np.float64).reshape(-1, 8)),
               cam=np.ascontiguousarray(np.asarray(cams, np.float64).reshape(-1, 8)),
               fix_scale=np.full(n_problems, int(fix_scale), np.int32), th2=np.full(n_problems, th2, np.float32),
               off=np.asarray(off, np.int32), its_first=5, its_more_outliers=10, its_more_clean=5)
    for k, v in acc.items():
        w = 3 if k[0] == "p" else (2 if k[0] == "o" else 1)
        a = np.concatenate(v) if v else np.zeros((0, w))
        out[k] = np.ascontiguousarray(f32(a).reshape(-1, w) if w > 1 else f32(a).reshape(-1))
    return out


def make_line_match_batch(n_pairs, n_lines, desc_dim, seed, tau=2.0, min_len=10, ragged=False):
    rng = np.random.default_rng(seed)
    P, N, D = n_pairs, n_lines, desc_dim
    baseline = float(np.float32(BF) / np.float32(FX))
    Pm = np.stack([rng.uniform(-12, 12, (P, N)), rng.uniform(-2, 3, (P, N)), rng.uniform(4, 40, (P, N))], -1)
    dc = rng.normal(0, 1, (P, N, 3)); dc /= np.linalg.norm(dc, axis=-1, keepdims=True)
    half = rng.uniform(0.3, 4, (P, N))
    E1 = Pm - half[..., None] * dc; E2 = Pm + half[..., None] * dc
    E1[..., 2] = np.maximum(E1[..., 2], 1.5); E2[..., 2] = np.maximum(E2[..., 2], 1.5)

    def seg(shift, noise):
        a = np.stack([FX * (E1[..., 0] - shift) / E1[..., 2] + CX, FY * E1[..., 1] / E1[..., 2] + CY], -1)
        b = np.stack([FX * (E2[..., 0] - shift) / E2[..., 2] + CX, FY * E2[..., 1] / E2[..., 2] + CY], -1)
        return np.concatenate([a, b], -1) + rng.normal(0, noise, (P, N, 4))

    left = seg(0.0, 0.5)
    right = seg(baseline, 0.5)
    octl = rng.integers(0, 3, (P, N)).astype(np.int32)
    octr = np.where(rng.random((P, N)) < 0.95, octl, (octl + 1) % 3).astype(np.int32)
    dl = rng.normal(0, 1, (P, N, D)); dl /= np.linalg.norm(dl, axis=-1, keepdims=True)
    dr = dl + rng.normal(0, 0.05, (P, N, D))
    unrel = rng.random((P, N)) < 0.2
    rnd = rng.normal(0, 1, (P, N, D)); rnd /= np.linalg.norm(rnd, axis=-1, keepdims=True)
    dr = np.where(unrel[..., None], rnd, dr)
    right = np.where(unrel[..., None], seg(baseline, 30.0), right)
    perm = np.argsort(rng.random((P, N)), axis=1)
    right = np.take_along_axis(right, perm[..., None], 1)
    dr = np.take_along_axis(dr, perm[..., None], 1)
    octr = np.take_along_axis(octr, perm, 1)
    K = np.array([FX, 0, CX, 0, FY, CY, 0, 0, 1.0])
    nl = np.full(P, N); nr = np.full(P, N)
    if ragged:
        nl = rng.integers(0, N + 1, P); nr = rng.integers(0, N + 1, P)
        nl[0] = 0
        if P > 1:
            nr[1] = 0
    lsel = np.concatenate([np.arange(N)[None, :] < nl[:, None]]).reshape(P, N)
    rsel = (np.arange(N)[None, :] < nr[:, None])
    return dict(
        n_pairs=P, desc_dim=D, left_off=_csr(nl), right_off=_csr(nr),
        left_seg=f32(left[lsel]), left_octave=np.ascontiguousarray(octl[lsel]),
        right_seg=f32(right[rsel]), right_octave=np.ascontiguousarray(octr[rsel]),
        left_desc=f32(dl[lsel]), right_desc=f32(dr[rsel]),
        K=K, baseline=baseline, tau=float(tau), min_line_length=int(min_len),
    )


# ---------------------------------------------------------------------------------------------
# stereo frames for Frame::ComputeStereoMatches (SURVEY §8(f) row 1)
# ---------------------------------------------------------------------------------------------
def make_stereo_frame(seed, n_kp=400, rows=240, cols=376, n_levels=4, sf=1.2):
    """A textured stereo pair (right = left shifted by a per-band disparity), its pyramids, keypoints at random places
    with random octaves and ORB-like descriptors (right = left with a few flipped bits; a share are outliers)."""
    import cv2
    rng = np.random.default_rng(seed)
    disp_of_row = 4 + (np.arange(rows) // 40) * 3            # 4, 7, 10, ... pixels
    extra = max(64, 32 + int(disp_of_row.max()))              # source columns beyond the frame: 64 up to 376 rows
    base = rng.integers(0, 256, (rows // 4 + 2, (cols + extra) // 4 + 2), dtype=np.uint8)
    wide = cv2.resize(base, (cols + extra, rows), interpolation=cv2.INTER_CUBIC)
    left = np.ascontiguousarray(wide[:, 32:32 + cols])
    right = np.empty_like(left)
    for y in range(rows):
        d = int(disp_of_row[y])
        right[y] = wide[y, 32 + d:32 + d + cols]             # x_R = x_L - d
    scale = np.array([sf ** i for i in range(n_levels)], np.float32)
    inv = (1.0 / scale).astype(np.float32)
    pyrL, pyrR = [left], [right]
    for i in range(1, n_levels):
        sz = (int(round(cols * float(inv[i]))), int(round(rows * float(inv[i]))))
        pyrL.append(np.ascontiguousarray(cv2.resize(left, sz, interpolation=cv2.INTER_LINEAR)))
        pyrR.append(np.ascontiguousarray(cv2.resize(right, sz, interpolation=cv2.INTER_LINEAR)))
    kpL = np.stack([rng.uniform(30, cols - 30, n_kp), rng.uniform(24, rows - 24, n_kp)], 1).astype(np.float32)
    octL = rng.integers(0, n_levels, n_kp).astype(np.int32)
    descL = rng.integers(0, 256, (n_kp, 32), dtype=np.uint8)
    d = disp_of_row[kpL[:, 1].astype(int)].astype(np.float32)
    kpR = kpL.copy()
    kpR[:, 0] -= d + rng.normal(0, 0.4, n_kp).astype(np.float32)
    kpR[:, 1] += rng.normal(0, 0.5, n_kp).astype(np.float32)
    octR = np.clip(octL + rng.integers(-1, 2, n_kp), 0, n_levels - 1).astype(np.int32)
    flips = np.where(rng.random(n_kp) < 0.8, rng.integers(0, 40, n_kp), 128)   # inliers: a few bits; outliers: unrelated
    descR = descL.copy()
    for i in range(n_kp):
        for bpos in rng.integers(0, 256, int(flips[i])):
            descR[i, bpos >> 3] ^= np.uint8(1 << (bpos & 7))
    perm = rng.permutation(n_kp)
    kpR, octR, descR = kpR[perm], octR[perm], np.ascontiguousarray(descR[perm])
    keep = kpR[:, 0] > 20
    return dict(kpL=kpL, octL=octL, descL=descL, kpR=np.ascontiguousarray(kpR[keep]), octR=np.ascontiguousarray(octR[keep]),
                descR=np.ascontiguousarray(descR[keep]), scale=scale, inv=inv, pyrL=pyrL, pyrR=pyrR, mb=np.float32(0.54),
                mbf=np.float32(0.54 * 45.0))


def batch_stereo(frames, pad=0):
    """frames from make_stereo_frame (same pyramid geometry) -> lld_stereo_problem field dict.  pad > 0 lays every level out
    as a region inside a wider buffer, row stride cols + pad, as ORBextractor's bordered pyramid (pad = 2 * EDGE_THRESHOLD =
    38): pad // 2 columns of noise left of the image, the rest right of it."""
    f0 = frames[0]
    n_levels = len(f0["pyrL"])
    rows = np.array([a.shape[0] for a in f0["pyrL"]], np.int32)
    cols = np.array([a.shape[1] for a in f0["pyrL"]], np.int32)
    stride = cols + np.int32(pad)
    rng = np.random.default_rng(12345)
    offs, blobs, pos = [], [], 0
    for f in frames:
        for side in ("pyrL", "pyrR"):
            for l in range(n_levels):
                a = np.asarray(f[side][l])
                assert a.shape == (rows[l], cols[l])
                buf = rng.integers(0, 256, (rows[l], stride[l]), dtype=np.uint8)
                buf[:, pad // 2:pad // 2 + cols[l]] = a
                offs.append(pos + pad // 2); blobs.append(buf.reshape(-1)); pos += buf.size
    pyr = np.concatenate(blobs)
    return dict(
        n_frames=len(frames), left_off=_csr([len(f["kpL"]) for f in frames]), right_off=_csr([len(f["kpR"]) for f in frames]),
        left_xy=np.ascontiguousarray(np.concatenate([f["kpL"] for f in frames]), np.float32),
        left_octave=np.ascontiguousarray(np.concatenate([f["octL"] for f in frames]), np.uint8),
        left_desc=np.ascontiguousarray(np.concatenate([f["descL"] for f in frames])),
        right_xy=np.ascontiguousarray(np.concatenate([f["kpR"] for f in frames]).reshape(-1, 2), np.float32),
        right_octave=np.ascontiguousarray(np.concatenate([f["octR"] for f in frames]), np.uint8),
        right_desc=np.ascontiguousarray(np.concatenate([f["descR"] for f in frames]).reshape(-1, 32)),
        n_levels=n_levels, scale_factors=f0["scale"], inv_scale_factors=f0["inv"],
        pyr=pyr, pyr_bytes=int(pyr.size), pyr_off=np.array(offs, np.int64), pyr_rows=rows, pyr_cols=cols, pyr_stride=stride,
        mb=float(f0["mb"]), mbf=float(f0["mbf"]), frames=frames)


# ---------------------------------------------------------------------------------------------
# temporal line association (Tracking::AddLinesFrom, SURVEY §8(f) row 3)
# ---------------------------------------------------------------------------------------------
def make_line_assoc_batch(n_frames, n_ml, n_cur, desc_dim, seed, n_cand=12):
    """Per frame: n_ml map lines in front of a stereo camera, n_cur current left lines (the projections of a subset of the
    map lines with pixel noise, plus clutter), right lines for most of them, candidate lists that contain the true line
    among random others, descriptors = map line descriptor + noise."""
    rng = np.random.default_rng(seed)
    K = np.array([[FX, 0, CX], [0, FY, CY], [0, 0, 1.0]])
    b = float(np.float32(BF) / np.float32(FX))
    out = dict(n_frames=n_frames, desc_dim=desc_dim, K=K.reshape(-1), thr_reproj_base=3.0, md_thr=2.0, monocular=0)
    ml_off, cur_off, right_off, cand_off = [0], [0], [0], [0]
    ml_valid, ml_xd, ml_x12, ml_desc, cand_idx = [], [], [], [], []
    cur_left, cur_oct, cur_lm, cur_taken, cur_desc, cur_right, Tc, Tr = [], [], [], [], [], [], [], []
    for f in range(n_frames):
        yaw = rng.normal(0, 0.05)
        R = _rot_y(np.array(yaw))                        # camera-to-world
        c = rng.normal(0, 0.3, 3)
        T = np.eye(4); T[:3, :3] = R; T[:3, 3] = c
        T2 = T.copy(); T2[:3, 3] = c + R @ np.array([b, 0, 0])
        Tc.append(T.reshape(-1)); Tr.append(T2.reshape(-1))
        X1c = np.stack([rng.uniform(-8, 8, n_ml), rng.uniform(-2, 2, n_ml), rng.uniform(4, 30, n_ml)], 1)
        dirc = rng.normal(0, 1, (n_ml, 3)); dirc[:, 2] *= 0.3
        dirc /= np.linalg.norm(dirc, axis=1, keepdims=True)
        X2c = X1c + dirc * rng.uniform(1, 4, n_ml)[:, None]
        X1 = (R @ X1c.T).T + c; X2 = (R @ X2c.T).T + c
        d = (X2 - X1) / np.linalg.norm(X2 - X1, axis=1, keepdims=True)
        X0 = X1 - (X1 * d).sum(1, keepdims=True) * d
        desc = rng.normal(0, 1, (n_ml, desc_dim)); desc /= np.linalg.norm(desc, axis=1, keepdims=True)

        def proj(Xc):
            x = (K @ Xc.T).T
            return x[:, :2] / x[:, 2:3]
        owner = rng.permutation(n_ml)[:n_cur] if n_cur <= n_ml else rng.integers(0, n_ml, n_cur)
        noise = lambda: rng.normal(0, 0.6, (n_cur, 2))   # noqa: E731
        s, e = proj(X1c[owner]) + noise(), proj(X2c[owner]) + noise()
        clutter = rng.random(n_cur) < 0.25
        s[clutter] += rng.uniform(-60, 60, (int(clutter.sum()), 2))
        left = np.concatenate([s, e], 1)
        shift = np.array([b, 0, 0])
        sr, er = proj(X1c[owner] - shift) + noise(), proj(X2c[owner] - shift) + noise()
        has_r = rng.random(n_cur) < 0.85
        lm = np.full(n_cur, -1, np.int64); lm[has_r] = np.arange(int(has_r.sum()))
        right = np.concatenate([sr, er], 1)[has_r]
        cdesc = desc[owner] + rng.normal(0, 0.05, (n_cur, desc_dim))
        cdesc[clutter] = rng.normal(0, 1, (int(clutter.sum()), desc_dim))
        inv = {int(o): i for i, o in enumerate(owner)}
        for i in range(n_ml):
            cs = list(rng.integers(0, n_cur, n_cand))
            if i in inv and rng.random() < 0.9:
                cs[int(rng.integers(0, n_cand))] = inv[i]
            cand_idx += cs
            cand_off.append(len(cand_idx))
        ml_valid.append((rng.random(n_ml) < 0.9).astype(np.uint8)); ml_xd.append(np.concatenate([X0, d], 1)); ml_x12.append(np.concatenate([X1, X2], 1))
        ml_desc.append(desc); cur_left.append(left); cur_oct.append(rng.integers(0, 3, n_cur)); cur_lm.append(lm)
        cur_taken.append((rng.random(n_cur) < 0.1).astype(np.uint8)); cur_desc.append(cdesc); cur_right.append(right)
        ml_off.append(ml_off[-1] + n_ml); cur_off.append(cur_off[-1] + n_cur); right_off.append(right_off[-1] + len(right))
    out.update(ml_off=np.array(ml_off, np.int32), ml_valid=np.concatenate(ml_valid), ml_x0_dir=np.ascontiguousarray(np.concatenate(ml_xd)),
               ml_x1x2=np.ascontiguousarray(np.concatenate(ml_x12)), ml_desc=np.ascontiguousarray(np.concatenate(ml_desc), np.float32),
               cand_off=np.array(cand_off, np.int32), cand_idx=np.array(cand_idx, np.int32), cur_off=np.array(cur_off, np.int32),
               cur_left=np.ascontiguousarray(np.concatenate(cur_left), np.float32), cur_octave=np.concatenate(cur_oct).astype(np.int32),
               cur_line_match=np.concatenate(cur_lm).astype(np.int32), cur_taken=np.concatenate(cur_taken),
               cur_desc=np.ascontiguousarray(np.concatenate(cur_desc), np.float32), right_off=np.array(right_off, np.int32),
               cur_right=np.ascontiguousarray(np.concatenate(cur_right), np.float32).reshape(-1, 4),
               T_curr=np.ascontiguousarray(np.stack(Tc)), T_right=np.ascontiguousarray(np.stack(Tr)))
    return out
