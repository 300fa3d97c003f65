"""Python-side callers of the C-ABI (include/lldba.h): allocate outputs, fill the ctypes structs, call.

`impl` selects the library:  "gpu" = the product (CUDA, needs a Context), "oracle" = the CPU oracle
(tests / cpu_baseline only).  The product path never routes through the oracle.
"""
from __future__ import annotations

import ctypes as C
from typing import Any, Dict, Optional

import numpy as np

from . import capi


def _lib(impl: str):
    if impl == "gpu":
        return capi.load_library()
    if impl == "oracle":
        return capi.load_oracle()
    raise ValueError(impl)


def _handle(impl: str, ctx: Optional[capi.Context]):
    if impl == "gpu":
        if ctx is None:
            raise ValueError("the CUDA library needs a Context (lld_ctx_create)")
        return ctx.handle
    return C.c_void_p()


def _check(impl, ctx, rc, what):
    if rc != 0:
        if impl == "gpu" and ctx is not None:
            ctx.check(rc, what)
        raise RuntimeError(f"{what} failed with {rc}")


def _stop_ptr(stop):
    if stop is None:
        return None, None
    arr = np.ascontiguousarray(stop, dtype=np.uint8)
    return arr.ctypes.data_as(capi.c_u8p), arr


def _ba_outputs(p: Dict[str, Any], log_stride: int):
    n_kf = int(p["kf_off"][-1]); n_pt = int(p["pt_off"][-1]); n_ln = int(p["ln_off"][-1])
    n_pe = int(p["pt_obs_off"][-1]); n_lc = int(p["ln_obs_off"][-1]); nw = int(p["n_win"])
    return dict(
        kf_Tcw=np.zeros((n_kf, 12)), pt_xyz=np.zeros((n_pt, 3)), ln_x0_dir=np.zeros((n_ln, 6)),
        pt_obs_bad=np.zeros(n_pe, np.uint8), ln_obs_bad=np.zeros((n_lc, 2), np.uint8), ln_removed=np.zeros(n_ln, np.uint8),
        log_stride=log_stride,
        chi2_log=np.zeros((nw, log_stride)), lambda_log=np.zeros((nw, log_stride)),
        trials_log=np.zeros((nw, log_stride), np.int32), n_iter_done=np.zeros((nw, 2), np.int32),
    )


def ba_local(p: Dict[str, Any], its1: int = 5, its2: int = 15, *, impl: str = "gpu", ctx=None, stop=None):
    lib = _lib(impl)
    prob, keep = capi.fill_struct(capi.BaProblem, p)
    out = _ba_outputs(p, its1 + its2 + 2)
    res, keep2 = capi.fill_struct(capi.BaResult, out)
    sp, sk = _stop_ptr(stop)
    rc = lib.ba_local(_handle(impl, ctx), C.byref(prob), its1, its2, sp, C.byref(res))
    _check(impl, ctx, rc, "lld_ba_local")
    return out


def ba_global(p: Dict[str, Any], n_iter: int = 10, *, impl: str = "gpu", ctx=None, stop=None):
    lib = _lib(impl)
    prob, keep = capi.fill_struct(capi.BaProblem, p)
    out = _ba_outputs(p, n_iter + 2)
    res, keep2 = capi.fill_struct(capi.BaResult, out)
    sp, sk = _stop_ptr(stop)
    rc = lib.ba_global(_handle(impl, ctx), C.byref(prob), n_iter, sp, C.byref(res))
    _check(impl, ctx, rc, "lld_ba_global")
    return out


def pose_opt(p: Dict[str, Any], *, impl: str = "gpu", ctx=None):
    lib = _lib(impl)
    prob, keep = capi.fill_struct(capi.PoseProblem, p)
    F = int(p["n_frames"])
    out = dict(Tcw=np.zeros((F, 12)), pt_outlier=np.zeros(int(p["pt_off"][-1]), np.uint8),
               ln_outlier=np.zeros(int(p["ln_off"][-1]), np.uint8), n_inliers=np.zeros(F, np.int32),
               chi2_final=np.zeros(F))
    res, keep2 = capi.fill_struct(capi.PoseResult, out)
    rc = lib.pose_opt(_handle(impl, ctx), C.byref(prob), C.byref(res))
    _check(impl, ctx, rc, "lld_pose_opt")
    return out


def _sbp_out(n_cur, n_q, n_pairs):
    return dict(match=np.full(n_cur, -1, np.int32), n_matches=np.zeros(n_pairs, np.int32),
                best_idx=np.full(n_q, -1, np.int32), best_dist=np.full(n_q, 256, np.int32))


def sbp_frame(p: Dict[str, Any], *, impl: str = "gpu", ctx=None):
    lib = _lib(impl)
    geom, gk = capi.make_geom(p["geom"])
    f = dict(p); f["geom"] = geom
    f.setdefault("th_high", 0); f.setdefault("allow_negative_depth", 0)
    prob, keep = capi.fill_struct(capi.SbpFrameProblem, f)
    out = _sbp_out(int(p["cur_off"][-1]), int(p["last_off"][-1]), int(p["n_pairs"]))
    res, keep2 = capi.fill_struct(capi.SbpResult, out)
    rc = lib.sbp_frame(_handle(impl, ctx), C.byref(prob), C.byref(res))
    _check(impl, ctx, rc, "lld_sbp_frame")
    return out


def sbp_mappoints(p: Dict[str, Any], *, impl: str = "gpu", ctx=None):
    lib = _lib(impl)
    geom, gk = capi.make_geom(p["geom"])
    f = dict(p); f["geom"] = geom
    prob, keep = capi.fill_struct(capi.SbpMpProblem, f)
    out = _sbp_out(int(p["cur_off"][-1]), int(p["mp_off"][-1]), int(p["n_pairs"]))
    res, keep2 = capi.fill_struct(capi.SbpResult, out)
    rc = lib.sbp_mappoints(_handle(impl, ctx), C.byref(prob), C.byref(res))
    _check(impl, ctx, rc, "lld_sbp_mappoints")
    return out


def kf_search(p: Dict[str, Any], *, impl: str = "gpu", ctx=None):
    """ORBmatcher::Fuse / Fuse(Scw) / SearchByProjection(KeyFrame*, Scw, ...): windowed search of projected map points in keyframes"""
    lib = _lib(impl)
    geom, gk = capi.make_geom(p["geom"])
    f = dict(p); f["geom"] = geom
    prob, keep = capi.fill_struct(capi.KfSearchProblem, f)
    out = _sbp_out(int(p["kp_off"][-1]), int(p["mp_off"][-1]), int(p["n_pairs"]))
    res, keep2 = capi.fill_struct(capi.SbpResult, out)
    rc = lib.kf_search(_handle(impl, ctx), C.byref(prob), C.byref(res))
    _check(impl, ctx, rc, "lld_kf_search")
    return out


def tri_search(p: Dict[str, Any], *, impl: str = "gpu", ctx=None):
    """ORBmatcher::SearchForTriangulation, batched over keyframe pairs"""
    lib = _lib(impl)
    prob, keep = capi.fill_struct(capi.TriSearchProblem, p)
    out = dict(match12=np.full(max(int(p["kp1_off"][-1]), 1), -1, np.int32), n_matches=np.zeros(int(p["n_pairs"]), np.int32))
    res, keep2 = capi.fill_struct(capi.TriSearchResult, out)
    rc = lib.tri_search(_handle(impl, ctx), C.byref(prob), C.byref(res))
    _check(impl, ctx, rc, "lld_tri_search")
    out["match12"] = out["match12"][:int(p["kp1_off"][-1])]
    return out


def bow_search(p: Dict[str, Any], *, impl: str = "gpu", ctx=None):
    """ORBmatcher::SearchByBoW (KeyFrame -> Frame, KeyFrame -> KeyFrame), batched over pairs"""
    lib = _lib(impl)
    prob, keep = capi.fill_struct(capi.BowSearchProblem, p)
    out = dict(match12=np.full(max(int(p["kp1_off"][-1]), 1), -1, np.int32), n_matches=np.zeros(int(p["n_pairs"]), np.int32))
    res, keep2 = capi.fill_struct(capi.TriSearchResult, out)
    rc = lib.bow_search(_handle(impl, ctx), C.byref(prob), C.byref(res))
    _check(impl, ctx, rc, "lld_bow_search")
    out["match12"] = out["match12"][:int(p["kp1_off"][-1])]
    return out


def init_search(p: Dict[str, Any], *, impl: str = "gpu", ctx=None):
    """ORBmatcher::SearchForInitialization, batched over frame pairs: match12 (vnMatches12), n_matches, prev_matched
    (vbPrevMatched after the call, [n1][2])"""
    lib = _lib(impl)
    geom, gk = capi.make_geom(p["geom"])
    f = dict(p); f["geom"] = geom
    prob, keep = capi.fill_struct(capi.InitSearchProblem, f)
    n1 = int(p["kp1_off"][-1])
    out = dict(match12=np.full(max(n1, 1), -2, np.int32), n_matches=np.zeros(int(p["n_pairs"]), np.int32),
               prev_matched=np.zeros((max(n1, 1), 2), np.float32))
    res, keep2 = capi.fill_struct(capi.InitSearchResult, out)
    rc = lib.init_search(_handle(impl, ctx), C.byref(prob), C.byref(res))
    _check(impl, ctx, rc, "lld_init_search")
    out["match12"] = out["match12"][:n1]
    out["prev_matched"] = out["prev_matched"][:n1]
    return out


def sim3_opt(p: Dict[str, Any], *, impl: str = "gpu", ctx=None):
    """Optimizer::OptimizeSim3, batched over loop candidates: S12 (g2oS12 after the call, [n][8] q t s), inlier (vpMatches1 kept,
    [m]), n_in (return value) and the LM trace of both rounds (include/lldba.h)"""
    lib = _lib(impl)
    prob, keep = capi.fill_struct(capi.Sim3Problem, p)
    n, m = int(p["n_problems"]), int(p["off"][-1])
    stride = int(p["its_first"]) + max(int(p["its_more_outliers"]), int(p["its_more_clean"])) + 2
    out = dict(S12=np.zeros((max(n, 1), 8)), inlier=np.full(max(m, 1), 2, np.uint8), n_in=np.full(max(n, 1), -1, np.int32),
               log_stride=stride, chi2_log=np.zeros((max(n, 1), stride)), lambda_log=np.zeros((max(n, 1), stride)),
               trials_log=np.zeros((max(n, 1), stride), np.int32), n_iter_done=np.zeros((max(n, 1), 2), np.int32))
    res, keep2 = capi.fill_struct(capi.Sim3Result, out)
    rc = lib.sim3_opt(_handle(impl, ctx), C.byref(prob), C.byref(res))
    _check(impl, ctx, rc, "lld_sim3_opt")
    for k in ("S12", "n_in", "chi2_log", "lambda_log", "trials_log", "n_iter_done"):
        out[k] = out[k][:n]
    out["inlier"] = out["inlier"][:m]
    return out


def line_match(p: Dict[str, Any], *, impl: str = "gpu", ctx=None):
    lib = _lib(impl)
    prob, keep = capi.fill_struct(capi.LineMatchProblem, p)
    n_left = int(p["left_off"][-1])
    out = dict(match=np.full(n_left, -1, np.int32), dist=np.full(n_left, np.inf, np.float32))
    res, keep2 = capi.fill_struct(capi.LineMatchResult, out)
    rc = lib.line_match(_handle(impl, ctx), C.byref(prob), C.byref(res))
    _check(impl, ctx, rc, "lld_line_match")
    return out


def descriptor_distance(a: np.ndarray, b: np.ndarray, *, impl: str = "gpu") -> int:
    lib = _lib(impl)
    a = np.ascontiguousarray(a, np.uint8); b = np.ascontiguousarray(b, np.uint8)
    assert a.size == 32 and b.size == 32
    return int(lib.descriptor_distance(a.ctypes.data_as(capi.c_u8p), b.ctypes.data_as(capi.c_u8p)))


def stereo_matches(p: Dict[str, Any], *, impl: str = "gpu", ctx=None):
    """Frame::ComputeStereoMatches on a batch (synth.batch_stereo).  The oracle has a per-frame entry point."""
    n_left = int(p["left_off"][-1]); F = int(p["n_frames"])
    out = dict(uright=np.full(n_left, -1, np.float32), depth=np.full(n_left, -1, np.float32), n_matched=np.zeros(F, np.int32))
    if impl == "gpu":
        lib = _lib(impl)
        prob, keep = capi.fill_struct(capi.StereoProblem, {k: v for k, v in p.items() if k != "frames"})
        res, keep2 = capi.fill_struct(capi.StereoResult, out)
        rc = lib.dll.lld_stereo_matches(_handle(impl, ctx), C.byref(prob), C.byref(res))
        _check(impl, ctx, rc, "lld_stereo_matches")
        return out
    dll = capi.load_oracle().dll
    fn = dll.lldo_stereo_matches
    fn.restype = C.c_int
    P = C.c_void_p
    fn.argtypes = [C.c_int, P, P, P, C.c_int, P, P, P, C.c_int, P, P, P, P, P, P, P, C.c_float, C.c_float, P, P]
    L = int(p["n_levels"])
    ptr = lambda a: a.ctypes.data_as(P)   # noqa: E731
    for f in range(F):
        a, b = int(p["left_off"][f]), int(p["left_off"][f + 1])
        ra, rb = int(p["right_off"][f]), int(p["right_off"][f + 1])
        base = p["pyr"].ctypes.data
        arrL = (P * L)(*[base + int(p["pyr_off"][(f * 2 + 0) * L + l]) for l in range(L)])
        arrR = (P * L)(*[base + int(p["pyr_off"][(f * 2 + 1) * L + l]) for l in range(L)])
        kl = np.ascontiguousarray(p["left_xy"][a:b]); ol = np.ascontiguousarray(p["left_octave"][a:b].astype(np.int32)); dl = np.ascontiguousarray(p["left_desc"][a:b])
        kr = np.ascontiguousarray(p["right_xy"][ra:rb]); orr = np.ascontiguousarray(p["right_octave"][ra:rb].astype(np.int32)); dr = np.ascontiguousarray(p["right_desc"][ra:rb])
        uR, dep = np.empty(b - a, np.float32), np.empty(b - a, np.float32)
        n = fn(b - a, ptr(kl), ptr(ol), ptr(dl), rb - ra, ptr(kr), ptr(orr), ptr(dr), L, ptr(p["scale_factors"]), ptr(p["inv_scale_factors"]),
               C.cast(arrL, P), C.cast(arrR, P), ptr(p["pyr_rows"]), ptr(p["pyr_cols"]), ptr(p["pyr_stride"]),
               C.c_float(float(p["mb"])), C.c_float(float(p["mbf"])), ptr(uR), ptr(dep))
        out["uright"][a:b] = uR; out["depth"][a:b] = dep; out["n_matched"][f] = n
    return out


def medoid_orb(off, desc, *, impl: str = "gpu", ctx=None):
    """MapPoint::ComputeDistinctiveDescriptors, batched: best descriptor index per landmark"""
    off = np.ascontiguousarray(off, np.int32); desc = np.ascontiguousarray(desc, np.uint8)
    best = np.full(len(off) - 1, -2, np.int32)
    dll = _lib(impl).dll
    fn = getattr(dll, ("lld_" if impl == "gpu" else "lldo_") + "medoid_orb")
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p, C.c_int32, capi.c_i32p, capi.c_u8p, capi.c_i32p]
    rc = fn(_handle(impl, ctx), len(off) - 1, off.ctypes.data_as(capi.c_i32p), desc.ctypes.data_as(capi.c_u8p), best.ctypes.data_as(capi.c_i32p))
    _check(impl, ctx, rc, "lld_medoid_orb")
    return best


def medoid_float(off, desc, *, impl: str = "gpu", ctx=None):
    """MapLine::ComputeDistinctiveDescriptors, batched"""
    off = np.ascontiguousarray(off, np.int32); desc = np.ascontiguousarray(desc, np.float32)
    best = np.full(len(off) - 1, -2, np.int32)
    dll = _lib(impl).dll
    fn = getattr(dll, ("lld_" if impl == "gpu" else "lldo_") + "medoid_float")
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p, C.c_int32, capi.c_i32p, C.c_int32, capi.c_f32p, capi.c_i32p]
    rc = fn(_handle(impl, ctx), len(off) - 1, off.ctypes.data_as(capi.c_i32p), int(desc.shape[1]), desc.ctypes.data_as(capi.c_f32p),
            best.ctypes.data_as(capi.c_i32p))
    _check(impl, ctx, rc, "lld_medoid_float")
    return best


class LineAssocProblem(C.Structure):
    _fields_ = [
        ("n_frames", C.c_int32), ("ml_off", capi.c_i32p), ("ml_valid", capi.c_u8p), ("ml_x0_dir", capi.c_f64p), ("ml_x1x2", capi.c_f64p),
        ("ml_desc", capi.c_f32p), ("cand_off", capi.c_i32p), ("cand_idx", capi.c_i32p), ("cur_off", capi.c_i32p), ("cur_left", capi.c_f32p),
        ("cur_octave", capi.c_i32p), ("cur_line_match", capi.c_i32p), ("cur_taken", capi.c_u8p), ("cur_desc", capi.c_f32p),
        ("right_off", capi.c_i32p), ("cur_right", capi.c_f32p), ("desc_dim", C.c_int32), ("T_curr", capi.c_f64p), ("T_right", capi.c_f64p),
        ("K", C.c_double * 9), ("thr_reproj_base", C.c_double), ("md_thr", C.c_double), ("monocular", C.c_int32),
    ]


class LineAssocResult(C.Structure):
    _fields_ = [("cur_assoc", capi.c_i32p), ("n_added", capi.c_i32p)]


def line_associate(p: Dict[str, Any], *, impl: str = "gpu", ctx=None):
    """Tracking::AddLinesFrom, batched over frames"""
    dll = _lib(impl).dll
    fn = getattr(dll, ("lld_" if impl == "gpu" else "lldo_") + "line_associate")
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p, C.POINTER(LineAssocProblem), C.POINTER(LineAssocResult)]
    prob, keep = capi.fill_struct(LineAssocProblem, p)
    out = dict(cur_assoc=np.full(int(p["cur_off"][-1]), -2, np.int32), n_added=np.zeros(int(p["n_frames"]), np.int32))
    res, keep2 = capi.fill_struct(LineAssocResult, out)
    rc = fn(_handle(impl, ctx), C.byref(prob), C.byref(res))
    _check(impl, ctx, rc, "lld_line_associate")
    return out
