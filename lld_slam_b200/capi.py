"""ctypes mirror of include/lldba.h.

This is the Python harness over the C-ABI used by tests/ and bench.py.  The product library is
lld_slam_b200/csrc/liblldba.so (CUDA, sm_100a); `load_library()` fails loudly when it is missing —
there is no CPU fallback.  `load_oracle()` loads the CPU oracle (oracle/liblld_oracle.so) which
exposes the same entry points with the `lldo_` prefix (lldo_init_search from tests/hostcheck/libinit_search_oracle.so, lldo_sim3_opt from
tests/hostcheck/libsim3_oracle.so); only tests, smoke() and the bench's
cpu_baseline / reference arm may call it.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Any, Dict

import numpy as np

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.environ.get("LLD_LIB_PATH") or os.path.join(_ROOT, "lld_slam_b200", "csrc", "liblldba.so")  # override: kernel A/B experiments
ORACLE_PATH = os.path.join(_ROOT, "oracle", "liblld_oracle.so")
# the oracle's SearchForInitialization (lldo_init_search) is a separate test-infrastructure library
INIT_SEARCH_ORACLE_PATH = os.path.join(_ROOT, "tests", "hostcheck", "libinit_search_oracle.so")
SIM3_ORACLE_PATH = os.path.join(_ROOT, "tests", "hostcheck", "libsim3_oracle.so")

c_i32p = C.POINTER(C.c_int32)
c_u8p = C.POINTER(C.c_uint8)
c_f32p = C.POINTER(C.c_float)
c_f64p = C.POINTER(C.c_double)

_NP2C = {
    np.dtype(np.int32): c_i32p,
    np.dtype(np.uint8): c_u8p,
    np.dtype(np.float32): c_f32p,
    np.dtype(np.float64): c_f64p,
}


class BaProblem(C.Structure):
    _fields_ = [
        ("n_win", C.c_int32),
        ("kf_off", c_i32p), ("pt_off", c_i32p), ("ln_off", c_i32p),
        ("kf_Tcw", c_f64p), ("kf_fixed", c_u8p), ("kf_intr", c_f64p), ("kf_line_cam", c_f64p),
        ("pt_xyz", c_f64p), ("pt_obs_off", c_i32p), ("pt_obs_kf", c_i32p),
        ("pt_obs_uvr", c_f32p), ("pt_obs_info", c_f32p),
        ("ln_x0_dir", c_f64p), ("ln_obs_off", c_i32p), ("ln_obs_kf", c_i32p),
        ("ln_obs_left", c_f32p), ("ln_obs_right", c_f32p), ("ln_obs_info", c_f64p), ("ln_obs_stereo", c_u8p),
        ("robust_points", C.c_int32),
        ("delta_pt_mono", C.c_double), ("delta_pt_stereo", C.c_double),
        ("delta_ln_mono", C.c_double), ("delta_ln_stereo", C.c_double),
        ("chi2_pt_mono", C.c_double), ("chi2_pt_stereo", C.c_double),
        ("ln_endpoints_normalized", C.c_int32), ("ln_filter", C.c_int32),
    ]


class BaResult(C.Structure):
    _fields_ = [
        ("kf_Tcw", c_f64p), ("pt_xyz", c_f64p), ("ln_x0_dir", c_f64p),
        ("pt_obs_bad", c_u8p), ("ln_obs_bad", c_u8p), ("ln_removed", c_u8p),
        ("log_stride", C.c_int32),
        ("chi2_log", c_f64p), ("lambda_log", c_f64p), ("trials_log", c_i32p), ("n_iter_done", c_i32p),
    ]


class PoseProblem(C.Structure):
    _fields_ = [
        ("n_frames", C.c_int32),
        ("Tcw", c_f64p), ("intr", c_f64p), ("line_cam", c_f64p),
        ("pt_off", c_i32p), ("pt_xw", c_f32p), ("pt_uvr", c_f32p), ("pt_info", c_f32p),
        ("ln_off", c_i32p), ("ln_x0_dir", c_f64p), ("ln_left", c_f32p), ("ln_right", c_f32p),
        ("ln_info", c_f64p), ("ln_stereo", c_u8p), ("ln_gate_stereo", c_u8p),
        ("delta_mono", C.c_double), ("delta_stereo", C.c_double),
        ("delta_ln_mono", C.c_double), ("delta_ln_stereo", C.c_double),
        ("chi2_mono", C.c_float), ("chi2_stereo", C.c_float),
        ("gate_ln_mono", C.c_double), ("gate_ln_stereo", C.c_double),
        ("n_rounds", C.c_int32), ("its", C.c_int32),
    ]


class PoseResult(C.Structure):
    _fields_ = [
        ("Tcw", c_f64p), ("pt_outlier", c_u8p), ("ln_outlier", c_u8p), ("n_inliers", c_i32p), ("chi2_final", c_f64p),
    ]


class FrameGeom(C.Structure):
    _fields_ = [
        ("fx", C.c_float), ("fy", C.c_float), ("cx", C.c_float), ("cy", C.c_float), ("bf", C.c_float), ("b", C.c_float),
        ("min_x", C.c_float), ("max_x", C.c_float), ("min_y", C.c_float), ("max_y", C.c_float),
        ("n_levels", C.c_int32), ("scale_factors", c_f32p),
    ]


class SbpFrameProblem(C.Structure):
    _fields_ = [
        ("n_pairs", C.c_int32), ("geom", FrameGeom), ("th", C.c_float), ("mono", C.c_int32), ("check_orientation", C.c_int32),
        ("cur_off", c_i32p), ("cur_xy", c_f32p), ("cur_octave", c_u8p), ("cur_angle", c_f32p), ("cur_uright", c_f32p),
        ("cur_desc", c_u8p), ("cur_claimed", c_u8p), ("cur_Tcw", c_f32p), ("last_Tcw", c_f32p),
        ("last_off", c_i32p), ("last_valid", c_u8p), ("last_xw", c_f32p), ("last_octave", c_u8p), ("last_angle", c_f32p),
        ("last_desc", c_u8p), ("last_has_obs", c_u8p),
        ("th_high", C.c_int32), ("allow_negative_depth", C.c_int32),
    ]


class SbpResult(C.Structure):
    _fields_ = [("match", c_i32p), ("n_matches", c_i32p), ("best_idx", c_i32p), ("best_dist", c_i32p)]


class SbpMpProblem(C.Structure):
    _fields_ = [
        ("n_pairs", C.c_int32), ("geom", FrameGeom), ("th", C.c_float), ("nn_ratio", C.c_float),
        ("cur_off", c_i32p), ("cur_xy", c_f32p), ("cur_octave", c_u8p), ("cur_uright", c_f32p),
        ("cur_desc", c_u8p), ("cur_claimed", c_u8p),
        ("mp_off", c_i32p), ("mp_valid", c_u8p), ("mp_proj", c_f32p), ("mp_level", c_i32p), ("mp_viewcos", c_f32p),
        ("mp_desc", c_u8p), ("mp_has_obs", c_u8p),
    ]


class KfSearchProblem(C.Structure):
    _fields_ = [
        ("n_pairs", C.c_int32), ("geom", FrameGeom), ("th", C.c_float), ("th_low", C.c_int32), ("chi2_gate", C.c_int32),
        ("sequential_claims", C.c_int32), ("inv_level_sigma2", C.c_float * 8),
        ("kp_off", c_i32p), ("kp_xy", c_f32p), ("kp_octave", c_u8p), ("kp_uright", c_f32p), ("kp_desc", c_u8p), ("kp_claimed", c_u8p),
        ("mp_off", c_i32p), ("mp_valid", c_u8p), ("mp_proj", c_f32p), ("mp_level", c_i32p), ("mp_desc", c_u8p),
    ]


class TriSearchProblem(C.Structure):
    _fields_ = [
        ("n_pairs", C.c_int32), ("only_stereo", C.c_int32), ("check_orientation", C.c_int32), ("n_levels", C.c_int32),
        ("scale_factors", C.c_float * 8), ("level_sigma2", C.c_float * 8), ("F12", c_f32p), ("epipole", c_f32p),
        ("kp1_off", c_i32p), ("kp1_xy", c_f32p), ("kp1_angle", c_f32p), ("kp1_uright", c_f32p), ("kp1_has_mp", c_u8p), ("kp1_desc", c_u8p),
        ("kp2_off", c_i32p), ("kp2_xy", c_f32p), ("kp2_octave", c_u8p), ("kp2_angle", c_f32p), ("kp2_uright", c_f32p), ("kp2_has_mp", c_u8p),
        ("kp2_desc", c_u8p),
        ("fv1_node_off", c_i32p), ("fv1_node", c_i32p), ("fv1_idx_off", c_i32p), ("fv1_idx", c_i32p),
        ("fv2_node_off", c_i32p), ("fv2_node", c_i32p), ("fv2_idx_off", c_i32p), ("fv2_idx", c_i32p),
    ]


class BowSearchProblem(C.Structure):
    _fields_ = [
        ("n_pairs", C.c_int32), ("strict_th", C.c_int32), ("check_orientation", C.c_int32), ("nn_ratio", C.c_float),
        ("kp1_off", c_i32p), ("kp1_angle", c_f32p), ("kp1_valid", c_u8p), ("kp1_desc", c_u8p),
        ("kp2_off", c_i32p), ("kp2_angle", c_f32p), ("kp2_valid", c_u8p), ("kp2_desc", c_u8p),
        ("fv1_node_off", c_i32p), ("fv1_node", c_i32p), ("fv1_idx_off", c_i32p), ("fv1_idx", c_i32p),
        ("fv2_node_off", c_i32p), ("fv2_node", c_i32p), ("fv2_idx_off", c_i32p), ("fv2_idx", c_i32p),
    ]


class InitSearchProblem(C.Structure):
    _fields_ = [
        ("n_pairs", C.c_int32), ("geom", FrameGeom), ("window_size", C.c_int32), ("nn_ratio", C.c_float), ("check_orientation", C.c_int32),
        ("kp1_off", c_i32p), ("kp1_octave", c_u8p), ("kp1_angle", c_f32p), ("kp1_desc", c_u8p), ("prev_matched", c_f32p),
        ("kp2_off", c_i32p), ("kp2_xy", c_f32p), ("kp2_octave", c_u8p), ("kp2_angle", c_f32p), ("kp2_desc", c_u8p),
    ]


class InitSearchResult(C.Structure):
    _fields_ = [("match12", c_i32p), ("n_matches", c_i32p), ("prev_matched", c_f32p)]


class Sim3Problem(C.Structure):
    _fields_ = [
        ("n_problems", C.c_int32), ("S12", c_f64p), ("cam", c_f64p), ("fix_scale", c_i32p), ("th2", c_f32p), ("off", c_i32p),
        ("p1c", c_f32p), ("p2c", c_f32p), ("obs1", c_f32p), ("obs2", c_f32p), ("info1", c_f32p), ("info2", c_f32p),
        ("its_first", C.c_int32), ("its_more_outliers", C.c_int32), ("its_more_clean", C.c_int32),
    ]


class Sim3Result(C.Structure):
    _fields_ = [
        ("S12", c_f64p), ("inlier", c_u8p), ("n_in", c_i32p), ("log_stride", C.c_int32),
        ("chi2_log", c_f64p), ("lambda_log", c_f64p), ("trials_log", c_i32p), ("n_iter_done", c_i32p),
    ]


class TriSearchResult(C.Structure):
    _fields_ = [("match12", c_i32p), ("n_matches", c_i32p)]


class LineMatchProblem(C.Structure):
    _fields_ = [
        ("n_pairs", C.c_int32), ("desc_dim", C.c_int32),
        ("left_off", c_i32p), ("right_off", c_i32p),
        ("left_seg", c_f32p), ("left_octave", c_i32p), ("right_seg", c_f32p), ("right_octave", c_i32p),
        ("left_desc", c_f32p), ("right_desc", c_f32p),
        ("K", C.c_double * 9), ("baseline", C.c_double), ("tau", C.c_double), ("min_line_length", C.c_int32),
    ]


class LineMatchResult(C.Structure):
    _fields_ = [("match", c_i32p), ("dist", c_f32p)]


c_i64p = C.POINTER(C.c_int64)
_NP2C[np.dtype(np.int64)] = c_i64p


class StereoProblem(C.Structure):
    _fields_ = [
        ("n_frames", C.c_int32), ("left_off", c_i32p), ("right_off", c_i32p),
        ("left_xy", c_f32p), ("left_octave", c_u8p), ("left_desc", c_u8p),
        ("right_xy", c_f32p), ("right_octave", c_u8p), ("right_desc", c_u8p),
        ("n_levels", C.c_int32), ("scale_factors", c_f32p), ("inv_scale_factors", c_f32p),
        ("pyr", c_u8p), ("pyr_bytes", C.c_int64), ("pyr_off", c_i64p),
        ("pyr_rows", c_i32p), ("pyr_cols", c_i32p), ("pyr_stride", c_i32p),
        ("mb", C.c_float), ("mbf", C.c_float),
    ]


class StereoResult(C.Structure):
    _fields_ = [("uright", c_f32p), ("depth", c_f32p), ("n_matched", c_i32p)]


def fill_struct(struct_cls, fields: Dict[str, Any]):
    """Build a ctypes struct from a dict of numpy arrays / scalars.  Returns (struct, keepalive list)."""
    s = struct_cls()
    keep = []
    for name, ctype in struct_cls._fields_:
        if name not in fields:
            if name == "geom":
                continue
            raise KeyError(f"{struct_cls.__name__}: missing field {name}")
        v = fields[name]
        if v is None:
            continue  # NULL pointer
        if isinstance(ctype, type) and issubclass(ctype, C.Array):
            setattr(s, name, ctype(*[float(x) for x in np.asarray(v).ravel()]))
            continue
        if isinstance(v, np.ndarray):
            want = _NP2C.get(v.dtype)
            if want is not ctype:
                raise TypeError(f"{struct_cls.__name__}.{name}: dtype {v.dtype} does not match {ctype}")
            if not v.flags["C_CONTIGUOUS"]:
                raise ValueError(f"{struct_cls.__name__}.{name}: array must be C-contiguous")
            keep.append(v)
            setattr(s, name, v.ctypes.data_as(ctype))
        elif isinstance(v, C.Structure):
            setattr(s, name, v)
        else:
            setattr(s, name, v)
    return s, keep


def make_geom(g: Dict[str, Any]):
    sf = np.ascontiguousarray(g["scale_factors"], dtype=np.float32)
    geom = FrameGeom(g["fx"], g["fy"], g["cx"], g["cy"], g["bf"], g["b"], g["min_x"], g["max_x"], g["min_y"], g["max_y"],
                     int(sf.shape[0]), sf.ctypes.data_as(c_f32p))
    return geom, sf


class _Lib:
    """Thin wrapper binding argtypes for one of the two libraries (prefix 'lld_' or 'lldo_')."""

    def __init__(self, path: str, prefix: str):
        if not os.path.exists(path):
            raise RuntimeError(
                f"{path} not found — build it first (python -c 'import __graft_entry__ as g; g.build()'). "
                "There is no fallback implementation.")
        self.path = path
        self.prefix = prefix
        self.dll = C.CDLL(path)
        self.is_oracle = prefix == "lldo_"
        d = self.dll
        vp = C.c_void_p
        self._sig("ba_local", [vp, C.POINTER(BaProblem), C.c_int, C.c_int, c_u8p, C.POINTER(BaResult)])
        self._sig("ba_global", [vp, C.POINTER(BaProblem), C.c_int, c_u8p, C.POINTER(BaResult)])
        self._sig("pose_opt", [vp, C.POINTER(PoseProblem), C.POINTER(PoseResult)])
        self._sig("sbp_frame", [vp, C.POINTER(SbpFrameProblem), C.POINTER(SbpResult)])
        self._sig("sbp_mappoints", [vp, C.POINTER(SbpMpProblem), C.POINTER(SbpResult)])
        self._sig("kf_search", [vp, C.POINTER(KfSearchProblem), C.POINTER(SbpResult)])
        self._sig("tri_search", [vp, C.POINTER(TriSearchProblem), C.POINTER(TriSearchResult)])
        self._sig("bow_search", [vp, C.POINTER(BowSearchProblem), C.POINTER(TriSearchResult)])
        init_sig = [vp, C.POINTER(InitSearchProblem), C.POINTER(InitSearchResult)]
        if self.is_oracle:
            if not os.path.exists(INIT_SEARCH_ORACLE_PATH):
                raise RuntimeError(f"{INIT_SEARCH_ORACLE_PATH} not found — build it first (python -c 'import __graft_entry__ as g; g.build()').")
            self.init_dll = C.CDLL(INIT_SEARCH_ORACLE_PATH)
            self.init_search = self.init_dll.lldo_init_search
            self.init_search.argtypes = init_sig
            self.init_search.restype = C.c_int
        else:
            self._sig("init_search", init_sig)
        sim3_sig = [vp, C.POINTER(Sim3Problem), C.POINTER(Sim3Result)]
        if self.is_oracle:
            if not os.path.exists(SIM3_ORACLE_PATH):
                raise RuntimeError(f"{SIM3_ORACLE_PATH} not found — build it first (python -c 'import __graft_entry__ as g; g.build()').")
            self.sim3_dll = C.CDLL(SIM3_ORACLE_PATH)
            self.sim3_opt = self.sim3_dll.lldo_sim3_opt
            self.sim3_opt.argtypes = sim3_sig
            self.sim3_opt.restype = C.c_int
        else:
            self._sig("sim3_opt", sim3_sig)
        self._sig("line_match", [vp, C.POINTER(LineMatchProblem), C.POINTER(LineMatchResult)])
        self._sig("descriptor_distance", [c_u8p, c_u8p])
        if not self.is_oracle:
            d.lld_ctx_create.argtypes = [C.c_int, C.POINTER(vp)]
            d.lld_ctx_create.restype = C.c_int
            d.lld_ctx_destroy.argtypes = [vp]
            d.lld_ctx_destroy.restype = None
            d.lld_ctx_last_error.argtypes = [vp]
            d.lld_ctx_last_error.restype = C.c_char_p
            d.lld_version.restype = C.c_char_p
            d.lld_ctx_launch_count.argtypes = [vp]
            d.lld_ctx_launch_count.restype = C.c_int64
            d.lld_ctx_last_timing.argtypes = [vp, c_f32p, c_f32p, c_f32p]
            d.lld_ctx_last_timing.restype = None
            d.lld_comm_unique_id.argtypes = [c_u8p]
            d.lld_comm_unique_id.restype = C.c_int
            d.lld_comm_init.argtypes = [vp, C.c_int, C.c_int, c_u8p]
            d.lld_comm_init.restype = C.c_int
            d.lld_ba_shard_bounds.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_int32, c_i32p]
            d.lld_ba_shard_bounds.restype = None
            d.lld_stereo_matches.argtypes = [vp, C.POINTER(StereoProblem), C.POINTER(StereoResult)]
            d.lld_stereo_matches.restype = C.c_int
            d.lld_ctx_set_topo_cache.argtypes = [vp, C.c_int]
            d.lld_ctx_set_topo_cache.restype = None
            d.lld_ctx_set_gba_sparse.argtypes = [vp, C.c_int]
            d.lld_ctx_set_gba_sparse.restype = None
            d.lld_gba_sparse_plan_report.argtypes = [C.POINTER(BaProblem), C.c_char_p, C.c_int]
            d.lld_gba_sparse_plan_report.restype = C.c_int
            d.lld_ctx_nccl_stats.argtypes = [vp, c_i64p, c_i64p]
            d.lld_ctx_nccl_stats.restype = None

    def _sig(self, name, argtypes):
        f = getattr(self.dll, self.prefix + name)
        f.argtypes = argtypes
        f.restype = C.c_int
        setattr(self, name, f)


_libs: Dict[str, _Lib] = {}


def load_library() -> _Lib:
    if "gpu" not in _libs:
        _libs["gpu"] = _Lib(LIB_PATH, "lld_")
    return _libs["gpu"]


def load_oracle() -> _Lib:
    if "oracle" not in _libs:
        _libs["oracle"] = _Lib(ORACLE_PATH, "lldo_")
    return _libs["oracle"]


class Context:
    """One CUDA stream + workspace (lld_ctx_create).  One per calling thread."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        self.handle = C.c_void_p()
        rc = self.lib.dll.lld_ctx_create(device, C.byref(self.handle))
        if rc != 0:
            raise RuntimeError(f"lld_ctx_create(device={device}) failed with {rc}: no usable CUDA device (no CPU fallback)")

    def check(self, rc: int, what: str):
        if rc != 0:
            msg = self.lib.dll.lld_ctx_last_error(self.handle)
            raise RuntimeError(f"{what} failed with {rc}: {msg.decode() if msg else ''}")

    def launch_count(self) -> int:
        return int(self.lib.dll.lld_ctx_launch_count(self.handle))

    def last_timing(self):
        a, b, c = C.c_float(), C.c_float(), C.c_float()
        self.lib.dll.lld_ctx_last_timing(self.handle, C.byref(a), C.byref(b), C.byref(c))
        return a.value, b.value, c.value

    def close(self):
        if self.handle:
            self.lib.dll.lld_ctx_destroy(self.handle)
            self.handle = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
