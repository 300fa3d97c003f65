"""ORBmatcher::SearchForInitialization (lld_init_search): an independent Python transcription pins the CPU oracle, small hand-built
frame pairs pin each rule of the sequential search (a later query taking an F2 keypoint away, the vMatchedDistance skip, ties,
the histogram counting displaced matches, the bin-30 wrap, windows clipped or outside the image, keypoints outside the grid,
tiny pairs, F1 keypoints above level 0), and the GPU is bit-exact against the oracle on match12, n_matches and prev_matched,
on both resolve arms (F2 state in shared memory / in global memory, told apart by the per-launch profile)."""
import ctypes as C
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import shim_io  # noqa: E402
from lld_slam_b200 import api, synth  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
f32 = np.float32
POP = np.array([bin(i).count("1") for i in range(256)], np.int64)
INT_MAX = 2**31 - 1
SMEM_MAX_KP = 57088   # largest F2 whose resolve state stays in shared memory (include/lldba.h)


# ------------------------------------------------------------------------------------------------------------------
# plain-Python transcription of the listing (float32 arithmetic, own grid, lists for the histogram)
# ------------------------------------------------------------------------------------------------------------------
def _round(v):
    """std::round: half away from zero"""
    return int(math.copysign(math.floor(abs(float(v)) + 0.5), float(v)))


def _three_max(sizes):
    max1 = max2 = max3 = 0
    i1 = i2 = i3 = -1
    for i, s in enumerate(sizes):
        if s > max1:
            max3, max2, max1, i3, i2, i1 = max2, max1, s, i2, i1, i
        elif s > max2:
            max3, max2, i3, i2 = max2, s, i2, i
        elif s > max3:
            max3, i3 = s, i
    if max2 < f32(0.1) * f32(max1):
        i2 = i3 = -1
    elif max3 < f32(0.1) * f32(max1):
        i3 = -1
    return i1, i2, i3


def _init_search_python(p, stats=None):
    g = p["geom"]
    minx, miny = f32(g["min_x"]), f32(g["min_y"])
    winv = f32(64) / (f32(g["max_x"]) - minx)
    hinv = f32(48) / (f32(g["max_y"]) - miny)
    r = f32(p["window_size"])
    ratio = f32(p["nn_ratio"])
    factor = f32(1.0) / f32(30)
    n1t = int(p["kp1_off"][-1])
    m12_all = np.full(n1t, -1, np.int32)
    prev_all = p["prev_matched"].astype(f32).copy()
    nm_all = np.zeros(int(p["n_pairs"]), np.int32)
    for pr in range(int(p["n_pairs"])):
        a0, a1 = int(p["kp1_off"][pr]), int(p["kp1_off"][pr + 1])
        b0, b1 = int(p["kp2_off"][pr]), int(p["kp2_off"][pr + 1])
        xy2 = p["kp2_xy"][b0:b1]
        oct2 = p["kp2_octave"][b0:b1]
        grid = {}
        for i in range(b1 - b0):   # Frame::AssignFeaturesToGrid / PosInGrid
            px = _round(f32(xy2[i, 0] - minx) * winv)
            py = _round(f32(xy2[i, 1] - miny) * hinv)
            if 0 <= px < 64 and 0 <= py < 48:
                grid.setdefault((px, py), []).append(i)
        n1 = a1 - a0
        m12 = [-1] * n1
        mdist = [INT_MAX] * (b1 - b0)
        m21 = [-1] * (b1 - b0)
        hist = [[] for _ in range(30)]
        prev = prev_all[a0:a1]
        nm = 0
        for i1 in range(n1):
            if p["kp1_octave"][a0 + i1] > 0:
                continue
            x, y = f32(prev[i1, 0]), f32(prev[i1, 1])
            cx0 = max(0, math.floor(f32(f32(x - minx) - r) * winv))
            cx1 = min(63, math.ceil(f32(f32(x - minx) + r) * winv))
            cy0 = max(0, math.floor(f32(f32(y - miny) - r) * hinv))
            cy1 = min(47, math.ceil(f32(f32(y - miny) + r) * hinv))
            cand = []
            if cx0 < 64 and cx1 >= 0 and cy0 < 48 and cy1 >= 0:
                for ix in range(cx0, cx1 + 1):
                    for iy in range(cy0, cy1 + 1):
                        for i2 in grid.get((ix, iy), []):
                            if oct2[i2] != 0:
                                continue
                            if abs(f32(xy2[i2, 0] - x)) < r and abs(f32(xy2[i2, 1] - y)) < r:
                                cand.append(i2)
            d1 = p["kp1_desc"][a0 + i1]
            best, best2, bidx = INT_MAX, INT_MAX, -1
            for i2 in cand:
                dist = int(POP[d1 ^ p["kp2_desc"][b0 + i2]].sum())
                if mdist[i2] <= dist:
                    continue
                if dist < best:
                    best2, best, bidx = best, dist, i2
                elif dist < best2:
                    best2 = dist
            if best <= 50 and f32(best) < f32(best2) * ratio:
                if m21[bidx] >= 0:
                    m12[m21[bidx]] = -1
                    nm -= 1
                    if stats is not None:
                        stats["displaced"] = stats.get("displaced", 0) + 1
                m12[i1] = bidx
                m21[bidx] = i1
                mdist[bidx] = best
                nm += 1
                if p["check_orientation"]:
                    rot = f32(p["kp1_angle"][a0 + i1]) - f32(p["kp2_angle"][b0 + bidx])
                    if rot < 0:
                        rot = rot + f32(360)
                    b = _round(f32(rot * factor))
                    hist[0 if b == 30 else b].append(i1)
        if p["check_orientation"]:
            keep = _three_max([len(h) for h in hist])
            for b in range(30):
                if b in keep:
                    continue
                for i1 in hist[b]:
                    if m12[i1] >= 0:
                        m12[i1] = -1
                        nm -= 1
                        if stats is not None:
                            stats["rot_removed"] = stats.get("rot_removed", 0) + 1
        for i1 in range(n1):
            if m12[i1] >= 0:
                prev[i1] = xy2[m12[i1]]
        m12_all[a0:a1] = m12
        nm_all[pr] = nm
    return dict(match12=m12_all, n_matches=nm_all, prev_matched=prev_all)


def _same(a, b):
    return (np.array_equal(a["match12"], b["match12"]) and np.array_equal(a["n_matches"], b["n_matches"])
            and np.array_equal(np.asarray(a["prev_matched"]).view(np.uint32), np.asarray(b["prev_matched"]).view(np.uint32)))


# ------------------------------------------------------------------------------------------------------------------
# hand-built frame pairs
# ------------------------------------------------------------------------------------------------------------------
_RNG = np.random.default_rng(2024)
_BASE = _RNG.integers(0, 256, (64, 32), dtype=np.uint8)


def _flip(d, n, first=0):
    """d with bits [first, first + n) flipped: Hamming distance n to d"""
    bits = np.unpackbits(d.copy())
    bits[first:first + n] ^= 1
    return np.packbits(bits)


def _pair(f1, f2, window=20, nn_ratio=0.9, ori=1):
    """f1: (prev x, prev y, octave, angle, desc); f2: (x, y, octave, angle, desc) -> one-pair problem"""
    g = synth.frame_geom()
    return dict(
        n_pairs=1, geom=g, window_size=window, nn_ratio=nn_ratio, check_orientation=ori,
        kp1_off=np.array([0, len(f1)], np.int32), kp2_off=np.array([0, len(f2)], np.int32),
        kp1_octave=np.array([k[2] for k in f1], np.uint8), kp1_angle=np.array([k[3] for k in f1], f32),
        kp1_desc=np.ascontiguousarray(np.array([k[4] for k in f1], np.uint8).reshape(-1, 32)),
        prev_matched=np.ascontiguousarray(np.array([k[:2] for k in f1], f32).reshape(-1, 2)),
        kp2_xy=np.ascontiguousarray(np.array([k[:2] for k in f2], f32).reshape(-1, 2)),
        kp2_octave=np.array([k[2] for k in f2], np.uint8), kp2_angle=np.array([k[3] for k in f2], f32),
        kp2_desc=np.ascontiguousarray(np.array([k[4] for k in f2], np.uint8).reshape(-1, 32)))


def _concat(parts):
    out = dict(parts[0])
    out["n_pairs"] = sum(int(q["n_pairs"]) for q in parts)
    for off, keys in (("kp1_off", ("kp1_octave", "kp1_angle", "kp1_desc", "prev_matched")),
                      ("kp2_off", ("kp2_xy", "kp2_octave", "kp2_angle", "kp2_desc"))):
        offs, base = [np.zeros(1, np.int32)], 0
        for q in parts:
            offs.append((q[off][1:] + base).astype(np.int32))
            base += int(q[off][-1])
        out[off] = np.concatenate(offs)
        for k in keys:
            out[k] = np.ascontiguousarray(np.concatenate([q[k] for q in parts], 0))
    return out


def _case_displacement():
    B = _BASE[0]
    p = _pair([(300, 100, 0, 0, _flip(B, 20)), (305, 100, 0, 0, _flip(B, 10))], [(300, 100, 0, 0, B)])
    return p, dict(match12=[-1, 0], n_matches=[1], prev_matched=[[300, 100], [300, 100]])


def _case_skip_flips_ratio():
    B0 = _BASE[1]
    q1 = _flip(B0, 20)
    k1 = _flip(q1, 21, 100)       # d(q1, k1) = 21, d(q0, k1) = 31
    p = _pair([(300, 100, 0, 0, _flip(B0, 10)), (305, 100, 0, 0, q1)], [(300, 100, 0, 0, B0), (310, 100, 0, 0, k1)])
    # without the skip, q1 would see best 20 (k0) / second 21 and fail the ratio test
    return p, dict(match12=[0, 1], n_matches=[2], prev_matched=[[300, 100], [310, 100]])


def _case_tie_by_traversal():
    Q, Q2 = _BASE[2], _BASE[3]
    f1 = [(320, 100, 0, 0, Q), (600, 200, 0, 0, Q2)]
    # equal distances: column 16 (x = 310) comes before column 17 (x = 330) whatever the indices; inside one cell insertion order
    f2 = [(330, 100, 0, 0, _flip(Q, 15, 0)), (310, 100, 0, 0, _flip(Q, 15, 50)),
          (600, 200, 0, 0, _flip(Q2, 12, 0)), (601, 200, 0, 0, _flip(Q2, 12, 80))]
    p = _pair(f1, f2, nn_ratio=1.5)
    return p, dict(match12=[1, 2], n_matches=[2], prev_matched=[[310, 100], [600, 200]])


def _case_displaced_entry_in_histogram():
    f1, f2, exp = [], [], []
    angles = [1.0, 1.0, 1.0, 30.0, 30.0, 60.0]   # bins 0, 0, 0, 1, 1, 2
    for j, a in enumerate(angles):
        x = 60 + 70 * j
        f2.append((x, 100, 0, 0.0, _BASE[10 + j]))
        f1.append((x, 100, 0, a, _flip(_BASE[10 + j], 5)))
        exp.append(j)
    Bx = _BASE[20]
    f2.append((700, 100, 0, 0.0, Bx))
    f1.append((700, 100, 0, 90.0, _flip(Bx, 20)))   # bin 3, displaced below: still counted
    f1.append((702, 100, 0, 91.0, _flip(Bx, 10)))   # bin 3, takes Bx
    # sizes with the displaced entry: [3, 2, 1, 2] -> bins 0, 1, 3 survive, the bin-2 match goes
    exp[5] = -1
    exp += [-1, 6]
    prev = [[k[0], k[1]] for k in f1]
    for i, m in enumerate(exp):
        if m >= 0:
            prev[i] = list(f2[m][:2])
    return _pair(f1, f2), dict(match12=exp, n_matches=[6], prev_matched=prev)


def _case_bin30_wraps():
    f1, f2 = [], []
    angles = [2.0] * 3 + [899.0] + [150.0] * 4 + [180.0] * 4 + [210.0] * 4   # 899 -> round(29.97) = 30 -> bin 0
    for j, a in enumerate(angles):
        x, y = 60 + 140 * (j % 8), 80 + 180 * (j // 8)
        f2.append((x, y, 0, 0.0, _BASE[30 + j]))
        f1.append((x, y, 0, a, _flip(_BASE[30 + j], 3)))
    # bin 0 holds 4 only through the wrap; ties keep the earlier bins: 0, 5, 6 survive, bin 7 goes
    exp = list(range(12)) + [-1] * 4
    prev = [list(f2[j][:2]) if exp[j] >= 0 else [f1[j][0], f1[j][1]] for j in range(16)]
    return _pair(f1, f2), dict(match12=exp, n_matches=[12], prev_matched=prev)


def _case_window_outside_image():
    K = _BASE[4:7]
    f2 = [(20, 150, 0, 0, K[0]), (1230, 150, 0, 0, K[1]), (600, 200, 0, 0, K[2])]
    f1 = [(-50, 150, 0, 0, _flip(K[0], 5)),      # window clipped at the left edge
          (1300, 150, 0, 0, _flip(K[1], 5)),     # clipped at the right edge
          (-500, -500, 0, 0, K[2]),              # entirely outside: no candidates
          (600, 600, 0, 0, K[2])]                # below the image
    p = _pair(f1, f2, window=100)
    return p, dict(match12=[0, 1, -1, -1], n_matches=[2], prev_matched=[[20, 150], [1230, 150], [-500, -500], [600, 600]])


def _case_keypoints_outside_grid():
    Q, Q2 = _BASE[7], _BASE[8]
    f2 = [(-20, 100, 0, 0, Q), (30, 100, 0, 0, _flip(Q, 30)),          # x = -20: PosInGrid column -1
          (1236, 100, 0, 0, Q2), (1200, 100, 0, 0, _flip(Q2, 25))]      # x = 1236: column round(63.74) = 64, outside too
    f1 = [(10, 100, 0, 0, Q), (1236, 100, 0, 0, Q2)]
    p = _pair(f1, f2, window=50)
    return p, dict(match12=[1, 3], n_matches=[2], prev_matched=[[30, 100], [1200, 100]])


def _case_tiny_pairs():
    Q = _BASE[9]
    parts = [_pair([], []), _pair([(100, 100, 0, 0, Q)], []), _pair([], [(100, 100, 0, 0, Q)]),
             _pair([(100, 100, 0, 0, Q)], [(104, 98, 0, 0, _flip(Q, 7))])]
    return _concat(parts), dict(match12=[-1, 0], n_matches=[0, 0, 0, 1], prev_matched=[[100, 100], [104, 98]])


def _case_upper_levels():
    Q, Q2 = _BASE[11], _BASE[12]
    f2 = [(200, 100, 0, 0, Q), (500, 100, 2, 0, Q2), (505, 100, 0, 0, _flip(Q2, 40))]
    f1 = [(200, 100, 1, 0, Q),      # F1 keypoint above level 0: skipped
          (500, 100, 0, 0, Q2)]     # its exact twin in F2 sits at level 2: not a candidate
    p = _pair(f1, f2)
    return p, dict(match12=[-1, 2], n_matches=[1], prev_matched=[[200, 100], [505, 100]])


CASES = {
    "displacement": _case_displacement, "skip_flips_ratio": _case_skip_flips_ratio, "tie_by_traversal": _case_tie_by_traversal,
    "displaced_entry_in_histogram": _case_displaced_entry_in_histogram, "bin30_wraps": _case_bin30_wraps,
    "window_outside_image": _case_window_outside_image, "keypoints_outside_grid": _case_keypoints_outside_grid,
    "tiny_pairs": _case_tiny_pairs, "upper_levels": _case_upper_levels,
}


def _global_arm_pad(p):
    """the same problem plus one pair whose F2 is too large for the shared-memory state: the batch takes the global arm"""
    rng = np.random.default_rng(77)
    n = SMEM_MAX_KP + 1
    g = synth.frame_geom()
    pad = _pair([], [])
    pad["kp2_off"] = np.array([0, n], np.int32)
    pad["kp2_xy"] = np.ascontiguousarray(np.stack([rng.uniform(0, g["max_x"], n), rng.uniform(0, g["max_y"], n)], 1).astype(f32))
    pad["kp2_octave"] = rng.integers(0, 8, n).astype(np.uint8)
    pad["kp2_angle"] = rng.uniform(0, 360, n).astype(f32)
    pad["kp2_desc"] = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    return _concat([p, pad])


# ------------------------------------------------------------------------------------------------------------------
# CPU: the oracle against the transcription
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("window", [50, 100, 200])
@pytest.mark.parametrize("ori", [0, 1])
@pytest.mark.parametrize("seed", [3, 4, 5])
def test_oracle_init_search_against_python(built, seed, ori, window):
    p = synth.make_init_search_batch(2, 500, seed, window_size=window, check_orientation=ori)
    stats = {}
    r = _init_search_python(p, stats)
    o = api.init_search(p, impl="oracle")
    assert _same(o, r)
    assert r["n_matches"].sum() > 50
    if window >= 100:
        assert stats.get("displaced", 0) > 0          # later queries take keypoints away
    if ori:
        assert stats.get("rot_removed", 0) > 0        # the rotated outliers are filtered


@pytest.mark.parametrize("name", sorted(CASES))
def test_hand_built_case_oracle_and_python(built, name):
    p, exp = CASES[name]()
    o = api.init_search(p, impl="oracle")
    r = _init_search_python(p)
    assert _same(o, r)
    assert o["match12"].tolist() == exp["match12"]
    assert o["n_matches"].tolist() == exp["n_matches"]
    assert np.array_equal(o["prev_matched"], np.asarray(exp["prev_matched"], f32).reshape(-1, 2))


def test_generator_shapes_and_ranges():
    p = synth.make_init_search_batch(3, [0, 1, 40], 9)
    assert p["kp1_off"].tolist() == [0, 0, 1, 41] and p["kp2_off"].tolist() == [0, 0, 1, 41]
    for k in ("kp1_angle", "kp2_angle"):
        assert p[k].dtype == f32 and (p[k] >= 0).all() and (p[k] < 360).all()
    assert p["kp1_desc"].shape == (41, 32) and p["prev_matched"].shape == (41, 2)


# ------------------------------------------------------------------------------------------------------------------
# shim
# ------------------------------------------------------------------------------------------------------------------
def _shim_build(tmp_path, oracle):
    src = os.path.join(ROOT, "tests", "hostcheck", "shim_init_search.cpp")
    exe = str(tmp_path / ("shim_init_oracle" if oracle else "shim_init_gpu"))
    if oracle:
        libdir, lib, extra = os.path.join(ROOT, "tests", "hostcheck"), "init_search_oracle", ["-DLLD_SHIM_ORACLE"]
    else:
        libdir, lib, extra = os.path.join(ROOT, "lld_slam_b200", "csrc"), "lldba", []
    r = subprocess.run(["g++", "-std=c++14", "-O1", "-Wall", *extra, src, "-o", exe, f"-L{libdir}", f"-l{lib}", f"-Wl,-rpath,{libdir}"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout
    return exe


def _check_shim(exe, tmp_path, impl, ctx=None):
    """two calls, as Tracking::MonocularInitialization makes them: the second takes vbPrevMatched from the first and a new F2"""
    p = synth.make_init_search_batch(1, 1500, 31)
    nxt = (p["kp2_xy"] + f32(6.0)).astype(f32)
    g = p["geom"]
    d = dict(bounds=np.array([g["min_x"], g["max_x"], g["min_y"], g["max_y"]], f32), scale_factors=np.asarray(g["scale_factors"], f32),
             config=np.array([p["window_size"], p["nn_ratio"], p["check_orientation"]], f32),
             kp1_octave=p["kp1_octave"], kp1_angle=p["kp1_angle"], kp1_desc=p["kp1_desc"], prev_matched=p["prev_matched"],
             kp2_xy=p["kp2_xy"], kp2_xy_next=nxt, kp2_octave=p["kp2_octave"], kp2_angle=p["kp2_angle"], kp2_desc=p["kp2_desc"])
    fin, fout = str(tmp_path / "init_in.bin"), str(tmp_path / "init_out.bin")
    shim_io.write(fin, d)
    r = subprocess.run([exe, fin, fout], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout
    got = shim_io.read(fout)
    ref0 = api.init_search(p, impl=impl, ctx=ctx)
    q = dict(p); q["prev_matched"] = ref0["prev_matched"]; q["kp2_xy"] = nxt
    ref1 = api.init_search(q, impl=impl, ctx=ctx)
    assert got["n_matches"].tolist() == [int(ref0["n_matches"][0]), int(ref1["n_matches"][0])] and ref0["n_matches"][0] > 100
    assert np.array_equal(got["match12_0"], ref0["match12"]) and np.array_equal(got["match12_1"], ref1["match12"])
    assert np.array_equal(got["prev_0"], ref0["prev_matched"].reshape(-1)) and np.array_equal(got["prev_1"], ref1["prev_matched"].reshape(-1))


def test_shim_search_for_initialization_on_host(built, tmp_path):
    _check_shim(_shim_build(tmp_path, True), tmp_path, "oracle")


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
def _profiled(p, ctx):
    d = ctx.lib.dll
    d.lld_ctx_profile.argtypes = [C.c_void_p, C.c_int]; d.lld_ctx_profile.restype = None
    d.lld_ctx_profile_report.argtypes = [C.c_void_p, C.c_char_p, C.c_int]; d.lld_ctx_profile_report.restype = C.c_int
    d.lld_ctx_profile(ctx.handle, 1)
    try:
        out = api.init_search(p, impl="gpu", ctx=ctx)
        buf = C.create_string_buffer(1 << 16)
        ctx.check(d.lld_ctx_profile_report(ctx.handle, buf, len(buf)), "lld_ctx_profile_report")
    finally:
        d.lld_ctx_profile(ctx.handle, 0)
    return out, set(json.loads(buf.value.decode()))


def _check_gpu(p, ctx, arm):
    g, names = _profiled(p, ctx)
    assert f"k_init_resolve_{arm}" in names and f"k_init_resolve_{'global' if arm == 'smem' else 'smem'}" not in names, names
    assert {"k_init_count", "k_init_scan", "k_init_fill", "k_init_finalize"} <= names
    o = api.init_search(p, impl="oracle")
    assert _same(g, o)
    assert _same(api.init_search(p, impl="gpu", ctx=ctx), g)     # unprofiled run: the same bits
    return g


@pytest.mark.gpu
@pytest.mark.parametrize("ori", [0, 1])
def test_gpu_init_search_kitti_batch(gpu_ctx, ori):
    p = synth.make_init_search_batch(256, 2000, 41, check_orientation=ori)
    g = _check_gpu(p, gpu_ctx, "smem")
    assert g["n_matches"].min() > 100


@pytest.mark.gpu
@pytest.mark.parametrize("arm", ["smem", "global"])
def test_gpu_init_search_ragged(gpu_ctx, arm):
    p = synth.make_init_search_batch(4, [0, 1, 37, 3000], 43)
    _check_gpu(p if arm == "smem" else _global_arm_pad(p), gpu_ctx, arm)


@pytest.mark.gpu
def test_gpu_init_search_large_frame_global_arm(gpu_ctx):
    p = synth.make_init_search_batch(1, 2000, 47, n_kp2=60000, window_size=50)
    _check_gpu(p, gpu_ctx, "global")


@pytest.mark.gpu
@pytest.mark.parametrize("arm", ["smem", "global"])
def test_gpu_init_search_two_call_chain(gpu_ctx, arm):
    p = synth.make_init_search_batch(16, 2000, 53)
    rng = np.random.default_rng(5)
    g0 = _check_gpu(p if arm == "smem" else _global_arm_pad(p), gpu_ctx, arm)
    q = dict(p)
    n1 = int(p["kp1_off"][-1])
    q["prev_matched"] = np.ascontiguousarray(g0["prev_matched"][:n1])
    q["kp2_xy"] = np.ascontiguousarray((p["kp2_xy"] + rng.normal(4.0, 1.0, p["kp2_xy"].shape)).astype(f32))
    g1 = _check_gpu(q if arm == "smem" else _global_arm_pad(q), gpu_ctx, arm)
    assert (g1["match12"][:n1] >= 0).sum() > 100


@pytest.mark.gpu
@pytest.mark.parametrize("arm", ["smem", "global"])
@pytest.mark.parametrize("name", sorted(CASES))
def test_gpu_init_search_hand_built_case(gpu_ctx, name, arm):
    p, exp = CASES[name]()
    g = _check_gpu(p if arm == "smem" else _global_arm_pad(p), gpu_ctx, arm)
    n1 = int(p["kp1_off"][-1])
    assert g["match12"][:n1].tolist() == exp["match12"]


@pytest.mark.gpu
def test_gpu_init_search_repeatable(gpu_ctx):
    p = synth.make_init_search_batch(64, 2000, 59)
    a = api.init_search(p, impl="gpu", ctx=gpu_ctx)
    b = api.init_search(p, impl="gpu", ctx=gpu_ctx)
    assert _same(a, b)


@pytest.mark.gpu
def test_gpu_init_search_prev_matched_in_place(gpu_ctx):
    """the result's prev_matched may be the problem's own array"""
    from lld_slam_b200 import capi
    p = synth.make_init_search_batch(8, 1000, 61)
    ref = api.init_search(p, impl="gpu", ctx=gpu_ctx)
    f = dict(p)
    geom, gk = capi.make_geom(p["geom"])
    f["geom"] = geom
    f["prev_matched"] = p["prev_matched"].copy()
    prob, keep = capi.fill_struct(capi.InitSearchProblem, f)
    out = dict(match12=np.full(int(p["kp1_off"][-1]), -2, np.int32), n_matches=np.zeros(8, np.int32), prev_matched=f["prev_matched"])
    res, keep2 = capi.fill_struct(capi.InitSearchResult, out)
    gpu_ctx.check(gpu_ctx.lib.init_search(gpu_ctx.handle, C.byref(prob), C.byref(res)), "lld_init_search")
    assert _same(out, ref)


@pytest.mark.gpu
def test_gpu_shim_search_for_initialization(gpu_ctx, tmp_path):
    _check_shim(_shim_build(tmp_path, False), tmp_path, "gpu", gpu_ctx)
