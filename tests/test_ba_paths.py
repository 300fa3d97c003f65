"""Every dispatch arm of local and global bundle adjustment against the CPU oracle.

`ba.cu` picks kernels and solvers from the shape of the problem: the cyclic-reduction solve (`k_cr_solve<15>` up to a
super-block of m = 120 scalars, `<20>` up to CR_MAX_M = 156), the single-CTA skyline LDL^T (`k_solve_env`, global BA
whose block half-bandwidth B is 27 or more), local sparse mode (more than 32 free keyframes in a window, or a landmark
seen twice by one free keyframe), the 1024-thread Schur rows, the sliced reductions of windows with 32k landmarks, the
lanes per line, the step schedules and the topology cache.  The windows of `synth.make_ba_window` reach only a few of
these, so the generators below build shapes that reach the others.

Each GPU case compares with the oracle through `check_ba` (the tolerances of test_gpu_parity.py) and proves that it ran
the arm it is named after: kernel names from the per-launch profile (`lld_ctx_profile`), the exact host-to-device byte
count of a topology-cache hit (`lld_ctx_last_bytes`), or the error code and message.  The shape claims each case rests
on (B, super-block count, neighbour counts, landmarks per window) are computed in numpy and asserted by CPU tests, so
that a generator change that moves a case off its arm fails without a GPU.
"""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from lld_slam_b200 import api, capi, synth
from test_gpu_parity import check_ba

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CR_MAX_M = 156            # cr_solver.cuh
SMEM_LIMIT = 220 * 1024   # ba.cu: dynamic shared memory the single-CTA global solvers may ask for
ERR_ARG, ERR_UNSUPPORTED = -2, -4


# ------------------------------------------------------------------------------------------------------------------
# generators
# ------------------------------------------------------------------------------------------------------------------
def _select(w, pt_keep, ln_keep, min_obs=2):
    """keep the selected observations of a window; landmarks left with fewer than min_obs observations are dropped"""
    w = dict(w)
    for pre, lm_key, obs_keys, keep in (("pt", "pt_xyz", ("pt_obs_kf", "pt_obs_uvr", "pt_obs_info"), pt_keep),
                                        ("ln", "ln_x0_dir", ("ln_obs_kf", "ln_obs_left", "ln_obs_right", "ln_obs_info", "ln_obs_stereo"), ln_keep)):
        off = w[f"{pre}_obs_off"]
        n_lm = len(off) - 1
        lm = np.repeat(np.arange(n_lm), np.diff(off))
        cnt = np.bincount(lm[keep], minlength=n_lm)
        lm_keep = cnt >= min_obs
        obs_keep = keep & lm_keep[lm]
        w[lm_key] = np.ascontiguousarray(w[lm_key][lm_keep])
        for k in obs_keys:
            w[k] = np.ascontiguousarray(w[k][obs_keep])
        w[f"{pre}_obs_off"] = synth._csr(cnt[lm_keep])
        w[f"n_{pre}"] = int(lm_keep.sum())
    return w


def _trim_tracks(w, B):
    """cut every track to the keyframes at most B after its first observation"""
    keep = []
    for pre in ("pt", "ln"):
        off, kf = w[f"{pre}_obs_off"], w[f"{pre}_obs_kf"]
        first = np.repeat(kf[off[:-1]], np.diff(off))
        keep.append(kf - first <= B)
    return _select(w, keep[0], keep[1])


def _truth_cam(w, k):
    T = w["truth"]["kf_Tcw"][k]
    return T[:9].reshape(3, 3), T[9:]


def _observe(w, X, k, rng, global_mode):
    """one point observation of X in keyframe k: true projection + pyramid-level noise, stereo when close enough"""
    R, t = _truth_cam(w, k)
    u, v, z, _ = synth._project(R, t, X)
    assert z > 0.5 and 0 <= u < synth.IMG_W and 0 <= v < synth.IMG_H, (k, u, v, z)
    octave = int(rng.integers(0, 4 if global_mode else synth.N_LEVELS))
    sig = synth.SCALE ** octave
    u = u + rng.normal() * sig
    v = v + rng.normal() * sig
    baseline = float(np.float32(synth.BF) / np.float32(synth.FX))
    ur = max(u - synth.BF / z + rng.normal() * sig, 0.0) if z < synth.TH_DEPTH * baseline else -1.0
    inv = synth.inv_level_sigma2()
    info = inv[octave * 2] if global_mode else inv[octave]   # GBA quirk of make_ba_window: mvInvLevelSigma2[octave * 2]
    return (u, v, ur), info


def add_points(w, kf_lists, rng, global_mode, ahead=6.0, side=(3.0, -1.0)):
    """append one map point per keyframe list, observed by every keyframe of the list.  The trajectory moves 1 m per
    keyframe along +z, so a point `ahead` metres in front of the last keyframe (a few metres off the optical axis) projects
    into all earlier ones."""
    w = dict(w)
    xyz, off, okf, uvr, info = [w["pt_xyz"]], list(w["pt_obs_off"]), [w["pt_obs_kf"]], [w["pt_obs_uvr"]], [w["pt_obs_info"]]
    for kfs in kf_lists:
        R, t = _truth_cam(w, kfs[-1])
        X = R.T @ (np.array([side[0], side[1], ahead]) - t)
        obs = [_observe(w, X, int(k), rng, global_mode) for k in kfs]
        xyz.append((X + rng.normal(0, 0.02, 3)).astype(np.float32).astype(np.float64)[None])
        off.append(off[-1] + len(kfs))
        okf.append(np.asarray(kfs, np.int32))
        uvr.append(synth.f32([o[0] for o in obs]))
        info.append(synth.f32([o[1] for o in obs]))
    w["pt_xyz"] = np.ascontiguousarray(np.concatenate(xyz))
    w["pt_obs_off"] = np.asarray(off, np.int32)
    w["pt_obs_kf"] = np.ascontiguousarray(np.concatenate(okf))
    w["pt_obs_uvr"] = np.ascontiguousarray(np.concatenate(uvr))
    w["pt_obs_info"] = np.ascontiguousarray(np.concatenate(info))
    w["n_pt"] = len(w["pt_xyz"])
    return w


def free_kfs(w):
    return np.nonzero(w["kf_fixed"] == 0)[0]


def banded_global(n_kf, B, n_pt, n_ln, seed, *, fixed=(), n_long=2, robust=False):
    """a global BA problem whose block half-bandwidth (largest free-keyframe span of one landmark) is exactly B: the tracks of
    make_ba_window(global_mode=True) cut to B keyframes after their first observation, plus n_long points seen by B + 1
    consecutive free keyframes.  `fixed` lists interior keyframes that are held fixed (free indices skip them)."""
    rng = np.random.default_rng(seed)
    w = synth.make_ba_window(n_kf, n_pt, n_ln, rng, mean_track=6.0, track_mode="geometric", global_mode=True)
    w["kf_fixed"] = w["kf_fixed"].copy()
    w["kf_fixed"][list(fixed)] = 1
    w = _trim_tracks(w, B)
    F = free_kfs(w)
    starts = np.linspace(0, len(F) - 1 - B, n_long).astype(int)
    w = add_points(w, [F[s:s + B + 1] for s in starts], rng, True)
    return synth.batch_ba([w], "global", 1.0, robust)


def long_local_window(n_kf, n_pt, n_ln, rng, *, mean_track=10.0, n_fixed_extra=0):
    """a local window with long tracks and one point seen by every free keyframe (the longest possible upper row)"""
    w = synth.make_ba_window(n_kf, n_pt, n_ln, rng, mean_track=mean_track, n_fixed_extra=n_fixed_extra)
    return add_points(w, [free_kfs(w)], rng, False, ahead=8.0, side=(2.0, -1.0))


def duplicate_observation(w, i, du=0.7, kind="pt"):
    """landmark i (a point, or a line with kind="ln") observed a second time by the keyframe of its first free observation,
    with a slightly different measurement (the reference never does this)"""
    w = dict(w)
    off = w[f"{kind}_obs_off"]
    free = w["kf_fixed"][w[f"{kind}_obs_kf"][off[i]:off[i + 1]]] == 0
    e = int(off[i] + np.nonzero(free)[0][0])
    ins = lambda a, x: np.ascontiguousarray(np.insert(a, e + 1, x, axis=0))
    if kind == "pt":
        w["pt_obs_uvr"] = ins(w["pt_obs_uvr"], w["pt_obs_uvr"][e] + np.float32([du, -du, du if w["pt_obs_uvr"][e, 2] >= 0 else 0]))
        w["pt_obs_info"] = ins(w["pt_obs_info"], w["pt_obs_info"][e])
    else:
        w["ln_obs_left"] = ins(w["ln_obs_left"], w["ln_obs_left"][e] + np.float32([du, -du, du, du]))
        w["ln_obs_right"] = ins(w["ln_obs_right"], w["ln_obs_right"][e])
        w["ln_obs_info"] = ins(w["ln_obs_info"], w["ln_obs_info"][e])
        w["ln_obs_stereo"] = ins(w["ln_obs_stereo"], w["ln_obs_stereo"][e])
    w[f"{kind}_obs_kf"] = ins(w[f"{kind}_obs_kf"], w[f"{kind}_obs_kf"][e])
    w[f"{kind}_obs_off"] = (off + (np.arange(len(off)) > i)).astype(np.int32)
    return w


# ------------------------------------------------------------------------------------------------------------------
# shape claims, as ba.cu computes them
# ------------------------------------------------------------------------------------------------------------------
def _free_sets(p, w):
    """per landmark of window w: the sorted set of free block indices (window-local) that observe it, and whether one
    free keyframe observes it twice"""
    k0, k1 = int(p["kf_off"][w]), int(p["kf_off"][w + 1])
    g = np.cumsum(p["kf_fixed"][k0:k1] == 0) - 1
    g[p["kf_fixed"][k0:k1] != 0] = -1
    sets, dup = [], False
    for pre in ("pt", "ln"):
        off, kf, lo, hi = p[f"{pre}_obs_off"], p[f"{pre}_obs_kf"], int(p[f"{pre}_off"][w]), int(p[f"{pre}_off"][w + 1])
        for i in range(lo, hi):
            gs = g[kf[off[i]:off[i + 1]]]
            gs = np.sort(gs[gs >= 0])
            dup |= bool(np.any(gs[1:] == gs[:-1]))
            sets.append(np.unique(gs))
    return int(g.max()) + 1, sets, dup


def shape_claims(p):
    """the quantities ba_upload derives from the structure"""
    nw = int(p["n_win"])
    n_free, dup, max_nnb, n_lm = [], False, 0, []
    B, fb = 1, None
    for w in range(nw):
        nG, sets, d = _free_sets(p, w)
        n_free.append(nG)
        dup |= d
        n_lm.append(int(p["pt_off"][w + 1] - p["pt_off"][w] + p["ln_off"][w + 1] - p["ln_off"][w]))
        if nw == 1:
            fb = np.arange(nG)
            cov = np.eye(nG, dtype=bool)
            for s in sets:
                if len(s):
                    cov[np.ix_(s, s)] = True
                    fb[s] = np.minimum(fb[s], s[0])
                    B = max(B, int(s[-1] - s[0]))
            global_nnb = int(np.triu(cov).sum(1).max())
    c = dict(n_free=n_free, max_n=6 * max(n_free), dup_free=dup, n_lm=n_lm,
             n_slices=max(1, min(128, max(n_lm) // 16384)),
             local_nnb=max(n_free))           # local mode: every later free keyframe of the window is a neighbour
    if nw == 1:
        nG = n_free[0]
        last = np.arange(nG)
        for b in range(nG):
            last[fb[b]:b + 1] = np.maximum(last[fb[b]:b + 1], b)
        ph = max(6, 6 * int((last - np.arange(nG)).max()))
        maxlen = 6 * int((np.arange(nG) - fb).max()) + 6
        env_smem = 8 * (6 * ph + 8 + 32 * maxlen + 6 * nG) + 64
        c.update(B=B, m=6 * B, N=-(-nG // B), global_nnb=global_nnb, env_smem=env_smem)
        c["solver"] = "cr" if 6 * B <= CR_MAX_M else "env" if env_smem <= SMEM_LIMIT else "too wide"
    return c


# cyclic reduction: (B, free keyframes).  m = 6B covers both k_cr_solve instances and their edges (12, 60, 96: RHS columns an
# exact multiple of 64, 120: last <15>, 126: first <20>, 156 = CR_MAX_M); N = ceil(n_free / B) covers 2, 3, 4, 5, 8, 9, 17
# with the last super-block partial and exactly full, and a power of two
CR_CASES = [(2, 34), (10, 85), (16, 64), (20, 50), (21, 42), (26, 130), (26, 200)]
ENV_CASES = [dict(B=27, n_kf=101, fixed=()), dict(B=45, n_kf=151, fixed=(40, 41, 90))]


def cr_problem(B, n_free, robust=False):
    """(short tracks chain the keyframes weakly: B = 2 gets 60 points per keyframe, so that the problem determines its chi2 to
    1e-11, measured as the oracle's own change under a landmark permutation; at 12 points per keyframe that is 2e-9, and
    two correct solvers drift apart to 2e-6 by iteration 7)"""
    return banded_global(n_free + 1, B, max(12, 120 // B) * (n_free + 1), 2 * (n_free + 1), 1000 + 7 * B + n_free, robust=robust)


def env_problem(B, n_kf, fixed, robust=False):
    return banded_global(n_kf, B, 12 * n_kf, 2 * n_kf, 2000 + B, fixed=fixed, robust=robust)


def too_wide_problem():
    """200 keyframes; one landmark seen by the free keyframes 5 and n_free - 5 (a loop closure across the whole map)"""
    rng = np.random.default_rng(77)
    w = synth.make_ba_window(200, 2400, 400, rng, mean_track=6.0, track_mode="geometric", global_mode=True)
    F = free_kfs(w)
    w = add_points(w, [[F[5], F[len(F) - 5]]], rng, True, ahead=150.0, side=(0.0, -2.0))
    return synth.batch_ba([w], "global")


def sparse_windows(n_free, seed):
    rng = np.random.default_rng(seed)
    return synth.batch_ba([long_local_window(n_free + 1, 1500, 200, rng)], "local")


def mixed_batch():
    """one 40-keyframe window next to small ones: the whole batch leaves dense mode"""
    rng = np.random.default_rng(41)
    return synth.batch_ba([synth.make_ba_window(8, 400, 80, rng), long_local_window(40, 1500, 200, rng),
                           synth.make_ba_window(5, 200, 40, rng)], "local")


def dup_local():
    """a point and a line each observed twice by one free keyframe"""
    rng = np.random.default_rng(43)
    w = synth.make_ba_window(10, 1200, 200, rng)
    return synth.batch_ba([duplicate_observation(duplicate_observation(w, 17), 5, kind="ln")], "local")


def many_points_window():
    """32 769 points + lines in one window: points take one lane each, the reductions run in two slices"""
    rng = np.random.default_rng(45)
    return synth.batch_ba([synth.make_ba_window(6, 32769, 400, rng)], "local")


def ragged_batch():
    rng = np.random.default_rng(5)    # the batch of test_gpu_parity.py::test_local_ba_batch_ragged
    return synth.batch_ba([synth.make_ba_window(8, 500, 100, rng, n_fixed_extra=2), synth.make_ba_window(5, 300, 0, rng),
                           synth.make_ba_window(12, 50, 200, rng), synth.make_ba_window(20, 800, 150, rng, n_fixed_extra=1),
                           synth.make_ba_window(3, 40, 10, rng)], "local")


def target_batch():
    return synth.make_local_ba_batch(1, 10, 5000, 1000, 77)


# ------------------------------------------------------------------------------------------------------------------
# CPU tests: the shapes the GPU cases rest on
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,n_free", CR_CASES)
def test_cr_shapes(B, n_free):
    c = shape_claims(cr_problem(B, n_free))
    assert (c["B"], c["n_free"][0], c["solver"]) == (B, n_free, "cr")
    assert c["N"] == -(-n_free // B) and c["m"] <= CR_MAX_M


def test_cr_cases_cover_the_solver_edges():
    ms = {6 * B for B, _ in CR_CASES}
    assert {12, 60, 96, 120, 126, 156} <= ms
    Ns = {-(-n // B) for B, n in CR_CASES}
    assert {2, 3, 4, 5, 8, 9, 17} <= Ns
    full = [n % B == 0 for B, n in CR_CASES]
    assert any(full) and not all(full)


@pytest.mark.parametrize("case", ENV_CASES, ids=lambda c: f"B{c['B']}")
def test_env_shapes(case):
    c = shape_claims(env_problem(**case))
    assert c["B"] == case["B"] and c["solver"] == "env", c
    assert c["n_free"][0] == case["n_kf"] - 1 - len(case["fixed"])


def test_envelope_limit_shapes():
    c = shape_claims(too_wide_problem())
    assert c["B"] == c["n_free"][0] - 10 and c["solver"] == "too wide", c
    assert 6 * c["global_nnb"] <= 1024      # the neighbour limit is not what rejects it


def test_envelope_width_limit_in_the_header():
    """include/lldba.h states the widest envelope the skyline solver takes; check the numbers against ba.cu's formula for a
    pure band of half-bandwidth B (panel 6B rows, row length 6B + 6)"""
    def fits(B, nG):
        return 8 * (6 * 6 * B + 8 + 32 * (6 * B + 6) + 6 * nG) + 64 <= SMEM_LIMIT
    assert fits(117, 200) and not fits(118, 200)
    assert fits(83, 1500) and not fits(84, 1500)
    assert fits(122, 1) and not fits(123, 1)
    hdr = open(os.path.join(ROOT, "include", "lldba.h")).read()
    assert "228 B + 6 n_free <= 27952" in hdr


def test_dup_global_shape():
    p = cr_problem(10, 85)
    w = dict(p, n_kf=int(p["kf_off"][-1]), n_pt=int(p["pt_off"][-1]), n_ln=int(p["ln_off"][-1]))
    q = dict(p); q.update({k: v for k, v in duplicate_observation(w, 3).items() if k.startswith("pt_")})
    assert shape_claims(q)["dup_free"] and not shape_claims(p)["dup_free"]


@pytest.mark.parametrize("n_free", [32, 33, 64, 65])
def test_sparse_switch_shapes(n_free):
    c = shape_claims(sparse_windows(n_free, n_free))
    assert c["n_free"] == [n_free] and not c["dup_free"]
    assert c["max_n"] > 156                                            # k_solve<false> (global-memory scratch)
    assert (6 * c["local_nnb"] > 256) == (n_free > 42)                 # k_schur_rows<., 1024>


def test_mixed_batch_shapes():
    c = shape_claims(mixed_batch())
    assert c["n_free"] == [7, 39, 4] and c["max_n"] > 6 * 32


def test_dup_local_shapes():
    c = shape_claims(dup_local())
    assert c["dup_free"] and c["max_n"] <= 6 * 32


def test_many_points_shapes():
    c = shape_claims(many_points_window())
    p = many_points_window()
    assert int(p["pt_off"][-1]) > 32768 and c["n_slices"] == 2 and c["max_n"] <= 156


@pytest.mark.parametrize("n_free", [170, 171])
def test_neighbour_limit_shapes(n_free):
    p = sparse_windows(n_free, 170)
    c = shape_claims(p)
    assert c["local_nnb"] == n_free and (6 * c["local_nnb"] <= 1024) == (n_free == 170)
    n_obs_longest = int(np.diff(p["pt_obs_off"]).max())
    assert n_obs_longest == n_free                         # the appended point is seen by every free keyframe


def test_ragged_and_target_are_dense_single():
    for p in (ragged_batch(), target_batch()):
        c = shape_claims(p)
        assert c["max_n"] <= 156 and not c["dup_free"] and c["n_slices"] == 1


# ------------------------------------------------------------------------------------------------------------------
# GPU harness
# ------------------------------------------------------------------------------------------------------------------
def _bind(lib):
    d = lib.dll
    vp = C.c_void_p
    d.lld_ctx_profile.argtypes = [vp, C.c_int]; d.lld_ctx_profile.restype = None
    d.lld_ctx_profile_report.argtypes = [vp, C.c_char_p, C.c_int]; d.lld_ctx_profile_report.restype = C.c_int
    d.lld_ctx_last_bytes.argtypes = [vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]; d.lld_ctx_last_bytes.restype = None
    d.lld_ctx_set_topo_cache.argtypes = [vp, C.c_int]; d.lld_ctx_set_topo_cache.restype = None
    return d


def _context(topo_cache):
    c = capi.Context(0)
    _bind(c.lib).lld_ctx_set_topo_cache(c.handle, topo_cache)
    return c


@pytest.fixture(scope="module")
def ctx(built):
    """cache off: every call indexes its problem again, so switches read at upload take effect"""
    c = _context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def ctx_cached(built):
    c = _context(1)
    yield c
    c.close()


def h2d_bytes(c):
    h, d = C.c_int64(), C.c_int64()
    c.lib.dll.lld_ctx_last_bytes(c.handle, C.byref(h), C.byref(d))
    return h.value


def value_bytes(p):
    """what a topology-cache hit uploads: the value arrays only (ba.cu, cache-hit branch of ba_upload)"""
    n_kf, n_pt, n_ln = int(p["kf_off"][-1]), int(p["pt_off"][-1]), int(p["ln_off"][-1])
    n_pe, n_lc = int(p["pt_obs_off"][-1]), int(p["ln_obs_off"][-1])
    return (40 + 32 + 96) * n_kf + 16 * n_pe + 24 * n_pt + 49 * n_lc + 48 * n_ln


def run(p, c, mode, its=(5, 15)):
    if mode == "global":
        return api.ba_global(p, its[0], impl="gpu", ctx=c)
    return api.ba_local(p, its[0], its[1], impl="gpu", ctx=c)


def oracle(p, mode, its=(5, 15)):
    if mode == "global":
        return api.ba_global(p, its[0], impl="oracle")
    return api.ba_local(p, its[0], its[1], impl="oracle")


def profiled(p, c, mode, its=(5, 15)):
    d = c.lib.dll
    d.lld_ctx_profile(c.handle, 1)
    try:
        out = run(p, c, mode, its)
        buf = C.create_string_buffer(1 << 16)
        c.check(d.lld_ctx_profile_report(c.handle, buf, len(buf)), "lld_ctx_profile_report")
    finally:
        d.lld_ctx_profile(c.handle, 0)
    return out, set(json.loads(buf.value.decode()))


def assert_identical(a, b, what=""):
    for k in ("kf_Tcw", "pt_xyz", "ln_x0_dir", "pt_obs_bad", "ln_obs_bad", "ln_removed", "chi2_log", "lambda_log", "trials_log", "n_iter_done"):
        assert np.array_equal(a[k], b[k]), f"{what}: {k} differs"


def checked(p, c, mode, its=(5, 15), what=""):
    """GPU run checked against the oracle, plus a profiled run that must be bit-identical (profiling only turns off graph
    replay and the forked streams); returns the result and the names of the launched kernels"""
    g = run(p, c, mode, its)
    gp, names = profiled(p, c, mode, its)
    assert_identical(g, gp, f"{what} profiled vs unprofiled")
    check_ba(g, oracle(p, mode, its), what)
    return g, names


def expect_error(p, c, mode, code, *words):
    with pytest.raises(RuntimeError) as ei:
        run(p, c, mode)
    msg = str(ei.value)
    assert f"failed with {code}" in msg, msg
    for wd in words:
        assert wd in msg, msg
    return msg


# ------------------------------------------------------------------------------------------------------------------
# global BA
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("B,n_free", CR_CASES)
def test_global_cr(ctx, B, n_free):
    p = cr_problem(B, n_free)
    _, names = checked(p, ctx, "global", (8,), f"CR B={B} n_free={n_free}")
    want = "k_cr_solve<15>" if 6 * B <= 120 else "k_cr_solve<20>"
    assert {"k_cr_factor", "k_cr_assemble", "k_cr_update", want} <= names, names
    assert not names & {"k_solve_env", "k_cr_solve<15>", "k_cr_solve<20>"} - {want}, names


@pytest.mark.gpu
@pytest.mark.parametrize("case", ENV_CASES, ids=lambda c: f"B{c['B']}")
def test_global_skyline(ctx, case):
    p = env_problem(**case)
    _, names = checked(p, ctx, "global", (8,), f"skyline B={case['B']}")
    assert "k_solve_env" in names and not any(n.startswith("k_cr_") for n in names), names


@pytest.mark.gpu
@pytest.mark.parametrize("robust", [False, True])
@pytest.mark.parametrize("kind", ["cr", "skyline"])
def test_global_robust_flag(ctx, kind, robust):
    p = cr_problem(16, 64, robust=robust) if kind == "cr" else env_problem(**ENV_CASES[0], robust=robust)
    _, names = checked(p, ctx, "global", (8,), f"{kind} robust={robust}")
    assert ("k_cr_factor" if kind == "cr" else "k_solve_env") in names


@pytest.mark.gpu
def test_global_envelope_too_wide(ctx):
    """a loop-closure landmark across the map: rejected on the host before any kernel runs, with the limit in the message;
    the context then solves a valid problem correctly"""
    p = too_wide_problem()
    msg = expect_error(p, ctx, "global", ERR_UNSUPPORTED, "envelope", "bytes of shared memory")
    assert str(SMEM_LIMIT) in msg, msg
    q = cr_problem(10, 85)
    check_ba(run(q, ctx, "global", (8,)), oracle(q, "global", (8,)), "after the rejection")


@pytest.mark.gpu
def test_global_duplicate_observation_rejected(ctx):
    p = cr_problem(10, 85)
    w = dict(p, n_kf=int(p["kf_off"][-1]), n_pt=int(p["pt_off"][-1]), n_ln=int(p["ln_off"][-1]))
    q = dict(p); q.update({k: v for k, v in duplicate_observation(w, 3).items() if k.startswith("pt_")})
    expect_error(q, ctx, "global", ERR_ARG)
    check_ba(run(p, ctx, "global", (8,)), oracle(p, "global", (8,)), "after the rejection")


# ------------------------------------------------------------------------------------------------------------------
# local BA
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n_free", [32, 33, 64, 65])
def test_local_dense_sparse_switch(ctx, n_free):
    """32 free keyframes: dense mode (k_schur_tile); 33: sparse rows.  64 / 65: the co-visibility signature is a bitmask /
    a hash of the block list.  Every one of them solves with k_solve<false> (6 n_free > 156, see test_sparse_switch_shapes)."""
    _, names = checked(sparse_windows(n_free, n_free), ctx, "local", what=f"local n_free={n_free}")
    rows = "(k_schur_rows<3, 1024>)" if n_free > 42 else "(k_schur_rows<3, 256>)"
    if n_free <= 32:
        assert "k_schur_tile<3>" in names and not any(n.startswith("(k_schur_rows") for n in names), names
    else:
        assert {rows, "k_reduce_rows"} <= names and "k_schur_tile<3>" not in names, names


@pytest.mark.gpu
def test_local_mixed_batch_goes_sparse(ctx):
    _, names = checked(mixed_batch(), ctx, "local", what="mixed batch")
    assert {"(k_schur_rows<3, 256>)", "(k_schur_rows<4, 256>)", "k_reduce_rows"} <= names and "k_schur_tile<3>" not in names, names


@pytest.mark.gpu
def test_local_duplicate_observation_goes_sparse(ctx):
    """the Schur rows pair each edge with one co-edge per keyframe; the W blocks of the twice-observed (landmark, keyframe)
    pairs are summed first (k_fold_dup), as g2o sums both edges into one Hessian block"""
    _, names = checked(dup_local(), ctx, "local", what="dup_free")
    assert {"(k_schur_rows<3, 256>)", "(k_schur_rows<4, 256>)", "k_fold_dup"} <= names and "k_schur_tile<3>" not in names, names


@pytest.mark.gpu
def test_local_neighbour_limit(ctx):
    """170 free keyframes in one window: 6 * 170 = 1020 threads per Schur row, passes; 171 is rejected on the host"""
    _, names = checked(sparse_windows(170, 170), ctx, "local", (5, 5), what="170 neighbours")
    assert "(k_schur_rows<3, 1024>)" in names, names
    expect_error(sparse_windows(171, 170), ctx, "local", ERR_UNSUPPORTED, "171", "170")


@pytest.mark.gpu
def test_local_many_points_slices(ctx):
    _, names = checked(many_points_window(), ctx, "local", what="32769 points")
    assert {"k_lin_points<1>", "k_reduce_lin", "k_sum_lin", "k_begin", "k_decide"} <= names, names
    assert "k_lin_points<4>" not in names and "k_begin_fused" not in names, names


_SUB = """
import sys, json, numpy as np
sys.path.insert(0, 'tests')
import test_ba_paths as t
c = t._context(0)
out = {}
for name in ('ragged', 'target'):
    p = getattr(t, name + '_batch')()
    g = t.run(p, c, 'local')
    gp, names = t.profiled(p, c, 'local')
    t.assert_identical(g, gp, name + ' profiled')
    t.check_ba(g, t.oracle(p, 'local'), name)
    out[name] = sorted(names)
    np.savez(sys.argv[1] + '/' + name + '.npz', **{k: v for k, v in g.items() if isinstance(v, np.ndarray)})
print('SUB-OK ' + json.dumps(out))
"""


def run_subprocess(tmp_path, **env):
    r = subprocess.run([sys.executable, "-c", _SUB, str(tmp_path)], cwd=ROOT, env=dict(os.environ, **env),
                       capture_output=True, text=True, timeout=900)
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("SUB-OK ")]
    assert r.returncode == 0 and line, r.stdout[-3000:] + r.stderr[-3000:]
    names = json.loads(line[0][7:])
    res = {n: dict(np.load(tmp_path / f"{n}.npz")) for n in ("ragged", "target")}
    return res, names


@pytest.mark.gpu
@pytest.mark.parametrize("lanes", [1, 2, 4, 8])
def test_local_lanes_per_line(tmp_path, lanes):
    """LLD_LN_G forces the lanes per map line of k_lin_lines / k_backsub_lines (read once per process: a subprocess)"""
    _, names = run_subprocess(tmp_path, LLD_LN_G=str(lanes))
    for n in names.values():
        assert f"k_backsub_lines<{lanes}>" in n and any(x.startswith(f"(k_lin_lines<{lanes},") for x in n), n


@pytest.mark.gpu
@pytest.mark.parametrize("env", [{"LLD_BA_GRAPH": "0"}], ids=["eager"])
def test_local_step_schedules(ctx, monkeypatch, env):
    """graph replay against eager launches: the same kernels in the same order of sums, bit-identical.  Both batches are
    dense and single-rank, so the default runs graph replay on forked streams and lean steps
    (test_ragged_and_target_are_dense_single)."""
    for name in ("ragged", "target"):
        p = globals()[f"{name}_batch"]()
        ref = run(p, ctx, "local")
        with monkeypatch.context() as m:
            for k, v in env.items():
                m.setenv(k, v)
            g, names = checked(p, ctx, "local", what=f"{name} {env}")
        assert_identical(g, ref, f"{name} eager vs graph")
        assert "k_decide_carry" in names


@pytest.mark.gpu
@pytest.mark.parametrize("group", [1, 3])
def test_local_step_group_length(ctx, tmp_path, group):
    """LM steps enqueued in groups of 1 or 3 instead of 2 (LLD_BA_GROUP, read once per process): bit-identical"""
    res, _ = run_subprocess(tmp_path, LLD_BA_GROUP=str(group))
    for name in ("ragged", "target"):
        ref = run(globals()[f"{name}_batch"](), ctx, "local")
        assert_identical(res[name], ref, f"{name} group {group}")


# ------------------------------------------------------------------------------------------------------------------
# topology cache
# ------------------------------------------------------------------------------------------------------------------
def new_values(p, seed, what):
    """the same structure with new values: initial estimates, observation noise, stereo / mono and line right-edge flips, or
    information weights"""
    rng = np.random.default_rng(seed)
    q = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in p.items()}
    if "perturb" in what:
        q["kf_Tcw"][:, 9:] += rng.normal(0, 0.01, q["kf_Tcw"][:, 9:].shape)
        q["kf_Tcw"] = q["kf_Tcw"].astype(np.float32).astype(np.float64)
        q["pt_xyz"] = (q["pt_xyz"] + rng.normal(0, 0.03, q["pt_xyz"].shape)).astype(np.float32).astype(np.float64)
        q["ln_x0_dir"][:, :3] += rng.normal(0, 0.02, (len(q["ln_x0_dir"]), 3))
        d = q["ln_x0_dir"]; d[:, :3] -= (d[:, :3] * d[:, 3:]).sum(1, keepdims=True) * d[:, 3:]
    if "noise" in what:
        uvr = q["pt_obs_uvr"].astype(np.float64)
        dn = rng.normal(0, 0.4, (len(uvr), 2))
        uvr[:, :2] += dn
        st = uvr[:, 2] >= 0
        uvr[st, 2] = np.maximum(uvr[st, 2] + dn[st, 0], 0.0)
        q["pt_obs_uvr"] = synth.f32(uvr)
        q["ln_obs_left"] = synth.f32(q["ln_obs_left"] + rng.normal(0, 0.4, q["ln_obs_left"].shape))
    if "flips" in what:
        uvr = q["pt_obs_uvr"].copy()
        st = np.nonzero(uvr[:, 2] >= 0)[0]
        mono = st[rng.random(len(st)) < 0.15]                 # stereo -> mono
        uvr[mono, 2] = -1.0
        q["pt_obs_uvr"] = uvr
        rt = q["ln_obs_right"].copy(); ls = q["ln_obs_stereo"].copy()
        has = np.nonzero(rt[:, 0] >= 0)[0]
        drop = has[rng.random(len(has)) < 0.15]               # right segment present -> absent
        rt[drop] = -1.0
        if "global" not in what:
            ls[drop] = 0
        q["ln_obs_right"] = rt; q["ln_obs_stereo"] = ls
    if "info" in what:
        q["pt_obs_info"] = synth.f32(q["pt_obs_info"] * rng.choice([0.5, 1.0, 1.44, 2.0], len(q["pt_obs_info"])))
        q["ln_obs_info"] = q["ln_obs_info"] * rng.choice([0.7, 1.0, 1.3], (len(q["ln_obs_info"]), 1))
    return q


def undo_flips(p, base):
    """stereo / right-edge observations that `base` has and `p` lacks come back (mono -> stereo, absent -> present)"""
    q = dict(p)
    uvr = p["pt_obs_uvr"].copy(); back = (uvr[:, 2] < 0) & (base["pt_obs_uvr"][:, 2] >= 0)
    uvr[back, 2] = base["pt_obs_uvr"][back, 2]
    q["pt_obs_uvr"] = uvr
    rt = p["ln_obs_right"].copy(); ls = p["ln_obs_stereo"].copy(); back = (rt[:, 0] < 0) & (base["ln_obs_right"][:, 0] >= 0)
    rt[back] = base["ln_obs_right"][back]; ls[back] = base["ln_obs_stereo"][back]
    q["ln_obs_right"] = rt; q["ln_obs_stereo"] = ls
    return q


def warm_vs_cold(p, mode, ctx_cached, ctx, its=(5, 15), hit=True, what=""):
    """a call on the cache-on context against a cold call on the cache-off one: bit-identical; the upload is exactly the
    value arrays (hit) or exactly what the cold call uploads (miss)"""
    g = run(p, ctx_cached, mode, its)
    h = h2d_bytes(ctx_cached)
    cold = run(p, ctx, mode, its)
    if hit:
        assert h == value_bytes(p), f"{what}: {h} bytes uploaded, a cache hit uploads {value_bytes(p)}"
    else:
        assert h == h2d_bytes(ctx) > value_bytes(p), f"{what}: {h} bytes uploaded, a cold upload is {h2d_bytes(ctx)}"
    assert_identical(g, cold, f"{what} warm vs cold")
    check_ba(g, oracle(p, mode, its), what)
    return g


def cache_sequence(p0, mode, ctx_cached, ctx, its=(5, 15), flips_key="flips"):
    run(p0, ctx_cached, mode, its)                                   # index the structure
    seq = [new_values(p0, 1, "perturb"), new_values(p0, 2, "noise"), new_values(p0, 3, flips_key)]
    seq.append(undo_flips(new_values(p0, 4, flips_key), seq[2]))     # mono -> stereo and absent -> present right edges
    seq.append(new_values(p0, 5, "info"))
    for i, q in enumerate(seq):
        warm_vs_cold(q, mode, ctx_cached, ctx, its, what=f"{mode} warm #{i}")


@pytest.mark.gpu
def test_topo_cache_local_window(ctx_cached, ctx):
    rng = np.random.default_rng(61)
    cache_sequence(synth.batch_ba([synth.make_ba_window(10, 2000, 400, rng)], "local"), "local", ctx_cached, ctx)


@pytest.mark.gpu
def test_topo_cache_local_pipelined_batch(ctx_cached, ctx):
    """16 windows, cut into two sub-batches by two worker contexts; the halves share one structure (same window shapes, new
    values), so whichever worker takes a half finds it in its cache.  5 + 5 iterations: over ten iterations these windows
    determine chi2 to 1e-13 (the oracle's own change under a landmark permutation); over twenty, the float invz of the
    stereo edges lets two correct solvers drift apart to ~1e-6 on windows this small (see smoke() in __graft_entry__.py)"""
    rng = np.random.default_rng(62)
    wins = [synth.make_ba_window(int(rng.integers(8, 12)), int(rng.integers(1500, 2500)), int(rng.integers(200, 400)), rng)
            for _ in range(8)]
    half = synth.batch_ba(wins, "local")
    twin = new_values(half, 9, "perturb noise")
    wins2 = []
    for w in range(8):
        d = dict(wins[w])
        for key, off_key, per in (("kf_Tcw", "kf_off", None), ("pt_xyz", "pt_off", None), ("ln_x0_dir", "ln_off", None),
                                  ("pt_obs_uvr", "pt_obs_off", "pt_off"), ("ln_obs_left", "ln_obs_off", "ln_off")):
            if per is None:
                a, b = int(half[off_key][w]), int(half[off_key][w + 1])
            else:
                a, b = int(half[off_key][half[per][w]]), int(half[off_key][half[per][w + 1]])
            d[key] = twin[key][a:b]
        wins2.append(d)
    p0 = synth.batch_ba(wins + wins2, "local")
    assert int(p0["n_win"]) >= 16
    cache_sequence(p0, "local", ctx_cached, ctx, (5, 5))


@pytest.mark.gpu
def test_topo_cache_global_cr(ctx_cached, ctx):
    cache_sequence(cr_problem(16, 64), "global", ctx_cached, ctx, (8,), flips_key="flips global")


@pytest.mark.gpu
def test_topo_cache_structure_change_misses(ctx_cached, ctx):
    """same sizes, different structure: two observations swap their keyframes, or one keyframe changes its fixed flag"""
    rng = np.random.default_rng(63)
    w = synth.make_ba_window(10, 2000, 400, rng)
    p0 = synth.batch_ba([w], "local")
    run(p0, ctx_cached, "local")
    q = dict(p0); kf = p0["pt_obs_kf"].copy(); off = p0["pt_obs_off"]
    # two points with disjoint keyframe sets swap the keyframe of their first observations (both become outliers there)
    sets = [set(kf[off[i]:off[i + 1]]) for i in range(len(off) - 1)]
    i, j = next((a, b) for a in range(50) for b in range(a + 1, 200) if kf[off[a]] not in sets[b] and kf[off[b]] not in sets[a])
    kf[off[i]], kf[off[j]] = kf[off[j]], kf[off[i]]
    q["pt_obs_kf"] = kf
    warm_vs_cold(q, "local", ctx_cached, ctx, hit=False, what="swapped observations")
    r = dict(p0); fx = p0["kf_fixed"].copy(); fx[4] = 1; r["kf_fixed"] = fx
    warm_vs_cold(r, "local", ctx_cached, ctx, hit=False, what="fixed flag toggled")
    warm_vs_cold(new_values(r, 7, "noise"), "local", ctx_cached, ctx, hit=True, what="toggled structure, new values")


@pytest.mark.gpu
def test_topo_cache_parameters(ctx_cached, ctx):
    """same structure, other parameters (the captured LM steps carry them and are dropped) or another split of the same
    number of iterations: a cache hit, and oracle parity"""
    p0 = target_batch()
    run(p0, ctx_cached, "local")
    q = dict(p0, robust_points=0)
    warm_vs_cold(q, "local", ctx_cached, ctx, what="robust_points=0")
    q = dict(p0, chi2_pt_mono=5.0, chi2_pt_stereo=7.0, delta_pt_mono=2.0, delta_pt_stereo=2.5, delta_ln_mono=2.0, delta_ln_stereo=2.5)
    warm_vs_cold(q, "local", ctx_cached, ctx, what="thresholds")
    warm_vs_cold(p0, "local", ctx_cached, ctx, (10, 10), what="10 + 10")
    warm_vs_cold(p0, "local", ctx_cached, ctx, (5, 15), what="5 + 15 again")
