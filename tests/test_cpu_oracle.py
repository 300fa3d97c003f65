"""CPU tests (-m "not gpu"): the oracle against independent checks and the committed golden vectors, the
host-compiled device math against the oracle, and the C-ABI library's exported symbols (no compute without a GPU)."""
import ctypes as C
import json
import os
import re

import numpy as np
import pytest

from lld_slam_b200 import api, capi, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
dp = C.POINTER(C.c_double)
fp = C.POINTER(C.c_float)
P = lambda a: a.ctypes.data_as(dp)  # noqa: E731
PF = lambda a: a.ctypes.data_as(fp)  # noqa: E731
INTR = np.array([707.0912, 707.0912, 601.8873, 183.1104, 379.8145]).astype(np.float32).astype(np.float64)


def rand_pose(rng):
    w = rng.normal(0, 0.3, 3)
    return np.concatenate([synth._rodrigues(w[None])[0].reshape(-1), rng.normal(0, 1, 3)]).astype(np.float32).astype(np.float64)


def oracle_edge(ol, kind, T, lm, lcam, obs, want_jl=True):
    err = np.zeros(3); Jl = np.zeros(12); Jp = np.zeros(18)
    d = ol.lldo_edge_eval(kind, P(T), P(lm), P(INTR), P(lcam), P(obs), P(err), P(Jl) if want_jl else None, P(Jp))
    nl = 4 if kind == 2 else 3
    return err[:d].copy(), Jl[:d * nl].reshape(d, nl).copy(), Jp[:d * 6].reshape(d, 6).copy()


def test_oracle_jacobians_numeric(built):
    """analytic Jacobians of the oracle's edges against central differences through the vertex oplus."""
    ol = capi.load_oracle().dll
    rng = np.random.default_rng(0)
    lcam = np.array([INTR[0], INTR[2], INTR[3], -0.5371])

    def oplus_pose(T, u):
        o = np.zeros(12); ol.lldo_pose_oplus(P(T), P(np.asarray(u, float)), P(o)); return o

    def oplus_line(l, u):
        o = np.zeros(6); ol.lldo_line_oplus(P(l), P(np.asarray(u, float)), P(o)); return o

    for _ in range(20):
        T = rand_pose(rng)
        R = T[:9].reshape(3, 3)
        Xc = np.array([rng.uniform(-8, 8), rng.uniform(-2, 3), rng.uniform(3, 40)])
        X = R.T @ (Xc - T[9:])
        obs = np.array([rng.uniform(0, 1241), rng.uniform(0, 376), rng.uniform(0, 1241)])
        # mono: tight; stereo: the residual rounds 1/z to float32, so use a larger step and tolerance
        for kind, h, tol in ((0, 1e-6, 1e-5), (1, 1e-3, 2e-2)):
            e, Jl, Jp = oracle_edge(ol, kind, T, X, lcam, obs)
            nJl = np.zeros_like(Jl); nJp = np.zeros_like(Jp)
            for i in range(3):
                dd = np.zeros(3); dd[i] = h
                nJl[:, i] = (oracle_edge(ol, kind, T, X + dd, lcam, obs)[0] - oracle_edge(ol, kind, T, X - dd, lcam, obs)[0]) / (2 * h)
            for i in range(6):
                dd = np.zeros(6); dd[i] = h
                nJp[:, i] = (oracle_edge(ol, kind, oplus_pose(T, dd), X, lcam, obs)[0] - oracle_edge(ol, kind, oplus_pose(T, -dd), X, lcam, obs)[0]) / (2 * h)
            assert np.abs(Jl - nJl).max() <= tol * max(1.0, np.abs(Jl).max())
            assert np.abs(Jp - nJp).max() <= tol * max(1.0, np.abs(Jp).max())
        d = rng.normal(0, 1, 3); d /= np.linalg.norm(d)
        Pw = R.T @ (np.array([rng.uniform(-8, 8), rng.uniform(-2, 3), rng.uniform(4, 30)]) - T[9:])
        ln = np.concatenate([Pw - (Pw @ d) * d, d])
        ob = np.array([rng.uniform(0, 1241), rng.uniform(0, 376), 1.0, rng.uniform(0, 1241), rng.uniform(0, 376), 1.0])
        e, Jl, Jp = oracle_edge(ol, 2, T, ln, lcam, ob)
        h = 1e-6
        nJl = np.zeros_like(Jl); nJp = np.zeros_like(Jp)
        for i in range(4):
            dd = np.zeros(4); dd[i] = h
            nJl[:, i] = (oracle_edge(ol, 2, T, oplus_line(ln, dd), lcam, ob)[0] - oracle_edge(ol, 2, T, oplus_line(ln, -dd), lcam, ob)[0]) / (2 * h)
        for i in range(6):
            dd = np.zeros(6); dd[i] = h
            nJp[:, i] = (oracle_edge(ol, 2, oplus_pose(T, dd), ln, lcam, ob)[0] - oracle_edge(ol, 2, oplus_pose(T, -dd), ln, lcam, ob)[0]) / (2 * h)
        assert np.abs(Jl - nJl).max() <= 1e-4 * max(1.0, np.abs(Jl).max())
        assert np.abs(Jp - nJp).max() <= 1e-4 * max(1.0, np.abs(Jp).max())


def test_device_math_matches_oracle(built):
    """lld_slam_b200/csrc/lld_math.cuh compiled for the host (tests/hostcheck) against the oracle, edge by edge."""
    ol = capi.load_oracle().dll
    dm = C.CDLL(os.path.join(ROOT, "tests", "hostcheck", "libdevmath_host.so"))
    rng = np.random.default_rng(1)
    for it in range(500):
        T = rand_pose(rng)
        R = T[:9].reshape(3, 3)
        Xc = np.array([rng.uniform(-10, 10), rng.uniform(-2, 3), rng.uniform(2, 60)])
        X = R.T @ (Xc - T[9:])
        obs = np.array([rng.uniform(0, 1241), rng.uniform(0, 376), rng.uniform(0, 1241)], np.float32)
        for kind in (0, 1, 3):
            e1, Jl1, Jp1 = oracle_edge(ol, kind, T, X, np.zeros(4), obs.astype(np.float64), want_jl=kind != 3)
            e2 = np.zeros(3); Jl2 = np.zeros(9); Jp2 = np.zeros(18)
            d = dm.dm_point(kind, P(T), P(X), P(INTR), PF(obs), P(e2), P(Jl2), P(Jp2))
            assert np.abs(e1 - e2[:d]).max() <= 1e-10
            if kind != 3:
                assert np.abs(Jl1 - Jl2[:d * 3].reshape(d, 3)).max() <= 1e-12 * np.abs(Jl1).max()
            assert np.abs(Jp1 - Jp2[:d * 6].reshape(d, 6)).max() <= 1e-12 * np.abs(Jp1).max()
        dd = rng.normal(0, 1, 3); dd /= np.linalg.norm(dd)
        Pw = R.T @ (np.array([rng.uniform(-10, 10), rng.uniform(-2, 3), rng.uniform(4, 40)]) - T[9:])
        ln = np.concatenate([Pw - (Pw @ dd) * dd, dd])
        lcam = np.array([INTR[0], INTR[2], INTR[3], rng.choice([0.0, -0.5371])])
        ob = np.array([rng.uniform(0, 1241), rng.uniform(0, 376), 1.0, rng.uniform(0, 1241), rng.uniform(0, 376), 1.0])
        e1, Jl1, Jp1 = oracle_edge(ol, 2, T, ln, lcam, ob)
        e2 = np.zeros(2); Jl2 = np.zeros(8); Jp2 = np.zeros(12); e3 = np.zeros(2); dpz = C.c_int()
        dm.dm_line(P(T), P(ln), P(lcam), P(ob), P(e2), P(Jl2), P(Jp2), P(e3), C.byref(dpz))
        assert np.abs(e1 - e2).max() <= 1e-9 * max(1.0, np.abs(e1).max())
        assert np.array_equal(e2, e3)
        assert np.abs(Jl1 - Jl2.reshape(2, 4)).max() <= 1e-9 * np.abs(Jl1).max()
        assert np.abs(Jp1 - Jp2.reshape(2, 6)).max() <= 1e-9 * np.abs(Jp1).max()
        assert ol.lldo_line_depth_positive(P(T), P(ln), P(lcam), P(ob)) == dpz.value
        u = rng.normal(0, 0.05, 6) if it % 10 else rng.normal(0, 1e-7, 6)
        o1 = np.zeros(12); o2 = np.zeros(12)
        ol.lldo_pose_oplus(P(T), P(u), P(o1)); dm.dm_pose_oplus(P(T), P(u), P(o2))
        assert np.abs(o1 - o2).max() <= 1e-14
        u4 = rng.normal(0, 0.05, 4)
        o1 = np.zeros(6); o2 = np.zeros(6)
        ol.lldo_line_oplus(P(ln), P(u4), P(o1)); dm.dm_line_oplus(P(ln), P(u4), P(o2))
        assert np.abs(o1 - o2).max() <= 1e-12
    for d in (3, 4):
        A = rng.normal(0, 1, (d, d)); A = A @ A.T + np.eye(d)
        I = np.zeros((d, d))
        dm.dm_inv(d, P(np.ascontiguousarray(A)), P(I))
        assert np.abs(I - np.linalg.inv(A)).max() <= 1e-12


def test_descriptor_distance_vs_cv2_and_numpy(built):
    """ORBmatcher::DescriptorDistance == popcount == cv2.NORM_HAMMING, for the oracle and the library's host inline."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(2)
    for _ in range(200):
        a = rng.integers(0, 256, 32, dtype=np.uint8); b = rng.integers(0, 256, 32, dtype=np.uint8)
        ref = int(np.unpackbits(a ^ b).sum())
        assert ref == int(cv2.norm(a, b, cv2.NORM_HAMMING))
        assert api.descriptor_distance(a, b, impl="oracle") == ref
        assert api.descriptor_distance(a, b, impl="gpu") == ref  # host inline of the product library, no device needed


def test_oracle_lm_step_against_numpy_dense(built):
    """one Gauss-Newton/LM iteration of the oracle reproduces a dense numpy normal-equation solve of the same problem."""
    p = synth.make_local_ba_batch(1, 4, 30, 8, 3, outlier_frac=0.0)
    p["robust_points"] = 0
    p["delta_ln_mono"] = p["delta_ln_stereo"] = 1e9   # Huber never active -> plain least squares
    o = api.ba_local(p, 1, 0, impl="oracle")
    ol = capi.load_oracle().dll
    nk, npnt, nl = 4, 30, 8
    free = [k for k in range(nk) if not p["kf_fixed"][k]]
    n = 6 * len(free) + 3 * npnt + 4 * nl
    H = np.zeros((n, n)); b = np.zeros(n)
    col_p = {k: 6 * i for i, k in enumerate(free)}
    off_pt, off_ln = 6 * len(free), 6 * len(free) + 3 * npnt
    chi0 = 0.0

    def add(Jl, Jp, e, info, lc, pc):
        nonlocal chi0
        chi0 += info * float(e @ e)
        J = np.zeros((len(e), n))
        J[:, lc:lc + Jl.shape[1]] = Jl
        if pc is not None:
            J[:, pc:pc + 6] = Jp
        H[:] += info * J.T @ J
        b[:] += -info * J.T @ e

    for i in range(npnt):
        for e in range(p["pt_obs_off"][i], p["pt_obs_off"][i + 1]):
            kf = p["pt_obs_kf"][e]; obs = p["pt_obs_uvr"][e].astype(np.float64)
            kind = 0 if obs[2] < 0 else 1
            er, Jl, Jp = oracle_edge(ol, kind, p["kf_Tcw"][kf], p["pt_xyz"][i], np.zeros(4), obs)
            add(Jl, Jp, er, float(p["pt_obs_info"][e]), off_pt + 3 * i, col_p.get(kf))
    for i in range(nl):
        for c in range(p["ln_obs_off"][i], p["ln_obs_off"][i + 1]):
            kf = p["ln_obs_kf"][c]; cam = p["kf_line_cam"][kf]
            for side, seg in ((0, p["ln_obs_left"][c]), (1, p["ln_obs_right"][c])):
                if side == 1 and seg[0] < 0:
                    continue
                lcam = np.array([cam[0], cam[1], cam[2], -cam[3] if side else 0.0])
                ob = np.array([seg[0], seg[1], 1.0, seg[2], seg[3], 1.0], np.float64)
                er, Jl, Jp = oracle_edge(ol, 2, p["kf_Tcw"][kf], p["ln_x0_dir"][i], lcam, ob)
                add(Jl, Jp, er, float(p["ln_obs_info"][c, side]), off_ln + 4 * i, col_p.get(kf))
    assert abs(chi0 - o["chi2_log"][0, 0]) <= 1e-9 * chi0
    lam = 1e-5 * np.abs(np.diag(H)).max()
    x = np.linalg.solve(H + lam * np.eye(n), b)
    # apply to the first free pose and compare with the oracle's result after its single iteration
    k = free[0]
    Tn = np.zeros(12)
    ol.lldo_pose_oplus(P(p["kf_Tcw"][k]), P(np.ascontiguousarray(x[col_p[k]:col_p[k] + 6])), P(Tn))
    if o["trials_log"][0, 0] == 1 and o["chi2_log"][0, 1] < o["chi2_log"][0, 0]:
        assert np.abs(Tn - o["kf_Tcw"][k]).max() <= 1e-7
        Xn = p["pt_xyz"][0] + x[off_pt:off_pt + 3]
        assert np.abs(Xn - o["pt_xyz"][0]).max() <= 1e-6


GOLDEN = os.path.join(ROOT, "tests", "golden", "oracle_golden.json")


def test_oracle_golden_vectors(built):
    """committed fixtures (tests/golden/make_golden.py): the oracle must keep reproducing them bit-for-bit / to 1e-12."""
    g = json.load(open(GOLDEN))
    p = synth.make_local_ba_batch(1, 5, 120, 30, g["ba_local"]["seed"])
    o = api.ba_local(p, 5, 15, impl="oracle")
    assert o["n_iter_done"].tolist() == g["ba_local"]["n_iter_done"]
    assert np.allclose(o["chi2_log"][0], g["ba_local"]["chi2_log"], rtol=1e-10, atol=0)
    assert int(o["pt_obs_bad"].sum()) == g["ba_local"]["n_pt_bad"] and int(o["ln_obs_bad"].sum()) == g["ba_local"]["n_ln_bad"]
    assert np.allclose(o["kf_Tcw"], np.array(g["ba_local"]["kf_Tcw"]), rtol=0, atol=1e-10)
    q = synth.make_pose_batch(3, 80, 20, g["pose"]["seed"])
    r = api.pose_opt(q, impl="oracle")
    assert r["n_inliers"].tolist() == g["pose"]["n_inliers"]
    assert np.allclose(r["Tcw"], np.array(g["pose"]["Tcw"]), rtol=0, atol=1e-10)
    m = synth.make_sbp_frame_batch(2, 300, g["sbp"]["seed"])
    s = api.sbp_frame(m, impl="oracle")
    assert s["n_matches"].tolist() == g["sbp"]["n_matches"]
    assert int(s["best_dist"][s["best_idx"] >= 0].sum()) == g["sbp"]["dist_sum"]
    assert s["match"].tolist() == g["sbp"]["match"]
    lm = synth.make_line_match_batch(2, 60, 64, g["lines"]["seed"])
    t = api.line_match(lm, impl="oracle")
    assert t["match"].tolist() == g["lines"]["match"]


def test_matching_oracle_properties(built):
    """domain properties of the matcher: every match within TH_HIGH, claimed keypoints never matched, matches are a
    partial injection when every query has observations."""
    m = synth.make_sbp_frame_batch(4, 800, 5)
    m["last_has_obs"][:] = 1
    m["check_orientation"] = 0
    s = api.sbp_frame(m, impl="oracle")
    assert (s["best_dist"][s["best_idx"] >= 0] <= 100).all()
    for pr in range(4):
        q0, q1 = m["last_off"][pr], m["last_off"][pr + 1]
        bi = s["best_idx"][q0:q1]
        bi = bi[bi >= 0]
        assert len(np.unique(bi)) == len(bi)
        c0 = m["cur_off"][pr]
        assert not m["cur_claimed"][c0 + bi].any()
    lm = synth.make_line_match_batch(3, 100, 64, 8)
    t = api.line_match(lm, impl="oracle")
    for pr in range(3):
        a0, a1 = lm["left_off"][pr], lm["left_off"][pr + 1]
        mm = t["match"][a0:a1]; mm = mm[mm >= 0]
        assert len(np.unique(mm)) == len(mm)
        assert (t["dist"][a0:a1][t["match"][a0:a1] >= 0] < lm["tau"]).all()


def test_library_exports_every_declared_symbol(built):
    """the C-ABI shared library loads and exports every function include/lldba.h declares."""
    hdr = open(os.path.join(ROOT, "include", "lldba.h")).read()
    names = set(re.findall(r"\b(lld_[a-z0-9_]+)\s*\(", hdr))
    assert {"lld_ba_local", "lld_ba_global", "lld_pose_opt", "lld_sbp_frame", "lld_sbp_mappoints", "lld_line_match",
            "lld_descriptor_distance", "lld_ctx_create", "lld_ctx_destroy", "lld_comm_init"} <= names
    dll = capi.load_library().dll
    for n in sorted(names):
        assert hasattr(dll, n), f"liblldba.so does not export {n}"
    assert dll.lld_version().startswith(b"lldba")


def test_product_never_routes_through_the_oracle():
    """the product sources must not reference the oracle (no CPU fallback)."""
    for dirpath, _, files in os.walk(os.path.join(ROOT, "lld_slam_b200", "csrc")):
        for f in files:
            if f.endswith((".cu", ".cuh", ".h", "Makefile")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "lldo_" not in txt and "liblld_oracle" not in txt, f
    import torch
    with pytest.raises(RuntimeError):   # without a device even device 0 must fail; with one, an index that does not exist
        capi.Context(0 if torch.cuda.device_count() == 0 else 9999)


def test_cpp_shim_compiles_and_links(built, tmp_path):
    """lld_slam_b200/host/lld_shim.h (reference class names over the C-ABI) compiles as C++14 and links to liblldba.so."""
    import subprocess
    exe = str(tmp_path / "shim_test")
    csrc = os.path.join(ROOT, "lld_slam_b200", "csrc")
    r = subprocess.run(["g++", "-std=c++14", "-Wall", os.path.join(ROOT, "tests", "hostcheck", "shim_compile.cpp"), "-o", exe,
                        "-L" + csrc, "-llldba", "-Wl,-rpath," + csrc], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    assert subprocess.run([exe]).returncode == 0


def test_host_indexing_stage_runs_without_a_device(built):
    """lld_ba_index_only drives the whole host stage of lld_ba_local / lld_ba_global (flattening, signature sort, keyframe lists,
    dense pieces, gather lists, worker pool, persistent scratch) with the device calls stubbed out: it must accept
    well-formed problems, repeatedly, and reject malformed ones — no GPU needed."""
    import ctypes as C
    from lld_slam_b200 import capi, synth
    lib = capi.load_library()
    f = lib.dll.lld_ba_index_only
    f.argtypes = [C.POINTER(capi.BaProblem), C.c_int]
    f.restype = C.c_int
    p = synth.make_local_ba_batch(6, 8, 300, 60, 17)
    prob, keep = capi.fill_struct(capi.BaProblem, p)
    for _ in range(3):   # persistent scratch: repeated calls reuse it
        assert f(C.byref(prob), 0) == 0
    g = synth.make_global_ba(30, 800, 150, 5)
    gprob, keep2 = capi.fill_struct(capi.BaProblem, g)
    assert f(C.byref(gprob), 1) == 0
    bad = dict(p)
    bad["pt_obs_kf"] = p["pt_obs_kf"].copy()
    bad["pt_obs_kf"][5] = 10 ** 6           # keyframe index outside its window
    bprob, keep3 = capi.fill_struct(capi.BaProblem, bad)
    assert f(C.byref(bprob), 0) == -2       # LLD_ERR_ARG


def test_host_indexing_is_deterministic(built, capfd, monkeypatch):
    """The host stage runs per-window work on a thread pool; every index array it uploads must not depend on the thread
    schedule: LLD_UP_TRACE prints an FNV hash of each uploaded array, two runs (and a run after an unrelated problem has
    reused the persistent scratch) must print the same hashes."""
    import ctypes as C
    from lld_slam_b200 import capi, synth
    lib = capi.load_library()
    f = lib.dll.lld_ba_index_only
    f.argtypes = [C.POINTER(capi.BaProblem), C.c_int]
    f.restype = C.c_int
    monkeypatch.setenv("LLD_UP_TRACE", "1")
    p = synth.make_local_ba_batch(9, 12, 700, 150, 23)
    q = synth.make_local_ba_batch(4, 6, 200, 40, 5)
    prob, keep = capi.fill_struct(capi.BaProblem, p)
    qrob, keep2 = capi.fill_struct(capi.BaProblem, q)

    def hashes(pr):
        capfd.readouterr()
        assert f(C.byref(pr), 0) == 0
        err = capfd.readouterr().err
        # arrays that are only sized, not filled, in dense mode (sparse-mode tables) are skipped: their bytes are scratch
        skip = ("pe_pos", "lc_pos", "pl_tab", "ll_tab")
        return [ln for ln in err.splitlines() if ln.startswith("[up]") and not any(k in ln for k in skip)]

    a = hashes(prob)
    assert len(a) > 40
    b = hashes(prob)
    hashes(qrob)
    c2 = hashes(prob)
    assert a == b == c2


# ------------------------------------------------------------------------------------------------
# SURVEY §8(f) row 1 (next round's kernel): Frame::ComputeStereoMatches, oracle pinned ahead of the product
# ------------------------------------------------------------------------------------------------
def _stereo_frame(seed, **kw):
    return synth.make_stereo_frame(seed, **kw)


def _stereo_matches_numpy(f):
    """Independent transcription of src/Frame.cc:530-704 with cv2 for the two distances."""
    import cv2
    f32 = np.float32
    N = len(f["kpL"])
    uRight = np.full(N, -1.0, f32)
    depth = np.full(N, -1.0, f32)
    nRows = f["pyrL"][0].shape[0]
    rowidx = [[] for _ in range(nRows)]
    for iR, (kp, o) in enumerate(zip(f["kpR"], f["octR"])):
        r = f32(2.0) * f["scale"][o]
        for yi in range(int(np.floor(kp[1] - r)), int(np.ceil(kp[1] + r)) + 1):
            if 0 <= yi < nRows:
                rowidx[yi].append(iR)
    maxD = f32(f["mbf"] / f["mb"])
    cand = []
    for iL in range(N):
        uL, vL = f["kpL"][iL]
        lvl = int(f["octL"][iL])
        if not vL >= 0 or int(vL) >= nRows:      # rowidx would be indexed outside the image: no match (as the oracle)
            continue
        cs = rowidx[int(vL)]
        if not cs or uL < 0:
            continue
        minU, maxU = f32(uL - maxD), uL
        best, bestR = 100, 0
        for iR in cs:
            if abs(int(f["octR"][iR]) - lvl) > 1:
                continue
            uR = f["kpR"][iR, 0]
            if minU <= uR <= maxU:
                dist = int(cv2.norm(f["descL"][iL], f["descR"][iR], cv2.NORM_HAMMING))
                if dist < best:
                    best, bestR = dist, iR
        if best >= 75:
            continue
        s = f["inv"][lvl]
        rnd = lambda x: f32(np.floor(abs(x) + 0.5) * np.sign(x))       # C round(): half away from zero
        su, sv, sr = rnd(f32(uL * s)), rnd(f32(vL * s)), rnd(f32(f["kpR"][bestR, 0] * s))
        imL, imR = f["pyrL"][lvl], f["pyrR"][lvl]
        rows, cols = imL.shape
        r0, c0 = int(sv) - 5, int(su) - 5
        if r0 < 0 or r0 + 11 > rows or c0 < 0 or c0 + 11 > cols:
            continue
        IL = imL[r0:r0 + 11, c0:c0 + 11].astype(f32)
        IL = IL - IL[5, 5]
        if sr < 0 or sr + 11 >= cols:
            continue
        dists, ok = [], True
        bestS, bestinc = 2 ** 31 - 1, 0
        for inc in range(-5, 6):
            cr = int(sr) + inc - 5
            if cr < 0 or cr + 11 > cols:
                ok = False
                break
            IR = imR[r0:r0 + 11, cr:cr + 11].astype(f32)
            IR = IR - IR[5, 5]
            dist = f32(cv2.norm(IL, IR, cv2.NORM_L1))
            if dist < f32(bestS):
                bestS, bestinc = int(dist), inc
            dists.append(dist)
        if not ok or bestinc in (-5, 5):
            continue
        d1, d2, d3 = dists[5 + bestinc - 1], dists[5 + bestinc], dists[5 + bestinc + 1]
        with np.errstate(divide="ignore", invalid="ignore"):
            delta = f32(f32(d1 - d3) / f32(f32(2.0) * f32(f32(d1 + d3) - f32(f32(2.0) * d2))))
        if delta < -1 or delta > 1:
            continue
        bu = f32(f["scale"][lvl] * f32(f32(sr + f32(bestinc)) + delta))
        disp = f32(uL - bu)
        if disp >= 0 and disp < maxD:
            if disp <= 0:
                disp = f32(0.01)
                bu = f32(np.float64(uL) - 0.01)
            depth[iL] = f32(f["mbf"] / disp)
            uRight[iL] = bu
            cand.append((bestS, iL))
    if cand:
        cand.sort()
        th = f32(f32(1.5) * f32(1.4)) * f32(cand[len(cand) // 2][0])
        for dS, iL in reversed(cand):
            if f32(dS) < th:
                break
            uRight[iL] = -1
            depth[iL] = -1
    return uRight, depth


def _stereo_matches_oracle(f):
    import ctypes as C
    dll = capi.load_oracle().dll
    fn = dll.lldo_stereo_matches
    fn.restype = C.c_int
    P = C.c_void_p
    n_levels = len(f["pyrL"])
    ptr = lambda a: a.ctypes.data_as(P)
    arrL = (P * n_levels)(*[a.ctypes.data for a in f["pyrL"]])
    arrR = (P * n_levels)(*[a.ctypes.data for a in f["pyrR"]])
    rows = np.array([a.shape[0] for a in f["pyrL"]], np.int32)
    cols = np.array([a.shape[1] for a in f["pyrL"]], np.int32)
    stride = np.array([a.strides[0] for a in f["pyrL"]], np.int32)
    N, Nr = len(f["kpL"]), len(f["kpR"])
    uR, dep = np.empty(N, np.float32), np.empty(N, np.float32)
    fn.argtypes = [C.c_int, P, P, P, C.c_int, P, P, P, C.c_int, P, P, P, P, P, P, P, C.c_float, C.c_float, P, P]
    n = fn(N, ptr(f["kpL"]), ptr(f["octL"]), ptr(f["descL"]), Nr, ptr(f["kpR"]), ptr(f["octR"]), ptr(f["descR"]), n_levels,
           ptr(f["scale"]), ptr(f["inv"]), C.cast(arrL, P), C.cast(arrR, P), ptr(rows), ptr(cols), ptr(stride),
           C.c_float(float(f["mb"])), C.c_float(float(f["mbf"])), ptr(uR), ptr(dep))
    return n, uR, dep


def test_oracle_stereo_matches_against_numpy(built):
    """Frame::ComputeStereoMatches (src/Frame.cc:530-704): the C++ oracle and an independent numpy / cv2 transcription give
    the same mvuRight / mvDepth bit for bit, on frames where most points match and the disparity is recovered."""
    for seed in (1, 2, 3):
        f = _stereo_frame(seed)
        n, uR, dep = _stereo_matches_oracle(f)
        uR2, dep2 = _stereo_matches_numpy(f)
        assert np.array_equal(uR, uR2) and np.array_equal(dep, dep2)
        got = uR >= 0
        assert n == int(got.sum()) and n > 0.4 * len(uR)
        # the synthetic disparity is 4 + 3 * (row // 40): sub-pixel refinement must land within a pixel of it
        true_d = 4 + (f["kpL"][got, 1].astype(int) // 40) * 3
        err = np.abs((f["kpL"][got, 0] - uR[got]) - true_d)
        assert np.median(err) < 0.6 and (err < 1.6).mean() > 0.9
    # no keypoints on the right: nothing matches, nothing is read out of range
    f = _stereo_frame(4)
    f["kpR"], f["octR"], f["descR"] = f["kpR"][:0], f["octR"][:0], f["descR"][:0]
    n, uR, dep = _stereo_matches_oracle(f)
    assert n == 0 and (uR == -1).all() and (dep == -1).all()


# ------------------------------------------------------------------------------------------------
# SURVEY §8(f) row 4: medoid (distinctive) descriptors of map points / map lines
# ------------------------------------------------------------------------------------------------
def _medoid_landmarks(seed, n_lm=150, max_obs=14, dim=None):
    rng = np.random.default_rng(seed)
    cnt = rng.integers(0, max_obs, n_lm)
    off = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int32)
    if dim is None:
        base = rng.integers(0, 256, (n_lm, 32), dtype=np.uint8)
        desc = np.zeros((int(off[-1]), 32), np.uint8)
        for l in range(n_lm):
            for j in range(off[l], off[l + 1]):
                d = base[l].copy()
                for b in rng.integers(0, 256, int(rng.integers(0, 60))):
                    d[b >> 3] ^= np.uint8(1 << (b & 7))
                desc[j] = d
        return off, desc
    base = rng.normal(0, 1, (n_lm, dim))
    desc = np.zeros((int(off[-1]), dim), np.float32)
    for l in range(n_lm):
        for j in range(off[l], off[l + 1]):
            desc[j] = (base[l] * rng.uniform(0.5, 3.0) + rng.normal(0, 0.6, dim)).astype(np.float32)   # distances straddle 1, 2, 3 ...
    return off, desc


def _medoid_numpy(off, desc, ham):
    """transcription of the reference with cv2.norm (NORM_HAMMING / NORM_L2), float distance table, truncated int median,
    first index on ties"""
    import cv2
    out = []
    for l in range(len(off) - 1):
        N = int(off[l + 1] - off[l])
        if N == 0:
            out.append(-1)
            continue
        d = desc[off[l]:off[l + 1]]
        Dm = np.zeros((N, N), np.float32)
        for i in range(N):
            for j in range(i + 1, N):
                Dm[i, j] = Dm[j, i] = cv2.norm(d[i], d[j], cv2.NORM_HAMMING) if ham else cv2.norm(d[i] - d[j])
        bm, bi = 2 ** 31 - 1, 0
        for i in range(N):
            m = int(np.sort(Dm[i])[int(0.5 * (N - 1))])
            if m < bm:
                bm, bi = m, i
        out.append(bi)
    return np.array(out, np.int32)


def test_oracle_medoid_descriptors_against_numpy(built):
    """MapPoint / MapLine::ComputeDistinctiveDescriptors (src/MapPoint.cc:242-307, src/MapLine.cc:133-201): the oracle against
    _medoid_numpy"""
    off, desc = _medoid_landmarks(1)
    assert np.array_equal(api.medoid_orb(off, desc, impl="oracle"), _medoid_numpy(off, desc, True))
    off, desc = _medoid_landmarks(2, dim=64)
    got = api.medoid_float(off, desc, impl="oracle")
    assert np.array_equal(got, _medoid_numpy(off, desc, False))
    assert len(set(got.tolist())) > 3     # not everything collapses onto index 0


# ------------------------------------------------------------------------------------------------
# SURVEY §8(f) row 3: temporal line association (Tracking::AddLinesFrom)
# ------------------------------------------------------------------------------------------------
def _add_lines_from_numpy(p):
    """transcription of src/Tracking.cc:996-1124 with vgl::LineReprojErrorL1 (src/vgl.cc:548-559) in numpy"""
    K = np.asarray(p["K"], np.float64).reshape(3, 3)
    out = np.full(int(p["cur_off"][-1]), -1, np.int32)
    added = []

    def map_point(T, X):
        return T[:3, :3].T @ (X - T[:3, 3])

    def err_l1(seg, T, X0, d):
        Xc1 = K @ map_point(T, X0)
        Xc2 = K @ map_point(T, X0 + d)
        leq = np.cross(Xc1, Xc2)
        leq = leq / np.linalg.norm(leq[:2])
        return abs(np.dot(seg[:2].astype(np.float64), leq[:2]) + leq[2]) + abs(np.dot(seg[2:].astype(np.float64), leq[:2]) + leq[2])

    for f in range(int(p["n_frames"])):
        T = p["T_curr"][f].reshape(4, 4); Tr = p["T_right"][f].reshape(4, 4)
        c0, r0 = int(p["cur_off"][f]), int(p["right_off"][f])
        taken = p["cur_taken"][c0:int(p["cur_off"][f + 1])].astype(bool).copy()
        n = 0
        for i in range(int(p["ml_off"][f]), int(p["ml_off"][f + 1])):
            if not p["ml_valid"][i]:
                continue
            X0, d = p["ml_x0_dir"][i, :3], p["ml_x0_dir"][i, 3:]
            X1c, X2c = map_point(T, p["ml_x1x2"][i, :3]), map_point(T, p["ml_x1x2"][i, 3:])
            match_id, md = -1, 1e10
            for si in p["cand_idx"][int(p["cand_off"][i]):int(p["cand_off"][i + 1])]:
                si = int(si)
                if taken[si]:
                    continue
                ri = int(p["cur_line_match"][c0 + si])
                if ri < 0 and not p["monocular"]:
                    continue
                if X1c[2] < 0 or X2c[2] < 0:
                    continue
                thr = float(p["thr_reproj_base"])
                for _ in range(int(p["cur_octave"][c0 + si])):
                    thr *= 1.44
                se = err_l1(p["cur_left"][c0 + si], T, X0, d)
                se2 = 0.0 if p["monocular"] else err_l1(p["cur_right"][r0 + ri], Tr, X0, d)
                if se > thr or se2 > thr:
                    continue
                cd = float(np.linalg.norm(p["ml_desc"][i].astype(np.float64) - p["cur_desc"][c0 + si].astype(np.float64)))
                if cd < md:
                    md, match_id = cd, si
            if md > p["md_thr"]:
                continue
            if match_id >= 0 and not taken[match_id]:
                taken[match_id] = True
                out[c0 + match_id] = i - int(p["ml_off"][f])
                n += 1
        added.append(n)
    return out, np.array(added, np.int32)


def test_oracle_line_association_against_numpy(built):
    p = synth.make_line_assoc_batch(4, 150, 120, 32, 3)
    o = api.line_associate(p, impl="oracle")
    ref, added = _add_lines_from_numpy(p)
    assert np.array_equal(o["cur_assoc"], ref) and np.array_equal(o["n_added"], added)
    assert added.min() > 20
    # the true map line is what gets associated for the unambiguous (non-clutter) lines
    assert (ref >= 0).sum() > 100


# ------------------------------------------------------------------------------------------------------------------
# SURVEY §8(f) row 2: keyframe searches (Fuse, Fuse with Sim3, SearchByProjection with Sim3)
# ------------------------------------------------------------------------------------------------------------------
def _kf_search_python(p):
    """Independent transcription of the loop bodies of ORBmatcher::Fuse (src/ORBmatcher.cc:886-972), Fuse(Scw) (:1040-1097) and
    SearchByProjection(KeyFrame*, Scw, ...) (:350-399) from KeyFrame::GetFeaturesInArea (src/KeyFrame.cc: cell range by floor / ceil of
    (x - mnMinX -+ r) * mfGridElementWidthInv, |dx| < r && |dy| < r) on, in float32 arithmetic, plain loops, its own grid."""
    f = np.float32
    g = p["geom"]
    minx, miny = f(g["min_x"]), f(g["min_y"])
    winv = f(64) / (f(g["max_x"]) - minx)
    hinv = f(48) / (f(g["max_y"]) - miny)
    sf = np.asarray(g["scale_factors"], np.float32)
    inv = np.asarray(p["inv_level_sigma2"], np.float32)
    n_mp = int(p["mp_off"][-1])
    best_idx = np.full(n_mp, -1, np.int32); best_dist = np.full(n_mp, 256, np.int32)
    match = np.full(int(p["kp_off"][-1]), -1, np.int32); n_matches = np.zeros(p["n_pairs"], np.int32)
    for pr in range(p["n_pairs"]):
        c0, c1 = int(p["kp_off"][pr]), int(p["kp_off"][pr + 1])
        xy = p["kp_xy"][c0:c1]; octv = p["kp_octave"][c0:c1]; kur = p["kp_uright"][c0:c1]; kd = p["kp_desc"][c0:c1]
        cells = {}
        for i in range(c1 - c0):                                   # KeyFrame keeps Frame::AssignFeaturesToGrid's grid
            px = int(np.round((xy[i, 0] - minx) * winv)); py = int(np.round((xy[i, 1] - miny) * hinv))
            if 0 <= px < 64 and 0 <= py < 48:
                cells.setdefault((px, py), []).append(i)
        matched = p["kp_claimed"][c0:c1].astype(bool).copy()
        for q in range(int(p["mp_off"][pr]), int(p["mp_off"][pr + 1])):
            if not p["mp_valid"][q]:
                continue
            u, v, ur = (f(x) for x in p["mp_proj"][q]); lvl = int(p["mp_level"][q])
            r = f(p["th"]) * sf[lvl]
            x0 = max(0, int(np.floor((u - minx - r) * winv))); x1 = min(63, int(np.ceil((u - minx + r) * winv)))
            y0 = max(0, int(np.floor((v - miny - r) * hinv))); y1 = min(47, int(np.ceil((v - miny + r) * hinv)))
            if x0 >= 64 or x1 < 0 or y0 >= 48 or y1 < 0:
                continue
            bd, bi = 256, -1
            for ix in range(x0, x1 + 1):
                for iy in range(y0, y1 + 1):
                    for idx in cells.get((ix, iy), ()):
                        if not (abs(xy[idx, 0] - u) < r and abs(xy[idx, 1] - v) < r):
                            continue
                        if matched[idx]:
                            continue
                        kl = int(octv[idx])
                        if kl < lvl - 1 or kl > lvl:
                            continue
                        if p["chi2_gate"]:
                            ex = u - xy[idx, 0]; ey = v - xy[idx, 1]
                            if kur[idx] >= 0:
                                er = ur - kur[idx]
                                e2 = f(f(ex * ex) + f(ey * ey)) + f(er * er)
                                if float(f(e2) * inv[kl]) > 7.8:
                                    continue
                            else:
                                e2 = f(ex * ex) + f(ey * ey)
                                if float(f(e2) * inv[kl]) > 5.99:
                                    continue
                        d = int(np.unpackbits(np.bitwise_xor(p["mp_desc"][q], kd[idx])).sum())
                        if d < bd:
                            bd, bi = d, idx
            if bd <= p["th_low"]:
                match[c0 + bi] = q - int(p["mp_off"][pr])
                if p["sequential_claims"]:
                    matched[bi] = True
                n_matches[pr] += 1
                best_idx[q] = bi; best_dist[q] = bd
    return dict(match=match, n_matches=n_matches, best_idx=best_idx, best_dist=best_dist)


@pytest.mark.parametrize("mode", [(1, 0), (0, 0), (0, 1)])
def test_oracle_kf_search_against_python(built, mode):
    from lld_slam_b200 import api, synth
    p = synth.make_kf_search_batch(2, 500, 400, 41 + mode[0] + 2 * mode[1], chi2_gate=mode[0], sequential_claims=mode[1])
    o = api.kf_search(p, impl="oracle")
    r = _kf_search_python(p)
    for k in ("match", "n_matches", "best_idx", "best_dist"):
        assert np.array_equal(o[k], r[k]), k
    assert int(o["n_matches"].sum()) > 100


def _tri_search_python(p):
    """Independent transcription of ORBmatcher::SearchForTriangulation (src/ORBmatcher.cc:657-823) and CheckDistEpipolarLine
    (:140-157): dictionaries for the feature vectors, float32 arithmetic, the rotation histogram as lists"""
    f = np.float32
    match12 = np.full(int(p["kp1_off"][-1]), -1, np.int32); nm = np.zeros(p["n_pairs"], np.int32)
    for pr in range(p["n_pairs"]):
        a0, a1 = int(p["kp1_off"][pr]), int(p["kp1_off"][pr + 1]); b0 = int(p["kp2_off"][pr])
        F = p["F12"][pr].reshape(3, 3); ex, ey = p["epipole"][pr]

        def fv(k):
            d = {}
            for n in range(int(p[f"fv{k}_node_off"][pr]), int(p[f"fv{k}_node_off"][pr + 1])):
                d[int(p[f"fv{k}_node"][n])] = [int(i) for i in p[f"fv{k}_idx"][int(p[f"fv{k}_idx_off"][n]):int(p[f"fv{k}_idx_off"][n + 1])]]
            return d
        fv1, fv2 = fv(1), fv(2)
        m12 = np.full(a1 - a0, -1, np.int32)
        hist = [[] for _ in range(30)]
        n = 0
        for node in sorted(set(fv1) & set(fv2)):
            for idx1 in fv1[node]:
                if p["kp1_has_mp"][a0 + idx1]:
                    continue
                s1 = p["kp1_uright"][a0 + idx1] >= 0
                if p["only_stereo"] and not s1:
                    continue
                x1, y1 = p["kp1_xy"][a0 + idx1]
                best, bi = 50, -1
                for idx2 in fv2[node]:
                    if p["kp2_has_mp"][b0 + idx2]:
                        continue
                    s2 = p["kp2_uright"][b0 + idx2] >= 0
                    if p["only_stereo"] and not s2:
                        continue
                    dist = int(np.unpackbits(np.bitwise_xor(p["kp1_desc"][a0 + idx1], p["kp2_desc"][b0 + idx2])).sum())
                    if dist > 50 or dist > best:
                        continue
                    x2, y2 = p["kp2_xy"][b0 + idx2]; o2 = int(p["kp2_octave"][b0 + idx2])
                    if not s1 and not s2:
                        dx = f(ex) - x2; dy = f(ey) - y2
                        if f(dx * dx) + f(dy * dy) < f(100) * p["scale_factors"][o2]:
                            continue
                    a = f(f(x1 * F[0, 0]) + f(y1 * F[1, 0])) + F[2, 0]
                    b = f(f(x1 * F[0, 1]) + f(y1 * F[1, 1])) + F[2, 1]
                    c = f(f(x1 * F[0, 2]) + f(y1 * F[1, 2])) + F[2, 2]
                    num = f(f(a * x2) + f(b * y2)) + c
                    den = f(a * a) + f(b * b)
                    if den == 0:
                        continue
                    dsqr = f(f(num * num) / den)
                    if float(dsqr) < 3.84 * float(p["level_sigma2"][o2]):
                        bi, best = idx2, dist
                if bi >= 0:
                    m12[idx1] = bi; n += 1
                    if p["check_orientation"]:
                        rot = p["kp1_angle"][a0 + idx1] - p["kp2_angle"][b0 + bi]
                        if rot < 0:
                            rot = f(rot + f(360))
                        b_ = int(np.floor(float(f(rot * f(1.0 / 30))) + 0.5))     # C round(): half away from zero, rot >= 0
                        if b_ == 30:
                            b_ = 0
                        hist[b_].append(idx1)
        if p["check_orientation"]:
            sizes = [len(h) for h in hist]
            m1 = m2 = m3 = 0; i1 = i2 = i3 = -1
            for i, s_ in enumerate(sizes):
                if s_ > m1:
                    m3, m2, m1 = m2, m1, s_; i3, i2, i1 = i2, i1, i
                elif s_ > m2:
                    m3, m2 = m2, s_; i3, i2 = i2, i
                elif s_ > m3:
                    m3, i3 = s_, i
            if m2 < 0.1 * m1:
                i2 = i3 = -1
            elif m3 < 0.1 * m1:
                i3 = -1
            for i in range(30):
                if i in (i1, i2, i3):
                    continue
                for j in hist[i]:
                    m12[j] = -1; n -= 1
        match12[a0:a1] = m12; nm[pr] = n
    return dict(match12=match12, n_matches=nm)


@pytest.mark.parametrize("mode", [(0, 1), (1, 0)])
def test_oracle_tri_search_against_python(built, mode):
    from lld_slam_b200 import api, synth
    p = synth.make_tri_search_batch(2, 500, 61 + mode[0], n_nodes=120, only_stereo=mode[0], check_orientation=mode[1])
    o = api.tri_search(p, impl="oracle")
    r = _tri_search_python(p)
    assert np.array_equal(o["match12"], r["match12"]) and np.array_equal(o["n_matches"], r["n_matches"])
    assert int(o["n_matches"].sum()) > (60 if mode[0] else 150)


def _bow_search_python(p):
    """Independent transcription of the two ORBmatcher::SearchByBoW overloads (src/ORBmatcher.cc:159-288, :522-655)"""
    f = np.float32
    match12 = np.full(int(p["kp1_off"][-1]), -1, np.int32); nm = np.zeros(p["n_pairs"], np.int32)
    for pr in range(p["n_pairs"]):
        a0, a1 = int(p["kp1_off"][pr]), int(p["kp1_off"][pr + 1]); b0, b1 = int(p["kp2_off"][pr]), int(p["kp2_off"][pr + 1])

        def fv(k):
            d = {}
            for n in range(int(p[f"fv{k}_node_off"][pr]), int(p[f"fv{k}_node_off"][pr + 1])):
                d[int(p[f"fv{k}_node"][n])] = [int(i) for i in p[f"fv{k}_idx"][int(p[f"fv{k}_idx_off"][n]):int(p[f"fv{k}_idx_off"][n + 1])]]
            return d
        fv1, fv2 = fv(1), fv(2)
        m12 = np.full(a1 - a0, -1, np.int32); taken = np.zeros(b1 - b0, bool)
        hist = [[] for _ in range(30)]
        n = 0
        for node in sorted(set(fv1) & set(fv2)):
            for idx1 in fv1[node]:
                if not p["kp1_valid"][a0 + idx1]:
                    continue
                bd1, bi, bd2 = 256, -1, 256
                for idx2 in fv2[node]:
                    if taken[idx2] or not p["kp2_valid"][b0 + idx2]:
                        continue
                    dist = int(np.unpackbits(np.bitwise_xor(p["kp1_desc"][a0 + idx1], p["kp2_desc"][b0 + idx2])).sum())
                    if dist < bd1:
                        bd2, bd1, bi = bd1, dist, idx2
                    elif dist < bd2:
                        bd2 = dist
                ok = bd1 < 50 if p["strict_th"] else bd1 <= 50
                if ok and f(bd1) < f(p["nn_ratio"]) * f(bd2):
                    m12[idx1] = bi; taken[bi] = True; n += 1
                    if p["check_orientation"]:
                        rot = p["kp1_angle"][a0 + idx1] - p["kp2_angle"][b0 + bi]
                        if rot < 0:
                            rot = f(rot + f(360))
                        b_ = int(np.floor(float(f(rot * f(1.0 / 30))) + 0.5))
                        hist[0 if b_ == 30 else b_].append(idx1)
        if p["check_orientation"]:
            sizes = [len(h) for h in hist]
            m1 = m2 = m3 = 0; i1 = i2 = i3 = -1
            for i, s_ in enumerate(sizes):
                if s_ > m1:
                    m3, m2, m1 = m2, m1, s_; i3, i2, i1 = i2, i1, i
                elif s_ > m2:
                    m3, m2 = m2, s_; i3, i2 = i2, i
                elif s_ > m3:
                    m3, i3 = s_, i
            if m2 < 0.1 * m1:
                i2 = i3 = -1
            elif m3 < 0.1 * m1:
                i3 = -1
            for i in range(30):
                if i not in (i1, i2, i3):
                    for j in hist[i]:
                        m12[j] = -1; n -= 1
        match12[a0:a1] = m12; nm[pr] = n
    return dict(match12=match12, n_matches=nm)


@pytest.mark.parametrize("strict", [0, 1])
def test_oracle_bow_search_against_python(built, strict):
    from lld_slam_b200 import api, synth
    p = synth.make_bow_search_batch(2, 500, 71 + strict, n_nodes=40, strict_th=strict, nn_ratio=0.7 if strict else 0.75)
    o = api.bow_search(p, impl="oracle")
    r = _bow_search_python(p)
    assert np.array_equal(o["match12"], r["match12"]) and np.array_equal(o["n_matches"], r["n_matches"])
    assert int(o["n_matches"].sum()) > 150
    m = o["match12"][o["match12"] >= 0]           # a side-2 keypoint is matched at most once per pair
    assert len(np.unique(m + 100000 * np.repeat(np.arange(2), 500)[o["match12"] >= 0])) == len(m)


# ------------------------------------------------------------------------------------------------------------------
# SURVEY §8 rows a8 / a9: the two Frame-level SearchByProjection variants, pinned by plain-Python transcriptions
# ------------------------------------------------------------------------------------------------------------------
class _PyGrid:
    """Frame::AssignFeaturesToGrid / PosInGrid / GetFeaturesInArea (src/Frame.cc:294-309, 391-456) in float32, dictionary of cells"""

    def __init__(self, g, xy):
        f = np.float32
        self.minx, self.miny = f(g["min_x"]), f(g["min_y"])
        self.winv = f(64) / (f(g["max_x"]) - self.minx)
        self.hinv = f(48) / (f(g["max_y"]) - self.miny)
        self.xy = xy
        self.cells = {}
        for i in range(len(xy)):
            px = int(np.round((xy[i, 0] - self.minx) * self.winv)); py = int(np.round((xy[i, 1] - self.miny) * self.hinv))
            if 0 <= px < 64 and 0 <= py < 48:
                self.cells.setdefault((px, py), []).append(i)

    def area(self, x, y, r, min_level, max_level, octv):
        x0 = max(0, int(np.floor((x - self.minx - r) * self.winv)))
        x1 = min(63, int(np.ceil((x - self.minx + r) * self.winv)))
        y0 = max(0, int(np.floor((y - self.miny - r) * self.hinv)))
        y1 = min(47, int(np.ceil((y - self.miny + r) * self.hinv)))
        if x0 >= 64 or x1 < 0 or y0 >= 48 or y1 < 0:
            return []
        check = min_level > 0 or max_level >= 0
        out = []
        for ix in range(x0, x1 + 1):
            for iy in range(y0, y1 + 1):
                for idx in self.cells.get((ix, iy), ()):
                    if check:
                        if int(octv[idx]) < min_level:
                            continue
                        if max_level >= 0 and int(octv[idx]) > max_level:
                            continue
                    if abs(self.xy[idx, 0] - x) < r and abs(self.xy[idx, 1] - y) < r:
                        out.append(idx)
        return out


def _three_maxima(sizes):
    m1 = m2 = m3 = 0; i1 = i2 = i3 = -1
    for i, s_ in enumerate(sizes):
        if s_ > m1:
            m3, m2, m1 = m2, m1, s_; i3, i2, i1 = i2, i1, i
        elif s_ > m2:
            m3, m2 = m2, s_; i3, i2 = i2, i
        elif s_ > m3:
            m3, i3 = s_, i
    if m2 < 0.1 * m1:
        i2 = i3 = -1
    elif m3 < 0.1 * m1:
        i3 = -1
    return i1, i2, i3


def _ham(a, b):
    return int(np.unpackbits(np.bitwise_xor(a, b)).sum())


def _sbp_frame_python(p):
    """ORBmatcher::SearchByProjection(Frame&, const Frame&, th, bMono) src/ORBmatcher.cc:1328-1470: cv::Mat float products as
    double-accumulating gemms rounded once, everything else float32 in source order"""
    f, f64 = np.float32, np.float64
    g = p["geom"]
    fx, fy, cx, cy, bf, b = (f(g[k]) for k in ("fx", "fy", "cx", "cy", "bf", "b"))
    sf = np.asarray(g["scale_factors"], f)
    nq = int(p["last_off"][-1])
    best_idx = np.full(nq, -1, np.int32); best_dist = np.full(nq, 256, np.int32)
    match = np.full(int(p["cur_off"][-1]), -1, np.int32); nm = np.zeros(p["n_pairs"], np.int32)
    for pr in range(p["n_pairs"]):
        c0, c1 = int(p["cur_off"][pr]), int(p["cur_off"][pr + 1]); l0, l1 = int(p["last_off"][pr]), int(p["last_off"][pr + 1])
        xy = p["cur_xy"][c0:c1]; octv = p["cur_octave"][c0:c1]
        G = _PyGrid(g, xy)
        Tc = p["cur_Tcw"][pr]; Tl = p["last_Tcw"][pr]
        Rcw = Tc[:9].reshape(3, 3).astype(f64); tcw = Tc[9:].astype(f64)
        Rlw = Tl[:9].reshape(3, 3).astype(f64); tlw = Tl[9:].astype(f64)
        twc = (-(Rcw.T @ tcw)).astype(f)
        tlc = (Rlw @ twc.astype(f64) + tlw).astype(f)
        fwd = bool(tlc[2] > b) and not p["mono"]
        bwd = bool(-tlc[2] > b) and not p["mono"]
        claimed = p["cur_claimed"][c0:c1].astype(bool).copy()
        m = np.full(c1 - c0, -1, np.int32)
        hist = [[] for _ in range(30)]
        n = 0
        for i in range(l1 - l0):
            q = l0 + i
            if not p["last_valid"][q]:
                continue
            pc = (Rcw @ p["last_xw"][q].astype(f64) + tcw).astype(f)
            invz = f(f64(1.0) / f64(pc[2]))
            if invz < 0 and not p.get("allow_negative_depth", 0):
                continue
            u = f(f(fx * pc[0]) * invz) + cx; v = f(f(fy * pc[1]) * invz) + cy
            if u < f(g["min_x"]) or u > f(g["max_x"]) or v < f(g["min_y"]) or v > f(g["max_y"]):
                continue
            lo = int(p["last_octave"][q])
            r = f(p["th"]) * sf[lo]
            if fwd:
                cand = G.area(u, v, r, lo, -1, octv)
            elif bwd:
                cand = G.area(u, v, r, 0, lo, octv)
            else:
                cand = G.area(u, v, r, lo - 1, lo + 1, octv)
            bd, bi = 256, -1
            for i2 in cand:
                if claimed[i2]:
                    continue
                if p["cur_uright"][c0 + i2] > 0:
                    ur = u - f(bf * invz)
                    if abs(ur - p["cur_uright"][c0 + i2]) > r:
                        continue
                d = _ham(p["last_desc"][q], p["cur_desc"][c0 + i2])
                if d < bd:
                    bd, bi = d, i2
            th_high = p.get("th_high", 0) or 100
            if bd <= th_high:
                m[bi] = i
                if p["last_has_obs"][q]:
                    claimed[bi] = True
                n += 1
                best_idx[q] = bi; best_dist[q] = bd
                if p["check_orientation"]:
                    rot = p["last_angle"][q] - p["cur_angle"][c0 + bi]
                    if rot < 0:
                        rot = f(rot + f(360))
                    b_ = int(np.floor(float(f(rot * f(1.0 / 30))) + 0.5))
                    hist[0 if b_ == 30 else b_].append(bi)
        if p["check_orientation"]:
            keep = _three_maxima([len(h) for h in hist])
            for i in range(30):
                if i not in keep:
                    for j in hist[i]:
                        m[j] = -1; n -= 1
        match[c0:c1] = m; nm[pr] = n
    return dict(match=match, n_matches=nm, best_idx=best_idx, best_dist=best_dist)


def _sbp_mappoints_python(p):
    """ORBmatcher::SearchByProjection(Frame&, const vector<MapPoint*>&, th) src/ORBmatcher.cc:45-129"""
    f = np.float32
    g = p["geom"]
    sf = np.asarray(g["scale_factors"], f)
    nq = int(p["mp_off"][-1])
    best_idx = np.full(nq, -1, np.int32); best_dist = np.full(nq, 256, np.int32)
    match = np.full(int(p["cur_off"][-1]), -1, np.int32); nm = np.zeros(p["n_pairs"], np.int32)
    for pr in range(p["n_pairs"]):
        c0, c1 = int(p["cur_off"][pr]), int(p["cur_off"][pr + 1])
        xy = p["cur_xy"][c0:c1]; octv = p["cur_octave"][c0:c1]
        G = _PyGrid(g, xy)
        claimed = p["cur_claimed"][c0:c1].astype(bool).copy()
        m = np.full(c1 - c0, -1, np.int32)
        n = 0
        for q in range(int(p["mp_off"][pr]), int(p["mp_off"][pr + 1])):
            if not p["mp_valid"][q]:
                continue
            lvl = int(p["mp_level"][q])
            r = f(2.5) if float(p["mp_viewcos"][q]) > 0.998 else f(4.0)
            if p["th"] != 1.0:
                r = f(r * f(p["th"]))
            u, v, ur = (f(x) for x in p["mp_proj"][q])
            rs = f(r * sf[lvl])
            cand = G.area(u, v, rs, lvl - 1, lvl, octv)
            bd = bd2 = 256; bl = bl2 = -1; bi = -1
            for idx in cand:
                if claimed[idx]:
                    continue
                if p["cur_uright"][c0 + idx] > 0:
                    if abs(ur - p["cur_uright"][c0 + idx]) > f(r * sf[lvl]):
                        continue
                d = _ham(p["mp_desc"][q], p["cur_desc"][c0 + idx])
                if d < bd:
                    bd2, bd = bd, d; bl2, bl = bl, int(octv[idx]); bi = idx
                elif d < bd2:
                    bl2 = int(octv[idx]); bd2 = d
            if bd <= 100:
                if bl == bl2 and bd > f(p["nn_ratio"]) * f(bd2):
                    continue
                m[bi] = q - int(p["mp_off"][pr])
                if p["mp_has_obs"][q]:
                    claimed[bi] = True
                n += 1
                best_idx[q] = bi; best_dist[q] = bd
        match[c0:c1] = m; nm[pr] = n
    return dict(match=match, n_matches=nm, best_idx=best_idx, best_dist=best_dist)


def test_oracle_sbp_frame_against_python(built):
    from lld_slam_b200 import api, synth
    p = synth.make_sbp_frame_batch(5, 400, 51)          # forward / backward / static pairs
    o = api.sbp_frame(p, impl="oracle"); r = _sbp_frame_python(p)
    for k in ("match", "n_matches", "best_idx", "best_dist"):
        assert np.array_equal(o[k], r[k]), k
    assert int(o["n_matches"].sum()) > 400
    q = dict(p); q["mono"] = 1; q["th_high"] = 30; q["allow_negative_depth"] = 1     # the relocalisation variant (:1472-1599)
    q["cur_uright"] = np.full_like(p["cur_uright"], -1.0); q["last_has_obs"] = np.ones_like(p["last_has_obs"])
    o = api.sbp_frame(q, impl="oracle"); r = _sbp_frame_python(q)
    for k in ("match", "n_matches", "best_idx", "best_dist"):
        assert np.array_equal(o[k], r[k]), k


def test_oracle_sbp_mappoints_against_python(built):
    from lld_slam_b200 import api, synth
    p = synth.make_sbp_mp_batch(4, 500, 400, 53)
    o = api.sbp_mappoints(p, impl="oracle"); r = _sbp_mappoints_python(p)
    for k in ("match", "n_matches", "best_idx", "best_dist"):
        assert np.array_equal(o[k], r[k]), k
    assert int(o["n_matches"].sum()) > 300


def _line_match_numpy(p):
    """TwoFrameLineMatcher::MatchLines / CheckLinePair (src/TwoFrameLineMatcher.cc:26-124) with vgl::TriangulateLine (src/vgl.cc:78-108),
    ReprojectKeyLineTo3D (src/LineMatching.cc:277-291), vgl::ReprojectLinePointTo3D (src/vgl.cc:336-346) and NormalizedLineEquation
    (:578-585), written with numpy's own solvers (np.linalg.solve for the 3x3 system, np.linalg.lstsq for the 3x2 one) where the
    reference uses colPivHouseholderQr -- the oracle uses closed forms, so the two only share the formulas.  T = I, T_right = T with
    t + R (b, 0, 0) (GetTForRight, src/LineMatching.cc:228-237); descriptor distance = L2 norm of the float rows (the oracle's definition
    of the un-vendored LBDMOD function)."""
    K = np.asarray(p["K"], np.float64).reshape(3, 3)
    b = float(p["baseline"]); tau = float(p["tau"]); min_len = float(p["min_line_length"])
    n_left = int(p["left_off"][-1])
    match = np.full(n_left, -1, np.int32); dist = np.full(n_left, np.inf, np.float32)

    def leq(seg):
        l = K.T @ np.cross(np.array([seg[0], seg[1], 1.0]), np.array([seg[2], seg[3], 1.0]))
        return l / np.linalg.norm(l[:2])

    def length(seg):
        return float(np.hypot(float(seg[0]) - float(seg[2]), float(seg[1]) - float(seg[3])))

    t2 = np.array([b, 0.0, 0.0])
    for pr in range(int(p["n_pairs"])):
        a0, a1 = int(p["left_off"][pr]), int(p["left_off"][pr + 1]); b0, b1 = int(p["right_off"][pr]), int(p["right_off"][pr + 1])
        L = [leq(p["left_seg"][i].astype(np.float64)) for i in range(a0, a1)]
        R = [leq(p["right_seg"][i].astype(np.float64)) for i in range(b0, b1)]
        taken = np.zeros(b1 - b0, bool)
        for j in range(a1 - a0):
            s1 = p["left_seg"][a0 + j].astype(np.float64)
            min_d, min_j = np.finfo(np.float64).max, -1
            for oi in range(b1 - b0):
                if taken[oi]:
                    continue
                if int(p["left_octave"][a0 + j]) != int(p["right_octave"][b0 + oi]):
                    continue
                if length(s1) < min_len or length(p["right_seg"][b0 + oi]) < min_len:
                    continue
                n1, n2 = L[j], R[oi]
                if abs(n1 @ n2) / np.linalg.norm(n1) / np.linalg.norm(n2) > 0.975:
                    continue
                d = np.cross(n1, n2); d = d / np.linalg.norm(d)
                M = np.stack([n1, n2, d]); rhs = np.array([0.0, n2 @ t2, 0.0])
                if np.linalg.matrix_rank(M) < 3:
                    continue
                X0 = np.linalg.solve(M, rhs)
                if np.linalg.norm(X0) < 0.5:
                    continue
                ok = True
                for px, py in ((s1[0], s1[1]), (s1[2], s1[3])):
                    A = np.stack([np.array([px, py, 1.0]), -(K @ d)], 1)
                    sol = np.linalg.lstsq(A, K @ X0, rcond=None)[0]
                    if (X0 + sol[1] * d)[2] < 0:
                        ok = False
                if not ok:
                    continue
                df = p["left_desc"][a0 + j].astype(np.float64) - p["right_desc"][b0 + oi].astype(np.float64)
                dd = float(np.sqrt(df @ df))
                if dd < min_d and dd < tau:
                    min_d, min_j = dd, oi
            if min_j >= 0:
                taken[min_j] = True
                dist[a0 + j] = np.float32(min_d)
            match[a0 + j] = min_j
    return dict(match=match, dist=dist)


def test_oracle_line_match_against_numpy(built):
    from lld_slam_b200 import api, synth
    p = synth.make_line_match_batch(2, 120, 32, 61)
    o = api.line_match(p, impl="oracle"); r = _line_match_numpy(p)
    assert np.array_equal(o["match"], r["match"]) and (o["match"] >= 0).sum() > 40
    fin = np.isfinite(r["dist"])
    assert np.array_equal(np.isfinite(o["dist"]), fin) and np.abs(o["dist"][fin] - r["dist"][fin]).max() <= 1e-6
