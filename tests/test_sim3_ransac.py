"""Sim3Solver (lld_sim3_ransac): an independent Python transcription of iterate / ComputeSim3 / CheckInliers that calls cv2
itself (cv2.reduce, cv2.gemm, cv2.eigen, cv2.norm, cv2.Rodrigues on float32 arrays) pins the CPU oracle; hand-built problems
pin one rule each; the host build of the device math equals the oracle's pieces; on the GPU the batched kernel matches the
oracle with the full budget in one call and as ComputeSim3 rounds of 5, and its winners feed lld_sim3_opt."""
import ctypes as C
import math
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from lld_slam_b200 import api, capi, synth  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HC = os.path.join(ROOT, "tests", "hostcheck")
DEVMATH = os.path.join(HC, "libdevmath_sim3_ransac_host.so")
f32, f64 = np.float32, np.float64


@pytest.fixture(scope="session")
def built_ransac(built):
    """the session's `built` checks only the older libraries: build when the Sim3Solver pieces are missing"""
    if not (os.path.exists(capi.SIM3_RANSAC_ORACLE_PATH) and os.path.exists(DEVMATH) and os.path.exists(capi.LIB_PATH)):
        import __graft_entry__ as g
        g.build()
    return True


# ------------------------------------------------------------------------------------------------------------------
# Python transcription with cv2
# ------------------------------------------------------------------------------------------------------------------
def _horn_cv(P1, P2, fix):
    """Sim3Solver::ComputeSim3 on P1, P2 (3x3 float32, column = point): R, t, s, and T12 / T21 as (A, b) pairs"""
    import cv2
    O1 = f32(cv2.reduce(P1, 1, cv2.REDUCE_SUM) * f32(1.0 / 3))
    O2 = f32(cv2.reduce(P2, 1, cv2.REDUCE_SUM) * f32(1.0 / 3))
    Pr1, Pr2 = f32(P1 - O1), f32(P2 - O2)
    M = cv2.gemm(Pr2, Pr1, 1.0, None, 0.0, flags=cv2.GEMM_2_T)
    m = lambda i, j: f32(M[i, j])   # noqa: E731
    N11 = (m(0, 0) + m(1, 1)) + m(2, 2); N12 = m(1, 2) - m(2, 1); N13 = m(2, 0) - m(0, 2); N14 = m(0, 1) - m(1, 0)
    N22 = (m(0, 0) - m(1, 1)) - m(2, 2); N23 = m(0, 1) + m(1, 0); N24 = m(2, 0) + m(0, 2)
    N33 = (-m(0, 0) + m(1, 1)) - m(2, 2); N34 = m(1, 2) + m(2, 1); N44 = (-m(0, 0) - m(1, 1)) + m(2, 2)
    N = f32([[N11, N12, N13, N14], [N12, N22, N23, N24], [N13, N23, N33, N34], [N14, N24, N34, N44]])
    _, _, evec = cv2.eigen(N)
    vec = np.ascontiguousarray(evec[0, 1:4].reshape(1, 3))
    nrm = cv2.norm(vec)
    ang = math.atan2(nrm, float(evec[0, 0]))
    with np.errstate(all="ignore"):
        vec = f32((2 * ang * (1.0 / nrm) if nrm != 0 else float("nan")) * vec.astype(f64))
    R = cv2.Rodrigues(vec.reshape(3, 1))[0]
    s = f32(1.0)
    if not fix:
        P3 = cv2.gemm(R, Pr2, 1.0, None, 0.0)
        nom = den = 0.0
        for i in range(3):
            for k in range(3):
                nom += float(Pr1[i, k]) * float(P3[i, k])
        for i in range(3):
            for k in range(3):
                den += float(f32(P3[i, k] * P3[i, k]))
        with np.errstate(all="ignore"):
            s = f32(nom / den) if den != 0 else f32(np.nan)
    t = cv2.gemm(R, O2, -float(s), O1, 1.0)
    with np.errstate(all="ignore"):
        sR = f32(s * R)
        sRinv = f32((1.0 / float(s)) * R.T.astype(f64))
    tinv = cv2.gemm(sRinv, t, -1.0, None, 0.0)
    return R, t[:, 0], s, (sR, t[:, 0]), (sRinv, tinv[:, 0])


def _proj(A, b, X, K):
    """Sim3Solver::Project over all points (float32; the 3-long float product as cv::gemm forms it)"""
    Y = []
    for r in range(3):
        acc = f32(f32(A[r, 0] * X[:, 0]) + f32(A[r, 1] * X[:, 1]))
        acc = f32(acc + f32(A[r, 2] * X[:, 2]))
        Y.append(f32(acc.astype(f64) + float(b[r])))
    invz = f32(1) / Y[2]
    return np.stack([f32(K[0] * f32(Y[0] * invz)) + K[2], f32(K[1] * f32(Y[1] * invz)) + K[3]], 1)


def _own(X, K):
    invz = f32(1) / X[:, 2]
    return np.stack([f32(K[0] * f32(X[:, 0] * invz)) + K[2], f32(K[1] * f32(X[:, 1] * invz)) + K[3]], 1)


def _err(a, b):
    d = f32(a - b).astype(f64)
    return f32(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1])


def _check_errors(est, K, x1, x2, thr1, thr2):
    with np.errstate(all="ignore"):
        e1 = _err(_own(x1, K[:4]), _proj(est[3][0], est[3][1], x2, K[:4]))
        e2 = _err(_proj(est[4][0], est[4][1], x1, K[4:]), _own(x2, K[4:]))
    return e1, e2, (e1 < thr1) & (e2 < thr2)


def ransac_python(p):
    """iterate() per problem, in the reference's order; per problem: dict of found, no_more, n_inliers, T12, inlier, its,
    best, hyp counts and the (errors, thresholds) of every evaluated set"""
    res = []
    for pb in range(int(p["n_problems"])):
        a, z = int(p["off"][pb]), int(p["off"][pb + 1])
        h0, h1 = int(p["hyp_off"][pb]), int(p["hyp_off"][pb + 1])
        N = z - a
        K = p["cam"][pb]
        x1, x2 = p["x1c"][a:z], p["x2c"][a:z]
        thr1 = f32(np.floor(9.210 * p["sigma2_1"][a:z].astype(f64)))
        thr2 = f32(np.floor(9.210 * p["sigma2_2"][a:z].astype(f64)))
        its, best = int(p["its_done"][pb]), int(p["best_inliers"][pb])
        r = dict(found=0, no_more=0, n_inliers=0, T12=np.zeros(13, f32), inlier=np.zeros(N, np.uint8), hyp=[], detail=[])
        if N < p["min_inliers"]:
            r["no_more"] = 1
        else:
            cur = 0
            while its < p["max_its"][pb] and cur < p["n_iterations"]:
                idx = p["hyp_idx"][h0 + cur]
                cur += 1
                its += 1
                est = _horn_cv(np.ascontiguousarray(x1[idx].T), np.ascontiguousarray(x2[idx].T), bool(p["fix_scale"][pb]))
                e1, e2, inl = _check_errors(est, K, x1, x2, thr1, thr2)
                c = int(inl.sum())
                r["hyp"].append(c)
                r["detail"].append((e1, e2, thr1, thr2))
                if c >= best:
                    best = c
                    if c > p["min_inliers"]:
                        r.update(found=1, n_inliers=c, inlier=inl.astype(np.uint8),
                                 T12=np.concatenate([est[0].reshape(-1), est[1], [est[2]]]).astype(f32))
                        break
            if not r["found"] and its >= p["max_its"][pb]:
                r["no_more"] = 1
            assert h1 - h0 >= cur
        r["its"], r["best"] = its, best
        res.append(r)
    return res


def _near_threshold(detail, k, tol=1e-5):
    e1, e2, t1, t2 = detail[k]
    return int((np.abs(e1 - t1) <= tol * t1).sum() + (np.abs(e2 - t2) <= tol * t2).sum())


def _compare_python(o, p, py):
    """oracle against the transcription: identical per-set counts except where correspondences lie within 1e-5 of their
    threshold, identical flags / iterations / masks, R t s to float tolerance; returns the number of explained divergences"""
    explained = 0
    for pb, r in enumerate(py):
        h0 = int(p["hyp_off"][pb])
        got = o["hyp_inliers"][h0:h0 + len(r["hyp"])]
        diff = [k for k in range(len(r["hyp"])) if got[k] != r["hyp"][k]]
        if diff:
            k = diff[0]
            assert abs(int(got[k]) - r["hyp"][k]) <= _near_threshold(r["detail"], k), (pb, k, got[k], r["hyp"][k])
            explained += 1
            continue
        a, z = int(p["off"][pb]), int(p["off"][pb + 1])
        assert int(o["found"][pb]) == r["found"] and int(o["no_more"][pb]) == r["no_more"], pb
        assert int(o["its_done"][pb]) == r["its"] and int(o["best_inliers"][pb]) == r["best"], pb
        assert int(o["n_inliers"][pb]) == r["n_inliers"] and np.array_equal(o["inlier"][a:z], r["inlier"]), pb
        if r["found"]:
            T, U = o["T12"][pb], r["T12"]
            assert np.abs(T[:9] - U[:9]).max() < 1e-5, pb
            assert np.abs(T[9:12] - U[9:12]).max() <= 1e-5 * max(1.0, np.abs(U[9:12]).max()), pb
            assert abs(T[12] - U[12]) <= 1e-5 * abs(U[12]), pb
        assert (got[len(r["hyp"]):] == -1).all()
    return explained


@pytest.mark.parametrize("fix", [1, 0])
@pytest.mark.parametrize("seed", [3, 4, 5])
def test_oracle_sim3_ransac_against_python(built_ransac, seed, fix):
    pytest.importorskip("cv2")
    p = synth.make_sim3_ransac_batch(12, 60, seed, fix_scale=fix)
    o = api.sim3_ransac(p, impl="oracle")
    py = ransac_python(p)
    assert _compare_python(o, p, py) <= 1
    assert o["found"].any() and (o["no_more"] == 1).any()   # both outcomes are exercised
    if fix:
        assert (o["T12"][o["found"] == 1, 12] == 1).all()


def test_max_its_against_formula(built_ransac):
    for n in (20, 21, 25, 100, 1000, 5000):
        want = synth.sim3_ransac_max_its_py(n)
        eps = float(f32(f32(20) / f32(n)))
        if n == 20:
            assert want == 1
        else:
            assert want == max(1, min(math.ceil(math.log(0.01) / math.log(1 - eps ** 3)), 300))
        assert api.sim3_ransac_max_its(n) == want, n
    assert api.sim3_ransac_max_its(21) == api.sim3_ransac_max_its(21, 0.99, 20, 300) < 300
    assert api.sim3_ransac_max_its(100) == 300 and api.sim3_ransac_max_its(1000) == 300   # the clamp
    assert api.sim3_ransac_max_its(21, 0.99, 21, 300) == 1
    assert api.sim3_ransac_max_its(100, 0.99, 20, 7) == 7


# ------------------------------------------------------------------------------------------------------------------
# hand-built problems, one rule each
# ------------------------------------------------------------------------------------------------------------------
K0 = f32([500, 500, 320, 240, 500, 500, 320, 240])


def _problem(x1, x2, sets, fix=1, sig1=None, sig2=None, its_done=0, best=0, max_its=300, n_iterations=None):
    x1, x2 = f32(x1).reshape(-1, 3), f32(x2).reshape(-1, 3)
    m = len(x1)
    sets = np.asarray(sets, np.int32).reshape(-1, 3)
    return dict(n_problems=1, cam=K0[None].copy(), fix_scale=np.array([fix], np.int32), off=np.array([0, m], np.int32),
                x1c=np.ascontiguousarray(x1), x2c=np.ascontiguousarray(x2),
                sigma2_1=f32(np.ones(m) if sig1 is None else sig1), sigma2_2=f32(np.ones(m) if sig2 is None else sig2),
                min_inliers=20, max_its=np.array([max_its], np.int32), its_done=np.array([its_done], np.int32),
                best_inliers=np.array([best], np.int32), n_iterations=len(sets) if n_iterations is None else n_iterations,
                hyp_off=np.array([0, len(sets)], np.int32), hyp_idx=np.ascontiguousarray(sets))


def _cloud(m, seed):
    rng = np.random.default_rng(seed)
    return f32(np.stack([rng.uniform(-4, 4, m), rng.uniform(-2, 2, m), rng.uniform(5, 20, m)], 1))


def _shift(x):
    """keyframe 2 = keyframe 1 turned by 5 degrees about y and moved 0.5 m along x (a pure translation makes M symmetric,
    the quaternion's vector part exactly 0 and the reference's v / |v| NaN)"""
    c, s = math.cos(math.radians(5)), math.sin(math.radians(5))
    R = np.array([[c, 0, s], [0, 1, 0], [-s, 0, c]])
    return f32(x.astype(f64) @ R.T - [0.5, 0, 0])


def _scramble(x, bad):
    y = x.copy()
    y[bad] = y[np.roll(bad, 1)]
    return y


def _case_too_few():
    x = _cloud(19, 1)
    return _problem(x, _shift(x), np.zeros((0, 3))), dict(found=0, no_more=1, its=0)


def _case_twenty_vs_twenty_one():
    x = _cloud(40, 2)
    y20 = _scramble(_shift(x), np.arange(20, 40))       # exactly 20 consistent: no success
    y21 = _scramble(_shift(x), np.arange(21, 40))       # 21: success
    p20 = _problem(x, y20, [[0, 1, 2]])
    p21 = _problem(x, y21, [[0, 1, 2]])
    return [p20, p21], [dict(found=0, hyp=[20], best=20), dict(found=1, hyp=[21], n_inliers=21)]


def _case_carried_best():
    x = _cloud(60, 3)
    y = _scramble(_shift(x), np.arange(30, 60))          # 30 consistent
    return _problem(x, y, [[0, 1, 2]], best=31, its_done=4), dict(found=0, hyp=[30], best=31, its=5)


def _case_last_iteration():
    x = _cloud(40, 4)
    y = _shift(x)
    p = _problem(x, y, [[0, 1, 2]], its_done=6, max_its=7, n_iterations=5)
    return p, dict(found=1, no_more=0, its=7)


def _case_integer_threshold():
    # correspondence 0 of keyframe 1 lies 3.0178 px off (err 9.107 in (9, 9.21)): an outlier at octave 0, an inlier at 9.21
    x = _cloud(30, 5)
    y = _shift(x)
    x = x.copy()
    z = x[0, 2]
    x[0, 0] += f32(3.0178 * z / 500)
    return _problem(x, y, [[1, 2, 3]]), dict(found=1, first_out=True)


def _case_behind_camera():
    # a rigid motion that puts the whole cloud behind keyframe 2: projections with a negative depth still agree (no depth test)
    x = _cloud(30, 6)
    y = f32(x * f32([-1, 1, -1]))                       # 180 degrees about y
    return _problem(x, y, [[0, 1, 2]]), dict(found=1, n_inliers=30)


def _case_degenerate():
    x = _cloud(30, 7)
    y = _shift(x)
    x = x.copy(); y = y.copy()
    x[1] = x[0]; y[1] = y[0]; x[2] = x[0]; y[2] = y[0]     # coincident triple (0, 1, 2)
    x[4] = x[3] + f32([1, 1, 1]); y[4] = y[3] + f32([1, 1, 1])   # collinear triple (3, 4, 5)
    x[5] = x[3] + f32([2, 2, 2]); y[5] = y[3] + f32([2, 2, 2])
    return _problem(x, y, [[0, 1, 2], [3, 4, 5]], fix=0), dict(no_nan=True)


def _case_fixed_scale():
    x = _cloud(30, 8)
    return _problem(x, _shift(x), [[0, 1, 2]], fix=1), dict(found=1, s=1.0)


CASES = {"too_few": _case_too_few, "twenty_vs_twenty_one": _case_twenty_vs_twenty_one, "carried_best": _case_carried_best,
         "last_iteration": _case_last_iteration, "integer_threshold": _case_integer_threshold, "behind_camera": _case_behind_camera,
         "degenerate": _case_degenerate, "fixed_scale": _case_fixed_scale}


def _check_case(run, name):
    ps, exps = CASES[name]()
    if isinstance(ps, dict):
        ps, exps = [ps], [exps]
    for p, exp in zip(ps, exps):
        o = run(p)
        if "found" in exp:
            assert int(o["found"][0]) == exp["found"], (name, o)
        if "no_more" in exp:
            assert int(o["no_more"][0]) == exp["no_more"], (name, o)
        if "its" in exp:
            assert int(o["its_done"][0]) == exp["its"], (name, o)
        if "best" in exp:
            assert int(o["best_inliers"][0]) == exp["best"], (name, o)
        if "hyp" in exp:
            assert list(o["hyp_inliers"]) == exp["hyp"], (name, o)
        if "n_inliers" in exp:
            assert int(o["n_inliers"][0]) == exp["n_inliers"], (name, o)
        if exp.get("first_out"):
            e = np.zeros(2, f32)
            est = o["T12"][0]
            dm = C.CDLL(DEVMATH)
            dm.dm_sim3r_errors.restype = C.c_int
            flag = dm.dm_sim3r_errors(_p(est), _p(p["cam"][0]), _p(p["x1c"][0]), _p(p["x2c"][0]), C.c_float(1.0), C.c_float(1.0), _p(e))
            assert 9.0 < e[0] < 9.21 and flag == 0 and o["inlier"][0] == 0 and o["inlier"][1:].all(), e
        if exp.get("no_nan"):
            assert int(o["found"][0]) == 0 or o["n_inliers"][0] > 20
            assert list(o["hyp_inliers"][:1]) == [0]           # the coincident triple: NaN estimate, no inliers
        if "s" in exp:
            assert o["T12"][0, 12] == exp["s"]
        if p is ps[-1] and name == "last_iteration":             # the next call draws nothing and sets bNoMore
            q = dict(p, its_done=o["its_done"].copy(), best_inliers=o["best_inliers"].copy(),
                     hyp_off=np.array([0, 0], np.int32), hyp_idx=np.zeros((0, 3), np.int32))
            o2 = run(q)
            assert int(o2["found"][0]) == 0 and int(o2["no_more"][0]) == 1 and int(o2["its_done"][0]) == 7


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.mark.parametrize("name", sorted(CASES))
def test_hand_built_case(built_ransac, name):
    _check_case(lambda p: api.sim3_ransac(p, impl="oracle"), name)


# ------------------------------------------------------------------------------------------------------------------
# host build of the device math against the oracle's pieces
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fix", [1, 0])
def test_device_math_host_equals_oracle(built_ransac, fix):
    """host g++ builds of both: the Horn estimate agrees to the bit except where glibc's atan2 / sin / cos are reached through
    different but equal-valued expressions (there: 2 ulp of float); projection errors and flags are bit-identical"""
    dm, orc = C.CDLL(DEVMATH), C.CDLL(capi.SIM3_RANSAC_ORACLE_PATH)
    for f in (dm.dm_sim3r_horn, orc.lldo_sim3r_horn, dm.dm_sym4_top_eigvec, orc.lldo_sym4_top_eigvec, dm.dm_rodrigues,
              orc.lldo_rodrigues):
        f.restype = None
    dm.dm_sim3r_errors.restype = C.c_int
    orc.lldo_sim3r_errors.restype = C.c_int
    p = synth.make_sim3_ransac_batch(1, 200, 31 + fix, fix_scale=fix)
    rng = np.random.default_rng(5 + fix)
    n = int(p["off"][1])
    for trial in range(200):
        idx = rng.choice(n, 3, replace=False)
        P1, P2 = np.ascontiguousarray(p["x1c"][idx]), np.ascontiguousarray(p["x2c"][idx])
        a, b = np.zeros(13, f32), np.zeros(13, f32)
        dm.dm_sim3r_horn(_p(P1), _p(P2), fix, _p(a)); orc.lldo_sim3r_horn(_p(P1), _p(P2), fix, _p(b))
        assert np.array_equal(a, b), (trial, a, b)
        Nm = f32(rng.normal(0, 1, (4, 4))); Nm = np.ascontiguousarray(f32(Nm + Nm.T))
        qa, qb = np.zeros(4, f32), np.zeros(4, f32)
        dm.dm_sym4_top_eigvec(_p(Nm), _p(qa)); orc.lldo_sym4_top_eigvec(_p(Nm), _p(qb))
        assert np.array_equal(qa, qb)
        w, V = np.linalg.eigh(Nm.astype(f64))
        assert abs(abs(float(qa.astype(f64) @ V[:, -1])) - 1) < 1e-6   # the largest eigenpair
        v = f32(rng.normal(0, 1, 3)); Ra, Rb = np.zeros(9, f32), np.zeros(9, f32)
        dm.dm_rodrigues(_p(v), _p(Ra)); orc.lldo_rodrigues(_p(v), _p(Rb))
        assert np.array_equal(Ra, Rb)
        for i in rng.choice(n, 4, replace=False):
            ea, eb = np.zeros(2, f32), np.zeros(2, f32)
            fa = dm.dm_sim3r_errors(_p(a), _p(p["cam"][0]), _p(p["x1c"][i]), _p(p["x2c"][i]), C.c_float(p["sigma2_1"][i]),
                                    C.c_float(p["sigma2_2"][i]), _p(ea))
            fb = orc.lldo_sim3r_errors(_p(a), _p(p["cam"][0]), _p(p["x1c"][i]), _p(p["x2c"][i]), C.c_float(p["sigma2_1"][i]),
                                       C.c_float(p["sigma2_2"][i]), _p(eb))
            assert fa == fb and np.array_equal(ea, eb, equal_nan=True)


def test_generator(built_ransac):
    p = synth.make_sim3_ransac_batch(64, [0, 19, 20, 21, 37] + [100] * 59, 9, fix_scale=0)
    N = np.diff(p["off"])
    assert list(N[:5]) == [0, 19, 20, 21, 37]
    assert list(synth.sim3_ransac_budget(p)[:5]) == [0, 0, 1, synth.sim3_ransac_max_its_py(21), synth.sim3_ransac_max_its_py(37)]
    idx = p["hyp_idx"]
    assert (idx[:, 0] != idx[:, 1]).all() and (idx[:, 0] != idx[:, 2]).all() and (idx[:, 1] != idx[:, 2]).all()
    assert set(np.unique(p["sigma2_1"])) <= set(synth.level_sigma2())
    s = iter([0, synth.RAND_MAX, 0])   # swap-with-back: first, last of the remaining, first
    assert synth.draw_minimal_set(5, s) == [0, 3, 4]


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
def _subset(p, keep):
    keep = np.asarray(keep)
    q = dict(p, n_problems=len(keep))
    N = np.diff(p["off"])
    rows = np.concatenate([np.arange(p["off"][i], p["off"][i + 1]) for i in keep]) if len(keep) else np.zeros(0, int)
    q["off"] = np.concatenate([[0], np.cumsum(N[keep])]).astype(np.int32)
    for k in ("x1c", "x2c", "sigma2_1", "sigma2_2"):
        q[k] = np.ascontiguousarray(p[k][rows])
    for k in ("cam", "fix_scale", "max_its", "its_done", "best_inliers"):
        q[k] = np.ascontiguousarray(p[k][keep])
    return q


def _same(g, o, p, strict, py=None):
    """GPU against the oracle, problem by problem; a problem may diverge (not strict: at most 1 in 1000) only when the first
    differing per-set count is explained by a correspondence within 1e-5 of its threshold in the Python transcription"""
    diverged = 0
    for pb in range(int(p["n_problems"])):
        a, z = int(p["off"][pb]), int(p["off"][pb + 1])
        h0, h1 = int(p["hyp_off"][pb]), int(p["hyp_off"][pb + 1])
        ok = (g["found"][pb] == o["found"][pb] and g["no_more"][pb] == o["no_more"][pb] and g["its_done"][pb] == o["its_done"][pb]
              and g["best_inliers"][pb] == o["best_inliers"][pb] and g["n_inliers"][pb] == o["n_inliers"][pb]
              and np.array_equal(g["inlier"][a:z], o["inlier"][a:z]) and np.array_equal(g["hyp_inliers"][h0:h1], o["hyp_inliers"][h0:h1]))
        if ok:
            T, U = g["T12"][pb], o["T12"][pb]
            assert np.all(np.abs(T - U) <= 1e-5 * np.maximum(np.abs(U), 1.0)), (pb, T, U)
            continue
        assert not strict, pb
        k = int(np.argmax(g["hyp_inliers"][h0:h1] != o["hyp_inliers"][h0:h1]))
        r = ransac_python(_subset(dict(p, hyp_off=np.array([0, h1 - h0], np.int32), hyp_idx=p["hyp_idx"][h0:h1]), [pb]))[0]
        assert k < len(r["detail"]) and _near_threshold(r["detail"], k) >= abs(int(g["hyp_inliers"][h0 + k]) - int(o["hyp_inliers"][h0 + k])) > 0, pb
        diverged += 1
    assert diverged <= int(p["n_problems"]) // 1000, diverged


def _profiled(p, ctx):
    out, prof = ctx.profile(lambda: api.sim3_ransac(p, impl="gpu", ctx=ctx))
    return out, set(prof)


def run_rounds(p, run, n_iterations=5, seed=0):
    """LoopClosing::ComputeSim3's loop: rounds of iterate(5) over the candidates neither found nor exhausted, drawing each
    round's sets from one stream; returns the per-candidate final state and the per-round outputs"""
    n = int(p["n_problems"])
    its, best = p["its_done"].copy(), p["best_inliers"].copy()
    found = np.zeros(n, np.uint8); no_more = np.zeros(n, np.uint8); n_in = np.zeros(n, np.int32)
    live = np.arange(n)
    stream = synth.rand_stream(seed)
    rounds = []
    while len(live):
        q = _subset(dict(p, its_done=its, best_inliers=best), live)
        q["n_iterations"] = n_iterations
        synth.draw_sim3_ransac_sets(q, stream)
        o = run(q)
        rounds.append((q, o))
        its[live] = o["its_done"]; best[live] = o["best_inliers"]
        found[live] = o["found"]; no_more[live] = o["no_more"]; n_in[live] = o["n_inliers"]
        live = live[(o["found"] == 0) & (o["no_more"] == 0)]
    return dict(its=its, best=best, found=found, no_more=no_more, n_in=n_in), rounds


@pytest.mark.gpu
@pytest.mark.parametrize("fix", [1, 0])
def test_gpu_sim3_ransac_4096x300(gpu_ctx, fix):
    p = synth.make_sim3_ransac_batch(4096, 300, 201 + fix, fix_scale=fix)
    g, names = _profiled(p, gpu_ctx)
    assert "k_sim3_ransac" in names, names
    o = api.sim3_ransac(p, impl="oracle")
    _same(g, o, p, strict=False)
    assert 0.2 < g["found"].mean() < 0.98 and (g["its_done"] == 300).any()
    # the same candidates as ComputeSim3 rounds of 5
    fg, rg = run_rounds(p, lambda q: api.sim3_ransac(q, impl="gpu", ctx=gpu_ctx), seed=fix)
    fo, ro = run_rounds(p, lambda q: api.sim3_ransac(q, impl="oracle"), seed=fix)
    if len(rg) == len(ro) and all(np.array_equal(a[0]["hyp_idx"], b[0]["hyp_idx"]) for a, b in zip(rg, ro)):
        for (q, a), (_, b) in zip(rg, ro):
            _same(a, b, q, strict=False)
    for k in ("its", "best", "found", "no_more", "n_in"):
        assert (fg[k] != fo[k]).sum() <= 4096 // 1000, k


@pytest.mark.gpu
@pytest.mark.parametrize("fix", [1, 0])
def test_gpu_sim3_ransac_ragged(gpu_ctx, fix):
    p = synth.make_sim3_ransac_batch(6, [0, 19, 20, 21, 37, 2048], 301 + fix, fix_scale=fix)
    _same(api.sim3_ransac(p, impl="gpu", ctx=gpu_ctx), api.sim3_ransac(p, impl="oracle"), p, strict=True)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_gpu_sim3_ransac_hand_built_case(gpu_ctx, name):
    def run(p):
        g = api.sim3_ransac(p, impl="gpu", ctx=gpu_ctx)
        _same(g, api.sim3_ransac(p, impl="oracle"), p, strict=True)
        return g
    _check_case(run, name)


@pytest.mark.gpu
def test_gpu_sim3_ransac_repeated(gpu_ctx):
    p = synth.make_sim3_ransac_batch(256, 300, 401, fix_scale=0)
    a = api.sim3_ransac(p, impl="gpu", ctx=gpu_ctx)
    api.sim3_ransac(synth.make_sim3_ransac_batch(3, [5, 50, 900], 402, fix_scale=1), impl="gpu", ctx=gpu_ctx)
    b = api.sim3_ransac(p, impl="gpu", ctx=gpu_ctx)
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def _bad_inputs():
    base = synth.make_sim3_ransac_batch(3, [30, 40, 50], 501, fix_scale=1)
    base["n_iterations"] = 5
    synth.draw_sim3_ransac_sets(base, synth.rand_stream(1))
    out = []
    def mod(**kw):
        q = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in base.items()}
        for k, v in kw.items():
            if callable(v):
                v(q)
            else:
                q[k] = v
        out.append(q)
    mod(n_problems=-1)
    mod(min_inliers=-1)
    mod(n_iterations=-1)
    mod(off=np.array([0, 40, 30, 120], np.int32))
    mod(off=np.array([1, 31, 71, 121], np.int32))
    mod(hyp_off=np.array([0, 10, 5, 15], np.int32))
    mod(fix_scale=np.array([1, 2, 1], np.int32))
    mod(max_its=np.array([0, 300, 300], np.int32))
    mod(its_done=np.array([-1, 0, 0], np.int32))
    mod(best_inliers=np.array([0, -3, 0], np.int32))
    mod(n_iterations=6)                                                    # set count != budget
    def out_of_range(q): q["hyp_idx"][7, 1] = 30
    mod(x=out_of_range)
    def negative(q): q["hyp_idx"][2, 0] = -1
    mod(x=negative)
    def repeated(q): q["hyp_idx"][11, 2] = q["hyp_idx"][11, 0]
    mod(x=repeated)
    return base, out


@pytest.mark.gpu
def test_gpu_sim3_ransac_rejects_bad_arguments(gpu_ctx):
    base, bad = _bad_inputs()
    for q in bad:
        q.pop("x", None)
        with pytest.raises(RuntimeError):
            api.sim3_ransac(q, impl="gpu", ctx=gpu_ctx)
    _same(api.sim3_ransac(base, impl="gpu", ctx=gpu_ctx), api.sim3_ransac(base, impl="oracle"), base, strict=True)


def _to_sim3(T):
    """lld::ToSim3: g2o::Sim3(R, t, s) with Eigen's Quaterniond(Matrix3d) branch order -> [q (x y z w), t, s]"""
    m = T[:9].astype(f64).reshape(3, 3)
    tr = m[0, 0] + m[1, 1] + m[2, 2]
    q = [0.0] * 4
    if tr > 0:
        t = math.sqrt(tr + 1.0); q[3] = 0.5 * t; t = 0.5 / t
        q[0] = (m[2, 1] - m[1, 2]) * t; q[1] = (m[0, 2] - m[2, 0]) * t; q[2] = (m[1, 0] - m[0, 1]) * t
    else:
        i = 0
        if m[1, 1] > m[0, 0]:
            i = 1
        if m[2, 2] > m[i, i]:
            i = 2
        j, k = (i + 1) % 3, (i + 2) % 3
        t = math.sqrt(m[i, i] - m[j, j] - m[k, k] + 1.0); q[i] = 0.5 * t; t = 0.5 / t
        q[3] = (m[k, j] - m[j, k]) * t; q[j] = (m[j, i] + m[i, j]) * t; q[k] = (m[k, i] + m[i, k]) * t
    return np.array(q + [float(T[9]), float(T[10]), float(T[11]), float(T[12])])


@pytest.mark.gpu
def test_gpu_chain_ransac_then_optimize_sim3(gpu_ctx):
    p = synth.make_sim3_ransac_batch(512, 300, 601, fix_scale=0, outlier_range=(0.05, 0.3))
    g = api.sim3_ransac(p, impl="gpu", ctx=gpu_ctx)
    won = np.where(g["found"] == 1)[0]
    assert len(won) > 0.9 * 512
    q = _subset(p, won)
    K = q["cam"].astype(f64)
    obs1 = np.concatenate([_own(q["x1c"][q["off"][i]:q["off"][i + 1]], q["cam"][i][:4]) for i in range(len(won))])
    obs2 = np.concatenate([_own(q["x2c"][q["off"][i]:q["off"][i + 1]], q["cam"][i][4:]) for i in range(len(won))])
    s = dict(n_problems=len(won), S12=np.ascontiguousarray(np.stack([_to_sim3(g["T12"][i]) for i in won])), cam=np.ascontiguousarray(K),
             fix_scale=q["fix_scale"], th2=np.full(len(won), 10.0, f32), off=q["off"], p1c=q["x1c"], p2c=q["x2c"],
             obs1=np.ascontiguousarray(f32(obs1)), obs2=np.ascontiguousarray(f32(obs2)),
             info1=np.ascontiguousarray(f32(1) / q["sigma2_1"]), info2=np.ascontiguousarray(f32(1) / q["sigma2_2"]),
             its_first=5, its_more_outliers=10, its_more_clean=5)
    r = api.sim3_opt(s, impl="gpu", ctx=gpu_ctx)
    assert (r["n_in"] >= 20).mean() >= 0.9, (r["n_in"] >= 20).mean()


# ------------------------------------------------------------------------------------------------------------------
# shim: lld::Sim3Solver in LoopClosing::ComputeSim3's loop, then lld::Optimizer::OptimizeSim3
# ------------------------------------------------------------------------------------------------------------------
def _shim_build(tmp_path, oracle):
    import subprocess
    src = os.path.join(HC, "shim_sim3_ransac.cpp")
    exe = str(tmp_path / ("shim_sim3_ransac_oracle" if oracle else "shim_sim3_ransac_gpu"))
    if oracle:
        libs, extra = [f"-L{HC}", "-lsim3_ransac_oracle", "-lsim3_oracle", f"-Wl,-rpath,{HC}"], ["-DLLD_SHIM_ORACLE"]
    else:
        d = os.path.join(ROOT, "lld_slam_b200", "csrc")
        libs, extra = [f"-L{d}", "-llldba", f"-Wl,-rpath,{d}"], []
    r = subprocess.run(["g++", "-std=c++14", "-O1", "-Wall", *extra, src, "-o", exe, *libs], stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout
    return exe


def _shim_input(fix, seed, n_cand=6):
    """n_cand loop candidates as keyframe objects (world poses, map points with world positions, keypoints with octaves) and
    vpMatched12 with entries the constructor skips; the candidates' outlier shares rise so that early ones fail"""
    rng = np.random.default_rng(seed)
    p = synth.make_sim3_ransac_batch(n_cand, 60, seed, fix_scale=fix, outlier_range=(0.6, 0.8))
    sig, isig = synth.level_sigma2(), synth.inv_level_sigma2()
    rows = {k: [] for k in ("kind", "X1w", "X2w", "kp1", "kp2", "oct1", "oct2")}
    T1s, T2s, coff, valid = [], [], [0], []
    for c in range(n_cand):
        a, z = int(p["off"][c]), int(p["off"][c + 1])
        m = z - a
        R1 = synth._rodrigues(rng.normal(0, 0.05, 3)); t1 = rng.normal(0, 1, 3)
        R2 = synth._rodrigues(rng.normal(0, 0.05, 3)); t2 = rng.normal(0, 1, 3)
        T1s.append(f32(np.concatenate([R1.reshape(-1), t1]))); T2s.append(f32(np.concatenate([R2.reshape(-1), t2])))
        kind = np.zeros(m + 6, np.int32); kind[m:] = [1, 2, 3, 4, 5, 1]
        kind = kind[rng.permutation(m + 6)]
        X1w = np.zeros((m + 6, 3), f32); X2w = np.zeros((m + 6, 3), f32)
        oct1 = np.zeros(m + 6, np.int32); oct2 = np.zeros(m + 6, np.int32)
        vr = np.where(kind == 0)[0]
        X1w[vr] = f32((p["x1c"][a:z].astype(f64) - t1) @ R1); X2w[vr] = f32((p["x2c"][a:z].astype(f64) - t2) @ R2)
        oct1[vr] = np.searchsorted(sig, p["sigma2_1"][a:z]); oct2[vr] = np.searchsorted(sig, p["sigma2_2"][a:z])
        kp1 = f32(rng.uniform(0, 1241, (m + 6, 2))); kp2 = f32(rng.uniform(0, 376, (m + 6, 2)))
        for k, v in (("kind", kind), ("X1w", X1w), ("X2w", X2w), ("kp1", kp1), ("kp2", kp2), ("oct1", oct1), ("oct2", oct2)):
            rows[k].append(v)
        valid.append(vr)
        coff.append(coff[-1] + m + 6)
    d = {k: np.ascontiguousarray(np.concatenate(v)) for k, v in rows.items()}
    d.update(coff=np.asarray(coff, np.int32), T1=np.ascontiguousarray(np.stack(T1s)), T2=np.ascontiguousarray(np.stack(T2s)),
             cam=f32(p["cam"][0][:4]), fix=np.array([fix], np.int32), level_sigma2=sig, inv_level_sigma2=isig,
             rands=np.asarray([next(s) for s in [synth.rand_stream(seed + 1)] for _ in range(200000)], np.int32))
    return d, valid


def _cv_cam(T, X, double_acc):
    R, t = T[:9].reshape(3, 3), T[9:]
    if double_acc:   # lld::Optimizer::OptimizeSim3's cam_frame
        return f32(np.stack([R[r, 0].astype(f64) * X[:, 0] + R[r, 1].astype(f64) * X[:, 1] + R[r, 2].astype(f64) * X[:, 2] + t[r].astype(f64)
                             for r in range(3)], 1))
    return f32(np.stack([f32(f32(f32(R[r, 0] * X[:, 0]) + f32(R[r, 1] * X[:, 1])) + f32(R[r, 2] * X[:, 2])).astype(f64) + float(t[r])
                         for r in range(3)], 1))


def _direct(d, valid, run_ransac, run_opt):
    """the driver's loop restated with the entry points called directly: one solver per candidate over its valid rows"""
    n_cand = len(valid)
    sig, isig = d["level_sigma2"], d["inv_level_sigma2"]
    cands = []
    for c in range(n_cand):
        a = int(d["coff"][c]); rows = a + valid[c]
        x1 = _cv_cam(d["T1"][c], d["X1w"][rows], False); x2 = _cv_cam(d["T2"][c], d["X2w"][rows], False)
        cands.append(dict(rows=rows, x1=x1, x2=x2, s1=sig[d["oct1"][rows]], s2=sig[d["oct2"][rows]]))
    cam8 = np.concatenate([d["cam"], d["cam"]])
    its = np.zeros(n_cand, np.int32); best = np.zeros(n_cand, np.int32)
    max_its = np.asarray([synth.sim3_ransac_max_its_py(len(c["rows"])) for c in cands], np.int32)
    discarded = np.zeros(n_cand, bool); successes = np.zeros(n_cand, np.int32)
    stream = iter(int(r) for r in d["rands"])
    rounds = 0
    while (~discarded).any():
        rounds += 1
        live = np.where(~discarded)[0]
        q = dict(n_problems=len(live), cam=np.ascontiguousarray(np.tile(cam8, (len(live), 1))),
                 fix_scale=np.full(len(live), int(d["fix"][0]), np.int32),
                 off=np.concatenate([[0], np.cumsum([len(cands[c]["rows"]) for c in live])]).astype(np.int32),
                 x1c=np.ascontiguousarray(np.concatenate([cands[c]["x1"] for c in live])),
                 x2c=np.ascontiguousarray(np.concatenate([cands[c]["x2"] for c in live])),
                 sigma2_1=np.ascontiguousarray(np.concatenate([cands[c]["s1"] for c in live])),
                 sigma2_2=np.ascontiguousarray(np.concatenate([cands[c]["s2"] for c in live])),
                 min_inliers=20, max_its=max_its[live].copy(), its_done=its[live].copy(), best_inliers=best[live].copy(), n_iterations=5)
        synth.draw_sim3_ransac_sets(q, stream)
        o = run_ransac(q)
        its[live] = o["its_done"]; best[live] = o["best_inliers"]
        for j, c in enumerate(live):
            if o["no_more"][j]:
                discarded[c] = True
            if not o["found"][j]:
                continue
            successes[c] += 1
            a0, z0 = int(q["off"][j]), int(q["off"][j + 1])
            rows = cands[c]["rows"][o["inlier"][a0:z0] == 1]
            s = dict(n_problems=1, S12=_to_sim3(o["T12"][j])[None].copy(), cam=cam8.astype(f64)[None].copy(),
                     fix_scale=d["fix"].copy(), th2=np.array([10.0], f32), off=np.array([0, len(rows)], np.int32),
                     p1c=np.ascontiguousarray(_cv_cam(d["T1"][c], d["X1w"][rows], True)),
                     p2c=np.ascontiguousarray(_cv_cam(d["T2"][c], d["X2w"][rows], True)),
                     obs1=np.ascontiguousarray(d["kp1"][rows]), obs2=np.ascontiguousarray(d["kp2"][rows]),
                     info1=np.ascontiguousarray(isig[d["oct1"][rows]]), info2=np.ascontiguousarray(isig[d["oct2"][rows]]),
                     its_first=5, its_more_outliers=10, its_more_clean=5)
            r = run_opt(s)
            if r["n_in"][0] >= 20:
                return dict(matched=c, n_in=int(r["n_in"][0]), S12=r["S12"][0], successes=successes, rounds=rounds)
    return dict(matched=-1, n_in=0, S12=np.zeros(8), successes=successes, rounds=rounds)


def _check_shim(exe, tmp_path, run_ransac, run_opt):
    import subprocess
    import shim_io
    for fix, seed in ((1, 71), (0, 72)):
        d, valid = _shim_input(fix, seed)
        # keypoints at the points' own projections (OptimizeSim3 needs observations that agree with the geometry)
        for c, vr in enumerate(valid):
            rows = int(d["coff"][c]) + vr
            d["kp1"][rows] = _own(_cv_cam(d["T1"][c], d["X1w"][rows], False), d["cam"])
            d["kp2"][rows] = _own(_cv_cam(d["T2"][c], d["X2w"][rows], False), d["cam"])
        fin, fout = str(tmp_path / "ransac_in.bin"), str(tmp_path / "ransac_out.bin")
        shim_io.write(fin, d)
        r = subprocess.run([exe, fin, fout], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        assert r.returncode == 0, r.stdout
        got = shim_io.read(fout)
        ref = _direct(d, valid, run_ransac, run_opt)
        assert int(got["matched"][0]) == ref["matched"] >= 0
        assert int(got["n_in"][0]) == ref["n_in"] and int(got["rounds"][0]) == ref["rounds"]
        assert np.array_equal(got["successes"], ref["successes"])
        assert np.array_equal(got["S12"], ref["S12"])


def test_shim_sim3_solver_on_host(built_ransac, tmp_path):
    _check_shim(_shim_build(tmp_path, True), tmp_path, lambda q: api.sim3_ransac(q, impl="oracle"),
                lambda s: api.sim3_opt(s, impl="oracle"))


@pytest.mark.gpu
def test_gpu_shim_sim3_solver(gpu_ctx, tmp_path):
    _check_shim(_shim_build(tmp_path, False), tmp_path, lambda q: api.sim3_ransac(q, impl="gpu", ctx=gpu_ctx),
                lambda s: api.sim3_opt(s, impl="gpu", ctx=gpu_ctx))
