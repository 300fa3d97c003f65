"""PnPsolver (lld_pnp_ransac): an independent Python transcription of iterate / Refine / CheckInliers and of EPnP's
compute_pose that calls cv2 itself (cv2.SVDecomp, cv2.invert and cv2.solve with DECOMP_SVD) pins the CPU oracle; hand-built
problems pin one rule each; the host build of the device math equals the oracle's pieces; on the GPU the batched kernel
matches the oracle with the full budget in one call and as relocalisation rounds of 5, and its poses feed lld_pose_opt."""
import ctypes as C
import itertools
import math
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from lld_slam_b200 import api, capi, synth  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HC = os.path.join(ROOT, "tests", "hostcheck")
DEVMATH = os.path.join(HC, "libdevmath_pnp_ransac_host.so")
f32, f64 = np.float32, np.float64
RELOC = (0.99, 10, 300, 4, 0.5)   # Tracking::Relocalization's SetRansacParameters


@pytest.fixture(scope="session")
def built_pnp(built):
    """the session's `built` checks only the older libraries: build when the PnPsolver pieces are missing"""
    if not (os.path.exists(capi.PNP_RANSAC_ORACLE_PATH) and os.path.exists(DEVMATH) and os.path.exists(capi.LIB_PATH)):
        import __graft_entry__ as g
        g.build()
    return True


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


# ------------------------------------------------------------------------------------------------------------------
# Python transcription with cv2
# ------------------------------------------------------------------------------------------------------------------
def _qr_solve(A, b):
    A, b = A.copy(), b.copy()
    nr, nc = 6, 4
    A1, A2, x = np.zeros(4), np.zeros(4), np.zeros(4)
    for k in range(nc):
        eta = np.abs(A[k:, k]).max()
        if eta == 0:
            return x
        A[k:, k] /= eta
        sigma = math.sqrt(float((A[k:, k] ** 2).sum()))
        if A[k, k] < 0:
            sigma = -sigma
        A[k, k] += sigma
        A1[k] = sigma * A[k, k]
        A2[k] = -eta * sigma
        for j in range(k + 1, nc):
            tau = float(A[k:, k] @ A[k:, j]) / A1[k]
            A[k:, j] -= tau * A[k:, k]
    for j in range(nc):
        tau = float(A[j:, j] @ b[j:]) / A1[j]
        b[j:] -= tau * A[j:, j]
    x[nc - 1] = b[nc - 1] / A2[nc - 1]
    for i in range(nc - 2, -1, -1):
        x[i] = (b[i] - float(A[i, i + 1:] @ x[i + 1:])) / A2[i]
    return x


def epnp_cv(pw, uv, cam):
    """Lepetit's compute_pose with OpenCV's SVD, invert and solve: R (3x3), t (double)"""
    import cv2
    fu, fv, uc, vc = (float(c) for c in cam)
    pw, uv = pw.astype(f64), uv.astype(f64)
    n = len(pw)
    c0 = pw.mean(0)
    PW0 = pw - c0
    dc, uct, _ = cv2.SVDecomp(PW0.T @ PW0)
    cws = np.vstack([c0] + [c0 + math.sqrt(float(dc[i, 0]) / n) * uct[:, i] for i in range(3)])
    CC = (cws[1:] - cws[0]).T
    _, cci = cv2.invert(CC, flags=cv2.DECOMP_SVD)
    al = np.zeros((n, 4))
    al[:, 1:] = (pw - cws[0]) @ cci.T
    al[:, 0] = 1.0 - al[:, 1] - al[:, 2] - al[:, 3]
    M = np.zeros((2 * n, 12))
    for j in range(4):
        M[0::2, 3 * j] = al[:, j] * fu
        M[0::2, 3 * j + 2] = al[:, j] * (uc - uv[:, 0])
        M[1::2, 3 * j + 1] = al[:, j] * fv
        M[1::2, 3 * j + 2] = al[:, j] * (vc - uv[:, 1])
    _, U, _ = cv2.SVDecomp(M.T @ M)
    ut = U.T
    v = [ut[11], ut[10], ut[9], ut[8]]
    pairs = [(0, 1), (0, 2), (0, 3), (1, 2), (1, 3), (2, 3)]
    dv = [[v[i][3 * a:3 * a + 3] - v[i][3 * b:3 * b + 3] for a, b in pairs] for i in range(4)]
    L = np.zeros((6, 10))
    for i in range(6):
        d = [dv[k][i] for k in range(4)]
        L[i] = [d[0] @ d[0], 2 * d[0] @ d[1], d[1] @ d[1], 2 * d[0] @ d[2], 2 * d[1] @ d[2], d[2] @ d[2], 2 * d[0] @ d[3],
                2 * d[1] @ d[3], 2 * d[2] @ d[3], d[3] @ d[3]]
    rho = np.array([((cws[a] - cws[b]) ** 2).sum() for a, b in pairs])
    sols = []
    for s, cols in enumerate(([0, 1, 3, 6], [0, 1, 2], [0, 1, 2, 3, 4])):
        _, bb = cv2.solve(np.ascontiguousarray(L[:, cols]), rho.reshape(6, 1), flags=cv2.DECOMP_SVD)
        bb = bb[:, 0]
        with np.errstate(all="ignore"):
            if s == 0:
                b0 = math.sqrt(-bb[0]) if bb[0] < 0 else math.sqrt(bb[0])
                sg = -1 if bb[0] < 0 else 1
                betas = np.array([b0, sg * bb[1] / b0, sg * bb[2] / b0, sg * bb[3] / b0])
            else:
                if bb[0] < 0:
                    betas = [math.sqrt(-bb[0]), math.sqrt(-bb[2]) if bb[2] < 0 else 0.0]
                else:
                    betas = [math.sqrt(bb[0]), math.sqrt(bb[2]) if bb[2] > 0 else 0.0]
                if bb[1] < 0:
                    betas[0] = -betas[0]
                betas = np.array(betas + [bb[3] / betas[0] if s == 2 else 0.0, 0.0])
            for _ in range(5):
                B = betas
                A = np.stack([2 * L[:, 0] * B[0] + L[:, 1] * B[1] + L[:, 3] * B[2] + L[:, 6] * B[3],
                              L[:, 1] * B[0] + 2 * L[:, 2] * B[1] + L[:, 4] * B[2] + L[:, 7] * B[3],
                              L[:, 3] * B[0] + L[:, 4] * B[1] + 2 * L[:, 5] * B[2] + L[:, 8] * B[3],
                              L[:, 6] * B[0] + L[:, 7] * B[1] + L[:, 8] * B[2] + 2 * L[:, 9] * B[3]], 1)
                q = np.array([B[0] * B[0], B[0] * B[1], B[1] * B[1], B[0] * B[2], B[1] * B[2], B[2] * B[2], B[0] * B[3], B[1] * B[3],
                              B[2] * B[3], B[3] * B[3]])
                betas = betas + _qr_solve(A, rho - L @ q)
            ccs = sum(betas[i] * v[i] for i in range(4)).reshape(4, 3)
            pcs = al @ ccs
            if pcs[0, 2] < 0:
                pcs = -pcs
            pc0, pw0 = pcs.mean(0), pw.mean(0)
            ABt = (pcs - pc0).T @ (pw - pw0)
            _, u, vt = cv2.SVDecomp(ABt)
            R = u @ vt
            if np.linalg.det(R) < 0:
                R[2] = -R[2]
            t = pc0 - R @ pw0
            Xc = pw @ R.T + t
            err = np.sqrt((uv[:, 0] - (uc + fu * Xc[:, 0] / Xc[:, 2])) ** 2 + (uv[:, 1] - (vc + fv * Xc[:, 1] / Xc[:, 2])) ** 2).mean()
        sols.append((R, t, err))
    k = 0
    if sols[1][2] < sols[0][2]:
        k = 1
    if sols[2][2] < sols[k][2]:
        k = 2
    return sols[k][0], sols[k][1]


def check_inliers_py(R, t, pw, uv, max_err, cam):
    """PnPsolver::CheckInliers: float Xc / Yc / invZc from double expressions, double ue / ve, float distances"""
    fu, fv, uc, vc = (float(c) for c in cam)
    P = pw.astype(f64)
    with np.errstate(all="ignore"):
        Xc = f32(R[0, 0] * P[:, 0] + R[0, 1] * P[:, 1] + R[0, 2] * P[:, 2] + t[0])
        Yc = f32(R[1, 0] * P[:, 0] + R[1, 1] * P[:, 1] + R[1, 2] * P[:, 2] + t[1])
        iz = f32(1 / (R[2, 0] * P[:, 0] + R[2, 1] * P[:, 1] + R[2, 2] * P[:, 2] + t[2]))
        ue = uc + fu * Xc.astype(f64) * iz.astype(f64)
        ve = vc + fv * Yc.astype(f64) * iz.astype(f64)
        dx, dy = f32(uv[:, 0].astype(f64) - ue), f32(uv[:, 1].astype(f64) - ve)
        e2 = f32(f32(dx * dx) + f32(dy * dy))
    return (e2 < max_err).astype(np.uint8), e2


def epnp_oracle(pw, uv, cam):
    """the oracle's compute_pose (lldo_pnp_epnp): R (3x3), t"""
    orc = C.CDLL(capi.PNP_RANSAC_ORACLE_PATH)
    orc.lldo_pnp_epnp.restype = None
    out = np.zeros(12)
    orc.lldo_pnp_epnp(_p(np.ascontiguousarray(pw, f32)), _p(np.ascontiguousarray(uv, f32)), len(pw), _p(np.asarray(cam, f64)), _p(out))
    return out[:9].reshape(3, 3), out[9:]


def ransac_python(p, epnp=epnp_oracle):
    """iterate() per problem in the reference's order, with the given compute_pose; per problem a dict of the outputs, the
    per-set counts and, per set, the errors of its correspondences"""
    res = []
    for pb in range(int(p["n_problems"])):
        a, z = int(p["off"][pb]), int(p["off"][pb + 1])
        h0 = int(p["hyp_off"][pb])
        N = z - a
        cam, pw, uv, me = p["cam"][pb], p["p3dw"][a:z], p["p2d"][a:z], p["max_err"][a:z]
        mi, mx = int(p["min_inliers"][pb]), int(p["max_its"][pb])
        its, best = int(p["its_done"][pb]), int(p["best_inliers"][pb])
        bmask, bT = p["best_mask"][a:z].copy(), p["best_Tcw"][pb].copy()
        r = dict(found=0, no_more=0, n_inliers=0, Tcw=np.zeros(12, f32), inlier=np.zeros(N, np.uint8), hyp=[], errs=[])
        if N < mi:
            r["no_more"] = 1
        else:
            cur = 0
            while its < mx or cur < p["n_iterations"]:
                idx = p["hyp_idx"][h0 + cur]
                cur += 1
                its += 1
                R, t = epnp(pw[idx], uv[idx], cam)
                inl, e2 = check_inliers_py(R, t, pw, uv, me, cam)
                c = int(inl.sum())
                r["hyp"].append(c)
                r["errs"].append(e2)
                if c >= mi:
                    if c > best:
                        bmask, best = inl, c
                        bT = f32(np.concatenate([R.reshape(-1), t]))
                    sel = np.where(bmask == 1)[0]
                    R, t = epnp(pw[sel], uv[sel], cam)
                    inl, _ = check_inliers_py(R, t, pw, uv, me, cam)
                    if inl.sum() > mi:
                        r.update(found=1, n_inliers=int(inl.sum()), inlier=inl, Tcw=f32(np.concatenate([R.reshape(-1), t])))
                        break
            if not r["found"] and its >= mx:
                r["no_more"] = 1
                if best >= mi:
                    r.update(found=1, n_inliers=best, inlier=bmask.copy(), Tcw=bT.copy())
        r.update(its=its, best=best, best_mask=bmask, best_Tcw=bT)
        res.append(r)
    return res


def _compare_python(o, p, py):
    """oracle against the transcription of iterate / Refine / CheckInliers driven by the oracle's compute_pose: every count,
    flag, mask and pose is identical"""
    for pb, r in enumerate(py):
        a, z = int(p["off"][pb]), int(p["off"][pb + 1])
        h0 = int(p["hyp_off"][pb])
        assert list(o["hyp_inliers"][h0:h0 + len(r["hyp"])]) == r["hyp"], pb
        assert (o["hyp_inliers"][h0 + len(r["hyp"]):int(p["hyp_off"][pb + 1])] == -1).all(), pb
        assert int(o["found"][pb]) == r["found"] and int(o["no_more"][pb]) == r["no_more"], pb
        assert int(o["its_done"][pb]) == r["its"] and int(o["best_inliers"][pb]) == r["best"], pb
        assert int(o["n_inliers"][pb]) == r["n_inliers"] and np.array_equal(o["inlier"][a:z], r["inlier"]), pb
        assert np.array_equal(o["best_mask"][a:z], r["best_mask"]) and np.array_equal(o["best_Tcw"][pb], r["best_Tcw"]), pb
        assert np.array_equal(o["Tcw"][pb], r["Tcw"]), pb


@pytest.mark.parametrize("seed", [3, 4, 5])
def test_oracle_iterate_against_python(built_pnp, seed):
    """iterate(), Refine() and CheckInliers (float / double mix) transcribed in Python over the oracle's compute_pose, on fresh
    solvers and on a second round that carries the state"""
    p = synth.make_pnp_ransac_batch(10, 60, seed, n_iterations=5)
    o = api.pnp_ransac(p, impl="oracle")
    _compare_python(o, p, ransac_python(p))
    assert o["found"].any() and (o["no_more"] == 1).any()
    q = dict(p, its_done=o["its_done"], best_inliers=o["best_inliers"], best_mask=o["best_mask"], best_Tcw=o["best_Tcw"])
    synth.draw_pnp_ransac_sets(q, synth.rand_stream(seed + 50))
    _compare_python(api.pnp_ransac(q, impl="oracle"), q, ransac_python(q))


@pytest.mark.parametrize("n", [6, 12, 60, 200])
def test_oracle_epnp_against_cv2(built_pnp, n):
    """the oracle's compute_pose against the Python transcription of Lepetit's epnp.cpp that calls cv2.SVDecomp, cv2.invert
    and cv2.solve (DECOMP_SVD).  With exact correspondences (noise-free keypoints rounded to float32) both recover the true
    pose to 1e-5 (relative) from six correspondences on (four or five leave EPnP's approximations short of it).  Under
    keypoint noise EPnP's answer depends on the control points, whose axes are eigenvectors of PW0^T PW0 with a
    solver-dependent sign: one of the eight sign choices of the transcription's axes reproduces the oracle's pose to 1e-9."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(n)
    real = cv2.SVDecomp
    for noise, trials in ((0.0, 10), (1.0, 10)):
        p = synth.make_pnp_ransac_batch(1, 200, 40 + n, outlier_range=(0.0, 0.0), noise=noise)
        cam, T = p["cam"][0], p["truth_Tcw"][0].astype(f64)
        for _ in range(trials):
            idx = rng.choice(200, n, replace=False)
            pw, uv = p["p3dw"][idx], p["p2d"][idx]
            Ro, to = epnp_oracle(pw, uv, cam)
            if noise == 0.0:
                Rc, tc = epnp_cv(pw, uv, cam)
                for R, t in ((Ro, to), (Rc, tc)):
                    assert np.abs(R.reshape(-1) - T[:9]).max() < 1e-5 and np.abs(t - T[9:]).max() < 1e-5 * max(1.0, np.abs(T[9:]).max())
                continue
            PW0 = pw.astype(f64) - pw.astype(f64).mean(0)
            best = np.inf
            for sg in itertools.product([1.0, -1.0], repeat=3):
                def svd(A, _s=np.array(sg)):
                    w, u, vt = real(A)
                    return (w, u * _s, vt) if A.shape == (3, 3) and np.array_equal(A, PW0.T @ PW0) else (w, u, vt)
                cv2.SVDecomp = svd
                try:
                    Rc, tc = epnp_cv(pw, uv, cam)
                finally:
                    cv2.SVDecomp = real
                best = min(best, max(np.abs(Rc - Ro).max(), np.abs(tc - to).max() / max(1.0, np.abs(to).max())))
            assert best < 1e-9, best


def test_oracle_epnp_four_points(built_pnp):
    """the minimal set: on exact correspondences EPnP from four points does not always recover the pose (its null space is
    four-dimensional and the beta approximations use part of it), so this pins a share.  Over 200 four-point sets of one
    KITTI frame, the oracle's and the cv2 transcription's poses each make all 200 correspondences inliers for at least 30 %
    of the sets (measured: 37 % and 48 %), and every such pose is the true one"""
    pytest.importorskip("cv2")
    p = synth.make_pnp_ransac_batch(1, 200, 44, outlier_range=(0.0, 0.0), noise=0.0)
    cam, T = p["cam"][0], p["truth_Tcw"][0].astype(f64)
    rng = np.random.default_rng(4)
    ok = {"oracle": 0, "cv2": 0}
    for _ in range(200):
        idx = rng.choice(200, 4, replace=False)
        pw, uv = p["p3dw"][idx], p["p2d"][idx]
        for name, (R, t) in (("oracle", epnp_oracle(pw, uv, cam)), ("cv2", epnp_cv(pw, uv, cam))):
            inl, _ = check_inliers_py(R, t, p["p3dw"], p["p2d"], p["max_err"], cam)
            if inl.all():
                ok[name] += 1
                assert np.abs(R.reshape(-1) - T[:9]).max() < 1e-3 and np.abs(t - T[9:]).max() < 0.05, (name, R, t)
    assert ok["oracle"] >= 60 and ok["cv2"] >= 60, ok


@pytest.mark.parametrize("tilt", [0.0, 0.3])
def test_epnp_coplanar_points(built_pnp, tilt):
    """world points on a plane (a wall): PW0^T PW0 has a vanishing axis, so CC is singular; as in OpenCV the pseudo-inverse
    drops that axis and the SVD of ABt has rank 2.  On exact correspondences the oracle recovers the rotation for a plane
    along the image axes and the whole pose for a tilted one, as the cv2 transcription does, and the host build of the device
    math gives the same bits"""
    pytest.importorskip("cv2")
    dm = C.CDLL(DEVMATH)
    dm.dm_pnp_epnp.restype = None
    rng = np.random.default_rng(int(tilt * 10))
    cam = f32([synth.FX, synth.FY, synth.CX, synth.CY])
    for n in (4, 6, 12, 60):
        Xc = np.stack([rng.uniform(-5, 5, n), rng.uniform(-2, 2, n), np.zeros(n)], 1)
        Xc[:, 2] = 20 + tilt * Xc[:, 0]
        Xw = f32(Xc)
        uv = f32(np.stack([cam[0] * Xc[:, 0] / Xc[:, 2] + cam[2], cam[1] * Xc[:, 1] / Xc[:, 2] + cam[3]], 1))
        Ro, to = epnp_oracle(Xw, uv, cam)
        a = np.zeros(12)
        dm.dm_pnp_epnp(_p(np.ascontiguousarray(Xw)), _p(uv), n, _p(cam.astype(f64)), _p(a))
        assert np.array_equal(a, np.concatenate([Ro.reshape(-1), to]))
        assert np.isfinite(a).all()
        if n == 6 or (tilt != 0.0 and n == 4):
            continue   # six points on a plane: EPnP's approximations stop short of the pose here, as in the cv2 transcription
        assert np.abs(Ro - np.eye(3)).max() < 1e-5, (n, Ro)
        if tilt != 0.0:
            Rc, tc = epnp_cv(Xw, uv, cam)
            assert np.abs(to).max() < 1e-4 and np.abs(tc).max() < 1e-4, (n, to, tc)


def test_params_against_formula(built_pnp):
    for n in (0, 3, 9, 10, 11, 19, 20, 21, 25, 60, 100, 200, 1000, 5000):
        for prm in (RELOC, (0.99, 8, 300, 4, 0.4), (0.9, 4, 50, 6, 0.7)):
            assert api.pnp_ransac_params(n, *prm) == synth.pnp_ransac_params_py(n, *prm), (n, prm)
    # relocalisation: min_inliers = (int)(N * 0.5f), at least 10; pow(epsilon, 3): 35 iterations at epsilon 0.5
    assert api.pnp_ransac_params(200, *RELOC) == (100, 35)
    assert api.pnp_ransac_params(21, *RELOC) == (10, math.ceil(math.log(0.01) / math.log(1 - 0.5 ** 3)))
    assert api.pnp_ransac_params(15, *RELOC)[0] == 10                                # raised to minInliers
    assert api.pnp_ransac_params(100, 0.99, 2, 300, 6, 0.01)[0] == 6                 # the minSet floor
    mi, its = api.pnp_ransac_params(40, 0.99, 30, 300, 4, 0.5)                      # epsilon raised to 30 / 40
    assert mi == 30 and its == math.ceil(math.log(0.01) / math.log(1 - float(f32(f32(30) / f32(40))) ** 3))
    assert api.pnp_ransac_params(10, *RELOC) == (10, 1)                              # nMinInliers == N
    assert api.pnp_ransac_params(9, *RELOC)[1] == 1                                  # N < nMinInliers
    assert api.pnp_ransac_params(7, 0.99, 1, 300, 1, 0.45)[0] == 3                  # 7 * 0.45f = 3.15 truncated
    assert api.pnp_ransac_params(1000, 0.99, 10, 300, 4, 0.05)[1] == 300             # the clamp
    # the exponent is 3, not the minimal set's 4
    e = 0.5
    assert api.pnp_ransac_params(200, *RELOC)[1] != math.ceil(math.log(0.01) / math.log(1 - e ** 4))


# ------------------------------------------------------------------------------------------------------------------
# hand-built problems, one rule each
# ------------------------------------------------------------------------------------------------------------------
CAM = f32([500, 500, 320, 240])


def _cloud(m, seed):
    rng = np.random.default_rng(seed)
    return f32(np.stack([rng.uniform(-4, 4, m), rng.uniform(-2, 2, m), rng.uniform(5, 20, m)], 1))


def _project(X, noise=0.0, seed=0):
    rng = np.random.default_rng(seed)
    X = X.astype(f64)
    return f32(np.stack([500 * X[:, 0] / X[:, 2] + 320, 500 * X[:, 1] / X[:, 2] + 240], 1) + rng.normal(0, noise, (len(X), 2)))


def _problem(X, uv, sets, min_inliers=10, max_its=35, its_done=0, best=0, best_mask=None, best_Tcw=None, n_iterations=None,
             max_err=5.991):
    X, uv = f32(X).reshape(-1, 3), f32(uv).reshape(-1, 2)
    m = len(X)
    sets = np.asarray(sets, np.int32).reshape(-1, 4)
    return dict(n_problems=1, cam=CAM[None].copy(), min_inliers=np.array([min_inliers], np.int32),
                max_its=np.array([max_its], np.int32), its_done=np.array([its_done], np.int32),
                best_inliers=np.array([best], np.int32), off=np.array([0, m], np.int32), p2d=np.ascontiguousarray(uv),
                p3dw=np.ascontiguousarray(X), max_err=np.full(m, f32(max_err), f32),
                best_mask=np.zeros(m, np.uint8) if best_mask is None else np.asarray(best_mask, np.uint8),
                best_Tcw=np.zeros((1, 12), f32) if best_Tcw is None else f32(best_Tcw).reshape(1, 12),
                n_iterations=len(sets) if n_iterations is None else n_iterations,
                hyp_off=np.array([0, len(sets)], np.int32), hyp_idx=np.ascontiguousarray(sets))


def _scramble(uv, bad):
    y = uv.copy()
    y[bad] = y[np.roll(bad, 1)]
    return y


def _sets(good, k, seed, X=None, uv=None):
    """k minimal sets from the correspondences good; with X / uv only sets whose EPnP pose (the oracle's compute_pose) makes
    every one of good an inlier: EPnP on four points does not always recover the pose, and a case that pins a rule of
    iterate() needs sets whose counts it knows"""
    rng = np.random.default_rng(seed)
    out = []
    while len(out) < k:
        s = rng.choice(good, 4, replace=False)
        if X is not None:
            R, t = epnp_oracle(X[s], uv[s], CAM)
            inl, _ = check_inliers_py(R, t, X, uv, np.full(len(X), f32(5.991)), CAM)
            if not inl[good].all():
                continue
        out.append(s)
    return out


def _case_too_few():
    X = _cloud(9, 1)
    return _problem(X, _project(X), np.zeros((0, 4))), dict(found=0, no_more=1, its=0)


def _case_or_loop():
    # 35 sets that all fail (count 0 < 10): the first iterate(5) evaluates all 35; the next call exactly 5 more
    X = _cloud(40, 2)
    uv = _project(X)
    uv = _scramble(uv, np.arange(40))
    p = _problem(X, uv, _sets(np.arange(40), 35, 2), n_iterations=5)
    return p, dict(found=0, no_more=1, its=35, next_call=5)


def _two_groups(seed):
    """60 correspondences: 0..29 agree with the identity pose (group A), 30..59 with the camera moved 0.5 m along x (group B,
    12 to 50 px from A's projections)"""
    X = _cloud(60, seed)
    uv = _project(X)
    uv[30:] = _project(X[30:] - f32([0.5, 0.0, 0.0]))
    return X, uv


def _case_refine_carried_from_set():
    # set 0 (group A) counts 30 and becomes the best; its Refine lands on 30, not > min_inliers 30.  Set 1 (group B) ties at
    # 30: not a new best (strict >), it still refines (on A's mask) and fails.  After the budget the call returns set 0's
    # mask and pose: group A, not B
    X, uv = _two_groups(3)
    sets = _sets(np.arange(30), 1, 3, X, uv) + _sets(np.arange(30, 60), 1, 3, X, uv)
    p = _problem(X, uv, sets, min_inliers=30, max_its=2)
    return p, dict(found=1, no_more=1, hyp=[30, 30], best=30, n_inliers=30, mask=np.arange(60) < 30, returns_best=True)
def _case_refine_exactly_min():
    # 25 consistent: every good set counts 25 >= min_inliers 25, Refine lands on 25, not > 25: it fails and the loop goes on
    X = _cloud(50, 4)
    uv = _scramble(_project(X), np.arange(25, 50))
    p = _problem(X, uv, _sets(np.arange(25), 3, 4, X, uv), min_inliers=25, max_its=3)
    return p, dict(found=1, no_more=1, its=3, hyp=[25, 25, 25], best=25, n_inliers=25)


def _case_refine_carried_from_call():
    # the best comes from an earlier call: 30 inliers, mask = group B.  The one set of this call (group A) counts 30: >=
    # min_inliers 20 and a tie, so no new best; Refine runs on the carried mask (group B), not on the set's own (group A),
    # succeeds and returns group B's mask with a pose 0.5 m away from the set's
    X, uv = _two_groups(5)
    mask = (np.arange(60) >= 30).astype(np.uint8)
    p = _problem(X, uv, _sets(np.arange(30), 1, 5, X, uv), min_inliers=20, max_its=35, its_done=35, best=30, best_mask=mask,
                 best_Tcw=np.zeros(12), n_iterations=1)
    return p, dict(found=1, no_more=0, its=36, best=30, hyp=[30], n_inliers=30, mask=np.arange(60) >= 30, tx=-0.5)


def _case_budget_exhausted_with_best():
    # min_inliers 12 and 12 consistent correspondences: every set reaches 12 and its Refine lands on 12 (not > 12); after the
    # budget the call returns mBestTcw with the best mask and count, no_more = 1
    X = _cloud(40, 6)
    uv = _scramble(_project(X), np.arange(12, 40))
    p = _problem(X, uv, _sets(np.arange(12), 2, 6, X, uv), min_inliers=12, max_its=2)
    return p, dict(found=1, no_more=1, its=2, best=12, n_inliers=12, returns_best=True)


def _case_budget_exhausted_below_min():
    X = _cloud(40, 7)
    uv = _scramble(_project(X), np.arange(8, 40))
    p = _problem(X, uv, _sets(np.arange(8), 3, 7, X, uv), min_inliers=10, max_its=3)
    return p, dict(found=0, no_more=1, its=3, best=0, hyp=[8, 8, 8])


def _case_degenerate():
    X = _cloud(30, 8)
    X = X.copy()
    X[1] = X[0]; X[2] = X[0]; X[3] = X[0]                        # four coincident points: NaN, all outliers
    X[5] = X[4] + f32([1, 1, 1]); X[6] = X[4] + f32([2, 2, 2]); X[7] = X[4] + f32([3, 3, 3])   # collinear
    p = _problem(X, _project(X), [[0, 1, 2, 3], [4, 5, 6, 7]], max_its=2)
    return p, dict(degenerate=True)


def _case_behind_camera():
    # 10 world points mirrored through the camera centre (behind it) project where their originals do: CheckInliers has no
    # depth test, so the sets of front points count them as inliers
    X = _cloud(30, 9)
    uv = _project(X)
    Xb = np.concatenate([X, -X[:10]])
    uvb = np.concatenate([uv, uv[:10]])
    return _problem(Xb, uvb, [[10, 11, 12, 13]], max_its=1), dict(found=1, n_inliers=40)


CASES = {"too_few": _case_too_few, "or_loop": _case_or_loop, "refine_tie_carried_from_set": _case_refine_carried_from_set,
         "refine_exactly_min": _case_refine_exactly_min, "refine_carried_from_call": _case_refine_carried_from_call,
         "budget_exhausted_with_best": _case_budget_exhausted_with_best,
         "budget_exhausted_below_min": _case_budget_exhausted_below_min, "degenerate": _case_degenerate,
         "behind_camera": _case_behind_camera}


def _check_case(run, name):
    p, exp = CASES[name]()
    o = run(p)
    for k, ok in (("found", "found"), ("no_more", "no_more"), ("its", "its_done"), ("best", "best_inliers"),
                  ("n_inliers", "n_inliers")):
        if k in exp:
            assert int(o[ok][0]) == exp[k], (name, k, o)
    if "hyp" in exp:
        assert list(o["hyp_inliers"]) == exp["hyp"], (name, o)
    if "mask" in exp:
        assert np.array_equal(o["inlier"], exp["mask"].astype(np.uint8)), (name, o["inlier"])
    if "tx" in exp:
        assert abs(float(o["Tcw"][0, 9]) - exp["tx"]) < 1e-3, o["Tcw"]
    if exp.get("returns_best"):
        assert np.array_equal(o["Tcw"][0], o["best_Tcw"][0]) and np.array_equal(o["inlier"], o["best_mask"])
    if exp.get("degenerate"):
        assert int(o["hyp_inliers"][0]) == 0 and int(o["hyp_inliers"][1]) < 10 and int(o["found"][0]) == 0
    if "next_call" in exp:
        q = dict(p, its_done=o["its_done"].copy(), best_inliers=o["best_inliers"].copy(), best_mask=o["best_mask"].copy(),
                 best_Tcw=o["best_Tcw"].copy())
        synth.draw_pnp_ransac_sets(q, synth.rand_stream(1))
        assert int(q["hyp_off"][-1]) == exp["next_call"]
        o2 = run(q)
        assert (o2["hyp_inliers"] >= 0).sum() == exp["next_call"] and int(o2["its_done"][0]) == exp["its"] + exp["next_call"]
        assert int(o2["no_more"][0]) == 1


@pytest.mark.parametrize("name", sorted(CASES))
def test_hand_built_case(built_pnp, name):
    _check_case(lambda p: api.pnp_ransac(p, impl="oracle"), name)


# ------------------------------------------------------------------------------------------------------------------
# host build of the device math against the oracle's pieces
# ------------------------------------------------------------------------------------------------------------------
def test_device_math_host_equals_oracle(built_pnp):
    """host g++ builds of both, -ffp-contract=off: EPnP poses over 4 to 200 correspondences, the Jacobi eigen solver, the SVD
    solves and CheckInliers are bit-identical"""
    dm, orc = C.CDLL(DEVMATH), C.CDLL(capi.PNP_RANSAC_ORACLE_PATH)
    for f in (dm.dm_pnp_epnp, orc.lldo_pnp_epnp, dm.dm_pnp_sym_jacobi, orc.lldo_pnp_sym_jacobi, dm.dm_pnp_svd_solve,
              orc.lldo_pnp_svd_solve):
        f.restype = None
    dm.dm_pnp_inlier.restype = C.c_int
    orc.lldo_pnp_inlier.restype = C.c_int
    p = synth.make_pnp_ransac_batch(1, 200, 31)
    cam = p["cam"][0].astype(f64)
    rng = np.random.default_rng(5)
    for trial in range(120):
        n = [4, 4, 4, 5, 12, 200][trial % 6]
        idx = rng.choice(200, n, replace=False)
        X, uv = np.ascontiguousarray(p["p3dw"][idx]), np.ascontiguousarray(p["p2d"][idx])
        a, b = np.zeros(12), np.zeros(12)
        dm.dm_pnp_epnp(_p(X), _p(uv), n, _p(cam), _p(a)); orc.lldo_pnp_epnp(_p(X), _p(uv), n, _p(cam), _p(b))
        assert np.array_equal(a, b, equal_nan=True), (trial, a, b)
        for i in rng.choice(200, 8, replace=False):
            fa = dm.dm_pnp_inlier(_p(a), _p(p["p3dw"][i]), _p(p["p2d"][i]), C.c_float(p["max_err"][i]), _p(cam))
            fb = orc.lldo_pnp_inlier(_p(a), _p(p["p3dw"][i]), _p(p["p2d"][i]), C.c_float(p["max_err"][i]), _p(cam))
            assert fa == fb
        k = [3, 12][trial % 2]
        S = rng.normal(0, 1, (2 * k, k)); S = S.T @ S
        A1, A2, V1, V2 = S.copy(), S.copy(), np.zeros((k, k)), np.zeros((k, k))
        o1, o2 = np.zeros(k, np.int32), np.zeros(k, np.int32)
        dm.dm_pnp_sym_jacobi(_p(A1), _p(V1), k, _p(o1)); orc.lldo_pnp_sym_jacobi(_p(A2), _p(V2), k, _p(o2))
        assert np.array_equal(A1, A2) and np.array_equal(V1, V2) and np.array_equal(o1, o2)
        w = np.linalg.eigvalsh(S)[::-1]
        assert np.allclose(np.diag(A1)[o1], w, rtol=1e-10, atol=1e-10 * w[0])
        kk = [3, 4, 5][trial % 3]
        L, r = rng.normal(0, 1, (6, kk)), rng.normal(0, 1, 6)
        x1, x2 = np.zeros(kk), np.zeros(kk)
        dm.dm_pnp_svd_solve(_p(L.copy()), 6, kk, _p(r), _p(x1)); orc.lldo_pnp_svd_solve(_p(L.copy()), 6, kk, _p(r), _p(x2))
        assert np.array_equal(x1, x2) and np.allclose(x1, np.linalg.lstsq(L, r, rcond=None)[0], atol=1e-10)


def test_generator(built_pnp):
    p = synth.make_pnp_ransac_batch(40, [0, 9, 10, 11, 20, 200] + [100] * 34, 9)
    N = np.diff(p["off"])
    assert list(N[:6]) == [0, 9, 10, 11, 20, 200]
    assert list(p["min_inliers"][:6]) == [10, 10, 10, 10, 10, 100]
    assert list(synth.pnp_ransac_budget(p)[:6]) == [0, 0, 5, max(5, p["max_its"][3]), max(5, p["max_its"][4]), 35]
    idx = p["hyp_idx"]
    assert all(len(set(r)) == 4 for r in idx.tolist())
    assert set(np.unique(p["max_err"])) <= set(f32(synth.level_sigma2() * f32(5.991)))
    T = p["truth_Tcw"].astype(f64)
    a, z = int(p["off"][5]), int(p["off"][6])
    Xc = p["p3dw"][a:z].astype(f64) @ T[5, :9].reshape(3, 3).T + T[5, 9:]
    assert (Xc[:, 2] > 0).mean() > 0.5
    s = iter([0, synth.RAND_MAX, 0, 0])   # swap-with-back: first, last of the remaining, first, first
    assert synth.draw_minimal_set(6, s, 4) == [0, 4, 5, 3]


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
STATE = ("found", "no_more", "n_inliers", "its_done", "best_inliers")


def _subset(p, keep):
    keep = np.asarray(keep)
    q = dict(p, n_problems=len(keep))
    N = np.diff(p["off"])
    rows = np.concatenate([np.arange(p["off"][i], p["off"][i + 1]) for i in keep]) if len(keep) else np.zeros(0, int)
    q["off"] = np.concatenate([[0], np.cumsum(N[keep])]).astype(np.int32)
    for k in ("p2d", "p3dw", "max_err", "best_mask"):
        q[k] = np.ascontiguousarray(p[k][rows])
    for k in ("cam", "min_inliers", "max_its", "its_done", "best_inliers", "best_Tcw", "truth_Tcw"):
        if k in p:
            q[k] = np.ascontiguousarray(p[k][keep])
    return q


def _same(g, o):
    """device against the oracle: the same algorithm and the same summation order, so every output is identical"""
    for k in g:
        assert np.array_equal(g[k], o[k], equal_nan=True), (k, np.where(g[k] != o[k])[0][:10])


def run_rounds(p, run, n_iterations=5, seed=0):
    """Tracking::Relocalization's loop: rounds of iterate(5) over the candidates neither found nor exhausted, drawing each
    round's sets from one stream and carrying the solver state; returns the final state and the number of rounds"""
    n = int(p["n_problems"])
    st = dict(its_done=p["its_done"].copy(), best_inliers=p["best_inliers"].copy(), best_mask=p["best_mask"].copy(),
              best_Tcw=p["best_Tcw"].copy())
    fin = dict(found=np.zeros(n, np.uint8), no_more=np.zeros(n, np.uint8), n_inliers=np.zeros(n, np.int32),
               Tcw=np.zeros((n, 12), f32), inlier=np.zeros(int(p["off"][-1]), np.uint8))
    live = np.arange(n)
    stream = synth.rand_stream(seed)
    rounds = 0
    while len(live):
        rounds += 1
        q = _subset(dict(p, **st), live)
        q["n_iterations"] = n_iterations
        synth.draw_pnp_ransac_sets(q, stream)
        o = run(q)
        rows = np.concatenate([np.arange(p["off"][i], p["off"][i + 1]) for i in live])
        st["its_done"][live] = o["its_done"]; st["best_inliers"][live] = o["best_inliers"]
        st["best_mask"][rows] = o["best_mask"]; st["best_Tcw"][live] = o["best_Tcw"]
        for k in ("found", "no_more", "n_inliers", "Tcw"):
            fin[k][live] = o[k]
        fin["inlier"][rows] = o["inlier"]
        live = live[(o["found"] == 0) & (o["no_more"] == 0)]
    fin.update(st)
    return fin, rounds


@pytest.mark.gpu
def test_gpu_pnp_ransac_4096x200(gpu_ctx):
    p = synth.make_pnp_ransac_batch(4096, 200, 201, n_iterations=5)
    g, prof = gpu_ctx.profile(lambda: api.pnp_ransac(p, impl="gpu", ctx=gpu_ctx))
    assert "k_pnp_ransac" in prof, prof
    _same(g, api.pnp_ransac(p, impl="oracle"))
    assert 0.2 < g["found"].mean() < 0.98
    fg, ng = run_rounds(p, lambda q: api.pnp_ransac(q, impl="gpu", ctx=gpu_ctx))
    fo, no = run_rounds(p, lambda q: api.pnp_ransac(q, impl="oracle"))
    assert ng == no
    _same(fg, fo)


@pytest.mark.gpu
def test_gpu_pnp_ransac_carried_state(gpu_ctx):
    """a second iterate(5) on every candidate after the first call: its_done from the first call (at or past max_its where it
    spent its budget, below where a Refine succeeded early, so the budget is 5 or the rest of max_its), the carried best
    count, mask and pose (found or not); then a third call carrying the second's"""
    p = synth.make_pnp_ransac_batch(1024, 200, 211)
    q = p
    for rnd in range(2):
        o = api.pnp_ransac(q, impl="oracle")
        q = dict(q, its_done=o["its_done"], best_inliers=o["best_inliers"], best_mask=o["best_mask"], best_Tcw=o["best_Tcw"],
                 n_iterations=5)
        synth.draw_pnp_ransac_sets(q, synth.rand_stream(212 + rnd))
        live = np.diff(q["off"]) >= q["min_inliers"]
        B = synth.pnp_ransac_budget(q)[live]
        assert (q["its_done"][live] > 0).all() and (B == 5).any() and (B > 5).any()
        assert (q["best_inliers"] >= q["min_inliers"]).any() and (q["best_mask"] == 1).any()
        g = api.pnp_ransac(q, impl="gpu", ctx=gpu_ctx)
        _same(g, api.pnp_ransac(q, impl="oracle"))
        assert g["found"].any() and (g["its_done"][live] > q["its_done"][live]).all()


@pytest.mark.gpu
def test_gpu_pnp_ransac_ragged(gpu_ctx):
    p = synth.make_pnp_ransac_batch(7, [0, 9, 10, 11, 37, 200, 2048], 301)
    _same(api.pnp_ransac(p, impl="gpu", ctx=gpu_ctx), api.pnp_ransac(p, impl="oracle"))
    for i in range(7):
        q = _subset(p, [i])
        q["n_iterations"] = 5
        synth.draw_pnp_ransac_sets(q, synth.rand_stream(i))
        _same(api.pnp_ransac(q, impl="gpu", ctx=gpu_ctx), api.pnp_ransac(q, impl="oracle"))


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_gpu_pnp_ransac_hand_built_case(gpu_ctx, name):
    def run(p):
        g = api.pnp_ransac(p, impl="gpu", ctx=gpu_ctx)
        _same(g, api.pnp_ransac(p, impl="oracle"))
        return g
    _check_case(run, name)


@pytest.mark.gpu
def test_gpu_pnp_ransac_repeated(gpu_ctx):
    p = synth.make_pnp_ransac_batch(256, 200, 401)
    a = api.pnp_ransac(p, impl="gpu", ctx=gpu_ctx)
    api.pnp_ransac(synth.make_pnp_ransac_batch(3, [5, 50, 900], 402), impl="gpu", ctx=gpu_ctx)
    b = api.pnp_ransac(p, impl="gpu", ctx=gpu_ctx)
    _same(a, b)


def _bad_inputs():
    base = synth.make_pnp_ransac_batch(3, [30, 40, 50], 501)
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
    mod(n_iterations=-1)
    mod(off=np.array([0, 40, 30, 120], np.int32))
    mod(off=np.array([1, 31, 71, 121], np.int32))
    mod(hyp_off=np.array([0, 10, 5, 15], np.int32))
    mod(min_inliers=np.array([3, 20, 25], np.int32))
    mod(max_its=np.array([0, 35, 35], np.int32))
    mod(its_done=np.array([-1, 0, 0], np.int32))
    mod(best_inliers=np.array([0, -3, 0], np.int32))
    mod(n_iterations=int(base["max_its"].max()) + 1)                     # set count != budget
    def out_of_range(q): q["hyp_idx"][7, 1] = 30
    mod(x=out_of_range)
    def negative(q): q["hyp_idx"][2, 0] = -1
    mod(x=negative)
    def repeated(q): q["hyp_idx"][11, 3] = q["hyp_idx"][11, 0]
    mod(x=repeated)
    return base, out


@pytest.mark.gpu
def test_gpu_pnp_ransac_rejects_bad_arguments(gpu_ctx):
    base, bad = _bad_inputs()
    lib = capi.load_library()
    for q in bad:
        q.pop("x", None)
        prob, keep = capi.fill_struct(capi.PnpRansacProblem, q)
        n, m, h = max(int(base["n_problems"]), 1), int(base["off"][-1]), int(base["hyp_off"][-1]) + 8
        out = dict(found=np.full(n, 7, np.uint8), no_more=np.full(n, 7, np.uint8), n_inliers=np.full(n, 7, np.int32),
                   Tcw=np.full((n, 12), 7, f32), inlier=np.full(m, 7, np.uint8), its_done=np.full(n, 7, np.int32),
                   best_inliers=np.full(n, 7, np.int32), best_mask=np.full(m, 7, np.uint8), best_Tcw=np.full((n, 12), 7, f32),
                   hyp_inliers=np.full(h, 7, np.int32))
        res, keep2 = capi.fill_struct(capi.PnpRansacResult, out)
        assert lib.pnp_ransac(gpu_ctx.handle, C.byref(prob), C.byref(res)) == -2
        for k, v in out.items():
            assert (v == 7).all(), k                                           # outputs untouched
    _same(api.pnp_ransac(base, impl="gpu", ctx=gpu_ctx), api.pnp_ransac(base, impl="oracle"))


@pytest.mark.gpu
def test_gpu_chain_ransac_then_pose_optimization(gpu_ctx):
    """lld_pnp_ransac -> lld_pose_opt on the returned pose and inliers (Tracking::Relocalization's next step) recovers the
    synthetic pose"""
    p = synth.make_pnp_ransac_batch(512, 200, 601, outlier_range=(0.05, 0.4))
    g, _ = run_rounds(p, lambda q: api.pnp_ransac(q, impl="gpu", ctx=gpu_ctx))
    won = np.where(g["found"] == 1)[0]
    assert len(won) > 0.7 * 512
    q = _subset(p, won)
    rows = [np.arange(p["off"][i], p["off"][i + 1]) for i in won]
    sel = [r[g["inlier"][r] == 1] for r in rows]
    n_pt = [len(s) for s in sel]
    allr = np.concatenate(sel)
    F = len(won)
    isig = f32(1) / f32(p["max_err"][allr] / f32(5.991))
    intr = np.array([f32(synth.FX), f32(synth.FY), f32(synth.CX), f32(synth.CY), f32(synth.BF)], f64)
    pose = dict(n_frames=F, Tcw=np.ascontiguousarray(g["Tcw"][won].astype(f64)), intr=np.tile(intr, (F, 1)),
                line_cam=np.tile(np.array([intr[0], intr[2], intr[3], float(f32(synth.BF) / f32(synth.FX))]), (F, 1)),
                pt_off=np.concatenate([[0], np.cumsum(n_pt)]).astype(np.int32), pt_xw=np.ascontiguousarray(p["p3dw"][allr]),
                pt_uvr=np.ascontiguousarray(f32(np.concatenate([p["p2d"][allr], -np.ones((len(allr), 1))], 1))),
                pt_info=np.ascontiguousarray(isig), ln_off=np.zeros(F + 1, np.int32), ln_x0_dir=np.zeros((0, 6)),
                ln_left=np.zeros((0, 4), f32), ln_right=np.zeros((0, 4), f32), ln_info=np.zeros((0, 2)),
                ln_stereo=np.zeros(0, np.uint8), ln_gate_stereo=np.zeros((0, 2), np.uint8),
                delta_mono=float(f32(math.sqrt(5.991))), delta_stereo=float(f32(math.sqrt(7.815))), delta_ln_mono=1.0,
                delta_ln_stereo=1.0, chi2_mono=float(f32(5.991)), chi2_stereo=float(f32(7.815)), gate_ln_mono=1.0,
                gate_ln_stereo=1.0, n_rounds=4, its=10)
    r = api.pose_opt(pose, impl="gpu", ctx=gpu_ctx)
    T, U = r["Tcw"], q["truth_Tcw"].astype(f64)
    rot = np.abs(T[:, :9] - U[:, :9]).max(1)
    tr = np.linalg.norm(T[:, 9:] - U[:, 9:], axis=1)
    assert np.median(rot) < 5e-3 and np.median(tr) < 0.1, (np.median(rot), np.median(tr))
    assert (r["n_inliers"] >= 10).mean() > 0.9


# ------------------------------------------------------------------------------------------------------------------
# shim: lld::PnPsolver in Tracking::Relocalization's loop
# ------------------------------------------------------------------------------------------------------------------
def _shim_build(tmp_path, oracle):
    import subprocess
    src = os.path.join(HC, "shim_pnp_ransac.cpp")
    exe = str(tmp_path / ("shim_pnp_ransac_oracle" if oracle else "shim_pnp_ransac_gpu"))
    if oracle:
        libs, extra = [f"-L{HC}", "-lpnp_ransac_oracle", f"-Wl,-rpath,{HC}"], ["-DLLD_SHIM_ORACLE"]
    else:
        d = os.path.join(ROOT, "lld_slam_b200", "csrc")
        libs, extra = [f"-L{d}", "-llldba", f"-Wl,-rpath,{d}"], []
    r = subprocess.run(["g++", "-std=c++14", "-O1", "-Wall", *extra, src, "-o", exe, *libs], stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout
    return exe


def _shim_input(seed, n_cand=8):
    """one current frame whose keypoints are the candidates' correspondences in turn, each candidate's block with entries the
    constructor skips (no map point, a bad map point); keypoint octaves recovered from max_err"""
    p = synth.make_pnp_ransac_batch(n_cand, [60, 80, 9, 120, 40, 60, 200, 100][:n_cand], seed)
    rng = np.random.default_rng(seed)
    sig = synth.level_sigma2()
    oct_all = np.searchsorted(f32(sig * f32(5.991)), p["max_err"]).astype(np.int32)
    assert np.array_equal(f32(sig[oct_all] * f32(5.991)), p["max_err"])
    kind, Xw, kp, oc, coff = [], [], [], [], [0]
    for c in range(n_cand):
        a, z = int(p["off"][c]), int(p["off"][c + 1])
        m = z - a
        k = np.zeros(m + 6, np.int32); k[m:] = [1, 2, 1, 2, 1, 1]
        perm = rng.permutation(m + 6)
        k = k[perm]
        X = np.zeros((m + 6, 3), f32); u = f32(rng.uniform(0, 1000, (m + 6, 2))); o = rng.integers(0, 8, m + 6).astype(np.int32)
        good = np.where(k == 0)[0]
        X[good] = p["p3dw"][a:z]; u[good] = p["p2d"][a:z]; o[good] = oct_all[a:z]
        kind.append(k); Xw.append(X); kp.append(u); oc.append(o)
        coff.append(coff[-1] + m + 6)
    rands = np.asarray([next(s) for s in [synth.rand_stream(seed + 1)] for _ in range(60000)], np.int32)
    d = dict(coff=np.asarray(coff, np.int32), kind=np.concatenate(kind), Xw=np.ascontiguousarray(np.concatenate(Xw)),
             kp=np.ascontiguousarray(np.concatenate(kp)), oct=np.concatenate(oc), cam=p["cam"][0].copy(), level_sigma2=sig,
             rands=rands)
    return d


def _direct_shim(d, run):
    """the driver's loop restated with lld_pnp_ransac called directly: one problem per candidate over its kept rows"""
    coff, kind = d["coff"], d["kind"]
    nc, NF = len(coff) - 1, int(coff[-1])
    rows = [np.arange(coff[c], coff[c + 1])[kind[coff[c]:coff[c + 1]] == 0] for c in range(nc)]
    me = [f32(d["level_sigma2"][d["oct"][r]] * f32(5.991)) for r in rows]
    prm = [synth.pnp_ransac_params_py(len(r), *RELOC) for r in rows]
    st = dict(its=np.zeros(nc, np.int32), best=np.zeros(nc, np.int32), mask=[np.zeros(len(r), np.uint8) for r in rows],
              T=np.zeros((nc, 12), f32))
    res = dict(found_round=np.full(nc, -1, np.int32), n_in=np.zeros(nc, np.int32), its=np.zeros(nc, np.int32),
               Tcw=np.zeros((nc, 12), f32), inlier=np.zeros((nc, NF), np.uint8))
    stream = iter(int(r) for r in d["rands"])
    live, rounds = list(range(nc)), 0
    while live:
        q = dict(n_problems=len(live), cam=np.ascontiguousarray(np.tile(d["cam"], (len(live), 1))),
                 min_inliers=np.asarray([prm[c][0] for c in live], np.int32), max_its=np.asarray([prm[c][1] for c in live], np.int32),
                 its_done=st["its"][live].copy(), best_inliers=st["best"][live].copy(),
                 off=np.concatenate([[0], np.cumsum([len(rows[c]) for c in live])]).astype(np.int32),
                 p2d=np.ascontiguousarray(np.concatenate([d["kp"][rows[c]] for c in live])),
                 p3dw=np.ascontiguousarray(np.concatenate([d["Xw"][rows[c]] for c in live])),
                 max_err=np.ascontiguousarray(np.concatenate([me[c] for c in live])),
                 best_mask=np.ascontiguousarray(np.concatenate([st["mask"][c] for c in live])),
                 best_Tcw=np.ascontiguousarray(st["T"][live]), n_iterations=5)
        synth.draw_pnp_ransac_sets(q, stream)
        o = run(q)
        nxt = []
        for j, c in enumerate(live):
            a, z = int(q["off"][j]), int(q["off"][j + 1])
            st["its"][c], st["best"][c] = o["its_done"][j], o["best_inliers"][j]
            st["mask"][c] = o["best_mask"][a:z].copy(); st["T"][c] = o["best_Tcw"][j]
            res["its"][c] = o["its_done"][j]
            if o["found"][j]:
                res["found_round"][c] = rounds; res["n_in"][c] = o["n_inliers"][j]; res["Tcw"][c] = o["Tcw"][j]
                res["inlier"][c, rows[c]] = o["inlier"][a:z]
            if not (o["found"][j] or o["no_more"][j]):
                nxt.append(c)
        live, rounds = nxt, rounds + 1
    res["rounds"] = rounds
    return res


def _check_shim(exe, tmp_path, run):
    import subprocess
    import shim_io
    for seed in (71, 72):
        d = _shim_input(seed)
        fin, fout = str(tmp_path / "pnp_in.bin"), str(tmp_path / "pnp_out.bin")
        shim_io.write(fin, d)
        r = subprocess.run([exe, fin, fout], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        assert r.returncode == 0, r.stdout
        got = shim_io.read(fout)
        ref = _direct_shim(d, run)
        nc, NF = len(d["coff"]) - 1, int(d["coff"][-1])
        assert int(got["rounds"][0]) == ref["rounds"]
        for k in ("found_round", "n_in", "its"):
            assert np.array_equal(got[k], ref[k]), (k, got[k], ref[k])
        assert np.array_equal(got["Tcw"].reshape(nc, 12), ref["Tcw"])
        assert np.array_equal(got["inlier"].reshape(nc, NF), ref["inlier"])
        assert (ref["found_round"] >= 0).any() and (ref["found_round"] < 0).any()   # both outcomes: found and discarded
        # iterate() alone on candidate 0 with the same draws equals its IterateBatch result
        fl = got["one_flags"]
        assert int(fl[0]) == int(ref["found_round"][0] == 0) and int(fl[1]) == 1 - int(fl[0])
        if fl[0]:
            assert int(fl[2]) == ref["n_in"][0] and np.array_equal(got["one_Tcw"], ref["Tcw"][0])
            assert int(got["one_n_vb"][0]) == NF and np.array_equal(got["one_inlier"], ref["inlier"][0])
        else:
            assert int(fl[2]) == 0 and int(got["one_n_vb"][0]) == 0


def test_shim_pnp_solver_on_host(built_pnp, tmp_path):
    _check_shim(_shim_build(tmp_path, True), tmp_path, lambda q: api.pnp_ransac(q, impl="oracle"))


@pytest.mark.gpu
def test_gpu_shim_pnp_solver(gpu_ctx, tmp_path):
    _check_shim(_shim_build(tmp_path, False), tmp_path, lambda q: api.pnp_ransac(q, impl="gpu", ctx=gpu_ctx))
