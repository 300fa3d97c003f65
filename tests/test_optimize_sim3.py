"""Optimizer::OptimizeSim3 (lld_sim3_opt): an independent Python transcription of the listing (g2o::Sim3, the two Sim3 edges
with g2o's numeric Jacobian, Levenberg-Marquardt with a dense 7x7 LDL^T and its stop rule, the stale-error chi2 tests and the
early return) pins the CPU oracle; hand-built problems pin one rule each; the host build of the device math equals the oracle's
Sim3 pieces; the shim writes back what the reference writes; on the GPU the batched kernel matches the oracle on both staging
arms (edge records in shared memory / in global memory, told apart by the per-launch profile)."""
import ctypes as C
import math
import os
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import shim_io  # noqa: E402
from lld_slam_b200 import api, capi, synth  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HC = os.path.join(ROOT, "tests", "hostcheck")
f32 = np.float32
SMEM_MAX_CORR = 4266   # largest problem whose edge records are staged in shared memory (include/lldba.h)


# ------------------------------------------------------------------------------------------------------------------
# plain-Python transcription of the listing (Python floats are IEEE doubles; math.* is the C library's)
# ------------------------------------------------------------------------------------------------------------------
def _cross(a, b):
    return [a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]]


def _rot(q, v):
    """Quaternion::_transformVector"""
    uv = _cross(q[:3], v)
    uv = [x + x for x in uv]
    c = _cross(q[:3], uv)
    return [v[k] + q[3] * uv[k] + c[k] for k in range(3)]


def _qmul(a, b):
    return [a[3] * b[0] + a[0] * b[3] + a[1] * b[2] - a[2] * b[1],
            a[3] * b[1] + a[1] * b[3] + a[2] * b[0] - a[0] * b[2],
            a[3] * b[2] + a[2] * b[3] + a[0] * b[1] - a[1] * b[0],
            a[3] * b[3] - a[0] * b[0] - a[1] * b[1] - a[2] * b[2]]


def _quat_from(m):
    """Quaterniond(Matrix3d)"""
    t = m[0][0] + m[1][1] + m[2][2]
    q = [0.0, 0.0, 0.0, 0.0]
    if t > 0:
        t = math.sqrt(t + 1.0)
        q[3] = 0.5 * t
        t = 0.5 / t
        q[0] = (m[2][1] - m[1][2]) * t
        q[1] = (m[0][2] - m[2][0]) * t
        q[2] = (m[1][0] - m[0][1]) * t
    else:
        i = 0
        if m[1][1] > m[0][0]:
            i = 1
        if m[2][2] > m[i][i]:
            i = 2
        j, k = (i + 1) % 3, (i + 2) % 3
        t = math.sqrt(m[i][i] - m[j][j] - m[k][k] + 1.0)
        q[i] = 0.5 * t
        t = 0.5 / t
        q[3] = (m[k][j] - m[j][k]) * t
        q[j] = (m[j][i] + m[i][j]) * t
        q[k] = (m[k][i] + m[i][k]) * t
    return q


def sim3_exp(u, branches=None):
    """g2o::Sim3(const Vector7d&) -> [q (4), t (3), s]"""
    w, ups, sigma = u[0:3], u[3:6], u[6]
    theta = math.sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2])
    Om = [[0.0, -w[2], w[1]], [w[2], 0.0, -w[0]], [-w[1], w[0], 0.0]]
    Om2 = [[Om[i][0] * Om[0][j] + Om[i][1] * Om[1][j] + Om[i][2] * Om[2][j] for j in range(3)] for i in range(3)]
    I = [[1.0 if i == j else 0.0 for j in range(3)] for i in range(3)]
    s = math.exp(sigma)
    eps = 0.00001
    small_angle = theta < eps
    if small_angle:
        R = [[I[i][j] + Om[i][j] + Om2[i][j] for j in range(3)] for i in range(3)]
    else:
        ra, rb = math.sin(theta) / theta, (1 - math.cos(theta)) / (theta * theta)
        R = [[I[i][j] + ra * Om[i][j] + rb * Om2[i][j] for j in range(3)] for i in range(3)]
    if abs(sigma) < eps:
        C = 1.0
        if small_angle:
            A, B = 1. / 2., 1. / 6.
        else:
            th2 = theta * theta
            A = (1 - math.cos(theta)) / th2
            B = (theta - math.sin(theta)) / (th2 * theta)
    else:
        C = (s - 1) / sigma
        if small_angle:
            sg2 = sigma * sigma
            A = ((sigma - 1) * s + 1) / sg2
            B = ((0.5 * sg2 - sigma + 1) * s) / (sg2 * sigma)
        else:
            a, b = s * math.sin(theta), s * math.cos(theta)
            th2, sg2 = theta * theta, sigma * sigma
            c = th2 + sg2
            A = (a * sigma + (1 - b) * theta) / (theta * c)
            B = (C - ((b - 1) * sigma + a * theta) / c) * 1. / th2
    if branches is not None:
        branches.add((abs(sigma) < eps, small_angle))
    W = [[A * Om[i][j] + B * Om2[i][j] + C * I[i][j] for j in range(3)] for i in range(3)]
    t = [W[i][0] * ups[0] + W[i][1] * ups[1] + W[i][2] * ups[2] for i in range(3)]
    return _quat_from(R) + t + [s]


def sim3_mul(A, B):
    rt = _rot(A[:4], B[4:7])
    return _qmul(A[:4], B[:4]) + [A[7] * rt[k] + A[4 + k] for k in range(3)] + [A[7] * B[7]]


def sim3_inv(S):
    qc = [-S[0], -S[1], -S[2], S[3]]
    c = -1. / S[7]
    return qc + _rot(qc, [c * S[4], c * S[5], c * S[6]]) + [1. / S[7]]


def sim3_map(S, x):
    r = _rot(S[:4], x)
    return [S[7] * r[k] + S[4 + k] for k in range(3)]


class _Prob:
    """one loop candidate: the Sim3 vertex and its edges (e12, e21 per correspondence)"""

    def __init__(self, S, cam, fix, P1, P2, o1, o2, i1, i2, branches=None):
        self.S, self.cam, self.fix, self.branches = list(S), [float(c) for c in cam], fix, branches
        self.P1, self.P2 = [[float(v) for v in r] for r in P1], [[float(v) for v in r] for r in P2]
        self.o1, self.o2 = [[float(v) for v in r] for r in o1], [[float(v) for v in r] for r in o2]
        self.info = [(float(a), float(b)) for a, b in zip(i1, i2)]

    def oplus(self, S, u):
        if self.fix:
            u[6] = 0.0
        return sim3_mul(sim3_exp(u, self.branches), S)

    def err(self, S, Sinv, i, side):
        P, o, K = (self.P2[i], self.o1[i], self.cam[0:4]) if side == 0 else (self.P1[i], self.o2[i], self.cam[4:8])
        x = sim3_map(S if side == 0 else Sinv, P)
        p0, p1 = x[0] / x[2], x[1] / x[2]
        return [o[0] - (p0 * K[0] + K[2]), o[1] - (p1 * K[1] + K[3])]


def _chi2(e, info):
    return e[0] * (info * e[0]) + e[1] * (info * e[1])


def _huber(e, delta):
    d2 = delta * delta
    if e <= d2:
        return e, 1.0
    se = math.sqrt(e)
    return 2 * se * delta - d2, delta / se


def _ldlt_solve(H, lam, b):
    A = [[H[r][c] + (lam if r == c else 0.0) for c in range(7)] for r in range(7)]
    D = [0.0] * 7
    for j in range(7):
        d = A[j][j]
        for q in range(j):
            d -= A[j][q] * A[j][q] * D[q]
        if not (d > 0.0) or not math.isfinite(d):
            return None
        D[j] = d
        for i in range(j + 1, 7):
            s = A[i][j]
            for q in range(j):
                s -= A[i][q] * A[j][q] * D[q]
            A[i][j] = s / d
    y = [0.0] * 7
    for i in range(7):
        s = b[i]
        for q in range(i):
            s -= A[i][q] * y[q]
        y[i] = s
    z = [y[i] / D[i] for i in range(7)]
    x = [0.0] * 7
    for i in range(6, -1, -1):
        s = z[i]
        for q in range(i + 1, 7):
            s -= A[q][i] * x[q]
        x[i] = s
    return x


def _optimize(pr, active, its, delta, stale, log):
    """initializeOptimization(); optimize(its): returns iterations run; stale[i] = [chi2 e12, chi2 e21] of the last evaluation"""
    if not any(active):
        return 0
    x = [0.0] * 7
    lam, ni, nbad_it = 0.0, 2.0, 0
    done = 0
    for it in range(its):
        done += 1
        Sinv = sim3_inv(pr.S)
        errs = {}
        cur = 0.0
        for i in range(len(active)):
            if active[i]:
                for side in (0, 1):
                    e = pr.err(pr.S, Sinv, i, side)
                    errs[(i, side)] = e
                    cur += _huber(_chi2(e, pr.info[i][side]), delta)[0]
        ini = cur
        # numeric Jacobians (push / oplus(+-delta e_d) / computeError / pop) and the normal equations
        H = [[0.0] * 7 for _ in range(7)]
        b = [0.0] * 7
        pert = []
        for d in range(7):
            for sgn in (1e-9, -1e-9):
                u = [0.0] * 7
                u[d] = sgn
                Sk = pr.oplus(pr.S, u)
                pert.append((Sk, sim3_inv(Sk)))
        scalar = 1.0 / (2 * 1e-9)
        for i in range(len(active)):
            if not active[i]:
                continue
            for side in (0, 1):
                e = errs[(i, side)]
                J = [[0.0] * 7, [0.0] * 7]
                for d in range(7):
                    ep = pr.err(pert[2 * d][0], pert[2 * d][1], i, side)
                    em = pr.err(pert[2 * d + 1][0], pert[2 * d + 1][1], i, side)
                    J[0][d] = scalar * (ep[0] - em[0])
                    J[1][d] = scalar * (ep[1] - em[1])
                info = pr.info[i][side]
                wo = _huber(_chi2(e, info), delta)[1] * info
                for r in range(7):
                    for c in range(7):
                        H[r][c] += wo * (J[0][r] * J[0][c] + J[1][r] * J[1][c])
                    b[r] -= wo * (J[0][r] * e[0] + J[1][r] * e[1])
        if it == 0:
            lam = 1e-5 * max(abs(H[j][j]) for j in range(7))
            ni, nbad_it = 2.0, 0
            log["chi2"].append(cur)
        qmax = 0
        while True:
            xn = _ldlt_solve(H, lam, b)
            if xn is not None:
                x = xn
            Sn = pr.oplus(pr.S, x)          # x[6] is zeroed in place with a fixed scale
            Sni = sim3_inv(Sn)
            tmp = 0.0
            for i in range(len(active)):
                if active[i]:
                    c = [_chi2(pr.err(Sn, Sni, i, s), pr.info[i][s]) for s in (0, 1)]
                    stale[i] = c
                    tmp += _huber(c[0], delta)[0]
                    tmp += _huber(c[1], delta)[0]
            if xn is None:
                tmp = sys.float_info.max
            rho = cur - tmp
            scale = 0.0
            for j in range(7):
                scale += x[j] * (lam * x[j] + b[j])
            scale += 1e-3
            rho /= scale
            if rho > 0 and math.isfinite(tmp):
                alpha = min(1. - (2 * rho - 1) ** 3, 2. / 3.)
                lam *= max(1. / 3., alpha)
                ni = 2.0
                cur = tmp
                pr.S = Sn
            else:
                lam *= ni
                ni *= 2
            qmax += 1
            if not (rho < 0 and qmax < 10):
                break
        log["chi2"].append(cur); log["lambda"].append(lam); log["trials"].append(qmax)
        if qmax == 10 or rho == 0:
            break
        nbad_it = nbad_it + 1 if (ini - cur) * 1e3 < ini else 0
        if nbad_it >= 3:
            break
    return done


def sim3_python(p, branches=None, stale_out=None):
    n = int(p["n_problems"])
    its1, itsb, itsc = int(p["its_first"]), int(p["its_more_outliers"]), int(p["its_more_clean"])
    stride = its1 + max(itsb, itsc) + 2
    m_all = int(p["off"][-1])
    out = dict(S12=np.zeros((n, 8)), inlier=np.ones(m_all, np.uint8), n_in=np.zeros(n, np.int32),
               chi2_log=np.zeros((n, stride)), lambda_log=np.zeros((n, stride)), trials_log=np.zeros((n, stride), np.int32),
               n_iter_done=np.zeros((n, 2), np.int32))
    for pb in range(n):
        a, z = int(p["off"][pb]), int(p["off"][pb + 1])
        m = z - a
        pr = _Prob([float(v) for v in p["S12"][pb]], p["cam"][pb], bool(p["fix_scale"][pb]), p["p1c"][a:z], p["p2c"][a:z],
                   p["obs1"][a:z], p["obs2"][a:z], p["info1"][a:z], p["info2"][a:z], branches)
        th2 = float(f32(p["th2"][pb]))
        delta = float(np.sqrt(f32(th2)))          # const float deltaHuber = sqrt(th2)
        S0 = list(pr.S)
        active = [True] * m
        stale = [[0.0, 0.0] for _ in range(m)]
        for r, base in ((0, 0), (1, its1 + 1)):
            log = dict(chi2=[], **{"lambda": []}, trials=[])
            if r == 0:
                its = its1
            else:
                its = itsb if nbad > 0 else itsc
            done = _optimize(pr, active, its, delta, stale, log)
            out["n_iter_done"][pb, r] = done
            for k, v in enumerate(log["chi2"]):
                out["chi2_log"][pb, base + k] = v
            for k, v in enumerate(log["lambda"]):
                out["lambda_log"][pb, base + 1 + k] = v
            for k, v in enumerate(log["trials"]):
                out["trials_log"][pb, base + 1 + k] = v
            drop = [i for i in range(m) if active[i] and (stale[i][0] > th2 or stale[i][1] > th2)]
            if stale_out is not None:
                stale_out.append(dict(pb=pb, round=r, stale=[list(s) for s in stale], S=list(pr.S), active=list(active)))
            for i in drop:
                active[i] = False
                out["inlier"][a + i] = 0
            if r == 0:
                nbad = len(drop)
                if m - nbad < 10:
                    break
            else:
                out["n_in"][pb] = sum(active)
        out["S12"][pb] = S0 if m - nbad < 10 else pr.S
    return out


def _rel(a, b):
    return np.abs(a - b) / np.maximum(np.abs(b), 1e-300)


def _same_pin(o, r):
    """the oracle against the transcription: logs to 1e-12 relative, identical counts and flags, S12 to 1e-12"""
    assert np.array_equal(o["n_iter_done"], r["n_iter_done"]), (o["n_iter_done"], r["n_iter_done"])
    assert np.array_equal(o["trials_log"], r["trials_log"])
    assert np.array_equal(o["inlier"], r["inlier"])
    assert np.array_equal(o["n_in"], r["n_in"])
    assert _rel(o["chi2_log"], r["chi2_log"]).max(initial=0) < 1e-12
    assert _rel(o["lambda_log"], r["lambda_log"]).max(initial=0) < 1e-12
    assert np.abs(o["S12"] - r["S12"]).max(initial=0) < 1e-12


# ------------------------------------------------------------------------------------------------------------------
# hand-built problems
# ------------------------------------------------------------------------------------------------------------------
def _one(S, P1, P2, o1, o2, fix=1, th2=10.0, info=None, its=(5, 10, 5), cam=(500.0, 500.0, 320.0, 240.0)):
    m = len(P1)
    info = np.ones(m, f32) if info is None else np.asarray(info, f32)
    return dict(n_problems=1, S12=np.asarray([S], np.float64), cam=np.asarray([list(cam) * 2], np.float64),
                fix_scale=np.array([fix], np.int32), th2=np.array([th2], f32), off=np.array([0, m], np.int32),
                p1c=np.ascontiguousarray(np.asarray(P1, f32).reshape(-1, 3)), p2c=np.ascontiguousarray(np.asarray(P2, f32).reshape(-1, 3)),
                obs1=np.ascontiguousarray(np.asarray(o1, f32).reshape(-1, 2)), obs2=np.ascontiguousarray(np.asarray(o2, f32).reshape(-1, 2)),
                info1=info.copy(), info2=info.copy(), its_first=its[0], its_more_outliers=its[1], its_more_clean=its[2])


def _exact_grid(m, seed):
    """points whose projections through the identity Sim3 are exact in float: zero residuals at S12 = identity"""
    rng = np.random.default_rng(seed)
    a = rng.integers(-256, 256, m) / 512.0
    b = rng.integers(-192, 192, m) / 512.0
    z = 2.0 ** rng.integers(0, 4, m)
    P = np.stack([a * z, b * z, z], 1)
    o = np.stack([a * 500.0 + 320.0, b * 500.0 + 240.0], 1)
    return P, o


IDENT = [0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0]


def _near_ident(deg=2.0, tr=0.05, ds=0.0):
    th = math.radians(deg) / math.sqrt(3)
    q = [math.sin(th / 2) / math.sqrt(3)] * 3 + [math.cos(th / 2)]
    return q + [tr, -tr, tr] + [1.0 + ds]


def _case_few_survivors():
    P, o = _exact_grid(14, 1)
    o1 = o.copy(); o1[[1, 4, 7, 9, 12]] += 150.0          # 5 gross outliers: 9 survivors
    return _one(_near_ident(), P, P, o1, o), dict(n_in=0, kept=9, ran2=False)


def _case_exactly_ten():
    P, o = _exact_grid(15, 2)
    o1 = o.copy(); o1[[0, 3, 6, 9, 13]] += 150.0          # 10 survivors: round 2 runs
    return _one(_near_ident(), P, P, o1, o, its=(5, 7, 2)), dict(n_in=10, kept=10, ran2=True, its2=7)


def _case_no_outliers():
    P, o = _exact_grid(30, 3)
    return _one(_near_ident(), P, P, o, o, its=(5, 7, 2)), dict(n_in=30, kept=30, ran2=True, its2=2)


def _case_outliers_more_iterations():
    P, o = _exact_grid(30, 4)
    rng = np.random.default_rng(4)
    o1 = o + rng.normal(0, 0.5, o.shape); o2 = o + rng.normal(0, 0.5, o.shape)
    o2[[2, 11, 20]] -= 120.0
    return _one(_near_ident(4.0, 0.2), P, P, o1, o2, its=(5, 7, 2)), dict(n_in=27, kept=27, ran2=True, its2=7)


def _case_at_optimum():
    P, o = _exact_grid(20, 5)
    return _one(IDENT, P, P, o, o), dict(n_in=20, kept=20, ran2=True, done=[1, 1], chi2_zero=True)


def _case_negative_depth():
    P, o = _exact_grid(20, 6)
    P1, P2 = P.copy(), P.copy()
    P2[5] = [0.1, 0.1, -2.0]                                 # behind keyframe 1 after the map: e12 is huge, no depth test
    return _one(_near_ident(1.0, 0.02), P1, P2, o, o), dict(n_in=19, kept=19, ran2=True, dropped=[5])


def _case_zero():
    return _one(_near_ident(), np.zeros((0, 3)), np.zeros((0, 3)), np.zeros((0, 2)), np.zeros((0, 2))), dict(n_in=0, kept=0, ran2=False, done=[0, 0])


CASES = {"few_survivors": _case_few_survivors, "exactly_ten": _case_exactly_ten, "no_outliers": _case_no_outliers,
         "outliers_more_iterations": _case_outliers_more_iterations, "at_optimum": _case_at_optimum,
         "negative_depth": _case_negative_depth, "zero_correspondences": _case_zero}


def _check_case(o, p, exp):
    m = int(p["off"][-1])
    assert int(o["n_in"][0]) == exp["n_in"]
    assert int(o["inlier"].sum()) == exp["kept"]
    if not exp["ran2"]:
        assert np.array_equal(o["S12"][0], p["S12"][0])          # g2oS12 unchanged
        assert int(o["n_iter_done"][0, 1]) == 0
    else:
        assert 0 < int(o["n_iter_done"][0, 1]) <= exp.get("its2", 10)
    if "its2" in exp and exp["its2"] == 7:
        assert int(o["n_iter_done"][0, 1]) > 2                     # more than the clean count: the outlier count ran
    if "done" in exp:
        assert o["n_iter_done"][0].tolist() == exp["done"]
    if exp.get("chi2_zero"):
        assert o["chi2_log"][0, 0] == 0.0 and np.array_equal(o["S12"][0], p["S12"][0])
    for i in exp.get("dropped", []):
        assert o["inlier"][i] == 0
    assert o["inlier"].shape == (m,)


def _rejected_round_problem():
    """a batch in which a round ends in ten rejected trials: the chi2 tests then read the errors of the last rejected trial"""
    return synth.make_sim3_batch(6, 40, 227, fix_scale=1)


# ------------------------------------------------------------------------------------------------------------------
# CPU: the oracle against the transcription
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fix", [1, 0])
@pytest.mark.parametrize("seed", [3, 4, 5])
def test_oracle_sim3_against_python(built, seed, fix):
    p = synth.make_sim3_batch(4, [120, 60, 14, 35], seed, fix_scale=fix)
    branches = set()
    r = sim3_python(p, branches)
    o = api.sim3_opt(p, impl="oracle")
    _same_pin(o, r)
    assert (r["n_in"] > 0).sum() >= 3 and (r["inlier"] == 0).sum() > 0
    assert r["n_iter_done"][:, 1].max() >= 2
    # fixed scale: every oplus has sigma = 0; the small-angle perturbations and the larger LM steps take both rotation branches
    want = {(True, True), (True, False)} if fix else {(False, True), (False, False)}
    assert want <= branches, branches


@pytest.mark.parametrize("name", sorted(CASES))
def test_hand_built_case(built, name):
    p, exp = CASES[name]()
    o = api.sim3_opt(p, impl="oracle")
    _same_pin(o, sim3_python(p))
    _check_case(o, p, exp)


def test_round_ending_in_rejected_trials_uses_stale_errors(built):
    p = _rejected_round_problem()
    snaps = []
    r = sim3_python(p, stale_out=snaps)
    o = api.sim3_opt(p, impl="oracle")
    _same_pin(o, r)
    # some round ends with an iteration whose ten trials were all rejected ...
    its1 = int(p["its_first"])
    ends = []
    for pb in range(int(p["n_problems"])):
        for rr, base in ((0, 0), (1, its1 + 1)):
            d = int(r["n_iter_done"][pb, rr])
            if d and r["trials_log"][pb, base + d] == 10:
                ends.append((pb, rr))
    assert ends
    # ... and in one of them the stale chi2 differ from the chi2 at the state the round ended in
    diffs = []
    for pb, rr in ends:
        snap = next(s for s in snaps if s["pb"] == pb and s["round"] == rr)
        a, z = int(p["off"][pb]), int(p["off"][pb + 1])
        pr = _Prob(snap["S"], p["cam"][pb], bool(p["fix_scale"][pb]), p["p1c"][a:z], p["p2c"][a:z], p["obs1"][a:z], p["obs2"][a:z],
                   p["info1"][a:z], p["info2"][a:z])
        Si = sim3_inv(pr.S)
        diffs += [abs(_chi2(pr.err(pr.S, Si, i, 0), pr.info[i][0]) - snap["stale"][i][0]) for i in range(z - a) if snap["active"][i]]
    assert max(diffs) > 0


def test_generator_shapes_and_scale():
    p = synth.make_sim3_batch(3, [0, 1, 40], 9, fix_scale=0)
    assert p["off"].tolist() == [0, 0, 1, 41]
    assert p["p1c"].shape == (41, 3) and p["obs2"].shape == (41, 2) and p["info1"].shape == (41,)
    assert (p["S12"][:, 7] > 0.45).all() and (p["S12"][:, 7] < 2.1).all()
    assert np.allclose(np.linalg.norm(p["S12"][:, :4], axis=1), 1.0)
    q = synth.make_sim3_batch(2, 10, 9, fix_scale=1)
    assert (q["S12"][:, 7] == 1.0).all()


# ------------------------------------------------------------------------------------------------------------------
# host build of the device math against the oracle's pieces
# ------------------------------------------------------------------------------------------------------------------
def _libs():
    dm = C.CDLL(os.path.join(HC, "libdevmath_sim3_host.so"))
    orc = C.CDLL(capi.SIM3_ORACLE_PATH)
    return dm, orc


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def _call(f, *arrays):
    f.restype = None
    f(*[a if isinstance(a, int) else _ptr(a) for a in arrays])


@pytest.mark.parametrize("fix", [1, 0])
def test_device_math_host_equals_oracle(built, fix):
    dm, orc = _libs()
    rng = np.random.default_rng(17 + fix)
    p = synth.make_sim3_batch(1, 64, 23 + fix, fix_scale=fix)
    for trial in range(64):
        scale_u = [0.0, 1e-6, 0.3][trial % 3] * (1 - fix)
        u = np.concatenate([rng.normal(0, [0.0, 1e-7, 0.2][trial % 3], 3), rng.normal(0, 0.5, 3), [rng.normal(0, 1) * scale_u]])
        A, B = np.zeros(8), np.zeros(8)
        _call(dm.dm_sim3_exp, u, A); _call(orc.lldo_sim3_exp, u, B)
        assert np.array_equal(A, B)
        S, T = p["S12"][0].copy(), np.zeros(8)
        _call(dm.dm_sim3_mul, A, S, T); R = np.zeros(8); _call(orc.lldo_sim3_mul, A, S, R)
        assert np.array_equal(T, R)
        _call(dm.dm_sim3_inverse, T, A); _call(orc.lldo_sim3_inverse, T, B)
        assert np.array_equal(A, B)
        x = rng.normal(0, 5, 3); y1, y2 = np.zeros(3), np.zeros(3)
        _call(dm.dm_sim3_map, T, x, y1); _call(orc.lldo_sim3_map, T, x, y2)
        assert np.array_equal(y1, y2)
        i = trial
        outs = [[np.zeros(2), np.zeros(2), np.zeros(14), np.zeros(14)] for _ in range(2)]
        for lib, (e12, e21, J12, J21), name in ((dm, outs[0], "dm_sim3_edges"), (orc, outs[1], "lldo_sim3_edges")):
            f = getattr(lib, name)
            f.restype = None
            f(_ptr(T), fix, _ptr(p["cam"][0]), _ptr(p["p1c"][i]), _ptr(p["p2c"][i]), _ptr(p["obs1"][i]), _ptr(p["obs2"][i]),
              _ptr(e12), _ptr(e21), _ptr(J12), _ptr(J21))
        for a, b in zip(*outs):
            if fix:
                assert np.array_equal(a, b)        # theta < eps perturbations: no transcendental function, the same bits
            else:
                assert np.allclose(a, b, rtol=1e-6, atol=1e-9)
        if fix:
            assert (outs[0][2].reshape(2, 7)[:, 6] == 0).all() and (outs[0][3].reshape(2, 7)[:, 6] == 0).all()


# ------------------------------------------------------------------------------------------------------------------
# shim
# ------------------------------------------------------------------------------------------------------------------
def _shim_build(tmp_path, oracle):
    src = os.path.join(HC, "shim_sim3.cpp")
    exe = str(tmp_path / ("shim_sim3_oracle" if oracle else "shim_sim3_gpu"))
    if oracle:
        libdir, lib, extra = HC, "sim3_oracle", ["-DLLD_SHIM_ORACLE"]
    else:
        libdir, lib, extra = os.path.join(ROOT, "lld_slam_b200", "csrc"), "lldba", []
    r = subprocess.run(["g++", "-std=c++14", "-O1", "-Wall", *extra, src, "-o", exe, f"-L{libdir}", f"-l{lib}", f"-Wl,-rpath,{libdir}"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout
    return exe


def _shim_input(fix, seed):
    """one loop candidate as keyframe objects: KF1 / KF2 world poses, map points with world positions, keypoints, and
    vpMatches1 with entries the reference skips (no match, no map point in KF1, a bad point, a point not in KF2)"""
    rng = np.random.default_rng(seed)
    p = synth.make_sim3_batch(1, 80, seed, fix_scale=fix)
    m = 80
    R1 = synth._rodrigues(rng.normal(0, 0.05, 3)); t1 = rng.normal(0, 1, 3)
    R2 = synth._rodrigues(rng.normal(0, 0.05, 3)); t2 = rng.normal(0, 1, 3)
    T1 = f32(np.concatenate([R1.reshape(-1), t1])); T2 = f32(np.concatenate([R2.reshape(-1), t2]))
    # world positions whose camera-frame images the shim recomputes in float
    X1w = f32((p["p1c"].astype(np.float64) - t1) @ R1); X2w = f32((p["p2c"].astype(np.float64) - t2) @ R2)
    octs = rng.integers(0, 8, (2, m)).astype(np.int32)
    kind = np.zeros(m + 6, np.int32)            # 0 valid, 1 no match, 2 no KF1 point, 3 KF1 point bad, 4 match bad, 5 not in KF2
    kind[m:] = [1, 2, 3, 4, 5, 1]
    order = rng.permutation(m + 6)
    d = dict(fix=np.array([fix], np.int32), th2=np.array([10.0], f32), S12=p["S12"][0].copy(), cam=f32(p["cam"][0]),
             T1=T1, T2=T2, kind=kind[order], X1w=np.zeros((m + 6, 3), f32), X2w=np.zeros((m + 6, 3), f32),
             kp1=np.zeros((m + 6, 2), f32), kp2=np.zeros((m + 6, 2), f32), oct1=np.zeros(m + 6, np.int32), oct2=np.zeros(m + 6, np.int32),
             inv_level_sigma2=synth.inv_level_sigma2())
    valid_rows = np.where(d["kind"] == 0)[0]
    for j, row in enumerate(valid_rows):
        d["X1w"][row] = X1w[j]; d["X2w"][row] = X2w[j]; d["kp1"][row] = p["obs1"][j]; d["kp2"][row] = p["obs2"][j]
        d["oct1"][row] = octs[0, j]; d["oct2"][row] = octs[1, j]
    return d, valid_rows


def _flat_from_shim_input(d, valid_rows):
    """the problem the shim must pass, built here with numpy float arithmetic (cv::Mat products accumulate in double and
    round once)"""
    def cam_frame(T, X):
        R, t, X = T[:9].reshape(3, 3).astype(np.float64), T[9:].astype(np.float64), X.astype(np.float64)
        return f32(np.stack([R[r, 0] * X[:, 0] + R[r, 1] * X[:, 1] + R[r, 2] * X[:, 2] + t[r] for r in range(3)], 1))
    isig = d["inv_level_sigma2"]
    rows = valid_rows
    return dict(n_problems=1, S12=d["S12"][None].copy(), cam=d["cam"].astype(np.float64)[None].copy(), fix_scale=d["fix"].copy(),
                th2=d["th2"].copy(), off=np.array([0, len(rows)], np.int32),
                p1c=np.ascontiguousarray(cam_frame(d["T1"], d["X1w"][rows])), p2c=np.ascontiguousarray(cam_frame(d["T2"], d["X2w"][rows])),
                obs1=np.ascontiguousarray(d["kp1"][rows]), obs2=np.ascontiguousarray(d["kp2"][rows]),
                info1=np.ascontiguousarray(isig[d["oct1"][rows]]), info2=np.ascontiguousarray(isig[d["oct2"][rows]]),
                its_first=5, its_more_outliers=10, its_more_clean=5)


def _check_shim(exe, tmp_path, impl, ctx=None):
    for fix, seed in ((1, 61), (0, 62)):
        d, rows = _shim_input(fix, seed)
        fin, fout = str(tmp_path / "sim3_in.bin"), str(tmp_path / "sim3_out.bin")
        shim_io.write(fin, d)
        r = subprocess.run([exe, fin, fout], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        assert r.returncode == 0, r.stdout
        got = shim_io.read(fout)
        ref = api.sim3_opt(_flat_from_shim_input(d, rows), impl=impl, ctx=ctx)
        assert int(got["n_in"][0]) == int(ref["n_in"][0]) and ref["n_in"][0] > 20
        assert np.array_equal(got["S12"], ref["S12"][0])
        # vpMatches1 after the call: cleared where the optimiser dropped the correspondence, untouched elsewhere
        want = np.where(d["kind"] == 1, 0, 1).astype(np.int32)
        want[rows] = ref["inlier"]
        assert np.array_equal(got["matched"], want)
        # the early return (fewer than 10 survivors) leaves g2oS12 as it was
        assert np.array_equal(got["S12_early"], d["S12"]) and int(got["n_in_early"][0]) == 0


def test_shim_optimize_sim3_on_host(built, tmp_path):
    _check_shim(_shim_build(tmp_path, True), tmp_path, "oracle")


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
def _profiled(p, ctx):
    out, prof = ctx.profile(lambda: api.sim3_opt(p, impl="gpu", ctx=ctx))
    return out, set(prof)


def _rel_log(g, o, pb, its1):
    """relative difference of the chi2 logs; chi2 below 1e-4 of its round's start (a round converging to zero residual, where
    chi2 is the square of the step's own noise) is compared against that level"""
    floor = np.zeros(o["chi2_log"].shape[1])
    floor[:its1 + 1] = 1e-4 * o["chi2_log"][pb, 0]
    floor[its1 + 1:] = max(1e-4 * o["chi2_log"][pb, its1 + 1], 1e-12 * o["chi2_log"][pb, 0])   # round 1 may end at zero residual
    return np.abs(g["chi2_log"][pb] - o["chi2_log"][pb]) / np.maximum(np.abs(o["chi2_log"][pb]), np.maximum(floor, 1e-300))


def _zero_residual_stop(g, o, pb, its1):
    """the rounds stop at different iterations only where chi2 has reached 1e-12 of the round's start: rounding noise"""
    for r, base in ((0, 0), (1, its1 + 1)):
        dg, do = int(g["n_iter_done"][pb, r]), int(o["n_iter_done"][pb, r])
        if dg != do and not o["chi2_log"][pb, base + min(dg, do)] <= 1e-12 * o["chi2_log"][pb, base]:
            return False
    return True


def _converged_tie(g, o, pb, its1):
    """the two runs of problem pb took a different number of trials in some LM iteration at which chi2 had converged: whether
    that iteration's last trial is accepted, and so which errors the chi2 test reads and when a round stops, is then decided by
    rounding (the fixed-order device reduction and the device sin / cos / exp against the sequential oracle and glibc)"""
    for r, base in ((0, 0), (1, its1 + 1)):
        for k in range(1, min(int(g["n_iter_done"][pb, r]), int(o["n_iter_done"][pb, r])) + 1):
            if g["trials_log"][pb, base + k] != o["trials_log"][pb, base + k]:
                prev, cur = o["chi2_log"][pb, base + k - 1], o["chi2_log"][pb, base + k]
                if abs(prev - cur) <= 1e-9 * abs(prev):
                    return True
    return False


def _check_gpu(p, ctx, arm="smem", o=None, strict=False):
    """GPU against the oracle, problem by problem.  A problem agrees when inlier, n_in and the iterations per round are
    identical (a round that has converged to zero residual may stop at another iteration), the robust chi2 of every iteration
    is within 1e-6 relative (within 1e-4 at the start of round 2, whose state is the end of a converged round 1) and S12
    within 1e-6 rad, 1e-5 |t| and 1e-5 relative scale.  Unless strict, a problem may instead diverge when a converged LM
    iteration took a different number of trials (_converged_tie), at most 1 in 1000 problems; round 1 must still agree."""
    g, names = _profiled(p, ctx)
    other = "global" if arm == "smem" else "smem"
    assert f"k_sim3_opt_{arm}" in names and f"k_sim3_opt_{other}" not in names, names
    o = api.sim3_opt(p, impl="oracle") if o is None else o
    n, its1 = int(p["n_problems"]), int(p["its_first"])
    diverged = 0
    for pb in range(n):
        a, z = int(p["off"][pb]), int(p["off"][pb + 1])
        rel = _rel_log(g, o, pb, its1)
        same = (np.array_equal(g["inlier"][a:z], o["inlier"][a:z]) and g["n_in"][pb] == o["n_in"][pb]
                and _zero_residual_stop(g, o, pb, its1))
        if same:
            for r, base in ((0, 0), (1, its1 + 1)):
                k = min(int(g["n_iter_done"][pb, r]), int(o["n_iter_done"][pb, r]))
                rr = rel[base:base + k + 1]
                assert rr[1:].max(initial=0) < 1e-6 and rr[:1].max(initial=0) < (1e-6 if r == 0 else 1e-4), (pb, r, rel)
            qg, qo = g["S12"][pb, :4], o["S12"][pb, :4]
            assert 2 * np.arccos(min(1.0, abs(qg @ qo) / (np.linalg.norm(qg) * np.linalg.norm(qo)))) < 1e-6, pb
            assert np.linalg.norm(g["S12"][pb, 4:7] - o["S12"][pb, 4:7]) <= 1e-5 * np.linalg.norm(o["S12"][pb, 4:7]) + 1e-12, pb
            assert abs(g["S12"][pb, 7] - o["S12"][pb, 7]) <= 1e-5 * abs(o["S12"][pb, 7]), pb
        else:
            assert not strict and _converged_tie(g, o, pb, its1), pb
            assert rel[:its1 + 1][o["chi2_log"][pb, :its1 + 1] > 0].max(initial=0) < 1e-6, pb
            diverged += 1
    assert diverged <= n // 1000, diverged
    return g


def _concat(parts):
    out = dict(parts[0])
    out["n_problems"] = sum(int(q["n_problems"]) for q in parts)
    for k in ("S12", "cam", "fix_scale", "th2", "p1c", "p2c", "obs1", "obs2", "info1", "info2"):
        out[k] = np.ascontiguousarray(np.concatenate([q[k] for q in parts], 0))
    offs, base = [np.zeros(1, np.int32)], 0
    for q in parts:
        offs.append((q["off"][1:] + base).astype(np.int32))
        base += int(q["off"][-1])
    out["off"] = np.concatenate(offs)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("fix", [1, 0])
def test_gpu_sim3_4096x300(gpu_ctx, fix):
    p = synth.make_sim3_batch(4096, 300, 101 + fix, fix_scale=fix)
    g = _check_gpu(p, gpu_ctx)
    assert (g["n_in"] > 200).mean() > 0.9


@pytest.mark.gpu
@pytest.mark.parametrize("fix", [1, 0])
def test_gpu_sim3_ragged(gpu_ctx, fix):
    p = synth.make_sim3_batch(7, [0, 1, 9, 10, 11, 37, 2048], 103, fix_scale=fix)
    _check_gpu(p, gpu_ctx)


@pytest.mark.gpu
@pytest.mark.parametrize("fix", [1, 0])
def test_gpu_sim3_global_arm(gpu_ctx, fix):
    big = synth.make_sim3_batch(1, SMEM_MAX_CORR + 1, 107, fix_scale=fix)
    small = synth.make_sim3_batch(3, [40, 300, 12], 109, fix_scale=fix)
    _check_gpu(big, gpu_ctx, "global")
    _check_gpu(_concat([small, big]), gpu_ctx, "global")
    _check_gpu(synth.make_sim3_batch(1, SMEM_MAX_CORR, 107, fix_scale=fix), gpu_ctx, "smem")


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_gpu_sim3_hand_built_case(gpu_ctx, name):
    p, exp = CASES[name]()
    g = _check_gpu(p, gpu_ctx, strict=True)
    _check_case(g, p, exp)


@pytest.mark.gpu
def test_gpu_sim3_round_ending_in_rejected_trials(gpu_ctx):
    _check_gpu(_rejected_round_problem(), gpu_ctx)


@pytest.mark.gpu
def test_gpu_sim3_repeated_calls(gpu_ctx):
    p = synth.make_sim3_batch(256, 300, 113, fix_scale=0)
    a = api.sim3_opt(p, impl="gpu", ctx=gpu_ctx)
    api.sim3_opt(synth.make_sim3_batch(3, [5000, 20, 0], 114), impl="gpu", ctx=gpu_ctx)   # another shape in between
    b = api.sim3_opt(p, impl="gpu", ctx=gpu_ctx)
    for k in a:
        if isinstance(a[k], np.ndarray):
            assert np.array_equal(a[k], b[k]), k


@pytest.mark.gpu
def test_gpu_sim3_argument_checks(gpu_ctx):
    p = synth.make_sim3_batch(3, [20, 20, 20], 117)
    bad = [("n_problems", -1), ("off", np.array([0, 20, 10, 60], np.int32)), ("fix_scale", np.array([0, 2, 1], np.int32)),
           ("th2", np.array([10, 0, 10], f32)), ("th2", np.array([10, -1, 10], f32)), ("its_first", -1)]
    for k, v in bad:
        q = dict(p); q[k] = v
        with pytest.raises(RuntimeError, match="bad argument"):
            api.sim3_opt(q, impl="gpu", ctx=gpu_ctx)
    g = api.sim3_opt(p, impl="gpu", ctx=gpu_ctx)          # the context is usable after a refused call
    assert np.array_equal(g["n_in"], api.sim3_opt(p, impl="oracle")["n_in"])


@pytest.mark.gpu
def test_gpu_shim_optimize_sim3(gpu_ctx, tmp_path):
    _check_shim(_shim_build(tmp_path, False), tmp_path, "gpu", gpu_ctx)
