"""Global BA across loop closures: the block-elimination solver of `sp_solver.cuh` (`lld_ctx_set_gba_sparse`).

After a loop closure some landmarks are seen by keyframes at both ends of the map.  The reduced camera system is then no
longer banded and the on-chip solvers reject it ("envelope ... too wide").  With the switch on, `ba.cu` groups the free
keyframes into super-blocks, plans an elimination over the super-block graph on the host and runs it with the `k_sp_*`
kernels.

CPU tests check the plan (through the host-only hook `lld_gba_sparse_plan_report`) against an independent numpy derivation,
run the plan in numpy on a random block-SPD matrix, and pin the shapes of the GPU cases.  GPU tests compare with the FP64
oracle through `check_ba` and prove from the per-launch profile that the `k_sp_*` kernels ran.
"""
import ctypes as C
import json

import numpy as np
import pytest

from lld_slam_b200 import capi, synth
from test_ba_paths import (ERR_UNSUPPORTED, SMEM_LIMIT, _bind, _free_sets, add_points, assert_identical, checked, cr_problem,
                           expect_error, free_kfs, h2d_bytes, new_values, oracle, profiled, run, shape_claims,
                           too_wide_problem, value_bytes)
from test_gpu_parity import check_ba

SP_MAX_MB = 26                 # ba.cu: super-blocks of at most 26 keyframes (6 * 26 = CR_MAX_M)
SP_MAX_BYTES = 2 << 30         # ba.cu / include/lldba.h: device storage of one plan


# ------------------------------------------------------------------------------------------------------------------
# generators
# ------------------------------------------------------------------------------------------------------------------
def loop_problem(n_kf, seed, *, robust=False, fixed=(), chords=False, n_loop=40):
    """a geometric-track window plus n_loop points linking the first and the last 10 free keyframes; `chords` adds three
    groups of points across the middle of the map, so that super-blocks get three or more neighbours"""
    rng = np.random.default_rng(seed)
    w = synth.make_ba_window(n_kf, 12 * n_kf, 2 * n_kf, rng, mean_track=6.0, track_mode="geometric", global_mode=True)
    if fixed:
        w["kf_fixed"] = w["kf_fixed"].copy()
        w["kf_fixed"][list(fixed)] = 1
    F = free_kfs(w)
    for _ in range(n_loop):
        w = add_points(w, [[F[rng.integers(0, 10)], F[len(F) - 1 - rng.integers(0, 10)]]], rng, True,
                       ahead=150.0, side=(rng.uniform(-1, 1), -2.0))
    if chords:
        n = len(F)
        for a, b in ((n // 5, 3 * n // 5), (2 * n // 5, 4 * n // 5), (n // 4, n // 2)):
            for _ in range(4):
                w = add_points(w, [[F[a + rng.integers(0, 5)], F[b + rng.integers(0, 5)]]], rng, True,
                               ahead=150.0, side=(rng.uniform(-1, 1), -2.0))
    return synth.batch_ba([w], "global", 1.0, robust)


GPU_CASES = {
    "too_wide": lambda: too_wide_problem(),
    "loop200": lambda: loop_problem(200, 7),
    "loop400": lambda: loop_problem(400, 8),
    "loop200_robust": lambda: loop_problem(200, 9, robust=True),
    "loop200_fixed": lambda: loop_problem(200, 10, fixed=(60, 61, 130)),
    "loop300_chords": lambda: loop_problem(300, 11, chords=True),
}
# (mb, N, levels) of each GPU case, from the numpy derivation below
GPU_SHAPES = {"too_wide": (19, 11, 5), "loop200": (19, 11, 5), "loop400": (19, 21, 6), "loop200_robust": (19, 11, 5),
              "loop200_fixed": (19, 11, 5), "loop300_chords": (19, 16, 7)}


# ------------------------------------------------------------------------------------------------------------------
# the plan, derived independently in numpy
# ------------------------------------------------------------------------------------------------------------------
def plan_report(p):
    lib = capi.load_library()
    prob, keep = capi.fill_struct(capi.BaProblem, p)
    buf = C.create_string_buffer(1 << 25)
    rc = lib.dll.lld_gba_sparse_plan_report(C.byref(prob), buf, len(buf))
    return rc, buf.value.decode()


def plan_numpy(p):
    nG, sets, _ = _free_sets(p, 0)
    pairs = set()
    for s in sets:
        for x in range(len(s)):
            for y in range(x, len(s)):
                pairs.add((int(s[x]), int(s[y])))
    mb = max([1] + [h - a for a, h in pairs if h - a <= SP_MAX_MB])
    N = -(-nG // mb)
    adj = [set() for _ in range(N)]
    for a, h in pairs:
        I, J = a // mb, h // mb
        if I != J:
            adj[I].add(J)
            adj[J].add(I)
    n_orig = sum(len(x) for x in adj) // 2
    alive, levels = set(range(N)), []
    while alive:
        order = sorted(alive, key=lambda i: (len(adj[i] & alive), i))
        E, blocked = [], set()
        for i in order:
            if i not in blocked:
                E.append(i)
                blocked |= adj[i] | {i}
        E.sort()
        nbrs = [sorted(adj[i] & alive) for i in E]
        for nb in nbrs:
            for a in nb:
                adj[a] |= set(nb) - {a}
        alive -= set(E)
        levels.append((E, nbrs))
    blocks = sorted((I, J) for I in range(N) for J in adj[I] if J > I)
    slot = {b: N + k for k, b in enumerate(blocks)}
    slot.update({(i, i): i for i in range(N)})
    items = []
    for E, nbrs in levels:
        blk, rhs = {}, {}
        for i, nb in zip(E, nbrs):
            for x, j in enumerate(nb):
                s2 = (slot[(min(i, j), max(i, j))], int(j < i))
                rhs.setdefault(j, []).append([i, *s2, x])
                for y in range(x, len(nb)):
                    blk.setdefault((j, nb[y]), []).append([i, *s2, y])
        items.append([[slot[k], blk[k]] for k in sorted(blk)] + [[j, rhs[j]] for j in sorted(rhs)])
    return dict(mb=mb, N=N, n_orig=n_orig, blocks=[list(b) for b in blocks], levels=levels, items=items)


def run_plan_numpy(r, rng):
    """the plan on a random block-SPD matrix with its original pattern; writes go only to the plan's slots"""
    N, m = r["N"], r["m"]
    orig = [tuple(b) for b in r["blocks"]][:]
    A = np.zeros((N * m, N * m))
    blk = lambda M, I, J: M[I * m:(I + 1) * m, J * m:(J + 1) * m]
    pattern = [(i, i) for i in range(N)] + [b for b in orig if b in r["_orig_pattern"]]
    for I, J in pattern:
        X = rng.normal(size=(m, m))
        blk(A, I, J)[:] = X
        blk(A, J, I)[:] = X.T
    A = (A + A.T) / 2 + 3 * m * np.sqrt(len(r["blocks"]) + N) * np.eye(N * m)
    b = rng.normal(size=N * m)
    W = {i: blk(A, i, i).copy() for i in range(N)}
    W.update({N + k: blk(A, I, J).copy() for k, (I, J) in enumerate(orig)})
    rb = {i: b[i * m:(i + 1) * m].copy() for i in range(N)}
    Z, zc = {}, {}
    U = lambda s, tr: W[s].T if tr else W[s]          # U_ij from its slot
    for lv in r["levels"]:
        for i, nb in zip(lv["nodes"], lv["nbrs"]):
            Di = W[i]
            cols = [U(*_slot2(r, i, j)) for j in nb]
            Z[i] = np.linalg.solve(Di, np.hstack(cols)) if cols else np.zeros((m, 0))
            zc[i] = np.linalg.solve(Di, rb[i])
        for k, (out, cs) in enumerate(lv["items"]):
            if k < lv["n_blk"]:
                acc = sum(U(s, tr).T @ Z[i][:, col * m:(col + 1) * m] for i, s, tr, col in cs)
                W[out] = W[out] - acc                      # KeyError: a write outside the plan's blocks
            else:
                rb[out] = rb[out] - sum(U(s, tr).T @ zc[i] for i, s, tr, col in cs)
    x = {}
    for lv in reversed(r["levels"]):
        for i, nb in zip(lv["nodes"], lv["nbrs"]):
            x[i] = zc[i] - sum((Z[i][:, a * m:(a + 1) * m] @ x[j] for a, j in enumerate(nb)), np.zeros(m))
    xs = np.concatenate([x[i] for i in range(N)])
    ref = np.linalg.solve(A, b)
    return np.abs(xs - ref).max() / np.abs(ref).max()


def _slot2(r, i, j):
    I, J = min(i, j), max(i, j)
    return (i if i == j else r["N"] + r["blocks"].index([I, J])), int(j < i)


def checked_plan(p):
    rc, s = plan_report(p)
    assert rc == 0, s
    r = json.loads(s)
    want = plan_numpy(p)
    assert (r["mb"], r["N"], r["m"], r["n_orig_blocks"]) == (want["mb"], want["N"], 6 * want["mb"], want["n_orig"])
    assert r["blocks"] == want["blocks"]
    assert len(r["levels"]) == len(want["levels"])
    for lv, (E, nbrs), items in zip(r["levels"], want["levels"], want["items"]):
        assert lv["nodes"] == E and lv["nbrs"] == nbrs
        assert lv["items"] == items
    z = [o for lv in r["levels"] for o in lv["z_off"]]
    deg = [len(nb) for lv in r["levels"] for nb in lv["nbrs"]]
    assert z == list(np.cumsum([0] + [r["m"] ** 2 * d for d in deg])[:-1])
    return r


# ------------------------------------------------------------------------------------------------------------------
# CPU tests
# ------------------------------------------------------------------------------------------------------------------
def test_plan_of_the_too_wide_problem(built):
    r = checked_plan(too_wide_problem())
    assert (r["mb"], r["N"], r["n_orig_blocks"], len(r["blocks"]), len(r["levels"])) == (19, 11, 11, 19, 5)


@pytest.mark.parametrize("name", [k for k in GPU_CASES if k != "too_wide"])
def test_plan_of_the_loop_problems(built, name):
    checked_plan(GPU_CASES[name]())


@pytest.mark.parametrize("name", list(GPU_CASES))
def test_gpu_case_shapes(built, name):
    p = GPU_CASES[name]()
    assert shape_claims(p)["solver"] == "too wide"
    r = checked_plan(p)
    shape = (r["mb"], r["N"], len(r["levels"]))
    assert shape == GPU_SHAPES[name], shape
    if name == "loop300_chords":
        assert max(len(nb) for lv in r["levels"] for nb in lv["nbrs"]) >= 3


@pytest.mark.parametrize("name", ["too_wide", "loop200_fixed", "loop300_chords"])
def test_plan_solves_a_random_block_spd_system(built, name):
    p = GPU_CASES[name]()
    r = checked_plan(p)
    want = plan_numpy(p)
    # the original (pre-fill) off-diagonal blocks: rebuild them from the keyframe pattern
    nG, sets, _ = _free_sets(p, 0)
    mb = r["mb"]
    orig = set()
    for s in sets:
        I = sorted(set((s // mb).tolist()))
        orig |= {(a, b) for a in I for b in I if a < b}
    assert len(orig) == want["n_orig"]
    r["_orig_pattern"] = orig
    err = run_plan_numpy(r, np.random.default_rng(3))
    assert err < 1e-10, err


def structure_only_problem(n_super, mb):
    """n_super * mb free keyframes (plus one fixed), with no tracks: one point at distance mb sets the super-block size, and
    one point links every pair of super-blocks (a different keyframe of each block per pair, within the neighbour limit).
    Only the structure is meaningful."""
    nG = n_super * mb
    lists = [[1, 1 + mb]]
    for I in range(n_super):
        for J in range(I + 1, n_super):
            lists.append([1 + I * mb + J % mb, 1 + J * mb + I % mb])
    n_kf, n_pt = nG + 1, len(lists)
    obs = np.asarray(lists, np.int32).ravel()
    return dict(n_win=1, kf_off=np.int32([0, n_kf]), pt_off=np.int32([0, n_pt]), ln_off=np.int32([0, 0]),
                kf_Tcw=np.tile(np.float64([1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0]), (n_kf, 1)),
                kf_fixed=np.uint8([1] + [0] * nG), kf_intr=np.tile(np.float64([500, 500, 320, 240, 40]), (n_kf, 1)),
                kf_line_cam=np.zeros((n_kf, 4)), pt_xyz=np.zeros((n_pt, 3)), pt_obs_off=np.arange(0, 2 * n_pt + 1, 2, dtype=np.int32),
                pt_obs_kf=obs, pt_obs_uvr=np.zeros((2 * n_pt, 3), np.float32), pt_obs_info=np.ones(2 * n_pt, np.float32),
                ln_x0_dir=np.zeros((0, 6)), ln_obs_off=np.int32([0]), ln_obs_kf=np.zeros(0, np.int32),
                ln_obs_left=np.zeros((0, 4), np.float32), ln_obs_right=np.zeros((0, 4), np.float32),
                ln_obs_info=np.zeros((0, 2)), ln_obs_stereo=np.zeros(0, np.uint8), robust_points=0, delta_pt_mono=1.0,
                delta_pt_stereo=1.0, delta_ln_mono=1.0, delta_ln_stereo=1.0, chi2_pt_mono=5.991, chi2_pt_stereo=7.815,
                ln_endpoints_normalized=0, ln_filter=0)


def test_capacity_limit(built):
    """a super-block graph that is complete from the start: the plan stores every block and the Z factors of every pair.
    20 super-blocks fit; 110 need 12 210 blocks of 156 x 156 doubles, over the 2 GiB limit."""
    rc, s = plan_report(structure_only_problem(20, 26))
    assert rc == 0, s
    r = json.loads(s)
    assert (r["mb"], r["N"], len(r["blocks"]), len(r["levels"])) == (26, 20, 190, 20) and r["bytes"] < SP_MAX_BYTES
    rc, msg = plan_report(structure_only_problem(110, 26))
    assert rc == ERR_UNSUPPORTED, msg
    assert str(SP_MAX_BYTES) in msg and "110 super-blocks of 26 keyframes" in msg and "5995 off-diagonal blocks" in msg, msg


# ------------------------------------------------------------------------------------------------------------------
# GPU tests
# ------------------------------------------------------------------------------------------------------------------
SP_KERNELS = {"k_sp_assemble", "k_sp_factor", "k_sp_solve<15>", "k_sp_update", "k_sp_backsub"}   # m = 6 * 19 <= 120


def _context(topo_cache, sparse):
    c = capi.Context(0)
    d = _bind(c.lib)
    d.lld_ctx_set_topo_cache(c.handle, topo_cache)
    c.lib.dll.lld_ctx_set_gba_sparse(c.handle, sparse)
    return c


@pytest.fixture(scope="module")
def sctx(built):
    """switch on, cache off: every call indexes its problem again"""
    c = _context(0, 1)
    yield c
    c.close()


def assert_sparse_arm(names):
    assert SP_KERNELS <= names, names
    assert not names & {"k_cr_factor", "k_cr_solve<15>", "k_cr_solve<20>", "k_cr_update", "k_solve_env"}, names


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(GPU_CASES))
def test_global_loop_sparse(sctx, name):
    p = GPU_CASES[name]()
    _, names = checked(p, sctx, "global", (10,), name)
    assert_sparse_arm(names)


@pytest.mark.gpu
def test_switch_on_the_same_context(sctx):
    """switch off: the existing rejection again; a cyclic-reduction problem keeps its arm and its bits with the switch on"""
    d = sctx.lib.dll
    d.lld_ctx_set_gba_sparse(sctx.handle, 0)
    try:
        msg = expect_error(too_wide_problem(), sctx, "global", ERR_UNSUPPORTED, "envelope", "bytes of shared memory")
        assert str(SMEM_LIMIT) in msg, msg
        q = cr_problem(10, 85)
        off, names_off = profiled(q, sctx, "global", (8,))
    finally:
        d.lld_ctx_set_gba_sparse(sctx.handle, 1)
    on, names_on = profiled(q, sctx, "global", (8,))
    assert_identical(on, off, "CR with the switch on vs off")
    assert names_on == names_off and "k_cr_factor" in names_on and not any(n.startswith("k_sp_") for n in names_on), names_on
    check_ba(on, oracle(q, "global", (8,)), "CR with the switch on")


@pytest.mark.gpu
def test_topo_cache_loop(sctx):
    """warm calls with new values are bit-identical to cold calls and upload the value arrays only; the switch is part of
    the cache key"""
    c = _context(1, 1)
    try:
        p0 = GPU_CASES["loop200"]()
        run(p0, c, "global", (10,))                                   # index the structure
        for i, what in enumerate(("perturb", "noise", "info")):
            q = new_values(p0, 20 + i, what)
            g = run(q, c, "global", (10,))
            assert h2d_bytes(c) == value_bytes(q), (what, h2d_bytes(c), value_bytes(q))
            assert_identical(g, run(q, sctx, "global", (10,)), f"loop warm {what} vs cold")
            check_ba(g, oracle(q, "global", (10,)), f"loop warm {what}")
        # switch off on the same structure: not a cache hit but the rejection
        c.lib.dll.lld_ctx_set_gba_sparse(c.handle, 0)
        expect_error(p0, c, "global", ERR_UNSUPPORTED, "envelope")
        # a cyclic-reduction structure indexed with the switch off misses the cache when the switch turns on
        q = cr_problem(10, 85)
        run(q, c, "global", (8,))
        run(q, c, "global", (8,))
        assert h2d_bytes(c) == value_bytes(q)
        c.lib.dll.lld_ctx_set_gba_sparse(c.handle, 1)
        run(q, c, "global", (8,))
        assert h2d_bytes(c) > value_bytes(q)
    finally:
        c.close()
