#!/usr/bin/env python
"""Global BA after a loop closure at the BASELINE configs[4] size: 1.5k keyframes / 300k points / 60k lines plus points that
link the first and the last free keyframes, solved by block elimination over the super-block graph
(lld_ctx_set_gba_sparse, sp_solver.cuh).  Reports the resident time of the LM iterations and the end-to-end time, the
share of the solver kernels from the per-launch profile, the same problem without the loop points (cyclic reduction),
the CPU oracle's time, and the GPU with its power limit.

  python tools/gba_loop.py --out profiles/r3_gba_loop.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
from lld_slam_b200 import api, capi, synth  # noqa: E402
from test_ba_paths import add_points, free_kfs, shape_claims  # noqa: E402


def problems(n_kf, n_pt, n_ln, n_loop, seed):
    rng = np.random.default_rng(seed)
    w = synth.make_ba_window(n_kf, n_pt, n_ln, rng, mean_track=6.0, track_mode="geometric", global_mode=True)
    base = synth.batch_ba([w], "global")
    F = free_kfs(w)
    for _ in range(n_loop):
        w = add_points(w, [[F[rng.integers(0, 10)], F[len(F) - 1 - rng.integers(0, 10)]]], rng, True,
                       ahead=150.0, side=(rng.uniform(-1, 1), -2.0))
    return base, synth.batch_ba([w], "global")


def measure(p, iters, reps, sparse):
    ctx = capi.Context(0)
    d = ctx.lib.dll
    d.lld_ctx_set_gba_sparse(ctx.handle, 1 if sparse else 0)
    d.lld_ctx_profile.argtypes = [C.c_void_p, C.c_int]; d.lld_ctx_profile.restype = None
    d.lld_ctx_profile_report.argtypes = [C.c_void_p, C.c_char_p, C.c_int]; d.lld_ctx_profile_report.restype = C.c_int
    api.ba_global(p, iters, impl="gpu", ctx=ctx)   # warm-up (indexes the structure; later calls hit the topology cache)
    e2e, res = [], []
    for _ in range(reps):
        t = time.perf_counter()
        g = api.ba_global(p, iters, impl="gpu", ctx=ctx)
        e2e.append(1e3 * (time.perf_counter() - t))
        res.append(ctx.last_timing()[1])
    d.lld_ctx_profile(ctx.handle, 1)
    api.ba_global(p, iters, impl="gpu", ctx=ctx)
    buf = C.create_string_buffer(1 << 16)
    ctx.check(d.lld_ctx_profile_report(ctx.handle, buf, len(buf)), "lld_ctx_profile_report")
    d.lld_ctx_profile(ctx.handle, 0)
    prof = json.loads(buf.value.decode())
    ctx.close()
    total = sum(v["ms"] for v in prof.values())
    solver = {k: v for k, v in prof.items() if k.startswith("k_sp_") or k.startswith("k_cr_")}
    return g, dict(resident_ms_median=float(np.median(res)), e2e_ms_median=float(np.median(e2e)), resident_ms=res, e2e_ms=e2e,
                   profiled_kernel_ms=total, solver_kernel_ms=sum(v["ms"] for v in solver.values()),
                   solver_share=sum(v["ms"] for v in solver.values()) / total if total else None, solver_kernels=solver,
                   n_iter_done=g["n_iter_done"].tolist())


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        pl = f"unavailable ({e})"
    return name, pl


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--kf", type=int, default=1500)
    ap.add_argument("--pts", type=int, default=300000)
    ap.add_argument("--lines", type=int, default=60000)
    ap.add_argument("--loop", type=int, default=60, help="points linking the first and the last 10 free keyframes")
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--seed", type=int, default=5)
    ap.add_argument("--no-oracle", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_gba_loop.json"))
    a = ap.parse_args()
    base, loop = problems(a.kf, a.pts, a.lines, a.loop, a.seed)
    cb, cl = shape_claims(base), shape_claims(loop)
    name, pl = gpu_info()
    out = dict(gpu=name, power_limit=pl, shape=dict(kf=a.kf, pts=a.pts, lines=a.lines, loop_points=a.loop, iters=a.iters),
               loop_free=dict(B=cb["B"], solver=cb["solver"]), loop=dict(B=cl["B"], solver_without_switch=cl["solver"]))
    lib = capi.load_library()
    prob, keep = capi.fill_struct(capi.BaProblem, loop)
    buf = C.create_string_buffer(1 << 26)
    rc = lib.dll.lld_gba_sparse_plan_report(C.byref(prob), buf, len(buf))
    plan = json.loads(buf.value.decode()) if rc == 0 else {"error": buf.value.decode()}
    out["plan"] = {k: plan.get(k) for k in ("mb", "N", "n_orig_blocks", "bytes")}
    if "levels" in plan:
        out["plan"].update(blocks_with_fill=len(plan["blocks"]), levels=[len(lv["nodes"]) for lv in plan["levels"]])
    g_loop, out["loop"]["gpu_sparse"] = measure(loop, a.iters, a.reps, True)
    _, out["loop_free"]["gpu_cr"] = measure(base, a.iters, a.reps, False)
    if not a.no_oracle:
        t = time.perf_counter()
        o = api.ba_global(loop, a.iters, impl="oracle")
        out["loop"]["oracle_s"] = time.perf_counter() - t
        k = int(o["n_iter_done"][0][0]) + 1
        rel = np.abs(g_loop["chi2_log"][0, :k] - o["chi2_log"][0, :k]) / o["chi2_log"][0, :k]
        out["loop"]["max_rel_chi2_vs_oracle"] = float(rel.max())
        out["loop"]["same_iterations_as_oracle"] = bool(np.array_equal(g_loop["n_iter_done"], o["n_iter_done"]))
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: v for k, v in out.items() if k != "plan"} | {"plan": out["plan"]}, indent=1))


if __name__ == "__main__":
    main()
