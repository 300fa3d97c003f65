#!/usr/bin/env python
"""Timing of the SURVEY §8(f) kernels (ComputeStereoMatches, relocalisation / map-point SearchByProjection, temporal line
association, distinctive descriptors, SearchForInitialization, OptimizeSim3, Sim3Solver, PnPsolver): device compute time from the library's own CUDA events (host buffers in, results
out through the public call), wall clock of the same call, and the CPU oracle on the same or a smaller sample.
Prints one JSON object; results are compared with the oracle where the sample is the same.
Usage: aux_kernels.py [section ...]   (default: every section)"""
import json, os, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
from lld_slam_b200 import api, capi, synth

ctx = capi.Context(0)
out = {}


def timed(fn, reps=5):
    fn()
    ms, wall = [], []
    for _ in range(reps):
        t0 = time.perf_counter(); r = fn(); wall.append((time.perf_counter() - t0) * 1e3); ms.append(ctx.last_timing()[1])
    return r, float(np.median(ms)), float(np.median(wall))


def cpu(fn):
    t0 = time.perf_counter(); r = fn(); return r, (time.perf_counter() - t0) * 1e3


# sections to run: all by default, or the ones named on the command line
SECTIONS = set(sys.argv[1:])
want = lambda name: not SECTIONS or name in SECTIONS   # noqa: E731

# ---- Frame::ComputeStereoMatches, KITTI-sized frames
if want("compute_stereo_matches"):
    nf = 32
    frames = [synth.make_stereo_frame(100 + s, n_kp=2000, rows=376, cols=1241, n_levels=8) for s in range(nf)]
    p = synth.batch_stereo(frames)
    g, ms, wall = timed(lambda: api.stereo_matches(p, impl="gpu", ctx=ctx))
    p4 = synth.batch_stereo(frames[:4])
    o, tc = cpu(lambda: api.stereo_matches(p4, impl="oracle"))
    out["compute_stereo_matches"] = {"frames": nf, "keypoints": 2000, "image": "1241x376, 8 levels", "device_ms": ms, "call_ms": wall,
                                     "frames_per_s_device": nf / ms * 1e3, "cpu_oracle_ms_per_frame": tc / 4,
                                     "bit_exact_on_sample": bool(np.array_equal(api.stereo_matches(p4, impl="gpu", ctx=ctx)["uright"], o["uright"]))}

# ---- relocalisation variant of SearchByProjection
if want("sbp_relocalisation"):
    pr = synth.make_sbp_frame_batch(256, 2000, 777, th=10.0)
    pr["mono"] = 1
    pr["cur_uright"] = np.full_like(pr["cur_uright"], -1.0)
    pr["last_has_obs"] = np.ones_like(pr["last_has_obs"])
    pr["th_high"] = 100; pr["allow_negative_depth"] = 1
    g, ms, wall = timed(lambda: api.sbp_frame(pr, impl="gpu", ctx=ctx))
    out["sbp_relocalisation"] = {"pairs": 256, "keypoints": 2000, "device_ms": ms, "call_ms": wall, "queries_per_s_device": 256 * 2000 / ms * 1e3}

# ---- map points -> frame
if want("sbp_mappoints"):
    pm = synth.make_sbp_mp_batch(256, 2000, 1500, 5)
    g, ms, wall = timed(lambda: api.sbp_mappoints(pm, impl="gpu", ctx=ctx))
    o, tc = cpu(lambda: api.sbp_mappoints(synth.make_sbp_mp_batch(8, 2000, 1500, 5), impl="oracle"))
    out["sbp_mappoints"] = {"frames": 256, "keypoints": 2000, "map_points": 1500, "device_ms": ms, "call_ms": wall,
                            "queries_per_s_device": 256 * 1500 / ms * 1e3, "cpu_oracle_ms_per_frame": tc / 8}

# ---- keyframe searches (Fuse with the reprojection gate; SearchByProjection(KeyFrame*, Scw) with sequential claims)
if want("kf_search"):
    for name, gate, claims in (("fuse_search", 1, 0), ("sim3_search_by_projection", 0, 1)):
        pk = synth.make_kf_search_batch(256, 2000, 1500, 9, chi2_gate=gate, sequential_claims=claims)
        g, ms, wall = timed(lambda: api.kf_search(pk, impl="gpu", ctx=ctx))
        o, tc = cpu(lambda: api.kf_search(synth.make_kf_search_batch(8, 2000, 1500, 9, chi2_gate=gate, sequential_claims=claims), impl="oracle"))
        out[name] = {"keyframes": 256, "keypoints": 2000, "map_points": 1500, "device_ms": ms, "call_ms": wall,
                     "queries_per_s_device": 256 * 1500 / ms * 1e3, "cpu_oracle_ms_per_keyframe": tc / 8}

# ---- SearchForTriangulation
if want("search_for_triangulation"):
    pt = synth.make_tri_search_batch(256, 2000, 13)
    g, ms, wall = timed(lambda: api.tri_search(pt, impl="gpu", ctx=ctx))
    o, tc = cpu(lambda: api.tri_search(synth.make_tri_search_batch(8, 2000, 13), impl="oracle"))
    out["search_for_triangulation"] = {"keyframe_pairs": 256, "keypoints": 2000, "vocabulary_nodes": 300, "device_ms": ms, "call_ms": wall,
                                       "pairs_per_s_device": 256 / ms * 1e3, "cpu_oracle_ms_per_pair": tc / 8}

# ---- SearchByBoW (keyframe -> frame)
if want("search_by_bow"):
    pb = synth.make_bow_search_batch(256, 2000, 17, n_nodes=300)
    g, ms, wall = timed(lambda: api.bow_search(pb, impl="gpu", ctx=ctx))
    o, tc = cpu(lambda: api.bow_search(synth.make_bow_search_batch(8, 2000, 17, n_nodes=300), impl="oracle"))
    out["search_by_bow"] = {"pairs": 256, "keypoints": 2000, "vocabulary_nodes": 300, "device_ms": ms, "call_ms": wall,
                            "pairs_per_s_device": 256 / ms * 1e3, "cpu_oracle_ms_per_pair": tc / 8}

# ---- temporal line association
if want("line_association"):
    pa = synth.make_line_assoc_batch(256, 300, 250, 64, 21, n_cand=40)
    g, ms, wall = timed(lambda: api.line_associate(pa, impl="gpu", ctx=ctx))
    pa8 = synth.make_line_assoc_batch(8, 300, 250, 64, 21, n_cand=40)
    o, tc = cpu(lambda: api.line_associate(pa8, impl="oracle"))
    out["line_association"] = {"frames": 256, "map_lines": 300, "current_lines": 250, "candidates": 40, "device_ms": ms, "call_ms": wall,
                               "frames_per_s_device": 256 / ms * 1e3, "cpu_oracle_ms_per_frame": tc / 8}

# ---- distinctive descriptors
if want("medoid"):
    import test_cpu_oracle as tco
    off, desc = tco._medoid_landmarks(11, n_lm=100000, max_obs=40)
    g, ms, wall = timed(lambda: api.medoid_orb(off, desc, impl="gpu", ctx=ctx))
    off8, desc8 = tco._medoid_landmarks(11, n_lm=5000, max_obs=40)
    o, tc = cpu(lambda: api.medoid_orb(off8, desc8, impl="oracle"))
    out["medoid_orb"] = {"map_points": 100000, "observations": int(off[-1]), "device_ms": ms, "call_ms": wall,
                         "map_points_per_s_device": 100000 / ms * 1e3, "cpu_oracle_us_per_point": tc / 5000 * 1e3}
    off, desc = tco._medoid_landmarks(12, n_lm=20000, max_obs=30, dim=64)
    g, ms, wall = timed(lambda: api.medoid_float(off, desc, impl="gpu", ctx=ctx))
    out["medoid_float"] = {"map_lines": 20000, "observations": int(off[-1]), "dim": 64, "device_ms": ms, "call_ms": wall,
                           "map_lines_per_s_device": 20000 / ms * 1e3}

# ---- SearchForInitialization (Tracking::MonocularInitialization: ORBmatcher(0.9, true), windowSize = 100)
if want("search_for_initialization"):
    import subprocess
    import torch
    pi = synth.make_init_search_batch(256, 2000, 71)
    g, ms, wall = timed(lambda: api.init_search(pi, impl="gpu", ctx=ctx))
    p8 = synth.make_init_search_batch(8, 2000, 71)          # the first 8 pairs of the batch above
    o, tc = cpu(lambda: api.init_search(p8, impl="oracle"))
    n8 = int(p8["kp1_off"][-1])
    exact = (np.array_equal(g["match12"][:n8], o["match12"]) and np.array_equal(g["n_matches"][:8], o["n_matches"])
             and np.array_equal(g["prev_matched"][:n8].view(np.uint32), o["prev_matched"].view(np.uint32)))
    _, prof = ctx.profile(lambda: api.init_search(pi, impl="gpu", ctx=ctx))   # separate, profiled run: per-launch CUDA events
    part = lambda names: sum(prof[k]["ms"] for k in names if k in prof)   # noqa: E731
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True).stdout
    out["search_for_initialization"] = {
        "pairs": 256, "keypoints": 2000, "window": 100, "image": "1241x376 (KITTI)", "device_ms": ms, "call_ms": wall,
        "pairs_per_s_device": 256 / ms * 1e3, "matches_per_pair": float(g["n_matches"].mean()),
        "cpu_oracle_ms_per_pair": tc / 8, "bit_exact_on_sample": bool(exact),
        "profile_ms": {k: v["ms"] for k, v in prof.items()},
        "split_ms": {"grid": part(["k_cell_count", "k_cell_scan", "k_cell_fill"]),
                     "candidate_listing": part(["k_init_count", "k_init_scan", "k_init_fill"]),
                     "resolve": part(["k_init_resolve_smem", "k_init_resolve_global"]), "histogram_and_output": part(["k_init_finalize"])},
        "gpu": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": smi.strip()}
# ---- OptimizeSim3 (LoopClosing::ComputeSim3: th2 = 10, 5 / 10 / 5 iterations), both scale modes
if want("optimize_sim3"):
    import subprocess
    import torch
    res = {}
    for fix in (1, 0):
        ps = synth.make_sim3_batch(4096, 300, 131 + fix, fix_scale=fix)
        g, ms, wall = timed(lambda: api.sim3_opt(ps, impl="gpu", ctx=ctx))
        _, prof = ctx.profile(lambda: api.sim3_opt(ps, impl="gpu", ctx=ctx))   # separate, profiled run: per-launch CUDA events
        p1 = synth.make_sim3_batch(1, 300, 131 + fix, fix_scale=fix)   # the batch-of-one call the shim makes per candidate
        one = []
        api.sim3_opt(p1, impl="gpu", ctx=ctx)
        for _ in range(50):
            t0 = time.perf_counter(); api.sim3_opt(p1, impl="gpu", ctx=ctx); one.append((time.perf_counter() - t0) * 1e3)
        one_dev = ctx.last_timing()[1]
        p16 = synth.make_sim3_batch(16, 300, 131 + fix, fix_scale=fix)  # the first 16 problems of the batch above
        o, tc = cpu(lambda: api.sim3_opt(p16, impl="oracle"))
        same = (np.array_equal(g["inlier"][:int(p16["off"][-1])], o["inlier"]) and np.array_equal(g["n_in"][:16], o["n_in"])
                and np.array_equal(g["n_iter_done"][:16], o["n_iter_done"]))
        rel = float((np.abs(g["chi2_log"][:16] - o["chi2_log"]) / np.maximum(np.abs(o["chi2_log"]), 1e-300)).max())
        res["fixed_scale" if fix else "free_scale"] = {
            "problems": 4096, "correspondences": 300, "device_ms": ms, "call_ms_from_host_buffers": wall,
            "problems_per_s_device": 4096 / ms * 1e3, "kernel_profile_ms": {k: v["ms"] for k, v in prof.items()},
            "batch_of_one_call_ms_median": float(np.median(one)), "batch_of_one_device_ms": one_dev,
            "cpu_oracle_ms_per_problem": tc / 16, "mean_inliers": float(g["n_in"].mean()),
            "oracle_sample_16": {"inlier_n_in_iterations_identical": bool(same), "chi2_log_max_rel": rel}}
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True).stdout
    res["gpu"] = torch.cuda.get_device_name(0)
    res["nvidia_smi_name_power_limit"] = smi.strip()
    res["cpu"] = next((l.split(":", 1)[1].strip() for l in open("/proc/cpuinfo") if l.startswith("model name")), "")
    out["optimize_sim3"] = res
# ---- Sim3Solver (LoopClosing::ComputeSim3: SetRansacParameters(0.99, 20, 300), iterate(5) per round), both scale modes
if want("sim3_ransac"):
    import subprocess
    import torch
    from test_sim3_ransac import run_rounds
    res = {}
    for fix in (1, 0):
        ps = synth.make_sim3_ransac_batch(4096, 300, 701 + fix, fix_scale=fix)
        g, ms, wall = timed(lambda: api.sim3_ransac(ps, impl="gpu", ctx=ctx))
        _, prof = ctx.profile(lambda: api.sim3_ransac(ps, impl="gpu", ctx=ctx))   # separate, profiled run: per-launch CUDA events
        # ComputeSim3 rounds of 5 over the same candidates (each round one call; draws on the host are not timed)
        dev, calls = [], []
        def gpu_round(q):
            t0 = time.perf_counter(); o = api.sim3_ransac(q, impl="gpu", ctx=ctx); calls.append((time.perf_counter() - t0) * 1e3)
            dev.append(ctx.last_timing()[1]); return o
        run_rounds(ps, gpu_round, seed=fix)
        # the batch-of-one round (5 sets) a caller without batching makes per candidate
        p1 = synth.make_sim3_ransac_batch(1, 300, 711 + fix, fix_scale=fix, outlier_range=(0.9, 0.9), n_iterations=5)
        one = []
        api.sim3_ransac(p1, impl="gpu", ctx=ctx)
        for _ in range(50):
            t0 = time.perf_counter(); api.sim3_ransac(p1, impl="gpu", ctx=ctx); one.append((time.perf_counter() - t0) * 1e3)
        one_dev = ctx.last_timing()[1]
        o1, t1 = cpu(lambda: [api.sim3_ransac(p1, impl="oracle") for _ in range(50)])
        sub = synth.make_sim3_ransac_batch(64, 300, 701 + fix, fix_scale=fix)   # the first 64 problems of the batch above
        o, tc = cpu(lambda: api.sim3_ransac(sub, impl="oracle"))
        h = int(sub["hyp_off"][-1])
        same = all(np.array_equal(g[k][:len(o[k])], o[k]) for k in ("found", "no_more", "n_inliers", "its_done", "inlier"))
        res["fixed_scale" if fix else "free_scale"] = {
            "problems": 4096, "correspondences": 300, "minimal_sets_in_call": int(ps["hyp_off"][-1]),
            "sets_evaluated": int((g["hyp_inliers"] >= 0).sum()), "found": int(g["found"].sum()),
            "full_budget_one_call": {"device_ms": ms, "call_ms_from_host_buffers": wall, "problems_per_s_device": 4096 / ms * 1e3,
                                     "kernel_profile_ms": {k: v["ms"] for k, v in prof.items()}},
            "rounds_of_5": {"rounds": len(dev), "device_ms_total": float(np.sum(dev)), "call_ms_total": float(np.sum(calls)),
                            "first_round_call_ms": calls[0], "last_round_call_ms": calls[-1]},
            "batch_of_one_round_of_5": {"call_ms_median": float(np.median(one)), "device_ms": one_dev,
                                        "cpu_oracle_ms": t1 / 50},
            "cpu_oracle_ms_per_problem_full_budget": tc / 64, "cpu_oracle_sets_evaluated_sample": int((o["hyp_inliers"] >= 0).sum()),
            "oracle_sample_64_identical": bool(same)}
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True).stdout
    res["gpu"] = torch.cuda.get_device_name(0)
    res["nvidia_smi_name_power_limit"] = smi.strip()
    res["cpu"] = next((l.split(":", 1)[1].strip() for l in open("/proc/cpuinfo") if l.startswith("model name")), "")
    out["sim3_ransac"] = res
# ---- PnPsolver (Tracking::Relocalization: SetRansacParameters(0.99, 10, 300, 4, 0.5, 5.991), iterate(5) per round)
if want("pnp_ransac"):
    import subprocess
    import torch
    from test_pnp_ransac import run_rounds
    res = {}
    ps = synth.make_pnp_ransac_batch(4096, 200, 801)
    g, ms, wall = timed(lambda: api.pnp_ransac(ps, impl="gpu", ctx=ctx))
    _, prof = ctx.profile(lambda: api.pnp_ransac(ps, impl="gpu", ctx=ctx))   # separate, profiled run: per-launch CUDA events
    # relocalisation rounds of 5 over the same candidates (each round one call; draws on the host are not timed)
    dev, calls = [], []
    def gpu_round(q):
        t0 = time.perf_counter(); o = api.pnp_ransac(q, impl="gpu", ctx=ctx); calls.append((time.perf_counter() - t0) * 1e3)
        dev.append(ctx.last_timing()[1]); return o
    fin, n_rounds = run_rounds(ps, gpu_round)
    # the batch-of-one round (iterate(5) on one candidate) a caller without batching makes
    p1 = synth.make_pnp_ransac_batch(1, 200, 811, outlier_range=(0.9, 0.9))
    one = []
    api.pnp_ransac(p1, impl="gpu", ctx=ctx)
    for _ in range(50):
        t0 = time.perf_counter(); api.pnp_ransac(p1, impl="gpu", ctx=ctx); one.append((time.perf_counter() - t0) * 1e3)
    one_dev = ctx.last_timing()[1]
    o1, t1 = cpu(lambda: [api.pnp_ransac(p1, impl="oracle") for _ in range(50)])
    sub = synth.make_pnp_ransac_batch(4096, 200, 801)
    o, tc = cpu(lambda: api.pnp_ransac(sub, impl="oracle"))
    same = all(np.array_equal(g[k], o[k], equal_nan=True) for k in g)
    fo, _ = run_rounds(ps, lambda q: api.pnp_ransac(q, impl="oracle"))
    same_rounds = all(np.array_equal(fin[k], fo[k]) for k in fin)
    res["reloc"] = {
        "problems": 4096, "correspondences": 200, "minimal_sets_in_call": int(ps["hyp_off"][-1]),
        "sets_evaluated": int((g["hyp_inliers"] >= 0).sum()), "found": int(g["found"].sum()),
        "full_budget_one_call": {"device_ms": ms, "call_ms_from_host_buffers": wall, "problems_per_s_device": 4096 / ms * 1e3,
                                 "kernel_profile_ms": {k: v["ms"] for k, v in prof.items()}, "cpu_oracle_ms": tc,
                                 "identical_to_oracle": bool(same)},
        "rounds_of_5": {"rounds": n_rounds, "device_ms_total": float(np.sum(dev)), "call_ms_total": float(np.sum(calls)),
                        "first_round_call_ms": calls[0], "last_round_call_ms": calls[-1], "identical_to_oracle": bool(same_rounds)},
        "batch_of_one_round_of_5": {"call_ms_median": float(np.median(one)), "device_ms": one_dev, "cpu_oracle_ms": t1 / 50}}
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True).stdout
    res["gpu"] = torch.cuda.get_device_name(0)
    res["nvidia_smi_name_power_limit"] = smi.strip()
    res["cpu"] = next((l.split(":", 1)[1].strip() for l in open("/proc/cpuinfo") if l.startswith("model name")), "")
    out["pnp_ransac"] = res
print(json.dumps(out))
