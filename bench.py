#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native point+line BA / descriptor-matching core.

A "step" is one full pass of the hot path over one batch of synthetic input:
  workload "batched_local_ba" (BASELINE.json configs[3] shape, weak scaling): per GPU `--windows` independent local-BA
  windows of 20 keyframes / 5 000 points / 1 000 lines, the reference schedule 5 + 15 LM iterations with the outlier
  round in between (Optimizer::LocalBundleAdjustment).  metric = LM outer iterations per second over all windows.
  workload "global_ba" (--workload global_ba; BASELINE.json configs[4], STRONG scaling): one global BA of 1.5k keyframes /
  300k points / 60k lines, 10 LM iterations, landmarks sharded over the ranks, reduced camera system all-reduced over NCCL.
Secondary workloads of BASELINE.json's metric (descriptor matches/s, pose-only frames/s, single-window local BA at the
north_star target shape 10 / 5k / 1k) are measured in the same run and reported under "extra"; at N > 1 the frame-pair
and frame batches (configs[1], configs[2]) are sharded over the ranks (no collective) and reported as whole-job rates.

`value`   : inputs resident in HBM, device-timed with CUDA events on the library's stream.
`e2e`     : the same step through the reference-shaped C-ABI call (lld_ba_local) with pinned HOST buffers: host indexing,
            H2D, compute, D2H all inside the timed region.
`roofline`: dominant kernel of the step from per-launch CUDA events (lld_ctx_profile), against MEASURED_PEAKS.json.
`cpu_baseline`: the CPU oracle (a restatement of the reference's g2o path; the reference itself cannot be built here)
            on one host core per problem, on a bounded sample of the same workload.
--impl reference : the CPU oracle on all host cores (rank 0 only).
--dump-outputs DIR : the results of the last timed step as .npy files (inputs are seeded: two builds compare one to one).
"""
import argparse
import atexit
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from lld_slam_b200 import api, capi, synth  # noqa: E402

WIN_KF, WIN_PT, WIN_LN = 20, 5000, 1000
ITS1, ITS2 = 5, 15


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, device):
        self.device = device
        self.proc = None
        self.lines = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.terminate)   # an exception before stop() must not leave the sampler running
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, val in zip(names, f[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def bind_resident(lib):
    d = lib.dll
    vp = C.c_void_p
    d.lld_ba_upload.argtypes = [vp, C.POINTER(capi.BaProblem), C.c_int, C.c_int]; d.lld_ba_upload.restype = C.c_int
    d.lld_ba_run_local.argtypes = [vp, C.c_int, C.c_int, capi.c_u8p]; d.lld_ba_run_local.restype = C.c_int
    d.lld_ba_sync.argtypes = [vp]; d.lld_ba_sync.restype = C.c_int
    d.lld_ba_download.argtypes = [vp, C.POINTER(capi.BaProblem), C.POINTER(capi.BaResult), C.c_int]; d.lld_ba_download.restype = C.c_int
    d.lld_ctx_profile.argtypes = [vp, C.c_int]; d.lld_ctx_profile.restype = None
    d.lld_ctx_profile_report.argtypes = [vp, C.c_char_p, C.c_int]; d.lld_ctx_profile_report.restype = C.c_int
    d.lld_ctx_last_bytes.argtypes = [vp, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]; d.lld_ctx_last_bytes.restype = None
    d.lld_ctx_event_record.argtypes = [vp, C.c_int]; d.lld_ctx_event_record.restype = C.c_int
    d.lld_ctx_event_elapsed_ms.argtypes = [vp]; d.lld_ctx_event_elapsed_ms.restype = C.c_float
    d.lld_sbp_frame_upload.argtypes = [vp, C.POINTER(capi.SbpFrameProblem)]; d.lld_sbp_frame_upload.restype = C.c_int
    d.lld_sbp_run.argtypes = [vp, C.POINTER(C.c_int)]; d.lld_sbp_run.restype = C.c_int
    d.lld_pose_upload.argtypes = [vp, C.POINTER(capi.PoseProblem)]; d.lld_pose_upload.restype = C.c_int
    d.lld_pose_run.argtypes = [vp]; d.lld_pose_run.restype = C.c_int
    return d


def profile_report(d, ctx):
    buf = C.create_string_buffer(1 << 16)
    ctx.check(d.lld_ctx_profile_report(ctx.handle, buf, len(buf)), "profile_report")
    return json.loads(buf.value.decode())


def pin(arr):
    """copy a numpy array into pinned host memory (torch-owned) and return the numpy view + keepalive"""
    import torch
    t = torch.from_numpy(np.ascontiguousarray(arr)).pin_memory()
    return t.numpy(), t


def pinned_problem(p):
    keep, out = [], {}
    for k, v in p.items():
        if isinstance(v, np.ndarray):
            a, t = pin(v)
            out[k] = a
            keep.append(t)
        else:
            out[k] = v
    return out, keep


DUMP_BYTES = 60 << 20   # array data written by --dump-outputs; with the .npy headers the files stay under 64 MB


def dump_outputs(path, out):
    """Write the result arrays of the timed path (an lld_ba_result filled by lld_ba_download) as <path>/<name>.npy so that
    two builds can be compared output for output.  Float arrays keep their dtype; integer and flag arrays are widened
    exactly (uint8 -> float32, int32 -> float64).  When the whole result exceeds DUMP_BYTES, every array keeps the same
    fraction of its rows, chosen by a fixed seed and kept in order: the sample depends only on the shapes."""
    arrs = {k: v if v.dtype.kind == "f" else v.astype(np.float32 if v.itemsize <= 2 else np.float64)
            for k, v in out.items() if isinstance(v, np.ndarray)}
    frac = min(1.0, DUMP_BYTES / sum(v.nbytes for v in arrs.values()))
    os.makedirs(path, exist_ok=True)
    for k, v in arrs.items():
        if frac < 1.0:
            n = len(v)
            v = v[np.sort(np.random.default_rng(0).choice(n, int(n * frac), replace=False))]
        np.save(os.path.join(path, k + ".npy"), v)


def edge_counts(p):
    n_pe = int(p["pt_obs_off"][-1])
    n_le = int(p["ln_obs_off"][-1]) + int((p["ln_obs_right"][:, 0] >= 0).sum())
    return n_pe, n_le


def free_edge_counts(p):
    """point edges / line cells whose keyframe is free (only those carry a W block into the Schur complement)"""
    fixed = p["kf_fixed"].astype(bool)
    kf_off = p["kf_off"]

    def count(lm_off, obs_off, obs_kf):
        n = 0
        for w in range(int(p["n_win"])):
            e0, e1 = int(obs_off[lm_off[w]]), int(obs_off[lm_off[w + 1]])
            n += int((~fixed[kf_off[w] + obs_kf[e0:e1]]).sum())
        return n
    return count(p["pt_off"], p["pt_obs_off"], p["pt_obs_kf"]), count(p["ln_off"], p["ln_obs_off"], p["ln_obs_kf"])


def algorithmic_bytes_step(p, iters_total, trials_total):
    """SURVEY.md §8(d), summed over the LM iterations actually executed in one step:
    per window and iteration with t trials  (1+t)(24 Ep + 36 El) + 2(1+t)(24 P + 40 L) + 96 Nkf + 8 (6 Nkf)^2.
    Every window has the same shape, so the batch total is the per-window figure times the iterations (and trials)
    summed over the windows."""
    n_pe, n_le = edge_counts(p)
    P, L, K = int(p["pt_off"][-1]), int(p["ln_off"][-1]), int(p["kf_off"][-1])
    nw = int(p["n_win"])
    edge = (24 * n_pe + 36 * n_le) / nw
    lm = 2 * (24 * P + 40 * L) / nw
    cam = 96 * K / nw + 8 * (6 * K / nw) ** 2
    return (iters_total + trials_total) * (edge + lm) + iters_total * cam


# per-kernel algorithmic bytes of OUR decomposition (DESIGN.md §kernels): what each launch must read + write once
def kernel_bytes(name, p):
    n_pe, n_le = edge_counts(p)
    n_lc = int(p["ln_obs_off"][-1])
    n_pw, n_lw = free_edge_counts(p)
    P, L, K = int(p["pt_off"][-1]), int(p["ln_off"][-1]), int(p["kf_off"][-1])
    nw = int(p["n_win"])
    nf = K / nw - 1
    tbl = {
        "k_lin_points<1>": n_pe * 24 + n_pw * 144 + P * (24 + 72),
        "k_lin_points<4>": n_pe * 24 + n_pw * 144 + P * (24 + 72),
        "k_lin_lines<1>": n_lc * 56 + n_lw * 192 + L * (40 + 112),
        "k_lin_lines<2>": n_lc * 56 + n_lw * 192 + L * (40 + 112),
        "k_lin_lines<4>": n_lc * 56 + n_lw * 192 + L * (40 + 112),
        "k_lin_lines<8>": n_lc * 56 + n_lw * 192 + L * (40 + 112),
        "k_lin_poses": n_pe * 24 + n_lc * 56 + (n_pe + n_lc) * 24,
        "k_schur_points": P * (72 + 80),
        "k_schur_lines": L * (112 + 112),
        # dense-mode Schur complement by co-visibility class: every W block and every landmark inverse record once
        "k_schur_piece<3>": n_pw * 144 + P * 80,
        "k_schur_piece<4>": n_lw * 192 + L * 112,
        "k_schur_tile<3>": n_pw * 144 + P * 80,
        "k_schur_tile<4>": n_lw * 192 + L * 112,
        "k_schur_rows": n_pe * (144 + 144) + n_lc * (192 + 192) + nw * 8 * 36 * nf * (nf + 1) / 2,
        "k_backsub_points<1>": n_pw * 144 + n_pe * (24 + 8) + P * (24 + 24 + 80),
        "k_backsub_points<4>": n_pw * 144 + n_pe * (24 + 8) + P * (24 + 24 + 80),
        "k_backsub_lines<1>": n_lw * 192 + n_lc * (56 + 16) + L * (40 + 40 + 112),
        "k_backsub_lines<2>": n_lw * 192 + n_lc * (56 + 16) + L * (40 + 40 + 112),
        "k_backsub_lines<4>": n_lw * 192 + n_lc * (56 + 16) + L * (40 + 40 + 112),
        "k_backsub_lines<8>": n_lw * 192 + n_lc * (56 + 16) + L * (40 + 40 + 112),
    }
    return tbl.get(name)


def make_batch(n_win, seed):
    return synth.make_local_ba_batch(n_win, WIN_KF, WIN_PT, WIN_LN, seed)


FP64_PEAK_TFLOPS = 36.3   # measured on this part: 62.5 DFMA / clk / SM (tools/ubench/fp64_probe.cu) x 148 SMs x 1.965 GHz x 2
GBA_SHAPE = (1500, 300000, 60000)
GBA_ITERS = 10


def algorithmic_flops_step(p, iters_total, trials_total):
    """SURVEY.md §8(d): ~400 flop per point edge, ~1100 per line edge (linearisation, once per iteration; the trial passes
    re-evaluate residuals only: ~90 / ~250), Schur 216 n(n+1)/2 + 160 n per point with n observing free keyframes
    (288 / 250 for lines), per trial."""
    n_pe, n_le = edge_counts(p)
    nw = int(p["n_win"])
    lin = (400.0 * n_pe + 1100.0 * n_le) / nw
    res = (90.0 * n_pe + 250.0 * n_le) / nw
    fixed = p["kf_fixed"].astype(bool)

    def schur(lm_off, obs_off, obs_kf, a, b):
        tot = 0.0
        w = 0   # every window has the same shape: evaluate the first one
        e0, e1 = int(obs_off[lm_off[w]]), int(obs_off[lm_off[w + 1]])
        free = ~fixed[p["kf_off"][w] + obs_kf[e0:e1]]
        cnt = np.add.reduceat(free.astype(np.int64), (obs_off[lm_off[w]:lm_off[w + 1]] - e0).astype(np.int64)) if e1 > e0 else np.zeros(0)
        tot = float((a * cnt * (cnt + 1) / 2 + b * cnt).sum())
        return tot
    sch = schur(p["pt_off"], p["pt_obs_off"], p["pt_obs_kf"], 216.0, 160.0) + schur(p["ln_off"], p["ln_obs_off"], p["ln_obs_kf"], 288.0, 250.0)
    return iters_total * lin + trials_total * (res + sch)


def run_reference_arm(args):
    """CPU oracle on the host cores (rank 0 only).  batched_local_ba: one window per worker thread (ctypes releases the
    GIL), all cores; global_ba: the reference's BundleAdjustment is single-threaded, one run per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    if args.workload == "global_ba":
        p = synth.make_global_ba(*GBA_SHAPE, synth.seed_for(5))
        steps = args.steps      # ~17 s per run on one core
        t0 = time.perf_counter()
        its = 0
        for _ in range(steps):
            o = api.ba_global(p, GBA_ITERS, impl="oracle")
            its += int(o["n_iter_done"][0, 0])
        dt = time.perf_counter() - t0
        val = its / dt
        line = {
            "impl": "reference", "metric": "global_ba_lm_iters_per_sec", "value": val, "unit": "LM iterations/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": 0, "ms_per_step": 1e3 * dt / steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"global_ba: {GBA_SHAPE[0]} KF / {GBA_SHAPE[1]} points / {GBA_SHAPE[2]} lines, {GBA_ITERS} LM iterations (BASELINE configs[4])",
                       "note": "CPU oracle (restatement of the reference g2o path); the reference BundleAdjustment is single-threaded"},
            "cpu_baseline": {"value": val, "unit": "LM iterations/s", "cores": 1, "kind": "port", "sample": f"{steps} full run(s)"},
            "e2e": {"value": val, "unit": "LM iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        print(json.dumps(line))
        return
    n_win = max(cores, 1)
    wins = [make_batch(1, synth.seed_for(4) + 1000 + i) for i in range(n_win)]
    api.ba_local(wins[0], ITS1, ITS2, impl="oracle")  # load + warm

    def one(p):
        o = api.ba_local(p, ITS1, ITS2, impl="oracle")
        return int(o["n_iter_done"].sum())

    with ThreadPoolExecutor(cores) as ex:
        for _ in range(args.warmup):
            list(ex.map(one, wins[:cores]))
        t0 = time.perf_counter()
        iters = 0
        for _ in range(args.steps):
            iters += sum(ex.map(one, wins))
        dt = time.perf_counter() - t0
    val = iters / dt
    line = {
        "impl": "reference", "metric": "local_ba_lm_iters_per_sec", "value": val, "unit": "LM iterations/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"batched_local_ba: windows of {WIN_KF} KF / {WIN_PT} points / {WIN_LN} lines, schedule {ITS1}+{ITS2}",
                   "note": "CPU oracle (restatement of the reference g2o path; the reference needs Eigen/OpenCV/LBDMOD, absent here)"},
        "cpu_baseline": {"value": val, "unit": "LM iterations/s", "cores": cores, "kind": "port",
                         "sample": f"{n_win} windows per step, one per host thread"},
        "e2e": {"value": val, "unit": "LM iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


class Ranks:
    """rank plumbing: barrier, max / sum over ranks (identity on one GPU)"""

    def __init__(self):
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.dist = None
        if self.world > 1:
            import torch
            import torch.distributed as dist
            torch.cuda.set_device(self.local_rank)
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
            self.dist = dist

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()

    def reduce(self, vals, op):
        if self.dist is None:
            return [float(x) for x in vals]
        import torch
        t = torch.tensor([float(x) for x in vals], device=f"cuda:{self.local_rank}", dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX if op == "max" else self.dist.ReduceOp.SUM)
        return [float(x) for x in t.cpu()]

    def share(self, n):
        """this rank's [a, b) of n units"""
        return (n * self.rank) // self.world, (n * (self.rank + 1)) // self.world

    def close(self):
        if self.dist is not None:
            self.dist.barrier()
            self.dist.destroy_process_group()


def timed_e2e(R, call, steps, count):
    """wall-clock over `steps` calls of the reference-shaped entry point (host buffers), max over ranks / sum of units"""
    for _ in range(2):
        call()
    R.barrier()
    t0 = time.perf_counter()
    units = 0
    for _ in range(steps):
        call()
        units += count()
    dt = time.perf_counter() - t0
    dt = R.reduce([dt], "max")[0]
    units = R.reduce([units], "sum")[0]
    return units / dt, 1e3 * dt / steps


def bench_global_ba(args, R, lib, d, ctx, hbm_peak, peak_src):
    """BASELINE configs[4]: strong scaling of one global BA; landmarks sharded, one packed all-reduce per LM trial."""
    world, rank = R.world, R.rank
    if world > 1:
        import torch
        idb = np.zeros(128, np.uint8)
        if rank == 0:
            assert lib.dll.lld_comm_unique_id(idb.ctypes.data_as(capi.c_u8p)) == 0
        t = torch.from_numpy(idb).cuda()
        R.dist.broadcast(t, 0)
        idb = t.cpu().numpy()
        ctx.check(lib.dll.lld_comm_init(ctx.handle, world, rank, idb.ctypes.data_as(capi.c_u8p)), "comm_init")
    p = synth.make_global_ba(*GBA_SHAPE, synth.seed_for(5))
    n_pe, n_le = edge_counts(p)
    prob, keep = capi.fill_struct(capi.BaProblem, p)
    log_stride = GBA_ITERS + 2
    out = api._ba_outputs(p, log_stride)
    res, keep2 = capi.fill_struct(capi.BaResult, out)
    d.lld_ba_upload_global.argtypes = [C.c_void_p, C.POINTER(capi.BaProblem), C.c_int]; d.lld_ba_upload_global.restype = C.c_int
    d.lld_ba_run_global.argtypes = [C.c_void_p, C.c_int, capi.c_u8p]; d.lld_ba_run_global.restype = C.c_int
    d.lld_ctx_nccl_stats.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]; d.lld_ctx_nccl_stats.restype = None
    ctx.check(d.lld_ba_upload_global(ctx.handle, C.byref(prob), log_stride), "upload_global")

    def step():
        ctx.check(d.lld_ba_run_global(ctx.handle, GBA_ITERS, None), "run_global")

    sampler = ClockSampler(R.local_rank)
    sampler.start()
    t_w, n_w = time.perf_counter(), 0
    while n_w < max(args.warmup, 3) or time.perf_counter() - t_w < 0.6:
        step()
        n_w += 1
    ctx.check(d.lld_ba_sync(ctx.handle), "sync")
    l0 = ctx.launch_count()
    R.barrier()
    ctx.check(d.lld_ba_sync(ctx.handle), "sync")
    d.lld_ctx_event_record(ctx.handle, 0)
    for _ in range(args.steps):
        step()
    d.lld_ctx_event_record(ctx.handle, 1)
    ctx.check(d.lld_ba_sync(ctx.handle), "sync")
    ms = float(d.lld_ctx_event_elapsed_ms(ctx.handle))
    clocks = sampler.stop()
    launches = ctx.launch_count() - l0
    nc, nb = C.c_int64(), C.c_int64()
    d.lld_ctx_nccl_stats(ctx.handle, C.byref(nc), C.byref(nb))
    if args.dump_outputs:
        ctx.check(d.lld_ba_download(ctx.handle, C.byref(prob), C.byref(res), 0), "download")
        dump_outputs(args.dump_outputs, out)
    # the landmark outputs of the other ranks are not needed for the metric: download this rank's view of the trace
    ms = R.reduce([ms], "max")[0]
    launches = int(R.reduce([launches], "sum")[0])
    # per-kernel profile of one run (rank 0's shard)
    d.lld_ctx_profile(ctx.handle, 1)
    step()
    prof = profile_report(d, ctx)
    d.lld_ctx_profile(ctx.handle, 0)
    # end to end: lld_ba_global with pinned host buffers (host indexing of the rank's shard, H2D, LM, D2H)
    pp, keep3 = pinned_problem(p)
    prob_h, keep4 = capi.fill_struct(capi.BaProblem, pp)
    outp, keep5 = pinned_problem(out)
    res_h, keep6 = capi.fill_struct(capi.BaResult, outp)
    lib.dll.lld_ctx_set_topo_cache(ctx.handle, 0)

    def call():
        ctx.check(lib.ba_global(ctx.handle, C.byref(prob_h), GBA_ITERS, None, C.byref(res_h)), "ba_global")
    e_val, e_ms = timed_e2e(R, call, max(2, min(args.steps, 5)), lambda: int(outp["n_iter_done"][0, 0]) if rank == 0 else 0)
    its = int(outp["n_iter_done"][0, 0]); trials = int(outp["trials_log"].sum())
    h2d, d2h = C.c_int64(), C.c_int64()
    d.lld_ctx_last_bytes(ctx.handle, C.byref(h2d), C.byref(d2h))
    lib.dll.lld_ctx_set_topo_cache(ctx.handle, -1)
    value = its * args.steps / (ms * 1e-3)
    tot_ms = sum(v["ms"] for v in prof.values())
    kernel_table = {k: {"ms": round(v["ms"], 4), "n": v["n"], "share": round(v["ms"] / tot_ms, 4)} for k, v in
                    sorted(prof.items(), key=lambda kv: -kv[1]["ms"])}
    # SURVEY §8(d): per iteration with t trials (1+t)(24 Ep + 36 El) + 2(1+t)(24 P + 40 L) + 8 nnz(Hschur)
    P, L = int(p["pt_off"][-1]), int(p["ln_off"][-1])
    step_bytes = (its + trials) * (24.0 * n_pe + 36.0 * n_le + 2 * (24.0 * P + 40.0 * L))
    roofline = {"bound": "hbm", "what": "whole run vs SURVEY §8(d) algorithmic bytes (edge stream + landmark state per pass)",
                "achieved": step_bytes / (ms * 1e-3 / args.steps) / 1e9, "peak": hbm_peak * world, "peak_source": peak_src, "unit": "GB/s",
                "traffic": None}
    roofline["frac"] = roofline["achieved"] / roofline["peak"]
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_extra:
        t0 = time.perf_counter()
        o = api.ba_global(p, GBA_ITERS, impl="oracle")
        tc = time.perf_counter() - t0
        cpu_baseline = {"value": int(o["n_iter_done"][0, 0]) / tc, "unit": "LM iterations/s", "cores": 1, "kind": "port",
                        "sample": "one full run of the same problem (the reference BundleAdjustment is single-threaded)"}
    line = {
        "metric": "global_ba_lm_iters_per_sec", "value": value, "unit": "LM iterations/s", "n_gpus": world,
        "steps": args.steps, "warmup": n_w, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"global_ba: {GBA_SHAPE[0]} KF / {GBA_SHAPE[1]} points / {GBA_SHAPE[2]} lines, {GBA_ITERS} LM iterations, bRobust=false "
                               "(BASELINE configs[4], strong scaling)",
                   "point_edges": n_pe, "line_edges": n_le, "iters_per_step": its, "lm_trials_per_step": trials,
                   "l2": "inputs larger than L2 (edge + landmark arrays > 150 MB per pass)",
                   "parallelism": f"landmarks block-sharded over {world} GPU(s); reduced camera system (block cyclic reduction) replicated; "
                                  "one packed ncclAllReduce of S + b_schur per LM trial"},
        "nccl": {"allreduce_calls_per_step": int(nc.value), "allreduce_bytes_per_step_per_rank": int(nb.value)},
        "e2e": {"value": e_val, "unit": "LM iterations/s", "h2d_bytes_per_step": int(h2d.value), "d2h_bytes_per_step": int(d2h.value),
                "ms_per_step": e_ms, "note": "lld_ba_global with pinned host buffers, topology cache off"},
        "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "kernels": kernel_table, "cpu_baseline": cpu_baseline,
    }
    if rank == 0:
        print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="batched_local_ba", choices=["batched_local_ba", "global_ba"])
    ap.add_argument("--windows", type=int, default=64, help="local-BA windows per GPU")
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary workloads and the CPU baselines")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the results of the last one (rank 0's batch) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or (args.workload == "global_ba" and int(os.environ.get("WORLD_SIZE", "1")) > 1)):
        ap.error("--dump-outputs needs --impl ours, and one GPU for --workload global_ba (its landmarks are sharded)")
    if args.impl == "reference":
        run_reference_arm(args)
        return

    R = Ranks()
    rank, world, local_rank = R.rank, R.world, R.local_rank
    hbm_peak, peak_src = load_peaks()
    lib = capi.load_library()
    d = bind_resident(lib)
    lib.dll.lld_ctx_set_topo_cache.argtypes = [C.c_void_p, C.c_int]; lib.dll.lld_ctx_set_topo_cache.restype = None
    ctx = capi.Context(local_rank)
    if args.workload == "global_ba":
        bench_global_ba(args, R, lib, d, ctx, hbm_peak, peak_src)
        R.close()
        ctx.close()
        return

    p = make_batch(args.windows, synth.seed_for(4) + rank)
    prob, keep = capi.fill_struct(capi.BaProblem, p)
    log_stride = ITS1 + ITS2 + 2
    out = api._ba_outputs(p, log_stride)
    res, keep2 = capi.fill_struct(capi.BaResult, out)
    barrier = R.barrier

    # ---------------- resident (value) ----------------
    ctx.check(d.lld_ba_upload(ctx.handle, C.byref(prob), 0, log_stride), "upload")

    def step():
        ctx.check(d.lld_ba_run_local(ctx.handle, ITS1, ITS2, None), "run_local")

    sampler = ClockSampler(local_rank)     # started before the warm-up: nvidia-smi needs ~0.2 s to produce its first line
    sampler.start()
    t_w = time.perf_counter()
    n_w = 0
    while n_w < max(args.warmup, 3) or time.perf_counter() - t_w < 0.6:   # same load as the timed region
        step()
        n_w += 1
        if n_w % 4 == 0:
            ctx.check(d.lld_ba_sync(ctx.handle), "sync")
    ctx.check(d.lld_ba_sync(ctx.handle), "sync")
    l0 = ctx.launch_count()
    barrier()
    ctx.check(d.lld_ba_sync(ctx.handle), "sync")
    d.lld_ctx_event_record(ctx.handle, 0)
    for _ in range(args.steps):
        step()
    d.lld_ctx_event_record(ctx.handle, 1)
    ctx.check(d.lld_ba_sync(ctx.handle), "sync")
    ms = float(d.lld_ctx_event_elapsed_ms(ctx.handle))
    clocks = sampler.stop()
    launches = ctx.launch_count() - l0
    ctx.check(d.lld_ba_download(ctx.handle, C.byref(prob), C.byref(res), 1), "download")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)
    iters_per_step = int(out["n_iter_done"].sum())
    trials_per_step = int(out["trials_log"].sum())
    ms = R.reduce([ms], "max")[0]
    iters_total, launches = R.reduce([iters_per_step, launches], "sum")
    launches = int(launches)
    value = iters_total * args.steps / (ms * 1e-3)

    # ---------------- per-kernel profile ----------------
    d.lld_ctx_profile(ctx.handle, 1)
    step()
    prof = profile_report(d, ctx)
    d.lld_ctx_profile(ctx.handle, 0)
    tot_ms = sum(v["ms"] for v in prof.values())
    top = max(prof.items(), key=lambda kv: kv[1]["ms"])
    top_name, top_ms, top_n = top[0], top[1]["ms"], top[1]["n"]
    key = top_name.strip("()")
    kb = kernel_bytes(key, p) or kernel_bytes(key.split("<")[0], p)
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r2_traffic.json")
    tinfo = json.load(open(tpath)) if os.path.exists(tpath) else {}
    if args.windows == 64:  # ncu dram bytes per launch of this exact workload (committed capture)
        traffic = tinfo.get("batched_local_ba_64", {}).get(top_name.strip("()"))
    roofline_kernel = {"bound": "hbm", "kernel": top_name, "share_of_step": top_ms / tot_ms if tot_ms else None,
                       "avg_launch_us": 1e3 * top_ms / max(top_n, 1), "peak": hbm_peak, "peak_source": peak_src, "unit": "GB/s",
                       "traffic": traffic, "traffic_source": tinfo.get("source") if traffic else None,
                       "note": "algorithmic bytes of OUR decomposition for this kernel (W blocks are its inputs), not of SURVEY §8(d)"}
    if kb:
        ach = kb / (1e-3 * top_ms / max(top_n, 1)) / 1e9
        roofline_kernel.update({"achieved": ach, "frac": ach / hbm_peak, "algorithmic_bytes_per_launch": kb})
    # headline roofline: the whole step against SURVEY §8(d) (minimal traffic of a perfectly fused implementation), HBM and FP64
    step_bytes = algorithmic_bytes_step(p, iters_per_step, trials_per_step)
    step_flops = algorithmic_flops_step(p, iters_per_step, trials_per_step)
    step_s = ms * 1e-3 / args.steps
    roofline = {"bound": "hbm", "what": "whole LM step sequence vs SURVEY §8(d) algorithmic bytes, summed over the executed iterations and trials "
                                        "(rank 0's batch); the path is FP64-issue / latency bound, see fp64",
                "achieved": step_bytes / step_s / 1e9, "peak": hbm_peak, "peak_source": peak_src, "unit": "GB/s",
                "traffic": tinfo.get("batched_local_ba_64_step_bytes") if args.windows == 64 else None,
                "traffic_note": "ncu dram bytes of all launches of one LM step with every window active" if tinfo else None,
                "fp64": {"achieved_tflops": step_flops / step_s / 1e12, "peak_tflops": FP64_PEAK_TFLOPS,
                         "frac": step_flops / step_s / 1e12 / FP64_PEAK_TFLOPS, "peak_source": "DFMA micro-benchmark on this part (tools/ubench)"}}
    roofline["frac"] = roofline["achieved"] / hbm_peak
    kernel_table = {k: {"ms": round(v["ms"], 4), "n": v["n"], "share": round(v["ms"] / tot_ms, 4)} for k, v in
                    sorted(prof.items(), key=lambda kv: -kv[1]["ms"])}

    # ---------------- end to end through the reference-shaped call, pinned host buffers ----------------
    pp, keep3 = pinned_problem(p)
    prob_h, keep4 = capi.fill_struct(capi.BaProblem, pp)
    outp, keep5 = pinned_problem(out)
    res_h, keep6 = capi.fill_struct(capi.BaResult, outp)

    def call():
        ctx.check(lib.ba_local(ctx.handle, C.byref(prob_h), ITS1, ITS2, None, C.byref(res_h)), "ba_local")
    h2d, d2h = C.c_int64(), C.c_int64()
    # headline: topology cache OFF — every call indexes its input from scratch, as a SLAM thread whose window changes with
    # every keyframe would see it
    lib.dll.lld_ctx_set_topo_cache(ctx.handle, 0)
    e_val, e_ms = timed_e2e(R, call, args.steps, lambda: int(outp["n_iter_done"].sum()))
    d.lld_ctx_last_bytes(ctx.handle, C.byref(h2d), C.byref(d2h))
    e2e = {"value": e_val, "unit": "LM iterations/s", "h2d_bytes_per_step": int(h2d.value), "d2h_bytes_per_step": int(d2h.value),
           "ms_per_step": e_ms, "note": "lld_ba_local, pinned host buffers, host indexing + H2D + LM + D2H per call (topology cache off)"}
    # the same call when the structure repeats (re-optimisation of an unchanged window): index tables stay on the device
    lib.dll.lld_ctx_set_topo_cache(ctx.handle, 1)
    w_val, w_ms = timed_e2e(R, call, args.steps, lambda: int(outp["n_iter_done"].sum()))
    d.lld_ctx_last_bytes(ctx.handle, C.byref(h2d), C.byref(d2h))
    e2e_same = {"value": w_val, "unit": "LM iterations/s", "h2d_bytes_per_step": int(h2d.value), "d2h_bytes_per_step": int(d2h.value),
                "ms_per_step": w_ms, "note": "same call, same structure as the previous call: topology cache hit, only values are uploaded"}
    lib.dll.lld_ctx_set_topo_cache(ctx.handle, -1)

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_extra:
        # ---------------- CPU baseline: oracle, one core, bounded sample ----------------
        sample = make_batch(1, synth.seed_for(4) + 999)
        t0 = time.perf_counter()
        api.ba_local(sample, ITS1, ITS2, impl="oracle")
        t1 = time.perf_counter() - t0
        n_s = int(max(2, min(16, 12.0 / max(t1, 1e-3))))
        sample = make_batch(n_s, synth.seed_for(4) + 998)
        t0 = time.perf_counter()
        o = api.ba_local(sample, ITS1, ITS2, impl="oracle")
        tc = time.perf_counter() - t0
        cpu_baseline = {"value": int(o["n_iter_done"].sum()) / tc, "unit": "LM iterations/s", "cores": 1, "kind": "port",
                        "sample": f"{n_s} windows of {WIN_KF}/{WIN_PT}/{WIN_LN}, schedule {ITS1}+{ITS2}, sequential on one core"}
    extra = {} if args.no_extra else run_extra(lib, d, ctx, hbm_peak, R)
    line = {
        "metric": "local_ba_lm_iters_per_sec", "value": value, "unit": "LM iterations/s", "n_gpus": world,
        "steps": args.steps, "warmup": n_w, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"batched_local_ba: {args.windows} windows/GPU of {WIN_KF} KF / {WIN_PT} points / {WIN_LN} lines, "
                               f"schedule {ITS1}+{ITS2} (BASELINE configs[3] shape, weak scaling)",
                   "windows_per_gpu": args.windows, "iters_per_step": iters_total, "lm_trials_per_step_rank0": trials_per_step,
                   "l2": "inputs larger than L2 (per-GPU working set > 500 MB)", "parallelism": f"windows sharded over {world} GPU(s), no collective"},
        "e2e": e2e, "e2e_same_structure": e2e_same, "gpu_launches": launches, "clocks": clocks, "roofline": roofline,
        "roofline_kernel": roofline_kernel, "kernels": kernel_table, "cpu_baseline": cpu_baseline, "extra": extra,
    }
    if rank == 0:
        print(json.dumps(line))
    R.close()
    ctx.close()


def run_extra(lib, d, ctx, hbm_peak, R):
    """secondary workloads of the BASELINE metric.  configs[1] (frame pairs) and configs[2] (frames) are sharded over the
    ranks with no collective (strong scaling of the BASELINE batch: 1024 pairs, 4096 frames); the single window is
    replicas-only and measured on one GPU."""
    ex = {}
    world, rank = R.world, R.rank
    one = world == 1

    def whole_job(ms_local, units_total):
        ms = R.reduce([ms_local], "max")[0]
        return units_total / (ms * 1e-3), ms

    # --- Hamming SearchByProjection, BASELINE configs[1]: 2k ORB / frame, batch of 1024 pairs
    try:
        PT, N = 1024, 2000
        a, b = R.share(PT)
        P = b - a
        m = synth.make_sbp_frame_batch(P, N, synth.seed_for(2) + 31 * rank)
        geom, gk = capi.make_geom(m["geom"])
        f = dict(m); f["geom"] = geom
        f.setdefault("th_high", 0); f.setdefault("allow_negative_depth", 0)
        prob, keep = capi.fill_struct(capi.SbpFrameProblem, f)
        ctx.check(d.lld_sbp_frame_upload(ctx.handle, C.byref(prob)), "sbp upload")
        passes = C.c_int()
        for _ in range(3):
            ctx.check(d.lld_sbp_run(ctx.handle, C.byref(passes)), "sbp run")
        d.lld_ba_sync(ctx.handle)
        R.barrier()
        d.lld_ctx_event_record(ctx.handle, 0)
        K = 20
        for _ in range(K):
            ctx.check(d.lld_sbp_run(ctx.handle, C.byref(passes)), "sbp run")
        d.lld_ctx_event_record(ctx.handle, 1)
        d.lld_ba_sync(ctx.handle)
        val, ms = whole_job(float(d.lld_ctx_event_elapsed_ms(ctx.handle)) / K, PT * N)
        alg = PT * (2 * N * 32 + 2 * N * 16 + N * 8)  # SURVEY §8(d): 208 KB / pair
        d.lld_ctx_profile(ctx.handle, 1)
        ctx.check(d.lld_sbp_run(ctx.handle, C.byref(passes)), "sbp run")
        prof = profile_report(d, ctx)
        d.lld_ctx_profile(ctx.handle, 0)
        # end to end: lld_sbp_frame with host buffers (H2D of the pair batch + matching + D2H of the match table)
        mp_, keepm = pinned_problem({k: v for k, v in m.items() if k != "geom"})
        mp_["geom"] = m["geom"]
        for _ in range(2):
            api.sbp_frame(mp_, impl="gpu", ctx=ctx)
        R.barrier()
        t0 = time.perf_counter()
        for _ in range(5):
            api.sbp_frame(mp_, impl="gpu", ctx=ctx)
        e_ms = R.reduce([1e3 * (time.perf_counter() - t0) / 5], "max")[0]
        ex["hamming_search_by_projection"] = {
            "metric": "descriptor_matches_per_sec", "value": val, "unit": "queries resolved/s", "n_gpus": world, "scaling": "strong",
            "config": f"{PT} frame pairs x {N} ORB keypoints (BASELINE configs[1]), th=7, {P} pairs on this rank, claim passes={passes.value}",
            "ms_per_batch": ms,
            "e2e": {"value": PT * N / (e_ms * 1e-3), "unit": "queries resolved/s", "ms_per_batch": e_ms,
                    "note": "lld_sbp_frame, pinned host buffers, H2D + match + D2H per call"},
            "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": hbm_peak * world, "unit": "GB/s",
                         "frac": alg / (ms * 1e-3) / 1e9 / (hbm_peak * world), "what": "whole matcher (grid build + all claim passes) vs 208 KB/pair"},
            "kernels": {k: {"ms": round(v["ms"], 4), "n": v["n"]} for k, v in prof.items()},
        }
        if one and rank == 0:
            ms_ = synth.make_sbp_frame_batch(32, N, synth.seed_for(2) + 1)
            t0 = time.perf_counter(); api.sbp_frame(ms_, impl="oracle"); tc = time.perf_counter() - t0
            ex["hamming_search_by_projection"]["cpu_baseline"] = {"value": 32 * N / tc, "unit": "queries resolved/s", "cores": 1, "kind": "port", "sample": "32 pairs"}
    except Exception as e:  # noqa: BLE001
        ex["hamming_search_by_projection"] = {"error": str(e)}
    # --- stereo line matching with float descriptors, BASELINE configs[1]: 500 lines / frame, D = 64, batch of 1024 pairs
    try:
        PT, N, D = 1024, 500, 64
        a, b = R.share(PT)
        P = b - a
        lm = synth.make_line_match_batch(P, N, D, synth.seed_for(2) + 7 + 31 * rank)
        for _ in range(2):
            api.line_match(lm, impl="gpu", ctx=ctx)
        comp, wall = [], []
        R.barrier()
        for _ in range(5):
            t0 = time.perf_counter()
            api.line_match(lm, impl="gpu", ctx=ctx)
            wall.append(1e3 * (time.perf_counter() - t0))
            comp.append(ctx.last_timing()[1])
        val, ms = whole_job(float(np.median(comp)), PT * N)
        e_ms = R.reduce([float(np.median(wall))], "max")[0]
        d.lld_ctx_profile(ctx.handle, 1)
        api.line_match(lm, impl="gpu", ctx=ctx)
        prof = profile_report(d, ctx)
        d.lld_ctx_profile(ctx.handle, 0)
        alg = PT * (2 * N * D * 4 + N * 8)          # SURVEY §8(d): 260 KB / pair at D = 64
        flops = PT * 2.0 * N * N * D                # dense contraction
        ex["line_descriptor_matching"] = {
            "metric": "descriptor_matches_per_sec", "value": val, "unit": "left lines resolved/s", "n_gpus": world, "scaling": "strong",
            "config": f"{PT} stereo pairs x {N} x {N} lines, D={D} float descriptors (BASELINE configs[1]), CheckLinePair gates + greedy assignment",
            "ms_per_batch": ms, "note": "device time between the library's own CUDA events on its stream (compute only)",
            "e2e": {"value": PT * N / (e_ms * 1e-3), "unit": "left lines resolved/s", "ms_per_batch": e_ms,
                    "note": "lld_line_match wall clock, host buffers in, matches out"},
            "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": hbm_peak * world, "unit": "GB/s",
                         "frac": alg / (ms * 1e-3) / 1e9 / (hbm_peak * world), "what": "whole matcher vs 260 KB/pair"},
            "contraction_tflops": flops / (ms * 1e-3) / 1e12,
            "kernels": {k: {"ms": round(v["ms"], 4), "n": v["n"]} for k, v in prof.items()},
        }
        if one and rank == 0:
            lms = synth.make_line_match_batch(8, N, D, synth.seed_for(2) + 8)
            t0 = time.perf_counter(); api.line_match(lms, impl="oracle"); tc = time.perf_counter() - t0
            ex["line_descriptor_matching"]["cpu_baseline"] = {"value": 8 * N / tc, "unit": "left lines resolved/s", "cores": 1, "kind": "port", "sample": "8 pairs"}
    except Exception as e:  # noqa: BLE001
        ex["line_descriptor_matching"] = {"error": str(e)}
    # --- pose-only LM, BASELINE configs[2]: 4096 frames x (1.5k points + 300 lines), 4 x 10 schedule
    try:
        FT = 4096
        a, b = R.share(FT)
        F = b - a
        pz = synth.make_pose_batch(F, 1500, 300, synth.seed_for(3) + 31 * rank)
        prob, keep = capi.fill_struct(capi.PoseProblem, pz)
        ctx.check(d.lld_pose_upload(ctx.handle, C.byref(prob)), "pose upload")
        for _ in range(2):
            ctx.check(d.lld_pose_run(ctx.handle), "pose run")
        d.lld_ba_sync(ctx.handle)
        R.barrier()
        d.lld_ctx_event_record(ctx.handle, 0)
        K = 3
        for _ in range(K):
            ctx.check(d.lld_pose_run(ctx.handle), "pose run")
        d.lld_ctx_event_record(ctx.handle, 1)
        d.lld_ba_sync(ctx.handle)
        val, ms = whole_job(float(d.lld_ctx_event_elapsed_ms(ctx.handle)) / K, FT)
        ex["pose_optimization"] = {"metric": "frames_per_sec", "value": val, "unit": "frames/s", "n_gpus": world, "scaling": "strong",
                                   "config": f"{FT} frames x (1500 points + 300 lines), 4x10 LM (BASELINE configs[2]), {F} frames on this rank",
                                   "ms_per_batch": ms}
        if one and rank == 0:
            ps = synth.make_pose_batch(16, 1500, 300, synth.seed_for(3) + 1)
            t0 = time.perf_counter(); api.pose_opt(ps, impl="oracle"); tc = time.perf_counter() - t0
            ex["pose_optimization"]["cpu_baseline"] = {"value": 16 / tc, "unit": "frames/s", "cores": 1, "kind": "port", "sample": "16 frames"}
    except Exception as e:  # noqa: BLE001
        ex["pose_optimization"] = {"error": str(e)}
    if not one or rank != 0:
        return ex
    # --- single local-BA window at the north_star target shape 10 KF / 5k points / 1k lines (replicas only: one GPU)
    try:
        p1 = synth.make_local_ba_batch(1, 10, 5000, 1000, synth.seed_for(1) + 5)
        prob, keep = capi.fill_struct(capi.BaProblem, p1)
        out = api._ba_outputs(p1, ITS1 + ITS2 + 2)
        res, keep2 = capi.fill_struct(capi.BaResult, out)
        ctx.check(d.lld_ba_upload(ctx.handle, C.byref(prob), 0, ITS1 + ITS2 + 2), "upload")
        for _ in range(3):
            ctx.check(d.lld_ba_run_local(ctx.handle, ITS1, ITS2, None), "run")
        d.lld_ba_sync(ctx.handle)
        d.lld_ctx_event_record(ctx.handle, 0)
        K = 10
        for _ in range(K):
            ctx.check(d.lld_ba_run_local(ctx.handle, ITS1, ITS2, None), "run")
        d.lld_ctx_event_record(ctx.handle, 1)
        d.lld_ba_sync(ctx.handle)
        ms = float(d.lld_ctx_event_elapsed_ms(ctx.handle)) / K
        ctx.check(d.lld_ba_download(ctx.handle, C.byref(prob), C.byref(res), 1), "download")
        its = int(out["n_iter_done"].sum())
        d.lld_ctx_profile(ctx.handle, 1)
        ctx.check(d.lld_ba_run_local(ctx.handle, ITS1, ITS2, None), "run")
        prof1 = profile_report(d, ctx)
        d.lld_ctx_profile(ctx.handle, 0)
        # the call a SLAM thread makes: lld_ba_local with host buffers, one window (topology cache off: a new window every call)
        pp1, k1 = pinned_problem(p1)
        prob1, k2 = capi.fill_struct(capi.BaProblem, pp1)
        out1, k3 = pinned_problem(out)
        res1, k4 = capi.fill_struct(capi.BaResult, out1)
        lib.dll.lld_ctx_set_topo_cache(ctx.handle, 0)
        for _ in range(3):
            ctx.check(lib.ba_local(ctx.handle, C.byref(prob1), ITS1, ITS2, None, C.byref(res1)), "ba_local")
        t0 = time.perf_counter()
        for _ in range(K):
            ctx.check(lib.ba_local(ctx.handle, C.byref(prob1), ITS1, ITS2, None, C.byref(res1)), "ba_local")
        e_ms = 1e3 * (time.perf_counter() - t0) / K
        lib.dll.lld_ctx_set_topo_cache(ctx.handle, -1)
        t0 = time.perf_counter(); o = api.ba_local(p1, ITS1, ITS2, impl="oracle"); tc = time.perf_counter() - t0
        cpu = int(o["n_iter_done"].sum()) / tc
        ex["single_window_local_ba"] = {"metric": "lm_iters_per_sec", "value": its / (ms * 1e-3), "unit": "LM iterations/s",
                                        "config": "1 window 10 KF / 5000 points / 1000 lines, schedule 5+15 (latency bound; north_star target shape)",
                                        "ms_per_call": ms, "iters": its,
                                        "e2e": {"value": its / (e_ms * 1e-3), "unit": "LM iterations/s", "ms_per_call": e_ms,
                                                "note": "lld_ba_local with pinned host buffers: host indexing + H2D + 5+15 LM + D2H, topology cache off"},
                                        "cpu_baseline": {"value": cpu, "unit": "LM iterations/s", "cores": 1, "kind": "port", "sample": "the same window"}}
        ex["single_window_local_ba"]["kernels_us_per_launch"] = {k: round(1e3 * v["ms"] / max(v["n"], 1), 2) for k, v in
                                                                 sorted(prof1.items(), key=lambda kv: -kv[1]["ms"])}
        ex["single_window_local_ba"]["speedup_vs_cpu_1core"] = ex["single_window_local_ba"]["value"] / cpu
        ex["single_window_local_ba"]["e2e_speedup_vs_cpu_1core"] = ex["single_window_local_ba"]["e2e"]["value"] / cpu
    except Exception as e:  # noqa: BLE001
        ex["single_window_local_ba"] = {"error": str(e)}
    return ex


if __name__ == "__main__":
    main()
