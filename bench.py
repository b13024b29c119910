#!/usr/bin/env python
"""bench.py — frames/s through detect -> match -> local BA at 1920x1080 mono (BASELINE.json metric), one JSON line.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A step is one frame through the whole hot path: ORB extract (2000 kp) of a NEW 1080p frame, 256-bit Hamming match against the
previous frame's descriptors, and one local bundle adjustment (50 keyframes / 2000 landmarks / 10 000 observations, 10 LM
iterations, 50-iteration block-Jacobi PCG cap).

  value        every input already resident in HBM (a ring of frames larger than L2), device time (CUDA events), the two stages
               of a SLAM front/back end PIPELINED on one GPU exactly as their data dependencies allow: the tracking ctx
               (extract + match) and the mapping ctx (local BA) are two streams; BA(k) waits for match(k), extract(k+1) does not
               wait for BA(k).  `serial` holds the same K steps on ONE stream (round 1's definition).
  e2e          the same pipeline through the C-ABI host-buffer entry points from two host threads (tracking / mapping) with
               PAGEABLE host frames (GImage memory is malloc'd, GImage.h:394-402): H2D + D2H inside the timed region.
  roofline     the BA Jacobian sweep at config-5 size (the BASELINE metric's second clause), outside the timed step.
  global_ba    BASELINE config 5 (500 cams / 100k landmarks / 1M obs), landmark-sharded over the N ranks with one NCCL
               all-reduce of the compact reduced camera system per LM iteration -- STRONG scaling (total work fixed).
N>1 for the per-frame path: independent replicas, one rank per GPU, no data-path collective -> weak scaling.

The timed block is exactly K steps (bracketed by barrier + synchronize, max over ranks); the clock sampler starts before the warm-up.
The default 1000 steps time about a second (1.08 ms per step on a B200 at a 1000 W power limit): a much shorter window would show
clock ramp and scheduler noise in the one number reported.

--dump-outputs DIR writes what the pipelined timed path computed in its last step, as a caller of that path receives it, to DIR/<name>.npy
(float32 / float64): the keypoints and descriptors of the last frame, its matches against the previous frame and the local BA window's
poses, points and costs.  The inputs depend only on the arguments, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import queue
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H, NKP = 1920, 1080, 2000
BA_CAMS, BA_PTS, BA_OBS_PER_PT, BA_ITERS, PCG_ITERS = 50, 2000, 5, 10, 50
RING = 72  # frames resident in HBM: 72 * 2.07 MB = 149 MB > 126 MB L2
GBA_CAMS, GBA_PTS, GBA_OBS_PER_PT, GBA_ITERS, GBA_PCG = 500, 100000, 10, 5, 30
METRIC = "frames/sec detect+match+local-BA @1920x1080 mono"


def level_sizes(w, h, nlevels=8, sf=1.2):
    out = []
    for l in range(nlevels):
        inv = np.float32(1.0) / np.float32(np.float64(np.float32(sf)) ** l)  # cv2: cols * (1/scale) in float, half-even
        out.append((int(np.rint(np.float32(w) * inv)), int(np.rint(np.float32(h) * inv))))
    return out


def algorithmic_bytes():
    """SURVEY.md §8d per-unit figures."""
    lv = level_sizes(W, H)
    p0 = lv[0][0] * lv[0][1]
    prest = sum(a * b for a, b in lv[1:])
    b_ext = p0 + 2 * prest + NKP * (43 * 43 + 60) + 2 * NKP * 81
    b_match = 32 * (NKP + NKP) + 12 * NKP
    n_obs = BA_PTS * BA_OBS_PER_PT
    b_ba = 168 * n_obs + 96 * BA_PTS + 272 * BA_CAMS
    return dict(extract=b_ext, match=b_match, ba_sweep=b_ba)


def workload_config(world):
    """The `config` object: identical keys in both arms (the driver compares them)."""
    return {"workload": (f"{W}x{H} mono, {NKP} kp ORB extract + {NKP}x{NKP} Hamming match + local BA "
                         f"({BA_CAMS} KF/{BA_PTS} pts/{BA_PTS * BA_OBS_PER_PT} obs, {BA_ITERS} LM it, PCG cap {PCG_ITERS})"),
            "l2": f"input ring of {RING} frames ({RING * W * H / 1e6:.0f} MB) > 126 MB L2",
            "parallelism": f"replicas x{world}; tracking (extract+match) and mapping (local BA) pipelined"}


class ClockSampler(threading.Thread):
    def __init__(self, gpu_index: int):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples = []
        self.stop_flag = False
        self.proc = None
        self.t_mark = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.samples.append((time.perf_counter(), [x.strip() for x in line.split(",")]))
        except Exception:
            pass

    def mark(self):
        """Samples from here on belong to the timed region."""
        self.t_mark = time.perf_counter()

    def finish(self):
        self.stop_flag = True
        if self.proc:
            try:
                self.proc.terminate()
            except Exception:
                pass
        sm, mx, reasons = [], 0, set()
        for t, s in self.samples:
            if self.t_mark is not None and t < self.t_mark:
                continue
            try:
                sm.append(float(s[0])); mx = max(mx, float(s[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm), "samples_total": len(self.samples)}


# ---------------------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's CPU path, organised the way a CPU SLAM runs it -- a tracking thread (OpenCV ORB + BFMatcher, all
# cores inside OpenCV) and a mapping thread (local BA) working concurrently, frame k+1's tracking overlapping window k's BA.
# ---------------------------------------------------------------------------------------------------------------------------
def cpu_path(frames, ba_problem, steps, threads):
    import oracle
    try:
        import cv2
        cv2.setNumThreads(threads)
        orb = cv2.ORB_create(nfeatures=NKP)
        bf = cv2.BFMatcher(cv2.NORM_HAMMING)

        def extract(img):
            return orb.detectAndCompute(img, None)[1]

        def match(a, b):
            return bf.match(a, b)
        what = f"cv2 {cv2.__version__} ORB+BFMatcher ({threads} threads)"
    except Exception:
        def extract(img):
            return oracle.orb_extract(img, NKP)[1]

        def match(a, b):
            return oracle.match_hamming(a, b)
        what = "oracle orb_ref+hamming_ref (1 thread)"
    ba_threads = max(1, min(16, threads // 4))  # the BA port's OpenMP loops (linearisation, Schur complement, dense mat-vec)
    oracle.ba_set_threads(ba_threads)
    what += f" on the tracking thread || oracle ba_ref ({ba_threads} OpenMP threads) on the mapping thread"
    prev = extract(frames[0])
    q: queue.Queue = queue.Queue(maxsize=2)

    def mapper():
        while True:
            k = q.get()
            if k is None:
                return
            pb = ba_problem.copy()
            oracle.ba_solve(pb, max_iterations=BA_ITERS, function_tolerance=0.0, pcg_max_iters=PCG_ITERS, pcg_tol=1e-10)

    th = threading.Thread(target=mapper, daemon=True)
    t0 = time.perf_counter()
    th.start()
    for k in range(steps):
        d = extract(frames[(k + 1) % len(frames)])
        match(d, prev)
        prev = d
        q.put(k)
    q.put(None)
    th.join()
    dt = time.perf_counter() - t0
    oracle.ba_set_threads(1)
    return steps / dt, what


def dump_outputs(out_dir, feats, graph, res):
    """The last timed step's results, as Features.download / Features.matches / BAGraph.download and the BaResult give them."""
    from gslam_b200.capi import KP_DTYPE
    kps, desc = feats.download()
    idx, d1, d2 = feats.matches()
    poses, points = graph.download()
    out = {"keypoints": np.stack([kps[f].astype(np.float32) for f in KP_DTYPE.names], axis=1),   # x y size angle response octave class_id
           "descriptors": desc.astype(np.float32), "match_train_index": idx.astype(np.float32), "match_distance": d1.astype(np.float32),
           "match_second_distance": d2.astype(np.float32), "ba_poses_wc": poses, "ba_points": points,
           "ba_cost": np.array([res.initial_cost, res.final_cost], np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def median(xs):
    return float(np.median(np.asarray(xs, dtype=np.float64)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--no-global-ba", action="store_true", help="skip the config-5 global BA section")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    from gslam_b200 import synth
    ba_problem = synth.synth_ba(BA_CAMS, BA_PTS, BA_OBS_PER_PT, seed=42, n_fixed=2)
    cores = os.cpu_count() or 1

    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the outputs of the GPU path; the reference arm has none to write")
    if args.impl == "reference":
        if rank != 0:
            return
        steps = max(1, min(args.steps, 20))
        warm = max(1, min(args.warmup, 3))
        frames = synth.synth_stream(W, H, 4, seed=7)
        cpu_path(frames, ba_problem, warm, cores)
        fps, what = cpu_path(frames, ba_problem, steps, cores)
        line = {"impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s",
                "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": 1e3 / fps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8+f64", "data": "synthetic",
                "config": workload_config(world),
                "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                                 "sample": f"{steps} frames after {warm} warm-up (bounded sample of the --steps/--warmup asked): {what}"},
                "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from gslam_b200.api import BAGraph, Context, Features, OptimzeConfig
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()  # before the warm-up: nvidia-smi needs a few hundred ms to deliver its first sample
    ctx = Context(local)    # tracking: extract + match
    ctx_m = Context(local, high_priority=True)  # mapping: local BA (its few-CTA kernels go ahead of the tracking grids)
    cfg = ctx.orb_cfg(nfeatures=NKP)
    ba_cfg = OptimzeConfig(maxIterations=BA_ITERS, functionTolerance=0.0, pcgMaxIterations=PCG_ITERS, pcgTolerance=1e-10)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world > 1:
            t = torch.tensor([x], device="cuda", dtype=torch.float64); dist.all_reduce(t, op=dist.ReduceOp.MAX); return float(t.item())
        return x

    # ---- device-resident inputs: a ring of distinct frames larger than L2 ----------------------------------------------
    base = synth.synth_stream(W, H, 8, seed=7 + rank)
    ring = torch.empty((RING, H, W), dtype=torch.uint8, device="cuda")
    for k in range(RING):  # distinct content per slot: shifted copies of 8 generated frames (cheap, still cold in L2)
        ring[k] = torch.from_numpy(np.roll(base[k % 8], shift=(k // 8) * 7, axis=1)).cuda()
    feats = [Features(ctx, 2 * NKP + 256), Features(ctx, 2 * NKP + 256)]
    graph_s = BAGraph(ctx, ba_problem)    # serial mode: BA on the tracking stream
    graph_p = BAGraph(ctx_m, ba_problem)  # pipelined mode: BA on the mapping stream
    torch.cuda.synchronize()

    def track(k):
        f, fp = feats[k & 1], feats[(k + 1) & 1]
        f.extract(ring[k % RING].data_ptr(), W, H, cfg, device_ptr=True, pitch=W)
        f.match(fp)

    def step_serial(k):
        track(k)
        graph_s.reset()
        graph_s.solve(ba_cfg)

    def run_serial(k0, n):
        for k in range(k0, k0 + n):
            step_serial(k)

    res_last = [None]

    def run_pipelined(k0, n):
        """n frames from two host threads, like a SLAM's tracking and mapping threads: the tracking thread enqueues extract(k) +
        match(k) (no host synchronisation: the matcher reads the keypoint counts on the device) and orders the mapping stream
        after match(k); the mapping thread runs BA(k) (one host synchronisation per window: the LM scalars come back with it)."""
        qq: queue.Queue = queue.Queue(maxsize=2)
        err = []

        def mapper():
            try:
                while True:
                    k = qq.get()
                    if k is None:
                        return
                    graph_p.reset()
                    res_last[0] = graph_p.solve(ba_cfg)
            except Exception as e:
                err.append(e)
        th = threading.Thread(target=mapper, daemon=True)
        th.start()
        for k in range(k0, k0 + n):
            track(k)
            ctx_m.wait_for(ctx)          # BA(k) after match(k); extract(k+1) does not wait for BA(k)
            qq.put(k)
        qq.put(None)
        th.join()
        if err:
            raise err[0]
        ctx.wait_for(ctx_m)              # the timing events live on the tracking stream

    def timed_block(run, steps):
        """[barrier, K steps, barrier] -> ms (max over ranks) and the launch count of the block."""
        barrier()
        l0 = ctx.launch_count() + ctx_m.launch_count()
        ctx.timer_begin()
        run(args.warmup, steps)
        ms = ctx.timer_end()
        torch.cuda.synchronize()
        return max_over_ranks(ms), ctx.launch_count() + ctx_m.launch_count() - l0

    feats[1].extract(ring[RING - 1].data_ptr(), W, H, cfg, device_ptr=True, pitch=W)
    run_serial(0, max(3, args.warmup))
    run_pipelined(0, max(3, args.warmup))
    ctx.sync(); ctx_m.sync()
    if sampler:
        sampler.mark()
    ms_serial, ser_launches = timed_block(run_serial, args.steps)
    ms_pipe, pip_launches = timed_block(run_pipelined, args.steps)
    clocks = sampler.finish() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, feats[(args.warmup + args.steps - 1) & 1], graph_p, res_last[0])

    # ---- per-stage device timing (CUDA events on the ctx stream) ------------------------------------------------------------
    def time_stage(fn, reps, c=ctx):
        fn(); c.sync()
        c.timer_begin()
        for r in range(reps):
            fn(r)
        return c.timer_end() / reps
    reps = 50
    t_ext = time_stage(lambda r=0: feats[0].extract(ring[(r * 7 + 3) % RING].data_ptr(), W, H, cfg, device_ptr=True, pitch=W), reps)
    t_match = time_stage(lambda r=0: feats[0].match(feats[1]), reps)

    def ba_once(r=0):
        graph_s.reset(); graph_s.solve(ba_cfg)
    t_ba = time_stage(ba_once, 10)
    # the same window with the DIRECT linear solver (block-skyline Cholesky in one CTA instead of 50 PCG iterations): reported for
    # comparison; the timed step keeps the PCG configuration BASELINE.json's workload names
    ba_cfg_direct = OptimzeConfig(maxIterations=BA_ITERS, functionTolerance=0.0, linearSolver=1)
    res_direct = [None]

    def ba_direct(r=0):
        graph_s.reset(); res_direct[0] = graph_s.solve(ba_cfg_direct)
    t_ba_direct = time_stage(ba_direct, 10)
    graph_s.reset(); res_pcg = graph_s.solve(ba_cfg)
    t_sweep_local = time_stage(lambda r=0: graph_s.sweep(0.01), 50)
    popc_peak = ctx.popc_peak() if rank == 0 else None
    # the BASELINE metric's second clause, "BA Jacobian-eval HBM GB/s": the fused residual+Jacobian sweep (K6a+K6b) on the
    # config-5-shaped graph (500 cams / 100k landmarks / 1M observations: 177.7 MB algorithmic per sweep > L2, so every
    # repetition is cold).  Rank 0 only.  NOT part of the timed step.
    gba_problem = None
    if rank == 0 or not args.no_global_ba:
        gba_problem = synth.synth_ba(GBA_CAMS, GBA_PTS, GBA_OBS_PER_PT, seed=42, n_fixed=2)
    t_sweep_big, big_bytes = None, None
    if rank == 0:
        gbig = BAGraph(ctx, gba_problem)
        t_sweep_big = time_stage(lambda r=0: gbig.sweep(0.01), 20)
        big_bytes = 168 * gba_problem.n_obs + 96 * gba_problem.n_points + 272 * gba_problem.n_cams
        gbig.close()

    # ---- global BA, config 5, landmark-sharded over the ranks (strong scaling) ---------------------------------------------------
    global_ba = None
    if not args.no_global_ba:
        from gslam_b200.dist import DistributedBA
        gcfg = OptimzeConfig(maxIterations=GBA_ITERS, functionTolerance=0.0, pcgMaxIterations=GBA_PCG)
        t_setup = time.perf_counter()
        dba = DistributedBA(ctx, gba_problem, rank, world)
        t_setup = time.perf_counter() - t_setup
        times, res = [], None
        for rep in range(4):  # rep 0 warms up (NCCL channels, first launches)
            dba.graph.reset()
            barrier()
            ctx.timer_begin()
            res = dba.solve(gcfg)
            ms = max_over_ranks(ctx.timer_end())
            if rep > 0:
                times.append(ms)
        global_ba = {"workload": f"{GBA_CAMS} cams / {GBA_PTS} landmarks / {gba_problem.n_obs} obs, {GBA_ITERS} LM it, PCG cap {GBA_PCG}",
                     "nranks": world, "ms_per_lm_iteration": median(times) / GBA_ITERS, "ms_total": median(times),
                     "allreduce_bytes": dba.reduce_bytes + 8, "cost": res.final_cost, "initial_cost": res.initial_cost,
                     "accepted": res.accepted, "pcg_iterations": res.pcg_iterations, "scaling": "strong",
                     "host_setup_ms": t_setup * 1e3,
                     "collective": "NCCL all-reduce (f64 sum) of the compact block-CSR reduced camera system, under the C-ABI"}
        dba.close()
        if world > 1 and rank == 0:  # the same solve on rank 0's GPU alone: the strong-scaling denominator + the parity of the sharding
            d1 = DistributedBA(ctx, gba_problem, 0, 1)
            t1 = []
            for rep in range(3):
                d1.graph.reset(); ctx.sync()
                ctx.timer_begin(); r1 = d1.solve(gcfg); t1.append(ctx.timer_end())
            d1.close()
            rel = abs(res.final_cost - r1.final_cost) / abs(r1.final_cost)
            global_ba.update({"ms_per_lm_iteration_n1": median(t1[1:]) / GBA_ITERS, "cost_n1": r1.final_cost, "cost_rel_diff_vs_n1": rel,
                              "cost_agrees_1e-12": bool(rel < 1e-12)})
        if world > 1:
            dist.barrier()
    del gba_problem

    # ---- BASELINE config 4: EuRoC-shaped stereo 752x480, 2000 kp per eye, stereo match + temporal match + PnP-RANSAC + local BA;
    #      frames shard over the ranks (independent replicas, no collective).  Device-resident frames; the PnP call is the host-buffer
    #      C-ABI entry point (its 80 KB of 3D-2D matches travel inside the timed region).
    SW, SH = 752, 480
    sbase = synth.synth_stream(SW, SH, 8, seed=21 + rank)
    sring = torch.empty((16, 2, SH, SW), dtype=torch.uint8, device="cuda")
    for k in range(16):
        left = np.roll(sbase[k % 8], shift=(k // 8) * 5, axis=1)
        sring[k, 0] = torch.from_numpy(left).cuda(); sring[k, 1] = torch.from_numpy(np.roll(left, -14, axis=1)).cuda()
    fl = [Features(ctx, 2 * NKP + 256), Features(ctx, 2 * NKP + 256)]
    fr_ = Features(ctx, 2 * NKP + 256)
    rng4 = np.random.default_rng(4)
    n4 = 2000   # 3D-2D matches of the tracking step: 30 % outliers, 1 px noise at f = 458 (EuRoC)
    Xc = np.column_stack([rng4.uniform(-4, 4, n4), rng4.uniform(-3, 3, n4), rng4.uniform(3, 20, n4)])
    xy4 = Xc[:, :2] / Xc[:, 2:3] + rng4.normal(0, 1 / 458.0, (n4, 2))
    bad4 = rng4.permutation(n4)[:600]
    xy4[bad4] = np.column_stack([rng4.uniform(-0.8, 0.8, 600), rng4.uniform(-0.5, 0.5, 600)])
    Xw4 = np.ascontiguousarray(Xc + np.array([0.3, -0.1, 0.2])); xy4 = np.ascontiguousarray(xy4)
    pnp_inliers = [0]

    def step_config4(k):
        a, b = fl[k & 1], fl[(k + 1) & 1]
        a.extract(sring[k % 16, 0].data_ptr(), SW, SH, cfg, device_ptr=True, pitch=SW)
        fr_.extract(sring[k % 16, 1].data_ptr(), SW, SH, cfg, device_ptr=True, pitch=SW)
        a.match_stereo(fr_, 2.0, 0.0, 96.0)
        a.match(b)
        pose, mask, st = ctx.pnp_ransac(Xw4, xy4, threshold=4 / 458.0, confidence=0.99, max_hypotheses=512, seed=k + 1)
        pnp_inliers[0] = int(st.inliers_refined)
        graph_s.reset()
        graph_s.solve(ba_cfg)
    fl[1].extract(sring[15, 0].data_ptr(), SW, SH, cfg, device_ptr=True, pitch=SW)
    for k in range(3):
        step_config4(k)
    c4_steps = max(10, min(args.steps, 50))
    c4_ms = []
    for rep in range(3):
        barrier()
        ctx.timer_begin()
        for k in range(c4_steps):
            step_config4(3 + k)
        c4_ms.append(max_over_ranks(ctx.timer_end()))
    config4 = {"workload": f"stereo {SW}x{SH}, {NKP} kp per eye: 2 x ORB extract + row-band stereo match + temporal match + PnP-RANSAC ({n4} matches, 30 % outliers, "
                           f"<= 512 hypotheses) + local BA ({BA_CAMS} KF/{BA_PTS} pts/{BA_PTS * BA_OBS_PER_PT} obs, {BA_ITERS} LM it)",
               "value": world * c4_steps / (median(c4_ms) * 1e-3), "unit": "frames/s", "ms_per_step": median(c4_ms) / c4_steps, "steps": c4_steps,
               "scaling": "weak (frames shard over the ranks, no collective)", "n_gpus": world, "pnp_inliers": pnp_inliers[0],
               "note": "single stream per rank; device-resident stereo pairs; BASELINE.json configs[3]"}

    # ---- bag-of-words transform (SURVEY.md section 8f-4; published CPU figure 615.5 us, doc/doxygen/4_2_tools.dox:43 "Trans ORB-4"):
    #      GSLAM::Vocabulary::transform(features, BowVector&, FeatureVector&, levelsup) of the frame's 2000 descriptors on a k = 10,
    #      L = 5 vocabulary (111 111 nodes, 3.6 MB of node descriptors), through the host-buffer C-ABI (descriptors in, maps out) and
    #      chained on the device after the extraction.  Rank 0 only.
    bow = None
    if rank == 0:
        from gslam_b200.api import Vocabulary
        vt = synth.synth_vocabulary(10, 5, seed=1)
        dv = Vocabulary(ctx, vt.k, vt.L, vt.weighting, vt.scoring, vt.child_num, vt.weight, vt.desc)
        rngb = np.random.default_rng(0)
        fb = np.ascontiguousarray(vt.desc[rngb.integers(1, vt.n_nodes, NKP)] ^ np.packbits(rngb.random((NKP, 256)) < 0.05, axis=1))
        for _ in range(5):
            dv.transform(fb, 2)
        t0 = time.perf_counter()
        for _ in range(200):
            out_b = dv.transform(fb, 2)
        bow_host_us = (time.perf_counter() - t0) / 200 * 1e6
        fcur = feats[0]
        fcur.extract(ring[0].data_ptr(), W, H, cfg, device_ptr=True, pitch=W)
        for _ in range(3):
            dv.transform(fcur, 2)
        t0 = time.perf_counter()
        for _ in range(100):
            dv.transform(fcur, 2)
        bow_dev_us = (time.perf_counter() - t0) / 100 * 1e6
        bow = {"workload": f"{NKP} ORB descriptors -> BowVector + FeatureVector (levelsup 2), vocabulary k=10 L=5 ({vt.n_nodes} nodes), TF_IDF / L1",
               "us_per_transform_host_buffers": bow_host_us, "us_per_transform_device_resident_descriptors": bow_dev_us,
               "words": int(out_b["words"].shape[0]), "published_cpu_us": 615.5,
               "note": "wall clock of the Python call around gb_bow_transform (ctypes + numpy allocation of the outputs included); "
                       "outputs are the reference's std::map contents in map order"}
        try:
            import oracle
            from oracle import oracle as O
            va = O.VocabularyArrays(vt.k, vt.L, vt.weighting, vt.scoring, vt.child_num, vt.weight, vt.desc)
            if oracle.have_ref():
                R = O.RefVocabulary.from_arrays(va)
                bow["cpu_reference_us"] = R.transform(fb, 2, repeat=20)["seconds"] * 1e6
                bow["cpu_reference_kind"] = "reference (GSLAM::Vocabulary::transform compiled from the reference headers, oracle/_ref, 1 thread)"
                R.close()
            else:
                t0 = time.perf_counter(); O.bow_transform(va, fb, 2); bow["cpu_reference_us"] = (time.perf_counter() - t0) * 1e6
                bow["cpu_reference_kind"] = "port (oracle/bow_ref.c, 1 thread)"
            want_b = O.bow_transform(va, fb, 2)
            bow["parity"] = bool(all(np.array_equal(out_b[k], want_b[k]) for k in ("words", "values", "fv_node", "fv_feat")))
        except Exception as e:  # the GPU numbers stand on their own
            bow["cpu_reference_error"] = repr(e)
        dv.close()

    # ---- end to end through the host-buffer C-ABI, PAGEABLE frames, tracking thread || mapping thread ---------------------------
    pageable = [np.array(base[k], copy=True) for k in range(8)]           # malloc'd, like GImage (GImage.h:394-402)
    pinned_t = [torch.from_numpy(base[k]).pin_memory() for k in range(8)]
    pinned = [x.numpy() for x in pinned_t]
    e2e_steps = max(10, min(args.steps, 100))

    def e2e_serial(frames_h, n):
        prev = ctx.orb_extract(frames_h[0], NKP)[1]
        t0 = time.perf_counter()
        for k in range(n):
            kps, desc = ctx.orb_extract(frames_h[(k + 1) % 8], NKP)
            ctx.match_hamming(desc, prev)
            prev = desc
            pb = ba_problem.copy()
            ctx.ba_solve(pb, ba_cfg)
        return time.perf_counter() - t0

    def e2e_pipelined(frames_h, n):
        prev = ctx.orb_extract(frames_h[0], NKP)[1]
        qq: queue.Queue = queue.Queue(maxsize=2)
        err = []

        def mapper():
            try:
                while True:
                    k = qq.get()
                    if k is None:
                        return
                    pb = ba_problem.copy()
                    ctx_m.ba_solve(pb, ba_cfg)
            except Exception as e:  # surfaced after the join
                err.append(e)
        th = threading.Thread(target=mapper, daemon=True)
        t0 = time.perf_counter()
        th.start()
        for k in range(n):
            kps, desc = ctx.orb_extract(frames_h[(k + 1) % 8], NKP)
            ctx.match_hamming(desc, prev)
            prev = desc
            qq.put(k)
        qq.put(None)
        th.join()
        if err:
            raise err[0]
        return time.perf_counter() - t0

    def e2e_measure(fn, frames_h):
        fn(frames_h, 3)
        ts = []
        for rep in range(3):
            if world > 1:
                dist.barrier()
            ts.append(max_over_ranks(fn(frames_h, e2e_steps)))
        return world * e2e_steps / median(ts)
    e2e_pipe_pageable = e2e_measure(e2e_pipelined, pageable)
    e2e_pipe_pinned = e2e_measure(e2e_pipelined, pinned)
    e2e_serial_pageable = e2e_measure(e2e_serial, pageable)
    e2e_serial_pinned = e2e_measure(e2e_serial, pinned)
    h2d = W * H + 2 * NKP * 32 + ba_problem.n_cams * 57 + ba_problem.n_points * 25 + ba_problem.n_obs * (8 + 24)
    d2h = NKP * 60 + NKP * 12 + ba_problem.n_cams * 56 + ba_problem.n_points * 24

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    fps = world * args.steps / (ms_pipe * 1e-3)
    ab = algorithmic_bytes()
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        peak, peak_src = float(peaks["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"

    def gbs(nbytes, ms_):
        return nbytes / (ms_ * 1e-3) / 1e9
    ach = gbs(big_bytes, t_sweep_big)
    traffic = None
    try:  # per-launch DRAM bytes of the sweep from the committed ncu capture of this round (profiles/r02_sweep_traffic.json)
        traffic = float(json.load(open(os.path.join(ROOT, "profiles", "r02_sweep_traffic.json")))["dram_bytes_per_launch"])
        traffic_src = "profiles/r02_sweep_traffic.json (dram__bytes_read.sum + dram__bytes_write.sum of one launch, ncu --set full)"
    except Exception:
        traffic, traffic_src = 150.6e6, "profiles/r01_ncu_summary.md (44.25 MB read + 106.36 MB written, one launch, ncu --set full; round-1 kernel)"
    line = {"metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_pipe / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8+f64", "data": "synthetic",
            "config": workload_config(world),
            "timing": {"blocks": 1, "block_ms": ms_pipe,
                       "rule": "one block of exactly --steps steps between barrier+synchronize, CUDA events, max over ranks"},
            "serial": {"value": world * args.steps / (ms_serial * 1e-3), "ms_per_step": ms_serial / args.steps, "blocks": 1,
                       "note": "the same steps on ONE stream (round-1 definition of `value`)", "gpu_launches": int(ser_launches)},
            "clocks": clocks, "gpu_launches": int(pip_launches),
            "e2e": {"value": e2e_pipe_pageable, "unit": "frames/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "steps": e2e_steps, "host_memory": "pageable (malloc'd like GImage); tracking thread || mapping thread, two gb_ctx",
                    "pinned": e2e_pipe_pinned, "serial_pageable": e2e_serial_pageable, "serial_pinned": e2e_serial_pinned},
            "stages_ms": {"extract": t_ext, "match": t_match, "local_ba": t_ba},
            "local_ba_direct_solver": {"ms": t_ba_direct, "final_cost": res_direct[0].final_cost, "accepted": res_direct[0].accepted,
                                       "pcg_final_cost": res_pcg.final_cost, "pcg_accepted": res_pcg.accepted,
                                       "note": "linear_solver=1 (exact block-skyline Cholesky, csrc/ba_chol.cu) on the same window and LM iteration count; "
                                               "not the timed configuration"},
            # dominant HBM-bound kernel of the path = the BA Jacobian sweep (BASELINE metric, 2nd clause), at config-5 size
            "roofline": {"kernel": "BA Jacobian sweep K6 (ba_sweep_kernel: camera items + landmark items in one persistent launch), 500 cams/100k pts/1M obs",
                         "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "frac_on_measured_dram_bytes": (traffic / (t_sweep_big * 1e-3) / 1e9) / peak if traffic else None,
                         "in_timed_step": False,
                         "peak_source": peak_src, "algorithmic_bytes": int(big_bytes), "ms_per_sweep": t_sweep_big},
            # the same quantity for the kernels as they run inside the timed step (one frame / one 10k-observation window:
            # launch-latency-bound, reported for completeness)
            "roofline_step": {"extract_chain": {"algorithmic_bytes": ab["extract"], "ms": t_ext, "achieved_gbs": gbs(ab["extract"], t_ext),
                                                "frac": gbs(ab["extract"], t_ext) / peak},
                              "ba_sweep_local": {"algorithmic_bytes": ab["ba_sweep"], "ms": t_sweep_local,
                                                 "achieved_gbs": gbs(ab["ba_sweep"], t_sweep_local), "frac": gbs(ab["ba_sweep"], t_sweep_local) / peak},
                              "match": {"algorithmic_bytes": ab["match"], "popc32": 8 * NKP * NKP, "ms": t_match,
                                        "gpopc_per_s": 8 * NKP * NKP / (t_match * 1e-3) / 1e9, "bound": "integer POPC pipe",
                                        "peak_gpopc_per_s": popc_peak / 1e9 if popc_peak else None,
                                        "peak_source": "measured on this device (gb_dbg_popc_peak: 16 independent LOP3+POPC chains per thread, all SMs)",
                                        "frac": (8 * NKP * NKP / (t_match * 1e-3)) / popc_peak if popc_peak else None}},
            }
    line["config4_stereo"] = config4
    line["bow_transform"] = bow
    if global_ba is not None:
        line["global_ba"] = global_ba
    # CPU baseline on a bounded sample, rank 0 only, N=1 only
    if world == 1:
        try:
            n_cpu = 10
            cfps, what = cpu_path(base, ba_problem, n_cpu, cores)
            line["cpu_baseline"] = {"value": cfps, "unit": "frames/s", "cores": cores, "kind": "port", "sample": f"{n_cpu} frames: {what}"}
        except Exception as e:  # the GPU numbers stand on their own
            line["cpu_baseline"] = {"value": None, "error": repr(e)}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
