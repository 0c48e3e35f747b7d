#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on its config, on N GPUs of one node.

Metric: Gauss-Newton iterations/sec on the 10-keyframe x 500-landmark window (BASELINE config 2:
reprojection-only, frames 0 and 1 fixed, K_res = 4500).  One "step" = one full GN iteration
(linearise all factors + Cauchy weights -> Schur-eliminate inverse depths -> solve the reduced
system -> back-substitute -> Plus -> candidate cost) over a batch of W independent cfg2 windows
per GPU; value = windows * iterations / second over all GPUs, inputs resident in HBM, timed with CUDA events.
W = 4096 by default so that the inputs exceed the 126 MB L2.

e2e = the same metric through the reference-facing C-ABI call with HOST buffers
(pvio_b200_batch_solve_host: pinned host staging -> device, the device-side trust-region solve of up to 10
iterations per window, solved states back), host <-> device copies inside the timed region.

Extra keys of the same line: the other BASELINE configurations with the CPU port timed beside them (single cfg3 / cfg4
windows, marginalisation, literal config 5), single-window latency, a heterogeneous batch, KLT, PnP, IMU pre-integration.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--windows W] [--dump-outputs DIR]
--dump-outputs DIR writes what the last timed step computed, as a caller of the batched GN step receives it
(dump_outputs below), so that two builds run with the same arguments can be compared output for output.
Multi-GPU: python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N (one rank per GPU;
windows are independent, so there is no data-path collective: scaling is weak, NCCL carries only
the start barrier and the max-over-ranks of the device time).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "GN iters/sec on 10-KF x 500-landmark window (window-iterations/s)"
UNIT = "window-iterations/s"
WORKLOAD = "cfg2: 10 KF x 500 landmarks, K_res = 4500, reprojection-only Gauss-Newton, frames 0-1 fixed; independent windows"


def bytes_alg(N, M, K, D):
    """SURVEY.md 8(d): compulsory bytes of one GN iteration of one window in the fp32 device layout."""
    return 16 * K + 16 * M + 64 * N + 4 * (D * D + D) + 4 * M


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.rows, self.proc = [], None
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
                for nme, v in zip(names, f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def pin_to_gpu_numa(local_rank):
    """Run this rank (and the pinned staging it allocates from now on) on the CPUs of its GPU's NUMA node: the
    host -> device copies of the end-to-end path then do not cross the socket interconnect."""
    try:
        out = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=20).stdout
        for line in out.splitlines():
            f = line.replace("\x1b[4m", "").replace("\x1b[0m", "").split("\t")
            if f and f[0].strip() == f"GPU{local_rank}":
                cand = [x.strip() for x in f if x.strip() and all(c in "0123456789,-" for c in x.strip()) and ("-" in x or "," in x)]
                if not cand:
                    return None
                cpus = set()
                for part in cand[0].split(","):
                    a, _, b = part.partition("-")
                    cpus.update(range(int(a), int(b or a) + 1))
                cpus &= os.sched_getaffinity(0)
                if cpus:
                    os.sched_setaffinity(0, cpus)
                    return f"{cand[0]} ({len(cpus)} usable)"
    except Exception:
        return None
    return None


def cpu_rate(kind, win, st, n_sample, threads=0, **kw):
    """The reference's CPU implementation of the path: oracle/ba_oracle.c (Ceres / Eigen are absent, so the fp64 C
    restatement stands in, kind = "port"), n_sample independent windows over `threads` host threads (0: all usable)."""
    from oracle import c_oracle
    c_oracle.batch(kind, win, st, max(2, min(8, n_sample)), threads, **kw)          # warm-up / page-in
    t = time.perf_counter()
    used, units = c_oracle.batch(kind, win, st, n_sample, threads, **kw)
    dt = time.perf_counter() - t
    return units / dt, used, dt, units


def run_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return 0
    from oracle import c_oracle
    from synthetic import synth
    win, st, _ = synth.make_cfg2()
    cores = c_oracle.usable_cores()
    # bounded sample: ~1 s of work per step on this box's cores (one window-iteration is ~0.8 ms on one core)
    n_sample = int(max(64, min(args.windows, 1024 * max(1, cores // 8))))
    times = []
    for i in range(args.warmup + args.steps):
        v, used, dt, units = cpu_rate("gn_step", win, st, n_sample)
        if i >= args.warmup:
            times.append(dt)
    tot = sum(times)
    value = n_sample * args.steps / tot
    one, _, _, _ = cpu_rate("gn_step", win, st, 32, threads=1)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * tot / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "windows_per_step": n_sample,
                   "note": "bounded sample of the same workload: independent cfg2 windows over every usable host core"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": used, "kind": "port",
                         "sample": f"{n_sample} independent cfg2 window-iterations per step over {used} host threads "
                                   f"(usable cores: sched_getaffinity capped by the cgroup quota = {cores}); "
                                   "oracle/ba_oracle.c (fp64 restatement; Ceres/Eigen are not installed)",
                         "single_thread_value": one},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


DUMP_BYTES = 64 * 10**6


def dump_outputs(out_dir, dx, costs):
    """Writes the batched GN step's results as pvio_b200_batch_download returns them: dx.npy [windows, 15 N + M]
    (the step of every window) and costs.npy [windows, 2] (cost at the state, cost at the candidate), float64.
    If all windows exceed DUMP_BYTES, a fixed seeded sample of windows (ascending) is written instead, the same
    rows for the same --windows."""
    n = len(dx)
    keep = np.arange(n)
    per_window = dx.itemsize * dx.shape[1] + costs.itemsize * costs.shape[1]
    if n * per_window > DUMP_BYTES - 4096:          # room for the two .npy headers
        keep = np.sort(np.random.default_rng(0).choice(n, (DUMP_BYTES - 4096) // per_window, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "dx.npy"), np.ascontiguousarray(dx[keep], dtype=np.float64))
    np.save(os.path.join(out_dir, "costs.npy"), np.ascontiguousarray(costs[keep], dtype=np.float64))


def time_call(fn, reps, warm=1):
    for _ in range(warm):
        fn()
    t0 = time.perf_counter()
    for _ in range(reps):
        out = fn()
    return (time.perf_counter() - t0) / reps, out


def run_gpu(args):
    rank, local_rank, world = dist_env()
    numa = pin_to_gpu_numa(local_rank)
    import torch
    use_dist = world > 1
    if use_dist:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from pvio_b200 import klt, pnp, imu
    from synthetic import synth
    from pvio_b200.bundle_adjustor import BundleAdjustor
    from pvio_b200 import _lib as L
    import ctypes as C

    W = args.windows
    win, st, _ = synth.make_cfg2()
    N, M, K = win.N, win.M, win.K
    D = 6 * int(np.sum(win.frame_fixed == 0))
    ba = BundleAdjustor(device=local_rank, max_windows=W, max_frames=N, max_landmarks=512, max_obs=4608)
    # pack: the shim's per-window gather -> device layout in the pinned staging (host work, outside every timed region)
    pa = L.PackedArgs(win, st)
    n_pack = min(W, 256)
    t0 = time.perf_counter()
    for i in range(n_pack):
        ba.lib.pvio_b200_batch_set_window(ba.h, i, C.byref(pa.cw), C.byref(pa.cs))
    pack_us = (time.perf_counter() - t0) / n_pack * 1e6
    ba.batch_replicate(W)
    ba.batch_upload(W)
    ba.sync()

    def barrier():
        if use_dist:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        if not use_dist:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(x):
        if not use_dist:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    warm = max(args.warmup, 3)
    for _ in range(warm):
        ba.batch_gn_step(W, 1e-8, apply=False)
    ba.sync()
    ba.last_kernel_ms(-1)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    barrier()
    l0 = ba.kernel_launches
    ba.timer_start()
    for _ in range(args.steps):
        ba.batch_gn_step(W, 1e-8, apply=False)
    ms = ba.timer_stop()
    barrier()
    launches = ba.kernel_launches - l0
    if args.dump_outputs and rank == 0:         # before the e2e calls below replace the batch on the device
        dump_outputs(args.dump_outputs, *ba.batch_download(W, 15 * N + M))
    stage_ms, lin_ms, schur_ms = ba.last_kernel_ms(1), ba.last_kernel_ms(2), ba.last_kernel_ms(3)
    clocks = sampler.stop() if sampler else None
    ms_max = allmax(ms)
    launches = int(allsum(launches))
    value = world * W * args.steps / (ms_max * 1e-3)

    # ---- end to end through the C-ABI with HOST buffers: H2D of the packed batch + device-side solve + D2H of the states
    fr_out = np.zeros((W, N * 16)); rho_out = np.zeros((W, M))
    ba.batch_solve_host(W, N, M, max_iterations=10, frames=fr_out, rho=rho_out)
    barrier()
    e2e_steps = max(2, min(args.steps, 4))
    t0 = time.perf_counter()
    its = 0
    for _ in range(e2e_steps):
        _, _, sm = ba.batch_solve_host(W, N, M, max_iterations=10, frames=fr_out, rho=rho_out)
        its += sum(x.iterations for x in sm)
    e2e_s = allmax(time.perf_counter() - t0)
    barrier()
    e2e_value = allsum(its) / e2e_s
    its_per_window = its / (e2e_steps * W)
    # one GN iteration per upload (round 1's end-to-end figure, transfer-bound), for continuity
    stride = 15 * N + M
    dx = np.zeros((W, stride)); costs = np.zeros((W, 2))
    ba.batch_gn_step_host(W, stride, 1e-8, dx, costs)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        ba.batch_gn_step_host(W, stride, 1e-8, dx, costs)
    e2e1_s = allmax(time.perf_counter() - t0)
    barrier()
    e2e1_value = world * W * e2e_steps / e2e1_s
    h2d = W * (8 * 4608 + 16 * 512 + 8 * 512 + 8 * 16 * N + 832 + 224)
    d2h = W * (8 * 16 * N + 8 * 512 + 216)

    # ---- heterogeneous batch (5 window kinds: sizes, anchors, visibility, fixed sets differ), same GN step
    kinds = [synth.make_cfg2(N=10, M=500, seed=41)[:2], synth.make_cfg2(N=10, M=420, staggered=True, seed=42)[:2],
             synth.make_cfg2(N=8, M=300, seed=43)[:2], synth.make_cfg2(N=9, M=350, staggered=True, seed=44)[:2],
             synth.make_cfg2(N=10, M=500, seed=45)[:2]]
    kinds[2][0].frame_fixed[:] = 0; kinds[2][0].frame_fixed[0] = 1; kinds[2][0].frame_fixed[5] = 1
    pas = [L.PackedArgs(w_, s_) for w_, s_ in kinds]
    for i in range(W):
        p_ = pas[i % len(pas)]
        ba.lib.pvio_b200_batch_set_window(ba.h, i, C.byref(p_.cw), C.byref(p_.cs))
    ba.batch_upload(W)
    for _ in range(3):
        ba.batch_gn_step(W, 1e-8, apply=False)
    ba.sync(); ba.timer_start()
    for _ in range(max(3, args.steps // 2)):
        ba.batch_gn_step(W, 1e-8, apply=False)
    het_ms = ba.timer_stop() / max(3, args.steps // 2)
    barrier()

    if rank != 0:
        # literal config 5 needs every rank (below); the other extras are rank 0's
        run_cfg5(local_rank, rank, world, use_dist, allmax if use_dist else (lambda x: x))
        if use_dist:
            dist.destroy_process_group()
        return 0

    # ---- roofline of the dominant stage (linearise + Schur), CUDA events around every launch
    balg = bytes_alg(N, M, K, D)
    peak, peak_src = measured_peak()
    achieved = balg * W / (stage_ms * 1e-3) / 1e9
    traffic = warp_instr = None
    counters_src = None
    tp = os.path.join(ROOT, "profiles", "r02_stage_counters.json")
    if os.path.exists(tp):
        try:
            cj = json.load(open(tp))
            traffic = cj["dram_bytes_per_window"] * W
            warp_instr = cj["warp_instructions_per_window"]
            counters_src = cj.get("source")
        except Exception:
            pass
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    issue_frac = None
    if warp_instr:
        # issue-slot roofline: warp instructions issued / (SMs x 4 schedulers x clock x time)
        issue_frac = warp_instr * W / (148 * 4 * sm_mhz * 1e6 * stage_ms * 1e-3)
    roofline = {"bound": "hbm", "kernel": "lin_obs_kernel + schur_kernel (linearise + Schur stage, timed together)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "peak_source": peak_src, "bytes_alg_per_window": balg, "windows_per_launch": W,
                "kernel_ms": stage_ms, "linearise_ms": lin_ms, "schur_ms": schur_ms,
                "kernel_share_of_step": stage_ms / (ms / args.steps),
                "issue_slot_frac": issue_frac, "warp_instructions_per_window": warp_instr, "counters_source": counters_src,
                "note": "achieved = algorithmic bytes (SURVEY 8d) / CUDA-event time of the stage measured in this run; "
                        "issue_slot_frac = ncu-counted warp instructions of both kernels per window x windows / "
                        "(148 SMs x 4 schedulers x SM clock x the same time): the stage is latency / issue bound, not HBM bound "
                        "(arithmetic intensity ~33 flop/B, above the fp32 ridge) -- see DESIGN.md 4"}

    # ---- single window, one at a time (the reference's real use): latency through the C-ABI
    from oracle import c_oracle
    ba1 = BundleAdjustor(device=local_rank, max_windows=1, max_frames=N, max_landmarks=512, max_obs=4608)
    ba1.batch_set(0, win, st); ba1.batch_upload(1)
    for _ in range(5):
        ba1.batch_gn_step(1, 1e-8, apply=False)
    ba1.sync(); ba1.timer_start()
    for _ in range(50):
        ba1.batch_gn_step(1, 1e-8, apply=False)
    us_iter = ba1.timer_stop() * 1e3 / 50
    solve_s, (_, summ) = time_call(lambda: ba1.solve(win, st, max_iterations=10), 20, warm=2)
    cpu1 = time_call(lambda: c_oracle.solve(win, st, max_iter=10), 5)
    single = {"gn_iters_per_s": 1e6 / us_iter, "us_per_iteration": us_iter, "solve_call_ms": solve_s * 1e3,
              "solve_device_ms": summ["solve_seconds"] * 1e3, "solve_iterations": int(summ["iterations"]),
              "solve_iters_per_s_e2e": summ["iterations"] / solve_s,
              "cpu_port_solve_ms_1_thread": cpu1[0] * 1e3, "cpu_port_iterations": int(cpu1[1][2]["iterations"])}
    ba1.close()

    # ---- BASELINE configs 3 and 4 (inertial windows with prior / planes) and the marginaliser, CPU port beside the GPU
    extras = {}
    for name, maker in (("cfg3_inertial_prior", synth.make_cfg3), ("cfg4_planes", synth.make_cfg4)):
        try:
            w3, s3, _ = maker()
            b3 = BundleAdjustor(device=local_rank, max_windows=1, max_frames=w3.N, max_landmarks=320, max_obs=2560)
            for _ in range(3):
                b3.solve(w3, s3, max_iterations=10)
            samples = []
            for _ in range(100):        # per-call samples: the host thread of a shared box is descheduled now and then
                t0 = time.perf_counter()    # (tens of ms, device time unaffected), which a mean would smear over every call
                _, sm3 = b3.solve(w3, s3, max_iterations=10)
                samples.append(time.perf_counter() - t0)
            samples.sort()
            ts, worst = samples[len(samples) // 2], samples[-1]
            tc, cs = time_call(lambda: c_oracle.solve(w3, s3, max_iter=10), 5)
            entry = {"N": int(w3.N), "M": int(w3.M), "K_res": int(w3.K), "gpu_solve_call_ms": ts * 1e3,
                     "gpu_solve_call_ms_p90": samples[89] * 1e3, "gpu_solve_call_ms_worst_of_100": worst * 1e3,
                     "gpu_solve_call_ms_note": "median / 90th percentile / worst wall time of 100 calls through the C-ABI (pack, upload, "
                                               "one graph launch, download)",
                     "gpu_solve_device_ms": sm3["solve_seconds"] * 1e3,
                     "iterations": int(sm3["iterations"]), "cpu_port_solve_ms_1_thread": tc * 1e3,
                     "cpu_port_iterations": int(cs[2]["iterations"]), "speedup_vs_1_thread": tc / ts}
            if name == "cfg3_inertial_prior":
                tm, _ = time_call(lambda: b3.marginalize_frame(w3, s3, 0), 20, warm=2)
                tcm, _ = time_call(lambda: c_oracle.marginalize(w3, s3, 0), 10)
                extras["marginalize_frame"] = {"gpu_call_ms": tm * 1e3, "cpu_port_ms_1_thread": tcm * 1e3, "D": 15 * int(w3.N)}
            b3.close()
            extras[name] = entry
        except Exception as e:          # an extra never takes the headline line down
            extras[name] = {"error": str(e)}

    # ---- SURVEY 8(f) rank 1: a keyframe cycle (solve, marginalise the oldest frame, shift) with the window RESIDENT in
    # the handle (prior left on the device) against re-packing the whole window and carrying S / e through the host
    try:
        from synthetic.sequence import Run, Chain, ResidentPlayer
        run = Run(F=30, N=9, M=420, seed=701)
        br = BundleAdjustor(device=local_rank, max_windows=1, max_frames=10, max_landmarks=512, max_obs=4096)
        bp = BundleAdjustor(device=local_rank, max_windows=1, max_frames=10, max_landmarks=512, max_obs=4096)
        player, chain, t_repack, nkf = ResidentPlayer(br, run), Chain(run), 0.0, 16
        for k in range(nkf + 2):
            wk, sk, lmk = chain.window(k)
            t0 = time.perf_counter()
            outk, _ = bp.solve(wk, sk, max_iterations=10, postpass=False)
            Sk, ek = bp.marginalize_frame(wk, outk, index=0)
            if k >= 2:
                t_repack += time.perf_counter() - t0
            chain.store(k, outk, lmk); chain.set_prior(k, Sk, ek, outk)
            if k == 2:
                player.seconds = 0.0
            player.solve(10)
            player.shift(k)
        extras["keyframe_cycle"] = {"frames": int(run.N), "landmarks_in_window": int(wk.M), "keyframes": nkf,
                                    "resident_ms_per_keyframe": player.seconds / nkf * 1e3,
                                    "repack_ms_per_keyframe": t_repack / nkf * 1e3,
                                    "note": "wall time inside the C-ABI calls: resident = window_solve + window_drop_victim + "
                                            "append_frame (prior stays on the device); repack = ba_solve + ba_marginalize with "
                                            "the whole window and the prior (S, e) through host buffers"}
        br.close(); bp.close()
    except Exception as e:
        extras["keyframe_cycle"] = {"error": str(e)}

    # ---- literal BASELINE config 5: 8 independent cfg3 windows (seeds 648..655), window i -> GPU i mod G, full solves
    cfg5 = run_cfg5(local_rank, rank, world, use_dist, allmax)

    # ---- KLT tracks/s (752x480, 500 points, 21x21, 4 levels) through the C-ABI with host images
    prev, nxt, pts, _ = synth.make_klt_pair()
    kb = BundleAdjustor(device=local_rank, max_windows=1, max_frames=4, max_landmarks=8, max_obs=16)
    klt_s, _ = time_call(lambda: klt.track_keypoints(kb, prev, nxt, pts), 20)
    klt_info = {"tracks_per_s_e2e": len(pts) / klt_s, "ms_per_frame_pair": klt_s * 1e3, "points": int(len(pts))}
    raw_s, _ = time_call(lambda: klt.track_keypoints(kb, prev, nxt, pts, clahe_clip=6.0), 20)
    klt_info["raw_frames_tracks_per_s_e2e"] = len(pts) / raw_s
    klt_info["raw_frames_ms_per_frame_pair"] = raw_s * 1e3
    try:
        import cv2
        crit = (cv2.TERM_CRITERIA_COUNT + cv2.TERM_CRITERIA_EPS, 30, 0.01)
        p0 = pts.reshape(-1, 1, 2)
        cv_call = lambda: cv2.calcOpticalFlowPyrLK(prev, nxt, p0.copy(), p0.copy(), winSize=(21, 21), maxLevel=3, criteria=crit,
                                                   flags=cv2.OPTFLOW_USE_INITIAL_FLOW)
        cv_s, _ = time_call(cv_call, 10)
        klt_info["cv2_tracks_per_s"] = len(pts) / cv_s
        klt_info["cv2_threads"] = cv2.getNumThreads()
    except Exception as e:      # cv2 is the reference's KLT; report if it is unavailable
        klt_info["cv2_tracks_per_s"] = None
        klt_info["cv2_error"] = str(e)
    try:
        # steady state of the tracker: prev = the previous call's next, already on the device (pyramid cache by frame id)
        klt.track_keypoints(kb, prev, nxt, pts, clahe_clip=6.0, prev_id=1, next_id=2)
        fid = [2]

        def cached_pair():
            fid[0] += 1
            return klt.track_keypoints(kb, None, nxt if fid[0] % 2 else prev, pts, clahe_clip=6.0, prev_id=fid[0] - 1,
                                       next_id=fid[0], shape=prev.shape)
        c_s, _ = time_call(cached_pair, 20)
        klt_info["cached_prev_tracks_per_s_e2e"] = len(pts) / c_s
        klt_info["cached_prev_ms_per_frame_pair"] = c_s * 1e3
        kb.timer_start()
        for _ in range(20):
            klt.track_keypoints(kb, None, None, pts, clahe_clip=6.0, prev_id=fid[0] - 1, next_id=fid[0], shape=prev.shape)
        lk_ms = kb.timer_stop() / 20
        klt_bytes = 16384.0 * len(pts)                # SURVEY 8(d): ~16 KB of patch + gradient loads per point over 4 levels
        klt_info["roofline"] = {"bound": "hbm", "kernel": "klt_track_kernel (+ border test), both pyramids resident",
                                "achieved": klt_bytes / (lk_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                "frac": klt_bytes / (lk_ms * 1e-3) / 1e9 / peak, "device_us_per_pair": lk_ms * 1e3,
                                "note": "latency-bound, not bandwidth-bound: one warp per keypoint walks 4 levels x <= 30 "
                                        "dependent iterations; 476 warps occupy 5 % of the GPU's warp slots and the pyramids "
                                        "(0.5 MB) sit in L2 (profiles/r02g_klt.md: 0.9 MB of DRAM reads per launch)"}
        from pvio_b200.detect import detect_keypoints
        have = pts[::4]
        d_s, newk = time_call(lambda: detect_keypoints(kb, None, have, keypoint_distance=25.0, clahe_clip=6.0, frame_id=fid[0],
                                                       shape=prev.shape), 20)
        klt_info["detect_keypoints"] = {"ms_per_frame_e2e": d_s * 1e3, "existing": int(len(have)), "new_keypoints": int(len(newk)),
                                        "note": "frame taken from the tracker's device cache"}
        try:
            import cv2
            eq = cv2.createCLAHE(6.0, (8, 8)).apply(nxt)
            g_s, _ = time_call(lambda: cv2.goodFeaturesToTrack(eq, 1000, 1e-3, 20, blockSize=3, useHarrisDetector=True, k=0.04), 10)
            klt_info["detect_keypoints"]["cv2_gftt_ms"] = g_s * 1e3
        except Exception as e:
            klt_info["detect_keypoints"]["cv2_error"] = str(e)
    except Exception as e:
        klt_info["cached_error"] = str(e)
    try:
        # the F-matrix outlier rejection of track_keypoints (opencv_image.cpp:121-129) and the whole call with it
        fp, fq = synth.make_fm_matches(seed=652, n=400, outlier_frac=0.2)
        f_s, (fmask, _, finfo) = time_call(lambda: klt.find_fundamental_mask(kb, fp, fq, return_info=True), 50, warm=3)
        klt_info["f_ransac"] = {"ms_per_call_e2e": f_s * 1e3, "matches": int(len(fp)), "inliers": int(fmask.sum()),
                                "serial_iterations": finfo["iterations"], "iterations_evaluated_on_device": 1000}
        w_s, _ = time_call(lambda: klt.track_keypoints_ransac(kb, prev, nxt, pts, prev_id=901, next_id=902), 20, warm=2)
        klt_info["track_keypoints_whole_call_ms"] = w_s * 1e3
        try:
            import cv2
            cf_s, _ = time_call(lambda: cv2.findFundamentalMat(fp, fq, cv2.FM_RANSAC, 1.0, 0.99), 50, warm=3)
            klt_info["f_ransac"]["cv2_ms"] = cf_s * 1e3
        except Exception as e:
            klt_info["f_ransac"]["cv2_error"] = str(e)
    except Exception as e:
        klt_info["f_ransac_error"] = str(e)

    # ---- visual_inertial_pnp (150 points + IMU prior): one kernel launch per solve, host buffers in/out
    d = synth.make_pnp()
    pargs = (d['frame'], d['last'], d['imu'], d['pts'], d['zs'], d['cam_q'], d['cam_p'], d['imu_q'], d['imu_p'], d['W'], True)
    pnp_s, (_, psum) = time_call(lambda: pnp.visual_inertial_pnp(kb, *pargs), 20)
    pnp_info = {"ms_per_solve_e2e": pnp_s * 1e3, "kernel_ms": psum["solve_seconds"] * 1e3,
                "iterations": int(psum["iterations"]), "points": int(len(d['pts']))}
    kb.close()

    # ---- CPU baseline beside it (bounded sample, all usable host cores; plus one thread like num_threads = 1)
    cores = c_oracle.usable_cores()
    n_sample = int(max(256, 1024 * max(1, cores // 8)))
    cpu_v, cpu_used, cpu_dt, _ = cpu_rate("gn_step", win, st, n_sample)
    cpu_one, _, _, _ = cpu_rate("gn_step", win, st, 64, threads=1)
    cpu_solve_v, _, _, _ = cpu_rate("solve", win, st, max(64, n_sample // 8), max_iter=10)
    cpu_baseline = {"value": cpu_v, "unit": UNIT, "cores": cpu_used, "kind": "port",
                    "sample": f"{n_sample} independent cfg2 window-iterations over {cpu_used} host threads "
                              f"({cpu_dt:.2f} s wall; usable cores = sched_getaffinity capped by the cgroup quota = {cores}); "
                              "oracle/ba_oracle.c, fp64, Ceres/Eigen unavailable",
                    "single_thread_value": cpu_one, "full_solve_value": cpu_solve_v}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
        "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 Jacobians + f64 residuals/accumulation/solve (visual-only windows); f64 throughout for inertial windows",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "windows_per_gpu": W,
                   "l2_policy": f"device-resident inputs {(8 * K + 24 * M + 128 * N + 1056) * W / 1e6:.0f} MB + "
                                f"{(16 * K + 32 * 6 * K // 6) * W / 1e6:.0f} MB of intermediate records per step exceed the 126 MB L2",
                   "parallelism": f"independent windows, {world} GPU(s), no data-path collective",
                   "cpu_affinity": numa},
        "clocks": clocks, "gpu_launches": int(launches),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "iterations_per_upload": its_per_window, "pack_us_per_window": pack_us,
                "one_iteration_per_upload_value": e2e1_value,
                "note": "pvio_b200_batch_solve_host: pinned host staging -> device, device-side trust-region solve "
                        "(<= 10 iterations per window, per-window termination), solved states back; "
                        "pack_us_per_window (the shim-side gather into the staging, host) is outside the timed region"},
        "roofline": roofline, "cpu_baseline": cpu_baseline,
        "heterogeneous_batch": {"ms_per_step": het_ms, "window_iterations_per_s": W / (het_ms * 1e-3),
                                "kinds": "5 window shapes (N 8-10, M 300-500, staggered anchors, non-contiguous fixed frames)"},
        "single_window": single, "configs": extras, "config5_8_windows": cfg5, "klt": klt_info, "pnp": pnp_info,
    }
    print(json.dumps(line))
    ba.close()
    if use_dist:
        dist.destroy_process_group()
    return 0


def run_cfg5(local_rank, rank, world, use_dist, allmax):
    """BASELINE config 5 as written: 8 independent cfg3-shaped windows (seeds 648..655), window i -> GPU i mod G, a full
    solve each; time = max over ranks of the host-buffer call (upload + device-side solves + download)."""
    try:
        from synthetic import synth
        from pvio_b200.bundle_adjustor import BundleAdjustor
        wins = [synth.make_cfg3(seed=648 + i)[:2] for i in range(8)]
        mine = [wins[i] for i in range(8) if i % world == rank]
        b5 = BundleAdjustor(device=local_rank, max_windows=len(mine), max_frames=9, max_landmarks=320, max_obs=2560)
        for i, (w_, s_) in enumerate(mine):
            b5.batch_set(i, w_, s_)
        N5, M5 = 9, 320
        b5.batch_solve_host(len(mine), N5, M5, max_iterations=10)
        if use_dist:
            import torch.distributed as dist
            import torch
            dist.barrier(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        reps = 10
        its = 0
        for _ in range(reps):
            _, _, sm = b5.batch_solve_host(len(mine), N5, M5, max_iterations=10)
            its += sum(x.iterations for x in sm)
        dt = allmax((time.perf_counter() - t0) / reps)
        b5.close()
        out = {"windows": 8, "gpus": world, "ms_per_batch_e2e": dt * 1e3, "windows_per_s": 8 / dt,
               "iterations_rank0": its / reps}
        if rank == 0:
            from oracle import c_oracle
            t0 = time.perf_counter()
            tot = 0
            for w_, s_ in wins:
                tot += c_oracle.solve(w_, s_, max_iter=10)[2]["iterations"]
            t1 = time.perf_counter() - t0
            out["cpu_port_ms_1_thread_8_windows"] = t1 * 1e3
            out["cpu_port_iterations"] = int(tot)
        return out
    except Exception as e:
        return {"error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--windows", type=int, default=4096, help="independent cfg2 windows per GPU per step")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's dx and costs as DIR/<name>.npy (at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the GPU path's outputs; it does not apply to --impl reference")
    if args.impl == "reference":
        return run_reference(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
