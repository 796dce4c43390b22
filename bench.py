#!/usr/bin/env python
"""bench.py — sliding-window continuous-time BA hot path (BASELINE.json metric) on B200.

    python bench.py --gpus N --steps K --warmup W            # CUDA engine (this repo)
    python bench.py --impl reference --gpus N --steps K ...  # CPU restatement of the reference path

A "step" is one pass of the hot path over one window: solve(15) of the BASELINE configs[1] window
(C2: 30 control points, 300 landmarks, 2 700 rolling-shutter observations, 270 IMU samples).
value  = residual-block Jacobian evaluations per second with the window resident in HBM
         (residual blocks x linearisation passes / solve time, CUDA events on the engine stream).
e2e    = the same metric through the C-ABI with HOST buffers: state + factors H2D, solve, state D2H
         inside the timed region (a fresh problem per window, like the reference's TrajectoryManager).
N > 1  = N independent replicas (one window per GPU, no data-path collective; "weak"); the
         landmark-sharded C4 run with its NCCL all-reduce is reported under "c4".
One JSON line on stdout (rank 0).
--dump-outputs DIR writes what the last timed solve returned to its caller (rank 0) as DIR/<name>.npy in float64:
the state read back after it (control points, biases, inverse depths, line delay) and its summary, and the same for
the last e2e step under the prefix "e2e_".  The inputs are seeded, so two builds run with the same arguments can be
compared array for array.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
pkg = importlib.import_module("ctrl-vio_b200")
syn = pkg.synthetic

MAX_ITERS = 15  # odometry_manager.cpp:277 budget of the full VIO solve


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region: NVML in a thread (a sample every ~10 ms, the timed
    region of the C2 window is only tens of milliseconds), `nvidia-smi -lms` as the fallback."""

    def __init__(self, index):
        self.index = index
        self.rows = []      # (sm_mhz, sm_max_mhz, reasons bitmask or list)
        self.stop_flag = threading.Event()
        self.thread = None
        self.mode = None
        self.proc = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            self.mode = "nvml"

            def loop():
                while True:
                    try:
                        sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                        rs = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                        self.rows.append((float(sm), float(mx), int(rs)))
                    except Exception:
                        pass
                    if self.stop_flag.wait(0.01):
                        break

            self.thread = threading.Thread(target=loop, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.mode = None
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.mode = "smi"
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.mode == "nvml":
            self.stop_flag.set()
            self.thread.join(timeout=1)
            import pynvml
            names = {"hw_slowdown": getattr(pynvml, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                     "hw_thermal_slowdown": getattr(pynvml, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                     "sw_thermal_slowdown": getattr(pynvml, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                     "sw_power_cap": getattr(pynvml, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
            reasons = sorted(n for n, bit in names.items() if any(r[2] & bit for r in self.rows))
            sm = [r[0] for r in self.rows]
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.rows[0][1] if self.rows else None,
                    "reasons": reasons, "samples": len(sm), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def oracle_lib():
    so = os.path.join(ROOT, "oracle", "liboracle.so")
    if not os.path.exists(so):
        subprocess.run(["make", "-C", os.path.join(ROOT, "oracle")], check=True, capture_output=True)
    return pkg.CtvioLib(so, "ctvo_", optional=pkg.binding.DEVICE_ONLY_SYMBOLS)


def solve_outputs(prefix, summary, q, p, biases, inv_depths, line_delay):
    """What a caller of solve receives: the summary and the state read back after it."""
    return {prefix + "knots_q": q, prefix + "knots_p": p, prefix + "biases": biases, prefix + "inv_depths": inv_depths,
            prefix + "line_delay": [line_delay], prefix + "cost": [summary.initial_cost, summary.final_cost],
            prefix + "lm_steps": [summary.iterations, summary.num_successful_steps, summary.num_unsuccessful_steps,
                                  summary.termination, summary.num_jacobian_evals]}


def dump_outputs(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def cpu_solve_rate(w, threads, budget_s):
    """Oracle (CPU port of the reference path) on a bounded sample: repeated solve(15) of window w."""
    import ctypes as C
    lib = oracle_lib()
    est = pkg.setup_estimator(lib, w)
    lib.raw("set_num_threads")(est.h, C.c_int32(threads))
    est.SaveState()
    t_total, evals, iters, solves = 0.0, 0, 0, 0
    while t_total < budget_s or solves < 2:
        est.RestoreState()
        t0 = time.perf_counter()
        s = est.Solve(MAX_ITERS)
        t_total += time.perf_counter() - t0
        evals += w.n_residual_blocks * s.num_jacobian_evals
        iters += s.iterations
        solves += 1
    return {"evals_per_s": evals / t_total, "lm_iters_per_s": iters / t_total, "solve_ms": 1e3 * t_total / solves,
            "solves": solves, "seconds": t_total}


def workload_desc(w):
    return (f"{w.name}: {w.n_knots} ctrl pts, {len(w.kf_times)} keyframes, {len(w.rho0)} landmarks, {w.n_obs} RS obs, "
            f"{len(w.imu_t)} IMU samples @200Hz, {len(w.bf_i)} bias factors, solve({MAX_ITERS})")


def algorithmic_bytes_visual(w):
    """SURVEY §8d per-unit figures x units of one K1 launch: 72 B per observation read, 408 B per landmark
    written, (np^2 + np) * 8 B camera system."""
    n_p = 6 * w.n_knots + 6 * len(w.kf_times) + 1
    return 72 * w.n_obs + 408 * len(w.rho0) + (n_p * n_p + n_p) * 8


VISUAL_KFLOP = 11.1  # SURVEY 8(d): ~6.0 kflop residual + analytic Jacobians (with the line-delay column) + ~5.1 kflop J'J


def roofline_k1_fp64(w_n_obs, visual_ms, fp64_tflops):
    """SURVEY 8(d) asks for K1's fp64 fraction next to its (by design tiny) HBM fraction: algorithmic flops of one
    launch = 11.1 kflop per visual block, over the kernel's CUDA-event time, against the fp64 rate measured in-run."""
    ach = VISUAL_KFLOP * 1e3 * w_n_obs / (visual_ms * 1e-3) / 1e12
    return {"bound": "fp64", "achieved": ach, "peak": fp64_tflops, "unit": "TFLOP/s", "frac": ach / fp64_tflops,
            "algorithmic_flops": VISUAL_KFLOP * 1e3 * w_n_obs, "kernel_ms": visual_ms, "kernel": "visual_kernel<true> (K1)"}


def best_thread_count(lib, est, candidates, solve):
    """The port's threaded residual assembly stops scaling well before the core count on small windows: calibrate."""
    import ctypes as C
    best = (float("inf"), 1)
    for cand in candidates:
        lib.raw("set_num_threads")(est.h, C.c_int32(cand))
        est.RestoreState()
        t0 = time.perf_counter()
        solve()
        best = min(best, (time.perf_counter() - t0, cand))
    return best[1]


def run_c3(lib, device, reps, is_oracle=False, threads=1):
    """BASELINE configs[2]: the C2-scale window with the line delay free: solve(15), 4-DoF re-alignment, marginalization
    of keyframe 0 (2 control points, bias node 0, the 100 landmarks anchored in it) into the next prior.  Wall-clock ms of
    the two C-ABI calls, state resident (SaveState / RestoreState between repetitions)."""
    import ctypes as C
    st = importlib.import_module("ctrl-vio_b200.streaming")
    e, seq, wa, nowk = st.c3_window_a(lib, device=device)
    if is_oracle:
        lib.raw("set_num_threads")(e.h, C.c_int32(threads))
    R0 = syn.qrot(wa.q0[nowk][None], np.eye(3)).T.copy(); t0 = wa.p0[nowk].copy()
    e.SaveState()
    t_solve, t_marg, dev, n = [], [], [], None
    for it in range(reps + (0 if is_oracle else 2)):
        e.RestoreState()
        a = time.perf_counter()
        s = e.Solve(MAX_ITERS)
        b = time.perf_counter()
        e.GaugeRealign(nowk, R0, t0)
        pr = e.SaveMarginalizationInfo()
        c = time.perf_counter()
        if is_oracle or it >= 2:
            t_solve.append(b - a); t_marg.append(c - b); dev.append(s.device_ms)
        n = pr.n
    return {"solve_ms": 1e3 * float(np.mean(t_solve)), "marginalize_ms": 1e3 * float(np.mean(t_marg)),
            "solve_device_ms": float(np.mean(dev)), "iterations": s.iterations, "prior_dim": n, "reps": len(t_solve),
            "n_obs": wa.n_obs}


def shard_window(w, rank, world):
    """Landmark-sharded view of a window: contiguous landmark ranges, global landmark ids kept (every rank holds the
    full inverse-depth array); IMU / bias factors stay on rank 0 (ctvio_comm_init contract)."""
    nL = len(w.rho0)
    lo, hi = rank * nL // world, (rank + 1) * nL // world
    return (w.lm >= lo) & (w.lm < hi)


def run_c4_sharded(lib, rank, world, local_rank, flush, dist, torch, fp64_tflops=None, n_landmarks=10_000, check_parity=True):
    """BASELINE configs[3]: C4 with residuals sharded by landmark over `world` GPUs; per LM step ONE NCCL all-reduce of the
    lower-triangular tiles of the reduced camera system (+ rhs + diagonal) and ONE all-gather of 8 scalars per rank.
    n_landmarks = 100 000 gives the 1 M-observation variant "c4x" (same control points: where sharding pays)."""
    w4 = syn.config_c4(n_landmarks=n_landmarks)
    sel = shard_window(w4, rank, world)
    est = pkg.Estimator(lib, pkg.make_config(device=local_rank, **w4.config_kwargs()))
    est.SetOptions(pkg.make_options(fix_ld=w4.fix_ld, ld_lower=w4.ld_lower, ld_upper=w4.ld_upper))
    est.SetKnots(w4.q0, w4.p0); est.SetBiases(w4.bias0); est.SetInvDepths(w4.rho0); est.SetLineDelay(w4.ld0)
    est.AddImageFeatureDelayAnalytic(w4.ti[sel], w4.rowi[sel], w4.pi[sel], w4.tj[sel], w4.rowj[sel], w4.pj[sel], w4.lm[sel])
    if rank == 0:
        est.AddIMUMeasurementAnalytic(w4.imu_t, w4.imu_gyro, w4.imu_accel, w4.imu_node)
        est.AddBiasFactor(w4.bf_i, w4.bf_j, w4.bf_sqrt_info)
    if world > 1:
        ids = [est.NcclUniqueId() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        est.CommInit(rank, world, ids[0])
    est.SaveState()
    w4_npad = ((6 * w4.n_knots + 6 * len(w4.kf_times) + 1 + 63) // 64) * 64
    ms, iters, passes = [], 0, 0
    for it in range(2 + 3):
        est.RestoreState()
        flush.fill_(it)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        s4 = est.Solve(MAX_ITERS)
        if it >= 2:
            ms.append(s4.device_ms); iters += s4.iterations; passes += s4.num_jacobian_evals
    t = torch.tensor([sum(ms)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    tot_s = t.item() * 1e-3
    out = {"workload": workload_desc(w4), "n_gpus": world, "value": w4.n_residual_blocks * passes / tot_s,
           "unit": "evals/s", "lm_iters_per_s": iters / tot_s, "solve_ms": 1e3 * tot_s / len(ms),
           "ms_per_lm_iter": 1e3 * tot_s / iters, "final_cost": s4.final_cost,
           "parallelism": f"landmark shards x{world}; per LM step one NCCL all-reduce of the packed lower-triangular reduced "
                          f"system ({8 * (w4_npad // 64) * (w4_npad // 64 + 1) // 2 * 4096 / 1e6:.1f} MB) + one all-gather of 8 scalars"}
    if world > 1 and check_parity:
        # in-bench parity of the sharded solve (the driver's GPU test box has one GPU): the same window solved by ONE
        # engine on rank 0 without sharding; state compared after the same number of LM steps
        qs, ps = est.GetKnots()
        diff = None
        if rank == 0:
            ref = pkg.setup_estimator(lib, w4, device=local_rank)
            sr = ref.Solve(MAX_ITERS)
            qr, pr = ref.GetKnots()
            dq = syn.qmul(syn.qconj(qr), qs)
            diff = {"iterations": [int(s4.iterations), int(sr.iterations)], "termination": [int(s4.termination), int(sr.termination)],
                    "final_cost_rel": abs(s4.final_cost - sr.final_cost) / sr.final_cost,
                    "max_translation_rel": float(np.abs(ps - pr).max() / np.abs(pr).max()),
                    "max_rotation_rad": float((2 * np.arctan2(np.linalg.norm(dq[:, :3], axis=1), np.abs(dq[:, 3]))).max())}
            del ref
        out["parity_vs_single_gpu"] = diff
    # K1 on this rank's shard (every N): algorithmic bytes / flops of the shard over the kernel's CUDA-event time
    n_shard = int(sel.sum())
    if world == 1:
        prof4 = est.ProfileKernels(reps=10, flush_l2=True)
        out["stage_ms"] = prof4
        vis_ms = prof4["visual"]
    else:
        vis_ms = est.ProfileVisual(reps=10, flush_l2=True)
    peaks, how = measured_peaks()
    n_p = 6 * w4.n_knots + 6 * len(w4.kf_times) + 1
    lm_shard = len(np.unique(w4.lm[sel]))
    alg = 72 * n_shard + 408 * lm_shard + (n_p * n_p + n_p) * 8
    ach4 = alg / (vis_ms * 1e-3) / 1e9
    out["roofline_visual"] = {"bound": "hbm", "achieved": ach4, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                              "frac": ach4 / peaks["hbm_gbs"], "algorithmic_bytes": alg, "kernel_ms": vis_ms,
                              "obs_on_this_rank": n_shard, "rank": rank}
    out["roofline_visual_fp64"] = roofline_k1_fp64(n_shard, vis_ms, fp64_tflops) if fp64_tflops else None
    del est
    return out


def cpu_c4_baseline(budget_s):
    """Oracle on the full C4 window: one solve(15) single-threaded (the reference's num_threads = 1) and one at the best
    thread count (bounded sample: the solve takes seconds)."""
    import ctypes as C
    w4 = syn.config_c4()
    lib = oracle_lib()
    est = pkg.setup_estimator(lib, w4)
    est.SaveState()
    out = {}
    ncpu = os.cpu_count() or 1
    for label, threads in (("threads_1", 1), ("threads_best", None)):
        if threads is None:
            threads = best_thread_count(lib, est, [c for c in (4, 8, 16, 32) if c <= ncpu] or [1], lambda: est.Solve(2))
        lib.raw("set_num_threads")(est.h, C.c_int32(threads))
        est.RestoreState()
        t0 = time.perf_counter()
        s = est.Solve(MAX_ITERS)
        dt = time.perf_counter() - t0
        out[label] = {"cores": threads, "solve_ms": 1e3 * dt, "value": w4.n_residual_blocks * s.num_jacobian_evals / dt,
                      "unit": "evals/s", "iterations": s.iterations, "final_cost": s.final_cost}
    out["kind"] = "port"
    out["sample"] = "1 x solve(15) of the full C4 window per thread count"
    return out


def c5_summary(records, skip):
    r = records[skip:]
    ms = np.array([x["ms"] for x in r])
    f = lambda k: float(np.mean([x[k] for x in r]))
    return {"windows": len(r), "ms_per_window_mean": float(ms.mean()), "ms_per_window_p50": float(np.median(ms)),
            "ms_per_window_p99": float(np.percentile(ms, 99)), "ms_build_and_predict_mean": f("ms_build_and_predict"),
            "ms_solve_mean": f("ms_solve"), "ms_realign_marginalize_mean": f("ms_realign_marginalize"),
            "ms_readback_mean": f("ms_readback"), "solve_device_ms_mean": f("device_ms"),
            "init_device_ms_mean": f("init_device_ms"), "lm_iterations_mean": f("iterations"),
            "h2d_bytes_per_window": f("h2d_bytes"), "d2h_bytes_per_window": f("d2h_bytes")}


def run_c5_streaming(lib, n_windows, device, cpu_windows):
    """BASELINE configs[4]: streaming sliding window at 20 Hz keyframes through the reference's per-image cycle
    (ExtendTrajectory -> InitTrajectory Solve(8) with fixed control points -> UpdateTrajectory Solve(15) -> 4-DoF
    re-alignment -> marginalization of the oldest keyframe -> slide), end-to-end ms per window through the public API with
    host buffers, everything that crosses the C-ABI inside the timed region.  The CPU oracle runs the IDENTICAL cycle on
    the first `cpu_windows` windows of the same sequence (bounded sample), single-threaded like the reference."""
    st = importlib.import_module("ctrl-vio_b200.streaming")
    seq = st.quantize_wire(st.config_c5_sequence(n_windows))  # bearings as the tracker's float32 PointCloud carries them
    r = st.StreamingRunner(lib, seq, device=device)
    r.run(n_windows)
    rr = st.ResidentRunner(lib, seq, device=device)   # SURVEY 8f-1 / 8f-4: the window lives in HBM, wire formats go up as they are
    rr.run(n_windows)
    last = r.records[-1]
    out = {"workload": f"C5: {n_windows} windows of 11 keyframes @20 Hz, ~{last['n_obs']} RS obs, {last['n_imu']} IMU samples, "
                       f"{last['n_knots']} ctrl pts, prior dim {last['prior_dim']}; per window: IMU-only predictor solve(8) + "
                       f"solve({MAX_ITERS}) + re-align + marginalize + slide",
           "gpu": c5_summary(r.records, min(5, n_windows // 2)), "final_cost_last": last["final_cost"],
           "rms_translation_error_vs_truth_m": r.state_error()}
    out["gpu"]["realtime_factor_at_20hz"] = 50.0 / out["gpu"]["ms_per_window_mean"]
    out["gpu"]["path"] = "host buffers: state, factors and prior re-uploaded every window through the Add* calls"
    out["gpu_resident"] = c5_summary(rr.records, min(5, n_windows // 2))
    out["gpu_resident"]["path"] = ("device-resident window: PointCloud / IMUData ingested as they are, control points extended / "
                                   "dropped on the device, prior handed over device-to-device, factor payload gathered from "
                                   "resident tables (index tables + the new frame cross the boundary)")
    out["gpu_resident"]["realtime_factor_at_20hz"] = 50.0 / out["gpu_resident"]["ms_per_window_mean"]
    out["gpu_resident"]["max_abs_translation_difference_to_host_buffer_path_m"] = float(
        np.abs(r.p[:r.ncp] - rr.p[:rr.ncp]).max())
    if cpu_windows > 0:
        ro = st.StreamingRunner(oracle_lib(), seq)
        ro.run(min(cpu_windows, n_windows))
        out["cpu_baseline"] = dict(c5_summary(ro.records, 1), cores=1, kind="port",
                                   sample=f"the first {len(ro.records)} windows of the same sequence, identical cycle")
        out["speedup_ms_per_window"] = out["cpu_baseline"]["ms_per_window_mean"] / out["gpu"]["ms_per_window_mean"]
        out["speedup_ms_per_window_resident"] = out["cpu_baseline"]["ms_per_window_mean"] / out["gpu_resident"]["ms_per_window_mean"]
    return out


def run_reference(args, rank, world):
    if rank != 0:
        return
    w = syn.config_c2()
    per_step = []
    evals = iters = 0
    lib = oracle_lib()
    import ctypes as C
    est = pkg.setup_estimator(lib, w)
    est.SaveState()
    # "All the host threads it can use": the port's threaded residual assembly stops scaling (and then degrades) well
    # before the box's core count on a window this small, so calibrate once and keep the fastest thread count.
    ncpu = os.cpu_count() or 1
    best = (float("inf"), 1)
    for cand in [c for c in (1, 2, 4, 8, 16, 32, 64, ncpu) if c <= ncpu]:
        lib.raw("set_num_threads")(est.h, C.c_int32(cand))
        ts = []
        for _ in range(2):
            est.RestoreState()
            t0 = time.perf_counter()
            est.Solve(MAX_ITERS)
            ts.append(time.perf_counter() - t0)
        best = min(best, (min(ts), cand))
    threads = best[1]
    lib.raw("set_num_threads")(est.h, C.c_int32(threads))
    for it in range(args.warmup + args.steps):
        est.RestoreState()
        t0 = time.perf_counter()
        s = est.Solve(MAX_ITERS)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            per_step.append(dt)
            evals += w.n_residual_blocks * s.num_jacobian_evals
            iters += s.iterations
    if args.dump_outputs:
        q, p = est.GetKnots()
        dump_outputs(args.dump_outputs, solve_outputs("", s, q, p, est.GetBiases(), est.GetInvDepths(), est.GetLineDelay()))
    total = sum(per_step)
    value = evals / total
    line = {
        "impl": "reference", "metric": "residual+Jacobian block evaluations per second (sliding-window LM solve)",
        "value": value, "unit": "evals/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / len(per_step), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_desc(w), "parallelism": f"cpu x{threads} threads (residual assembly)"},
        "lm_iters_per_s": iters / total,
        "cpu_baseline": {"value": value, "unit": "evals/s", "cores": threads, "kind": "port",
                         "sample": f"{len(per_step)} x solve({MAX_ITERS}) of the C2 window; CPU restatement of the "
                                   "reference path (the reference needs Eigen+Ceres, not buildable here); dense Schur + "
                                   "dense Cholesky instead of CHOLMOD"},
        "e2e": {"value": value, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--c5-windows", type=int, default=1000)
    ap.add_argument("--c5-cpu-windows", type=int, default=40)
    ap.add_argument("--no-c3", action="store_true")
    ap.add_argument("--no-c4x", action="store_true")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ctvio", choices=["ctvio", "reference"])
    ap.add_argument("--cpu-budget-s", type=float, default=10.0)
    ap.add_argument("--no-c4", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ctvio" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ctvio needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        # one window per GPU, each driven by its own host thread (launches + a spin on mapped memory once per LM step):
        # give every rank its own slice of the host cores so that the ranks do not migrate onto each other
        try:
            cpus = sorted(os.sched_getaffinity(0))
            per = len(cpus) // world
            if per >= 4:
                os.sched_setaffinity(0, cpus[local_rank * per:(local_rank + 1) * per])
        except (AttributeError, OSError):
            pass
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    lib = pkg.load()
    w = syn.config_c2(seed=syn.SEED0 + 2 + 1000 * rank)  # rank r solves its own window (replicas)
    n_blocks = w.n_residual_blocks

    # ---------------- resident path (value) ----------------
    est = pkg.setup_estimator(lib, w, device=local_rank)
    est.SaveState()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    sampler = ClockSampler(local_rank)
    per_ms, evals, iters, launches, wall = [], 0, 0, 0, 0.0
    for it in range(args.warmup + args.steps):
        if it == args.warmup:
            barrier()
            sampler.start()
            t_region0 = time.perf_counter()
        est.RestoreState()
        flush.fill_(it & 0xFF)          # L2 flush between timed iterations
        torch.cuda.synchronize()
        s = est.Solve(MAX_ITERS)        # timed by CUDA events on the engine stream (summary.device_ms)
        if it >= args.warmup:
            per_ms.append(s.device_ms)
            evals += n_blocks * s.num_jacobian_evals
            iters += s.iterations
            launches += s.kernel_launches
    barrier()
    wall = time.perf_counter() - t_region0
    clocks = sampler.stop()
    dev_s = sum(per_ms) * 1e-3
    summ = s
    if args.dump_outputs and rank == 0:
        q, p = est.GetKnots()
        outputs = solve_outputs("", s, q, p, est.GetBiases(), est.GetInvDepths(), est.GetLineDelay())

    # ---------------- e2e path: host buffers through the C-ABI ----------------
    e2e_est = pkg.Estimator(lib, pkg.make_config(device=local_rank, **w.config_kwargs()))
    e2e_est.SetOptions(pkg.make_options(fix_ld=w.fix_ld, ld_lower=w.ld_lower, ld_upper=w.ld_upper))
    pin = lambda a: a  # numpy arrays; the C-ABI stages them itself
    h2d = (w.q0.nbytes + w.p0.nbytes + w.bias0.nbytes + w.rho0.nbytes + 8 + w.ti.nbytes + w.tj.nbytes + w.rowi.nbytes +
           w.rowj.nbytes + w.pi.nbytes + w.pj.nbytes + w.lm.nbytes + w.imu_t.nbytes + w.imu_gyro.nbytes +
           w.imu_accel.nbytes + w.imu_node.nbytes + w.bf_i.nbytes + w.bf_j.nbytes + w.bf_sqrt_info.nbytes)
    d2h = w.q0.nbytes + w.p0.nbytes + w.bias0.nbytes + w.rho0.nbytes + 8
    e2e_times, e2e_evals = [], 0
    for it in range(args.warmup + args.steps):
        if it == args.warmup:
            barrier()
        t0 = time.perf_counter()
        e2e_est.SetKnots(w.q0, w.p0); e2e_est.SetBiases(w.bias0); e2e_est.SetInvDepths(w.rho0); e2e_est.SetLineDelay(w.ld0)
        e2e_est.ClearFactors()
        e2e_est.AddImageFeatureDelayAnalytic(w.ti, w.rowi, w.pi, w.tj, w.rowj, w.pj, w.lm)
        e2e_est.AddIMUMeasurementAnalytic(w.imu_t, w.imu_gyro, w.imu_accel, w.imu_node)
        e2e_est.AddBiasFactor(w.bf_i, w.bf_j, w.bf_sqrt_info)
        s2 = e2e_est.Solve(MAX_ITERS)
        q, p = e2e_est.GetKnots(); b = e2e_est.GetBiases(); r = e2e_est.GetInvDepths(); ld = e2e_est.GetLineDelay()
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            e2e_times.append(dt)
            e2e_evals += n_blocks * s2.num_jacobian_evals
    barrier()
    e2e_s = sum(e2e_times)
    if args.dump_outputs and rank == 0:
        outputs.update(solve_outputs("e2e_", s2, q, p, b, r, ld))
        dump_outputs(args.dump_outputs, outputs)

    # ---------------- kernel stage timings + roofline of the dominant kernel ----------------
    prof = est.ProfileKernels(reps=20, flush_l2=True) if rank == 0 else None
    fp64_tflops = est.MeasureFp64Tflops() if rank == 0 else None
    if world > 1:  # every rank needs the measured fp64 rate for its shard's K1 fraction
        fp64_tflops = est.MeasureFp64Tflops()
    c4 = None
    c4_clocks = None
    if not args.no_c4:
        s4 = ClockSampler(local_rank); s4.start()
        c4 = run_c4_sharded(lib, rank, world, local_rank, flush, dist, torch, fp64_tflops)
        c4_clocks = s4.stop()
        c4["clocks"] = c4_clocks
        if not args.no_c4x:
            c4["c4x"] = run_c4_sharded(lib, rank, world, local_rank, flush, dist, torch, fp64_tflops, n_landmarks=100_000,
                                       check_parity=False)
    c3 = c5 = None
    if rank == 0 and not args.no_c3:
        c3 = {"workload": "C3: C2-scale window (30 ctrl pts, 2700 RS obs, 270 IMU), line delay free, solve(15) + re-align + "
                          "marginalize keyframe 0", "gpu": run_c3(lib, local_rank, 10)}
    if rank == 0 and args.c5_windows > 0:
        s5 = ClockSampler(local_rank); s5.start()
        c5 = run_c5_streaming(lib, args.c5_windows, local_rank, args.c5_cpu_windows if world == 1 else 0)
        c5["clocks"] = s5.stop()

    # ---------------- reduce over ranks ----------------
    t = torch.tensor([dev_s, e2e_s, wall], dtype=torch.float64, device="cuda")
    c = torch.tensor([float(evals), float(iters), float(launches), float(e2e_evals)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
    dev_s_max, e2e_s_max, wall_max = t.tolist()
    evals_all, iters_all, launches_all, e2e_evals_all = c.tolist()

    if rank == 0:
        peaks, how = measured_peaks()
        # dominant kernel of the step: the dense solve (K5, chol_dag_kernel; > 50 % of the LM iteration, see
        # profiles/r1/e_launches_c2.csv).  It computes on the fp64 tensor/FMA pipe: algorithmic flops of one launch =
        # n^3/3 (factor) + 2 n^2 (two triangular solves), n = n_p; the denominator is the fp64 rate measured in this run
        # (MEASURED_PEAKS.json only has HBM and bf16 numbers).  K1's HBM-side roofline is reported next to it.
        n_p = 6 * w.n_knots + 6 * len(w.kf_times) + 1
        chol_flops = n_p ** 3 / 3.0 + 2.0 * n_p ** 2
        ach_tf = chol_flops / (prof["cholesky_solve"] * 1e-3) / 1e12
        alg = algorithmic_bytes_visual(w)
        ach = alg / (prof["visual"] * 1e-3) / 1e9
        traffic, traffic_k1, traffic_src = None, None, None
        try:
            with open(os.path.join(ROOT, "profiles", "kernel_traffic.json")) as f:
                tj = json.load(f)
                traffic, traffic_k1 = tj.get("c2_chol_dag_dram_bytes_per_launch"), tj.get("c2_visual_dram_bytes_per_launch")
                traffic_src = "STATIC: dram__bytes_read+write per launch from the committed ncu --set full capture " + \
                              str(tj.get("source", "profiles/kernel_traffic.json")) + " (not re-measured in this run)"
        except Exception:
            pass
        cpu1 = cpu_solve_rate(w, 1, args.cpu_budget_s) if world == 1 else None
        line = {
            "metric": "residual+Jacobian block evaluations per second (sliding-window LM solve)",
            "value": evals_all / dev_s_max, "unit": "evals/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dev_s_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_desc(w), "parallelism": f"replicas x{world} (one window per GPU)",
                       "l2": "256 MiB buffer written between timed solves (inputs are < L2)",
                       "timing": "CUDA events on the engine stream around each solve; max over ranks"},
            "lm_iters_per_s": iters_all / dev_s_max, "solve_ms": 1e3 * dev_s_max / args.steps,
            "wall_ms_per_step_incl_flush": 1e3 * wall_max / args.steps,
            "e2e": {"value": e2e_evals_all / e2e_s_max, "unit": "evals/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * e2e_s_max / args.steps},
            "gpu_launches": int(launches_all),
            "clocks": clocks,
            "roofline": {"bound": "tensor", "achieved": ach_tf, "peak": fp64_tflops, "unit": "TFLOP/s",
                         "frac": ach_tf / fp64_tflops, "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "chol_dag_kernel (K5)",
                         "peak_source": "fp64 DFMA/DMMA rate measured in this run (ctvio_measure_fp64_tflops); "
                                        "MEASURED_PEAKS.json has no fp64 figure",
                         "algorithmic_flops": chol_flops, "kernel_ms": prof["cholesky_solve"],
                         "note": "serial pivot chain of an n=%d factorisation: latency bound, not pipe bound "
                                 "(floor ~126 cycles per column = %.1f us, see DESIGN.md)" % (n_p, n_p * 126 / 1.965e3)},
            "roofline_k1": {"bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                            "frac": ach / peaks["hbm_gbs"], "traffic": traffic_k1, "kernel": "visual_kernel<true> (K1)",
                            "peak_source": how, "algorithmic_bytes": alg, "kernel_ms": prof["visual"],
                            "traffic_source": traffic_src},
            "roofline_k1_fp64": roofline_k1_fp64(w.n_obs, prof["visual"], fp64_tflops),
            "stage_ms": prof,
            "fp64_peak_tflops_measured": fp64_tflops,
            "solver": {"iterations": summ.iterations, "jacobian_passes": summ.num_jacobian_evals,
                       "termination": summ.as_dict()["termination_name"], "final_cost": summ.final_cost},
        }
        if cpu1 is not None:
            nmt = min(16, os.cpu_count() or 1)
            cpu_all = cpu_solve_rate(w, nmt, max(2.0, args.cpu_budget_s / 3))
            line["cpu_baseline"] = {"value": cpu1["evals_per_s"], "unit": "evals/s", "cores": 1, "kind": "port",
                                    "sample": f"{cpu1['solves']} x solve({MAX_ITERS}) of the same C2 window "
                                              f"({cpu1['seconds']:.1f} s), single thread like the reference's "
                                              "num_threads=1 (trajectory_estimator.cpp:379-383)",
                                    "lm_iters_per_s": cpu1["lm_iters_per_s"], "solve_ms": cpu1["solve_ms"],
                                    "multi_thread": {"cores": nmt, "value": cpu_all["evals_per_s"],
                                                  "solve_ms": cpu_all["solve_ms"]}}
        if c4 is not None:
            if world == 1:
                c4["cpu_baseline"] = cpu_c4_baseline(args.cpu_budget_s)
            line["c4"] = c4
        if c3 is not None:
            if world == 1:
                c3["cpu_baseline"] = dict(run_c3(oracle_lib(), 0, 3, is_oracle=True, threads=1), cores=1, kind="port")
                c3["speedup_solve"] = c3["cpu_baseline"]["solve_ms"] / c3["gpu"]["solve_ms"]
                c3["speedup_marginalize"] = c3["cpu_baseline"]["marginalize_ms"] / c3["gpu"]["marginalize_ms"]
            line["c3"] = c3
        if c5 is not None:
            line["c5"] = c5
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
