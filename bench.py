#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native camera<-laser extrinsic solve.

Workload (BASELINE.json configs[1]): 10^4 frames x 10^3 laser points per GPU, synthetic boards from the reference's
simulation generator (main/calibr_simulation.cpp:10-108, exact-M mode, 1 cm range noise), identity initial guess.
A "step" is one complete CamLaserCalibration-equivalent solve: the on-device Levenberg-Marquardt loop to Ceres'
convergence criteria, one fused residual+Jacobian+reduce sweep over every point per LM iteration.

One JSON line; everything the driver's parser keeps is nested under the contract keys:
  value     residual+Jacobian evaluations / s over the whole job, data already resident in HBM (CUDA-event time, max over ranks)
  e2e       the same through the reference's OWN C++ call: host/dropin_bench.cpp builds a std::vector<Oberserve> (one pageable
            heap array per frame) and times CamLaserCalibration(obs, Tcl, false) of the drop-in, entry to return -- gather/pack,
            PCIe, HBM layout, LM solve, analysis tail, tear-down; N ranks: rank 0 runs it on N devices of one process
  roofline  the fused sweep kernel alone: algorithmic bytes (24 B/residual + 40 B/frame + 224 B) / CUDA-event time per launch,
            L2 flushed between launches, against the measured HBM copy bandwidth (MEASURED_PEAKS.json); nested: .planar (16 B per
            residual, own denominator), .config3 (10^5 x 2000, 4.8 GB), .config5 (+ board-edge residuals, camera-chain poses)
  config    workload + .check (noise-free ground truth < 1e-9; collective evaluation = sum of the shards'), .strong_scaling
            (BASELINE configs[3], 2*10^9 residuals split over the N ranks), .step_device_ms (min / median / max of the K solves)
  cpu_baseline / --impl reference   the CPU oracle port of the reference algorithm (Ceres-shaped: materialised Jacobian + dense
            QR, evaluation threaded over the host cores) on a bounded sample of the same workload.

Multi-GPU (torchrun, one rank per GPU): weak scaling -- every rank holds 10^4 frames of a 10^4 x N frame problem; the 28
normal-equation sums are exchanged inside the sweep kernel (NVLink peer stores) and every rank runs the identical LM update.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FRAMES_PER_GPU = 10_000
BEAMS = 1_000
SEED = 7
SIGMA = 0.01
X0 = np.array([0, 0, 0, 0, 0, 0, 1.0])
CPU_SAMPLE_FRAMES = 1_000
METRIC = "residual+Jacobian evals/sec (full LM solves)"
UNIT = "residual evals/s"


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError(f"must be >= 1, got {v}")
    return v


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=200, help="timed steps (full LM solves), exactly this many")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--frames", type=int, default=FRAMES_PER_GPU, help="frames per GPU")
    ap.add_argument("--beams", type=int, default=BEAMS)
    ap.add_argument("--kernel-launches", type=int, default=100, help="timed launches of the sweep kernel for the roofline")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--nccl-allreduce", action="store_true", help="N>1: ncclAllReduce between kernels instead of the fused peer exchange")
    ap.add_argument("--no-config3", action="store_true", help="skip the supplementary 4.8 GB rows (configs[2] and configs[4])")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling leg (configs[3], 48 GB over the N ranks)")
    ap.add_argument("--strong-frames", type=int, default=1_000_000)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed solve returned as DIR/<name>.npy (rank 0)")
    return ap.parse_args()


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


# ---- clocks during the timed region (B200_PROFILING.md) ----------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); smax.append(float(parts[1])); power.append(float(parts[2]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        os.unlink(self.path)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        # "under load": samples in the upper half of the observed power range
        thr = min(power) + 0.5 * (max(power) - min(power))
        loaded = [c for c, p in zip(sm, power) if p >= thr] or sm
        return {"sm_mhz": statistics.median(loaded), "sm_max_mhz": max(smax), "reasons": sorted(reasons),
                "power_w_max": max(power), "samples": len(sm)}


# ---- CPU baseline: the oracle port of the reference algorithm ------------------------------------------------------
def cpu_reference_problem(frames, beams):
    from oracle import oracle as O

    return O.generate(frames, beams, seed=SEED, sigma=SIGMA, exact_m=True)


def time_cpu_solve(p, threads, linear_solver):
    """One full LM solve with the oracle; returns (seconds, residual evaluations, iterations, (pose7, summary, trace))."""
    from oracle import oracle as O

    opt = O.default_options(linear_solver=linear_solver, num_threads=threads)
    t0 = time.perf_counter()
    x, s, tr = O.solve(p, X0, opt)
    dt = time.perf_counter() - t0
    return dt, s.num_residual_evaluations * p.num_residuals(), s.num_iterations, (x, s, tr)


def pick_threads(p):
    """Thread count that makes the oracle's residual sweep fastest on this host (a container may expose more CPUs than
    its quota lets it use, in which case all-cores OpenMP is slower than a few threads)."""
    from oracle import oracle as O

    cores = os.cpu_count() or 1
    cands = sorted({1, 2, 4, 8, 16, 32, 64, cores} & set(range(1, cores + 1)))
    best, best_t = 1, None
    for th in cands:
        O.evaluate_normal(p, X0, num_threads=th)
        t0 = time.perf_counter()
        for _ in range(3):
            O.evaluate_normal(p, X0, num_threads=th)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = th, dt
    return best


def cpu_baseline(frames, beams, quick=False):
    """Times the oracle port on a bounded sample.  Primary number: the Ceres-shaped solve (materialised P x 6
    Jacobian + Householder QR -- the work the reference does) with the better of {1 thread (what the reference uses:
    Ceres num_threads is never set), all host threads for the residual/Jacobian evaluation}."""
    n = min(frames, CPU_SAMPLE_FRAMES)
    p = cpu_reference_problem(n, beams)
    cores = pick_threads(p)
    dt1, ev1, iters, _ = time_cpu_solve(p, 1, 0)
    best = dict(value=ev1 / dt1, cores=1)
    extras = {"ceres_shaped_1_thread": {"value": ev1 / dt1, "unit": UNIT, "cores": 1}}
    if cores > 1:
        dta, eva, _, _ = time_cpu_solve(p, cores, 0)
        extras["ceres_shaped_best_thread_count"] = {"value": eva / dta, "unit": UNIT, "cores": cores}
        if eva / dta > best["value"]:
            best = dict(value=eva / dta, cores=cores)
    if not quick:
        dts, evs, _, _ = time_cpu_solve(p, cores, 1)  # most favourable CPU variant: streaming normal equations
        extras["streaming_normal_equations_best_thread_count"] = {"value": evs / dts, "unit": UNIT, "cores": cores}
    extras["host_cpus_visible"] = os.cpu_count()
    out = dict(value=best["value"], unit=UNIT, cores=best["cores"], kind="port",
               sample=f"first {n} of {frames} frames x {beams} points ({n * beams} residuals), one full LM solve "
                      f"({iters} iterations, {ev1 // (n * beams)} sweeps), Ceres-shaped (materialised Jacobian + dense QR)")
    out.update(extras)
    return out


def workload_config(args, world):
    """The `config` both arms print (the reference arm runs a bounded sample of it; see its cpu_baseline.sample)."""
    return {"workload": f"BASELINE configs[1]: {args.frames} frames x {args.beams} points per GPU, calibr_simulation generator "
                        f"(exact-M), sigma={SIGMA} m, identity start, full LM solve to Ceres convergence"}


def run_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return
    n = min(args.frames, CPU_SAMPLE_FRAMES)
    p = cpu_reference_problem(n, args.beams)
    cores = pick_threads(p)
    # threads: the better of 1 (what the reference uses) and all host threads, decided on the warm-up solves
    rates = {}
    for th in sorted({1, cores}):
        dt, ev, _, _ = time_cpu_solve(p, th, 0)
        rates[th] = ev / dt
    cores = max(rates, key=rates.get)
    for _ in range(max(0, args.warmup - len(rates))):
        time_cpu_solve(p, cores, 0)
    t_tot, ev_tot, iters, steps_done = 0.0, 0, 0, 0
    for _ in range(args.steps):
        dt, ev, iters, result = time_cpu_solve(p, cores, 0)
        t_tot += dt
        ev_tot += ev
        steps_done += 1
    if args.dump_outputs:
        from oracle import oracle as O

        dump_solve_outputs(args.dump_outputs, *result, O.Iteration)
    value = ev_tot / t_tot
    sample = (f"each step = one full LM solve on the first {n} of {args.frames} frames x {args.beams} points "
              f"({n * args.beams} residuals, {iters} iterations); Ceres-shaped oracle port, evaluation on {cores} threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps_done,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / steps_done, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "the reference itself (Ceres+Eigen+ROS) cannot be built in this image; this is the CPU oracle port",
    }
    print(json.dumps(line))


# ---- our arm ----------------------------------------------------------------------------------------------------------
GT_TLC = np.array([[0.0, 0.0, 1.0, 0.1], [-1.0, 0.0, 0.0, 0.2], [0.0, -1.0, 0.0, 0.3], [0.0, 0.0, 0.0, 1.0]])  # calibr_simulation.cpp:15-20


def pose_error_vs_ground_truth(x):
    """(rotation angle [rad], translation distance [m]) between pose7 x (T_cl) and the generator's ground truth."""
    from camlasercalibratool_b200.api import pose7_to_T

    T = np.asarray(pose7_to_T(x)).reshape(4, 4)
    Tgt = np.linalg.inv(GT_TLC)
    dR = T[:3, :3].T @ Tgt[:3, :3]
    # angle from the skew part (arccos of the trace loses half the digits near zero)
    w = 0.5 * np.array([dR[2, 1] - dR[1, 2], dR[0, 2] - dR[2, 0], dR[1, 0] - dR[0, 1]])
    sn, cs = float(np.linalg.norm(w)), float((np.trace(dR) - 1.0) / 2.0)
    return float(np.arctan2(sn, cs)), float(np.linalg.norm(T[:3, 3] - Tgt[:3, 3]))


def run_dropin(frames, beams, steps, warmup, devices=None, edges=0, sigma=SIGMA, seed=SEED, timeout=900):
    """Runs the C++ end-to-end driver (host/dropin_bench.cpp: std::vector<Oberserve> -> CamLaserCalibration() of the drop-in)
    as a child process and returns its JSON."""
    from camlasercalibratool_b200 import _build

    exe = _build.BENCH_EXE
    if not os.path.exists(exe):
        exe = _build.build_dropin_bench()
    env = dict(os.environ)
    if devices is not None:
        env["CLC_DEVICES"] = ",".join(str(d) for d in devices)
    cmd = [exe, str(frames), str(beams), repr(sigma), str(seed), str(steps), str(warmup), str(edges)]
    res = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=timeout)
    for line in res.stdout.splitlines():
        if line.startswith("CLC_DROPIN_JSON "):
            out = json.loads(line[len("CLC_DROPIN_JSON "):])
            out["rc"] = res.returncode
            return out
    raise RuntimeError(f"clc_dropin_bench failed (rc {res.returncode}): {res.stderr[-400:]}")


def kernel_row(prob, x, n_launch, peaks, label):
    """Roofline row of the sweep kernel on `prob` as configured: per-launch CUDA events, L2 flushed between launches."""
    prob.bench_eval(x, 5, flush_l2=True)
    ms = prob.bench_eval(x, n_launch, flush_l2=True)
    mean = float(np.mean(ms))
    nbytes = prob.streamed_bytes()
    n_points = prob.sizes()[1]
    ach = nbytes / (mean * 1e-3) / 1e9
    return {"kernel": label, "bound": "hbm", "achieved": ach, "peak": peaks, "unit": "GB/s", "frac": ach / peaks,
            "kernel_ms_mean": mean, "kernel_ms_min": float(np.min(ms)), "kernel_ms_median": float(np.median(ms)),
            "algorithmic_bytes_per_launch": nbytes, "residuals_per_s_kernel": n_points / (mean * 1e-3), "launches_timed": n_launch}


def solve_row(prob, opt, reps, n_points_total, max_over_ranks, barrier):
    """K full LM solves; returns throughput figures (device time, max over ranks)."""
    prob.solve(X0, opt)
    barrier()
    ms, sweeps, iters, per = 0.0, 0, 0, []
    x = X0
    for _ in range(reps):
        x, s, _ = prob.solve(X0, opt)
        ms += s.device_ms
        per.append(s.device_ms)
        sweeps += s.num_sweeps
        iters += s.num_iterations - 1
    barrier()
    ms = max_over_ranks(ms)
    return x, {"ms_per_solve": ms / reps, "sweeps_per_solve": sweeps / reps, "lm_iterations_per_solve": iters / reps,
               "residual_evals_per_s": n_points_total * sweeps / (ms * 1e-3), "lm_iters_per_s": iters / (ms * 1e-3),
               "termination": int(s.termination)}


def dump_solve_outputs(out_dir, x, summary, trace, iteration_type):
    """What a solve returned (Problem.solve, or the oracle's for --impl reference), one float64 .npy per quantity: pose7
    (T_cl), summary_<field> and trace_<field> (one entry per LM iteration, fields of iteration_type).  The timing
    (device_ms) and padding fields are left out: they are not results."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"pose7": x}
    for name, _ in type(summary)._fields_:
        if name not in ("reserved", "device_ms"):
            arrays["summary_" + name] = getattr(summary, name)
    for name, _ in iteration_type._fields_:
        if name != "reserved":
            arrays["trace_" + name] = [getattr(t, name) for t in trace]
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def run_ours(args):
    import torch
    import torch.distributed as dist

    from camlasercalibratool_b200 import Comm, Problem, comm_unique_id, default_options, launch_count

    rank, local_rank, world = dist_env()
    if args.gpus != world:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local_rank)
    # clocks: 100 ms sampling period and nvidia-smi needs ~1 s to deliver its first line, the timed region lasts ~20 ms -- the
    # sampler therefore runs from here (problem generation, communicator set-up, warm-up, timed solves, roofline legs)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    cpu_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        cpu_group = dist.new_group(backend="gloo")  # host-only rendezvous: does not put a spinning kernel on the GPUs

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(a):
        a = np.atleast_1d(np.asarray(a, dtype=np.float64))
        if world == 1:
            return a
        t = torch.tensor(a, dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return t.cpu().numpy()

    peaks, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks, peak_src = float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy burst)"
    except Exception:
        pass
    traffic = {}
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            traffic = json.load(f)
    except Exception:
        pass

    frames_total = args.frames * world
    f0, f1 = rank * args.frames, (rank + 1) * args.frames
    prob = Problem.synthetic(frames_total, args.beams, seed=SEED, sigma=SIGMA, frame_begin=f0, frame_end=f1, device=local_rank)
    n_frames, n_points, _ = prob.sizes()
    # The simulated laser is two-dimensional, so the library would drop the z stream (16 B per residual).  SURVEY.md 8(d)
    # fixes the contract figure at 24 B per residual: the headline legs run the general three-stream kernels; the planar
    # kernels are reported as their own row (roofline.planar) with their own byte count.
    prob.set_planar_mode(0)
    comm = None
    if world > 1:
        uid = [comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        comm = Comm(uid[0], world, rank, device=local_rank)

        def all_gather(blob):
            out = [None] * world
            dist.all_gather_object(out, blob)
            return out

        if not args.nccl_allreduce:
            try:
                comm.enable_p2p(all_gather)  # fused in-kernel all-reduce over NVLink peer memory
            except Exception:  # no peer access between these GPUs: the NCCL path still works
                args.nccl_allreduce = True
            ok = torch.tensor([0 if args.nccl_allreduce else 1], device="cuda")
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)  # all ranks must use the same mode
            if int(ok.item()) == 0 and not args.nccl_allreduce:
                args.nccl_allreduce = True
                comm.close()
                uid = [comm_unique_id() if rank == 0 else None]
                dist.broadcast_object_list(uid, src=0)
                comm = Comm(uid[0], world, rank, device=local_rank)
        prob.attach_comm(comm)
        # the first collective sweeps after the peer mappings were created are slow (lazy peer-access set-up, cold mailboxes):
        # run them outside every timed region
        for _ in range(20):
            prob.eval(X0)
    opt = default_options()
    total_points = float(sum_over_ranks(float(n_points))[0])

    # ---- resident-data leg: K full solves ----
    for _ in range(args.warmup):
        prob.solve(X0, opt)
    launches0 = launch_count()
    barrier()
    t0 = time.perf_counter()
    dev_ms, sweeps, iters, per_step = 0.0, 0, 0, []
    x = X0
    for _ in range(args.steps):
        x, s, trace = prob.solve(X0, opt)
        dev_ms += s.device_ms
        per_step.append(s.device_ms)
        sweeps += s.num_sweeps
        iters += s.num_iterations - 1
    barrier()
    wall_ms = 1e3 * (time.perf_counter() - t0)
    launches = launch_count() - launches0
    if args.dump_outputs and rank == 0:
        from camlasercalibratool_b200._lib import LmIteration

        dump_solve_outputs(args.dump_outputs, x, s, trace, LmIteration)
    dev_ms = max_over_ranks(dev_ms)
    wall_ms = max_over_ranks(wall_ms)
    value = total_points * sweeps / (dev_ms * 1e-3)
    lm_iters_per_s = iters / (dev_ms * 1e-3)
    step_stats = {"min": float(np.min(per_step)), "median": float(np.median(per_step)), "max": float(np.max(per_step)),
                  "first": float(per_step[0]), "what": "device ms per solve on rank 0"}

    # ---- clocks: the timed region lasts ~20 ms, nvidia-smi samples every 100 ms and needs a second or so before its first line:
    #      keep the device in exactly the timed region's state (the same solves, untimed) for ~2 s so that the sampler sees it ----
    for _ in range(2500):
        prob.solve(X0, opt)
    barrier()

    # ---- check block (outside every timed region): the answer, at this N ----
    check = {}
    cost_c, H_c, g_c = prob.eval(x)  # collective (fused exchange when world > 1)
    if world > 1:
        prob.attach_comm(None)
        cost_l, H_l, g_l = prob.eval(x)  # this shard alone
        prob.attach_comm(comm)
        tot = sum_over_ranks(np.concatenate([[cost_l], H_l.ravel(), g_l]))
        ref = np.concatenate([[cost_c], H_c.ravel(), g_c])
        scale = max(np.abs(H_c).max(), abs(cost_c))
        check["collective_vs_sum_of_shards_rel"] = float(np.abs(tot - ref).max() / scale)
        check["collective_ok"] = bool(check["collective_vs_sum_of_shards_rel"] <= 1e-11)
    with Problem.synthetic(frames_total, args.beams, seed=SEED, sigma=0.0, frame_begin=f0, frame_end=f1, device=local_rank) as clean:
        clean.set_planar_mode(0)
        clean.attach_comm(comm)
        xc, sc, _ = clean.solve(X0, opt)
        ang, dt = pose_error_vs_ground_truth(xc)
        check.update({"noise_free_rot_err_rad": ang, "noise_free_trans_err_m": dt, "noise_free_ok": bool(ang < 1e-9 and dt < 1e-9),
                      "noise_free_iterations": int(sc.num_iterations - 1)})
        clean.attach_comm(None)
    ang_n, dt_n = pose_error_vs_ground_truth(x)
    check.update({"noisy_rot_err_rad": ang_n, "noisy_trans_err_m": dt_n})

    # ---- roofline leg: the sweep kernel alone, L2 flushed between launches (local shard, no collective) ----
    roofline = kernel_row(prob, x, args.kernel_launches, peaks, "clc_sweep_kernel<LOSS,LM> general, 24 B/residual")
    k_b2b = prob.bench_eval(x, args.kernel_launches, flush_l2=False)
    roofline.update({"traffic": traffic.get("dram_bytes_per_launch"), "traffic_source": traffic.get("source"),
                     "peak_source": peak_src,
                     "l2": "flushed between launches (256 MiB written, then read back: no dirty lines left)",
                     "back_to_back_no_flush_ms": float(np.mean(k_b2b))})

    # ---- separate row: the planar (two-stream) kernels the library picks by itself for z == 0 data (16 B/residual) ----
    prob.set_planar_mode(1)
    if prob.planar:
        row = kernel_row(prob, x, args.kernel_launches, peaks, "clc_sweep_kernel<LOSS,LM,PLANAR>, 16 B/residual (own denominator)")
        row["traffic"] = (traffic.get("planar") or {}).get("dram_bytes_per_launch")
        row["speedup_over_24B_kernel"] = roofline["kernel_ms_mean"] / row["kernel_ms_mean"]
        _, srow = solve_row(prob, opt, args.steps, total_points, max_over_ranks, barrier)
        row["full_lm_solve"] = srow
        roofline["planar"] = row
    # the sampler ran from process start over the warm-up, the timed solves and the roofline legs (nvidia-smi needs a second or
    # two before its first line, the timed solves last 20 ms); it stops here: the 48 GB strong-scaling leg below runs into
    # the software power cap and is not what `value` / `roofline` were measured under
    clocks = sampler.stop() if rank == 0 else None

    # ---- strong scaling: BASELINE configs[3] (10^6 frames x 2*10^3 points = 2*10^9 residuals, 48 GB) over the N ranks ----
    strong = None
    if not args.no_strong:
        prob.close()
        prob = None
        SF, SB = args.strong_frames, 2_000
        sf0, sf1 = SF * rank // world, SF * (rank + 1) // world
        with Problem.synthetic(SF, SB, seed=SEED, sigma=SIGMA, frame_begin=sf0, frame_end=sf1, device=local_rank) as big:
            big.set_planar_mode(0)
            big.attach_comm(comm)
            xs, srow = solve_row(big, opt, 3, float(SF) * SB, max_over_ranks, barrier)
            srow["gt_rot_err_rad"], srow["gt_trans_err_m"] = pose_error_vs_ground_truth(xs)
            big.set_planar_mode(1)
            _, prow = solve_row(big, opt, 3, float(SF) * SB, max_over_ranks, barrier)
            big.attach_comm(None)
        strong = {"workload": f"BASELINE configs[3]: {SF} frames x {SB} points, the SAME total problem at every N (frames sharded by rank)",
                  "general_24B": srow, "planar_16B": prow}
    elif prob is not None:
        prob.close()
        prob = None

    # ---- end-to-end leg: std::vector<Oberserve> (pageable, one heap array per frame) -> CamLaserCalibration() of the C++
    #      drop-in (the reference's own signature) on N devices of ONE process; rank 0 runs it, the others stay off the GPUs ----
    e2e, config1 = None, None
    if rank == 0:
        e2e_steps = max(3, min(args.steps, 10))
        dj = run_dropin(frames_total, args.beams, e2e_steps, 3, devices=list(range(world)))
        pts = float(dj["points"])
        e2e = {"value": pts * dj["sweeps_per_call"] / (dj["body_ms_median"] * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": int(dj["h2d_bytes_per_call"]), "d2h_bytes_per_step": int(dj["d2h_bytes_per_call"]),
               "ms_per_step": dj["body_ms_median"], "ms_per_step_mean": dj["body_ms_mean"], "ms_per_step_min": dj["body_ms_min"],
               "ms_per_step_max": dj["body_ms_max"], "steps": e2e_steps,
               "statistic": "median over the steps (the host side shares a 16-CPU container quota with the launcher; single "
                            "steps that hit a scheduler stall are visible in ms_per_step_max / _mean)",
               "what": "C++ drop-in, pageable std::vector<Oberserve> input: CamLaserCalibration() entry to return",
               "phases_ms": dj["phases_ms_median"], "raw_h2d_ms_same_bytes": dj["raw_h2d_ms_same_bytes"],
               "upload_over_raw_h2d": dj["phases_ms_median"]["upload"] / max(dj["raw_h2d_ms_same_bytes"], 1e-9),
               "sweeps_per_call": dj["sweeps_per_call"], "n_devices": dj["n_devices"], "pack_threads": dj["pack_threads"],
               "call_expr_moved_ms": dj["call_expr_moved_ms_median"], "call_expr_lvalue_ms": dj["call_expr_lvalue_ms_median"],
               "caller_copy_of_obs_ms": dj["caller_copy_of_obs_ms"], "caller_destruction_of_obs_ms": dj["caller_destruction_of_obs_ms"],
               "by_value_note": "call_expr_* add what the reference's by-value signature makes the CALLER do (deep copy / destruction "
                                "of the vector<Oberserve>); identical for the reference, none of it library code",
               "max_abs_dev_vs_c_abi_solve": dj["max_abs_dev_vs_c_abi_solve"], "rc": dj["rc"]}
        if world == 1:
            c1 = run_dropin(50, 180, 20, 3, devices=[0], seed=1)
            config1 = {"workload": "BASELINE configs[0]: 50 frames x 180 beams through the C++ drop-in",
                       "body_ms": c1["body_ms_mean"], "call_expr_lvalue_ms": c1["call_expr_lvalue_ms_median"],
                       "lm_device_ms": c1["lm_device_ms"], "lm_iterations": c1["lm_iterations"], "phases_ms": c1["phases_ms_median"]}
            e2e["config1"] = config1
    if world > 1:
        dist.barrier(group=cpu_group)

    # ---- supplementary rows (one GPU): BASELINE configs[2] and configs[4] ----
    if world == 1 and not args.no_config3:
        with Problem.synthetic(100_000, 2_000, seed=SEED, sigma=SIGMA, device=local_rank) as big:
            big.set_planar_mode(0)  # contract row first (24 B per residual)
            r3 = kernel_row(big, x, 20, peaks, "general, 24 B/residual")
            _, r3["full_lm_solve"] = solve_row(big, opt, 2, 2e8, max_over_ranks, barrier)
            big.set_planar_mode(1)
            r3p = kernel_row(big, x, 20, peaks, "planar, 16 B/residual")
            _, r3p["full_lm_solve"] = solve_row(big, opt, 2, 2e8, max_over_ranks, barrier)
            r3["traffic"] = (traffic.get("config3") or {}).get("dram_bytes_per_launch")
            r3p["traffic"] = ((traffic.get("config3") or {}).get("planar") or {}).get("dram_bytes_per_launch")
            r3["planar"] = r3p
            r3["workload"] = "BASELINE configs[2]: 100000 frames x 2000 points (4.8 GB)"
            roofline["config3"] = r3
        with Problem.synthetic(100_000, 2_000, seed=SEED, sigma=SIGMA, with_edges=True, camera="equi", pixel_sigma=0.3,
                               device=local_rank) as c5:
            c5.set_planar_mode(0)
            r5 = kernel_row(c5, x, 20, peaks, "general + edge tail, 24 B/residual + 56 B/edge residual")
            x5, r5["full_lm_solve"] = solve_row(c5, opt, 2, 2e8 + 2e5, max_over_ranks, barrier)
            r5["gt_rot_err_rad"], r5["gt_trans_err_m"] = pose_error_vs_ground_truth(x5)
            c5.set_planar_mode(1)
            r5p = kernel_row(c5, x, 20, peaks, "planar + edge tail, 16 B/residual + 56 B/edge residual")
            r5["traffic"] = (traffic.get("config5") or {}).get("dram_bytes_per_launch")
            r5["planar"] = r5p
            r5["workload"] = ("BASELINE configs[4]: 100000 frames x 2000 points + 200000 board-edge residuals, board poses from "
                              "the equidistant (Kannala-Brandt) camera chain with 0.3 px corner noise")
            roofline["config5"] = r5

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(args.frames, args.beams)
    if world > 1:
        dist.barrier(group=cpu_group)

    if rank == 0:
        cfg = workload_config(args, world)
        cfg.update({"sharding": (f"frames by rank, {world} ranks, 28-double all-reduce per sweep: " +
                                 ("ncclAllReduce between kernels" if args.nccl_allreduce else
                                  "fused into the sweep kernel (NVLink peer stores, rank-order sum)")) if world > 1 else "single GPU",
                    "l2": f"inputs ({roofline['algorithmic_bytes_per_launch'] / 1e6:.0f} MB/GPU) > 126 MB L2; roofline leg also flushes L2 between launches",
                    "lm": "one fused residual+Jacobian+reduce sweep per LM iteration",
                    "kernels": "general three-stream kernels (24 B/residual contract row); planar rows separate",
                    "check": check, "strong_scaling": strong, "step_device_ms": step_stats})
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": len(per_step), "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": cfg,
            "lm_iters_per_s": lm_iters_per_s, "sweeps_per_solve": sweeps / args.steps, "lm_iterations_per_solve": iters / args.steps,
            "wall_ms_per_step": wall_ms / args.steps, "value_on_wall_clock": total_points * sweeps / (wall_ms * 1e-3),
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "clocks": clocks,
            "gpu_launches": int(launches),
        }
        print(json.dumps(line))
    if comm is not None:
        comm.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return
    _, _, world = dist_env()
    if args.gpus > 1 and world == 1 and "RANK" not in os.environ:
        # convenience: self-launch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    run_ours(args)


if __name__ == "__main__":
    main()
