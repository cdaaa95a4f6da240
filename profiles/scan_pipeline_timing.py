"""Raw LaserScan ranges -> the two calibration problems -> closed form -> LM: the device path
(api.problems_from_scans, one upload of the ranges) against the host chain (formats.segments_from_scans ->
observations_from_segments -> CamLaserCalClosedSolution / CamLaserCalibration), in one process, alternating.

    python profiles/scan_pipeline_timing.py [out.json]

Sessions come from the seeded ray-caster of tests/test_scan_problems.py: 1081-beam scans at 40 Hz, tag poses at 20 Hz,
the board redrawn every 8 poses (key-frame thinning keeps about one pose in 8).  Phase times of problems_from_scans are
CUDA events inside the library (clc_scan_last_stats); everything else is host wall clock around synchronous calls."""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from camlasercalibratool_b200 import api, formats as fmt  # noqa: E402
from camlasercalibratool_b200.api import pinned_array  # noqa: E402
from oracle import oracle as O  # noqa: E402
import test_scan_problems as gen  # noqa: E402


def device_path(tagpose, stamps, ranges):
    t0 = time.perf_counter()
    kf = fmt.select_keyframes(tagpose)
    tp, pw = gen._pose_arrays(kf)
    t1 = time.perf_counter()
    pts, onl, _, _ = api.problems_from_scans(ranges, stamps, gen.A0, gen.INC, gen.RMIN, tp, pw)
    t2 = time.perf_counter()
    stats = api.scan_stats()
    with pts, onl:
        Tlc0 = np.eye(4)
        api.closed_form_on(onl, Tlc0, verbose=False)
        t3 = time.perf_counter()
        Tcl = np.linalg.inv(Tlc0)
        rep = api.calibrate_on(pts, Tcl, verbose=False)
        t4 = time.perf_counter()
        nf, npts, _ = pts.sizes()
        planar = pts.planar
    return dict(keyframes_ms=1e3 * (t1 - t0), problems_from_scans_ms=1e3 * (t2 - t1), closed_form_ms=1e3 * (t3 - t2),
                lm_and_information_ms=1e3 * (t4 - t3), total_ms=1e3 * (t4 - t0), phases=stats, n_frames=nf, n_points=npts,
                planar=bool(planar), lm_iterations=rep["iterations"], Tlc=np.linalg.inv(Tcl))


def host_path(tagpose, stamps, ranges):
    t0 = time.perf_counter()
    segs = fmt.segments_from_scans(stamps, ranges, gen.A0, gen.INC, gen.RMIN)
    t1 = time.perf_counter()
    obs = fmt.observations_from_segments(fmt.select_keyframes(tagpose), segs)
    t2 = time.perf_counter()
    Tlc0 = np.eye(4)
    api.CamLaserCalClosedSolution(obs, Tlc0, verbose=False)
    t3 = time.perf_counter()
    Tcl = np.linalg.inv(Tlc0)
    rep = api.CamLaserCalibration(obs, Tcl, False, verbose=False)
    t4 = time.perf_counter()
    n_pts = sum(len(o.points) for o in obs)
    return dict(segments_from_scans_ms=1e3 * (t1 - t0), observations_ms=1e3 * (t2 - t1), closed_form_ms=1e3 * (t3 - t2),
                lm_and_information_ms=1e3 * (t4 - t3), total_ms=1e3 * (t4 - t0), n_frames=len(obs), n_points=n_pts,
                lm_iterations=rep["iterations"], Tlc=np.linalg.inv(Tcl),
                # ranges once, then every segment point twice at 24 B (line fit upload, LM upload) + the end points
                bytes_h2d=int(ranges.nbytes + 24 * 2 * n_pts + 48 * len(obs)))


def gpu_identity():
    import torch

    out = dict(device=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        out["nvidia_smi"] = q
    except Exception as exc:  # the query is informational
        out["nvidia_smi"] = f"not available: {exc}"
    return out


def med(rows, key):
    return float(np.median([r[key] for r in rows]))


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "scan_pipeline_timing.json")
    O.build()
    result = dict(gpu=gpu_identity(), sizes=[])
    for name, n_poses, reps in (("session_5e3_scans", 2500, 5), ("batch_1e5_scans", 50000, 3)):
        tagpose, stamps, ranges = gen._session(O, n_poses, seed=21, hold=8)
        dev, host, pinned = [], [], []
        buf = pinned_array(ranges.shape, np.float32)
        buf.array[...] = ranges
        device_path(tagpose, stamps, ranges)  # warm-up (module load, memory pool)
        for _ in range(reps):
            dev.append(device_path(tagpose, stamps, ranges))
            host.append(host_path(tagpose, stamps, ranges))
            pinned.append(device_path(tagpose, stamps, buf.array))
        buf.free()
        d, h = dev[-1], host[-1]
        assert d["n_frames"] == h["n_frames"] and d["n_points"] == h["n_points"], (d["n_frames"], h["n_frames"])
        row = dict(
            name=name, n_scans=int(ranges.shape[0]), n_beams=int(ranges.shape[1]), ranges_MB=ranges.nbytes / 1e6,
            n_poses=n_poses, n_keyframes=len(fmt.select_keyframes(tagpose)), n_frames=d["n_frames"], n_points=d["n_points"],
            planar=d["planar"], reps=reps,
            device_pageable=dict(total_ms=med(dev, "total_ms"), keyframes_ms=med(dev, "keyframes_ms"),
                                 problems_from_scans_ms=med(dev, "problems_from_scans_ms"),
                                 phases_ms={k: float(np.median([r["phases"][k] for r in dev])) for k in dev[0]["phases"] if k.endswith("_ms")},
                                 closed_form_ms=med(dev, "closed_form_ms"), lm_and_information_ms=med(dev, "lm_and_information_ms"),
                                 bytes_h2d=dev[-1]["phases"]["bytes_h2d"], bytes_d2h=dev[-1]["phases"]["bytes_d2h"]),
            device_pinned=dict(total_ms=med(pinned, "total_ms"), problems_from_scans_ms=med(pinned, "problems_from_scans_ms"),
                               phases_ms={k: float(np.median([r["phases"][k] for r in pinned])) for k in pinned[0]["phases"] if k.endswith("_ms")}),
            host_chain=dict(total_ms=med(host, "total_ms"), segments_from_scans_ms=med(host, "segments_from_scans_ms"),
                            observations_ms=med(host, "observations_ms"), closed_form_ms=med(host, "closed_form_ms"),
                            lm_and_information_ms=med(host, "lm_and_information_ms"), bytes_h2d=h["bytes_h2d"]),
            speedup_total=med(host, "total_ms") / med(dev, "total_ms"),
            max_abs_Tlc_difference=float(np.abs(d["Tlc"] - h["Tlc"]).max()),
            lm_iterations=(d["lm_iterations"], h["lm_iterations"]),
        )
        result["sizes"].append(row)
        print(json.dumps(row), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["gpu"]))


if __name__ == "__main__":
    main()
