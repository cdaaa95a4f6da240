"""bench.py's reference arm runs on the CPU (it times the oracle port), so its JSON contract can be checked here:
one line, the keys the driver reads, the metric/unit of BASELINE.json, `impl: reference`, zero-byte e2e."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--frames", "200",
                                   "--beams", "100", "--steps", "2", "--warmup", "1"], text=True, timeout=600, cwd=ROOT)
    lines = [ln for ln in out.splitlines() if ln.strip().startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert d["impl"] == "reference" and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["dtype"] == "f64" and d["data"] == "synthetic"
    assert d["value"] > 0 and d["unit"] == "residual evals/s" and "workload" in d["config"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"] and cb["cores"] >= 1 and cb["sample"]
    # the metric is the one BASELINE.json names
    assert "residual" in d["metric"].lower() and "residual" in json.dumps(base).lower()


def test_both_arms_print_the_same_config():
    """The driver compares the two arms' `config`: both come from one function (the reference arm's bounded sample is described
    in its cpu_baseline.sample, not in config)."""
    sys.path.insert(0, ROOT)
    import argparse

    import bench

    a = argparse.Namespace(frames=10_000, beams=1_000)
    c = bench.workload_config(a, 1)
    assert set(c) == {"workload"} and "10000 frames x 1000 points" in c["workload"]
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert src.count("workload_config(args, world)") == 3  # the definition + run_reference + run_ours


def test_ground_truth_pose_error_is_accurate_near_zero():
    """bench.py's check block measures the distance to the generator's ground truth: it must resolve 1e-12 rad (an arccos of
    the trace would stop at 1e-8)."""
    sys.path.insert(0, ROOT)
    import numpy as np

    import bench
    from oracle import oracle as O

    gt = O.ground_truth()[1]
    ang, dt = bench.pose_error_vs_ground_truth(gt)
    assert ang < 1e-15 and dt < 1e-15
    x = O.pose_plus(gt, np.array([0, 0, 1e-9, 2e-12, 0, 0]))
    ang, dt = bench.pose_error_vs_ground_truth(x)
    assert abs(ang - 2e-12) < 1e-14 and abs(dt - 1e-9) < 1e-14


def test_dump_outputs_writes_what_solve_returned(tmp_path):
    """--dump-outputs: one float64 .npy per returned quantity, the timing and padding fields left out."""
    sys.path.insert(0, ROOT)
    import numpy as np

    import bench
    from camlasercalibratool_b200._lib import LmIteration, LmSummary

    x = np.array([0.1, 0.2, 0.3, 0.0, 0.0, 0.6, 0.8])
    s = LmSummary(termination=1, num_iterations=2, num_successful_steps=2, num_sweeps=3, initial_cost=5.0,
                  final_cost=0.25, device_ms=1.5)
    tr = [LmIteration(iteration=i, step_is_successful=1, cost=c, trust_region_radius=1e4 * 3**i) for i, c in enumerate((5.0, 0.25))]
    bench.dump_solve_outputs(str(tmp_path / "out"), x, s, tr, LmIteration)
    got = {f[:-4]: np.load(tmp_path / "out" / f) for f in os.listdir(tmp_path / "out")}
    assert all(a.dtype == np.float64 for a in got.values())
    assert not any("device_ms" in k or "reserved" in k for k in got)
    np.testing.assert_array_equal(got["pose7"], x)
    assert got["summary_termination"] == 1 and got["summary_num_sweeps"] == 3 and got["summary_final_cost"] == 0.25
    np.testing.assert_array_equal(got["trace_cost"], [5.0, 0.25])
    np.testing.assert_array_equal(got["trace_trust_region_radius"], [1e4, 3e4])
    np.testing.assert_array_equal(got["trace_iteration"], [0, 1])


@pytest.mark.gpu
def test_dump_outputs_of_the_cuda_arm_are_the_solve_and_repeat(tmp_path):
    """`bench.py --dump-outputs`: --steps timed solves (`steps` counts the solves of the timed loop), the last one's result on
    disk, identical in a second run, and equal to a direct Problem.solve of the same seeded workload."""
    sys.path.insert(0, ROOT)
    import numpy as np

    import bench
    from camlasercalibratool_b200 import Problem, default_options

    frames, beams = 300, 200
    dumps = []
    for run in range(2):
        out = tmp_path / f"run{run}"
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "1",
                              "--frames", str(frames), "--beams", str(beams), "--kernel-launches", "5", "--no-cpu-baseline",
                              "--no-config3", "--no-strong", "--dump-outputs", str(out)],
                             capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert res.returncode == 0, res.stderr[-2000:]
        lines = [ln for ln in res.stdout.splitlines() if ln.strip().startswith("{")]
        assert len(lines) == 1 and json.loads(lines[0])["steps"] == 3
        dumps.append({f[:-4]: np.load(out / f) for f in os.listdir(out)})
    assert dumps[0].keys() == dumps[1].keys()
    for k in dumps[0]:
        np.testing.assert_array_equal(dumps[0][k], dumps[1][k], err_msg=k)
    d = dumps[0]
    with Problem.synthetic(frames, beams, seed=bench.SEED, sigma=bench.SIGMA) as p:
        p.set_planar_mode(0)
        x, s, tr = p.solve(bench.X0, default_options())
    np.testing.assert_array_equal(d["pose7"], x)
    assert d["summary_num_iterations"] == s.num_iterations == len(d["trace_cost"])
    np.testing.assert_array_equal(d["trace_cost"], [t.cost for t in tr])


def test_reference_arm_dumps_the_oracle_solve_under_the_same_names(tmp_path):
    sys.path.insert(0, ROOT)
    import numpy as np

    import bench
    from camlasercalibratool_b200._lib import LmIteration
    from oracle import oracle as O

    out = tmp_path / "out"
    subprocess.check_call([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--frames", "200", "--beams",
                           "100", "--steps", "2", "--warmup", "1", "--dump-outputs", str(out)],
                          stdout=subprocess.DEVNULL, timeout=600, cwd=ROOT)
    got = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert all(a.dtype == np.float64 for a in got.values())
    assert {k for k in got if k.startswith("trace_")} == {"trace_" + n for n, _ in LmIteration._fields_ if n != "reserved"}
    x, s, tr = O.solve(bench.cpu_reference_problem(200, 100), bench.X0)
    ang, dt = O.pose_error(got["pose7"], x)  # the timed solves may evaluate on several threads: summation order only
    assert ang < 1e-12 and dt < 1e-12
    assert got["summary_num_iterations"] == s.num_iterations == len(got["trace_cost"])
    assert got["summary_termination"] == s.termination
    np.testing.assert_allclose(got["trace_cost"], [t.cost for t in tr], rtol=1e-12)


def test_reference_arm_runs_exactly_steps_solves(monkeypatch, capsys):
    """--steps N times N solves however long each takes (no wall-clock cut-off); --steps 0 is refused."""
    sys.path.insert(0, ROOT)
    import bench

    solves = []

    def slow_solve(p, threads, linear_solver):
        solves.append(threads)
        return 100.0, 10**6, 5, None  # 100 s per solve

    monkeypatch.setattr(bench, "cpu_reference_problem", lambda n, beams: None)
    monkeypatch.setattr(bench, "pick_threads", lambda p: 1)
    monkeypatch.setattr(bench, "time_cpu_solve", slow_solve)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--steps", "5", "--warmup", "2"])
    bench.main()
    d = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert d["steps"] == 5 and len(solves) == 2 + 5 and d["ms_per_step"] == 1e5
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "0"])
    with pytest.raises(SystemExit):
        bench.parse_args()


def test_reference_arm_under_torchrun_only_rank0_works():
    """`bench.py --impl reference` launched with N ranks: rank 0 alone runs and prints, the others exit 0 without work."""
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert res.returncode == 0 and res.stdout.strip() == ""
