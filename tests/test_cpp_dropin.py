"""The C++ drop-in (camlasercalibratool_b200/host/LaseCamCalB200.cpp) behind the reference's own signatures.
CPU: it compiles against the reference interface (Eigen stand-in) and links against libclc_b200.so.
GPU: a C++ caller shaped like calibr_simulation.cpp / calibr_offline.cpp gets the oracle's T_cl."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def build_driver(out_dir):
    from camlasercalibratool_b200 import _build, _lib

    _lib.load()
    exe = os.path.join(out_dir, "host_dropin_test")
    # against the reference's own include/LaseCamCalCeres.h when CLC_REFERENCE_INCLUDE names it, else the stand-in
    subprocess.check_call(_build.cxx_command([os.path.join(ROOT, "tests", "host_dropin_test.cpp"), _build.DROPIN_SRC], exe))
    return exe


def test_dropin_compiles_against_the_reference_header_when_present(tmp_path, monkeypatch):
    from camlasercalibratool_b200 import _build

    stubs = os.path.join(ROOT, "tests", "stubs")
    monkeypatch.delenv("CLC_REFERENCE_INCLUDE", raising=False)
    assert _build.interface_include_dirs()[0] == stubs
    ref = tmp_path / "include"
    ref.mkdir()
    monkeypatch.setenv("CLC_REFERENCE_INCLUDE", str(ref))  # no header there: the stand-in stays
    assert _build.interface_include_dirs()[0] == stubs
    # a directory with the interface header wins over tests/stubs/LaseCamCalCeres.h, and the drop-in builds against it; the
    # probe lives outside that directory, so only the include path can lead it to the marked header
    with open(os.path.join(stubs, "LaseCamCalCeres.h")) as f:
        header = f.read()
    (ref / "LaseCamCalCeres.h").write_text("#define CLC_TEST_REFERENCE_HEADER_USED 1\n" + header)
    assert _build.interface_include_dirs()[0] == str(ref)
    probe = tmp_path / "probe.cpp"
    probe.write_text('#include "LaseCamCalCeres.h"\n#ifndef CLC_TEST_REFERENCE_HEADER_USED\n#error stand-in header used\n#endif\n')
    for src in (str(probe), _build.DROPIN_SRC):
        subprocess.check_call(_build.cxx_command([src], str(tmp_path / "obj.o"), extra=("-c",)))


def test_bench_driver_builds():
    from camlasercalibratool_b200 import _build

    exe = _build.build_dropin_bench(force=True)
    out = subprocess.check_output(["nm", "-C", "--defined-only", exe], text=True)
    assert "CamLaserCalibration(" in out


def test_dropin_compiles_and_links(tmp_path):
    exe = build_driver(str(tmp_path))
    out = subprocess.check_output(["nm", "-C", "--defined-only", exe], text=True)
    for sym in ("CamLaserCalibration(", "CamLaserCalClosedSolution(", "LineFittingCeres(", "CalibrationTool_SavePlanePoints("):
        assert sym in out, sym


def _matrices(text):
    res = {}
    for line in text.splitlines():
        if line.startswith("RESULT_"):
            tag, *vals = line.split()
            res[tag] = np.array([float(v) for v in vals]).reshape(4, 4)
    return res


@pytest.mark.gpu
@pytest.mark.parametrize("sigma,edges", [(0.0, 0), (0.01, 0), (0.01, 1)])
def test_dropin_matches_oracle(oracle, tmp_path, sigma, edges):
    exe = build_driver(str(tmp_path))
    out = subprocess.check_output([exe, "50", "180", str(sigma), str(edges)], text=True, timeout=120)
    assert "Termination: CONVERGENCE" in out and "recover chi2" in out and "Closed-form solution Tlc" in out
    m = _matrices(out)
    p = oracle.generate(50, 180, seed=1, sigma=sigma, exact_m=True, with_edges=bool(edges))
    x0 = np.array([0, 0, 0, 0, 0, 0, 1.0])
    plain = oracle.Problem(p.frame_pose, p.offsets, p.points)
    if edges:  # the driver overwrote points.front()/back() with the edge points, as the reference would read them
        pts = p.points.copy()
        pts[p.offsets[:-1]] = p.edge_points[:, :3]
        pts[p.offsets[1:] - 1] = p.edge_points[:, 3:]
        plain = oracle.Problem(p.frame_pose, p.offsets, pts)
    xs, _, _ = oracle.solve(plain, x0)
    np.testing.assert_allclose(m["RESULT_SIM_TCL"], oracle.pose7_to_T(xs), atol=1e-8)
    # closed form on points_on_line (= the untouched points in the driver)
    Tlc, _, _, _ = oracle.closed_form(oracle.Problem(p.frame_pose, p.offsets, p.points))
    np.testing.assert_allclose(m["RESULT_CLOSED_TLC"], Tlc, atol=1e-8)
    xo, _, _ = oracle.solve(plain, oracle.T_to_pose7(np.linalg.inv(m["RESULT_CLOSED_TLC"])))
    np.testing.assert_allclose(m["RESULT_OFFLINE_TCL"], oracle.pose7_to_T(xo), atol=1e-8)
    if sigma == 0.0:
        gtT, gt = oracle.ground_truth()
        np.testing.assert_allclose(np.linalg.inv(m["RESULT_SIM_TCL"]), gtT, atol=1e-8)
    if edges:
        pe = oracle.Problem(p.frame_pose, p.offsets, p.points, p.edge_points)
        xe, _, _ = oracle.solve(pe, oracle.T_to_pose7(np.linalg.inv(m["RESULT_CLOSED_TLC"])))
        np.testing.assert_allclose(m["RESULT_EDGES_TCL"], oracle.pose7_to_T(xe), atol=1e-8)
