"""The offline driver's scan loop on the device (clc_problems_create_from_scans; reference main/calibr_offline.cpp:86-155):
LaserScan ranges + tag poses -> the points problem and the on-line problem, against the host chain
observations_from_segments(select_keyframes(tagpose), segments_from_scans(...)) -> Problem.from_observations."""
import ctypes as C
import math

import numpy as np
import pytest

A0, INC = -3 * math.pi / 4, (3 * math.pi / 2) / 1080  # 1081 beams over 270 degrees
RMIN = 0.05
BOARD = (-0.042, 0.458)  # the board square in the tag frame (corners of the reference's edge residuals)


# ---- a seeded ray-caster ------------------------------------------------------------------------------------------------
def _session(oracle, n_poses, seed=0, sigma=0.003, drop=0.01, board=True, hold=1):
    """Tag poses at 20 Hz and 1081-beam scans at 40 Hz.  Board orientations are oracle.generate's draw (yaw, pitch, roll
    within 30 degrees); its position is redrawn 0.7-1.4 m in front of the camera so that the scan plane of
    oracle.ground_truth()'s T_lc crosses it.  Every scan sees the board of the pose it is nearest to, in a room whose walls
    are 3.5-6.5 m away; odd scans lie 21 / 29 ms from the neighbouring poses, so only even ones can be matched.  hold > 1:
    the board is redrawn every `hold` poses and only moves by up to 1 cm in between, so that key-frame thinning keeps about
    one pose in `hold` (a real session).  Returns (tagpose, scan_stamps, ranges float32)."""
    from camlasercalibratool_b200 import formats as fmt

    rng = np.random.default_rng(seed)
    Tlc, _ = oracle.ground_truth()
    Rlc, tlc = Tlc[:3, :3], Tlc[:3, 3]
    qca = oracle.generate(n_poses, 1, seed=seed + 1).frame_pose[:, :4].copy() if n_poses else np.zeros((0, 4))
    tagpose = []
    board_pose = []
    centre = np.array([0.208, 0.208, 0.0])
    for k in range(n_poses):
        Rca = oracle.quat_to_rot(qca[k - k % hold])
        if k % hold == 0:
            tca = np.array([rng.uniform(-0.4, 0.4), 0.0, rng.uniform(0.7, 1.4)])
            tca[1] = 0.3 - (Rca @ centre)[1] + rng.uniform(-0.12, 0.12)  # the scan plane is y_c = 0.3
            tca[0] -= (Rca @ centre)[0]
            t0 = tca
        else:
            tca = t0 + rng.uniform(-0.005, 0.005, 3)
        board_pose.append((Rca, tca))
        qwc = fmt.quat_inverse(qca[k - k % hold])
        tagpose.append(fmt.CamPose(100.0 + 0.05 * k, qwc, -fmt.quat_to_rot(qwc) @ tca))
    n_scans = 2 * n_poses
    stamps = 100.0 + 0.025 * np.arange(n_scans) + 0.004
    ang = A0 + np.arange(1081) * INC
    d = np.stack([np.cos(ang), np.sin(ang), np.zeros_like(ang)])
    ranges = np.empty((n_scans, 1081), dtype=np.float32)
    for j in range(n_scans):
        r = 5.0 + 1.5 * np.sin(3 * ang + rng.uniform(0, 6))
        if board:
            Rca, tca = board_pose[j // 2]
            Rla, tla = Rlc @ Rca, Rlc @ tca + tlc
            n = Rla[:, 2]
            den = n @ d
            with np.errstate(divide="ignore", invalid="ignore"):
                lam = (n @ tla) / den
                pa = Rla.T @ (lam * d - tla[:, None])
            hit = (lam > 0) & (np.abs(den) > 1e-9) & (pa[0] >= BOARD[0]) & (pa[0] <= BOARD[1]) & (pa[1] >= BOARD[0]) & (pa[1] <= BOARD[1])
            r = np.where(hit & (lam < r), lam, r)
        if sigma:
            r = r + rng.normal(size=r.shape) * sigma
        r = r.astype(np.float32)
        if drop:
            r[rng.random(r.shape) < drop] = np.inf
        ranges[j] = r
    return tagpose, stamps, ranges


def _pose_arrays(poses):
    return (np.array([p.timestamp for p in poses]),
            np.array([np.concatenate([p.qwc, p.twc]) for p in poses]).reshape(-1, 7))


def _host_chain(tagpose, stamps, ranges, with_edges=False):
    from camlasercalibratool_b200 import Problem
    from camlasercalibratool_b200 import formats as fmt

    segs = fmt.segments_from_scans(stamps, ranges, A0, INC, RMIN)
    obs = fmt.observations_from_segments(fmt.select_keyframes(tagpose), segs)
    return obs, Problem.from_observations(obs, False, False), Problem.from_observations(obs, True, with_edges)


def _nearest_restated(pose_t, t):
    """main/calibr_offline.cpp:103-116, literally."""
    min_dt, best = 10000.0, -1
    for i, pt in enumerate(pose_t):
        d = abs(pt - t)
        if d < min_dt:
            min_dt, best = d, i
    return best, min_dt


POSES = [np.array([0.1, 0.2, 0.3, 1.0, 0.5, -0.2, 1.5]), np.array([0.3, -0.5, 0.1, 0.8, -1.0, 2.0, 0.3])]


# ---- CPU tier: the host build of the CLC_HD helpers ------------------------------------------------------------------------
def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


@pytest.fixture(scope="module")
def scan_harness(tmp_path_factory):
    """tests/scan_harness.cpp (the CLC_HD helpers of csrc/clc_scans.cuh) compiled with g++ for the host."""
    import os
    import subprocess

    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "scan_harness.cpp")
    out = str(tmp_path_factory.mktemp("scan_harness") / "libclc_scan_harness.so")
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    subprocess.check_call([cxx, "-O2", "-std=c++17", "-Wno-unknown-pragmas", "-shared", "-fPIC", "-o", out, src])
    L = C.CDLL(out)
    dp = C.POINTER(C.c_double)
    L.harness_nearest_pose.restype = C.c_int64
    L.harness_nearest_pose.argtypes = [dp, C.c_int64, C.c_double, dp]
    L.harness_tag_to_frame_pose.argtypes = [dp, dp]
    L.harness_line_end_points.argtypes = [C.c_double, C.c_double, C.c_double, C.c_double, dp, dp]
    return L


def test_nearest_pose_is_the_reference_linear_search(scan_harness):
    L = scan_harness
    rng = np.random.default_rng(1)
    cases = []
    for _ in range(300):
        n = int(rng.choice([0, 1, 2, 7, 50, 300]))
        s = rng.uniform(0, 10, n)
        kind = int(rng.integers(0, 4))
        if kind == 1 and n > 2:  # ties: repeated stamps at different indices
            s[rng.integers(0, n, n // 2)] = s[0]
        if kind == 2 and n:
            s[rng.random(n) < 0.3] = np.nan
        if kind == 3:
            s = np.sort(s)
        t = float(rng.choice([rng.uniform(-1, 11), s[0] if n else 0.0, np.nan]))
        cases.append((s, t))
    # equidistant on both sides (exactly representable): the lower index wins
    cases.append((np.array([2.0, 1.0, 3.0]), 2.5))
    cases.append((np.array([3.0, 1.0, 2.0]), 2.5))
    cases.append((np.array([20000.0]), 0.0))  # beyond the 10000 start value: no pose
    for s, t in cases:
        s = np.ascontiguousarray(s, dtype=np.float64)
        md = C.c_double()
        got = L.harness_nearest_pose(_dp(s), len(s), t, C.byref(md))
        want, want_dt = _nearest_restated(s, t)
        assert got == want and md.value == want_dt, (s, t)
    # the keep rule is strict: dt == max_dt drops the scan (stamps exactly representable)
    s = np.array([1.0, 1.5])
    for t, keep in ((1.015625, False), (1.0078125, True), (0.984375, False)):
        md = C.c_double()
        k = L.harness_nearest_pose(_dp(s), 2, t, C.byref(md))
        assert k == 0 and (md.value < 0.015625) == keep


def test_tag_to_frame_pose_matches_eigen_restatement(scan_harness):
    from camlasercalibratool_b200 import formats as fmt

    L = scan_harness
    rng = np.random.default_rng(2)
    for _ in range(200):
        q = rng.normal(size=4) * rng.choice([1.0, 0.3, 3.0])  # not normalised: Eigen's inverse divides by squaredNorm
        pw = np.concatenate([q, rng.uniform(-3, 3, 3)])
        fp = np.empty(7)
        L.harness_tag_to_frame_pose(_dp(pw), _dp(fp))
        qca = fmt.quat_inverse(q)
        tca = -fmt.quat_to_rot(qca) @ pw[4:]
        np.testing.assert_allclose(fp[:4], qca, rtol=0, atol=1e-15)
        np.testing.assert_allclose(fp[4:], tca, rtol=0, atol=1e-15 * max(1.0, np.abs(tca).max()))


def test_line_end_points_follow_the_driver_rule(scan_harness):
    L = scan_harness
    rng = np.random.default_rng(3)
    branches = set()
    for _ in range(400):
        xs, ys, xe, ye = rng.uniform(-2, 2, 4)
        line = np.ascontiguousarray(rng.normal(size=2))
        out = np.empty(4)
        L.harness_line_end_points(xs, ys, xe, ye, _dp(line), _dp(out))
        # formats.observations_from_segments, :126-142
        x_s, x_e, y_s, y_e = xs, xe, ys, ye
        if abs(x_e - x_s) > abs(y_e - y_s):
            y_s = -(x_s * line[0] + 1) / line[1]
            y_e = -(x_e * line[0] + 1) / line[1]
            branches.add("x")
        else:
            x_s = -(y_s * line[1] + 1) / line[0]
            x_e = -(y_e * line[1] + 1) / line[0]
            branches.add("y")
        np.testing.assert_array_equal(out, [x_s, y_s, x_e, y_e])
    assert branches == {"x", "y"}


def test_offline_from_scans_refuses_few_poses():
    """reference main/calibr_offline.cpp:55-59: the refusal comes before any device work."""
    from camlasercalibratool_b200 import formats as fmt

    poses = [fmt.CamPose(0.1 * i, np.array([0, 0, 0, 1.0]), np.zeros(3)) for i in range(9)]
    Tlc, why = fmt.calibrate_offline_from_scans(poses, np.zeros(0), np.zeros((0, 1081), np.float32), A0, INC, RMIN)
    assert Tlc is None and why == "apriltag pose less than 10."


def _raw_create(**over):
    from camlasercalibratool_b200 import _lib

    L = _lib.load()
    r = np.ones((2, 100), dtype=np.float32)
    ts = np.zeros(2)
    tp, pw = np.zeros(1), np.array([[0, 0, 0, 1.0, 0, 0, 0]])
    d = _lib.ScanDesc()
    d.n_scans, d.n_beams, d.ranges, d.scan_stamp = 2, 100, r.ctypes.data_as(C.POINTER(C.c_float)), ts.ctypes.data_as(_lib.c_double_p)
    d.angle_min, d.angle_increment, d.range_min = A0, INC, RMIN
    d.n_poses, d.pose_stamp, d.pose_wc = 1, tp.ctypes.data_as(_lib.c_double_p), pw.ctypes.data_as(_lib.c_double_p)
    d.max_dt, d.line_fit_max_iterations, d.with_edges, d.use_loss, d.cauchy_a, d.device = 0.02, 10, 0, 1, 0.05, -1
    for k, v in over.items():
        setattr(d, k, v)
    hp, hl = C.c_void_p(0x10), C.c_void_p(0x20)  # sentinels: must come back NULL
    rc = L.clc_problems_create_from_scans(C.byref(d), C.byref(hp), C.byref(hl), None, None)
    return rc, L.clc_last_error().decode(), hp.value, hl.value, (r, ts, tp, pw)


@pytest.mark.parametrize("over", [
    dict(ranges=None), dict(scan_stamp=None), dict(pose_stamp=None), dict(pose_wc=None), dict(n_beams=(1 << 31)),
    dict(angle_increment=float("nan")), dict(angle_increment=float("inf")), dict(max_dt=0.0), dict(max_dt=-1.0),
    dict(max_dt=float("nan")), dict(cauchy_a=0.0), dict(cauchy_a=-1.0), dict(n_scans=-1), dict(n_poses=-2),
    dict(line_fit_max_iterations=-1)])
def test_invalid_scan_arguments_are_refused(over):
    """Argument checks come before any CUDA call: status CLC_ERR_INVALID, a message, both outputs NULL."""
    rc, msg, hp, hl, _ = _raw_create(**over)
    assert rc == 1 and msg and hp is None and hl is None


# ---- GPU tier -------------------------------------------------------------------------------------------------------------
def _bitwise_eval_equal(p, use_edges=False):
    from camlasercalibratool_b200 import Problem

    d = p.download()
    with Problem.from_arrays(d["frame_pose"], d["offsets"], d["points"], d["edge_points"] if use_edges else None) as q:
        assert q.planar == p.planar
        for pose in ([0, 0, 0, 0, 0, 0, 1.0], [0.1, -0.2, 0.05, 0.01, 0.7, -0.02, 0.714], [-0.4, 0.1, 0.3, 0.5, -0.5, 0.5, 0.5]):
            c1, H1, g1 = p.eval(np.array(pose))
            c2, H2, g2 = q.eval(np.array(pose))
            assert c1 == c2 and np.array_equal(H1, H2) and np.array_equal(g1, g2)
    return d


@pytest.mark.gpu
@pytest.mark.parametrize("with_edges", [False, True])
def test_device_problems_equal_the_host_chain(oracle, with_edges):
    from camlasercalibratool_b200 import formats as fmt
    from camlasercalibratool_b200 import problems_from_scans

    tagpose, stamps, ranges = _session(oracle, 150, seed=11)
    kf = fmt.select_keyframes(tagpose)
    tp, pw = _pose_arrays(kf)
    pts, onl, info, lines = problems_from_scans(ranges, stamps, A0, INC, RMIN, tp, pw, with_edges=with_edges)
    obs, hp, hl = _host_chain(tagpose, stamps, ranges, with_edges)
    with pts, onl, hp, hl:
        assert 100 < len(obs) and pts.sizes()[0] == len(obs) == onl.sizes()[0]
        a, b = pts.download(), hp.download()
        # frames: scans with a segment whose nearest key-frame pose is < 20 ms away, in scan order
        kept = []
        for k in range(len(stamps)):
            seg = oracle.auto_get_line_pts(oracle.scan_to_points(ranges[k], A0, INC, RMIN))
            assert (seg is None and info[k, 0] == -1 and info[k, 1] == -1) or seg == (info[k, 0], info[k, 1]), k
            if seg is None:
                assert info[k, 2] == -1 and info[k, 3] == -1
                continue
            near, dt = _nearest_restated(tp, stamps[k])
            assert info[k, 2] == near
            if dt < 0.02:
                kept.append(k)
        assert np.array_equal(np.nonzero(info[:, 3] >= 0)[0], kept) and np.array_equal(info[kept, 3], np.arange(len(kept)))
        assert np.array_equal(a["offsets"], b["offsets"])
        np.testing.assert_allclose(a["frame_pose"], b["frame_pose"], rtol=0, atol=1e-15 * 4)
        np.testing.assert_allclose(a["points"], b["points"], rtol=0, atol=1e-12)
        assert np.all(a["points"][:, 2] == 0.0)
        c, e = onl.download(), hl.download()
        assert np.array_equal(c["offsets"], np.arange(len(obs) + 1) * 2)
        assert np.array_equal(c["frame_pose"], a["frame_pose"])
        np.testing.assert_allclose(c["points"], e["points"], rtol=0, atol=1e-9)
        if with_edges:
            # exactly the first and last point of the frame's segment, as marshal(obs, True, True) takes them
            assert np.array_equal(c["edge_points"], a["points"][np.stack([a["offsets"][:-1], a["offsets"][1:] - 1], 1)].reshape(-1, 6))
            np.testing.assert_allclose(c["edge_points"], e["edge_points"], rtol=0, atol=1e-12)
        assert np.all(np.isnan(lines[info[:, 3] < 0]))
        host_lines, _ = hp.line_fit(np.zeros((len(obs), 2)))
        np.testing.assert_allclose(lines[kept], host_lines, rtol=1e-7, atol=1e-9)
        # layout: the device-built problems evaluate bit for bit like the same arrays uploaded from the host
        _bitwise_eval_equal(pts)
        _bitwise_eval_equal(onl, use_edges=with_edges)
    # bit-reproducible
    p2, o2, info2, lines2 = problems_from_scans(ranges, stamps, A0, INC, RMIN, tp, pw, with_edges=with_edges)
    with p2, o2:
        assert np.array_equal(info, info2) and np.array_equal(lines, lines2, equal_nan=True)
        for x, y in ((a, p2.download()), (c, o2.download())):
            for k in ("frame_pose", "offsets", "points", "planes"):
                assert x[k].tobytes() == y[k].tobytes(), k


@pytest.mark.gpu
def test_pose_search_ties_unsorted_and_many_tiles(oracle):
    """More poses than one shared-memory tile, shuffled, with duplicated stamps far apart: the lowest index still wins."""
    from camlasercalibratool_b200 import problems_from_scans

    tagpose, stamps, ranges = _session(oracle, 60, seed=12, drop=0)
    tp, pw = _pose_arrays(tagpose)
    rng = np.random.default_rng(4)
    perm = rng.permutation(len(tp))
    tp, pw = tp[perm], pw[perm]
    tp = np.concatenate([rng.uniform(0, 99, 5000), tp, tp])  # the duplicates at the end lose every tie
    pw = np.concatenate([np.tile(POSES[0], (5000, 1)), pw, np.tile(POSES[1], (len(perm), 1))])
    tp[17] = np.nan
    pts, onl, info, _ = problems_from_scans(ranges, stamps, A0, INC, RMIN, tp, pw)
    with pts, onl:
        fp = pts.download()["frame_pose"]
        for k in range(len(stamps)):
            if info[k, 0] < 0:
                continue
            near, dt = _nearest_restated(tp, stamps[k])
            assert info[k, 2] == near and 5000 <= near < 5000 + len(perm)
            assert (info[k, 3] >= 0) == (dt < 0.02)
        assert pts.sizes()[0] > 20 and np.all(fp[:, 3] != 0)


@pytest.mark.gpu
def test_offline_from_scans_equals_the_host_driver(oracle, tmp_path):
    from camlasercalibratool_b200 import formats as fmt

    tagpose, stamps, ranges = _session(oracle, 200, seed=13)
    Tlc, rep = fmt.calibrate_offline_from_scans(tagpose, stamps, ranges, A0, INC, RMIN, result_yaml=str(tmp_path / "r.yaml"))
    Tlc_h, rep_h = fmt.calibrate_offline(tagpose, fmt.segments_from_scans(stamps, ranges, A0, INC, RMIN))
    assert rep["n_obs"] == rep_h["n_obs"] > 100
    np.testing.assert_allclose(rep["Tlc_closed_form"], rep_h["Tlc_closed_form"], rtol=0, atol=1e-9)
    np.testing.assert_allclose(Tlc, Tlc_h, rtol=0, atol=1e-9)
    assert rep["termination"] == rep_h["termination"] and rep["iterations"] == rep_h["iterations"]
    np.testing.assert_array_equal(fmt.read_result_yaml(str(tmp_path / "r.yaml"))["extrinsicTlc"], Tlc)
    assert np.abs(Tlc - oracle.ground_truth()[0]).max() < 2e-3  # 3 mm range noise, 1 % dropped beams kept as (1000, 1000)


@pytest.mark.gpu
def test_noise_free_ranges_recover_ground_truth(oracle):
    """Without noise the only error left is the float32 range (LaserScan::ranges): half an ulp is 6e-8 relative, about
    1e-7 m at 1.5 m.  Averaged over ~2*10^4 points in 200 frames that leaves a few 1e-9 on T_lc (measured on a B200:
    4.3e-9 for both the closed form and the LM result); the bound is 1e-7, the single-point quantisation."""
    from camlasercalibratool_b200 import formats as fmt

    tagpose, stamps, ranges = _session(oracle, 200, seed=14, sigma=0.0, drop=0.0)
    Tlc, rep = fmt.calibrate_offline_from_scans(tagpose, stamps, ranges, A0, INC, RMIN)
    err = np.abs(Tlc - oracle.ground_truth()[0]).max()
    print(f"noise-free ranges: n_obs {rep['n_obs']}, max |Tlc - T_gt| = {err:.3e}, closed form "
          f"{np.abs(rep['Tlc_closed_form'] - oracle.ground_truth()[0]).max():.3e}")
    assert err < 1e-7


@pytest.mark.gpu
def test_planar_family_engages_on_a_large_batch(oracle):
    from camlasercalibratool_b200 import problems_from_scans

    tagpose, stamps, ranges = _session(oracle, 12000, seed=15, sigma=0.002, drop=0.0)
    tp, pw = _pose_arrays(tagpose)
    pts, onl, info, _ = problems_from_scans(ranges, stamps, A0, INC, RMIN, tp, pw)
    with pts, onl:
        nf, npts, _ = pts.sizes()
        assert nf > 9000 and npts >= 6e5 and pts.planar
        assert pts.streamed_bytes() - (40 * nf + 224) == 16 * npts
        _bitwise_eval_equal(pts)


@pytest.mark.gpu
def test_pinned_and_pageable_ranges_give_the_same_problems(oracle):
    from camlasercalibratool_b200 import problems_from_scans
    from camlasercalibratool_b200.api import pinned_array

    tagpose, stamps, ranges = _session(oracle, 80, seed=16)
    tp, pw = _pose_arrays(tagpose)
    buf = pinned_array(ranges.shape, np.float32)
    try:
        buf.array[...] = ranges
        out = []
        for r in (ranges, buf.array):
            p, o, info, lines = problems_from_scans(r, stamps, A0, INC, RMIN, tp, pw, with_edges=True)
            with p, o:
                out.append((p.download(), o.download(), info, lines))
    finally:
        buf.free()
    (a, b, i1, l1), (c, d, i2, l2) = out
    assert np.array_equal(i1, i2) and np.array_equal(l1, l2, equal_nan=True)
    for x, y in ((a, c), (b, d)):
        for k in ("frame_pose", "offsets", "points", "planes"):
            assert x[k].tobytes() == y[k].tobytes()
    assert b["edge_points"].tobytes() == d["edge_points"].tobytes()


@pytest.mark.gpu
def test_scan_edge_cases(oracle):
    from camlasercalibratool_b200 import formats as fmt
    from camlasercalibratool_b200 import problems_from_scans

    tagpose, stamps, ranges = _session(oracle, 30, seed=17, drop=0)
    tp, pw = _pose_arrays(tagpose)

    def frames(r, ts, tps, pws, **kw):
        p, o, info, lines = problems_from_scans(r, ts, A0, INC, RMIN, tps, pws, **kw)
        with p, o:
            assert p.sizes()[0] == o.sizes()[0]
            d = p.download()
            assert d["offsets"][0] == 0 and len(d["offsets"]) == p.sizes()[0] + 1
            return p.sizes()[0], info

    n, info = frames(ranges[:0], stamps[:0], tp, pw)  # zero scans
    assert n == 0 and info.shape == (0, 4)
    n, info = frames(ranges, stamps, tp[:0], pw[:0])  # zero poses
    assert n == 0 and np.all(info[:, 2:] == -1) and np.any(info[:, 0] >= 0)
    _, s2, walls = _session(oracle, 30, seed=17, drop=0, board=False)  # no board anywhere
    n, info = frames(walls, s2, tp, pw)
    assert n == 0 and np.all(info == -1)
    n, info = frames(ranges, stamps + 10.0, tp, pw)  # every scan outside max_dt
    assert n == 0 and np.all(info[:, 3] == -1) and np.any(info[:, 2] >= 0)
    # the strict boundary, exactly representable: dt == max_dt is dropped, dt < max_dt kept
    one = ranges[[0, 0, 0]]
    n, info = frames(one, np.array([1.015625, 1.0078125, 0.984375]), np.array([1.0]), pw[:1], max_dt=0.015625)
    assert n == 1 and list(info[:, 3]) == [-1, 0, -1]
    # the driver's refusal: fewer than 5 observations
    Tlc, why = fmt.calibrate_offline_from_scans(tagpose, stamps + 10.0, ranges, A0, INC, RMIN)
    assert Tlc is None and why == "Valid Calibra Data Less"
