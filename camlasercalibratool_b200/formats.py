"""On-disk formats and the glue of the reference's offline driver, without ROS (SURVEY.md 8(f) rank 3).

Host-side only (text I/O and O(frames) bookkeeping); every numeric step of the calibration itself -- line fits,
closed form, LM solve, information matrix -- goes through the CUDA library.

* ``apriltag_pose.txt``  one pose per line ``ts x y z qx qy qz qw [roll pitch yaw]`` -- written by reference
  main/kalibratag_detector_node.cpp:202-236, read by src/utilities.cpp:6-54 (trailing Euler columns ignored).
* ``result.yaml``        OpenCV FileStorage YAML with ``extrinsicTlc`` (4x4), ``RollPitchYaw`` (3x1), ``txtytz`` (3x1)
  -- reference main/calibr_offline.cpp:186-197.
* ``calibrate_offline``  reference main/calibr_offline.cpp:52-170 from key-frame thinning to the LM solve, taking the
  already-extracted laser segments (the output of AutoGetLinePts) instead of a rosbag.
* ``calibrate_offline_from_scans``  the same from the raw LaserScan ranges: the scan loop (segment, nearest pose, line fit,
  end points) runs on the device and builds both problems there (clc_problems_create_from_scans).
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np

from .api import CamLaserCalClosedSolution, CamLaserCalibration, Oberserve, Problem


@dataclass
class CamPose:
    """reference include/utilities.h:15-26 (the fields this path uses)."""

    timestamp: float
    qwc: np.ndarray  # x, y, z, w
    twc: np.ndarray


# ---- quaternion helpers (Eigen semantics, coefficient order x,y,z,w) ------------------------------------------------
def quat_mul(a, b):
    ax, ay, az, aw = a
    bx, by, bz, bw = b
    return np.array([aw * bx + ax * bw + ay * bz - az * by, aw * by + ay * bw + az * bx - ax * bz,
                     aw * bz + az * bw + ax * by - ay * bx, aw * bw - ax * bx - ay * by - az * bz])


def quat_inverse(q):
    q = np.asarray(q, dtype=float)
    return np.array([-q[0], -q[1], -q[2], q[3]]) / float(q @ q)  # Eigen: conjugate / squaredNorm


def quat_to_rot(q):
    x, y, z, w = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


def to_euler_angles(q):
    """reference src/utilities.cpp:234-257 ToEulerAngles: (roll, pitch, yaw)."""
    x, y, z, w = q
    roll = math.atan2(2.0 * (w * x + y * z), 1.0 - 2.0 * (x * x + y * y))
    sinp = 2.0 * (w * y - z * x)
    pitch = math.copysign(math.pi / 2, sinp) if abs(sinp) >= 1 else math.asin(sinp)
    yaw = math.atan2(2.0 * (w * z + x * y), 1.0 - 2.0 * (y * y + z * z))
    return roll, pitch, yaw


# ---- apriltag_pose.txt ----------------------------------------------------------------------------------------------
def load_cam_pose_txt(path) -> list[CamPose]:
    """reference src/utilities.cpp:6-54: blank lines skipped, columns beyond the eighth ignored."""
    out = []
    with open(path) as f:
        for line in f:
            v = line.split()
            if not v:
                continue
            ts, x, y, z, q1, q2, q3, qw = (float(t) for t in v[:8])
            out.append(CamPose(ts, np.array([q1, q2, q3, qw]), np.array([x, y, z])))
    return out


def save_cam_pose_txt(path, poses):
    """reference main/kalibratag_detector_node.cpp:205-232: fixed notation, timestamp with 9 decimals, the rest with 10."""
    with open(path, "w") as f:
        for p in poses:
            r, pi, yw = to_euler_angles(p.qwc)
            vals = [p.twc[0], p.twc[1], p.twc[2], p.qwc[0], p.qwc[1], p.qwc[2], p.qwc[3], r, pi, yw]
            f.write(f"{p.timestamp:.9f} " + " ".join(f"{v:.10f}" for v in vals) + "\n")


# ---- result.yaml -------------------------------------------------------------------------------------------------------
def _cv_matrix(name, m):
    m = np.atleast_2d(np.asarray(m, dtype=float))
    data = ", ".join(repr(float(v)) for v in m.reshape(-1))
    return f"{name}: !!opencv-matrix\n   rows: {m.shape[0]}\n   cols: {m.shape[1]}\n   dt: d\n   data: [ {data} ]\n"


def write_result_yaml(path, Tlc):
    """reference main/calibr_offline.cpp:173-197: extrinsicTlc, RollPitchYaw (of R_lc), txtytz, readable by cv::FileStorage."""
    Tlc = np.asarray(Tlc, dtype=float)
    from .api import T_to_pose7

    q = T_to_pose7(Tlc)[3:]  # Eigen::Quaterniond(Rlc)
    rpy = to_euler_angles(q)
    with open(path, "w") as f:
        f.write("%YAML:1.0\n---\n")
        f.write(_cv_matrix("extrinsicTlc", Tlc))
        f.write(_cv_matrix("RollPitchYaw", np.array(rpy).reshape(3, 1)))
        f.write(_cv_matrix("txtytz", Tlc[:3, 3].reshape(3, 1)))
    return rpy


def read_result_yaml(path):
    """Minimal reader of the file above (cv::FileStorage reads it too): {name: ndarray}."""
    import re

    text = open(path).read()
    out = {}
    for m in re.finditer(r"(\w+): !!opencv-matrix\s+rows: (\d+)\s+cols: (\d+)\s+dt: d\s+data: \[([^\]]*)\]", text):
        out[m.group(1)] = np.array([float(v) for v in m.group(4).replace("\n", " ").split(",")]).reshape(int(m.group(2)), int(m.group(3)))
    return out


# ---- board poses from tag detections (the arithmetic of kalibratag_detector_node) ---------------------------------------
def estimate_board_poses(camera, detections, intrinsics=None, grid=(6, 6, 0.055, 0.3), device=-1):
    """Batched CamPoseEst::calcCamPose minus the tag detector (reference src/calcCamPose.cpp:270-294, :211-236) on the
    GPU.  ``camera``: "radtan" | "equi"; ``detections``: per frame a pair (tag_ids[k], corners[k,4,2] pixel coordinates)
    in ascending id order, as the AprilTag detector of the reference delivers them.  Returns (pose_wc[n,7] =
    qx qy qz qw x y z of T_wc, ok[n] bool); frames with fewer than 4 points or a bad id get the identity pose, ok False."""
    import ctypes as C

    from . import _lib
    from .api import CAMERA_DEFAULTS

    d = _lib.CameraDesc()
    d.camera_model = {"radtan": 1, "pinhole": 1, "equi": 2}[camera]
    k = CAMERA_DEFAULTS["radtan" if d.camera_model == 1 else "equi"] if intrinsics is None else intrinsics
    d.intrinsics = (C.c_double * 8)(*[float(v) for v in k])
    d.grid_rows, d.grid_cols, d.tag_size, d.tag_spacing = int(grid[0]), int(grid[1]), float(grid[2]), float(grid[3])
    n = len(detections)
    counts = [len(np.atleast_1d(ids)) for ids, _ in detections]
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    ids = np.ascontiguousarray(np.concatenate([np.atleast_1d(i) for i, _ in detections]) if n else [], dtype=np.int32)
    uv = np.ascontiguousarray(np.concatenate([np.asarray(c, dtype=np.float32).reshape(-1, 8) for _, c in detections])
                              if n else np.zeros((0, 8)), dtype=np.float32)
    pose = np.zeros((n, 7))
    ok = np.zeros(n, dtype=np.int32)
    _lib.check(_lib.load().clc_estimate_board_poses(C.byref(d), n, off.ctypes.data_as(C.POINTER(C.c_int64)),
                                                    ids.ctypes.data_as(C.POINTER(C.c_int32)), uv.ctypes.data_as(C.POINTER(C.c_float)),
                                                    pose.ctypes.data_as(C.POINTER(C.c_double)), ok.ctypes.data_as(C.POINTER(C.c_int32)),
                                                    int(device)), "clc_estimate_board_poses")
    return pose, ok.astype(bool)


def cam_poses_from_detections(timestamps, camera, detections, **kw) -> list[CamPose]:
    """reference main/kalibratag_detector_node.cpp:206-234: the CamPose list (frames without a usable detection dropped)
    that save_cam_pose_txt writes as apriltag_pose.txt."""
    pose, ok = estimate_board_poses(camera, detections, **kw)
    return [CamPose(float(t), pose[i, :4].copy(), pose[i, 4:].copy()) for i, t in enumerate(timestamps) if ok[i]]


# ---- planar.txt / RoiPoints.txt / RoiPtOnLines.txt ------------------------------------------------------------------------
def save_plane_points(obs, Tcl, path):
    """reference src/LaseCamCalCeres.cpp:68-110 CalibrationTool_SavePlanePoints: per frame the board plane in the camera
    frame (``i nx ny nz d`` -> planar.txt) and the laser points / fitted-line points moved into the camera frame by Tcl
    (``i x y z`` -> RoiPoints.txt, RoiPtOnLines.txt); std::setprecision(3) on a default-format stream = ``%.3g``.
    The planes come from the library (the same device kernel that feeds the solve)."""
    from .api import marshal

    Tcl = np.asarray(Tcl, dtype=float)
    fp, off, pts, _ = marshal(obs, False, False)
    with Problem.from_arrays(fp, off, pts) as g:
        planes = g.download()["planes"]

    def g3(v):
        return "%.3g" % v

    with open(path + "planar.txt", "w") as fa, open(path + "RoiPoints.txt", "w") as fb, open(path + "RoiPtOnLines.txt", "w") as fc:
        for i, o in enumerate(obs):
            fa.write(f"{i} " + " ".join(g3(v) for v in planes[i]) + "\n")
            for f, arr in ((fb, o.points), (fc, o.points_on_line)):
                arr = np.asarray(arr, dtype=float).reshape(-1, 3)
                cam = arr @ Tcl[:3, :3].T + Tcl[:3, 3]
                for q in cam:
                    f.write(f"{i} " + " ".join(g3(v) for v in q) + "\n")


# ---- scans: LaserScan ranges -> points -> board segment ---------------------------------------------------------------
def scan_to_points(ranges, angle_min, angle_increment, range_min):
    """reference src/utilities.cpp:181-215 TranScanToPoints (host data preparation; invalid beams -> (1000,1000,0))."""
    r = np.asarray(ranges, dtype=np.float32)
    ang = angle_min + np.arange(r.shape[-1], dtype=float) * angle_increment
    ok = (r < 30.0) & (r >= range_min)
    with np.errstate(invalid="ignore"):
        x = np.where(ok, r.astype(float) * np.cos(ang), 1000.0)
        y = np.where(ok, r.astype(float) * np.sin(ang), 1000.0)
    return np.stack([x, y, np.zeros_like(x)], axis=-1)


def auto_get_line_segments(ranges, angle_min, angle_increment, range_min, device=-1):
    """Batched AutoGetLinePts (reference src/selectScanPoints.cpp:17-190) on the GPU: ranges[n_scans, n_beams] float32 ->
    (seg_start[n_scans], seg_end[n_scans]) inclusive beam indices, -1 where no board segment was found."""
    import ctypes as C

    from . import _lib

    r = np.ascontiguousarray(ranges, dtype=np.float32).reshape(len(ranges), -1)
    s = np.empty(r.shape[0], dtype=np.int32)
    e = np.empty(r.shape[0], dtype=np.int32)
    _lib.check(_lib.load().clc_scan_segments(r.ctypes.data_as(C.POINTER(C.c_float)), r.shape[0], r.shape[1], float(angle_min),
                                             float(angle_increment), float(range_min), s.ctypes.data_as(C.POINTER(C.c_int32)),
                                             e.ctypes.data_as(C.POINTER(C.c_int32)), int(device)), "clc_scan_segments")
    return s, e


def segments_from_scans(timestamps, ranges, angle_min, angle_increment, range_min):
    """reference main/calibr_offline.cpp:88-100: [(timestamp, points[n,3])] of the scans in which a board segment was found."""
    pts = scan_to_points(ranges, angle_min, angle_increment, range_min)
    s, e = auto_get_line_segments(ranges, angle_min, angle_increment, range_min)
    return [(float(t), pts[k, s[k]:e[k] + 1]) for k, t in enumerate(timestamps) if s[k] >= 0]


# ---- the offline driver, without ROS -----------------------------------------------------------------------------------
def select_keyframes(tagpose, dist_min=0.20, theta_min=3.1415926 * 10 / 180.0):
    """reference main/calibr_offline.cpp:62-78."""
    sparse = [tagpose[0]]
    older = tagpose[0]
    for newer in tagpose[1:]:
        dist = float(np.linalg.norm(older.twc - newer.twc))
        w = quat_mul(quat_inverse(older.qwc), newer.qwc)[3]
        theta = 2 * math.acos(max(-1.0, min(1.0, w)))
        if dist > dist_min or abs(theta) > theta_min:
            older = newer
            sparse.append(older)
    return sparse


def observations_from_segments(tagpose, scans, max_dt=0.02, lines=None):
    """reference main/calibr_offline.cpp:84-155: ``scans`` = [(timestamp, points[n,3])] are the laser segments on the
    board (the output of AutoGetLinePts).  Every scan is matched to the nearest tag pose (accepted within 20 ms), its
    line is fitted by LineFittingCeres -- here for all accepted scans in ONE batched GPU call -- and the two end points
    on the fitted line become points_on_line.  Returns list[Oberserve]."""
    ts_pose = np.array([p.timestamp for p in tagpose])
    picked = []
    for ts, pts in scans:
        pts = np.asarray(pts, dtype=float).reshape(-1, 3)
        if len(pts) == 0:
            continue
        k = int(np.argmin(np.abs(ts_pose - ts)))  # :105-115
        if abs(ts_pose[k] - ts) < max_dt:
            picked.append((tagpose[k], pts))
    if not picked:
        return []
    if lines is None:
        off = np.concatenate([[0], np.cumsum([len(p) for _, p in picked])])
        fp = np.tile([0, 0, 0, 1, 0, 0, 1.0], (len(picked), 1))
        with Problem.from_arrays(fp, off, np.concatenate([p for _, p in picked])) as g:
            lines, _ = g.line_fit(np.zeros((len(picked), 2)))  # :123-124 (start value: zeros)
    obs = []
    for (pose, pts), line in zip(picked, lines):
        # :126-142 -- NB the reference reads points.end() (one past the last point, UB); the last point is meant
        x_s, x_e, y_s, y_e = pts[0, 0], pts[-1, 0], pts[0, 1], pts[-1, 1]
        if abs(x_e - x_s) > abs(y_e - y_s):
            y_s = -(x_s * line[0] + 1) / line[1]
            y_e = -(x_e * line[0] + 1) / line[1]
        else:
            x_s = -(y_s * line[1] + 1) / line[0]
            x_e = -(y_e * line[1] + 1) / line[0]
        qca = quat_inverse(pose.qwc)  # :145
        tca = -quat_to_rot(qca) @ pose.twc  # :146
        obs.append(Oberserve(qca, tca, pts, np.array([[x_s, y_s, 0.0], [x_e, y_e, 0.0]])))
    return obs


def calibrate_offline(tagpose, scans, result_yaml=None, verbose=False):
    """reference main/calibr_offline.cpp:52-197 without the rosbag: returns (Tlc, report) or (None, reason)."""
    if len(tagpose) < 10:  # :55-59
        return None, "apriltag pose less than 10."
    obs = observations_from_segments(select_keyframes(tagpose), scans)
    if len(obs) < 5:  # :158-163
        return None, "Valid Calibra Data Less"
    Tlc0 = np.eye(4)
    CamLaserCalClosedSolution(obs, Tlc0, verbose=verbose)  # :166-167
    Tcl = np.linalg.inv(Tlc0)
    report = CamLaserCalibration(obs, Tcl, False, verbose=verbose)  # :169-170
    Tlc = np.linalg.inv(Tcl)
    if result_yaml is not None:
        write_result_yaml(result_yaml, Tlc)
    report["n_obs"] = len(obs)
    report["Tlc_closed_form"] = Tlc0
    return Tlc, report


def calibrate_offline_from_scans(tagpose, scan_stamps, ranges, angle_min, angle_increment, range_min, result_yaml=None,
                                 verbose=False):
    """reference main/calibr_offline.cpp:52-197 from the raw LaserScan ranges[n_scans, n_beams] (float32) and their stamps:
    the same result as ``calibrate_offline(tagpose, segments_from_scans(scan_stamps, ranges, ...))``, but the scan loop
    (segment, nearest key-frame pose, line fit, end points) runs on the device and the points never leave it -- one upload
    of the ranges.  Key-frame thinning stays on the host (sequential, O(poses)).  Returns (Tlc, report) or (None, reason)."""
    from .api import calibrate_on, closed_form_on, problems_from_scans

    if len(tagpose) < 10:  # :55-59
        return None, "apriltag pose less than 10."
    kf = select_keyframes(tagpose)
    stamps = np.array([p.timestamp for p in kf], dtype=np.float64)
    pose_wc = np.array([np.concatenate([p.qwc, p.twc]) for p in kf], dtype=np.float64).reshape(-1, 7)
    points, on_line, _, _ = problems_from_scans(ranges, scan_stamps, angle_min, angle_increment, range_min, stamps, pose_wc)
    with points, on_line:
        n_obs = points.sizes()[0]
        if n_obs < 5:  # :158-163
            return None, "Valid Calibra Data Less"
        Tlc0 = np.eye(4)
        closed_form_on(on_line, Tlc0, verbose=verbose)  # :166-167
        Tcl = np.linalg.inv(Tlc0)
        report = calibrate_on(points, Tcl, verbose=verbose)  # :169-170
    Tlc = np.linalg.inv(Tcl)
    if result_yaml is not None:
        write_result_yaml(result_yaml, Tlc)
    report["n_obs"] = n_obs
    report["Tlc_closed_form"] = Tlc0
    return Tlc, report
