"""Python mirror of the reference's solver interface, on top of the C ABI (include/clc_b200.h).

Mirrors reference include/LaseCamCalCeres.h:11-29: the ``Oberserve`` struct (sic) and the free functions
``CamLaserCalibration`` / ``CamLaserCalClosedSolution`` with the same argument meaning (in/out 4x4 transform,
``use_linefitting_data``, ``use_boundary_constraint``).  Everything numeric happens in libclc_b200.so on the GPU;
this module only marshals ``list[Oberserve]`` into the flat arrays of the ABI.  (The C++ drop-in with the exact
reference signatures is camlasercalibratool_b200/host/LaseCamCalB200.cpp.)
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np

from . import _lib
from ._lib import ClcError, GatherDesc, LmIteration, LmOptions, LmSummary, ProblemDesc, ScanDesc, SyntheticDesc, TERMINATION


def _dp(a):
    return a.ctypes.data_as(_lib.c_double_p) if a is not None else None


def _ip(a):
    return a.ctypes.data_as(_lib.c_int64_p) if a is not None else None


@dataclass
class Oberserve:
    """reference include/LaseCamCalCeres.h:11-24 (the misspelling is the reference's)."""

    tagPose_Qca: np.ndarray = field(default_factory=lambda: np.array([0.0, 0.0, 0.0, 1.0]))  # Eigen coeffs x,y,z,w
    tagPose_tca: np.ndarray = field(default_factory=lambda: np.zeros(3))
    points: np.ndarray = field(default_factory=lambda: np.zeros((0, 3)))
    points_on_line: np.ndarray = field(default_factory=lambda: np.zeros((0, 3)))


def marshal(obs, use_linefitting_data=True, use_boundary_constraint=False):
    """list[Oberserve] -> (frame_pose[N,7], offsets[N+1], points[P,3], edge_points[N,6] | None).

    Point-set selection as reference src/LaseCamCalCeres.cpp:233-237; the edge residuals exist only when both
    flags are set (:258) and use obs.points.front()/back() (:278-279)."""
    n = len(obs)
    frame_pose = np.zeros((n, 7))
    counts = np.zeros(n + 1, dtype=np.int64)
    chunks = []
    want_edges = bool(use_boundary_constraint and use_linefitting_data)
    edge = np.zeros((n, 6)) if want_edges else None
    for i, ob in enumerate(obs):
        frame_pose[i, :4] = np.asarray(ob.tagPose_Qca, dtype=np.float64)
        frame_pose[i, 4:] = np.asarray(ob.tagPose_tca, dtype=np.float64)
        pts = np.asarray(ob.points_on_line if use_linefitting_data else ob.points, dtype=np.float64).reshape(-1, 3)
        counts[i + 1] = pts.shape[0]
        chunks.append(pts)
        if want_edges and pts.shape[0] > 0:
            raw = np.asarray(ob.points, dtype=np.float64).reshape(-1, 3)
            if raw.shape[0] == 0:
                raise ValueError("use_boundary_constraint needs obs.points (reference :278 calls points.at(0))")
            edge[i, :3] = raw[0]
            edge[i, 3:] = raw[-1]
    offsets = np.cumsum(counts)
    points = np.concatenate(chunks, axis=0) if chunks else np.zeros((0, 3))
    return frame_pose, offsets, np.ascontiguousarray(points), edge


# intrinsics of the reference's two shipped configurations
CAMERA_DEFAULTS = {
    # config/calibra_config_pinhole.yaml (its distortion block is all zeros; a mild radtan distortion is used instead so that
    # the undistortion step does something)
    "radtan": [367.049931000148, 366.94446918887405, 368.7202381120387, 241.13814795878562, -0.05, 0.01, 0.0005, -0.0005],
    # config/calibra_config.yaml (KANNALA_BRANDT)
    "equi": [367.049931000148, 366.94446918887405, 368.7202381120387, 241.13814795878562, -0.02276964, -0.00056958, -0.0026224,
             0.00017455],
}


class _Gather:
    """Keeps the arrays of a clc_gather_desc alive: one separate [n_i, 3] array per frame, as std::vector<Oberserve> holds
    them (reference include/LaseCamCalCeres.h:22-23)."""

    def __init__(self, frame_pose, frames, edge_points=None, use_loss=True, cauchy_a=0.05, device=-1):
        self.frame_pose = np.ascontiguousarray(frame_pose, dtype=np.float64).reshape(-1, 7)
        self.frames = [np.ascontiguousarray(f, dtype=np.float64).reshape(-1, 3) for f in frames]
        n = self.frame_pose.shape[0]
        if len(self.frames) != n:
            raise ValueError("one point array per frame is needed")
        self.counts = np.array([f.shape[0] for f in self.frames], dtype=np.int64)
        self.ptrs = (_lib.c_double_p * max(n, 1))(*[_dp(f) for f in self.frames])
        self.edge = None
        if edge_points is not None:
            self.edge = np.ascontiguousarray(edge_points, dtype=np.float64).reshape(-1, 6)
            if self.edge.shape[0] != n:
                raise ValueError("edge_points must be [n_frames, 6]")
        d = GatherDesc()
        d.n_frames = n
        d.frame_pose, d.frame_points, d.frame_counts, d.edge_points = _dp(self.frame_pose), self.ptrs, _ip(self.counts), _dp(self.edge)
        d.use_loss, d.cauchy_a, d.device = int(bool(use_loss)), float(cauchy_a), int(device)
        self.desc = d


def _synthetic_desc(n_frames_total, beams, seed, sigma, with_edges, frame_begin, frame_end, use_loss, cauchy_a, device, camera,
                    pixel_sigma, intrinsics, image_size, grid):
    d = SyntheticDesc()
    d.n_frames_total = int(n_frames_total)
    d.frame_begin = int(frame_begin)
    d.frame_end = int(n_frames_total if frame_end is None else frame_end)
    d.beams, d.seed, d.sigma = int(beams), int(seed), float(sigma)
    d.with_edges, d.use_loss, d.cauchy_a, d.device = int(bool(with_edges)), int(bool(use_loss)), float(cauchy_a), int(device)
    d.camera_model = {None: 0, "none": 0, "radtan": 1, "pinhole": 1, "equi": 2}[camera]
    if d.camera_model:
        k = CAMERA_DEFAULTS["radtan" if d.camera_model == 1 else "equi"] if intrinsics is None else intrinsics
        d.camera_intrinsics = (C.c_double * 8)(*[float(v) for v in k])
        d.pixel_sigma = float(pixel_sigma)
        d.image_width, d.image_height = int(image_size[0]), int(image_size[1])
        d.grid_rows, d.grid_cols, d.tag_size, d.tag_spacing = int(grid[0]), int(grid[1]), float(grid[2]), float(grid[3])
    return d


def default_options(**kw) -> LmOptions:
    o = LmOptions()
    _lib.load().clc_lm_default_options(C.byref(o))
    for k, v in kw.items():
        setattr(o, k, v)
    return o


class Problem:
    """A device-resident problem (one per GPU / rank).  Thin wrapper over clc_problem*."""

    def __init__(self, handle):
        self._h = handle
        self._L = _lib.load()
        self._comm = None

    # ---- construction ----
    @classmethod
    def from_arrays(cls, frame_pose, offsets, points, edge_points=None, use_loss=True, cauchy_a=0.05, device=-1):
        L = _lib.load()
        frame_pose = np.ascontiguousarray(frame_pose, dtype=np.float64).reshape(-1, 7)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        points = np.ascontiguousarray(points, dtype=np.float64).reshape(-1, 3)
        if edge_points is not None:
            edge_points = np.ascontiguousarray(edge_points, dtype=np.float64).reshape(-1, 6)
            if edge_points.shape[0] != frame_pose.shape[0]:
                raise ValueError("edge_points must be [n_frames, 6]")
        if offsets.shape[0] != frame_pose.shape[0] + 1 or (offsets.size and offsets[-1] != points.shape[0]):
            raise ValueError("offsets do not match frame_pose / points")
        d = ProblemDesc()
        d.n_frames = frame_pose.shape[0]
        d.frame_pose, d.offsets, d.points, d.edge_points = _dp(frame_pose), _ip(offsets), _dp(points), _dp(edge_points)
        d.use_loss, d.cauchy_a, d.device = int(bool(use_loss)), float(cauchy_a), int(device)
        h = C.c_void_p()
        _lib.check(L.clc_problem_create(C.byref(h), C.byref(d)), "clc_problem_create")
        return cls(h)

    @classmethod
    def from_frames(cls, frame_pose, frames, edge_points=None, use_loss=True, cauchy_a=0.05, device=-1):
        """One separate [n_i, 3] array per frame (clc_problem_create_gather): the library gathers them itself."""
        g = _Gather(frame_pose, frames, edge_points, use_loss, cauchy_a, device)
        h = C.c_void_p()
        _lib.check(_lib.load().clc_problem_create_gather(C.byref(h), C.byref(g.desc)), "clc_problem_create_gather")
        return cls(h)

    @classmethod
    def from_observations(cls, obs, use_linefitting_data=True, use_boundary_constraint=False, **kw):
        fp, off, pts, edge = marshal(obs, use_linefitting_data, use_boundary_constraint)
        return cls.from_arrays(fp, off, pts, edge, **kw)

    @classmethod
    def synthetic(cls, n_frames_total, beams, seed=1, sigma=0.0, with_edges=False, frame_begin=0, frame_end=None,
                  use_loss=True, cauchy_a=0.05, device=-1, camera=None, pixel_sigma=0.0, intrinsics=None,
                  image_size=(752, 480), grid=(6, 6, 0.055, 0.3)):
        """camera: None (exact board poses, the reference simulation), "radtan" (pinhole, fx fy cx cy k1 k2 p1 p2) or "equi"
        (Kannala-Brandt, mu mv u0 v0 k2 k3 k4 k5): the poses handed to the solver are then estimated from noisy corner
        pixels by the reference's undistort + PnP chain.  Default intrinsics: the reference's config/*.yaml."""
        L = _lib.load()
        d = _synthetic_desc(n_frames_total, beams, seed, sigma, with_edges, frame_begin, frame_end, use_loss, cauchy_a, device,
                            camera, pixel_sigma, intrinsics, image_size, grid)
        h = C.c_void_p()
        _lib.check(L.clc_problem_create_synthetic(C.byref(h), C.byref(d)), "clc_problem_create_synthetic")
        return cls(h)

    def close(self):
        if self._h is not None:
            self._L.clc_problem_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- introspection ----
    def sizes(self):
        nf, npts, he = C.c_int64(), C.c_int64(), C.c_int()
        _lib.check(self._L.clc_problem_sizes(self._h, C.byref(nf), C.byref(npts), C.byref(he)), "clc_problem_sizes")
        return nf.value, npts.value, bool(he.value)

    def algorithmic_bytes(self):
        b = C.c_int64()
        _lib.check(self._L.clc_problem_algorithmic_bytes(self._h, C.byref(b)), "clc_problem_algorithmic_bytes")
        return b.value

    def streamed_bytes(self):
        """Bytes one sweep really streams (16 B per point when the planar two-stream kernels are active)."""
        b = C.c_int64()
        _lib.check(self._L.clc_problem_streamed_bytes(self._h, C.byref(b)), "clc_problem_streamed_bytes")
        return b.value

    @property
    def planar(self):
        """True if the z stream was dropped (every z exactly 0) and the two-stream kernels run."""
        return self.streamed_bytes() != self.algorithmic_bytes()

    def set_planar_mode(self, mode):
        """1 = automatic (default): planar data runs the two-stream kernels; 0 = always the general kernels."""
        _lib.check(self._L.clc_problem_set_planar_mode(self._h, int(mode)), "clc_problem_set_planar_mode")

    def download(self):
        nf, npts, he = self.sizes()
        fp, off, pts = np.empty((nf, 7)), np.empty(nf + 1, dtype=np.int64), np.empty((npts, 3))
        edge = np.empty((nf, 6)) if he else None
        planes = np.empty((nf, 4))
        _lib.check(self._L.clc_problem_download(self._h, _dp(fp), _ip(off), _dp(pts), _dp(edge), _dp(planes)),
                   "clc_problem_download")
        return dict(frame_pose=fp, offsets=off, points=pts, edge_points=edge, planes=planes)

    def download_true_poses(self):
        """Synthetic problems with a camera model: the poses the laser points were generated from."""
        fp = np.empty((self.sizes()[0], 7))
        _lib.check(self._L.clc_problem_download_true_poses(self._h, _dp(fp)), "clc_problem_download_true_poses")
        return fp

    # ---- the hot path ----
    def eval(self, pose7):
        pose7 = np.ascontiguousarray(pose7, dtype=np.float64)
        H, g, cost = np.empty((6, 6)), np.empty(6), C.c_double()
        _lib.check(self._L.clc_eval(self._h, _dp(pose7), _dp(H), _dp(g), C.byref(cost)), "clc_eval")
        return cost.value, H, g

    def solve(self, pose7, options: LmOptions | None = None, trace_cap=256):
        x = np.ascontiguousarray(pose7, dtype=np.float64).copy()
        o = options if options is not None else default_options()
        s = LmSummary()
        tr = (LmIteration * trace_cap)()
        _lib.check(self._L.clc_solve_lm(self._h, _dp(x), C.byref(o), C.byref(s), tr, trace_cap), "clc_solve_lm")
        return x, s, [tr[i] for i in range(min(s.num_iterations, trace_cap))]

    def information(self, pose7):
        pose7 = np.ascontiguousarray(pose7, dtype=np.float64)
        H, b, sv, chi = np.empty((6, 6)), np.empty(6), np.empty(6), C.c_double()
        self.last_V = np.empty((6, 6))  # right singular vectors of H, columns ordered like sv
        _lib.check(self._L.clc_information(self._h, _dp(pose7), _dp(H), _dp(b), C.byref(chi), _dp(sv), _dp(self.last_V)),
                   "clc_information")
        return H, b, chi.value, sv

    def closed_form(self):
        T, AtA, Atb, un = np.empty(16), np.empty((9, 9)), np.empty(9), C.c_int()
        _lib.check(self._L.clc_closed_form(self._h, _dp(T), C.byref(un), _dp(AtA), _dp(Atb)), "clc_closed_form")
        return T.reshape(4, 4), bool(un.value), AtA, Atb

    def line_fit(self, lines0=None, max_num_iterations=10):
        """Batched LineFittingCeres over the frames' points: returns (lines[N,2], info[N,4])."""
        nf = self.sizes()[0]
        lines = np.zeros((nf, 2)) if lines0 is None else np.ascontiguousarray(lines0, dtype=np.float64).reshape(nf, 2).copy()
        info = np.empty((nf, 4))
        _lib.check(self._L.clc_problem_line_fit(self._h, _dp(lines), int(max_num_iterations), _dp(info)), "clc_problem_line_fit")
        return lines, info

    # ---- multi-GPU ----
    def set_allreduce_mode(self, mode: int):
        """0 = NCCL all-reduce between kernels, 1 = fused in-kernel peer exchange (default once p2p is enabled)."""
        _lib.check(self._L.clc_problem_set_allreduce_mode(self._h, int(mode)), "clc_problem_set_allreduce_mode")

    def attach_comm(self, comm: "Comm | None"):
        """Borrow a communicator: every sweep's 28 sums are then all-reduced over its ranks."""
        self._comm = comm  # keep it alive
        _lib.check(self._L.clc_problem_attach_comm(self._h, comm._h if comm is not None else None), "clc_problem_attach_comm")

    # ---- measurement ----
    def bench_eval(self, pose7, n, flush_l2=True):
        pose7 = np.ascontiguousarray(pose7, dtype=np.float64)
        ms = (C.c_float * n)()
        _lib.check(self._L.clc_bench_eval(self._h, _dp(pose7), int(n), int(bool(flush_l2)), ms), "clc_bench_eval")
        return np.array(ms[:], dtype=np.float64)


class Group:
    """G devices of THIS process solving one problem (clc_group_*): frames sharded by point count, the 28 sums exchanged
    over NVLink inside the sweep kernel, one host thread.  A group of one device is a plain problem."""

    def __init__(self, handle):
        self._h = handle
        self._L = _lib.load()

    @staticmethod
    def _devices(devices):
        devs = [int(d) for d in devices]
        return (C.c_int * len(devs))(*devs), len(devs)

    @classmethod
    def from_frames(cls, frame_pose, frames, edge_points=None, devices=(-1,), use_loss=True, cauchy_a=0.05):
        g = _Gather(frame_pose, frames, edge_points, use_loss, cauchy_a)
        arr, n = cls._devices(devices)
        h = C.c_void_p()
        _lib.check(_lib.load().clc_group_create_gather(C.byref(h), C.byref(g.desc), arr, n), "clc_group_create_gather")
        return cls(h)

    @classmethod
    def from_arrays(cls, frame_pose, offsets, points, edge_points=None, devices=(-1,), **kw):
        points = np.ascontiguousarray(points, dtype=np.float64).reshape(-1, 3)
        offsets = np.asarray(offsets, dtype=np.int64)
        frames = [points[offsets[f]:offsets[f + 1]] for f in range(len(offsets) - 1)]
        return cls.from_frames(frame_pose, frames, edge_points, devices, **kw)

    @classmethod
    def synthetic(cls, n_frames, beams, seed=1, sigma=0.0, with_edges=False, devices=(-1,), use_loss=True, cauchy_a=0.05,
                  n_frames_total=None, frame_begin=0, camera=None, pixel_sigma=0.0, intrinsics=None, image_size=(752, 480),
                  grid=(6, 6, 0.055, 0.3)):
        total = int(n_frames_total if n_frames_total is not None else frame_begin + n_frames)
        d = _synthetic_desc(total, beams, seed, sigma, with_edges, frame_begin, frame_begin + n_frames, use_loss, cauchy_a, -1,
                            camera, pixel_sigma, intrinsics, image_size, grid)
        arr, n = cls._devices(devices)
        h = C.c_void_p()
        _lib.check(_lib.load().clc_group_create_synthetic(C.byref(h), C.byref(d), arr, n), "clc_group_create_synthetic")
        return cls(h)

    def close(self):
        if self._h is not None:
            self._L.clc_group_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def sizes(self):
        n, nf, npts = C.c_int(), C.c_int64(), C.c_int64()
        _lib.check(self._L.clc_group_size(self._h, C.byref(n), C.byref(nf), C.byref(npts)), "clc_group_size")
        return n.value, nf.value, npts.value

    def problem(self, index):
        """Borrowed view of shard `index` (do not close it)."""
        h = C.c_void_p()
        _lib.check(self._L.clc_group_problem(self._h, int(index), C.byref(h)), "clc_group_problem")
        p = Problem(h)
        p.close = lambda: None  # owned by the group
        return p

    def eval(self, pose7):
        pose7 = np.ascontiguousarray(pose7, dtype=np.float64)
        H, g, cost = np.empty((6, 6)), np.empty(6), C.c_double()
        _lib.check(self._L.clc_group_eval(self._h, _dp(pose7), _dp(H), _dp(g), C.byref(cost)), "clc_group_eval")
        return cost.value, H, g

    def solve(self, pose7, options: LmOptions | None = None, trace_cap=256):
        x = np.ascontiguousarray(pose7, dtype=np.float64).copy()
        o = options if options is not None else default_options()
        s = LmSummary()
        tr = (LmIteration * trace_cap)()
        _lib.check(self._L.clc_group_solve_lm(self._h, _dp(x), C.byref(o), C.byref(s), tr, trace_cap), "clc_group_solve_lm")
        return x, s, [tr[i] for i in range(min(s.num_iterations, trace_cap))]

    def information(self, pose7):
        pose7 = np.ascontiguousarray(pose7, dtype=np.float64)
        H, b, sv, chi = np.empty((6, 6)), np.empty(6), np.empty(6), C.c_double()
        self.last_V = np.empty((6, 6))
        _lib.check(self._L.clc_group_information(self._h, _dp(pose7), _dp(H), _dp(b), C.byref(chi), _dp(sv), _dp(self.last_V)),
                   "clc_group_information")
        return H, b, chi.value, sv

    def closed_form(self):
        T, AtA, Atb, un = np.empty(16), np.empty((9, 9)), np.empty(9), C.c_int()
        _lib.check(self._L.clc_group_closed_form(self._h, _dp(T), C.byref(un), _dp(AtA), _dp(Atb)), "clc_group_closed_form")
        return T.reshape(4, 4), bool(un.value), AtA, Atb


def upload_stats():
    """Statistics of this process's most recent host -> HBM upload (clc_upload_last_stats)."""
    t, w, b = C.c_double(), C.c_double(), C.c_int64()
    ch, th, di = C.c_int(), C.c_int(), C.c_int()
    _lib.load().clc_upload_last_stats(C.byref(t), C.byref(w), C.byref(b), C.byref(ch), C.byref(th), C.byref(di))
    return dict(total_ms=t.value, pack_wait_ms=w.value, bytes_h2d=b.value, chunks=ch.value, pack_threads=th.value, direct=bool(di.value))


def debug_pack(frames, a, b, xy):
    """What the pack threads write for the local point range [a, b) (test hook; no CUDA)."""
    g = _Gather(np.zeros((len(frames), 7)), frames)
    out = np.empty((b - a) * (2 if xy else 3))
    nonplanar = C.c_int(-1)
    _lib.check(_lib.load().clc_debug_pack(len(frames), g.ptrs, _ip(g.counts), int(a), int(b), int(bool(xy)), _dp(out),
                                          C.byref(nonplanar)), "clc_debug_pack")
    return out.reshape(-1, 2 if xy else 3), nonplanar.value


class Comm:
    """NCCL communicator of the solve (one per rank / GPU), shareable between problems on the same device."""

    def __init__(self, unique_id: bytes, nranks: int, rank: int, device: int = -1):
        self._L = _lib.load()
        self._h = C.c_void_p()
        buf = C.create_string_buffer(unique_id, 128)
        _lib.check(self._L.clc_comm_create(C.byref(self._h), buf, int(nranks), int(rank), int(device)), "clc_comm_create")
        self.nranks, self.rank = int(nranks), int(rank)

    def p2p_export(self) -> bytes:
        """64-byte CUDA IPC handle of this rank's mailbox (for the fused in-kernel all-reduce over NVLink)."""
        buf = C.create_string_buffer(64)
        _lib.check(self._L.clc_comm_p2p_export(self._h, buf), "clc_comm_p2p_export")
        return buf.raw

    def p2p_import(self, handles):
        """handles: the exported handles of all ranks, in rank order."""
        blob = b"".join(handles)
        if len(blob) != 64 * self.nranks:
            raise ValueError("need one 64-byte handle per rank")
        _lib.check(self._L.clc_comm_p2p_import(self._h, C.create_string_buffer(blob, len(blob))), "clc_comm_p2p_import")

    def enable_p2p(self, all_gather):
        """all_gather(bytes) -> list[bytes] over the ranks (e.g. torch.distributed.all_gather_object)."""
        self.p2p_import(all_gather(self.p2p_export()))

    def close(self):
        if self._h is not None:
            self._L.clc_comm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def comm_unique_id() -> bytes:
    buf = C.create_string_buffer(128)
    _lib.check(_lib.load().clc_comm_unique_id(buf), "clc_comm_unique_id")
    return buf.raw


def shard_range(n_frames, nranks, rank, offsets=None):
    b, e = C.c_int64(), C.c_int64()
    off = None if offsets is None else np.ascontiguousarray(offsets, dtype=np.int64)
    _lib.check(_lib.load().clc_shard_range(int(n_frames), _ip(off), int(nranks), int(rank), C.byref(b), C.byref(e)),
               "clc_shard_range")
    return b.value, e.value


def T_to_pose7(T):
    T = np.ascontiguousarray(T, dtype=np.float64).reshape(16)
    p = np.empty(7)
    _lib.load().clc_T_to_pose7(_dp(T), _dp(p))
    return p


def pose7_to_T(p):
    p = np.ascontiguousarray(p, dtype=np.float64)
    T = np.empty(16)
    _lib.load().clc_pose7_to_T(_dp(p), _dp(T))
    return T.reshape(4, 4)


def launch_count() -> int:
    return int(_lib.load().clc_launch_count())


class pinned_array:
    """numpy view of CUDA pinned host memory (upload buffers for the end-to-end measurement)."""

    def __init__(self, shape, dtype=np.float64):
        self._L = _lib.load()
        self.nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        self._ptr = C.c_void_p()
        _lib.check(self._L.clc_host_alloc(C.byref(self._ptr), self.nbytes), "clc_host_alloc")
        buf = (C.c_char * max(self.nbytes, 1)).from_address(self._ptr.value)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def free(self):
        if self._ptr is not None and self._ptr.value:
            self.array = None
            self._L.clc_host_free(self._ptr)
            self._ptr = None


def problems_from_scans(ranges, scan_stamps, angle_min, angle_increment, range_min, pose_stamps, pose_wc, max_dt=0.02,
                        line_fit_max_iterations=10, with_edges=False, use_loss=True, cauchy_a=0.05, device=-1):
    """The offline driver's scan loop on the device (clc_problems_create_from_scans, reference main/calibr_offline.cpp:86-155):
    ranges[n_scans, n_beams] float32 (a pinned_array's array is used as the DMA source), scan_stamps[n_scans],
    pose_stamps[n_poses], pose_wc[n_poses, 7] = qx qy qz qw x y z of T_wc.  Returns (points_problem, on_line_problem,
    scan_info[n_scans, 4] int32 = seg_start, seg_end, nearest pose, frame (-1: none), scan_line[n_scans, 2] (NaN where no
    frame)).  The points problem holds Oberserve::points, the on-line problem Oberserve::points_on_line (+ edge residuals
    when with_edges)."""
    L = _lib.load()
    r = np.asarray(ranges)
    if r.dtype != np.float32:
        raise ValueError("ranges must be float32 (sensor_msgs/LaserScan::ranges)")
    r = np.ascontiguousarray(r)
    if r.ndim != 2:
        raise ValueError("ranges must be [n_scans, n_beams]")
    ts = np.ascontiguousarray(scan_stamps, dtype=np.float64).reshape(-1)
    if ts.shape[0] != r.shape[0]:
        raise ValueError("one stamp per scan is needed")
    tp = np.ascontiguousarray(pose_stamps, dtype=np.float64).reshape(-1)
    pw = np.ascontiguousarray(pose_wc, dtype=np.float64).reshape(-1, 7)
    if pw.shape[0] != tp.shape[0]:
        raise ValueError("one pose per pose stamp is needed")
    d = ScanDesc()
    d.n_scans, d.n_beams = r.shape
    d.ranges = r.ctypes.data_as(C.POINTER(C.c_float))
    d.scan_stamp = _dp(ts)
    d.angle_min, d.angle_increment, d.range_min = float(angle_min), float(angle_increment), float(range_min)
    d.n_poses, d.pose_stamp, d.pose_wc = tp.shape[0], _dp(tp), _dp(pw)
    d.max_dt, d.line_fit_max_iterations, d.with_edges = float(max_dt), int(line_fit_max_iterations), int(bool(with_edges))
    d.use_loss, d.cauchy_a, d.device = int(bool(use_loss)), float(cauchy_a), int(device)
    info = np.empty((r.shape[0], 4), dtype=np.int32)
    lines = np.empty((r.shape[0], 2))
    hp, hl = C.c_void_p(), C.c_void_p()
    _lib.check(L.clc_problems_create_from_scans(C.byref(d), C.byref(hp), C.byref(hl), info.ctypes.data_as(C.POINTER(C.c_int32)),
                                                _dp(lines)), "clc_problems_create_from_scans")
    return Problem(hp), Problem(hl), info, lines


def scan_stats():
    """Phase times (ms) and PCIe bytes of this thread's most recent problems_from_scans (clc_scan_last_stats)."""
    ms, h2d, d2h = (C.c_float * 6)(), C.c_int64(), C.c_int64()
    _lib.check(_lib.load().clc_scan_last_stats(ms, C.byref(h2d), C.byref(d2h)), "clc_scan_last_stats")
    names = ("h2d", "classify", "scan", "gather", "line_fit", "finish")
    return dict(**{k + "_ms": float(v) for k, v in zip(names, ms)}, bytes_h2d=h2d.value, bytes_d2h=d2h.value)


def LineFittingCeres(Points, Line: np.ndarray, max_num_iterations=10):
    """reference src/LaseCamCalCeres.cpp:401-433: ``Line`` (2,) is the start value on entry and the fit on exit."""
    pts = np.ascontiguousarray(Points, dtype=np.float64).reshape(-1, 3)
    line = np.ascontiguousarray(Line, dtype=np.float64).copy()
    _lib.check(_lib.load().clc_line_fit_points(_dp(pts), pts.shape[0], _dp(line), int(max_num_iterations)), "clc_line_fit_points")
    Line[...] = line


# ---- the reference's two entry points -------------------------------------------------------------------------

def CamLaserCalClosedSolution(obs, Tlc: np.ndarray, verbose=True):
    """reference src/LaseCamCalCeres.cpp:112-203.  Writes T_lc (4x4) into ``Tlc``; uses obs[i].points_on_line."""
    with Problem.from_observations(obs, use_linefitting_data=True, use_boundary_constraint=False) as p:
        return closed_form_on(p, Tlc, verbose)


def closed_form_on(p: Problem, Tlc: np.ndarray, verbose=True):
    """CamLaserCalClosedSolution on a problem that already holds the points_on_line (e.g. from problems_from_scans)."""
    T, unobservable, _, _ = p.closed_form()
    if unobservable and verbose:
        print("\n~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~")
        print(" Notice Notice Notice: system unobservable !!!!!!!")
        print("~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~~\n")
    Tlc[...] = T
    if verbose:
        print("------- Closed-form solution Tlc: -------\n", Tlc)
    return unobservable


def CamLaserCalibration(obs, Tcl: np.ndarray, use_linefitting_data=True, use_boundary_constraint=False, verbose=True,
                        options: LmOptions | None = None):
    """reference src/LaseCamCalCeres.cpp:213-383.  ``Tcl`` (4x4) is the initial guess on entry and the result on
    exit (bottom row untouched, :313-314).  Returns a dict with the solver summary and the analysis-tail outputs the
    reference prints (H singular values, null-space basis, chi2/2)."""
    with Problem.from_observations(obs, use_linefitting_data, use_boundary_constraint) as p:
        return calibrate_on(p, Tcl, verbose, options)


def calibrate_on(p: Problem, Tcl: np.ndarray, verbose=True, options: LmOptions | None = None):
    """CamLaserCalibration on a problem that already holds the selected point set (e.g. from problems_from_scans)."""
    pose = T_to_pose7(Tcl)  # :215-219
    x, s, trace = p.solve(pose, options)
    T = pose7_to_T(x)
    Tcl[:3, :] = T[:3, :]  # :311-314
    H, b, chi, sv = p.information(x)  # :318-362
    V = p.last_V
    report = dict(termination=TERMINATION.get(s.termination, "?"), iterations=s.num_iterations,
                  initial_cost=s.initial_cost, final_cost=s.final_cost, trace=trace, H=H, b=b, chi2=chi / 2.0,
                  singular_values=sv, V=V, pose7=x, device_ms=s.device_ms, num_sweeps=s.num_sweeps)
    if verbose:
        print(f"LM (on device): {report['termination']}, {s.num_iterations} iterations, cost {s.initial_cost:.6e} -> "
              f"{s.final_cost:.6e}, {s.device_ms:.3f} ms")
        print("----- H singular values--------:\n", sv)
        n_null = int(np.sum(sv < 1e-8))  # :368-379
        if n_null > 0:
            print("====== null space basis, it's means the unobservable direction for Tcl ======")
            print("       please note the unobservable direction is for Tcl, not for Tlc        ")
            print(V[:, 6 - n_null:])  # svd.matrixV().rightCols(n), :378
        print("\nrecover chi2: ", chi / 2.0)
    return report
