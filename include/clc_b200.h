/*
 * clc_b200.h -- C ABI of libclc_b200.so: the B200-native (sm_100a) implementation of the camera<-laser
 * extrinsic solve of MegviiRobot/CamLaserCalibraTool.
 *
 * The reference has no FFI: its "operator API" for this path is four C++ free functions plus one struct
 * (reference include/LaseCamCalCeres.h:11-29).  This header is the boundary a replacement of
 * reference src/LaseCamCalCeres.cpp binds to; camlasercalibratool_b200/host/LaseCamCalB200.cpp is that
 * replacement (same signatures, same Oberserve struct) and INTEGRATION.md shows the CMake change.
 *
 * Plain C, POD only, int status codes (0 = CLC_OK), no exceptions cross the boundary, no torch types.
 * There is NO CPU fallback: every entry point fails with CLC_ERR_CUDA if no sm_100 device is usable.
 *
 * Data conventions (identical to the marshalled form of std::vector<Oberserve>):
 *   frame_pose[f*7 .. +7] = qx,qy,qz,qw (Eigen coeff order of Oberserve::tagPose_Qca), tx,ty,tz (tagPose_tca)
 *                           -- reference include/LaseCamCalCeres.h:20-21
 *   offsets[n_frames+1]   = CSR delimiters of the frames inside `points`
 *   points[P*3]           = AoS x,y,z doubles: the calibration point set the reference selects at
 *                           src/LaseCamCalCeres.cpp:233-237 (obs.points or obs.points_on_line)
 *   edge_points[f*6..+6]  = obs[f].points.front() then obs[f].points.back() (src/LaseCamCalCeres.cpp:278-279);
 *                           non-NULL enables the board-edge residuals of :258-294
 *   pose7                 = tx,ty,tz,qx,qy,qz,qw: the Ceres parameter block of T_cl (:219)
 *   4x4 matrices are row-major.
 */
#ifndef CLC_B200_H
#define CLC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CLC_OK 0
#define CLC_ERR_INVALID 1  /* bad argument */
#define CLC_ERR_CUDA 2     /* CUDA runtime / no usable device */
#define CLC_ERR_NCCL 3     /* NCCL missing or a collective failed */
#define CLC_ERR_STATE 4    /* call not valid in this state */

typedef struct clc_problem clc_problem; /* opaque, device-resident problem (one per GPU / rank) */

/* replaces: the argument marshalling of CamLaserCalibration()/CamLaserCalClosedSolution(),
 * reference src/LaseCamCalCeres.cpp:213-295 and :112-159 */
typedef struct {
  int64_t n_frames;
  const double* frame_pose;  /* host [n_frames*7] */
  const int64_t* offsets;    /* host [n_frames+1] */
  const double* points;      /* host [offsets[n_frames]*3]; pinned memory uploads at full PCIe rate */
  const double* edge_points; /* host [n_frames*6] or NULL */
  int use_loss;              /* 1: CauchyLoss(cauchy_a*scale), reference :212,:249 */
  double cauchy_a;           /* 0.05 */
  int device;                /* CUDA ordinal, -1 = current device */
} clc_problem_desc;

/* The same problem as the caller of the reference holds it: one separate array of Vector3d per frame -- Oberserve::points or
 * ::points_on_line of every element of the std::vector<Oberserve> the reference's functions take BY VALUE
 * (reference include/LaseCamCalCeres.h:22-23,28; Eigen::Vector3d is three contiguous doubles, so
 * obs[f].points.data() is frame_points[f]).  The library gathers the frames itself (pack threads -> pinned ring -> PCIe
 * -> layout kernel, all overlapped); pageable memory is fine.  replaces: the per-point loops of
 * reference src/LaseCamCalCeres.cpp:233-254 (one heap CostFunction + LossFunction per point). */
typedef struct {
  int64_t n_frames;
  const double* frame_pose;          /* host [n_frames*7] */
  const double* const* frame_points; /* host [n_frames]: AoS xyz of frame f, frame_counts[f] points */
  const int64_t* frame_counts;       /* host [n_frames] */
  const double* edge_points;         /* host [n_frames*6] or NULL */
  int use_loss;
  double cauchy_a;
  int device;                        /* ignored by the clc_group_* entry points (they take a device list) */
} clc_gather_desc;

/* replaces: GenerateSimData(), reference main/calibr_simulation.cpp:10-108, scaled to n_frames x beams and run
 * on the device (the 48 GB of BASELINE config 4 cannot pass through std::vector<Oberserve>). */
typedef struct {
  int64_t n_frames_total; /* frames of the whole (all-rank) problem; RNG counters are global frame ids */
  int64_t frame_begin;    /* this problem holds frames [frame_begin, frame_end) */
  int64_t frame_end;
  int64_t beams;          /* points per frame (exact-M mode: every frame has exactly `beams` points) */
  uint64_t seed;
  double sigma;           /* range noise along the ray, metres */
  int with_edges;         /* also generate the two board-edge residual points per frame */
  int use_loss;
  double cauchy_a;
  int device;
  /* Optional camera measurement chain (SURVEY.md 8(f) rank 2): the board pose the calibration sees is then ESTIMATED from
   * noisy corner pixels -- kalibr-grid corners -> Camera::spaceToPlane -> pixel noise -> Camera::liftProjective -> planar
   * PnP, as reference src/calcCamPose.cpp:279-292,211-236 does with cv::solvePnP -- while the laser hits the true board.
   * camera_model 0: exact poses (the reference simulation); 1: pinhole + radtan, intrinsics = fx fy cx cy k1 k2 p1 p2
   * (reference config/calibra_config_pinhole.yaml); 2: equidistant (Kannala-Brandt), intrinsics = mu mv u0 v0 k2 k3 k4 k5
   * (reference config/calibra_config.yaml).  Boards are redrawn until all grid corners fall inside the image. */
  int camera_model;
  double camera_intrinsics[8];
  double pixel_sigma;     /* std of the corner noise in pixels */
  int image_width, image_height; /* 752 x 480 in the reference configs */
  int grid_rows, grid_cols;      /* 6 x 6 */
  double tag_size, tag_spacing;  /* 0.055 m, 0.3 */
} clc_synthetic_desc;

/* Ceres Solver::Options subset, defaults = reference src/LaseCamCalCeres.cpp:302-304 + Ceres defaults */
typedef struct {
  int max_num_iterations;           /* 100 */
  double initial_trust_region_radius; /* 1e4 */
  double max_trust_region_radius;   /* 1e16 */
  double min_trust_region_radius;   /* 1e-32 */
  double min_relative_decrease;     /* 1e-3 */
  double min_lm_diagonal;           /* 1e-6 */
  double max_lm_diagonal;           /* 1e32 */
  double function_tolerance;        /* 1e-6 */
  double gradient_tolerance;        /* 1e-10 */
  double parameter_tolerance;       /* 1e-8 */
  int max_num_consecutive_invalid_steps; /* 5 */
  int jacobi_scaling;               /* 1 */
  int iterations_per_sync;          /* LM iterations enqueued between host polls of the device `done` flag (8; the first batch of a solve is twice as long) */
  int reserved;
} clc_lm_options;

/* termination codes (Ceres TerminationType + the tolerance that fired) */
#define CLC_TERM_RUNNING 0
#define CLC_TERM_CONVERGENCE_FUNCTION 1
#define CLC_TERM_CONVERGENCE_PARAMETER 2
#define CLC_TERM_CONVERGENCE_GRADIENT 3
#define CLC_TERM_CONVERGENCE_MIN_RADIUS 4
#define CLC_TERM_NO_CONVERGENCE 5
#define CLC_TERM_FAILURE 6

/* one row of Ceres' IterationSummary */
typedef struct {
  int iteration;
  int step_is_valid;
  int step_is_successful;
  int reserved;
  double cost;
  double cost_change;
  double gradient_max_norm;
  double step_norm;
  double relative_decrease;
  double trust_region_radius;
} clc_lm_iteration;

typedef struct {
  int termination;
  int num_iterations;          /* rows written to the trace (iteration 0 included) */
  int num_successful_steps;
  int num_unsuccessful_steps;
  int num_sweeps;              /* launches of the fused residual+Jacobian+reduce kernel that did work */
  int reserved;
  double initial_cost;
  double final_cost;
  double device_ms;            /* CUDA-event time of the whole on-device solve on this rank */
} clc_lm_summary;

const char* clc_last_error(void);
int clc_device_count(int* count);

void clc_lm_default_options(clc_lm_options* opt);

/* Uploads (H2D) and lays the problem out in HBM (SoA points, per-frame planes).  replaces: problem assembly,
 * reference src/LaseCamCalCeres.cpp:222-295 (no per-residual heap objects are created). */
int clc_problem_create(clc_problem** out, const clc_problem_desc* desc);
/* Same from per-frame arrays (the marshalled form of std::vector<Oberserve> without flattening it on the host). */
int clc_problem_create_gather(clc_problem** out, const clc_gather_desc* desc);
/* Same, generated on the device. */
int clc_problem_create_synthetic(clc_problem** out, const clc_synthetic_desc* desc);
int clc_problem_destroy(clc_problem* p);

/* Sizes and read-back (tests / the C++ simulation driver). Any output pointer may be NULL. */
int clc_problem_sizes(const clc_problem* p, int64_t* n_frames, int64_t* n_points, int* has_edges);
int clc_problem_download(const clc_problem* p, double* frame_pose, int64_t* offsets, double* points,
                         double* edge_points, double* planes /* [n_frames*4] n,d in the camera frame */);
/* Synthetic problems with a camera model: the TRUE board poses [n_frames*7] (frame_pose above holds the estimated ones). */
int clc_problem_download_true_poses(const clc_problem* p, double* frame_pose_true);

/* THE FUSED KERNEL (K1): one sweep over every residual at `pose7` -> H = sum J~^T J~ (row-major 6x6),
 * g = sum J~^T r~, cost = 1/2 sum rho, with the Cauchy correction applied.  All-reduced over the ranks when a
 * communicator is attached.  replaces: one ceres Evaluate over all PointInPlaneFactor residual blocks,
 * reference src/LaseCamCalCeres.cpp:43-66 + Ceres Corrector.  Synchronous.  H36/g6 may be NULL. */
int clc_eval(clc_problem* p, const double pose7[7], double H36[36], double g6[6], double* cost);

/* replaces: ceres::Solve() at reference src/LaseCamCalCeres.cpp:306-307 with the options of :302-304.
 * pose7 is in/out.  trace may be NULL.  Collective over the communicator's ranks.
 * The whole Levenberg-Marquardt loop runs on the device: one K1 sweep per iteration, chained with programmatic dependent
 * launch, the host only polls a `done` flag; problems of the reference's own size (<= 16384 residuals, single rank) are solved
 * by ONE launch of the one-cluster kernel K2 (csrc/clc_small.cuh) that keeps the residuals in registers. */
int clc_solve_lm(clc_problem* p, double pose7[7], const clc_lm_options* opt, clc_lm_summary* summary,
                 clc_lm_iteration* trace, int trace_cap);

/* replaces: the analysis tail, reference src/LaseCamCalCeres.cpp:318-381: un-robustified H, b = -J^T r,
 * chi = sum r^2 (scale kept, no edge residuals), singular values of H (descending) and the matching right singular
 * vectors as the columns of V36 (row-major 6x6): the last n columns span the null space the reference prints when n
 * singular values are below 1e-8 (:368-379).  Any output may be NULL. */
int clc_information(clc_problem* p, const double pose7[7], double H36[36], double b6[6], double* chi,
                    double singular_values6[6], double V36[36]);

/* replaces: CamLaserCalClosedSolution(), reference src/LaseCamCalCeres.cpp:112-203.  Tlc16 row-major.
 * AtA81/Atb9 (the 9x9 normal equations) may be NULL. */
int clc_closed_form(clc_problem* p, double Tlc16[16], int* unobservable, double AtA81[81], double Atb9[9]);

/* replaces: LineFittingCeres(), reference src/LaseCamCalCeres.cpp:385-433 (the step before the solve: SURVEY.md 8(f)),
 * batched: fits m0 x + m1 y + 1 = 0 (CauchyLoss(0.05), <= max_num_iterations Ceres LM iterations, reference: 10) to
 * the x,y of every frame's points of the problem, one warp per frame, the whole loop on the device.
 * lines[n_frames*2] (host): start values in (the reference's caller passes them uninitialised), fits out.
 * info[n_frames*4] (host, optional): termination code, LM iterations, sweeps, final cost per frame.
 * Local to the rank's shard (no collective). */
int clc_problem_line_fit(clc_problem* p, double* lines, int max_num_iterations, double* info);
/* The reference's per-scan call shape: one scan of n points (AoS xyz, z ignored), line[2] in/out. */
int clc_line_fit_points(const double* points_xyz, int64_t n, double line[2], int max_num_iterations);

/* replaces: TranScanToPoints() + AutoGetLinePts(), reference src/utilities.cpp:181-215 and src/selectScanPoints.cpp:17-190
 * (without the OpenCV debug drawing), batched over scans: for every LaserScan (n_beams float ranges, angle of beam i =
 * angle_min + i * angle_increment) the inclusive beam-index range [seg_start, seg_end] of the laser segment on the board,
 * or -1/-1 when none is found.  Host arrays in/out; device = CUDA ordinal or -1. */
int clc_scan_segments(const float* ranges, int64_t n_scans, int64_t n_beams, double angle_min, double angle_increment,
                      double range_min, int32_t* seg_start, int32_t* seg_end, int device);

/* replaces: the scan loop of the offline driver, reference main/calibr_offline.cpp:86-155 -- TranScanToPoints
 * (src/utilities.cpp:181-215), AutoGetLinePts (src/selectScanPoints.cpp:17-190), the nearest tag pose (:103-116),
 * LineFittingCeres (src/LaseCamCalCeres.cpp:385-433), the line end points (:126-142) and the Oberserve it fills (:144-150)
 * -- for a whole batch of LaserScans, on the device.  Only the ranges, the stamps and the poses cross PCIe; the two problems
 * the driver then solves are built device to device:
 *   *points  : Oberserve::points of every frame (CamLaserCalibration(obs, Tcl, false), :170), no edge residuals;
 *   *on_line : Oberserve::points_on_line, two per frame (CamLaserCalClosedSolution, :167), with the board-edge residuals
 *              (front and back of obs.points) when with_edges.
 * A frame is a scan with a board segment whose nearest pose (linear search: strict <, ties to the lowest index, NaN stamps
 * never match, poses in any order) lies strictly within max_dt; frames keep scan order.  frame_pose = (qwc^-1, -R(qwc^-1) twc)
 * with Eigen semantics (no normalisation).  Points are the beams seg_start..seg_end of the scan (invalid beams inside a
 * segment included as (1000, 1000), as the reference keeps them), z = 0.  The lines are fitted from a zero start with
 * CauchyLoss(0.05).  Both problems are planar by construction.  Either output may be NULL; on failure both are NULL.
 * scan_info[n_scans*4] (optional) = seg_start, seg_end, nearest pose (-1: no segment or no pose), frame (-1: not kept);
 * scan_line[n_scans*2] (optional) = the fitted line of a kept scan, NaN otherwise.  Bit-reproducible. */
typedef struct {
  int64_t n_scans, n_beams;
  const float* ranges;          /* host [n_scans*n_beams], LaserScan::ranges row by row; pinned memory is the DMA source */
  const double* scan_stamp;     /* host [n_scans], header.stamp.toSec() */
  double angle_min, angle_increment, range_min; /* the LaserScan fields */
  int64_t n_poses;
  const double* pose_stamp;     /* host [n_poses] */
  const double* pose_wc;        /* host [n_poses*7] qx qy qz qw x y z of T_wc (the layout of clc_estimate_board_poses) */
  double max_dt;                /* 0.02 s in the reference (:116) */
  int line_fit_max_iterations;  /* 10 */
  int with_edges;               /* board-edge residuals on the on-line problem (use_boundary_constraint) */
  int use_loss;
  double cauchy_a;
  int device;
} clc_scan_desc;
int clc_problems_create_from_scans(const clc_scan_desc* d, clc_problem** points, clc_problem** on_line, int32_t* scan_info,
                                   double* scan_line);

/* Board poses from detected tag corners, batched: the arithmetic of CamPoseEst::calcCamPose after the tag detector
 * (reference src/calcCamPose.cpp:270-294: liftProjective of every corner, x/z y/z as cv::Point2f) and of
 * CamPoseEst::EstimatePose (:211-236: solvePnP with identity intrinsics on the kalibr-grid object points :114-136,
 * T_wc = T_cw^-1) -- what main/kalibratag_detector_node.cpp turns into apriltag_pose.txt.  No image processing.
 * camera_model 1 = pinhole + radtan (fx fy cx cy k1 k2 p1 p2), 2 = equidistant / Kannala-Brandt (mu mv u0 v0 k2 k3 k4 k5).
 * Frame f owns detections det_offsets[f] .. det_offsets[f+1] (ascending tag id); corners_uv[D*8] = 4 corners (u, v) per
 * detection in detector order.  pose_wc[n_frames*7] = (qx qy qz qw x y z) of T_wc; ok[f] = 0 (identity pose) for fewer
 * than 4 points, a tag id outside the grid or a degenerate configuration. */
typedef struct clc_camera_desc {
  int camera_model;
  double intrinsics[8];
  int grid_rows, grid_cols; /* april grid; a single tag is a 1 x 1 grid */
  double tag_size;          /* metres */
  double tag_spacing;       /* gap / tag_size (kalibr convention) */
} clc_camera_desc;
int clc_estimate_board_poses(const clc_camera_desc* cam, int64_t n_frames, const int64_t* det_offsets, const int32_t* tag_ids,
                             const float* corners_uv, double* pose_wc, int32_t* ok, int device);

/* Eigen-equivalent conversions used on both sides of the boundary (reference :215-219 and :311-314). */
void clc_T_to_pose7(const double T16[16], double pose7[7]);
void clc_pose7_to_T(const double pose7[7], double T16[16]);

/* ---- multi-GPU: one process per GPU, frames sharded by the caller, 28-double all-reduce per sweep ---------- */
/* Balanced contiguous frame range of `rank` (by point count when offsets != NULL, else by frame count). */
int clc_shard_range(int64_t n_frames, const int64_t* offsets, int nranks, int rank, int64_t* begin, int64_t* end);
/* NCCL bootstrap: rank 0 calls clc_comm_unique_id, ships the 128 bytes to every rank by any means
 * (torch.distributed, MPI, a file); every rank creates its communicator (collective) and attaches it to any number
 * of problems on that device.  The communicator is borrowed: it must outlive the problems it is attached to.
 * Attaching NULL detaches. */
typedef struct clc_comm clc_comm;
int clc_comm_unique_id(void* id128);
int clc_comm_create(clc_comm** out, const void* id128, int nranks, int rank, int device);
int clc_comm_destroy(clc_comm* comm);
int clc_problem_attach_comm(clc_problem* p, clc_comm* comm);
/* Fused all-reduce over NVLink peer memory: every rank exports a 64-byte IPC handle of its mailbox, the handles of
 * all ranks (rank order, nranks*64 bytes) are shipped to every rank by any means, and every rank imports them.  From
 * then on the last block of every sweep kernel exchanges the 28 sums with direct peer stores and runs the LM update in
 * the same launch (no NCCL call, no extra kernel).  Requires one process per GPU on one NVLink/NVSwitch node. */
int clc_comm_p2p_export(clc_comm* comm, void* handle64);
int clc_comm_p2p_import(clc_comm* comm, const void* handles /* [nranks*64] */);
/* all-reduce mode of a problem: 0 = ncclAllReduce on the solve stream between the kernels,
 * 1 = fused in-kernel peer exchange (needs clc_comm_p2p_import; the default once it has been called) */
int clc_problem_set_allreduce_mode(clc_problem* p, int mode);

/* ---- in-process multi-GPU: ONE process (one host thread) drives G devices ---------------------------------------
 * What lets the unmodified reference callers (main/calibr_simulation.cpp:130, main/calibr_offline.cpp:170 -- one call of
 * CamLaserCalibration() from one process) use every GPU of the box: the frames are sharded over the devices by point
 * count (clc_shard_range), every device holds its shard for the whole solve, and the last block of every sweep kernel
 * exchanges the 28 sums with plain peer stores (cudaDeviceEnablePeerAccess; the same sequence-tagged mailbox protocol as
 * the multi-process path, no IPC handles, no NCCL).  All devices run the identical LM update.  A group of one device is
 * a plain problem.  devices[i] = CUDA ordinal (-1 = current); an ordinal may appear only once. */
typedef struct clc_group clc_group;
int clc_group_create_gather(clc_group** out, const clc_gather_desc* desc, const int* devices, int n_devices);
/* desc->frame_begin..frame_end is the range the GROUP holds (split evenly over its devices); desc->device is ignored */
int clc_group_create_synthetic(clc_group** out, const clc_synthetic_desc* desc, const int* devices, int n_devices);
int clc_group_destroy(clc_group* g);
int clc_group_size(const clc_group* g, int* n_devices, int64_t* n_frames, int64_t* n_points);
int clc_group_problem(clc_group* g, int index, clc_problem** out); /* borrowed: shard `index` (tests, measurement) */
/* the collective forms of clc_eval / clc_solve_lm / clc_information / clc_closed_form (same outputs) */
int clc_group_eval(clc_group* g, const double pose7[7], double H36[36], double g6[6], double* cost);
int clc_group_solve_lm(clc_group* g, double pose7[7], const clc_lm_options* opt, clc_lm_summary* summary,
                       clc_lm_iteration* trace, int trace_cap);
int clc_group_information(clc_group* g, const double pose7[7], double H36[36], double b6[6], double* chi,
                          double singular_values6[6], double V36[36]);
int clc_group_closed_form(clc_group* g, double Tlc16[16], int* unobservable, double AtA81[81], double Atb9[9]);
/* The device list the reference-facing drop-in uses (its signatures have no device argument): environment variable
 * CLC_DEVICES = "0,1,2,3" | "all" | unset (the current device only).  Writes at most `cap` ordinals. */
int clc_default_devices(int* devices, int cap, int* n);

/* ---- measurement hooks (bench.py) ---------------------------------------------------------------------- */
/* Launches K1 `n` times at pose7 on the problem's stream; each launch is bracketed by its own CUDA events.
 * flush_l2 != 0 overwrites a buffer larger than L2 between launches (outside the timed brackets).
 * ms_each[n] receives the per-launch device times.  No collective, local shard only. */
int clc_bench_eval(clc_problem* p, const double pose7[7], int n, int flush_l2, float* ms_each);
/* Algorithmic bytes of one K1 launch on this problem: 24*P + 40*N + 56*edges + 224 (SURVEY.md section 8(d)). */
int clc_problem_algorithmic_bytes(const clc_problem* p, int64_t* bytes);
/* Bytes one K1 launch actually streams: the figure above with 16 instead of 24 bytes per point when the planar
 * (two-stream) kernels are active. */
int clc_problem_streamed_bytes(const clc_problem* p, int64_t* bytes);
/* Planar data.  A 2-D laser delivers z == 0 for every point (reference src/utilities.cpp:207, main/calibr_simulation.cpp:82,88,
 * main/calibr_offline.cpp:141-142) although Oberserve::points is a Vector3d.  The upload detects this; the library then
 * drops the z stream from HBM and runs two-stream kernels whose results equal the general ones (up to summation order) on such
 * data (SURVEY.md 8(d): a separate roofline row, 16 B per residual).  mode 1 = automatic (default), 0 = always the
 * general three-stream kernels (an all-zero z stream is re-materialised if it was dropped).  Problems too small to give
 * every warp of the grid a 256-point stage (about 6*10^5 points on a B200) are latency-bound and stay on the general
 * kernels in either mode (environment override for tests: CLC_PLANAR_MIN_POINTS). */
int clc_problem_set_planar_mode(clc_problem* p, int mode);
/* Statistics of this process's most recent host -> HBM point upload: wall time of the pipeline, time the issuing thread
 * waited for the pack threads, bytes that crossed PCIe (16 per point while every z is 0, else 24), chunks, pack threads,
 * direct = 1 when the caller's buffer was pinned and used as the DMA source.  Any pointer may be NULL. */
int clc_upload_last_stats(double* total_ms, double* pack_wait_ms, int64_t* bytes_h2d, int* chunks, int* pack_threads,
                          int* direct);
/* Test hook, no CUDA: what the pack threads write for the local point range [a, b) of a gathered problem -- packed x,y
 * pairs (xy != 0; *nonplanar = a z != 0 or NaN was met) or packed x,y,z. */
int clc_debug_pack(int64_t n_frames, const double* const* frame_points, const int64_t* frame_counts, int64_t a, int64_t b,
                   int xy, double* out, int* nonplanar);
/* Phase times (CUDA events, ms) of this thread's most recent clc_problems_create_from_scans: H2D, classify, scan (+ the
 * D2H of the totals), gather (+ allocation), line fit (+ on-line build), finish; and the bytes it moved H2D / D2H. */
int clc_scan_last_stats(float phase_ms6[6], int64_t* bytes_h2d, int64_t* bytes_d2h);
/* Raw PCIe yardstick: `reps` host(pinned) -> device copies of `bytes` on `device`, each timed with CUDA events. */
int clc_bench_h2d(int64_t bytes, int device, int reps, float* ms_each);
/* Bytes clc_solve_lm reads back per solve (LM state + iteration trace). */
int64_t clc_solve_readback_bytes(void);
/* Pinned host memory for upload buffers. */
int clc_host_alloc(void** ptr, int64_t bytes);
int clc_host_free(void* ptr);
/* Number of kernel launches issued by this library since load (bench.py's gpu_launches). */
int64_t clc_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* CLC_B200_H */
