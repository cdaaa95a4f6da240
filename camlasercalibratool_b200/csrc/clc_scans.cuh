// clc_scans.cuh -- the two calibration problems built on the device straight from LaserScan ranges: the glue of the
// reference's offline driver (main/calibr_offline.cpp:86-155) between TranScanToPoints / AutoGetLinePts (clc_linefit.cuh),
// the nearest-pose match, LineFittingCeres and the Oberserve it fills.
//
// Pipeline (clc_problems_create_from_scans): classify (one thread per scan: segment + nearest pose) -> exclusive scan of the
// kept flags and segment lengths (frame index, offsets) -> gather (one warp per scan: SoA x, y of the kept segments, the
// frame pose) -> batched line fit -> on-line problem (two end points per frame), all device to device.
#pragma once

#if defined(__CUDACC__)
#include <math_constants.h>
#endif

#include "clc_linefit.cuh"

namespace clc {

// Round-to-nearest products and sums that nvcc does not contract into FMAs, so that the device and a host build (and
// numpy, which evaluates the same expressions) agree bit for bit on the few values below.
CLC_HD double mul_rn(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dmul_rn(a, b);
#else
  return a * b;
#endif
}
CLC_HD double add_rn(double a, double b) {
#if defined(__CUDA_ARCH__)
  return __dadd_rn(a, b);
#else
  return a + b;
#endif
}

// reference main/calibr_offline.cpp:103-116: the first pose with the smallest |t_pose - t_scan| (strict <, starting from
// 10000; a NaN stamp never matches; poses need not be sorted).  Returns the index or -1, and that smallest difference.
CLC_HD int64_t nearest_pose(const double* pose_stamp, int64_t n_poses, double t, double* min_dt_out) {
  double min_dt = 10000.0;
  int64_t best = -1;
  for (int64_t k = 0; k < n_poses; ++k) {
    const double dt = fabs(pose_stamp[k] - t);
    if (dt < min_dt) {
      min_dt = dt;
      best = k;
    }
  }
  *min_dt_out = min_dt;
  return best;
}

// reference main/calibr_offline.cpp:145-146 with Eigen semantics: qca = qwc.inverse() (conjugate / squaredNorm, no
// normalisation), tca = -R(qca) twc.  pose_wc = qx qy qz qw x y z; fp = qx qy qz qw tx ty tz (Oberserve::tagPose_Qca, _tca).
CLC_HD void tag_to_frame_pose(const double* pose_wc, double* fp) {
  const double x = pose_wc[0], y = pose_wc[1], z = pose_wc[2], w = pose_wc[3];
  const double n2 = add_rn(add_rn(add_rn(mul_rn(x, x), mul_rn(y, y)), mul_rn(z, z)), mul_rn(w, w));
  const double q[4] = {-x / n2, -y / n2, -z / n2, w / n2};
  // QuaternionBase::toRotationMatrix (the form of clc::quat_to_rot), without contractions
  const double qx = q[0], qy = q[1], qz = q[2], qw = q[3];
  const double R[9] = {1.0 - 2.0 * add_rn(mul_rn(qy, qy), mul_rn(qz, qz)), 2.0 * (mul_rn(qx, qy) - mul_rn(qz, qw)),
                       2.0 * add_rn(mul_rn(qx, qz), mul_rn(qy, qw)),
                       2.0 * add_rn(mul_rn(qx, qy), mul_rn(qz, qw)), 1.0 - 2.0 * add_rn(mul_rn(qx, qx), mul_rn(qz, qz)),
                       2.0 * (mul_rn(qy, qz) - mul_rn(qx, qw)),
                       2.0 * (mul_rn(qx, qz) - mul_rn(qy, qw)), 2.0 * add_rn(mul_rn(qy, qz), mul_rn(qx, qw)),
                       1.0 - 2.0 * add_rn(mul_rn(qx, qx), mul_rn(qy, qy))};
  for (int i = 0; i < 4; ++i) fp[i] = q[i];
  for (int r = 0; r < 3; ++r)
    fp[4 + r] = -add_rn(add_rn(mul_rn(R[3 * r], pose_wc[4]), mul_rn(R[3 * r + 1], pose_wc[5])), mul_rn(R[3 * r + 2], pose_wc[6]));
}

// reference main/calibr_offline.cpp:126-142: the first and the last segment point moved onto the fitted line
// m0 x + m1 y + 1 = 0 along the axis the segment spans least.  (The reference reads points.end(), one past the last
// point; the last point is meant.)  out = x_s, y_s, x_e, y_e.
CLC_HD void line_end_points(double x_s, double y_s, double x_e, double y_e, const double* line, double* out) {
  if (fabs(x_e - x_s) > fabs(y_e - y_s)) {
    y_s = -add_rn(mul_rn(x_s, line[0]), 1.0) / line[1];
    y_e = -add_rn(mul_rn(x_e, line[0]), 1.0) / line[1];
  } else {
    x_s = -add_rn(mul_rn(y_s, line[1]), 1.0) / line[0];
    x_e = -add_rn(mul_rn(y_e, line[1]), 1.0) / line[0];
  }
  out[0] = x_s; out[1] = y_s; out[2] = x_e; out[3] = y_e;
}

#if defined(__CUDACC__)
constexpr int kClassifyThreads = 128;
constexpr int kPoseTile = 2048;  // pose stamps staged in shared memory per pass (16 KB)

// One thread per scan: AutoGetLinePts, then -- for a scan with a segment -- the linear nearest-pose search over the
// stamps, staged tile by tile through shared memory (every thread reads the same stamp: a broadcast).
// info[s*4] = seg_start, seg_end, nearest pose (-1: no segment or no pose), frame (filled by the gather);
// cnt[s] = kept (0/1), cnt[n_scans + 1 + s] = points of a kept scan; the two trailing entries are 0 (exclusive scans
// of n_scans + 1 items leave the totals there), so the grid covers n_scans + 1 threads.
__global__ void __launch_bounds__(kClassifyThreads) clc_scan_classify_kernel(
    const float* __restrict__ ranges, int64_t n_scans, int64_t n_beams, double angle_min, double angle_increment,
    double range_min, const double* __restrict__ scan_stamp, const double* __restrict__ pose_stamp, int64_t n_poses,
    double max_dt, int* __restrict__ info, int64_t* __restrict__ cnt) {
  __shared__ double tile[kPoseTile];
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = s < n_scans;
  int a = -1, b = -1;
  if (active) auto_get_line_pts(ranges + s * n_beams, n_beams, angle_min, angle_increment, range_min, &a, &b);
  const bool want = active && a >= 0;
  const double t = active ? scan_stamp[s] : 0.0;
  double min_dt = 10000.0;
  int64_t best = -1;
  // the block searches only if one of its scans has a segment; the tile loop is uniform over the block
  if (__syncthreads_or(want ? 1 : 0)) {
    for (int64_t k0 = 0; k0 < n_poses; k0 += kPoseTile) {
      const int m = (int)(n_poses - k0 < kPoseTile ? n_poses - k0 : kPoseTile);
      __syncthreads();
      for (int i = threadIdx.x; i < m; i += blockDim.x) tile[i] = pose_stamp[k0 + i];
      __syncthreads();
      if (want) {
        double tile_dt;
        const int64_t k = nearest_pose(tile, m, t, &tile_dt);
        if (k >= 0 && tile_dt < min_dt) {  // strict: an earlier tile keeps a tie
          min_dt = tile_dt;
          best = k0 + k;
        }
      }
    }
  }
  if (!active) {
    if (s == n_scans) { cnt[n_scans] = 0; cnt[2 * n_scans + 1] = 0; }
    return;
  }
  const bool keep = want && best >= 0 && min_dt < max_dt;  // calibr_offline.cpp:116, strict
  info[4 * s] = a;
  info[4 * s + 1] = b;
  info[4 * s + 2] = want ? (int)best : -1;
  cnt[s] = keep ? 1 : 0;
  cnt[n_scans + 1 + s] = keep ? (int64_t)(b - a + 1) : 0;
}

// One warp per scan: a kept scan writes its segment points (x, y of scan_point, coalesced) at its offset, its frame pose
// and the CSR delimiter; every scan writes its frame index (or -1) into info.
__global__ void __launch_bounds__(256) clc_scan_gather_kernel(
    const float* __restrict__ ranges, int64_t n_scans, int64_t n_beams, double angle_min, double angle_increment,
    double range_min, const double* __restrict__ pose_wc, const int64_t* __restrict__ cnt, const int64_t* __restrict__ excl,
    int* __restrict__ info, double* __restrict__ x, double* __restrict__ y, double* __restrict__ frame_pose,
    int64_t* __restrict__ offsets) {
  const int64_t s = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (s == 0 && lane == 0) offsets[excl[n_scans]] = excl[2 * n_scans + 1];  // offsets[F] = P
  if (s >= n_scans) return;
  const bool keep = cnt[s] != 0;
  const int64_t f = excl[s];
  if (lane == 0) info[4 * s + 3] = keep ? (int)f : -1;
  if (!keep) return;
  const int64_t a = info[4 * s], b = info[4 * s + 1], o = excl[n_scans + 1 + s];
  const float* r = ranges + s * n_beams;
  for (int64_t i = a + lane; i <= b; i += 32) scan_point(r, i, angle_min, angle_increment, range_min, x + o + (i - a), y + o + (i - a));
  if (lane < 7) {
    double fp[7];
    tag_to_frame_pose(pose_wc + 7 * (int64_t)info[4 * s + 2], fp);
    frame_pose[7 * f + lane] = fp[lane];
  }
  if (lane == 0) offsets[f] = o;
}

// One thread per frame: the on-line problem (points_on_line of calibr_offline.cpp:126-142, two points per frame, the same
// frame pose; with edges the first and last segment point, LaseCamCalCeres.cpp:278-279) from the points problem.
__global__ void clc_scan_on_line_kernel(const double* __restrict__ x, const double* __restrict__ y,
                                        const int64_t* __restrict__ offsets, const double* __restrict__ frame_pose,
                                        const double* __restrict__ lines, int64_t n_frames, double* __restrict__ lx,
                                        double* __restrict__ ly, double* __restrict__ lframe_pose, int64_t* __restrict__ loffsets,
                                        double* __restrict__ edge_pt) {
  const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (f == 0) loffsets[0] = 0;
  if (f >= n_frames) return;
  const int64_t a = offsets[f], e = offsets[f + 1] - 1;
  double ends[4];
  line_end_points(x[a], y[a], x[e], y[e], lines + 2 * f, ends);
  lx[2 * f] = ends[0]; ly[2 * f] = ends[1];
  lx[2 * f + 1] = ends[2]; ly[2 * f + 1] = ends[3];
  loffsets[f + 1] = 2 * (f + 1);
  for (int i = 0; i < 7; ++i) lframe_pose[7 * f + i] = frame_pose[7 * f + i];
  if (edge_pt != nullptr) {
    double* ep = edge_pt + 6 * f;
    ep[0] = x[a]; ep[1] = y[a]; ep[2] = 0.0;
    ep[3] = x[e]; ep[4] = y[e]; ep[5] = 0.0;
  }
}

// per scan: the fitted line of a kept scan, NaN otherwise
__global__ void clc_scan_lines_kernel(const int* __restrict__ info, int64_t n_scans, const double* __restrict__ lines,
                                      double* __restrict__ scan_line) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n_scans) return;
  const int f = info[4 * s + 3];
  scan_line[2 * s] = f >= 0 ? lines[2 * (int64_t)f] : CUDART_NAN;
  scan_line[2 * s + 1] = f >= 0 ? lines[2 * (int64_t)f + 1] : CUDART_NAN;
}
#endif

}  // namespace clc
