// Test-only harness for the scan loop of the offline driver (csrc/clc_scans.cuh): compiles its CLC_HD helpers with g++ so
// that the exact source the GPU runs -- the nearest-pose search, the frame pose, the line end points -- can be checked on a
// machine without a GPU.  Never shipped, never linked into libclc_b200.so.
#include "../camlasercalibratool_b200/csrc/clc_scans.cuh"

extern "C" {

int64_t harness_nearest_pose(const double* stamps, int64_t n, double t, double* min_dt) {
  return clc::nearest_pose(stamps, n, t, min_dt);
}
void harness_tag_to_frame_pose(const double* pose_wc, double* fp) { clc::tag_to_frame_pose(pose_wc, fp); }
void harness_line_end_points(double xs, double ys, double xe, double ye, const double* line, double* out) {
  clc::line_end_points(xs, ys, xe, ye, line, out);
}

}  // extern "C"
