// Arithmetic of the tracker glue that the host form of a single handle (fe_context.cu) and the device form of the stream
// group (kernels_glue.cu, kernels_track.cu) must evaluate identically: the group's rows are compared bit for bit with the
// handle's.  Include it only from host code (built with -ffp-contract=off) and from device files built with --fmad=false,
// so that every float expression rounds where the reference's SSE build rounds it.
#pragma once
#include <cmath>
#include <vector>

#include "fe_kernels.h"
#include "ransac_core.h"   // PLVIWO_HD

namespace plviwo {

// cv::undistortPoints with a 4-coefficient radtan model: 5 fixed-point iterations in double (SURVEY.md Appendix A6).
PLVIWO_HD inline float2 undistort_radtan(float2 uv, const double K[4], const double D[4]) {
  const double x0 = ((double)uv.x - K[2]) / K[0], y0 = ((double)uv.y - K[3]) / K[1];
  double x = x0, y = y0;
  const double k1 = D[0], k2 = D[1], p1 = D[2], p2 = D[3];
#pragma unroll 1
  for (int j = 0; j < 5; j++) {
    const double r2 = x * x + y * y;
    const double icdist = 1.0 / (1.0 + (k2 * r2 + k1) * r2);
    const double dx = 2 * p1 * x * y + p2 * (r2 + 2 * x * x);
    const double dy = p1 * (r2 + 2 * y * y) + 2 * p2 * x * y;
    x = (x0 - dx) * icdist;
    y = (y0 - dy) * icdist;
  }
  return make_float2((float)x, (float)y);
}

// TrackLSD::PointLineDistance (TrackLSD.cpp:794-814): float arithmetic; the last branch mixes in double through
// std::pow(float, int), which promotes to double and is correctly rounded for an exponent of 2, so it is dy * dy.
PLVIWO_HD inline float point_line_distance(const float4 &line, float x0, float y0) {
  const float x1 = line.x, y1 = line.y, x2 = line.z, y2 = line.w;
  const float cross = (x2 - x1) * (x0 - x1) + (y2 - y1) * (y0 - y1);
  if (cross <= 0) return sqrtf((x0 - x1) * (x0 - x1) + (y0 - y1) * (y0 - y1));
  const float d = (x2 - x1) * (x2 - x1) + (y2 - y1) * (y2 - y1);
  if (cross > d) return sqrtf((x0 - x2) * (x0 - x2) + (y0 - y2) * (y0 - y2));
  const double dy = (double)(y2 - y1), dx = (double)(x1 - x2);
  return (float)fabs((double)fabsf((y2 - y1) * x0 + (x1 - x2) * y0 + ((x2 * y1) - (x1 * y2))) / sqrt(dy * dy + dx * dx));
}

// TrackLSD::LineSimilar (:816-830)
PLVIWO_HD inline bool line_similar(const float4 &line2, const float4 &line1) {
  const float mx = (line1.x + line1.z) / 2, my = (line1.y + line1.w) / 2;
  return point_line_distance(line2, mx, my) <= 6;
}

// TrackLSD::LineClass (:335-366), including atan(dy) / dx at :350-351 as written there
PLVIWO_HD inline bool line_class(const float4 &line, double vx, double vy) {
  const double s[3] = {line.x, line.y, 1}, e[3] = {line.z, line.w, 1};
  const double mid[3] = {(s[0] + e[0]) / 2, (s[1] + e[1]) / 2, (s[2] + e[2]) / 2};
  const double v3[3] = {vx, vy, 1};
  const double ln[3] = {mid[1] * v3[2] - mid[2] * v3[1], mid[2] * v3[0] - mid[0] * v3[2], mid[0] * v3[1] - mid[1] * v3[0]};
  double dis_error = (fabs(ln[0] * s[0] + ln[1] * s[1] + ln[2] * s[2]) + fabs(ln[0] * e[0] + ln[1] * e[1] + ln[2] * e[2])) /
                     (2 * sqrt(ln[0] * ln[0] + ln[1] * ln[1]));
  dis_error = fabs(dis_error);
  const double angle1 = atanf(line.y - line.w) / (line.x - line.z);   // float arithmetic
  const double angle2 = atan(mid[1] - vy) / (mid[0] - vx);
  const double angle_error = fabs(angle1 - angle2);
  return dis_error <= 5.0 && angle_error <= 0.35;
}

// TrackLSD::LineClassification (:318-333)
PLVIWO_HD inline int line_classification(const float4 &line, const double vp[6]) {
  if (line_class(line, vp[4], vp[5])) return 3;
  if (line_class(line, vp[2], vp[3])) return 2;
  if (line_class(line, vp[0], vp[1])) return 1;
  return 0;
}

// Grider_GRID geometry (Grider_GRID.h:88-100): the grider may shrink ITS grid when num_features < grid_x * grid_y while the
// cell indices still come from the caller's grid; cells that leave the image are skipped (:117-118).
struct GriderLayout {
  std::vector<FastCell> cells;   // every in-image cell, x-major like valid_locs
  std::vector<int> cell_of_loc;  // caller-grid (x * grid_y + y) -> index into cells or -1
  int nfg = 0;                   // num_features_grid: candidates kept per cell
  int csx = 0, csy = 0;          // cell size
  int n_bands = 0;               // FAST bands of kFastBandRows rows per cell
};
inline GriderLayout grider_layout(int W, int H, int grid_x, int grid_y, int num_features) {
  GriderLayout L;
  int ggx = grid_x, ggy = grid_y;
  if (num_features < ggx * ggy) {
    double ratio = (double)ggx / (double)ggy;
    ggy = (int)std::ceil(std::sqrt(num_features / ratio));
    ggx = (int)std::ceil(ggy * ratio);
  }
  L.nfg = (int)((double)num_features / (double)(ggx * ggy)) + 1;
  L.csx = W / ggx;
  L.csy = H / ggy;
  L.cell_of_loc.assign((size_t)grid_x * grid_y, -1);
  if (L.csx > 0 && L.csy > 0)
    for (int x = 0; x < grid_x; x++)
      for (int y = 0; y < grid_y; y++) {
        const int px = x * L.csx, py = y * L.csy;
        if (px + L.csx > W || py + L.csy > H) continue;
        L.cell_of_loc[(size_t)x * grid_y + y] = (int)L.cells.size();
        L.cells.push_back(FastCell{px, py, L.csx, L.csy});
      }
  L.n_bands = L.csy > 0 ? (L.csy + kFastBandRows - 1) / kFastBandRows : 0;
  return L;
}

}  // namespace plviwo
