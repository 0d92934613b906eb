// Arithmetic of the tracker glue that the host form of a single handle (fe_context.cu) and the device form of the stream
// group (kernels_glue.cu, kernels_track.cu) must evaluate identically: the group's rows are compared bit for bit with the
// handle's.  Include it only from host code (built with -ffp-contract=off) and from device files built with --fmad=false,
// so that every float expression rounds where the reference's SSE build rounds it.
#pragma once
#include <cmath>
#include <cstdint>
#include <cstring>
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

// tan(x) in plain IEEE double arithmetic: fdlibm's __kernel_tan after the medium-range reduction of __ieee754_rem_pio2
// (n = rint(x * 2 / pi), pi / 2 in three parts).  libm's tan and CUDA's tan are different functions; this one rounds the same
// on the host and on the device, so a handle (host) and a stream group (device) undistort line endpoints identically.
// Beyond |x| ~ 1.6e6 the reduction loses accuracy; only points that end up at (-1e6, -1e6) get there.
PLVIWO_HD inline uint64_t f64_bits(double x) {
#ifdef __CUDA_ARCH__
  return (uint64_t)__double_as_longlong(x);
#else
  uint64_t u;
  memcpy(&u, &x, 8);
  return u;
#endif
}
PLVIWO_HD inline double f64_from_bits(uint64_t u) {
#ifdef __CUDA_ARCH__
  return __longlong_as_double((long long)u);
#else
  double x;
  memcpy(&x, &u, 8);
  return x;
#endif
}
PLVIWO_HD inline double f64_clear_lo(double x) { return f64_from_bits(f64_bits(x) & 0xffffffff00000000ull); }

// fdlibm k_tan.c: tan(x + y) for |x + y| <= pi / 4; iy = 1 tan, iy = -1 -1 / tan
PLVIWO_HD inline double kernel_tan(double x, double y, int iy) {
  const double T[13] = {3.33333333333334091986e-01, 1.33333333333201242699e-01, 5.39682539762260521377e-02,
                        2.18694882948595424599e-02, 8.86323982359930005737e-03, 3.59207910759131235356e-03,
                        1.45620945432529025516e-03, 5.88041240820264096874e-04, 2.46463134818469906812e-04,
                        7.81794442939557092300e-05, 7.14072491382608190305e-05, -1.85586374855275456654e-05,
                        2.59073051863633712884e-05};
  const double pio4 = 7.85398163397448278999e-01, pio4lo = 3.06161699786838301793e-17;
  const int hx = (int)(f64_bits(x) >> 32), ix = hx & 0x7fffffff;
  double z, r, v, w, s;
  if (ix < 0x3e300000) {   // |x| < 2^-28
    if (iy == 1) return x;
    if (x == 0) return 1.0 / fabs(x);
    z = w = x + y;
    z = f64_clear_lo(z);
    v = y - (z - x);
    double a = -1.0 / w, t = f64_clear_lo(a);
    s = 1.0 + t * z;
    return t + a * (s + t * v);
  }
  if (ix >= 0x3FE59428) {   // |x| >= 0.6744
    if (hx < 0) {
      x = -x;
      y = -y;
    }
    z = pio4 - x;
    w = pio4lo - y;
    x = z + w;
    y = 0.0;
  }
  z = x * x;
  w = z * z;
  r = T[1] + w * (T[3] + w * (T[5] + w * (T[7] + w * (T[9] + w * T[11]))));
  v = z * (T[2] + w * (T[4] + w * (T[6] + w * (T[8] + w * (T[10] + w * T[12])))));
  s = z * x;
  r = y + z * (s * (r + v) + y);
  r += T[0] * s;
  w = x + r;
  if (ix >= 0x3FE59428) {
    v = (double)iy;
    return (double)(1 - ((hx >> 30) & 2)) * (v - 2.0 * (x - (w * w / (w + v) - r)));
  }
  if (iy == 1) return w;
  z = f64_clear_lo(w);
  v = r - (z - x);
  double a = -1.0 / w, t = f64_clear_lo(a);
  s = 1.0 + t * z;
  return t + a * (s + t * v);
}

PLVIWO_HD inline double tan_ieee(double x) {
  const int ix = (int)(f64_bits(x) >> 32) & 0x7fffffff;
  if (ix <= 0x3fe921fb) return kernel_tan(x, 0.0, 1);   // |x| <= pi / 4
  if (ix >= 0x7ff00000) return x - x;                   // inf, NaN
  const double invpio2 = 6.36619772367581382433e-01, pio2_1 = 1.57079632673412561417e+00, pio2_1t = 6.07710050650619224932e-11,
               pio2_2 = 6.07710050630396597660e-11, pio2_2t = 2.02226624879595063154e-21, pio2_3 = 2.02226624871116645580e-21,
               pio2_3t = 8.47842766036889956997e-32;
  const double fn = rint(x * invpio2);
  double r = x - fn * pio2_1, w = fn * pio2_1t, y0 = r - w;
  const int j = ix >> 20;
  if (j - (int)((f64_bits(y0) >> 52) & 0x7ff) > 16) {   // second step, 118 bits
    double t = r;
    w = fn * pio2_2;
    r = t - w;
    w = fn * pio2_2t - ((t - r) - w);
    y0 = r - w;
    if (j - (int)((f64_bits(y0) >> 52) & 0x7ff) > 49) {   // third step, 151 bits
      t = r;
      w = fn * pio2_3;
      r = t - w;
      w = fn * pio2_3t - ((t - r) - w);
      y0 = r - w;
    }
  }
  const double y1 = (r - y0) - w;
  const double half = fn * 0.5;   // parity of n without converting fn to an integer
  return kernel_tan(y0, y1, half != floor(half) ? -1 : 1);
}

// cv::fisheye::undistortPoints with identity R / P and the default criteria (10 iterations, eps 1e-8), as CamEqui::undistort_f
// calls it (cam/CamEqui.h:108-129): Newton on theta (1 + k1 theta^2 + k2 theta^4 + k3 theta^6 + k4 theta^8) = theta_d, the
// point is pw tan(theta) / theta_d, or (-1e6, -1e6) when the iteration did not converge or theta changed sign.  The clamp of
// theta_d is std::min(std::max(-pi/2, theta_d), pi/2) with std::'s operand order, so a NaN theta_d becomes -pi/2 there as well.
PLVIWO_HD inline float2 undistort_equi(float2 uv, const double K[4], const double D[4]) {
  const double pwx = ((double)uv.x - K[2]) / K[0], pwy = ((double)uv.y - K[3]) / K[1];
  const double half_pi = 3.14159265358979323846 / 2.0;
  double td = sqrt(pwx * pwx + pwy * pwy);
  td = (-half_pi < td) ? td : -half_pi;
  td = (half_pi < td) ? half_pi : td;
  bool converged = false;
  double theta = td, scale = 0.0;
  if (fabs(td) > 1e-8) {
#pragma unroll 1
    for (int j = 0; j < 10; j++) {
      const double t2 = theta * theta, t4 = t2 * t2, t6 = t4 * t2, t8 = t6 * t2;
      const double k0 = D[0] * t2, k1 = D[1] * t4, k2 = D[2] * t6, k3 = D[3] * t8;
      const double fix = (theta * (1 + k0 + k1 + k2 + k3) - td) / (1 + 3 * k0 + 5 * k1 + 7 * k2 + 9 * k3);
      theta = theta - fix;
      if (fabs(fix) < 1e-8) {
        converged = true;
        break;
      }
    }
    scale = tan_ieee(theta) / td;
  } else {
    converged = true;
  }
  const bool flipped = (td < 0 && theta > 0) || (td > 0 && theta < 0);
  if (!converged || flipped) return make_float2(-1000000.0f, -1000000.0f);
  return make_float2((float)(pwx * scale), (float)(pwy * scale));
}

// The camera model of a handle / rig / group (FeCameraModel), fixed at creation; uniform per launch.
PLVIWO_HD inline float2 undistort_point(int model, float2 uv, const double K[4], const double D[4]) {
  return model == FE_CAM_EQUI ? undistort_equi(uv, K, D) : undistort_radtan(uv, K, D);
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
