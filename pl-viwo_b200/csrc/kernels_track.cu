// Per-feature kernels (sm_100a): sub-pixel corner refinement, pyramidal Lucas-Kanade with on-the-fly Scharr
// derivatives, and undistortion (radtan or equidistant).  One warp per feature; compiled with --fmad=false so that float
// expressions round exactly where the reference's SSE build rounds.
//
// Reference ops replaced (SURVEY.md Appendix A3, A5, A6):
//   cv::cornerSubPix(img, pts, (5,5), (-1,-1), {COUNT+EPS, 20, 0.001})             Grider_GRID.h:163-174
//   cv::calcOpticalFlowPyrLK(.., win, maxLevel, {COUNT|EPS, 30, 0.01}, USE_INITIAL_FLOW)  TrackKLT.cpp:855-858
//   CamRadtan::undistort_f -> cv::undistortPoints (one Mat per point)               cam/CamRadtan.h:99-120
//   CamEqui::undistort_f -> cv::fisheye::undistortPoints (one Mat per point)        cam/CamEqui.h:108-129
#include "fe_kernels.h"
#include "fe_group_dev.h"
#include "tracker_core.h"

#include <algorithm>
#include <mutex>
#include <cfloat>
#include <climits>
#include <cmath>

namespace plviwo {

__device__ __forceinline__ int reflect101(int i, int n) {
  // BORDER_REFLECT_101; the final clamp only guards reads that the algorithm discards (far-outside halo)
  if (i < 0) i = -i;
  if (i >= n) i = 2 * n - 2 - i;
  return min(max(i, 0), n - 1);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
  return v;
}

// ============================================================================================ cornerSubPix
// win = (5,5): 11 x 11 window, 13 x 13 bilinear patch (cv::getRectSubPix, BORDER_REPLICATE at the image edge),
// Gaussian-like mask exp(-x^2/25) exp(-y^2/25), double-precision normal equations, <= 20 iterations, eps 1e-3.
constexpr int kSpWin = 5;
constexpr int kSpW = 2 * kSpWin + 1;   // 11
constexpr int kSpP = kSpW + 2;         // 13
constexpr int kSpWarps = 4;

__constant__ float c_subpix_mask[kSpW * kSpW];
static bool g_subpix_mask_ready[64] = {false};

__device__ __forceinline__ void corner_subpix_body(const uint8_t *__restrict__ img, int w, int h, int pitch, const float2 *pts_in,
                                                   float2 *pts, int n, const int *__restrict__ cnt, int stride) {
  __shared__ float patch_s[kSpWarps][kSpP * kSpP];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int pi = blockIdx.x * kSpWarps + warp;
  if (pi >= n) return;
  if (cnt != nullptr) {   // fixed-stride candidate table: dead slots are skipped
    const int cell = pi / stride;
    if (pi - cell * stride >= cnt[cell]) return;
  }
  float *patch = patch_s[warp];
  const float2 cT = pts_in[pi];
  float2 cI = cT;
  const double eps = 0.001 * 0.001;
  int iter = 0;
  double err = 0;
  do {
    // getRectSubPix(src, 13x13, cI): top-left = cI - 6, bilinear weights in float, replicate outside
    float cx = cI.x - (kSpP - 1) * 0.5f, cy = cI.y - (kSpP - 1) * 0.5f;
    int ipx = __float2int_rd(cx), ipy = __float2int_rd(cy);
    float a = cx - ipx, b = cy - ipy;
    float a11 = (1.f - a) * (1.f - b), a12 = a * (1.f - b), a21 = (1.f - a) * b, a22 = a * b;
    for (int i = lane; i < kSpP * kSpP; i += 32) {
      int r = i / kSpP, c = i - r * kSpP;
      int x0 = min(max(ipx + c, 0), w - 1), x1 = min(max(ipx + c + 1, 0), w - 1);
      int y0 = min(max(ipy + r, 0), h - 1), y1 = min(max(ipy + r + 1, 0), h - 1);
      const uint8_t *r0 = img + (size_t)y0 * pitch, *r1 = img + (size_t)y1 * pitch;
      patch[i] = r0[x0] * a11 + r0[x1] * a12 + r1[x0] * a21 + r1[x1] * a22;
    }
    __syncwarp();
    double sa = 0, sb = 0, sc = 0, sbb1 = 0, sbb2 = 0;
    for (int k = lane; k < kSpW * kSpW; k += 32) {
      int i = k / kSpW, j = k - i * kSpW;
      const float *sp = patch + (i + 1) * kSpP + (j + 1);
      double m = c_subpix_mask[k];
      double tgx = sp[1] - sp[-1];
      double tgy = sp[kSpP] - sp[-kSpP];
      double gxx = tgx * tgx * m, gxy = tgx * tgy * m, gyy = tgy * tgy * m;
      double px = j - kSpWin, py = i - kSpWin;
      sa += gxx; sb += gxy; sc += gyy;
      sbb1 += gxx * px + gxy * py;
      sbb2 += gxy * px + gyy * py;
    }
    sa = warp_sum(sa); sb = warp_sum(sb); sc = warp_sum(sc); sbb1 = warp_sum(sbb1); sbb2 = warp_sum(sbb2);
    __syncwarp();
    double det = sa * sc - sb * sb;
    if (fabs(det) <= DBL_EPSILON * DBL_EPSILON) break;
    double scale = 1.0 / det;
    float2 cI2;
    cI2.x = (float)(cI.x + sc * scale * sbb1 - sb * scale * sbb2);
    cI2.y = (float)(cI.y - sb * scale * sbb1 + sa * scale * sbb2);
    err = (double)((cI2.x - cI.x) * (cI2.x - cI.x) + (cI2.y - cI.y) * (cI2.y - cI.y));
    cI = cI2;
    if (cI.x < 0 || cI.x >= w || cI.y < 0 || cI.y >= h) break;
  } while (++iter < 20 && err > eps);
  if (fabsf(cI.x - cT.x) > kSpWin || fabsf(cI.y - cT.y) > kSpWin) cI = cT;
  if (lane == 0) pts[pi] = cI;
}

__global__ void __launch_bounds__(kSpWarps * 32)
    k_corner_subpix(const uint8_t *__restrict__ img, int w, int h, int pitch, const float2 *pts_in, float2 *pts, int n,
                    const int *__restrict__ cnt, int stride) {
  corner_subpix_body(img, w, h, pitch, pts_in, pts, n, cnt, stride);
}

void init_device_constants() {
  DevImage dummy;
  launch_corner_subpix(dummy, nullptr, nullptr, -1, 0);
  init_fld_constants();
}

void launch_corner_subpix(const DevImage &img, const float2 *d_in, float2 *d_out, int n, cudaStream_t s, const int *d_cnt,
                          int stride) {
  if (n == 0) return;
  int dev = 0;
  cudaGetDevice(&dev);
  static std::mutex mu;   // handles may be created from several host threads
  std::unique_lock<std::mutex> lk(mu);
  if (!g_subpix_mask_ready[dev & 63]) {
    float m[kSpW * kSpW];
    for (int i = 0; i < kSpW; i++) {
      float y = (float)(i - kSpWin) / kSpWin;
      float vy = std::exp(-y * y);
      for (int j = 0; j < kSpW; j++) {
        float x = (float)(j - kSpWin) / kSpWin;
        m[i * kSpW + j] = (float)(vy * std::exp(-x * x));
      }
    }
    cudaMemcpyToSymbol(c_subpix_mask, m, sizeof(m));
    g_subpix_mask_ready[dev & 63] = true;
  }
  lk.unlock();
  if (n < 0) return;
  PLVIWO_CARVEOUT(k_corner_subpix);
  k_corner_subpix<<<(n + kSpWarps - 1) / kSpWarps, kSpWarps * 32, 0, s>>>(img.p, img.w, img.h, img.pitch, d_in, d_out, n, d_cnt,
                                                                          stride);
}

// Stream group: cornerSubPix of the candidates the top-off detection of a frame really considers (the corners of the valid
// cells that pass the mask test: a few dozen per frame), between the two halves of the detection.  Same body, same result
// per corner as refining the whole candidate table ahead of time, at a tenth of the work.
__global__ void __launch_bounds__(kSpWarps * 32)
    k_corner_subpix_g(const __grid_constant__ GroupDev g, const TrackJob *__restrict__ jobs) {
  const TrackJob &job = jobs[blockIdx.y];
  const int s = job.stream;
  const int n = g.winfo[4 * s + 3];
  if ((int)blockIdx.x * kSpWarps >= n) return;
  const bool first = g.wmode[s] == 1;
  const DevImage &im = g.slots[first ? job.cur_slot : job.prev_slot].lvl[0];
  const size_t o = (size_t)s * g.cand_cap;
  corner_subpix_body(im.p, im.w, im.h, im.pitch, g.ext_in + o, g.ext_pt + o, n, nullptr, 0);
}
void launch_group_subpix(const GroupDev &g, const TrackJob *jobs, int n_jobs, cudaStream_t s) {
  if (n_jobs <= 0 || g.cand_cap <= 0) return;
  launch_corner_subpix(DevImage(), nullptr, nullptr, -1, 0);   // constant table of this device
  PLVIWO_CARVEOUT(k_corner_subpix_g);
  k_corner_subpix_g<<<dim3((g.cand_cap + kSpWarps - 1) / kSpWarps, n_jobs), kSpWarps * 32, 0, s>>>(g, jobs);
}

// ============================================================================================== undistort
struct CalibArgs {
  double K[4], D[4];
};

// The equidistant model out of line: its Newton loop and tan stay out of the register budget of the LK kernels, whose
// epilogue calls it for one point per lane at most.  The calibration goes by value (registers): a pointer into a kernel's
// parameter block would make the caller copy the whole block to its stack.
__device__ __noinline__ float2 undistort_equi_call(float2 uv, double fx, double fy, double cx, double cy, double k1, double k2,
                                                   double k3, double k4) {
  const double K[4] = {fx, fy, cx, cy}, D[4] = {k1, k2, k3, k4};
  return undistort_equi(uv, K, D);
}
// undistort_point of the kernels: `model` is uniform per launch
__device__ __forceinline__ float2 undistort_dev(int model, float2 uv, const CalibArgs &c) {
  if (model == FE_CAM_EQUI)
    return undistort_equi_call(uv, c.K[0], c.K[1], c.K[2], c.K[3], c.D[0], c.D[1], c.D[2], c.D[3]);
  return undistort_radtan(uv, c.K, c.D);
}

__global__ void k_undistort(const float2 *__restrict__ pts, float2 *__restrict__ out, int n, int model, CalibArgs c) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = undistort_point(model, pts[i], c.K, c.D);
}

void launch_undistort(const float2 *d_pts, float2 *d_out, int n, int model, const double K[4], const double D[4], cudaStream_t s) {
  if (n <= 0) return;
  CalibArgs c;
  for (int i = 0; i < 4; i++) { c.K[i] = K[i]; c.D[i] = D[i]; }
  PLVIWO_CARVEOUT(k_undistort);
  k_undistort<<<(n + 127) / 128, 128, 0, s>>>(d_pts, d_out, n, model, c);
}

// ===================================================================================================== LK
// One warp per feature, every pyramid level in ONE launch.  Per level the warp
//   1. loads the (win+3)^2 neighbourhood of the previous image (REFLECT_101 like OpenCV's padded pyramid),
//   2. forms Scharr derivatives at the (win+1)^2 integer positions on the fly (zero outside the frame, exactly
//      what the reference's zero-padded derivative planes hold),
//   3. builds the fixed-point (W_BITS = 14) bilinear patches I, Ix, Iy (int16) and the 2x2 normal matrix,
//   4. iterates <= 30 times: bilinear J patch, mismatch vector b (shuffle-reduced), 2x2 solve.
// Nothing but the two 8-bit pyramids is read from HBM: no derivative planes, no padded copies.
constexpr int kLkWarps = 4;   // features (warps) per CTA of the warp-per-feature kernels

struct LkArgs {
  const uint8_t *p0[kMaxLevels];
  const uint8_t *p1[kMaxLevels];
  int w[kMaxLevels], h[kMaxLevels], pitch0[kMaxLevels], pitch1[kMaxLevels];
  int win, max_level, max_count, undistort;
  int flow_is_zero;   // the initial guess is the previous position itself: pts1 is output only
  unsigned cell_mask[8];   // table mode: cells whose candidates are tracked at all (bit c of word c / 32)
  float eps_sq, min_eig;
  int model;          // FeCameraModel of calib (in the padding before it: LkArgs keeps its size)
  CalibArgs calib;
};

// The arguments of one pair of pyramids: `levels` images of l0 (previous) and l1 (next), prm's window and criteria,
// calibration K / D (undistort: also write the undistorted positions), cell_mask null = every cell.
__host__ __device__ inline void lk_args(LkArgs &a, const DevImage *l0, const DevImage *l1, int levels, const LkParams &prm,
                                        const double *K, const double *D, int undistort, int flow_is_zero, const unsigned *cell_mask) {
  for (int l = 0; l < levels; l++) {
    a.p0[l] = l0[l].p;
    a.p1[l] = l1[l].p;
    a.w[l] = l0[l].w;
    a.h[l] = l0[l].h;
    a.pitch0[l] = l0[l].pitch;
    a.pitch1[l] = l1[l].pitch;
  }
  a.win = prm.win;
  a.max_level = levels - 1;
  a.max_count = prm.max_count;
  a.eps_sq = prm.eps_sq;
  a.min_eig = prm.min_eig;
  a.undistort = undistort;
  a.model = prm.model;
  a.flow_is_zero = flow_is_zero;
  for (int i = 0; i < 8; i++) a.cell_mask[i] = cell_mask ? cell_mask[i] : 0xffffffffu;
  for (int i = 0; i < 4; i++) {
    a.calib.K[i] = K[i];
    a.calib.D[i] = D[i];
  }
}

// lk_body's shared memory per warp: raw[np*np] u8 | dx[nd*nd] s16 | dy[nd*nd] s16 | Iw[nw] s16 | Ix[nw] s16 | Iy[nw] s16,
// each part rounded up to 16 bytes.  Its launches size their dynamic shared memory with it.
struct LkLayout {
  int raw, d, w, per_warp;   // bytes of the raw patch, of one derivative plane, of one window patch, of a warp's slice
  __host__ __device__ explicit LkLayout(int win)
      : raw(((win + 3) * (win + 3) + 15) & ~15), d(((win + 1) * (win + 1) * 2 + 15) & ~15), w((win * win * 2 + 15) & ~15),
        per_warp(raw + 2 * d + 3 * w) {}
};

// feature pi of the warp's launch; the warp's shared memory is its slice of the dynamic buffer
template <class Args>
__device__ __forceinline__ void lk_body(const Args &a, const float2 *__restrict__ pts0, float2 *__restrict__ pts1,
                                        uint8_t *__restrict__ status, float2 *__restrict__ p0n, float2 *__restrict__ p1n, int pi) {
  extern __shared__ __align__(16) uint8_t lk_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int win = a.win;
  const int np = win + 3;        // raw patch side
  const int nd = win + 1;        // derivative grid side
  const int nw = win * win;
  const LkLayout lay(win);
  const int raw_bytes = lay.raw, d_bytes = lay.d, w_bytes = lay.w;
  uint8_t *base = lk_smem + warp * lay.per_warp;
  uint8_t *raw = base;
  short *ddx = reinterpret_cast<short *>(base + raw_bytes);
  short *ddy = reinterpret_cast<short *>(base + raw_bytes + d_bytes);
  short *Iw = reinterpret_cast<short *>(base + raw_bytes + 2 * d_bytes);
  short *Ixw = reinterpret_cast<short *>(base + raw_bytes + 2 * d_bytes + w_bytes);
  short *Iyw = reinterpret_cast<short *>(base + raw_bytes + 2 * d_bytes + 2 * w_bytes);

  const float2 prev_in = pts0[pi];
  float2 next = a.flow_is_zero ? prev_in : pts1[pi];   // OPTFLOW_USE_INITIAL_FLOW
  bool ok = true;
  const float half = (win - 1) * 0.5f;
  const float FLT_SCALE = 1.f / (1 << 20);

  for (int level = a.max_level; level >= 0; level--) {
    const int cols = a.w[level], rows = a.h[level];
    const float lscale = 1.f / (float)(1 << level);
    float2 prevPt = make_float2(prev_in.x * lscale, prev_in.y * lscale);
    if (level == a.max_level) {
      next.x = next.x * lscale;
      next.y = next.y * lscale;
    } else {
      next.x = next.x * 2.f;
      next.y = next.y * 2.f;
    }
    prevPt.x -= half;
    prevPt.y -= half;
    const int ipx = __float2int_rd(prevPt.x), ipy = __float2int_rd(prevPt.y);
    if (ipx < -win || ipx >= cols || ipy < -win || ipy >= rows) {
      if (level == 0) ok = false;
      continue;
    }
    float fa = prevPt.x - ipx, fb = prevPt.y - ipy;
    int iw00 = __float2int_rn((1.f - fa) * (1.f - fb) * 16384.f);
    int iw01 = __float2int_rn(fa * (1.f - fb) * 16384.f);
    int iw10 = __float2int_rn((1.f - fa) * fb * 16384.f);
    int iw11 = 16384 - iw00 - iw01 - iw10;

    // 1. raw neighbourhood, origin (ipx - 1, ipy - 1)
    const uint8_t *I = a.p0[level];
    const int pitchI = a.pitch0[level];
    for (int i = lane; i < np * np; i += 32) {
      int r = i / np, c = i - r * np;
      int x = reflect101(ipx - 1 + c, cols), y = reflect101(ipy - 1 + r, rows);
      raw[i] = I[(size_t)y * pitchI + x];
    }
    __syncwarp();
    // 2. Scharr derivatives at (ipx + c, ipy + r), c, r in [0, win]; zero outside the frame
    for (int i = lane; i < nd * nd; i += 32) {
      int r = i / nd, c = i - r * nd;
      int gx = ipx + c, gy = ipy + r;
      int vx = 0, vy = 0;
      if (gx >= 0 && gx < cols && gy >= 0 && gy < rows) {
        const uint8_t *q = raw + (r + 1) * np + (c + 1);
        int tl = q[-np - 1], tc = q[-np], tr = q[-np + 1];
        int ml = q[-1], mr = q[1];
        int bl = q[np - 1], bc = q[np], br = q[np + 1];
        vx = 3 * (tr + br) + 10 * mr - 3 * (tl + bl) - 10 * ml;
        vy = 3 * (bl + br) + 10 * bc - 3 * (tl + tr) - 10 * tc;
      }
      ddx[i] = (short)vx;
      ddy[i] = (short)vy;
    }
    __syncwarp();
    // 3. interpolated patches + normal matrix
    float A11 = 0, A12 = 0, A22 = 0;
    for (int i = lane; i < nw; i += 32) {
      int y = i / win, x = i - y * win;
      const uint8_t *q = raw + (y + 1) * np + (x + 1);
      int ival = (q[0] * iw00 + q[1] * iw01 + q[np] * iw10 + q[np + 1] * iw11 + (1 << 8)) >> 9;
      int di = y * nd + x;
      int ixval = (ddx[di] * iw00 + ddx[di + 1] * iw01 + ddx[di + nd] * iw10 + ddx[di + nd + 1] * iw11 + (1 << 13)) >> 14;
      int iyval = (ddy[di] * iw00 + ddy[di + 1] * iw01 + ddy[di + nd] * iw10 + ddy[di + nd + 1] * iw11 + (1 << 13)) >> 14;
      Iw[i] = (short)ival;
      Ixw[i] = (short)ixval;
      Iyw[i] = (short)iyval;
      A11 += (float)(ixval * ixval);
      A12 += (float)(ixval * iyval);
      A22 += (float)(iyval * iyval);
    }
    A11 = warp_sum(A11) * FLT_SCALE;
    A12 = warp_sum(A12) * FLT_SCALE;
    A22 = warp_sum(A22) * FLT_SCALE;
    __syncwarp();
    float Dt = A11 * A22 - A12 * A12;
    float minEig = (A22 + A11 - sqrtf((A11 - A22) * (A11 - A22) + 4.f * A12 * A12)) / (float)(2 * win * win);
    if (minEig < a.min_eig || Dt < FLT_EPSILON) {
      if (level == 0) ok = false;
      continue;
    }
    Dt = 1.f / Dt;
    float2 result = next;   // nextPts[ptidx] as stored by OpenCV; only rewritten after an update step
    next.x -= half;
    next.y -= half;
    float2 prevDelta = make_float2(0.f, 0.f);
    const uint8_t *J = a.p1[level];
    const int pitchJ = a.pitch1[level];
    for (int j = 0; j < a.max_count; j++) {
      const int inx = __float2int_rd(next.x), iny = __float2int_rd(next.y);
      if (inx < -win || inx >= cols || iny < -win || iny >= rows) {
        if (level == 0) ok = false;
        break;
      }
      float ja = next.x - inx, jb = next.y - iny;
      int jw00 = __float2int_rn((1.f - ja) * (1.f - jb) * 16384.f);
      int jw01 = __float2int_rn(ja * (1.f - jb) * 16384.f);
      int jw10 = __float2int_rn((1.f - ja) * jb * 16384.f);
      int jw11 = 16384 - jw00 - jw01 - jw10;
      float b1 = 0, b2 = 0;
      const bool inside = inx >= 0 && iny >= 0 && inx + win < cols && iny + win < rows;
      if (inside) {
        const uint8_t *Jp = J + (size_t)iny * pitchJ + inx;
        for (int i = lane; i < nw; i += 32) {
          int y = i / win, x = i - y * win;
          const uint8_t *q = Jp + (size_t)y * pitchJ + x;
          int jv = (q[0] * jw00 + q[1] * jw01 + q[pitchJ] * jw10 + q[pitchJ + 1] * jw11 + (1 << 8)) >> 9;
          int diff = jv - Iw[i];
          b1 += (float)(diff * Ixw[i]);
          b2 += (float)(diff * Iyw[i]);
        }
      } else {
        for (int i = lane; i < nw; i += 32) {
          int y = i / win, x = i - y * win;
          int x0 = reflect101(inx + x, cols), x1 = reflect101(inx + x + 1, cols);
          const uint8_t *r0 = J + (size_t)reflect101(iny + y, rows) * pitchJ;
          const uint8_t *r1 = J + (size_t)reflect101(iny + y + 1, rows) * pitchJ;
          int jv = (r0[x0] * jw00 + r0[x1] * jw01 + r1[x0] * jw10 + r1[x1] * jw11 + (1 << 8)) >> 9;
          int diff = jv - Iw[i];
          b1 += (float)(diff * Ixw[i]);
          b2 += (float)(diff * Iyw[i]);
        }
      }
      b1 = warp_sum(b1) * FLT_SCALE;
      b2 = warp_sum(b2) * FLT_SCALE;
      float2 delta = make_float2((A12 * b2 - A22 * b1) * Dt, (A12 * b1 - A11 * b2) * Dt);
      next.x += delta.x;
      next.y += delta.y;
      result = make_float2(next.x + half, next.y + half);
      if ((double)delta.x * (double)delta.x + (double)delta.y * (double)delta.y <= (double)a.eps_sq) break;
      if (j > 0 && fabs((double)(delta.x + prevDelta.x)) < 0.01 && fabs((double)(delta.y + prevDelta.y)) < 0.01) {
        result.x -= delta.x * 0.5f;
        result.y -= delta.y * 0.5f;
        break;
      }
      prevDelta = delta;
    }
    next = result;
    if (level == 0 && ok) {
      // the reference asks for the error vector, so OpenCV re-checks the final position (lkpyramid.cpp err block)
      int fx = __float2int_rd(next.x - half), fy = __float2int_rd(next.y - half);
      if (fx < -win || fx >= cols || fy < -win || fy >= rows) ok = false;
    }
  }
  if (lane == 0) {
    pts1[pi] = next;
    status[pi] = ok ? 1 : 0;
  }
  if (a.undistort) {
    if (lane == 0) p0n[pi] = undistort_dev(a.model, prev_in, a.calib);
    if (lane == 1) p1n[pi] = undistort_dev(a.model, next, a.calib);
  }
}

// ------------------------------------------------------------------------------------------ LK, 15 x 15 window
// Specialisation for the reference's window (TrackKLT.h:144): ONE CTA PER FEATURE, one warp per pyramid level.
//
// The kernel's duration is the latency of its slowest feature, so the dependent chain of one feature is what counts:
//   set-up   everything that depends only on the PREVIOUS image and the previous position — per level the raw
//            neighbourhood, the Scharr derivatives, the fixed-point I / Ix / Iy patches and the 2 x 2 normal matrix —
//            is built by warp l for level l, all levels at the same time (it used to be 5 x ~4.5k cycles in a row);
//            lane i owns the 2 x 4 block of window pixels at rows 2*(i/4).., columns 4*(i%4).. (the 16th row / column
//            is masked off), its 8 values per patch are parked in shared memory as int16;
//   chain    warps 0..3 then run the coarse-to-fine iterations together, which only touch the NEXT image.  Per level a
//            25 x 25 region of it (REFLECT_101 applied while staging) is copied to shared memory around the start
//            position; of the 15 x 16 window slots each of the 120 active lanes owns two horizontally adjacent pixels,
//            keeps the 2 x 3 block of the next image it interpolates them from in registers and re-reads it — from
//            shared memory — only when the integer window position moves; the region is re-staged if the window leaves
//            it.  The mismatch sums are exact integers (redux.sync per warp, 4 partials through shared memory, one named
//            barrier per iteration), so splitting the window over several warps cannot change a single bit of the
//            result; every warp repeats the scalar part of the iteration (position, weights, 2 x 2 solve, convergence
//            tests) and they stay in lock step.
// The per-pixel arithmetic is that of the generic kernel above; the only difference is that it accumulates the integer
// products in float32 while this kernel sums them exactly.
constexpr int kW15 = 15;
constexpr int kLk15MaxLevels = 6;   // pyramid images (the reference's pyr_levels 5); deeper pyramids take the generic body
constexpr int kJMargin = 4;         // the staged region of the next image extends this far around a window
constexpr int kJSpan = kW15 + 2;    // rows / columns a window touches: 15 + 1 (bilinear) + 1 (the lanes' masked 16th row)
constexpr int kJR = kJSpan + 2 * kJMargin;   // 25
constexpr int kChainWarps = 4;      // warps that share one feature's iteration chain

template <class Args>
__device__ __forceinline__ void lk15_body(const Args &a, const float2 *__restrict__ pts0, float2 *__restrict__ pts1,
                                          uint8_t *__restrict__ status, float2 *__restrict__ p0n, float2 *__restrict__ p1n, int n,
                                          int *host_flag, int flag_value, unsigned *done_counter, const int *__restrict__ tab_cnt,
                                          int tab_stride) {
  constexpr int win = kW15, np = win + 3, nd = win + 1;
  constexpr int kRawLoads = (np * np + 31) / 32;   // 11
  __shared__ uint8_t raw_s[kLk15MaxLevels][np * np + 12];
  __shared__ short ddx_s[kLk15MaxLevels][nd * nd];
  __shared__ short ddy_s[kLk15MaxLevels][nd * nd];
  __shared__ short patch_s[kLk15MaxLevels][3][kW15][16];   // [level][I, Ix, Iy][window row][window column (15 used)]
  __shared__ int red_s[2][kChainWarps][4];                 // per-warp partial sums, double-buffered by iteration parity
  __shared__ float amat_s[kLk15MaxLevels][4];           // [level][A11, A12, A22, level usable]
  __shared__ uint8_t jreg_s[kJR * kJR + 7];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int pi = blockIdx.x;
  const int r0 = (lane >> 2) * 2, c0 = (lane & 3) * 4;
  if (tab_cnt != nullptr) {   // pts0 is a fixed-stride table (cell c at c * stride, tab_cnt[c] live entries)
    const int cell = pi / tab_stride;
    const bool cell_on = cell < 256 && ((a.cell_mask[cell >> 5] >> (cell & 31)) & 1u);
    if (!cell_on || pi - cell * tab_stride >= tab_cnt[cell]) {   // dead slot: only the completion count
      if (threadIdx.x == 0 && host_flag != nullptr && atomicAdd(done_counter, 1u) == (unsigned)n - 1u) {
        *done_counter = 0;
        __threadfence_system();
        *reinterpret_cast<volatile int *>(host_flag) = flag_value;
      }
      return;
    }
  }
  const float2 prev_in = pts0[pi];
  const float half = (win - 1) * 0.5f;
  const float FLT_SCALE = 1.f / (1 << 20);

  // ---- set-up of level `warp`
  if (warp <= a.max_level) {
    const int l = warp;
    const int cols = a.w[l], rows = a.h[l];
    const float lscale = 1.f / (float)(1 << l);
    const float px = prev_in.x * lscale - half, py = prev_in.y * lscale - half;
    const int ipx = __float2int_rd(px), ipy = __float2int_rd(py);
    const bool in_range = !(ipx < -win || ipx >= cols || ipy < -win || ipy >= rows);
    float A11 = 0, A12 = 0, A22 = 0;
    if (in_range) {
      uint8_t *raw = raw_s[l];
      short *ddx = ddx_s[l], *ddy = ddy_s[l];
      {  // raw neighbourhood, origin (ipx - 1, ipy - 1): all loads in flight before the first store
        const uint8_t *I = a.p0[l];
        const int pitchI = a.pitch0[l];
        uint8_t v[kRawLoads];
#pragma unroll
        for (int j = 0; j < kRawLoads; j++) {
          const int i = lane + 32 * j;
          v[j] = 0;
          if (i < np * np) {
            const int r = i / np, c = i - r * np;
            v[j] = I[(size_t)reflect101(ipy - 1 + r, rows) * pitchI + reflect101(ipx - 1 + c, cols)];
          }
        }
#pragma unroll
        for (int j = 0; j < kRawLoads; j++)
          if (lane + 32 * j < np * np) raw[lane + 32 * j] = v[j];
      }
      const float fa = px - ipx, fb = py - ipy;
      const int iw00 = __float2int_rn((1.f - fa) * (1.f - fb) * 16384.f);
      const int iw01 = __float2int_rn(fa * (1.f - fb) * 16384.f);
      const int iw10 = __float2int_rn((1.f - fa) * fb * 16384.f);
      const int iw11 = 16384 - iw00 - iw01 - iw10;
      __syncwarp();
      // Scharr derivatives at (ipx + c, ipy + r), c, r in [0, win]; zero outside the frame
      for (int i = lane; i < nd * nd; i += 32) {
        int r = i / nd, c = i - r * nd;
        int gx = ipx + c, gy = ipy + r;
        int vx = 0, vy = 0;
        if (gx >= 0 && gx < cols && gy >= 0 && gy < rows) {
          const uint8_t *q = raw + (r + 1) * np + (c + 1);
          int tl = q[-np - 1], tc = q[-np], tr = q[-np + 1];
          int ml = q[-1], mr = q[1];
          int bl = q[np - 1], bc = q[np], br = q[np + 1];
          vx = 3 * (tr + br) + 10 * mr - 3 * (tl + bl) - 10 * ml;
          vy = 3 * (bl + br) + 10 * bc - 3 * (tl + tr) - 10 * tc;
        }
        ddx[i] = (short)vx;
        ddy[i] = (short)vy;
      }
      __syncwarp();
#pragma unroll
      for (int k = 0; k < 8; k++) {
        const int y = r0 + (k >> 2), x = c0 + (k & 3);
        int ival = 0, ixval = 0, iyval = 0;
        if (y < win && x < win) {
          const uint8_t *q = raw + (y + 1) * np + (x + 1);
          ival = (q[0] * iw00 + q[1] * iw01 + q[np] * iw10 + q[np + 1] * iw11 + (1 << 8)) >> 9;
          const int di = y * nd + x;
          ixval = (ddx[di] * iw00 + ddx[di + 1] * iw01 + ddx[di + nd] * iw10 + ddx[di + nd + 1] * iw11 + (1 << 13)) >> 14;
          iyval = (ddy[di] * iw00 + ddy[di + 1] * iw01 + ddy[di + nd] * iw10 + ddy[di + nd + 1] * iw11 + (1 << 13)) >> 14;
        }
        if (y < win && x < 16) {
          patch_s[l][0][y][x] = (short)ival;
          patch_s[l][1][y][x] = (short)ixval;
          patch_s[l][2][y][x] = (short)iyval;
        }
        A11 += (float)(ixval * ixval);
        A12 += (float)(ixval * iyval);
        A22 += (float)(iyval * iyval);
      }
      A11 = warp_sum(A11) * FLT_SCALE;
      A12 = warp_sum(A12) * FLT_SCALE;
      A22 = warp_sum(A22) * FLT_SCALE;
    }
    if (lane == 0) {
      amat_s[l][0] = A11;
      amat_s[l][1] = A12;
      amat_s[l][2] = A22;
      amat_s[l][3] = in_range ? 1.f : 0.f;
    }
  }
  __syncthreads();
  if (warp >= kChainWarps) return;

  // ---- the iteration chain (warps 0..3 in lock step; named barrier 1 over 128 threads)
  const int gid = warp * 32 + lane;                 // 0..127; slots 120..127 idle
  const int wy = gid >> 3, wx = (gid & 7) * 2;      // this lane's pixels: (wy, wx) and (wy, wx + 1)
  const bool own0 = wy < win, own1 = wy < win && wx + 1 < win;
  auto chain_sync = [] { asm volatile("bar.sync 1, %0;" ::"n"(kChainWarps * 32) : "memory"); };
  float2 next = a.flow_is_zero ? prev_in : pts1[pi];   // OPTFLOW_USE_INITIAL_FLOW
  bool ok = true;
  int parity = 0;
#pragma unroll 1
  for (int level = a.max_level; level >= 0; level--) {
    const int cols = a.w[level], rows = a.h[level];
    const float lscale = 1.f / (float)(1 << level);
    if (level == a.max_level) {
      next.x = next.x * lscale;
      next.y = next.y * lscale;
    } else {
      next.x = next.x * 2.f;
      next.y = next.y * 2.f;
    }
    if (amat_s[level][3] == 0.f) {
      if (level == 0) ok = false;
      continue;
    }
    const float A11 = amat_s[level][0], A12 = amat_s[level][1], A22 = amat_s[level][2];
    float Dt = A11 * A22 - A12 * A12;
    const float minEig = (A22 + A11 - sqrtf((A11 - A22) * (A11 - A22) + 4.f * A12 * A12)) / (float)(2 * win * win);
    if (minEig < a.min_eig || Dt < FLT_EPSILON) {
      if (level == 0) ok = false;
      continue;
    }
    Dt = 1.f / Dt;
    int Iw0 = 0, Iw1 = 0, Ix0 = 0, Ix1 = 0, Iy0 = 0, Iy1 = 0;
    if (own0) {
      Iw0 = patch_s[level][0][wy][wx];
      Ix0 = patch_s[level][1][wy][wx];
      Iy0 = patch_s[level][2][wy][wx];
    }
    if (own1) {
      Iw1 = patch_s[level][0][wy][wx + 1];
      Ix1 = patch_s[level][1][wy][wx + 1];
      Iy1 = patch_s[level][2][wy][wx + 1];
    }
    float2 result = next;   // nextPts[ptidx] as stored by OpenCV; only rewritten after an update step
    next.x -= half;
    next.y -= half;
    float2 prevDelta = make_float2(0.f, 0.f);
    const uint8_t *J = a.p1[level];
    const int pitchJ = a.pitch1[level];
    int j00 = 0, j01 = 0, j02 = 0, j10 = 0, j11 = 0, j12 = 0;   // the 2 x 3 block of the next image under this lane's pixels
    int cached_x = INT_MIN, cached_y = INT_MIN;
    int reg_x0 = INT_MIN / 2, reg_y0 = INT_MIN / 2;   // origin of the staged region (none yet)
    for (int j = 0; j < a.max_count; j++) {
      const int inx = __float2int_rd(next.x), iny = __float2int_rd(next.y);
      if (inx < -win || inx >= cols || iny < -win || iny >= rows) {
        if (level == 0) ok = false;
        break;
      }
      const float ja = next.x - inx, jbf = next.y - iny;
      const int jw00 = __float2int_rn((1.f - ja) * (1.f - jbf) * 16384.f);
      const int jw01 = __float2int_rn(ja * (1.f - jbf) * 16384.f);
      const int jw10 = __float2int_rn((1.f - ja) * jbf * 16384.f);
      const int jw11 = 16384 - jw00 - jw01 - jw10;
      if (inx != cached_x || iny != cached_y) {   // uniform over the four warps
        cached_x = inx;
        cached_y = iny;
        if (inx < reg_x0 || inx + kJSpan > reg_x0 + kJR || iny < reg_y0 || iny + kJSpan > reg_y0 + kJR) {
          // (re)stage the region around the window; pixel (rx, ry) of it is J(reflect(reg_x0 + rx), reflect(reg_y0 + ry))
          reg_x0 = inx - kJMargin;
          reg_y0 = iny - kJMargin;
          chain_sync();   // everybody is done reading the old region
          constexpr int kJLoads = (kJR * kJR + kChainWarps * 32 - 1) / (kChainWarps * 32);
          uint8_t t[kJLoads];
#pragma unroll
          for (int q = 0; q < kJLoads; q++) {
            const int i = gid + kChainWarps * 32 * q;
            const int ry = i / kJR, rx = i - ry * kJR;
            t[q] = 0;
            if (i < kJR * kJR) t[q] = J[(size_t)reflect101(reg_y0 + ry, rows) * pitchJ + reflect101(reg_x0 + rx, cols)];
          }
#pragma unroll
          for (int q = 0; q < kJLoads; q++)
            if (gid + kChainWarps * 32 * q < kJR * kJR) jreg_s[gid + kChainWarps * 32 * q] = t[q];
          chain_sync();
        }
        if (own0) {
          const uint8_t *Jp = jreg_s + (iny - reg_y0 + wy) * kJR + (inx - reg_x0 + wx);
          j00 = Jp[0]; j01 = Jp[1]; j02 = Jp[2];
          j10 = Jp[kJR]; j11 = Jp[kJR + 1]; j12 = Jp[kJR + 2];
        }
      }
      // mismatch vector b = sum over the window of diff * (Ix, Iy).  Every term is an integer, so the sum is formed
      // EXACTLY: per-lane int32 sums, hardware warp reductions on the 16-bit halves (the window total needs 34 bits),
      // four warp partials through shared memory, one rounding to float at the end.  OpenCV accumulates the same
      // integers in float32 (order depends on its SIMD width); this is that sum without the accumulated rounding error.
      int sb1 = 0, sb2 = 0;
      {
        const int jv0 = (j00 * jw00 + j01 * jw01 + j10 * jw10 + j11 * jw11 + (1 << 8)) >> 9;
        const int jv1 = (j01 * jw00 + j02 * jw01 + j11 * jw10 + j12 * jw11 + (1 << 8)) >> 9;
        const int d0 = own0 ? jv0 - Iw0 : 0, d1 = own1 ? jv1 - Iw1 : 0;
        sb1 = d0 * Ix0 + d1 * Ix1;
        sb2 = d0 * Iy0 + d1 * Iy1;
      }
      const int p1h = __reduce_add_sync(0xffffffffu, sb1 >> 16), p1l = __reduce_add_sync(0xffffffffu, sb1 & 0xffff);
      const int p2h = __reduce_add_sync(0xffffffffu, sb2 >> 16), p2l = __reduce_add_sync(0xffffffffu, sb2 & 0xffff);
      if (lane == 0) {
        red_s[parity][warp][0] = p1h;
        red_s[parity][warp][1] = p1l;
        red_s[parity][warp][2] = p2h;
        red_s[parity][warp][3] = p2l;
      }
      chain_sync();
      long long t1h = 0, t1l = 0, t2h = 0, t2l = 0;
#pragma unroll
      for (int w = 0; w < kChainWarps; w++) {
        t1h += red_s[parity][w][0];
        t1l += red_s[parity][w][1];
        t2h += red_s[parity][w][2];
        t2l += red_s[parity][w][3];
      }
      parity ^= 1;
      const float b1 = (float)((t1h << 16) + t1l) * FLT_SCALE;
      const float b2 = (float)((t2h << 16) + t2l) * FLT_SCALE;
      const float2 delta = make_float2((A12 * b2 - A22 * b1) * Dt, (A12 * b1 - A11 * b2) * Dt);
      next.x += delta.x;
      next.y += delta.y;
      result = make_float2(next.x + half, next.y + half);
      // delta.dot(delta) <= epsilon in double, decided in float whenever the float value is not within rounding distance
      // of the threshold (the double expression is evaluated only then: same decision, no fp64 on the common path)
      {
        const float d2 = delta.x * delta.x + delta.y * delta.y;
        bool stop;
        if (d2 < a.eps_sq * 0.999999f) stop = true;
        else if (d2 > a.eps_sq * 1.000001f) stop = false;
        else stop = (double)delta.x * (double)delta.x + (double)delta.y * (double)delta.y <= (double)a.eps_sq;
        if (stop) break;
      }
      // |float| < 0.01 (a double constant): 0.01f is the largest float below 0.01, so this is |float| <= 0.01f
      if (j > 0 && fabsf(delta.x + prevDelta.x) <= 0.01f && fabsf(delta.y + prevDelta.y) <= 0.01f) {
        result.x -= delta.x * 0.5f;
        result.y -= delta.y * 0.5f;
        break;
      }
      prevDelta = delta;
    }
    next = result;
    if (level == 0 && ok) {
      // the reference asks for the error vector, so OpenCV re-checks the final position (lkpyramid.cpp err block)
      int fx = __float2int_rd(next.x - half), fy = __float2int_rd(next.y - half);
      if (fx < -win || fx >= cols || fy < -win || fy >= rows) ok = false;
    }
  }
  if (warp != 0) return;
  if (lane == 0) {
    pts1[pi] = next;
    status[pi] = ok ? 1 : 0;
  }
  if (a.undistort) {
    if (lane == 0) p0n[pi] = undistort_dev(a.model, prev_in, a.calib);
    if (lane == 1) p1n[pi] = undistort_dev(a.model, next, a.calib);
  }
  // ---- completion signal: the last feature to finish publishes the sequence number (results first, system-wide)
  if (host_flag != nullptr) {
    __threadfence_system();
    __syncwarp();
    if (lane == 0) {
      if (atomicAdd(done_counter, 1u) == (unsigned)n - 1u) {
        *done_counter = 0;
        __threadfence_system();
        *reinterpret_cast<volatile int *>(host_flag) = flag_value;
      }
    }
  }
}

__global__ void __launch_bounds__(kLk15MaxLevels * 32)
    k_lk15(LkArgs a, const float2 *__restrict__ pts0, float2 *__restrict__ pts1, uint8_t *__restrict__ status,
           float2 *__restrict__ p0n, float2 *__restrict__ p1n, int n, int *host_flag, int flag_value, unsigned *done_counter,
           const int *__restrict__ tab_cnt, int tab_stride) {
  lk15_body(a, pts0, pts1, status, p0n, p1n, n, host_flag, flag_value, done_counter, tab_cnt, tab_stride);
}

// ------------------------------------------------------------------------------ LK, 15 x 15 window, one warp per feature
// The throughput form of k_lk15, for launches that carry thousands of features (stream groups).  k_lk15 minimises the
// LATENCY of one feature: a CTA per feature, six warps building the levels side by side, four warps sharing the iteration
// chain with a barrier per iteration — every warp repeats the scalar part of an iteration, and an SM holds 10 features.
// Here ONE warp owns a feature: it builds level l (the same code, so the float normal matrix is summed in the same order),
// then runs level l's iterations alone — lane (row, half) owns 8 (7) adjacent window pixels of one row, their I / Ix / Iy
// values and the 2 x 9 block of the next image under them stay in registers, no barrier, no exchange through shared memory
// — and moves on to level l - 1.  The mismatch sums are exact integers (per-lane 32-bit, warp reductions on 16-bit halves),
// so the split of the window over lanes cannot change a bit: results are identical to k_lk15's (tests/test_group_gpu.py
// compares a group, which runs this kernel, with single handles, which run k_lk15).  An SM holds 32+ features.
// Staged rows of the previous image (18 x 18 pixels) and of the region of the next image (25 x 25) are kept with a row
// stride that is a multiple of 4 bytes and their first word aligned like the image's (it holds the region's first column,
// x0 & 3 bytes in).  Rows are reflected through their row pointer; a word that lies inside the image row is one 32-bit
// load, and only the words that cross or lie beyond its left or right edge are assembled from REFLECT_101 columns byte by
// byte.  Interior and border neighbourhoods take the same path, and the bytes in shared memory are the reference's.
constexpr int kRawStride = 24;   // >= 18 + 3
constexpr int kJStride = 28;     // >= 25 + 3
// One buffer per warp, used three ways in turn (each hand-over is separated by a __syncwarp): the staged rows of the previous
// image + the Scharr planes (set-up), the fixed-point patches I / Ix / Iy (written once every lane has read what it needs of
// the former, read back row-wise into registers), the staged region of the next image (iterations).  1.5 KB per feature
// instead of 3.6 KB: a CTA of four features needs 6 KB of shared memory, so the kernel's residency does not depend on what
// the long-lived kernels of the pipeline (the chain walkers) leave free.
constexpr int kLkwDdxOff = ((kW15 + 3) * kRawStride + 8 + 15) & ~15;                  // 448
constexpr int kLkwDdyOff = kLkwDdxOff + (kW15 + 1) * (kW15 + 1) * 2;                   // 960
constexpr int kLkwBytes = kLkwDdyOff + (kW15 + 1) * (kW15 + 1) * 2;                    // 1472
static_assert(3 * kW15 * 16 * 2 <= kLkwBytes && kJR * kJStride + 4 <= kLkwBytes, "patches and the J region fit the buffer");
struct LkwSmem {
  __align__(16) uint8_t buf[kLkwBytes];
};

// kRows staged rows of kStride bytes: image rows y0.., columns from the word that holds column x0 (see above).  `aligned`:
// the image pointer and pitch are multiples of 4 (group pyramids are 256-byte aligned); otherwise every word is assembled
// byte by byte.
template <int kRows, int kStride>
__device__ __forceinline__ void lkw_stage(uint8_t *dst, const uint8_t *__restrict__ img, int pitch, int cols, int rows, int x0,
                                          int y0, bool aligned, int lane) {
  constexpr int kW = kStride / 4, kN = kRows * kW, kL = (kN + 31) / 32;
  const int xw = x0 & ~3;
  unsigned v[kL];
#pragma unroll
  for (int j = 0; j < kL; j++) {
    const int i = lane + 32 * j;
    v[j] = 0;
    if (i < kN) {
      const int r = i / kW, x = xw + 4 * (i - r * kW);
      const uint8_t *row = img + (size_t)reflect101(y0 + r, rows) * pitch;
      if (aligned && x >= 0 && x + 4 <= cols) {
        v[j] = __ldg(reinterpret_cast<const unsigned *>(row + x));
      } else {
#pragma unroll
        for (int k = 0; k < 4; k++) v[j] |= (unsigned)__ldg(row + reflect101(x + k, cols)) << (8 * k);
      }
    }
  }
#pragma unroll
  for (int j = 0; j < kL; j++)
    if (lane + 32 * j < kN) reinterpret_cast<unsigned *>(dst)[lane + 32 * j] = v[j];
}

// Bilinear taps as 2-way dot products: w holds two signed 16-bit weights, px four unsigned 8-bit pixels, of which the low
// (dp2a_lo) or high (dp2a_hi) pair is used: c + w.h0 * px.b0 + w.h1 * px.b1.  Exact in int32 (|weight| <= 16384).
__device__ __forceinline__ int dp2a_lo(int w, unsigned px, int c) {
  int d;
  asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(w), "r"(px), "r"(c));
  return d;
}
__device__ __forceinline__ int dp2a_hi(int w, unsigned px, int c) {
  int d;
  asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(w), "r"(px), "r"(c));
  return d;
}
__device__ __forceinline__ int pack_w16(int lo, int hi) { return (int)(((unsigned)lo & 0xffffu) | ((unsigned)hi << 16)); }

template <class Args>
__device__ __forceinline__ void lk15w_body(const Args &a, const float2 *__restrict__ pts0, float2 *__restrict__ pts1,
                                           uint8_t *__restrict__ status, float2 *__restrict__ p0n, float2 *__restrict__ p1n, int pi,
                                           LkwSmem &sm) {
  constexpr int win = kW15, np = win + 3, nd = win + 1;
  const int lane = threadIdx.x & 31;
  const int r0 = (lane >> 2) * 2, c0 = (lane & 3) * 4;   // set-up: this lane's 2 x 4 block of window pixels
  const int wy = lane >> 1, wx = (lane & 1) * 8;         // chain: this lane's row and its 8 adjacent pixels
  const bool own = wy < win;
  const float2 prev_in = pts0[pi];
  const float half = (win - 1) * 0.5f;
  const float FLT_SCALE = 1.f / (1 << 20);
  float2 next = a.flow_is_zero ? prev_in : pts1[pi];   // OPTFLOW_USE_INITIAL_FLOW
  bool ok = true;
#pragma unroll 1
  for (int level = a.max_level; level >= 0; level--) {
    const int cols = a.w[level], rows = a.h[level];
    const float lscale = 1.f / (float)(1 << level);
    if (level == a.max_level) {
      next.x = next.x * lscale;
      next.y = next.y * lscale;
    } else {
      next.x = next.x * 2.f;
      next.y = next.y * 2.f;
    }
    // ---- set-up of this level (k_lk15's integers and float sums): raw neighbourhood, Scharr derivatives, fixed-point
    // patches, A
    const float px = prev_in.x * lscale - half, py = prev_in.y * lscale - half;
    const int ipx = __float2int_rd(px), ipy = __float2int_rd(py);
    const bool in_range = !(ipx < -win || ipx >= cols || ipy < -win || ipy >= rows);
    if (!in_range) {
      if (level == 0) ok = false;
      continue;
    }
    float A11 = 0, A12 = 0, A22 = 0;
    __syncwarp();   // the previous level's patches have been read by every lane
    {
      uint8_t *const raw_s = sm.buf;
      short *ddx = reinterpret_cast<short *>(sm.buf + kLkwDdxOff), *ddy = reinterpret_cast<short *>(sm.buf + kLkwDdyOff);
      // raw neighbourhood, origin (ipx - 1, ipy - 1): 18 rows x 6 words, column ipx - 1 at byte roff of each row
      const uint8_t *I = a.p0[level];
      const int pitchI = a.pitch0[level];
      const int roff = (ipx - 1) & 3;
      lkw_stage<np, kRawStride>(raw_s, I, pitchI, cols, rows, ipx - 1, ipy - 1, ((((size_t)I) | (size_t)pitchI) & 3) == 0, lane);
      const float fa = px - ipx, fb = py - ipy;
      const int iw00 = __float2int_rn((1.f - fa) * (1.f - fb) * 16384.f);
      const int iw01 = __float2int_rn(fa * (1.f - fb) * 16384.f);
      const int iw10 = __float2int_rn((1.f - fa) * fb * 16384.f);
      const int iw11 = 16384 - iw00 - iw01 - iw10;
      __syncwarp();
      {
        // Scharr derivatives of the 16 x 16 positions (ipx + c, ipy + r): this lane's row r and 8 adjacent columns from
        // three staged rows of 10 pixels, each taken as four aligned words and shifted into place; zero outside the frame,
        // which is what the reference's zero-padded derivative planes hold
        const int r = lane >> 1, cb = (lane & 1) * 8;
        unsigned X[3][3];
#pragma unroll
        for (int k = 0; k < 3; k++) {
          const uint2 *rp = reinterpret_cast<const uint2 *>(raw_s + (r + k) * kRawStride + cb);   // 8-byte aligned (stride 24)
          const uint2 wa = rp[0], wb = rp[1];
          X[k][0] = __funnelshift_r(wa.x, wa.y, 8 * roff);
          X[k][1] = __funnelshift_r(wa.y, wb.x, 8 * roff);
          X[k][2] = __funnelshift_r(wb.x, wb.y, 8 * roff);
        }
        int S[10], Dv[10];   // column smoothing 3 t + 10 m + 3 b and column difference b - t
#pragma unroll
        for (int c = 0; c < 10; c++) {
          const int t = (X[0][c >> 2] >> (8 * (c & 3))) & 0xff, m = (X[1][c >> 2] >> (8 * (c & 3))) & 0xff,
                    bb = (X[2][c >> 2] >> (8 * (c & 3))) & 0xff;
          S[c] = 3 * (t + bb) + 10 * m;
          Dv[c] = bb - t;
        }
        const int gy = ipy + r, gx = ipx + cb;
        const bool inside = gy >= 0 && gy < rows && gx >= 0 && gx + 8 <= cols;
        unsigned qx[4], qy[4];
#pragma unroll
        for (int c = 0; c < 8; c += 2) {
          int vx0 = S[c + 2] - S[c], vx1 = S[c + 3] - S[c + 1];
          int vy0 = 3 * (Dv[c] + Dv[c + 2]) + 10 * Dv[c + 1], vy1 = 3 * (Dv[c + 1] + Dv[c + 3]) + 10 * Dv[c + 2];
          if (!inside) {
            const bool row_in = gy >= 0 && gy < rows;
            if (!(row_in && (unsigned)(gx + c) < (unsigned)cols)) vx0 = vy0 = 0;
            if (!(row_in && (unsigned)(gx + c + 1) < (unsigned)cols)) vx1 = vy1 = 0;
          }
          qx[c >> 1] = ((unsigned)vx0 & 0xffffu) | ((unsigned)vx1 << 16);
          qy[c >> 1] = ((unsigned)vy0 & 0xffffu) | ((unsigned)vy1 << 16);
        }
        *reinterpret_cast<uint4 *>(&ddx[r * nd + cb]) = make_uint4(qx[0], qx[1], qx[2], qx[3]);
        *reinterpret_cast<uint4 *>(&ddy[r * nd + cb]) = make_uint4(qy[0], qy[1], qy[2], qy[3]);
      }
      __syncwarp();
      short pv[3][8];   // this lane's 2 x 4 block of I, Ix, Iy: stored once every lane is done with the rows and planes
      {
        // bilinear taps of I: staged rows r0 + 1 .. r0 + 3 from column c0 + 1 on, P = bytes 0..3 and Q = bytes 1..4 of it
        const int wI0 = pack_w16(iw00, iw01), wI1 = pack_w16(iw10, iw11);
        const int off = roff + c0 + 1;
        unsigned P[3], Q[3];
#pragma unroll
        for (int k = 0; k < 3; k++) {
          const unsigned *rp = reinterpret_cast<const unsigned *>(raw_s + (r0 + 1 + k) * kRawStride) + (off >> 2);
          const unsigned w0 = rp[0], w1 = rp[1];
          P[k] = __funnelshift_r(w0, w1, 8 * (off & 3));
          Q[k] = __funnelshift_rc(w0, w1, 8 * (off & 3) + 8);   // clamped: a shift of 32 yields w1
        }
        // derivative rows r0 .. r0 + 2 (clamped to the plane), columns c0 .. c0 + 4, read as int16 pairs
        int dx[3][5], dy[3][5];
#pragma unroll
        for (int k = 0; k < 3; k++) {
          const int rr = min(r0 + k, nd - 1);
          const uint2 xa = *reinterpret_cast<const uint2 *>(&ddx[rr * nd + c0]);
          const uint2 ya = *reinterpret_cast<const uint2 *>(&ddy[rr * nd + c0]);
          const unsigned xe = *reinterpret_cast<const unsigned *>(&ddx[rr * nd + min(c0 + 4, nd - 2)]);
          const unsigned ye = *reinterpret_cast<const unsigned *>(&ddy[rr * nd + min(c0 + 4, nd - 2)]);
          dx[k][0] = (short)(xa.x & 0xffffu); dx[k][1] = (int)xa.x >> 16;
          dx[k][2] = (short)(xa.y & 0xffffu); dx[k][3] = (int)xa.y >> 16;
          dx[k][4] = (short)(xe & 0xffffu);
          dy[k][0] = (short)(ya.x & 0xffffu); dy[k][1] = (int)ya.x >> 16;
          dy[k][2] = (short)(ya.y & 0xffffu); dy[k][3] = (int)ya.y >> 16;
          dy[k][4] = (short)(ye & 0xffffu);
        }
#pragma unroll
        for (int k = 0; k < 8; k++) {
          const int t = k >> 2, m = k & 3;
          const int y = r0 + t, x = c0 + m;
          int ival = 0, ixval = 0, iyval = 0;
          if (y < win && x < win) {
            const unsigned top = (m & 1) ? Q[t] : P[t], bot = (m & 1) ? Q[t + 1] : P[t + 1];
            ival = ((m & 2) ? dp2a_hi(wI0, top, dp2a_hi(wI1, bot, 1 << 8)) : dp2a_lo(wI0, top, dp2a_lo(wI1, bot, 1 << 8))) >> 9;
            ixval = (dx[t][m] * iw00 + dx[t][m + 1] * iw01 + dx[t + 1][m] * iw10 + dx[t + 1][m + 1] * iw11 + (1 << 13)) >> 14;
            iyval = (dy[t][m] * iw00 + dy[t][m + 1] * iw01 + dy[t + 1][m] * iw10 + dy[t + 1][m + 1] * iw11 + (1 << 13)) >> 14;
          }
          pv[0][k] = (short)ival;
          pv[1][k] = (short)ixval;
          pv[2][k] = (short)iyval;
          A11 += (float)(ixval * ixval);
          A12 += (float)(ixval * iyval);
          A22 += (float)(iyval * iyval);
        }
      }
      __syncwarp();   // the patches take the place of the rows and planes they were computed from
      {
        short(*patch)[kW15][16] = reinterpret_cast<short(*)[kW15][16]>(sm.buf);
#pragma unroll
        for (int pl = 0; pl < 3; pl++)
#pragma unroll
          for (int rr = 0; rr < 2; rr++) {
            const int y = r0 + rr;
            if (y < win) {
              const unsigned lo = ((unsigned)(unsigned short)pv[pl][4 * rr]) | ((unsigned)(unsigned short)pv[pl][4 * rr + 1] << 16);
              const unsigned hi = ((unsigned)(unsigned short)pv[pl][4 * rr + 2]) | ((unsigned)(unsigned short)pv[pl][4 * rr + 3] << 16);
              *reinterpret_cast<uint2 *>(&patch[pl][y][c0]) = make_uint2(lo, hi);
            }
          }
      }
      A11 = warp_sum(A11) * FLT_SCALE;
      A12 = warp_sum(A12) * FLT_SCALE;
      A22 = warp_sum(A22) * FLT_SCALE;
    }
    __syncwarp();
    float Dt = A11 * A22 - A12 * A12;
    const float minEig = (A22 + A11 - sqrtf((A11 - A22) * (A11 - A22) + 4.f * A12 * A12)) / (float)(2 * win * win);
    if (minEig < a.min_eig || Dt < FLT_EPSILON) {
      if (level == 0) ok = false;
      continue;
    }
    Dt = 1.f / Dt;
    // ---- this lane's 8 window pixels: Ix, Iy (int16 pairs, one 16-byte load per patch) and the constant part of the
    // mismatch sums, ci1 = sum I * Ix and ci2 = sum I * Iy
    int Ix[8], Iy[8], ci1 = 0, ci2 = 0;
    {
      uint4 q0 = make_uint4(0, 0, 0, 0), q1 = q0, q2 = q0;
      if (own) {
        const short(*patch)[kW15][16] = reinterpret_cast<const short(*)[kW15][16]>(sm.buf);
        q0 = *reinterpret_cast<const uint4 *>(&patch[0][wy][wx]);
        q1 = *reinterpret_cast<const uint4 *>(&patch[1][wy][wx]);
        q2 = *reinterpret_cast<const uint4 *>(&patch[2][wy][wx]);
      }
      const unsigned w0[4] = {q0.x, q0.y, q0.z, q0.w}, w1[4] = {q1.x, q1.y, q1.z, q1.w}, w2[4] = {q2.x, q2.y, q2.z, q2.w};
#pragma unroll
      for (int k = 0; k < 4; k++) {
        Ix[2 * k] = (short)(w1[k] & 0xffffu);
        Ix[2 * k + 1] = (short)(w1[k] >> 16);
        Iy[2 * k] = (short)(w2[k] & 0xffffu);
        Iy[2 * k + 1] = (short)(w2[k] >> 16);
        const int i0 = (short)(w0[k] & 0xffffu), i1 = (short)(w0[k] >> 16);
        ci1 += i0 * Ix[2 * k] + i1 * Ix[2 * k + 1];
        ci2 += i0 * Iy[2 * k] + i1 * Iy[2 * k + 1];
      }
    }
    float2 result = next;   // nextPts[ptidx] as stored by OpenCV; only rewritten after an update step
    next.x -= half;
    next.y -= half;
    float2 prevDelta = make_float2(0.f, 0.f);
    const uint8_t *J = a.p1[level];
    const int pitchJ = a.pitch1[level];
    const bool alignedJ = ((((size_t)J) | (size_t)pitchJ) & 3) == 0;
    // the 2 x 9 block of the next image under this lane's pixels, byte-packed: per row, columns 0..3, 1..4, 4..7, 5..8
    unsigned jt[4] = {0, 0, 0, 0}, jb[4] = {0, 0, 0, 0};
    int cached_x = INT_MIN, cached_y = INT_MIN;
    int reg_x0 = INT_MIN / 2, reg_y0 = INT_MIN / 2;   // origin of the staged region (none yet)
    for (int j = 0; j < a.max_count; j++) {
      const int inx = __float2int_rd(next.x), iny = __float2int_rd(next.y);
      if (inx < -win || inx >= cols || iny < -win || iny >= rows) {
        if (level == 0) ok = false;
        break;
      }
      const float ja = next.x - inx, jbf = next.y - iny;
      const int jw00 = __float2int_rn((1.f - ja) * (1.f - jbf) * 16384.f);
      const int jw01 = __float2int_rn(ja * (1.f - jbf) * 16384.f);
      const int jw10 = __float2int_rn((1.f - ja) * jbf * 16384.f);
      const int jw11 = 16384 - jw00 - jw01 - jw10;
      if (inx != cached_x || iny != cached_y) {   // warp-uniform
        cached_x = inx;
        cached_y = iny;
        if (inx < reg_x0 || inx + kJSpan > reg_x0 + kJR || iny < reg_y0 || iny + kJSpan > reg_y0 + kJR) {
          // (re)stage the region around the window; pixel (rx, ry) of it is J(reflect(reg_x0 + rx), reflect(reg_y0 + ry))
          reg_x0 = inx - kJMargin;
          reg_y0 = iny - kJMargin;
          __syncwarp();   // every lane is done reading the old region
          lkw_stage<kJR, kJStride>(sm.buf, J, pitchJ, cols, rows, reg_x0, reg_y0, alignedJ, lane);
          __syncwarp();
        }
        if (own) {
          const int o = inx - reg_x0 + (reg_x0 & 3) + wx;   // byte of this lane's first pixel in its staged row
          const unsigned *rp = reinterpret_cast<const unsigned *>(sm.buf + (iny - reg_y0 + wy) * kJStride) + (o >> 2);
          const int sh = 8 * (o & 3);
          unsigned w0 = rp[0], w1 = rp[1], w2 = rp[2];
          jt[0] = __funnelshift_r(w0, w1, sh);
          jt[1] = __funnelshift_rc(w0, w1, sh + 8);   // clamped: a shift of 32 yields w1
          jt[2] = __funnelshift_r(w1, w2, sh);
          jt[3] = __funnelshift_rc(w1, w2, sh + 8);
          w0 = rp[kJStride / 4];
          w1 = rp[kJStride / 4 + 1];
          w2 = rp[kJStride / 4 + 2];
          jb[0] = __funnelshift_r(w0, w1, sh);
          jb[1] = __funnelshift_rc(w0, w1, sh + 8);
          jb[2] = __funnelshift_r(w1, w2, sh);
          jb[3] = __funnelshift_rc(w1, w2, sh + 8);
        }
      }
      // mismatch vector b = sum (J - I) * (Ix, Iy) = sum J * (Ix, Iy) - (ci1, ci2), in exact integers (the pixels a lane
      // does not own have Ix = Iy = 0 and I = 0).  Bounds: the four bilinear weights sum to 16384 and none is below -2,
      // so |J|, |I| <= 8161 and |Ix|, |Iy| <= 16 * 255 = 4080 (Scharr of 8-bit pixels); every product is below 2^25, a
      // lane's eight-term sums below 2^28 and their difference below 2^29: 32-bit per lane, the warp total through 16-bit
      // halves as in k_lk15
      const int wJ0 = pack_w16(jw00, jw01), wJ1 = pack_w16(jw10, jw11);
      int s1 = -ci1, s2 = -ci2;
#pragma unroll
      for (int k = 0; k < 8; k++) {
        const int q = ((k >> 2) << 1) | (k & 1);   // pixel k's pair (k, k + 1): low or high half of jt[q] / jb[q]
        const int jv = ((k & 2) ? dp2a_hi(wJ0, jt[q], dp2a_hi(wJ1, jb[q], 1 << 8)) : dp2a_lo(wJ0, jt[q], dp2a_lo(wJ1, jb[q], 1 << 8))) >> 9;
        s1 += jv * Ix[k];
        s2 += jv * Iy[k];
      }
      const long long t1 = ((long long)__reduce_add_sync(0xffffffffu, s1 >> 16) << 16) + (long long)__reduce_add_sync(0xffffffffu, s1 & 0xffff);
      const long long t2 = ((long long)__reduce_add_sync(0xffffffffu, s2 >> 16) << 16) + (long long)__reduce_add_sync(0xffffffffu, s2 & 0xffff);
      const float b1 = (float)t1 * FLT_SCALE;
      const float b2 = (float)t2 * FLT_SCALE;
      const float2 delta = make_float2((A12 * b2 - A22 * b1) * Dt, (A12 * b1 - A11 * b2) * Dt);
      next.x += delta.x;
      next.y += delta.y;
      result = make_float2(next.x + half, next.y + half);
      {
        const float d2 = delta.x * delta.x + delta.y * delta.y;
        bool stop;
        if (d2 < a.eps_sq * 0.999999f) stop = true;
        else if (d2 > a.eps_sq * 1.000001f) stop = false;
        else stop = (double)delta.x * (double)delta.x + (double)delta.y * (double)delta.y <= (double)a.eps_sq;
        if (stop) break;
      }
      if (j > 0 && fabsf(delta.x + prevDelta.x) <= 0.01f && fabsf(delta.y + prevDelta.y) <= 0.01f) {
        result.x -= delta.x * 0.5f;
        result.y -= delta.y * 0.5f;
        break;
      }
      prevDelta = delta;
    }
    next = result;
    if (level == 0 && ok) {
      int fx = __float2int_rd(next.x - half), fy = __float2int_rd(next.y - half);
      if (fx < -win || fx >= cols || fy < -win || fy >= rows) ok = false;
    }
  }
  if (lane == 0) {
    pts1[pi] = next;
    status[pi] = ok ? 1 : 0;
  }
  if (a.undistort) {
    if (lane == 0) p0n[pi] = undistort_dev(a.model, prev_in, a.calib);
    if (lane == 1) p1n[pi] = undistort_dev(a.model, next, a.calib);
  }
}

// ------------------------------------------------------------------------------------- LK, one warp per feature
// Two kernel templates, one per body — k_lk_g (lk_body, any window) and k_lk15w_g (lk15w_body) — over a point source that
// gives CTA (blockIdx.x, blockIdx.y) its job (grid.y) and features blockIdx.x * kLkWarps + warp of that job:
//   Cta                  the source's shared per-CTA state
//   setup(c, first)      thread 0, once per CTA: the job's feature count; c is set up when feature `first` is below it
//   track(c, pi, body)   runs body(args, pts0, pts1, status, p0n, p1n, i) on feature pi of the job and stores what it leaves

// n points in explicit arrays over one pyramid pair (launch_lk's generic form, launch_lk_warp)
struct LkArrays {
  LkArgs a;
  const float2 *pts0;
  float2 *pts1;
  uint8_t *status;
  float2 *p0n, *p1n;
  int n;
  struct Cta {};
  __device__ int setup(Cta &, int) const { return n; }
  template <class Body>
  __device__ void track(Cta &, int pi, Body body) const { body(a, pts0, pts1, status, p0n, p1n, pi); }
};

// The group sources assemble a job's LkArgs in shared memory from the slot table, through the prm.max_level + 1 images every
// slot's pyramid holds (FeGroup clamps max_level to them), so a stream's tracks are bit-identical to those of a single handle.
struct GroupSrc {
  GroupDev g;
  const TrackJob *jobs;
  LkParams prm;
  // previous image = slot s0, next image = slot s1, calibration of `cal`, initial guess = the previous position
  __device__ void args(LkArgs &a, int s0, int s1, const TrackJob &cal, int undistort) const {
    lk_args(a, g.slots[s0].lvl, g.slots[s1].lvl, prm.max_level + 1, prm, cal.K, cal.D, undistort, 1, nullptr);
  }
};

// Stream group: the working list of every stream of a tracking launch, previous -> current image (pts_new = pts_old,
// TrackKLT.cpp:134); a stream with fewer than 10 points runs no LK (TrackKLT.cpp:848-852).
struct GroupPoints : GroupSrc {
  struct Cta {
    LkArgs a;
  };
  __device__ int setup(Cta &c, int first) const {
    const TrackJob &job = jobs[blockIdx.y];
    const int n = g.wn[job.stream];
    if (g.wmode[job.stream] != 0 || n < 10) return 0;
    if (first < n) args(c.a, job.prev_slot, job.cur_slot, job, 1);
    return n;
  }
  template <class Body>
  __device__ void track(Cta &c, int pi, Body body) const {
    const size_t o = (size_t)jobs[blockIdx.y].stream * g.pts_cap;
    body(c.a, g.wpts + o, g.lk_pts1 + o, g.lk_status + o, g.lk_p0n + o, g.lk_p1n + o, pi);
  }
};

// Stereo group: the left -> right KLT of the new left points of a rig's detection (perform_detection_stereo :658-666,
// FeStereo's lk_launch(L.pyr, R.pyr, new0, ..., false)): previous image = the left image of the detection pair, next image =
// its right image, initial flow = the left position, no undistortion.  The new points are the tail k_group_accept appended
// to the left working list; the results go to the RIGHT stream's LK arrays (k_stereo_pair reads them).  grid.y = rig, on
// the left half of the lane's jobs.
struct StereoLr : GroupSrc {
  struct Cta {
    LkArgs a;
    int start;   // the first new point in the left working list
  };
  __device__ int setup(Cta &c, int first) const {
    const TrackJob &lj = jobs[blockIdx.y], &rj = jobs[blockIdx.y + gridDim.y];
    const int n = g.winfo[4 * lj.stream + 1];
    c.start = g.wn[lj.stream] - n;
    if (first < n) {
      const bool first_frame = g.wmode[lj.stream] == 1;
      args(c.a, first_frame ? lj.cur_slot : lj.prev_slot, first_frame ? rj.cur_slot : rj.prev_slot, lj, 0);
    }
    return n;
  }
  template <class Body>
  __device__ void track(Cta &c, int pi, Body body) const {
    const size_t ol = (size_t)jobs[blockIdx.y].stream * g.pts_cap, orr = (size_t)jobs[blockIdx.y + gridDim.y].stream * g.pts_cap;
    body(c.a, g.wpts + ol + c.start, g.lk_pts1 + orr, g.lk_status + orr, nullptr, nullptr, pi);
  }
};

// Stream group, cfg.line_samples: the samples a handle appends to its point LK launch (fe_context.cu perform_matching),
// grid.y = job.  Samples exist when the frame's point LK ran — the gate then wrote n_lk_in = n >= 10 into the frame's
// header, 0 otherwise — and lie along the stream's last detected segments (lnew, n_lnew: k_group_lines of the latest frame
// fed with vanishing points), k = 0..S-1 per segment, cut where the handle's LK buffer ends: ns = min(S * L, max_pts - n).
// Same LK parameters and pyramids as the points, initial guess = the sample itself, no undistortion (the handle computes
// the samples' undistorted positions and discards them).  CTAs past the job's samples read nothing but n_lnew.
struct LineSamples : GroupSrc {
  struct Cta {
    LkArgs a;
    float2 p1[kLkWarps];   // the body's result, stored to the record afterwards (no record pointer held through it)
    uint8_t st[kLkWarps];
  };
  __device__ int setup(Cta &c, int first) const {
    const TrackJob &job = jobs[blockIdx.y];
    const long long all = (long long)g.line_samples * g.n_lnew[job.stream];
    if (first >= all) return 0;
    GroupOutHeader *hdr = reinterpret_cast<GroupOutHeader *>(g.out + (size_t)job.out * g.out_stride);
    const int n = hdr->info.n_lk_in;
    if (n < 10) return 0;
    const int ns = (int)max(0ll, min(all, (long long)(g.sample_max_pts - n)));
    if (blockIdx.x == 0) hdr->n_samples = ns;
    if (first < ns) args(c.a, job.prev_slot, job.cur_slot, job, 0);
    return ns;
  }
  // sample pi: a = k / (S - 1) (0.5 for S = 1) along segment pi / S, rounded as the host rounds it (no contraction)
  template <class Body>
  __device__ void track(Cta &c, int pi, Body body) const {
    const TrackJob &job = jobs[blockIdx.y];
    const int warp = threadIdx.x >> 5, S = g.line_samples, k = pi % S;
    const float4 l = g.lnew[(size_t)job.stream * g.lines_cap + pi / S];
    const float a = S > 1 ? (float)k / (float)(S - 1) : 0.5f;
    const float2 p0 = make_float2(l.x + (l.z - l.x) * a, l.y + (l.w - l.y) * a);
    body(c.a, &p0, &c.p1[warp], &c.st[warp], nullptr, nullptr, 0);
    if ((threadIdx.x & 31) == 0) {   // the lane that wrote the result
      uint8_t *const rec = g.out + (size_t)job.out * g.out_stride;
      reinterpret_cast<float2 *>(rec + g.off_sp0)[pi] = p0;
      reinterpret_cast<float2 *>(rec + g.off_sp1)[pi] = c.p1[warp];
      rec[g.off_sst + pi] = c.st[warp];
    }
  }
};

template <class Src>
__global__ void __launch_bounds__(kLkWarps * 32) k_lk_g(const __grid_constant__ Src src) {
  __shared__ typename Src::Cta c;
  __shared__ int s_n;
  if (threadIdx.x == 0) s_n = src.setup(c, blockIdx.x * kLkWarps);
  __syncthreads();
  const int pi = blockIdx.x * kLkWarps + (threadIdx.x >> 5);
  if (pi >= s_n) return;
  src.track(c, pi, [&](const LkArgs &a, const float2 *p0, float2 *p1, uint8_t *st, float2 *p0n, float2 *p1n, int i) {
    lk_body(a, p0, p1, st, p0n, p1n, i);
  });
}

// 5 resident CTAs per SM: 96 registers, no spills
template <class Src>
__global__ void __launch_bounds__(kLkWarps * 32, 5) k_lk15w_g(const __grid_constant__ Src src) {
  __shared__ typename Src::Cta c;
  __shared__ LkwSmem sm[kLkWarps];
  __shared__ int s_n;
  if (threadIdx.x == 0) s_n = src.setup(c, blockIdx.x * kLkWarps);
  __syncthreads();
  const int warp = threadIdx.x >> 5;
  const int pi = blockIdx.x * kLkWarps + warp;
  if (pi >= s_n) return;
  src.track(c, pi, [&](const LkArgs &a, const float2 *p0, float2 *p1, uint8_t *st, float2 *p0n, float2 *p1n, int i) {
    lk15w_body(a, p0, p1, st, p0n, p1n, i, sm[warp]);
  });
}

bool lk_w15_form(int win, int pyramid_images) { return win == kW15 && pyramid_images <= kLk15MaxLevels; }

// src's features, at most per_job of each of n_jobs jobs: the 15 x 15 body where lk_w15_form allows it, the generic body
// otherwise.  `images`: the pyramid images the source's LkArgs hold.
template <class Src>
static void launch_lk_warps(const Src &src, int win, int images, int per_job, int n_jobs, cudaStream_t s) {
  const dim3 grid((per_job + kLkWarps - 1) / kLkWarps, n_jobs);
  if (lk_w15_form(win, images)) {
    PLVIWO_CARVEOUT(k_lk15w_g<Src>);
    k_lk15w_g<Src><<<grid, kLkWarps * 32, 0, s>>>(src);
    return;
  }
  const size_t smem = (size_t)LkLayout(win).per_warp * kLkWarps;
  static SmemOptIn optin;
  optin.ensure(k_lk_g<Src>, smem);
  PLVIWO_CARVEOUT(k_lk_g<Src>);
  k_lk_g<Src><<<grid, kLkWarps * 32, smem, s>>>(src);
}

void launch_group_lk(const GroupDev &g, const TrackJob *jobs, int n_jobs, const LkParams &prm, cudaStream_t s) {
  if (n_jobs > 0) launch_lk_warps(GroupPoints{{g, jobs, prm}}, prm.win, prm.max_level + 1, g.pts_cap, n_jobs, s);
}

void launch_stereo_lr_lk(const GroupDev &g, const TrackJob *jobs, int n_rigs, const LkParams &prm, cudaStream_t s) {
  if (n_rigs > 0) launch_lk_warps(StereoLr{{g, jobs, prm}}, prm.win, prm.max_level + 1, g.pts_cap, n_rigs, s);
}

void launch_group_line_samples(const GroupDev &g, const TrackJob *jobs, int n_jobs, const LkParams &prm, cudaStream_t s) {
  if (n_jobs > 0 && g.sample_cap > 0) launch_lk_warps(LineSamples{{g, jobs, prm}}, prm.win, prm.max_level + 1, g.sample_cap, n_jobs, s);
}

bool launch_lk(const Pyramid &prev, const Pyramid &next, const float2 *d_pts0, float2 *d_pts1, uint8_t *d_status,
               float2 *d_p0n, float2 *d_p1n, int n, const LkParams &prm, cudaStream_t s, int *host_flag, int flag_value,
               unsigned *d_done_counter, const int *d_tab_cnt, int tab_stride, bool flow_is_zero, const unsigned *cell_mask) {
  if (n <= 0) return false;
  const int levels = std::min(prm.max_level + 1, prev.n);
  LkArgs a;
  lk_args(a, prev.lvl, next.lvl, levels, prm, prm.K, prm.D, prm.undistort, flow_is_zero ? 1 : 0, cell_mask);
  if (lk_w15_form(prm.win, levels)) {   // one CTA per feature, one warp per level
    PLVIWO_CARVEOUT(k_lk15);
    k_lk15<<<n, std::max(levels, kChainWarps) * 32, 0, s>>>(a, d_pts0, d_pts1, d_status, d_p0n, d_p1n, n, host_flag, flag_value, d_done_counter,
                                     d_tab_cnt, tab_stride);
    return host_flag != nullptr;
  }
  if (d_tab_cnt != nullptr || flow_is_zero) return false;   // table mode exists for the 15 x 15 kernel only (caller checks)
  launch_lk_warps(LkArrays{a, d_pts0, d_pts1, d_status, d_p0n, d_p1n, n}, prm.win, levels, n, 1, s);
  return false;
}

// k_lk15w_g on arbitrary points over one image pair: lets tests reach the border paths of the group kernel with points a
// tracker would not produce
bool launch_lk_warp(const Pyramid &prev, const Pyramid &next, const float2 *d_pts0, float2 *d_pts1, uint8_t *d_status, int n,
                    const LkParams &prm, cudaStream_t s) {
  const int levels = std::min(prm.max_level + 1, prev.n);
  if (!lk_w15_form(prm.win, levels) || prm.undistort) return false;
  if (n <= 0) return true;
  LkArgs a;
  lk_args(a, prev.lvl, next.lvl, levels, prm, prm.K, prm.D, 0, 0, nullptr);
  launch_lk_warps(LkArrays{a, d_pts0, d_pts1, d_status, nullptr, nullptr, n}, prm.win, levels, n, 1, s);
  return true;
}

}  // namespace plviwo
