// extern "C" surface declared in include/plviwo_fe.h.  Thin: argument checks, exception firewall, and the
// stand-alone kernel entry points used by the parity tests and micro-benchmarks.
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "fe_context.h"
#include "fe_stereo.h"
#include "fe_group.h"

using namespace plviwo;

struct FeHandle {
  FeContext *ctx;
};

struct FeStereoHandle {
  FeStereo *st;
};

struct FeGroupHandle {
  FeGroup *grp;
};

struct FeStereoGroupHandle {
  FeGroup *grp;
};

static thread_local std::string g_create_error;

// See bench.py / INTEGRATION.md: one hardware queue per stream.  Only effective if no CUDA context exists yet.
namespace {
struct EnvInit {
  EnvInit() { setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0); }
} g_env_init;
}  // namespace

#define API_BEGIN try {
#define API_END                                   \
  }                                               \
  catch (const std::bad_alloc &) {                \
    return FE_INTERNAL;                           \
  }                                               \
  catch (...) {                                   \
    return FE_INTERNAL;                           \
  }

// Creation errors: the reason goes to plviwo_*_last_error(NULL).
static int create_error(int code, const char *why) {
  g_create_error = why;
  return code;
}

// The config rules of every creator; tw x th is the size the tracker runs at (the handle's downsampled size, the raw size
// elsewhere).  nullptr when they hold, otherwise the reason.
static const char *check_config(const FeConfig &c, int tw, int th) {
  if (c.width < 64 || c.height < 64 || c.width > 4095 || c.height > 4095) return "image size must be in [64, 4095]";
  if (c.win_size < 3 || c.win_size > kMaxWin || (c.win_size & 1) == 0) return "win_size must be odd and in [3, 31]";
  if (c.pyr_levels < 0 || c.pyr_levels >= kMaxLevels) return "pyr_levels must be in [0, 7]";
  if (c.grid_x < 1 || c.grid_y < 1 || c.min_px_dist < 1 || c.num_features < 1) return "bad grid / distance / feature count";
  if (c.histogram_method != FE_HIST_NONE && c.histogram_method != FE_HIST_HISTOGRAM && c.histogram_method != FE_HIST_CLAHE)
    return "bad histogram_method";
  if (c.use_lines) {
    if ((tw & 1) || (th & 1)) return "line tracker needs even (tracking) image dimensions (exact 2x decimation)";
    if (c.canny_th1 != c.canny_th2) return "canny_th1 != canny_th2: hysteresis pass is not implemented";
    if (c.fld_length_threshold < 2) return "bad fld_length_threshold";
  }
  return nullptr;
}

// The camera model of a creator (FeCameraModel): nullptr when it is one the library implements, otherwise the reason.
static const char *check_model(int model) {
  if (model != FE_CAM_RADTAN && model != FE_CAM_EQUI) return "camera model must be FE_CAM_RADTAN (0) or FE_CAM_EQUI (1)";
  return nullptr;
}
static const char *model_name(int model) { return model == FE_CAM_EQUI ? "equidistant" : "radtan"; }
// set_camera's refusal of a model other than the one the object was created with (a CamBase keeps its class for life)
static std::string model_mismatch(int created) {
  return std::string("set_camera: created with the ") + model_name(created) +
         " model; the model is fixed at creation (use the _create_model functions to pick it)";
}

// After the config checks: the device a creator is asked for exists.
static int check_device(int device) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
    cudaGetLastError();
    return create_error(FE_NO_DEVICE, "no CUDA device: this front end has no CPU fallback");
  }
  if (device < 0 || device >= ndev) return create_error(FE_BAD_ARG, "device index out of range");
  return FE_OK;
}

static int copy_rows(const void *src, int n, size_t elem, void *out, int cap, int *n_out) {
  if (n_out) *n_out = n;
  if (!out) return FE_OK;
  if (cap < n) return FE_OVERFLOW;
  if (n) std::memcpy(out, src, (size_t)n * elem);
  return FE_OK;
}

extern "C" {

int plviwo_fe_abi_version(void) { return PLVIWO_FE_ABI_VERSION; }

void plviwo_fe_default_config(FeConfig *cfg) {
  if (!cfg) return;
  std::memset(cfg, 0, sizeof(*cfg));
  cfg->width = 1280;
  cfg->height = 560;
  cfg->num_features = 150;      // OptionsCamera.h:77-89
  cfg->fast_threshold = 20;
  cfg->grid_x = 5;
  cfg->grid_y = 5;
  cfg->min_px_dist = 10;
  cfg->pyr_levels = 5;          // TrackKLT.h:143
  cfg->win_size = 15;           // TrackKLT.h:144
  cfg->histogram_method = FE_HIST_HISTOGRAM;
  cfg->numaruco = 0;
  cfg->use_lines = 1;           // OptionsCamera.h:108
  cfg->fld_length_threshold = 20;
  cfg->fld_distance_threshold = 1.414213562f;
  cfg->canny_th1 = 50.f;
  cfg->canny_th2 = 50.f;
  cfg->line_min_length = 40.f;
  cfg->line_samples = 0;
  cfg->lookahead = 0;
  const double K[4] = {8.1690378992770002e+02, 8.1156803828490001e+02, 6.0850726281690004e+02, 2.6347599764440002e+02};
  const double D[4] = {-5.6143027800000002e-02, 1.3952563200000001e-01, -1.2155906999999999e-03, -9.7281389999999998e-04};
  for (int i = 0; i < 4; i++) {
    cfg->K[i] = K[i];
    cfg->D[i] = D[i];
  }
}

int plviwo_fe_device_count(int *n) {
  int c = 0;
  cudaError_t e = cudaGetDeviceCount(&c);
  if (n) *n = e == cudaSuccess ? c : 0;
  if (e != cudaSuccess) {
    cudaGetLastError();
    return FE_NO_DEVICE;
  }
  return c > 0 ? FE_OK : FE_NO_DEVICE;
}

int plviwo_fe_create(const FeConfig *cfg, int device, FeHandle **out) {
  return plviwo_fe_create_model(cfg, FE_CAM_RADTAN, device, out);
}

int plviwo_fe_create_model(const FeConfig *cfg, int model, int device, FeHandle **out) {
  API_BEGIN
  if (!cfg || !out) return FE_BAD_ARG;
  *out = nullptr;
  if (const char *why = check_model(model)) return create_error(FE_BAD_ARG, why);
  const int tw = cfg->downsample ? (int)(cfg->width / 2.0) : cfg->width, th = cfg->downsample ? (int)(cfg->height / 2.0) : cfg->height;
  if (cfg->downsample && (tw < 64 || th < 64)) return create_error(FE_BAD_ARG, "downsampled image would be smaller than 64 pixels");
  if (const char *why = check_config(*cfg, tw, th)) return create_error(FE_BAD_ARG, why);
  if (int rc = check_device(device)) return rc;
  FeContext *ctx = new FeContext(*cfg, device, model);
  int rc = ctx->init();
  if (rc != FE_OK) {
    g_create_error = ctx->last_error;
    delete ctx;
    return rc;
  }
  FeHandle *h = new FeHandle{ctx};
  *out = h;
  return FE_OK;
  API_END
}

int plviwo_fe_destroy(FeHandle *h) {
  API_BEGIN
  if (!h) return FE_BAD_ARG;
  delete h->ctx;
  delete h;
  return FE_OK;
  API_END
}

const char *plviwo_fe_last_error(const FeHandle *h) { return h ? h->ctx->last_error.c_str() : g_create_error.c_str(); }

int plviwo_fe_set_calib(FeHandle *h, const double K[4], const double D[4]) {
  if (!h || !K || !D) return FE_BAD_ARG;
  return h->ctx->set_calib(K, D);
}

int plviwo_fe_set_camera(FeHandle *h, int model, const double K[4], const double D[4]) {
  if (!h || !K || !D) return FE_BAD_ARG;
  if (model != h->ctx->model()) {
    h->ctx->last_error = model_mismatch(h->ctx->model());
    return FE_BAD_ARG;
  }
  return h->ctx->set_calib(K, D);
}

int plviwo_fe_get_currid(FeHandle *h, uint64_t *currid) {
  if (!h || !currid) return FE_BAD_ARG;
  *currid = h->ctx->currid();
  return FE_OK;
}

int plviwo_fe_set_currid(FeHandle *h, uint64_t currid) {
  if (!h) return FE_BAD_ARG;
  return h->ctx->set_currid(currid);
}
int plviwo_fe_set_num_features(FeHandle *h, int n) {
  if (!h || n < 1) return FE_BAD_ARG;
  return h->ctx->set_num_features(n);
}
int plviwo_fe_change_feat_id(FeHandle *h, uint64_t id_old, uint64_t id_new) {
  if (!h) return FE_BAD_ARG;
  return h->ctx->change_feat_id(id_old, id_new);
}

int plviwo_fe_feed(FeHandle *h, double timestamp, const uint8_t *image, int width, int height, int stride,
                   const uint8_t *mask, int mask_stride, const double vp[6], FeFrameInfo *info) {
  API_BEGIN
  if (!h) return FE_BAD_ARG;
  return h->ctx->feed(timestamp, image, width, height, stride, false, mask, mask_stride, vp, info);
  API_END
}
int plviwo_fe_feed_device(FeHandle *h, double timestamp, const void *d_image, int width, int height, int pitch,
                          const uint8_t *mask, int mask_stride, const double vp[6], FeFrameInfo *info) {
  API_BEGIN
  if (!h) return FE_BAD_ARG;
  return h->ctx->feed(timestamp, static_cast<const uint8_t *>(d_image), width, height, pitch, true, mask, mask_stride, vp, info);
  API_END
}
int plviwo_fe_submit(FeHandle *h, double timestamp, const uint8_t *image, int stride, int on_device, const uint8_t *mask,
                     int mask_stride, const double vp[6]) {
  API_BEGIN
  if (!h || !image || stride < h->ctx->cfg().width || (mask && mask_stride < h->ctx->cfg().width)) return FE_BAD_ARG;
  return h->ctx->submit(timestamp, image, stride, on_device != 0, mask, mask_stride, vp);
  API_END
}
int plviwo_fe_play(FeHandle *h, int n_frames, const uint8_t *const *images, int stride, int on_device, const double *timestamps,
                   const double *vps, FePlayStats *out) {
  API_BEGIN
  if (!h || n_frames < 0 || (n_frames > 0 && (!images || !timestamps)) || stride < h->ctx->cfg().width) return FE_BAD_ARG;
  return h->ctx->play(n_frames, images, stride, on_device != 0, timestamps, vps, out);
  API_END
}
int plviwo_fe_collect(FeHandle *h, FeFrameInfo *info) {
  API_BEGIN
  if (!h) return FE_BAD_ARG;
  return h->ctx->collect(info);
  API_END
}

}  // extern "C"
template <class T>
static int copy_out(const std::vector<T> &v, T *out, int cap, int *n_out) {
  if (n_out) *n_out = (int)v.size();
  if (!out) return FE_OK;
  if (cap < (int)v.size()) return FE_OVERFLOW;
  if (!v.empty()) std::memcpy(out, v.data(), v.size() * sizeof(T));
  return FE_OK;
}
extern "C" {

int plviwo_fe_get_point_rows(FeHandle *h, FePointRow *out, int cap, int *n_out) {
  if (!h) return FE_BAD_ARG;
  return copy_out(h->ctx->result().point_rows, out, cap, n_out);
}
int plviwo_fe_get_last_obs(FeHandle *h, uint64_t *ids, float *uv, int cap, int *n_out) {
  if (!h) return FE_BAD_ARG;
  const auto &p = h->ctx->result().obs;
  const auto &id = h->ctx->result().obs_ids;
  if (n_out) *n_out = (int)p.size();
  if (!ids && !uv) return FE_OK;
  if (cap < (int)p.size()) return FE_OVERFLOW;
  for (size_t i = 0; i < p.size(); i++) {
    if (ids) ids[i] = id[i];
    if (uv) {
      uv[2 * i] = p[i].x;
      uv[2 * i + 1] = p[i].y;
    }
  }
  return FE_OK;
}
int plviwo_fe_get_line_rows(FeHandle *h, FeLineRow *out, int cap, int *n_out) {
  if (!h) return FE_BAD_ARG;
  return copy_out(h->ctx->result().line_rows, out, cap, n_out);
}
int plviwo_fe_get_line_points(FeHandle *h, FeLinePoint *out, int cap, int *n_out) {
  if (!h) return FE_BAD_ARG;
  return copy_out(h->ctx->result().line_points, out, cap, n_out);
}
int plviwo_fe_classify_lines(FeHandle *h, const double vp[6]) {
  if (!h || !vp) return FE_BAD_ARG;
  return h->ctx->classify_lines(vp);
}
int plviwo_fe_get_line_samples(FeHandle *h, float *uv01, uint8_t *status, int cap, int *n_out) {
  if (!h) return FE_BAD_ARG;
  const auto &s = h->ctx->result().sample_status;
  if (n_out) *n_out = (int)s.size();
  if (!uv01 && !status) return FE_OK;
  if (cap < (int)s.size()) return FE_OVERFLOW;
  if (uv01 && !s.empty()) std::memcpy(uv01, h->ctx->result().sample_uv.data(), s.size() * 4 * sizeof(float));
  if (status && !s.empty()) std::memcpy(status, s.data(), s.size());
  return FE_OK;
}

int plviwo_fe_get_state(FeHandle *h, void *buf, size_t cap, size_t *n_bytes) {
  API_BEGIN
  if (!h) return FE_BAD_ARG;
  return h->ctx->get_state(buf, cap, n_bytes);
  API_END
}
int plviwo_fe_set_state(FeHandle *h, const void *buf, size_t n_bytes) {
  API_BEGIN
  if (!h) return FE_BAD_ARG;
  return h->ctx->set_state(buf, n_bytes);
  API_END
}
int plviwo_fe_tap(FeHandle *h, int what, void *buf, size_t cap, size_t *n_bytes) {
  API_BEGIN
  if (!h) return FE_BAD_ARG;
  return h->ctx->tap(what, buf, cap, n_bytes);
  API_END
}
int plviwo_fe_enable_timing(FeHandle *h, int on) {
  if (!h) return FE_BAD_ARG;
  h->ctx->timing = on != 0;
  return FE_OK;
}
int plviwo_fe_enable_taps(FeHandle *h, int on) {
  if (!h) return FE_BAD_ARG;
  h->ctx->taps = on != 0;
  return FE_OK;
}
int plviwo_fe_get_stage_times(FeHandle *h, FeStageTimes *out, int reset) {
  if (!h || !out) return FE_BAD_ARG;
  *out = h->ctx->snapshot_times();
  if (reset) h->ctx->reset_times();
  return FE_OK;
}

// --------------------------------------------------------------------------------- stand-alone kernels
#define OP_CUDA(call)                              \
  do {                                             \
    cudaError_t e__ = (call);                      \
    if (e__ != cudaSuccess) {                      \
      g_create_error = std::string(#call) + ": " + cudaGetErrorString(e__); \
      return e__ == cudaErrorNoDevice || e__ == cudaErrorInsufficientDriver ? FE_NO_DEVICE : FE_CUDA_ERROR; \
    }                                              \
  } while (0)

}  // extern "C"
namespace {
struct TmpImage {
  DevImage im;
  ~TmpImage() { cudaFree(im.p); }
  int alloc(int w, int h) {
    im.w = w;
    im.h = h;
    im.pitch = (w + 255) / 256 * 256;
    return cudaMalloc(&im.p, (size_t)im.pitch * h + 256) == cudaSuccess ? 0 : 1;
  }
  int upload(const uint8_t *src) {
    return cudaMemcpy2D(im.p, im.pitch, src, im.w, im.w, im.h, cudaMemcpyHostToDevice) == cudaSuccess ? 0 : 1;
  }
};
struct TmpPyr {
  Pyramid pyr;
  ~TmpPyr() {
    for (int l = 0; l < pyr.n; l++) cudaFree(pyr.lvl[l].p);
  }
  int alloc(int w, int h, int levels, int win) {
    pyr.n = 0;
    for (int l = 0; l <= levels && l < kMaxLevels; l++) {
      DevImage &im = pyr.lvl[l];
      im.w = w;
      im.h = h;
      im.pitch = (w + 255) / 256 * 256;
      if (cudaMalloc(&im.p, (size_t)im.pitch * h + 256) != cudaSuccess) return 1;
      pyr.n = l + 1;
      w = (w + 1) / 2;
      h = (h + 1) / 2;
      if (win > 0 && (w <= win || h <= win)) break;
      if (w < 2 || h < 2) break;
    }
    return 0;
  }
};
template <class T>
struct DevBuf {
  T *p = nullptr;
  ~DevBuf() { cudaFree(p); }
  int alloc(size_t n) { return cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T)) == cudaSuccess ? 0 : 1; }
};
int build_pyramid(const uint8_t *img, int w, int h, int levels, int win, int equalize, TmpImage &raw, TmpPyr &pyr,
                  TmpImage *half) {
  if (raw.alloc(w, h) || raw.upload(img) || pyr.alloc(w, h, levels, win)) return 1;
  DevBuf<unsigned> hist, counters;
  DevBuf<uint8_t> lut;
  if (hist.alloc(256) || counters.alloc(4) || lut.alloc(256)) return 1;
  cudaMemset(hist.p, 0, 256 * sizeof(unsigned));
  cudaMemset(counters.p, 0, 4 * sizeof(unsigned));
  if (equalize) launch_hist(raw.im, hist.p, counters.p, lut.p, 0);
  DevImage l1 = pyr.pyr.n > 1 ? pyr.pyr.lvl[1] : DevImage();
  launch_eq_pyr1(raw.im, lut.p, equalize, pyr.pyr.lvl[0], l1, half ? half->im : DevImage(), 0);
  launch_pyr_rest(pyr.pyr, counters.p + 1, 0);
  return cudaDeviceSynchronize() == cudaSuccess ? 0 : 1;
}
}  // namespace
extern "C" {

int plviwo_op_clahe(int device, const uint8_t *img, int w, int h, uint8_t *out) {
  API_BEGIN
  if (!img || !out || w < 8 || h < 8) return FE_BAD_ARG;
  OP_CUDA(cudaSetDevice(device));
  TmpImage raw, l0;
  DevBuf<uint8_t> luts;
  if (raw.alloc(w, h) || raw.upload(img) || l0.alloc(w, h) || luts.alloc(64 * 256)) return FE_CUDA_ERROR;
  launch_clahe_lut(raw.im, luts.p, 0);
  launch_eq_pyr1(raw.im, nullptr, 2, l0.im, DevImage(), DevImage(), 0, luts.p);
  OP_CUDA(cudaDeviceSynchronize());
  OP_CUDA(cudaMemcpy2D(out, w, l0.im.p, l0.im.pitch, w, h, cudaMemcpyDeviceToHost));
  return FE_OK;
  API_END
}

int plviwo_op_equalize_pyramid(int device, const uint8_t *img, int w, int h, int levels, uint8_t *out_levels, uint8_t *out_half) {
  API_BEGIN
  if (!img || !out_levels || w < 8 || h < 8 || levels < 1 || levels >= kMaxLevels) return FE_BAD_ARG;
  OP_CUDA(cudaSetDevice(device));
  TmpImage raw, half;
  TmpPyr pyr;
  if (out_half && half.alloc(w / 2, h / 2)) return FE_CUDA_ERROR;
  if (build_pyramid(img, w, h, levels, 0, 1, raw, pyr, out_half ? &half : nullptr)) {
    g_create_error = cudaGetErrorString(cudaGetLastError());
    return FE_CUDA_ERROR;
  }
  uint8_t *o = out_levels;
  for (int l = 0; l < pyr.pyr.n; l++) {
    const DevImage &im = pyr.pyr.lvl[l];
    OP_CUDA(cudaMemcpy2D(o, im.w, im.p, im.pitch, im.w, im.h, cudaMemcpyDeviceToHost));
    o += (size_t)im.w * im.h;
  }
  if (out_half) OP_CUDA(cudaMemcpy2D(out_half, half.im.w, half.im.p, half.im.pitch, half.im.w, half.im.h, cudaMemcpyDeviceToHost));
  return FE_OK;
  API_END
}

int plviwo_op_fast_cell(int device, const uint8_t *img, int w, int h, int threshold, int32_t *xys, int cap, int *n_out) {
  API_BEGIN
  if (!img || !n_out || w < 7 || h < 7 || w > 4095 || h > 4095) return FE_BAD_ARG;
  OP_CUDA(cudaSetDevice(device));
  TmpImage raw;
  if (raw.alloc(w, h) || raw.upload(img)) return FE_CUDA_ERROR;
  const int nb = (h + kFastBandRows - 1) / kFastBandRows;
  const int kcap = w * h / 4 + 1024;
  DevBuf<FastCell> cells;
  DevBuf<unsigned> total, kps;
  DevBuf<int> off, cnt;
  if (cells.alloc(1) || total.alloc(1) || kps.alloc(kcap) || off.alloc(nb) || cnt.alloc(nb)) return FE_CUDA_ERROR;
  FastCell c{0, 0, w, h};
  OP_CUDA(cudaMemcpy(cells.p, &c, sizeof(c), cudaMemcpyHostToDevice));
  OP_CUDA(cudaMemset(total.p, 0, sizeof(unsigned)));
  launch_fast(raw.im, cells.p, 1, nb, w, threshold, total.p, off.p, cnt.p, kps.p, kcap, 0);
  OP_CUDA(cudaDeviceSynchronize());
  std::vector<int> hoff(nb), hcnt(nb);
  unsigned htotal = 0;
  OP_CUDA(cudaMemcpy(&htotal, total.p, sizeof(unsigned), cudaMemcpyDeviceToHost));
  OP_CUDA(cudaMemcpy(hoff.data(), off.p, nb * sizeof(int), cudaMemcpyDeviceToHost));
  OP_CUDA(cudaMemcpy(hcnt.data(), cnt.p, nb * sizeof(int), cudaMemcpyDeviceToHost));
  std::vector<unsigned> hk(std::min<unsigned>(htotal, kcap));
  if (!hk.empty()) OP_CUDA(cudaMemcpy(hk.data(), kps.p, hk.size() * sizeof(unsigned), cudaMemcpyDeviceToHost));
  int n = 0;
  for (int b = 0; b < nb; b++)
    for (int k = 0; k < hcnt[b]; k++, n++) {
      if (xys && n < cap) {
        unsigned v = hk[hoff[b] + k];
        xys[3 * n] = v & 0xfff;
        xys[3 * n + 1] = (v >> 12) & 0xfff;
        xys[3 * n + 2] = v >> 24;
      }
    }
  *n_out = n;
  return (xys && n > cap) ? FE_OVERFLOW : FE_OK;
  API_END
}

int plviwo_op_sort_corners(int device, const uint32_t *packed, int n, int nfg, uint32_t *sorted, float *cand, int *n_cand) {
  API_BEGIN
  if (!packed || n < 0 || nfg < 1) return FE_BAD_ARG;
  if (device < 0) {   // host instantiation of introsort.h
    if (!sorted) return FE_BAD_ARG;
    std::memcpy(sorted, packed, (size_t)n * sizeof(uint32_t));
    host_sort_corners(sorted, n);
    if (n_cand) *n_cand = std::min(n, nfg);
    if (cand) {   // the pruned form the selection kernel runs (isort::sort_prefix): x, y of its first nfg elements
      std::vector<uint32_t> tmp(packed, packed + n);
      host_sort_corners(tmp.data(), n, nfg);
      for (int i = 0; i < std::min(n, nfg); i++) {
        cand[2 * i] = (float)(tmp[i] & 0xfffu);
        cand[2 * i + 1] = (float)((tmp[i] >> 12) & 0xfffu);
      }
    }
    return FE_OK;
  }
  if (!cand || !n_cand) return FE_BAD_ARG;
  OP_CUDA(cudaSetDevice(device));
  DevBuf<FastCell> cells;
  DevBuf<unsigned> total, kps, scratch;
  DevBuf<int> off, cnt, ccnt;
  DevBuf<float2> csel;
  if (cells.alloc(1) || total.alloc(2) || kps.alloc(n) || scratch.alloc(n) || off.alloc(1) || cnt.alloc(1) || ccnt.alloc(1) ||
      csel.alloc(nfg))
    return FE_CUDA_ERROR;
  FastCell c{0, 0, 4095, 4095};
  const unsigned tot[2] = {(unsigned)n, 0u};
  const int zero = 0;
  OP_CUDA(cudaMemcpy(cells.p, &c, sizeof(c), cudaMemcpyHostToDevice));
  OP_CUDA(cudaMemcpy(total.p, tot, sizeof(tot), cudaMemcpyHostToDevice));
  OP_CUDA(cudaMemcpy(off.p, &zero, sizeof(int), cudaMemcpyHostToDevice));
  OP_CUDA(cudaMemcpy(cnt.p, &n, sizeof(int), cudaMemcpyHostToDevice));
  if (n) OP_CUDA(cudaMemcpy(kps.p, packed, (size_t)n * sizeof(uint32_t), cudaMemcpyHostToDevice));
  launch_fast_select(cells.p, 1, 1, total.p, off.p, cnt.p, kps.p, std::max(n, 1), scratch.p, nfg, csel.p, ccnt.p, 0);
  OP_CUDA(cudaDeviceSynchronize());
  OP_CUDA(cudaMemcpy(n_cand, ccnt.p, sizeof(int), cudaMemcpyDeviceToHost));
  if (*n_cand > 0) OP_CUDA(cudaMemcpy(cand, csel.p, (size_t)*n_cand * sizeof(float2), cudaMemcpyDeviceToHost));
  return FE_OK;
  API_END
}

int plviwo_op_corner_subpix(int device, const uint8_t *img, int w, int h, float *pts, int n) {
  API_BEGIN
  if (!img || !pts || n < 0) return FE_BAD_ARG;
  OP_CUDA(cudaSetDevice(device));
  TmpImage raw;
  DevBuf<float2> d;
  if (raw.alloc(w, h) || raw.upload(img) || d.alloc(n)) return FE_CUDA_ERROR;
  OP_CUDA(cudaMemcpy(d.p, pts, (size_t)n * sizeof(float2), cudaMemcpyHostToDevice));
  launch_corner_subpix(raw.im, d.p, d.p, n, 0);
  OP_CUDA(cudaDeviceSynchronize());
  OP_CUDA(cudaMemcpy(pts, d.p, (size_t)n * sizeof(float2), cudaMemcpyDeviceToHost));
  return FE_OK;
  API_END
}

static int op_lk(int device, const uint8_t *img0, const uint8_t *img1, int w, int h, int win, int max_level, const float *pts0,
                 float *pts1, uint8_t *status, int n, bool warp) {
  API_BEGIN
  if (!img0 || !img1 || !pts0 || !pts1 || !status || n < 0 || win < 3 || win > kMaxWin || !(win & 1) || max_level < 0 ||
      max_level >= kMaxLevels)
    return FE_BAD_ARG;
  OP_CUDA(cudaSetDevice(device));
  TmpImage r0, r1;
  TmpPyr p0, p1;
  if (build_pyramid(img0, w, h, max_level, win, 0, r0, p0, nullptr) || build_pyramid(img1, w, h, max_level, win, 0, r1, p1, nullptr)) {
    g_create_error = cudaGetErrorString(cudaGetLastError());
    return FE_CUDA_ERROR;
  }
  DevBuf<float2> d0, d1, dn0, dn1;
  DevBuf<uint8_t> ds;
  if (d0.alloc(n) || d1.alloc(n) || dn0.alloc(n) || dn1.alloc(n) || ds.alloc(n)) return FE_CUDA_ERROR;
  OP_CUDA(cudaMemcpy(d0.p, pts0, (size_t)n * sizeof(float2), cudaMemcpyHostToDevice));
  OP_CUDA(cudaMemcpy(d1.p, pts1, (size_t)n * sizeof(float2), cudaMemcpyHostToDevice));
  const LkParams prm = lk_params(win, max_level, nullptr, nullptr, false);
  if (!warp) launch_lk(p0.pyr, p1.pyr, d0.p, d1.p, ds.p, dn0.p, dn1.p, n, prm, 0);
  else if (!launch_lk_warp(p0.pyr, p1.pyr, d0.p, d1.p, ds.p, n, prm, 0)) return FE_BAD_ARG;
  OP_CUDA(cudaDeviceSynchronize());
  OP_CUDA(cudaMemcpy(pts1, d1.p, (size_t)n * sizeof(float2), cudaMemcpyDeviceToHost));
  OP_CUDA(cudaMemcpy(status, ds.p, (size_t)n, cudaMemcpyDeviceToHost));
  return FE_OK;
  API_END
}

int plviwo_op_lk(int device, const uint8_t *img0, const uint8_t *img1, int w, int h, int win, int max_level,
                 const float *pts0, float *pts1, uint8_t *status, int n) {
  return op_lk(device, img0, img1, w, h, win, max_level, pts0, pts1, status, n, false);
}

int plviwo_op_lk_warp(int device, const uint8_t *img0, const uint8_t *img1, int w, int h, int win, int max_level,
                      const float *pts0, float *pts1, uint8_t *status, int n) {
  return op_lk(device, img0, img1, w, h, win, max_level, pts0, pts1, status, n, true);
}

int plviwo_op_undistort(int device, const float *pts, int n, const double K[4], const double D[4], float *out) {
  API_BEGIN
  if (!pts || !out || !K || !D || n < 0) return FE_BAD_ARG;
  OP_CUDA(cudaSetDevice(device));
  DevBuf<float2> a, b;
  if (a.alloc(n) || b.alloc(n)) return FE_CUDA_ERROR;
  OP_CUDA(cudaMemcpy(a.p, pts, (size_t)n * sizeof(float2), cudaMemcpyHostToDevice));
  launch_undistort(a.p, b.p, n, FE_CAM_RADTAN, K, D, 0);
  OP_CUDA(cudaDeviceSynchronize());
  OP_CUDA(cudaMemcpy(out, b.p, (size_t)n * sizeof(float2), cudaMemcpyDeviceToHost));
  return FE_OK;
  API_END
}

int plviwo_op_undistort_equi(int device, const float *pts, int n, const double K[4], const double D[4], float *out) {
  API_BEGIN
  if (!pts || !out || !K || !D || n < 0) return FE_BAD_ARG;
  if (device < 0) {   // host instantiation of tracker_core.h's undistort_equi
    for (int i = 0; i < n; i++) {
      const float2 r = undistort_equi(make_float2(pts[2 * i], pts[2 * i + 1]), K, D);
      out[2 * i] = r.x;
      out[2 * i + 1] = r.y;
    }
    return FE_OK;
  }
  OP_CUDA(cudaSetDevice(device));
  DevBuf<float2> a, b;
  if (a.alloc(n) || b.alloc(n)) return FE_CUDA_ERROR;
  OP_CUDA(cudaMemcpy(a.p, pts, (size_t)n * sizeof(float2), cudaMemcpyHostToDevice));
  launch_undistort(a.p, b.p, n, FE_CAM_EQUI, K, D, 0);
  OP_CUDA(cudaDeviceSynchronize());
  OP_CUDA(cudaMemcpy(out, b.p, (size_t)n * sizeof(float2), cudaMemcpyDeviceToHost));
  return FE_OK;
  API_END
}

namespace {
struct TmpFld {
  FldBuffers fb;
  ~TmpFld() { fb.release(); }
  int alloc(int w, int h, int T, int out_cap) { return fb.alloc(w, h, T, out_cap); }
};
}  // namespace

int plviwo_op_canny_half(int device, const uint8_t *img, int w, int h, float th, uint8_t *edges) {
  API_BEGIN
  if (!img || !edges || w < 8 || h < 8) return FE_BAD_ARG;
  OP_CUDA(cudaSetDevice(device));
  TmpImage raw;
  TmpFld f;
  DevBuf<uint8_t> out;
  if (raw.alloc(w, h) || raw.upload(img) || f.alloc(w, h, 20, 16) || out.alloc((size_t)w * h)) return FE_CUDA_ERROR;
  launch_canny(raw.im, th, th, f.fb, 0);
  launch_unpack_edges(f.fb, w, h, out.p, 0);
  OP_CUDA(cudaDeviceSynchronize());
  OP_CUDA(cudaMemcpy(edges, out.p, (size_t)w * h, cudaMemcpyDeviceToHost));
  return FE_OK;
  API_END
}

int plviwo_op_ccl_tiles(int device, const uint32_t *edge_words, int w, int h, int32_t *label, int32_t *cnt, int32_t *bbox,
                        int32_t *roots, int cap, int *n_roots) {
  API_BEGIN
  if (!edge_words || !label || !cnt || !bbox || !n_roots || (cap > 0 && !roots) || cap < 0 || w < 1 || h < 1 ||
      (size_t)w * h > (size_t)1 << 28)
    return FE_BAD_ARG;
  OP_CUDA(cudaSetDevice(device));
  TmpFld f;
  if (f.alloc(w, h, 20, 16)) return FE_CUDA_ERROR;
  const size_t n = (size_t)w * h;
  OP_CUDA(cudaMemcpy(f.fb.edges, edge_words, (size_t)f.fb.words_per_row * h * sizeof(unsigned), cudaMemcpyHostToDevice));
  OP_CUDA(cudaMemset(f.fb.label, 0xff, n * sizeof(int)));
  launch_ccl_tiles(f.fb, w, h, 0);
  OP_CUDA(cudaDeviceSynchronize());
  int nr = 0;
  OP_CUDA(cudaMemcpy(&nr, f.fb.lroot_n, sizeof(int), cudaMemcpyDeviceToHost));
  OP_CUDA(cudaMemcpy(label, f.fb.label, n * sizeof(int), cudaMemcpyDeviceToHost));
  OP_CUDA(cudaMemcpy(cnt, f.fb.cnt, n * sizeof(int), cudaMemcpyDeviceToHost));
  OP_CUDA(cudaMemcpy(bbox, f.fb.bbox, 3 * n * sizeof(int), cudaMemcpyDeviceToHost));
  *n_roots = nr;
  if (nr > cap) return FE_OVERFLOW;
  if (nr) OP_CUDA(cudaMemcpy(roots, f.fb.lroots, (size_t)nr * sizeof(int), cudaMemcpyDeviceToHost));
  return FE_OK;
  API_END
}

int plviwo_op_fld(int device, const uint8_t *img, int w, int h, int length_threshold, float distance_threshold,
                  float canny_th, float *lines, int cap, int *n_out) {
  API_BEGIN
  if (!img || !n_out || w < 16 || h < 16 || length_threshold < 2) return FE_BAD_ARG;
  OP_CUDA(cudaSetDevice(device));
  TmpImage raw;
  TmpFld f;
  const int out_cap = 8192;
  if (raw.alloc(w, h) || raw.upload(img) || f.alloc(w, h, length_threshold, out_cap)) return FE_CUDA_ERROR;
  launch_canny(raw.im, canny_th, canny_th, f.fb, 0);
  launch_fld(raw.im, length_threshold, distance_threshold, f.fb, 0);
  OP_CUDA(cudaDeviceSynchronize());
  int counts[2] = {0, 0};
  OP_CUDA(cudaMemcpy(counts, f.fb.counters + 3, sizeof(counts), cudaMemcpyDeviceToHost));
  int n = std::min(counts[1], out_cap);
  *n_out = n;
  if (lines) {
    if (n > cap) return FE_OVERFLOW;
    if (n) OP_CUDA(cudaMemcpy(lines, f.fb.out, (size_t)n * sizeof(float4), cudaMemcpyDeviceToHost));
  }
  return FE_OK;
  API_END
}

int plviwo_op_image_kernels_time(int device, int w, int h, int iters, float ms[4]) {
  API_BEGIN
  if (!ms || w < 64 || h < 64 || (w & 3) || (h & 3) || iters < 1) return FE_BAD_ARG;
  OP_CUDA(cudaSetDevice(device));
  TmpImage raw, l0, l1, half;
  DevBuf<unsigned> hist, counters, total, kps;
  DevBuf<uint8_t> eq_lut;
  DevBuf<int> off, cnt;
  DevBuf<FastCell> cells;
  TmpFld f;
  const int cw = 256, ch = 112;                       // the 5 x 5 grid cell of a 1280 x 560 frame
  const int gx = w / cw, gy = h / ch, ncell = gx * gy;
  const int nb = (ch + kFastBandRows - 1) / kFastBandRows;
  const int kcap = 1 << 22;
  if (raw.alloc(w, h) || l0.alloc(w, h) || l1.alloc((w + 1) / 2, (h + 1) / 2) || half.alloc(w / 2, h / 2) || hist.alloc(256) ||
      counters.alloc(4) || eq_lut.alloc(256) || total.alloc(2) || kps.alloc(kcap) || off.alloc((size_t)ncell * nb) || cnt.alloc((size_t)ncell * nb) ||
      cells.alloc(std::max(ncell, 1)) || f.alloc(w / 2, h / 2, 20, 16))
    return FE_CUDA_ERROR;
  {  // synthetic texture: smooth ramps + hash noise (uploaded once)
    std::vector<uint8_t> row((size_t)w);
    std::vector<uint8_t> img((size_t)w * h);
    for (int y = 0; y < h; y++)
      for (int x = 0; x < w; x++) {
        unsigned v = (unsigned)(x * 2654435761u) ^ (unsigned)(y * 40503u);
        v ^= v >> 13; v *= 0x5bd1e995u; v ^= v >> 15;
        img[(size_t)y * w + x] = (uint8_t)(40 + ((x / 7 + y / 5) & 63) + (v & 63));
      }
    if (raw.upload(img.data())) return FE_CUDA_ERROR;
  }
  std::vector<FastCell> hc;
  for (int x = 0; x < gx; x++)
    for (int y = 0; y < gy; y++) hc.push_back(FastCell{x * cw, y * ch, cw, ch});
  if (ncell) OP_CUDA(cudaMemcpy(cells.p, hc.data(), hc.size() * sizeof(FastCell), cudaMemcpyHostToDevice));
  OP_CUDA(cudaMemset(hist.p, 0, 256 * sizeof(unsigned)));
  OP_CUDA(cudaMemset(counters.p, 0, 4 * sizeof(unsigned)));
  cudaEvent_t e0, e1;
  OP_CUDA(cudaEventCreate(&e0));
  OP_CUDA(cudaEventCreate(&e1));
  auto time_it = [&](int which) -> float {
    float tot = 0;
    for (int it = 0; it < iters + 3; it++) {
      if (which == 0) cudaMemsetAsync(hist.p, 0, 256 * sizeof(unsigned), 0);
      if (which == 2) cudaMemsetAsync(total.p, 0, 2 * sizeof(unsigned), 0);
      cudaEventRecord(e0, 0);
      if (which == 0) launch_hist(raw.im, hist.p, counters.p, eq_lut.p, 0);
      if (which == 1) launch_eq_pyr1(raw.im, eq_lut.p, 0, l0.im, l1.im, half.im, 0);
      if (which == 2) launch_fast(l0.im, cells.p, ncell, nb, cw, 20, total.p, off.p, cnt.p, kps.p, kcap, 0);
      if (which == 3) launch_canny(half.im, 50.f, 50.f, f.fb, 0);
      cudaEventRecord(e1, 0);
      cudaEventSynchronize(e1);
      float t = 0;
      cudaEventElapsedTime(&t, e0, e1);
      if (it >= 3) tot += t;
    }
    return tot / iters;
  };
  for (int k = 0; k < 4; k++) ms[k] = time_it(k);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  OP_CUDA(cudaDeviceSynchronize());
  return FE_OK;
  API_END
}

int plviwo_op_ransac_fundamental(const float *p0n, const float *p1n, int n, double threshold, double confidence,
                                 uint8_t *mask, int *n_inliers) {
  API_BEGIN
  if (!p0n || !p1n || !mask || n < 0) return FE_BAD_ARG;
  int valid = 0;
  int good = ransac_fundamental(p0n, p1n, n, threshold, confidence, mask, &valid);
  if (n_inliers) *n_inliers = valid ? good : -1;
  return FE_OK;
  API_END
}

// TrackLSD::AssignPointToLines (host-side step; tests).  kept[i] = 1 if line i keeps at least one point; the points of
// the kept lines follow in CSR form in (line, ascending point id) order: off[k] .. off[k + 1] for the k-th kept line.
int plviwo_op_assign_points(int n_lines, const float *lines, int n_pts, const float *pts, const uint64_t *pids, int32_t *kept,
                            int32_t *off, int32_t *pid_out, float *dist_out, int cap, int *n_out) {
  API_BEGIN
  if (n_lines < 0 || n_pts < 0 || !kept || !off || !n_out || (n_lines && !lines) || (n_pts && (!pts || !pids))) return FE_BAD_ARG;
  std::vector<float4> ln((size_t)n_lines);
  std::vector<uint64_t> ids((size_t)n_lines);
  for (int i = 0; i < n_lines; i++) {
    ln[(size_t)i] = make_float4(lines[4 * i], lines[4 * i + 1], lines[4 * i + 2], lines[4 * i + 3]);
    ids[(size_t)i] = (uint64_t)i;
  }
  std::vector<Pt> p((size_t)n_pts);
  std::vector<uint64_t> pid(pids, pids + n_pts);
  for (int j = 0; j < n_pts; j++) p[(size_t)j] = Pt{pts[2 * j], pts[2 * j + 1]};
  std::vector<std::map<int, double>> pol;
  std::vector<std::vector<Pt>> positions;
  std::vector<float4> fl;
  std::vector<uint64_t> fid;
  std::vector<float> sx, sy;
  std::vector<uint8_t> pass;
  assign_points_to_lines_host(ln, ids, p, pid, pol, positions, fl, fid, sx, sy, pass);
  for (int i = 0; i < n_lines; i++) kept[i] = 0;
  int n = 0;
  off[0] = 0;
  for (size_t k = 0; k < pol.size(); k++) {
    kept[fid[k]] = 1;
    for (auto &kv : pol[k]) {
      if (n < cap && pid_out && dist_out) {
        pid_out[n] = kv.first;
        dist_out[n] = (float)kv.second;
      }
      n++;
    }
    off[k + 1] = n;
  }
  *n_out = n;
  return n > cap ? FE_OVERFLOW : FE_OK;
  API_END
}

// TrackLSD::LineMatch on CSR inputs (host-side step; tests)
int plviwo_op_line_match(int n_last, const int32_t *last_off, const int32_t *last_pids, const float *last_lines, int n_new,
                         const int32_t *new_off, const int32_t *new_pids, const float *new_lines, int32_t *match_out) {
  API_BEGIN
  if (n_last < 0 || n_new < 0 || !match_out || (n_last && (!last_off || !last_lines)) || (n_new && (!new_off || !new_lines)))
    return FE_BAD_ARG;
  std::vector<std::map<int, double>> pl((size_t)n_last), pn((size_t)n_new);
  std::vector<float4> ll((size_t)n_last), ln((size_t)n_new);
  for (int j = 0; j < n_last; j++) {
    for (int k = last_off[j]; k < last_off[j + 1]; k++) pl[(size_t)j][last_pids[k]] = 0.0;
    ll[(size_t)j] = make_float4(last_lines[4 * j], last_lines[4 * j + 1], last_lines[4 * j + 2], last_lines[4 * j + 3]);
  }
  for (int i = 0; i < n_new; i++) {
    for (int k = new_off[i]; k < new_off[i + 1]; k++) pn[(size_t)i][new_pids[k]] = 0.0;
    ln[(size_t)i] = make_float4(new_lines[4 * i], new_lines[4 * i + 1], new_lines[4 * i + 2], new_lines[4 * i + 3]);
  }
  std::map<int, int> matches;
  std::vector<std::pair<int, int>> inv;
  std::vector<int> shared, touched;
  line_match_host(pl, pn, ln, ll, matches, inv, shared, touched);
  for (int i = 0; i < n_new; i++) match_out[i] = -1;
  for (auto &m : matches) match_out[m.first] = m.second;
  return FE_OK;
  API_END
}

// ---- stream group (many camera streams of one device, csrc/fe_group.h) ---------------------------------------------
int plviwo_fe_group_create(const FeConfig *cfg, int n_streams, int device, FeGroupHandle **out) {
  return plviwo_fe_group_create_model(cfg, n_streams, FE_CAM_RADTAN, device, out);
}

int plviwo_fe_group_create_model(const FeConfig *cfg, int n_streams, int model, int device, FeGroupHandle **out) {
  API_BEGIN
  if (!cfg || !out) return FE_BAD_ARG;
  *out = nullptr;
  if (const char *why = check_model(model)) return create_error(FE_BAD_ARG, why);
  if (n_streams < 1 || n_streams > 4096) return create_error(FE_BAD_ARG, "n_streams must be in [1, 4096]");
  if (cfg->downsample) return create_error(FE_BAD_ARG, "cfg.downsample is not supported in a stream group");
  if (const char *why = check_config(*cfg, cfg->width, cfg->height)) return create_error(FE_BAD_ARG, why);
  if (cfg->grid_x * cfg->grid_y > 256) return create_error(FE_BAD_ARG, "a stream group supports at most 256 grid cells");
  if (int rc = check_device(device)) return rc;
  FeGroup *grp = new FeGroup(*cfg, n_streams, device, false, model);
  int rc = grp->init();
  if (rc != FE_OK) {
    g_create_error = grp->last_error;
    delete grp;
    return rc;
  }
  *out = new FeGroupHandle{grp};
  return FE_OK;
  API_END
}

int plviwo_fe_group_destroy(FeGroupHandle *g) {
  API_BEGIN
  if (!g) return FE_BAD_ARG;
  delete g->grp;
  delete g;
  return FE_OK;
  API_END
}

const char *plviwo_fe_group_last_error(const FeGroupHandle *g) { return g ? g->grp->last_error.c_str() : g_create_error.c_str(); }

int plviwo_fe_group_set_calib(FeGroupHandle *g, int stream, const double K[4], const double D[4]) {
  if (!g) return FE_BAD_ARG;
  return g->grp->set_calib(stream, K, D);
}

int plviwo_fe_group_set_camera(FeGroupHandle *g, int stream, int model, const double K[4], const double D[4]) {
  if (!g) return FE_BAD_ARG;
  if (model != g->grp->model()) {   // as plviwo_fe_set_camera
    g->grp->last_error = model_mismatch(g->grp->model());
    return FE_BAD_ARG;
  }
  return g->grp->set_calib(stream, K, D);
}

int plviwo_fe_group_submit(FeGroupHandle *g, const double *timestamps, const uint8_t *const *images, int stride, int on_device,
                           const uint8_t *const *masks, int mask_stride, const double *vps) {
  API_BEGIN
  if (!g) return FE_BAD_ARG;
  return g->grp->submit(timestamps, images, stride, on_device != 0, masks, mask_stride, vps);
  API_END
}

int plviwo_fe_group_collect(FeGroupHandle *g, FeFrameInfo *infos) {
  API_BEGIN
  if (!g) return FE_BAD_ARG;
  return g->grp->collect(infos);
  API_END
}

int plviwo_fe_group_play(FeGroupHandle *g, int n_ticks, const uint8_t *const *images, int stride, int on_device,
                         const double *timestamps, const double *vps, FePlayStats *out) {
  API_BEGIN
  if (!g || n_ticks < 0 || !images || !timestamps) return FE_BAD_ARG;
  return g->grp->play(n_ticks, images, stride, on_device != 0, timestamps, vps, out);
  API_END
}

int plviwo_fe_group_get_point_rows(FeGroupHandle *g, int stream, FePointRow *out, int cap, int *n_out) {
  if (!g) return FE_BAD_ARG;
  const GroupOutHeader *h = g->grp->header(stream);
  if (!h) return FE_BAD_ARG;
  return copy_rows(g->grp->point_rows(stream), h->info.n_point_rows, sizeof(FePointRow), out, cap, n_out);
}
int plviwo_fe_group_get_last_obs(FeGroupHandle *g, int stream, uint64_t *ids, float *uv, int cap, int *n_out) {
  if (!g) return FE_BAD_ARG;
  const GroupOutHeader *h = g->grp->header(stream);
  if (!h) return FE_BAD_ARG;
  const int n = h->n_obs;
  if (n_out) *n_out = n;
  if (!ids && !uv) return FE_OK;
  if (cap < n) return FE_OVERFLOW;
  if (ids && n) std::memcpy(ids, g->grp->obs_ids(stream), (size_t)n * sizeof(uint64_t));
  if (uv && n) std::memcpy(uv, g->grp->obs_uv(stream), (size_t)n * 2 * sizeof(float));
  return FE_OK;
}
int plviwo_fe_group_get_line_rows(FeGroupHandle *g, int stream, FeLineRow *out, int cap, int *n_out) {
  if (!g) return FE_BAD_ARG;
  const GroupOutHeader *h = g->grp->header(stream);
  if (!h) return FE_BAD_ARG;
  return copy_rows(g->grp->line_rows(stream), h->info.n_line_rows, sizeof(FeLineRow), out, cap, n_out);
}
int plviwo_fe_group_get_line_points(FeGroupHandle *g, int stream, FeLinePoint *out, int cap, int *n_out) {
  if (!g) return FE_BAD_ARG;
  const GroupOutHeader *h = g->grp->header(stream);
  if (!h) return FE_BAD_ARG;
  return copy_rows(g->grp->line_points(stream), h->info.n_line_rows > 0 ? h->n_line_points : 0, sizeof(FeLinePoint), out, cap, n_out);
}
int plviwo_fe_group_get_line_samples(FeGroupHandle *g, int stream, float *uv01, uint8_t *status, int cap, int *n_out) {
  if (!g) return FE_BAD_ARG;
  return g->grp->line_samples(stream, uv01, status, cap, n_out);
}
int plviwo_fe_group_get_state(FeGroupHandle *g, int stream, void *buf, size_t cap, size_t *n_bytes) {
  API_BEGIN
  if (!g) return FE_BAD_ARG;
  return g->grp->get_state(stream, buf, cap, n_bytes);
  API_END
}
int plviwo_fe_group_set_state(FeGroupHandle *g, int stream, const void *buf, size_t n_bytes) {
  API_BEGIN
  if (!g) return FE_BAD_ARG;
  return g->grp->set_state(stream, buf, n_bytes);
  API_END
}
int plviwo_fe_group_tap(FeGroupHandle *g, int stream, int what, void *buf, size_t cap, size_t *n_bytes) {
  API_BEGIN
  if (!g) return FE_BAD_ARG;
  return g->grp->tap(stream, what, buf, cap, n_bytes);
  API_END
}
int plviwo_fe_group_enable_timing(FeGroupHandle *g, int on) {
  if (!g) return FE_BAD_ARG;
  g->grp->enable_timing(on != 0);
  return FE_OK;
}
int plviwo_fe_group_get_times(FeGroupHandle *g, FeGroupTimes *out, int reset) {
  if (!g || !out) return FE_BAD_ARG;
  *out = g->grp->times(reset != 0);
  return FE_OK;
}

// ---- stereo group (many stereo rigs of one device, csrc/fe_group.h) ---------------------------------------------
int plviwo_fe_stereo_group_create(const FeConfig *cfg, int n_rigs, int device, FeStereoGroupHandle **out) {
  return plviwo_fe_stereo_group_create_model(cfg, n_rigs, FE_CAM_RADTAN, device, out);
}

int plviwo_fe_stereo_group_create_model(const FeConfig *cfg, int n_rigs, int model, int device, FeStereoGroupHandle **out) {
  API_BEGIN
  if (!cfg || !out) return FE_BAD_ARG;
  *out = nullptr;
  if (const char *why = check_model(model)) return create_error(FE_BAD_ARG, why);
  if (n_rigs < 1 || n_rigs > 2048) return create_error(FE_BAD_ARG, "n_rigs must be in [1, 2048] (2 camera streams per rig, at most 4096)");
  if (const char *why = check_config(*cfg, cfg->width, cfg->height)) return create_error(FE_BAD_ARG, why);
  if (cfg->grid_x * cfg->grid_y > 256) return create_error(FE_BAD_ARG, "a stream group supports at most 256 grid cells");
  // the stereo handle ignores both; a stereo group refuses them rather than run something else than asked
  if (cfg->downsample) return create_error(FE_BAD_ARG, "cfg.downsample is not supported in a stereo group");
  if (cfg->line_samples) return create_error(FE_BAD_ARG, "cfg.line_samples is not supported in a stereo group");
  if (int rc = check_device(device)) return rc;
  FeGroup *grp = new FeGroup(*cfg, 2 * n_rigs, device, true, model);
  int rc = grp->init();
  if (rc != FE_OK) {
    g_create_error = grp->last_error;
    delete grp;
    return rc;
  }
  *out = new FeStereoGroupHandle{grp};
  return FE_OK;
  API_END
}

int plviwo_fe_stereo_group_destroy(FeStereoGroupHandle *g) {
  API_BEGIN
  if (!g) return FE_BAD_ARG;
  delete g->grp;
  delete g;
  return FE_OK;
  API_END
}

const char *plviwo_fe_stereo_group_last_error(const FeStereoGroupHandle *g) { return g ? g->grp->last_error.c_str() : g_create_error.c_str(); }

// stream of (rig, cam), or -1 with the reason in last_error
static int rig_stream(FeStereoGroupHandle *g, int rig, int cam) {
  if (rig < 0 || rig >= g->grp->n_streams() / 2 || cam < 0 || cam > 1) {
    g->grp->last_error = "rig or cam out of range (cam: 0 left, 1 right)";
    return -1;
  }
  return 2 * rig + cam;
}

int plviwo_fe_stereo_group_set_calib(FeStereoGroupHandle *g, int rig, int cam, const double K[4], const double D[4]) {
  if (!g) return FE_BAD_ARG;
  const int s = rig_stream(g, rig, cam);
  if (s < 0) return FE_BAD_ARG;
  return g->grp->set_calib(s, K, D);
}

int plviwo_fe_stereo_group_set_camera(FeStereoGroupHandle *g, int rig, int cam, int model, const double K[4], const double D[4]) {
  if (!g) return FE_BAD_ARG;
  if (model != g->grp->model()) {   // as plviwo_fe_set_camera
    g->grp->last_error = model_mismatch(g->grp->model());
    return FE_BAD_ARG;
  }
  return plviwo_fe_stereo_group_set_calib(g, rig, cam, K, D);
}

int plviwo_fe_stereo_group_submit(FeStereoGroupHandle *g, const double *timestamps, const uint8_t *const *images_left,
                                  const uint8_t *const *images_right, int stride, int on_device, const uint8_t *const *masks_left,
                                  const uint8_t *const *masks_right, int mask_stride, const double *vps) {
  API_BEGIN
  if (!g) return FE_BAD_ARG;
  return g->grp->stereo_submit(timestamps, images_left, images_right, stride, on_device != 0, masks_left, masks_right, mask_stride, vps);
  API_END
}

int plviwo_fe_stereo_group_collect(FeStereoGroupHandle *g, FeStereoInfo *infos) {
  API_BEGIN
  if (!g) return FE_BAD_ARG;
  return g->grp->stereo_collect(infos);
  API_END
}

int plviwo_fe_stereo_group_play(FeStereoGroupHandle *g, int n_ticks, const uint8_t *const *images, int stride, int on_device,
                                const double *timestamps, const double *vps, FePlayStats *out) {
  API_BEGIN
  if (!g || n_ticks < 0 || !images || !timestamps) return FE_BAD_ARG;
  return g->grp->play(n_ticks, images, stride, on_device != 0, timestamps, vps, out);
  API_END
}

int plviwo_fe_stereo_group_get_point_rows(FeStereoGroupHandle *g, int rig, int cam, FePointRow *out, int cap, int *n_out) {
  if (!g) return FE_BAD_ARG;
  const int s = rig_stream(g, rig, cam);
  const GroupOutHeader *h = s < 0 ? nullptr : g->grp->header(s);
  if (!h) return FE_BAD_ARG;
  return copy_rows(g->grp->point_rows(s), h->info.n_point_rows, sizeof(FePointRow), out, cap, n_out);
}
int plviwo_fe_stereo_group_get_last_obs(FeStereoGroupHandle *g, int rig, int cam, uint64_t *ids, float *uv, int cap, int *n_out) {
  if (!g) return FE_BAD_ARG;
  const int s = rig_stream(g, rig, cam);
  if (s < 0) return FE_BAD_ARG;
  FeGroupHandle view{g->grp};   // the group's getter on the rig's stream
  return plviwo_fe_group_get_last_obs(&view, s, ids, uv, cap, n_out);
}
int plviwo_fe_stereo_group_get_line_rows(FeStereoGroupHandle *g, int rig, FeLineRow *out, int cap, int *n_out) {
  if (!g) return FE_BAD_ARG;
  const int s = rig_stream(g, rig, 0);
  if (s < 0) return FE_BAD_ARG;
  FeGroupHandle view{g->grp};   // the group's getter on the rig's stream
  return plviwo_fe_group_get_line_rows(&view, s, out, cap, n_out);
}
int plviwo_fe_stereo_group_get_line_points(FeStereoGroupHandle *g, int rig, FeLinePoint *out, int cap, int *n_out) {
  if (!g) return FE_BAD_ARG;
  const int s = rig_stream(g, rig, 0);
  if (s < 0) return FE_BAD_ARG;
  FeGroupHandle view{g->grp};   // the group's getter on the rig's stream
  return plviwo_fe_group_get_line_points(&view, s, out, cap, n_out);
}
int plviwo_fe_stereo_group_get_state(FeStereoGroupHandle *g, int rig, void *buf, size_t cap, size_t *n_bytes) {
  API_BEGIN
  if (!g) return FE_BAD_ARG;
  return g->grp->stereo_get_state(rig, buf, cap, n_bytes);
  API_END
}
int plviwo_fe_stereo_group_set_state(FeStereoGroupHandle *g, int rig, const void *buf, size_t n_bytes) {
  API_BEGIN
  if (!g) return FE_BAD_ARG;
  return g->grp->stereo_set_state(rig, buf, n_bytes);
  API_END
}

// ---- stereo rig (TrackKLT with use_stereo = true) -----------------------------------------------------------
int plviwo_fe_stereo_create(const FeConfig *cfg, const double K_right[4], const double D_right[4], int device,
                            FeStereoHandle **out) {
  return plviwo_fe_stereo_create_model(cfg, FE_CAM_RADTAN, K_right, D_right, device, out);
}

int plviwo_fe_stereo_create_model(const FeConfig *cfg, int model, const double K_right[4], const double D_right[4], int device,
                                  FeStereoHandle **out) {
  API_BEGIN
  if (!cfg || !out) return FE_BAD_ARG;
  *out = nullptr;
  if (const char *why = check_model(model)) return create_error(FE_BAD_ARG, why);
  // the rig tracks at the raw size: it zeroes cfg.downsample
  if (const char *why = check_config(*cfg, cfg->width, cfg->height)) return create_error(FE_BAD_ARG, why);
  if (int rc = check_device(device)) return rc;
  FeStereo *st = new FeStereo(*cfg, K_right, D_right, device, model);
  int rc = st->init();
  if (rc != FE_OK) {
    g_create_error = st->last_error;
    delete st;
    return rc;
  }
  *out = new FeStereoHandle{st};
  return FE_OK;
  API_END
}

int plviwo_fe_stereo_destroy(FeStereoHandle *h) {
  API_BEGIN
  if (!h) return FE_BAD_ARG;
  delete h->st;
  delete h;
  return FE_OK;
  API_END
}

const char *plviwo_fe_stereo_last_error(const FeStereoHandle *h) { return h ? h->st->last_error.c_str() : g_create_error.c_str(); }

int plviwo_fe_stereo_set_calib(FeStereoHandle *h, int cam, const double K[4], const double D[4]) {
  if (!h || !K || !D) return FE_BAD_ARG;
  return h->st->set_calib(cam, K, D);
}
int plviwo_fe_stereo_set_camera(FeStereoHandle *h, int cam, int model, const double K[4], const double D[4]) {
  if (!h || !K || !D) return FE_BAD_ARG;
  if (model != h->st->model()) {
    h->st->last_error = model_mismatch(h->st->model());
    return FE_BAD_ARG;
  }
  return plviwo_fe_stereo_set_calib(h, cam, K, D);
}

int plviwo_fe_stereo_set_num_features(FeStereoHandle *h, int n) {
  if (!h || n < 1) return FE_BAD_ARG;
  return h->st->set_num_features(n);
}
int plviwo_fe_stereo_change_feat_id(FeStereoHandle *h, uint64_t id_old, uint64_t id_new) {
  if (!h) return FE_BAD_ARG;
  return h->st->change_feat_id(id_old, id_new);
}

int plviwo_fe_stereo_feed(FeStereoHandle *h, double timestamp, const uint8_t *image_left, const uint8_t *image_right, int width,
                          int height, int stride, const uint8_t *mask_left, const uint8_t *mask_right, int mask_stride,
                          const double vp[6], FeStereoInfo *info) {
  API_BEGIN
  if (!h) return FE_BAD_ARG;
  const uint8_t *img[2] = {image_left, image_right};
  const uint8_t *msk[2] = {mask_left, mask_right};
  return h->st->feed(timestamp, img, width, height, stride, false, msk, mask_stride, vp, info);
  API_END
}

int plviwo_fe_stereo_submit(FeStereoHandle *h, double timestamp, const uint8_t *image_left, const uint8_t *image_right, int stride,
                            int on_device, const uint8_t *mask_left, const uint8_t *mask_right, int mask_stride, const double vp[6]) {
  API_BEGIN
  if (!h || !image_left || !image_right) return FE_BAD_ARG;
  const uint8_t *img[2] = {image_left, image_right};
  const uint8_t *msk[2] = {mask_left, mask_right};
  return h->st->submit(timestamp, img, stride, on_device != 0, msk, mask_stride, vp);
  API_END
}

int plviwo_fe_stereo_collect(FeStereoHandle *h, FeStereoInfo *info) {
  API_BEGIN
  if (!h) return FE_BAD_ARG;
  return h->st->collect(info);
  API_END
}

int plviwo_fe_stereo_get_point_rows(FeStereoHandle *h, int cam, FePointRow *out, int cap, int *n_out) {
  if (!h || cam < 0 || cam > 1) return FE_BAD_ARG;
  return copy_out(h->st->rows(cam), out, cap, n_out);
}

int plviwo_fe_stereo_get_last_obs(FeStereoHandle *h, int cam, uint64_t *ids, float *uv, int cap, int *n_out) {
  if (!h || cam < 0 || cam > 1) return FE_BAD_ARG;
  const auto &p = h->st->last_obs(cam);
  const auto &id = h->st->last_ids(cam);
  if (n_out) *n_out = (int)p.size();
  if (!ids && !uv) return FE_OK;
  if (cap < (int)p.size()) return FE_OVERFLOW;
  for (size_t i = 0; i < p.size(); i++) {
    if (ids) ids[i] = id[i];
    if (uv) {
      uv[2 * i] = p[i].x;
      uv[2 * i + 1] = p[i].y;
    }
  }
  return FE_OK;
}

int plviwo_fe_stereo_get_line_rows(FeStereoHandle *h, FeLineRow *out, int cap, int *n_out) {
  if (!h) return FE_BAD_ARG;
  return copy_out(h->st->left_result().line_rows, out, cap, n_out);
}
int plviwo_fe_stereo_get_line_points(FeStereoHandle *h, FeLinePoint *out, int cap, int *n_out) {
  if (!h) return FE_BAD_ARG;
  return copy_out(h->st->left_result().line_points, out, cap, n_out);
}
int plviwo_fe_stereo_classify_lines(FeStereoHandle *h, const double vp[6]) {
  if (!h || !vp) return FE_BAD_ARG;
  return h->st->classify_lines(vp);
}

int plviwo_fe_stereo_get_state(FeStereoHandle *h, void *buf, size_t cap, size_t *n_bytes) {
  API_BEGIN
  if (!h) return FE_BAD_ARG;
  return h->st->get_state(buf, cap, n_bytes);
  API_END
}
int plviwo_fe_stereo_set_state(FeStereoHandle *h, const void *buf, size_t n_bytes) {
  API_BEGIN
  if (!h) return FE_BAD_ARG;
  return h->st->set_state(buf, n_bytes);
  API_END
}
int plviwo_fe_stereo_get_stage_times(FeStereoHandle *h, FeStageTimes *out, int reset) {
  if (!h || !out) return FE_BAD_ARG;
  *out = h->st->snapshot_times(reset != 0);
  return FE_OK;
}

}  // extern "C"
