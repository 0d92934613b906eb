/*
 * plviwo_fe.h — C ABI of the B200-native PL-VIWO visual front end.
 *
 * One FeHandle = one camera stream (one ov_core::TrackKLT + one viw::TrackLSD for the same camera) bound to one
 * CUDA device and its own CUDA streams.  The entry points are what a binding of the reference's tracker API
 * would call (see INTEGRATION.md for the header-only ov_core adaptor):
 *
 *   reference interface                                               file:line                      replaced by
 *   ----------------------------------------------------------------  -----------------------------  -------------------------
 *   TrackKLT::TrackKLT(cameras, numfeats, numaruco, stereo, hist,     ov_core/src/track/TrackKLT.h:54-57,       plviwo_fe_create
 *       fast_threshold, gridx, gridy, minpxdist)                      TrackBase.cpp:30-41
 *   viw::TrackLSD::TrackLSD(cameras, stereo, hist, trackFEATS)        PL-VIWO/src/update/cam/TrackLSD.cpp:30-37  plviwo_fe_create (use_lines)
 *   CamBase::set_value(calib) on the shared camera object             ov_core/src/cam/CamBase.h:56-82            plviwo_fe_set_calib
 *   TrackKLT::feed_new_camera(const CameraData&)                      ov_core/src/track/TrackKLT.cpp:34-94       plviwo_fe_feed
 *   TrackLSD::feed_new_camera(const CameraData&, vanishing_points)    PL-VIWO/src/update/cam/TrackLSD.cpp:39-68  plviwo_fe_feed (vp != NULL)
 *   FeatureDatabase::update_feature(id,t,cam,u,v,un,vn) rows          ov_core/src/feat/FeatureDatabase.cpp:60-85 plviwo_fe_get_point_rows
 *   TrackBase::get_last_obs() / get_last_ids()                        ov_core/src/track/TrackBase.h:137-146      plviwo_fe_get_last_obs
 *   LineFeatureDatabase::update_feature(id,t,cam,line,line_n,...)     linefeat/LineFeatureDatabase.cpp:40-76     plviwo_fe_get_line_rows (+ _line_points)
 *   TrackLSD::LineClassification(line, vanishing_points)              PL-VIWO/src/update/cam/TrackLSD.cpp:318-333 plviwo_fe_classify_lines
 *   TrackBase::set_num_features / change_feat_id                      ov_core/src/track/TrackBase.cpp:267-285    plviwo_fe_set_num_features / _change_feat_id
 *   the bag loop feeding frames in order                               PL-VIWO/src/run_bag.cpp:272-340            plviwo_fe_submit / _collect / _play
 *   tracker members pts_last/ids_last/currid, lines_last/...          TrackBase.h:173-192, TrackLSD.h:248-279    plviwo_fe_get_state / _set_state
 *
 * No C++ types, no exceptions, no exit() cross this boundary: malformed input is FE_BAD_ARG where the reference
 * calls std::exit(EXIT_FAILURE) (TrackKLT.cpp:37-43).  All pixel work runs in hand-written CUDA kernels for
 * sm_100a; there is no CPU fallback — every entry point fails with FE_NO_DEVICE / FE_CUDA_ERROR instead.
 *
 * Threading (TrackBase.h:58-65): a handle is not re-entrant; distinct handles are independent and may be
 * driven from different host threads and live on different GPUs (streams never exchange data).
 */
#ifndef PLVIWO_FE_H
#define PLVIWO_FE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PLVIWO_FE_ABI_VERSION 1

typedef struct FeHandle FeHandle;

enum FeStatus {
  FE_OK = 0,
  FE_BAD_ARG = 1,        /* malformed message / sizes do not match the handle          */
  FE_NO_DEVICE = 2,      /* no usable CUDA device (never falls back to the CPU)        */
  FE_CUDA_ERROR = 3,     /* a CUDA call failed; see plviwo_fe_last_error               */
  FE_OVERFLOW = 4,       /* caller-provided output array too small (n_out = required)  */
  FE_INTERNAL = 5
};

enum FeHistogramMethod { FE_HIST_NONE = 0, FE_HIST_HISTOGRAM = 1, FE_HIST_CLAHE = 2 }; /* TrackBase.h:78 */

/* Every front-end knob: options/OptionsCamera.h:77-108 plus the constants the reference hard-codes
 * (TrackKLT.h:143-144 pyr_levels/win_size, TrackLSD.h:269-273 FLD parameters, TrackLSD.cpp:231 length). */
typedef struct FeConfig {
  int32_t width, height;        /* image size; fixed for the lifetime of the handle                     */
  int32_t num_features;         /* n_pts                                                                */
  int32_t fast_threshold;
  int32_t grid_x, grid_y;
  int32_t min_px_dist;
  int32_t pyr_levels;           /* OpenCV maxLevel (reference: 5) => pyr_levels + 1 images              */
  int32_t win_size;             /* LK window (reference: 15); odd, <= 31                                */
  int32_t histogram_method;     /* FeHistogramMethod (CLAHE = cv::createCLAHE(10.0, 8x8), TrackKLT.cpp:60-64) */
  int32_t numaruco;             /* first point id = 4 * numaruco + 2 (TrackBase.cpp:34)                 */
  int32_t use_lines;            /* OptionsCamera.h:108                                                  */
  int32_t fld_length_threshold; /* 20                                                                   */
  float fld_distance_threshold; /* 1.414213562f                                                         */
  float canny_th1, canny_th2;   /* 50, 50 (aperture 3, L1 gradient)                                     */
  float line_min_length;        /* 40 (TrackLSD.cpp:231)                                                */
  int32_t line_samples;         /* extension (BASELINE.json configs[2], not in the reference): LK over this many   */
                                /* points sampled evenly along every segment the line detector kept in the previous */
                                /* frame (longer than line_min_length), previous -> current image; 0 = off          */
  int32_t lookahead;            /* frames that plviwo_fe_submit may run ahead of plviwo_fe_collect      */
  int32_t downsample;           /* UpdaterCamera::feed_measurement's pre-step (UpdaterCamera.cpp:86-95): cv::pyrDown of */
                                /* image and mask to (width/2, height/2) before tracking; width/height above are the    */
                                /* INPUT size, K is the (already halved, OptionsCamera.cpp:123-126) tracking calibration */
  double K[4];                  /* fx fy cx cy                                                          */
  double D[4];                  /* radtan k1 k2 p1 p2                                                   */
} FeConfig;

/* One FeatureDatabase::update_feature call (TrackKLT.cpp:176-179). */
typedef struct FePointRow {
  uint64_t id;
  float u, v;     /* raw pixel                     */
  float un, vn;   /* undistorted normalised coords */
} FePointRow;

/* One LineFeatureDatabase::update_feature call (TrackLSD.cpp:163-167).  The points attached to the line
 * (point_on_lines map in ascending point id, and point_position in detection order) are stored contiguously;
 * fetch them with plviwo_fe_get_line_points using [pt_offset, pt_offset + n_pts). */
typedef struct FeLineRow {
  uint64_t id;
  float line[4];    /* x1 y1 x2 y2, full-resolution pixels */
  float line_n[4];  /* undistorted normalised endpoints    */
  int32_t D;        /* LineClassification: 3 z, 2 y, 1 x, 0 none */
  int32_t n_pts;
  int32_t pt_offset;
  int32_t matched;  /* 1 if the id was inherited from last frame's line (LineMatch) */
} FeLineRow;

typedef struct FeLinePoint {
  int32_t pid;      /* key of point_on_lines (ascending within a line)          */
  float dist;       /* value of point_on_lines: point-to-segment distance       */
  float u, v;       /* point_position entry k of the same line (detection order)*/
} FeLinePoint;

/* Per-frame outcome flags / counters (the reference only prints these). */
typedef struct FeFrameInfo {
  double timestamp;
  int32_t n_point_rows;
  int32_t n_line_rows;
  int32_t n_last_obs;       /* size of pts_last after the frame                          */
  int32_t reset;            /* 1: tracker cleared itself (TrackKLT.cpp:143-152)          */
  int32_t first_frame;      /* 1: detection-only frame (TrackKLT.cpp:110-123)            */
  int32_t n_detected;       /* points added by the top-off detection                    */
  int32_t n_lk_in, n_klt_ok, n_ransac_ok;
  int32_t n_lines_detected; /* segments longer than line_min_length                      */
  int32_t n_line_matches;
  int32_t detection_ran;
  int32_t reserved;
} FeFrameInfo;

/* Stage timings accumulated with CUDA events on the handle's own streams (ms, and launch counts). */
enum FeStage {
  FE_STAGE_H2D = 0, FE_STAGE_HIST, FE_STAGE_EQ_PYR, FE_STAGE_PYR_REST, FE_STAGE_FAST, FE_STAGE_SUBPIX, FE_STAGE_LK,
  FE_STAGE_CANNY, FE_STAGE_FLD /* whole segment extraction: CCL + WALK + SEG */, FE_STAGE_FLD_CCL, FE_STAGE_FLD_WALK,
  FE_STAGE_FLD_SEG, FE_STAGE_COUNT,
  FE_STAGE_LINE_FRAMES = FE_STAGE_COUNT /* launches[] only: frames carried by the timed line-path launches (a launch of the
                                           line path carries a batch of frames; ms[] / launches[] of CANNY..FLD_SEG is per launch) */
};
/* indices of FeStageTimes.host_ms: wall time of the host-side steps of a single handle */
enum FeHostStage {
  FE_HOST_SUBMIT = 0, FE_HOST_DETECTION, FE_HOST_MATCHING, FE_HOST_RANSAC, FE_HOST_LINES, FE_HOST_COLLECT, FE_HOST_LINE_WAIT,
  FE_HOST_CAND_WAIT /* candidate table */, FE_HOST_SPECULATE /* speculative LK launch */, FE_HOST_ASSEMBLE /* result assembly */,
  FE_HOST_LINE_ASSIGN /* AssignPointToLines */, FE_HOST_SPEC_LAUNCH, FE_HOST_LK_LAUNCH, FE_HOST_LK_WAIT, FE_HOST_LINE_MATCH,
  FE_HOST_LINE_ROWS, FE_HOST_COUNT
};
typedef struct FeStageTimes {
  double ms[16];
  uint64_t launches[16];
  uint64_t frames;
  uint64_t kernel_launches_total;
  uint64_t h2d_bytes, d2h_bytes;   /* bytes moved by the handle's own cudaMemcpyAsync calls */
  double host_ms[16];              /* host wall time per FeHostStage */
} FeStageTimes;

/* ---- lifetime ----------------------------------------------------------------------------------------- */
int plviwo_fe_abi_version(void);
void plviwo_fe_default_config(FeConfig *cfg);                 /* reference defaults, KAIST cam0 calibration */
int plviwo_fe_device_count(int *n);
int plviwo_fe_create(const FeConfig *cfg, int device, FeHandle **out);
int plviwo_fe_destroy(FeHandle *h);
const char *plviwo_fe_last_error(const FeHandle *h);          /* h may be NULL: last create() error         */

/* ---- per-frame ---------------------------------------------------------------------------------------- */
/* Intrinsics are refined online by the estimator (StateHelper.cpp:166): call before feed whenever they change. */
int plviwo_fe_set_calib(FeHandle *h, const double K[4], const double D[4]);
/* The same with the camera model named (ov_core::CamBase subclasses, cam/CamRadtan.h / cam/CamEqui.h).  Only the radtan
 * model is implemented: FE_CAM_EQUI is rejected with FE_BAD_ARG instead of being undistorted with the wrong formula. */
enum FeCameraModel { FE_CAM_RADTAN = 0, FE_CAM_EQUI = 1 };
int plviwo_fe_set_camera(FeHandle *h, int model, const double K[4], const double D[4]);
/* TrackBase::currid (TrackBase.h:192) is one counter per tracker object, shared by all its cameras: a caller that owns
 * several handles hands the counter from handle to handle around every feed (between frames only). */
int plviwo_fe_get_currid(FeHandle *h, uint64_t *currid);
int plviwo_fe_set_currid(FeHandle *h, uint64_t currid);
int plviwo_fe_set_num_features(FeHandle *h, int num_features);
int plviwo_fe_change_feat_id(FeHandle *h, uint64_t id_old, uint64_t id_new);

/* Synchronous drop-in for feed_new_camera: image and mask are HOST buffers (8UC1, borrowed for the call);
 * mask may be NULL (all zero); vp = 3 vanishing points (x0 y0 x1 y1 x2 y2) or NULL to skip the line tracker. */
int plviwo_fe_feed(FeHandle *h, double timestamp, const uint8_t *image, int width, int height, int stride,
                   const uint8_t *mask, int mask_stride, const double vp[6], FeFrameInfo *info);

/* Same, with the image already resident in this handle's device memory (device pointer, pitch in bytes). */
int plviwo_fe_feed_device(FeHandle *h, double timestamp, const void *d_image, int width, int height, int pitch,
                          const uint8_t *mask, int mask_stride, const double vp[6], FeFrameInfo *info);

/* Pipelined form for offline playback (run_bag.cpp indexes the whole bag first): submit() enqueues the
 * state-independent work of a frame (copy, equalisation, pyramid, edge map, segment extraction) up to
 * cfg.lookahead frames ahead; collect() finishes the oldest submitted frame in order and exposes its rows.
 * Results are identical to calling plviwo_fe_feed frame by frame. */
int plviwo_fe_submit(FeHandle *h, double timestamp, const uint8_t *image, int stride, int on_device,
                     const uint8_t *mask, int mask_stride, const double vp[6]);
int plviwo_fe_collect(FeHandle *h, FeFrameInfo *info);

/* Whole-sequence playback (run_bag.cpp:272-340 feeds a bag frame by frame): submit/collect over n_frames frames with the
 * handle's lookahead, entirely inside the library.  images[i] is a host or device pointer (on_device), vps has 6 doubles
 * per frame or is NULL (no line tracker).  Rows are counted and folded into a checksum instead of being returned; the
 * rows of the LAST frame stay available through the getters.  Results are identical to feeding frame by frame. */
typedef struct FePlayStats {
  uint64_t frames, point_rows, line_rows, resets;
  double checksum;   /* sum over point rows of (id + u + v) plus sum over line rows of (id + x1 + y1 + x2 + y2) */
} FePlayStats;
int plviwo_fe_play(FeHandle *h, int n_frames, const uint8_t *const *images, int stride, int on_device, const double *timestamps,
                   const double *vps, FePlayStats *out);

/* ---- results of the last completed frame -------------------------------------------------------------- */
int plviwo_fe_get_point_rows(FeHandle *h, FePointRow *out, int cap, int *n_out);
int plviwo_fe_get_last_obs(FeHandle *h, uint64_t *ids, float *uv /* 2 per point */, int cap, int *n_out);
int plviwo_fe_get_line_rows(FeHandle *h, FeLineRow *out, int cap, int *n_out);
int plviwo_fe_get_line_points(FeHandle *h, FeLinePoint *out, int cap, int *n_out);
/* Re-runs LineClassification (TrackLSD.cpp:318-366) on the line rows of the last completed frame with these vanishing
 * points.  For callers that, like UpdaterCamera.cpp:105-110, only know the vanishing points after the point tracker was
 * fed: feed with any vp (e.g. zeros), then classify, then read the rows. */
int plviwo_fe_classify_lines(FeHandle *h, const double vp[6]);
/* extension: LK-tracked samples of the previous frame's detected segments, segment-major (line_samples consecutive
 * entries per segment, in detection order): u0 v0 (previous image) u1 v1 (current image) and the KLT status */
int plviwo_fe_get_line_samples(FeHandle *h, float *uv01 /* 4 per sample */, uint8_t *status, int cap, int *n_out);

/* ---- tracker state: teacher-forced parity tests, checkpoint / resume ---------------------------------- */
/* Serialised into a caller buffer; *n_bytes returns the size needed / written.  Includes the previous frame's
 * equalised image (the pyramid is rebuilt on set_state). */
int plviwo_fe_get_state(FeHandle *h, void *buf, size_t cap, size_t *n_bytes);
int plviwo_fe_set_state(FeHandle *h, const void *buf, size_t n_bytes);

/* ---- debug / test taps (device results copied to host) ------------------------------------------------ */
enum FeTap {
  FE_TAP_PYR_LEVEL0 = 0,   /* .. FE_TAP_PYR_LEVEL0 + level : current pyramid images (8U, tight rows)          */
  FE_TAP_HALF = 32,        /* half-resolution equalised image fed to the line detector                        */
  FE_TAP_EDGES = 33,       /* Canny edge map, one byte per pixel (0 / 255), half resolution                   */
  FE_TAP_FAST_LAST = 34,   /* last detection: int32 records (cell_x, cell_y, x, y, score) in reference order  */
  FE_TAP_LK_LAST = 35,     /* last LK: float records (x0, y0, x1, y1, status_klt, status_ransac)              */
  FE_TAP_SUBPIX_LAST = 36, /* last detection: float records (x_sel, y_sel, x_ref, y_ref)                      */
  FE_TAP_FLD_LAST = 37     /* last line detection: float records (x1, y1, x2, y2) at half resolution          */
};
int plviwo_fe_enable_taps(FeHandle *h, int on);   /* taps cost host time: off by default, enable BEFORE feeding */
int plviwo_fe_tap(FeHandle *h, int what, void *buf, size_t cap, size_t *n_bytes);

/* ---- measurement -------------------------------------------------------------------------------------- */
int plviwo_fe_enable_timing(FeHandle *h, int on);   /* CUDA-event stage timing (adds event records only)   */
int plviwo_fe_get_stage_times(FeHandle *h, FeStageTimes *out, int reset);

/* ---- stereo rig: TrackKLT with use_stereo = true ------------------------------------------------------- */
/*
 *   reference interface                                               file:line                                   replaced by
 *   ----------------------------------------------------------------  ------------------------------------------  -----------------------------
 *   TrackKLT::TrackKLT(cameras {0, 1}, ..., stereo = true, ...)       ov_core/src/track/TrackKLT.h:54-57          plviwo_fe_stereo_create
 *   TrackKLT::feed_new_camera(message with two images) -> feed_stereo ov_core/src/track/TrackKLT.cpp:34-94, 202-393 plviwo_fe_stereo_feed
 *   TrackKLT::perform_detection_stereo                                TrackKLT.cpp:530-827                        (inside feed / collect)
 *   FeatureDatabase::update_feature rows of cam_id_left / _right      TrackKLT.cpp:352-363                        plviwo_fe_stereo_get_point_rows
 *   TrackBase::get_last_obs()[cam] / get_last_ids()[cam]              TrackBase.h:137-146                         plviwo_fe_stereo_get_last_obs
 *
 * One FeStereoHandle = one stereo pair (camera 0 = left, 1 = right; OptionsCamera stereo_pairs) on one device.  Both
 * images have the size given in FeConfig; cfg->K / cfg->D calibrate the left camera, K_right / D_right the right one
 * (NULL: same as left).  The reference's line tracker has no stereo path: with two images it runs its monocular code
 * on the LEFT image against the stereo tracker's left points (TrackLSD.cpp:57-60, :127-129).  cfg->use_lines = 1 and a
 * non-NULL vp do exactly that here; the line rows come back through plviwo_fe_stereo_get_line_rows.  line_samples and
 * downsample are ignored.
 */
typedef struct FeStereoHandle FeStereoHandle;
typedef struct FeStereoInfo {
  double timestamp;
  int32_t n_point_rows[2];   /* rows of the left / right camera                                   */
  int32_t n_last_obs[2];     /* pts_last sizes after the pair                                     */
  int32_t reset;             /* 1: both temporal masks empty, tracker cleared (TrackKLT.cpp:286-300) */
  int32_t first_frame;       /* 1: detection-only pair (:221-241)                                 */
  int32_t detection_ran[2];
  int32_t n_detected[2];     /* points added per camera by the top-off detection                  */
  int32_t n_stereo_new;      /* new left points that were also found in the right image (:668-678) */
  int32_t n_lk_in[2], n_klt_ok[2], n_ransac_ok[2];
  int32_t n_stereo_rows;     /* ids present in both cameras' rows of this pair                    */
  int32_t n_line_rows, n_lines_detected, n_line_matches;   /* left-image line tracker (0 when off)   */
} FeStereoInfo;

int plviwo_fe_stereo_create(const FeConfig *cfg, const double K_right[4], const double D_right[4], int device,
                            FeStereoHandle **out);
int plviwo_fe_stereo_destroy(FeStereoHandle *h);
const char *plviwo_fe_stereo_last_error(const FeStereoHandle *h);
int plviwo_fe_stereo_set_calib(FeStereoHandle *h, int cam, const double K[4], const double D[4]);
int plviwo_fe_stereo_set_camera(FeStereoHandle *h, int cam, int model, const double K[4], const double D[4]);
int plviwo_fe_stereo_set_num_features(FeStereoHandle *h, int num_features);
int plviwo_fe_stereo_change_feat_id(FeStereoHandle *h, uint64_t id_old, uint64_t id_new);
/* Synchronous drop-in for feed_new_camera with two images (HOST buffers, 8UC1, same stride; masks may be NULL). */
int plviwo_fe_stereo_feed(FeStereoHandle *h, double timestamp, const uint8_t *image_left, const uint8_t *image_right, int width,
                          int height, int stride, const uint8_t *mask_left, const uint8_t *mask_right, int mask_stride,
                          const double vp[6], FeStereoInfo *info);
/* Pipelined form (as plviwo_fe_submit / _collect): the frame-independent work of both images runs up to cfg.lookahead
 * pairs ahead; images are host or device pointers (on_device). */
int plviwo_fe_stereo_submit(FeStereoHandle *h, double timestamp, const uint8_t *image_left, const uint8_t *image_right, int stride,
                            int on_device, const uint8_t *mask_left, const uint8_t *mask_right, int mask_stride, const double vp[6]);
int plviwo_fe_stereo_collect(FeStereoHandle *h, FeStereoInfo *info);
int plviwo_fe_stereo_get_point_rows(FeStereoHandle *h, int cam, FePointRow *out, int cap, int *n_out);
int plviwo_fe_stereo_get_last_obs(FeStereoHandle *h, int cam, uint64_t *ids, float *uv /* 2 per point */, int cap, int *n_out);
/* line rows of the LEFT camera (cam id 0), as plviwo_fe_get_line_rows / _line_points / _classify_lines */
int plviwo_fe_stereo_get_line_rows(FeStereoHandle *h, FeLineRow *out, int cap, int *n_out);
int plviwo_fe_stereo_get_line_points(FeStereoHandle *h, FeLinePoint *out, int cap, int *n_out);
int plviwo_fe_stereo_classify_lines(FeStereoHandle *h, const double vp[6]);
/* State blob: 32-byte header (magic 'PLVS', currid, sizes) followed by one monocular state blob per camera. */
int plviwo_fe_stereo_get_state(FeStereoHandle *h, void *buf, size_t cap, size_t *n_bytes);
int plviwo_fe_stereo_set_state(FeStereoHandle *h, const void *buf, size_t n_bytes);
int plviwo_fe_stereo_get_stage_times(FeStereoHandle *h, FeStageTimes *out, int reset);   /* both cameras summed */

/* ---- stream group: many camera streams of one device tracked together ------------------------------------ */
/*
 *   reference interface                                               file:line                                   replaced by
 *   ----------------------------------------------------------------  ------------------------------------------  -----------------------------
 *   one TrackKLT + one TrackLSD per camera, built in a loop           PL-VIWO/src/update/cam/UpdaterCamera.cpp:36-66  plviwo_fe_group_create
 *   the bag loop feeding every camera's frame in time order           PL-VIWO/src/run_bag.cpp:56-95, 272-340      plviwo_fe_group_submit / _collect / _play
 *   trackFEATS[cam]->feed_new_camera + trackLSDS[cam]->feed_new_camera UpdaterCamera.cpp:105-110                   (one tick = one frame of every stream)
 *   FeatureDatabase / LineFeatureDatabase ::update_feature rows       FeatureDatabase.cpp:60-85, LineFeatureDatabase.cpp:40-76  plviwo_fe_group_get_*_rows
 *
 * BASELINE.json configs[4] ("64 independent camera streams, multi-session batch throughput").  Stream s of a group is what
 * one FeHandle is — its rows are bit-identical to those of a handle fed the same frames — but the frames of all streams
 * of a tick share their kernel launches and the tracker state lives on the device (csrc/fe_group.h).  All streams share
 * the FeConfig (image size, knobs); the calibration is per stream.  cfg->lookahead = ticks that submit may run ahead of
 * collect.  Not supported in a group: cfg->downsample, set_num_features / change_feat_id.
 * cfg->line_samples > 0 (with use_lines): each stream's samples come back through plviwo_fe_group_get_line_samples, equal to a
 * handle's; every output record then holds a sample region of min(line_samples * 1024, max(4096, 8 * num_features) + 32768)
 * samples (17 bytes each: at line_samples = 10, 170 KB per record, n_streams * (lookahead + 2) records of pinned memory).
 */
typedef struct FeGroupHandle FeGroupHandle;
enum FeGroupKernel {
  FE_GK_HIST = 0, FE_GK_EQ_PYR1, FE_GK_PYR_REST, FE_GK_FAST, FE_GK_SELECT, FE_GK_SUBPIX, FE_GK_CANNY, FE_GK_CCL, FE_GK_WALK,
  FE_GK_SEGMENTS, FE_GK_DETECT, FE_GK_LK, FE_GK_GATE, FE_GK_LINES, FE_GK_ACCEPT, FE_GK_CANDS, FE_GK_COUNT
};
typedef struct FeGroupTimes {
  double ms[16];             /* CUDA-event time per kernel (FeGroupKernel), summed over launches (timing enabled) */
  uint64_t launches[16];
  uint64_t frames[16];       /* frames carried by those launches                                                   */
  uint64_t ticks, frames_total, kernel_launches_total;
  uint64_t h2d_bytes, d2h_bytes;   /* frames copied in; rows written back to pinned host memory                    */
  uint64_t fast_cells;       /* grid cells FAST ran on (the valid cells of the detections, Grider_GRID.h:108-125)  */
} FeGroupTimes;

int plviwo_fe_group_create(const FeConfig *cfg, int n_streams, int device, FeGroupHandle **out);
int plviwo_fe_group_destroy(FeGroupHandle *g);
const char *plviwo_fe_group_last_error(const FeGroupHandle *g);
int plviwo_fe_group_set_calib(FeGroupHandle *g, int stream, const double K[4], const double D[4]);
/* as plviwo_fe_set_camera (CamBase::camera_k_OPENCV / camera_d_OPENCV + the model of the CamBase subclass, cam/CamBase.h:47-60):
 * FE_CAM_EQUI is refused with FE_BAD_ARG */
int plviwo_fe_group_set_camera(FeGroupHandle *g, int stream, int model, const double K[4], const double D[4]);
/* One tick: images[s] = frame of stream s (host or device pointer, NULL: no frame for that stream), timestamps[s] its
 * time; masks = NULL or per-stream host pointers (NULL entries allowed); vps = NULL (line tracker not fed) or 6 doubles per
 * stream.  Device frames are read in place and must stay valid until the tick is collected. */
int plviwo_fe_group_submit(FeGroupHandle *g, const double *timestamps, const uint8_t *const *images, int stride, int on_device,
                           const uint8_t *const *masks, int mask_stride, const double *vps);
/* Completes the oldest submitted tick; infos = NULL or n_streams records (timestamp -1 for a stream without a frame). */
int plviwo_fe_group_collect(FeGroupHandle *g, FeFrameInfo *infos);
/* n_ticks ticks of every stream inside the library: images[t * n_streams + s], timestamps[t], vps = 6 doubles per stream
 * (fixed) or NULL; out = n_streams records. */
int plviwo_fe_group_play(FeGroupHandle *g, int n_ticks, const uint8_t *const *images, int stride, int on_device,
                         const double *timestamps, const double *vps, FePlayStats *out);
/* rows of the last collected tick */
int plviwo_fe_group_get_point_rows(FeGroupHandle *g, int stream, FePointRow *out, int cap, int *n_out);
int plviwo_fe_group_get_last_obs(FeGroupHandle *g, int stream, uint64_t *ids, float *uv, int cap, int *n_out);
int plviwo_fe_group_get_line_rows(FeGroupHandle *g, int stream, FeLineRow *out, int cap, int *n_out);
int plviwo_fe_group_get_line_points(FeGroupHandle *g, int stream, FeLinePoint *out, int cap, int *n_out);
/* as plviwo_fe_get_line_samples, for stream `stream` of the last collected tick */
int plviwo_fe_group_get_line_samples(FeGroupHandle *g, int stream, float *uv01 /* 4 per sample */, uint8_t *status, int cap,
                                     int *n_out);
/* per-stream tracker state, same blob as plviwo_fe_get_state / _set_state (teacher forcing, checkpoint / resume) */
int plviwo_fe_group_get_state(FeGroupHandle *g, int stream, void *buf, size_t cap, size_t *n_bytes);
int plviwo_fe_group_set_state(FeGroupHandle *g, int stream, const void *buf, size_t n_bytes);
int plviwo_fe_group_tap(FeGroupHandle *g, int stream, int what /* FE_TAP_PYR_LEVEL0 + l, FE_TAP_HALF */, void *buf, size_t cap,
                        size_t *n_bytes);
int plviwo_fe_group_enable_timing(FeGroupHandle *g, int on);
int plviwo_fe_group_get_times(FeGroupHandle *g, FeGroupTimes *out, int reset);

/* ---- stand-alone kernels (tests / micro-benchmarks; all pointers are HOST buffers) --------------------- */
int plviwo_op_equalize_pyramid(int device, const uint8_t *img, int w, int h, int levels /* maxLevel */,
                               uint8_t *out_levels /* concatenated tight levels 0..maxLevel */, uint8_t *out_half);
int plviwo_op_clahe(int device, const uint8_t *img, int w, int h, uint8_t *out /* w*h */);   /* createCLAHE(10, 8x8)->apply */
int plviwo_op_fast_cell(int device, const uint8_t *img, int w, int h, int threshold, int32_t *xys /* x y score */,
                        int cap, int *n_out);
/* std::sort(corners, compare_response) + first nfg (Grider_GRID.h:128-133) on packed corners x | y << 12 | score << 24.
 * device < 0: the host instantiation of the sort (sorted[] = whole sorted list; cand, if not NULL, = x, y of the first nfg
 * elements as the pruned selection the kernel runs computes them); device >= 0: the selection kernel (cand[] = x, y of
 * the survivors, n_cand of them; sorted may be NULL). */
int plviwo_op_sort_corners(int device, const uint32_t *packed, int n, int nfg, uint32_t *sorted, float *cand, int *n_cand);
int plviwo_op_corner_subpix(int device, const uint8_t *img, int w, int h, float *pts /* in/out 2 per point */, int n);
int plviwo_op_lk(int device, const uint8_t *img0, const uint8_t *img1, int w, int h, int win, int max_level,
                 const float *pts0, float *pts1 /* in: initial flow, out */, uint8_t *status, int n);
/* The same tracking by the stream group's one-warp-per-feature kernel (win 15 and maxLevel <= 5 only): bit-identical results */
int plviwo_op_lk_warp(int device, const uint8_t *img0, const uint8_t *img1, int w, int h, int win, int max_level,
                      const float *pts0, float *pts1 /* in: initial flow, out */, uint8_t *status, int n);
int plviwo_op_undistort(int device, const float *pts, int n, const double K[4], const double D[4], float *out);
int plviwo_op_canny_half(int device, const uint8_t *img, int w, int h, float th, uint8_t *edges /* w*h bytes */);
int plviwo_op_fld(int device, const uint8_t *img, int w, int h, int length_threshold, float distance_threshold,
                  float canny_th, float *lines /* 4 per segment */, int cap, int *n_out);
/* Micro-benchmark of the image-domain kernels on a DEVICE-resident synthetic image of any size (w, h multiples of 4):
 * equalise + pyramid level 1 + half image (k_hist, k_eq_pyr1), FAST over one grid of cells, Canny of the half image.
 * Each kernel is timed alone with CUDA events over `iters` launches after 3 warm-up launches; ms[0..3] = hist, eq_pyr1,
 * fast, canny (mean per launch).  Used by bench.py to report what the kernels reach when a launch carries enough
 * bytes (a batch of frames' worth) instead of one 0.7 MB frame. */
int plviwo_op_image_kernels_time(int device, int w, int h, int iters, float ms[4]);
/* TrackLSD::AssignPointToLines (TrackLSD.cpp:744-792): kept[i] = 1 if line i (x1 y1 x2 y2) keeps at least one of the points;
 * the k-th kept line's (point id, distance) pairs, in ascending point id, are entries off[k] .. off[k + 1] of pid_out /
 * dist_out (off has n_lines + 1 entries).  Host-side step, no GPU needed. */
int plviwo_op_assign_points(int n_lines, const float *lines, int n_pts, const float *pts /* 2 per point */, const uint64_t *pids,
                            int32_t *kept, int32_t *off, int32_t *pid_out, float *dist_out, int cap, int *n_out);
/* TrackLSD::LineMatch (TrackLSD.cpp:368-407) on CSR inputs: line j of the last frame holds point ids
 * last_pids[last_off[j] .. last_off[j + 1]), lines are x1 y1 x2 y2; match_out[i] = index of the last-frame line whose id new
 * line i inherits, or -1.  Host-side step, no GPU needed. */
int plviwo_op_line_match(int n_last, const int32_t *last_off, const int32_t *last_pids, const float *last_lines, int n_new,
                         const int32_t *new_off, const int32_t *new_pids, const float *new_lines, int32_t *match_out);
int plviwo_op_ransac_fundamental(const float *p0n, const float *p1n, int n, double threshold, double confidence,
                                 uint8_t *mask, int *n_inliers); /* host-side sequential step (K9) */

#ifdef __cplusplus
}
#endif
#endif /* PLVIWO_FE_H */
