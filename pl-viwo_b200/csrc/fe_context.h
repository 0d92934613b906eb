// Host side of the front end: one FeContext per camera stream.  Mirrors the reference's tracker objects
// (ov_core::TrackKLT, viw::TrackLSD) with the same method names and the same per-frame state machine, but every
// pixel-touching step is a kernel launch on the context's own CUDA streams (fe_kernels.h).
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <condition_variable>
#include <cstdint>
#include <deque>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/plviwo_fe.h"
#include "fe_kernels.h"
#include "tracker_core.h"

namespace plviwo {

struct Pt {
  float x, y;
};

void pyr_down_host(const uint8_t *src, int sw, int sh, int stride, uint8_t *dst, int dw, int dh);
int line_candidates(const float *px, const float *py, int n, float min_lx, float max_lx, float min_ly, float max_ly, float pa,
                    float pb, float pc, float plen2, uint8_t *pass);
void assign_points_to_lines_host(const std::vector<float4> &lines_new, const std::vector<uint64_t> &ids_new,
                                 const std::vector<Pt> &points, const std::vector<uint64_t> &pids,
                                 std::vector<std::map<int, double>> &pol_new, std::vector<std::vector<Pt>> &positions,
                                 std::vector<float4> &filt_lines, std::vector<uint64_t> &filt_ids, std::vector<float> &spx,
                                 std::vector<float> &spy, std::vector<uint8_t> &pass);
void line_match_host(const std::vector<std::map<int, double>> &pol_last, const std::vector<std::map<int, double>> &pol_new,
                     const std::vector<float4> &lines_new, const std::vector<float4> &lines_last, std::map<int, int> &matches,
                     std::vector<std::pair<int, int>> &inv, std::vector<int> &shared, std::vector<int> &touched);
int ransac_fundamental(const float *m1, const float *m2, int count, double threshold, double confidence, uint8_t *mask,
                       int *mask_valid);

// Everything one frame hands back to the caller: the rows the reference would push into its two databases, the
// tracker's "last" observations after the frame, and the optional debug taps.  Filled by the tracker threads, exposed
// by collect().
struct FrameResult {
  FeFrameInfo info{};
  std::vector<FePointRow> point_rows;
  std::vector<FeLineRow> line_rows;
  std::vector<FeLinePoint> line_points;
  std::vector<float> sample_uv;
  std::vector<uint8_t> sample_status;
  std::vector<Pt> obs;              // pts_last / ids_last after this frame (TrackBase::get_last_obs / get_last_ids)
  std::vector<uint64_t> obs_ids;
  std::vector<int32_t> tap_fast;
  std::vector<float> tap_lk, tap_subpix, tap_fld;
  int rc = FE_OK;
  std::string error;
  void clear() {
    info = FeFrameInfo{};
    point_rows.clear(); line_rows.clear(); line_points.clear(); sample_uv.clear(); sample_status.clear();
    obs.clear(); obs_ids.clear(); tap_fast.clear(); tap_lk.clear(); tap_subpix.clear(); tap_fld.clear();
    rc = FE_OK;
    error.clear();
  }
};

// Hand-off between the threads of one handle: the consumer spins briefly (steady-state pipelining never sleeps) and
// then blocks on a condition variable (an idle handle costs no CPU).
class WorkQueue {
 public:
  void push(int v);
  bool pop(int *v);   // false: stop requested and nothing left
  bool peek(int *v);  // front element without taking it; false if empty
  void stop();
 private:
  std::mutex mu_;
  std::condition_variable cv_;
  std::deque<int> q_;
  std::atomic<int> n_{0};
  std::atomic<bool> stop_{false};
};

// Everything that belongs to one submitted frame and can be produced without tracker state.
struct FrameSlot {
  DevImage raw;          // staged input (device), tracking size
  DevImage raw_in;       // cfg.downsample: the full-size input, raw = pyrDown(raw_in)
  Pyramid pyr;           // equalised pyramid, level 0 = equalised frame
  DevImage half;         // half-resolution equalised frame (line detector input)
  FldBuffers fld;
  uint8_t *h_raw = nullptr;      // pinned staging for the host image
  float4 *h_segs = nullptr;      // pinned: detected segments (half-res)
  int *h_fld_counts = nullptr;   // pinned: [n_chains, n_segments]
  std::vector<uint8_t> mask;     // host copy of the caller's mask (empty = all zero)
  double timestamp = 0;
  double vp[6] = {0, 0, 0, 0, 0, 0};
  bool has_vp = false;
  bool busy = false;
  int line_timed = 0;            // > 0: ev_t[5..9] hold the stage events of a line-path launch that carried this many frames
  bool line_pending = false;     // the frame waits in the handle's line batch (its line path is not launched yet)
  double K[4] = {0, 0, 0, 0}, D[4] = {0, 0, 0, 0};   // calibration in force when the frame was submitted
  FrameResult res;
  std::atomic<int> stage{0};     // 0 idle, 1 submitted, 2 point tracker done, 3 complete (line tracker done)
  int index = 0;
  cudaEvent_t ev_pyr = nullptr, ev_lines = nullptr;
  cudaStream_t s_line = nullptr;   // per-slot streams: the frame-independent work of different frames overlaps
  cudaStream_t s_a = nullptr, s_b = nullptr;
  unsigned *d_hist = nullptr, *d_counters = nullptr;
  uint8_t *d_eq_lut = nullptr;     // cv::equalizeHist LUT of this frame (launch_hist -> launch_eq_pyr1)
  uint8_t *d_clahe = nullptr;      // CLAHE: 64 tile LUTs of this frame
  int *d_seq = nullptr;            // device-side sequence numbers of the completion signals [fast, -, lines]
  cudaGraphExec_t g_image = nullptr, g_fast = nullptr, g_lines = nullptr;
  int graph_version = -1;
  bool warmed = false;
  bool lines_recorded = false;   // ev_lines has been recorded at least once
  cudaEvent_t ev_t[10] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  bool timed = false;

  // ---- pre-detection: everything perform_griding computes that does NOT depend on tracker state.  FAST runs on
  // every grid cell of the frame as soon as level 0 exists; a second kernel sorts each cell's corners with the
  // reference's std::sort (introsort.h), takes the first num_features_grid of each and a third refines them
  // (cornerSubPix).  The top-off detection of the point tracker then only applies the state-dependent tests (valid
  // cells, mask, min distance) to this candidate table.
  unsigned *d_fast_total = nullptr, *d_kps = nullptr, *h_kps = nullptr;
  int *d_band_off = nullptr, *d_band_cnt = nullptr, *h_band = nullptr;   // h_band: [total, off..., cnt...]
  float2 *d_cand = nullptr, *d_cand_ref = nullptr, *h_cand_in = nullptr, *h_cand_out = nullptr;   // fixed stride: cell c at c * nfg
  int *d_cand_cnt = nullptr, *h_cand_cnt = nullptr;
  unsigned *d_sort_scratch = nullptr;
  bool fast_taps = false;                 // the full corner lists were copied back too (debug taps)
  // tracks of the PREVIOUS submitted frame's candidates into this frame (FeContext::track_candidates), by table slot
  float2 *h_sc_pts1 = nullptr, *h_sc_p0n = nullptr, *h_sc_p1n = nullptr;   // pinned
  uint8_t *h_sc_status = nullptr;
  unsigned *d_sc_done = nullptr;
  int sc_prev = -1, sc_ntab = 0, seq_sc = 0;   // slot whose candidates were tracked (-1: none); completion flag h_flags[3]
  cudaEvent_t ev_l0 = nullptr, ev_fast = nullptr;
  cudaEvent_t ev_fast_t[2] = {nullptr, nullptr};
  cudaEvent_t ev_sp_t[2] = {nullptr, nullptr};   // cornerSubPix stage timing
  int *h_flags = nullptr;                 // pinned: [0] FAST done, [1] sub-pixel done, [2] lines done (sequence numbers)
  int seq_fast = 0, seq_subpix = 0, seq_lines = 0;
  std::atomic<int> predet_state{0};        // 0 none, 1 queued, 2 ready, -1 failed
  int predet_nfg = 0, predet_ncell = 0, predet_nb = 0, predet_num_features = -1;
  std::vector<FastCell> cells;            // cell layout this frame's FAST ran on
  std::vector<int> cell_of_loc;
  std::vector<int32_t> cell_kps_tap;       // optional (taps on): every cell's FAST list as (x, y, score), cell_kps_first
  std::vector<int> cell_kps_first;
};

// Occupancy bookkeeping of one top-off detection (TrackKLT.cpp:401-408): the min-distance grid, the per-cell counts and
// the squares that mask0_updated gets around every kept point.
struct OccGrids {
  int d = 1;   // min_px_dist: the min-distance cell size
  int close_w = 0, close_h = 0;
  std::vector<uint8_t> close, grid;
  std::vector<std::pair<int, int>> rects;
  // A new point is added only if its min-distance cell is inside the grid and free; the cell is then taken
  // (TrackKLT.cpp:497-512; stereo: :631-645 left, :779-793 right)
  bool take(const Pt &kp) {
    const int x = (int)(kp.x / (float)d), y = (int)(kp.y / (float)d);
    if (x < 0 || x >= close_w || y < 0 || y >= close_h) return false;
    uint8_t &c = close[(size_t)y * close_w + x];
    if (c > 127) return false;
    c = 255;
    return true;
  }
};

// Results of FeContext::lk_launch in the context's pinned tracking buffers, valid until its next launch
struct LkTracks {
  const float2 *pts1, *p0n, *p1n;
  const uint8_t *status;
};

class FeContext {
 public:
  // model: the FeCameraModel of the camera (ov_core's CamBase subclass), fixed for the context's lifetime
  FeContext(const FeConfig &cfg, int device, int model = FE_CAM_RADTAN);
  ~FeContext();
  int init();  // allocates; returns FeStatus

  // ---- reference-shaped API ----
  int set_calib(const double K[4], const double D[4]);
  int submit(double t, const uint8_t *image, int stride, bool on_device, const uint8_t *mask, int mask_stride,
             const double vp[6]);
  int collect(FeFrameInfo *info);
  int play(int n_frames, const uint8_t *const *images, int stride, bool on_device, const double *timestamps, const double *vps,
           FePlayStats *out);
  int feed(double t, const uint8_t *image, int w, int h, int stride, bool on_device, const uint8_t *mask,
           int mask_stride, const double vp[6], FeFrameInfo *info);

  // results of the last collected frame (TrackBase::get_last_obs / get_last_ids are result().obs / obs_ids)
  const FrameResult &result() const { return *cur_res_; }
  int set_num_features(int n);
  int set_currid(uint64_t id);
  uint64_t currid() const { return currid_; }
  int cand_table_size(int num_features) const;
  int classify_lines(const double vp[6]);
  int change_feat_id(uint64_t id_old, uint64_t id_new);

  int get_state(void *buf, size_t cap, size_t *n_bytes);
  int set_state(const void *buf, size_t n_bytes);
  int tap(int what, void *buf, size_t cap, size_t *n_bytes);

  const FeConfig &cfg() const { return cfg_; }
  int model() const { return model_; }
  static std::string &thread_error();   // error text of the calling thread (what last_error is filled from)
  std::string last_error;
  std::atomic<bool> timing{false};
  std::atomic<bool> taps{false};     // record the debug taps (FAST lists, sub-pixel, LK, FLD) — off on the hot path
  FeStageTimes snapshot_times();
  void reset_times();

  // ---- building blocks for an owner that runs its own point tracker on this context's frames (FeStereo).  Errors
  // leave their text in thread_error() (write_state / load_state: in last_error).
  // Takes a free slot (*slot_out; -1 if none) and enqueues the frame's frame-independent work.  If this fails after a
  // slot was taken, unstage_frame() gives the slot back.
  int stage_frame(double t, const uint8_t *image, int stride, bool on_device, const uint8_t *mask, int mask_stride,
                  const double vp[6], int *slot_out);
  void unstage_frame(int si);   // undoes a staged frame whose submit failed: nothing of it stays pending
  void release_slot(int si) { slots_[si].busy = false; }
  FrameSlot &slot(int si) { return slots_[si]; }
  cudaStream_t track_stream() const { return s_pt_; }
  int flush_line_batch();   // launches the line paths of the frames waiting in the line batch as ONE batch
  // hands a tracked frame to the line tracker thread with the points it is associated against
  void queue_lines(int si, const std::vector<Pt> &pts, const std::vector<uint64_t> &ids);
  // LK of pts from p0 into p1 (initial guess: pts) on track_stream(), in the tracking buffers; lk_wait() waits for it.
  // Launch and wait are separate so that the launches of several contexts run side by side.
  int lk_launch(const Pyramid &p0, const Pyramid &p1, const std::vector<Pt> &pts, const double K[4], const double D[4],
                bool undistort);
  int lk_wait(LkTracks *out);
  // the two halves of the top-off detection that the monocular and the stereo state machines share
  void filter_existing(const std::vector<uint8_t> &mask_test, std::vector<Pt> &pts, std::vector<uint64_t> &ids, std::vector<int> *src,
                       const std::vector<uint64_t> *stereo_ids, OccGrids &g) const;
  int grid_candidates(FrameSlot &slot, const std::vector<uint8_t> &mask_resize, const std::vector<uint8_t> &mask_clone,
                      const OccGrids &g, std::vector<Pt> &ext, std::vector<int> &ext_cand, FrameResult &res);
  void flush_tracker_stats();   // thread that runs the point tracker: lk_launch / grid_candidates statistics
  // State blob (state_blob.h) from point-tracker state passed in (image_slot: the slot holding the previous image, -1
  // none) and this context's line-tracker state; load_state() loads one, the image into a slot, and hands the
  // point-tracker state back.  Only legal while nothing is in flight.
  int write_state(const std::vector<Pt> &pts, const std::vector<uint64_t> &ids, uint64_t currid, int image_slot, void *buf,
                  size_t cap, size_t *n_bytes);
  int load_state(const void *buf, size_t n_bytes, std::vector<Pt> &pts, std::vector<uint64_t> &ids, uint64_t *currid,
                 int *image_slot);

 private:
  int fail(cudaError_t e, const char *what);
  int err(int code, const std::string &msg);
  int collect_impl(FeFrameInfo *info);
  void flush_stats(FeStageTimes &local);
  void klt_main();
  void line_main();
  int wait_flag(volatile int *flag, int value, cudaStream_t st, std::string *err);
  int enqueue_frame_independent(FrameSlot &s);
  int record_image_path(FrameSlot &s, cudaStream_t st);
  int record_fast_path(FrameSlot &s, cudaStream_t st);
  int record_line_path(FrameSlot &s, cudaStream_t st);
  int build_graphs(FrameSlot &s);
  void destroy_graphs(FrameSlot &s);
  void layout_cells();                       // all grid cells of the frame (Grider_GRID geometry)
  int enqueue_fast_all_cells(FrameSlot &s);  // main thread, stream s_det_
  int wait_predetection(FrameSlot &s);
  // TrackKLT
  int klt_feed(FrameSlot &cur);
  int perform_detection(const FrameSlot &img, std::vector<Pt> &pts, std::vector<uint64_t> &ids, std::vector<int> &src,
                        FrameResult &res);
  int perform_matching(const FrameSlot &f0, FrameSlot &f1, std::vector<Pt> &pts0, const std::vector<int> &src, bool spec,
                       std::vector<Pt> &pts1, std::vector<uint8_t> &mask_out, bool &mask_empty, FrameResult &res);
  int speculate(FrameSlot &prev, const float2 *lk_pts, const uint8_t *lk_status, int n);
  int track_candidates(FrameSlot &prev, FrameSlot &s);
  // TrackLSD
  int lsd_feed(FrameSlot &cur);

  FeConfig cfg_;
  int device_;
  int model_;            // FeCameraModel (undistortion of the LK epilogue and of the line rows)
  int W_, H_;            // tracking size (= input size, or half of it with cfg.downsample)
  int Win_, Hin_;        // input size
  cudaStream_t s_pt_ = nullptr;
  std::deque<FrameSlot> slots_;           // deque: FrameSlot holds an atomic and never moves
  std::vector<int> queue_;      // submitted, not yet collected (slot indices, FIFO) — caller's thread only
  int last_slot_ = -1;          // slot of the last COLLECTED frame (kept until the next collect: its rows are exposed)
  int klt_last_slot_ = -1;      // point-tracker thread: slot holding the previous frame's pyramid (img_pyramid_last)
  FrameResult state_res_;       // what result() shows before the first collect / after set_state
  const FrameResult *cur_res_ = &state_res_;
  // ---- the two tracker threads: frames flow submit -> point tracker -> line tracker -> collect, each stage in frame
  // order; the point tracker of frame t+1 overlaps the line association of frame t
  std::thread klt_thread_, line_thread_;
  WorkQueue klt_q_, line_q_;
  FeStageTimes times_{};        // merged statistics (stat_mu_)
  FeStageTimes mst_{}, kst_{}, lst_{};   // per-thread accumulators: caller, point tracker, line tracker

  // ---- point tracker state (TrackBase.h:173-192)
  std::vector<Pt> pts_last_;
  std::vector<uint64_t> ids_last_;
  uint64_t currid_ = 1;
  // ---- line tracker state (TrackLSD.h:248-279)
  std::vector<float4> lines_det_last_;   // cfg.line_samples: the segments detected in the last fed frame (not part of the state blob)
  std::vector<float4> lines_last_;
  std::vector<uint64_t> line_ids_last_;
  std::vector<std::map<int, double>> pol_last_;
  uint64_t line_currid_ = 1;

  // ---- detection: static cell layout + worker
  FastCell *d_cells_ = nullptr;
  GriderLayout cells_;                     // the layout of cells_num_features_
  int cells_num_features_ = -1;
  int max_cells_ = 0, max_bands_ = 0, kps_cap_ = 0, cand_cap_ = 0;
  bool cells_uploaded_ = false;
  int layout_version_ = 0;
  bool use_graphs_ = true;
  int line_batch_ = 1;                  // frames per line-path launch (PLVIWO_LINE_BATCH; 1 = per-frame graph replay)
  std::vector<int> pending_lines_;      // caller's thread: slots whose line path waits for the batch to fill
  std::vector<uint64_t> occ_bits_;
  std::mutex wstat_mu_;
  std::vector<float> sc_px_, sc_py_;      // scratch of the line tracker
  std::vector<uint8_t> sc_pass_;
  std::vector<std::pair<int, int>> sc_inv_;
  std::vector<int> sc_shared_, sc_touched_;
  // ---- tracking scratch
  int max_pts_ = 0;
  unsigned *d_lk_done_ = nullptr;   // features finished in the running LK launches (completion signals) [ordinary, speculative]
  // ---- speculative tracking (FeContext::speculate): LK(t -> t+1) for every point that may be tracked, launched before
  // frame t's RANSAC gate
  float2 *h_sp_pts0_ = nullptr, *h_sp_pts1_ = nullptr, *h_sp_p0n_ = nullptr, *h_sp_p1n_ = nullptr;   // pinned
  uint8_t *h_sp_status_ = nullptr;
  static constexpr int kCandBase = 1 << 24;   // src >= kCandBase: result of candidate table slot (src - kCandBase)
  int prev_submit_slot_ = -1;                 // caller's thread: slot of the frame submitted last
  int spec_n_ = 0, seq_sp_ = 0;
  int spec_prev_slot_ = -1, spec_next_slot_ = -1;
  bool spec_valid_ = false, spec_timed_ = false, use_spec_ = true;
  std::vector<int> spec_of_lk_;     // per point of this frame's LK arrays: its index in the speculative launch, or -1
  std::vector<int> last_src_;       // parallel to pts_last_: the same for the surviving points
  std::vector<int> lk2_;            // points that go through the ordinary launch
  std::vector<float2> a_pts1_, a_p0n_, a_p1n_;   // this frame's tracking results in the reference's order
  std::vector<uint8_t> a_status_;
  float2 *h_pts0_ = nullptr, *h_pts1_ = nullptr, *h_p0n_ = nullptr, *h_p1n_ = nullptr;
  uint8_t *h_status_ = nullptr;
  cudaEvent_t ev_pt_[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  int *h_flag_lk_ = nullptr;
  int seq_lk_ = 0;
  int cur_slot_ = -1;
};

}  // namespace plviwo
