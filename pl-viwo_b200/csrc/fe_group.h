// Stream group: many camera streams of one device tracked together (BASELINE.json configs[4], "multi-session batch
// throughput").  Each stream is what one FeContext is — one ov_core::TrackKLT + one viw::TrackLSD for one camera, same
// results bit for bit — but
//   * the state-independent work of a frame of EVERY stream (equalise, pyramid, Canny, connected components, chain walk,
//     segments) is one set of launches per tick (grid.z = stream), and
//   * the tracker state (pts_last / ids_last / currid, lines_last / point_on_lines_last) lives in device memory and the
//     state machine of a frame (top-off detection on the previous image, with FAST + std::sort / top-k + cornerSubPix on
//     the cells it leaves open, LK, RANSAC gate, row filter, line association) is one set of launches per tick for all
//     streams (kernels_glue.cu, kernels_fast.cu, k_lk15w_g) — no host thread sees a feature before the
//     rows of the frame are complete in pinned host memory.
// The caller's thread only enqueues launches (submit) and waits for a tick's completion event (collect).
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <string>
#include <vector>

#include "../../include/plviwo_fe.h"
#include "fe_group_dev.h"

namespace plviwo {

class FeGroup {
 public:
  FeGroup(const FeConfig &cfg, int n_streams, int device);
  ~FeGroup();
  int init();

  int n_streams() const { return S_; }
  const FeConfig &cfg() const { return cfg_; }
  int set_calib(int stream, const double K[4], const double D[4]);
  // One tick: a frame of every stream whose images[s] is not null.  vps: 6 doubles per stream (all streams) or null (the line
  // tracker is not fed); masks: per-stream host pointers or null.
  int submit(const double *timestamps, const uint8_t *const *images, int stride, bool on_device, const uint8_t *const *masks,
             int mask_stride, const double *vps);
  int collect(FeFrameInfo *infos);   // the oldest submitted tick; infos: n_streams entries or null
  int play(int n_ticks, const uint8_t *const *images, int stride, bool on_device, const double *timestamps, const double *vps,
           FePlayStats *out);
  int in_flight() const { return submitted_ - collected_; }

  // results of the last collected tick (valid until the next collect)
  const GroupOutHeader *header(int stream) const;
  const FePointRow *point_rows(int stream) const;
  const uint64_t *obs_ids(int stream) const;
  const float *obs_uv(int stream) const;
  const FeLineRow *line_rows(int stream) const;
  const FeLinePoint *line_points(int stream) const;
  // cfg.line_samples: u0 v0 u1 v1 and status per sample, as plviwo_fe_get_line_samples
  int line_samples(int stream, float *uv01, uint8_t *status, int cap, int *n_out) const;

  int get_state(int stream, void *buf, size_t cap, size_t *n_bytes);
  int set_state(int stream, const void *buf, size_t n_bytes);
  int tap(int stream, int what, void *buf, size_t cap, size_t *n_bytes);

  void enable_timing(bool on) { timing_ = on; }
  FeGroupTimes times(bool reset);
  std::string last_error;

 private:
  struct TickRec {
    int ring = 0;                       // output / job ring entry
    std::vector<int> cur_slot;          // per stream: global slot index of the frame, -1 none
    bool track_launched = false;
    int batch = -1;                     // front batch the tick belongs to
  };
  struct FrontBatch {
    std::vector<FrontJob> jobs;
    std::vector<int> line_slots;
    std::vector<int> ticks;             // tick numbers carried
    bool launched = false;
  };
  int fail(cudaError_t e, const char *what);
  int err(int code, const std::string &msg);
  int alloc_image(DevImage &im, int w, int h);
  void layout_cells();
  int flush_front();                     // launches the pending front batch and the tracking of its ticks
  int launch_front(FrontBatch &b, int buf);
  int launch_track(int tick);
  int ensure_mask_buffer(int slot);
  void account(int k, cudaEvent_t a, cudaEvent_t b, int frames);

  FeConfig cfg_;
  int S_, device_, W_, H_;
  int la_ = 0, R_ = 2, RB_ = 2, B_ = 1, lanes_ = 1;
  std::vector<double> K_, D_;            // per stream, 4 each
  // ---- device data
  GroupDev g_{};
  FrontGeom fg_{};
  std::vector<SlotRec> slots_;           // host copy of the table (S * R entries, stream-major)
  SlotRec *d_slots_ = nullptr;
  int *d_slot_flags_ = nullptr;
  FastCell *d_cells_ = nullptr;
  std::vector<FastCell> cells_;
  int cells_nb_ = 0, cells_csx_ = 0, cells_csy_ = 0;
  std::vector<void *> dev_allocs_, host_allocs_;
  std::vector<uint8_t *> h_raw_;         // pinned staging per slot for pageable host frames (lazy)
  std::vector<uint8_t *> h_mask_;        // pinned staging per slot (lazy)
  uint8_t *h_out_ = nullptr;             // pinned output ring: record (ring * S + stream)
  // job rings: pinned + device, entry = ring index
  FrontJob *h_fjobs_ = nullptr, *d_fjobs_ = nullptr;   // RB * B * S
  int *h_ljobs_ = nullptr, *d_ljobs_ = nullptr;        // RB * B * S
  TrackJob *h_tjobs_ = nullptr, *d_tjobs_ = nullptr;   // RB * S
  std::vector<cudaStream_t> s_copy_;                   // frames go in round-robin over a few copy streams (a 0.7 MB copy has a fixed cost that only overlaps across streams)
  unsigned copy_rr_ = 0;
  // PLVIWO_GROUP_TRACE=1: device-side latency of every front batch (first kernel .. segments) and the interval between
  // consecutive batches, printed when the group is destroyed (diagnostics; two timed events per batch)
  bool trace_ = false;
  std::vector<cudaEvent_t> ev_tr0_, ev_tr1_, ev_trs_;   // ev_trs_: 4 per batch (after the pyramid, Canny + tiles, components, walk)
  double tr_stage_ms_[5] = {0, 0, 0, 0, 0};
  double tr_host_copy_us_ = 0, tr_host_submit_us_ = 0, tr_host_wait_us_ = 0;   // host time: issuing the frame copies, the whole of submit, waiting in collect
  long tr_host_ticks_ = 0;
  std::vector<char> tr_valid_;
  int tr_prev_ = -1;
  double tr_lat_ms_ = 0, tr_period_ms_ = 0, tr_lane_ms_ = 0;
  long tr_n_ = 0, tr_np_ = 0;
  std::vector<int> prev_rec_;                          // per stream: the state record that holds its pts_last (fe_group_dev.h)
  std::vector<cudaStream_t> s_front_, s_track_, s_lines_;
  std::vector<cudaEvent_t> ev_gate_;                   // per ring entry * lanes: the point chain of the tick is done
  std::vector<cudaEvent_t> ev_copy_, ev_front_, ev_pyr_;   // per front-batch buffer (ev_pyr_: the batch's pyramids are built)
  std::vector<cudaEvent_t> ev_done_;                   // per ring entry * lanes
  std::vector<cudaEvent_t> ev_lane_prev_;              // per lane: previous tick's tracking done (front may reuse its slots)
  // ---- bookkeeping (caller's thread)
  std::vector<long long> frame_count_;
  std::vector<int> prev_slot_;
  long long submitted_ = 0, collected_ = 0, batch_seq_ = 0;
  std::vector<TickRec> ticks_;           // ring of RB entries indexed by tick % RB
  std::vector<FrontBatch> batches_;      // ring of RB entries
  int pending_batch_ = -1;               // batch being filled (index into batches_)
  long long last_collected_ = -1;
  // ---- timing
  bool timing_ = false;
  FeGroupTimes times_{};
  struct TimedLaunch { int k; cudaEvent_t a, b; int frames; };
  std::vector<TimedLaunch> timed_;
  std::vector<cudaEvent_t> ev_pool_;
  size_t ev_next_ = 0;
  cudaEvent_t timing_event();
  int drain_timing();
  uint64_t launches_ = 0, h2d_bytes_ = 0, d2h_bytes_ = 0, frames_done_ = 0, fast_cells_base_ = 0;
};

}  // namespace plviwo
