// Stereo point tracker: ov_core::TrackKLT with use_stereo = true fed two images per message
// (open_vins/ov_core/src/track/TrackKLT.cpp:202-393 feed_stereo, :530-827 perform_detection_stereo).
// One FeStereo = one stereo rig on one device.  It owns two FeContext objects and stages each camera's frames in one of
// them — each runs the frame-independent pipeline of one camera (copy, equalise, pyramid, FAST on every cell, std::sort +
// top-k, cornerSubPix) on its own streams at submit() — and runs the stereo state machine itself on its tracker thread.
#pragma once
#include <atomic>
#include <deque>
#include <memory>
#include <thread>
#include <string>
#include <utility>
#include <vector>

#include "fe_context.h"

namespace plviwo {

class FeStereo {
 public:
  // model: the FeCameraModel of both cameras, fixed for the rig's lifetime
  FeStereo(const FeConfig &cfg, const double K_right[4], const double D_right[4], int device, int model = FE_CAM_RADTAN);
  ~FeStereo();
  int init();
  int model() const { return cam_[0]->model(); }

  int set_calib(int cam, const double K[4], const double D[4]);
  int set_num_features(int n);
  int change_feat_id(uint64_t id_old, uint64_t id_new);
  int submit(double t, const uint8_t *const image[2], int stride, bool on_device, const uint8_t *const mask[2], int mask_stride,
             const double vp[6]);
  int collect(FeStereoInfo *info);
  int feed(double t, const uint8_t *const image[2], int w, int h, int stride, bool on_device, const uint8_t *const mask[2],
           int mask_stride, const double vp[6], FeStereoInfo *info);
  int get_state(void *buf, size_t cap, size_t *n_bytes);
  int set_state(const void *buf, size_t n_bytes);
  FeStageTimes snapshot_times(bool reset);

  // results of the last collected pair
  const std::vector<FePointRow> &rows(int cam) const { return rows_[cam]; }
  const std::vector<Pt> &last_obs(int cam) const { return obs_[cam]; }
  const std::vector<uint64_t> &last_ids(int cam) const { return obs_ids_[cam]; }
  const FrameResult &left_result() const { return *left_res_; }   // line rows / line points of the left image
  int classify_lines(const double vp[6]);
  std::string last_error;

 private:
  struct Match {   // one perform_matching call (TrackKLT.cpp:829-886)
    int n = 0;
    bool launched = false, mask_empty = true;
    std::vector<Pt> pts1;
    std::vector<uint8_t> mask;
    std::vector<float2> p1n;
  };
  // One submitted pair: where its images live, and what the tracker thread hands back for it
  struct Pair {
    int slot[2] = {-1, -1};
    double t = 0;
    FeStereoInfo info{};
    std::vector<FePointRow> rows[2];
    std::vector<Pt> obs[2];              // pts_last / ids_last after the pair (TrackBase::get_last_obs / get_last_ids)
    std::vector<uint64_t> obs_ids[2];
    int rc = FE_OK;
    std::string error;
    bool lines_queued = false;           // the left frame went to the line thread (its slot's stage reaches 3 when done)
    std::atomic<int> stage{0};           // 0 free, 1 submitted, 2 tracked (point results complete)
  };
  int err(int code, const std::string &msg);
  void track_main();
  int collect_impl(Pair &p);
  int detection_stereo(FrameSlot &L, FrameSlot &R, std::vector<Pt> &pts0, std::vector<Pt> &pts1, std::vector<uint64_t> &ids0,
                       std::vector<uint64_t> &ids1, FeStereoInfo &info);
  int matching_begin(int cam, FrameSlot &f0, FrameSlot &f1, const std::vector<Pt> &pts0, Match &m);
  int matching_end(int cam, FrameSlot &f1, const std::vector<Pt> &pts0, Match &m, FeStereoInfo &info);

  FeConfig cfg_;
  int device_;
  std::unique_ptr<FeContext> cam_[2];
  // submit() -> tracker thread -> collect(), pairs in order.  The tracker thread owns the tracker state while pairs are
  // in flight; the state is only touched from the caller's thread when nothing is pending (setters, state blobs).
  std::vector<std::unique_ptr<Pair>> ring_;  // lookahead + 2 records
  std::deque<int> queue_;                    // caller's thread: ring indices submitted, not yet collected
  std::thread worker_;
  WorkQueue work_q_;
  int last_[2] = {-1, -1};                   // tracker thread: slots holding the previous pair (img_pyramid_last)
  int released_[2] = {-1, -1};               // caller's thread: slots of the last COLLECTED pair (freed at the next collect)
  // tracker state (TrackBase.h:173-192; one currid for both cameras)
  std::vector<Pt> pts_last_[2];
  std::vector<uint64_t> ids_last_[2];
  uint64_t currid_ = 1;
  std::vector<FePointRow> rows_[2];          // of the last collected pair
  std::vector<Pt> obs_[2];
  std::vector<uint64_t> obs_ids_[2];
  FrameResult *left_res_ = &no_lines_;      // the left image's result of the last collected pair
  FrameResult no_lines_;                     // ... before the first collect and after set_state
  FrameResult scratch_res_;
  FeStageTimes st_{};
};

}  // namespace plviwo
