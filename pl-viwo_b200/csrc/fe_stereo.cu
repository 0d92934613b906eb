// Stereo point tracker.  Line-by-line counterpart of the reference's stereo glue with every OpenCV call replaced by a
// kernel launch:
//   ov_core::TrackKLT::feed_new_camera (two images)   open_vins/ov_core/src/track/TrackKLT.cpp:34-94
//   TrackKLT::feed_stereo                             TrackKLT.cpp:202-393
//   TrackKLT::perform_detection_stereo                TrackKLT.cpp:530-827
//   TrackKLT::perform_matching                        TrackKLT.cpp:829-886
// Per pair: the frame-independent work of BOTH images is enqueued at submit() by the two per-camera contexts (their own
// streams, CUDA graphs); collect() runs the state machine: top-off detection on the previous pair (left, then a
// left->right LK launch for the new points, then right), the two temporal LK launches side by side on two streams,
// the two RANSAC gates, and the left/right merge.
#include "fe_stereo.h"
#include "state_blob.h"

#include <algorithm>
#include <cmath>
#include <cstring>

namespace plviwo {

#define ST_CUDA(call)                                                             \
  do {                                                                            \
    cudaError_t e__ = (call);                                                     \
    if (e__ != cudaSuccess) return err(FE_CUDA_ERROR, std::string(#call) + ": " + cudaGetErrorString(e__)); \
  } while (0)

FeStereo::FeStereo(const FeConfig &cfg, const double K_right[4], const double D_right[4], int device, int model)
    : cfg_(cfg), device_(device) {
  cfg_.line_samples = 0;
  cfg_.downsample = 0;
  FeConfig cr = cfg_;
  cr.use_lines = 0;   // TrackLSD.cpp:57-60: with two images the line tracker runs on the left one only
  for (int i = 0; i < 4; i++) {
    if (K_right) cr.K[i] = K_right[i];
    if (D_right) cr.D[i] = D_right[i];
  }
  cam_[0].reset(new FeContext(cfg_, device, model));
  cam_[1].reset(new FeContext(cr, device, model));
  currid_ = 4 * (uint64_t)cfg.numaruco + 1;   // TrackBase.cpp:34
}

FeStereo::~FeStereo() {
  if (worker_.joinable()) {
    cudaSetDevice(device_);
    cam_[0]->flush_line_batch();   // the tracker thread may be waiting for the line result of an unlaunched batch
    work_q_.stop();
    worker_.join();
  }
}

// error text of the calling thread; the tracker thread's ends up in the pair's record, the caller's in last_error
static thread_local std::string t_serr;
static thread_local bool t_on_worker = false;

int FeStereo::err(int code, const std::string &msg) {
  t_serr = msg;
  if (!t_on_worker) last_error = msg;
  return code;
}

int FeStereo::init() {
  for (int c = 0; c < 2; c++) {
    int rc = cam_[c]->init();
    if (rc) return err(rc, cam_[c]->last_error.empty() ? FeContext::thread_error() : cam_[c]->last_error);
  }
  const int n = std::max(cfg_.lookahead, 0) + 2;
  for (int i = 0; i < n; i++) ring_.emplace_back(new Pair());
  worker_ = std::thread([this] { track_main(); });
  return FE_OK;
}

int FeStereo::set_calib(int cam, const double K[4], const double D[4]) {
  if (cam < 0 || cam > 1) return err(FE_BAD_ARG, "set_calib: cam must be 0 (left) or 1 (right)");
  return cam_[cam]->set_calib(K, D);
}

int FeStereo::set_num_features(int n) {
  if (!queue_.empty()) return err(FE_BAD_ARG, "set_num_features: collect the pending pairs first");
  // both cameras have the same image size, grid and capacity: the right one accepts what the left one accepts
  if (cam_[0]->set_num_features(n) || cam_[1]->set_num_features(n))
    return err(FE_BAD_ARG, "set_num_features: the candidate table of that feature count exceeds the capacity this rig was created with");
  cfg_.num_features = n;
  return FE_OK;
}

int FeStereo::classify_lines(const double vp[6]) {
  for (FeLineRow &row : left_res_->line_rows) row.D = line_classification(make_float4(row.line[0], row.line[1], row.line[2], row.line[3]), vp);
  return FE_OK;
}

int FeStereo::change_feat_id(uint64_t id_old, uint64_t id_new) {   // TrackBase.cpp:267-285 (tracker side)
  if (!queue_.empty()) return err(FE_BAD_ARG, "change_feat_id: collect the pending pairs first");
  for (int c = 0; c < 2; c++) {
    for (uint64_t &id : ids_last_[c])
      if (id == id_old) id = id_new;
    for (uint64_t &id : obs_ids_[c])   // keep get_last_ids in step
      if (id == id_old) id = id_new;
  }
  return FE_OK;
}

int FeStereo::submit(double t, const uint8_t *const image[2], int stride, bool on_device, const uint8_t *const mask[2],
                     int mask_stride, const double vp[6]) {
  int ri = -1;
  for (int i = 0; i < (int)ring_.size(); i++)
    if (ring_[i]->stage.load(std::memory_order_acquire) == 0 && std::find(queue_.begin(), queue_.end(), i) == queue_.end()) {
      ri = i;
      break;
    }
  if (ri < 0) return err(FE_BAD_ARG, "submit: lookahead window full (collect a pair first)");
  int slot[2] = {-1, -1};
  for (int c = 0; c < 2; c++) {
    int rc = cam_[c]->stage_frame(t, image[c], stride, on_device, mask ? mask[c] : nullptr, mask_stride, c == 0 ? vp : nullptr,
                                  &slot[c]);
    if (rc) {   // a failed submit leaves no trace: neither image stays staged
      for (int k = 0; k <= c; k++)
        if (slot[k] >= 0) cam_[k]->unstage_frame(slot[k]);
      return err(rc, FeContext::thread_error());
    }
  }
  Pair &p = *ring_[ri];
  p.slot[0] = slot[0];
  p.slot[1] = slot[1];
  p.t = t;
  p.rc = FE_OK;
  p.error.clear();
  std::memset(&p.info, 0, sizeof(p.info));
  p.info.timestamp = t;
  queue_.push_back(ri);
  p.stage.store(1, std::memory_order_release);
  work_q_.push(ri);
  return FE_OK;
}

int FeStereo::feed(double t, const uint8_t *const image[2], int w, int h, int stride, bool on_device, const uint8_t *const mask[2],
                   int mask_stride, const double vp[6], FeStereoInfo *info) {
  // TrackKLT.cpp:37-43 exits on a malformed message
  if (!image || !image[0] || !image[1] || w != cfg_.width || h != cfg_.height || stride < w ||
      (mask && (mask[0] || mask[1]) && mask_stride < w))
    return err(FE_BAD_ARG, "feed: image/mask size does not match the handle");
  if (!queue_.empty()) return err(FE_BAD_ARG, "feed: pairs submitted with plviwo_fe_stereo_submit are still pending");
  int rc = submit(t, image, stride, on_device, mask, mask_stride, vp);
  if (rc) return rc;
  return collect(info);
}

// Tracker thread: pairs in submission order.  Owns pts_last_ / ids_last_ / currid_ / last_ while pairs are in flight.
void FeStereo::track_main() {
  t_on_worker = true;
  cudaSetDevice(device_);
  int ri;
  while (work_q_.pop(&ri)) {
    Pair &p = *ring_[ri];
    int rc = collect_impl(p);
    for (int c = 0; c < 2; c++) {
      p.obs[c] = pts_last_[c];
      p.obs_ids[c] = ids_last_[c];
      p.info.n_point_rows[c] = (int)p.rows[c].size();
      p.info.n_last_obs[c] = (int)pts_last_[c].size();
    }
    // UpdaterCamera.cpp:105-110: the line tracker runs after the point tracker, on the LEFT image, against the left points
    // the stereo tracker has just produced (TrackLSD.cpp:57-60, :127-129): hand the frame to the left context's line
    // thread (the association of pair t overlaps the tracking of pair t + 1).  Its line path was launched by the
    // caller's thread (at submit, or by collect() when the batch never filled).
    p.lines_queued = false;
    if (rc == FE_OK && cfg_.use_lines && cam_[0]->slot(p.slot[0]).has_vp) {
      p.lines_queued = true;
      cam_[0]->queue_lines(p.slot[0], pts_last_[0], ids_last_[0]);
    }
    for (int c = 0; c < 2; c++) cam_[c]->flush_tracker_stats();
    last_[0] = p.slot[0];   // move forward in time whatever happened (:366-378)
    last_[1] = p.slot[1];
    p.rc = rc;
    if (rc) p.error = t_serr;
    p.stage.store(2, std::memory_order_release);
  }
}

int FeStereo::collect(FeStereoInfo *info) {
  if (cudaSetDevice(device_) != cudaSuccess) return err(FE_CUDA_ERROR, "cudaSetDevice failed");
  if (queue_.empty()) return err(FE_BAD_ARG, "collect: nothing submitted");
  const int ri = queue_.front();
  Pair &p = *ring_[ri];
  FrameSlot &L = cam_[0]->slot(p.slot[0]);
  if (L.line_pending) {   // its line batch never filled up: launch what is there
    int rc = cam_[0]->flush_line_batch();
    if (rc) return err(rc, FeContext::thread_error());
  }
  for (unsigned spins = 0; p.stage.load(std::memory_order_acquire) != 2; spins++) {
    if (spins < 256) {
#if defined(__x86_64__)
      __builtin_ia32_pause();
#endif
    } else {
      std::this_thread::yield();
    }
  }
  if (p.lines_queued) {   // ... and for the line thread
    for (unsigned spins = 0; L.stage.load(std::memory_order_acquire) != 3; spins++) {
      if (spins >= 256) std::this_thread::yield();
    }
    L.stage.store(0, std::memory_order_relaxed);
    p.info.n_line_rows = (int)L.res.line_rows.size();
    p.info.n_lines_detected = L.res.info.n_lines_detected;
    p.info.n_line_matches = L.res.info.n_line_matches;
    if (L.res.rc && p.rc == FE_OK) {
      p.rc = L.res.rc;
      p.error = L.res.error;
    }
  }
  queue_.pop_front();
  for (int c = 0; c < 2; c++) {
    rows_[c].swap(p.rows[c]);
    obs_[c].swap(p.obs[c]);
    obs_ids_[c].swap(p.obs_ids[c]);
  }
  left_res_ = &L.res;   // line rows / line points of the left image (plviwo_fe_stereo_get_line_rows)
  // the previous collected pair's slots become free: its pyramids are no longer the tracker's "last" pair (the tracker
  // finished THIS pair, which was the last one to read them)
  for (int c = 0; c < 2; c++) {
    if (released_[c] >= 0) cam_[c]->release_slot(released_[c]);
    released_[c] = p.slot[c];
  }
  st_.frames++;
  if (info) *info = p.info;
  const int rc = p.rc;
  if (rc) last_error = p.error;
  p.stage.store(0, std::memory_order_release);
  return rc;
}

// TrackKLT.cpp:829-868: the launch half ...
int FeStereo::matching_begin(int cam, FrameSlot &f0, FrameSlot &f1, const std::vector<Pt> &pts0, Match &m) {
  m = Match();
  m.n = (int)pts0.size();
  m.pts1 = pts0;
  if (m.n == 0) return FE_OK;        // :836-837 (mask stays empty)
  m.mask_empty = false;
  m.mask.assign(m.n, 0);
  if (m.n < 10) return FE_OK;        // :848-852
  int rc = cam_[cam]->lk_launch(f0.pyr, f1.pyr, pts0, f1.K, f1.D, true);
  if (rc) return err(rc, FeContext::thread_error());
  m.launched = true;
  return FE_OK;
}

// ... and the gate half (:869-885)
int FeStereo::matching_end(int cam, FrameSlot &f1, const std::vector<Pt> &pts0, Match &m, FeStereoInfo &info) {
  (void)pts0;
  if (!m.launched) return FE_OK;
  LkTracks c;
  int rc = cam_[cam]->lk_wait(&c);
  if (rc) return err(rc, FeContext::thread_error());
  const int n = m.n;
  const double max_focal = std::max(f1.K[0], f1.K[1]);   // id0 == id1 for the temporal tracks
  std::vector<uint8_t> mask_rsc(n, 0);
  int mask_valid = 0;
  const int n_in = ransac_fundamental(reinterpret_cast<const float *>(c.p0n), reinterpret_cast<const float *>(c.p1n), n,
                                      2.0 / max_focal, 0.999, mask_rsc.data(), &mask_valid);
  m.p1n.assign(c.p1n, c.p1n + n);
  int n_klt = 0;
  for (int i = 0; i < n; i++) {
    m.mask[i] = (c.status[i] && mask_valid && mask_rsc[i]) ? 1 : 0;
    n_klt += c.status[i] ? 1 : 0;
    m.pts1[i] = Pt{c.pts1[i].x, c.pts1[i].y};
  }
  info.n_lk_in[cam] = n;
  info.n_klt_ok[cam] = n_klt;
  info.n_ransac_ok[cam] = n_in;
  return FE_OK;
}

// ------------------------------------------------------------------------------------ perform_detection_stereo
int FeStereo::detection_stereo(FrameSlot &L, FrameSlot &R, std::vector<Pt> &pts0, std::vector<Pt> &pts1, std::vector<uint64_t> &ids0,
                               std::vector<uint64_t> &ids1, FeStereoInfo &info) {
  const int cols = cfg_.width, rows = cfg_.height;
  const int thr = std::min(20, (int)(0.50 * cfg_.num_features));
  std::vector<Pt> ext;
  std::vector<int> ext_cand;
  // ---- LEFT (:537-682)
  OccGrids g0;
  cam_[0]->filter_existing(L.mask, pts0, ids0, nullptr, nullptr, g0);
  if (cfg_.num_features - (int)pts0.size() > thr) {   // :606 (strictly greater; the monocular path uses >=)
    info.detection_ran[0] = 1;
    int rc = cam_[0]->grid_candidates(L, L.mask, L.mask, g0, ext, ext_cand, scratch_res_);
    if (rc) return err(rc, FeContext::thread_error());
    std::vector<Pt> new0;
    for (const Pt &kp : ext)   // :631-645
      if (g0.take(kp)) new0.push_back(kp);
    if (!new0.empty()) {
      // left -> right KLT of the new points, initial guess = the left position, no RANSAC gate (:658-666)
      LkTracks c;
      rc = cam_[0]->lk_launch(L.pyr, R.pyr, new0, L.K, L.D, false);
      if (rc == FE_OK) rc = cam_[0]->lk_wait(&c);
      if (rc) return err(rc, FeContext::thread_error());
      for (size_t i = 0; i < new0.size(); i++) {   // :669-699
        const Pt p0 = new0[i];
        const Pt p1 = Pt{c.pts1[i].x, c.pts1[i].y};
        const bool oob_left = (int)p0.x < 0 || (int)p0.x >= cols || (int)p0.y < 0 || (int)p0.y >= rows;
        const bool oob_right = (int)p1.x < 0 || (int)p1.x >= cols || (int)p1.y < 0 || (int)p1.y >= rows;
        if (!oob_left && !oob_right && c.status[i] == 1) {
          const uint64_t id = ++currid_;
          pts0.push_back(p0);
          pts1.push_back(p1);
          ids0.push_back(id);
          ids1.push_back(id);
          info.n_detected[0]++;
          info.n_stereo_new++;
        } else if (!oob_left) {
          pts0.push_back(p0);
          ids0.push_back(++currid_);
          info.n_detected[0]++;
        }
      }
    }
  }
  // ---- RIGHT (:684-826).  A right point on an occupied min-distance cell survives if its id is also in the left image
  // (:720-726); the working mask starts as a clone of the LEFT mask (:691)
  OccGrids g1;
  cam_[1]->filter_existing(R.mask, pts1, ids1, nullptr, &ids0, g1);
  if (cfg_.num_features - (int)pts1.size() > thr) {   // :753
    info.detection_ran[1] = 1;
    int rc = cam_[1]->grid_candidates(R, R.mask, L.mask, g1, ext, ext_cand, scratch_res_);
    if (rc) return err(rc, FeContext::thread_error());
    for (const Pt &kp : ext) {   // :779-793
      if (!g1.take(kp)) continue;
      pts1.push_back(kp);
      ids1.push_back(++currid_);
      info.n_detected[1]++;
    }
  }
  return FE_OK;
}

// ------------------------------------------------------------------------------------------------ feed_stereo
int FeStereo::collect_impl(Pair &pair) {
  FeStereoInfo *info = &pair.info;
  FrameSlot &L = cam_[0]->slot(pair.slot[0]), &R = cam_[1]->slot(pair.slot[1]);
  std::vector<FePointRow> *rows_out = pair.rows;
  rows_out[0].clear();
  rows_out[1].clear();
  // every tracking stream may read either image of the pair (the left->right launch runs on the left stream)
  for (int c = 0; c < 2; c++) {
    ST_CUDA(cudaStreamWaitEvent(cam_[c]->track_stream(), L.ev_pyr, 0));
    ST_CUDA(cudaStreamWaitEvent(cam_[c]->track_stream(), R.ev_pyr, 0));
  }
  const int cols = cfg_.width, rows = cfg_.height;
  // :221-241 — nothing tracked last time: detect on the CURRENT pair only
  if ((pts_last_[0].empty() && pts_last_[1].empty()) || last_[0] < 0 || last_[1] < 0) {
    std::vector<Pt> gl, gr;
    std::vector<uint64_t> il, ir;
    int rc = detection_stereo(L, R, gl, gr, il, ir, *info);
    if (rc) return rc;
    pts_last_[0] = gl; pts_last_[1] = gr;
    ids_last_[0] = il; ids_last_[1] = ir;
    info->first_frame = 1;
    return FE_OK;
  }
  FrameSlot &L0 = cam_[0]->slot(last_[0]), &R0 = cam_[1]->slot(last_[1]);
  // top-off on the PREVIOUS pair (:245-252)
  std::vector<Pt> pl_old = pts_last_[0], pr_old = pts_last_[1];
  std::vector<uint64_t> il_old = ids_last_[0], ir_old = ids_last_[1];
  int rc = detection_stereo(L0, R0, pl_old, pr_old, il_old, ir_old, *info);
  if (rc) return rc;
  // temporal tracking of both cameras (:261-270): two launches on two streams, then the two gates
  Match ml, mr;
  rc = matching_begin(0, L0, L, pl_old, ml);
  if (rc) return rc;
  rc = matching_begin(1, R0, R, pr_old, mr);
  if (rc) return rc;
  rc = matching_end(0, L, pl_old, ml, *info);
  if (rc) return rc;
  rc = matching_end(1, R, pr_old, mr, *info);
  if (rc) return rc;
  if (ml.mask_empty && mr.mask_empty) {   // :286-300
    pts_last_[0].clear(); pts_last_[1].clear();
    ids_last_[0].clear(); ids_last_[1].clear();
    info->reset = 1;
    return FE_OK;
  }
  std::vector<Pt> good_l, good_r;
  std::vector<uint64_t> gid_l, gid_r;
  auto push_row = [&](int cam, uint64_t id, const Pt &p, const Match &m, size_t i) {
    // :352-363 — undistort_cv(pt) of a tracked point is the p1n the LK epilogue produced; a point of a matching call
    // that never launched (fewer than 10 points) has an all-zero mask and never gets here
    FePointRow r;
    r.id = id;
    r.u = p.x;
    r.v = p.y;
    r.un = m.p1n[i].x;
    r.vn = m.p1n[i].y;
    rows_out[cam].push_back(r);
  };
  std::vector<std::pair<size_t, size_t>> row_src[2];   // (index into the matching call) per good point, for the rows
  for (size_t i = 0; i < ml.pts1.size(); i++) {   // :298-334
    const Pt &p = ml.pts1[i];
    if (p.x < 0 || p.y < 0 || (int)p.x > cols || (int)p.y > rows) continue;   // '>' as in the reference (:302-303)
    bool found_right = false;
    size_t index_right = 0;
    for (size_t n = 0; n < ir_old.size(); n++)
      if (il_old[i] == ir_old[n]) {
        found_right = true;
        index_right = n;
        break;
      }
    if (ml.mask[i] && found_right && !mr.mask_empty && mr.mask[index_right]) {
      const Pt &q = mr.pts1[index_right];
      if (q.x < 0 || q.y < 0 || (int)q.x >= cols || (int)q.y >= rows) continue;
      good_l.push_back(p);
      good_r.push_back(q);
      gid_l.push_back(il_old[i]);
      gid_r.push_back(ir_old[index_right]);
      row_src[0].emplace_back(i, 0);
      row_src[1].emplace_back(index_right, 0);
      info->n_stereo_rows++;
    } else if (ml.mask[i]) {
      good_l.push_back(p);
      gid_l.push_back(il_old[i]);
      row_src[0].emplace_back(i, 0);
    }
  }
  for (size_t i = 0; i < mr.pts1.size(); i++) {   // :337-349
    const Pt &q = mr.pts1[i];
    if (q.x < 0 || q.y < 0 || (int)q.x >= cols || (int)q.y >= rows) continue;
    const bool added_already = std::find(gid_r.begin(), gid_r.end(), ir_old[i]) != gid_r.end();
    if (mr.mask[i] && !added_already) {
      good_r.push_back(q);
      gid_r.push_back(ir_old[i]);
      row_src[1].emplace_back(i, 0);
    }
  }
  for (size_t k = 0; k < good_l.size(); k++) push_row(0, gid_l[k], good_l[k], ml, row_src[0][k].first);
  for (size_t k = 0; k < good_r.size(); k++) push_row(1, gid_r[k], good_r[k], mr, row_src[1][k].first);
  pts_last_[0] = good_l; pts_last_[1] = good_r;
  ids_last_[0] = gid_l; ids_last_[1] = gid_r;
  return FE_OK;
}

// ------------------------------------------------------------------------------------------------ state

int FeStereo::get_state(void *buf, size_t cap, size_t *n_bytes) {
  if (!queue_.empty()) return err(FE_BAD_ARG, "get_state: collect the pending pairs first");
  size_t sz[2] = {0, 0};
  for (int c = 0; c < 2; c++) {
    int rc = cam_[c]->write_state(pts_last_[c], ids_last_[c], currid_, last_[c], nullptr, 0, &sz[c]);
    if (rc) return err(rc, cam_[c]->last_error);
  }
  const size_t need = sizeof(StereoStateHeader) + sz[0] + sz[1];
  if (n_bytes) *n_bytes = need;
  if (!buf) return FE_OK;
  if (cap < need) return FE_OVERFLOW;
  StereoStateHeader hd;
  hd.magic = kStereoStateMagic;
  hd.version = kStereoStateVersion;
  hd.currid = currid_;
  hd.size[0] = sz[0];
  hd.size[1] = sz[1];
  uint8_t *p = static_cast<uint8_t *>(buf);
  std::memcpy(p, &hd, sizeof(hd));
  p += sizeof(hd);
  for (int c = 0; c < 2; c++) {
    size_t got = 0;
    int rc = cam_[c]->write_state(pts_last_[c], ids_last_[c], currid_, last_[c], p, sz[c], &got);
    if (rc) return err(rc, cam_[c]->last_error);
    p += sz[c];
  }
  return FE_OK;
}

int FeStereo::set_state(const void *buf, size_t n_bytes) {
  if (!buf || n_bytes < sizeof(StereoStateHeader) || !queue_.empty()) return err(FE_BAD_ARG, "set_state: bad blob or pairs pending");
  StereoStateHeader hd;
  const uint8_t *p = static_cast<const uint8_t *>(buf);
  std::memcpy(&hd, p, sizeof(hd));
  p += sizeof(hd);
  if (hd.magic != kStereoStateMagic || sizeof(hd) + hd.size[0] + hd.size[1] > n_bytes) return err(FE_BAD_ARG, "set_state: not a stereo state blob");
  for (int c = 0; c < 2; c++) {
    FeContext &x = *cam_[c];
    uint64_t cam_currid = 0;   // one id counter for both cameras: the envelope's
    int rc = x.load_state(p, hd.size[c], pts_last_[c], ids_last_[c], &cam_currid, &last_[c]);
    if (rc) return err(rc, x.last_error.empty() ? "set_state: camera blob rejected" : x.last_error);
    p += hd.size[c];
    obs_[c] = pts_last_[c];
    obs_ids_[c] = ids_last_[c];
    released_[c] = last_[c];   // the slot the image was loaded into is busy until the next pair has been collected
    left_res_ = &no_lines_;
  }
  currid_ = hd.currid;
  rows_[0].clear();
  rows_[1].clear();
  return FE_OK;
}

FeStageTimes FeStereo::snapshot_times(bool reset) {
  FeStageTimes t = cam_[0]->snapshot_times();
  const FeStageTimes r = cam_[1]->snapshot_times();
  for (int i = 0; i < 16; i++) {
    t.ms[i] += r.ms[i];
    t.launches[i] += r.launches[i];
    t.host_ms[i] += r.host_ms[i];
  }
  t.kernel_launches_total += r.kernel_launches_total;
  t.h2d_bytes += r.h2d_bytes;
  t.d2h_bytes += r.d2h_bytes;
  t.frames = st_.frames;
  if (reset) {
    cam_[0]->reset_times();
    cam_[1]->reset_times();
    st_ = FeStageTimes{};
  }
  return t;
}

}  // namespace plviwo
