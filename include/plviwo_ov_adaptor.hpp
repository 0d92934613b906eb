// plviwo_ov_adaptor.hpp — header-only adaptor that puts the B200 front end behind the reference's own tracker classes.
//
// Compiled DOWNSTREAM, inside the PL-VIWO catkin workspace (it needs ov_core's, OpenCV's and Eigen's headers, none of
// which exist in the authoring image; tests/test_adaptor_syntax.py compiles it against minimal stand-in headers).
//
//   plviwo::TrackB200     : public ov_core::TrackBase      replaces  ov_core::TrackKLT   (track/TrackKLT.h:54-57)
//   plviwo::TrackLSDB200  : public viw::TrackLSD            replaces  viw::TrackLSD       (update/cam/TrackLSD.h:84-99)
//
// Both write into the UNCHANGED containers (ov_core::FeatureDatabase, viw::LineFeatureDatabase) with exactly the calls
// the reference makes (TrackKLT.cpp:176-179, TrackLSD.cpp:163-167), so UpdaterCamera, CamHelper, LineHelper and the
// initialisers keep working on the same objects.  One FeHandle per camera id for monocular feeds; a message with two
// images and stereo = true goes through one FeStereoHandle (TrackKLT::feed_stereo, TrackKLT.cpp:202-393).
#pragma once

#include <array>
#include <map>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <vector>

#include "cam/CamBase.h"
#include "cam/CamEqui.h"
#include "cam/CamRadtan.h"
#include "feat/FeatureDatabase.h"
#include "plviwo_fe.h"
#include "track/TrackBase.h"
#include "update/cam/TrackLSD.h"
#include "update/cam/linefeat/LineFeatureDatabase.h"
#include "utils/sensor_data.h"

namespace plviwo {

class TrackB200 : public ov_core::TrackBase {
 public:
  // same argument list as TrackKLT (track/TrackKLT.h:54-57) plus the line switch and the CUDA device
  TrackB200(std::unordered_map<size_t, std::shared_ptr<ov_core::CamBase>> cameras, int numfeats, int numaruco, bool stereo,
            HistogramMethod histmethod, int fast_threshold, int gridx, int gridy, int minpxdist, bool use_lines = true,
            int device = 0)
      : TrackBase(cameras, numfeats, numaruco, stereo, histmethod), threshold_(fast_threshold), grid_x_(gridx), grid_y_(gridy),
        min_px_dist_(minpxdist), use_lines_(use_lines), device_(device) {}
  ~TrackB200() override {
    for (auto &kv : handles_) plviwo_fe_destroy(kv.second);
    if (stereo_) plviwo_fe_stereo_destroy(stereo_);
  }

  // TrackKLT::feed_new_camera (TrackKLT.cpp:34-94): validates the message, then the same dispatch as :80-93
  void feed_new_camera(const ov_core::CameraData &message) override {
    if (message.sensor_ids.empty() || message.sensor_ids.size() != message.images.size() ||
        message.images.size() != message.masks.size())
      throw std::invalid_argument("plviwo::TrackB200: message data sizes do not match or are empty");   // reference: std::exit
    const size_t num_images = message.images.size();
    if (num_images == 1) {
      feed_monocular(message, 0);
    } else if (num_images == 2 && use_stereo) {
      feed_stereo(message, 0, 1);
    } else if (!use_stereo) {
      for (size_t i = 0; i < num_images; i++) feed_monocular(message, i);
    } else {
      throw std::invalid_argument("plviwo::TrackB200: invalid number of images, only mono or stereo tracking");   // reference: std::exit
    }
  }

  // TrackBase::change_feat_id (TrackBase.cpp:267-285) is not virtual: callers that rename a feature use this wrapper, which
  // also renames it inside the handles (the next frame would re-emit the old id otherwise)
  void change_feat_id_b200(size_t id_old, size_t id_new) {
    change_feat_id(id_old, id_new);
    for (auto &kv : handles_) plviwo_fe_change_feat_id(kv.second, (uint64_t)id_old, (uint64_t)id_new);
    if (stereo_) plviwo_fe_stereo_change_feat_id(stereo_, (uint64_t)id_old, (uint64_t)id_new);
  }

  // line rows of the last frame of a camera (consumed by TrackLSDB200)
  FeHandle *handle(size_t cam_id) { return handles_.at(cam_id); }
  FeStereoHandle *stereo_handle() { return stereo_; }   // non-null once a two-image message was fed
  bool lines_enabled() const { return use_lines_; }

 private:
  FeHandle *handle_for(size_t cam_id, const cv::Mat &img) {
    auto it = handles_.find(cam_id);
    if (it != handles_.end()) return it->second;
    FeConfig cfg = make_config(img);
    FeHandle *h = nullptr;
    if (plviwo_fe_create_model(&cfg, camera_model(cam_id), device_, &h) != FE_OK)
      throw std::runtime_error(std::string("plviwo_fe_create_model: ") + plviwo_fe_last_error(nullptr));
    handles_[cam_id] = h;
    return h;
  }
  FeConfig make_config(const cv::Mat &img) const {
    FeConfig cfg;
    plviwo_fe_default_config(&cfg);
    cfg.width = img.cols;
    cfg.height = img.rows;
    cfg.num_features = num_features;
    cfg.fast_threshold = threshold_;
    cfg.grid_x = grid_x_;
    cfg.grid_y = grid_y_;
    cfg.min_px_dist = min_px_dist_;
    cfg.histogram_method = histogram_method == HISTOGRAM ? FE_HIST_HISTOGRAM : (histogram_method == CLAHE ? FE_HIST_CLAHE : FE_HIST_NONE);
    cfg.numaruco = numaruco_of_currid();
    cfg.use_lines = use_lines_ ? 1 : 0;
    cfg.lookahead = 0;   // online use: one frame in, one frame out
    return cfg;
  }
  int numaruco_of_currid() const { return (int)((currid.load() - 1) / 4); }   // TrackBase.cpp:34: currid = 4 * numaruco + 1
  // the FeCameraModel of a camera's CamBase subclass (fixed for the camera's lifetime); any other subclass is refused, not
  // undistorted with the wrong formula
  int camera_model(size_t cam_id) const {
    const std::shared_ptr<ov_core::CamBase> &cam = camera_calib.at(cam_id);
    if (std::dynamic_pointer_cast<ov_core::CamRadtan>(cam)) return FE_CAM_RADTAN;
    if (std::dynamic_pointer_cast<ov_core::CamEqui>(cam)) return FE_CAM_EQUI;
    throw std::invalid_argument("plviwo::TrackB200: camera " + std::to_string(cam_id) +
                                " is neither an ov_core::CamRadtan nor an ov_core::CamEqui");
  }

  void feed_monocular(const ov_core::CameraData &message, size_t msg_id) {
    const size_t cam_id = (size_t)message.sensor_ids.at(msg_id);
    const cv::Mat &img = message.images.at(msg_id);
    const cv::Mat &mask = message.masks.at(msg_id);
    const int model = camera_model(cam_id);
    FeHandle *h = handle_for(cam_id, img);
    // intrinsics are refined online (StateHelper.cpp:166): hand over the current values every frame
    const Eigen::MatrixXd calib = camera_calib.at(cam_id)->get_value();
    const double K[4] = {calib(0), calib(1), calib(2), calib(3)}, D[4] = {calib(4), calib(5), calib(6), calib(7)};
    if (plviwo_fe_set_camera(h, model, K, D) != FE_OK) throw std::runtime_error(std::string("plviwo_fe_set_camera: ") + plviwo_fe_last_error(h));
    int &last_nf = last_num_features_[cam_id];   // per handle: every camera's handle follows set_num_features
    if (num_features != last_nf) {
      if (plviwo_fe_set_num_features(h, num_features) != FE_OK)
        throw std::runtime_error(std::string("plviwo_fe_set_num_features: ") + plviwo_fe_last_error(h));
      last_nf = num_features;
    }
    // one id counter for all cameras of the tracker (TrackBase.h:192): the handle continues from the shared counter ...
    plviwo_fe_set_currid(h, (uint64_t)currid.load());
    // the vanishing points are only known to the caller of TrackLSD: feed with zeros, TrackLSDB200 re-classifies
    const double vp0[6] = {0, 0, 0, 0, 0, 0};
    FeFrameInfo info;
    const int rc = plviwo_fe_feed(h, message.timestamp, img.data, img.cols, img.rows, (int)img.step, mask.empty() ? nullptr : mask.data,
                                  mask.empty() ? 0 : (int)mask.step, use_lines_ ? vp0 : nullptr, &info);
    if (rc != FE_OK) throw std::runtime_error(std::string("plviwo_fe_feed: ") + plviwo_fe_last_error(h));
    {   // ... and hands it back, so that code reading TrackBase::currid sees the ids that were given out
      uint64_t c = 0;
      plviwo_fe_get_currid(h, &c);
      currid = (size_t)c;
    }
    // rows -> FeatureDatabase::update_feature (TrackKLT.cpp:176-179)
    rows_.resize((size_t)info.n_point_rows);
    int n = 0;
    plviwo_fe_get_point_rows(h, rows_.data(), (int)rows_.size(), &n);
    for (int i = 0; i < n; i++) database->update_feature((size_t)rows_[i].id, message.timestamp, cam_id, rows_[i].u, rows_[i].v, rows_[i].un, rows_[i].vn);
    // move forward in time (TrackKLT.cpp:182-189): what display_* and TrackLSD read
    ids_.resize((size_t)info.n_last_obs);
    uv_.resize(2 * (size_t)info.n_last_obs);
    plviwo_fe_get_last_obs(h, ids_.data(), uv_.data(), info.n_last_obs, &n);
    std::vector<cv::KeyPoint> kps((size_t)n);
    std::vector<size_t> ids((size_t)n);
    for (int i = 0; i < n; i++) {
      kps[(size_t)i].pt.x = uv_[2 * (size_t)i];
      kps[(size_t)i].pt.y = uv_[2 * (size_t)i + 1];
      ids[(size_t)i] = (size_t)ids_[(size_t)i];
    }
    std::lock_guard<std::mutex> lckv(mtx_last_vars);
    img_last[cam_id] = img;
    img_mask_last[cam_id] = mask;
    pts_last[cam_id] = kps;
    ids_last[cam_id] = ids;
  }

  // TrackKLT::feed_stereo (TrackKLT.cpp:202-393) behind one FeStereoHandle.  The line tracker has no stereo path in the
  // reference (TrackLSD.cpp:57-60 feeds the left image to its monocular code): the handle runs it on the left image.
  void feed_stereo(const ov_core::CameraData &message, size_t msg_id_left, size_t msg_id_right) {
    const size_t cam[2] = {(size_t)message.sensor_ids.at(msg_id_left), (size_t)message.sensor_ids.at(msg_id_right)};
    const cv::Mat *img[2] = {&message.images.at(msg_id_left), &message.images.at(msg_id_right)};
    const cv::Mat *mask[2] = {&message.masks.at(msg_id_left), &message.masks.at(msg_id_right)};
    if (img[0]->cols != img[1]->cols || img[0]->rows != img[1]->rows || img[0]->step != img[1]->step)
      throw std::invalid_argument("plviwo::TrackB200: stereo images must have the same size and step");
    // one camera model per rig
    const int model = camera_model(cam[0]);
    if (camera_model(cam[1]) != model)
      throw std::invalid_argument("plviwo::TrackB200: the two cameras of a stereo pair must have the same camera model");
    double K[2][4], D[2][4];
    for (int c = 0; c < 2; c++) {
      const Eigen::MatrixXd calib = camera_calib.at(cam[c])->get_value();
      for (int i = 0; i < 4; i++) {
        K[c][i] = calib(i);
        D[c][i] = calib(4 + i);
      }
    }
    if (!stereo_) {
      FeConfig cfg = make_config(*img[0]);
      for (int i = 0; i < 4; i++) {
        cfg.K[i] = K[0][i];
        cfg.D[i] = D[0][i];
      }
      if (plviwo_fe_stereo_create_model(&cfg, model, K[1], D[1], device_, &stereo_) != FE_OK)
        throw std::runtime_error(std::string("plviwo_fe_stereo_create_model: ") + plviwo_fe_stereo_last_error(nullptr));
    }
    for (int c = 0; c < 2; c++)
      if (plviwo_fe_stereo_set_camera(stereo_, c, model, K[c], D[c]) != FE_OK)
        throw std::runtime_error(std::string("plviwo_fe_stereo_set_camera: ") + plviwo_fe_stereo_last_error(stereo_));
    if (num_features != last_num_features_stereo_) {
      if (plviwo_fe_stereo_set_num_features(stereo_, num_features) != FE_OK)
        throw std::runtime_error(std::string("plviwo_fe_stereo_set_num_features: ") + plviwo_fe_stereo_last_error(stereo_));
      last_num_features_stereo_ = num_features;
    }
    const bool has_mask = !mask[0]->empty() && !mask[1]->empty();
    const double vp0[6] = {0, 0, 0, 0, 0, 0};   // TrackLSDB200 re-classifies with the real vanishing points
    FeStereoInfo info;
    const int rc = plviwo_fe_stereo_feed(stereo_, message.timestamp, img[0]->data, img[1]->data, img[0]->cols, img[0]->rows,
                                         (int)img[0]->step, has_mask ? mask[0]->data : nullptr, has_mask ? mask[1]->data : nullptr,
                                         has_mask ? (int)mask[0]->step : 0, use_lines_ ? vp0 : nullptr, &info);
    if (rc != FE_OK) throw std::runtime_error(std::string("plviwo_fe_stereo_feed: ") + plviwo_fe_stereo_last_error(stereo_));
    std::lock_guard<std::mutex> lckv(mtx_last_vars);
    for (int c = 0; c < 2; c++) {   // left rows first, then right (TrackKLT.cpp:352-363)
      rows_.resize((size_t)info.n_point_rows[c]);
      int n = 0;
      plviwo_fe_stereo_get_point_rows(stereo_, c, rows_.data(), (int)rows_.size(), &n);
      for (int i = 0; i < n; i++) database->update_feature((size_t)rows_[i].id, message.timestamp, cam[c], rows_[i].u, rows_[i].v, rows_[i].un, rows_[i].vn);
      ids_.resize((size_t)info.n_last_obs[c]);
      uv_.resize(2 * (size_t)info.n_last_obs[c]);
      plviwo_fe_stereo_get_last_obs(stereo_, c, ids_.data(), uv_.data(), info.n_last_obs[c], &n);
      std::vector<cv::KeyPoint> kps((size_t)n);
      std::vector<size_t> ids((size_t)n);
      for (int i = 0; i < n; i++) {
        kps[(size_t)i].pt.x = uv_[2 * (size_t)i];
        kps[(size_t)i].pt.y = uv_[2 * (size_t)i + 1];
        ids[(size_t)i] = (size_t)ids_[(size_t)i];
      }
      img_last[cam[c]] = *img[c];
      img_mask_last[cam[c]] = *mask[c];
      pts_last[cam[c]] = kps;
      ids_last[cam[c]] = ids;
    }
  }

  int threshold_, grid_x_, grid_y_, min_px_dist_;
  bool use_lines_;
  FeStereoHandle *stereo_ = nullptr;
  int device_;
  std::map<size_t, int> last_num_features_;   // per camera handle (a fresh entry is 0: the first feed sets it)
  int last_num_features_stereo_ = -1;
  std::map<size_t, FeHandle *> handles_;
  std::vector<FePointRow> rows_;
  std::vector<uint64_t> ids_;
  std::vector<float> uv_;
};

// viw::TrackLSD's feed_new_camera is not virtual (TrackLSD.h:94), so UpdaterCamera holds this type directly (see
// INTEGRATION.md for the two-line change); the base class only provides the LineFeatureDatabase.
class TrackLSDB200 : public viw::TrackLSD {
 public:
  TrackLSDB200(std::unordered_map<size_t, std::shared_ptr<ov_core::CamBase>> cameras, bool stereo,
               ov_core::TrackBase::HistogramMethod histmethod, std::map<int, std::shared_ptr<ov_core::TrackBase>> track_feats)
      : viw::TrackLSD(cameras, stereo, histmethod, track_feats), feats_(track_feats) {}

  // TrackLSD::feed_new_camera (TrackLSD.cpp:39-68): the segments of this frame were extracted and associated while the
  // point tracker ran; classify them with the vanishing points and push the rows (TrackLSD.cpp:163-167)
  void feed_new_camera(const ov_core::CameraData &message, std::vector<Eigen::Vector2d> &vanishing_points) {
    const int cam_id = message.sensor_ids.at(0);
    auto b200 = std::dynamic_pointer_cast<TrackB200>(feats_.at(cam_id));
    if (!b200 || !b200->lines_enabled()) throw std::invalid_argument("plviwo::TrackLSDB200 needs a plviwo::TrackB200 with lines enabled");
    const double vp[6] = {vanishing_points.at(0)(0), vanishing_points.at(0)(1), vanishing_points.at(1)(0),
                          vanishing_points.at(1)(1), vanishing_points.at(2)(0), vanishing_points.at(2)(1)};
    int n = 0, np = 0;
    std::vector<FeLineRow> rows;
    std::vector<FeLinePoint> pts;
    if (message.images.size() == 2 && b200->stereo_handle()) {   // TrackLSD.cpp:57-60: the left image of the pair
      FeStereoHandle *h = b200->stereo_handle();
      plviwo_fe_stereo_classify_lines(h, vp);
      plviwo_fe_stereo_get_line_rows(h, nullptr, 0, &n);
      plviwo_fe_stereo_get_line_points(h, nullptr, 0, &np);
      rows.resize((size_t)n);
      pts.resize((size_t)np);
      plviwo_fe_stereo_get_line_rows(h, rows.data(), n, &n);
      plviwo_fe_stereo_get_line_points(h, pts.data(), np, &np);
    } else {
      FeHandle *h = b200->handle((size_t)cam_id);
      plviwo_fe_classify_lines(h, vp);
      plviwo_fe_get_line_rows(h, nullptr, 0, &n);
      plviwo_fe_get_line_points(h, nullptr, 0, &np);
      rows.resize((size_t)n);
      pts.resize((size_t)np);
      plviwo_fe_get_line_rows(h, rows.data(), n, &n);
      plviwo_fe_get_line_points(h, pts.data(), np, &np);
    }
    for (const FeLineRow &r : rows) {
      Eigen::Vector4f line(r.line[0], r.line[1], r.line[2], r.line[3]), line_n(r.line_n[0], r.line_n[1], r.line_n[2], r.line_n[3]);
      std::map<int, double> points_line;
      std::vector<Eigen::Vector2f> points;
      for (int k = 0; k < r.n_pts; k++) {
        const FeLinePoint &p = pts[(size_t)(r.pt_offset + k)];
        points_line[p.pid] = (double)p.dist;
        points.emplace_back(p.u, p.v);
      }
      database->update_feature((size_t)r.id, message.timestamp, (size_t)cam_id, line, line_n, points_line, points, r.D);
    }
  }

 private:
  std::map<int, std::shared_ptr<ov_core::TrackBase>> feats_;
};

}  // namespace plviwo
