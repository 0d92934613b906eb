// Stream group host side (see fe_group.h).  Reference call sites mirrored per stream:
//   ov_core::TrackKLT::feed_new_camera / feed_monocular      open_vins/ov_core/src/track/TrackKLT.cpp:34-200
//   viw::TrackLSD::feed_new_camera / feed_monocular          PL-VIWO/src/update/cam/TrackLSD.cpp:39-192
//   the bag loop feeding every camera in time order           PL-VIWO/src/run_bag.cpp:272-340
#include "fe_group.h"
#include "state_blob.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>

namespace plviwo {

#define FG_CUDA(call)                                  \
  do {                                                 \
    cudaError_t e__ = (call);                          \
    if (e__ != cudaSuccess) return fail(e__, #call);   \
  } while (0)

static inline int align_up(int v, int a) { return (v + a - 1) / a * a; }
static inline size_t align_up_sz(size_t v, size_t a) { return (v + a - 1) / a * a; }

FeGroup::FeGroup(const FeConfig &cfg, int n_streams, int device, bool stereo, int model)
    : cfg_(cfg), S_(n_streams), device_(device), W_(cfg.width), H_(cfg.height), stereo_(stereo), model_(model) {}

int FeGroup::fail(cudaError_t e, const char *what) {
  last_error = std::string(what) + ": " + cudaGetErrorString(e);
  return FE_CUDA_ERROR;
}
int FeGroup::err(int code, const std::string &msg) {
  last_error = msg;
  return code;
}

void FeGroup::layout_cells() {
  cells_ = grider_layout(W_, H_, cfg_.grid_x, cfg_.grid_y, cfg_.num_features);
  g_.nfg = cells_.nfg;
  g_.n_cells = (int)cells_.cells.size();
  for (int i = 0; i < 256; i++) g_.cell_of_loc[i] = -1;
  std::copy(cells_.cell_of_loc.begin(), cells_.cell_of_loc.end(), g_.cell_of_loc);   // grid_x * grid_y <= 256
}

template <class T>
static cudaError_t dev_alloc(std::vector<void *> &keep, T **p, size_t count, bool zero = true) {
  cudaError_t e = cudaMalloc((void **)p, std::max<size_t>(count, 1) * sizeof(T));
  if (e != cudaSuccess) return e;
  keep.push_back(*p);
  if (zero) e = cudaMemset(*p, 0, std::max<size_t>(count, 1) * sizeof(T));
  return e;
}

int FeGroup::init() {
  FG_CUDA(cudaSetDevice(device_));
  init_device_constants();
  la_ = std::max(cfg_.lookahead, 0);
  R_ = la_ + 2;
  RB_ = la_ + 2;
  {   // ticks whose state-independent work shares one set of launches: enough frames per launch to fill the device
    const char *e = std::getenv("PLVIWO_GROUP_FRONT_TICKS");
    // measured on B200 (profiles/sweep_group.sh): launches that carry >= 128-256 frames run the image / FAST / line kernels
    // at their best (64 streams: 1 tick per batch 33.6 k frames/s, 2: 37.8 k, 4: 38.3 k; 32 streams, 4 ticks: 36.0 k)
    int b = e ? std::atoi(e) : std::max(1, (256 + S_ - 1) / std::max(S_, 1));
    B_ = std::max(1, std::min(b, std::max(la_ / 3, 1)));
    // tracking lanes: the streams are split over this many CUDA streams, each running its own detect -> LK -> gate -> lines
    // chain; the chain is latency bound (~0.4 ms per tick whatever the number of streams), so lanes overlap
    e = std::getenv("PLVIWO_GROUP_LANES");
    lanes_ = e ? std::atoi(e) : 4;
    lanes_ = std::max(1, std::min(lanes_, stereo_ ? S_ / 2 : S_));   // a rig's two streams share a lane
  }
  K_.resize(4 * (size_t)S_);
  D_.resize(4 * (size_t)S_);
  for (int s = 0; s < S_; s++)
    for (int i = 0; i < 4; i++) {
      K_[4 * s + i] = cfg_.K[i];
      D_[4 * s + i] = cfg_.D[i];
    }
  frame_count_.assign(S_, 0);
  prev_slot_.assign(S_, -1);
  ticks_.resize(RB_);
  batches_.resize(RB_);

  // ---- geometry
  g_.W = W_;
  g_.H = H_;
  g_.n_streams = S_;
  g_.num_features = cfg_.num_features;
  g_.grid_x = cfg_.grid_x;
  g_.grid_y = cfg_.grid_y;
  g_.min_px_dist = cfg_.min_px_dist;
  g_.close_w = (int)((float)W_ / (float)cfg_.min_px_dist);
  g_.close_h = (int)((float)H_ / (float)cfg_.min_px_dist);
  g_.line_min_length = cfg_.line_min_length;
  g_.use_lines = cfg_.use_lines;
  g_.cam_model = model_;
  layout_cells();
  const int ncell = g_.n_cells, nfg = g_.nfg;
  g_.cand_cap = std::max(ncell * nfg, 1);
  g_.pts_cap = align_up(cfg_.num_features + ncell * nfg + 32, 32);
  // a stereo rig's right list is not bounded by its own top-off (it also receives the new stereo points of the left): hold
  // as many points per camera as the stereo handle's tracking buffers (fe_context.cu, max_pts without line samples)
  if (stereo_) g_.pts_cap = align_up(std::max(g_.pts_cap, std::max(4096, 8 * cfg_.num_features)), 32);
  g_.lines_cap = 1024;
  g_.pol_cap = 8192;
  g_.segs_cap = 4096;
  const int kps_cap = W_ * H_ / 4 + 1024;
  const int max_bands = (H_ + kFastBandRows - 1) / kFastBandRows;
  FG_CUDA(dev_alloc(dev_allocs_, &d_cells_, std::max(ncell, 1)));
  if (ncell) FG_CUDA(cudaMemcpy(d_cells_, cells_.cells.data(), ncell * sizeof(FastCell), cudaMemcpyHostToDevice));
  fg_.w = W_;
  fg_.h = H_;
  fg_.n_cells = ncell;
  fg_.max_bands = cells_.n_bands;
  fg_.max_cell_w = cells_.csx;
  fg_.fast_threshold = cfg_.fast_threshold;
  fg_.kps_cap = kps_cap;
  fg_.nfg = nfg;
  fg_.cells = d_cells_;
  (void)max_bands;

  // ---- slots
  const int nslots = S_ * R_;
  slots_.assign(nslots, SlotRec{});
  h_raw_.assign(nslots, nullptr);
  h_mask_.assign(nslots, nullptr);
  for (int i = 0; i < nslots; i++) {
    SlotRec &sl = slots_[i];
    FG_CUDA(alloc_image(sl.raw, W_, H_));
    dev_allocs_.push_back(sl.raw.p);
    int w = W_, h = H_;
    sl.n_lvl = 0;
    for (int l = 0; l <= cfg_.pyr_levels && l < kMaxLevels; l++) {   // cv::buildOpticalFlowPyramid: a level is kept while both sides stay > winSize
      FG_CUDA(alloc_image(sl.lvl[l], w, h));
      dev_allocs_.push_back(sl.lvl[l].p);
      sl.n_lvl = l + 1;
      w = (w + 1) / 2;
      h = (h + 1) / 2;
      if (w <= cfg_.win_size || h <= cfg_.win_size) break;
    }
    sl.mask = nullptr;
    FG_CUDA(dev_alloc(dev_allocs_, &sl.hist, 256));
    FG_CUDA(dev_alloc(dev_allocs_, &sl.counters, 4));
    FG_CUDA(dev_alloc(dev_allocs_, &sl.eq_lut, 256));
    FG_CUDA(dev_alloc(dev_allocs_, &sl.clahe, cfg_.histogram_method == FE_HIST_CLAHE ? 64 * 256 : 1));
    FG_CUDA(dev_alloc(dev_allocs_, &sl.fast_total, 2));
    FG_CUDA(dev_alloc(dev_allocs_, &sl.kps, kps_cap, false));
    FG_CUDA(dev_alloc(dev_allocs_, &sl.sort_scratch, kps_cap, false));
    FG_CUDA(dev_alloc(dev_allocs_, &sl.band_off, std::max(ncell * cells_.n_bands, 1)));
    FG_CUDA(dev_alloc(dev_allocs_, &sl.band_cnt, std::max(ncell * cells_.n_bands, 1)));
    FG_CUDA(dev_alloc(dev_allocs_, &sl.cand, g_.cand_cap));
    FG_CUDA(dev_alloc(dev_allocs_, &sl.cand_cnt, std::max(ncell, 1)));
    if (cfg_.use_lines) {
      FG_CUDA(alloc_image(sl.half, W_ / 2, H_ / 2));
      dev_allocs_.push_back(sl.half.p);
      if (sl.fld.alloc(W_ / 2, H_ / 2, cfg_.fld_length_threshold, g_.segs_cap)) return fail(cudaGetLastError(), "FldBuffers::alloc");
    }
  }
  FG_CUDA(dev_alloc(dev_allocs_, &d_slots_, nslots, false));
  FG_CUDA(cudaMemcpy(d_slots_, slots_.data(), nslots * sizeof(SlotRec), cudaMemcpyHostToDevice));
  FG_CUDA(dev_alloc(dev_allocs_, &d_slot_flags_, nslots));
  g_.slots = d_slots_;
  g_.slot_flags = d_slot_flags_;
  // every slot's pyramid holds n_lvl images: LK tracks through all of them (cv::calcOpticalFlowPyrLK on a prebuilt pyramid),
  // and the body of its launches is chosen by that count, as a handle chooses it (fe_kernels.h lk_w15_form)
  lk_prm_ = lk_params(cfg_.win_size, slots_[0].n_lvl - 1, nullptr, nullptr, true, model_);

  // ---- tracker state and work arrays
  const size_t P = (size_t)S_ * g_.pts_cap;
  FG_CUDA(dev_alloc(dev_allocs_, &g_.pts, P * RB_));   // ring of state records, one per output record (fe_group_dev.h)
  FG_CUDA(dev_alloc(dev_allocs_, &g_.ids, P * RB_));
  FG_CUDA(dev_alloc(dev_allocs_, &g_.n_pts, (size_t)S_ * RB_));
  prev_rec_.resize(S_);
  for (int s = 0; s < S_; s++) prev_rec_[s] = s;       // record (ring 0, stream s): zero points
  FG_CUDA(dev_alloc(dev_allocs_, &g_.currid, S_));
  FG_CUDA(dev_alloc(dev_allocs_, &g_.wpts, P));
  FG_CUDA(dev_alloc(dev_allocs_, &g_.wids, P));
  FG_CUDA(dev_alloc(dev_allocs_, &g_.wn, S_));
  FG_CUDA(dev_alloc(dev_allocs_, &g_.wmode, S_));
  FG_CUDA(dev_alloc(dev_allocs_, &g_.winfo, 4 * (size_t)S_));
  FG_CUDA(dev_alloc(dev_allocs_, &g_.lk_pts1, P));
  FG_CUDA(dev_alloc(dev_allocs_, &g_.lk_p0n, P));
  FG_CUDA(dev_alloc(dev_allocs_, &g_.lk_p1n, P));
  FG_CUDA(dev_alloc(dev_allocs_, &g_.lk_status, P));
  FG_CUDA(dev_alloc(dev_allocs_, &g_.close, (size_t)S_ * std::max(g_.close_w * g_.close_h, 1)));
  FG_CUDA(dev_alloc(dev_allocs_, &g_.valid, (size_t)S_ * kValidStride));
  FG_CUDA(dev_alloc(dev_allocs_, &g_.stats, 4));
  FG_CUDA(dev_alloc(dev_allocs_, &g_.ext_in, (size_t)S_ * g_.cand_cap));
  FG_CUDA(dev_alloc(dev_allocs_, &g_.ext_pt, (size_t)S_ * g_.cand_cap));
  {
    std::vector<uint64_t> cur(S_, 4 * (uint64_t)cfg_.numaruco + 1);   // TrackBase.cpp:34
    FG_CUDA(cudaMemcpy(g_.currid, cur.data(), S_ * sizeof(uint64_t), cudaMemcpyHostToDevice));
  }
  if (cfg_.use_lines) {
    const size_t L2 = 2 * (size_t)S_;
    FG_CUDA(dev_alloc(dev_allocs_, &g_.lines, L2 * g_.lines_cap));
    FG_CUDA(dev_alloc(dev_allocs_, &g_.line_ids, L2 * g_.lines_cap));
    FG_CUDA(dev_alloc(dev_allocs_, &g_.pol_off, L2 * (g_.lines_cap + 1)));
    FG_CUDA(dev_alloc(dev_allocs_, &g_.pol_pid, L2 * g_.pol_cap));
    FG_CUDA(dev_alloc(dev_allocs_, &g_.pol_dist, L2 * g_.pol_cap));
    FG_CUDA(dev_alloc(dev_allocs_, &g_.n_lines, L2));
    FG_CUDA(dev_alloc(dev_allocs_, &g_.line_buf, S_));
    FG_CUDA(dev_alloc(dev_allocs_, &g_.line_currid, S_));
    FG_CUDA(dev_alloc(dev_allocs_, &g_.lnew, (size_t)S_ * g_.lines_cap));
    FG_CUDA(dev_alloc(dev_allocs_, &g_.n_lnew, S_));   // zero: no segments before the first frame fed with vanishing points
    FG_CUDA(dev_alloc(dev_allocs_, &g_.lcnt, (size_t)S_ * (g_.lines_cap + 1)));
    FG_CUDA(dev_alloc(dev_allocs_, &g_.loff, (size_t)S_ * (g_.lines_cap + 1)));
    FG_CUDA(dev_alloc(dev_allocs_, &g_.lpos, (size_t)S_ * g_.pol_cap));
    FG_CUDA(dev_alloc(dev_allocs_, &g_.lmatch, (size_t)S_ * g_.lines_cap));
    std::vector<uint64_t> one(S_, 1);                                 // TrackLSD.cpp:32
    FG_CUDA(cudaMemcpy(g_.line_currid, one.data(), S_ * sizeof(uint64_t), cudaMemcpyHostToDevice));
  }

  // ---- output ring (pinned, device-mapped): header | point rows | obs ids | obs uv | line rows | line points
  //      [| sample p0 | sample p1 | sample status: cfg.line_samples only]
  g_.off_rows = align_up_sz(sizeof(GroupOutHeader), 64);
  g_.off_obs_ids = align_up_sz(g_.off_rows + (size_t)g_.pts_cap * sizeof(FePointRow), 64);
  g_.off_obs_uv = align_up_sz(g_.off_obs_ids + (size_t)g_.pts_cap * sizeof(uint64_t), 64);
  g_.off_lrows = align_up_sz(g_.off_obs_uv + (size_t)g_.pts_cap * sizeof(float2), 64);
  g_.off_lpts = align_up_sz(g_.off_lrows + (size_t)(cfg_.use_lines ? g_.lines_cap : 0) * sizeof(FeLineRow), 64);
  const size_t end_lpts = g_.off_lpts + (size_t)(cfg_.use_lines ? g_.pol_cap : 0) * sizeof(FeLinePoint);
  if (cfg_.use_lines && cfg_.line_samples > 0) {
    // a handle tracks its samples in its LK buffer, after the n points: ns = min(S * L, max_pts - n) (fe_context.cu init /
    // perform_matching); L <= lines_cap here.  At S = 10: 10240 samples, 170 KB per record.
    g_.line_samples = cfg_.line_samples;
    g_.sample_max_pts = std::max(4096, 8 * cfg_.num_features) + 4096 * 8;
    g_.sample_cap = (int)std::min<long long>((long long)cfg_.line_samples * g_.lines_cap, g_.sample_max_pts);
    g_.off_sp0 = align_up_sz(end_lpts, 64);
    g_.off_sp1 = g_.off_sp0 + (size_t)g_.sample_cap * sizeof(float2);
    g_.off_sst = g_.off_sp1 + (size_t)g_.sample_cap * sizeof(float2);
    g_.out_stride = align_up_sz(g_.off_sst + (size_t)g_.sample_cap, 256);
  } else if (stereo_) {
    g_.off_sinfo = align_up_sz(end_lpts, 64);
    g_.out_stride = align_up_sz(g_.off_sinfo + sizeof(FeStereoInfo), 256);
  } else {
    g_.out_stride = align_up_sz(end_lpts, 256);
  }
  if (stereo_ && stereo_rows_smem(g_.pts_cap) > 227 * 1024)
    return err(FE_BAD_ARG, "stereo group: the id table of num_features + the grid's candidates exceeds shared memory");
  FG_CUDA(cudaHostAlloc((void **)&h_out_, g_.out_stride * (size_t)RB_ * S_, cudaHostAllocMapped));
  host_allocs_.push_back(h_out_);
  std::memset(h_out_, 0, g_.out_stride * (size_t)RB_ * S_);
  {
    void *dp = nullptr;
    FG_CUDA(cudaHostGetDevicePointer(&dp, h_out_, 0));
    g_.out = static_cast<uint8_t *>(dp);
  }
  // ---- job rings
  const size_t nfj = (size_t)RB_ * B_ * S_;
  FG_CUDA(cudaMallocHost((void **)&h_fjobs_, nfj * sizeof(FrontJob)));
  host_allocs_.push_back(h_fjobs_);
  FG_CUDA(cudaMallocHost((void **)&h_ljobs_, nfj * sizeof(int)));
  host_allocs_.push_back(h_ljobs_);
  FG_CUDA(cudaMallocHost((void **)&h_tjobs_, (size_t)RB_ * S_ * sizeof(TrackJob)));
  host_allocs_.push_back(h_tjobs_);
  FG_CUDA(dev_alloc(dev_allocs_, &d_fjobs_, nfj));
  FG_CUDA(dev_alloc(dev_allocs_, &d_ljobs_, nfj));
  FG_CUDA(dev_alloc(dev_allocs_, &d_tjobs_, (size_t)RB_ * S_));

  // ---- streams and events
  int lo = 0, hi = 0;
  FG_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
  {
    int ncopy = 4;
    if (const char *e = std::getenv("PLVIWO_GROUP_COPY_STREAMS")) ncopy = std::max(1, std::min(std::atoi(e), 8));
    s_copy_.resize(ncopy);
    for (auto &st : s_copy_) FG_CUDA(cudaStreamCreateWithPriority(&st, cudaStreamNonBlocking, lo));
  }
  // front batches of consecutive ticks run on different streams: the tail of one batch's chain walk (a few long
  // components, milliseconds) overlaps the next batches' kernels
  int nfront = std::min(RB_, 6);
  if (const char *e = std::getenv("PLVIWO_GROUP_FRONT_STREAMS")) nfront = std::max(1, std::min(std::atoi(e), RB_));
  s_front_.resize(nfront);
  for (auto &st : s_front_) FG_CUDA(cudaStreamCreateWithPriority(&st, cudaStreamNonBlocking, lo));
  s_track_.resize(lanes_);
  for (auto &st : s_track_) FG_CUDA(cudaStreamCreateWithPriority(&st, cudaStreamNonBlocking, hi));
  // the line association of tick t only needs tick t's points: it runs beside the point chain of tick t + 1
  s_lines_.resize(lanes_);
  for (auto &st : s_lines_) FG_CUDA(cudaStreamCreateWithPriority(&st, cudaStreamNonBlocking, hi));
  ev_gate_.resize((size_t)RB_ * lanes_);
  for (auto &e : ev_gate_) FG_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  ev_copy_.resize((size_t)RB_ * s_copy_.size());
  ev_front_.resize(RB_);
  trace_ = std::getenv("PLVIWO_GROUP_TRACE") != nullptr;
  if (trace_) {
    ev_tr0_.resize(RB_);
    ev_tr1_.resize(RB_);
    tr_valid_.assign(RB_, 0);
    for (auto &e : ev_tr0_) FG_CUDA(cudaEventCreate(&e));
    for (auto &e : ev_tr1_) FG_CUDA(cudaEventCreate(&e));
    ev_trs_.resize((size_t)RB_ * 4);
    for (auto &e : ev_trs_) FG_CUDA(cudaEventCreate(&e));
  }
  ev_pyr_.resize(RB_);
  for (auto &e : ev_pyr_) FG_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  for (auto &e : ev_copy_) FG_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  for (auto &e : ev_front_) FG_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  ev_done_.resize((size_t)RB_ * lanes_);
  for (auto &e : ev_done_) FG_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  FG_CUDA(cudaDeviceSynchronize());
  return FE_OK;
}

FeGroup::~FeGroup() {
  cudaSetDevice(device_);
  cudaDeviceSynchronize();
  if (trace_ && tr_n_ > 0)
    std::fprintf(stderr, "[plviwo group trace] %ld front batches (%d ticks each): device latency %.3f ms, interval between batches %.3f ms\n",
                 tr_n_, B_, tr_lat_ms_ / tr_n_, tr_np_ ? tr_period_ms_ / tr_np_ : 0.0);
  if (trace_ && tr_n_ > 0)
    std::fprintf(stderr, "[plviwo group trace] stages of a front batch, ms: equalise + pyramid %.3f, Canny + tiles %.3f, components %.3f, walk %.3f, "
                 "segments %.3f\n", tr_stage_ms_[0] / tr_n_, tr_stage_ms_[1] / tr_n_, tr_stage_ms_[2] / tr_n_, tr_stage_ms_[3] / tr_n_,
                 tr_stage_ms_[4] / tr_n_);
  if (trace_ && tr_host_ticks_ > 0)
    std::fprintf(stderr, "[plviwo group trace] host per tick, us: submit %.1f (of which issuing frame copies %.1f), waiting in collect %.1f\n",
                 tr_host_submit_us_ / tr_host_ticks_, tr_host_copy_us_ / tr_host_ticks_, tr_host_wait_us_ / tr_host_ticks_);
  for (auto e : ev_tr0_) cudaEventDestroy(e);
  for (auto e : ev_tr1_) cudaEventDestroy(e);
  for (auto e : ev_trs_) cudaEventDestroy(e);
  for (SlotRec &sl : slots_)
    if (cfg_.use_lines) sl.fld.release();
  for (void *p : dev_allocs_) cudaFree(p);
  for (void *p : host_allocs_) cudaFreeHost(p);
  for (uint8_t *p : h_raw_) if (p) cudaFreeHost(p);
  for (uint8_t *p : h_mask_) if (p) cudaFreeHost(p);
  for (auto st : s_copy_) cudaStreamDestroy(st);
  for (auto st : s_front_) cudaStreamDestroy(st);
  for (auto st : s_track_) cudaStreamDestroy(st);
  for (auto st : s_lines_) cudaStreamDestroy(st);
  for (auto e : ev_gate_) cudaEventDestroy(e);
  for (auto e : ev_copy_) cudaEventDestroy(e);
  for (auto e : ev_front_) cudaEventDestroy(e);
  for (auto e : ev_pyr_) cudaEventDestroy(e);
  for (auto e : ev_done_) cudaEventDestroy(e);
  for (auto e : ev_pool_) cudaEventDestroy(e);
}

int FeGroup::set_calib(int stream, const double K[4], const double D[4]) {
  if (stream < 0 || stream >= S_ || !K || !D) return err(FE_BAD_ARG, "set_calib: bad stream");
  for (int i = 0; i < 4; i++) {
    K_[4 * stream + i] = K[i];
    D_[4 * stream + i] = D[i];
  }
  return FE_OK;
}

int FeGroup::ensure_mask_buffer(int slot) {
  if (slots_[slot].mask != nullptr) return FE_OK;
  FG_CUDA(cudaMalloc((void **)&slots_[slot].mask, (size_t)W_ * H_));
  dev_allocs_.push_back(slots_[slot].mask);
  // the table entry on the device: a plain copy (nothing that is in flight uses this slot's mask pointer)
  FG_CUDA(cudaMemcpy(&d_slots_[slot], &slots_[slot], sizeof(SlotRec), cudaMemcpyHostToDevice));
  FG_CUDA(cudaMallocHost((void **)&h_mask_[slot], (size_t)W_ * H_));
  return FE_OK;
}

cudaEvent_t FeGroup::timing_event() {
  if (ev_next_ == ev_pool_.size()) {
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    ev_pool_.push_back(e);
  }
  return ev_pool_[ev_next_++];
}

int FeGroup::drain_timing() {
  for (const TimedLaunch &t : timed_) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, t.a, t.b) == cudaSuccess) {
      times_.ms[t.k] += ms;
      times_.launches[t.k]++;
      times_.frames[t.k] += (uint64_t)t.frames;
    } else {
      cudaGetLastError();
    }
  }
  timed_.clear();
  ev_next_ = 0;
  return FE_OK;
}

FeGroupTimes FeGroup::times(bool reset) {
  cudaSetDevice(device_);   // the counter below lives on the group's device (a process may hold groups on several)
  FeGroupTimes t = times_;
  t.kernel_launches_total = launches_;
  t.h2d_bytes = h2d_bytes_;
  t.d2h_bytes = d2h_bytes_;
  t.frames_total = frames_done_;
  t.ticks = (uint64_t)collected_;
  {   // grid cells the detector ran on (device counter; everything collected has finished)
    unsigned long long v = 0;
    if (g_.stats && cudaMemcpy(&v, g_.stats, sizeof(v), cudaMemcpyDeviceToHost) == cudaSuccess) t.fast_cells = v - fast_cells_base_;
    if (reset) fast_cells_base_ = v;
    cudaGetLastError();
  }
  if (reset) {
    times_ = FeGroupTimes{};
    launches_ = h2d_bytes_ = d2h_bytes_ = frames_done_ = 0;
  }
  return t;
}

// ------------------------------------------------------------------------------------------------ submit
int FeGroup::submit(const double *timestamps, const uint8_t *const *images, int stride, bool on_device, const uint8_t *const *masks,
                    int mask_stride, const double *vps) {
  FG_CUDA(cudaSetDevice(device_));
  const auto t_sub0 = std::chrono::steady_clock::now();
  double copy_us = 0;
  if (!timestamps || !images || stride < W_) return err(FE_BAD_ARG, "submit: bad arguments");
  if (submitted_ - collected_ > la_) return err(FE_BAD_ARG, "submit: lookahead window full (collect a tick first)");
  const long long tick = submitted_;
  const int ring = (int)(tick % RB_);
  TickRec &tr = ticks_[ring];
  tr.ring = ring;
  tr.cur_slot.assign(S_, -1);
  tr.track_launched = false;
  if (pending_batch_ < 0) {
    pending_batch_ = (int)(batch_seq_++ % RB_);
    FrontBatch &nb = batches_[pending_batch_];
    nb.jobs.clear();
    nb.line_slots.clear();
    nb.ticks.clear();
    nb.launched = false;
  }
  FrontBatch &b = batches_[pending_batch_];
  tr.batch = pending_batch_;
  const int eq = cfg_.histogram_method == FE_HIST_HISTOGRAM ? 1 : (cfg_.histogram_method == FE_HIST_CLAHE ? 2 : 0);
  TrackJob *tj = h_tjobs_ + (size_t)ring * S_;
  int nj = 0;
  for (int s = 0; s < S_; s++) {
    if (!images[s]) continue;
    const int slot = s * R_ + (int)(frame_count_[s] % R_);
    SlotRec &sl = slots_[slot];
    FrontJob fj;
    fj.slot = slot;
    fj.eq_mode = eq;
    fj.flags = 0;
    if (on_device) {
      fj.src = images[s];
      fj.src_pitch = stride;
    } else {
      cudaPointerAttributes attr;
      const bool pinned = cudaPointerGetAttributes(&attr, images[s]) == cudaSuccess && attr.type == cudaMemoryTypeHost;
      cudaGetLastError();
      const uint8_t *src = images[s];
      int sstride = stride;
      if (!pinned) {   // pageable caller memory: stage through the slot's pinned buffer
        if (!h_raw_[slot]) FG_CUDA(cudaMallocHost((void **)&h_raw_[slot], (size_t)W_ * H_));
        for (int y = 0; y < H_; y++) std::memcpy(h_raw_[slot] + (size_t)y * W_, images[s] + (size_t)y * stride, W_);
        src = h_raw_[slot];
        sstride = W_;
      }
      // a tight frame into a tight staging image is ONE contiguous transfer (a 2-D copy is issued row by row: 1280-byte
      // rows reach less than half of the link's bandwidth)
      const auto t_c0 = std::chrono::steady_clock::now();
      cudaStream_t cs = s_copy_[copy_rr_++ % s_copy_.size()];
      if (sstride == W_ && sl.raw.pitch == W_) FG_CUDA(cudaMemcpyAsync(sl.raw.p, src, (size_t)W_ * H_, cudaMemcpyHostToDevice, cs));
      else FG_CUDA(cudaMemcpy2DAsync(sl.raw.p, sl.raw.pitch, src, sstride, W_, H_, cudaMemcpyHostToDevice, cs));
      h2d_bytes_ += (size_t)W_ * H_;
      if (trace_) copy_us += std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t_c0).count();
      fj.src = sl.raw.p;
      fj.src_pitch = sl.raw.pitch;
    }
    if (masks && masks[s]) {
      if (mask_stride < W_) return err(FE_BAD_ARG, "submit: bad mask stride");
      int rc = ensure_mask_buffer(slot);
      if (rc) return rc;
      for (int y = 0; y < H_; y++) std::memcpy(h_mask_[slot] + (size_t)y * W_, masks[s] + (size_t)y * mask_stride, W_);
      FG_CUDA(cudaMemcpyAsync(slots_[slot].mask, h_mask_[slot], (size_t)W_ * H_, cudaMemcpyHostToDevice, s_copy_[copy_rr_++ % s_copy_.size()]));
      h2d_bytes_ += (size_t)W_ * H_;
      fj.flags |= 1;
    }
    b.jobs.push_back(fj);
    const bool lines = cfg_.use_lines && vps != nullptr && !(stereo_ && (s & 1));   // stereo: the left image only
    if (lines) b.line_slots.push_back(slot);
    TrackJob &j = tj[nj++];
    std::memset(&j, 0, sizeof(j));
    j.stream = s;
    j.cur_slot = slot;
    j.prev_slot = prev_slot_[s];
    j.flags = lines ? 1 : 0;
    j.out = ring * S_ + s;
    j.prev_rec = prev_rec_[s];
    prev_rec_[s] = j.out;
    j.timestamp = timestamps[s];
    for (int i = 0; i < 4; i++) {
      j.K[i] = K_[4 * s + i];
      j.D[i] = D_[4 * s + i];
    }
    if (vps) std::memcpy(j.vp, vps + 6 * (size_t)(stereo_ ? s / 2 : s), 6 * sizeof(double));
    tr.cur_slot[s] = slot;
    prev_slot_[s] = slot;
    frame_count_[s]++;
  }
  // streams without a frame in this tick: an empty record
  for (int s = 0; s < S_; s++)
    if (tr.cur_slot[s] < 0) std::memset(h_out_ + (size_t)(ring * S_ + s) * g_.out_stride, 0, sizeof(GroupOutHeader));
  b.ticks.push_back((int)tick);
  submitted_++;
  int rc_flush = FE_OK;
  if ((int)b.ticks.size() >= B_) rc_flush = flush_front();
  if (trace_) {
    tr_host_copy_us_ += copy_us;
    tr_host_submit_us_ += std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t_sub0).count();
    tr_host_ticks_++;
  }
  return rc_flush;
}

int FeGroup::flush_front() {
  if (pending_batch_ < 0) return FE_OK;
  const int buf = pending_batch_;
  FrontBatch &b = batches_[buf];
  pending_batch_ = -1;
  int rc = launch_front(b, buf);
  if (rc) return rc;
  for (int t : b.ticks) {
    rc = launch_track(t);
    if (rc) return rc;
  }
  return FE_OK;
}

void FeGroup::account(int k, cudaEvent_t a, cudaEvent_t b, int frames) { timed_.push_back(TimedLaunch{k, a, b, frames}); }

int FeGroup::launch_front(FrontBatch &b, int buf) {
  const int nj = (int)b.jobs.size(), nl = (int)b.line_slots.size();
  b.launched = true;
  if (nj == 0) return FE_OK;
  // stage timing: everything on ONE stream, so that a kernel's event interval holds that kernel alone
  cudaStream_t st = timing_ ? s_front_[0] : s_front_[buf % s_front_.size()];
  FrontJob *hj = h_fjobs_ + (size_t)buf * B_ * S_, *dj = d_fjobs_ + (size_t)buf * B_ * S_;
  int *hl = h_ljobs_ + (size_t)buf * B_ * S_, *dl = d_ljobs_ + (size_t)buf * B_ * S_;
  int n_half = cfg_.use_lines ? nj : 0;   // jobs [0, n_half) get the half-resolution image of the line front work
  if (stereo_ && cfg_.use_lines) {        // ... in a stereo group the left images only (TrackLSD.cpp:57-60): left jobs first
    auto right_image = [this](const FrontJob &j) { return (j.slot / R_) & 1; };
    n_half = (int)(std::stable_partition(b.jobs.begin(), b.jobs.end(), [&](const FrontJob &j) { return !right_image(j); }) - b.jobs.begin());
  }
  std::memcpy(hj, b.jobs.data(), nj * sizeof(FrontJob));
  if (nl) std::memcpy(hl, b.line_slots.data(), nl * sizeof(int));
  // the frames (and masks) of the batch are on their way on the copy stream
  for (size_t c = 0; c < s_copy_.size(); c++) {
    cudaEvent_t ev = ev_copy_[(size_t)buf * s_copy_.size() + c];
    FG_CUDA(cudaEventRecord(ev, s_copy_[c]));
    FG_CUDA(cudaStreamWaitEvent(st, ev, 0));
  }
  FG_CUDA(cudaMemcpyAsync(dj, hj, nj * sizeof(FrontJob), cudaMemcpyHostToDevice, st));
  if (nl) FG_CUDA(cudaMemcpyAsync(dl, hl, nl * sizeof(int), cudaMemcpyHostToDevice, st));
  if (trace_) {
    if (tr_valid_[buf]) {   // the buffer's previous batch has been collected: read its events before they are re-recorded
      float ms = 0;
      if (cudaEventElapsedTime(&ms, ev_tr0_[buf], ev_tr1_[buf]) == cudaSuccess) { tr_lat_ms_ += ms; tr_n_++; }
      cudaEvent_t *es = &ev_trs_[(size_t)buf * 4];
      cudaEvent_t seq[6] = {ev_tr0_[buf], es[0], es[1], es[2], es[3], ev_tr1_[buf]};
      for (int k = 0; k < 5; k++)
        if (cudaEventElapsedTime(&ms, seq[k], seq[k + 1]) == cudaSuccess) tr_stage_ms_[k] += ms;
      const int nxt = (buf + 1) % RB_;
      if (tr_valid_[nxt] && cudaEventElapsedTime(&ms, ev_tr0_[buf], ev_tr0_[nxt]) == cudaSuccess && ms > 0) { tr_period_ms_ += ms; tr_np_++; }
      cudaGetLastError();
    }
    tr_valid_[buf] = 1;
    cudaEventRecord(ev_tr0_[buf], st);
  }
  const bool tm = timing_;
  cudaEvent_t e0 = nullptr;
  auto mark = [&]() -> cudaEvent_t {
    cudaEvent_t e = timing_event();
    cudaEventRecord(e, st);
    return e;
  };
  auto step = [&](int k, int frames) {
    if (!tm) return;
    cudaEvent_t e1 = mark();
    account(k, e0, e1, frames);
    e0 = e1;
  };
  if (tm) e0 = mark();
  const int eq = cfg_.histogram_method;
  launch_hist_batch(d_slots_, dj, nj, fg_, d_slot_flags_, st);
  launches_++;
  step(FE_GK_HIST, nj);
  if (eq == FE_HIST_CLAHE) {
    launch_clahe_lut_batch(d_slots_, dj, nj, fg_, st);
    launches_++;
    if (tm) e0 = mark();
  }
  if (n_half > 0) {
    launch_eq_pyr1_batch(d_slots_, dj, n_half, fg_, true, st);
    launches_++;
  }
  if (n_half < nj) {
    launch_eq_pyr1_batch(d_slots_, dj + n_half, nj - n_half, fg_, false, st);
    launches_++;
  }
  step(FE_GK_EQ_PYR1, nj);
  const SlotRec &s0 = slots_[0];
  for (int l = 2; l < s0.n_lvl; l++) {
    launch_pyr_level_batch(d_slots_, dj, nj, l, s0.lvl[l].w, s0.lvl[l].h, st);
    launches_++;
  }
  step(FE_GK_PYR_REST, nj);
  // the point chains of the batch's ticks need nothing else (launch_track); only the line association waits for the rest
  FG_CUDA(cudaEventRecord(ev_pyr_[buf], st));
  if (trace_) for (int k = 0; k < 4; k++) cudaEventRecord(ev_trs_[(size_t)buf * 4 + k], st);   // (re-recorded below where the stage exists)
  // FAST is NOT here: the reference runs it on the cells the detection finds short of features only (Grider_GRID.h:108-125,
  // 1-3 of 25 cells on a tracked sequence), so it runs inside the detection of the tick (launch_track)
  if (nl > 0) {
    launch_canny_table(d_slots_, dl, nl, W_ / 2, H_ / 2, cfg_.canny_th1, st);   // + tile-local component labels (fused)
    launches_ += 2;
    step(FE_GK_CANNY, nl);
    cudaEvent_t ev2[2] = {nullptr, nullptr};
    if (tm) {
      ev2[0] = timing_event();
      ev2[1] = timing_event();
    } else if (trace_) {
      cudaEventRecord(ev_trs_[(size_t)buf * 4 + 1], st);
      ev2[0] = ev_trs_[(size_t)buf * 4 + 2];
      ev2[1] = ev_trs_[(size_t)buf * 4 + 3];
    }
    launch_fld_table(d_slots_, dl, nl, W_ / 2, H_ / 2, s0.fld.max_chains, cfg_.fld_length_threshold, cfg_.fld_distance_threshold, st,
                     (tm || trace_) ? ev2 : nullptr);
    launches_ += 7 + (nl >= 16 ? 1 : 0);
    if (tm) {
      cudaEvent_t e1 = mark();
      account(FE_GK_CCL, e0, ev2[0], nl);
      account(FE_GK_WALK, ev2[0], ev2[1], nl);
      account(FE_GK_SEGMENTS, ev2[1], e1, nl);
      e0 = e1;
    }
  }
  FG_CUDA(cudaGetLastError());
  FG_CUDA(cudaEventRecord(ev_front_[buf], st));
  if (trace_) cudaEventRecord(ev_tr1_[buf], st);
  return FE_OK;
}

int FeGroup::launch_track(int tick) {
  if (stereo_) return launch_track_stereo(tick);
  const int ring = tick % RB_;
  TickRec &tr = ticks_[ring];
  tr.track_launched = true;
  TrackJob *hj = h_tjobs_ + (size_t)ring * S_, *dj = d_tjobs_ + (size_t)ring * S_;
  int nj = 0;
  for (int s = 0; s < S_; s++) nj += tr.cur_slot[s] >= 0 ? 1 : 0;
  const LkParams &prm = lk_prm_;
  const bool tm = timing_;
  // jobs are stored in stream order; lane l owns streams [S l / lanes, S (l + 1) / lanes) for the lifetime of the group
  // (a stream's frames are tracked in order on ONE CUDA stream), i.e. a contiguous range of the tick's jobs
  int jpos = 0;
  for (int l = 0; l < lanes_; l++) {
    const int s_end = (int)((long long)S_ * (l + 1) / lanes_);
    const int j0 = jpos;
    while (jpos < nj && hj[jpos].stream < s_end) jpos++;
    const int j1 = jpos;
    cudaStream_t st = timing_ ? s_front_[0] : s_track_[l];
    const int n = j1 - j0;
    if (n > 0) {
      FG_CUDA(cudaStreamWaitEvent(st, ev_pyr_[tr.batch], 0));
      FG_CUDA(cudaMemcpyAsync(dj + j0, hj + j0, (size_t)n * sizeof(TrackJob), cudaMemcpyHostToDevice, st));
      cudaEvent_t e0 = nullptr;
      auto step = [&](int k) {
        if (!tm) return;
        cudaEvent_t e1 = timing_event();
        cudaEventRecord(e1, st);
        account(k, e0, e1, n);
        e0 = e1;
      };
      if (tm) {
        e0 = timing_event();
        cudaEventRecord(e0, st);
      }
      launch_group_detect(g_, dj + j0, n, st);
      step(FE_GK_DETECT);
      if (fg_.n_cells > 0) {
        launch_group_fast(g_, dj + j0, n, fg_, st);
        step(FE_GK_FAST);
        launch_group_fast_select(g_, dj + j0, n, fg_, st);
        step(FE_GK_SELECT);
        launches_ += 2;
      }
      launch_group_cands(g_, dj + j0, n, st);
      step(FE_GK_CANDS);
      launch_group_subpix(g_, dj + j0, n, st);
      step(FE_GK_SUBPIX);
      launch_group_accept(g_, dj + j0, n, st);
      step(FE_GK_ACCEPT);
      launches_ += 3;
      launch_group_lk(g_, dj + j0, n, prm, st);
      step(FE_GK_LK);
      // (the gate writes this tick's state record; the previous tick's line association reads ITS record: no ordering needed)
      launch_group_gate(g_, dj + j0, n, st);
      step(FE_GK_GATE);
      launches_ += 3;
      cudaStream_t sl = st;
      if (cfg_.use_lines) {
        if (!tm) {   // side stream: ordered after this tick's gate and (stream order) after the previous tick's association
          sl = s_lines_[l];
          FG_CUDA(cudaEventRecord(ev_gate_[(size_t)ring * lanes_ + l], st));
          FG_CUDA(cudaStreamWaitEvent(sl, ev_gate_[(size_t)ring * lanes_ + l], 0));
        }
        if (g_.sample_cap > 0) {
          // cfg.line_samples: needs the gate's header and the segments the previous association left in lnew, which this
          // tick's association rewrites next on the same stream; the point chain never waits for it, collect does (ev_done_)
          launch_group_line_samples(g_, dj + j0, n, prm, sl);
          launches_++;
          step(FE_GK_LK);
        }
        if (!tm) FG_CUDA(cudaStreamWaitEvent(sl, ev_front_[tr.batch], 0));   // the frame's segments (chain walk + fit of the batch)
        launch_group_lines(g_, dj + j0, n, sl);
        launches_++;
        step(FE_GK_LINES);
      }
      FG_CUDA(cudaGetLastError());
      FG_CUDA(cudaEventRecord(ev_done_[(size_t)ring * lanes_ + l], sl));
      continue;
    }
    FG_CUDA(cudaEventRecord(ev_done_[(size_t)ring * lanes_ + l], st));
  }
  return FE_OK;
}

// ------------------------------------------------------------------------------------------------ collect
int FeGroup::collect(FeFrameInfo *infos) {
  FG_CUDA(cudaSetDevice(device_));
  if (collected_ >= submitted_) return err(FE_BAD_ARG, "collect: nothing submitted");
  const long long tick = collected_;
  const int ring = (int)(tick % RB_);
  TickRec &tr = ticks_[ring];
  if (!tr.track_launched) {   // its front batch never filled up: launch what is there
    int rc = flush_front();
    if (rc) return rc;
  }
  const auto t_w0 = std::chrono::steady_clock::now();
  for (int l = 0; l < lanes_; l++) FG_CUDA(cudaEventSynchronize(ev_done_[(size_t)ring * lanes_ + l]));
  if (trace_) tr_host_wait_us_ += std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t_w0).count();
  collected_++;
  last_collected_ = tick;
  int status = FE_OK;
  for (int s = 0; s < S_; s++) {
    const GroupOutHeader *h = reinterpret_cast<const GroupOutHeader *>(h_out_ + (size_t)(ring * S_ + s) * g_.out_stride);
    if (infos) {
      infos[s] = h->info;
      if (tr.cur_slot[s] < 0) infos[s].timestamp = -1.0;
    }
    if (tr.cur_slot[s] < 0) continue;
    frames_done_++;
    d2h_bytes_ += sizeof(GroupOutHeader) + (size_t)h->info.n_point_rows * sizeof(FePointRow) +
                  (size_t)h->n_obs * (sizeof(uint64_t) + sizeof(float2)) + (size_t)h->info.n_line_rows * sizeof(FeLineRow) +
                  (size_t)h->n_line_points * sizeof(FeLinePoint) + (size_t)h->n_samples * (2 * sizeof(float2) + 1);
    if (h->status != FE_OK && status == FE_OK) {
      status = h->status;
      static const char *what[] = {"?", "points", "lines", "point / line pairs", "candidates"};
      last_error = (stereo_ ? "rig " + std::to_string(s / 2) + (s & 1 ? " right" : " left") : "stream " + std::to_string(s)) + ": more " +
                   what[std::min(std::max(h->overflow_what, 0), 4)] + " than the group's buffers hold";
    }
  }
  if (timing_ && submitted_ == collected_) {   // everything launched has finished: read the stage events
    FG_CUDA(cudaDeviceSynchronize());
    drain_timing();
  }
  return status;
}

const GroupOutHeader *FeGroup::header(int s) const {
  if (last_collected_ < 0 || s < 0 || s >= S_) return nullptr;
  return reinterpret_cast<const GroupOutHeader *>(h_out_ + (size_t)((int)(last_collected_ % RB_) * S_ + s) * g_.out_stride);
}
const FePointRow *FeGroup::point_rows(int s) const {
  const uint8_t *r = reinterpret_cast<const uint8_t *>(header(s));
  return r ? reinterpret_cast<const FePointRow *>(r + g_.off_rows) : nullptr;
}
const uint64_t *FeGroup::obs_ids(int s) const {
  const uint8_t *r = reinterpret_cast<const uint8_t *>(header(s));
  return r ? reinterpret_cast<const uint64_t *>(r + g_.off_obs_ids) : nullptr;
}
const float *FeGroup::obs_uv(int s) const {
  const uint8_t *r = reinterpret_cast<const uint8_t *>(header(s));
  return r ? reinterpret_cast<const float *>(r + g_.off_obs_uv) : nullptr;
}
const FeLineRow *FeGroup::line_rows(int s) const {
  const uint8_t *r = reinterpret_cast<const uint8_t *>(header(s));
  return r ? reinterpret_cast<const FeLineRow *>(r + g_.off_lrows) : nullptr;
}
const FeLinePoint *FeGroup::line_points(int s) const {
  const uint8_t *r = reinterpret_cast<const uint8_t *>(header(s));
  return r ? reinterpret_cast<const FeLinePoint *>(r + g_.off_lpts) : nullptr;
}
int FeGroup::line_samples(int s, float *uv01, uint8_t *status, int cap, int *n_out) const {
  const GroupOutHeader *h = header(s);
  if (!h) return FE_BAD_ARG;
  const int n = h->n_samples;
  if (n_out) *n_out = n;
  if (!uv01 && !status) return FE_OK;
  if (cap < n) return FE_OVERFLOW;
  if (n == 0) return FE_OK;
  const uint8_t *r = reinterpret_cast<const uint8_t *>(h);
  if (uv01) {
    const float2 *p0 = reinterpret_cast<const float2 *>(r + g_.off_sp0), *p1 = reinterpret_cast<const float2 *>(r + g_.off_sp1);
    for (int k = 0; k < n; k++) {
      uv01[4 * k + 0] = p0[k].x;
      uv01[4 * k + 1] = p0[k].y;
      uv01[4 * k + 2] = p1[k].x;
      uv01[4 * k + 3] = p1[k].y;
    }
  }
  if (status) std::memcpy(status, r + g_.off_sst, (size_t)n);
  return FE_OK;
}

// Whole-sequence playback of every stream (run_bag.cpp:272-340 feeds the cameras in time order): images[t * S + s].
int FeGroup::play(int n_ticks, const uint8_t *const *images, int stride, bool on_device, const double *timestamps, const double *vps,
                  FePlayStats *out) {
  if (submitted_ != collected_) return err(FE_BAD_ARG, "play: ticks submitted with submit are still pending");
  if (stereo_)
    for (size_t k = 0; k < (size_t)n_ticks * S_; k += 2)
      if (!images[k] != !images[k + 1]) return err(FE_BAD_ARG, "play: a rig's pair has exactly one image");
  const int per = stereo_ ? 2 : 1, U = S_ / per;   // a stereo rig's statistics cover both cameras' point rows
  std::vector<FePlayStats> st(U);
  for (auto &x : st) std::memset(&x, 0, sizeof(x));
  std::vector<double> ts(S_);
  int sub = 0;
  for (int i = 0; i < n_ticks; i++) {
    while (sub < n_ticks && sub <= i + la_) {
      for (int s = 0; s < S_; s++) ts[s] = timestamps[sub];
      int rc = submit(ts.data(), images + (size_t)sub * S_, stride, on_device, nullptr, 0, vps);
      if (rc) return rc;
      sub++;
    }
    int rc = collect(nullptr);
    if (rc) return rc;
    for (int s = 0; s < S_; s++) {
      const GroupOutHeader *h = header(s);
      if (!images[(size_t)i * S_ + s]) continue;
      FePlayStats &x = st[s / per];
      if (s % per == 0) {
        x.frames++;
        x.resets += (stereo_ ? stereo_info(s / 2).reset : h->info.reset) ? 1 : 0;
      }
      x.point_rows += (uint64_t)h->info.n_point_rows;
      x.line_rows += (uint64_t)h->info.n_line_rows;
      const FePointRow *pr = point_rows(s);
      for (int k = 0; k < h->info.n_point_rows; k++) x.checksum += (double)pr[k].id + pr[k].u + pr[k].v;
      const FeLineRow *lr = line_rows(s);
      for (int k = 0; k < h->info.n_line_rows; k++) x.checksum += (double)lr[k].id + lr[k].line[0] + lr[k].line[1] + lr[k].line[2] + lr[k].line[3];
    }
  }
  if (out) std::memcpy(out, st.data(), U * sizeof(FePlayStats));
  return FE_OK;
}

// ------------------------------------------------------------------------------------------ state / taps
// One stream's blob, in the format of a single handle's (state_blob.h): the device's per-line point lists (CSR, float
// distances) go through the handle's point maps.
int FeGroup::get_state(int s, void *buf, size_t cap, size_t *n_bytes) {
  FG_CUDA(cudaSetDevice(device_));
  if (s < 0 || s >= S_) return err(FE_BAD_ARG, "get_state: bad stream");
  if (submitted_ != collected_) return err(FE_BAD_ARG, "get_state: collect the pending ticks first");
  FG_CUDA(cudaDeviceSynchronize());
  int n_pts = 0, lb = 0, n_lines = 0;
  uint64_t currid = 0, line_currid = 1;
  const size_t rec = (size_t)prev_rec_[s];   // the stream's current state record
  FG_CUDA(cudaMemcpy(&n_pts, g_.n_pts + rec, sizeof(int), cudaMemcpyDeviceToHost));
  FG_CUDA(cudaMemcpy(&currid, g_.currid + s, sizeof(uint64_t), cudaMemcpyDeviceToHost));
  std::vector<float4> lines;
  std::vector<uint64_t> lids;
  PointsOnLines pol;
  if (cfg_.use_lines) {
    FG_CUDA(cudaMemcpy(&lb, g_.line_buf + s, sizeof(int), cudaMemcpyDeviceToHost));
    FG_CUDA(cudaMemcpy(&n_lines, g_.n_lines + 2 * s + lb, sizeof(int), cudaMemcpyDeviceToHost));
    FG_CUDA(cudaMemcpy(&line_currid, g_.line_currid + s, sizeof(uint64_t), cudaMemcpyDeviceToHost));
    const size_t b = (size_t)(2 * s + lb);
    lines.resize(n_lines);
    lids.resize(n_lines);
    std::vector<int> poff(n_lines + 1);
    FG_CUDA(cudaMemcpy(lines.data(), g_.lines + b * g_.lines_cap, n_lines * sizeof(float4), cudaMemcpyDeviceToHost));
    FG_CUDA(cudaMemcpy(lids.data(), g_.line_ids + b * g_.lines_cap, n_lines * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    FG_CUDA(cudaMemcpy(poff.data(), g_.pol_off + b * (g_.lines_cap + 1), (n_lines + 1) * sizeof(int), cudaMemcpyDeviceToHost));
    if (n_lines == 0) poff[0] = 0;
    const int ne = poff[n_lines];
    std::vector<int> ppid(ne);
    std::vector<float> pdist(ne);
    FG_CUDA(cudaMemcpy(ppid.data(), g_.pol_pid + b * g_.pol_cap, ne * sizeof(int), cudaMemcpyDeviceToHost));
    FG_CUDA(cudaMemcpy(pdist.data(), g_.pol_dist + b * g_.pol_cap, ne * sizeof(float), cudaMemcpyDeviceToHost));
    pol.resize(n_lines);
    for (int i = 0; i < n_lines; i++)
      for (int e = poff[i]; e < poff[i + 1]; e++) pol[i][ppid[e]] = (double)pdist[e];
  }
  const int ps = prev_slot_[s];
  int flags = 0;
  if (ps >= 0) FG_CUDA(cudaMemcpy(&flags, d_slot_flags_ + ps, sizeof(int), cudaMemcpyDeviceToHost));
  const StateHeader hd = state_header(W_, H_, currid, line_currid, n_pts, n_lines, pol, ps >= 0, (flags & 1) != 0);
  const StateLayout at = state_layout(hd);
  if (n_bytes) *n_bytes = at.size;
  if (!buf || cap < at.size) return buf ? FE_OVERFLOW : FE_OK;
  std::vector<float2> pts(n_pts);
  std::vector<uint64_t> ids(n_pts);
  FG_CUDA(cudaMemcpy(pts.data(), g_.pts + rec * g_.pts_cap, n_pts * sizeof(float2), cudaMemcpyDeviceToHost));
  FG_CUDA(cudaMemcpy(ids.data(), g_.ids + rec * g_.pts_cap, n_pts * sizeof(uint64_t), cudaMemcpyDeviceToHost));
  uint8_t *p = static_cast<uint8_t *>(buf);
  state_write(p, hd, pts.data(), ids.data(), lines.data(), lids.data(), pol);
  if (hd.has_image) {
    const DevImage &l0 = slots_[ps].lvl[0];
    FG_CUDA(cudaMemcpy2D(p + at.image, W_, l0.p, l0.pitch, W_, H_, cudaMemcpyDeviceToHost));
  }
  if (hd.has_mask) FG_CUDA(cudaMemcpy(p + at.mask, slots_[ps].mask, (size_t)W_ * H_, cudaMemcpyDeviceToHost));
  return FE_OK;
}

const char *FeGroup::check_state(const void *buf, size_t n_bytes, StateView &v) const {
  if (const char *why = state_read(buf, n_bytes, W_, H_, v)) return why;
  if (v.hd.n_pts > g_.pts_cap || v.hd.n_lines > g_.lines_cap || v.hd.n_pol_entries > g_.pol_cap)
    return "set_state: more points / lines than the group's buffers hold";
  return nullptr;
}

int FeGroup::set_state(int s, const void *buf, size_t n_bytes) {
  FG_CUDA(cudaSetDevice(device_));
  if (s < 0 || s >= S_) return err(FE_BAD_ARG, "set_state: bad stream");
  if (submitted_ != collected_) return err(FE_BAD_ARG, "set_state: collect the pending ticks first");
  // ---- parse and validate everything before any of it is applied
  StateView v;
  if (const char *why = check_state(buf, n_bytes, v)) return err(FE_BAD_ARG, why);
  const StateHeader &hd = v.hd;
  std::vector<int> poff(hd.n_lines + 1, 0), ppid;
  std::vector<float> pdist;
  for (int i = 0; i < hd.n_lines; i++) {
    poff[i] = (int)ppid.size();
    for (const auto &kv : v.pol[i]) {
      ppid.push_back(kv.first);
      pdist.push_back((float)kv.second);
    }
  }
  poff[hd.n_lines] = (int)ppid.size();
  // ---- apply
  FG_CUDA(cudaDeviceSynchronize());
  const int n = hd.n_pts;
  const size_t rec = (size_t)prev_rec_[s];   // nothing is in flight: the stream's current state record is rewritten in place
  FG_CUDA(cudaMemcpy(g_.pts + rec * g_.pts_cap, v.base + v.at.pts, n * sizeof(float2), cudaMemcpyHostToDevice));
  FG_CUDA(cudaMemcpy(g_.ids + rec * g_.pts_cap, v.base + v.at.ids, n * sizeof(uint64_t), cudaMemcpyHostToDevice));
  FG_CUDA(cudaMemcpy(g_.n_pts + rec, &n, sizeof(int), cudaMemcpyHostToDevice));
  FG_CUDA(cudaMemcpy(g_.currid + s, &hd.currid, sizeof(uint64_t), cudaMemcpyHostToDevice));
  if (cfg_.use_lines) {
    const int lb = 0;
    const size_t b = (size_t)(2 * s + lb);
    FG_CUDA(cudaMemcpy(g_.line_buf + s, &lb, sizeof(int), cudaMemcpyHostToDevice));
    FG_CUDA(cudaMemcpy(g_.n_lines + 2 * s + lb, &hd.n_lines, sizeof(int), cudaMemcpyHostToDevice));
    FG_CUDA(cudaMemcpy(g_.line_currid + s, &hd.line_currid, sizeof(uint64_t), cudaMemcpyHostToDevice));
    FG_CUDA(cudaMemcpy(g_.lines + b * g_.lines_cap, v.base + v.at.lines, hd.n_lines * sizeof(float4), cudaMemcpyHostToDevice));
    FG_CUDA(cudaMemcpy(g_.line_ids + b * g_.lines_cap, v.base + v.at.line_ids, hd.n_lines * sizeof(uint64_t), cudaMemcpyHostToDevice));
    FG_CUDA(cudaMemcpy(g_.pol_off + b * (g_.lines_cap + 1), poff.data(), (hd.n_lines + 1) * sizeof(int), cudaMemcpyHostToDevice));
    FG_CUDA(cudaMemcpy(g_.pol_pid + b * g_.pol_cap, ppid.data(), ppid.size() * sizeof(int), cudaMemcpyHostToDevice));
    FG_CUDA(cudaMemcpy(g_.pol_dist + b * g_.pol_cap, pdist.data(), pdist.size() * sizeof(float), cudaMemcpyHostToDevice));
  }
  prev_slot_[s] = -1;
  if (hd.has_image) {   // the stored image is already equalised: rebuild its pyramid and candidate table without a LUT
    const int slot = s * R_ + (int)(frame_count_[s] % R_);
    SlotRec &sl = slots_[slot];
    FG_CUDA(cudaMemcpy2D(sl.raw.p, sl.raw.pitch, v.base + v.at.image, W_, W_, H_, cudaMemcpyHostToDevice));
    FrontJob fj;
    fj.src = sl.raw.p;
    fj.src_pitch = sl.raw.pitch;
    fj.slot = slot;
    fj.eq_mode = 0;
    fj.flags = 0;
    if (hd.has_mask) {
      int rc = ensure_mask_buffer(slot);
      if (rc) return rc;
      FG_CUDA(cudaMemcpy(slots_[slot].mask, v.base + v.at.mask, (size_t)W_ * H_, cudaMemcpyHostToDevice));
      fj.flags |= 1;
    }
    cudaStream_t st = s_front_[0];
    FG_CUDA(cudaMemcpy(d_fjobs_, &fj, sizeof(fj), cudaMemcpyHostToDevice));
    launch_hist_batch(d_slots_, d_fjobs_, 1, fg_, d_slot_flags_, st);
    launch_eq_pyr1_batch(d_slots_, d_fjobs_, 1, fg_, cfg_.use_lines != 0 && !(stereo_ && (s & 1)), st);
    for (int l = 2; l < sl.n_lvl; l++) launch_pyr_level_batch(d_slots_, d_fjobs_, 1, l, sl.lvl[l].w, sl.lvl[l].h, st);
    FG_CUDA(cudaGetLastError());
    FG_CUDA(cudaStreamSynchronize(st));
    prev_slot_[s] = slot;
    frame_count_[s]++;
  }
  return FE_OK;
}

int FeGroup::tap(int s, int what, void *buf, size_t cap, size_t *n_bytes) {
  FG_CUDA(cudaSetDevice(device_));
  if (s < 0 || s >= S_ || prev_slot_[s] < 0) return err(FE_BAD_ARG, "tap: bad stream / no frame yet");
  if (submitted_ != collected_) return err(FE_BAD_ARG, "tap: collect the pending ticks first");
  FG_CUDA(cudaDeviceSynchronize());
  const SlotRec &sl = slots_[prev_slot_[s]];
  const DevImage *im = nullptr;
  if (what >= FE_TAP_PYR_LEVEL0 && what < FE_TAP_PYR_LEVEL0 + kMaxLevels && what - FE_TAP_PYR_LEVEL0 < sl.n_lvl) im = &sl.lvl[what - FE_TAP_PYR_LEVEL0];
  if (what == FE_TAP_HALF && cfg_.use_lines) im = &sl.half;
  if (!im) return err(FE_BAD_ARG, "tap: not available");
  const int rc = tap_image(*im, buf, cap, n_bytes);
  return rc == FE_CUDA_ERROR ? fail(cudaGetLastError(), "tap: cudaMemcpy2D") : rc;
}

// ------------------------------------------------------------------------------------------------ stereo rigs
// The tracking phase of a tick for the rigs of each lane (fe_group_dev.h has the sequence and the job layout).
int FeGroup::launch_track_stereo(int tick) {
  const int ring = tick % RB_;
  TickRec &tr = ticks_[ring];
  tr.track_launched = true;
  TrackJob *hj = h_tjobs_ + (size_t)ring * S_, *dj = d_tjobs_ + (size_t)ring * S_;
  int nj = 0;
  for (int s = 0; s < S_; s++) nj += tr.cur_slot[s] >= 0 ? 1 : 0;
  const LkParams &prm = lk_prm_;
  const int n_rigs = S_ / 2;
  std::vector<TrackJob> pairs;
  int jpos = 0;
  for (int l = 0; l < lanes_; l++) {
    const int s_end = 2 * (int)((long long)n_rigs * (l + 1) / lanes_);
    const int j0 = jpos;
    while (jpos < nj && hj[jpos].stream < s_end) jpos++;
    const int n = (jpos - j0) / 2;   // rigs with a pair in this tick: their left and right jobs are adjacent (stream order)
    cudaStream_t st = s_track_[l];
    if (n == 0) {
      FG_CUDA(cudaEventRecord(ev_done_[(size_t)ring * lanes_ + l], st));
      continue;
    }
    pairs.assign(hj + j0, hj + j0 + 2 * n);
    for (int k = 0; k < n; k++) {
      hj[j0 + k] = pairs[2 * k];
      hj[j0 + n + k] = pairs[2 * k + 1];
    }
    FG_CUDA(cudaStreamWaitEvent(st, ev_pyr_[tr.batch], 0));
    FG_CUDA(cudaMemcpyAsync(dj + j0, hj + j0, (size_t)2 * n * sizeof(TrackJob), cudaMemcpyHostToDevice, st));
    const TrackJob *jl = dj + j0, *jr = dj + j0 + n;
    auto detect_tail = [&](const TrackJob *jobs, bool right) {   // FAST .. accept of one camera of the lane's rigs
      if (fg_.n_cells > 0) {
        launch_group_fast(g_, jobs, n, fg_, st);
        launch_group_fast_select(g_, jobs, n, fg_, st);
        launches_ += 2;
      }
      if (right) launch_stereo_cands_right(g_, jobs, n, st);
      else launch_group_cands(g_, jobs, n, st);
      launch_group_subpix(g_, jobs, n, st);
      launch_group_accept(g_, jobs, n, st);
      launches_ += 3;
    };
    launch_stereo_detect(g_, jl, n, false, st);
    detect_tail(jl, false);
    launch_stereo_lr_lk(g_, jl, n, prm, st);
    launch_stereo_pair(g_, jl, n, st);
    launch_stereo_detect(g_, jr, n, true, st);
    detect_tail(jr, true);
    launch_group_lk(g_, jl, 2 * n, prm, st);
    launch_stereo_gate(g_, jl, 2 * n, st);
    launch_stereo_rows(g_, jl, n, st);
    launches_ += 7;
    cudaStream_t sl = st;
    if (cfg_.use_lines) {   // the left image's line tracker, against the left points the rig has just produced
      sl = s_lines_[l];
      FG_CUDA(cudaEventRecord(ev_gate_[(size_t)ring * lanes_ + l], st));
      FG_CUDA(cudaStreamWaitEvent(sl, ev_gate_[(size_t)ring * lanes_ + l], 0));
      FG_CUDA(cudaStreamWaitEvent(sl, ev_front_[tr.batch], 0));
      launch_group_lines(g_, jl, n, sl);
      launches_++;
    }
    FG_CUDA(cudaGetLastError());
    FG_CUDA(cudaEventRecord(ev_done_[(size_t)ring * lanes_ + l], sl));
  }
  return FE_OK;
}

int FeGroup::stereo_submit(const double *timestamps, const uint8_t *const *left, const uint8_t *const *right, int stride, bool on_device,
                           const uint8_t *const *masks_left, const uint8_t *const *masks_right, int mask_stride, const double *vps) {
  if (!stereo_ || !timestamps || !left || !right) return err(FE_BAD_ARG, "submit: bad arguments");
  if (!masks_left != !masks_right) return err(FE_BAD_ARG, "submit: masks are given for both cameras or for neither");
  const int n_rigs = S_ / 2;
  std::vector<const uint8_t *> img(S_), msk(masks_left ? S_ : 0);
  std::vector<double> ts(S_);
  for (int r = 0; r < n_rigs; r++) {
    if (!left[r] != !right[r]) return err(FE_BAD_ARG, "submit: rig " + std::to_string(r) + " has exactly one image of its pair");
    img[2 * r] = left[r];
    img[2 * r + 1] = right[r];
    ts[2 * r] = ts[2 * r + 1] = timestamps[r];
    if (masks_left) {
      if (!masks_left[r] != !masks_right[r]) return err(FE_BAD_ARG, "submit: rig " + std::to_string(r) + " has exactly one mask");
      if (masks_left[r] && left[r] && mask_stride < W_) return err(FE_BAD_ARG, "submit: bad mask stride");
      msk[2 * r] = masks_left[r];
      msk[2 * r + 1] = masks_right[r];
    }
  }
  return submit(ts.data(), img.data(), stride, on_device, masks_left ? msk.data() : nullptr, mask_stride, vps);
}

FeStereoInfo FeGroup::stereo_info(int rig) const {
  FeStereoInfo si;
  std::memset(&si, 0, sizeof(si));
  si.timestamp = -1.0;
  const GroupOutHeader *h = header(2 * rig);
  if (!stereo_ || !h || ticks_[(int)(last_collected_ % RB_)].cur_slot[2 * rig] < 0) return si;   // no pair in the tick
  std::memcpy(&si, reinterpret_cast<const uint8_t *>(h) + g_.off_sinfo, sizeof(si));
  si.n_line_rows = h->info.n_line_rows;   // k_group_lines writes the left record's header
  si.n_lines_detected = h->info.n_lines_detected;
  si.n_line_matches = h->info.n_line_matches;
  return si;
}

int FeGroup::stereo_collect(FeStereoInfo *infos) {
  if (!stereo_) return err(FE_BAD_ARG, "collect: not a stereo group");
  const int rc = collect(nullptr);
  if (infos && last_collected_ >= 0)
    for (int r = 0; r < S_ / 2; r++) infos[r] = stereo_info(r);
  return rc;
}

int FeGroup::stereo_get_state(int rig, void *buf, size_t cap, size_t *n_bytes) {
  if (!stereo_ || rig < 0 || rig >= S_ / 2) return err(FE_BAD_ARG, "get_state: bad rig");
  size_t sz[2] = {0, 0};
  for (int c = 0; c < 2; c++) {
    int rc = get_state(2 * rig + c, nullptr, 0, &sz[c]);
    if (rc) return rc;
  }
  const size_t need = sizeof(StereoStateHeader) + sz[0] + sz[1];
  if (n_bytes) *n_bytes = need;
  if (!buf) return FE_OK;
  if (cap < need) return FE_OVERFLOW;
  StereoStateHeader hd;
  hd.magic = kStereoStateMagic;
  hd.version = kStereoStateVersion;
  FG_CUDA(cudaMemcpy(&hd.currid, g_.currid + 2 * rig, sizeof(uint64_t), cudaMemcpyDeviceToHost));   // the rig's counter
  hd.size[0] = sz[0];
  hd.size[1] = sz[1];
  uint8_t *p = static_cast<uint8_t *>(buf);
  std::memcpy(p, &hd, sizeof(hd));
  p += sizeof(hd);
  for (int c = 0; c < 2; c++) {
    int rc = get_state(2 * rig + c, p, sz[c], nullptr);
    if (rc) return rc;
    p += sz[c];
  }
  return FE_OK;
}

int FeGroup::stereo_set_state(int rig, const void *buf, size_t n_bytes) {
  if (!stereo_ || rig < 0 || rig >= S_ / 2) return err(FE_BAD_ARG, "set_state: bad rig");
  if (submitted_ != collected_) return err(FE_BAD_ARG, "set_state: collect the pending ticks first");
  // ---- both cameras' blobs are checked before either is applied
  StereoStateHeader hd;
  if (!buf || n_bytes < sizeof(hd)) return err(FE_BAD_ARG, "set_state: blob shorter than the stereo header");
  std::memcpy(&hd, buf, sizeof(hd));
  if (hd.magic != kStereoStateMagic) return err(FE_BAD_ARG, "set_state: not a stereo state blob (magic)");
  if (hd.version != kStereoStateVersion) return err(FE_BAD_ARG, "set_state: unknown stereo state version");
  if (hd.size[0] > n_bytes || hd.size[1] > n_bytes || sizeof(hd) + hd.size[0] + hd.size[1] > n_bytes)
    return err(FE_BAD_ARG, "set_state: truncated stereo blob (its camera blobs end past its size)");
  const uint8_t *cam[2] = {static_cast<const uint8_t *>(buf) + sizeof(hd), static_cast<const uint8_t *>(buf) + sizeof(hd) + hd.size[0]};
  for (int c = 0; c < 2; c++) {
    StateView v;
    if (const char *why = check_state(cam[c], hd.size[c], v)) return err(FE_BAD_ARG, std::string(c ? "right camera: " : "left camera: ") + why);
  }
  // ---- apply
  for (int c = 0; c < 2; c++) {
    int rc = set_state(2 * rig + c, cam[c], hd.size[c]);
    if (rc) return rc;
    FG_CUDA(cudaMemcpy(g_.currid + 2 * rig + c, &hd.currid, sizeof(uint64_t), cudaMemcpyHostToDevice));   // one counter per rig
  }
  return FE_OK;
}

}  // namespace plviwo
