// Host-side trackers of the B200 front end.  Line-by-line counterparts of the reference's glue, with every
// OpenCV call replaced by a kernel launch (fe_kernels.h):
//   ov_core::TrackKLT::feed_new_camera / feed_monocular      open_vins/ov_core/src/track/TrackKLT.cpp:34-200
//   TrackKLT::perform_detection_monocular                    TrackKLT.cpp:395-528
//   Grider_GRID::perform_griding                             open_vins/ov_core/src/track/Grider_GRID.h:74-180
//   TrackKLT::perform_matching                               TrackKLT.cpp:829-886
//   viw::TrackLSD::feed_monocular and helpers                PL-VIWO/src/update/cam/TrackLSD.cpp:70-236, 318-448, 744-830
// The frame-independent work of a frame (copy, equalise, pyramid, edge map, segment extraction) is enqueued at
// submit() on its own streams; collect() runs the state-dependent chain (top-off detection on the previous
// image, LK, RANSAC gate, line association) in frame order.
#include "fe_context.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>

namespace plviwo {

#define FE_CUDA(call)                                  \
  do {                                                 \
    cudaError_t e__ = (call);                          \
    if (e__ != cudaSuccess) return fail(e__, #call);   \
  } while (0)

static inline int align_up(int v, int a) { return (v + a - 1) / a * a; }

namespace {
struct HostTimer {  // accumulates wall time into FeStageTimes::host_ms[idx]
  double *acc;
  std::chrono::steady_clock::time_point t0;
  explicit HostTimer(double *a) : acc(a), t0(std::chrono::steady_clock::now()) {}
  ~HostTimer() { *acc += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); }
};
}  // namespace

// cudaMemcpyAsync with byte accounting (FeStageTimes::h2d_bytes / d2h_bytes) into the calling thread's statistics
#define FE_COPY(st, dst, src, bytes, kind, stream)                               \
  do {                                                                           \
    size_t b__ = (bytes);                                                        \
    if ((kind) == cudaMemcpyHostToDevice) (st).h2d_bytes += b__;                 \
    if ((kind) == cudaMemcpyDeviceToHost) (st).d2h_bytes += b__;                 \
    FE_CUDA(cudaMemcpyAsync((dst), (src), b__, (kind), (stream)));               \
  } while (0)

// Error text of the calling thread; the public entry points copy it into FeContext::last_error, the tracker threads
// into the frame's FrameResult.
static thread_local std::string t_err;

std::string &FeContext::thread_error() { return t_err; }

static inline void cpu_pause() {
#if defined(__x86_64__)
  __builtin_ia32_pause();
#endif
}

// How long a waiting thread spins before it starts yielding.  A handle keeps three host threads busy (caller, point
// tracker, line tracker); on a host with fewer free cores than that (8 ranks on one box) a long pure spin steals the core
// from the thread it is waiting for, while sched_yield on an idle core returns at once — so the pure spin is short.
static const unsigned kSpin = [] {
  const char *e = std::getenv("PLVIWO_SPIN");
  return e ? (unsigned)std::max(0, std::atoi(e)) : 256u;
}();

// ------------------------------------------------------------------------------------------------ WorkQueue
void WorkQueue::push(int v) {
  {
    std::lock_guard<std::mutex> lk(mu_);
    q_.push_back(v);
  }
  n_.fetch_add(1, std::memory_order_release);
  cv_.notify_one();
}
bool WorkQueue::pop(int *v) {
  for (unsigned spins = 0; spins < 20000; spins++) {   // ~1 ms, then sleep on the condition variable
    if (n_.load(std::memory_order_acquire) > 0 || stop_.load(std::memory_order_relaxed)) break;
    if (spins < kSpin) cpu_pause();
    else std::this_thread::yield();
  }
  std::unique_lock<std::mutex> lk(mu_);
  cv_.wait(lk, [this] { return stop_.load() || !q_.empty(); });
  if (q_.empty()) return false;
  *v = q_.front();
  q_.pop_front();
  n_.fetch_sub(1, std::memory_order_relaxed);
  return true;
}
bool WorkQueue::peek(int *v) {
  if (n_.load(std::memory_order_acquire) <= 0) return false;
  std::lock_guard<std::mutex> lk(mu_);
  if (q_.empty()) return false;
  *v = q_.front();
  return true;
}
void WorkQueue::stop() {
  {
    std::lock_guard<std::mutex> lk(mu_);
    stop_.store(true);
  }
  cv_.notify_all();
}

FeContext::FeContext(const FeConfig &cfg, int device)
    : cfg_(cfg), device_(device), W_(cfg.width), H_(cfg.height), Win_(cfg.width), Hin_(cfg.height) {
  if (cfg.downsample) {   // cv::Size(img.cols / 2.0, img.rows / 2.0): truncation (UpdaterCamera.cpp:91)
    W_ = (int)(cfg.width / 2.0);
    H_ = (int)(cfg.height / 2.0);
  }
  currid_ = 4 * (uint64_t)cfg.numaruco + 1;  // TrackBase.cpp:34
  line_currid_ = 1;                          // TrackLSD.cpp:32
}

int FeContext::fail(cudaError_t e, const char *what) {
  t_err = std::string(what) + ": " + cudaGetErrorString(e);
  return FE_CUDA_ERROR;
}
int FeContext::err(int code, const std::string &msg) {
  t_err = msg;
  return code;
}

void FeContext::flush_stats(FeStageTimes &l) {
  std::lock_guard<std::mutex> lk(wstat_mu_);
  for (int i = 0; i < 16; i++) {
    times_.ms[i] += l.ms[i];
    times_.launches[i] += l.launches[i];
    times_.host_ms[i] += l.host_ms[i];
  }
  times_.frames += l.frames;
  times_.kernel_launches_total += l.kernel_launches_total;
  times_.h2d_bytes += l.h2d_bytes;
  times_.d2h_bytes += l.d2h_bytes;
  l = FeStageTimes{};
}
void FeContext::reset_times() {
  std::lock_guard<std::mutex> lk(wstat_mu_);
  times_ = FeStageTimes{};
}

int FeContext::alloc_image(DevImage &im, int w, int h) {
  im.w = w;
  im.h = h;
  im.pitch = align_up(w, 256);
  FE_CUDA(cudaMalloc(&im.p, (size_t)im.pitch * h + 256));
  FE_CUDA(cudaMemset(im.p, 0, (size_t)im.pitch * h + 256));
  return FE_OK;
}

int FeContext::init() {
  FE_CUDA(cudaSetDevice(device_));
  int lo = 0, hi = 0;
  FE_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
  FE_CUDA(cudaStreamCreateWithPriority(&s_pt_, cudaStreamNonBlocking, hi));
  init_device_constants();
  use_graphs_ = std::getenv("PLVIWO_NO_GRAPHS") == nullptr;
  // Line-path batching: the segment extraction of a frame is > 2 ms of kernel TIME (the sequential chain walk), and the
  // device runs a bounded number of kernels at once, so a pipelined stream launches the line paths of consecutive frames
  // together (kernel time per frame / batch).  Needs frames in flight: off for the synchronous drop-in (lookahead 0).
  {
    const char *e = std::getenv("PLVIWO_LINE_BATCH");
    int v = e ? std::atoi(e) : (cfg_.lookahead >= 8 ? 4 : 1);
    v = std::min(v, std::max(cfg_.lookahead / 2, 1));
    line_batch_ = std::max(1, std::min(v, kMaxLineBatch));
  }

  const int nslots = std::max(cfg_.lookahead, 0) + 2;
  slots_.resize(nslots);
  for (int i = 0; i < nslots; i++) slots_[i].index = i;
  for (FrameSlot &s : slots_) {
    int rc = alloc_image(s.raw, W_, H_);
    if (rc) return rc;
    if (cfg_.downsample) {
      rc = alloc_image(s.raw_in, Win_, Hin_);
      if (rc) return rc;
    }
    // cv::buildOpticalFlowPyramid: a level is kept while both sides stay > winSize
    int w = W_, h = H_;
    s.pyr.n = 0;
    for (int l = 0; l <= cfg_.pyr_levels && l < kMaxLevels; l++) {
      rc = alloc_image(s.pyr.lvl[l], w, h);
      if (rc) return rc;
      s.pyr.n = l + 1;
      w = (w + 1) / 2;
      h = (h + 1) / 2;
      if (w <= cfg_.win_size || h <= cfg_.win_size) break;
    }
    if (cfg_.use_lines) {
      rc = alloc_image(s.half, W_ / 2, H_ / 2);
      if (rc) return rc;
      FldBuffers &fb = s.fld;
      if (fb.alloc(W_ / 2, H_ / 2, cfg_.fld_length_threshold, 4096)) return fail(cudaGetLastError(), "FldBuffers::alloc");
      FE_CUDA(cudaMallocHost(&s.h_segs, (size_t)fb.out_cap * sizeof(float4)));
      FE_CUDA(cudaMallocHost(&s.h_fld_counts, 2 * sizeof(int)));
    }
    FE_CUDA(cudaMallocHost(&s.h_raw, (size_t)Win_ * Hin_));
    // One stream per slot and path.  Measured on B200 (profiles/experiments_r1.md): sharing streams between the slots
    // LOWERS single-stream throughput — the line path needs ~2.5 ms of kernel time per frame, so its throughput is
    // (streams in flight) / 2.5 ms: 12 line streams 5.7k frames/s, 16: 7.3k, 24: 8.0k, one per slot (26): 9.3k.
    if (cfg_.use_lines) FE_CUDA(cudaStreamCreateWithPriority(&s.s_line, cudaStreamNonBlocking, lo));
    FE_CUDA(cudaStreamCreateWithPriority(&s.s_a, cudaStreamNonBlocking, lo));
    FE_CUDA(cudaStreamCreateWithPriority(&s.s_b, cudaStreamNonBlocking, lo));
    FE_CUDA(cudaMalloc(&s.d_hist, 256 * sizeof(unsigned)));
    FE_CUDA(cudaMemset(s.d_hist, 0, 256 * sizeof(unsigned)));
    FE_CUDA(cudaMalloc(&s.d_clahe, 64 * 256));
    FE_CUDA(cudaMalloc(&s.d_counters, 4 * sizeof(unsigned)));
    FE_CUDA(cudaMemset(s.d_counters, 0, 4 * sizeof(unsigned)));
    FE_CUDA(cudaMalloc(&s.d_seq, 4 * sizeof(int)));
    FE_CUDA(cudaMemset(s.d_seq, 0, 4 * sizeof(int)));
    FE_CUDA(cudaEventCreateWithFlags(&s.ev_pyr, cudaEventDisableTiming));
    FE_CUDA(cudaEventCreateWithFlags(&s.ev_lines, cudaEventDisableTiming));
    for (auto &e : s.ev_t) FE_CUDA(cudaEventCreate(&e));
  }
  for (auto &e : ev_pt_) FE_CUDA(cudaEventCreate(&e));
  FE_CUDA(cudaEventCreateWithFlags(&ev_sync_, cudaEventDisableTiming));
  FE_CUDA(cudaMallocHost(&h_flag_lk_, 16 * sizeof(int)));
  std::memset(h_flag_lk_, 0, 16 * sizeof(int));

  // detection: FAST output buffers live in the frame slots (pre-detection runs ahead of the tracker)
  max_cells_ = std::max(cfg_.grid_x * cfg_.grid_y, 1);
  max_bands_ = (H_ + kFastBandRows - 1) / kFastBandRows;
  kps_cap_ = W_ * H_ / 4 + 1024;
  cand_cap_ = std::max(max_cells_ * (cfg_.num_features + 1), 1024);   // set_num_features() is checked against this
  if (cand_cap_ > 65536) cand_cap_ = 65536;
  FE_CUDA(cudaMalloc(&d_cells_, (size_t)max_cells_ * sizeof(FastCell)));
  for (FrameSlot &s : slots_) {
    FE_CUDA(cudaMalloc(&s.d_fast_total, 2 * sizeof(unsigned)));
    FE_CUDA(cudaMalloc(&s.d_sort_scratch, (size_t)kps_cap_ * sizeof(unsigned)));
    FE_CUDA(cudaMalloc(&s.d_cand_cnt, (size_t)max_cells_ * sizeof(int)));
    FE_CUDA(cudaMallocHost(&s.h_cand_cnt, (size_t)max_cells_ * sizeof(int)));
    FE_CUDA(cudaMalloc(&s.d_cand_ref, (size_t)cand_cap_ * sizeof(float2)));
    FE_CUDA(cudaMalloc(&s.d_kps, (size_t)kps_cap_ * sizeof(unsigned)));
    FE_CUDA(cudaMallocHost(&s.h_kps, (size_t)kps_cap_ * sizeof(unsigned)));
    FE_CUDA(cudaMalloc(&s.d_band_off, (size_t)max_cells_ * max_bands_ * sizeof(int)));
    FE_CUDA(cudaMalloc(&s.d_band_cnt, (size_t)max_cells_ * max_bands_ * sizeof(int)));
    FE_CUDA(cudaMallocHost(&s.h_band, (size_t)(1 + 2 * max_cells_ * max_bands_) * sizeof(int)));
    FE_CUDA(cudaMalloc(&s.d_cand, (size_t)cand_cap_ * sizeof(float2)));
    FE_CUDA(cudaMallocHost(&s.h_cand_in, (size_t)cand_cap_ * sizeof(float2)));
    FE_CUDA(cudaMallocHost(&s.h_cand_out, (size_t)cand_cap_ * sizeof(float2)));
    FE_CUDA(cudaMallocHost(&s.h_flags, 16 * sizeof(int)));
    std::memset(s.h_flags, 0, 16 * sizeof(int));
    FE_CUDA(cudaEventCreateWithFlags(&s.ev_l0, cudaEventDisableTiming));
    FE_CUDA(cudaEventCreateWithFlags(&s.ev_fast, cudaEventDisableTiming));
    for (auto &e : s.ev_fast_t) FE_CUDA(cudaEventCreate(&e));
    for (auto &e : s.ev_sp_t) FE_CUDA(cudaEventCreate(&e));
  }
  occ_bits_.assign((size_t)((W_ + 63) / 64) * H_, 0);
  layout_cells();
  if (!external_) {
    klt_thread_ = std::thread([this] { klt_main(); });
    line_thread_ = std::thread([this] { line_main(); });
  } else if (cfg_.use_lines) {
    line_thread_ = std::thread([this] { line_main(); });   // the owner queues frames whose points are known (line_q_)
  }

  max_pts_ = std::max(4096, 8 * cfg_.num_features) + 4096 * (cfg_.line_samples > 0 ? 8 : 0);
  FE_CUDA(cudaMalloc(&d_pts0_, (size_t)max_pts_ * sizeof(float2)));
  FE_CUDA(cudaMalloc(&d_pts1_, (size_t)max_pts_ * sizeof(float2)));
  FE_CUDA(cudaMalloc(&d_p0n_, (size_t)max_pts_ * sizeof(float2)));
  FE_CUDA(cudaMalloc(&d_p1n_, (size_t)max_pts_ * sizeof(float2)));
  FE_CUDA(cudaMalloc(&d_status_, (size_t)max_pts_));
  FE_CUDA(cudaMalloc(&d_lk_done_, 4 * sizeof(unsigned)));   // [ordinary, speculative, candidates set 0, set 1]
  FE_CUDA(cudaMemset(d_lk_done_, 0, 4 * sizeof(unsigned)));
  FE_CUDA(cudaMallocHost(&h_sp_pts0_, (size_t)max_pts_ * sizeof(float2)));
  FE_CUDA(cudaMallocHost(&h_sp_pts1_, (size_t)max_pts_ * sizeof(float2)));
  FE_CUDA(cudaMallocHost(&h_sp_p0n_, (size_t)max_pts_ * sizeof(float2)));
  FE_CUDA(cudaMallocHost(&h_sp_p1n_, (size_t)max_pts_ * sizeof(float2)));
  FE_CUDA(cudaMallocHost(&h_sp_status_, (size_t)max_pts_));
  for (FrameSlot &s : slots_) {
    FE_CUDA(cudaMallocHost(&s.h_sc_pts1, (size_t)cand_cap_ * sizeof(float2)));
    FE_CUDA(cudaMallocHost(&s.h_sc_p0n, (size_t)cand_cap_ * sizeof(float2)));
    FE_CUDA(cudaMallocHost(&s.h_sc_p1n, (size_t)cand_cap_ * sizeof(float2)));
    FE_CUDA(cudaMallocHost(&s.h_sc_status, (size_t)cand_cap_));
    FE_CUDA(cudaMalloc(&s.d_sc_done, sizeof(unsigned)));
    FE_CUDA(cudaMemset(s.d_sc_done, 0, sizeof(unsigned)));
  }
  // Speculative tracking is on whenever frames are pipelined: it takes RANSAC and the detection glue off the point
  // tracker's dependent chain (100 -> 67 us per frame) at ~40 % more LK work.  It only pays when the line path keeps up —
  // which it does since consecutive frames share their line-path launches (line_batch_) and the lookahead is deep enough
  // (profiles/experiments_r1.md: 9.3 k -> 12.4 k frames/s).  Results are bit-identical to the synchronous handle's
  // (tests/test_frontend_gpu.py), which (lookahead 0) never has a next frame to speculate into.
  use_spec_ = cfg_.lookahead >= 1;
  FE_CUDA(cudaMallocHost(&h_pts0_, (size_t)max_pts_ * sizeof(float2)));
  FE_CUDA(cudaMallocHost(&h_pts1_, (size_t)max_pts_ * sizeof(float2)));
  FE_CUDA(cudaMallocHost(&h_p0n_, (size_t)max_pts_ * sizeof(float2)));
  FE_CUDA(cudaMallocHost(&h_p1n_, (size_t)max_pts_ * sizeof(float2)));
  FE_CUDA(cudaMallocHost(&h_status_, (size_t)max_pts_));
  FE_CUDA(cudaDeviceSynchronize());
  return FE_OK;
}

FeContext::~FeContext() {
  cudaSetDevice(device_);
  flush_line_batch();   // a line thread waiting for the flag of an unlaunched batch would never be joined
  klt_q_.stop();
  if (klt_thread_.joinable()) klt_thread_.join();
  line_q_.stop();
  if (line_thread_.joinable()) line_thread_.join();
  cudaSetDevice(device_);
  cudaDeviceSynchronize();
  for (FrameSlot &s : slots_) {
    cudaFree(s.raw.p);
    cudaFree(s.raw_in.p);
    for (int l = 0; l < s.pyr.n; l++) cudaFree(s.pyr.lvl[l].p);
    cudaFree(s.half.p);
    s.fld.release();
    cudaFreeHost(s.h_segs); cudaFreeHost(s.h_fld_counts); cudaFreeHost(s.h_raw);
    cudaFree(s.d_sort_scratch); cudaFree(s.d_cand_cnt); cudaFreeHost(s.h_cand_cnt); cudaFree(s.d_cand_ref);
    cudaFree(s.d_fast_total); cudaFree(s.d_kps); cudaFreeHost(s.h_kps); cudaFree(s.d_band_off); cudaFree(s.d_band_cnt);
    cudaFreeHost(s.h_flags);
    cudaFreeHost(s.h_band); cudaFree(s.d_cand); cudaFreeHost(s.h_cand_in); cudaFreeHost(s.h_cand_out);
    if (s.ev_l0) cudaEventDestroy(s.ev_l0);
    if (s.ev_fast) cudaEventDestroy(s.ev_fast);
    for (auto &e : s.ev_fast_t) if (e) cudaEventDestroy(e);
    for (auto &e : s.ev_sp_t) if (e) cudaEventDestroy(e);
    destroy_graphs(s);
    cudaFree(s.d_hist); cudaFree(s.d_counters); cudaFree(s.d_seq); cudaFree(s.d_clahe);
    if (s.s_a) cudaStreamDestroy(s.s_a);
    if (s.s_b) cudaStreamDestroy(s.s_b);
    if (s.s_line) cudaStreamDestroy(s.s_line);
    if (s.ev_pyr) cudaEventDestroy(s.ev_pyr);
    if (s.ev_lines) cudaEventDestroy(s.ev_lines);
    for (auto &e : s.ev_t) if (e) cudaEventDestroy(e);
  }
  for (auto &e : ev_pt_) if (e) cudaEventDestroy(e);
  if (ev_sync_) cudaEventDestroy(ev_sync_);
  cudaFreeHost(h_flag_lk_);
  cudaFree(d_cells_);
  cudaFree(d_lk_done_);
  cudaFreeHost(h_sp_pts0_); cudaFreeHost(h_sp_pts1_); cudaFreeHost(h_sp_p0n_); cudaFreeHost(h_sp_p1n_); cudaFreeHost(h_sp_status_);
  for (FrameSlot &s : slots_) {
    cudaFreeHost(s.h_sc_pts1); cudaFreeHost(s.h_sc_p0n); cudaFreeHost(s.h_sc_p1n); cudaFreeHost(s.h_sc_status);
    cudaFree(s.d_sc_done);
  }
  cudaFree(d_pts0_); cudaFree(d_pts1_); cudaFree(d_p0n_); cudaFree(d_p1n_); cudaFree(d_status_);
  cudaFreeHost(h_pts0_); cudaFreeHost(h_pts1_); cudaFreeHost(h_p0n_); cudaFreeHost(h_p1n_); cudaFreeHost(h_status_);
  if (s_pt_) cudaStreamDestroy(s_pt_);
}

// Low-latency wait: poll an event instead of a blocking synchronise (the tracker thread has nothing else to do)
int FeContext::spin_sync(cudaStream_t st) {
  FE_CUDA(cudaEventRecord(ev_sync_, st));
  while (true) {
    cudaError_t e = cudaEventQuery(ev_sync_);
    if (e == cudaSuccess) return FE_OK;
    if (e != cudaErrorNotReady) return fail(e, "cudaEventQuery");
    cpu_pause();
  }
}

// Waits for a k_signal sequence number.  Polls memory only; every ~2M polls it asks the driver whether the stream
// died, so a faulting kernel turns into an error instead of a hang.
int FeContext::wait_flag(volatile int *flag, int value, cudaStream_t st, std::string *err) {
  unsigned spins = 0;
  while (*flag != value) {
    // a few microseconds of pure spinning (the usual wait is shorter than a context switch), then let other threads of
    // an oversubscribed host run between polls
    if (spins < kSpin) cpu_pause();
    else std::this_thread::yield();
    if ((++spins & 0x1fffff) == 0) {
      cudaError_t e = cudaStreamQuery(st);
      if (e != cudaSuccess && e != cudaErrorNotReady) {
        *err = std::string("stream failed while waiting for a completion signal: ") + cudaGetErrorString(e);
        return FE_CUDA_ERROR;
      }
    }
  }
  return FE_OK;
}

int FeContext::set_calib(const double K[4], const double D[4]) {
  for (int i = 0; i < 4; i++) {
    cfg_.K[i] = K[i];
    cfg_.D[i] = D[i];
  }
  return FE_OK;
}

// The tracker state belongs to the tracker threads while frames are in flight: the two setters below are only legal
// between frames (nothing submitted and not yet collected), which is the only place the reference can call them too.
int FeContext::change_feat_id(uint64_t id_old, uint64_t id_new) {  // TrackBase.cpp:267-285 (tracker side)
  if (!queue_.empty()) {
    last_error = "change_feat_id: collect the pending frames first";
    return FE_BAD_ARG;
  }
  for (uint64_t &id : ids_last_)
    if (id == id_old) id = id_new;
  if (cur_res_ != &state_res_) {   // keep get_last_obs / get_last_ids in step
    FrameResult &r = const_cast<FrameResult &>(*cur_res_);
    for (uint64_t &id : r.obs_ids)
      if (id == id_old) id = id_new;
  }
  for (uint64_t &id : state_res_.obs_ids)
    if (id == id_old) id = id_new;
  return FE_OK;
}
int FeContext::set_num_features(int n) {
  if (!queue_.empty()) {
    last_error = "set_num_features: collect the pending frames first";
    return FE_BAD_ARG;
  }
  if (n < 1) {
    last_error = "set_num_features: bad feature count";
    return FE_BAD_ARG;
  }
  // the candidate table (cells x num_features_grid) of the new layout must fit the buffers sized at creation
  if (cand_table_size(n) > cand_cap_) {
    last_error = "set_num_features: the candidate table of that feature count exceeds the capacity this handle was created with";
    return FE_BAD_ARG;
  }
  cfg_.num_features = n;
  return FE_OK;
}

// cells x num_features_grid of the Grider_GRID layout for a feature count (layout_cells)
int FeContext::cand_table_size(int num_features) const {
  const int gx = cfg_.grid_x, gy = cfg_.grid_y;
  int ggx = gx, ggy = gy;
  if (num_features < ggx * ggy) {
    double ratio = (double)ggx / (double)ggy;
    ggy = (int)std::ceil(std::sqrt(num_features / ratio));
    ggx = (int)std::ceil(ggy * ratio);
  }
  const int nfg = (int)((double)num_features / (double)(ggx * ggy)) + 1;
  const int csx = W_ / ggx, csy = H_ / ggy;
  int ncell = 0;
  if (csx > 0 && csy > 0)
    for (int x = 0; x < gx; x++)
      for (int y = 0; y < gy; y++)
        if (x * csx + csx <= W_ && y * csy + csy <= H_) ncell++;
  return ncell * nfg;
}

int FeContext::set_currid(uint64_t id) {
  if (!queue_.empty()) {
    last_error = "set_currid: collect the pending frames first";
    return FE_BAD_ARG;
  }
  currid_ = id;
  return FE_OK;
}

// cv::undistortPoints on one point (Appendix A6) — only for the two endpoints of each line row
void FeContext::undistort_host(const double K[4], const double D[4], float u, float v, float &un, float &vn) {
  double x0 = ((double)u - K[2]) / K[0], y0 = ((double)v - K[3]) / K[1];
  double x = x0, y = y0;
  for (int j = 0; j < 5; j++) {
    double r2 = x * x + y * y;
    double icdist = 1.0 / (1.0 + (D[1] * r2 + D[0]) * r2);
    double dx = 2 * D[2] * x * y + D[3] * (r2 + 2 * x * x);
    double dy = D[2] * (r2 + 2 * y * y) + 2 * D[3] * x * y;
    x = (x0 - dx) * icdist;
    y = (y0 - dy) * icdist;
  }
  un = (float)x;
  vn = (float)y;
}

// ------------------------------------------------------------------------------------------------ submit
// The frame-independent work of a frame, as three recordable paths.  Each is issued on a per-slot stream either
// directly (first use of a slot, or while the cell layout changes) or as a replay of a CUDA graph captured from
// exactly these calls: ~30 launches per frame collapse into three graph launches.  Stage-timing events are part of
// the paths, so timings can be read whether or not the graphs are used.
int FeContext::record_image_path(FrameSlot &s, cudaStream_t st) {
  const int eq = cfg_.histogram_method == FE_HIST_HISTOGRAM ? 1 : (cfg_.histogram_method == FE_HIST_CLAHE ? 2 : 0);
  if (eq == 1) launch_hist(s.raw, s.d_hist, st);
  if (eq == 2) launch_clahe_lut(s.raw, s.d_clahe, st);
  if (timing) cudaEventRecord(s.ev_t[2], st);
  DevImage half = cfg_.use_lines ? s.half : DevImage();
  launch_eq_pyr1(s.raw, s.d_hist, s.d_counters, eq, s.pyr.lvl[0], s.pyr.n > 1 ? s.pyr.lvl[1] : DevImage(), half, st, s.d_clahe);
  if (timing) cudaEventRecord(s.ev_t[3], st);
  if (s.pyr.n > 2) launch_pyr_rest(s.pyr, s.d_counters + 1, st);
  if (timing) cudaEventRecord(s.ev_t[4], st);
  FE_CUDA(cudaGetLastError());
  return FE_OK;
}

int FeContext::record_fast_path(FrameSlot &s, cudaStream_t st) {
  const int ncell = (int)cells_.size(), nb = cells_nb_;
  if (ncell > 0) {
    const int nfg = cells_nfg_, ntab_c = ncell * nfg;
    FE_CUDA(cudaMemsetAsync(s.d_fast_total, 0, 2 * sizeof(unsigned), st));
    if (timing) cudaEventRecord(s.ev_fast_t[0], st);
    launch_fast(s.pyr.lvl[0], d_cells_, ncell, nb, cells_csx_, cfg_.fast_threshold, s.d_fast_total, s.d_band_off, s.d_band_cnt,
                s.d_kps, kps_cap_, st);
    // Grider_GRID.h:128-133 and :163-179 on the device: per-cell std::sort + top num_features_grid, then cornerSubPix of
    // every survivor.  Only the candidate table (a few KB) goes back to the host.
    launch_fast_select(d_cells_, ncell, nb, s.d_fast_total, s.d_band_off, s.d_band_cnt, s.d_kps, kps_cap_, s.d_sort_scratch, nfg,
                       s.d_cand, s.d_cand_cnt, st);
    if (timing) cudaEventRecord(s.ev_fast_t[1], st);
    if (timing) cudaEventRecord(s.ev_sp_t[0], st);
    launch_corner_subpix(s.pyr.lvl[0], s.d_cand, s.d_cand_ref, ntab_c, st, s.d_cand_cnt, nfg);
    if (timing) cudaEventRecord(s.ev_sp_t[1], st);
    FE_CUDA(cudaMemcpyAsync(s.h_cand_cnt, s.d_cand_cnt, (size_t)ncell * sizeof(int), cudaMemcpyDeviceToHost, st));
    FE_CUDA(cudaMemcpyAsync(s.h_cand_in, s.d_cand, (size_t)ntab_c * sizeof(float2), cudaMemcpyDeviceToHost, st));
    FE_CUDA(cudaMemcpyAsync(s.h_cand_out, s.d_cand_ref, (size_t)ntab_c * sizeof(float2), cudaMemcpyDeviceToHost, st));
    if (taps) {   // debug tap: every cell's full corner list in the reference's order
      const int ntab = ncell * nb;
      FE_CUDA(cudaMemcpyAsync(s.h_band, s.d_fast_total, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
      FE_CUDA(cudaMemcpyAsync(s.h_band + 1, s.d_band_off, (size_t)ntab * sizeof(int), cudaMemcpyDeviceToHost, st));
      FE_CUDA(cudaMemcpyAsync(s.h_band + 1 + ntab, s.d_band_cnt, (size_t)ntab * sizeof(int), cudaMemcpyDeviceToHost, st));
      FE_CUDA(cudaMemcpyAsync(s.h_kps, s.d_kps, (size_t)kps_cap_ * sizeof(unsigned), cudaMemcpyDeviceToHost, st));
    }
  }
  s.fast_taps = taps;
  launch_signal_inc(&s.h_flags[0], s.d_seq + 0, st);
  FE_CUDA(cudaGetLastError());
  return FE_OK;
}

int FeContext::record_line_path(FrameSlot &s, cudaStream_t st) {
  if (timing) cudaEventRecord(s.ev_t[5], st);
  launch_canny(s.half, cfg_.canny_th1, cfg_.canny_th2, s.fld, st);
  if (timing) cudaEventRecord(s.ev_t[6], st);
  launch_fld(s.half, cfg_.fld_length_threshold, cfg_.fld_distance_threshold, s.fld, st, timing ? &s.ev_t[8] : nullptr);
  if (timing) cudaEventRecord(s.ev_t[7], st);
  FE_CUDA(cudaMemcpyAsync(s.h_fld_counts, s.fld.counters + 3, 2 * sizeof(int), cudaMemcpyDeviceToHost, st));
  FE_CUDA(cudaMemcpyAsync(s.h_segs, s.fld.out, 1024 * sizeof(float4), cudaMemcpyDeviceToHost, st));
  launch_signal_inc(&s.h_flags[2], s.d_seq + 2, st);
  FE_CUDA(cudaGetLastError());
  return FE_OK;
}

void FeContext::destroy_graphs(FrameSlot &s) {
  if (s.g_image) cudaGraphExecDestroy(s.g_image);
  if (s.g_fast) cudaGraphExecDestroy(s.g_fast);
  if (s.g_lines) cudaGraphExecDestroy(s.g_lines);
  s.g_image = s.g_fast = s.g_lines = nullptr;
  s.graph_version = -1;
}

int FeContext::build_graphs(FrameSlot &s) {
  destroy_graphs(s);
  auto capture = [&](cudaStream_t st, int (FeContext::*fn)(FrameSlot &, cudaStream_t), cudaGraphExec_t *out) -> int {
    // thread-local capture mode: the worker thread keeps issuing its own CUDA calls meanwhile
    FE_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    int rc = (this->*fn)(s, st);
    cudaGraph_t g = nullptr;
    cudaError_t e = cudaStreamEndCapture(st, &g);
    if (rc) {
      if (g) cudaGraphDestroy(g);
      return rc;
    }
    if (e != cudaSuccess) return fail(e, "cudaStreamEndCapture");
    e = cudaGraphInstantiate(out, g, 0);
    cudaGraphDestroy(g);
    if (e != cudaSuccess) return fail(e, "cudaGraphInstantiate");
    return FE_OK;
  };
  int rc = capture(s.s_a, &FeContext::record_image_path, &s.g_image);
  if (rc) return rc;
  rc = capture(s.s_b, &FeContext::record_fast_path, &s.g_fast);
  if (rc) return rc;
  if (cfg_.use_lines) {
    rc = capture(s.s_line, &FeContext::record_line_path, &s.g_lines);
    if (rc) return rc;
  }
  s.graph_version = layout_version_;
  return FE_OK;
}

int FeContext::enqueue_frame_independent(FrameSlot &s) {
  s.timed = timing;
  const bool lines = cfg_.use_lines && s.has_vp;
  // a slot replays its graphs from its second use on (the first use runs the same calls directly, which also gets
  // every lazy one-time initialisation out of the way before anything is captured)
  bool replay = use_graphs_ && s.warmed && !timing && !taps;   // stage timing / taps: direct launches of the same calls
  if (replay && s.graph_version != layout_version_) {
    int rc = build_graphs(s);
    if (rc) return rc;
  }
  if (replay) {
    FE_CUDA(cudaGraphLaunch(s.g_image, s.s_a));
  } else {
    int rc = record_image_path(s, s.s_a);
    if (rc) return rc;
  }
  FE_CUDA(cudaEventRecord(s.ev_pyr, s.s_a));
  FE_CUDA(cudaStreamWaitEvent(s.s_b, s.ev_pyr, 0));
  if (replay) {
    FE_CUDA(cudaGraphLaunch(s.g_fast, s.s_b));
  } else {
    int rc = record_fast_path(s, s.s_b);
    if (rc) return rc;
  }
  s.seq_fast++;
  FE_CUDA(cudaEventRecord(s.ev_fast, s.s_b));
  bool batched = false;
  if (lines) {
    s.seq_lines++;
    s.line_timed = 0;
    if (line_batch_ > 1 && !taps) {   // joins the batch; launched when it is full (or when collect needs it)
      batched = true;
      s.line_pending = true;
      pending_lines_.push_back(s.index);
      if ((int)pending_lines_.size() >= line_batch_) {
        int rc = flush_line_batch();
        if (rc) return rc;
      }
    } else {
      FE_CUDA(cudaStreamWaitEvent(s.s_line, s.ev_pyr, 0));
      if (replay) {
        FE_CUDA(cudaGraphLaunch(s.g_lines, s.s_line));
      } else {
        int rc = record_line_path(s, s.s_line);
        if (rc) return rc;
        if (timing) s.line_timed = 1;
      }
      FE_CUDA(cudaEventRecord(s.ev_lines, s.s_line));
      s.lines_recorded = true;
    }
  }
  s.warmed = true;
  // bookkeeping (identical for both ways of issuing the work)
  const int ncell = (int)cells_.size(), ntab = ncell * cells_nb_;
  mst_.kernel_launches_total += (cfg_.histogram_method != FE_HIST_NONE ? 1 : 0) + 1 + std::max(s.pyr.n - 2, 0) +
                                 (ncell > 0 ? 3 : 0) + 1 + (lines && !batched ? 13 : 0);
  (void)ntab;
  if (ncell > 0) mst_.d2h_bytes += (size_t)ncell * sizeof(int) + (size_t)2 * ncell * cells_nfg_ * sizeof(float2);
  if (lines) mst_.d2h_bytes += 2 * sizeof(int) + 1024 * sizeof(float4);
  return FE_OK;
}

int FeContext::flush_line_batch() {
  const int n = (int)pending_lines_.size();
  if (n == 0) return FE_OK;
  cudaStream_t st = slots_[pending_lines_[0]].s_line;
  FldBatch b;
  b.n = n;
  for (int k = 0; k < n; k++) {
    FrameSlot &s = slots_[pending_lines_[k]];
    FE_CUDA(cudaStreamWaitEvent(st, s.ev_pyr, 0));
    b.half[k] = s.half;
    b.f[k] = s.fld;
  }
  FrameSlot &first = slots_[pending_lines_[0]];
  const bool timed = timing;
  if (timed) cudaEventRecord(first.ev_t[5], st);
  launch_canny_batch(b, cfg_.canny_th1, cfg_.canny_th2, st);
  if (timed) cudaEventRecord(first.ev_t[6], st);
  launch_fld_batch(b, cfg_.fld_length_threshold, cfg_.fld_distance_threshold, st, timed ? &first.ev_t[8] : nullptr);
  if (timed) {
    cudaEventRecord(first.ev_t[7], st);
    first.line_timed = n;
  }
  for (int k = 0; k < n; k++) {
    FrameSlot &s = slots_[pending_lines_[k]];
    FE_CUDA(cudaMemcpyAsync(s.h_fld_counts, s.fld.counters + 3, 2 * sizeof(int), cudaMemcpyDeviceToHost, st));
    FE_CUDA(cudaMemcpyAsync(s.h_segs, s.fld.out, 1024 * sizeof(float4), cudaMemcpyDeviceToHost, st));
    launch_signal_inc(&s.h_flags[2], s.d_seq + 2, st);
    FE_CUDA(cudaEventRecord(s.ev_lines, st));
    s.lines_recorded = true;
    s.line_pending = false;
  }
  FE_CUDA(cudaGetLastError());
  mst_.kernel_launches_total += 11 + n + (n >= 16 ? 1 : 0);   // canny, 5 x components, walk (+ thread walk for a large batch), order, segments, compact + one signal per frame
  pending_lines_.clear();
  return FE_OK;
}

// The second half of the speculation.  Every refined corner candidate of the PREVIOUS submitted frame — the only points
// the top-off detection can add when this frame is tracked — is tracked into this frame straight from that frame's
// device-side candidate table.  It depends on nothing but the two frames' images, so it is issued here, at submit time,
// as part of this frame's state-independent work (typically many frames ahead of the trackers); the point tracker only
// reads the few results that belong to candidates the detection really adds.
int FeContext::track_candidates(FrameSlot &prev, FrameSlot &s) {
  s.sc_prev = -1;
  if (!use_spec_ || cfg_.line_samples > 0) return FE_OK;
  LkParams prm;
  prm.win = cfg_.win_size;
  prm.max_level = cfg_.pyr_levels;
  prm.max_count = 30;
  prm.eps_sq = 0.01f * 0.01f;
  prm.min_eig = 1e-4f;
  prm.undistort = 1;
  for (int i = 0; i < 4; i++) { prm.K[i] = s.K[i]; prm.D[i] = s.D[i]; }
  const int ntab = prev.predet_ncell * prev.predet_nfg;
  if (ntab <= 0 || ntab > cand_cap_ || prev.predet_num_features != cfg_.num_features || !lk_table_mode_ok(prm, prev.pyr.n))
    return FE_OK;
  FE_CUDA(cudaStreamWaitEvent(s.s_b, prev.ev_fast, 0));   // the candidate table of the previous frame
  launch_lk(prev.pyr, s.pyr, prev.d_cand_ref, s.h_sc_pts1, s.h_sc_status, s.h_sc_p0n, s.h_sc_p1n, ntab, prm, s.s_b, &s.h_flags[3],
            ++s.seq_sc, s.d_sc_done, prev.d_cand_cnt, prev.predet_nfg, true);
  FE_CUDA(cudaGetLastError());
  mst_.kernel_launches_total++;
  mst_.d2h_bytes += (size_t)ntab * (3 * sizeof(float2) + 1);
  s.sc_prev = prev.index;
  s.sc_ntab = ntab;
  return FE_OK;
}

int FeContext::submit(double t, const uint8_t *image, int stride, bool on_device, const uint8_t *mask, int mask_stride,
                      const double vp[6]) {
  int si = -1;
  int rc = submit_impl(t, image, stride, on_device, mask, mask_stride, vp, &si);
  if (rc) {
    last_error = t_err;
    if (si >= 0 && !external_) {   // a failed submit leaves no trace: the slot is free again, nothing of it is pending
      FrameSlot &s = slots_[si];
      cudaStreamSynchronize(s.s_a);
      cudaStreamSynchronize(s.s_b);
      if (s.s_line) cudaStreamSynchronize(s.s_line);
      cudaGetLastError();
      pending_lines_.erase(std::remove(pending_lines_.begin(), pending_lines_.end(), si), pending_lines_.end());
      s.line_pending = false;
      s.busy = false;
    }
  }
  flush_stats(mst_);
  return rc;
}

int FeContext::submit_impl(double t, const uint8_t *image, int stride, bool on_device, const uint8_t *mask, int mask_stride,
                           const double vp[6], int *slot_out) {
  HostTimer ht(&mst_.host_ms[FE_HOST_SUBMIT]);
  FE_CUDA(cudaSetDevice(device_));
  int si = -1;
  for (int i = 0; i < (int)slots_.size(); i++)
    if (!slots_[i].busy && i != last_slot_) { si = i; break; }
  if (si < 0) return err(FE_BAD_ARG, "submit: lookahead window full (collect a frame first)");
  FrameSlot &s = slots_[si];
  if (slot_out) *slot_out = si;
  s.busy = true;
  s.timestamp = t;
  s.res.clear();
  // the slot's previous frame: its FAST / selection / sub-pixel path (s_b) and line path read level 0 / the half image that
  // the image path (s_a) is about to overwrite
  if (s.warmed) {
    FE_CUDA(cudaStreamWaitEvent(s.s_a, s.ev_fast, 0));
    if (cfg_.use_lines && s.lines_recorded) FE_CUDA(cudaStreamWaitEvent(s.s_a, s.ev_lines, 0));
  }
  for (int i = 0; i < 4; i++) {
    s.K[i] = cfg_.K[i];
    s.D[i] = cfg_.D[i];
  }
  s.has_vp = vp != nullptr;
  if (vp) std::memcpy(s.vp, vp, sizeof(s.vp));
  if (mask) {
    s.mask.resize((size_t)W_ * H_);
    if (cfg_.downsample) {   // cv::pyrDown(mask, .., Size(cols / 2.0, rows / 2.0)) (UpdaterCamera.cpp:92-93)
      pyr_down_host(mask, Win_, Hin_, mask_stride, s.mask.data(), W_, H_);
    } else {
      for (int y = 0; y < H_; y++) std::memcpy(&s.mask[(size_t)y * W_], mask + (size_t)y * mask_stride, W_);
    }
  } else {
    s.mask.clear();
  }
  if (timing) cudaEventRecord(s.ev_t[0], s.s_a);
  DevImage &dst = cfg_.downsample ? s.raw_in : s.raw;
  if (on_device) {
    FE_CUDA(cudaMemcpy2DAsync(dst.p, dst.pitch, image, stride, Win_, Hin_, cudaMemcpyDeviceToDevice, s.s_a));
  } else {
    cudaPointerAttributes attr;
    bool pinned = cudaPointerGetAttributes(&attr, image) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    const uint8_t *src = image;
    int sstride = stride;
    if (!pinned) {  // pageable caller memory: stage through the slot's pinned buffer
      for (int y = 0; y < Hin_; y++) std::memcpy(s.h_raw + (size_t)y * Win_, image + (size_t)y * stride, Win_);
      src = s.h_raw;
      sstride = Win_;
    }
    if (sstride == Win_ && dst.pitch == Win_) FE_CUDA(cudaMemcpyAsync(dst.p, src, (size_t)Win_ * Hin_, cudaMemcpyHostToDevice, s.s_a));   // one contiguous transfer
    else FE_CUDA(cudaMemcpy2DAsync(dst.p, dst.pitch, src, sstride, Win_, Hin_, cudaMemcpyHostToDevice, s.s_a));
    mst_.h2d_bytes += (size_t)Win_ * Hin_;
  }
  if (cfg_.downsample) {   // cv::pyrDown(img, .., Size(cols / 2.0, rows / 2.0)) (UpdaterCamera.cpp:90-91)
    launch_pyr_down(s.raw_in, s.raw, s.s_a);
    mst_.kernel_launches_total++;
  }
  if (timing) cudaEventRecord(s.ev_t[1], s.s_a);
  int rc = enqueue_fast_all_cells(s);   // layout bookkeeping first: it decides whether the graphs are still valid
  if (rc) return rc;
  rc = enqueue_frame_independent(s);
  if (rc) return rc;
  s.sc_prev = -1;
  if (slot_out) *slot_out = si;
  if (external_) return FE_OK;   // the owner (FeStereo) runs the state machine and releases the slot
  if (prev_submit_slot_ >= 0) {
    rc = track_candidates(slots_[prev_submit_slot_], s);
    if (rc) return rc;
  }
  prev_submit_slot_ = si;
  queue_.push_back(si);
  s.stage.store(1, std::memory_order_release);
  klt_q_.push(si);
  return FE_OK;
}

// ------------------------------------------------------------------------------------------ pre-detection
void FeContext::layout_cells() {
  // Grider_GRID geometry (Grider_GRID.h:88-100): the grider may shrink ITS grid when num_features < grid_x * grid_y
  // while the cell indices still come from the caller's grid; cells that leave the image are skipped (:117-118)
  const int gx = cfg_.grid_x, gy = cfg_.grid_y;
  int ggx = gx, ggy = gy;
  if (cfg_.num_features < ggx * ggy) {
    double ratio = (double)ggx / (double)ggy;
    ggy = (int)std::ceil(std::sqrt(cfg_.num_features / ratio));
    ggx = (int)std::ceil(ggy * ratio);
  }
  cells_nfg_ = (int)((double)cfg_.num_features / (double)(ggx * ggy)) + 1;
  cells_csx_ = W_ / ggx;
  cells_csy_ = H_ / ggy;
  cells_.clear();
  cell_of_loc_.assign((size_t)gx * gy, -1);
  if (cells_csx_ > 0 && cells_csy_ > 0) {
    for (int x = 0; x < gx; x++)
      for (int y = 0; y < gy; y++) {
        int px = x * cells_csx_, py = y * cells_csy_;
        if (px + cells_csx_ > W_ || py + cells_csy_ > H_) continue;
        if ((int)cells_.size() >= max_cells_) continue;
        cell_of_loc_[(size_t)x * gy + y] = (int)cells_.size();
        cells_.push_back(FastCell{px, py, cells_csx_, cells_csy_});
      }
  }
  cells_nb_ = cells_csy_ > 0 ? (cells_csy_ + kFastBandRows - 1) / kFastBandRows : 0;
  cells_num_features_ = cfg_.num_features;
  cells_uploaded_ = false;
}

// Host-side part of starting a frame's pre-detection: make sure the device cell table matches the current
// num_features, remember the layout the frame is processed with.  The FAST launch itself is record_fast_path().
int FeContext::enqueue_fast_all_cells(FrameSlot &s) {
  if (cells_num_features_ != cfg_.num_features) {
    FE_CUDA(cudaDeviceSynchronize());   // d_cells_ may still be read by an earlier frame's FAST
    layout_cells();
    layout_version_++;
  }
  if (!cells_uploaded_ && !cells_.empty()) {
    FE_CUDA(cudaMemcpy(d_cells_, cells_.data(), cells_.size() * sizeof(FastCell), cudaMemcpyHostToDevice));
    cells_uploaded_ = true;
  }
  s.cells = cells_;
  s.cell_of_loc = cell_of_loc_;
  s.predet_ncell = (int)cells_.size();
  s.predet_nb = cells_nb_;
  s.predet_nfg = cells_nfg_;
  s.predet_num_features = cfg_.num_features;
  s.predet_state.store(1);
  return FE_OK;
}

// The frame's candidate table (per cell: the first num_features_grid corners after the reference's std::sort, before and
// after cornerSubPix) was produced on the device by record_fast_path; wait for its completion signal and unpack it.
// Called by the thread that needs the table (the point tracker; set_state).
int FeContext::wait_predetection(FrameSlot &s) {
  const int st = s.predet_state.load(std::memory_order_acquire);
  if (st == 2) return FE_OK;
  if (st == 0) return err(FE_INTERNAL, "pre-detection was never queued for this frame");
  if (wait_flag(&s.h_flags[0], s.seq_fast, s.s_b, &t_err)) return FE_CUDA_ERROR;
  const int ncell = s.predet_ncell, nb = s.predet_nb, nfg = s.predet_nfg;
  // the table itself (h_cand_cnt / h_cand_in / h_cand_out, fixed stride nfg per cell) is read in place by the top-off
  // detection, and only for the cells that turn out to be valid
  (void)nfg;
  s.cell_kps_tap.clear();
  s.cell_kps_first.assign(ncell + 1, 0);
  if (s.fast_taps && ncell > 0) {
    const int ntab = ncell * nb;
    const int total = std::min(s.h_band[0], kps_cap_);
    const int *band_off = s.h_band + 1, *band_cnt = s.h_band + 1 + ntab;
    for (int c = 0; c < ncell; c++) {
      for (int b = 0; b < nb; b++) {
        const int off = band_off[c * nb + b], cnt = band_cnt[c * nb + b];
        for (int k = 0; k < cnt && off + k < total; k++) {
          const unsigned v = s.h_kps[off + k];
          s.cell_kps_tap.insert(s.cell_kps_tap.end(), {(int)(v & 0xfff), (int)((v >> 12) & 0xfff), (int)(v >> 24)});
        }
      }
      s.cell_kps_first[c + 1] = (int)s.cell_kps_tap.size() / 3;
    }
  }
  s.predet_state.store(2, std::memory_order_release);
  return FE_OK;
}

FeStageTimes FeContext::snapshot_times() {
  std::lock_guard<std::mutex> lk(wstat_mu_);
  FeStageTimes t = times_;
  return t;
}

static void acc_time(FeStageTimes &t, int stage, cudaEvent_t a, cudaEvent_t b) {
  float ms = 0;
  if (cudaEventElapsedTime(&ms, a, b) == cudaSuccess) {
    t.ms[stage] += ms;
    t.launches[stage]++;
  } else {
    cudaGetLastError();
  }
}

// ------------------------------------------------------------------------------------- tracker threads
// Point tracker: frames in submission order.  Owns pts_last_ / ids_last_ / currid_ while frames are in flight.
void FeContext::klt_main() {
  cudaSetDevice(device_);
  int si;
  while (klt_q_.pop(&si)) {
    FrameSlot &cur = slots_[si];
    cur.res.info.timestamp = cur.timestamp;
    int rc = cudaStreamWaitEvent(s_pt_, cur.ev_pyr, 0) == cudaSuccess ? FE_OK : fail(cudaGetLastError(), "cudaStreamWaitEvent");
    if (rc == FE_OK) rc = klt_feed(cur);
    if (rc) {
      cur.res.rc = rc;
      cur.res.error = t_err;
    }
    cur.res.obs = pts_last_;
    cur.res.obs_ids = ids_last_;
    klt_last_slot_ = si;   // move forward in time (TrackKLT.cpp:182-189)
    flush_stats(kst_);
    if (rc == FE_OK && cfg_.use_lines && cur.has_vp) {
      cur.stage.store(2, std::memory_order_release);
      line_q_.push(si);
    } else {
      cur.stage.store(3, std::memory_order_release);
    }
  }
}

// Line tracker: runs one frame behind the point tracker at most (it needs that frame's tracked points).
void FeContext::line_main() {
  cudaSetDevice(device_);
  int si;
  while (line_q_.pop(&si)) {
    FrameSlot &cur = slots_[si];
    int rc = lsd_feed(cur);
    if (rc) {
      cur.res.rc = rc;
      cur.res.error = t_err;
    }
    flush_stats(lst_);
    cur.stage.store(3, std::memory_order_release);
  }
}

int FeContext::collect(FeFrameInfo *info) {
  int rc = collect_impl(info);
  if (rc) last_error = t_err;
  flush_stats(mst_);
  return rc;
}

int FeContext::collect_impl(FeFrameInfo *info) {
  HostTimer ht(&mst_.host_ms[FE_HOST_COLLECT]);
  FE_CUDA(cudaSetDevice(device_));
  if (queue_.empty()) return err(FE_BAD_ARG, "collect: nothing submitted");
  const int si = queue_.front();
  queue_.erase(queue_.begin());
  FrameSlot &cur = slots_[si];
  if (cur.line_pending) {   // its line batch never filled up: launch what is there
    int rc = flush_line_batch();
    if (rc) return rc;
  }
  // wait for the tracker threads: spin (the result is normally there already, or a few microseconds away), then yield
  for (unsigned spins = 0; cur.stage.load(std::memory_order_acquire) != 3; spins++) {
    if (spins < kSpin) cpu_pause();
    else std::this_thread::yield();
  }
  cur.stage.store(0, std::memory_order_relaxed);
  // the candidate tracks into this frame read the previous frame's pyramid and candidate table: that slot is released
  // below, so the launch must be over (it was issued at submit time and normally finished long ago)
  if (cur.sc_prev >= 0 && wait_flag(&cur.h_flags[3], cur.seq_sc, cur.s_b, &t_err)) return FE_CUDA_ERROR;
  cur_slot_ = si;
  cur_res_ = &cur.res;
  FrameResult &res = cur.res;
  // the previous collected frame's slot becomes free: its pyramid is no longer the point tracker's "last" image and its
  // rows are no longer exposed
  if (last_slot_ >= 0) slots_[last_slot_].busy = false;
  last_slot_ = si;
  if (res.rc) return err(res.rc, res.error);
  if (cur.timed) {
    FE_CUDA(cudaEventSynchronize(cur.ev_pyr));
    acc_time(mst_, FE_STAGE_H2D, cur.ev_t[0], cur.ev_t[1]);
    if (cur.predet_ncell > 0) {
      FE_CUDA(cudaStreamSynchronize(cur.s_b));
      acc_time(mst_, FE_STAGE_FAST, cur.ev_fast_t[0], cur.ev_fast_t[1]);
      acc_time(mst_, FE_STAGE_SUBPIX, cur.ev_sp_t[0], cur.ev_sp_t[1]);
    }
    if (cfg_.histogram_method != FE_HIST_NONE) acc_time(mst_, FE_STAGE_HIST, cur.ev_t[1], cur.ev_t[2]);
    acc_time(mst_, FE_STAGE_EQ_PYR, cur.ev_t[2], cur.ev_t[3]);
    acc_time(mst_, FE_STAGE_PYR_REST, cur.ev_t[3], cur.ev_t[4]);
  }
  // line stages: one set of events per LAUNCH — a batched line path is timed on the first frame of its batch, so
  // launches[] counts batches and ms[] / launches[] is the duration of a launch that carries line_timed frames
  if (cur.line_timed > 0) {
    acc_time(mst_, FE_STAGE_CANNY, cur.ev_t[5], cur.ev_t[6]);
    acc_time(mst_, FE_STAGE_FLD, cur.ev_t[6], cur.ev_t[7]);
    acc_time(mst_, FE_STAGE_FLD_CCL, cur.ev_t[6], cur.ev_t[8]);
    acc_time(mst_, FE_STAGE_FLD_WALK, cur.ev_t[8], cur.ev_t[9]);
    acc_time(mst_, FE_STAGE_FLD_SEG, cur.ev_t[9], cur.ev_t[7]);
    mst_.launches[FE_STAGE_LINE_FRAMES] += (uint64_t)cur.line_timed;
    cur.line_timed = 0;
  }
  mst_.frames++;
  res.info.n_point_rows = (int)res.point_rows.size();
  res.info.n_line_rows = (int)res.line_rows.size();
  res.info.n_last_obs = (int)res.obs.size();
  if (info) *info = res.info;
  return FE_OK;
}

int FeContext::play(int n_frames, const uint8_t *const *images, int stride, bool on_device, const double *timestamps,
                    const double *vps, FePlayStats *out) {
  if (!queue_.empty()) {
    last_error = "play: frames submitted with plviwo_fe_submit are still pending";
    return FE_BAD_ARG;
  }
  FePlayStats st;
  std::memset(&st, 0, sizeof(st));
  const int la = std::max(cfg_.lookahead, 0);
  int sub = 0;
  for (int i = 0; i < n_frames; i++) {
    while (sub < n_frames && sub <= i + la) {
      int rc = submit(timestamps[sub], images[sub], stride, on_device, nullptr, 0, vps ? vps + 6 * (size_t)sub : nullptr);
      if (rc) return rc;
      sub++;
    }
    FeFrameInfo info;
    int rc = collect(&info);
    if (rc) return rc;
    const FrameResult &r = result();
    st.frames++;
    st.point_rows += r.point_rows.size();
    st.line_rows += r.line_rows.size();
    st.resets += info.reset ? 1 : 0;
    for (const FePointRow &p : r.point_rows) st.checksum += (double)p.id + p.u + p.v;
    for (const FeLineRow &l : r.line_rows) st.checksum += (double)l.id + l.line[0] + l.line[1] + l.line[2] + l.line[3];
  }
  if (out) *out = st;
  return FE_OK;
}

int FeContext::feed(double t, const uint8_t *image, int w, int h, int stride, bool on_device, const uint8_t *mask,
                    int mask_stride, const double vp[6], FeFrameInfo *info) {
  if (!image || w != Win_ || h != Hin_ || stride < w || (mask && mask_stride < w)) {
    last_error = "feed: image/mask size does not match the handle";   // TrackKLT.cpp:37-43 exits here
    return FE_BAD_ARG;
  }
  if (!queue_.empty()) {
    last_error = "feed: frames submitted with plviwo_fe_submit are still pending";
    return FE_BAD_ARG;
  }
  int rc = submit(t, image, stride, on_device, mask, mask_stride, vp);
  if (rc) return rc;
  return collect(info);
}

// -------------------------------------------------------------------------------------------- TrackKLT
static inline bool mask_hit(const FrameSlot &s, int W, int y, int x) { return !s.mask.empty() && s.mask[(size_t)y * W + x] > 127; }

int FeContext::klt_feed(FrameSlot &cur) {
  FrameResult &res = cur.res;
  FeFrameInfo *info = &res.info;
  std::vector<FePointRow> &point_rows = res.point_rows;
  // A speculative LK launch (perform_matching) may be tracking last frame's points into THIS frame already
  const bool spec = spec_valid_ && spec_prev_slot_ == klt_last_slot_ && spec_next_slot_ == cur.index;
  if (spec_valid_ && !spec) {   // launched for another pair of frames (cannot happen in order): drain it, do not use it
    if (wait_flag(&h_flag_lk_[1], seq_sp_, s_pt_, &t_err)) return FE_CUDA_ERROR;
  }
  if (!spec) spec_n_ = 0;
  spec_valid_ = false;
  // candidate tracks of the previous frame into this one were issued when this frame was submitted (track_candidates)
  const bool spec_cand = cur.sc_prev >= 0 && cur.sc_prev == klt_last_slot_;
  auto resolve = [&](std::vector<int> &src, bool have_cand) {   // candidate codes -(2 + table slot) -> kCandBase + slot
    for (int &v : src)
      if (v <= -2) v = have_cand ? kCandBase + (-(v + 2)) : -1;
  };
  // TrackKLT.cpp:110-123 — nothing tracked last time: detect on the CURRENT image only
  if (pts_last_.empty() || klt_last_slot_ < 0) {
    if (spec_n_ > 0 && wait_flag(&h_flag_lk_[1], seq_sp_, s_pt_, &t_err)) return FE_CUDA_ERROR;
    std::vector<Pt> good;
    std::vector<uint64_t> good_ids;
    std::vector<int> src;
    int rc = perform_detection(cur, good, good_ids, src, res);
    if (rc) return rc;
    pts_last_ = good;
    ids_last_ = good_ids;
    info->first_frame = 1;
    // the new points are candidates of THIS frame: track them into the next one right away
    resolve(src, true);   // candidates of THIS frame; whether they were tracked into the next one is checked there
    last_src_ = src;
    return FE_OK;
  }
  FrameSlot &last = slots_[klt_last_slot_];
  // top-off on the PREVIOUS image with the previous points (:127-130)
  std::vector<Pt> pts_old = pts_last_;
  std::vector<uint64_t> ids_old = ids_last_;
  std::vector<int> src_old = last_src_;
  src_old.resize(pts_old.size(), -1);
  if (!spec) std::fill(src_old.begin(), src_old.end(), -1);
  int rc = perform_detection(last, pts_old, ids_old, src_old, res);
  if (rc) return rc;
  resolve(src_old, spec_cand);
  std::vector<Pt> pts_new = pts_old;
  std::vector<uint8_t> mask_ll;
  bool mask_empty = true;
  if (!spec_cand)
    for (int &v : src_old)
      if (v >= kCandBase) v = -1;
  rc = perform_matching(last, cur, pts_old, src_old, spec || spec_cand, pts_new, mask_ll, mask_empty, res);
  if (rc) return rc;
  if (mask_empty) {  // :143-152
    pts_last_.clear();
    ids_last_.clear();
    last_src_.clear();
    info->reset = 1;
    return FE_OK;
  }
  std::vector<Pt> good;
  std::vector<uint64_t> good_ids;
  std::vector<int> good_src;
  good.reserve(pts_new.size());
  good_ids.reserve(pts_new.size());
  good_src.reserve(pts_new.size());
  for (size_t i = 0; i < pts_new.size(); i++) {  // :159-173
    const Pt &p = pts_new[i];
    if (p.x < 0 || p.y < 0 || (int)p.x >= W_ || (int)p.y >= H_) continue;
    if (mask_hit(cur, W_, (int)p.y, (int)p.x)) continue;
    if (mask_ll[i]) {
      good.push_back(p);
      good_ids.push_back(ids_old[i]);
      good_src.push_back(i < spec_of_lk_.size() ? spec_of_lk_[i] : -1);
      // :176-179 — undistort_cv(pt) of the tracked point is exactly the p1n the LK epilogue produced
      FePointRow r;
      r.id = ids_old[i];
      r.u = p.x;
      r.v = p.y;
      r.un = a_p1n_[i].x;
      r.vn = a_p1n_[i].y;
      point_rows.push_back(r);
    }
  }
  pts_last_ = good;
  ids_last_ = good_ids;
  last_src_ = good_src;
  return FE_OK;
}

// Speculative tracking.  LK treats every point on its own, so the tracks of frame t+1 do not depend on WHICH points
// survive frame t's RANSAC gate, bounds / mask filter and top-off detection — only their positions matter, and every
// point that can possibly be tracked into t+1 is known the moment frame t's LK finishes: the points whose KLT status is
// good, and the refined corner candidates of frame t (the top-off detection can only add those).  So LK(t -> t+1) is
// launched for that superset BEFORE frame t's RANSAC runs, and the host work of frame t (RANSAC, rows, next frame's
// detection glue) overlaps the GPU's tracking instead of waiting for it.  Frame t+1 then picks its points' results out
// of the speculative arrays by index; a point without a speculative result (no next frame was queued yet, or the layout
// changed) goes through an ordinary launch.  Results are bit-identical either way.
int FeContext::speculate(FrameSlot &prev, const float2 *lk_pts, const uint8_t *lk_status, int n) {
  HostTimer hs(&kst_.host_ms[FE_HOST_SPECULATE]);
  spec_of_lk_.assign((size_t)n, -1);
  if (!use_spec_ || cfg_.line_samples > 0) return FE_OK;
  int nxt = -1;
  if (!klt_q_.peek(&nxt)) return FE_OK;          // the next frame has not been submitted yet
  FrameSlot &fn = slots_[nxt];
  LkParams prm;
  prm.win = cfg_.win_size;
  prm.max_level = cfg_.pyr_levels;
  prm.max_count = 30;
  prm.eps_sq = 0.01f * 0.01f;
  prm.min_eig = 1e-4f;
  prm.undistort = 1;
  for (int i = 0; i < 4; i++) { prm.K[i] = fn.K[i]; prm.D[i] = fn.D[i]; }
  // ---- (A) the points tracked into `prev` whose KLT status is good: latency-critical stream
  int k = 0;
  for (int i = 0; i < n && k < max_pts_; i++)
    if (lk_status[i]) {
      h_sp_pts0_[k] = lk_pts[i];
      spec_of_lk_[(size_t)i] = k++;
    }
  spec_n_ = k;
  spec_timed_ = false;
  if (k > 0) {
    HostTimer h11(&kst_.host_ms[FE_HOST_SPEC_LAUNCH]);
    FE_CUDA(cudaStreamWaitEvent(s_pt_, fn.ev_pyr, 0));
    spec_timed_ = fn.timed;
    if (spec_timed_) cudaEventRecord(ev_pt_[2], s_pt_);
    const bool flow0 = lk_table_mode_ok(prm, prev.pyr.n);   // pts1 = pts0 is implicit for the 15 x 15 kernel
    if (!flow0) std::memcpy(h_sp_pts1_, h_sp_pts0_, (size_t)k * sizeof(float2));
    const bool self_signal = launch_lk(prev.pyr, fn.pyr, h_sp_pts0_, h_sp_pts1_, h_sp_status_, h_sp_p0n_, h_sp_p1n_, k, prm, s_pt_,
                                       &h_flag_lk_[1], ++seq_sp_, d_lk_done_ + 1, nullptr, 0, flow0);
    if (spec_timed_) cudaEventRecord(ev_pt_[3], s_pt_);
    if (!self_signal) launch_signal(&h_flag_lk_[1], seq_sp_, s_pt_);
    FE_CUDA(cudaGetLastError());
    kst_.kernel_launches_total++;
    kst_.h2d_bytes += (size_t)k * sizeof(float2);
    kst_.d2h_bytes += (size_t)k * (3 * sizeof(float2) + 1);
  }
  spec_valid_ = k > 0;
  spec_prev_slot_ = prev.index;
  spec_next_slot_ = nxt;
  return FE_OK;
}

// First loop of the top-off detection (TrackKLT.cpp:411-464; stereo: :545-598 left, :692-748 right): drop points near the
// border, outside the grids, on an occupied min-distance cell (unless stereo_ids holds their id, :720-726) or on the mask.
void FeContext::filter_existing(const std::vector<uint8_t> &mask_test, std::vector<Pt> &pts0, std::vector<uint64_t> &ids0,
                                std::vector<int> *src, const std::vector<uint64_t> *stereo_ids, OccGrids &g) const {
  const int d = cfg_.min_px_dist;
  const int cols = W_, rows = H_;
  const int close_w = (int)((float)cols / (float)d), close_h = (int)((float)rows / (float)d);
  g.close_w = close_w;
  g.close_h = close_h;
  g.close.assign((size_t)close_w * close_h, 0);
  const float size_x = (float)cols / (float)cfg_.grid_x, size_y = (float)rows / (float)cfg_.grid_y;
  const int gx = cfg_.grid_x, gy = cfg_.grid_y;
  g.grid.assign((size_t)gx * gy, 0);
  g.rects.clear();
  size_t keep = 0;
  for (size_t k = 0; k < pts0.size(); k++) {
    const Pt kp = pts0[k];
    int x = (int)kp.x, y = (int)kp.y;
    const int edge = 10;
    if (x < edge || x >= cols - edge || y < edge || y >= rows - edge) continue;
    int x_close = (int)(kp.x / (float)d), y_close = (int)(kp.y / (float)d);
    if (x_close < 0 || x_close >= close_w || y_close < 0 || y_close >= close_h) continue;
    int x_grid = (int)std::floor(kp.x / size_x), y_grid = (int)std::floor(kp.y / size_y);
    if (x_grid < 0 || x_grid >= gx || y_grid < 0 || y_grid >= gy) continue;
    if (g.close[(size_t)y_close * close_w + x_close] > 127) {
      if (!stereo_ids || std::find(stereo_ids->begin(), stereo_ids->end(), ids0[k]) == stereo_ids->end()) continue;
    }
    if (!mask_test.empty() && mask_test[(size_t)y * cols + x] > 127) continue;
    g.close[(size_t)y_close * close_w + x_close] = 255;
    uint8_t &c = g.grid[(size_t)y_grid * gx + x_grid];
    if (c < 255) c += 1;
    if (x - d >= 0 && x + d < cols && y - d >= 0 && y + d < rows) g.rects.emplace_back(x, y);
    pts0[keep] = kp;
    ids0[keep] = ids0[k];
    if (src) (*src)[keep] = (*src)[k];
    keep++;
  }
  pts0.resize(keep);
  ids0.resize(keep);
  if (src) src->resize(keep);
}

// Valid cells (:479-492) + Grider_GRID::perform_griding (Grider_GRID.h:74-180) on the frame's candidate table.  FAST, the
// unstable sort, the top-num_features_grid cut and cornerSubPix do not depend on tracker state and were computed for
// EVERY cell when the frame was submitted; only the state-dependent part is left: which cells are valid and the mask
// test (:140-147).  mask_resize is the mask the reference resizes to the grid, mask_clone the one it clones into
// mask_updated (the same for the monocular path; the stereo path clones the LEFT mask for the right image, :691).
int FeContext::grid_candidates(FrameSlot &slot, const std::vector<uint8_t> &mask_resize, const std::vector<uint8_t> &mask_clone,
                               const OccGrids &g, std::vector<Pt> &ext, std::vector<int> &ext_cand, FrameResult &res) {
  std::vector<int32_t> &tap_fast_ = res.tap_fast;
  std::vector<float> &tap_subpix_ = res.tap_subpix;
  const bool taps = this->taps.load(std::memory_order_relaxed);
  const int d = cfg_.min_px_dist;
  const int cols = W_, rows = H_;
  const int gx = cfg_.grid_x, gy = cfg_.grid_y;
  const int bw = (cols + 63) / 64;
  const double min_feat_percent = 0.50;
  // mask0_grid = resize(mask0, grid, INTER_NEAREST) (:479-480)
  std::vector<uint8_t> mask_grid((size_t)gx * gy, 0);
  if (!mask_resize.empty()) {
    const double ifx = 1.0 / ((double)gx / (double)cols), ify = 1.0 / ((double)gy / (double)rows);
    for (int y = 0; y < gy; y++) {
      int sy = std::min((int)std::floor(y * ify), rows - 1);
      for (int x = 0; x < gx; x++) {
        int sx = std::min((int)std::floor(x * ifx), cols - 1);
        mask_grid[(size_t)y * gx + x] = mask_resize[(size_t)sy * cols + sx];
      }
    }
  }
  int num_features_grid = (int)((double)cfg_.num_features / (double)(gx * gy)) + 1;
  int num_features_grid_req = std::max(1, (int)(min_feat_percent * num_features_grid));
  std::vector<std::pair<int, int>> valid_locs;
  for (int x = 0; x < gx; x++)        // x-major order (:486-492)
    for (int y = 0; y < gy; y++)
      if ((int)g.grid[(size_t)y * gx + x] < num_features_grid_req && (int)mask_grid[(size_t)y * gx + x] != 255)
        valid_locs.emplace_back(x, y);

  ext.clear();        // pts0_ext after sub-pixel refinement
  ext_cand.clear();   // ... and which candidate of the frame's table each one is
  if (taps) {
    tap_fast_.clear();
    tap_subpix_.clear();
  }
  if (valid_locs.empty()) return FE_OK;
  if (slot.predet_num_features != cfg_.num_features) {   // set_num_features() after the frame was submitted
    int rc = wait_predetection(slot);
    if (rc) return rc;
    rc = enqueue_fast_all_cells(slot);
    if (rc) return rc;
    rc = record_fast_path(slot, slot.s_b);
    if (rc) return rc;
    slot.seq_fast++;
    FE_CUDA(cudaEventRecord(slot.ev_fast, slot.s_b));
  }
  {
    HostTimer hw(&kst_.host_ms[FE_HOST_CAND_WAIT]);
    int rc = wait_predetection(slot);
    if (rc) return rc;
  }
  bool any_cell = false;
  for (auto &loc : valid_locs) any_cell = any_cell || slot.cell_of_loc[(size_t)loc.first * gy + loc.second] >= 0;
  if (!any_cell) return FE_OK;
  // mask0_updated as a bit mask: caller mask > 127 or inside a (2d+1)^2 square of a kept point (:457-461)
  std::fill(occ_bits_.begin(), occ_bits_.end(), 0);
  if (!mask_clone.empty())
    for (int y = 0; y < rows; y++)
      for (int x = 0; x < cols; x++)
        if (mask_clone[(size_t)y * cols + x] > 127) occ_bits_[(size_t)y * bw + (x >> 6)] |= 1ull << (x & 63);
  for (auto &rc : g.rects) {
    int x0 = rc.first - d, x1 = rc.first + d;
    for (int y = rc.second - d; y <= rc.second + d; y++) {
      uint64_t *row = &occ_bits_[(size_t)y * bw];
      int w0 = x0 >> 6, w1 = x1 >> 6;
      uint64_t m0 = ~0ull << (x0 & 63), m1 = (x1 & 63) == 63 ? ~0ull : ((1ull << ((x1 & 63) + 1)) - 1);
      if (w0 == w1) {
        row[w0] |= m0 & m1;
      } else {
        row[w0] |= m0;
        for (int w = w0 + 1; w < w1; w++) row[w] = ~0ull;
        row[w1] |= m1;
      }
    }
  }
  for (auto &loc : valid_locs) {     // cells in valid_locs order (:108-156)
    const int c = slot.cell_of_loc[(size_t)loc.first * gy + loc.second];
    if (c < 0) continue;
    if (taps)
      for (int k = slot.cell_kps_first[c]; k < slot.cell_kps_first[c + 1]; k++)
        tap_fast_.insert(tap_fast_.end(), {loc.first, loc.second, slot.cell_kps_tap[3 * k], slot.cell_kps_tap[3 * k + 1],
                                           slot.cell_kps_tap[3 * k + 2]});
    const int nfg_t = slot.predet_nfg, cnt = std::min(slot.h_cand_cnt[c], nfg_t);
    for (int k = 0; k < cnt; k++) {   // :133-149
      const int i = c * nfg_t + k;    // slot of the candidate in the frame's fixed-stride table
      const Pt p = Pt{slot.h_cand_in[i].x, slot.h_cand_in[i].y};
      if ((int)p.x < 0 || (int)p.x > cols || (int)p.y < 0 || (int)p.y > rows) continue;
      const int ix = (int)p.x, iy = (int)p.y;
      if (iy >= rows || ix >= cols) continue;  // the reference would read out of bounds here; cannot happen
      if ((occ_bits_[(size_t)iy * bw + (ix >> 6)] >> (ix & 63)) & 1ull) continue;
      const Pt pr = Pt{slot.h_cand_out[i].x, slot.h_cand_out[i].y};
      ext.push_back(pr);                    // cornerSubPix result of exactly this point (:163-179)
      ext_cand.push_back(i);
      if (taps) tap_subpix_.insert(tap_subpix_.end(), {p.x, p.y, pr.x, pr.y});
    }
  }
  return FE_OK;
}

int FeContext::perform_detection(const FrameSlot &img, std::vector<Pt> &pts0, std::vector<uint64_t> &ids0, std::vector<int> &src,
                                 FrameResult &res) {
  src.resize(pts0.size(), -1);   // per point: index into the speculative LK arrays, -1 none, -(2 + i) = candidate i
  HostTimer ht(&kst_.host_ms[FE_HOST_DETECTION]);
  FeFrameInfo *info = &res.info;
  const int d = cfg_.min_px_dist;
  OccGrids g;
  filter_existing(img.mask, pts0, ids0, &src, nullptr, g);   // TrackKLT.cpp:411-464
  const double min_feat_percent = 0.50;
  int num_featsneeded = cfg_.num_features - (int)pts0.size();
  if (num_featsneeded < std::min(20, (int)(min_feat_percent * cfg_.num_features))) return FE_OK;  // :468-471
  info->detection_ran = 1;
  std::vector<Pt> ext;
  std::vector<int> ext_cand;
  int rc = grid_candidates(const_cast<FrameSlot &>(img), img.mask, img.mask, g, ext, ext_cand, res);
  if (rc) return rc;
  // reject new points that are close to an existing one (:497-512), then hand out ids (:519-527)
  int added = 0;
  for (size_t e = 0; e < ext.size(); e++) {
    const Pt &kp = ext[e];
    int x_grid = (int)(kp.x / (float)d), y_grid = (int)(kp.y / (float)d);
    if (x_grid < 0 || x_grid >= g.close_w || y_grid < 0 || y_grid >= g.close_h) continue;
    if (g.close[(size_t)y_grid * g.close_w + x_grid] > 127) continue;
    g.close[(size_t)y_grid * g.close_w + x_grid] = 255;
    pts0.push_back(kp);
    ids0.push_back(++currid_);
    src.push_back(-(2 + ext_cand[e]));   // slot of the candidate in the frame's fixed-stride table
    added++;
  }
  info->n_detected += added;
  return FE_OK;
}

int FeContext::perform_matching(const FrameSlot &f0, FrameSlot &f1, std::vector<Pt> &pts0, const std::vector<int> &src, bool spec,
                                std::vector<Pt> &pts1, std::vector<uint8_t> &mask_out, bool &mask_empty, FrameResult &res) {
  HostTimer ht(&kst_.host_ms[FE_HOST_MATCHING]);
  FeFrameInfo *info = &res.info;
  std::vector<float> &tap_lk_ = res.tap_lk, &sample_uv = res.sample_uv;
  std::vector<uint8_t> &sample_status = res.sample_status;
  const bool taps = this->taps.load(std::memory_order_relaxed);
  const bool timing = f1.timed;
  mask_out.clear();
  mask_empty = true;
  spec_of_lk_.clear();
  const int n = (int)pts0.size();
  if (n == 0 || n < 10) {
    // the speculative launch (if any) is not used: let it finish before its buffers are reused
    if (spec_n_ > 0 && wait_flag(&h_flag_lk_[1], seq_sp_, s_pt_, &t_err)) return FE_CUDA_ERROR;
    if (n == 0) return FE_OK;                // :836-837 (mask stays empty => caller resets)
    mask_empty = false;
    mask_out.assign(n, 0);                   // :848-852
    return FE_OK;
  }
  mask_empty = false;
  if (n > max_pts_) return err(FE_INTERNAL, "perform_matching: more points than the tracking buffers hold");
  a_pts1_.resize(n);
  a_status_.resize(n);
  a_p0n_.resize(n);
  a_p1n_.resize(n);
  // points without a speculative result go through an ordinary launch (compact arrays; lk2_[k] = point index)
  lk2_.clear();
  bool need_a = false, need_b = false;
  for (int i = 0; i < n; i++) {
    const int v = spec ? src[i] : -1;
    if (v >= kCandBase && v - kCandBase < f1.sc_ntab) need_b = true;
    else if (v >= 0 && v < spec_n_) need_a = true;
    else lk2_.push_back(i);
  }
  const int n2 = (int)lk2_.size();
  // extension: samples along last frame's segments ride in the same launch (not part of the RANSAC gate)
  int ns = 0;
  if (cfg_.line_samples > 0) {
    // the segments belong to the line tracker's thread: wait until it is done with the previous frame
    for (unsigned spins = 0; f0.stage.load(std::memory_order_acquire) == 2; spins++) {
      if (spins < kSpin) cpu_pause();
      else std::this_thread::yield();
    }
    const int S = cfg_.line_samples;
    for (const float4 &l : lines_det_last_) {   // every segment the detector kept in the previous frame (> line_min_length)
      for (int k = 0; k < S && n2 + ns < max_pts_; k++) {
        float a = S > 1 ? (float)k / (float)(S - 1) : 0.5f;
        h_pts0_[n2 + ns] = make_float2(l.x + (l.z - l.x) * a, l.y + (l.w - l.y) * a);
        ns++;
      }
    }
  }
  const int nt = n2 + ns;
  for (int k = 0; k < n2; k++) {
    h_pts0_[k] = make_float2(pts0[lk2_[k]].x, pts0[lk2_[k]].y);
    h_pts1_[k] = h_pts0_[k];   // OPTFLOW_USE_INITIAL_FLOW with pts1 = pts0 (:134-138)
  }
  for (int k = 0; k < ns; k++) h_pts1_[n2 + k] = h_pts0_[n2 + k];
  LkParams prm;
  prm.win = cfg_.win_size;
  prm.max_level = cfg_.pyr_levels;
  prm.max_count = 30;
  prm.eps_sq = 0.01f * 0.01f;
  prm.min_eig = 1e-4f;
  prm.undistort = 1;
  for (int i = 0; i < 4; i++) { prm.K[i] = f1.K[i]; prm.D[i] = f1.D[i]; }
  // The feature arrays are a few KB: the kernel reads and writes them in pinned, device-mapped host memory directly
  // (no copy-engine operation queued behind the next frame's 700 KB upload, one synchronisation per frame).
  if (nt > 0) {
    kst_.h2d_bytes += (size_t)nt * 2 * sizeof(float2);
    kst_.d2h_bytes += (size_t)nt * (3 * sizeof(float2) + 1);
    if (timing) cudaEventRecord(ev_pt_[4], s_pt_);
    HostTimer tl(&kst_.host_ms[FE_HOST_LK_LAUNCH]);
    // the LK kernel publishes the completion sequence number itself (its last feature writes the pinned flag)
    const bool self_signal = launch_lk(f0.pyr, f1.pyr, h_pts0_, h_pts1_, h_status_, h_p0n_, h_p1n_, nt, prm, s_pt_, h_flag_lk_,
                                       ++seq_lk_, d_lk_done_);
    kst_.kernel_launches_total++;
    if (timing) cudaEventRecord(ev_pt_[5], s_pt_);
    if (!self_signal) launch_signal(h_flag_lk_, seq_lk_, s_pt_);
    FE_CUDA(cudaGetLastError());
  }
  {
    HostTimer tw(&kst_.host_ms[FE_HOST_LK_WAIT]);
    if (spec_n_ > 0 && wait_flag(&h_flag_lk_[1], seq_sp_, s_pt_, &t_err)) return FE_CUDA_ERROR;
    if (need_b && wait_flag(&f1.h_flags[3], f1.seq_sc, f1.s_b, &t_err)) return FE_CUDA_ERROR;
    if (nt > 0 && wait_flag(h_flag_lk_, seq_lk_, s_pt_, &t_err)) return FE_CUDA_ERROR;
  }
  (void)need_a;
  if (timing && nt > 0) {
    FE_CUDA(cudaEventSynchronize(ev_pt_[5]));
    acc_time(kst_, FE_STAGE_LK, ev_pt_[4], ev_pt_[5]);
  }
  if (spec && spec_timed_) {
    FE_CUDA(cudaEventSynchronize(ev_pt_[3]));
    acc_time(kst_, FE_STAGE_LK, ev_pt_[2], ev_pt_[3]);
  }
  // assemble the per-point results in the reference's order
  HostTimer *ha = new HostTimer(&kst_.host_ms[FE_HOST_ASSEMBLE]);
  if (spec)
    for (int i = 0; i < n; i++) {
      const int k = src[i];
      if (k >= kCandBase && k - kCandBase < f1.sc_ntab) {
        const int j = k - kCandBase;
        a_pts1_[i] = f1.h_sc_pts1[j];
        a_status_[i] = f1.h_sc_status[j];
        a_p0n_[i] = f1.h_sc_p0n[j];
        a_p1n_[i] = f1.h_sc_p1n[j];
      } else if (k >= 0 && k < spec_n_) {
        a_pts1_[i] = h_sp_pts1_[k];
        a_status_[i] = h_sp_status_[k];
        a_p0n_[i] = h_sp_p0n_[k];
        a_p1n_[i] = h_sp_p1n_[k];
      }
    }
  for (int k = 0; k < n2; k++) {
    const int i = lk2_[k];
    a_pts1_[i] = h_pts1_[k];
    a_status_[i] = h_status_[k];
    a_p0n_[i] = h_p0n_[k];
    a_p1n_[i] = h_p1n_[k];
  }
  for (int k = 0; k < ns; k++) {
    sample_uv.insert(sample_uv.end(), {h_pts0_[n2 + k].x, h_pts0_[n2 + k].y, h_pts1_[n2 + k].x, h_pts1_[n2 + k].y});
    sample_status.push_back(h_status_[n2 + k]);
  }
  delete ha;
  // this frame's tracks are known: start tracking into the NEXT frame before the host-side gate below
  {
    int rc = speculate(f1, a_pts1_.data(), a_status_.data(), n);
    if (rc) return rc;
  }

  // RANSAC gate on the normalised coordinates (:869-873)
  const double max_focal = std::max(f1.K[0], f1.K[1]);
  std::vector<uint8_t> mask_rsc(n, 0);
  int mask_valid = 0;
  int n_in;
  {
    HostTimer hr(&kst_.host_ms[FE_HOST_RANSAC]);
    n_in = ransac_fundamental(reinterpret_cast<const float *>(a_p0n_.data()), reinterpret_cast<const float *>(a_p1n_.data()), n,
                              2.0 / max_focal, 0.999, mask_rsc.data(), &mask_valid);
  }
  mask_out.resize(n);
  int n_klt = 0;
  if (taps) tap_lk_.clear();
  for (int i = 0; i < n; i++) {  // :876-885
    mask_out[i] = (a_status_[i] && mask_valid && mask_rsc[i]) ? 1 : 0;
    n_klt += a_status_[i] ? 1 : 0;
    pts1[i] = Pt{a_pts1_[i].x, a_pts1_[i].y};
    if (taps) tap_lk_.insert(tap_lk_.end(), {pts0[i].x, pts0[i].y, pts1[i].x, pts1[i].y, (float)a_status_[i], (float)(mask_valid && mask_rsc[i])});
  }
  info->n_lk_in = n;
  info->n_klt_ok = n_klt;
  info->n_ransac_ok = n_in;
  return FE_OK;
}

// -------------------------------------------------------------------------------------------- TrackLSD
namespace {
// TrackLSD::PointLineDistance (TrackLSD.cpp:794-814): float arithmetic, std::pow(float,int) promotes to double
float point_line_distance(const float4 &line, float x0, float y0) {
  float x1 = line.x, y1 = line.y, x2 = line.z, y2 = line.w;
  float cross = (x2 - x1) * (x0 - x1) + (y2 - y1) * (y0 - y1);
  if (cross <= 0) return std::sqrt((x0 - x1) * (x0 - x1) + (y0 - y1) * (y0 - y1));
  float d = (x2 - x1) * (x2 - x1) + (y2 - y1) * (y2 - y1);
  if (cross > d) return std::sqrt((x0 - x2) * (x0 - x2) + (y0 - y2) * (y0 - y2));
  return (float)std::abs(std::fabs((y2 - y1) * x0 + (x1 - x2) * y0 + ((x2 * y1) - (x1 * y2))) /
                         (std::sqrt(std::pow((double)(y2 - y1), 2) + std::pow((double)(x1 - x2), 2))));
}
// TrackLSD::LineSimilar (:816-830)
bool line_similar(const float4 &line2, const float4 &line1) {
  float mx = (line1.x + line1.z) / 2, my = (line1.y + line1.w) / 2;
  return point_line_distance(line2, mx, my) <= 6;
}
// TrackLSD::LineClass (:335-366), including atan(dy) / dx at :350-351
bool line_class(const float4 &line, double vx, double vy) {
  double s[3] = {line.x, line.y, 1}, e[3] = {line.z, line.w, 1};
  double mid[3] = {(s[0] + e[0]) / 2, (s[1] + e[1]) / 2, (s[2] + e[2]) / 2};
  double v3[3] = {vx, vy, 1};
  double ln[3] = {mid[1] * v3[2] - mid[2] * v3[1], mid[2] * v3[0] - mid[0] * v3[2], mid[0] * v3[1] - mid[1] * v3[0]};
  double dis_error = (std::abs(ln[0] * s[0] + ln[1] * s[1] + ln[2] * s[2]) + std::abs(ln[0] * e[0] + ln[1] * e[1] + ln[2] * e[2])) /
                     (2 * std::sqrt(ln[0] * ln[0] + ln[1] * ln[1]));
  dis_error = std::abs(dis_error);
  double angle1 = std::atan(line.y - line.w) / (line.x - line.z);   // float arithmetic, as written in the reference
  double angle2 = std::atan(mid[1] - vy) / (mid[0] - vx);
  double angle_error = std::abs(angle1 - angle2);
  return dis_error <= 5.0 && angle_error <= 0.35;
}
int line_classification(const float4 &line, const double vp[6]) {  // :318-333
  if (line_class(line, vp[4], vp[5])) return 3;
  if (line_class(line, vp[2], vp[3])) return 2;
  if (line_class(line, vp[0], vp[1])) return 1;
  return 0;
}
}  // namespace

// TrackLSD::AssignPointToLines (:744-792): per line the points inside its (mis-indexed, :754-757) bounding box and within
// 5 px of the SEGMENT; lines without a point are dropped.  The candidate test of one line against all points is
// vectorised (line_candidates, host_simd.cpp); survivors go through the exact PointLineDistance.
void assign_points_to_lines_host(const std::vector<float4> &lines_new, const std::vector<uint64_t> &ids_new,
                                 const std::vector<Pt> &points, const std::vector<uint64_t> &pids,
                                 std::vector<std::map<int, double>> &pol_new, std::vector<std::vector<Pt>> &positions,
                                 std::vector<float4> &filt_lines, std::vector<uint64_t> &filt_ids, std::vector<float> &spx,
                                 std::vector<float> &spy, std::vector<uint8_t> &pass) {
  const int npt = (int)points.size();
  spx.assign((size_t)npt + 16, 0.f);   // padded to whole groups of 16 points (line_candidates reads them)
  spy.assign((size_t)npt + 16, 0.f);
  pass.assign((size_t)npt / 8 + 4, 0);   // one bit per point
  pol_new.clear();
  positions.clear();
  filt_lines.clear();
  filt_ids.clear();
  pol_new.reserve(64);
  positions.reserve(64);
  filt_lines.reserve(64);
  filt_ids.reserve(64);
  for (int j = 0; j < npt; j++) {
    spx[j] = points[j].x;
    spy[j] = points[j].y;
  }
  for (size_t i = 0; i < lines_new.size(); i++) {
    const float4 &l = lines_new[i];
    float lx1 = l.x, lx2 = l.y, ly1 = l.z, ly2 = l.w;  // index mix-up reproduced (:754-757)
    float min_lx = lx1, max_lx = lx2, min_ly = ly1, max_ly = ly2;
    if (lx1 > lx2) std::swap(min_lx, max_lx);
    if (ly1 > ly2) std::swap(min_ly, max_ly);
    const float pa = l.w - l.y, pb = l.x - l.z, pc = l.z * l.y - l.x * l.w;
    const float plen2 = 36.f * (pa * pa + pb * pb);
    if (!line_candidates(spx.data(), spy.data(), npt, min_lx, max_lx, min_ly, max_ly, pa, pb, pc, plen2, pass.data())) continue;
    bool find_point = false;   // the line's containers are only created once a point is really within 5 px
    for (int j = 0; j < npt; j++) {
      const unsigned grp = pass[j >> 3];
      if (grp == 0) { j |= 7; continue; }
      if (!((grp >> (j & 7)) & 1u)) continue;
      float dist = point_line_distance(l, spx[j], spy[j]);
      if (dist > 5) continue;
      if (!find_point) {
        pol_new.emplace_back();
        positions.emplace_back();
        filt_lines.push_back(l);
        filt_ids.push_back(ids_new[i]);
        find_point = true;
      }
      pol_new.back()[(int)pids[j]] = dist;
      positions.back().push_back(points[j]);
    }
  }
}

// TrackLSD::LineMatch (:368-407): i over new lines, j over last lines, the LAST satisfying j wins.  The reference walks
// every (i, j) pair and every point id of line j; a pair can only match if the two lines share a point id — j matches i
// iff they share >= 2 ids, or >= 1 id and LineSimilar holds (the inner loop stops at the first shared id when the lines
// are similar, at the second otherwise) — so the candidates come from an inverted index id -> last lines holding it.
void line_match_host(const std::vector<std::map<int, double>> &pol_last, const std::vector<std::map<int, double>> &pol_new,
                     const std::vector<float4> &lines_new, const std::vector<float4> &lines_last, std::map<int, int> &matches,
                     std::vector<std::pair<int, int>> &inv, std::vector<int> &shared, std::vector<int> &touched) {
  matches.clear();
  const size_t n0 = pol_last.size(), n1 = pol_new.size();
  if (n0 == 0 || n1 == 0) return;
  inv.clear();   // (point id, last line), sorted
  for (size_t j = 0; j < n0; j++)
    for (auto &pt : pol_last[j]) inv.emplace_back(pt.first, (int)j);
  std::sort(inv.begin(), inv.end());
  shared.assign(n0, 0);
  for (size_t i = 0; i < n1; i++) {
    touched.clear();
    for (auto &pt : pol_new[i]) {
      auto lo = std::lower_bound(inv.begin(), inv.end(), std::make_pair(pt.first, -1));
      for (; lo != inv.end() && lo->first == pt.first; ++lo)
        if (shared[lo->second]++ == 0) touched.push_back(lo->second);
    }
    int best = -1;
    for (int j : touched) {
      if (j > best && (shared[j] >= 2 || line_similar(lines_new[i], lines_last[j]))) best = j;
      shared[j] = 0;
    }
    if (best >= 0) matches[(int)i] = best;
  }
}

int FeContext::lsd_feed(FrameSlot &cur) {
  HostTimer ht(&lst_.host_ms[FE_HOST_LINES]);
  FrameResult &res = cur.res;
  FeFrameInfo *info = &res.info;
  std::vector<FeLineRow> &line_rows = res.line_rows;
  std::vector<FeLinePoint> &line_points = res.line_points;
  std::vector<float> &tap_fld_ = res.tap_fld;
  const bool taps = this->taps.load(std::memory_order_relaxed);
  {
    HostTimer hw(&lst_.host_ms[FE_HOST_LINE_WAIT]);
    int rc = wait_flag(&cur.h_flags[2], cur.seq_lines, cur.s_line, &t_err);
    if (rc) return rc;
  }
  int nseg = std::min(cur.h_fld_counts[1], cur.fld.out_cap);
  if (nseg > 1024) {
    // rare: more segments than the asynchronous copy carries.  The data is complete (the flag above), and the line stream
    // is shared with other slots (the caller's thread may be capturing a graph on it), so this is a plain blocking copy
    lst_.d2h_bytes += (size_t)(nseg - 1024) * sizeof(float4);
    FE_CUDA(cudaMemcpy(cur.h_segs + 1024, cur.fld.out + 1024, (size_t)(nseg - 1024) * sizeof(float4), cudaMemcpyDeviceToHost));
  }
  if (taps) tap_fld_.assign(reinterpret_cast<float *>(cur.h_segs), reinterpret_cast<float *>(cur.h_segs) + 4 * (size_t)nseg);
  // perform_detection_monocular (:194-236): x2, FilterShortLines(40), a fresh id for EVERY detected line
  std::vector<float4> lines_new;
  std::vector<uint64_t> ids_new;
  const float thr_sq = cfg_.line_min_length * cfg_.line_min_length;
  for (int i = 0; i < nseg; i++) {
    float4 l = cur.h_segs[i];
    l.x *= 2; l.y *= 2; l.z *= 2; l.w *= 2;
    float lsq = (l.z - l.x) * (l.z - l.x) + (l.w - l.y) * (l.w - l.y);
    if (lsq > thr_sq) lines_new.push_back(l);
  }
  for (size_t i = 0; i < lines_new.size(); i++) ids_new.push_back(++line_currid_);
  info->n_lines_detected = (int)lines_new.size();
  if (cfg_.line_samples > 0) lines_det_last_ = lines_new;   // the next frame's LK samples points along these

  // AssignPointToLines (:744-792) against the CURRENT points of the point tracker (:127-129)
  const std::vector<Pt> &points = res.obs;        // the point tracker's pts_last / ids_last after THIS frame
  const std::vector<uint64_t> &pids = res.obs_ids;
  std::vector<std::map<int, double>> pol_new;
  std::vector<std::vector<Pt>> positions;
  std::vector<float4> filt_lines;
  std::vector<uint64_t> filt_ids;
  HostTimer *t_assign = new HostTimer(&lst_.host_ms[FE_HOST_LINE_ASSIGN]);
  assign_points_to_lines_host(lines_new, ids_new, points, pids, pol_new, positions, filt_lines, filt_ids, sc_px_, sc_py_, sc_pass_);
  delete t_assign;
  if (lines_last_.empty()) {  // first frame / lost (:95-115): no database rows
    lines_last_ = filt_lines;
    line_ids_last_ = filt_ids;
    pol_last_ = pol_new;
    return FE_OK;
  }
  // LineMatch (:368-407)
  std::map<int, int> matches;
  {
    HostTimer tm(&lst_.host_ms[FE_HOST_LINE_MATCH]);
    line_match_host(pol_last_, pol_new, filt_lines, lines_last_, matches, sc_inv_, sc_shared_, sc_touched_);
  }
  HostTimer t_rows(&lst_.host_ms[FE_HOST_LINE_ROWS]);
  info->n_line_matches = (int)matches.size();
  std::vector<uint64_t> good_ids(filt_lines.size());
  for (size_t i = 0; i < filt_lines.size(); i++) {  // :146-158
    auto it = matches.find((int)i);
    int id = it != matches.end() ? (int)line_ids_last_[it->second] : (int)filt_ids[i];
    good_ids[i] = (uint64_t)(size_t)id;
  }
  for (size_t i = 0; i < filt_lines.size(); i++) {  // :163-167
    FeLineRow r;
    std::memset(&r, 0, sizeof(r));
    r.id = good_ids[i];
    const float4 &l = filt_lines[i];
    r.line[0] = l.x; r.line[1] = l.y; r.line[2] = l.z; r.line[3] = l.w;
    undistort_host(cur.K, cur.D, l.x, l.y, r.line_n[0], r.line_n[1]);
    undistort_host(cur.K, cur.D, l.z, l.w, r.line_n[2], r.line_n[3]);
    r.D = line_classification(l, cur.vp);
    r.n_pts = (int)pol_new[i].size();
    r.pt_offset = (int)line_points.size();
    r.matched = matches.count((int)i) ? 1 : 0;
    size_t k = 0;
    for (auto &pt : pol_new[i]) {
      FeLinePoint lp;
      lp.pid = pt.first;
      lp.dist = (float)pt.second;
      lp.u = positions[i][k].x;
      lp.v = positions[i][k].y;
      line_points.push_back(lp);
      k++;
    }
    line_rows.push_back(r);
  }
  lines_last_.swap(filt_lines);  // :175-182
  line_ids_last_.swap(good_ids);
  pol_last_.swap(pol_new);
  return FE_OK;
}

int FeContext::classify_lines(const double vp[6]) {
  FrameResult &r = const_cast<FrameResult &>(*cur_res_);
  for (FeLineRow &row : r.line_rows) row.D = line_classification(make_float4(row.line[0], row.line[1], row.line[2], row.line[3]), vp);
  return FE_OK;
}

// ------------------------------------------------------------------------------------------ state / taps
namespace {
struct StateHeader {
  uint32_t magic, version;
  int32_t w, h;
  uint64_t currid, line_currid;
  int32_t n_pts, n_lines, has_image, has_mask;
  int32_t n_pol_entries, reserved;
};
}  // namespace

// Both are only legal between frames (nothing in flight): the tracker threads are idle then and their state is visible
// to the caller's thread through the release/acquire pair on FrameSlot::stage.
int FeContext::get_state(void *buf, size_t cap, size_t *n_bytes) {
  if (!queue_.empty()) {
    last_error = "get_state: collect the pending frames first";
    return FE_BAD_ARG;
  }
  int rc = [&]() -> int {
  FE_CUDA(cudaSetDevice(device_));
  const int last_slot_ = klt_last_slot_;
  StateHeader hd;
  std::memset(&hd, 0, sizeof(hd));
  hd.magic = 0x504c5657u;
  hd.version = 1;
  hd.w = W_;
  hd.h = H_;
  hd.currid = currid_;
  hd.line_currid = line_currid_;
  hd.n_pts = (int)pts_last_.size();
  hd.n_lines = (int)lines_last_.size();
  hd.has_image = last_slot_ >= 0 ? 1 : 0;
  hd.has_mask = (last_slot_ >= 0 && !slots_[last_slot_].mask.empty()) ? 1 : 0;
  int npol = 0;
  for (auto &m : pol_last_) npol += (int)m.size();
  hd.n_pol_entries = npol;
  size_t need = sizeof(hd) + (size_t)hd.n_pts * (sizeof(Pt) + sizeof(uint64_t)) +
                (size_t)hd.n_lines * (sizeof(float4) + sizeof(uint64_t) + sizeof(int32_t)) +
                (size_t)npol * (sizeof(int32_t) + sizeof(double)) + (hd.has_image ? (size_t)W_ * H_ : 0) +
                (hd.has_mask ? (size_t)W_ * H_ : 0);
  if (n_bytes) *n_bytes = need;
  if (!buf || cap < need) return buf ? FE_OVERFLOW : FE_OK;
  uint8_t *p = static_cast<uint8_t *>(buf);
  auto put = [&](const void *src, size_t n) { std::memcpy(p, src, n); p += n; };
  put(&hd, sizeof(hd));
  put(pts_last_.data(), pts_last_.size() * sizeof(Pt));
  put(ids_last_.data(), ids_last_.size() * sizeof(uint64_t));
  put(lines_last_.data(), lines_last_.size() * sizeof(float4));
  put(line_ids_last_.data(), line_ids_last_.size() * sizeof(uint64_t));
  for (auto &m : pol_last_) { int32_t k = (int32_t)m.size(); put(&k, sizeof(k)); }
  for (auto &m : pol_last_)
    for (auto &kv : m) { int32_t k = kv.first; put(&k, sizeof(k)); put(&kv.second, sizeof(double)); }
  if (hd.has_image) {
    const DevImage &l0 = slots_[last_slot_].pyr.lvl[0];
    FE_CUDA(cudaMemcpy2D(p, W_, l0.p, l0.pitch, W_, H_, cudaMemcpyDeviceToHost));
    p += (size_t)W_ * H_;
  }
  if (hd.has_mask) put(slots_[last_slot_].mask.data(), (size_t)W_ * H_);
  return FE_OK;
  }();
  if (rc == FE_CUDA_ERROR) last_error = t_err;
  return rc;
}

int FeContext::set_state(const void *buf, size_t n_bytes) {
  if (!buf || n_bytes < sizeof(StateHeader) || !queue_.empty()) return FE_BAD_ARG;
  int rc = [&]() -> int {
  FE_CUDA(cudaSetDevice(device_));
  const uint8_t *p = static_cast<const uint8_t *>(buf);
  StateHeader hd;
  std::memcpy(&hd, p, sizeof(hd));
  p += sizeof(hd);
  if (hd.magic != 0x504c5657u || hd.version != 1 || hd.w != W_ || hd.h != H_) return FE_BAD_ARG;
  if (hd.n_pts < 0 || hd.n_lines < 0 || hd.n_pol_entries < 0) return FE_BAD_ARG;
  {   // the blob must hold everything its header announces (a truncated or foreign buffer is rejected, not read past)
    const size_t need = sizeof(hd) + (size_t)hd.n_pts * (sizeof(Pt) + sizeof(uint64_t)) +
                        (size_t)hd.n_lines * (sizeof(float4) + sizeof(uint64_t) + sizeof(int32_t)) +
                        (size_t)hd.n_pol_entries * (sizeof(int32_t) + sizeof(double)) + (hd.has_image ? (size_t)W_ * H_ : 0) +
                        (hd.has_image && hd.has_mask ? (size_t)W_ * H_ : 0);
    if (n_bytes < need) return FE_BAD_ARG;
  }
  auto get = [&](void *dst, size_t n) { std::memcpy(dst, p, n); p += n; };
  // parse into temporaries: the tracker state is only replaced once the whole blob has been checked
  std::vector<Pt> t_pts(hd.n_pts);
  std::vector<uint64_t> t_ids(hd.n_pts);
  get(t_pts.data(), (size_t)hd.n_pts * sizeof(Pt));
  get(t_ids.data(), (size_t)hd.n_pts * sizeof(uint64_t));
  std::vector<float4> t_lines(hd.n_lines);
  std::vector<uint64_t> t_lids(hd.n_lines);
  get(t_lines.data(), (size_t)hd.n_lines * sizeof(float4));
  get(t_lids.data(), (size_t)hd.n_lines * sizeof(uint64_t));
  std::vector<int32_t> sizes(hd.n_lines);
  get(sizes.data(), (size_t)hd.n_lines * sizeof(int32_t));
  long long tot = 0;
  for (int32_t v : sizes) {
    if (v < 0) return FE_BAD_ARG;
    tot += v;
  }
  if (tot != hd.n_pol_entries) return FE_BAD_ARG;   // the entries the lines announce are the entries the blob holds
  std::vector<std::map<int, double>> t_pol(hd.n_lines);
  for (int i = 0; i < hd.n_lines; i++)
    for (int k = 0; k < sizes[i]; k++) {
      int32_t key;
      double val;
      get(&key, sizeof(key));
      get(&val, sizeof(val));
      t_pol[i][key] = val;
    }
  currid_ = hd.currid;
  line_currid_ = hd.line_currid;
  pts_last_.swap(t_pts);
  ids_last_.swap(t_ids);
  lines_last_.swap(t_lines);
  line_ids_last_.swap(t_lids);
  pol_last_.swap(t_pol);
  for (FrameSlot &s : slots_) {
    s.busy = false;
  }
  FE_CUDA(cudaDeviceSynchronize());
  last_slot_ = -1;
  klt_last_slot_ = -1;
  cur_slot_ = -1;
  spec_valid_ = false;
  prev_submit_slot_ = -1;
  last_src_.clear();
  state_res_.clear();
  state_res_.obs = pts_last_;
  state_res_.obs_ids = ids_last_;
  cur_res_ = &state_res_;
  if (hd.has_image) {
    FrameSlot &s = slots_[0];
    s.busy = true;
    FE_CUDA(cudaMemcpy2DAsync(s.raw.p, s.raw.pitch, p, W_, W_, H_, cudaMemcpyHostToDevice, s.s_a));
    p += (size_t)W_ * H_;
    // the stored image is already equalised: rebuild the pyramid from it without a LUT
    launch_eq_pyr1(s.raw, s.d_hist, s.d_counters, 0, s.pyr.lvl[0], s.pyr.n > 1 ? s.pyr.lvl[1] : DevImage(),
                   cfg_.use_lines ? s.half : DevImage(), s.s_a);
    if (s.pyr.n > 2) launch_pyr_rest(s.pyr, s.d_counters + 1, s.s_a);
    FE_CUDA(cudaEventRecord(s.ev_pyr, s.s_a));
    FE_CUDA(cudaStreamSynchronize(s.s_a));
    {
      int rc = enqueue_fast_all_cells(s);
      if (rc) return rc;
      FE_CUDA(cudaStreamWaitEvent(s.s_b, s.ev_pyr, 0));
      rc = record_fast_path(s, s.s_b);
      if (rc) return rc;
      s.seq_fast++;
      FE_CUDA(cudaEventRecord(s.ev_fast, s.s_b));
    }
    if (hd.has_mask) {
      s.mask.resize((size_t)W_ * H_);
      get(s.mask.data(), (size_t)W_ * H_);
    } else {
      s.mask.clear();
    }
    last_slot_ = 0;
    klt_last_slot_ = 0;
    prev_submit_slot_ = 0;
  }
  return FE_OK;
  }();
  if (rc == FE_CUDA_ERROR) last_error = t_err;
  return rc;
}

int FeContext::tap(int what, void *buf, size_t cap, size_t *n_bytes) {
  FE_CUDA(cudaSetDevice(device_));
  const int si = cur_slot_ >= 0 ? cur_slot_ : last_slot_;
  const FrameResult &res = *cur_res_;
  const std::vector<int32_t> &tap_fast_ = res.tap_fast;
  const std::vector<float> &tap_lk_ = res.tap_lk, &tap_subpix_ = res.tap_subpix, &tap_fld_ = res.tap_fld;
  auto copy_vec = [&](const void *src, size_t n) -> int {
    if (n_bytes) *n_bytes = n;
    if (!buf) return FE_OK;
    if (cap < n) return FE_OVERFLOW;
    std::memcpy(buf, src, n);
    return FE_OK;
  };
  if (what == FE_TAP_FAST_LAST) return copy_vec(tap_fast_.data(), tap_fast_.size() * sizeof(int32_t));
  if (what == FE_TAP_LK_LAST) return copy_vec(tap_lk_.data(), tap_lk_.size() * sizeof(float));
  if (what == FE_TAP_SUBPIX_LAST) return copy_vec(tap_subpix_.data(), tap_subpix_.size() * sizeof(float));
  if (what == FE_TAP_FLD_LAST) return copy_vec(tap_fld_.data(), tap_fld_.size() * sizeof(float));
  if (si < 0) return FE_BAD_ARG;
  FrameSlot &s = slots_[si];
  FE_CUDA(cudaDeviceSynchronize());
  if (what >= FE_TAP_PYR_LEVEL0 && what < FE_TAP_PYR_LEVEL0 + kMaxLevels) {
    int l = what - FE_TAP_PYR_LEVEL0;
    if (l >= s.pyr.n) return FE_BAD_ARG;
    const DevImage &im = s.pyr.lvl[l];
    size_t n = (size_t)im.w * im.h;
    if (n_bytes) *n_bytes = n;
    if (!buf) return FE_OK;
    if (cap < n) return FE_OVERFLOW;
    FE_CUDA(cudaMemcpy2D(buf, im.w, im.p, im.pitch, im.w, im.h, cudaMemcpyDeviceToHost));
    return FE_OK;
  }
  if (what == FE_TAP_HALF && cfg_.use_lines) {
    const DevImage &im = s.half;
    size_t n = (size_t)im.w * im.h;
    if (n_bytes) *n_bytes = n;
    if (!buf) return FE_OK;
    if (cap < n) return FE_OVERFLOW;
    FE_CUDA(cudaMemcpy2D(buf, im.w, im.p, im.pitch, im.w, im.h, cudaMemcpyDeviceToHost));
    return FE_OK;
  }
  return FE_BAD_ARG;
}

}  // namespace plviwo
