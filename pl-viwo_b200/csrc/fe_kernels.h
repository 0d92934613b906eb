// Internal C++ interface between the host-side trackers and the sm_100a kernels (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <cstdint>

namespace plviwo {

// Opt-in to more than 48 KB of dynamic shared memory.  The attribute is per DEVICE (handles of one process may live on
// different GPUs) and launches come from several host threads: remember the largest request per device.
struct SmemOptIn {
  std::atomic<size_t> granted[64];
  SmemOptIn() { for (auto &g : granted) g.store(0); }
  template <class Kernel>
  void ensure(Kernel kernel, size_t bytes) {
    if (bytes <= 48 * 1024) return;
    int dev = 0;
    cudaGetDevice(&dev);
    std::atomic<size_t> &g = granted[dev & 63];
    if (bytes > g.load(std::memory_order_relaxed)) {
      cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
      g.store(bytes, std::memory_order_relaxed);
    }
  }
};

// One shared-memory / L1 split for EVERY kernel of the library (PLVIWO_CARVEOUT = percent of the SM's unified storage
// preferred as shared memory; default 100, -1 = the driver's per-kernel default).  Kernels that prefer different splits cannot share
// an SM until it has drained and been reconfigured; with dozens of kernels of several frames resident at once — among
// them millisecond-long persistent ones that opt in to > 48 KB — a short latency-critical launch then only gets the SMs
// whose current split happens to suit it.
int carveout_percent();   // -1: leave the default
struct CarveoutOnce {
  std::atomic<bool> done[64];
  CarveoutOnce() { for (auto &d : done) d.store(false); }
  template <class Kernel>
  void apply(Kernel kernel) {
    const int pct = carveout_percent();
    if (pct < 0) return;
    int dev = 0;
    cudaGetDevice(&dev);
    std::atomic<bool> &d = done[dev & 63];
    if (d.load(std::memory_order_relaxed)) return;
    cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
    d.store(true, std::memory_order_relaxed);
  }
};
#define PLVIWO_CARVEOUT(kernel)   \
  do {                            \
    static CarveoutOnce c__;      \
    c__.apply(kernel);            \
  } while (0)

struct DevImage {
  uint8_t *p = nullptr;
  int w = 0, h = 0, pitch = 0;
};

constexpr int kMaxLevels = 8;       // pyramid images (maxLevel + 1)
constexpr int kFastBandRows = 16;   // rows per FAST CTA band
constexpr int kMaxWin = 31;

struct Pyramid {
  DevImage lvl[kMaxLevels];
  int n = 0;  // number of images actually built (maxLevel + 1, fewer if a level gets <= win)
};

// ---- image kernels (kernels_image.cu) -------------------------------------------------------------------
// hist[256] must be zero on entry (the equalise kernel re-zeroes it when it is done with it).
void launch_hist(const DevImage &src, unsigned *d_hist, cudaStream_t s);
// LUT from hist (cv::equalizeHist), level 0 = lut[src] (or a plain copy when equalize == 0), level 1 = pyrDown,
// half = exact 2x2 INTER_AREA of level 0 (may be null).  d_hist is cleared for the next frame by the last CTA.
// equalize: 0 copy, 1 cv::equalizeHist LUT from d_hist, 2 CLAHE blend of the 64 tile LUTs in d_clahe_luts.
void launch_eq_pyr1(const DevImage &src, unsigned *d_hist, unsigned *d_counter, int equalize, const DevImage &l0,
                    const DevImage &l1, const DevImage &half, cudaStream_t s, const uint8_t *d_clahe_luts = nullptr);
// cv::createCLAHE(10.0, 8x8): the 64 tile LUTs (64 * 256 bytes) of the frame
void launch_clahe_lut(const DevImage &src, uint8_t *d_luts, cudaStream_t s);
// levels 2..n-1, one short launch per level (4 outputs per thread).
void launch_pyr_rest(const Pyramid &pyr, unsigned *d_counter, cudaStream_t s);
// cv::pyrDown(src, dst, Size(dst.w, dst.h)) for one image (|2 dst - src| <= 2 per side)
void launch_pyr_down(const DevImage &src, const DevImage &dst, cudaStream_t s);

void launch_signal(int *host_flag, int value, cudaStream_t s);
void launch_signal_inc(int *host_flag, int *dev_seq, cudaStream_t s);
void init_fld_constants();      // chain-walk decision table (kernels_lines.cu)
void init_device_constants();   // constant-memory tables (sub-pixel mask); call once per device before capturing graphs

// ---- FAST (kernels_fast.cu) ------------------------------------------------------------------------------
struct FastCell {
  int x, y, w, h;  // ROI in level-0 pixels
};
// Output: d_total (1 counter, must be 0 on entry), per (cell, band) offset/count tables and packed keypoints
// (x | y << 12 | score << 24, cell-local coordinates) written compactly at [offset, offset + count).
void launch_fast(const DevImage &img, const FastCell *d_cells, int n_cells, int max_bands, int max_cell_w, int threshold,
                 unsigned *d_total, int *d_band_off, int *d_band_cnt, unsigned *d_kps, int kps_cap, cudaStream_t s);

// Per-cell std::sort + top num_features_grid (Grider_GRID.h:128-133) on the device.  d_total: 2 counters, both zero on
// entry of launch_fast ([0] corners, [1] scratch cursor); d_scratch: kps_cap words; output: cell c's survivors at
// d_cand_sel[c * nfg ..] (full-image coordinates), d_cand_cnt[c] of them.
void launch_fast_select(const FastCell *d_cells, int n_cells, int max_bands, unsigned *d_total, const int *d_band_off,
                        const int *d_band_cnt, const unsigned *d_kps, int kps_cap, unsigned *d_scratch, int nfg,
                        float2 *d_cand_sel, int *d_cand_cnt, cudaStream_t s);
void host_sort_corners(unsigned *v, int n, int keep = 0);   // the same introsort on the host (tests); keep > 0: sort_prefix

// ---- cornerSubPix (kernels_track.cu) ----------------------------------------------------------------------
// n points; with d_cnt != null the points are a fixed-stride table (slot i belongs to cell i / stride and is live only if
// i % stride < d_cnt[cell]).  d_in == d_out is allowed.
void launch_corner_subpix(const DevImage &img, const float2 *d_in, float2 *d_out, int n, cudaStream_t s,
                          const int *d_cnt = nullptr, int stride = 0);

// ---- pyramidal LK + undistort (kernels_track.cu) ----------------------------------------------------------
struct LkParams {
  int win;         // odd
  int max_level;   // pyramid images - 1
  int max_count;   // 30
  float eps_sq;    // 0.01^2
  float min_eig;   // 1e-4
  double K[4], D[4];
  int undistort;   // also write normalised coordinates of pts0 / pts1
};
// host_flag / flag_value / d_done_counter (optional): the kernel itself publishes flag_value to the pinned word when its
// last feature is done (d_done_counter: one zeroed device word).  Returns true if the kernel will do so; false means
// the caller has to queue its own completion signal (generic-window kernel).
bool launch_lk(const Pyramid &prev, const Pyramid &next, const float2 *d_pts0, float2 *d_pts1, uint8_t *d_status,
               float2 *d_p0n, float2 *d_p1n, int n, const LkParams &prm, cudaStream_t s, int *host_flag = nullptr,
               int flag_value = 0, unsigned *d_done_counter = nullptr, const int *d_tab_cnt = nullptr, int tab_stride = 0,
               bool flow_is_zero = false, const unsigned *cell_mask = nullptr);
// table mode (15 x 15 window, <= 6 pyramid images only — lk_table_mode_ok): d_pts0 is a fixed-stride candidate table (slot i
// belongs to cell i / tab_stride, live iff i % tab_stride < d_tab_cnt[cell]); flow_is_zero: the initial guess is the
// previous position, d_pts1 is written only; cell_mask (8 words, optional): only cells whose bit is set are tracked.
bool lk_table_mode_ok(const LkParams &prm, int pyramid_images);
// k_lk15w_g's one-warp-per-feature body on n points over one pyramid pair (15 x 15 window, <= 6 pyramid images, no
// undistortion; false otherwise): the same results as launch_lk's k_lk15, bit for bit
bool launch_lk_warp(const Pyramid &prev, const Pyramid &next, const float2 *d_pts0, float2 *d_pts1, uint8_t *d_status, int n,
                    const LkParams &prm, cudaStream_t s);
void launch_undistort(const float2 *d_pts, float2 *d_out, int n, const double K[4], const double D[4], cudaStream_t s);

// ---- lines (kernels_lines.cu) -------------------------------------------------------------------------------
struct FldBuffers {
  unsigned *edges = nullptr;      // bit-packed edge map, words_per_row * h
  int words_per_row = 0;
  int *label = nullptr;           // connected-component label per pixel (root = smallest raster index), -1 = no edge
  int *cnt = nullptr;             // pixels per component (at the root)
  int *bbox = nullptr;            // 3 planes at the root: max y, min x, max x (min y is the root's row)
  int *lroots = nullptr;          // tile-local roots of the connected-component pass (k_ccl_tile -> k_ccl_link)
  int *lroot_n = nullptr;
  int lroot_cap = 0;
  int *comp_root = nullptr;       // roots of the components big enough to hold a chain
  int *counters = nullptr;        // [0] components [1] - [2] chain-point cursor [3] chains [4] segments
  int2 *chain_pts = nullptr;      // chain points, one slice per component (capacity = w * h)
  int *chain_seed = nullptr, *chain_off = nullptr, *chain_len = nullptr, *order = nullptr;
  int max_chains = 0;
  float4 *segs = nullptr;         // segment slots (chain_off / 21 + j)
  int *seg_cnt = nullptr;         // [0, max_chains): segments per chain in seed order; [max_chains, 2 max_chains): slot base
  float4 *out = nullptr;          // compacted, ordered segments
  int out_cap = 0;
  int alloc(int w, int h, int length_threshold, int out_capacity);   // returns 0 on success
  void release();
};
// The line paths of several frames in one set of launches (grid.y / grid.z = frame): per-frame kernel TIME is what limits
// a stream (the chain walk alone is > 1 ms of latency per frame and the device runs a limited number of kernels at
// once), so frames submitted back to back share their launches.  All frames of a batch have the same size.
constexpr int kMaxLineBatch = 8;
struct FldBatch {
  int n = 0;
  DevImage half[kMaxLineBatch];
  FldBuffers f[kMaxLineBatch];
  __host__ __device__ const DevImage &half_of(int k) const { return half[k]; }
  __host__ __device__ const FldBuffers &fld_of(int k) const { return f[k]; }
};
void launch_canny_batch(const FldBatch &b, float th_low, float th_high, cudaStream_t s);
void launch_fld_batch(const FldBatch &b, int length_threshold, float distance_threshold, cudaStream_t s, cudaEvent_t *ev = nullptr);
constexpr int kSegsPerChainDiv = 21;  // a chain of n points yields at most n / 21 + 1 segments
void launch_canny(const DevImage &half, float th_low, float th_high, FldBuffers &fb, cudaStream_t s);
// ev (optional, 2 events): recorded after the connected-component kernels and after the chain walk (stage timing)
void launch_fld(const DevImage &half, int length_threshold, float distance_threshold, FldBuffers &fb, cudaStream_t s,
                cudaEvent_t *ev = nullptr);
void launch_unpack_edges(const FldBuffers &fb, int w, int h, uint8_t *d_out, cudaStream_t s);

// ---- batched multi-stream launches (FeGroup, fe_group.cu) ------------------------------------------------------
// A stream group processes one frame of MANY camera streams per launch (grid.z = job).  Every frame slot of every
// stream is described once, at creation, by a SlotRec in device memory; a launch gets a device array of jobs that name
// slots by index, so the same launch sequence serves any mix of streams without re-encoding kernel arguments.
struct SlotRec {
  DevImage raw;                  // staging of a host-fed frame (device-resident inputs are read in place)
  DevImage lvl[kMaxLevels];      // equalised pyramid, level 0 = equalised frame
  int n_lvl;
  DevImage half;                 // half-resolution equalised frame (line detector input)
  uint8_t *mask;                 // caller mask of the frame (w * h bytes, tight); valid iff the slot's flag bit 0 is set
  unsigned *hist, *counters;     // 256 bins (zero between frames), 4 counters
  uint8_t *clahe;                // 64 tile LUTs
  unsigned *fast_total;          // [0] corners [1] scratch cursor
  unsigned *kps, *sort_scratch;
  int *band_off, *band_cnt;
  float2 *cand;                  // per-cell candidate table (cell c at c * nfg)
  int *cand_cnt;
  FldBuffers fld;
};
struct FrontJob {
  const uint8_t *src;            // the frame: device pointer (caller's, or the slot's raw staging)
  int src_pitch;
  int slot;                      // index into the SlotRec table
  int eq_mode;                   // 0 copy, 1 cv::equalizeHist, 2 CLAHE
  int flags;                     // bit 0: the slot's mask buffer holds this frame's mask
};
struct FrontGeom {               // the same for every stream of a group
  int w, h;                      // tracking size
  int n_cells, max_bands, max_cell_w, fast_threshold, kps_cap, nfg;
  const FastCell *cells;
};
// State-independent work of n_jobs frames: histogram (+ CLAHE tile LUTs), equalise + pyramid (+ the half-resolution
// line input).  FAST, its per-cell selection and cornerSubPix run later, on demand, on the cells the tracker leaves
// open (fe_group_dev.h).
void launch_hist_batch(const SlotRec *slots, const FrontJob *jobs, int n_jobs, const FrontGeom &g, int *slot_flags, cudaStream_t s);
void launch_clahe_lut_batch(const SlotRec *slots, const FrontJob *jobs, int n_jobs, const FrontGeom &g, cudaStream_t s);
void launch_eq_pyr1_batch(const SlotRec *slots, const FrontJob *jobs, int n_jobs, const FrontGeom &g, bool want_half, cudaStream_t s);
void launch_pyr_level_batch(const SlotRec *slots, const FrontJob *jobs, int n_jobs, int level, int dw, int dh, cudaStream_t s);
// The line kernels take either a FldBatch by value (a few frames of one handle) or this view of the slot table
// (entry k of the launch = slot idx[k]); same kernel bodies, instantiated for both.
struct FldTable {
  const SlotRec *slots;
  const int *idx;
  __device__ const DevImage &half_of(int k) const { return slots[idx[k]].half; }
  __device__ const FldBuffers &fld_of(int k) const { return slots[idx[k]].fld; }
};
// Line paths of n_jobs frames; line_slots: device array of slot indices.  ev as launch_fld.  launch_canny_table also labels
// the connected components of every 64 x 16 tile (fused into the Canny kernel); launch_fld_table continues from there and
// must follow it on the same stream.
void launch_canny_table(const SlotRec *slots, const int *line_slots, int n_jobs, int w, int h, float th_low, cudaStream_t s);
void launch_fld_table(const SlotRec *slots, const int *line_slots, int n_jobs, int w, int h, int max_chains, int length_threshold,
                      float distance_threshold, cudaStream_t s, cudaEvent_t *ev = nullptr);

}  // namespace plviwo
