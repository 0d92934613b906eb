// Device-side data of a stream group (FeGroup, fe_group.cu): the per-stream tracker state that the reference keeps in
// TrackBase / TrackLSD members (TrackBase.h:173-192, TrackLSD.h:248-279) lives in device memory, so that a frame of every
// stream goes through the whole state machine — top-off detection, LK, RANSAC gate, row filter, line association — as a
// fixed sequence of kernel launches with no host round trip.  Not part of the C ABI.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

#include "../../include/plviwo_fe.h"
#include "fe_kernels.h"

namespace plviwo {

// One frame of one stream in a tracking launch (grid.y / grid.z = job).
struct TrackJob {
  int stream;
  int cur_slot, prev_slot;   // indices into the SlotRec table; prev_slot < 0: no previous image (first frame of the stream)
  int flags;                 // bit 0: run the line tracker (vanishing points given)
  int out;                   // index of the frame's output record = of the state record the frame WRITES (pts_last after it)
  int prev_rec;              // state record holding the stream's pts_last / ids_last BEFORE this frame
  double timestamp;
  double K[4], D[4];         // calibration in force when the frame was submitted
  double vp[6];
};

// Header of a frame's output record in pinned host memory; followed by the rows (fixed capacities, GroupDev).
struct GroupOutHeader {
  FeFrameInfo info;
  int32_t n_obs;             // pts_last / ids_last after the frame
  int32_t n_line_points;
  int32_t status;            // FE_OK or FE_INTERNAL (a capacity was exceeded: the message says which)
  int32_t overflow_what;     // 1 points, 2 lines, 3 point/line pairs, 4 candidates
  int32_t n_samples;         // cfg.line_samples: samples tracked in this frame (0 when the frame made no LK call)
  int32_t reserved[11];
};

constexpr int kValidStride = 260;

struct GroupDev {
  // ---- geometry / parameters (FeConfig)
  int W, H;
  int n_streams;
  int num_features, grid_x, grid_y, min_px_dist;
  int n_cells, nfg;              // Grider_GRID cell layout (fe_group.cu: layout_cells)
  int cell_of_loc[256];          // caller-grid (x * grid_y + y) -> cell index or -1
  int close_w, close_h;
  float line_min_length;
  int use_lines;
  // ---- capacities
  int pts_cap, lines_cap, pol_cap, cand_cap, segs_cap;
  // ---- slot table
  const SlotRec *slots;
  const int *slot_flags;
  // ---- point tracker state.  pts_last / ids_last live in a RING of records (one per output record: tick ring x stream), record
  // r at r * pts_cap: the frame of a tick reads its stream's previous record and writes its own, so the line association of a
  // tick — which reads the points of ITS tick and may run much later than the point chain, after the batch's chain walk —
  // never holds up the next tick's point chain.
  float2 *pts;
  uint64_t *ids;
  int *n_pts;                    // per record
  uint64_t *currid;              // per stream
  // ---- work arrays of the frame being tracked
  float2 *wpts;                  // pts_old after the top-off detection (LK input)
  uint64_t *wids;
  int *wn;
  int *wmode;                    // 0 track, 1 first frame (detection only), 2 nothing to do
  int *winfo;                    // per stream [detection_ran, n_detected, overflow, candidates to refine]
  float2 *lk_pts1, *lk_p0n, *lk_p1n;
  uint8_t *lk_status;
  int *close;                    // min-distance grid of the detection, stream s at s * close_w * close_h
  int *valid;                    // valid cells of the detection, stream s at s * kValidStride: [0] count, [4 + i] cell index (or -1)
  unsigned long long *stats;     // [0] grid cells FAST ran on (all streams, since creation)
  float2 *ext_in;                // candidates of the valid cells that passed the mask test, stream s at s * cand_cap
  float2 *ext_pt;                // ... after cornerSubPix
  // ---- line tracker state, double buffered (buffer b of stream s at (2 * s + b) * cap)
  float4 *lines;
  uint64_t *line_ids;
  int *pol_off;                  // lines_cap + 1 per buffer
  int *pol_pid;                  // pol_cap per buffer, ascending within a line
  float *pol_dist;
  int *n_lines;                  // per buffer
  int *line_buf;                 // per stream: which buffer holds lines_last
  uint64_t *line_currid;
  // scratch of the line association, per stream
  float4 *lnew;                  // lines_cap: detected lines longer than line_min_length (full-res)
  int *n_lnew;                   // per stream: lines in lnew, written with it (the segments the next frame's samples lie on)
  int *lcnt, *loff;              // lines_cap (+1): points per line, entry offsets
  float2 *lpos;                  // pol_cap: point_position entries (detection order)
  int *lmatch;                   // lines_cap
  // ---- outputs (pinned, device-mapped): record r at out + r * out_stride
  uint8_t *out;
  size_t out_stride;
  size_t off_rows, off_obs_ids, off_obs_uv, off_lrows, off_lpts;   // byte offsets inside a record
  // cfg.line_samples (0: off, no region): samples per segment, the handle's LK buffer size (max_pts, fe_context.cu) that
  // truncates them, and the record's sample region: sample_cap positions p0, p1 (float2) and status bytes
  int line_samples, sample_max_pts, sample_cap;
  size_t off_sp0, off_sp1, off_sst;
};

// tracking launches (kernels_glue.cu, kernels_track.cu)
// the top-off detection of a tick: k_group_detect (existing points, valid cells) -> FAST + selection on the VALID cells only
// (Grider_GRID.h:108-151 runs cv::FAST on valid_locs only) -> k_group_cands (mask / occupancy test of the candidates)
// -> cornerSubPix -> k_group_accept
void launch_group_detect(const GroupDev &g, const TrackJob *jobs, int n_jobs, cudaStream_t s);
void launch_group_fast(const GroupDev &g, const TrackJob *jobs, int n_jobs, const FrontGeom &fg, cudaStream_t s);          // kernels_fast.cu
void launch_group_fast_select(const GroupDev &g, const TrackJob *jobs, int n_jobs, const FrontGeom &fg, cudaStream_t s);   // kernels_fast.cu
void launch_group_cands(const GroupDev &g, const TrackJob *jobs, int n_jobs, cudaStream_t s);
void launch_group_subpix(const GroupDev &g, const TrackJob *jobs, int n_jobs, cudaStream_t s);   // kernels_track.cu
void launch_group_accept(const GroupDev &g, const TrackJob *jobs, int n_jobs, cudaStream_t s);
void launch_group_lk(const GroupDev &g, const TrackJob *jobs, int n_jobs, const LkParams &prm, cudaStream_t s);
void launch_group_gate(const GroupDev &g, const TrackJob *jobs, int n_jobs, cudaStream_t s);
// cfg.line_samples: LK of the samples along the stream's last detected segments (lnew), previous -> current pyramid, for the
// frames whose point LK ran; reads the header the gate wrote and lnew before this tick's k_group_lines rewrites it
void launch_group_line_samples(const GroupDev &g, const TrackJob *jobs, int n_jobs, const LkParams &prm, cudaStream_t s);
void launch_group_lines(const GroupDev &g, const TrackJob *jobs, int n_jobs, cudaStream_t s);

}  // namespace plviwo
