// State-dependent steps of the front end on the device (sm_100a), one CTA per camera stream of a stream group:
//
//   k_group_detect   TrackKLT::perform_detection_monocular (TrackKLT.cpp:395-528) — the occupancy loop and the valid-cell
//                    list; FAST + selection then run on the valid cells only (kernels_fast.cu: k_fast_g, k_fast_select_g);
//   k_group_cands    the mask test of Grider_GRID.h:140-147 on the candidates; k_group_accept (after cornerSubPix) the
//                    minimum-distance rejection and the id assignment
//   k_group_gate     the tail of TrackKLT::perform_matching (:862-885: cv::findFundamentalMat(FM_RANSAC) on the undistorted
//                    pairs, mask_klt && mask_rsc) and of feed_monocular (:143-189: reset, bounds / mask filter, the rows of
//                    FeatureDatabase::update_feature, pts_last / ids_last)
//   k_group_lines    viw::TrackLSD::feed_monocular after the detector (TrackLSD.cpp:127-182): x2 + FilterShortLines + ids
//                    (:218-236), AssignPointToLines (:744-792, bounding-box index mix-up kept), LineMatch (:368-407, the
//                    last satisfying line wins), LineClassification (:318-366, atan(dy)/dx kept), the rows of
//                    LineFeatureDatabase::update_feature
//
// The host glue of a single handle (fe_context.cu: filter_existing / grid_candidates / perform_detection / klt_feed /
// lsd_feed) is the sequential statement of the same steps; here every loop whose iterations only interact through "the
// first one in order wins" is run in parallel with an atomicMin on the order index plus an ordered compaction, which
// gives the sequential result exactly.  Compiled with --fmad=false: float expressions round where the host's do.
#include "fe_group_dev.h"
#include "ransac_core.h"

#include <cfloat>
#include <climits>

namespace plviwo {

constexpr int kGT = 256;           // threads per CTA (one CTA per stream)
constexpr int kExtBase = 1 << 24;  // min-distance grid: marks of new candidates are kExtBase + order index

struct BlockScan {
  int warp_tot[kGT / 32];
  int total;
};
// exclusive prefix of v over the CTA (all threads call); bs.total = sum, valid until the next call
__device__ __forceinline__ int block_excl(int v, BlockScan &bs) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int x = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, x, d);
    if (lane >= d) x += t;
  }
  __syncthreads();   // the previous call's total has been read by everybody
  if (lane == 31) bs.warp_tot[w] = x;
  __syncthreads();
  int base = 0;
  for (int k = 0; k < w; k++) base += bs.warp_tot[k];
  if (threadIdx.x == kGT - 1) bs.total = base + x;
  __syncthreads();
  return base + x - v;
}
__device__ __forceinline__ int block_sum(int v, BlockScan &bs) {
  block_excl(v, bs);
  return bs.total;
}

__device__ __forceinline__ GroupOutHeader *out_header(const GroupDev &g, const TrackJob &job) {
  return reinterpret_cast<GroupOutHeader *>(g.out + (size_t)job.out * g.out_stride);
}

// ======================================================================================== top-off detection
__global__ void __launch_bounds__(kGT)
    k_group_detect(const __grid_constant__ GroupDev g, const TrackJob *__restrict__ jobs) {
  __shared__ BlockScan bs;
  __shared__ int grid_cnt[256];
  const TrackJob &job = jobs[blockIdx.x];
  const int s = job.stream, tid = threadIdx.x;
  const int cols = g.W, rows = g.H, d = g.min_px_dist, gx = g.grid_x, gy = g.grid_y;
  const int close_w = g.close_w, close_h = g.close_h, close_n = close_w * close_h;
  const int n0 = g.n_pts[job.prev_rec];
  // TrackKLT.cpp:110-123 — nothing tracked last time (or no previous image): detect on the CURRENT image only
  const bool first = n0 == 0 || job.prev_slot < 0;
  const int islot = first ? job.cur_slot : job.prev_slot;
  const SlotRec &sl = g.slots[islot];
  const uint8_t *__restrict__ mask = (g.slot_flags[islot] & 1) ? sl.mask : nullptr;
  const size_t o = (size_t)s * g.pts_cap;
  const float2 *__restrict__ pts = g.pts + (size_t)job.prev_rec * g.pts_cap;
  const uint64_t *__restrict__ ids = g.ids + (size_t)job.prev_rec * g.pts_cap;
  float2 *__restrict__ wpts = g.wpts + o;
  uint64_t *__restrict__ wids = g.wids + o;
  int *__restrict__ close = g.close + (size_t)s * close_n;
  const int np = first ? 0 : n0;
  const float size_x = (float)cols / (float)gx, size_y = (float)rows / (float)gy;

  for (int i = tid; i < close_n; i += kGT) close[i] = INT_MAX;
  grid_cnt[tid] = 0;
  __syncthreads();

  // ---- first loop (:411-464).  A point is kept iff it passes the tests that do not depend on the other points (border,
  // grids, mask) and no EARLIER such point sits in its min-distance cell: first in order per cell wins.
  auto classify = [&](float2 kp, int &cell, int &gcell) -> bool {
    const int x = (int)kp.x, y = (int)kp.y;
    const int edge = 10;
    if (x < edge || x >= cols - edge || y < edge || y >= rows - edge) return false;
    const int xc = (int)(kp.x / (float)d), yc = (int)(kp.y / (float)d);
    if (xc < 0 || xc >= close_w || yc < 0 || yc >= close_h) return false;
    const int xg = (int)floorf(kp.x / size_x), yg = (int)floorf(kp.y / size_y);
    if (xg < 0 || xg >= gx || yg < 0 || yg >= gy) return false;
    if (mask != nullptr && mask[(size_t)y * cols + x] > 127) return false;
    cell = yc * close_w + xc;
    gcell = yg * gx + xg;
    return true;
  };
  for (int k = tid; k < np; k += kGT) {
    int cell, gcell;
    if (classify(pts[k], cell, gcell)) atomicMin(&close[cell], k);
  }
  __syncthreads();
  int nk = 0;
  for (int base = 0; base < np; base += kGT) {
    const int k = base + tid;
    int cell = 0, gcell = 0;
    float2 kp = make_float2(0.f, 0.f);
    bool keep = false;
    if (k < np) {
      kp = pts[k];
      keep = classify(kp, cell, gcell) && close[cell] == k;
    }
    const int e = block_excl(keep ? 1 : 0, bs);
    if (keep) {
      wpts[nk + e] = kp;
      wids[nk + e] = ids[k];
      atomicAdd(&grid_cnt[gcell], 1);   // the reference saturates at 255; only "< required" is ever asked
    }
    nk += bs.total;
  }
  __syncthreads();

  int detection_ran = 0;
  const double min_feat_percent = 0.50;
  const int need = g.num_features - nk;
  const int need_min = min(20, (int)(min_feat_percent * g.num_features));
  int *__restrict__ valid = g.valid + (size_t)s * kValidStride;
  if (need >= need_min) {   // :468-471
    detection_ran = 1;
    // ---- valid cells in x-major order (:479-492)
    if (tid == 0) {
      int nv = 0;
      const int nfg_caller = (int)((double)g.num_features / (double)(gx * gy)) + 1;
      const int req = max(1, (int)(min_feat_percent * nfg_caller));
      const double ifx = 1.0 / ((double)gx / (double)cols), ify = 1.0 / ((double)gy / (double)rows);
      for (int x = 0; x < gx; x++)
        for (int y = 0; y < gy; y++) {
          int mg = 0;
          if (mask != nullptr) {   // resize(mask0, grid, INTER_NEAREST)
            const int sy = min((int)floor(y * ify), rows - 1), sx = min((int)floor(x * ifx), cols - 1);
            mg = mask[(size_t)sy * cols + sx];
          }
          if (min(grid_cnt[y * gx + x], 255) < req && mg != 255) valid[4 + nv++] = g.cell_of_loc[x * gy + y];
        }
      valid[0] = nv;
      atomicAdd(g.stats, (unsigned long long)nv);
    }
  }
  if (tid == 0) {
    if (!detection_ran) valid[0] = 0;
    // the FAST counters of the image the detection is about (k_fast_g / k_fast_select_g follow on this CUDA stream)
    sl.fast_total[0] = 0;
    sl.fast_total[1] = 0;
    g.wn[s] = nk;                       // points kept so far; k_group_accept appends the new ones
    g.wmode[s] = first ? 1 : 0;
    g.winfo[4 * s + 0] = detection_ran;
    g.winfo[4 * s + 1] = 0;
    g.winfo[4 * s + 2] = 0;
    g.winfo[4 * s + 3] = 0;             // candidates waiting for cornerSubPix: k_group_cands
  }
}

// Grider_GRID.h:133-149 on the candidate table of the valid cells (k_fast_g + k_fast_select_g have just filled it): bounds and
// mask0_updated (caller mask, or inside the (2d+1)^2 square of a kept point whose square lies inside the image,
// TrackKLT.cpp:457-461), in (cell, rank) order.
__global__ void __launch_bounds__(kGT)
    k_group_cands(const __grid_constant__ GroupDev g, const TrackJob *__restrict__ jobs) {
  __shared__ BlockScan bs;
  const TrackJob &job = jobs[blockIdx.x];
  const int s = job.stream, tid = threadIdx.x;
  if (g.winfo[4 * s + 0] == 0) return;   // no detection this frame
  const int cols = g.W, rows = g.H, d = g.min_px_dist;
  const bool first = g.wmode[s] == 1;
  const int islot = first ? job.cur_slot : job.prev_slot;
  const SlotRec &sl = g.slots[islot];
  const uint8_t *__restrict__ mask = (g.slot_flags[islot] & 1) ? sl.mask : nullptr;
  const float2 *__restrict__ wpts = g.wpts + (size_t)s * g.pts_cap;
  const int *__restrict__ valid = g.valid + (size_t)s * kValidStride;
  const int nk = g.wn[s];
  const int nv = valid[0], nfg = g.nfg;
  float2 *__restrict__ ext = g.ext_in + (size_t)s * g.cand_cap;
  int next = 0;
  const int total_q = nv * nfg;
  // one WARP per candidate for the occupancy test (its lanes share the kept points), then the ordered compaction
  constexpr int kChunk = 2048;
  __shared__ uint8_t s_pass[kChunk];
  const int warp = tid >> 5, lane = tid & 31;
  for (int base = 0; base < total_q; base += kChunk) {
    const int nq = min(kChunk, total_q - base);
    for (int ql = warp; ql < nq; ql += kGT / 32) {
      const int q = base + ql;
      const int v = q / nfg, k = q - v * nfg, c = valid[4 + v];
      bool pass = false;
      if (c >= 0 && k < min(sl.cand_cnt[c], nfg)) {
        const float2 p = sl.cand[c * nfg + k];
        const int ix = (int)p.x, iy = (int)p.y;
        if (!(ix < 0 || ix > cols || iy < 0 || iy > rows) && iy < rows && ix < cols) {
          bool occ = mask != nullptr && mask[(size_t)iy * cols + ix] > 127;
          if (!occ) {
            for (int j = lane; j < nk; j += 32) {
              const float2 w = wpts[j];
              const int x = (int)w.x, y = (int)w.y;
              occ = occ || (x - d >= 0 && x + d < cols && y - d >= 0 && y + d < rows && abs(ix - x) <= d && abs(iy - y) <= d);
            }
            occ = __any_sync(0xffffffffu, occ);
          }
          pass = !occ;
        }
      }
      if (lane == 0) s_pass[ql] = pass ? 1 : 0;
    }
    __syncthreads();
    for (int b0 = 0; b0 < nq; b0 += kGT) {
      const int ql = b0 + tid;
      const bool pass = ql < nq && s_pass[ql];
      const int e = block_excl(pass ? 1 : 0, bs);
      if (pass) {
        const int q = base + ql;
        const int v = q / nfg, k = q - v * nfg;
        ext[next + e] = sl.cand[valid[4 + v] * nfg + k];   // refined by k_group_subpix before the distance test (Grider_GRID.h:163-179)
      }
      next += bs.total;
    }
    __syncthreads();
  }
  if (tid == 0) g.winfo[4 * s + 3] = next;
}

// Second half of the top-off detection, after cornerSubPix of the surviving candidates (Grider_GRID.h:163-179).
__global__ void __launch_bounds__(kGT)
    k_group_accept(const __grid_constant__ GroupDev g, const TrackJob *__restrict__ jobs) {
  __shared__ BlockScan bs;
  const TrackJob &job = jobs[blockIdx.x];
  const int s = job.stream, tid = threadIdx.x;
  const int d = g.min_px_dist;
  const int close_w = g.close_w, close_h = g.close_h, close_n = close_w * close_h;
  const size_t o = (size_t)s * g.pts_cap;
  float2 *__restrict__ wpts = g.wpts + o;
  uint64_t *__restrict__ wids = g.wids + o;
  int *__restrict__ close = g.close + (size_t)s * close_n;
  const float2 *__restrict__ ext = g.ext_pt + (size_t)s * g.cand_cap;
  const int nk = g.wn[s], next = g.winfo[4 * s + 3];
  int n_added = 0, overflow = 0, n_out = nk;
  if (next > 0) {
    // ---- minimum-distance rejection among the new points, in order (:497-512), then ids (:519-527)
    for (int e = tid; e < next; e += kGT) {
      const float2 kp = ext[e];
      const int xg = (int)(kp.x / (float)d), yg = (int)(kp.y / (float)d);
      if (xg < 0 || xg >= close_w || yg < 0 || yg >= close_h) continue;
      atomicMin(&close[yg * close_w + xg], kExtBase + e);
    }
    __syncthreads();
    const uint64_t currid = g.currid[s];
    for (int base = 0; base < next; base += kGT) {
      const int e0 = base + tid;
      bool acc = false;
      float2 kp = make_float2(0.f, 0.f);
      if (e0 < next) {
        kp = ext[e0];
        const int xg = (int)(kp.x / (float)d), yg = (int)(kp.y / (float)d);
        acc = !(xg < 0 || xg >= close_w || yg < 0 || yg >= close_h) && close[yg * close_w + xg] == kExtBase + e0;
      }
      const int r = block_excl(acc ? 1 : 0, bs);
      if (acc) {
        const int dst = nk + n_added + r;
        if (dst < g.pts_cap) {
          wpts[dst] = kp;
          wids[dst] = currid + 1 + (uint64_t)(n_added + r);
        }
      }
      n_added += bs.total;
    }
    if (nk + n_added > g.pts_cap) {
      overflow = 1;
      n_added = g.pts_cap - nk;
    }
    n_out = nk + n_added;
    if (tid == 0) g.currid[s] = currid + (uint64_t)n_added;
  }
  if (tid == 0) {
    g.wn[s] = n_out;
    g.winfo[4 * s + 1] = n_added;
    g.winfo[4 * s + 2] = overflow;
  }
}

void launch_group_detect(const GroupDev &g, const TrackJob *jobs, int n_jobs, cudaStream_t s) {
  if (n_jobs <= 0) return;
  PLVIWO_CARVEOUT(k_group_detect);
  k_group_detect<<<n_jobs, kGT, 0, s>>>(g, jobs);
}
void launch_group_cands(const GroupDev &g, const TrackJob *jobs, int n_jobs, cudaStream_t s) {
  if (n_jobs <= 0) return;
  PLVIWO_CARVEOUT(k_group_cands);
  k_group_cands<<<n_jobs, kGT, 0, s>>>(g, jobs);
}
void launch_group_accept(const GroupDev &g, const TrackJob *jobs, int n_jobs, cudaStream_t s) {
  if (n_jobs <= 0) return;
  PLVIWO_CARVEOUT(k_group_accept);
  k_group_accept<<<n_jobs, kGT, 0, s>>>(g, jobs);
}

// ============================================================================================= RANSAC gate + rows
namespace rc = ransac_core;
constexpr int kRounds = kGT / 32;   // samples solved side by side (one per warp)

// LMedSPointSetRegistrator::run (8 <= count < 15), one thread (ransac.cpp has the commentary)
__device__ int lmeds_gate(const float2 *m1, const float2 *m2, int count, uint8_t *mask) {
  const int model_points = 7, max_iters = 1000;
  float ms1[14], ms2[14], err[16], sorted[16];
  double F[27], bestF[9];
  rc::CvRng rng((uint64_t)-1);
  int niters = rc::ransac_update_num_iters(0.999, 0.45, model_points, max_iters);
  niters = max(niters, 3);
  double min_median = DBL_MAX;
  bool found = false;
  auto errors = [&](const double *Fm) {
    for (int i = 0; i < count; i++) err[i] = rc::epipolar_error(Fm, m1[i].x, m1[i].y, m2[i].x, m2[i].y);
  };
  for (int iter = 0; iter < niters; iter++) {
    if (!rc::get_subset(reinterpret_cast<const float *>(m1), reinterpret_cast<const float *>(m2), count, ms1, ms2, rng, 1000)) {
      if (iter == 0) return 0;
      break;
    }
    const int nmodels = rc::run_7point(ms1, ms2, F);
    if (nmodels <= 0) continue;
    for (int i = 0; i < nmodels; i++) {
      errors(F + 9 * i);
      for (int k = 0; k < count; k++) sorted[k] = err[k];
      for (int a = 1; a < count; a++) {   // insertion sort: only the (count / 2)-th smallest is used
        const float v = sorted[a];
        int b = a - 1;
        for (; b >= 0 && sorted[b] > v; b--) sorted[b + 1] = sorted[b];
        sorted[b + 1] = v;
      }
      const double median = sorted[count / 2];
      if (median < min_median) {
        min_median = median;
        for (int k = 0; k < 9; k++) bestF[k] = F[9 * i + k];
        found = true;
      }
    }
  }
  if (!found || min_median >= DBL_MAX) return 0;
  double sigma = 2.5 * 1.4826 * (1 + 5. / (count - model_points)) * sqrt(min_median);
  sigma = fmax(sigma, 0.001);
  errors(bestF);
  const float t = (float)(sigma * sigma);
  int good = 0;
  for (int k = 0; k < count; k++) {
    const uint8_t f = err[k] <= t;
    mask[k] = f;
    good += f;
  }
  return good;
}

__global__ void __launch_bounds__(kGT)
    k_group_gate(const __grid_constant__ GroupDev g, const TrackJob *__restrict__ jobs) {
  extern __shared__ uint8_t gate_smem[];   // two inlier masks of pts_cap bytes
  __shared__ BlockScan bs;
  __shared__ float s_ms1[kRounds][14], s_ms2[kRounds][14];
  __shared__ double s_F[kRounds][27];
  __shared__ int s_nm[kRounds], s_ok[kRounds], s_good[kRounds][3];
  __shared__ double s_bestF[9];
  __shared__ int s_niters, s_maxgood, s_R, s_stop, s_best;
  const TrackJob &job = jobs[blockIdx.x];
  const int s = job.stream, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n = g.wn[s], mode = g.wmode[s];
  const size_t o = (size_t)s * g.pts_cap;
  float2 *__restrict__ pts = g.pts + (size_t)job.out * g.pts_cap;      // this frame's state record
  uint64_t *__restrict__ ids = g.ids + (size_t)job.out * g.pts_cap;
  const float2 *__restrict__ wpts = g.wpts + o;
  const uint64_t *__restrict__ wids = g.wids + o;
  uint8_t *const rec = g.out + (size_t)job.out * g.out_stride;
  GroupOutHeader *hdr = reinterpret_cast<GroupOutHeader *>(rec);
  FePointRow *rows = reinterpret_cast<FePointRow *>(rec + g.off_rows);
  uint64_t *obs_ids = reinterpret_cast<uint64_t *>(rec + g.off_obs_ids);
  float2 *obs_uv = reinterpret_cast<float2 *>(rec + g.off_obs_uv);
  if (tid == 0) {
    GroupOutHeader h;
    memset(&h, 0, sizeof(h));
    h.info.timestamp = job.timestamp;
    h.info.detection_ran = g.winfo[4 * s + 0];
    h.info.n_detected = g.winfo[4 * s + 1];
    if (g.winfo[4 * s + 2]) {
      h.status = FE_INTERNAL;
      h.overflow_what = 1;
    }
    *hdr = h;
  }
  __syncthreads();
  if (mode == 1) {   // detection-only frame (:110-123): the new points ARE pts_last; no rows
    for (int i = tid; i < n; i += kGT) {
      pts[i] = wpts[i];
      ids[i] = wids[i];
      obs_ids[i] = wids[i];
      obs_uv[i] = wpts[i];
    }
    if (tid == 0) {
      g.n_pts[job.out] = n;
      hdr->info.first_frame = 1;
      hdr->info.n_last_obs = n;
      hdr->n_obs = n;
    }
    return;
  }
  if (n < 10) {   // n == 0: mask_out stays empty => reset (:143-152); 1..9: every point fails (:848-852)
    if (tid == 0) {
      g.n_pts[job.out] = 0;
      if (n == 0) hdr->info.reset = 1;
    }
    return;
  }
  const float2 *__restrict__ m1 = g.lk_p0n + o;
  const float2 *__restrict__ m2 = g.lk_p1n + o;
  const float2 *__restrict__ p1 = g.lk_pts1 + o;
  const uint8_t *__restrict__ st = g.lk_status + o;
  uint8_t *mcur = gate_smem, *mbest = gate_smem + g.pts_cap;
  for (int i = tid; i < n; i += kGT) mbest[i] = 0;
  // ---- cv::findFundamentalMat(p0n, p1n, FM_RANSAC, 2 / max focal, 0.999) (:869-873), ransac.cpp restated for one CTA:
  // the samples are drawn by one thread (the RNG sequence is the contract), kRounds of them are solved side by side, one
  // per warp, and the models are then scored in order by all threads with the sequential accept / iteration-count rule.
  const double threshold = 2.0 / fmax(job.K[0], job.K[1]);
  int n_in = 0, mask_valid = 1;
  {
    bool moved = false;
    for (int i = tid; i < n; i += kGT) moved = moved || m1[i].x != m2[i].x || m1[i].y != m2[i].y;
    const bool all_static = __syncthreads_or(moved ? 1 : 0) == 0;   // a repeated frame: every point is an inlier
    if (all_static) {
      for (int i = tid; i < n; i += kGT) mbest[i] = 1;
      n_in = n;
    } else if (n < 15) {
      if (tid == 0) s_best = lmeds_gate(m1, m2, n, mbest);
      __syncthreads();
      n_in = s_best;
    } else {
      const float t = (float)(threshold * threshold);
      rc::CvRng rng((uint64_t)-1);   // thread 0's copy is the one that advances
      if (tid == 0) {
        s_niters = 1000;
        s_maxgood = 0;
        s_stop = 0;
      }
      __syncthreads();
      int iter = 0;
      while (true) {
        if (tid == 0) {
          int R = 0;
          while (R < kRounds && iter + R < s_niters) {
            const bool ok = rc::get_subset(reinterpret_cast<const float *>(m1), reinterpret_cast<const float *>(m2), n, s_ms1[R],
                                           s_ms2[R], rng, 10000);
            s_ok[R] = ok ? 1 : 0;
            R++;
            if (!ok) break;   // the library leaves the loop here
          }
          s_R = R;
        }
        __syncthreads();
        const int R = s_R;
        if (R == 0) break;
        // warp r: the 7-point models of sample r (one lane), then their inlier counts over all points (all lanes)
        if (warp < R) {
          int nm = 0;
          if (lane == 0 && s_ok[warp]) nm = rc::run_7point(s_ms1[warp], s_ms2[warp], s_F[warp]);
          nm = __shfl_sync(0xffffffffu, nm, 0);
          if (lane == 0) s_nm[warp] = nm;
          __syncwarp();
          for (int i = 0; i < nm && i < 3; i++) {
            const double *F = s_F[warp] + 9 * i;
            int good = 0;
            for (int k = lane; k < n; k += 32) good += rc::epipolar_error(F, m1[k].x, m1[k].y, m2[k].x, m2[k].y) <= t ? 1 : 0;
            good = __reduce_add_sync(0xffffffffu, good);
            if (lane == 0) s_good[warp][i] = good;
          }
        }
        __syncthreads();
        // the sequential accept rule and adaptive iteration count, in sample order (RANSACPointSetRegistrator::run)
        if (tid == 0) {
          for (int r = 0; r < R; r++) {
            if (iter + r >= s_niters || !s_ok[r]) {   // the count dropped below the samples solved ahead / no sample
              s_stop = 1;
              break;
            }
            for (int i = 0; i < s_nm[r] && i < 3; i++) {
              const int good = s_good[r][i];
              if (good > max(s_maxgood, 6)) {
                s_maxgood = good;
                for (int q = 0; q < 9; q++) s_bestF[q] = s_F[r][9 * i + q];
                s_niters = rc::ransac_update_num_iters(0.999, (double)(n - good) / n, 7, s_niters);
              }
            }
          }
        }
        __syncthreads();
        iter += R;
        if (s_stop || iter >= s_niters) break;
      }
      n_in = s_maxgood;
      if (n_in > 0)   // the mask of the accepted model
        for (int k = tid; k < n; k += kGT) mbest[k] = rc::epipolar_error(s_bestF, m1[k].x, m1[k].y, m2[k].x, m2[k].y) <= t ? 1 : 0;
    }
  }
  __syncthreads();
  // ---- mask_out = mask_klt && mask_rsc (:876-879), then feed_monocular's filter (:159-173) and the rows (:176-179)
  const uint8_t *__restrict__ cmask = (g.slot_flags[job.cur_slot] & 1) ? g.slots[job.cur_slot].mask : nullptr;
  int n_good = 0, n_klt = 0;
  for (int base = 0; base < n; base += kGT) {
    const int i = base + tid;
    bool keep = false;
    float2 p = make_float2(0.f, 0.f);
    if (i < n) {
      p = p1[i];
      n_klt += st[i] ? 1 : 0;
      const bool ll = st[i] && mask_valid && mbest[i];
      const bool oob = p.x < 0 || p.y < 0 || (int)p.x >= g.W || (int)p.y >= g.H;
      keep = !oob && !(cmask != nullptr && cmask[(size_t)(int)p.y * g.W + (int)p.x] > 127) && ll;
    }
    const int e = block_excl(keep ? 1 : 0, bs);
    if (keep) {
      const int dst = n_good + e;
      const uint64_t id = wids[i];
      pts[dst] = p;
      ids[dst] = id;
      FePointRow r;
      r.id = id;
      r.u = p.x;
      r.v = p.y;
      r.un = m2[i].x;   // undistort_cv(pt) of the tracked point is the p1n the LK epilogue produced
      r.vn = m2[i].y;
      rows[dst] = r;
      obs_ids[dst] = id;
      obs_uv[dst] = p;
    }
    n_good += bs.total;
  }
  n_klt = block_sum(n_klt, bs);
  if (tid == 0) {
    g.n_pts[job.out] = n_good;
    hdr->info.n_lk_in = n;
    hdr->info.n_klt_ok = n_klt;
    hdr->info.n_ransac_ok = n_in;
    hdr->info.n_point_rows = n_good;
    hdr->info.n_last_obs = n_good;
    hdr->n_obs = n_good;
  }
}

void launch_group_gate(const GroupDev &g, const TrackJob *jobs, int n_jobs, cudaStream_t s) {
  if (n_jobs <= 0) return;
  PLVIWO_CARVEOUT(k_group_gate);
  k_group_gate<<<n_jobs, kGT, 2 * (size_t)g.pts_cap, s>>>(g, jobs);
}

// ==================================================================================================== lines
// TrackLSD::PointLineDistance (TrackLSD.cpp:794-814): float arithmetic, the last branch mixes in double (std::pow)
__device__ __forceinline__ float point_line_distance(const float4 &line, float x0, float y0) {
  const float x1 = line.x, y1 = line.y, x2 = line.z, y2 = line.w;
  const float cross = (x2 - x1) * (x0 - x1) + (y2 - y1) * (y0 - y1);
  if (cross <= 0) return sqrtf((x0 - x1) * (x0 - x1) + (y0 - y1) * (y0 - y1));
  const float d = (x2 - x1) * (x2 - x1) + (y2 - y1) * (y2 - y1);
  if (cross > d) return sqrtf((x0 - x2) * (x0 - x2) + (y0 - y2) * (y0 - y2));
  const double dy = (double)(y2 - y1), dx = (double)(x1 - x2);
  return (float)fabs((double)fabsf((y2 - y1) * x0 + (x1 - x2) * y0 + ((x2 * y1) - (x1 * y2))) / sqrt(dy * dy + dx * dx));
}
__device__ __forceinline__ bool line_similar(const float4 &line2, const float4 &line1) {   // :816-830
  const float mx = (line1.x + line1.z) / 2, my = (line1.y + line1.w) / 2;
  return point_line_distance(line2, mx, my) <= 6;
}
__device__ bool line_class(const float4 &line, double vx, double vy) {   // :335-366, atan(dy) / dx as written there
  const double s[3] = {line.x, line.y, 1}, e[3] = {line.z, line.w, 1};
  const double mid[3] = {(s[0] + e[0]) / 2, (s[1] + e[1]) / 2, (s[2] + e[2]) / 2};
  const double v3[3] = {vx, vy, 1};
  const double ln[3] = {mid[1] * v3[2] - mid[2] * v3[1], mid[2] * v3[0] - mid[0] * v3[2], mid[0] * v3[1] - mid[1] * v3[0]};
  double dis_error = (fabs(ln[0] * s[0] + ln[1] * s[1] + ln[2] * s[2]) + fabs(ln[0] * e[0] + ln[1] * e[1] + ln[2] * e[2])) /
                     (2 * sqrt(ln[0] * ln[0] + ln[1] * ln[1]));
  dis_error = fabs(dis_error);
  const double angle1 = atanf(line.y - line.w) / (line.x - line.z);   // float arithmetic
  const double angle2 = atan(mid[1] - vy) / (mid[0] - vx);
  const double angle_error = fabs(angle1 - angle2);
  return dis_error <= 5.0 && angle_error <= 0.35;
}
__device__ int line_classification(const float4 &line, const double vp[6]) {   // :318-333
  if (line_class(line, vp[4], vp[5])) return 3;
  if (line_class(line, vp[2], vp[3])) return 2;
  if (line_class(line, vp[0], vp[1])) return 1;
  return 0;
}
// cv::undistortPoints on one point (SURVEY.md Appendix A6): 5 fixed-point iterations in double
__device__ void undistort_pt(const double K[4], const double D[4], float u, float v, float &un, float &vn) {
  const double x0 = ((double)u - K[2]) / K[0], y0 = ((double)v - K[3]) / K[1];
  double x = x0, y = y0;
#pragma unroll 1
  for (int j = 0; j < 5; j++) {
    const double r2 = x * x + y * y;
    const double icdist = 1.0 / (1.0 + (D[1] * r2 + D[0]) * r2);
    const double dx = 2 * D[2] * x * y + D[3] * (r2 + 2 * x * x);
    const double dy = D[2] * (r2 + 2 * y * y) + 2 * D[3] * x * y;
    x = (x0 - dx) * icdist;
    y = (y0 - dy) * icdist;
  }
  un = (float)x;
  vn = (float)y;
}

// AssignPointToLines' test of one (line, point) pair (:770-781): inside the mis-indexed bounding box and not farther than
// 5 px from the SEGMENT
__device__ __forceinline__ bool on_line(const float4 &l, float min_lx, float max_lx, float min_ly, float max_ly, float2 p, float &dist) {
  if (p.x < min_lx || p.x > max_lx || p.y < min_ly || p.y > max_ly) return false;
  dist = point_line_distance(l, p.x, p.y);
  return !(dist > 5);
}

__global__ void __launch_bounds__(kGT)
    k_group_lines(const __grid_constant__ GroupDev g, const TrackJob *__restrict__ jobs) {
  __shared__ BlockScan bs;
  __shared__ int s_over;
  const TrackJob &job = jobs[blockIdx.x];
  if (!(job.flags & 1)) return;   // no vanishing points given: the line tracker is not fed (UpdaterCamera.cpp:106-110)
  const int s = job.stream, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const FldBuffers &fb = g.slots[job.cur_slot].fld;
  uint8_t *const rec = g.out + (size_t)job.out * g.out_stride;
  GroupOutHeader *hdr = reinterpret_cast<GroupOutHeader *>(rec);
  FeLineRow *lrows = reinterpret_cast<FeLineRow *>(rec + g.off_lrows);
  FeLinePoint *lpts = reinterpret_cast<FeLinePoint *>(rec + g.off_lpts);
  const int LC = g.lines_cap, PC = g.pol_cap;
  const int lastb = g.line_buf[s], newb = lastb ^ 1;
  const size_t bl = (size_t)(2 * s + lastb), bn = (size_t)(2 * s + newb);
  const float4 *__restrict__ lines_last = g.lines + bl * LC;
  const uint64_t *__restrict__ lids_last = g.line_ids + bl * LC;
  const int *__restrict__ poff_last = g.pol_off + bl * (LC + 1);
  const int *__restrict__ ppid_last = g.pol_pid + bl * PC;
  const int n_last = g.n_lines[2 * s + lastb];
  float4 *__restrict__ lines_new = g.lines + bn * LC;
  uint64_t *__restrict__ lids_new = g.line_ids + bn * LC;
  int *__restrict__ poff_new = g.pol_off + bn * (LC + 1);
  int *__restrict__ ppid_new = g.pol_pid + bn * PC;
  float *__restrict__ pdist_new = g.pol_dist + bn * PC;
  float4 *__restrict__ lnew = g.lnew + (size_t)s * LC;
  int *__restrict__ lcnt = g.lcnt + (size_t)s * (LC + 1);
  int *__restrict__ loff = g.loff + (size_t)s * (LC + 1);
  float2 *__restrict__ lpos = g.lpos + (size_t)s * PC;
  int *__restrict__ lmatch = g.lmatch + (size_t)s * LC;
  const float2 *__restrict__ pts = g.pts + (size_t)job.out * g.pts_cap;      // the point tracker's pts_last / ids_last after THIS frame (:127-129)
  const uint64_t *__restrict__ pids = g.ids + (size_t)job.out * g.pts_cap;
  const int npt = g.n_pts[job.out];
  if (tid == 0) s_over = 0;

  // ---- perform_detection_monocular (:218-236): x2, FilterShortLines(40), a fresh id for EVERY detected line
  const int nseg = min(fb.counters[4], fb.out_cap);
  const float thr_sq = g.line_min_length * g.line_min_length;
  int L = 0;
  for (int base = 0; base < nseg; base += kGT) {
    const int i = base + tid;
    bool keep = false;
    float4 l = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < nseg) {
      l = fb.out[i];
      l.x *= 2; l.y *= 2; l.z *= 2; l.w *= 2;
      const float lsq = (l.z - l.x) * (l.z - l.x) + (l.w - l.y) * (l.w - l.y);
      keep = lsq > thr_sq;
    }
    const int e = block_excl(keep ? 1 : 0, bs);
    if (keep && L + e < LC) lnew[L + e] = l;
    L += bs.total;
  }
  if (L > LC) {
    if (tid == 0) s_over = 2;
    L = LC;
  }
  const uint64_t lcurr = g.line_currid[s];   // line i gets id lcurr + 1 + i
  __syncthreads();

  // ---- AssignPointToLines, pass 1: points per line (one warp per line)
  for (int i = warp; i < L; i += kGT / 32) {
    const float4 l = lnew[i];
    float min_lx = l.x, max_lx = l.y, min_ly = l.z, max_ly = l.w;   // index mix-up reproduced (:754-757)
    if (l.x > l.y) { min_lx = l.y; max_lx = l.x; }
    if (l.z > l.w) { min_ly = l.w; max_ly = l.z; }
    int c = 0;
    for (int j0 = 0; j0 < npt; j0 += 32) {
      const int j = j0 + lane;
      float dist;
      const bool hit = j < npt && on_line(l, min_lx, max_lx, min_ly, max_ly, pts[j], dist);
      c += __popc(__ballot_sync(0xffffffffu, hit));
    }
    if (lane == 0) lcnt[i] = c;
  }
  __syncthreads();
  // ---- lines that keep at least one point survive, in order; entry offsets
  int nk = 0, ne = 0;
  for (int base = 0; base < L; base += kGT) {
    const int i = base + tid;
    const int c = i < L ? lcnt[i] : 0;
    const int ki = block_excl(c > 0 ? 1 : 0, bs);
    const int tk = bs.total;
    const int eo = block_excl(c, bs);
    const int te = bs.total;
    if (c > 0) {
      const int dst = nk + ki;
      lines_new[dst] = lnew[i];
      lids_new[dst] = lcurr + 1 + (uint64_t)i;   // filt_ids; replaced by the inherited id below
      poff_new[dst] = ne + eo;
      lmatch[dst] = -1;
    }
    nk += tk;
    ne += te;
  }
  __syncthreads();
  if (tid == 0) poff_new[nk] = ne;
  if (ne > PC) {   // more point / line pairs than the buffers hold: the frame is flagged, the association is cut short
    if (tid == 0) s_over = 3;
  }
  __syncthreads();
  // ---- pass 2: the entries of every surviving line, points in detection order; the map<int, double> is keyed by the
  // point id cast to int and iterates in ascending key order
  for (int i = warp; i < nk; i += kGT / 32) {
    const float4 l = lines_new[i];
    float min_lx = l.x, max_lx = l.y, min_ly = l.z, max_ly = l.w;
    if (l.x > l.y) { min_lx = l.y; max_lx = l.x; }
    if (l.z > l.w) { min_ly = l.w; max_ly = l.z; }
    const int off = poff_new[i];
    int c = 0;
    for (int j0 = 0; j0 < npt; j0 += 32) {
      const int j = j0 + lane;
      float dist = 0.f;
      const float2 p = j < npt ? pts[j] : make_float2(0.f, 0.f);
      const bool hit = j < npt && on_line(l, min_lx, max_lx, min_ly, max_ly, p, dist);
      const unsigned b = __ballot_sync(0xffffffffu, hit);
      if (hit) {
        const int dst = off + c + __popc(b & ((1u << lane) - 1u));
        if (dst < PC) {
          ppid_new[dst] = (int)pids[j];
          pdist_new[dst] = dist;
          lpos[dst] = p;
        }
      }
      c += __popc(b);
    }
    __syncwarp();
    if (lane == 0) {   // ids are handed out in increasing order and points keep their order, so this is a no-op unless ids
      const int end = min(off + c, PC);   // were renamed (change_feat_id); a duplicate key keeps the LAST value, as the map
      for (int a = off + 1; a < end; a++) {
        const int kp = ppid_new[a];
        const float kd = pdist_new[a];
        int b2 = a - 1;
        for (; b2 >= off && ppid_new[b2] > kp; b2--) {
          ppid_new[b2 + 1] = ppid_new[b2];
          pdist_new[b2 + 1] = pdist_new[b2];
        }
        ppid_new[b2 + 1] = kp;
        pdist_new[b2 + 1] = kd;
      }
    }
  }
  __syncthreads();
  const bool over_pairs = ne > PC;
  if (tid == 0) {
    g.line_currid[s] = lcurr + (uint64_t)L;
    g.n_lnew[s] = L;   // lines_det_last_ of a handle (fe_context.cu lsd_feed): cfg.line_samples samples the next frame along these
    hdr->info.n_lines_detected = L;
    if (s_over) {
      hdr->status = FE_INTERNAL;
      hdr->overflow_what = s_over;
    }
  }
  if (n_last == 0 || over_pairs) {   // first frame / lost (:95-115): the new lines become lines_last, no database rows
    if (tid == 0) {
      g.n_lines[2 * s + newb] = over_pairs ? 0 : nk;
      g.line_buf[s] = newb;
    }
    return;
  }
  // ---- LineMatch (:368-407): new line i inherits the id of the LAST line j of the previous frame that shares two point
  // ids with it, or one and LineSimilar.  One warp per new line, lanes over the previous frame's lines.
  for (int i = warp; i < nk; i += kGT / 32) {
    const int a0 = poff_new[i], a1 = poff_new[i + 1];
    const float4 li = lines_new[i];
    int best = -1;
    for (int j = lane; j < n_last; j += 32) {
      int b0 = poff_last[j];
      const int b1 = poff_last[j + 1];
      int shared = 0;
      for (int a = a0; a < a1 && b0 < b1; a++) {   // both lists ascend
        const int key = ppid_new[a];
        while (b0 < b1 && ppid_last[b0] < key) b0++;
        if (b0 < b1 && ppid_last[b0] == key) shared++;
      }
      if (shared >= 2 || (shared >= 1 && line_similar(li, lines_last[j]))) best = j;   // j ascends per lane
    }
    best = __reduce_max_sync(0xffffffffu, best);
    if (lane == 0) lmatch[i] = best;
  }
  __syncthreads();
  // ---- ids (:146-158, through int as in the reference), rows (:163-167) and the new lines_last (:175-182)
  int n_matches = 0;
  for (int i = tid; i < nk; i += kGT) {
    const int m = lmatch[i];
    const int id32 = m >= 0 ? (int)lids_last[m] : (int)lids_new[i];
    const uint64_t id = (uint64_t)(long long)id32;
    const float4 l = lines_new[i];
    FeLineRow r;
    memset(&r, 0, sizeof(r));
    r.id = id;
    r.line[0] = l.x; r.line[1] = l.y; r.line[2] = l.z; r.line[3] = l.w;
    undistort_pt(job.K, job.D, l.x, l.y, r.line_n[0], r.line_n[1]);
    undistort_pt(job.K, job.D, l.z, l.w, r.line_n[2], r.line_n[3]);
    r.D = line_classification(l, job.vp);
    r.n_pts = poff_new[i + 1] - poff_new[i];
    r.pt_offset = poff_new[i];
    r.matched = m >= 0 ? 1 : 0;
    lrows[i] = r;
    n_matches += m >= 0 ? 1 : 0;
  }
  for (int e = tid; e < ne; e += kGT) {
    FeLinePoint lp;
    lp.pid = ppid_new[e];
    lp.dist = pdist_new[e];
    lp.u = lpos[e].x;
    lp.v = lpos[e].y;
    lpts[e] = lp;
  }
  n_matches = block_sum(n_matches, bs);
  for (int i = tid; i < nk; i += kGT) {   // after every row has read lids_new / lids_last
    const int m = lmatch[i];
    if (m >= 0) lids_new[i] = (uint64_t)(long long)(int)lids_last[m];
    else lids_new[i] = (uint64_t)(long long)(int)lids_new[i];
  }
  if (tid == 0) {
    g.n_lines[2 * s + newb] = nk;
    g.line_buf[s] = newb;
    hdr->info.n_line_rows = nk;
    hdr->info.n_line_matches = n_matches;
    hdr->n_line_points = ne;
  }
}

void launch_group_lines(const GroupDev &g, const TrackJob *jobs, int n_jobs, cudaStream_t s) {
  if (n_jobs <= 0 || !g.use_lines) return;
  PLVIWO_CARVEOUT(k_group_lines);
  k_group_lines<<<n_jobs, kGT, 0, s>>>(g, jobs);
}

}  // namespace plviwo
