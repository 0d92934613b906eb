// Grid-bucketed FAST-9/16 with 3x3 non-max suppression, per cell ROI (sm_100a).
//
// Replaces cv::FAST(img(roi), pts, threshold, true) as called per valid grid cell at Grider_GRID.h:121-125.
// Arithmetic per SURVEY.md Appendix A4: the ROI is treated as a whole image, so only 3 <= x < cols-3,
// 3 <= y < rows-3 are tested (a 3 px band along every cell edge is never a corner), score = max over the 16
// contiguous 9-arcs of min(d) / of -max(d) minus 1, strict 3x3 NMS against the 8 neighbours' scores, output in
// row-major order — the order matters because the unstable std::sort at Grider_GRID.h:128 permutes ties.
//
// One CTA handles one band of kFastBandRows rows of one cell: the pixels are staged in shared memory with a
// halo that is CLAMPED TO THE CELL (rows outside the cell simply do not exist), scores go to a second shared
// plane, and survivors are emitted with an ordered block-wide compaction.  Bands of a cell reserve their slice
// of the compact output with one atomic; the host (or the selection kernel) walks bands in order.
#include "fe_group_dev.h"
#include "fe_kernels.h"
#include "introsort.h"

namespace plviwo {

constexpr int kFastThreads = 256;
constexpr int kBH = kFastBandRows;

__device__ __forceinline__ bool has_arc9(unsigned m16) {
  // 9 contiguous set bits in a circular 16-bit mask
  unsigned m = m16 | (m16 << 16);
  unsigned r = m & (m >> 1);
  r &= r >> 2;
  r &= r >> 4;
  r &= m >> 8;
  return (r & 0xffffu) != 0;
}

// FAST-9/16 test and score of one pixel; get(dx, dy) returns the neighbour at that offset (compile-time offsets after
// unrolling: shared-memory bytes in the generic path, byte extracts from registers in the 4-pixel path).
// Necessary condition (exact, OpenCV's own early exit): 9 contiguous ring positions always contain position k or k + 8 for
// every k, so a bright (dark) arc needs a brighter (darker) pixel in each opposite pair.  Two pairs — four pixels — reject
// most pixels of a natural image before the other twelve are looked at.
template <class Get>
__device__ __forceinline__ bool fast_quick_t(Get get, int threshold) {
  const int v = get(0, 0);
  const int hi = v + threshold, lo = v - threshold;
  const int p0 = get(0, 3), p8 = get(0, -3), p4 = get(3, 0), p12 = get(-3, 0);
  const bool br = (p0 > hi || p8 > hi) && (p4 > hi || p12 > hi);
  const bool dk = (p0 < lo || p8 < lo) && (p4 < lo || p12 < lo);
  return br || dk;
}

// the corner test proper: 9 contiguous ring pixels all brighter or all darker than the centre by more than the threshold
template <class Get>
__device__ __forceinline__ bool fast_arc_t(Get get, int threshold) {
  constexpr int dx[16] = {0, 1, 2, 3, 3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1};
  constexpr int dy[16] = {3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1, 0, 1, 2, 3};
  const int v = get(0, 0);
  unsigned bright = 0, dark = 0;
#pragma unroll
  for (int k = 0; k < 16; k++) {
    const int dk = v - get(dx[k], dy[k]);
    bright |= (dk > threshold ? 1u : 0u) << k;
    dark |= (dk < -threshold ? 1u : 0u) << k;
  }
  return has_arc9(bright) || has_arc9(dark);
}

// score of a pixel that passed fast_arc_t
template <class Get>
__device__ __forceinline__ int fast_full_t(Get get, int threshold) {
  // ring offsets in OpenCV's order (Appendix A4)
  constexpr int dx[16] = {0, 1, 2, 3, 3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1};
  constexpr int dy[16] = {3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1, 0, 1, 2, 3};
  const int v = get(0, 0);
  int d[16];
#pragma unroll
  for (int k = 0; k < 16; k++) d[k] = v - get(dx[k], dy[k]);
  (void)threshold;
  // a0 = max over arcs of min(d), b0 = min over arcs of max(d): sliding window of 9 over the circular ring
  int mn2[16], mx2[16];
#pragma unroll
  for (int k = 0; k < 16; k++) {
    mn2[k] = min(d[k], d[(k + 1) & 15]);
    mx2[k] = max(d[k], d[(k + 1) & 15]);
  }
  int mn4[16], mx4[16];
#pragma unroll
  for (int k = 0; k < 16; k++) {
    mn4[k] = min(mn2[k], mn2[(k + 2) & 15]);
    mx4[k] = max(mx2[k], mx2[(k + 2) & 15]);
  }
  int a0 = -256, b0 = 256;
#pragma unroll
  for (int k = 0; k < 16; k++) {
    int mn9 = min(min(mn4[k], mn4[(k + 4) & 15]), d[(k + 8) & 15]);
    int mx9 = max(max(mx4[k], mx4[(k + 4) & 15]), d[(k + 8) & 15]);
    a0 = max(a0, mn9);
    b0 = min(b0, mx9);
  }
  return max(a0, -b0) - 1;
}

__device__ __forceinline__ int fast_score(const uint8_t *__restrict__ px, int stride, int threshold) {
  auto get = [&](int dx, int dy) { return (int)px[dy * stride + dx]; };
  if (!fast_quick_t(get, threshold) || !fast_arc_t(get, threshold)) return 0;
  return fast_full_t(get, threshold);
}

constexpr int kFastPad = 16;   // bytes in front of the staged pixels: the 4-pixel path reads the word left of column 0

__device__ __forceinline__ void fast_body(const int cell_idx, const uint8_t *__restrict__ img, int pitch, const FastCell *__restrict__ cells, int max_bands,
                                          int threshold, unsigned *__restrict__ total, int *__restrict__ band_off,
                                          int *__restrict__ band_cnt, unsigned *__restrict__ kps, int kps_cap, int smem_w) {
  extern __shared__ __align__(16) uint8_t smem[];
  uint8_t *pix = smem + kFastPad;                              // (kBH + 8) rows x smem_w
  uint8_t *sc = smem + 2 * kFastPad + (kBH + 8) * smem_w;      // (kBH + 2) rows x smem_w
  __shared__ int warp_tot[kFastThreads / 32];
  __shared__ int s_base, s_nlist, s_nlist2;

  const FastCell cell = cells[cell_idx];
  const int band = blockIdx.x;
  const int slot = cell_idx * max_bands + band;
  const int y0 = band * kBH;
  const int cw = cell.w, ch = cell.h;
  if (y0 >= ch) {
    if (threadIdx.x == 0) { band_off[slot] = 0; band_cnt[slot] = 0; }
    return;
  }
  const int tid = threadIdx.x;
  // ---- stage pixel rows y0-4 .. y0+kBH+3 (cell-local), clipped to the cell
  const int py0 = y0 - 4;
  if (((cell.x | cw | pitch) & 3) == 0 && ((size_t)img & 3) == 0) {   // whole 32-bit words (coalesced 128-byte rows per warp)
    const int cww = cw >> 2;
    for (int i = tid; i < (kBH + 8) * cww; i += kFastThreads) {
      int r = i / cww, xw = i - r * cww;
      int y = py0 + r;
      unsigned v = 0;
      if (y >= 0 && y < ch) v = __ldg(reinterpret_cast<const unsigned *>(img + (size_t)(cell.y + y) * pitch + cell.x) + xw);
      *reinterpret_cast<unsigned *>(&pix[r * smem_w + 4 * xw]) = v;
    }
  } else {
    for (int i = tid; i < (kBH + 8) * cw; i += kFastThreads) {
      int r = i / cw, x = i - r * cw;
      int y = py0 + r;
      uint8_t v = 0;
      if (y >= 0 && y < ch) v = img[(size_t)(cell.y + y) * pitch + cell.x + x];
      pix[r * smem_w + x] = v;
    }
  }
  __syncthreads();
  // ---- scores for rows y0-1 .. y0+kBH
  const bool words = ((cell.x | cw | pitch) & 3) == 0 && ((size_t)img & 3) == 0 && cw <= 2048;
  if (words) {
    // Two phases, so that the expensive part only runs on lanes that have work (a warp pays for the arc test and the score
    // whenever ONE of its lanes needs them, and in a textured image there is such a pixel in nearly every 32):
    //  1. the four-pixel quick test on every pixel — four horizontally adjacent pixels per thread, the 7 x 10 pixels they look
    //     at are seven rows of three 32-bit words in registers (only the centre row and the rows 3 above / below are needed
    //     here) — survivors are appended to a list in shared memory (warp-aggregated);
    //  2. the full ring test and the score on the list, one survivor per lane.
    unsigned short *list = reinterpret_cast<unsigned short *>(smem + 3 * kFastPad + (2 * kBH + 10) * smem_w);
    const int cww = cw >> 2;
    const int items = (kBH + 2) * cww;
    for (int i = tid; i < (kBH + 2) * (smem_w >> 2); i += kFastThreads) reinterpret_cast<unsigned *>(sc)[i] = 0;
    if (tid == 0) s_nlist = s_nlist2 = 0;
    __syncthreads();
    const int lane = tid & 31;
    const unsigned t4 = (unsigned)min(max(threshold, 0), 255) * 0x01010101u;
    for (int i0 = 0; i0 < items; i0 += kFastThreads) {
      const int i = i0 + tid;
      const int r = i / cww, x0 = (i - r * cww) << 2;
      const int y = y0 - 1 + r;
      unsigned pass4 = 0;
      if (i < items && y >= 3 && y < ch - 3) {
        // the four pixels at once, one byte lane each: centre +- threshold with saturation (a pixel cannot exceed 255 or go
        // below 0, so the saturated bound decides the same), the four ring pixels at distance 3 as whole words (N, S) or
        // funnel shifts of the centre row (E, W), per-byte unsigned compares
        const unsigned *p0r = reinterpret_cast<const unsigned *>(&pix[(r + 0) * smem_w + x0]);
        const unsigned *p3r = reinterpret_cast<const unsigned *>(&pix[(r + 3) * smem_w + x0]);
        const unsigned *p6r = reinterpret_cast<const unsigned *>(&pix[(r + 6) * smem_w + x0]);
        const unsigned v4 = p3r[0], pS = p0r[0], pN = p6r[0];
        const unsigned pE = __funnelshift_r(v4, p3r[1], 24), pW = __funnelshift_r(p3r[-1], v4, 8);
        const unsigned hi4 = __vaddus4(v4, t4), lo4 = __vsubus4(v4, t4);
        const unsigned br = (__vcmpgtu4(pN, hi4) | __vcmpgtu4(pS, hi4)) & (__vcmpgtu4(pE, hi4) | __vcmpgtu4(pW, hi4));
        const unsigned dk = (__vcmpltu4(pN, lo4) | __vcmpltu4(pS, lo4)) & (__vcmpltu4(pE, lo4) | __vcmpltu4(pW, lo4));
        pass4 = br | dk;
        // columns 0..2 and cw-3..cw-1 of the cell are never tested
        if (x0 == 0) pass4 &= 0xff000000u;
        if (x0 + 4 >= cw - 3) {
#pragma unroll
          for (int j = 0; j < 4; j++)
            if (x0 + j >= cw - 3) pass4 &= ~(0xffu << (8 * j));
        }
      }
      const int mine = __popc(pass4 & 0x01010101u);
      int incl = mine;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += t;
      }
      const int tot = __shfl_sync(0xffffffffu, incl, 31);
      if (tot) {
        int base = 0;
        if (lane == 31) base = atomicAdd(&s_nlist, tot);
        base = __shfl_sync(0xffffffffu, base, 31) + incl - mine;
#pragma unroll
        for (int j = 0; j < 4; j++)
          if (pass4 & (0xffu << (8 * j))) list[base++] = (unsigned short)((r << 11) | (x0 + j));
      }
    }
    __syncthreads();
    //  2. the ring test on the survivors, one per lane; those with an arc go to a second list ...
    unsigned short *list2 = list + (kBH + 2) * smem_w;
    const int nlist = s_nlist;
    for (int k0 = 0; k0 < nlist; k0 += kFastThreads) {
      const int k = k0 + tid;
      bool pass = false;
      int e = 0;
      if (k < nlist) {
        e = list[k];
        const uint8_t *px = &pix[((e >> 11) + 3) * smem_w + (e & 2047)];
        pass = fast_arc_t([&](int dx, int dy) { return (int)px[dy * smem_w + dx]; }, threshold);
      }
      const unsigned bal = __ballot_sync(0xffffffffu, pass);
      if (bal) {
        int base = 0;
        if (lane == 0) base = atomicAdd(&s_nlist2, __popc(bal));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (pass) list2[base + __popc(bal & ((1u << lane) - 1u))] = (unsigned short)e;
      }
    }
    __syncthreads();
    //  3. ... and get their score, again one per lane
    const int nlist2 = s_nlist2;
    for (int k = tid; k < nlist2; k += kFastThreads) {
      const int e = list2[k], r = e >> 11, x = e & 2047;
      const uint8_t *px = &pix[(r + 3) * smem_w + x];
      sc[r * smem_w + x] = (uint8_t)fast_full_t([&](int dx, int dy) { return (int)px[dy * smem_w + dx]; }, threshold);
    }
    __syncthreads();
    //  4. strict 3 x 3 non-maximum suppression on the scored pixels (the second list holds exactly the non-zero scores), one
    //     per lane; the survivors' scores are parked in the pixel plane, which nobody reads any more
    const int brows = min(kBH, ch - y0);
    for (int i = tid; i < brows * (smem_w >> 2); i += kFastThreads) reinterpret_cast<unsigned *>(pix)[i] = 0;
    __syncthreads();
    for (int k = tid; k < nlist2; k += kFastThreads) {
      const int e = list2[k], r = e >> 11, x = e & 2047;
      if (r < 1 || r > brows) continue;
      const uint8_t *c = &sc[r * smem_w + x];
      const int sv = c[0];
      if (sv > c[-1] && sv > c[1] && sv > c[-smem_w - 1] && sv > c[-smem_w] && sv > c[-smem_w + 1] && sv > c[smem_w - 1] &&
          sv > c[smem_w] && sv > c[smem_w + 1])
        pix[(r - 1) * smem_w + x] = (uint8_t)sv;
    }
  } else {
    for (int i = tid; i < (kBH + 2) * cw; i += kFastThreads) {
      int r = i / cw, x = i - r * cw;
      int y = y0 - 1 + r;
      int s = 0;
      if (x >= 3 && x < cw - 3 && y >= 3 && y < ch - 3) s = fast_score(&pix[(r + 3) * smem_w + x], smem_w, threshold);
      sc[r * smem_w + x] = (uint8_t)s;
    }
  }
  __syncthreads();
  // ---- NMS + ordered compaction: thread t owns positions [t*R, (t+1)*R) of the band in row-major order
  const int rows = min(kBH, ch - y0);
  const int npos = rows * cw;
  // word path: runs of positions that start on a word boundary, scores read four at a time (most words are all zero), the
  // survivors' scores parked in the pixel plane (no longer needed) so that the second pass does not repeat the test
  const int R = words ? 4 * ((npos / 4 + kFastThreads - 1) / kFastThreads) : (npos + kFastThreads - 1) / kFastThreads;
  const int p0 = min(tid * R, npos), p1 = min(p0 + R, npos);
  int cnt = 0;
  if (words) {
    for (int p = p0; p < p1; p += 4) {
      const int r = p / cw, x = p - r * cw;
      const unsigned kept = *reinterpret_cast<const unsigned *>(&pix[r * smem_w + x]);
      cnt += __popc(__vcmpne4(kept, 0u) & 0x01010101u);
    }
  } else {
    for (int p = p0; p < p1; p++) {
      int r = p / cw, x = p - r * cw;
      int s = sc[(r + 1) * smem_w + x];
      if (s > 0 && x > 0 && x < cw - 1) {
        const uint8_t *c = &sc[(r + 1) * smem_w + x];
        bool keep = s > c[-1] && s > c[1] && s > c[-smem_w - 1] && s > c[-smem_w] && s > c[-smem_w + 1] &&
                    s > c[smem_w - 1] && s > c[smem_w] && s > c[smem_w + 1];
        cnt += keep ? 1 : 0;
      }
    }
  }
  // block exclusive scan of cnt
  int v = cnt;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, v, d);
    if ((tid & 31) >= d) v += t;
  }
  if ((tid & 31) == 31) warp_tot[tid >> 5] = v;
  __syncthreads();
  int base = 0;
  for (int k = 0; k < (tid >> 5); k++) base += warp_tot[k];
  int excl = base + v - cnt;
  if (tid == kFastThreads - 1) {
    int tot = base + v;
    int off = tot ? (int)atomicAdd(total, (unsigned)tot) : 0;
    s_base = off;
    band_off[slot] = off;
    band_cnt[slot] = tot;
  }
  __syncthreads();
  int w = s_base + excl;
  if (words) {
    for (int p = p0; p < p1; p += 4) {
      const int r = p / cw, x = p - r * cw;
      unsigned kept = *reinterpret_cast<const unsigned *>(&pix[r * smem_w + x]);
      while (kept) {
        const int k = (__ffs((int)kept) - 1) >> 3;
        const unsigned sv = (kept >> (8 * k)) & 0xffu;
        if (w < kps_cap) kps[w] = (unsigned)(x + k) | ((unsigned)(y0 + r) << 12) | (sv << 24);
        w++;
        kept &= ~(0xffu << (8 * k));
      }
    }
    return;
  }
  for (int p = p0; p < p1; p++) {
    int r = p / cw, x = p - r * cw;
    int s = sc[(r + 1) * smem_w + x];
    if (s > 0 && x > 0 && x < cw - 1) {
      const uint8_t *c = &sc[(r + 1) * smem_w + x];
      bool keep = s > c[-1] && s > c[1] && s > c[-smem_w - 1] && s > c[-smem_w] && s > c[-smem_w + 1] &&
                  s > c[smem_w - 1] && s > c[smem_w] && s > c[smem_w + 1];
      if (keep) {
        if (w < kps_cap) kps[w] = (unsigned)x | ((unsigned)(y0 + r) << 12) | ((unsigned)s << 24);
        w++;
      }
    }
  }
}

__global__ void __launch_bounds__(kFastThreads)
    k_fast(const uint8_t *__restrict__ img, int pitch, const FastCell *__restrict__ cells, int max_bands, int threshold,
           unsigned *__restrict__ total, int *__restrict__ band_off, int *__restrict__ band_cnt,
           unsigned *__restrict__ kps, int kps_cap, int smem_w) {
  fast_body(blockIdx.y, img, pitch, cells, max_bands, threshold, total, band_off, band_cnt, kps, kps_cap, smem_w);
}
// Stream group, FAST on demand: grid = (band, index into the stream's valid-cell list, job).  The reference runs cv::FAST on the
// valid cells only (Grider_GRID.h:108-125); which cells are valid is known once k_group_detect has counted the tracked points
// per cell, so the detector runs between the two halves of the detection, on the image the detection is about.
__global__ void __launch_bounds__(kFastThreads, 4)
    k_fast_g(const __grid_constant__ GroupDev gd, const TrackJob *__restrict__ jobs, FrontGeom g, int smem_w) {
  const TrackJob &job = jobs[blockIdx.z];
  const int s = job.stream;
  const int *__restrict__ valid = gd.valid + (size_t)s * kValidStride;
  if ((int)blockIdx.y >= valid[0]) return;
  const int c = valid[4 + blockIdx.y];
  if (c < 0) return;
  const SlotRec &sl = gd.slots[gd.wmode[s] == 1 ? job.cur_slot : job.prev_slot];
  fast_body(c, sl.lvl[0].p, sl.lvl[0].pitch, g.cells, g.max_bands, g.fast_threshold, sl.fast_total, sl.band_off, sl.band_cnt, sl.kps,
            g.kps_cap, smem_w);
}

// ------------------------------------------------------------------------------------- per-cell selection
// Grider_GRID.h:128-133: std::sort(cell corners, compare_response), keep the first num_features_grid.  One CTA per
// cell: the cell's corners (band slices of the compact list, i.e. row-major order — the order cv::FAST emits them in)
// are gathered into shared memory, ONE thread runs libstdc++'s introsort on them (introsort.h: the tie permutation is
// part of the contract) — pruned to the partitions that can reach the first num_features_grid positions, which is a
// selection, not a sort, with the identical result — and the survivors are written as full-image float coordinates to a fixed-stride table
// (cell c at c * nfg).  Cells with more corners than fit in shared memory sort in a global scratch slice.
constexpr int kSelThreads = 128;
constexpr int kSelSmemCap = 8192;
constexpr int kSelMaxBands = 256;   // 4095 rows / kFastBandRows

__device__ __forceinline__ void fast_select_body(const int c, const FastCell *__restrict__ cells, int max_bands,
                  unsigned *__restrict__ total /* [0] corners, [1] scratch cursor */,
                  const int *__restrict__ band_off, const int *__restrict__ band_cnt, const unsigned *__restrict__ kps,
                  int kps_cap, unsigned *__restrict__ scratch, int nfg, float2 *__restrict__ cand_sel,
                  int *__restrict__ cand_cnt) {
  __shared__ unsigned sv[kSelSmemCap];
  __shared__ int pref[kSelMaxBands + 1];
  __shared__ int s_base;
  const int tid = threadIdx.x;
  const int tot = min((int)total[0], kps_cap);
  if (tid == 0) {
    int acc = 0;
    for (int b = 0; b < max_bands; b++) {
      pref[b] = acc;
      const int off = band_off[c * max_bands + b];
      acc += max(0, min(band_cnt[c * max_bands + b], tot - off));
    }
    pref[max_bands] = acc;
    s_base = acc > kSelSmemCap ? (int)atomicAdd(total + 1, (unsigned)acc) : 0;
  }
  __syncthreads();
  const int n = pref[max_bands];
  unsigned *v = n > kSelSmemCap ? scratch + s_base : sv;
  for (int b = 0; b < max_bands; b++) {
    const int off = band_off[c * max_bands + b], cnt = pref[b + 1] - pref[b];
    for (int k = tid; k < cnt; k += kSelThreads) v[pref[b] + k] = kps[off + k];
  }
  __syncthreads();
  if (tid == 0) {
    isort::sort_prefix(v, n, nfg);   // exactly std::sort's first nfg elements (introsort.h), without sorting the rest
    cand_cnt[c] = min(n, nfg);
  }
  __syncthreads();
  const float x0 = (float)cells[c].x, y0 = (float)cells[c].y;
  for (int i = tid; i < min(n, nfg); i += kSelThreads) {
    const unsigned p = v[i];
    cand_sel[c * nfg + i] = make_float2((float)(p & 0xfffu) + x0, (float)((p >> 12) & 0xfffu) + y0);
  }
}

__global__ void __launch_bounds__(kSelThreads)
    k_fast_select(const FastCell *__restrict__ cells, int max_bands, unsigned *__restrict__ total,
                  const int *__restrict__ band_off, const int *__restrict__ band_cnt, const unsigned *__restrict__ kps,
                  int kps_cap, unsigned *__restrict__ scratch, int nfg, float2 *__restrict__ cand_sel,
                  int *__restrict__ cand_cnt) {
  fast_select_body(blockIdx.x, cells, max_bands, total, band_off, band_cnt, kps, kps_cap, scratch, nfg, cand_sel, cand_cnt);
}
// grid =(index into the stream's valid-cell list, job)
__global__ void __launch_bounds__(kSelThreads)
    k_fast_select_g(const __grid_constant__ GroupDev gd, const TrackJob *__restrict__ jobs, FrontGeom g) {
  const TrackJob &job = jobs[blockIdx.y];
  const int s = job.stream;
  const int *__restrict__ valid = gd.valid + (size_t)s * kValidStride;
  if ((int)blockIdx.x >= valid[0]) return;
  const int c = valid[4 + blockIdx.x];
  if (c < 0) return;
  const SlotRec &sl = gd.slots[gd.wmode[s] == 1 ? job.cur_slot : job.prev_slot];
  fast_select_body(c, g.cells, g.max_bands, sl.fast_total, sl.band_off, sl.band_cnt, sl.kps, g.kps_cap, sl.sort_scratch, g.nfg, sl.cand,
                   sl.cand_cnt);
}

void launch_group_fast(const GroupDev &gd, const TrackJob *jobs, int n_jobs, const FrontGeom &g, cudaStream_t s) {
  if (n_jobs <= 0 || g.n_cells <= 0) return;
  const int smem_w = (g.max_cell_w + 15) & ~15;
  const size_t smem = (size_t)(2 * kBH + 10) * smem_w + 3 * kFastPad + (size_t)(kBH + 2) * smem_w * 4;
  static SmemOptIn optin;
  optin.ensure(k_fast_g, smem);
  PLVIWO_CARVEOUT(k_fast_g);
  k_fast_g<<<dim3(g.max_bands, g.n_cells, n_jobs), kFastThreads, smem, s>>>(gd, jobs, g, smem_w);
}
void launch_group_fast_select(const GroupDev &gd, const TrackJob *jobs, int n_jobs, const FrontGeom &g, cudaStream_t s) {
  if (n_jobs <= 0 || g.n_cells <= 0 || g.max_bands > kSelMaxBands) return;
  PLVIWO_CARVEOUT(k_fast_select_g);
  k_fast_select_g<<<dim3(g.n_cells, n_jobs), kSelThreads, 0, s>>>(gd, jobs, g);
}

void launch_fast_select(const FastCell *d_cells, int n_cells, int max_bands, unsigned *d_total, const int *d_band_off,
                        const int *d_band_cnt, const unsigned *d_kps, int kps_cap, unsigned *d_scratch, int nfg,
                        float2 *d_cand_sel, int *d_cand_cnt, cudaStream_t s) {
  if (n_cells <= 0 || max_bands > kSelMaxBands) return;
  PLVIWO_CARVEOUT(k_fast_select);
  k_fast_select<<<n_cells, kSelThreads, 0, s>>>(d_cells, max_bands, d_total, d_band_off, d_band_cnt, d_kps, kps_cap, d_scratch,
                                                nfg, d_cand_sel, d_cand_cnt);
}

// host instantiation of the same sort (tests: compared with the real std::sort and with the kernel)
void host_sort_corners(unsigned *v, int n, int keep) {
  if (keep > 0) isort::sort_prefix(v, n, keep);
  else isort::sort(v, n);
}

void launch_fast(const DevImage &img, const FastCell *d_cells, int n_cells, int max_bands, int max_cell_w, int threshold,
                 unsigned *d_total, int *d_band_off, int *d_band_cnt, unsigned *d_kps, int kps_cap, cudaStream_t s) {
  if (n_cells <= 0) return;
  int smem_w = (max_cell_w + 15) & ~15;
  size_t smem = (size_t)(2 * kBH + 10) * smem_w + 3 * kFastPad + (size_t)(kBH + 2) * smem_w * 4;
  static SmemOptIn optin;
  optin.ensure(k_fast, smem);
  dim3 grid(max_bands, n_cells);
  PLVIWO_CARVEOUT(k_fast);
  k_fast<<<grid, kFastThreads, smem, s>>>(img.p, img.pitch, d_cells, max_bands, threshold, d_total, d_band_off, d_band_cnt,
                                          d_kps, kps_cap, smem_w);
}

}  // namespace plviwo
