// Line-segment extraction kernels (sm_100a): Canny edge map of the half-resolution equalised frame and the
// FastLineDetector chain walk + incremental segment fit.
//
// Reference ops replaced (both inside cv::ximgproc::FastLineDetector::detect, called at TrackLSD.cpp:200-205 with
// length 20, distance 1.414213562, Canny 50/50 aperture 3, no merge — TrackLSD.h:269-273):
//   cv::Canny(src, 50, 50, 3, L1)    SURVEY.md Appendix A8: low == high, so every gradient-direction local
//                                    maximum above the threshold is an edge and no hysteresis walk is needed
//   lineDetection / getPointChain / extractSegments / additionalOperationsOnSegment    Appendix B
//
// Structure.  The chain walk is order dependent (visited pixels are consumed, seeds are taken in raster order), but
// a walk never leaves the 8-connected component of its seed, so different components cannot influence each other:
// the sequential algorithm is exactly "for every connected component, run the raster-order walk on that component
// alone; then list all chains by the raster index of their seed".  So
//   1. connected components of the edge map by union-find (label = smallest raster index = the component's first seed),
//   2. every component with >= length_threshold + 1 pixels is copied into a private bit map in shared memory and walked
//      there: the small ones of a launch over many frames by one thread each (k_fld_walk_thread, one 64-bit word per
//      row), the others by one warp each (k_fld_walk_cc: its lanes scan for the next seed together and fetch the 5 x 5
//      window of every step together); both walks take their steps from the same two decision tables,
//   3. chains are ranked by seed index, segments are fitted by one thread per chain (running double-precision sums,
//      identical to refitting from scratch) and an ordered compaction restores the reference's output order.
// The first version walked the whole frame with a single thread: 14.6 ms per 640x280 frame.
#include "fe_kernels.h"

#include <cstdlib>

#include <algorithm>
#include <type_traits>
#include <mutex>
#include <cstdio>
#include <cmath>

namespace plviwo {

__global__ void k_unpack_edges(const unsigned *__restrict__ edges, int words_per_row, int w, int h,
                               uint8_t *__restrict__ out) {
  int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
  if (x < w && y < h) out[(size_t)y * w + x] = ((edges[(size_t)y * words_per_row + (x >> 5)] >> (x & 31)) & 1u) ? 255 : 0;
}
void launch_unpack_edges(const FldBuffers &fb, int w, int h, uint8_t *d_out, cudaStream_t s) {
  dim3 grid((w + 255) / 256, h);
  PLVIWO_CARVEOUT(k_unpack_edges);
  k_unpack_edges<<<grid, 256, 0, s>>>(fb.edges, fb.words_per_row, w, h, d_out);
}

// --------------------------------------------------------------------------- connected components (8-conn)
__device__ __forceinline__ int ccl_find(const int *parent, int i) {
  int p = __ldcg(parent + i);
  while (p != i) {
    i = p;
    p = __ldcg(parent + i);
  }
  return i;
}
__device__ __forceinline__ void ccl_union(int *parent, int a, int b) {
  while (true) {
    a = ccl_find(parent, a);
    b = ccl_find(parent, b);
    if (a == b) return;
    if (a < b) { int t = a; a = b; b = t; }   // link the larger root under the smaller index
    int old = atomicMin(parent + a, b);
    if (old == a) return;
    a = old;
  }
}

__device__ __forceinline__ bool edge_at(const unsigned *__restrict__ edges, int words_per_row, int x, int y) {
  return (__ldg(edges + (size_t)y * words_per_row + (x >> 5)) >> (x & 31)) & 1u;
}

// Connected components in three steps:
//   k_ccl_tile     every 64 x 16 tile labels ITS pixels in shared memory (union-find over the tile's horizontal runs) and
//                  counts pixels / bounding boxes per tile-local component: the label written out for a pixel is the raster
//                  index of its tile-local root, the aggregates go to the root's slot of the cnt / bbox planes;
//   k_ccl_border   unions across tile borders on the global label array (only border pixels: ~8 % of the frame);
//   k_ccl_link     tile-local roots that are not global roots point straight at their global root and hand it their
//                  aggregates (a pixel reaches its global root in two loads: label[label[p]]).
// Only edge pixels carry a label, a pixel count and a bounding box; everything asks the bit-packed edge map first.  The
// planes are written for the ~5-10 % of the pixels that are edges, and the hot global atomics of a large component are one
// per TILE it crosses instead of one per few pixels.
constexpr int kTileW = 64, kTileH = 16, kTilePx = kTileW * kTileH, kTileThreads = 256;
constexpr int kTileRuns = kTilePx / 2;                  // a 64-pixel row holds at most 32 runs
constexpr int kRunsPer = kTileRuns / kTileThreads;      // 2

__device__ __forceinline__ int sm_find(const int *lab, int i) {
  int p = lab[i];
  while (p != i) {
    i = p;
    p = lab[i];
  }
  return i;
}
__device__ __forceinline__ void sm_union(int *lab, int a, int b) {
  while (true) {
    a = sm_find(lab, a);
    b = sm_find(lab, b);
    if (a == b) return;
    if (a < b) { int t = a; a = b; b = t; }   // link the larger root under the smaller index
    const int old = atomicMin(lab + a, b);
    if (old == a) return;
    a = old;
  }
}

// Shared memory of the tile labelling, indexed by run id: the tile's horizontal runs numbered in raster order of their
// first pixels.  The first pixel of a component is the first pixel of a run, so the smallest run id of a component is the
// run of its smallest raster index.
struct CclTileSmem {
  unsigned start[kTileH * 2];    // first pixels of the runs, in the words of the edge bits
  int rpref[kTileH * 2 + 1];     // runs starting before word f (exclusive prefix); [32] = all runs of the tile
  int nroot, base;               // tile-local roots; their first slot in lroots
  int rpix[kTileRuns];           // run -> tile pixel index of its first pixel
  int lab[kTileRuns];            // union-find over the runs
  int glab[kTileRuns];           // run -> global raster index of its component's root pixel
  int a_cnt[kTileRuns], a_ymax[kTileRuns], a_xmin[kTileRuns], a_xmax[kTileRuns];
};

// Labels one 64 x 16 tile whose edge bits are bits[row][half] (block-wide call, kTileThreads threads, bits visible to all).
// The nodes of the union-find are the horizontal runs (~146 per tile on the bench scenes against ~247 edge pixels):
//   1. warp 0 numbers the runs in raster order (the first-pixel bits of each word, a scan of their population counts);
//   2. thread t takes run t (and t + 256): its length, and the aggregates of the run alone;
//   3. a run is 8-adjacent to every run of the row above that meets its pixels dilated by one; those are consecutive ids;
//   4. every run finds its root, adds its aggregates there and records the root's global index;
//   5. one lane per pixel writes the labels (a pixel's run id is a population count of the first-pixel bits before it),
//      the roots write cnt / bbox and take their lroots slots from one reservation per tile.
// Nothing depends on the order the runs are processed in (roots are minima, aggregates are sums / minima / maxima).
__device__ __forceinline__ void ccl_tile_body(const FldBuffers &fb, CclTileSmem &sm, const unsigned (*bits)[2], int x0, int y0,
                                              int w, int h) {
  int *__restrict__ label = fb.label, *__restrict__ cnt = fb.cnt, *__restrict__ bbox = fb.bbox /* maxy, minx, maxx planes */;
  int *lab = sm.lab, *a_cnt = sm.a_cnt, *a_ymax = sm.a_ymax, *a_xmin = sm.a_xmin, *a_xmax = sm.a_xmax;
  const int tid = threadIdx.x, lane = tid & 31, wv = tid >> 5;
  const unsigned *flat = &bits[0][0];   // word f = row f / 2, half f % 2: pixel index = 32 f + bit
  auto row_of = [&](const unsigned *v, int y) -> unsigned long long { return (unsigned long long)v[2 * y + 1] << 32 | v[2 * y]; };
  if (wv == 0) {
    const unsigned b = flat[lane];
    const unsigned lo = __shfl_sync(0xffffffffu, b, lane & ~1);   // a run of the high half may start in the low half
    const unsigned st = b & ~(b << 1 | ((lane & 1) ? lo >> 31 : 0u));
    const int c = __popc(st);
    int incl = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += t;
    }
    sm.start[lane] = st;
    sm.rpref[lane] = incl - c;
    if (lane == 31) sm.rpref[32] = incl;
    if (lane == 0) sm.nroot = 0;
    int q = incl - c;
    for (unsigned m = st; m; m &= m - 1) sm.rpix[q++] = 32 * lane + __ffs((int)m) - 1;
  }
  __syncthreads();
  const int nruns = sm.rpref[32];
  if (nruns == 0) return;   // no edge pixel in this tile
  int ry[kRunsPer], rx[kRunsPer], rlen[kRunsPer];
#pragma unroll
  for (int k = 0; k < kRunsPer; k++) {
    const int t = tid + k * kTileThreads;
    rlen[k] = 0;
    if (t < nruns) {
      const int p = sm.rpix[t];
      ry[k] = p >> 6;
      rx[k] = p & (kTileW - 1);
      rlen[k] = __clzll(__brevll(~(row_of(flat, ry[k]) >> rx[k])));   // trailing ones from the first pixel
      lab[t] = t;
      a_cnt[t] = rlen[k];
      a_ymax[t] = ry[k];
      a_xmin[t] = rx[k];
      a_xmax[t] = rx[k] + rlen[k] - 1;
    }
  }
  __syncthreads();
  // run id of the pixel at (x, y): the runs before row y, plus the runs of row y starting at or before x, minus one
  auto run_at = [&](int x, int y) -> int {
    return sm.rpref[2 * y] + __popcll(row_of(sm.start, y) & (~0ull >> (63 - x))) - 1;
  };
#pragma unroll
  for (int k = 0; k < kRunsPer; k++) {
    if (rlen[k] == 0 || ry[k] == 0) continue;
    const int lo = max(rx[k] - 1, 0), hi = min(rx[k] + rlen[k], kTileW - 1);
    const unsigned long long touch = row_of(flat, ry[k] - 1) & (~0ull >> (63 - hi)) & (~0ull << lo);
    if (touch == 0) continue;
    const int t = tid + k * kTileThreads;
    const int first = run_at(__clzll(__brevll(touch)), ry[k] - 1), last = run_at(63 - __clzll(touch), ry[k] - 1);
    for (int j = first; j <= last; j++) sm_union(lab, t, j);
  }
  __syncthreads();
  bool is_root[kRunsPer];
#pragma unroll
  for (int k = 0; k < kRunsPer; k++) {
    const int t = tid + k * kTileThreads;
    is_root[k] = false;
    if (rlen[k] == 0) continue;
    const int r = sm_find(lab, t);
    is_root[k] = r == t;
    if (!is_root[k]) {
      atomicAdd(&a_cnt[r], rlen[k]);
      atomicMax(&a_ymax[r], ry[k]);
      atomicMin(&a_xmin[r], rx[k]);
      atomicMax(&a_xmax[r], rx[k] + rlen[k] - 1);
    }
    const int rp = sm.rpix[r];
    sm.glab[t] = (y0 + (rp >> 6)) * w + x0 + (rp & (kTileW - 1));
  }
  int slot[kRunsPer];   // the root's place among the tile's roots
#pragma unroll
  for (int k = 0; k < kRunsPer; k++) {
    const unsigned m = __ballot_sync(0xffffffffu, is_root[k]);
    int q = 0;
    if (lane == 0 && m) q = atomicAdd(&sm.nroot, __popc(m));
    slot[k] = __shfl_sync(0xffffffffu, q, 0) + __popc(m & ((1u << lane) - 1));
  }
  __syncthreads();
  if (tid == 0) sm.base = atomicAdd(fb.lroot_n, sm.nroot);   // tile-local roots, for k_ccl_link
  // labels: warp wv writes rows 2 wv and 2 wv + 1, one lane per pixel, so a warp's stores are one row segment
#pragma unroll
  for (int j = 0; j < 4; j++) {
    const int f = 4 * wv + j;
    if ((flat[f] >> lane) & 1u) {
      const int id = sm.rpref[f] + __popc(sm.start[f] & (0xffffffffu >> (31 - lane))) - 1;
      label[(y0 + (f >> 1)) * w + x0 + 32 * (f & 1) + lane] = sm.glab[id];
    }
  }
  __syncthreads();
  const int n = w * h;
#pragma unroll
  for (int k = 0; k < kRunsPer; k++) {
    if (!is_root[k]) continue;
    const int t = tid + k * kTileThreads;
    const int gi = sm.glab[t];
    cnt[gi] = a_cnt[t];
    bbox[gi] = y0 + a_ymax[t];
    bbox[n + gi] = x0 + a_xmin[t];
    bbox[2 * n + gi] = x0 + a_xmax[t];
    const int q = sm.base + slot[k];
    if (q < fb.lroot_cap) fb.lroots[q] = gi;
  }
}

template <class B>
__global__ void __launch_bounds__(kTileThreads)
    k_ccl_tile(const __grid_constant__ B b, int w, int h) {
  const FldBuffers &fb = b.fld_of(blockIdx.z);
  const unsigned *__restrict__ edges = fb.edges;
  const int words_per_row = fb.words_per_row;
  __shared__ CclTileSmem sm;
  __shared__ unsigned s_bits[kTileH][2];
  const int tid = threadIdx.x;
  const int x0 = blockIdx.x * kTileW, y0 = blockIdx.y * kTileH;
  // (counters and the local-root count are zeroed by k_ccl_reset, ahead of this launch)
  if (tid < kTileH * 2) {
    const int r = tid >> 1, k = tid & 1;
    const int gy = y0 + r, gw = (x0 >> 5) + k;
    unsigned v = 0;
    if (gy < h && gw < words_per_row) v = edges[(size_t)gy * words_per_row + gw];
    if (gy < h && (gw << 5) + 32 > w) v &= (gw << 5) < w ? (0xffffffffu >> (32 - (w - (gw << 5)))) : 0u;   // beyond the frame
    s_bits[r][k] = v;
  }
  __syncthreads();
  ccl_tile_body(fb, sm, s_bits, x0, y0, w, h);
}

template <class B>
__global__ void k_ccl_reset(const __grid_constant__ B b) {
  const FldBuffers &fb = b.fld_of(blockIdx.x);
  if (threadIdx.x < 12) fb.counters[threadIdx.x] = 0;
  if (threadIdx.x == 12) *fb.lroot_n = 0;
}

// ------------------------------------------------------------------------------------------------ Canny
constexpr int kCnW = 64, kCnH = 16, kCnThreads = 256;

// Stream group (FldTable): the Canny CTA goes on to label its tile (the Canny tile IS the connected-component tile: same
// 64 x 16 pixels, same 256 threads), so the edge bits never make the trip through global memory before the first labelling
// step and the frame's tiles are launched once instead of twice; k_ccl_reset runs ahead of that Canny launch.  A handle's
// frames (FldBatch) are labelled by k_ccl_tile, at the start of the line launches.
template <class B>
constexpr bool kFusedLabels = std::is_same<B, FldTable>::value;
static_assert(kCnW == kTileW && kCnH == kTileH && kCnThreads == kTileThreads, "Canny tile = connected-component tile");
constexpr int kCnPixW = kCnW + 8;   // staged columns: x0 - 4 ... x0 + 67, whole aligned words (the Sobel halo is x0 - 2 ... x0 + 65)
struct CannySmem {
  uint8_t pix[kCnH + 4][kCnPixW];
  short sdx[kCnH + 2][kCnW + 2];
  short sdy[kCnH + 2][kCnW + 2];
  unsigned short mag[kCnH + 2][kCnW + 2];
};
template <class B>
__global__ void __launch_bounds__(kCnThreads)
    k_canny(const __grid_constant__ B b, int low) {
  constexpr bool kFuse = kFusedLabels<B>;
  const uint8_t *__restrict__ img = b.half_of(blockIdx.z).p;
  const int w = b.half_of(blockIdx.z).w, h = b.half_of(blockIdx.z).h, pitch = b.half_of(blockIdx.z).pitch;
  unsigned *__restrict__ edges = b.fld_of(blockIdx.z).edges;
  const int words_per_row = b.fld_of(blockIdx.z).words_per_row;
  // the labelling pass reuses the gradient planes' shared memory (they are dead once the edge bits exist)
  __shared__ __align__(16) uint8_t smem_raw[kFuse ? (sizeof(CclTileSmem) > sizeof(CannySmem) ? sizeof(CclTileSmem) : sizeof(CannySmem))
                                                  : sizeof(CannySmem)];
  __shared__ unsigned s_bits[kCnH][2];
  CannySmem &cs = *reinterpret_cast<CannySmem *>(smem_raw);
  auto &pix = cs.pix;
  auto &sdx = cs.sdx;
  auto &sdy = cs.sdy;
  auto &mag = cs.mag;
  const int tx0 = blockIdx.x * kCnW, ty0 = blockIdx.y * kCnH;
  const int tid = threadIdx.x;
  // pixels with a halo of 2, BORDER_REPLICATE: one 32-bit word per thread and step; a word that reaches beyond the frame
  // (or an unaligned image) is read byte by byte with the coordinates clamped
  const bool aligned = ((pitch | (int)(size_t)img) & 3) == 0;
  for (int i = tid; i < (kCnH + 4) * (kCnPixW / 4); i += kCnThreads) {
    const int r = i / (kCnPixW / 4), k = i - r * (kCnPixW / 4);
    const int gy = min(max(ty0 - 2 + r, 0), h - 1), gx = tx0 - 4 + 4 * k;
    const uint8_t *src = img + (size_t)gy * pitch;
    unsigned v;
    if (aligned && gx >= 0 && gx + 3 < w) {
      v = __ldg(reinterpret_cast<const unsigned *>(src + gx));
    } else {
      v = 0;
#pragma unroll
      for (int j = 0; j < 4; j++) v |= (unsigned)src[min(max(gx + j, 0), w - 1)] << (8 * j);
    }
    *reinterpret_cast<unsigned *>(&pix[r][4 * k]) = v;
  }
  __syncthreads();
  // Sobel + L1 magnitude with a halo of 1; zero outside the image
  for (int i = tid; i < (kCnH + 2) * (kCnW + 2); i += kCnThreads) {
    int r = i / (kCnW + 2), c = i - r * (kCnW + 2);
    int gx = tx0 - 1 + c, gy = ty0 - 1 + r;
    int dx = 0, dy = 0, m = 0;
    if (gx >= 0 && gx < w && gy >= 0 && gy < h) {
      const uint8_t *p = &pix[r + 1][c + 3];
      const int s = kCnPixW;
      dx = (p[-s + 1] + 2 * p[1] + p[s + 1]) - (p[-s - 1] + 2 * p[-1] + p[s - 1]);
      dy = (p[s - 1] + 2 * p[s] + p[s + 1]) - (p[-s - 1] + 2 * p[-s] + p[-s + 1]);
      m = abs(dx) + abs(dy);
    }
    sdx[r][c] = (short)dx;
    sdy[r][c] = (short)dy;
    mag[r][c] = (unsigned short)m;
  }
  __syncthreads();
  // non-maximum suppression; warp wv handles rows 2wv, 2wv+1; 32 pixels per ballot
  const int wv = tid >> 5, lane = tid & 31;
#pragma unroll
  for (int q = 0; q < 4; q++) {
    int r = 2 * wv + (q >> 1), c = (q & 1) * 32 + lane;
    int gx = tx0 + c, gy = ty0 + r;
    bool edge = false;
    if (gx < w && gy < h) {
      int m = mag[r + 1][c + 1];
      if (m > low) {
        int dx = sdx[r + 1][c + 1], dy = sdy[r + 1][c + 1];
        int x = abs(dx), y = abs(dy) << 15;
        int tg22x = x * 13573;
        if (y < tg22x) {
          edge = m > mag[r + 1][c] && m >= mag[r + 1][c + 2];
        } else {
          int tg67x = tg22x + (x << 16);
          if (y > tg67x) {
            edge = m > mag[r][c + 1] && m >= mag[r + 2][c + 1];
          } else {
            int s = (dx ^ dy) < 0 ? -1 : 1;
            edge = m > mag[r][c + 1 - s] && m > mag[r + 2][c + 1 + s];
          }
        }
      }
      // FastLineDetector clears the two corner blocks of the edge map before walking
      if (gy < 6 && gx < 6) edge = false;
      if (gy >= h - 5 && gx >= w - 5) edge = false;
    }
    unsigned bits = __ballot_sync(0xffffffffu, edge);
    if (lane == 0 && gy < h && (tx0 + (q & 1) * 32) < w) edges[(size_t)gy * words_per_row + ((tx0 + (q & 1) * 32) >> 5)] = bits;
    if (kFuse && lane == 0) s_bits[r][q & 1] = bits;   // pixels beyond the frame are not edges: the same bits k_ccl_tile would read
  }
  if constexpr (kFuse) {
    __syncthreads();   // every warp is done with the gradient planes; the tile's bits are complete
    ccl_tile_body(b.fld_of(blockIdx.z), *reinterpret_cast<CclTileSmem *>(smem_raw), s_bits, tx0, ty0, w, h);
  }
}

// Tile labelling of one frame's edge bits (fb.edges), as the line launches start it; for tests.
void launch_ccl_tiles(FldBuffers &fb, int w, int h, cudaStream_t s) {
  FldBatch b;
  b.n = 1;
  b.f[0] = fb;
  PLVIWO_CARVEOUT(k_ccl_reset<FldBatch>);
  k_ccl_reset<FldBatch><<<1, 32, 0, s>>>(b);
  PLVIWO_CARVEOUT(k_ccl_tile<FldBatch>);
  k_ccl_tile<FldBatch><<<dim3((w + kTileW - 1) / kTileW, (h + kTileH - 1) / kTileH, 1), kTileThreads, 0, s>>>(b, w, h);
}

template <class B>
static void launch_canny_any(const B &b, int n, int w, int h, float th_low, cudaStream_t s) {
  dim3 grid((w + kCnW - 1) / kCnW, (h + kCnH - 1) / kCnH, n);
  if constexpr (kFusedLabels<B>) {
    PLVIWO_CARVEOUT(k_ccl_reset<B>);
    k_ccl_reset<B><<<n, 32, 0, s>>>(b);
  }
  PLVIWO_CARVEOUT(k_canny<B>);
  k_canny<B><<<grid, kCnThreads, 0, s>>>(b, (int)floorf(th_low));
}
void launch_canny_batch(const FldBatch &b, float th_low, float th_high, cudaStream_t s) {
  (void)th_high;  // low == high is enforced at create time (no hysteresis pass is implemented)
  launch_canny_any(b, b.n, b.half[0].w, b.half[0].h, th_low, s);
}
void launch_canny_table(const SlotRec *slots, const int *line_slots, int n_jobs, int w, int h, float th_low, cudaStream_t s) {
  if (n_jobs <= 0) return;
  launch_canny_any(FldTable{slots, line_slots}, n_jobs, w, h, th_low, s);
}
void launch_canny(const DevImage &half, float th_low, float th_high, FldBuffers &fb, cudaStream_t s) {
  FldBatch b;
  b.n = 1;
  b.half[0] = half;
  b.f[0] = fb;
  launch_canny_batch(b, th_low, th_high, s);
}

// One thread per pixel of a tile border: rows y = 16 k (all x) first, then columns x = 64 m (all y).
template <class B>
__global__ void k_ccl_border(const __grid_constant__ B b, int w, int h) {
  const FldBuffers &fb = b.fld_of(blockIdx.y);
  const unsigned *__restrict__ edges = fb.edges;
  const int words_per_row = fb.words_per_row;
  int *__restrict__ label = fb.label;
  const int nrow = (h - 1) / kTileH, ncol = (w - 1) / kTileW;   // interior boundaries
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < nrow * w) {
    const int y = (t / w + 1) * kTileH, x = t % w;
    if (!edge_at(edges, words_per_row, x, y)) return;
    const int i = y * w + x;
    if (x > 0 && edge_at(edges, words_per_row, x - 1, y - 1)) ccl_union(label, i, i - w - 1);
    if (edge_at(edges, words_per_row, x, y - 1)) ccl_union(label, i, i - w);
    if (x < w - 1 && edge_at(edges, words_per_row, x + 1, y - 1)) ccl_union(label, i, i - w + 1);
    return;
  }
  const int u = t - nrow * w;
  if (u >= ncol * h) return;
  const int x = (u / h + 1) * kTileW, y = u % h;
  if (!edge_at(edges, words_per_row, x, y)) return;
  const int i = y * w + x;
  if (y > 0 && edge_at(edges, words_per_row, x - 1, y - 1)) ccl_union(label, i, i - w - 1);
  if (edge_at(edges, words_per_row, x - 1, y)) ccl_union(label, i, i - 1);
  if (y < h - 1 && edge_at(edges, words_per_row, x - 1, y + 1)) ccl_union(label, i, i + w - 1);
}

// One thread per tile-local root: find the global root once, point straight at it, hand the aggregates over.
template <class B>
__global__ void k_ccl_link(const __grid_constant__ B b, int w, int h) {
  const FldBuffers &fb = b.fld_of(blockIdx.y);
  int *__restrict__ label = fb.label, *__restrict__ cnt = fb.cnt, *__restrict__ bbox = fb.bbox;
  const int nl = min(*fb.lroot_n, fb.lroot_cap);
  const int n = w * h;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < nl; t += gridDim.x * blockDim.x) {
    const int i = fb.lroots[t];
    const int root = ccl_find(label, i);
    if (root == i) continue;
    atomicExch(label + i, root);   // other threads may be walking through this node: any ancestor is a valid parent
    atomicAdd(cnt + root, cnt[i]);
    atomicMax(bbox + root, bbox[i]);
    atomicMin(bbox + n + root, bbox[n + i]);
    atomicMax(bbox + 2 * n + root, bbox[2 * n + i]);
  }
}

// Components large enough to hold a chain of length_threshold + 1 pixels are queued for the walk in three classes:
//   BIG    the private bit map (bounding box rounded to 32-pixel words, plus padding) does not fit a warp's slice of the
//          walk kernel's shared-memory arena: a whole CTA gathers it and one warp walks it, these go first (they are also
//          the long ones: a walk is sequential and the longest component is the critical path of the launch);
//   W      fits a slice but not class T: one WARP per component, the warps of a CTA work side by side;
//   T      the bounding box is at most 62 x 44 pixels — nine components in ten, a third of the walked pixels: one THREAD per
//          component (k_fld_walk_thread), the bit map is one 64-bit word per row.  A warp instruction costs an issue slot
//          whether one lane or 32 have a pixel in hand: here 32 components advance per instruction instead of one.
constexpr int kPadRows = 2;             // zero rows above and below the private bit map (the walk looks 2 pixels ahead)
constexpr int kWalkThreads = 128;
constexpr int kWalkWarps = kWalkThreads / 32;
constexpr int kSliceWords = 1600;       // per-warp bit map slice (6.25 KB): e.g. 128 x 224 or 640 x 68 pixels of bounding box
constexpr int kTMaxW = 62, kTMaxH = 44; // class T bounding box
constexpr int kTRows = kTMaxH + 2;      // rows of a thread's bit map (one zero row above and below)
constexpr int kTLanes = 64;             // threads per CTA of the thread-walk kernel
// a BIG component spans > kSliceWords words, i.e. at least ~280 pixels in a row or column direction: at most n / 128 of them
__host__ __device__ inline int comp_cap_big(int n) { return n / 128 + 1; }
// comp_root: [0, comp_cap_big) BIG, then max_chains entries of class W, then max_chains entries of class T

// counters: [0] BIG components, [1] BIG cursor, [2] chain-point cursor, [3] chains, [4] segments, [5] class-W components,
//           [6] class-T components, [7] class-W cursor, [8] class-T cursor
template <class B>
__global__ void k_ccl_roots(const __grid_constant__ B b, int w, int h, int min_pixels, int thread_class) {   // strides over the tile-local roots
  const FldBuffers &fb = b.fld_of(blockIdx.y);
  const int *__restrict__ label = fb.label, *__restrict__ cnt = fb.cnt, *__restrict__ bbox = fb.bbox;
  int *__restrict__ comp_root = fb.comp_root, *__restrict__ counters = fb.counters;
  const int max_comps = fb.max_chains;
  const int nl = min(*fb.lroot_n, fb.lroot_cap);
  const int n = w * h;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < nl; t += gridDim.x * blockDim.x) {
    const int i = fb.lroots[t];
    if (label[i] != i) continue;   // a global root is the tile-local root of its own tile
    const int c = cnt[i];
    if (c < min_pixels) continue;
    const int bh = bbox[i] - i / w + 1;
    const int groups = (bbox[2 * n + i] >> 5) - (bbox[n + i] >> 5) + 1;
    const int bw = bbox[2 * n + i] - bbox[n + i] + 1;
    if (thread_class && bw <= kTMaxW && bh <= kTMaxH) {
      const int q = atomicAdd(counters + 6, 1);
      if (q < max_comps) comp_root[comp_cap_big(n) + max_comps + q] = i;
    } else if ((bh + 2 * kPadRows) * (groups + 2) > kSliceWords) {
      const int q = atomicAdd(counters + 0, 1);
      if (q < comp_cap_big(n)) comp_root[q] = i;
    } else {
      const int q = atomicAdd(counters + 5, 1);
      if (q < max_comps) comp_root[comp_cap_big(n) + q] = i;
    }
  }
}

// ------------------------------------------------------------------------------------------- chain walk
// getPointChain: among the set neighbours take the one whose direction is closest to the running direction (circular
// difference; ties go to the LATER neighbour index), accept only a difference < 2; the first step of a chain takes the
// first set neighbour.  Neighbour index i -> (dr, dc): 0 (+1,+1) 1 (+1,0) 2 (+1,-1) 3 (0,-1) 4 (-1,-1) 5 (-1,0) 6 (-1,+1)
// 7 (0,+1).  The whole decision is a table: [first step?][neighbour key][running direction + 3] -> i | (dr+1) << 4 |
// (dc+1) << 6 (i == 8: stop); the 8 direction entries of a key are one 8-byte load and the entry is picked with a byte
// permute once the direction is known, so the direction update is not on the path to the table address.
// The neighbour key is taken from a 5 x 5 bit window B (bit 5 (r + 2) + (c + 2) = pixel (r, c) relative to the window
// centre): for a pixel at offset (dr, dc) from the centre, Bs = B >> (6 + 5 dr + dc) has neighbour i at bit
// {12, 11, 10, 5, 0, 1, 2, 7}[i]; the key packs those 8 bits into one byte (bits 0-2 stay, 5 -> 3, 7 -> 4, 10-12 -> 5-7),
// so the tables are 4.5 KB (they were 33 KB with an 11-bit key, which cost the kernel its co-residency with everything
// else that needs shared memory).
static int choose_neighbour_host(unsigned mask, int direction) {
  const int i0 = direction < 0 ? direction + 8 : direction;      // neighbour index with difference 0
  if ((mask >> i0) & 1u) return i0;
  const int ia = (i0 + 1) & 7, ib = (i0 + 7) & 7;               // the two neighbours with difference 1
  const bool sa = (mask >> ia) & 1u, sb = (mask >> ib) & 1u;
  if (sa && sb) return ia > ib ? ia : ib;
  if (sa) return ia;
  if (sb) return ib;
  return 8;
}
static inline int nb_dr(int i) { return (i <= 2) ? 1 : ((i == 3 || i == 7) ? 0 : -1); }
static inline int nb_dc(int i) { return (i == 0 || i == 6 || i == 7) ? 1 : ((i == 1 || i == 5) ? 0 : -1); }

constexpr int kKeys = 256;
constexpr int kLut1 = 2 * kKeys * 8;    // [first step?][neighbour key][direction + 3] -> decision
constexpr int kLut2 = 8 * 8 * 8;        // [min(step, 7)][direction + 3][i] -> next direction + 3
constexpr int kLutSize = kLut1 + kLut2;
__device__ __align__(16) uint8_t g_walk_lut[kLutSize];
static bool g_walk_lut_ready[64] = {false};

void init_fld_constants() {
  static std::mutex mu;   // handles may be created from several host threads
  std::lock_guard<std::mutex> lk(mu);
  int dev = 0;
  cudaGetDevice(&dev);
  if (g_walk_lut_ready[dev & 63]) return;
  static uint8_t lut[kLutSize];
  static const int key_bit[8] = {7, 6, 5, 3, 0, 1, 2, 4};   // key bit of neighbour i (see above)
  for (int first = 0; first < 2; first++)
    for (unsigned key = 0; key < (unsigned)kKeys; key++) {
      unsigned mask = 0;
      for (int i = 0; i < 8; i++) mask |= ((key >> key_bit[i]) & 1u) << i;
      for (int d = 0; d < 8; d++) {
        int i = 8;
        if (mask) i = first ? __builtin_ffs((int)mask) - 1 : choose_neighbour_host(mask, d - 3);
        const int dr = i < 8 ? nb_dr(i) : 0, dc = i < 8 ? nb_dc(i) : 0;
        lut[(first * kKeys + key) * 8 + d] = (uint8_t)(i | ((dr + 1) << 4) | ((dc + 1) << 6));
      }
    }
  // running direction after taking neighbour i at step `step`: direction = (direction * step + cd) / (step + 1), C integer
  // division; from step 7 on the result no longer depends on step (|cd - direction| <= 7 < step + 1)
  for (int sc = 0; sc < 8; sc++)
    for (int d = 0; d < 8; d++)
      for (int i = 0; i < 8; i++) {
        const int cd = i > 4 ? i - 8 : i;
        const int nd = sc == 0 ? cd : ((d - 3) * sc + cd) / (sc + 1);
        lut[kLut1 + (sc * 8 + d) * 8 + i] = (uint8_t)(nd + 3);
      }
  cudaMemcpyToSymbol(g_walk_lut, lut, sizeof(lut));
  g_walk_lut_ready[dev & 63] = true;
}

// explicit shared-memory accesses by 32-bit shared address (keeps the address arithmetic out of the walk loop)
__device__ __forceinline__ unsigned lds_u32(unsigned addr) {
  unsigned v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ unsigned lds_u8(unsigned addr) {
  unsigned v;
  asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ uint2 lds_u64(unsigned addr) {
  uint2 v;
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void sts_u32(unsigned addr, unsigned v) {
  asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

struct WalkCtx {
  const unsigned *edges;
  int words_per_row;
  const int *label, *cnt, *bbox;
  int *counters;
  int2 *chain_pts;
  int *chain_seed, *chain_off, *chain_len;
  int max_chains, w, n, length_threshold;
  bool vec4;
};

// Gather of one component's private bit map by `nw` warps (this is warp `wi` of them): private word = edge word AND
// (label == root).  Row stride ws = groups + 2 words with one zero word on each side, kPadRows zero rows above and below;
// word g + 1 of row ly + kPadRows is the component's part of edge word (y0 + ly, g0 + g), so no shifting is needed.  A
// warp covers 128 pixels (4 words) per round with one 16-byte label load per lane, skipped where the edge map is empty.
__device__ __forceinline__ void walk_gather(const WalkCtx &c, unsigned *bm, int root, int y0, int g0, int groups, int bh, int ws,
                                            int wi, int nw, int lane) {
  const int segs = (groups + 3) >> 2;          // 4-word segments per row
  const int items = bh * segs;
  const unsigned gmask = 0xffu << (lane & 24);
  for (int it0 = wi * 4; it0 < items; it0 += nw * 4) {
    int4 lab[4];
    unsigned nib[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const int it = it0 + u;
      nib[u] = 0;
      lab[u] = make_int4(-2, -2, -2, -2);
      if (it < items) {
        const int ly = it / segs, sg = it - ly * segs;
        const int g = 4 * sg + (lane >> 3);
        if (g < groups) {
          const unsigned e = __ldg(c.edges + (size_t)(y0 + ly) * c.words_per_row + g0 + g);
          nib[u] = (e >> (4 * (lane & 7))) & 15u;
          if (nib[u]) {
            const int *lp = c.label + (size_t)(y0 + ly) * c.w + ((g0 + g) << 5) + 4 * (lane & 7);
            if (c.vec4) {
              lab[u] = *reinterpret_cast<const int4 *>(lp);
            } else {
              if (nib[u] & 1u) lab[u].x = lp[0];
              if (nib[u] & 2u) lab[u].y = lp[1];
              if (nib[u] & 4u) lab[u].z = lp[2];
              if (nib[u] & 8u) lab[u].w = lp[3];
            }
          }
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 4; u++) {
      const int it = it0 + u;
      // a pixel's label is its tile-local root (k_ccl_tile); the label of a tile-local root is the global root (k_ccl_link)
      const int l4[4] = {lab[u].x, lab[u].y, lab[u].z, lab[u].w};
      unsigned bits = 0;
#pragma unroll
      for (int k = 0; k < 4; k++) {
        if (!((nib[u] >> k) & 1u)) continue;
        int l = l4[k];
        if (l != root) l = __ldg(c.label + l);
        bits |= (l == root ? 1u : 0u) << k;
      }
      bits = (bits & nib[u]) << (4 * (lane & 7));
      const unsigned word = __reduce_or_sync(gmask, bits);
      if ((lane & 7) == 0 && word && it < items) {
        const int ly = it / segs, sg = it - ly * segs;
        bm[(ly + kPadRows) * ws + 1 + 4 * sg + (lane >> 3)] = word;
      }
    }
  }
}

// The sequential part, one warp: raster-order seeds, one chain per seed.  The walk is a chain of dependent steps and a GPU
// thread retires a dependent instruction every ~4 cycles, so the step is spread over the warp and software-pipelined:
// lane j < 25 reads pixel j of the 5 x 5 window around the CURRENT pixel (one shared load, one ballot) while the decision
// for the current pixel is taken from the window fetched around the PREVIOUS pixel (shift, 8-bit key, one table look-up).
// All state is warp-uniform.
__device__ __forceinline__ void walk_component(const WalkCtx &c, unsigned *bm, unsigned lut_addr, int root, int y0, int g0, int groups,
                                               int bh, int ws, int lane) {
  const int my_dr = lane < 25 ? lane / 5 - 2 : 0;   // this lane's pixel of the window (lanes >= 25 look at the centre; their
  const int my_dc = lane < 25 ? lane % 5 - 2 : 0;   // ballot bits are dropped)
  int npts = 0;
  if (lane == 0) npts = atomicAdd(c.counters + 2, c.cnt[root]);   // this component's slice of the chain-point pool
  npts = __shfl_sync(0xffffffffu, npts, 0);
  const int xbase = (g0 << 5) - 32;                // global x of bit 0 of a private row
  const unsigned bm_addr = (unsigned)__cvta_generic_to_shared(bm);
  const int my_off = my_dr * ws;
  int sy = 0, sg = 0;                              // scan position (row, word): everything before it is consumed
  while (sy < bh) {
    // next seed: first set bit at or after the scan position, 32 words per probe
    const int g = sg + lane;
    const unsigned v = g < groups ? bm[(sy + kPadRows) * ws + 1 + g] : 0u;
    const unsigned any = __ballot_sync(0xffffffffu, v != 0);
    __syncwarp();   // every lane's probe has been read before a lane consumes a pixel below (write after read)
    if (!any) {
      sg += 32;
      if (sg >= groups) { sg = 0; sy++; }
      continue;
    }
    const int first = __ffs(any) - 1;
    const unsigned wv = __shfl_sync(0xffffffffu, v, first);
    sg += first;
    // ---- walk one chain; p = bit position in the private row (pixel local x + 32), rb = word index of the row start
    int p = ((sg + 1) << 5) + __ffs(wv) - 1, cy = sy;
    int rb = (cy + kPadRows) * ws;
    const int start = npts;
    const int seed = (y0 + cy) * c.w + xbase + p;
    int step = 0;
    unsigned dsel = 0, sh = 6;              // dsel: running direction + 3 (byte selector)
    unsigned tb = lut_addr + kKeys * 8;     // first-step half of the table
    // consume the seed, then fetch its 5 x 5 window
    if (lane == 0) sts_u32(bm_addr + 4u * (unsigned)(rb + (p >> 5)), wv & ~(1u << (p & 31)));
    __syncwarp();   // the other lanes' window loads below must see the cleared bit (memory ordering inside the warp)
    unsigned Bw;
    {
      const int qb = p + my_dc;
      const unsigned word = lds_u32(bm_addr + 4u * (unsigned)(rb + my_off + (qb >> 5)));
      Bw = __ballot_sync(0xffffffffu, (word >> (qb & 31)) & 1u);
      __syncwarp();
    }
    while (true) {
      // Bw: window around the previous pixel (the seed itself in the first round); the current pixel sits at offset
      // (dr, dc) of the previous move inside it and sh = 6 + 5 dr + dc.  Start fetching the current pixel's window.
      const int qb = p + my_dc;
      const unsigned waddr = bm_addr + 4u * (unsigned)(rb + my_off + (qb >> 5));
      const unsigned word = lds_u32(waddr);
      const unsigned Bs = Bw >> sh;
      const unsigned key = (Bs & 7u) | ((Bs >> 2) & 8u) | ((Bs >> 3) & 16u) | ((Bs >> 5) & 0xE0u);
      const uint2 ev = lds_u64(tb + key * 8u);
      if (lane == 0) c.chain_pts[npts] = make_int2(xbase + p, y0 + cy);
      npts++;
      Bw = __ballot_sync(0xffffffffu, (word >> (qb & 31)) & 1u);
      __syncwarp();   // all window loads of this round are done before a lane rewrites its word below (write after read)
      const unsigned e = __byte_perm(ev.x, ev.y, dsel);   // byte dsel of the 8 entries
      const unsigned i = e & 15u;
      if (i == 8u) break;
      dsel = lds_u8(lut_addr + kLut1 + ((unsigned)min(step, 7) * 8u + dsel) * 8u + i);
      step++;
      tb = lut_addr;
      const unsigned r1 = (e >> 4) & 3u, c1 = (e >> 6) & 3u;   // dr + 1, dc + 1
      sh = 5u * r1 + c1;
      // consume the new pixel: the lane that just fetched it (window position 6 + sh) rewrites its word without it
      if (lane == (int)(sh + 6u)) sts_u32(waddr, word & ~(1u << (qb & 31)));
      __syncwarp();   // orders the store before the next round's window loads of the other lanes (and the seed scan)
      p += (int)c1 - 1;
      cy += (int)r1 - 1;
      rb += ((int)r1 - 1) * ws;
    }
    if (npts - start < c.length_threshold + 1) {
      npts = start;  // chain too short: dropped (its pixels stay consumed)
    } else if (lane == 0) {
      const int k = atomicAdd(c.counters + 3, 1);
      if (k < c.max_chains) {
        c.chain_seed[k] = seed;
        c.chain_off[k] = start;
        c.chain_len[k] = npts - start;
      }
    }
  }
}

// grid = (walkers, frame).  Phase 1: the CTA takes BIG components one at a time (all warps gather into the whole arena,
// warp 0 walks).  Phase 2: every warp takes components of its own from the common queue (B then C) and works in its slice
// of the arena; no block-wide synchronisation any more.  The 8 CTAs per SM of the launch bounds hold the kernel to 64
// registers without spills (up to 72 otherwise); its ~31 KB of shared memory allow 7 per SM anyway.
template <class B>
__global__ void __launch_bounds__(kWalkThreads, 8)
    k_fld_walk_cc(const __grid_constant__ B b, int w, int h, int length_threshold) {
  const FldBuffers &fb = b.fld_of(blockIdx.y);
  WalkCtx c;
  c.edges = fb.edges;
  c.words_per_row = fb.words_per_row;
  c.label = fb.label;
  c.cnt = fb.cnt;
  c.bbox = fb.bbox;
  c.counters = fb.counters;
  c.chain_pts = fb.chain_pts;
  c.chain_seed = fb.chain_seed;
  c.chain_off = fb.chain_off;
  c.chain_len = fb.chain_len;
  c.max_chains = fb.max_chains;
  c.w = w;
  c.n = w * h;
  c.length_threshold = length_threshold;
  c.vec4 = (w & 3) == 0;
  const int *__restrict__ comp_root = fb.comp_root;
  extern __shared__ __align__(16) uint8_t walk_smem[];   // decision tables, then the bit map arena
  uint8_t *lut = walk_smem;
  unsigned *arena = reinterpret_cast<unsigned *>(walk_smem + kLutSize);
  __shared__ int s_ci;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = c.n;
  const int nBig = min(c.counters[0], comp_cap_big(n));
  const int nSmall = min(c.counters[5], c.max_chains);   // class W
  // a CTA that can get neither a BIG component nor (as one of its warps) a small one has nothing to do
  if ((int)blockIdx.x >= nBig && (int)blockIdx.x * kWalkWarps >= nSmall) return;
  for (int i = tid; i < kLutSize / 4; i += kWalkThreads)
    reinterpret_cast<unsigned *>(lut)[i] = reinterpret_cast<const unsigned *>(g_walk_lut)[i];
  const unsigned lut_addr = (unsigned)__cvta_generic_to_shared(lut);
  // ---- phase 1
  while (true) {
    __syncthreads();   // the previous component's walk is finished (and the table is in place)
    if (tid == 0) s_ci = nBig > 0 ? atomicAdd(c.counters + 1, 1) : 0x7fffffff;
    __syncthreads();
    const int q = s_ci;
    if (q >= nBig) break;
    const int root = comp_root[q];
    const int y0 = root / w, y1 = c.bbox[root];
    const int g0 = c.bbox[n + root] >> 5, g1 = c.bbox[2 * n + root] >> 5;
    const int groups = g1 - g0 + 1, bh = y1 - y0 + 1, ws = groups + 2;
    for (int i = tid; i < (bh + 2 * kPadRows) * ws; i += kWalkThreads) arena[i] = 0;
    __syncthreads();
    walk_gather(c, arena, root, y0, g0, groups, bh, ws, warp, kWalkWarps, lane);
    __syncthreads();
    if (warp == 0) walk_component(c, arena, lut_addr, root, y0, g0, groups, bh, ws, lane);
  }
  // ---- phase 2
  unsigned *bm = arena + warp * kSliceWords;
  while (true) {
    int q = 0;
    if (lane == 0) q = atomicAdd(c.counters + 7, 1);
    q = __shfl_sync(0xffffffffu, q, 0);
    if (q >= nSmall) break;
    const int root = comp_root[comp_cap_big(n) + q];
    const int y0 = root / w, y1 = c.bbox[root];
    const int g0 = c.bbox[n + root] >> 5, g1 = c.bbox[2 * n + root] >> 5;
    const int groups = g1 - g0 + 1, bh = y1 - y0 + 1, ws = groups + 2;
    for (int i = lane; i < (bh + 2 * kPadRows) * ws; i += 32) bm[i] = 0;
    __syncwarp();
    walk_gather(c, bm, root, y0, g0, groups, bh, ws, 0, 1, lane);
    __syncwarp();
    walk_component(c, bm, lut_addr, root, y0, g0, groups, bh, ws, lane);
    __syncwarp();
  }
}

// Class T: one thread per component.  The component's bit map is one 64-bit word per row (bit b of row r = pixel
// (xmin - 1 + b, y0 - 1 + r): a zero column on either side, a zero row above and below), rows of the CTA's threads interleaved in
// shared memory.  The step is getPointChain through the same two tables as the warp walk — 3 x 3 neighbourhood -> key ->
// decision, (step, direction, neighbour) -> direction — on three row words, so the chains are the same; seeds are the lowest set
// bit of the first non-empty row (raster order).  No ballots, no warp synchronisation: a lane's walk touches only its own words.
template <class B>
__global__ void __launch_bounds__(kTLanes)
    k_fld_walk_thread(const __grid_constant__ B b, int w, int h, int length_threshold) {
  const FldBuffers &fb = b.fld_of(blockIdx.y);
  const unsigned *__restrict__ edges = fb.edges;
  const int words_per_row = fb.words_per_row;
  const int *__restrict__ label = fb.label, *__restrict__ cnt = fb.cnt, *__restrict__ bbox = fb.bbox;
  int *__restrict__ counters = fb.counters;
  int2 *__restrict__ chain_pts = fb.chain_pts;
  const int max_chains = fb.max_chains;
  const int n = w * h;
  __shared__ __align__(16) uint8_t lut[kLutSize];
  __shared__ unsigned long long bm[kTRows * kTLanes];
  const int tid = threadIdx.x;
  const int nT = min(counters[6], max_chains);
  if ((int)blockIdx.x * kTLanes >= nT) return;   // more walkers than components
  for (int i = tid; i < kLutSize / 4; i += kTLanes) reinterpret_cast<unsigned *>(lut)[i] = reinterpret_cast<const unsigned *>(g_walk_lut)[i];
  __syncthreads();
  const int *__restrict__ queue = fb.comp_root + comp_cap_big(n) + max_chains;
  unsigned long long *row = bm + tid;   // row r of this thread: row[r * kTLanes]
  while (true) {
    const int q = atomicAdd(counters + 8, 1);
    if (q >= nT) break;
    const int root = queue[q];
    const int y0 = root / w, y1 = bbox[root], xmin = bbox[n + root], xmax = bbox[2 * n + root];
    const int bh = y1 - y0 + 1, bw = xmax - xmin + 1;
    // ---- gather: the component's pixels of every row of the bounding box (edge bits whose label leads to this root)
    row[0] = 0ull;
    row[(bh + 1) * kTLanes] = 0ull;
    const int w0 = xmin >> 5, sh = xmin & 31;
    const unsigned long long wmask = (bw >= 64 ? ~0ull : ((1ull << bw) - 1ull));
    for (int r = 0; r < bh; r++) {
      const unsigned *er = edges + (size_t)(y0 + r) * words_per_row;
      const unsigned e0 = er[w0], e1 = w0 + 1 < words_per_row ? er[w0 + 1] : 0u, e2 = w0 + 2 < words_per_row ? er[w0 + 2] : 0u;
      unsigned long long v = ((unsigned long long)e0 | ((unsigned long long)e1 << 32)) >> sh;
      if (sh) v |= (unsigned long long)e2 << (64 - sh);
      v &= wmask;
      unsigned long long mine = 0ull;
      const int base = (y0 + r) * w + xmin;
      while (v) {
        const int bpos = __ffsll((long long)v) - 1;
        v &= v - 1;
        int l = label[base + bpos];
        if (l != root) l = label[l];   // tile-local root -> global root
        if (l == root) mine |= 1ull << bpos;
      }
      row[(r + 1) * kTLanes] = mine << 1;
    }
    // ---- walk
    int npts = atomicAdd(counters + 2, cnt[root]);   // this component's slice of the chain-point pool
    const int xorg = xmin - 1, yorg = y0 - 1;
    int sy = 1;
    bool in_chain = false;
    int cy = 0, cx = 0, start = 0, seed = 0, step = 0;
    unsigned dsel = 0;
    const uint8_t *tb = lut;
    while (true) {
      if (!in_chain) {
        if (sy > bh) break;
        const unsigned long long R = row[sy * kTLanes];
        if (R == 0ull) {
          sy++;
          continue;
        }
        cx = __ffsll((long long)R) - 1;
        cy = sy;
        row[sy * kTLanes] = R & ~(1ull << cx);   // the seed is consumed
        start = npts;
        seed = (yorg + cy) * w + xorg + cx;
        step = 0;
        dsel = 0;
        tb = lut + kKeys * 8;   // first-step half of the table
        in_chain = true;
      }
      chain_pts[npts++] = make_int2(xorg + cx, yorg + cy);
      const unsigned long long Ra = row[(cy - 1) * kTLanes], Rc = row[cy * kTLanes], Rb = row[(cy + 1) * kTLanes];
      const unsigned t3 = (unsigned)(Ra >> (cx - 1)) & 7u, c3 = (unsigned)(Rc >> (cx - 1)) & 7u, b3 = (unsigned)(Rb >> (cx - 1)) & 7u;
      const unsigned key = t3 | ((c3 & 1u) << 3) | ((c3 >> 2) << 4) | (b3 << 5);
      const unsigned e = tb[key * 8u + dsel];
      const unsigned i = e & 15u;
      if (i == 8u) {   // the chain ends here
        if (npts - start < length_threshold + 1) {
          npts = start;   // too short: dropped (its pixels stay consumed)
        } else {
          const int k = atomicAdd(counters + 3, 1);
          if (k < max_chains) {
            fb.chain_seed[k] = seed;
            fb.chain_off[k] = start;
            fb.chain_len[k] = npts - start;
          }
        }
        in_chain = false;
        continue;
      }
      dsel = lut[kLut1 + ((unsigned)min(step, 7) * 8u + dsel) * 8u + i];
      step++;
      tb = lut;
      const int dr = (int)((e >> 4) & 3u) - 1, dc = (int)((e >> 6) & 3u) - 1;
      cy += dr;
      cx += dc;
      const unsigned long long Rn = dr < 0 ? Ra : (dr > 0 ? Rb : Rc);
      row[cy * kTLanes] = Rn & ~(1ull << cx);   // the new pixel is consumed
    }
  }
}

// rank of every chain by the raster index of its seed (seeds are distinct pixels): order[rank] = chain
template <class B>
__global__ void k_fld_order(const __grid_constant__ B b) {
  const FldBuffers &fb = b.fld_of(blockIdx.y);
  const int *__restrict__ chain_seed = fb.chain_seed, *__restrict__ counters = fb.counters;
  int *__restrict__ order = fb.order;
  const int max_chains = fb.max_chains;
  const int n = min(counters[3], max_chains);
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n) return;
  const int mine = chain_seed[c];
  int rank = 0;
  for (int k = 0; k < n; k++) rank += chain_seed[k] < mine ? 1 : 0;
  order[rank] = c;
}

// --------------------------------------------------------------------------------- segments from chains
struct FitSums {
  double x, y, x2, y2, xy;
  int n;
};
__device__ __forceinline__ void fs_add(FitSums &s, int2 p) {
  float px = (float)p.x, py = (float)p.y;
  s.x += px; s.y += py;
  s.x2 += px * px; s.y2 += py * py; s.xy += px * py;
  s.n++;
}
// cv::fitLine(.., DIST_L2, 0, 0.01, 0.01) == fitLine2D_wods, then the homogeneous line through (x0,y0),(x0+vx,y0+vy)
__device__ __forceinline__ void fs_line(const FitSums &s, double l[3]) {
  double w = (float)s.n;
  double x = s.x / w, y = s.y / w, x2 = s.x2 / w, y2 = s.y2 / w, xy = s.xy / w;
  double dx2 = x2 - x * x, dy2 = y2 - y * y, dxy = xy - x * y;
  float t = (float)atan2(2 * dxy, dx2 - dy2) / 2;
  float l0 = cosf(t), l1 = sinf(t), l2 = (float)x, l3 = (float)y;
  double a[3] = {l2, l3, 1.0};
  double b[3] = {(double)(l2 + l0), (double)(l3 + l1), 1.0};
  l[0] = a[1] * b[2] - a[2] * b[1];
  l[1] = a[2] * b[0] - a[0] * b[2];
  l[2] = a[0] * b[1] - a[1] * b[0];
}
// distPointLine of the reference normalises the line IN PLACE on every call.  After the first call the norm is 1 up to
// rounding; when x * x + y * y is exactly 1.0 the square root is exactly 1 and the three divisions are identities, so
// they are skipped (bit-exact shortcut: a double-precision sqrt and three divisions per chain point otherwise).
__device__ __forceinline__ double dist_point_line(double px, double py, double l[3]) {
  double x = l[0], y = l[1];
  double n2 = x * x + y * y;
  if (n2 != 1.0) {
    double w = sqrt(n2);
    l[0] = x / w; l[1] = y / w; l[2] = l[2] / w;
  }
  return l[0] * px + l[1] * py + l[2];
}
__device__ __forceinline__ void incident_point(const double l[3], float &px, float &py, int W, int H) {
  double a[3] = {(double)px, (double)py, 1.0};
  double b[3] = {l[0], l[1], 0.0};
  double lk[3] = {a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]};
  double xk[3] = {lk[1] * l[2] - lk[2] * l[1], lk[2] * l[0] - lk[0] * l[2], lk[0] * l[1] - lk[1] * l[0]};
  double alpha = 1.0 / xk[2];
  float fx = (float)(xk[0] * alpha), fy = (float)(xk[1] * alpha);
  px = fx < 0.0f ? 0.0f : (fx >= (W - 1.0f) ? (W - 1.0f) : fx);
  py = fy < 0.0f ? 0.0f : (fy >= (H - 1.0f) ? (H - 1.0f) : fy);
}

// one thread per chain, in seed order; chain c writes its segments to slots chain_off[c] / 21 + j (collision free:
// every segment consumes at least 21 chain points and the chains' point ranges are disjoint)
template <class B>
__global__ void k_fld_segments(const __grid_constant__ B b, int T, float dist_thr) {
  const FldBuffers &fb = b.fld_of(blockIdx.y);
  const uint8_t *__restrict__ img = b.half_of(blockIdx.y).p;
  const int W = b.half_of(blockIdx.y).w, H = b.half_of(blockIdx.y).h, pitch = b.half_of(blockIdx.y).pitch;
  const int2 *__restrict__ chain_pts = fb.chain_pts;
  const int *__restrict__ chain_off = fb.chain_off, *__restrict__ chain_len = fb.chain_len, *__restrict__ order = fb.order;
  const int *__restrict__ counters = fb.counters;
  const int max_chains = fb.max_chains;
  float4 *__restrict__ segs = fb.segs;
  int *__restrict__ seg_cnt = fb.seg_cnt, *__restrict__ seg_base = fb.seg_cnt + fb.max_chains;
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= min(counters[3], max_chains)) return;
  const int c = order[r];
  const int2 *points = chain_pts + chain_off[c];
  const int total = chain_len[c];
  const int slot0 = chain_off[c] / kSegsPerChainDiv;
  int nseg = 0;
  int i, j;
  for (i = 0; i + T < total; i++) {
    int2 ps = points[i], pe = points[i + T];
    double l[3] = {(double)ps.y - (double)pe.y, (double)pe.x - (double)ps.x,
                   (double)ps.x * (double)pe.y - (double)ps.y * (double)pe.x};
    bool is_line = true;
    FitSums fs = {0, 0, 0, 0, 0, 0};
    fs_add(fs, ps);
    for (j = 1; j < T; j++) {
      int2 pt = points[i + j];
      double dist = dist_point_line((double)pt.x, (double)pt.y, l);
      if (fabs(dist) > dist_thr) { is_line = false; break; }
      fs_add(fs, pt);
    }
    if (!is_line) continue;
    fs_add(fs, pe);
    fs_line(fs, l);
    {  // incidentPoint(l, ps) on the INTEGER point: result rounded (cv::Point2i(Point2f) == cvRound)
      float fx = (float)ps.x, fy = (float)ps.y;
      incident_point(l, fx, fy, W, H);
      ps.x = __float2int_rn(fx);
      ps.y = __float2int_rn(fy);
    }
    for (j = T + 1; i + j < total; j++) {
      int2 pt = points[i + j];
      double dist = dist_point_line((double)pt.x, (double)pt.y, l);
      if (fabs(dist) > dist_thr) {
        fs_line(fs, l);
        dist = dist_point_line((double)pt.x, (double)pt.y, l);
        if (fabs(dist) > dist_thr) { j--; break; }
      }
      pe = pt;
      fs_add(fs, pt);
    }
    fs_line(fs, l);
    float e1x = (float)ps.x, e1y = (float)ps.y, e2x = (float)pe.x, e2y = (float)pe.y;
    incident_point(l, e1x, e1y, W, H);
    incident_point(l, e2x, e2y, W, H);
    i = i + j;
    // ---- per-segment filters of lineDetection
    float len = sqrtf((e1x - e2x) * (e1x - e2x) + (e1y - e2y) * (e1y - e2y));
    if (len < (float)T) continue;
    if ((e1x <= 5.0f && e2x <= 5.0f) || (e1y <= 5.0f && e2y <= 5.0f) || (e1x >= W - 5.0f && e2x >= W - 5.0f) ||
        (e1y >= H - 5.0f && e2y >= H - 5.0f))
      continue;
    // ---- additionalOperationsOnSegment: orient by the brighter side
    if (!(e1x == 0.0f && e2x == 0.0f && e1y == 0.0f && e2y == 0.0f)) {
      double ang = atan2((double)(e2y - e1y), (double)(e2x - e1x));
      double dx = (double)e2x - (double)e1x, dy = (double)e2y - (double)e1y;
      const double kPi = 3.1415926535897932384626433832795;
      double cs = cos(90.0 * kPi / 180.0 + ang), sn = sin(90.0 * kPi / 180.0 + ang);
      int iR = 0, iL = 0;
      for (int k = 0; k < 10; k++) {
        float qx, qy;
        if (k == 0) { qx = e1x; qy = e1y; }
        else if (k == 9) { qx = e2x; qy = e2y; }
        else {
          qx = e1x + ((float)dx / 9.0f * (float)k);
          qy = e1y + ((float)dy / 9.0f * (float)k);
        }
        int rx = __double2int_rn(qx + cs), ry = __double2int_rn(qy + sn);
        int lx = __double2int_rn(qx - cs), ly = __double2int_rn(qy - sn);
        rx = min(max(rx, 0), W - 1); ry = min(max(ry, 0), H - 1);
        lx = min(max(lx, 0), W - 1); ly = min(max(ly, 0), H - 1);
        iR += img[(size_t)ry * pitch + rx];
        iL += img[(size_t)ly * pitch + lx];
      }
      if (iR > iL) {
        float tx = e1x, ty = e1y;
        e1x = e2x; e1y = e2y; e2x = tx; e2y = ty;
      }
    }
    segs[slot0 + nseg] = make_float4(e1x, e1y, e2x, e2y);
    nseg++;
  }
  seg_cnt[r] = nseg;      // indexed by RANK so the compaction below walks chains in seed order
  seg_base[r] = slot0;
}

// ordered compaction of the per-chain segment slots (one block)
template <class B>
__global__ void __launch_bounds__(256)
    k_fld_compact(const __grid_constant__ B b) {
  const FldBuffers &fb = b.fld_of(blockIdx.y);
  const float4 *__restrict__ segs = fb.segs;
  const int *__restrict__ seg_cnt = fb.seg_cnt, *__restrict__ seg_base = fb.seg_cnt + fb.max_chains;
  int *__restrict__ counters = fb.counters;
  const int max_chains = fb.max_chains, out_cap = fb.out_cap;
  float4 *__restrict__ out = fb.out;
  __shared__ int warp_tot[8];
  __shared__ int s_running;
  const int n = min(counters[3], max_chains);
  const int tid = threadIdx.x;
  if (tid == 0) s_running = 0;
  __syncthreads();
  for (int base = 0; base < n; base += 256) {
    int c = base + tid;
    int cnt = c < n ? seg_cnt[c] : 0;
    int v = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      int t = __shfl_up_sync(0xffffffffu, v, d);
      if ((tid & 31) >= d) v += t;
    }
    if ((tid & 31) == 31) warp_tot[tid >> 5] = v;
    __syncthreads();
    int off = s_running;
    for (int k = 0; k < (tid >> 5); k++) off += warp_tot[k];
    off += v - cnt;
    for (int k = 0; k < cnt; k++)
      if (off + k < out_cap) out[off + k] = segs[seg_base[c] + k];
    __syncthreads();
    if (tid == 255) s_running = off + cnt;
    __syncthreads();
  }
  if (tid == 0) counters[4] = s_running;
}

int FldBuffers::alloc(int w, int h, int length_threshold, int out_capacity) {
  const size_t n = (size_t)w * h;
  words_per_row = (w + 31) / 32;
  max_chains = (int)(n / (length_threshold + 1)) + 1;
  out_cap = out_capacity;
  bool ok = true;
  auto A = [&](auto **p, size_t bytes) { ok = ok && cudaMalloc((void **)p, bytes) == cudaSuccess; };
  A(&edges, (size_t)words_per_row * h * sizeof(unsigned));
  A(&label, (n + 32) * sizeof(int));   // slack: the walk gathers labels with 16-byte loads
  A(&cnt, n * sizeof(int));
  A(&bbox, 3 * n * sizeof(int));
  A(&comp_root, (size_t)(2 * max_chains + comp_cap_big((int)n)) * sizeof(int));
  A(&counters, 12 * sizeof(int));
  lroot_cap = (int)(n / 4 + 1);
  A(&lroots, (size_t)lroot_cap * sizeof(int));
  A(&lroot_n, sizeof(int));
  A(&chain_pts, n * sizeof(int2));
  A(&chain_seed, (size_t)max_chains * sizeof(int));
  A(&chain_off, (size_t)max_chains * sizeof(int));
  A(&chain_len, (size_t)max_chains * sizeof(int));
  A(&order, (size_t)max_chains * sizeof(int));
  A(&segs, (n / kSegsPerChainDiv + 2) * sizeof(float4));
  A(&seg_cnt, (size_t)2 * max_chains * sizeof(int));
  A(&out, (size_t)out_cap * sizeof(float4));
  if (ok) ok = cudaMemset(counters, 0, 12 * sizeof(int)) == cudaSuccess;
  return ok ? 0 : 1;
}

void FldBuffers::release() {
  cudaFree(lroots); cudaFree(lroot_n);
  cudaFree(edges); cudaFree(label); cudaFree(cnt); cudaFree(bbox); cudaFree(comp_root); cudaFree(counters);
  cudaFree(chain_pts); cudaFree(chain_seed); cudaFree(chain_off); cudaFree(chain_len); cudaFree(order);
  cudaFree(segs); cudaFree(seg_cnt); cudaFree(out);
  *this = FldBuffers();
}

template <class B>
static void launch_fld_any(const B &b, int nb_frames, int w, int h, int max_chains, int length_threshold, float distance_threshold,
                           cudaStream_t s, cudaEvent_t *ev) {
  const int n = w * h;
  const int tpb = 256;
  const int lroot_cap = n / 4 + 1;
  if constexpr (!kFusedLabels<B>) {
    PLVIWO_CARVEOUT(k_ccl_reset<B>);
    k_ccl_reset<B><<<nb_frames, 32, 0, s>>>(b);
    PLVIWO_CARVEOUT(k_ccl_tile<B>);
    k_ccl_tile<B><<<dim3((w + kTileW - 1) / kTileW, (h + kTileH - 1) / kTileH, nb_frames), kTileThreads, 0, s>>>(b, w, h);
  }
  const int nborder = ((h - 1) / kTileH) * w + ((w - 1) / kTileW) * h;
  if (nborder > 0) {
    PLVIWO_CARVEOUT(k_ccl_border<B>);
    k_ccl_border<B><<<dim3((nborder + tpb - 1) / tpb, nb_frames), tpb, 0, s>>>(b, w, h);
  }
  // tile-local roots are a few thousand per frame (capacity n / 4): a fixed small grid strides over the list.  There is no
  // flatten pass: a pixel's label is its tile-local root and that root's label is the global root, which is all the walk's
  // gather needs (two loads for the pixels of the components that are walked instead of a pass over every edge pixel)
  const int root_ctas = std::max(1, std::min((lroot_cap + tpb - 1) / tpb, 12));
  PLVIWO_CARVEOUT(k_ccl_link<B>);
  k_ccl_link<B><<<dim3(root_ctas, nb_frames), tpb, 0, s>>>(b, w, h);
  PLVIWO_CARVEOUT(k_ccl_roots<B>);
  // class T (one thread per small component, a launch of its own ahead of the warp walk) pays when launches carry many frames
  // (a stream group: 32-256 per launch); one frame, or the few frames a single handle batches, are about latency — there
  // everything that is not BIG goes to the warps of the one walk launch (measured: one pipelined stream 12.7 k frames/s
  // without the extra launch, 11.6 k with it)
  // PLVIWO_WALK_THREAD_MIN = frames per launch from which class T is used (read at every launch: the tests switch it)
  const char *tmin_env = std::getenv("PLVIWO_WALK_THREAD_MIN");
  const int thread_class = nb_frames >= (tmin_env ? std::max(1, std::atoi(tmin_env)) : 16) ? 1 : 0;
  k_ccl_roots<B><<<dim3(root_ctas, nb_frames), tpb, 0, s>>>(b, w, h, length_threshold + 1, thread_class);
  if (ev) cudaEventRecord(ev[0], s);
  init_fld_constants();
  const int ws = ((w + 31) >> 5) + 2;
  const size_t arena_words = std::max<size_t>((size_t)(h + 2 * kPadRows) * ws, (size_t)kWalkWarps * kSliceWords);
  size_t smem = (size_t)kLutSize + arena_words * sizeof(unsigned);
  static SmemOptIn optin;
  optin.ensure(k_fld_walk_cc<B>, smem);
  // Walkers per frame: components are pulled from atomic queues (BIG ones by whole CTAs, the rest by single warps), the
  // launch lasts as long as its longest component; a batch of frames shares one launch (grid.y = frame).
  static const int walk_ctas_env = [] {
    const char *e = std::getenv("PLVIWO_WALK_CTAS");
    return e ? std::atoi(e) : 0;
  }();
  // A walker CTA holds 30 KB of shared memory for as long as its components last (milliseconds for the few long ones): in a
  // launch over many frames the walkers are kept scarce (256 per launch, < 2 per SM) so that the other kernels of the
  // pipeline — other streams, other ticks — stay resident beside them; the walk's WORK is small, its duration is the
  // latency of the longest component either way.
  const int walk_ctas = walk_ctas_env > 0 ? walk_ctas_env : (nb_frames > 1 ? std::max(2, std::min(74, 256 / nb_frames)) : 148);
  // class T first: a short launch (its longest component has a few hundred pixels), one thread per component
  const int walk_t = 4;   // CTAs of kTLanes threads per frame (about 250 class-T components per frame)
  if (thread_class) {
    PLVIWO_CARVEOUT(k_fld_walk_thread<B>);
    k_fld_walk_thread<B><<<dim3(walk_t, nb_frames), kTLanes, 0, s>>>(b, w, h, length_threshold);
  }
  PLVIWO_CARVEOUT(k_fld_walk_cc<B>);
  k_fld_walk_cc<B><<<dim3(walk_ctas, nb_frames), kWalkThreads, smem, s>>>(b, w, h, length_threshold);
  if (ev) cudaEventRecord(ev[1], s);
  PLVIWO_CARVEOUT(k_fld_order<B>);
  k_fld_order<B><<<dim3((max_chains + 127) / 128, nb_frames), 128, 0, s>>>(b);
  PLVIWO_CARVEOUT(k_fld_segments<B>);
  k_fld_segments<B><<<dim3((max_chains + 63) / 64, nb_frames), 64, 0, s>>>(b, length_threshold, distance_threshold);
  PLVIWO_CARVEOUT(k_fld_compact<B>);
  k_fld_compact<B><<<dim3(1, nb_frames), 256, 0, s>>>(b);
}
void launch_fld_batch(const FldBatch &b, int length_threshold, float distance_threshold, cudaStream_t s, cudaEvent_t *ev) {
  launch_fld_any(b, b.n, b.half[0].w, b.half[0].h, b.f[0].max_chains, length_threshold, distance_threshold, s, ev);
}
void launch_fld_table(const SlotRec *slots, const int *line_slots, int n_jobs, int w, int h, int max_chains, int length_threshold,
                      float distance_threshold, cudaStream_t s, cudaEvent_t *ev) {
  if (n_jobs <= 0) return;
  launch_fld_any(FldTable{slots, line_slots}, n_jobs, w, h, max_chains, length_threshold, distance_threshold, s, ev);
}

void launch_fld(const DevImage &half, int length_threshold, float distance_threshold, FldBuffers &fb, cudaStream_t s,
                cudaEvent_t *ev) {
  FldBatch b;
  b.n = 1;
  b.half[0] = half;
  b.f[0] = fb;
  launch_fld_batch(b, length_threshold, distance_threshold, s, ev);
}

}  // namespace plviwo
