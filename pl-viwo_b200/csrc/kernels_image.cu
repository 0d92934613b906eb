// Image-domain kernels of the front end (sm_100a): histogram, equalise + pyramid level 1 + half-resolution
// image in one pass, and the remaining pyramid levels in one launch.
//
// Reference ops replaced (all are OpenCV calls made by the reference; arithmetic per SURVEY.md Appendix A):
//   cv::equalizeHist                    TrackKLT.cpp:59, TrackLSD.cpp:83   (A1)  -> k_hist + k_eq_pyr1 (LUT)
//   cv::buildOpticalFlowPyramid         TrackKLT.cpp:71                    (A2)  -> k_eq_pyr1 (level 1) + k_pyr_rest
//   cv::resize(.., 0.5, 0.5, LINEAR)    TrackLSD.cpp:204                   (A7)  -> k_eq_pyr1 (half)
// The reference equalises the same frame twice (point and line tracker) and materialises Scharr derivative
// planes with a 15 px border; here the frame is read once, the equalised image is written once and shared,
// and derivatives are formed on the fly inside the LK kernel.
#include "fe_kernels.h"

#include <cstdlib>
#include "tma_bulk.h"

namespace plviwo {

__device__ __forceinline__ int reflect101(int i, int n) {
  // BORDER_REFLECT_101, valid for -n < i < 2n - 1
  if (i < 0) i = -i;
  if (i >= n) i = 2 * n - 2 - i;
  return i;
}

// ------------------------------------------------------------------------------------------------ histogram
// Each thread walks 16-byte chunks (uint4 = 16 pixels), four loads in flight per thread: a pass over a frame is a pure
// streaming read and one outstanding 16-byte load per thread (32 warps per SM) covers only half of bandwidth x latency.
// Per-warp shared sub-histograms keep shared-memory atomics off a single copy, one global atomic per non-empty bin per
// CTA at the end.  (Four bank-interleaved copies per warp were tried and measured slower: 2.1 vs 2.4 TB/s.)
constexpr int kHistThreads = 256;
constexpr int kHistWarps = kHistThreads / 32;
constexpr int kHistUnroll = 4;

__device__ __forceinline__ void hist_add16(unsigned *my, const uint4 &v) {
  const unsigned wds[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int k = 0; k < 4; k++) {
    atomicAdd(&my[wds[k] & 0xff], 1u);
    atomicAdd(&my[(wds[k] >> 8) & 0xff], 1u);
    atomicAdd(&my[(wds[k] >> 16) & 0xff], 1u);
    atomicAdd(&my[wds[k] >> 24], 1u);
  }
}

// The frame's 256-byte cv::equalizeHist LUT (Appendix A1) from its complete histogram, one bin per thread.
__device__ __forceinline__ void equalize_lut(const unsigned *__restrict__ hist, unsigned total, uint8_t *__restrict__ lut) {
  __shared__ unsigned warp_tot[kHistWarps];
  __shared__ int s_i0;
  __shared__ unsigned s_h0;
  const int tid = threadIdx.x;
  if (tid == 0) s_i0 = 256;
  __syncthreads();
  const unsigned hv = __ldcg(hist + tid);   // other CTAs' atomics: read at L2
  if (hv) atomicMin(&s_i0, tid);
  // inclusive scan over 256 bins
  unsigned v = hv;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    unsigned t = __shfl_up_sync(0xffffffffu, v, d);
    if ((tid & 31) >= d) v += t;
  }
  if ((tid & 31) == 31) warp_tot[tid >> 5] = v;
  __syncthreads();
  unsigned base = 0;
  for (int k = 0; k < (tid >> 5); k++) base += warp_tot[k];
  const unsigned cum = v + base;  // sum hist[0..tid]
  const int i0 = s_i0;
  if (tid == i0) s_h0 = hv;
  __syncthreads();
  const unsigned hist0 = s_h0;
  uint8_t out;
  if (hist0 == total) {
    out = (uint8_t)i0;  // single-valued image: dst.setTo(i0)
  } else if (tid <= i0) {
    out = 0;
  } else {
    float scale = __fdiv_rn(255.f, (float)(total - hist0));
    int sum = (int)(cum - hist0);  // bins i0+1..tid (bins below i0 are empty)
    int r = __float2int_rn(__fmul_rn((float)sum, scale));
    out = (uint8_t)min(max(r, 0), 255);
  }
  lut[tid] = out;
}

// hist (zero on entry) accumulates the frame; the last of the n_blocks CTAs to finish (counter: zero on entry) turns it into
// the LUT and leaves hist and counter zeroed for the next frame.  k_eq_pyr1 then only loads the 256 bytes.
__device__ __forceinline__ void hist_body(const uint8_t *__restrict__ src, int w, int h, int pitch, unsigned *__restrict__ hist,
                                          unsigned *__restrict__ counter, uint8_t *__restrict__ lut, int block, int n_blocks) {
  static_assert(kHistThreads == 256, "one LUT bin per thread");
  __shared__ unsigned sh[kHistWarps][256];
  __shared__ unsigned s_last;
  for (int i = threadIdx.x; i < kHistWarps * 256; i += kHistThreads) (&sh[0][0])[i] = 0;
  __syncthreads();
  unsigned *my = sh[threadIdx.x >> 5];
  const int chunks_per_row = (w + 15) >> 4;
  const int total = chunks_per_row * h;
  const int stride = n_blocks * kHistThreads;
  const bool full_rows = (w & 15) == 0 && (pitch & 15) == 0 && ((size_t)src & 15) == 0;   // every chunk is a whole, aligned uint4
  int c = block * kHistThreads + threadIdx.x;
  if (full_rows) {
    for (; c + (kHistUnroll - 1) * stride < total; c += kHistUnroll * stride) {
      uint4 v[kHistUnroll];
#pragma unroll
      for (int u = 0; u < kHistUnroll; u++) {
        const int cu = c + u * stride;
        const int y = cu / chunks_per_row;
        v[u] = __ldg(reinterpret_cast<const uint4 *>(src + (size_t)y * pitch + ((cu - y * chunks_per_row) << 4)));
      }
#pragma unroll
      for (int u = 0; u < kHistUnroll; u++) hist_add16(my, v[u]);
    }
  }
  for (; c < total; c += stride) {
    int y = c / chunks_per_row;
    int x = (c - y * chunks_per_row) << 4;
    const uint8_t *row = src + (size_t)y * pitch + x;
    if (x + 16 <= w && ((size_t)row & 15) == 0) {
      hist_add16(my, *reinterpret_cast<const uint4 *>(row));
    } else {
      for (int k = 0; x + k < w; k++) atomicAdd(&my[row[k]], 1u);
    }
  }
  __syncthreads();
  for (int b = threadIdx.x; b < 256; b += kHistThreads) {
    unsigned s = 0;
#pragma unroll
    for (int k = 0; k < kHistWarps; k++) s += sh[k][b];
    if (s) atomicAdd(&hist[b], s);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    s_last = (atomicAdd(counter, 1u) == (unsigned)n_blocks - 1) ? 1u : 0u;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  equalize_lut(hist, (unsigned)w * (unsigned)h, lut);
  hist[threadIdx.x] = 0;
  if (threadIdx.x == 0) *counter = 0;
}

__global__ void __launch_bounds__(kHistThreads) k_hist(const uint8_t *__restrict__ src, int w, int h, int pitch,
                                                       unsigned *__restrict__ hist, unsigned *__restrict__ counter,
                                                       uint8_t *__restrict__ lut) {
  hist_body(src, w, h, pitch, hist, counter, lut, blockIdx.x, gridDim.x);
}

// grid.z = job.  Block 0 of a job also publishes the frame's flags and zeroes the FAST counters of its slot (every later
// kernel of the frame is ordered after this one on the same stream).
__global__ void __launch_bounds__(kHistThreads)
    k_hist_b(const SlotRec *__restrict__ slots, const FrontJob *__restrict__ jobs, int w, int h, int *__restrict__ slot_flags) {
  const FrontJob job = jobs[blockIdx.z];
  const SlotRec &sl = slots[job.slot];
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    slot_flags[job.slot] = job.flags;
    sl.fast_total[0] = 0;
    sl.fast_total[1] = 0;
  }
  if (job.eq_mode != 1) return;
  hist_body(job.src, w, h, job.src_pitch, sl.hist, sl.counters, sl.eq_lut, blockIdx.x, gridDim.x);
}

void launch_hist_batch(const SlotRec *slots, const FrontJob *jobs, int n_jobs, const FrontGeom &g, int *slot_flags, cudaStream_t s) {
  if (n_jobs <= 0) return;
  const int chunks = ((g.w + 15) >> 4) * g.h;
  int grid = (chunks + kHistThreads * 4 - 1) / (kHistThreads * 4);   // one unrolled round of 4 chunks per thread
  if (grid < 1) grid = 1;
  PLVIWO_CARVEOUT(k_hist_b);
  k_hist_b<<<dim3(grid, 1, n_jobs), kHistThreads, 0, s>>>(slots, jobs, g.w, g.h, slot_flags);
}

void launch_hist(const DevImage &src, unsigned *d_hist, unsigned *d_counter, uint8_t *d_lut, cudaStream_t s) {
  int chunks = ((src.w + 15) >> 4) * src.h;
  int grid = (chunks + kHistThreads * 2 - 1) / (kHistThreads * 2);  // ~2 chunks per thread for one frame
  if (grid < 1) grid = 1;
  if (grid > 148 * 8) grid = 148 * 8;                               // 8 KB of shared memory per CTA: 8 CTAs per SM
  PLVIWO_CARVEOUT(k_hist);
  k_hist<<<grid, kHistThreads, 0, s>>>(src.p, src.w, src.h, src.pitch, d_hist, d_counter, d_lut);
}

// ------------------------------------------------------------------------------------------------ CLAHE
// cv::createCLAHE(10.0, Size(8, 8))->apply (TrackKLT.cpp:60-64, TrackLSD.cpp:84-88).  Arithmetic of OpenCV's clahe.cpp:
// the frame is extended to a multiple of the tile grid with BORDER_REFLECT_101 (both directions, even when only one is
// not divisible), per tile a 256-bin histogram is clipped at clipLimit * area / 256 (>= 1), the excess is spread evenly
// (the remainder one count every 256 / remainder bins), the LUT is cvRound(cumsum * (255 / area)) in float32; the output
// pixel blends the LUTs of the 4 nearest tile centres bilinearly, float32, in the order
// (l11 * xa1 + l12 * xa) * ya1 + (l21 * xa1 + l22 * xa) * ya.  The blend is part of k_eq_pyr1's staging; this kernel
// builds the tile LUTs: one CTA per tile.
struct ClaheGeom {
  int tiles_x, tiles_y, tile_w, tile_h, clip;
  float lut_scale, inv_tw, inv_th;
};

__device__ __forceinline__ void clahe_lut_body(const uint8_t *__restrict__ src, int w, int h, int pitch, const ClaheGeom &g,
                                               uint8_t *__restrict__ luts) {
  __shared__ unsigned sh[8][256];
  __shared__ unsigned warp_tot[8];
  __shared__ unsigned s_clipped;
  const int tid = threadIdx.x;
  const int tx = blockIdx.x % g.tiles_x, ty = blockIdx.x / g.tiles_x;
  for (int i = tid; i < 8 * 256; i += 256) (&sh[0][0])[i] = 0;
  if (tid == 0) s_clipped = 0;
  __syncthreads();
  unsigned *my = sh[tid >> 5];
  const int x0 = tx * g.tile_w, y0 = ty * g.tile_h;
  for (int i = tid; i < g.tile_w * g.tile_h; i += 256) {
    const int r = i / g.tile_w, c = i - r * g.tile_w;
    const int sx = reflect101(x0 + c, w), sy = reflect101(y0 + r, h);
    atomicAdd(&my[src[(size_t)sy * pitch + sx]], 1u);
  }
  __syncthreads();
  unsigned hv = 0;
#pragma unroll
  for (int k = 0; k < 8; k++) hv += sh[k][tid];
  // clip and redistribute
  const unsigned clip = (unsigned)g.clip;
  if (hv > clip) {
    atomicAdd(&s_clipped, hv - clip);
    hv = clip;
  }
  __syncthreads();
  const unsigned clipped = s_clipped;
  const unsigned batch = clipped / 256u, residual = clipped - batch * 256u;
  hv += batch;
  if (residual != 0) {
    const unsigned step = max(256u / residual, 1u);
    if ((unsigned)tid % step == 0 && (unsigned)tid / step < residual) hv += 1;
  }
  // inclusive scan over the 256 bins
  unsigned v = hv;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    unsigned t = __shfl_up_sync(0xffffffffu, v, d);
    if ((tid & 31) >= d) v += t;
  }
  if ((tid & 31) == 31) warp_tot[tid >> 5] = v;
  __syncthreads();
  unsigned base = 0;
  for (int k = 0; k < (tid >> 5); k++) base += warp_tot[k];
  const int r = __float2int_rn(__fmul_rn((float)(int)(v + base), g.lut_scale));
  luts[(size_t)blockIdx.x * 256 + tid] = (uint8_t)min(max(r, 0), 255);
}

__device__ __forceinline__ unsigned clahe_px(const uint8_t *__restrict__ luts, const ClaheGeom &g, int x, int y, int v) {
  const float txf = __fsub_rn(__fmul_rn((float)x, g.inv_tw), 0.5f), tyf = __fsub_rn(__fmul_rn((float)y, g.inv_th), 0.5f);
  int tx1 = __float2int_rd(txf), ty1 = __float2int_rd(tyf);
  const float xa = __fsub_rn(txf, (float)tx1), ya = __fsub_rn(tyf, (float)ty1);
  const float xa1 = __fsub_rn(1.f, xa), ya1 = __fsub_rn(1.f, ya);
  const int tx2 = min(tx1 + 1, g.tiles_x - 1), ty2 = min(ty1 + 1, g.tiles_y - 1);
  tx1 = max(tx1, 0);
  ty1 = max(ty1, 0);
  const float l11 = (float)__ldg(luts + ((ty1 * g.tiles_x + tx1) << 8) + v), l12 = (float)__ldg(luts + ((ty1 * g.tiles_x + tx2) << 8) + v);
  const float l21 = (float)__ldg(luts + ((ty2 * g.tiles_x + tx1) << 8) + v), l22 = (float)__ldg(luts + ((ty2 * g.tiles_x + tx2) << 8) + v);
  const float top = __fadd_rn(__fmul_rn(l11, xa1), __fmul_rn(l12, xa)), bot = __fadd_rn(__fmul_rn(l21, xa1), __fmul_rn(l22, xa));
  const int r = __float2int_rn(__fadd_rn(__fmul_rn(top, ya1), __fmul_rn(bot, ya)));
  return (unsigned)min(max(r, 0), 255);
}

__global__ void __launch_bounds__(256)
    k_clahe_lut(const uint8_t *__restrict__ src, int w, int h, int pitch, ClaheGeom g, uint8_t *__restrict__ luts) {
  clahe_lut_body(src, w, h, pitch, g, luts);
}
__global__ void __launch_bounds__(256)
    k_clahe_lut_b(const SlotRec *__restrict__ slots, const FrontJob *__restrict__ jobs, int w, int h, ClaheGeom g) {
  const FrontJob job = jobs[blockIdx.z];
  if (job.eq_mode != 2) return;
  clahe_lut_body(job.src, w, h, job.src_pitch, g, slots[job.slot].clahe);
}

static ClaheGeom clahe_geom(int w, int h) {
  ClaheGeom g;
  g.tiles_x = 8;
  g.tiles_y = 8;
  int ew = w, eh = h;
  if (w % 8 != 0 || h % 8 != 0) {
    ew = w + (8 - w % 8);
    eh = h + (8 - h % 8);
  }
  g.tile_w = ew / 8;
  g.tile_h = eh / 8;
  const int area = g.tile_w * g.tile_h;
  g.lut_scale = 255.f / (float)area;
  g.clip = (int)(10.0 * area / 256);
  if (g.clip < 1) g.clip = 1;
  g.inv_tw = 1.0f / (float)g.tile_w;
  g.inv_th = 1.0f / (float)g.tile_h;
  return g;
}

void launch_clahe_lut(const DevImage &src, uint8_t *d_luts, cudaStream_t s) {
  const ClaheGeom g = clahe_geom(src.w, src.h);
  PLVIWO_CARVEOUT(k_clahe_lut);
  k_clahe_lut<<<64, 256, 0, s>>>(src.p, src.w, src.h, src.pitch, g, d_luts);
}

void launch_clahe_lut_batch(const SlotRec *slots, const FrontJob *jobs, int n_jobs, const FrontGeom &g, cudaStream_t s) {
  if (n_jobs <= 0) return;
  PLVIWO_CARVEOUT(k_clahe_lut_b);
  k_clahe_lut_b<<<dim3(64, 1, n_jobs), 256, 0, s>>>(slots, jobs, g.w, g.h, clahe_geom(g.w, g.h));
}

// ------------------------------------------------------------------------- equalise + level 0/1 + half-res
// One CTA produces a 64 x 16 tile of level 1, i.e. consumes a (128 + 4) x (32 + 4) window of the raw frame
// (5-tap [1 4 6 4 1] pyrDown halo of 2), staged in shared memory AFTER the LUT so level 0, level 1 and the
// 2x2-mean half-resolution image all come from one read of the frame.
constexpr int kT1W = 64, kT1H = 16;            // level-1 tile
constexpr int kT0W = 2 * kT1W, kT0H = 2 * kT1H;  // level-0 interior of the tile
constexpr int kTileCols = kT0W + 8;            // staged columns: [2*tx0 - 4, 2*tx0 + 132), word aligned
constexpr int kTileRows = kT0H + 4;            // staged rows:    [2*ty0 - 2, 2*ty0 + 34)
constexpr int kEqThreads = 256;
// Interior tiles (no reflected row or column, the 16-byte aligned span inside the row) are staged by the TMA unit: one
// bulk copy per tile row of the span [2*tx0 - 16, 2*tx0 + 144), issued before the LUT is loaded so that the copy overlaps
// the load.  Border tiles take the per-thread path with BORDER_REFLECT_101.
constexpr int kBulkCols = kT0W + 32;           // 160 bytes per row
constexpr int kBulkLead = 12;                  // bulk column of tile column 0: (2*tx0 - 4) - (2*tx0 - 16)

// Packed 16-bit lanes.  A word of 4 consecutive pixels (b0 b1 b2 b3) splits into Ev = (b0, b2) and Od = (b1, b3), low lane
// first.  With pixel c0 at the first byte of wd[0], hpyr_words gives in hs[m] the [1 4 6 4 1] sums centred on pixels
// 4m + 4 and 4m + 6 (taps 4m + 2 .. 4m + 8): two horizontally adjacent pyrDown columns per word, each lane <= 16 * 255.
// Bytes c0, c1 and the last two of wd[N + 1] do not enter any sum.
template <int N>
__device__ __forceinline__ void hpyr_words(const unsigned (&wd)[N + 2], unsigned (&hs)[N]) {
  unsigned ev[N + 2], od[N + 1];
#pragma unroll
  for (int k = 0; k < N + 2; k++) ev[k] = __byte_perm(wd[k], 0, 0x4240);
#pragma unroll
  for (int k = 0; k < N + 1; k++) od[k] = __byte_perm(wd[k], 0, 0x4341);
#pragma unroll
  for (int m = 0; m < N; m++) {
    const unsigned e_m2 = __byte_perm(ev[m], ev[m + 1], 0x5432);       // pixels 4m + 2, 4m + 4
    const unsigned e_p2 = __byte_perm(ev[m + 1], ev[m + 2], 0x5432);   // 4m + 6, 4m + 8
    const unsigned o_m1 = __byte_perm(od[m], od[m + 1], 0x5432);       // 4m + 3, 4m + 5
    hs[m] = e_m2 + e_p2 + 4 * (o_m1 + od[m + 1]) + 6 * ev[m + 1];
  }
}
// Vertical [1 4 6 4 1] of five packed horizontal sums, rounded: each lane <= 16 * 4080 + 128 = 65408, so no carry crosses
// into the next lane and (s + 128) >> 8 is the lane's high byte.
__device__ __forceinline__ unsigned vpyr_words(unsigned a, unsigned b, unsigned c, unsigned d, unsigned e) {
  return a + e + 4 * (b + d) + 6 * c + 0x00800080u;
}
// The four output bytes of two vpyr_words results (lo lane, hi lane of v0, then of v1).
__device__ __forceinline__ unsigned pack_hi_bytes(unsigned v0, unsigned v1) { return __byte_perm(v0, v1, 0x7531); }

__device__ __forceinline__ void eq_pyr1_body(const uint8_t *__restrict__ src, int w, int h, int spitch,
              const uint8_t *__restrict__ eq_lut, int equalize, const uint8_t *__restrict__ clahe_luts, const ClaheGeom &cg,
              uint8_t *__restrict__ l0, int l0pitch,
              uint8_t *__restrict__ l1, int w1, int h1, int l1pitch, uint8_t *__restrict__ half, int wh, int hh,
              int hpitch) {
  __shared__ __align__(16) uint8_t tile[kTileRows][kTileCols];
  __shared__ __align__(16) uint8_t rawt[kTileRows][kBulkCols];
  __shared__ __align__(8) unsigned long long bulk_bar;
  __shared__ __align__(16) unsigned hbuf[kTileRows][kT1W / 2];   // packed horizontal sums, level-1 columns (2j, 2j + 1)
  __shared__ uint8_t lut[256];

  const int tid = threadIdx.x;
  const int tx0 = blockIdx.x * kT1W, ty0 = blockIdx.y * kT1H;
  const int gx_base = 2 * tx0 - 4, gy_base = 2 * ty0 - 2;
  // ---- interior tile: start the bulk copies of the raw window now
  const bool bulk = gy_base >= 0 && gy_base + kTileRows <= h && 2 * tx0 - 16 >= 0 && 2 * tx0 + kBulkCols - 16 <= w &&
                    (spitch & 15) == 0 && ((size_t)src & 15) == 0;
  if (bulk && tid == 0) {
    const unsigned bar = smem_u32(&bulk_bar);
    mbar_init(bar, 1);
    mbar_expect_tx(bar, kTileRows * kBulkCols);
    const uint8_t *g = src + (size_t)gy_base * spitch + (2 * tx0 - 16);
#pragma unroll 4
    for (int r = 0; r < kTileRows; r++) bulk_g2s(smem_u32(&rawt[r][0]), g + (size_t)r * spitch, kBulkCols, bar);
  }
  // ---- LUT (cv::equalizeHist, Appendix A1): built once per frame by the histogram's last CTA
  lut[tid] = equalize == 1 ? eq_lut[tid] : (uint8_t)tid;
  __syncthreads();

  // ---- stage the raw window through the LUT
  constexpr int kWordsPerRow = kTileCols / 4;
  if (bulk) {
    mbar_wait(smem_u32(&bulk_bar), 0);
    for (int i = tid; i < kTileRows * kWordsPerRow; i += kEqThreads) {
      const int r = i / kWordsPerRow, wi = i - r * kWordsPerRow;
      const unsigned v = *reinterpret_cast<const unsigned *>(&rawt[r][kBulkLead + 4 * wi]);
      unsigned out;
      if (equalize == 2) {
        const int gy = gy_base + r, gx = gx_base + 4 * wi;
        out = clahe_px(clahe_luts, cg, gx, gy, v & 0xff) | (clahe_px(clahe_luts, cg, gx + 1, gy, (v >> 8) & 0xff) << 8) |
              (clahe_px(clahe_luts, cg, gx + 2, gy, (v >> 16) & 0xff) << 16) | (clahe_px(clahe_luts, cg, gx + 3, gy, v >> 24) << 24);
      } else {
        out = (unsigned)lut[v & 0xff] | ((unsigned)lut[(v >> 8) & 0xff] << 8) | ((unsigned)lut[(v >> 16) & 0xff] << 16) |
              ((unsigned)lut[v >> 24] << 24);
      }
      *reinterpret_cast<unsigned *>(&tile[r][4 * wi]) = out;
    }
  } else
  for (int i = tid; i < kTileRows * kWordsPerRow; i += kEqThreads) {
    int r = i / kWordsPerRow, wi = i - r * kWordsPerRow;
    int gy = gy_base + r, gx = gx_base + 4 * wi;
    unsigned out = 0;
    if (gy > -h && gy < 2 * h - 1) {
      int ry = reflect101(gy, h);
      const uint8_t *row = src + (size_t)ry * spitch;
      if (equalize == 2) {   // CLAHE: the mapping depends on the pixel position (the REFLECTED one in the halo)
#pragma unroll
        for (int k = 0; k < 4; k++) {
          int x = gx + k;
          if (x > -w && x < 2 * w - 1) {
            const int rx = reflect101(x, w);
            out |= clahe_px(clahe_luts, cg, rx, ry, row[rx]) << (8 * k);
          }
        }
      } else if (gx >= 0 && gx + 4 <= w) {
        unsigned v = *reinterpret_cast<const unsigned *>(row + gx);
        out = (unsigned)lut[v & 0xff] | ((unsigned)lut[(v >> 8) & 0xff] << 8) | ((unsigned)lut[(v >> 16) & 0xff] << 16) |
              ((unsigned)lut[v >> 24] << 24);
      } else {
#pragma unroll
        for (int k = 0; k < 4; k++) {
          int x = gx + k;
          if (x > -w && x < 2 * w - 1) out |= (unsigned)lut[row[reflect101(x, w)]] << (8 * k);
        }
      }
    }
    *reinterpret_cast<unsigned *>(&tile[r][4 * wi]) = out;
  }
  __syncthreads();

  // ---- level 0 (equalised frame): interior words of the tile
  for (int i = tid; i < kT0H * (kT0W / 4); i += kEqThreads) {
    int r = i / (kT0W / 4), wi = i - r * (kT0W / 4);
    int gy = 2 * ty0 + r, gx = 2 * tx0 + 4 * wi;
    if (gy < h && gx < w) {
      unsigned v = *reinterpret_cast<const unsigned *>(&tile[r + 2][4 + 4 * wi]);
      uint8_t *dst = l0 + (size_t)gy * l0pitch + gx;
      if (gx + 4 <= w) {
        *reinterpret_cast<unsigned *>(dst) = v;
      } else {
        for (int k = 0; gx + k < w; k++) dst[k] = (uint8_t)(v >> (8 * k));
      }
    }
  }

  // ---- horizontal [1 4 6 4 1] on all staged rows, packed: a task is 4 words of hbuf (level-1 columns 8g .. 8g + 7)
  // from tile words 4g .. 4g + 5 of one row
  constexpr int kHGroups = kT1W / 8;
  for (int t = tid; t < kTileRows * kHGroups; t += kEqThreads) {
    const int r = t / kHGroups, g = t - r * kHGroups;
    const uint2 *p = reinterpret_cast<const uint2 *>(&tile[r][16 * g]);   // rows are 8-byte aligned (kTileCols = 136)
    const uint2 a = p[0], b = p[1], c = p[2];
    const unsigned wd[6] = {a.x, a.y, b.x, b.y, c.x, c.y};
    unsigned hs[4];
    hpyr_words<4>(wd, hs);
    *reinterpret_cast<uint4 *>(&hbuf[r][4 * g]) = make_uint4(hs[0], hs[1], hs[2], hs[3]);
  }
  __syncthreads();

  // ---- vertical pass -> level 1, and the 2x2 mean -> half-resolution image; one output word of each per thread
  {
    static_assert(kT1H * (kT1W / 4) == kEqThreads, "one level-1 word per thread");
    const int r = tid / (kT1W / 4), q = tid - r * (kT1W / 4);
    const int oy = ty0 + r, ox = tx0 + 4 * q;
    if (oy < h1 && ox < w1) {
      uint2 hv[5];
#pragma unroll
      for (int j = 0; j < 5; j++) hv[j] = *reinterpret_cast<const uint2 *>(&hbuf[2 * r + j][2 * q]);
      const unsigned packed = pack_hi_bytes(vpyr_words(hv[0].x, hv[1].x, hv[2].x, hv[3].x, hv[4].x),
                                            vpyr_words(hv[0].y, hv[1].y, hv[2].y, hv[3].y, hv[4].y));
      uint8_t *dst = l1 + (size_t)oy * l1pitch + ox;
      if (ox + 4 <= w1) {
        *reinterpret_cast<unsigned *>(dst) = packed;
      } else {
        for (int k = 0; ox + k < w1; k++) dst[k] = (uint8_t)(packed >> (8 * k));
      }
    }
    if (half != nullptr && oy < hh && ox < wh) {
      // (a + b + c + d + 2) >> 2 per lane: Ev + Od of a word are the sums of its two pixel pairs; each lane <= 1022
      const unsigned *p0 = reinterpret_cast<const unsigned *>(&tile[2 * r + 2][8 * q + 4]);
      const unsigned *p1 = reinterpret_cast<const unsigned *>(&tile[2 * r + 3][8 * q + 4]);
      const unsigned a0 = p0[0], a1 = p0[1], b0 = p1[0], b1 = p1[1];
      const unsigned s0 = __byte_perm(a0, 0, 0x4240) + __byte_perm(a0, 0, 0x4341) + __byte_perm(b0, 0, 0x4240) +
                          __byte_perm(b0, 0, 0x4341) + 0x00020002u;
      const unsigned s1 = __byte_perm(a1, 0, 0x4240) + __byte_perm(a1, 0, 0x4341) + __byte_perm(b1, 0, 0x4240) +
                          __byte_perm(b1, 0, 0x4341) + 0x00020002u;
      const unsigned packed = __byte_perm(s0 >> 2, s1 >> 2, 0x6420);
      uint8_t *dst = half + (size_t)oy * hpitch + ox;
      if (ox + 4 <= wh) {
        *reinterpret_cast<unsigned *>(dst) = packed;
      } else {
        for (int k = 0; ox + k < wh; k++) dst[k] = (uint8_t)(packed >> (8 * k));
      }
    }
  }
}

__global__ void __launch_bounds__(kEqThreads)
    k_eq_pyr1(const uint8_t *__restrict__ src, int w, int h, int spitch, const uint8_t *__restrict__ eq_lut, int equalize,
              const uint8_t *__restrict__ clahe_luts, ClaheGeom cg,
              uint8_t *__restrict__ l0, int l0pitch,
              uint8_t *__restrict__ l1, int w1, int h1, int l1pitch, uint8_t *__restrict__ half, int wh, int hh,
              int hpitch) {
  eq_pyr1_body(src, w, h, spitch, eq_lut, equalize, clahe_luts, cg, l0, l0pitch, l1, w1, h1, l1pitch, half, wh, hh, hpitch);
}
__global__ void __launch_bounds__(kEqThreads)
    k_eq_pyr1_b(const SlotRec *__restrict__ slots, const FrontJob *__restrict__ jobs, int w, int h, ClaheGeom cg, int want_half) {
  const FrontJob job = jobs[blockIdx.z];
  const SlotRec &sl = slots[job.slot];
  const DevImage &l1 = sl.lvl[1];
  const bool has1 = sl.n_lvl > 1;
  eq_pyr1_body(job.src, w, h, job.src_pitch, sl.eq_lut, job.eq_mode, sl.clahe, cg, sl.lvl[0].p, sl.lvl[0].pitch,
               has1 ? l1.p : nullptr, has1 ? l1.w : 0, has1 ? l1.h : 0, l1.pitch, want_half ? sl.half.p : nullptr, sl.half.w, sl.half.h,
               sl.half.pitch);
}

void launch_eq_pyr1_batch(const SlotRec *slots, const FrontJob *jobs, int n_jobs, const FrontGeom &g, bool want_half, cudaStream_t s) {
  if (n_jobs <= 0) return;
  const int w1 = (g.w + 1) / 2, h1 = (g.h + 1) / 2;
  dim3 grid((w1 + kT1W - 1) / kT1W, (h1 + kT1H - 1) / kT1H, n_jobs);
  PLVIWO_CARVEOUT(k_eq_pyr1_b);
  k_eq_pyr1_b<<<grid, kEqThreads, 0, s>>>(slots, jobs, g.w, g.h, clahe_geom(g.w, g.h), want_half ? 1 : 0);
}

void launch_eq_pyr1(const DevImage &src, const uint8_t *d_lut, int equalize, const DevImage &l0,
                    const DevImage &l1, const DevImage &half, cudaStream_t s, const uint8_t *d_clahe_luts) {
  // tiles are laid over the level-1 footprint of the frame even when level 1 itself is not wanted (l1.p == null)
  const int w1 = (src.w + 1) / 2, h1 = (src.h + 1) / 2;
  dim3 grid((w1 + kT1W - 1) / kT1W, (h1 + kT1H - 1) / kT1H);
  PLVIWO_CARVEOUT(k_eq_pyr1);
  k_eq_pyr1<<<grid, kEqThreads, 0, s>>>(src.p, src.w, src.h, src.pitch, d_lut, equalize, d_clahe_luts,
                                        clahe_geom(src.w, src.h), l0.p, l0.pitch, l1.p,
                                        l1.p ? l1.w : 0, l1.p ? l1.h : 0, l1.pitch, half.p, half.w, half.h, half.pitch);
}

// ---------------------------------------------------------------------------------------- remaining levels
constexpr int kRestThreads = 256;

// One level from the previous one: a thread produces 4 horizontally adjacent outputs (one 32-bit store).  The upper
// levels are tiny (320x140 and below), L2 resident, and each costs one short launch; an earlier version that let the
// last CTA of level 2 compute all remaining levels alone measured 51 us, this is ~3 us per level.
__device__ __forceinline__ void pyr_down_body(const uint8_t *__restrict__ src, int sw, int sh, int spitch, uint8_t *__restrict__ dst,
                                              int dw, int dh, int dpitch) {
  const int quads = (dw + 3) >> 2;
  const int i = blockIdx.x * kRestThreads + threadIdx.x;
  if (i >= quads * dh) return;
  const int y = i / quads, x0 = (i - y * quads) << 2;
  // 5 source rows x 11 source columns feed 4 outputs
  int col[11];
#pragma unroll
  for (int k = 0; k < 11; k++) col[k] = reflect101(2 * x0 + k - 2, sw);
  int hs[4] = {0, 0, 0, 0};
  const int wgt[5] = {1, 4, 6, 4, 1};
#pragma unroll
  for (int j = 0; j < 5; j++) {
    const uint8_t *row = src + (size_t)reflect101(2 * y + j - 2, sh) * spitch;
    int v[11];
#pragma unroll
    for (int k = 0; k < 11; k++) v[k] = row[col[k]];
#pragma unroll
    for (int o = 0; o < 4; o++)
      hs[o] += wgt[j] * (v[2 * o] + 4 * v[2 * o + 1] + 6 * v[2 * o + 2] + 4 * v[2 * o + 3] + v[2 * o + 4]);
  }
  uint8_t *d = dst + (size_t)y * dpitch + x0;
  if (x0 + 4 <= dw) {
    unsigned packed = 0;
#pragma unroll
    for (int o = 0; o < 4; o++) packed |= (unsigned)((hs[o] + 128) >> 8) << (8 * o);
    *reinterpret_cast<unsigned *>(d) = packed;
  } else {
    for (int o = 0; x0 + o < dw; o++) d[o] = (uint8_t)((hs[o] + 128) >> 8);
  }
}

__global__ void __launch_bounds__(kRestThreads)
    k_pyr_down(const uint8_t *__restrict__ src, int sw, int sh, int spitch, uint8_t *__restrict__ dst, int dw, int dh,
               int dpitch) {
  pyr_down_body(src, sw, sh, spitch, dst, dw, dh, dpitch);
}
__global__ void __launch_bounds__(kRestThreads)
    k_pyr_down_b(const SlotRec *__restrict__ slots, const FrontJob *__restrict__ jobs, int level) {
  const SlotRec &sl = slots[jobs[blockIdx.z].slot];
  const DevImage &a = sl.lvl[level - 1], &b = sl.lvl[level];
  pyr_down_body(a.p, a.w, a.h, a.pitch, b.p, b.w, b.h, b.pitch);
}
void launch_pyr_level_batch(const SlotRec *slots, const FrontJob *jobs, int n_jobs, int level, int dw, int dh, cudaStream_t s) {
  if (n_jobs <= 0) return;
  const int n = ((dw + 3) >> 2) * dh;
  PLVIWO_CARVEOUT(k_pyr_down_b);
  k_pyr_down_b<<<dim3((n + kRestThreads - 1) / kRestThreads, 1, n_jobs), kRestThreads, 0, s>>>(slots, jobs, level);
}

// Completion signal: a one-thread kernel at the tail of a stream writes a sequence number into pinned host memory.
// The host threads poll that word instead of calling into the driver (cudaEventQuery / cudaStreamSynchronize from
// two threads serialise on the context lock and cost 10-100 us each).
__global__ void k_signal(volatile int *flag, int value) {
  *flag = value;
  __threadfence_system();
}
int carveout_percent() {
  static const int pct = [] {
    const char *e = std::getenv("PLVIWO_CARVEOUT");
    if (!e) return 100;   // measured +3 % frames/s on one pipelined stream (profiles/experiments_r1.md)
    const int v = std::atoi(e);
    return v < 0 ? -1 : (v > 100 ? 100 : v);
  }();
  return pct;
}

void launch_signal(int *host_flag, int value, cudaStream_t s) {
  PLVIWO_CARVEOUT(k_signal);
  k_signal<<<1, 1, 0, s>>>(host_flag, value);
}
// Same, with the sequence number kept in device memory so that the launch can live in a replayed CUDA graph.
__global__ void k_signal_inc(volatile int *flag, int *dev_seq) {
  int v = *dev_seq + 1;
  *dev_seq = v;
  *flag = v;
  __threadfence_system();
}
void launch_signal_inc(int *host_flag, int *dev_seq, cudaStream_t s) {
  PLVIWO_CARVEOUT(k_signal_inc);
  k_signal_inc<<<1, 1, 0, s>>>(host_flag, dev_seq);
}

void launch_pyr_down(const DevImage &a, const DevImage &b, cudaStream_t s) {
  int n = ((b.w + 3) >> 2) * b.h;
  PLVIWO_CARVEOUT(k_pyr_down);
  k_pyr_down<<<(n + kRestThreads - 1) / kRestThreads, kRestThreads, 0, s>>>(a.p, a.w, a.h, a.pitch, b.p, b.w, b.h, b.pitch);
}

void launch_pyr_rest(const Pyramid &pyr, unsigned *d_counter, cudaStream_t s) {
  (void)d_counter;
  for (int l = 2; l < pyr.n; l++) {
    const DevImage &a = pyr.lvl[l - 1], &b = pyr.lvl[l];
    int n = ((b.w + 3) >> 2) * b.h;
    PLVIWO_CARVEOUT(k_pyr_down);
    k_pyr_down<<<(n + kRestThreads - 1) / kRestThreads, kRestThreads, 0, s>>>(a.p, a.w, a.h, a.pitch, b.p, b.w, b.h, b.pitch);
  }
}

}  // namespace plviwo
