// R1/P1: multi-level ROIAlign (NHWC).  R2+R3 (relation head) live in relation_tc.cu.
#include "common.cuh"
#include "tc05.cuh"

namespace fod {

// ------------------------------------------------------------------------------------------------
// ROIAlign, aligned=True, sampling_ratio=0 (adaptive grid), torchvision CPU semantics
// (torchvision/csrc/ops/cpu/roi_align_kernel.cpp + roi_align_common.h).
// One CTA per ROI; a warp owns a bin at a time; a lane owns 4 channels (16-byte loads, the
// four bilinear taps of a sample are four fully coalesced 512-byte rows of the NHWC map).
// ------------------------------------------------------------------------------------------------
struct RoiParams {
  const float* feat[FOD_MAX_LEVELS];
  int H[FOD_MAX_LEVELS], W[FOD_MAX_LEVELS], stride[FOD_MAX_LEVELS];
  int num_levels;
  int C;        // problems per image
  int roi_cap;
  int tiled;    // output layout, see roi_align_kernel
  int pix;      // floats per pixel of the maps = channels (a multiple of 128; blockIdx.z selects the 128-channel block)
};

// d2 poolers.py:50-58, fp32 like torch: floor(4 + log2(sqrt(area)/224 + 1e-8)) clamped to the
// available levels.  min level = log2(stride[0]).
__device__ __forceinline__ int assign_level(float4 b, int min_level, int num_levels) {
  float area = __fmul_rn(__fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y));
  float sz = __fsqrt_rn(area);
  float v = __fadd_rn(4.0f, log2f(__fadd_rn(__fdiv_rn(sz, 224.0f), 1e-8f)));
  v = floorf(v);
  v = fminf(fmaxf(v, (float)min_level), (float)(min_level + num_levels - 1));
  return (int)v - min_level;   // NaN area (negative) -> (int)NaN = 0 on CUDA; torch gives INT64_MIN: never valid input
}

// One bilinear sample coordinate along one axis (torchvision roi_align_common.h pre_calc_for_bilinear_interpolate):
// the two neighbouring rows / columns and their weights; w_low = w_high = 0 for a sample outside [-1, size].
struct AxisSample {
  int lo, hi;
  float w_hi, w_lo;  // weight of index `hi` (l) and of index `lo` (h = 1 - l)
};

__device__ __forceinline__ AxisSample axis_sample(float start, float bin, int p, int i, int grid, int size) {
  // coordinate = start + p*bin + (i+.5)*bin/grid     (left-to-right like the C++ expression)
  float v = __fadd_rn(__fadd_rn(start, __fmul_rn((float)p, bin)),
                      __fdiv_rn(__fmul_rn(__fadd_rn((float)i, 0.5f), bin), (float)grid));
  AxisSample s;
  if (v < -1.0f || v > (float)size) {
    s.lo = s.hi = 0;
    s.w_hi = s.w_lo = 0.f;
    return s;
  }
  if (v <= 0.f) v = 0.f;
  int lo = (int)v, hi;
  if (lo >= size - 1) {
    hi = lo = size - 1;
    v = (float)lo;
  } else {
    hi = lo + 1;
  }
  s.lo = lo;
  s.hi = hi;
  s.w_hi = __fsub_rn(v, (float)lo);
  s.w_lo = __fsub_rn(1.f, s.w_hi);
  return s;
}

constexpr int kMaxGrid = 7;             // sampling grid per bin handled by the shared-memory tables
constexpr int kMaxTaps = 8;             // distinct rows / columns one bin can touch (grid + 1)

// Per ROI and axis: for every bin the list of DISTINCT map rows (columns) its samples touch, with the summed
// interpolation weight of each.  Consecutive samples of a bin share a row (the upper neighbour of one is the lower
// neighbour of the next), so a bin with a g x g grid reads (g+1)^2 pixels instead of 4 g^2 taps.  Lists are padded
// to the ROI-wide maximum length with zero-weight entries so that the hot loop has a compile-time trip count.
#ifdef FOD_ROI_PROF
__device__ long long g_roi_prof[8];
#define RPROF(slot) do { if (threadIdx.x == 0 && blockIdx.y == 0 && blockIdx.x < 64) atomicAdd((unsigned long long*)&g_roi_prof[slot], (unsigned long long)(clock64() - t_start)); } while (0)
#else
#define RPROF(slot)
#endif

// Everything the pooling of one ROI needs besides the map: written once per ROI by roi_tables_kernel (all ROIs of a
// call in parallel, one thread per axis and bin) and copied into shared memory by the pooling CTA.  Without this pre-pass
// the same work is a serial prologue of every CTA - one thread for the box geometry, then 2R threads for the tap lists,
// 5 600 of the 13 900 cycles a CTA lives (tools/prof_roi.py).
template <int R>
struct alignas(16) RoiBlob {
  int xoff[R][kMaxTaps];
  float xw[R][kMaxTaps];
  int yoff[R][kMaxTaps];
  float yw[R][kMaxTaps];
  int xn[R], yn[R];
  float gbox[4];           // start_w, start_h, bin_w, bin_h
  int grid_w, grid_h, W, H;
  int level, tables;
  float inv_count;
  int pad;
};

struct BoxGeom {
  int lvl, H, W, grid_w, grid_h;
  float start_w, start_h, bin_w, bin_h;
  bool tables;       // the sampling grid fits the tap tables
  float inv_count;   // 1 / samples per bin
};

template <int R>
__device__ __forceinline__ BoxGeom box_geometry(const RoiParams& prm, const float4 box) {
  BoxGeom g;
  const int min_level = 31 - __clz(prm.stride[0]);
  g.lvl = assign_level(box, min_level, prm.num_levels);
  g.H = prm.H[0];
  g.W = prm.W[0];
  int stride = prm.stride[0];
  if (g.lvl == 1) { g.H = prm.H[1]; g.W = prm.W[1]; stride = prm.stride[1]; }
  if (g.lvl == 2) { g.H = prm.H[2]; g.W = prm.W[2]; stride = prm.stride[2]; }
  const float scale = 1.0f / (float)stride;
  g.start_w = __fsub_rn(__fmul_rn(box.x, scale), 0.5f);
  g.start_h = __fsub_rn(__fmul_rn(box.y, scale), 0.5f);
  const float end_w = __fsub_rn(__fmul_rn(box.z, scale), 0.5f);
  const float end_h = __fsub_rn(__fmul_rn(box.w, scale), 0.5f);
  const float roi_w = __fsub_rn(end_w, g.start_w), roi_h = __fsub_rn(end_h, g.start_h);
  g.grid_h = (int)ceilf(__fdiv_rn(roi_h, (float)R));
  g.grid_w = (int)ceilf(__fdiv_rn(roi_w, (float)R));
  g.bin_w = __fdiv_rn(roi_w, (float)R);
  g.bin_h = __fdiv_rn(roi_h, (float)R);
  g.tables = g.grid_h <= kMaxGrid && g.grid_w <= kMaxGrid;
  g.inv_count = 1.0f / fmaxf((float)(g.grid_h * g.grid_w), 1.0f);
  return g;
}

// Everything of the blob but the tap tables: all that pool_one_roi needs for a ROI beyond the tables.
template <int R>
__device__ __forceinline__ void write_blob_header(RoiBlob<R>& B, const BoxGeom& g) {
  B.gbox[0] = g.start_w; B.gbox[1] = g.start_h; B.gbox[2] = g.bin_w; B.gbox[3] = g.bin_h;
  B.grid_w = g.grid_w; B.grid_h = g.grid_h; B.W = g.W; B.H = g.H;
  B.level = g.lvl;
  B.tables = g.tables ? 1 : 0;
  B.inv_count = g.inv_count;
  B.pad = 0;
}

// The list of DISTINCT map rows (columns) the samples of one bin touch along one axis, with the summed interpolation
// weight of each, in the order torchvision adds them.  The indices are CONSECUTIVE (the sampling step bin / grid is at
// most one pixel and the clamped ends repeat the border index), so entry q is index first + q and a sample adds its two
// weights to the slots lo - first and hi - first: w[] stays in registers.  Returns the number of entries n (at most
// grid + 1 <= kMaxTaps); w[q] = 0 for q >= n.
__device__ __forceinline__ int build_axis_taps(const BoxGeom& g, bool is_x, int bin, int& first, float (&w)[kMaxTaps]) {
  int n = 0;
  first = 0;
#pragma unroll
  for (int q = 0; q < kMaxTaps; ++q) w[q] = 0.f;
  const int grid = is_x ? g.grid_w : g.grid_h, size = is_x ? g.W : g.H;
  const float start = is_x ? g.start_w : g.start_h, bsz = is_x ? g.bin_w : g.bin_h;
  for (int i = 0; i < grid; ++i) {
    const AxisSample s = axis_sample(start, bsz, bin, i, grid, size);
    if (s.w_lo == 0.f && s.w_hi == 0.f) continue;
    if (n == 0) first = s.lo;
    const int dlo = s.lo - first, dhi = s.hi - first;
#pragma unroll
    for (int q = 0; q < kMaxTaps; ++q)
      if (q == dlo) w[q] += s.w_lo;
#pragma unroll
    for (int q = 0; q < kMaxTaps; ++q)
      if (q == dhi) w[q] += s.w_hi;
    n = max(n, dhi + 1);
  }
  return n;
}

// One thread per (ROI, axis, bin): grid.x covers roi_cap * 2R threads of a problem, grid.y = problem.
template <int R>
__global__ void __launch_bounds__(256) roi_tables_kernel(RoiParams prm, const float* __restrict__ rois,
                                                         const int32_t* __restrict__ roi_count, RoiBlob<R>* __restrict__ blobs,
                                                         int32_t* __restrict__ out_level) {
  const int p = blockIdx.y;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int r = t / (2 * R), k = t - r * 2 * R;      // k < R: x bin k, else y bin k - R
  const int cnt = roi_count ? min(roi_count[p], prm.roi_cap) : prm.roi_cap;
  if (r >= cnt) return;
  const float4 box = *reinterpret_cast<const float4*>(rois + ((size_t)p * prm.roi_cap + r) * 4);
  const BoxGeom g = box_geometry<R>(prm, box);
  RoiBlob<R>& B = blobs[(size_t)p * prm.roi_cap + r];
  if (k == 0) {
    if (out_level) out_level[(size_t)p * prm.roi_cap + r] = g.lvl;
    write_blob_header(B, g);
  }
  if (!g.tables) return;
  const bool is_x = k < R;
  const int bin = is_x ? k : k - R;
  int first;
  float w[kMaxTaps];
  const int n = build_axis_taps(g, is_x, bin, first, w);
  const int pitch = is_x ? prm.pix : g.W * prm.pix;
  int* po = is_x ? B.xoff[bin] : B.yoff[bin];
  float* pw = is_x ? B.xw[bin] : B.yw[bin];
#pragma unroll
  for (int q = 0; q < kMaxTaps; ++q) {      // padding: offset 0, weight 0
    po[q] = q < n ? (first + q) * pitch : 0;
    pw[q] = w[q];
  }
  (is_x ? B.xn : B.yn)[bin] = n;
}

// NX = padded number of column taps per bin (compile time): the inner loop is 2 LDS.128 per bin and row plus
// LDG.128 + FMUL + 4 FFMA per tap.
template <int R, int NX>
__device__ __forceinline__ void roi_accumulate(const RoiBlob<R>& B, const float* __restrict__ f, int ph, int pw0, int ny,
                                               float4 (&acc)[R / 2]) {
  for (int kr = 0; kr < ny; ++kr) {
    const float wy = B.yw[ph][kr];
    const float* rowp = f + B.yoff[ph][kr];
#pragma unroll
    for (int j = 0; j < R / 2; ++j) {
      int off[kMaxTaps];
      float w[kMaxTaps];
      *reinterpret_cast<int4*>(off) = *reinterpret_cast<const int4*>(&B.xoff[pw0 + j][0]);
      *reinterpret_cast<float4*>(w) = *reinterpret_cast<const float4*>(&B.xw[pw0 + j][0]);
      if (NX > 4) {
        *reinterpret_cast<int4*>(off + 4) = *reinterpret_cast<const int4*>(&B.xoff[pw0 + j][4]);
        *reinterpret_cast<float4*>(w + 4) = *reinterpret_cast<const float4*>(&B.xw[pw0 + j][4]);
      }
      float4 v[NX];
#pragma unroll
      for (int k = 0; k < NX; ++k) v[k] = ldg4(rowp + off[k]);
#pragma unroll
      for (int k = 0; k < NX; ++k) {
        const float ww = wy * w[k];
        acc[j].x = fmaf(ww, v[k].x, acc[j].x);
        acc[j].y = fmaf(ww, v[k].y, acc[j].y);
        acc[j].z = fmaf(ww, v[k].z, acc[j].z);
        acc[j].w = fmaf(ww, v[k].w, acc[j].w);
      }
    }
  }
}

// Where a lane stores its 4 channels of bin 0 of a pooled ROI row (problem p, ROI r, 128-channel block cblock), and the
// stride from one bin to the next.  tiled == 0: [P][roi_cap][bins][pix] (row-major ROI rows).  tiled == 1 (8 x 8 bins,
// 128 channels, consumed by fod_relation_head): [P][units][256 k-chunks][128 rows][32], units = ceil(roi_cap / 128): the
// 16 KB A tile of one 32-wide K chunk of 128 ROI rows is contiguous, so one TMA box fetches it as a linear stream.
// The stride is a function of its own: as a separate select the compiler turns the tile kernel's per-bin multiply
// into a shift.
__device__ __forceinline__ float* pooled_row(float* pooled, bool tiled, int roi_cap, int bins, int pix, int p, int r,
                                             unsigned cblock, int lane) {
  const int units = (roi_cap + 127) >> 7;
  return tiled ? pooled + ((((size_t)p * units + (r >> 7)) * 256 + (lane >> 3)) * 128 + (r & 127)) * 32 + (lane & 7) * 4
               : pooled + ((size_t)p * roi_cap + r) * bins * pix + cblock * kC + lane * 4;
}
__device__ __forceinline__ size_t pooled_bin_stride(bool tiled, int pix) {
  return tiled ? (size_t)4 * 128 * 32 : (size_t)pix;   // tiled: next bin = 4 k-chunks further
}

// One CTA per ROI (and 128-channel block); warp = (bin row, half of the bin columns), lane = 4 channels: every tap is
// one fully coalesced 512-byte row of the NHWC map, 4 accumulators per lane keep the register count low enough for
// full occupancy.  The ROI's geometry and tap lists come from roi_tables_kernel.
template <int R>
__device__ __forceinline__ void pool_one_roi(const RoiParams& prm, const RoiBlob<R>* __restrict__ blobs,
                                             float* __restrict__ pooled, const int p, const int r, RoiBlob<R>& B) {
#ifdef FOD_ROI_PROF
  const long long t_start = clock64();
#endif
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  {
    const int4* src = reinterpret_cast<const int4*>(blobs + ((size_t)p * prm.roi_cap + r));
    int4* dst = reinterpret_cast<int4*>(&B);
    for (int i = threadIdx.x; i < (int)(sizeof(RoiBlob<R>) / 16); i += blockDim.x) dst[i] = __ldg(src + i);
  }
  __syncthreads();
  RPROF(1);
  const bool tables = B.tables != 0;
  const int W = B.W, H = B.H, grid_w = B.grid_w, grid_h = B.grid_h;
  const float* fbase = prm.feat[0];
  if (B.level == 1) fbase = prm.feat[1];
  if (B.level == 2) fbase = prm.feat[2];
  const float* f = fbase + (size_t)(p / prm.C) * H * W * prm.pix + blockIdx.z * kC + lane * 4;   // this CTA's 128-channel block
  const int ph = warp >> 1, pw0 = (warp & 1) * (R / 2);
  float4 acc[R / 2];
#pragma unroll
  for (int j = 0; j < R / 2; ++j) acc[j] = make_float4(0, 0, 0, 0);
  if (tables) {
    int nx = 0;
#pragma unroll
    for (int j = 0; j < R; ++j) nx = max(nx, B.xn[j]);
    const int ny = B.yn[ph];
    switch (nx) {
      case 0: break;
      case 1: case 2: roi_accumulate<R, 2>(B, f, ph, pw0, ny, acc); break;
      case 3: roi_accumulate<R, 3>(B, f, ph, pw0, ny, acc); break;
      case 4: roi_accumulate<R, 4>(B, f, ph, pw0, ny, acc); break;
      case 5: case 6: roi_accumulate<R, 6>(B, f, ph, pw0, ny, acc); break;
      default: roi_accumulate<R, 8>(B, f, ph, pw0, ny, acc); break;
    }
  } else {  // sampling grid beyond the tables (box much larger than the pyramid level expects): sample by sample
    for (int iy = 0; iy < grid_h; ++iy) {
      const AxisSample ys = axis_sample(B.gbox[1], B.gbox[3], ph, iy, grid_h, H);
      if (ys.w_lo == 0.f && ys.w_hi == 0.f) continue;
      const float* row_lo = f + (size_t)ys.lo * W * prm.pix;
      const float* row_hi = f + (size_t)ys.hi * W * prm.pix;
#pragma unroll
      for (int j = 0; j < R / 2; ++j) {
        for (int ix = 0; ix < grid_w; ++ix) {
          const AxisSample xs = axis_sample(B.gbox[0], B.gbox[2], pw0 + j, ix, grid_w, W);
          const float4 v1 = ldg4(row_lo + (size_t)xs.lo * prm.pix), v2 = ldg4(row_lo + (size_t)xs.hi * prm.pix);
          const float4 v3 = ldg4(row_hi + (size_t)xs.lo * prm.pix), v4 = ldg4(row_hi + (size_t)xs.hi * prm.pix);
          const float w1 = ys.w_lo * xs.w_lo, w2 = ys.w_lo * xs.w_hi, w3 = ys.w_hi * xs.w_lo, w4 = ys.w_hi * xs.w_hi;
          acc[j].x += w1 * v1.x + w2 * v2.x + w3 * v3.x + w4 * v4.x;
          acc[j].y += w1 * v1.y + w2 * v2.y + w3 * v3.y + w4 * v4.y;
          acc[j].z += w1 * v1.z + w2 * v2.z + w3 * v3.z + w4 * v4.z;
          acc[j].w += w1 * v1.w + w2 * v2.w + w3 * v3.w + w4 * v4.w;
        }
      }
    }
  }
  RPROF(2);
  float* out = pooled_row(pooled, prm.tiled, prm.roi_cap, R * R, prm.pix, p, r, blockIdx.z, lane);
  const size_t bin_stride = pooled_bin_stride(prm.tiled, prm.pix);
  const float inv_count = B.inv_count;
#pragma unroll
  for (int j = 0; j < R / 2; ++j) {
    float4 o = make_float4(acc[j].x * inv_count, acc[j].y * inv_count, acc[j].z * inv_count, acc[j].w * inv_count);
    *reinterpret_cast<float4*>(out + (size_t)(ph * R + pw0 + j) * bin_stride) = o;
  }
  RPROF(3);
}


template <int R>
__global__ void __launch_bounds__(R * 64, R > 8 ? 1 : 2)
roi_align_kernel(RoiParams prm, const int32_t* __restrict__ roi_count, const RoiBlob<R>* __restrict__ blobs,
                 float* __restrict__ pooled) {
  __shared__ RoiBlob<R> B;
  const int r = blockIdx.x, p = blockIdx.y;
  const int cnt = roi_count ? min(roi_count[p], prm.roi_cap) : prm.roi_cap;
  if (r >= cnt) return;
  pool_one_roi<R>(prm, blobs, pooled, p, r, B);
}

// The same pooling for a LIST of ROIs (list[0] = number of entries, list[1 + i] = p * roi_cap + r): the ROIs whose
// sampling grid is beyond the tap tables, which the tile-stationary kernel below leaves out.  Usually the list is empty.
__global__ void __launch_bounds__(512, 2)
roi_align_list_kernel(RoiParams prm, const int32_t* __restrict__ list, const RoiBlob<8>* __restrict__ blobs,
                      float* __restrict__ pooled) {
  __shared__ RoiBlob<8> B;
  const int n = list[0];
  for (int i = blockIdx.x; i < n; i += gridDim.x) {
    const int e = list[1 + i];
    pool_one_roi<8>(prm, blobs, pooled, e / prm.roi_cap, e % prm.roi_cap, B);
    __syncthreads();   // B is rewritten by the next entry
  }
}

// ------------------------------------------------------------------------------------------------
// Tile-stationary pooling (R = 8, 128 channels: the query path R1).
//
// The per-ROI kernel above gathers a ROI's ~17 x 17-pixel window out of L2 once per ROI; the windows of one image
// overlap ~9 times, and it is the L2 -> SM path (9.5 TB/s) plus the L1 data pipe that bound it, not HBM.  Here the MAP
// is stationary: a CTA owns an 8 x 8-pixel tile of one pyramid level of one image, TMA-stages the tile plus a 4-pixel
// halo to the right / below into shared memory ONCE (12 x 12 pixels x 512 B = 72 KB, three CTAs per SM) and pools
// every bin whose first tap lies inside its 8 x 8 pixels, whatever ROI (and class) the bin belongs to.  A bin reaches
// at most ceil(bin size) + 1 rows / columns, so everything up to 4-pixel bins - the whole range FPN level assignment
// produces - is served from shared memory; a longer bin (elongated boxes) reads the map directly, same arithmetic.
// Work is found by a scan: one thread per ROI compares the ROI's 8 + 8 first taps (RoiSum, written by the table
// pre-pass) with the tile; candidates go to a shared list and warp w takes bin row (w + i) & 7 of candidate i.
// Inside a (ROI, bin row) task the tap lists live in registers, lane-distributed (lane = (bin & 3) * 8 + tap) and
// broadcast with SHFL; a lane owns 4 channels, a tap is one conflict-free LDS.128 per lane.  The summation order of a
// bin is the per-ROI kernel's (rows outer, columns inner, one FMA per tap and channel): results are bit-identical.
// ------------------------------------------------------------------------------------------------
struct alignas(16) RoiTile {       // tap lists of one ROI, indices instead of offsets, padded with the LAST valid index
  int xi[8][kMaxTaps];             // (weight 0), so that entry [..][7] is the bin's largest column / row
  float xw[8][kMaxTaps];
  int yi[8][kMaxTaps];
  float yw[8][kMaxTaps];
};
struct alignas(16) RoiSum {        // what the scan and a task's prologue need (48 bytes)
  short x0[8], y0[8];              // first column / row of every bin (0 for a bin without samples inside the map)
  short level, nx, tables, pad;    // nx = largest number of distinct columns over the ROI's bins
  uint32_t yn;                     // number of distinct rows of bin row i in bits 4i .. 4i+3
  float inv_count;
};

namespace rt {
constexpr int kOwn = 8;                       // a CTA owns kOwn x kOwn pixels ...
constexpr int kEdge = 12;                     // ... and stages kEdge x kEdge
constexpr int kThreads = 256;
constexpr int kScan = 256;                    // ROIs per scan pass (one per thread)
constexpr uint32_t kTileBytes = kEdge * kEdge * kC * 4;
constexpr uint32_t kOffCand = kTileBytes;                    // uint32[kScan]: ROI of the pass | column mask << 8 | row mask << 16
constexpr uint32_t kOffBar = kOffCand + kScan * 4;           // mbarrier
constexpr uint32_t kOffCount = kOffBar + 8;                  // int[2]: candidates, next task
constexpr uint32_t kSmemBytes = kOffCount + 8;
constexpr uint32_t kSmemAlloc = kSmemBytes + 128;            // slack for the 128-byte alignment of the TMA destination
static_assert(3 * (kSmemAlloc + 1024) <= 233472, "three CTAs per SM");
struct Params {
  CUtensorMap map[FOD_MAX_LEVELS];
  const float* feat[FOD_MAX_LEVELS];
  int H[FOD_MAX_LEVELS], W[FOD_MAX_LEVELS], tiles_x[FOD_MAX_LEVELS], tile_end[FOD_MAX_LEVELS];
  int num_levels, C, roi_cap, tiled;
};
}  // namespace rt

// One thread per (ROI, axis, bin), 16 threads per ROI.  Tabled ROIs get a RoiTile; a ROI whose sampling grid is beyond
// the tables gets the per-ROI kernel's blob header and an entry in the slow list.  Every ROI gets a RoiSum.
__global__ void __launch_bounds__(256) roi_tile_tables_kernel(RoiParams prm, const float* __restrict__ rois,
                                                              const int32_t* __restrict__ roi_count,
                                                              RoiTile* __restrict__ tiles, RoiSum* __restrict__ sums,
                                                              RoiBlob<8>* __restrict__ blobs, int32_t* __restrict__ slow_list,
                                                              int32_t* __restrict__ out_level) {
  constexpr int R = 8;
  const int p = blockIdx.y;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int r = t >> 4, k = t & 15;                  // k < 8: x bin k, else y bin k - 8
  const int cnt = roi_count ? min(roi_count[p], prm.roi_cap) : prm.roi_cap;
  const bool valid = r < cnt;                        // no early exit: the shuffles below are warp-wide
  const size_t row = (size_t)p * prm.roi_cap + (valid ? r : 0);
  const float4 box = *reinterpret_cast<const float4*>(rois + row * 4);
  const BoxGeom g = box_geometry<R>(prm, box);
  const bool is_x = k < R;
  const int bin = k & 7;
  int first = 0;
  float w[kMaxTaps];
  int n = 0;
  if (valid && g.tables) n = build_axis_taps(g, is_x, bin, first, w);
  int nx = is_x ? n : 0;
  uint32_t yn = is_x ? 0u : ((uint32_t)n << (4 * bin));
#pragma unroll
  for (int d = 8; d >= 1; d >>= 1) {
    nx = max(nx, __shfl_xor_sync(0xffffffffu, nx, d));
    yn |= __shfl_xor_sync(0xffffffffu, yn, d);
  }
  if (!valid) return;
  RoiSum& S = sums[row];
  if (k == 0) {
    if (out_level) out_level[row] = g.lvl;
    S.level = (short)g.lvl;
    S.nx = (short)nx;
    S.tables = g.tables ? 1 : 0;
    S.pad = 0;
    S.yn = yn;
    S.inv_count = g.inv_count;
    if (!g.tables) {
      write_blob_header(blobs[row], g);
      slow_list[1 + atomicAdd(slow_list, 1)] = (int32_t)row;
    }
  }
  (is_x ? S.x0 : S.y0)[bin] = (short)first;
  if (!g.tables) return;
  RoiTile& T = tiles[row];
  int4* pi = reinterpret_cast<int4*>(is_x ? T.xi[bin] : T.yi[bin]);
  float4* pw = reinterpret_cast<float4*>(is_x ? T.xw[bin] : T.yw[bin]);
  const int last = n ? first + n - 1 : 0;
  int iv[kMaxTaps];
#pragma unroll
  for (int q = 0; q < kMaxTaps; ++q) iv[q] = min(first + q, last);      // w[q] is 0 for q >= n by construction
  pi[0] = make_int4(iv[0], iv[1], iv[2], iv[3]);
  pi[1] = make_int4(iv[4], iv[5], iv[6], iv[7]);
  pw[0] = make_float4(w[0], w[1], w[2], w[3]);
  pw[1] = make_float4(w[4], w[5], w[6], w[7]);
}

// One bin out of the staged tile with compile-time tap counts: NX column taps (fetched from the lanes that hold the
// ROI's lists) x NY rows (addresses and weights prepared once per task); the NY * NX loads are independent.
template <int NY, int NX>
__device__ __forceinline__ float4 tile_bin_fixed(const uint32_t (&rowa)[4], const float (&wy)[4], const int xb, const float xw,
                                                 const int src) {
  uint32_t off[NX];
  float w[NX];
#pragma unroll
  for (int k = 0; k < NX; ++k) {
    off[k] = (uint32_t)__shfl_sync(0xffffffffu, xb, src + k);
    w[k] = __shfl_sync(0xffffffffu, xw, src + k);
  }
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int kr = 0; kr < NY; ++kr) {
    float4 v[NX];
#pragma unroll
    for (int k = 0; k < NX; ++k) v[k] = tc::lds4s(rowa[kr] + off[k]);
#pragma unroll
    for (int k = 0; k < NX; ++k) {
      const float ww = wy[kr] * w[k];
      acc.x = fmaf(ww, v[k].x, acc.x);
      acc.y = fmaf(ww, v[k].y, acc.y);
      acc.z = fmaf(ww, v[k].z, acc.z);
      acc.w = fmaf(ww, v[k].w, acc.w);
    }
  }
  return acc;
}

// Any tap counts (bins wider / taller than 3 pixels, taps beyond the staged pixels): taps fetched inside the loops.
// xb = byte offset of the column inside the tile (relative column * 512), yr = relative row.
template <bool SM>
__device__ __forceinline__ float4 tile_bin_any(const int nx, const int xb, const float xw, const int src, const int yr,
                                               const float yw, const int ysrc, const int ny, const uint32_t tile_lane,
                                               const float* __restrict__ f_lane, const int tx0, const int ty0, const int W) {
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int kr = 0; kr < ny; ++kr) {
    const int yrel = __shfl_sync(0xffffffffu, yr, ysrc + kr);
    const float wy = __shfl_sync(0xffffffffu, yw, ysrc + kr);
    for (int k = 0; k < nx; ++k) {
      const int xo = __shfl_sync(0xffffffffu, xb, src + k);
      const float ww = wy * __shfl_sync(0xffffffffu, xw, src + k);
      float4 v;
      if (SM) v = tc::lds4s(tile_lane + (uint32_t)(yrel * (rt::kEdge * kC * 4) + xo));
      else v = ldg4(f_lane + ((size_t)(yrel + ty0) * W + ((xo >> 9) + tx0)) * kC);
      acc.x = fmaf(ww, v.x, acc.x);
      acc.y = fmaf(ww, v.y, acc.y);
      acc.z = fmaf(ww, v.z, acc.z);
      acc.w = fmaf(ww, v.w, acc.w);
    }
  }
  return acc;
}

__global__ void __launch_bounds__(rt::kThreads, 3)
roi_align_tiles_kernel(const __grid_constant__ rt::Params P, const int32_t* __restrict__ roi_count,
                       const RoiTile* __restrict__ tiles, const RoiSum* __restrict__ sums, float* __restrict__ pooled) {
  using namespace rt;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t sbase = (tc::smem_u32(smem_raw) + 127u) & ~127u;
  uint8_t* sgen = smem_raw + (sbase - tc::smem_u32(smem_raw));
  uint32_t* cand = reinterpret_cast<uint32_t*>(sgen + kOffCand);
  int* s_count = reinterpret_cast<int*>(sgen + kOffCount);    // [0] candidates, [1] next task
  const uint32_t bar = sbase + kOffBar;
  const int tid = threadIdx.x, lane = tid & 31;
  const int b = blockIdx.y;
  // which tile of which level
  int lvl = 0, id = blockIdx.x;
  if (P.num_levels > 1 && id >= P.tile_end[0]) { lvl = 1; }
  if (P.num_levels > 2 && id >= P.tile_end[1]) { lvl = 2; }
  if (lvl) id -= P.tile_end[lvl - 1];
  int W = P.W[0], H = P.H[0], tiles_x = P.tiles_x[0];
  const float* fmap = P.feat[0];
  if (lvl == 1) { W = P.W[1]; H = P.H[1]; tiles_x = P.tiles_x[1]; fmap = P.feat[1]; }
  if (lvl == 2) { W = P.W[2]; H = P.H[2]; tiles_x = P.tiles_x[2]; fmap = P.feat[2]; }
  const int ty = id / tiles_x, tx = id - ty * tiles_x;
  const int tx0 = tx * kOwn, ty0 = ty * kOwn;
  const float* f_lane = fmap + (size_t)b * H * W * kC + lane * 4;
  const uint32_t tile_lane = sbase + lane * 16;
  if (tid == 0) {                            // the tile is on its way while the ROIs are scanned
    tc::mbar_init(bar, 1);
    tc::fence_barrier_init();
    tc::mbar_arrive_expect_tx(bar, kTileBytes);
    tc::tma_load_4d(sbase, &P.map[lvl], bar, 0, tx0, ty0, b);
  }
  bool waited = false;
  for (int c = 0; c < P.C; ++c) {
    const int p = b * P.C + c;
    const int cnt = roi_count ? min(roi_count[p], P.roi_cap) : P.roi_cap;
    for (int base = 0; base < cnt; base += kScan) {
      if (tid < 2) s_count[tid] = 0;
      __syncthreads();                       // also orders the barrier initialisation before its first use
      {                                      // scan: which bins of ROI base + tid start inside this tile
        const int r = base + tid;
        if (tid < kScan && r < cnt) {
          const int4* sp = reinterpret_cast<const int4*>(sums + ((size_t)p * P.roi_cap + r));
          const int4 m = __ldg(sp + 2);      // level | nx, tables | pad, yn, inv_count
          const int level = (short)(m.x & 0xffff), tabled = (short)(m.y & 0xffff);
          if (level == lvl && tabled) {
            const int4 xa = __ldg(sp), ya = __ldg(sp + 1);
            const int xs[4] = {xa.x, xa.y, xa.z, xa.w}, ys[4] = {ya.x, ya.y, ya.z, ya.w};
            uint32_t xm = 0, ym = 0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int x_even = (short)(xs[j] & 0xffff), x_odd = xs[j] >> 16;
              const int y_even = (short)(ys[j] & 0xffff), y_odd = ys[j] >> 16;
              xm |= ((uint32_t)(x_even - tx0) < (uint32_t)kOwn ? 1u : 0u) << (2 * j);
              xm |= ((uint32_t)(x_odd - tx0) < (uint32_t)kOwn ? 1u : 0u) << (2 * j + 1);
              ym |= ((uint32_t)(y_even - ty0) < (uint32_t)kOwn ? 1u : 0u) << (2 * j);
              ym |= ((uint32_t)(y_odd - ty0) < (uint32_t)kOwn ? 1u : 0u) << (2 * j + 1);
            }
            if (xm && ym) cand[atomicAdd(&s_count[0], 1)] = (uint32_t)tid | (xm << 8) | (ym << 16);
          }
        }
      }
      __syncthreads();
      const int ntask = s_count[0];
      if (ntask > 0) {
        tc::mbar_wait(bar, 0);
        waited = true;
        for (;;) {                           // warps draw ROIs from a shared counter
          int ti = 0;
          if (lane == 0) ti = atomicAdd(&s_count[1], 1);
          ti = __shfl_sync(0xffffffffu, ti, 0);
          if (ti >= ntask) break;
          const uint32_t e = cand[ti];
          const int r = base + (int)(e & 255u);
          const uint32_t xm = (e >> 8) & 255u, ym = e >> 16;
          const size_t row = (size_t)p * P.roi_cap + r;
          const RoiTile& T = tiles[row];
          // lane = (bin & 3) * 8 + tap holds the taps of bins / bin rows 0-3 (a) and 4-7 (b)
          const int xa_r = __ldg(&T.xi[0][0] + lane) - tx0, xb_r = __ldg(&T.xi[0][0] + 32 + lane) - tx0;
          const float xa_w = __ldg(&T.xw[0][0] + lane), xb_w = __ldg(&T.xw[0][0] + 32 + lane);
          const int ya_r = __ldg(&T.yi[0][0] + lane) - ty0, yb_r = __ldg(&T.yi[0][0] + 32 + lane) - ty0;
          const float ya_w = __ldg(&T.yw[0][0] + lane), yb_w = __ldg(&T.yw[0][0] + 32 + lane);
          const uint32_t yn = __ldg(&sums[row].yn);
          const float inv_count = __ldg(&sums[row].inv_count);
          // a tap beyond the staged 12 x 12 pixels sends its bin (or the whole bin row) to the map
          const uint32_t xfar_a = __ballot_sync(0xffffffffu, (uint32_t)xa_r >= (uint32_t)kEdge);
          const uint32_t xfar_b = __ballot_sync(0xffffffffu, (uint32_t)xb_r >= (uint32_t)kEdge);
          const uint32_t yfar_a = __ballot_sync(0xffffffffu, (uint32_t)ya_r >= (uint32_t)kEdge);
          const uint32_t yfar_b = __ballot_sync(0xffffffffu, (uint32_t)yb_r >= (uint32_t)kEdge);
          const uint32_t nz_a = __ballot_sync(0xffffffffu, xa_w != 0.f);
          const uint32_t nz_b = __ballot_sync(0xffffffffu, xb_w != 0.f);
          const int xa_b = xa_r * (kC * 4), xb_b = xb_r * (kC * 4);                    // byte offsets inside the tile
          const int ya_b = ya_r * (kEdge * kC * 4), yb_b = yb_r * (kEdge * kC * 4);
          float* out_roi = pooled_row(pooled, P.tiled, P.roi_cap, 64, kC, p, r, 0, lane);
          const size_t bin_stride = pooled_bin_stride(P.tiled, kC);
          for (uint32_t rows = ym; rows; rows &= rows - 1) {
            const int by = __ffs(rows) - 1;
            const bool yhi = by >= 4;
            const int ysrc = (by & 3) * 8;
            const int ny = (int)((yn >> (4 * by)) & 15u);
            const bool rows_near = (((yhi ? yfar_b : yfar_a) >> ysrc) & 255u) == 0u;
            const int yb = yhi ? yb_b : ya_b, yr = yhi ? yb_r : ya_r;
            const float yw = yhi ? yb_w : ya_w;
            uint32_t rowa[4];
            float wy[4];
#pragma unroll
            for (int kr = 0; kr < 4; ++kr) {
              rowa[kr] = tile_lane + (uint32_t)__shfl_sync(0xffffffffu, yb, ysrc + kr);
              wy[kr] = __shfl_sync(0xffffffffu, yw, ysrc + kr);
            }
            float* out = out_roi + (size_t)(by * 8) * bin_stride;
            for (uint32_t mm = xm; mm; mm &= mm - 1) {
              const int bx = __ffs(mm) - 1;
              const bool hi = bx >= 4;
              const int src = (bx & 3) * 8;
              const bool near = rows_near && (((hi ? xfar_b : xfar_a) >> src) & 255u) == 0u;
              const int n = 32 - __clz(((hi ? nz_b : nz_a) >> src) & 255u);      // taps up to the last non-zero weight
              const int xb = hi ? xb_b : xa_b;
              const float xwv = hi ? xb_w : xa_w;
              float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
              if (n == 0 || ny == 0) {
              } else if (near && n <= 4 && ny <= 4) {
                switch ((ny - 1) * 3 + max(n, 2) - 2) {        // zero-weight padding taps lie inside the tile as well
                  case 0: a = tile_bin_fixed<1, 2>(rowa, wy, xb, xwv, src); break;
                  case 1: a = tile_bin_fixed<1, 3>(rowa, wy, xb, xwv, src); break;
                  case 2: a = tile_bin_fixed<1, 4>(rowa, wy, xb, xwv, src); break;
                  case 3: a = tile_bin_fixed<2, 2>(rowa, wy, xb, xwv, src); break;
                  case 4: a = tile_bin_fixed<2, 3>(rowa, wy, xb, xwv, src); break;
                  case 5: a = tile_bin_fixed<2, 4>(rowa, wy, xb, xwv, src); break;
                  case 6: a = tile_bin_fixed<3, 2>(rowa, wy, xb, xwv, src); break;
                  case 7: a = tile_bin_fixed<3, 3>(rowa, wy, xb, xwv, src); break;
                  case 8: a = tile_bin_fixed<3, 4>(rowa, wy, xb, xwv, src); break;
                  case 9: a = tile_bin_fixed<4, 2>(rowa, wy, xb, xwv, src); break;
                  case 10: a = tile_bin_fixed<4, 3>(rowa, wy, xb, xwv, src); break;
                  default: a = tile_bin_fixed<4, 4>(rowa, wy, xb, xwv, src); break;
                }
              } else if (near) {
                a = tile_bin_any<true>(n, xb, xwv, src, yr, yw, ysrc, ny, tile_lane, f_lane, tx0, ty0, W);
              } else {
                a = tile_bin_any<false>(n, xb, xwv, src, yr, yw, ysrc, ny, tile_lane, f_lane, tx0, ty0, W);
              }
              const float4 o = make_float4(a.x * inv_count, a.y * inv_count, a.z * inv_count, a.w * inv_count);
              *reinterpret_cast<float4*>(out + (size_t)bx * bin_stride) = o;
            }
          }
        }
      }
      if (base + kScan < cnt || c + 1 < P.C) __syncthreads();      // the list is rewritten by the next pass
    }
  }
  if (!waited) tc::mbar_wait(bar, 0);        // nothing started here: the copy must still land before the CTA's memory is released
}


}  // namespace fod

#ifdef FOD_ROI_PROF
extern "C" int fod_roi_prof(long long* out8, int reset) {
  if (reset) {
    long long z[8] = {0};
    cudaMemcpyToSymbol(fod::g_roi_prof, z, sizeof(z));
  } else {
    cudaMemcpyFromSymbol(out8, fod::g_roi_prof, sizeof(long long) * 8);
  }
  return 0;
}
#endif

using namespace fod;

// The workspace of one call of n = problems * roi_cap ROIs: blobs | tile tap lists | scan summaries | slow list (count +
// entries).  Only resolution 8, where the tile-stationary path can run, has the parts after the blobs.
struct RoiWorkspace {
  size_t tiles, sums, slow;   // byte offsets
  size_t bytes;
};
static RoiWorkspace roi_workspace(size_t n, int resolution) {
  static_assert(sizeof(RoiBlob<8>) % 16 == 0 && sizeof(RoiTile) == 1024 && sizeof(RoiSum) == 48, "workspace layout");
  RoiWorkspace w;
  w.tiles = n * (resolution == 4 ? sizeof(RoiBlob<4>) : resolution == 8 ? sizeof(RoiBlob<8>) : sizeof(RoiBlob<14>));
  w.sums = w.tiles + n * sizeof(RoiTile);
  w.slow = w.sums + n * sizeof(RoiSum);
  w.bytes = resolution == 8 ? w.slow + ((n + 1) * sizeof(int32_t) + 15) / 16 * 16 : w.tiles;
  return w;
}

// One CTA per ROI and 128-channel block, after the pre-pass has written every ROI's blob.
template <int R>
static void launch_per_roi(const RoiParams& prm, unsigned P, const float* rois, const int32_t* roi_count, void* workspace,
                           float* pooled, int32_t* out_level, cudaStream_t st) {
  auto* blobs = static_cast<RoiBlob<R>*>(workspace);
  roi_tables_kernel<R><<<dim3((unsigned)((prm.roi_cap * 2 * R + 255) / 256), P), 256, 0, st>>>(prm, rois, roi_count, blobs,
                                                                                             out_level);
  roi_align_kernel<R><<<dim3(prm.roi_cap, P, (unsigned)(prm.pix / kC)), R * 64, 0, st>>>(prm, roi_count, blobs, pooled);
}

// tile_stationary: 1 = the tile-stationary kernel where it applies (resolution 8, 128 channels), 0 = one CTA per ROI
static int roi_align_impl(const float* const* feat, const fod_level_t* levels, int num_levels, int batch,
                          int problems_per_image, const float* rois, const int32_t* roi_count, int roi_cap,
                          int resolution, int channels, int tiled, float* pooled, int32_t* out_level,
                          void* workspace, fod_stream_t stream, int tile_stationary) {
  FOD_REQUIRE(feat && levels && rois && pooled && workspace, "fod_roi_align: null pointer");
  FOD_REQUIRE(((uintptr_t)workspace & 15) == 0, "fod_roi_align: workspace must be 16-byte aligned");
  FOD_REQUIRE(num_levels >= 1 && num_levels <= FOD_MAX_LEVELS, "fod_roi_align: num_levels %d out of range", num_levels);
  FOD_REQUIRE(batch >= 0 && problems_per_image > 0 && roi_cap > 0, "fod_roi_align: bad sizes");
  FOD_REQUIRE(resolution == 8 || resolution == 4 || resolution == 14,
              "fod_roi_align: pooler resolution must be 8, 4 (POOLER_RESOLUTION / _2) or 14 (the C4 heads)");
  FOD_REQUIRE(channels >= kC && channels % kC == 0 && channels / kC <= 65535, "fod_roi_align: channels must be a multiple of 128");
  long P = (long)batch * problems_per_image;
  if (P == 0) return FOD_OK;
  FOD_REQUIRE(P <= 65535, "fod_roi_align: batch*classes %ld > 65535", P);
  RoiParams prm;
  for (int l = 0; l < num_levels; ++l) {
    FOD_REQUIRE(feat[l], "fod_roi_align: null level pointer");
    FOD_REQUIRE(levels[l].stride > 0 && (levels[l].stride & (levels[l].stride - 1)) == 0,
                "fod_roi_align: stride must be a power of two");
    if (l) FOD_REQUIRE(levels[l].stride == 2 * levels[l - 1].stride, "fod_roi_align: strides must form a pyramid");
    prm.feat[l] = feat[l];
    prm.H[l] = levels[l].height;
    prm.W[l] = levels[l].width;
    prm.stride[l] = levels[l].stride;
  }
  prm.num_levels = num_levels;
  prm.C = problems_per_image;
  prm.roi_cap = roi_cap;
  prm.pix = channels;
  FOD_REQUIRE(!tiled || (resolution == 8 && channels == kC), "fod_roi_align: the tiled layout needs resolution 8 and 128 channels");
  prm.tiled = tiled ? 1 : 0;
  cudaStream_t st = as_stream(stream);
  if (tile_stationary && resolution == 8 && channels == kC) {
    const RoiWorkspace ws = roi_workspace((size_t)P * roi_cap, resolution);
    uint8_t* base = static_cast<uint8_t*>(workspace);
    auto* blobs = reinterpret_cast<RoiBlob<8>*>(base);
    auto* tiles = reinterpret_cast<RoiTile*>(base + ws.tiles);
    auto* sums = reinterpret_cast<RoiSum*>(base + ws.sums);
    auto* slow = reinterpret_cast<int32_t*>(base + ws.slow);
    rt::Params tp;
    int total = 0;
    for (int l = 0; l < num_levels; ++l) {
      const int rc = make_nhwc_map(&tp.map[l], feat[l], batch, prm.H[l], prm.W[l], kC, kC, kC, rt::kEdge, rt::kEdge, 1,
                                   CU_TENSOR_MAP_SWIZZLE_NONE);
      if (rc != FOD_OK) return rc;
      tp.feat[l] = feat[l];
      tp.H[l] = prm.H[l];
      tp.W[l] = prm.W[l];
      tp.tiles_x[l] = (prm.W[l] + rt::kOwn - 1) / rt::kOwn;
      total += tp.tiles_x[l] * ((prm.H[l] + rt::kOwn - 1) / rt::kOwn);
      tp.tile_end[l] = total;
    }
    for (int l = num_levels; l < FOD_MAX_LEVELS; ++l) {
      tp.map[l] = tp.map[0];
      tp.feat[l] = feat[0];
      tp.H[l] = prm.H[0]; tp.W[l] = prm.W[0]; tp.tiles_x[l] = tp.tiles_x[0]; tp.tile_end[l] = total;
    }
    tp.num_levels = num_levels;
    tp.C = problems_per_image;
    tp.roi_cap = roi_cap;
    tp.tiled = tiled ? 1 : 0;
    FOD_CUDA_CALL(cudaFuncSetAttribute(roi_align_tiles_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rt::kSmemAlloc));
    FOD_CUDA_CALL(cudaFuncSetAttribute(roi_align_tiles_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                       (int)cudaSharedmemCarveoutMaxShared));
    FOD_CUDA_CALL(cudaMemsetAsync(slow, 0, sizeof(int32_t), st));
    const dim3 tgrid8((unsigned)((roi_cap * 16 + 255) / 256), (unsigned)P);
    roi_tile_tables_kernel<<<tgrid8, 256, 0, st>>>(prm, rois, roi_count, tiles, sums, blobs, slow, out_level);
    roi_align_tiles_kernel<<<dim3((unsigned)total, (unsigned)batch), rt::kThreads, rt::kSmemAlloc, st>>>(tp, roi_count, tiles,
                                                                                                     sums, pooled);
    roi_align_list_kernel<<<74, 512, 0, st>>>(prm, slow, blobs, pooled);
  } else if (resolution == 8) {
    launch_per_roi<8>(prm, (unsigned)P, rois, roi_count, workspace, pooled, out_level, st);
  } else if (resolution == 4) {
    launch_per_roi<4>(prm, (unsigned)P, rois, roi_count, workspace, pooled, out_level, st);
  } else {
    launch_per_roi<14>(prm, (unsigned)P, rois, roi_count, workspace, pooled, out_level, st);
  }
  FOD_CUDA_LAUNCH_CHECK("fod_roi_align");
  return FOD_OK;
}

extern "C" int fod_roi_align_wide(const float* const* feat, const fod_level_t* levels, int num_levels, int batch,
                                  int problems_per_image, const float* rois, const int32_t* roi_count, int roi_cap,
                                  int resolution, int channels, int tiled, float* pooled, int32_t* out_level,
                                  void* workspace, fod_stream_t stream) {
  return roi_align_impl(feat, levels, num_levels, batch, problems_per_image, rois, roi_count, roi_cap, resolution, channels,
                        tiled, pooled, out_level, workspace, stream, 1);
}

extern "C" int fod_roi_align_per_roi(const float* const* feat, const fod_level_t* levels, int num_levels, int batch,
                                     int problems_per_image, const float* rois, const int32_t* roi_count, int roi_cap,
                                     int resolution, int channels, int tiled, float* pooled, int32_t* out_level,
                                     void* workspace, fod_stream_t stream) {
  return roi_align_impl(feat, levels, num_levels, batch, problems_per_image, rois, roi_count, roi_cap, resolution, channels,
                        tiled, pooled, out_level, workspace, stream, 0);
}

extern "C" size_t fod_roi_align_workspace_bytes(int num_problems, int roi_cap, int resolution) {
  return roi_workspace((size_t)num_problems * roi_cap, resolution).bytes;
}

extern "C" int fod_roi_align(const float* const* feat, const fod_level_t* levels, int num_levels, int batch,
                             int problems_per_image, const float* rois, const int32_t* roi_count, int roi_cap,
                             int resolution, int tiled, float* pooled, int32_t* out_level, void* workspace,
                             fod_stream_t stream) {
  return fod_roi_align_wide(feat, levels, num_levels, batch, problems_per_image, rois, roi_count, roi_cap, resolution, kC,
                            tiled, pooled, out_level, workspace, stream);
}
