// stem_1 on the 5th-generation tensor cores: raw uint8 image -> (x - mean) / std -> 3x3 / stride 2 / pad 1 convolution,
// 3 -> 64 channels, bias, ReLU -> NHWC fp32.  Replaces the first convolution of the VoVNet stem and the normalisation of
// CenterNet2Detector.preprocess_image (d2!/modeling/backbone/vovnet.py stem_1, fewx/modeling/fsod/fsod_cen.py:540-555).
//
// The layer has K = 27: as a GEMM it is one 32-wide K chunk per 128-pixel tile, and its cost is the 256 bytes per output
// pixel it writes (1.68 GB at batch 64 x 640^2).  The generic convolution kernel (conv_tc.cu) cannot run it at that bound:
// with ONE chunk per tile its per-tile costs are exposed (profiles/r2_ncu_summary.md: 1.17 ms).  This kernel keeps the
// same arithmetic - fp16 hi / lo split of both operands, three kind::f16 MMAs per product, fp32 accumulation in tensor
// memory - around a skeleton made for one chunk per tile:
//   * one persistent CTA per SM, tile = 8 x 16 output pixels, M = 128, N = 64, cta_group::1;
//   * the weights ([64][32] fp16 hi and lo planes, 8 KB) are loaded ONCE by TMA and stay in shared memory;
//   * 8 converter warps (two sets that alternate over the tiles; TMEM quadrant = warp % 4, one pixel per lane) gather the
//     27 im2col columns of their pixel straight from the uint8 planes (independent byte loads, L1 / L2), normalise, scale,
//     split and store them into tensor memory (tcgen05.st): the A operand never exists in shared or global memory;
//   * one thread issues the 6 MMAs of a tile; a tile owns one of four SLOTS (32 A columns + 64 accumulator columns) whose
//     three barriers (A written / MMAs complete / accumulator read) are the whole protocol;
//   * 8 epilogue warps (quadrant x 32-channel half; the bias lives in registers): tcgen05.ld -> rescale, bias, ReLU,
//     max|y| -> the warp's OWN swizzled 4 KB staging box (32 pixels = two tile rows x 32 channels, two buffers) -> its own
//     TMA store, clipped at the image border: no barrier between the epilogue warps.
#include <cuda_fp16.h>

#include "common.cuh"
#include "split_format.cuh"
#include "tc05.cuh"

namespace fod {

using namespace tc;

namespace s1tc {

constexpr int kTileH = 8, kTileW = 16;
constexpr int kCout = 64, kK = 32, kKUsed = 27;
constexpr int kSlots = 4;
constexpr int kWarpMma = 0, kWarpAlloc = 1, kWarpConv0 = 4, kWarpEpi0 = 12;
constexpr int kConvWarps = 8, kEpiWarps = 8;
constexpr int kThreads = (kWarpEpi0 + kEpiWarps) * 32;   // 640

constexpr uint32_t kPlaneBytes = kCout * kK * 2;          // 4096: one fp16 weight plane
constexpr uint32_t kOffB = 0;                             // hi plane, lo plane
constexpr uint32_t kBoxBytes = 32 * 128;                   // 32 pixels x 32 channels fp32
constexpr uint32_t kOffStage = 8192;                      // [epilogue warp][buffer] boxes
constexpr uint32_t kOffLut = kOffStage + kEpiWarps * 2 * kBoxBytes;   // [3][256] normalised, scaled pixel values
constexpr uint32_t kOffBars = kOffLut + 3 * 256 * 4;
constexpr uint32_t kNumBars = 3 * kSlots + 1;
constexpr uint32_t kOffTmemPtr = kOffBars + kNumBars * 8;
constexpr uint32_t kSmemBytes = kOffTmemPtr + 16;
constexpr uint32_t kSmemAlloc = kSmemBytes + 1024;

constexpr uint32_t kTmemCols = 512;
constexpr uint32_t kColA = 0;                             // 4 slots x [hi 16 | lo 16] packed fp16 pairs
constexpr uint32_t kColAcc = kSlots * 32;                 // 4 slots x 64

struct Params {
  CUtensorMap out_map;   // [N][Ho][Wo][Cout] fp32, box 32 channels x 16 x 2 pixels (one epilogue warp's share of a tile)
  CUtensorMap whi_map;   // fp16 [64][32], box 32 x 64
  CUtensorMap wlo_map;
  const uint8_t* x;      // [N][3][H][W]
  const float* bias;     // [64] or null
  const float* w_inv;    // 1 / weight scale (tail of the packed buffer)
  float* y_amax;         // null, [1] or [N]
  int y_amax_per_image;
  const float* y_bound;   // split output: device float >= max(y); y is written as [16 x fp16 hi | 16 x fp16 lo] of y * 2^e per 16 channels
  int H, W, ho, wo;
  int tiles_x, tiles_per_img, tiles_total;
  int std_one;
  float mean[3], std[3];
  float xs, xs_inv;      // operand scale 2^e of the normalised pixels and its inverse
};

// Tile coordinates of a CTA's static schedule t = blockIdx.x, + gridDim.x, ...: carried along with additions and two
// compares instead of two integer divisions per tile and warp (every role walks the same sequence).
struct TileWalk {
  int n, ty, tx;        // image, tile row, tile column of the current tile
  int dn, dty, dtx;     // the same decomposition of the stride gridDim.x
  int tiles_x, tiles_y;
  __device__ __forceinline__ void init(int t0, int step, int tx_count, int ty_count) {
    tiles_x = tx_count;
    tiles_y = ty_count;
    const int per_img = tx_count * ty_count;
    n = t0 / per_img;
    int r = t0 - n * per_img;
    ty = r / tx_count;
    tx = r - ty * tx_count;
    dn = step / per_img;
    r = step - dn * per_img;
    dty = r / tx_count;
    dtx = r - dty * tx_count;
  }
  __device__ __forceinline__ void next() {
    tx += dtx;
    if (tx >= tiles_x) { tx -= tiles_x; ++ty; }
    ty += dty;
    if (ty >= tiles_y) { ty -= tiles_y; ++n; }
    n += dn;
  }
};

__global__ void __launch_bounds__(kThreads, 1) stem1_tc_kernel(const __grid_constant__ Params P) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const uint32_t sbase = smem_u32(smem);
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  const uint32_t bar0 = sbase + kOffBars;
  auto a_full = [&](int s) { return bar0 + 8u * s; };                     // converters -> MMA
  auto acc_full = [&](int s) { return bar0 + 8u * (kSlots + s); };        // MMA commit -> epilogue
  auto slot_free = [&](int s) { return bar0 + 8u * (2 * kSlots + s); };   // epilogue -> converters
  const uint32_t b_full = bar0 + 8u * (3 * kSlots);

  if (tid == 0) {
    for (int s = 0; s < kSlots; ++s) {
      mbar_init(a_full(s), 4);            // the four quadrant warps of one converter set
      mbar_init(acc_full(s), 1);
      mbar_init(slot_free(s), kEpiWarps);
    }
    mbar_init(b_full, 1);
    fence_barrier_init();
  }
  if (warp == kWarpAlloc) {
    tmem_alloc<1>(sbase + kOffTmemPtr, kTmemCols);
    tmem_relinquish<1>();
  }
  if (warp == kWarpMma && lane == 0) {
    tma_prefetch_desc(&P.out_map);
    tma_prefetch_desc(&P.whi_map);
    tma_prefetch_desc(&P.wlo_map);
  }
  {   // ((v - mean) / std) * 2^e for every byte value and channel: the reference's two roundings, then an exact scaling
    float* lut = reinterpret_cast<float*>(smem + kOffLut);
    for (int i = tid; i < 3 * 256; i += kThreads) {
      const int c = i >> 8;
      lut[i] = __fdiv_rn(__fsub_rn((float)(i & 255), P.mean[c]), P.std[c]) * P.xs;
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem + kOffTmemPtr);
  const int total = P.tiles_total, step = (int)gridDim.x;

  if (warp == kWarpMma) {
    // ------------------------------------------------------------------ weights once, then 6 MMAs per tile
    if (lane == 0) {
      mbar_arrive_expect_tx(b_full, 2 * kPlaneBytes);
      tma_load_2d(sbase + kOffB, &P.whi_map, b_full, 0, 0);
      tma_load_2d(sbase + kOffB + kPlaneBytes, &P.wlo_map, b_full, 0, 0);
    }
    mbar_wait(b_full, 0);
    const uint32_t idesc = idesc_f16(128, kCout);
    const uint64_t bhi = smem_desc_k_sw64(sbase + kOffB), blo = smem_desc_k_sw64(sbase + kOffB + kPlaneBytes);
    int i = 0;
    for (int t = (int)blockIdx.x; t < total; t += step, ++i) {
      const int s = i % kSlots;
      mbar_wait(a_full(s), (uint32_t)(i / kSlots) & 1u);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t d = tmem_base + kColAcc + (uint32_t)s * kCout, a0 = tmem_base + kColA + (uint32_t)s * 32;
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {   // K = 16 fp16 per MMA: 8 packed columns of A, 32 bytes of a B row
          const uint32_t ah = a0 + ks * 8, al = ah + 16;
          const uint64_t boff = (uint64_t)((ks * 32) >> 4);
          mma_f16_ts<1>(d, ah, bhi + boff, idesc, ks ? 1u : 0u);
          mma_f16_ts<1>(d, al, bhi + boff, idesc, 1u);
          mma_f16_ts<1>(d, ah, blo + boff, idesc, 1u);
        }
        mma_commit(acc_full(s));
      }
      __syncwarp();
    }
  } else if (warp >= kWarpConv0 && warp < kWarpConv0 + kConvWarps) {
    // ------------------------------------------------------------------ converters: uint8 gather -> tensor memory
    const int cw = warp - kWarpConv0, qd = warp & 3, set = cw >> 2;
    const int m = qd * 32 + lane, py = m >> 4, px = m & 15;
    const uint32_t trow = tmem_base + ((uint32_t)(qd * 32) << 16) + kColA;
    const int H = P.H, W = P.W;
    const size_t plane = (size_t)H * W;
    const float xs = P.xs;
    const float nm0 = -P.mean[0] * xs, nm1 = -P.mean[1] * xs, nm2 = -P.mean[2] * xs;   // exact: xs is a power of two
    const float* lut = reinterpret_cast<const float*>(smem + kOffLut);
    const int tiles_y = P.tiles_per_img / P.tiles_x;
    TileWalk tw;
    tw.init((int)blockIdx.x, step, P.tiles_x, tiles_y);
    int i = 0;
    for (int t = (int)blockIdx.x; t < total; t += step, ++i, tw.next()) {
      if ((i & 1) != set) continue;
      const int n = tw.n, ty = tw.ty, tx = tw.tx;
      const int oy = ty * kTileH + py, ox = tx * kTileW + px;
      const uint8_t* img = P.x + (size_t)n * 3 * plane;
      // a tile whose 17 x 33 input window lies inside the image needs neither clamps nor padding (uniform per warp)
      const bool interior = ty > 0 && tx > 0 && 2 * (ty * kTileH + kTileH - 1) + 1 < H && 2 * (tx * kTileW + kTileW - 1) + 1 < W;
      float v[kK];
      uint32_t raw[kKUsed];
      bool rok[3] = {true, true, true}, cok[3] = {true, true, true};
      if (interior) {
        const uint8_t* p0 = img + (size_t)(2 * oy - 1) * W + (2 * ox - 1);
#pragma unroll
        for (int k = 0; k < kKUsed; ++k) {   // k = (ky*3 + kx)*3 + c
          const int tap = k / 3, c = k - tap * 3, ky = tap / 3, kx = tap - ky * 3;
          raw[k] = __ldg(p0 + c * plane + ky * W + kx);
        }
      } else {
        // every load is issued unconditionally from a clamped address (27 independent loads in flight); the padding is
        // applied to the value
        int rowoff[3], col[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const int iy = 2 * oy - 1 + k, ix = 2 * ox - 1 + k;
          rok[k] = (unsigned)iy < (unsigned)H;
          cok[k] = (unsigned)ix < (unsigned)W;
          rowoff[k] = min(max(iy, 0), H - 1) * W;
          col[k] = min(max(ix, 0), W - 1);
        }
#pragma unroll
        for (int k = 0; k < kKUsed; ++k) {
          const int tap = k / 3, c = k - tap * 3, ky = tap / 3, kx = tap - ky * 3;
          raw[k] = __ldg(img + c * plane + rowoff[ky] + col[kx]);
        }
      }
      if (P.std_one) {
#pragma unroll
        for (int k = 0; k < kKUsed; ++k) {
          const int c = k % 3;
          // (raw - mean) * xs in one rounding: raw * xs and mean * xs are exact, so this is the rounded difference scaled
          v[k] = fmaf((float)raw[k], xs, c == 0 ? nm0 : (c == 1 ? nm1 : nm2));
        }
      } else {   // a division per value would dominate the converter: table look-up (same bits)
#pragma unroll
        for (int k = 0; k < kKUsed; ++k) v[k] = lut[(k % 3) * 256 + raw[k]];
      }
      if (!interior) {
#pragma unroll
        for (int k = 0; k < kKUsed; ++k) {
          const int tap = k / 3, ky = tap / 3, kx = tap - ky * 3;
          v[k] = (rok[ky] && cok[kx]) ? v[k] : 0.f;
        }
      }
#pragma unroll
      for (int k = kKUsed; k < kK; ++k) v[k] = 0.f;
      uint32_t hi[16], lo[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) split_f16x2(v[2 * j], v[2 * j + 1], hi[j], lo[j]);
      const int s = i % kSlots;
      mbar_wait(slot_free(s), ((uint32_t)(i / kSlots) & 1u) ^ 1u);   // the slot's previous accumulator has been read
      tc_fence_after();
      tmem_st16(trow + (uint32_t)s * 32, hi);
      tmem_st16(trow + (uint32_t)s * 32 + 16, lo);
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(a_full(s));
    }
  } else if (warp >= kWarpEpi0) {
    // ------------------------------------------------------------------ epilogue: (quadrant, 32-channel half)
    const int ew = warp - kWarpEpi0, qd = warp & 3, half = ew >> 2;
    const int m = qd * 32 + lane;
    const uint32_t trow = tmem_base + ((uint32_t)(qd * 32) << 16) + kColAcc + (uint32_t)half * 32;
    const uint32_t box0 = sbase + kOffStage + (uint32_t)ew * 2u * kBoxBytes;            // this warp's two staging boxes
    const uint32_t row0 = box0 + (uint32_t)((lane >> 3) * 1024 + (lane & 7) * 128);   // this lane's pixel row
    const float rescale = P.xs_inv * __ldg(P.w_inv);   // undoes the two power-of-two operand scales (exact)
    float ysplit = 0.f, unused;   // != 0: the output leaves as fp16 hi / lo of y * ysplit
    if (P.y_bound) pow2_scale(__ldg(P.y_bound), ysplit, unused);
    float bias[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) bias[j] = P.bias ? __ldg(P.bias + half * 32 + j) : 0.f;
    float vmax = 0.f;
    int vmax_n = -1;   // image the running maximum belongs to
    auto flush_amax = [&]() {   // one atomic per warp and image (outputs are >= 0 after the ReLU)
      const uint32_t wmax = __reduce_max_sync(0xffffffffu, __float_as_uint(vmax));
      if (lane == 0 && wmax && vmax_n >= 0)
        atomicMax(reinterpret_cast<unsigned int*>(P.y_amax + (P.y_amax_per_image ? vmax_n : 0)), wmax);
      vmax = 0.f;
    };
    TileWalk tw;
    tw.init((int)blockIdx.x, step, P.tiles_x, P.tiles_per_img / P.tiles_x);
    int i = 0;
    for (int t = (int)blockIdx.x; t < total; t += step, ++i, tw.next()) {
      const int n = tw.n, ty = tw.ty, tx = tw.tx;
      const int s = i % kSlots;
      const bool px_valid = ty * kTileH + (m >> 4) < P.ho && tx * kTileW + (m & 15) < P.wo;
      if (P.y_amax && n != vmax_n) {
        flush_amax();
        vmax_n = n;
      }
      mbar_wait(acc_full(s), (uint32_t)(i / kSlots) & 1u);
      tc_fence_after();
      uint32_t v[32];
      tmem_ld32(trow + (uint32_t)s * kCout, v);
      tmem_wait_ld();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(slot_free(s));
        tma_store_wait_read<1>();   // this warp's store of the tile before the previous one has left the buffer
      }
      __syncwarp();
      const uint32_t row_s = row0 + (uint32_t)(i & 1) * kBoxBytes;
      float lmax = 0.f;
      if (ysplit != 0.f) {
        // the split operand format (split_format.cuh): per 16 channels 64 bytes = [16 x fp16 hi | 16 x the exact remainders]
        // of y * 2^e
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint32_t hi[4], lo[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int j = c * 8 + q * 2;
            const float a = fmaxf(fmaf(__uint_as_float(v[j]), rescale, bias[j]), 0.f);
            const float b = fmaxf(fmaf(__uint_as_float(v[j + 1]), rescale, bias[j + 1]), 0.f);
            lmax = fmaxf(lmax, fmaxf(a, b));
            split_f16x2(a * ysplit, b * ysplit, hi[q], lo[q]);
          }
          const int hp = (c >> 1) * 4 + (c & 1);      // per 16 channels [16 x hi | 16 x lo]
          asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(row_s + (uint32_t)((hp ^ (lane & 7)) << 4)), "r"(hi[0]),
                       "r"(hi[1]), "r"(hi[2]), "r"(hi[3]) : "memory");
          asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(row_s + (uint32_t)(((hp + 2) ^ (lane & 7)) << 4)), "r"(lo[0]),
                       "r"(lo[1]), "r"(lo[2]), "r"(lo[3]) : "memory");
        }
      } else {
#pragma unroll
        for (int c4 = 0; c4 < 8; ++c4) {
          float4 o;
          o.x = fmaxf(fmaf(__uint_as_float(v[c4 * 4 + 0]), rescale, bias[c4 * 4 + 0]), 0.f);
          o.y = fmaxf(fmaf(__uint_as_float(v[c4 * 4 + 1]), rescale, bias[c4 * 4 + 1]), 0.f);
          o.z = fmaxf(fmaf(__uint_as_float(v[c4 * 4 + 2]), rescale, bias[c4 * 4 + 2]), 0.f);
          o.w = fmaxf(fmaf(__uint_as_float(v[c4 * 4 + 3]), rescale, bias[c4 * 4 + 3]), 0.f);
          lmax = fmaxf(fmaxf(lmax, fmaxf(o.x, o.y)), fmaxf(o.z, o.w));
          sts4s(row_s + (uint32_t)((c4 ^ (lane & 7)) << 4), o);
        }
      }
      if (px_valid) vmax = fmaxf(vmax, lmax);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        tma_store_4d(&P.out_map, box0 + (uint32_t)(i & 1) * kBoxBytes, half * 32, tx * kTileW, ty * kTileH + 2 * qd, n);
        tma_store_commit();
      }
    }
    if (lane == 0) tma_store_wait<0>();
    if (P.y_amax) flush_amax();
  }
  // ---------------------------------------------------------------------- teardown
  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == kWarpAlloc) tmem_dealloc<1>(tmem_base, kTmemCols);
}

}  // namespace s1tc
}  // namespace fod

using namespace fod;

static int stem1_u8_tc_impl(const uint8_t* x, int n, int h, int w, const float* mean3, const float* std3,
                            const float* packed, const float* bias, float* y, long y_pixel_stride, float* y_amax,
                            int amax_per_image, const float* y_bound, fod_stream_t stream) {
  FOD_REQUIRE(x && mean3 && std3 && packed && y, "fod_stem1_u8_tc: null pointer");
  FOD_REQUIRE(n >= 0 && h > 0 && w > 0, "fod_stem1_u8_tc: bad sizes");
  FOD_REQUIRE(y_pixel_stride >= s1tc::kCout && y_pixel_stride % 4 == 0, "fod_stem1_u8_tc: bad output pixel stride");
  FOD_REQUIRE((((uintptr_t)y | (uintptr_t)packed) & 15) == 0, "fod_stem1_u8_tc: pointers must be 16-byte aligned");
  if (n == 0) return FOD_OK;
  s1tc::Params prm;
  memset(&prm, 0, sizeof(prm));
  float bound = 0.f;
  prm.std_one = 1;
  for (int c = 0; c < 3; ++c) {
    FOD_REQUIRE(std3[c] != 0.f && std3[c] == std3[c], "fod_stem1_u8_tc: pixel_std must not be zero");
    prm.mean[c] = mean3[c];
    prm.std[c] = std3[c];
    if (std3[c] != 1.f) prm.std_one = 0;
    const float b = fmaxf(fabsf(0.f - mean3[c]), fabsf(255.f - mean3[c])) / fabsf(std3[c]);
    bound = fmaxf(bound, b);
  }
  {   // 2^e with bound * 2^e in [2^13, 2^14): fixed by the normalisation constants, the same for every image
    int e = 0;
    if (!(bound < 1e30f)) bound = 1e30f;
    const float fr = frexpf(bound > 1e-30f ? bound : 1.f, &e);   // bound = fr * 2^e, fr in [0.5, 1)
    (void)fr;
    prm.xs = ldexpf(1.f, 14 - e);
    prm.xs_inv = ldexpf(1.f, e - 14);
  }
  prm.x = x;
  prm.bias = bias;
  prm.y_amax = y_amax;
  prm.y_amax_per_image = amax_per_image ? 1 : 0;
  prm.y_bound = y_bound;
  prm.H = h;
  prm.W = w;
  prm.ho = (h - 1) / 2 + 1;
  prm.wo = (w - 1) / 2 + 1;
  prm.tiles_x = (prm.wo + s1tc::kTileW - 1) / s1tc::kTileW;
  prm.tiles_per_img = prm.tiles_x * ((prm.ho + s1tc::kTileH - 1) / s1tc::kTileH);
  const long tiles = (long)n * prm.tiles_per_img;
  FOD_REQUIRE(tiles < (1L << 30), "fod_stem1_u8_tc: too many tiles");
  prm.tiles_total = (int)tiles;
  int rc = make_nhwc_map(&prm.out_map, y, n, prm.ho, prm.wo, s1tc::kCout, y_pixel_stride, 32, s1tc::kTileW, 2, 1,
                         CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc != FOD_OK) return rc;
  const __half* whi = reinterpret_cast<const __half*>(packed);
  rc = make_matrix_map_f16(&prm.whi_map, whi, s1tc::kCout, s1tc::kK, s1tc::kK, s1tc::kCout);
  if (rc != FOD_OK) return rc;
  rc = make_matrix_map_f16(&prm.wlo_map, whi + (size_t)s1tc::kCout * s1tc::kK, s1tc::kCout, s1tc::kK, s1tc::kK, s1tc::kCout);
  if (rc != FOD_OK) return rc;
  prm.w_inv = packed + (size_t)s1tc::kCout * s1tc::kK;   // tail[0] = 1 / weight scale
  int dev = 0, sms = 0;
  FOD_CUDA_CALL(cudaGetDevice(&dev));
  FOD_CUDA_CALL(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int grid = tiles < sms ? (int)tiles : sms;
  FOD_CUDA_CALL(cudaFuncSetAttribute(s1tc::stem1_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s1tc::kSmemAlloc));
  s1tc::stem1_tc_kernel<<<grid, s1tc::kThreads, s1tc::kSmemAlloc, as_stream(stream)>>>(prm);
  FOD_CUDA_LAUNCH_CHECK("fod_stem1_u8_tc");
  return FOD_OK;
}

extern "C" int fod_stem1_u8_tc(const uint8_t* x, int n, int h, int w, const float* mean3, const float* std3,
                               const float* packed, const float* bias, float* y, long y_pixel_stride, float* y_amax,
                               int amax_per_image, fod_stream_t stream) {
  return stem1_u8_tc_impl(x, n, h, w, mean3, std3, packed, bias, y, y_pixel_stride, y_amax, amax_per_image, nullptr, stream);
}

extern "C" int fod_stem1_u8_tc_split(const uint8_t* x, int n, int h, int w, const float* mean3, const float* std3,
                                     const float* packed, const float* bias, float* y, long y_pixel_stride, float* y_amax,
                                     int amax_per_image, const float* y_bound, fod_stream_t stream) {
  FOD_REQUIRE(y_bound, "fod_stem1_u8_tc_split: y_bound is required");
  return stem1_u8_tc_impl(x, n, h, w, mean3, std3, packed, bias, y, y_pixel_stride, y_amax, amax_per_image, y_bound, stream);
}
