// Memory-bound glue between the tensor-core convolutions of the feature extractor (d2!/modeling/backbone/vovnet.py):
//   * fod_stem_patches   - im2col of the 3-channel stem convolution (3x3, stride 2, pad 1, vovnet.py stem_1): each output
//                          pixel gets its 27 input values (+5 zeros) as one 128-byte row, so stem_1 runs as a 1x1
//                          tensor-core convolution with K = 32 instead of a 3-channel cuDNN kernel.
//   * fod_maxpool3x3s2   - nn.MaxPool2d(3, stride 2, ceil_mode=True) of the OSA stages (vovnet.py _OSA_stage) over NHWC
//                          maps, optionally multiplied by the eSE gate of the producing stage (x * hsigmoid(fc(avg(x))),
//                          vovnet.py eSEModule; the gate is >= 0, so it commutes with the max), written straight into a
//                          channel slice of the next stage's concat buffer.
// One float4 (4 channels) per thread, coalesced 128-bit accesses; the 9-fold window overlap is served by L1/L2.
#include "common.cuh"
#include "split_format.cuh"

namespace fod {
namespace glue {

constexpr int kThreads = 256;

// x: [N][H][W][3] fp32 (normalised image, NHWC) -> p: [N][Ho][Wo][32], k = (ky*3 + kx)*3 + c, rows 27..31 zero
__global__ void __launch_bounds__(kThreads) stem_patches_kernel(const float* __restrict__ x, int H, int W, int Ho, int Wo,
                                                                float* __restrict__ p, size_t total) {
  for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < total; i += (size_t)gridDim.x * kThreads) {
    const int q = (int)(i & 7);  // float4 index inside the 32-wide row
    const size_t pix = i >> 3;
    const int ox = (int)(pix % Wo);
    const size_t r = pix / Wo;
    const int oy = (int)(r % Ho);
    const size_t n = r / Ho;
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = q * 4 + j;
      float val = 0.f;
      if (k < 27) {
        const int tap = k / 3, c = k - tap * 3;
        const int ky = tap / 3, kx = tap - ky * 3;
        const int iy = 2 * oy + ky - 1, ix = 2 * ox + kx - 1;
        if (iy >= 0 && iy < H && ix >= 0 && ix < W) val = __ldg(x + ((n * H + iy) * (size_t)W + ix) * 3 + c);
      }
      v[j] = val;
    }
    *reinterpret_cast<float4*>(p + i * 4) = make_float4(v[0], v[1], v[2], v[3]);
  }
}

// Same rows straight from the raw image: x [N][3][H][W] uint8 planar (the dataset mapper's CHW tensors, stacked),
// normalised on the fly as (x - mean[c]) / std[c] (fsod_cen.py:540-555; IEEE division, identical to the torch ops).
__global__ void __launch_bounds__(kThreads) stem_patches_u8_kernel(const uint8_t* __restrict__ x, int H, int W, int Ho, int Wo,
                                                                   float m0, float m1, float m2, float s0, float s1, float s2,
                                                                   float* __restrict__ p, size_t total) {
  for (size_t i = (size_t)blockIdx.x * kThreads + threadIdx.x; i < total; i += (size_t)gridDim.x * kThreads) {
    const int q = (int)(i & 7);
    const size_t pix = i >> 3;
    const int ox = (int)(pix % Wo);
    const size_t r = pix / Wo;
    const int oy = (int)(r % Ho);
    const size_t n = r / Ho;
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = q * 4 + j;
      float val = 0.f;
      if (k < 27) {
        const int tap = k / 3, c = k - tap * 3;
        const int ky = tap / 3, kx = tap - ky * 3;
        const int iy = 2 * oy + ky - 1, ix = 2 * ox + kx - 1;
        if (iy >= 0 && iy < H && ix >= 0 && ix < W) {
          const float raw = (float)__ldg(x + ((n * 3 + c) * (size_t)H + iy) * W + ix);
          const float mean = c == 0 ? m0 : (c == 1 ? m1 : m2), sd = c == 0 ? s0 : (c == 1 ? s1 : s2);
          val = __fdiv_rn(__fsub_rn(raw, mean), sd);
        }
      }
      v[j] = val;
    }
    *reinterpret_cast<float4*>(p + i * 4) = make_float4(v[0], v[1], v[2], v[3]);
  }
}

// stem_1 in one pass on the CUDA cores: raw uint8 planar image -> normalise -> 3x3 / stride 2 / pad 1 convolution with 64
// output channels (BN folded) -> ReLU -> NHWC fp32.  27 x 64 FMAs per output pixel are too few for the tensor-core
// pipeline to pay (the im2col rows alone are 2.5x the bytes of the result), and the layer is bound by writing its
// 1.7 GB result.  Four adjacent lanes share a pixel; lane j owns channels {16 i + 4 j .. + 3 : i = 0..3}, so every
// store instruction of a warp writes 8 x 64 contiguous bytes; the weights sit in shared memory as [27][64].
constexpr int kStemC = 64;
__global__ void __launch_bounds__(kThreads) stem1_u8_kernel(const uint8_t* __restrict__ x, int H, int W, int Ho, int Wo,
                                                            float m0, float m1, float m2, float s0, float s1, float s2,
                                                            const float* __restrict__ w /*[64][27] = OIHW*/,
                                                            const float* __restrict__ bias, float* __restrict__ y,
                                                            float* __restrict__ y_amax, size_t total_pairs, int pairs_per_row) {
  __shared__ __align__(16) float ws[27][kStemC];
  __shared__ __align__(16) float bs[kStemC];
  __shared__ float lut[3][257];   // (v - mean[c]) / std[c] for the 256 raw values (IEEE division, as torch); [256] = padding
  for (int i = threadIdx.x; i < 27 * kStemC; i += kThreads) {
    const int co = i % kStemC, k = i / kStemC;         // k = (ky*3 + kx)*3 + c  <-  OIHW index (c*3 + ky)*3 + kx
    const int tap = k / 3, c = k - tap * 3;
    ws[k][co] = w[co * 27 + c * 9 + tap];
  }
  for (int i = threadIdx.x; i < kStemC; i += kThreads) bs[i] = bias ? bias[i] : 0.f;
  for (int i = threadIdx.x; i < 3 * 257; i += kThreads) {
    const int c = i / 257, v = i - c * 257;
    lut[c][v] = v == 256 ? 0.f : __fdiv_rn(__fsub_rn((float)v, c == 0 ? m0 : (c == 1 ? m1 : m2)), c == 0 ? s0 : (c == 1 ? s1 : s2));
  }
  __syncthreads();
  const int j = threadIdx.x & 3;
  const size_t plane = (size_t)H * W;
  float vmax = 0.f;
  // a group of four lanes computes two horizontally adjacent output pixels (their windows share an input column)
  for (size_t pr = ((size_t)blockIdx.x * kThreads + threadIdx.x) >> 2; pr < total_pairs; pr += ((size_t)gridDim.x * kThreads) >> 2) {
    const int px = (int)(pr % pairs_per_row);
    const size_t r = pr / pairs_per_row;
    const int oy = (int)(r % Ho);
    const size_t n = r / Ho;
    const int ox = 2 * px;
    const bool second = ox + 1 < Wo;
    float4 acc[2][4];
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[0][i] = acc[1][i] = *reinterpret_cast<const float4*>(&bs[16 * i + 4 * j]);
    const uint8_t* img = x + n * 3 * plane;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      const int iy = 2 * oy + ky - 1;
      const bool rowin = iy >= 0 && iy < H;
      const uint8_t* rowp = img + (size_t)(rowin ? iy : 0) * W;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        float v[5];   // input columns 2*ox - 1 .. 2*ox + 3 of this row and channel
#pragma unroll
        for (int q = 0; q < 5; ++q) {
          const int ix = 2 * ox - 1 + q;
          const bool in = rowin && ix >= 0 && ix < W;
          const int raw = in ? (int)__ldg(rowp + c * plane + ix) : 256;
          v[q] = lut[c][raw];
        }
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const int k = (ky * 3 + kx) * 3 + c;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float4 wv = *reinterpret_cast<const float4*>(&ws[k][16 * i + 4 * j]);
            acc[0][i].x = fmaf(v[kx], wv.x, acc[0][i].x); acc[0][i].y = fmaf(v[kx], wv.y, acc[0][i].y);
            acc[0][i].z = fmaf(v[kx], wv.z, acc[0][i].z); acc[0][i].w = fmaf(v[kx], wv.w, acc[0][i].w);
            acc[1][i].x = fmaf(v[kx + 2], wv.x, acc[1][i].x); acc[1][i].y = fmaf(v[kx + 2], wv.y, acc[1][i].y);
            acc[1][i].z = fmaf(v[kx + 2], wv.z, acc[1][i].z); acc[1][i].w = fmaf(v[kx + 2], wv.w, acc[1][i].w);
          }
        }
      }
    }
    const size_t pix = (n * Ho + oy) * (size_t)Wo + ox;
#pragma unroll
    for (int p = 0; p < 2; ++p) {
      if (p == 1 && !second) break;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 a = acc[p][i];
        const float4 o = make_float4(fmaxf(a.x, 0.f), fmaxf(a.y, 0.f), fmaxf(a.z, 0.f), fmaxf(a.w, 0.f));
        vmax = fmaxf(fmaxf(vmax, fmaxf(o.x, o.y)), fmaxf(o.z, o.w));
        *reinterpret_cast<float4*>(y + (pix + p) * kStemC + 16 * i + 4 * j) = o;
      }
    }
  }
  if (y_amax) {
    const uint32_t wm = __reduce_max_sync(0xffffffffu, __float_as_uint(vmax));
    if ((threadIdx.x & 31) == 0 && wm) atomicMax(reinterpret_cast<unsigned int*>(y_amax), wm);
  }
}

// The same layer, tiled (the version fod_stem1_u8 launches).  The kernel above is bound by the shared-memory pipe (128
// bytes per cycle and SM delivered into registers): every lane re-reads the weights per two pixels and looks its inputs
// up one by one, ~580 LSU cycles per 1024 outputs against 216 FMA cycles, and its scalar FFMAs run at half of the FP32
// peak, which Blackwell only reaches with the packed FFMA2.  Here a CTA stages the normalised inputs of an 8 x 32 output
// tile ONCE (17 input rows x 3 channels), de-interleaved per input row into three 32-float arrays - column 2p-1, 2p and
// 2p+1 of output pixel p, i.e. the operand of kx = 0, 1, 2 - so that one LDS.128 yields the operands of four adjacent
// pixels as two aligned register pairs.  A warp owns one output row of the tile, a quarter warp 8 adjacent pixels, a
// lane 8 output channels {4l..4l+3, 32+4l..32+4l+3} of those pixels: per tap 4 LDS.128 (8 inputs, 8 weights) feed 32
// FFMA2 (accumulators are pixel pairs of one channel, the weight is duplicated into a register pair), which balances the
// two pipes, and the 8 lanes of a quarter write 128 contiguous bytes per store.  The summation order (bias, then ky, c,
// kx) is the order of the kernel above: identical results.
constexpr int kS1TileY = 8, kS1TileX = 32, kS1Rows = 2 * kS1TileY + 1;
__global__ void __launch_bounds__(kThreads, 2) stem1_u8_tile_kernel(const uint8_t* __restrict__ x, int H, int W, int Ho, int Wo,
                                                                    float m0, float m1, float m2, float s0, float s1, float s2,
                                                                    const float* __restrict__ w /*[64][27] = OIHW*/,
                                                                    const float* __restrict__ bias, float* __restrict__ y,
                                                                    float* __restrict__ y_amax, int amax_per_image,
                                                                    int tiles_x, int tiles_y, long total_tiles) {
  __shared__ __align__(16) float vs[kS1Rows][3][3 * kS1TileX];   // [input row][channel][kx][pixel]
  __shared__ __align__(16) float ws[27][kStemC];
  __shared__ __align__(16) float bs[kStemC];
  __shared__ float lut[3][257];
  for (int i = threadIdx.x; i < 27 * kStemC; i += kThreads) {
    const int co = i % kStemC, k = i / kStemC;         // k = (ky*3 + kx)*3 + c  <-  OIHW index (c*3 + ky)*3 + kx
    const int tap = k / 3, c = k - tap * 3;
    ws[k][co] = w[co * 27 + c * 9 + tap];
  }
  for (int i = threadIdx.x; i < kStemC; i += kThreads) bs[i] = bias ? bias[i] : 0.f;
  for (int i = threadIdx.x; i < 3 * 257; i += kThreads) {
    const int c = i / 257, v = i - c * 257;
    lut[c][v] = v == 256 ? 0.f : __fdiv_rn(__fsub_rn((float)v, c == 0 ? m0 : (c == 1 ? m1 : m2)), c == 0 ? s0 : (c == 1 ? s1 : s2));
  }
  const int lane = threadIdx.x & 31, wr = threadIdx.x >> 5;
  const int q = lane >> 3, cl = lane & 7;   // pixels 8q .. 8q+7 of the warp's row; channels 4cl .. +3 and 32 + 4cl .. +3
  const size_t plane = (size_t)H * W;
  float vmax = 0.f;
  // Staging item = (input row r, channel c, group t of four input columns 2*ox0 + 4t .. + 3), t = -1 .. 15 (t = -1 only
  // supplies column 2*ox0 - 1, the kx = 0 operand of the tile's first pixel): 17 x 3 x 17 = 867 items, <= 4 per thread.
  // The raw bytes of the NEXT tile are fetched into registers before the current tile is computed (the loads fly during
  // the FMAs); after the barrier they go through the normalisation table into shared memory.
  constexpr int kItems = kS1Rows * 3 * 17, kPerThread = (kItems + kThreads - 1) / kThreads;
  uint32_t raw[kPerThread];
  uint32_t okmask = 0;   // 4 validity bits per item (a byte outside the image is the zero padding)
  auto tile_origin = [&](int tile, int& oy0, int& ox0, size_t& n) {
    const int tx = tile % tiles_x, tr = tile / tiles_x;
    const int ty = tr % tiles_y;
    n = (size_t)(tr / tiles_y);
    oy0 = ty * kS1TileY;
    ox0 = tx * kS1TileX;
  };
  auto fetch = [&](int tile) {
    int oy0, ox0;
    size_t n;
    tile_origin(tile, oy0, ox0, n);
    const uint8_t* img = x + n * 3 * plane;
    okmask = 0;
#pragma unroll
    for (int k = 0; k < kPerThread; ++k) {
      const int idx = (int)threadIdx.x + k * kThreads;
      raw[k] = 0;
      if (idx < kItems) {
        const int t = idx % 17 - 1, rc = idx / 17;
        const int c = rc % 3, r = rc / 3;
        const int iy = 2 * oy0 - 1 + r, col0 = 2 * ox0 + 4 * t;
        if (iy >= 0 && iy < H) {
          const uint8_t* src = img + c * plane + (size_t)iy * W + col0;
          if (col0 >= 0 && col0 + 3 < W && ((reinterpret_cast<uintptr_t>(src) & 3) == 0)) {
            raw[k] = __ldg(reinterpret_cast<const uint32_t*>(src));
            okmask |= 0xFu << (4 * k);
          } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
              if (col0 + j >= 0 && col0 + j < W) {
                raw[k] |= (uint32_t)__ldg(src + j) << (8 * j);
                okmask |= 1u << (4 * k + j);
              }
          }
        }
      }
    }
  };
  auto stage = [&]() {
#pragma unroll
    for (int k = 0; k < kPerThread; ++k) {
      const int idx = (int)threadIdx.x + k * kThreads;
      if (idx < kItems) {
        const int t = idx % 17 - 1, rc = idx / 17;
        const int c = rc % 3, r = rc / 3;
        float* row = &vs[r][c][0];
        const float* lc = lut[c];
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = lc[((okmask >> (4 * k + j)) & 1u) ? (int)((raw[k] >> (8 * j)) & 255u) : 256];
        if (t < 0) {
          row[0] = v[3];
        } else {
          const int p = 2 * t;
          *reinterpret_cast<float2*>(row + kS1TileX + p) = make_float2(v[0], v[2]);       // kx = 1: columns 2p, 2p + 2
          *reinterpret_cast<float2*>(row + 2 * kS1TileX + p) = make_float2(v[1], v[3]);   // kx = 2: columns 2p + 1, 2p + 3
          row[p + 1] = v[1];                                                              // kx = 0 of pixel p + 1
          if (p + 2 < kS1TileX) row[p + 2] = v[3];                                        // kx = 0 of pixel p + 2
        }
      }
    }
  };
  const int total = (int)total_tiles;
  int tile = (int)blockIdx.x;
  if (tile < total) fetch(tile);
  for (; tile < total; tile += (int)gridDim.x) {
    int oy0, ox0;
    size_t n;
    tile_origin(tile, oy0, ox0, n);
    __syncthreads();   // the previous tile has been consumed (and, the first time, the tables above are written)
    stage();
    __syncthreads();
    if (tile + (int)gridDim.x < total) fetch(tile + (int)gridDim.x);
    const int oy = oy0 + wr;
    if (oy < Ho) {   // (uniform per warp; the barriers are at the top of the loop and every warp reaches them)
    float2 acc[4][8];         // [pixel pair m: pixels 8q + 2m, + 1][channel j]
    {
      const float4 b0 = *reinterpret_cast<const float4*>(&bs[4 * cl]), b1 = *reinterpret_cast<const float4*>(&bs[32 + 4 * cl]);
      const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int m = 0; m < 4; ++m)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[m][j] = make_float2(bb[j], bb[j]);
    }
#pragma unroll 1
    for (int ky = 0; ky < 3; ++ky) {
      const int r = 2 * wr + ky;
#pragma unroll 1
      for (int c = 0; c < 3; ++c) {
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const int k = (ky * 3 + kx) * 3 + c;
          const float4 w0 = *reinterpret_cast<const float4*>(&ws[k][4 * cl]);
          const float4 w1 = *reinterpret_cast<const float4*>(&ws[k][32 + 4 * cl]);
          const float* arr = &vs[r][c][kx * kS1TileX + 8 * q];
          const float4 va = *reinterpret_cast<const float4*>(arr), vb = *reinterpret_cast<const float4*>(arr + 4);
          const float2 vp[4] = {make_float2(va.x, va.y), make_float2(va.z, va.w), make_float2(vb.x, vb.y), make_float2(vb.z, vb.w)};
          const float wj[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
          // m outer: consecutive FFMA2s share the 64-bit input pair (operand-reuse cache), the weight is the 32-bit
          // scalar-broadcast operand: fewer register-file reads per instruction
#pragma unroll
          for (int m = 0; m < 4; ++m)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[m][j] = __ffma2_rn(vp[m], make_float2(wj[j], wj[j]), acc[m][j]);
        }
      }
    }
    float* out = y + ((n * Ho + oy) * (size_t)Wo + ox0 + 8 * q) * kStemC + 4 * cl;
#pragma unroll
    for (int m = 0; m < 4; ++m) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {   // pixel 8q + 2m + h
        if (ox0 + 8 * q + 2 * m + h >= Wo) continue;
        float4 lo, hi;
        if (h == 0) {
          lo = make_float4(acc[m][0].x, acc[m][1].x, acc[m][2].x, acc[m][3].x);
          hi = make_float4(acc[m][4].x, acc[m][5].x, acc[m][6].x, acc[m][7].x);
        } else {
          lo = make_float4(acc[m][0].y, acc[m][1].y, acc[m][2].y, acc[m][3].y);
          hi = make_float4(acc[m][4].y, acc[m][5].y, acc[m][6].y, acc[m][7].y);
        }
        lo = make_float4(fmaxf(lo.x, 0.f), fmaxf(lo.y, 0.f), fmaxf(lo.z, 0.f), fmaxf(lo.w, 0.f));
        hi = make_float4(fmaxf(hi.x, 0.f), fmaxf(hi.y, 0.f), fmaxf(hi.z, 0.f), fmaxf(hi.w, 0.f));
        vmax = fmaxf(vmax, fmaxf(fmaxf(fmaxf(lo.x, lo.y), fmaxf(lo.z, lo.w)), fmaxf(fmaxf(hi.x, hi.y), fmaxf(hi.z, hi.w))));
        float* o = out + (size_t)(2 * m + h) * kStemC;
        *reinterpret_cast<float4*>(o) = lo;
        *reinterpret_cast<float4*>(o + 32) = hi;
      }
    }
    }
    if (y_amax && amax_per_image) {   // this tile's image: max|y| per image, so that no image's scale depends on its batch mates
      const uint32_t wm = __reduce_max_sync(0xffffffffu, __float_as_uint(vmax));
      if ((threadIdx.x & 31) == 0 && wm) atomicMax(reinterpret_cast<unsigned int*>(y_amax + n), wm);
      vmax = 0.f;
    }
  }
  if (y_amax && !amax_per_image) {
    const uint32_t wm = __reduce_max_sync(0xffffffffu, __float_as_uint(vmax));
    if ((threadIdx.x & 31) == 0 && wm) atomicMax(reinterpret_cast<unsigned int*>(y_amax), wm);
  }
}

// x: [N][H][W] pixels of xs floats (first C used), gate: [N][C] or null -> y: [N][Ho][Wo] pixels of ys floats.
// Grid (x: blocks over one output row's (pixel, 4-channel group) items, y: output row, z: image): the only division left
// per thread is one 32-bit one (a flat 64-bit index cost three 64-bit div / mod pairs per output, more instructions than
// the nine loads and the maxima).  Consecutive threads take consecutive channel groups of one pixel: 16-byte loads,
// fully coalesced; the 3x3 windows of neighbouring outputs overlap by one column / row, which the L1 serves.
__global__ void __launch_bounds__(kThreads) maxpool_kernel(const float* __restrict__ x, long xs, int H, int W, int C,
                                                           const float* __restrict__ gate, float* __restrict__ y, long ys,
                                                           int Ho, int Wo, const float* __restrict__ y_bound) {
  const int c4n = C >> 2;
  const int item = (int)(blockIdx.x * kThreads + threadIdx.x);
  if (item >= Wo * c4n) return;
  const int ox = item / c4n, c4 = item - ox * c4n;
  const int oy = (int)blockIdx.y;
  const size_t n = blockIdx.z;
  const int y0 = 2 * oy, x0 = 2 * ox;
  const int y1 = min(y0 + 3, H), x1 = min(x0 + 3, W);
  const float* px = x + ((n * H + y0) * (size_t)W + x0) * xs + c4 * 4;
  float4 m = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
  if (y1 - y0 == 3 && x1 - x0 == 3) {   // the full window: nine independent loads
    float4 v[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) v[k] = ldg4(px + ((size_t)(k / 3) * W + (k % 3)) * xs);
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      m.x = fmaxf(m.x, v[k].x); m.y = fmaxf(m.y, v[k].y); m.z = fmaxf(m.z, v[k].z); m.w = fmaxf(m.w, v[k].w);
    }
  } else {
    for (int iy = 0; iy < y1 - y0; ++iy)
      for (int ix = 0; ix < x1 - x0; ++ix) {
        const float4 v = ldg4(px + ((size_t)iy * W + ix) * xs);
        m.x = fmaxf(m.x, v.x); m.y = fmaxf(m.y, v.y); m.z = fmaxf(m.z, v.z); m.w = fmaxf(m.w, v.w);
      }
  }
  if (gate) {
    const float4 g = ldg4(gate + n * C + c4 * 4);
    m.x *= g.x; m.y *= g.y; m.z *= g.z; m.w *= g.w;
  }
  float* out = y + ((n * Ho + oy) * (size_t)Wo + ox) * ys;
  if (y_bound) {
    // the split operand format of the convolutions that read this map (split_format.cuh), 2^e = pow2_scale(y_bound[n]):
    // the consumer derives the same scale
    float sc, unused;
    pow2_scale(__ldg(y_bound + n), sc, unused);
    uint2 hv, lv;
    split_f16x2(m.x * sc, m.y * sc, hv.x, lv.x);
    split_f16x2(m.z * sc, m.w * sc, hv.y, lv.y);
    const int ch = c4 * 4, grp = ch >> 4, q = ch & 15;       // 4 channels = 8 bytes of hi and 8 bytes of lo inside the group
    uint8_t* gb = reinterpret_cast<uint8_t*>(out) + grp * 64;
    *reinterpret_cast<uint2*>(gb + q * 2) = hv;
    *reinterpret_cast<uint2*>(gb + 32 + q * 2) = lv;
  } else {
    *reinterpret_cast<float4*>(out + c4 * 4) = m;
  }
}

}  // namespace glue
}  // namespace fod

using namespace fod;

static unsigned grid_for(size_t total, int threads) {
  size_t b = (total + threads - 1) / threads;
  const size_t cap = 148 * 32;
  return (unsigned)(b < cap ? (b ? b : 1) : cap);
}

extern "C" int fod_stem_patches(const float* x, int n, int h, int w, float* patches, fod_stream_t stream) {
  FOD_REQUIRE(x && patches, "fod_stem_patches: null pointer");
  FOD_REQUIRE(n >= 0 && h > 0 && w > 0, "fod_stem_patches: bad sizes");
  FOD_REQUIRE(((uintptr_t)patches & 15) == 0, "fod_stem_patches: output must be 16-byte aligned");
  if (n == 0) return FOD_OK;
  const int ho = (h - 1) / 2 + 1, wo = (w - 1) / 2 + 1;
  const size_t total = (size_t)n * ho * wo * 8;
  glue::stem_patches_kernel<<<grid_for(total, glue::kThreads), glue::kThreads, 0, as_stream(stream)>>>(x, h, w, ho, wo, patches,
                                                                                                    total);
  FOD_CUDA_LAUNCH_CHECK("fod_stem_patches");
  return FOD_OK;
}

extern "C" int fod_stem_patches_u8(const uint8_t* x, int n, int h, int w, const float* mean3, const float* std3, float* patches,
                                   fod_stream_t stream) {
  FOD_REQUIRE(x && patches && mean3 && std3, "fod_stem_patches_u8: null pointer");
  FOD_REQUIRE(n >= 0 && h > 0 && w > 0, "fod_stem_patches_u8: bad sizes");
  FOD_REQUIRE(((uintptr_t)patches & 15) == 0, "fod_stem_patches_u8: output must be 16-byte aligned");
  if (n == 0) return FOD_OK;
  const int ho = (h - 1) / 2 + 1, wo = (w - 1) / 2 + 1;
  const size_t total = (size_t)n * ho * wo * 8;
  glue::stem_patches_u8_kernel<<<grid_for(total, glue::kThreads), glue::kThreads, 0, as_stream(stream)>>>(
      x, h, w, ho, wo, mean3[0], mean3[1], mean3[2], std3[0], std3[1], std3[2], patches, total);
  FOD_CUDA_LAUNCH_CHECK("fod_stem_patches_u8");
  return FOD_OK;
}

extern "C" int fod_stem1_u8(const uint8_t* x, int n, int h, int w, const float* mean3, const float* std3, const float* weight,
                            const float* bias, float* y, float* y_amax, int amax_per_image, fod_stream_t stream) {
  FOD_REQUIRE(x && y && mean3 && std3 && weight, "fod_stem1_u8: null pointer");
  FOD_REQUIRE(n >= 0 && h > 0 && w > 0, "fod_stem1_u8: bad sizes");
  FOD_REQUIRE(((uintptr_t)y & 15) == 0, "fod_stem1_u8: output must be 16-byte aligned");
  if (n == 0) return FOD_OK;
  const int ho = (h - 1) / 2 + 1, wo = (w - 1) / 2 + 1;
  const int tiles_x = (wo + glue::kS1TileX - 1) / glue::kS1TileX, tiles_y = (ho + glue::kS1TileY - 1) / glue::kS1TileY;
  const long total_tiles = (long)n * tiles_x * tiles_y;
  FOD_REQUIRE(total_tiles < (1L << 31), "fod_stem1_u8: too many tiles");
  int dev = 0, sms = 0;
  FOD_CUDA_CALL(cudaGetDevice(&dev));
  FOD_CUDA_CALL(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const long resident = 2L * (sms > 0 ? sms : 148);   // two CTAs per SM (__launch_bounds__), each loops over tiles
  glue::stem1_u8_tile_kernel<<<(unsigned)(total_tiles < resident ? total_tiles : resident), glue::kThreads, 0, as_stream(stream)>>>(
      x, h, w, ho, wo, mean3[0], mean3[1], mean3[2], std3[0], std3[1], std3[2], weight, bias, y, y_amax, amax_per_image, tiles_x, tiles_y,
      total_tiles);
  FOD_CUDA_LAUNCH_CHECK("fod_stem1_u8");
  return FOD_OK;
}

static int maxpool_impl(const float* x, int n, int h, int w, int c, long x_pixel_stride, const float* gate, float* y,
                        long y_pixel_stride, const float* y_bound, fod_stream_t stream) {
  FOD_REQUIRE(x && y, "fod_maxpool3x3s2_nhwc: null pointer");
  FOD_REQUIRE(n >= 0 && h >= 3 && w >= 3 && c > 0 && c % 4 == 0 && x_pixel_stride % 4 == 0 && y_pixel_stride % 4 == 0 &&
                  x_pixel_stride >= c && y_pixel_stride >= c, "fod_maxpool3x3s2_nhwc: bad sizes (channels / strides multiples of 4)");
  FOD_REQUIRE((((uintptr_t)x | (uintptr_t)y | (uintptr_t)gate) & 15) == 0, "fod_maxpool3x3s2_nhwc: pointers must be 16-byte aligned");
  if (n == 0) return FOD_OK;
  // ceil_mode output size of nn.MaxPool2d(3, 2): ceil((H - 3) / 2) + 1 (the last window always starts inside the map)
  const int ho = (h - 3 + 1) / 2 + 1, wo = (w - 3 + 1) / 2 + 1;
  FOD_REQUIRE(ho <= 65535 && n <= 65535, "fod_maxpool3x3s2_nhwc: more than 65535 output rows or images");
  const dim3 grid((unsigned)(((long)wo * (c / 4) + glue::kThreads - 1) / glue::kThreads), (unsigned)ho, (unsigned)n);
  FOD_REQUIRE(!y_bound || (c % 16 == 0 && y_pixel_stride % 16 == 0), "fod_maxpool3x3s2_nhwc_split: whole 16-channel groups needed");
  glue::maxpool_kernel<<<grid, glue::kThreads, 0, as_stream(stream)>>>(x, x_pixel_stride, h, w, c, gate, y, y_pixel_stride, ho, wo,
                                                                       y_bound);
  FOD_CUDA_LAUNCH_CHECK("fod_maxpool3x3s2_nhwc");
  return FOD_OK;
}

extern "C" int fod_maxpool3x3s2_nhwc(const float* x, int n, int h, int w, int c, long x_pixel_stride, const float* gate,
                                     float* y, long y_pixel_stride, fod_stream_t stream) {
  return maxpool_impl(x, n, h, w, c, x_pixel_stride, gate, y, y_pixel_stride, nullptr, stream);
}

extern "C" int fod_maxpool3x3s2_nhwc_split(const float* x, int n, int h, int w, int c, long x_pixel_stride, const float* gate,
                                           float* y, long y_pixel_stride, const float* y_bound, fod_stream_t stream) {
  FOD_REQUIRE(y_bound, "fod_maxpool3x3s2_nhwc_split: y_bound is required");
  return maxpool_impl(x, n, h, w, c, x_pixel_stride, gate, y, y_pixel_stride, y_bound, stream);
}
