// H0 (and the convolutions either side of the head): 3x3 / 1x1 convolution over NHWC fp32 maps as an implicit GEMM on
// the 5th-generation tensor cores with fp32 accuracy, bias + ReLU epilogue.
// Replaces the F.conv2d -> cuDNN calls of CenterNetHead (CenterNet2/centernet/modeling/dense_heads/centernet_head.py:
// 141-161) and of the VoVNet/FPN modules that feed the head (d2!/modeling/backbone/vovnet.py, fpn.py), which cuDNN
// serves on sm_100 with fp32 SIMT / FFT engines when TF32 is off.
//
//   y[n][oy][ox][co] = act( bias[co] + sum_{ky,kx,ci} w[co][ky][kx][ci] * x[n][oy*s + ky - pad][ox*s + kx - pad][ci] )
//   (stride s in {1, 2}, pad = ksize / 2, zero padding)
//
// Arithmetic: every fp32 operand is split as x * 2^e = hi + lo with hi = fp16(x * 2^e), lo = fp16(x * 2^e - hi)
// (22 significant bits, the same as a tf32 hi/lo split) and the product is hi.hi + lo.hi + hi.lo on kind::f16 MMAs with
// fp32 accumulation.  The power-of-two scale 2^e puts the largest magnitude of the tensor into [2^13, 2^14), so nothing
// overflows fp16 and what underflows is below 2^-38 of that maximum; it is exact and is undone in the epilogue.  The
// caller passes an upper bound of max|x| (device scalar, normally written by the kernel that produced x: this kernel's
// own epilogue reports max|y|); the weights' scale is fixed when they are packed.  Against the 3xTF32 version of this
// kernel (K = 8 per MMA, one MMA per 45 cycles at best) kind::f16 moves K = 16 per MMA in 64 cycles at N = 128 and in
// 32 cycles at N = 64 (tools/f16_probe.cu): half the tensor time for the same accuracy (measured 4e-7 relative).
//
// Design (B200, sm_100a) - the skeleton of correlate_tc.cu / relation_tc.cu:
//   * work unit = tile of 8 x 16 output pixels of one image (128 GEMM rows) x one group of <= 128 output channels.
//     CTAs run as pairs (cluster of 2, tcgen05 cta_group::2): one MMA covers both CTAs' tiles (M = 256) against the
//     weight group whose rows are split between the two CTAs (each CTA stages only half of every weight chunk).
//   * K = taps x Cin is streamed in 32-channel chunks.  The input tile plus its halo (zero-filled outside the image
//     by TMA, which is the convolution's zero padding) is staged ONCE per 32-channel chunk into a 3-deep shared-memory
//     ring and serves all ksize^2 taps: the shifted A operands are read from it, never re-fetched from L2.
//     (Stride 2: a halo tile would be 17 x 33 pixels, so each tap's 8 x 16 pixels are fetched by their own TMA load
//     with element strides (2, 2) instead: one ring stage per tap.)
//   * 16 converter warps first convert the staged tile IN PLACE to scaled fp16 hi / lo (once per 32 channels, not once
//     per tap), then, per tap, one output pixel per lane (= TMEM lane), move the tap-shifted 128-byte row of their pixel
//     (conflict-free LDS.128 thanks to the TMA swizzle) into TENSOR MEMORY; the MMA reads A from tensor memory and only
//     the weights from shared memory.  Two sets of 8 warps alternate over the taps so that their latencies overlap.
//   * weights: pre-split fp16 hi / lo planes [Cout][taps][Cin_pad] (fod_conv2d_pack_weights), TMA-streamed per chunk
//     into a 6-stage ring (they are L2 resident: <= 0.6 MB per layer).
//   * the tensor core accumulates with round-toward-zero (tools/tc_probe.cu), so the K loop is cut into partial sums
//     of <= 16 chunks (96 MMAs) that the 4 epilogue warps add in IEEE fp32 into a running tile in shared memory; the
//     last part rescales, adds the bias, applies ReLU and the tile leaves through TMA stores (clipped at the image
//     border and at Cout by the tensor map, so the output may be a channel slice of a wider NHWC buffer: concatenation
//     is free).
#include <cuda_fp16.h>

#include "common.cuh"
#include "pair.cuh"
#include "split_format.cuh"

namespace fod {

using namespace tc;

namespace cvt {

constexpr int kTileH = 8, kTileW = 16;
constexpr int kChunk = 32;
constexpr int kQStages = 3, kStages = 6, kAccStages = 2;
constexpr int kPartChunks = 16;
constexpr uint32_t kQStageStrideS1 = ((kTileH + 2) * (kTileW + 2) * 128 + 1023) / 1024 * 1024;   // 23552
constexpr uint32_t kBPlaneMax = 64 * 64;                                    // 64 rows (half of a 128 group) x 32 fp16
constexpr uint32_t kBStageBytes = 2 * kBPlaneMax;                           // hi + lo
constexpr uint32_t kSlabBytes = 128 * 128;                                  // 128 pixels x 32 channels

// shared memory of the tensor-memory pipeline
constexpr uint32_t kOffQ = 0;
constexpr uint32_t kOffB = kOffQ + kQStages * kQStageStrideS1;              // 70656
constexpr uint32_t kOffSum = kOffB + kStages * kBStageBytes;                // running tile / store staging, 4 slabs
constexpr uint32_t kOffBias = kOffSum + 4 * kSlabBytes;
constexpr uint32_t kOffBars = kOffBias + 128 * 4;
constexpr uint32_t kNumBars = 2 * kQStages + 2 * kStages + 2 * kAccStages;
constexpr uint32_t kOffTmemPtr = kOffBars + kNumBars * 8;
constexpr uint32_t kSmemBytes = kOffTmemPtr + 16;
constexpr uint32_t kSmemAlloc = kSmemBytes + 1024;

constexpr int kConvWarps = 16;
constexpr int kWarpTma = 0, kWarpMma = 1, kWarpAlloc = 2, kWarpTmaB = 3, kWarpEpi0 = 4, kWarpConv0 = 8;
constexpr int kThreads = (kWarpConv0 + kConvWarps) * 32;  // 768

constexpr uint32_t kTmemCols = 512;
constexpr uint32_t kAStageCols = 32;                // [hi: 16 columns of packed fp16 pairs | lo: 16]
constexpr uint32_t kColA = 0;                       // 6 stages x 32
constexpr uint32_t kColAcc = kStages * kAStageCols; // 2 stages x 128

#ifdef FOD_DBG
__device__ long long* g_dbg = nullptr;   // [role][g][4] clock64 stamps of pair 0 / rank 0, chunks kDbg0 .. kDbg0 + kDbgN
constexpr uint32_t kDbg0 = 400, kDbgN = 64;
#define DBG_STAMP(role, g, slot)                                                                   \
  do {                                                                                             \
    if (dbg_buf && lane == 0 && (g) >= kDbg0 && (g) < kDbg0 + kDbgN)                               \
      dbg_buf[((role) * kDbgN + ((g) - kDbg0)) * 4 + (slot)] = clock64();                          \
  } while (0)
#else
#define DBG_STAMP(role, g, slot)
#endif

struct Params {   // what both pipelines read
  CUtensorMap in_map;   // [N][H][W][Cin] (pixel stride may exceed Cin), box 32 x halo_w x halo_h
  CUtensorMap out_map;  // [N][Ho][Wo][Cout], box 32 x 16 x 8
  CUtensorMap whi_map;  // fp16 [Cout][taps*Cin_pad], box 32 x nhalf
  CUtensorMap wlo_map;
  const float* bias;    // [Cout] or null
  const float* x_amax;  // [n_amax] upper bounds of max|x| (their maximum is used)
  const float* w_inv;   // 1 / weight scale (tail of the packed buffer)
  float* y_amax;        // null or: atomically raised to max|y|
  float* colsum;        // null or: [N][tiles_per_img][Cout] per-tile channel sums of the output (for the eSE average)
  float* colsumsq;      // null or: same shape, sums of squares (GroupNorm statistics of the output)
  const float* res;     // null or: residual [N][res_h][res_w][cout] (dense NHWC) added before the activation;
  int res_h, res_w, res_shift;   // read at (oy >> res_shift, ox >> res_shift): 0 = same size, 1 = nearest 2x upsampling
  int tiles_x, tiles_per_img, tiles_total;
  int taps, stride, per_tap;  // per_tap: stride 2, every tap (tap row) of a chunk is a TMA load of its own
  int cin_chunks, chunks, parts, chunks_per_part;
  int n_groups, n_group, nhalf, ncol32, cout;
  int relu, num_pairs, pair_units, n_amax, ho, wo;
  int x_amax_stride;    // 0: x_amax holds n_amax scalars (one scale for the whole batch); N: x_amax is [n_amax][N], the scale
                        // of image n comes from column n, so an image's result does not depend on its batch mates
  int y_amax_per_image; // y_amax is [N]: max|y| per image
  // Split hand-off between convolutions (the producer writes the consumer's operand format; same bytes as fp32):
  const float* x_actual;   // null or [N] / [1] like x_amax: the ACTUAL max|x| (x_amax may be the looser bound that fixed the scale
                           // of a pre-split x); only used for the output bound below
  float* y_bound;          // null or [N] / [1]: y is written as [16 x fp16 hi | 16 x fp16 lo] of y * 2^e per pixel and 16 channels,
                           // 2^e = pow2_scale(y_l1 * max|x| + y_beta); that bound is published here for the consumer
  float y_l1, y_beta;      // max_c sum|w[c]| and max|bias| (host constants of the layer)
};

struct TmemA {   // what only the tensor-memory pipeline reads: its input ring and the converters' operand transform
  const float* a_gate;  // null or: [N][Cin] factors multiplied into the input (the eSE gate of the producing stage, or the
                        // per-(image, channel) scale of a normalisation)
  const float* a_shift; // null or: [N][Cin] added after the factor, followed by ReLU if a_relu: x' = act(x * a_gate + a_shift)
                        // for pixels inside the image (the zero padding stays zero): GroupNorm + ReLU of the producer's map
  int a_relu, in_h, in_w, cin;
  int ksize, halo_w;
  uint32_t q_stage_bytes, q_stage_stride;
  int x_presplit;       // x already holds [16 x fp16 hi | 16 x fp16 lo] of x * 2^e per 16 channels (e from x_amax): no conversion pass
  int x_presplit_from;  // single-tap path: input channels >= this are pre-split, each slice at the scale of ITS x_amax row
  int slice_ch[8];      // first channel of the slice that x_amax row k bounds
};

// Shared-memory layout of the shared-memory A pipeline (sized per launch): an A stage is three TMA boxes of a_box_bytes
// at 0; the weights of one tap row (3 taps x hi / lo) form a B stage of b_stage_bytes at off_b, b_stages deep; the
// output staging starts at off_sum
struct SmemA {
  uint32_t a_box_bytes, b_stage_bytes, off_b, off_sum;
  int b_stages;
};

// ---------------------------------------------------------------------------------------------- rules every role shares
// Static schedule: iteration i of pair k owns pair-unit pu = i * num_pairs + k = (tile pair, channel group grp), grp
// innermost so that the pairs working on the same input tile run at the same time (L2 reuse of the halo).  The second
// CTA of the last pair of an odd tile count recomputes the last tile and stores nothing.
struct Unit {
  int n, tt, ty, tx;   // image, tile index within the image, tile row and column
  int ch0;             // first output channel of the group
  bool store;
};
__device__ __forceinline__ bool has_unit(const Params& P, int pair, int i) { return i * P.num_pairs + pair < P.pair_units; }
__device__ __forceinline__ Unit unit_of(const Params& P, int pair, uint32_t rank, int i) {
  const int pu = i * P.num_pairs + pair, t = 2 * (pu / P.n_groups) + (int)rank;
  const int tc = min(t, P.tiles_total - 1);
  Unit u;
  u.store = t < P.tiles_total;
  u.n = tc / P.tiles_per_img;
  u.tt = tc - u.n * P.tiles_per_img;
  u.ty = u.tt / P.tiles_x;
  u.tx = u.tt - u.ty * P.tiles_x;
  u.ch0 = (pu % P.n_groups) * P.n_group;
  return u;
}
// Chunk lc of a unit, the pc-th of its running partial sum, ends that partial sum.  The MMA issuer commits there, the
// watcher drains the next accumulator stage and the epilogue adds P.parts of them: all three must cut alike.
__device__ __forceinline__ bool ends_part(int pc, int lc, int chunks_per_part, int chunks) {
  return pc == chunks_per_part - 1 || lc == chunks - 1;
}
// Both CTAs allocate the pair's tensor memory while the TMA warp prefetches the tensor maps
__device__ __forceinline__ uint32_t conv_pair_setup(const Params& P, uint8_t* tmem_ptr, int warp, int lane) {
  return pair_setup(tmem_ptr, warp, kWarpAlloc, kTmemCols, [&] {
    if (warp == kWarpTma && lane == 0) {
      tma_prefetch_desc(&P.in_map);
      tma_prefetch_desc(&P.out_map);
      tma_prefetch_desc(&P.whi_map);
      tma_prefetch_desc(&P.wlo_map);
    }
  });
}

// TMA producer of the weights (lane 0): a B stage holds kTaps taps (one, or a tap row of three) of one 32-channel
// chunk, hi and lo planes of this CTA's half of the channel group.  Stage s at dst0 + s * stage_bytes is filled once
// free0 + 8 s released it and completes full0 + 8 s of the leader CTA, which expects the bytes of both CTAs.
template <int kTaps>
__device__ __forceinline__ void weight_producer(const Params& P, int pair, uint32_t rank, uint32_t dst0, uint32_t stage_bytes,
                                                uint32_t stages, uint32_t full0, uint32_t free0) {
#ifdef FOD_DBG
  long long* const dbg_buf = (pair == 0 && rank == 0) ? g_dbg : nullptr;
  constexpr int lane = 0;
#endif
  const uint32_t full_leader = map_to_cta(full0, 0);
  const uint32_t plane = (uint32_t)P.nhalf * 64u;
  uint32_t g = 0;
  for (int i = 0; has_unit(P, pair, i); ++i) {
    const int row0 = unit_of(P, pair, rank, i).ch0 + (int)rank * P.nhalf;
    for (int cc = 0; cc < P.cin_chunks; ++cc)
      for (int tap0 = 0; tap0 < P.taps; tap0 += kTaps, ++g) {
        const uint32_t s = ring_stage(g, stages);
        DBG_STAMP(0, g, 0);
        mbar_wait(free0 + 8u * s, ring_phase(g, stages) ^ 1);
        DBG_STAMP(0, g, 1);
        if (rank == 0) mbar_arrive_expect_tx(full0 + 8u * s, 4 * kTaps * plane);   // kTaps x hi / lo x 2 CTAs
#pragma unroll
        for (int k = 0; k < kTaps; ++k) {
          const int k0 = ((tap0 + k) * P.cin_chunks + cc) * kChunk;
          const uint32_t dst = dst0 + s * stage_bytes + k * 2 * plane;
          tma_load_2d_2sm(dst, &P.whi_map, full_leader + 8u * s, k0, row0);
          tma_load_2d_2sm(dst + plane, &P.wlo_map, full_leader + 8u * s, k0, row0);
        }
      }
  }
}

// Epilogue: one output pixel per lane; warp = (TMEM quadrant qd, slab phase sp) handles the 32-column slabs j = sp,
// sp + kEpiWarps / 4, ...  The partial sums are added in IEEE fp32 into the running tile at off_sum (ncol32 slabs),
// from which the last part leaves through TMA stores.
template <int kEpiWarps>
__device__ __forceinline__ void epilogue(const Params& P, uint8_t* smem, uint32_t off_sum, uint32_t off_bias, uint32_t acc_full0,
                                         uint32_t acc_empty0, uint32_t tmem_acc, int warp, int lane, int pair, uint32_t rank) {
  const uint32_t sbase = smem_u32(smem);
  const int qd = warp & 3, sp = (warp - kWarpEpi0) >> 2;
  constexpr int sstep = kEpiWarps / 4;
  const int m = qd * 32 + lane;
  const uint32_t acc_empty_leader = map_to_cta(acc_empty0, 0);
  const bool issuer = (warp == kWarpEpi0 && lane == 0);
  const uint32_t row_s = sbase + off_sum + (uint32_t)((m >> 3) * 1024 + (m & 7) * 128);
  const uint32_t bias_s = sbase + off_bias;
  const int ncol32 = P.ncol32, parts = P.parts;
  const float w_inv = __ldg(P.w_inv);
  float vmax = 0.f;                 // max |y| over the valid outputs this lane produced
  uint32_t gp = 0;
  for (int i = 0; has_unit(P, pair, i); ++i) {
    const Unit u = unit_of(P, pair, rank, i);
    const float x_bound = image_bound(P.x_amax, P.n_amax, P.x_amax_stride, u.n);
    float xs, xs_inv;
    pow2_scale(x_bound, xs, xs_inv);
    const float rescale = xs_inv * w_inv;   // undoes the two power-of-two operand scales (exact)
    float ysplit = 0.f;   // != 0: the final part leaves as fp16 hi / lo of y * ysplit
    if (P.y_bound) {
      const int bi = P.x_amax_stride ? u.n : 0;
      const float yb = fmaf(P.y_l1, P.x_actual ? __ldg(P.x_actual + bi) : x_bound, P.y_beta);
      float unused;
      pow2_scale(yb, ysplit, unused);
      if (issuer) P.y_bound[bi] = yb;   // every CTA that works on image n writes the same value
    }
    const int oy = u.ty * kTileH + (m >> 4), ox = u.tx * kTileW + (m & 15);
    const bool px_valid = u.store && oy < P.ho && ox < P.wo;
    const float* res_px = nullptr;   // this pixel's row of the residual map
    if (P.res && px_valid)
      res_px = P.res + (((size_t)u.n * P.res_h + (oy >> P.res_shift)) * P.res_w + (ox >> P.res_shift)) * P.cout;
    if (issuer) tma_store_wait_read<0>();  // the previous tile has left the staging slabs
    named_bar_sync(1, 32 * kEpiWarps);
    if (sp == 0) reinterpret_cast<float*>(smem + off_bias)[m] = (P.bias && u.ch0 + m < P.cout) ? __ldg(P.bias + u.ch0 + m) : 0.f;
    named_bar_sync(1, 32 * kEpiWarps);
#pragma unroll 1
    for (int part = 0; part < parts; ++part, ++gp) {
      const uint32_t as_ = ring_stage(gp, kAccStages);
      mbar_wait(acc_full0 + 8u * as_, ring_phase(gp, kAccStages));
      tc_fence_after();
      const uint32_t trow = tmem_acc + ((uint32_t)(qd * 32) << 16) + as_ * 128u;
      if (sp >= ncol32) acc_release(acc_empty_leader + 8u * as_, lane);   // a group narrower than the slab phases: nothing to read
      const bool final = part == parts - 1;
#pragma unroll 1
      for (int j = sp; j < ncol32; j += sstep) {
        uint32_t v[32];
        tmem_ld32(trow + j * 32, v);
        tmem_wait_ld();
        if (j + sstep >= ncol32) acc_release(acc_empty_leader + 8u * as_, lane);   // this warp's columns are read
        const uint32_t slab = row_s + (uint32_t)j * kSlabBytes;
        float4 xv[8];
#pragma unroll
        for (int c4 = 0; c4 < 8; ++c4) {
          const int cb = u.ch0 + j * 32 + c4 * 4;   // channel of x.x
          float4 x = make_float4(__uint_as_float(v[c4 * 4 + 0]), __uint_as_float(v[c4 * 4 + 1]), __uint_as_float(v[c4 * 4 + 2]),
                                 __uint_as_float(v[c4 * 4 + 3]));
          if (part > 0) {
            const float4 r = lds4s(slab + (uint32_t)((c4 ^ (m & 7)) << 4));
            x.x += r.x; x.y += r.y; x.z += r.z; x.w += r.w;
          }
          if (final) {
            const float4 bb = lds4s(bias_s + (j * 32 + c4 * 4) * 4);
            x.x = fmaf(x.x, rescale, bb.x); x.y = fmaf(x.y, rescale, bb.y);
            x.z = fmaf(x.z, rescale, bb.z); x.w = fmaf(x.w, rescale, bb.w);
            if (res_px && cb < P.cout) {
              const float4 rv = ldg4(res_px + cb);
              x.x += rv.x; x.y += rv.y; x.z += rv.z; x.w += rv.w;
            }
            if (P.relu) {
              x.x = fmaxf(x.x, 0.f); x.y = fmaxf(x.y, 0.f); x.z = fmaxf(x.z, 0.f); x.w = fmaxf(x.w, 0.f);
            }
            if (P.y_amax && px_valid) {   // columns beyond Cout hold whatever the accumulator columns held
              if (cb + 0 < P.cout) vmax = fmaxf(vmax, fabsf(x.x));
              if (cb + 1 < P.cout) vmax = fmaxf(vmax, fabsf(x.y));
              if (cb + 2 < P.cout) vmax = fmaxf(vmax, fabsf(x.z));
              if (cb + 3 < P.cout) vmax = fmaxf(vmax, fabsf(x.w));
            }
          }
          xv[c4] = x;
        }
        if (final && ysplit != 0.f) {
          // the consumer's operand format: all 32 channels of the row are formed first (the running sums sit where the
          // packed chunks go), then per 16 channels [16 x fp16 hi | 16 x the exact remainders]
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            uint32_t hi[4], lo[4];
            split_f16x2(xv[2 * c].x * ysplit, xv[2 * c].y * ysplit, hi[0], lo[0]);
            split_f16x2(xv[2 * c].z * ysplit, xv[2 * c].w * ysplit, hi[1], lo[1]);
            split_f16x2(xv[2 * c + 1].x * ysplit, xv[2 * c + 1].y * ysplit, hi[2], lo[2]);
            split_f16x2(xv[2 * c + 1].z * ysplit, xv[2 * c + 1].w * ysplit, hi[3], lo[3]);
            const int hp = (c >> 1) * 4 + (c & 1);      // per 16 channels [16 x hi | 16 x lo]: channels [8c, 8c + 8) -> chunk hp, hp + 2
            asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(slab + (uint32_t)((hp ^ (m & 7)) << 4)), "r"(hi[0]), "r"(hi[1]),
                         "r"(hi[2]), "r"(hi[3]) : "memory");
            asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(slab + (uint32_t)(((hp + 2) ^ (m & 7)) << 4)), "r"(lo[0]),
                         "r"(lo[1]), "r"(lo[2]), "r"(lo[3]) : "memory");
          }
        } else {
#pragma unroll
          for (int c4 = 0; c4 < 8; ++c4) sts4s(slab + (uint32_t)((c4 ^ (m & 7)) << 4), xv[c4]);
        }
      }
    }
    if (P.y_amax && P.y_amax_per_image) {   // this unit's image: one atomic per warp and unit
      const uint32_t wmax = __reduce_max_sync(0xffffffffu, __float_as_uint(vmax));
      if (lane == 0 && wmax) atomicMax(reinterpret_cast<unsigned int*>(P.y_amax + u.n), wmax);
      vmax = 0.f;
    }
    fence_proxy_async_smem();
    named_bar_sync(1, 32 * kEpiWarps);
    if (issuer && u.store) {
      for (int j = 0; j < ncol32 && u.ch0 + j * 32 < P.cout; ++j)
        tma_store_4d(&P.out_map, sbase + off_sum + j * kSlabBytes, u.ch0 + j * 32, u.tx * kTileW, u.ty * kTileH, u.n);
      tma_store_commit();
    }
    if (P.colsum && u.store && sp == 0 && qd < ncol32) {
      // Channel sums over the tile's pixels that lie inside the image, in a fixed order (deterministic, independent of
      // the batch).  Warp = 32-channel slab; lane = (row offset 0..3, 4-channel group): a warp reads four consecutive
      // 128-byte rows per step (conflict-free), 32 steps cover the tile; the four row offsets meet in two shuffles.
      const int vy = min(kTileH, P.ho - u.ty * kTileH), vx = min(kTileW, P.wo - u.tx * kTileW);
      const uint32_t c4 = (uint32_t)(lane & 7), ro = (uint32_t)(lane >> 3);
      const uint32_t sb = sbase + off_sum + (uint32_t)qd * kSlabBytes;
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f), acq = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
      for (uint32_t r0 = 0; r0 < 128; r0 += 4) {
        const uint32_t r = r0 + ro;
        if ((int)(r >> 4) < vy && (int)(r & 15) < vx) {
          const float4 v = lds4s(sb + (r >> 3) * 1024 + (r & 7) * 128 + ((c4 ^ (r & 7)) << 4));
          acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
          acq.x = fmaf(v.x, v.x, acq.x); acq.y = fmaf(v.y, v.y, acq.y);
          acq.z = fmaf(v.z, v.z, acq.z); acq.w = fmaf(v.w, v.w, acq.w);
        }
      }
#pragma unroll
      for (int sh = 8; sh <= 16; sh <<= 1) {
        acc.x += __shfl_xor_sync(0xffffffffu, acc.x, sh); acc.y += __shfl_xor_sync(0xffffffffu, acc.y, sh);
        acc.z += __shfl_xor_sync(0xffffffffu, acc.z, sh); acc.w += __shfl_xor_sync(0xffffffffu, acc.w, sh);
        acq.x += __shfl_xor_sync(0xffffffffu, acq.x, sh); acq.y += __shfl_xor_sync(0xffffffffu, acq.y, sh);
        acq.z += __shfl_xor_sync(0xffffffffu, acq.z, sh); acq.w += __shfl_xor_sync(0xffffffffu, acq.w, sh);
      }
      const int ch = u.ch0 + qd * 32 + (int)c4 * 4;
      if (ro == 0 && ch < P.cout) {
        const size_t o = ((size_t)u.n * P.tiles_per_img + u.tt) * P.cout + ch;
        *reinterpret_cast<float4*>(P.colsum + o) = acc;
        if (P.colsumsq) *reinterpret_cast<float4*>(P.colsumsq + o) = acq;
      }
    }
  }
  if (issuer) tma_store_wait<0>();
  if (P.y_amax && !P.y_amax_per_image) {   // non-negative floats order like their bit patterns; a NaN becomes a huge bound (scale 1 downstream)
    const uint32_t wmax = __reduce_max_sync(0xffffffffu, __float_as_uint(vmax));
    if (lane == 0 && wmax) atomicMax(reinterpret_cast<unsigned int*>(P.y_amax), wmax);
  }
}

// ---------------------------------------------------------------------------------------------- tensor-memory pipeline
// Barriers: q_full / q_empty: input ring, TMA -> converters -> TMA; ready: the converters of both CTAs + the weight
// bytes -> watcher (one barrier per stage); st_free: MMA commit -> A + B stage free; acc_full / acc_empty: MMA ->
// epilogue warps of both CTAs -> watcher.
__global__ void __launch_bounds__(kThreads, 1) conv_tc_kernel_tmem(const __grid_constant__ Params P, const __grid_constant__ TmemA T) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const uint32_t sbase = smem_u32(smem);
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  const uint32_t rank = blockIdx.x & 1;  // == %cluster_ctarank for cluster dims (2,1,1)
  const int pair = blockIdx.x >> 1;
#ifdef FOD_DBG
  long long* const dbg_buf = (pair == 0 && rank == 0) ? g_dbg : nullptr;
#endif
  const uint32_t bar0 = sbase + kOffBars, flag = sbase + kOffTmemPtr + 8;
  auto q_full = [&](int s) { return bar0 + 8u * s; };
  auto q_empty = [&](int s) { return bar0 + 8u * (kQStages + s); };
  auto ready = [&](int s) { return bar0 + 8u * (2 * kQStages + s); };
  auto st_free = [&](int s) { return bar0 + 8u * (2 * kQStages + kStages + s); };
  auto acc_full = [&](int s) { return bar0 + 8u * (2 * kQStages + 2 * kStages + s); };
  auto acc_empty = [&](int s) { return bar0 + 8u * (2 * kQStages + 2 * kStages + kAccStages + s); };
  if (tid == 0) {
    for (int s = 0; s < kQStages; ++s) {
      mbar_init(q_full(s), 1);
      mbar_init(q_empty(s), kConvWarps);
    }
    for (int s = 0; s < kStages; ++s) {
      mbar_init(ready(s), kConvWarps + 1);  // one set of 8 warps per CTA, both CTAs, + the weight producer's expect_tx
      mbar_init(st_free(s), 1);
    }
    for (int s = 0; s < kAccStages; ++s) {
      mbar_init(acc_full(s), 1);
      mbar_init(acc_empty(s), 2 * 4);  // epilogue warps x 2 CTAs
    }
    *reinterpret_cast<volatile uint32_t*>(smem + kOffTmemPtr + 8) = 0;
    fence_barrier_init();
  }
  const uint32_t tmem_base = conv_pair_setup(P, smem + kOffTmemPtr, warp, lane);

  if (warp == kWarpTma) {
    // ------------------------------------------------------------------ TMA producer: input tile + halo, per 32 channels
    if (lane == 0) {
      uint32_t g = 0;
      const int pad = T.ksize >> 1, loads = P.per_tap ? P.taps : 1;
      for (int i = 0; has_unit(P, pair, i); ++i) {
        const Unit u = unit_of(P, pair, rank, i);
        const int x0 = u.tx * kTileW * P.stride - pad, y0 = u.ty * kTileH * P.stride - pad;
        for (int cc = 0; cc < P.cin_chunks; ++cc)
          for (int tap = 0; tap < loads; ++tap, ++g) {
            const uint32_t s = ring_stage(g, kQStages);
            const int dy = tap / T.ksize, dx = tap - dy * T.ksize;   // (0, 0) when the halo tile serves every tap
            mbar_wait(q_empty(s), ring_phase(g, kQStages) ^ 1);
            mbar_arrive_expect_tx(q_full(s), T.q_stage_bytes);
            tma_load_4d(sbase + kOffQ + s * T.q_stage_stride, &P.in_map, q_full(s), cc * kChunk, x0 + dx, y0 + dy, u.n);
          }
      }
    }
  } else if (warp == kWarpTmaB) {
    if (lane == 0) weight_producer<1>(P, pair, rank, sbase + kOffB, kBStageBytes, kStages, ready(0), st_free(0));
  } else if (warp == kWarpMma) {
    // ------------------------------------------------------------------ MMA issuer (leader CTA)
    // The whole warp runs the loop converged and one elected lane issues: every operand of tcgen05.mma is then a
    // warp-uniform value that ptxas keeps in uniform registers.  (Inside an `if (lane == 0)` region the same code
    // compiles to a broadcast-and-retry loop around each MMA whose latency exceeds the 64 cycles of the MMA itself.)
    if (rank == 0) {
      const uint32_t idesc = idesc_f16(256, P.n_group);
      const uint32_t plane16 = ((uint32_t)P.nhalf * 64u) >> 4;
      const int cpp = P.chunks_per_part, chunks = P.chunks;
      // Everything a chunk's MMAs need is carried in (uniform) registers and advanced AFTER the chunk has been issued,
      // so nothing but the flag test sits between the last MMA of one chunk and the first MMA of the next: the
      // tensor pipe's queue is only an MMA or two deep and a 64-channel layer's MMA lasts 32 cycles.
      const uint64_t bhi0 = smem_desc_k_sw64(sbase + kOffB);
      const uint32_t a00 = tmem_base + kColA, d0 = tmem_base + kColAcc;
      uint64_t bhi = bhi0;
      uint32_t a0 = a00, d = d0, sf = st_free(0), af = acc_full(0);
      uint32_t upto = 0, g = 0, s = 0;
      int pc = 0, as_ = 0;
      for (int i = 0; has_unit(P, pair, i); ++i) {
        for (int lc = 0; lc < chunks; ++lc, ++g) {
          DBG_STAMP(1, g, 0);
          flag_wait(flag, upto, g);
          tc_fence_after();
          DBG_STAMP(1, g, 1);
          const bool last = ends_part(pc, lc, cpp, chunks);
          if (elect_one()) {
            const uint64_t blo = bhi + plane16;
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {  // K = 16 fp16 per MMA: 8 packed columns of A, 32 bytes of a B row
              const uint32_t ah = a0 + ks * 8, al = ah + 16;
              const uint64_t boff = (uint64_t)((ks * 32) >> 4);
              mma_f16_ts<2>(d, ah, bhi + boff, idesc, (pc | ks) ? 1u : 0u);
              mma_f16_ts<2>(d, al, bhi + boff, idesc, 1u);
              mma_f16_ts<2>(d, ah, blo + boff, idesc, 1u);
            }
            mma_commit_pair(sf, 3);
            if (last) mma_commit_pair(af, 3);
          }
          __syncwarp();
          DBG_STAMP(1, g, 2);
          s = ring_next(s, kStages);
          a0 = a00 + s * kAStageCols;
          bhi = bhi0 + s * (kBStageBytes >> 4);
          sf = st_free(s);
          pc = last ? 0 : pc + 1;
          if (last) {
            as_ ^= 1;
            d = d0 + (uint32_t)as_ * 128u;
            af = acc_full(as_);
          }
        }
      }
    }
  } else if (warp == kWarpAlloc) {
    // ------------------------------------------------------------------ barrier watcher of the MMA warp (leader)
    if (rank == 0 && lane == 0) {
      uint32_t g = 0, gp = 0;
      for (int i = 0; has_unit(P, pair, i); ++i) {
        int pc = 0;
        for (int lc = 0; lc < P.chunks; ++lc, ++g) {
          DBG_STAMP(2, g, 0);
          if (pc == 0) mbar_wait(acc_empty(ring_stage(gp, kAccStages)), ring_phase(gp, kAccStages) ^ 1);
          DBG_STAMP(2, g, 1);
          mbar_wait(ready(ring_stage(g, kStages)), ring_phase(g, kStages));
          DBG_STAMP(2, g, 3);
          flag_publish(flag, g + 1);
          const bool last = ends_part(pc, lc, P.chunks_per_part, P.chunks);
          pc = last ? 0 : pc + 1;
          gp += last;
        }
      }
    }
  } else if (warp < kWarpConv0) {
    epilogue<4>(P, smem, kOffSum, kOffBias, acc_full(0), acc_empty(0), tmem_base + kColAcc, warp, lane, pair, rank);
  } else {
    // ------------------------------------------------------------------ converters
    // Phase A, once per staged tile (i.e. once per 32 input channels, not once per tap): all 16 warps convert the tile
    // IN PLACE from fp32 to scaled fp16 hi / lo: a 128-byte pixel row of 32 floats becomes [32 x hi | 32 x lo], the
    // 16-byte chunks keep the position swizzle of the TMA (chunk c of row r at c ^ (r & 7)).  A row is shared by two
    // adjacent lanes (16 channels each) that read it completely before either writes.
    // Phase B, per tap: one set of 8 warps (the sets alternate over the chunks) moves the tap-shifted row of each
    // output pixel (one pixel per lane = TMEM lane; conflict-free LDS.128) into TENSOR MEMORY: no arithmetic.
    const int cw = warp - kWarpConv0;
    const int qd = cw & 3, half = (cw >> 2) & 1, set = cw >> 3;
    const int m = qd * 32 + lane;
    const int py = m >> 4, px = m & 15;  // position of this pixel's tap (0,0) in the halo tile
    const bool per_tap = P.per_tap != 0;
    // a tile that serves a single tap (1x1 kernels, stride 2) is converted on the way to tensor memory instead: no
    // shared-memory round trip and no barrier between the two warp sets
    const bool direct = per_tap || P.taps == 1;
    const uint32_t ready_leader = map_to_cta(ready(0), 0);
    const uint32_t trow = tmem_base + ((uint32_t)(qd * 32) << 16) + kColA + half * 8;
    const int ksz = T.ksize, hw = T.halo_w;
    const int stage_rows = (int)(T.q_stage_bytes >> 7);
    const int crow = (cw * 32 + lane) >> 1, chalf = lane & 1;   // phase A: (row, 16-channel half) of this lane
    float xs, xs_inv;   // input scale 2^e of this unit's image
    uint32_t g = 0, gq = 0;

    const float* gate_row = nullptr;    // a_gate row of this unit's image, at this chunk's first channel
    const float* shift_row = nullptr;   // a_shift likewise
    bool row_in = true;                 // the row being transformed lies inside the image (set by the caller)
    auto gated = [&](float4 v, int c4) {   // c4: index of the 4-channel group inside the 32-channel chunk
      if (gate_row) {
        const float4 gv = ldg4(gate_row + c4 * 4);
        v.x *= gv.x; v.y *= gv.y; v.z *= gv.z; v.w *= gv.w;
      }
      if (shift_row) {   // affine normalisation (+ ReLU) of the producer's map; the padding ring stays zero
        const float4 sv = ldg4(shift_row + c4 * 4);
        v.x += sv.x; v.y += sv.y; v.z += sv.z; v.w += sv.w;
        if (T.a_relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
        if (!row_in) v = make_float4(0.f, 0.f, 0.f, 0.f);
      }
      return v;
    };
    int in_y0 = 0, in_x0 = 0;   // image coordinates of row 0 of the staged tile (tile origin - padding)
    auto convert_stage = [&](uint32_t qt) {
      const uint32_t at = qt + (uint32_t)crow * 128u;
      const uint32_t key = (uint32_t)(crow & 7);
      {
        const int ry = crow / hw, rx = crow - ry * hw;
        row_in = in_y0 + ry >= 0 && in_y0 + ry < T.in_h && in_x0 + rx >= 0 && in_x0 + rx < T.in_w;
      }
      float4 x[4];
      if (crow < stage_rows) {
#pragma unroll
        for (int j = 0; j < 4; ++j) x[j] = gated(lds4s(at + ((((uint32_t)(chalf * 4 + j)) ^ key) << 4)), chalf * 4 + j);
      }
      __syncwarp();   // both lanes of a row have read it
      if (crow < stage_rows) {
        uint32_t hi[8], lo[8];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          split_f16x2(x[j].x * xs, x[j].y * xs, hi[2 * j + 0], lo[2 * j + 0]);
          split_f16x2(x[j].z * xs, x[j].w * xs, hi[2 * j + 1], lo[2 * j + 1]);
        }
        // logical chunks: hi of channels [8c, 8c+8) at c, lo at 4 + c; this lane owns c = 2*chalf, 2*chalf + 1.  The two
        // lanes of a row write in opposite orders (hi first / lo first) so that a quarter warp never hits a bank twice.
        const uint32_t c0 = (uint32_t)(2 * chalf);
        const uint4 h0 = make_uint4(hi[0], hi[1], hi[2], hi[3]), h1 = make_uint4(hi[4], hi[5], hi[6], hi[7]);
        const uint4 l0 = make_uint4(lo[0], lo[1], lo[2], lo[3]), l1 = make_uint4(lo[4], lo[5], lo[6], lo[7]);
        auto put = [&](uint32_t c, const uint4& v) {
          asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(at + ((c ^ key) << 4)), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
                       : "memory");
        };
        if (chalf == 0) {
          put(c0, h0); put(c0 + 1, h1); put(4 + c0, l0); put(5 + c0, l1);
        } else {
          put(4 + c0, l0); put(5 + c0, l1); put(c0, h0); put(c0 + 1, h1);
        }
      }
      named_bar_sync(2, kConvWarps * 32);   // the whole tile is converted before any warp copies a tap out of it
    };

    for (int i = 0; has_unit(P, pair, i); ++i) {
      const Unit u = unit_of(P, pair, rank, i);
      pow2_scale(image_bound(P.x_amax, P.n_amax, P.x_amax_stride, u.n), xs, xs_inv);
      in_y0 = u.ty * kTileH * P.stride - (ksz >> 1);
      in_x0 = u.tx * kTileW * P.stride - (ksz >> 1);
      for (int cc = 0; cc < P.cin_chunks; ++cc) {
        if (T.a_gate) gate_row = T.a_gate + (size_t)u.n * T.cin + cc * kChunk;
        if (T.a_shift) shift_row = T.a_shift + (size_t)u.n * T.cin + cc * kChunk;
        // single-tap path over a concat buffer whose later slices were written pre-split by their producers, each at the
        // scale of its own bound: the stored halves are brought to this launch's common scale by an exact power of two
        const int ch16 = cc * kChunk + half * 16;          // first channel of the 16-channel group this warp moves
        const bool pre = direct && ch16 >= T.x_presplit_from;
        __half2 pre_mult = __float2half2_rn(1.f);
        if (pre) {
          int k = P.n_amax - 1;
          while (k > 0 && ch16 < T.slice_ch[k]) --k;
          const int step = P.x_amax_stride ? P.x_amax_stride : 1;
          float sk, sk_inv;
          pow2_scale(__ldg(P.x_amax + (size_t)k * step + (P.x_amax_stride ? u.n : 0)), sk, sk_inv);
          pre_mult = __float2half2_rn(xs * sk_inv);
        }
        uint32_t qs = ring_stage(gq, kQStages);
        uint32_t qt = sbase + kOffQ + qs * T.q_stage_stride;
        if (!per_tap) {
          mbar_wait(q_full(qs), ring_phase(gq, kQStages));
          if (!direct && !T.x_presplit) convert_stage(qt);
        }
        int dy = 0, dx = 0;
        for (int tap = 0; tap < P.taps; ++tap, ++g) {
          if (per_tap) {  // this tap's own 8 x 16 tile
            qs = ring_stage(gq, kQStages);
            qt = sbase + kOffQ + qs * T.q_stage_stride;
            mbar_wait(q_full(qs), ring_phase(gq, kQStages));
          }
          if ((int)(g & 1) == set) {
            if (cw == 0 || cw == 8) DBG_STAMP(3, g, 0);
            const int r = per_tap ? m : (py + dy) * hw + px + dx;
            const uint32_t at = qt + (uint32_t)r * 128u;
            const uint32_t key = (uint32_t)(r & 7);
            uint32_t hi[8], lo[8];
            if (direct && !pre) {
              {   // image position of this pixel's input for this tap (a per-tap tile holds every stride-th pixel)
                const int iy = in_y0 + (per_tap ? py * P.stride + dy : py), ix = in_x0 + (per_tap ? px * P.stride + dx : px);
                row_in = iy >= 0 && iy < T.in_h && ix >= 0 && ix < T.in_w;
              }
              float4 x[4];
#pragma unroll
              for (int j = 0; j < 4; ++j) x[j] = gated(lds4s(at + ((((uint32_t)(half * 4 + j)) ^ key) << 4)), half * 4 + j);
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                split_f16x2(x[j].x * xs, x[j].y * xs, hi[2 * j + 0], lo[2 * j + 0]);
                split_f16x2(x[j].z * xs, x[j].w * xs, hi[2 * j + 1], lo[2 * j + 1]);
              }
            } else {
              // the converted tile holds [32 x hi | 32 x lo] per row, a pre-split one (written by its producer) per 16 channels
              // [16 x hi | 16 x lo] = chunks 4h, 4h+1 | 4h+2, 4h+3: 16-aligned slices of a concat buffer stay whole groups
              const bool split_in = pre || T.x_presplit;
              const uint32_t hi0 = split_in ? (uint32_t)(4 * half) : (uint32_t)(2 * half);
              const uint32_t lo0 = split_in ? (uint32_t)(4 * half + 2) : (uint32_t)(4 + 2 * half);
#pragma unroll
              for (int j = 0; j < 2; ++j) {
                asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];"
                             : "=r"(hi[4 * j]), "=r"(hi[4 * j + 1]), "=r"(hi[4 * j + 2]), "=r"(hi[4 * j + 3])
                             : "r"(at + (((hi0 + j) ^ key) << 4)));
                asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];"
                             : "=r"(lo[4 * j]), "=r"(lo[4 * j + 1]), "=r"(lo[4 * j + 2]), "=r"(lo[4 * j + 3])
                             : "r"(at + (((lo0 + j) ^ key) << 4)));
              }
              if (pre) {   // to this launch's scale
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  const __half2 h = __hmul2(*reinterpret_cast<const __half2*>(&hi[j]), pre_mult);
                  const __half2 l = __hmul2(*reinterpret_cast<const __half2*>(&lo[j]), pre_mult);
                  hi[j] = *reinterpret_cast<const uint32_t*>(&h);
                  lo[j] = *reinterpret_cast<const uint32_t*>(&l);
                }
              }
            }
            const uint32_t s = ring_stage(g, kStages);
            if (cw == 0 || cw == 8) DBG_STAMP(3, g, 1);
            mbar_wait(st_free(s), ring_phase(g, kStages) ^ 1);  // the MMAs that read this TMEM stage have completed
            tc_fence_after();
            if (cw == 0 || cw == 8) DBG_STAMP(3, g, 2);
            tmem_st8(trow + s * kAStageCols, hi);
            tmem_st8(trow + s * kAStageCols + 16, lo);
            tmem_wait_st();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_remote(ready_leader + 8u * s);
            if (cw == 0 || cw == 8) DBG_STAMP(3, g, 3);
          }
          if (++dx == ksz) { dx = 0; ++dy; }
          if (per_tap) {
            __syncwarp();
            if (lane == 0) mbar_arrive(q_empty(qs));
            ++gq;
          }
        }
        if (!per_tap) {
          __syncwarp();
          if (lane == 0) mbar_arrive(q_empty(qs));
          ++gq;
        }
      }
    }
  }
  pair_teardown(warp, kWarpAlloc, tmem_base, kTmemCols);
}

// ---------------------------------------------------------------------------------------------- shared-memory A pipeline
// For 3x3 layers whose input arrives pre-split at one scale: the stored fp16 halves are what the MMA multiplies, so the
// tensor core reads them straight from the TMA-staged tile instead of from tensor memory, and there are no converter
// warps.  A K-major SW128 descriptor has one stride between 8-row groups, so the 18-pixel-wide halo cannot serve as the
// operand; per 32-channel chunk three dx-shifted boxes of 16 x 10 pixels are staged instead, and the operand of tap
// (dy, dx) is box dx from pixel row dy on (start + dy * 2048 bytes, 1024-aligned).  Stride 2: the three taps of a tap
// row are three 8 x 16 boxes with element strides 2, one A stage per tap row.  In a 128-byte row the split format is
// [16 hi | 16 lo | 16 hi | 16 lo]: step ks of the K = 16 MMAs reads hi at +64 ks bytes and lo at +64 ks + 32, the K
// advance inside a swizzle atom.  MMAs, their order and the part boundaries are those of the tensor-memory pipeline, so
// the result is bit-identical to it.  The unit of synchronisation is the tap row (cc, dy): one weight stage, and a new
// A stage at dy == 0 (stride 1) or at every tap row (stride 2).  Barriers: a_full / b_full: TMA bytes of both CTAs ->
// watcher; a_empty / b_free: MMA commit -> TMA; acc_full / acc_empty as in the tensor-memory pipeline.
constexpr int kAStagesS = 2;
constexpr int kEpiWarpsS = 8;
constexpr int kThreadsS = (kWarpEpi0 + kEpiWarpsS) * 32;   // TMA A, MMA, watcher, TMA B, epilogue
constexpr uint32_t kRowBytesS1 = 16 * 128;   // one pixel row of a stride-1 box
constexpr uint32_t kMaxDynSmem = 232448;     // opt-in dynamic shared memory per block (sm_100)
constexpr uint32_t kNumBarsS = 2 * kAStagesS + 2 * kStages + 2 * kAccStages;
// shared memory from off_sum on: output staging, bias, barriers, TMEM address and watcher flag
__host__ __device__ constexpr uint32_t smem_a_tail_bytes(int ncol32) { return ncol32 * kSlabBytes + 128 * 4 + kNumBarsS * 8 + 16; }

__global__ void __launch_bounds__(kThreadsS, 1) conv_tc_kernel_smem(const __grid_constant__ Params P, const __grid_constant__ SmemA L) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const uint32_t sbase = smem_u32(smem);
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  const uint32_t rank = blockIdx.x & 1;  // == %cluster_ctarank for cluster dims (2,1,1)
  const int pair = blockIdx.x >> 1;
  const uint32_t off_bias = L.off_sum + (uint32_t)P.ncol32 * kSlabBytes, off_bars = off_bias + 128 * 4;
  const uint32_t off_tmem_ptr = off_bars + kNumBarsS * 8;
  const uint32_t bar0 = sbase + off_bars, flag = sbase + off_tmem_ptr + 8;
  auto a_full = [&](int s) { return bar0 + 8u * s; };
  auto a_empty = [&](int s) { return bar0 + 8u * (kAStagesS + s); };
  auto b_full = [&](int s) { return bar0 + 8u * (2 * kAStagesS + s); };
  auto b_free = [&](int s) { return bar0 + 8u * (2 * kAStagesS + kStages + s); };
  auto acc_full = [&](int s) { return bar0 + 8u * (2 * kAStagesS + 2 * kStages + s); };
  auto acc_empty = [&](int s) { return bar0 + 8u * (2 * kAStagesS + 2 * kStages + kAccStages + s); };
  if (tid == 0) {
    for (int s = 0; s < kAStagesS; ++s) {
      mbar_init(a_full(s), 1);
      mbar_init(a_empty(s), 1);
    }
    for (int s = 0; s < L.b_stages; ++s) {
      mbar_init(b_full(s), 1);
      mbar_init(b_free(s), 1);
    }
    for (int s = 0; s < kAccStages; ++s) {
      mbar_init(acc_full(s), 1);
      mbar_init(acc_empty(s), 2 * kEpiWarpsS);  // epilogue warps x 2 CTAs
    }
    *reinterpret_cast<volatile uint32_t*>(smem + off_tmem_ptr + 8) = 0;
    fence_barrier_init();
  }
  const uint32_t tmem_base = conv_pair_setup(P, smem + off_tmem_ptr, warp, lane);

  const bool per_row_a = P.per_tap != 0;
  const uint32_t a_stage_bytes = 3 * L.a_box_bytes;
  if (warp == kWarpTma) {
    // ------------------------------------------------------------------ TMA producer: A stages (three boxes each)
    if (lane == 0) {
      const uint32_t a_full_leader = map_to_cta(a_full(0), 0);
      uint32_t ga = 0;
      for (int i = 0; has_unit(P, pair, i); ++i) {
        const Unit u = unit_of(P, pair, rank, i);
        const int x0 = u.tx * kTileW * P.stride - 1, y0 = u.ty * kTileH * P.stride - 1;
        for (int cc = 0; cc < P.cin_chunks; ++cc)
          for (int dy = 0; dy < 3; dy += per_row_a ? 1 : 3, ++ga) {
            const uint32_t s = ring_stage(ga, kAStagesS);
            mbar_wait(a_empty(s), ring_phase(ga, kAStagesS) ^ 1);
            if (rank == 0) mbar_arrive_expect_tx(a_full(s), 2 * a_stage_bytes);
            for (int dx = 0; dx < 3; ++dx)
              tma_load_4d_2sm(sbase + s * a_stage_bytes + dx * L.a_box_bytes, &P.in_map, a_full_leader + 8u * s,
                              cc * kChunk, x0 + dx, y0 + dy, u.n);
          }
      }
    }
  } else if (warp == kWarpTmaB) {
    if (lane == 0) weight_producer<3>(P, pair, rank, sbase + L.off_b, L.b_stage_bytes, L.b_stages, b_full(0), b_free(0));
  } else if (warp == kWarpMma) {
    // ------------------------------------------------------------------ MMA issuer (leader CTA), A from shared memory
    if (rank == 0) {
      const uint32_t idesc = idesc_f16(256, P.n_group);
      const uint32_t plane16 = ((uint32_t)P.nhalf * 64u) >> 4, tap16 = 2 * plane16, bstep16 = L.b_stage_bytes >> 4;
      const uint32_t box16 = L.a_box_bytes >> 4, astep16 = a_stage_bytes >> 4, row16 = per_row_a ? 0u : kRowBytesS1 >> 4;
      const int cpp = P.chunks_per_part, chunks = P.chunks;
      const uint64_t a_desc0 = smem_desc_k_sw128(sbase), b_desc0 = smem_desc_k_sw64(sbase + L.off_b);
      const uint32_t d0 = tmem_base + kColAcc;
      uint64_t a_desc = a_desc0, b_desc = b_desc0;
      uint32_t d = d0, af = acc_full(0), sf = b_free(0), qf = a_empty(0);
      uint32_t upto = 0, g = 0, sb = 0, sa = 0;
      int pc = 0, as_ = 0;
      for (int i = 0; has_unit(P, pair, i); ++i) {
        int lc = 0;
        for (int cc = 0; cc < P.cin_chunks; ++cc)
          for (int dy = 0; dy < 3; ++dy, ++g) {
            flag_wait(flag, upto, g);
            tc_fence_after();
            const uint64_t a_row = a_desc + (uint64_t)(dy * row16);
#pragma unroll 1
            for (int dx = 0; dx < 3; ++dx, ++lc) {
              const bool last = ends_part(pc, lc, cpp, chunks);
              if (elect_one()) {
                const uint64_t a = a_row + dx * box16, bhi = b_desc + dx * tap16, blo = bhi + plane16;
#pragma unroll
                for (int ks = 0; ks < 2; ++ks) {   // A: [16 hi | 16 lo] per 64 bytes of the row; B: 32 bytes per step
                  const uint64_t ah = a + (uint64_t)(ks * 4), al = ah + 2u, boff = (uint64_t)(ks * 2);
                  mma_f16_ss<2>(d, ah, bhi + boff, idesc, (pc | ks) ? 1u : 0u);
                  mma_f16_ss<2>(d, al, bhi + boff, idesc, 1u);
                  mma_f16_ss<2>(d, ah, blo + boff, idesc, 1u);
                }
                if (last) mma_commit_pair(af, 3);
              }
              __syncwarp();
              pc = last ? 0 : pc + 1;
              if (last) {
                as_ ^= 1;
                d = d0 + (uint32_t)as_ * 128u;
                af = acc_full(as_);
              }
            }
            const bool a_done = per_row_a || dy == 2;
            if (elect_one()) {
              mma_commit_pair(sf, 3);
              if (a_done) mma_commit_pair(qf, 3);
            }
            __syncwarp();
            sb = ring_next(sb, L.b_stages);
            b_desc = b_desc0 + sb * bstep16;
            sf = b_free(sb);
            if (a_done) {
              sa = ring_next(sa, kAStagesS);
              a_desc = a_desc0 + sa * astep16;
              qf = a_empty(sa);
            }
          }
      }
    }
  } else if (warp == kWarpAlloc) {
    // ------------------------------------------------------------------ barrier watcher of the MMA warp, per tap row
    if (rank == 0 && lane == 0) {
      uint32_t g = 0, ga = 0, gp = 0;
      for (int i = 0; has_unit(P, pair, i); ++i) {
        int pc = 0, lc = 0;
        for (int cc = 0; cc < P.cin_chunks; ++cc)
          for (int dy = 0; dy < 3; ++dy, ++g) {
            for (int dx = 0; dx < 3; ++dx, ++lc) {   // a part that starts in this row needs its accumulator drained
              if (pc == 0) mbar_wait(acc_empty(ring_stage(gp, kAccStages)), ring_phase(gp, kAccStages) ^ 1);
              const bool last = ends_part(pc, lc, P.chunks_per_part, P.chunks);
              pc = last ? 0 : pc + 1;
              gp += last;
            }
            if (per_row_a || dy == 0) {
              mbar_wait(a_full(ring_stage(ga, kAStagesS)), ring_phase(ga, kAStagesS));
              ++ga;
            }
            mbar_wait(b_full(ring_stage(g, L.b_stages)), ring_phase(g, L.b_stages));
            flag_publish(flag, g + 1);
          }
      }
    }
  } else {
    epilogue<kEpiWarpsS>(P, smem, L.off_sum, off_bias, acc_full(0), acc_empty(0), tmem_base + kColAcc, warp, lane, pair, rank);
  }
  pair_teardown(warp, kWarpAlloc, tmem_base, kTmemCols);
}

// max |x| of a dense fp32 array into *out (non-negative floats order like their bit patterns); *out must start at 0.
// blockIdx.y selects one of several arrays of n floats laid end to end, and out[blockIdx.y] receives its maximum.
__global__ void absmax_kernel(const float* __restrict__ x, size_t n, float* __restrict__ out) {
  x += (size_t)blockIdx.y * n;
  out += blockIdx.y;
  float m = 0.f;
  const size_t n4 = n >> 2;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    const float4 v = ldg4(x + i * 4);
    m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
  }
  if (blockIdx.x == 0)
    for (size_t i = n4 * 4 + threadIdx.x; i < n; i += blockDim.x) m = fmaxf(m, fabsf(x[i]));
  const uint32_t w = __reduce_max_sync(0xffffffffu, __float_as_uint(m));
  if ((threadIdx.x & 31) == 0 && w) atomicMax(reinterpret_cast<unsigned int*>(out), w);
}

// eSE gate from the per-tile channel sums of a convolution (vovnet.py eSEModule: x * hsigmoid(fc(avg_pool(x)))):
// gate[n][o] = relu6(b[o] + sum_i W[o][i] * mean[n][i] + 3) / 6, mean = sum over tiles / hw.
// Grid (image, group of kEseOuts outputs): every CTA rebuilds the image's mean vector (a few KB out of L2) and then
// computes its own outputs, one warp per output - 64 x c/32 CTAs instead of 64, so the fc weights (1 MB at c = 512) are
// read by 16 CTAs per image in parallel instead of by one.  The summation orders are fixed (tiles w, w+8, ... per warp,
// then the 8 partials; lanes i, i+32, ... then the shuffle tree): results do not depend on the grid.
constexpr int kEseOuts = 32;
__global__ void __launch_bounds__(256) ese_gate_kernel(const float* __restrict__ colsum, int tiles, int c, float inv_hw,
                                                       const float* __restrict__ w, const float* __restrict__ b,
                                                       float* __restrict__ gate) {
  extern __shared__ __align__(16) float mean[];   // [c] means, then [8][c] partial sums
  float* part = mean + c;
  const float* cs = colsum + (size_t)blockIdx.x * tiles * c;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  const int c4 = c >> 2;
  for (int i = lane; i < c4; i += 32) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
    for (int t = warp; t < tiles; t += nw) {
      const float4 v = ldg4(cs + (size_t)t * c + i * 4);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    *reinterpret_cast<float4*>(part + warp * c + i * 4) = acc;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < c; i += blockDim.x) {
    float acc = 0.f;
    for (int w8 = 0; w8 < nw; ++w8) acc += part[w8 * c + i];
    mean[i] = acc * inv_hw;
  }
  __syncthreads();
  const int o1 = min(c, ((int)blockIdx.y + 1) * kEseOuts);
  for (int o = (int)blockIdx.y * kEseOuts + warp; o < o1; o += nw) {
    float acc = 0.f;
    for (int i = lane; i < c; i += 32) acc = fmaf(__ldg(w + (size_t)o * c + i), mean[i], acc);
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
    if (lane == 0) gate[(size_t)blockIdx.x * c + o] = fminf(fmaxf(acc + b[o] + 3.f, 0.f), 6.f) / 6.f;
  }
}

// OIHW fp32 weights -> scaled fp16 hi / lo planes [Cout][ky][kx][Cin_pad] (Cin_pad = Cin rounded up to 32, zero filled);
// tail[0] = 1 / scale, tail[1] = scale, tail[2] = max |w| (written by absmax_kernel before this kernel runs)
__global__ void pack_weights_kernel(const float* __restrict__ w, int cout, int cin, int ksize, int cin_pad,
                                    __half* __restrict__ hi, __half* __restrict__ lo, float* __restrict__ tail) {
  const int taps = ksize * ksize;
  const size_t total = (size_t)cout * taps * cin_pad;
  float scale, inv;
  pow2_scale(tail[2], scale, inv);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int ci = (int)(i % cin_pad);
    const size_t r = i / cin_pad;
    const int tap = (int)(r % taps), co = (int)(r / taps);
    float x = 0.f;
    if (ci < cin) x = w[((size_t)co * cin + ci) * taps + tap] * scale;
    const __half h = __float2half_rn(x);
    hi[i] = h;
    lo[i] = __float2half_rn(x - __half2float(h));
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    tail[0] = inv;
    tail[1] = scale;
  }
}

}  // namespace cvt
}  // namespace fod

using namespace fod;

#ifdef FOD_DBG
extern "C" int fod_conv2d_debug(long long* buf) {
  cudaMemcpyToSymbol(cvt::g_dbg, &buf, sizeof(buf));
  return 0;
}
#endif

extern "C" size_t fod_conv2d_packed_floats(int cout, int cin, int ksize) {
  const size_t cin_pad = (size_t)(cin + 31) / 32 * 32;
  return (size_t)cout * ksize * ksize * cin_pad + 4;   // two fp16 planes + {1/scale, scale, max|w|, 0}
}

extern "C" int fod_conv2d_tiles_per_image(int ho, int wo) {
  return ((wo + cvt::kTileW - 1) / cvt::kTileW) * ((ho + cvt::kTileH - 1) / cvt::kTileH);
}

extern "C" int fod_ese_gate(const float* colsum, int n, int tiles_per_img, int channels, long hw, const float* fc_weight,
                            const float* fc_bias, float* gate, fod_stream_t stream) {
  FOD_REQUIRE(colsum && fc_weight && fc_bias && gate, "fod_ese_gate: null pointer");
  FOD_REQUIRE(n >= 0 && tiles_per_img > 0 && channels > 0 && channels <= 1024 && hw > 0, "fod_ese_gate: bad sizes");
  if (n == 0) return FOD_OK;
  FOD_REQUIRE(channels % 4 == 0 && ((uintptr_t)colsum & 15) == 0, "fod_ese_gate: channels must be a multiple of 4, colsum 16-byte aligned");
  const dim3 grid((unsigned)n, (unsigned)((channels + cvt::kEseOuts - 1) / cvt::kEseOuts));
  cvt::ese_gate_kernel<<<grid, 256, 9 * channels * sizeof(float), as_stream(stream)>>>(colsum, tiles_per_img, channels,
                                                                                 1.f / (float)hw, fc_weight, fc_bias, gate);
  FOD_CUDA_LAUNCH_CHECK("fod_ese_gate");
  return FOD_OK;
}

extern "C" int fod_absmax(const float* x, size_t n, float* out, fod_stream_t stream) {
  return fod_absmax_rows(x, 1, n, out, stream);
}

extern "C" int fod_absmax_rows(const float* x, int rows, size_t row_len, float* out, fod_stream_t stream) {
  FOD_REQUIRE(x && out, "fod_absmax: null pointer");
  FOD_REQUIRE(((uintptr_t)x & 15) == 0, "fod_absmax: input must be 16-byte aligned");
  FOD_REQUIRE(rows >= 1 && rows <= 65535 && (rows == 1 || row_len % 4 == 0), "fod_absmax_rows: 1..65535 rows of a multiple of 4 floats");
  FOD_CUDA_CALL(cudaMemsetAsync(out, 0, sizeof(float) * rows, as_stream(stream)));
  if (row_len == 0) return FOD_OK;
  const size_t per_row = (148 * 8 + rows - 1) / rows;                  // about 148 * 8 CTAs in all
  const size_t blocks = (row_len / 4 + 255) / 256;
  const dim3 grid((unsigned)(blocks < per_row ? (blocks ? blocks : 1) : per_row), (unsigned)rows);
  cvt::absmax_kernel<<<grid, 256, 0, as_stream(stream)>>>(x, row_len, out);
  FOD_CUDA_LAUNCH_CHECK("fod_absmax");
  return FOD_OK;
}

extern "C" int fod_conv2d_pack_weights(const float* w_oihw, int cout, int cin, int ksize, float* packed, fod_stream_t stream) {
  FOD_REQUIRE(w_oihw && packed, "fod_conv2d_pack_weights: null pointer");
  FOD_REQUIRE(cout > 0 && cin > 0 && (ksize == 1 || ksize == 3), "fod_conv2d_pack_weights: bad sizes");
  FOD_REQUIRE((((uintptr_t)w_oihw | (uintptr_t)packed) & 15) == 0, "fod_conv2d_pack_weights: pointers must be 16-byte aligned");
  const int cin_pad = (cin + 31) / 32 * 32;
  const size_t plane = (size_t)cout * ksize * ksize * cin_pad;
  __half* hi = reinterpret_cast<__half*>(packed);
  float* tail = packed + plane;
  int rc = fod_absmax(w_oihw, (size_t)cout * cin * ksize * ksize, tail + 2, stream);
  if (rc != FOD_OK) return rc;
  const unsigned blocks = (unsigned)((plane + 255) / 256 < 4096 ? (plane + 255) / 256 : 4096);
  cvt::pack_weights_kernel<<<blocks, 256, 0, as_stream(stream)>>>(w_oihw, cout, cin, ksize, cin_pad, hi, hi + plane, tail);
  FOD_CUDA_LAUNCH_CHECK("fod_conv2d_pack_weights");
  return FOD_OK;
}

// The shared-memory A pipeline serves 3x3 layers whose input is pre-split at one scale (stride 1, or stride 2 with a single
// bound, where the stored halves are brought to the common scale by exactly 1), for the channel groups whose A stages,
// weight stages and output staging fit the shared memory.  Returns its layout, or false: the layer converts through
// tensor memory.
static bool smem_a_layout(const cvt::Params& P, bool presplit_one_scale, cvt::SmemA& L) {
  if (!presplit_one_scale || !(P.n_group <= 96 || (P.stride == 2 && P.n_group == 128))) return false;
  L.a_box_bytes = (uint32_t)(cvt::kTileW * (P.per_tap ? cvt::kTileH : cvt::kTileH + 2) * 128);
  L.b_stage_bytes = (uint32_t)(6 * P.nhalf * 64 + 1023) / 1024 * 1024;
  L.off_b = cvt::kAStagesS * 3 * L.a_box_bytes;
  const long room = (long)cvt::kMaxDynSmem - 1024 - L.off_b - cvt::smem_a_tail_bytes(P.ncol32);
  L.b_stages = (int)(room / (long)L.b_stage_bytes < cvt::kStages ? room / (long)L.b_stage_bytes : cvt::kStages);
  L.off_sum = L.off_b + (uint32_t)L.b_stages * L.b_stage_bytes;
  return L.b_stages >= 2;
}

static int conv2d_nhwc_impl(const float* x, int n, int h, int w, int cin, long x_pixel_stride, const float* x_amax,
                            int n_amax, int amax_per_image, const float* packed, const float* bias, int cout, int ksize, int stride,
                            int relu, float* y, long y_pixel_stride, float* y_amax, const float* residual,
                            int residual_upsample2, const float* a_gate, const float* a_shift, int a_relu, float* colsum,
                            float* colsumsq, const float* x_actual, float* y_bound, float y_l1, float y_beta,
                            int x_presplit_from, const int* slice_ch, fod_stream_t stream) {
  FOD_REQUIRE((((uintptr_t)a_gate | (uintptr_t)a_shift | (uintptr_t)colsum | (uintptr_t)colsumsq) & 15) == 0,
              "fod_conv2d_nhwc: a_gate / a_shift / colsum / colsumsq must be 16-byte aligned");
  FOD_REQUIRE((!a_gate && !a_shift) || cin % 32 == 0, "fod_conv2d_nhwc: a_gate / a_shift need cin to be a multiple of 32");
  FOD_REQUIRE(!colsumsq || colsum, "fod_conv2d_nhwc: colsumsq needs colsum");
  FOD_REQUIRE(x && packed && y && x_amax, "fod_conv2d_nhwc: null pointer");
  FOD_REQUIRE(((uintptr_t)residual & 15) == 0, "fod_conv2d_nhwc: residual must be 16-byte aligned");
  FOD_REQUIRE(n_amax >= 1 && n_amax <= 8, "fod_conv2d_nhwc: 1..8 input bounds");
  FOD_REQUIRE(n >= 0 && h > 0 && w > 0 && cin > 0 && cout > 0, "fod_conv2d_nhwc: bad sizes");
  FOD_REQUIRE(ksize == 1 || ksize == 3, "fod_conv2d_nhwc: ksize must be 1 or 3");
  FOD_REQUIRE(stride == 1 || (stride == 2 && ksize == 3), "fod_conv2d_nhwc: stride 1, or stride 2 with a 3x3 kernel");
  FOD_REQUIRE(cin % 4 == 0 && cout % 4 == 0 && x_pixel_stride % 4 == 0 && y_pixel_stride % 4 == 0 &&
                  x_pixel_stride >= cin && y_pixel_stride >= cout,
              "fod_conv2d_nhwc: channel counts and pixel strides must be multiples of 4 (16-byte TMA granularity)");
  FOD_REQUIRE((((uintptr_t)x | (uintptr_t)y | (uintptr_t)packed) & 15) == 0, "fod_conv2d_nhwc: pointers must be 16-byte aligned");
  if (n == 0) return FOD_OK;
  const int pad = ksize / 2;
  const int ho = (h + 2 * pad - ksize) / stride + 1, wo = (w + 2 * pad - ksize) / stride + 1;
  cvt::Params prm = {};
  cvt::TmemA tm = {};
  const int per_tap = stride != 1;
  // stride 1: tile + halo; stride 2: every second pixel of a (2*16-1) x (2*8-1) window = the 16 x 8 pixels of one tap
  const int halo_w = per_tap ? (cvt::kTileW - 1) * stride + 1 : cvt::kTileW + ksize - 1;
  const int halo_h = per_tap ? (cvt::kTileH - 1) * stride + 1 : cvt::kTileH + ksize - 1;
  prm.per_tap = per_tap;
  tm.halo_w = per_tap ? cvt::kTileW : halo_w;
  tm.q_stage_bytes = per_tap ? (uint32_t)(cvt::kTileW * cvt::kTileH * 128) : (uint32_t)(halo_w * halo_h * 128);
  tm.q_stage_stride = (tm.q_stage_bytes + 1023) / 1024 * 1024;
  FOD_REQUIRE(cvt::kQStages * tm.q_stage_stride <= cvt::kOffB, "fod_conv2d_nhwc: halo tile does not fit the input ring");
  const int cin_pad = (cin + 31) / 32 * 32;
  tm.ksize = ksize;
  prm.taps = ksize * ksize;
  prm.stride = stride;
  prm.cin_chunks = cin_pad / 32;
  prm.chunks = prm.taps * prm.cin_chunks;
  prm.parts = (prm.chunks + cvt::kPartChunks - 1) / cvt::kPartChunks;
  prm.chunks_per_part = (prm.chunks + prm.parts - 1) / prm.parts;
  prm.parts = (prm.chunks + prm.chunks_per_part - 1) / prm.chunks_per_part;
  const int n16 = (cout + 15) / 16 * 16;
  prm.n_group = n16 < 128 ? n16 : 128;
  prm.n_groups = (cout + prm.n_group - 1) / prm.n_group;
  prm.nhalf = prm.n_group / 2;
  prm.ncol32 = (prm.n_group + 31) / 32;
  prm.cout = cout;
  prm.relu = relu;
  prm.bias = bias;
  prm.x_amax = x_amax;
  prm.n_amax = n_amax;
  prm.y_amax = y_amax;
  prm.x_amax_stride = (amax_per_image & 1) ? n : 0;
  tm.x_presplit = (amax_per_image & 4) ? 1 : 0;
  FOD_REQUIRE(!tm.x_presplit || (ksize == 3 && stride == 1 && !a_gate && !a_shift && cin % 16 == 0 && x_pixel_stride % 16 == 0),
              "fod_conv2d_nhwc: a pre-split input needs a 3x3 stride-1 convolution over whole 16-channel groups without a_gate / a_shift");
  prm.y_amax_per_image = (amax_per_image & 2) ? 1 : 0;
  prm.x_actual = x_actual;
  prm.y_bound = y_bound;
  prm.y_l1 = y_l1;
  prm.y_beta = y_beta;
  tm.x_presplit_from = x_presplit_from >= 0 ? x_presplit_from : (1 << 30);
  for (int k = 0; k < 8; ++k) tm.slice_ch[k] = (slice_ch && k < n_amax) ? slice_ch[k] : 0;
  FOD_REQUIRE(!y_bound || (!residual && !colsum && cout % 16 == 0 && y_pixel_stride % 16 == 0 && relu),
              "fod_conv2d_nhwc_split: a split output needs ReLU, whole 16-channel groups and no residual / colsum");
  FOD_REQUIRE(x_presplit_from < 0 || ((ksize == 1 || stride != 1) && slice_ch && x_presplit_from % 16 == 0 && cin % 16 == 0 &&
                                      x_pixel_stride % 16 == 0 && !a_gate && !a_shift),
              "fod_conv2d_nhwc_split: pre-split slices need a single-tap-per-tile convolution (1x1 or stride 2) over whole "
              "16-channel groups without a_gate / a_shift");
  prm.ho = ho;
  prm.wo = wo;
  tm.a_gate = a_gate;
  tm.a_shift = a_shift;
  tm.a_relu = a_relu;
  tm.in_h = h;
  tm.in_w = w;
  prm.colsum = colsum;
  prm.colsumsq = colsumsq;
  tm.cin = cin;
  prm.res = residual;
  prm.res_shift = residual_upsample2 ? 1 : 0;
  prm.res_h = residual_upsample2 ? (ho + 1) / 2 : ho;
  prm.res_w = residual_upsample2 ? (wo + 1) / 2 : wo;
  prm.tiles_x = (wo + cvt::kTileW - 1) / cvt::kTileW;
  prm.tiles_per_img = prm.tiles_x * ((ho + cvt::kTileH - 1) / cvt::kTileH);
  const long tiles = (long)n * prm.tiles_per_img;
  FOD_REQUIRE(tiles * prm.n_groups < (1L << 30), "fod_conv2d_nhwc: too many tiles");
  prm.tiles_total = (int)tiles;
  prm.pair_units = (int)((tiles + 1) / 2) * prm.n_groups;
  cvt::SmemA sm = {};
  const bool smem_a = smem_a_layout(prm, tm.x_presplit || (stride == 2 && x_presplit_from == 0 && n_amax == 1), sm);
  // stride 1 with A in shared memory: three dx-shifted boxes of the tile's width instead of one halo-wide box
  int rc = make_nhwc_map(&prm.in_map, x, n, h, w, cin, x_pixel_stride, cvt::kChunk, smem_a && !per_tap ? cvt::kTileW : halo_w,
                         halo_h, stride, CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc != FOD_OK) return rc;
  rc = make_nhwc_map(&prm.out_map, y, n, ho, wo, cout, y_pixel_stride, cvt::kChunk, cvt::kTileW, cvt::kTileH, 1,
                     CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc != FOD_OK) return rc;
  const long ktot = (long)prm.taps * cin_pad;
  const __half* whi = reinterpret_cast<const __half*>(packed);
  rc = make_matrix_map_f16(&prm.whi_map, whi, cout, ktot, cvt::kChunk, prm.nhalf);
  if (rc != FOD_OK) return rc;
  rc = make_matrix_map_f16(&prm.wlo_map, whi + (size_t)cout * ktot, cout, ktot, cvt::kChunk, prm.nhalf);
  if (rc != FOD_OK) return rc;
  prm.w_inv = packed + (size_t)cout * ktot;   // tail[0] = 1 / weight scale
  rc = pair_count(prm.pair_units, &prm.num_pairs);
  if (rc != FOD_OK) return rc;
  const void* kernel = smem_a ? (const void*)cvt::conv_tc_kernel_smem : (const void*)cvt::conv_tc_kernel_tmem;
  void* args[] = {&prm, smem_a ? (void*)&sm : (void*)&tm};
  const uint32_t smem_bytes = smem_a ? sm.off_sum + cvt::smem_a_tail_bytes(prm.ncol32) + 1024 : cvt::kSmemAlloc;
  return launch_clusters(kernel, args, prm.num_pairs, 2, smem_a ? cvt::kThreadsS : cvt::kThreads, smem_bytes, stream,
                         "fod_conv2d_nhwc");
}

extern "C" int fod_conv2d_nhwc(const float* x, int n, int h, int w, int cin, long x_pixel_stride, const float* x_amax,
                               int n_amax, int amax_per_image, const float* packed, const float* bias, int cout, int ksize, int stride,
                               int relu, float* y, long y_pixel_stride, float* y_amax, const float* residual,
                               int residual_upsample2, const float* a_gate, const float* a_shift, int a_relu, float* colsum,
                               float* colsumsq, fod_stream_t stream) {
  return conv2d_nhwc_impl(x, n, h, w, cin, x_pixel_stride, x_amax, n_amax, amax_per_image, packed, bias, cout, ksize, stride, relu, y,
                          y_pixel_stride, y_amax, residual, residual_upsample2, a_gate, a_shift, a_relu, colsum, colsumsq, nullptr,
                          nullptr, 0.f, 0.f, -1, nullptr, stream);
}

extern "C" int fod_conv2d_nhwc_split(const float* x, int n, int h, int w, int cin, long x_pixel_stride, const float* x_amax,
                                     int n_amax, int amax_per_image, const float* packed, const float* bias, int cout, int ksize,
                                     int stride, int relu, float* y, long y_pixel_stride, float* y_amax, float* colsum,
                                     const float* x_actual, float* y_bound, float y_l1, float y_beta, int x_presplit_from,
                                     const int* slice_ch, fod_stream_t stream) {
  return conv2d_nhwc_impl(x, n, h, w, cin, x_pixel_stride, x_amax, n_amax, amax_per_image, packed, bias, cout, ksize, stride, relu, y,
                          y_pixel_stride, y_amax, nullptr, 0, nullptr, nullptr, 0, colsum, nullptr, x_actual, y_bound, y_l1, y_beta,
                          x_presplit_from, slice_ch, stream);
}
