// Q2+Q3 on the 5th-generation tensor cores: depthwise support correlation fused with the 1x1 relation
// conv (fsod_cen.py:463-470, 482-491, 502-509), all FPN levels and all (image, class) problems in ONE
// persistent launch.
//
//   attn[p][y][x][:] = relu( W3 . [ s(y,x,:) | q(y,x,:) ] + b3 ),   s = a + b + q,
//   a = relu(k11 * relu(k11 * q)),   b = relu(conv3x1_k31(relu(conv1x3_k13(q))))   (zero padding)
//
// Design (B200, sm_100a)
//   * work unit = tile of 8 x 16 pixels of one problem (128 rows of the GEMM).  CTAs run as pairs (cluster of 2,
//     tcgen05 cta_group::2): one MMA covers both CTAs' tiles (M = 256) against W3 (N = 128) whose rows are split
//     between the two CTAs, so each CTA keeps only half of the weights resident in shared memory (hi + lo tf32
//     parts of 64 x 256 fp32 = 128 KB) for the whole kernel.
//   * fp32 accuracy on tf32 tensor cores by operand splitting (3xTF32): x = hi + lo, A.B ~ Ahi.Bhi + Alo.Bhi +
//     Ahi.Blo, fp32 accumulation in tensor memory; measured error ~1e-6 relative (tools/tc_probe.cu).
//   * the query tile (+1 pixel halo, zero-filled outside the image by TMA) is staged channel-chunk-wise
//     (32 channels = one 128-byte swizzled row per pixel) into a 3-deep shared-memory ring by TMA.
//   * 16 "stencil" warps build the A operand: one pixel per lane (TMEM lane = pixel), they read the 3x3
//     neighbourhood from the ring (conflict-free LDS.128 thanks to the TMA swizzle), evaluate s with packed
//     f32x2 math, split s and q into hi/lo and write them straight into TENSOR MEMORY (tcgen05.st): the A operand
//     never exists in shared or global memory, and the MMA reads only the weights from shared memory.  The support
//     taps are warp-uniform: they sit in the constant bank and reach the FMAs through uniform registers (LDCU),
//     costing no shared-memory bandwidth.  A stages are 16 channels wide, 4 deep; warp k of a quadrant owns the
//     sub-chunks with index % 4 == k, so the warps of one SM sub-partition sit in different pipeline phases.
//   * one thread of the leader CTA issues the MMAs (12 per sub-chunk), completion is tracked with tcgen05.commit
//     multicast to both CTAs; accumulators are double buffered in tensor memory (2 x 128 columns).
//   * 4 epilogue warps: tcgen05.ld -> + bias, ReLU -> swizzled staging tile -> TMA store (clipped at the image
//     border by the tensor map).
//   HBM traffic = read q once + write attn once = 1024 B per pixel per problem (SURVEY 8d).
#include "common.cuh"
#include "tc05.cuh"

namespace fod {

using namespace tc;

namespace ctc {

constexpr int kTileH = 8, kTileW = 16, kTilePx = 128;
constexpr int kHaloH = kTileH + 2, kHaloW = kTileW + 2, kHaloPx = kHaloH * kHaloW;  // 10 x 18 = 180
constexpr int kChunk = 32;                                                           // channels per chunk
constexpr int kNumChunks = kC / kChunk;                                              // 4
constexpr int kQStages = 3, kAStages = 4, kAccStages = 2;
constexpr int kSub = 16;                      // channels per A stage (sub-chunk); 2 per 32-channel q box
constexpr int kNumSubs = kC / kSub;           // 8 per tile
constexpr uint32_t kAStageCols = 4 * kSub;    // [s_hi 16 | s_lo 16 | q_hi 16 | q_lo 16]
constexpr uint32_t kQStageBytes = kHaloPx * 128;         // 23040
constexpr uint32_t kQStageStride = 23552;                // rounded up to 1024
constexpr uint32_t kBHalfRows = 64;                      // W3 rows per CTA
constexpr uint32_t kBChunkBytes = kBHalfRows * 128;      // 8192: one 32-wide K chunk
constexpr uint32_t kBPartBytes = 8 * kBChunkBytes;       // 65536: K = 256
constexpr uint32_t kStageOutBytes = kTilePx * 128;       // 16384

// shared memory map (offsets from the 1024-aligned base)
constexpr uint32_t kOffBHi = 0;
constexpr uint32_t kOffBLo = kOffBHi + kBPartBytes;
constexpr uint32_t kOffQ = kOffBLo + kBPartBytes;
constexpr uint32_t kOffOut = kOffQ + kQStages * kQStageStride;
constexpr uint32_t kOffBias = kOffOut + kStageOutBytes;
constexpr uint32_t kOffBars = kOffBias + kC * 4;
constexpr uint32_t kNumBars = 2 * kQStages + 2 * kAStages + 2 * kAccStages;
constexpr uint32_t kOffTmemPtr = kOffBars + kNumBars * 8;
constexpr uint32_t kOffFlag = kOffTmemPtr + 8;  // sub-chunks released to the MMA thread by its barrier watcher
constexpr uint32_t kSmemBytes = kOffTmemPtr + 16;
constexpr uint32_t kSmemAlloc = kSmemBytes + 1024;

constexpr int kThreads = 768;
constexpr int kWarpTma = 0, kWarpMma = 1, kWarpAlloc = 2, kWarpEpi0 = 4, kWarpSten0 = 8;
constexpr int kStencilWarps = 16;

// tensor memory columns
constexpr uint32_t kTmemCols = 512;
constexpr uint32_t kColA = 0;      // 4 stages x [s_hi 16 | s_lo 16 | q_hi 16 | q_lo 16]
constexpr uint32_t kColAcc = 256;  // 2 stages x 128

// Support taps of every (level, class) set of one launch travel INSIDE THE LAUNCH PARAMETERS (constant bank 0): a tap is
// warp-uniform, so it reaches the FMA as a uniform / constant operand instead of costing shared-memory bandwidth per
// lane, and - unlike a __constant__ symbol - the values belong to the launch, not to the device: concurrent calls on
// different streams (or a graph replay next to an eager call) cannot overwrite each other's taps.
constexpr int kMaxTapSets = 6;     // 6 x 4 KB of the 32 764-byte parameter space (CUDA >= 12.1)
constexpr int kStencilUnroll = 1;  // measured: 1, 2 and 4 run at the same speed; 1 keeps the body inside the L0 I-cache
// rows 0..6: k11, k13 (left, centre, right), k31 (up, centre, down); row 7: c11 = k11 > 0 ? k11*k11 : 0
constexpr int kTapRows = 8;

struct Level {
  int H, W, tiles_x, tiles_per_problem, tiles_per_class, tile_begin;  // tiles_per_class = batch * tiles_per_problem
};

struct Params {
  CUtensorMap in_map[FOD_MAX_LEVELS];   // [B][H][W][128], box 32 x 18 x 10
  CUtensorMap out_map[FOD_MAX_LEVELS];  // [P][H][W][128], box 32 x 16 x 8
  Level lv[FOD_MAX_LEVELS];
  const float* w3;
  const float* b3;
  float* attn_amax[FOD_MAX_LEVELS];   // null or, per level, [B*C] device floats (zeroed by the caller): entry p is raised to
                                      // max(attn of problem p) - per problem, so that the operand scale of the convolution
                                      // that consumes a map does not depend on the other problems of the batch
  // problems of this launch: images x classes [class_begin, class_begin + class_count) of num_classes
  int num_levels, num_classes, class_begin, class_count, total_tiles, num_pairs;
  // tap sets of this launch, set = level * class_count + class (filled on the host from the caller's HOST taps)
  alignas(16) float taps[kMaxTapSets][kTapRows][kC];
};

// Tile order: level-major, then class, then image, then tile (all tiles that share one tap set are contiguous).
struct TileCoord {
  int level, b, cc, y0, x0;  // image, class index inside the launch's class group
};

__device__ __forceinline__ TileCoord decode_tile(const Params& P, int t) {
  int l = 0;
  if (P.num_levels > 1 && t >= P.lv[1].tile_begin) l = 1;
  if (P.num_levels > 2 && t >= P.lv[2].tile_begin) l = 2;
  const Level& L = P.lv[l];
  int r = t - L.tile_begin;
  int cc = r / L.tiles_per_class;
  r -= cc * L.tiles_per_class;
  int b = r / L.tiles_per_problem;
  int tt = r - b * L.tiles_per_problem;
  int ty = tt / L.tiles_x;
  TileCoord tc;
  tc.level = l;
  tc.b = b;
  tc.cc = cc;
  tc.y0 = ty * kTileH;
  tc.x0 = (tt - ty * L.tiles_x) * kTileW;
  return tc;
}

__device__ __forceinline__ float4 lds4(const uint8_t* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 f4_relu(float4 v) {
  return make_float4(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f), fmaxf(v.z, 0.f), fmaxf(v.w, 0.f));
}
__device__ __forceinline__ float4 f4_mul(float4 a, float4 b) { return make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w); }
__device__ __forceinline__ float4 f4_fma(float4 a, float4 b, float4 c) {
  return make_float4(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y), fmaf(a.z, b.z, c.z), fmaf(a.w, b.w, c.w));
}
__device__ __forceinline__ float4 f4_add(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

struct StencilCtx {
  uint8_t* smem;
  uint32_t sbase, tmem_base, bar0;
  int pair, rank;
};

__device__ __forceinline__ float2 relu2(float2 v) { return make_float2(fmaxf(v.x, 0.f), fmaxf(v.y, 0.f)); }
__device__ __forceinline__ void split2(float2 v, uint32_t& h0, uint32_t& h1, uint32_t& l0, uint32_t& l1) {
  h0 = (__float_as_uint(v.x) + 0x1000u) & 0xFFFFE000u;  // round to nearest tf32 (see tc05.cuh split_tf32)
  h1 = (__float_as_uint(v.y) + 0x1000u) & 0xFFFFE000u;
  float2 lo = __ffma2_rn(make_float2(__uint_as_float(h0), __uint_as_float(h1)), make_float2(-1.f, -1.f), v);
  l0 = __float_as_uint(lo.x);
  l1 = __float_as_uint(lo.y);
}

// One stencil warp: TMEM lane quadrant qd = warp & 3, one pixel per lane.  The four warps of a quadrant share every
// 32-channel chunk: warp k takes the 16-byte channel groups jj with (jj >> 1) == k.  The loops over chunks and
// groups stay ROLLED with uniform counters (one small code copy for all 16 warps -> instruction cache; the tap
// address set*3584 + ch*128 + jj*16 stays in uniform registers -> LDCU + uniform FFMA2 operands).
__device__ __forceinline__ void stencil_role(const Params& P, const StencilCtx& cx, const int warp) {
  const int lane = threadIdx.x & 31;
  const int qd = warp & 3, myk = (warp - kWarpSten0) >> 2;
  const int m = qd * 32 + lane;
  const int ty = m >> 4, tx = m & 15;
  const uint32_t bar0 = cx.bar0;
  const uint32_t a_full_leader = map_to_cta(bar0 + 8u * (2 * kQStages), 0);
  const uint32_t trow = cx.tmem_base + ((uint32_t)(qd * 32) << 16) + kColA;
  // A warp holds two tile rows (lanes 0..15: row 2 qd, lanes 16..31: row 2 qd + 1).  The 1x3 row pass of a halo row is
  // shared by the three 3x1 taps that read it, so a lane evaluates it for its own row and for the row on the far side
  // (above for the upper half warp, below for the lower one) and takes the third from lane ^ 16, whose own row it is:
  // 6 LDS.128 and 4 SHFL per four channels instead of 9 LDS.128 - the kernel's limiter is the shared-memory pipe.
  // byte offset of 16-byte chunk 0 of a neighbour's 128-byte row (swizzled); chunk jj is this ^ (jj << 4)
  const bool upper = lane < 16;
  uint32_t off_own[3], off_out[3];
#pragma unroll
  for (int dx = 0; dx < 3; ++dx) {
    const int r1 = (ty + 1) * kHaloW + tx + dx, r2 = (ty + (upper ? 0 : 2)) * kHaloW + tx + dx;
    off_own[dx] = (uint32_t)(r1 * 128 + ((r1 & 7) << 4));
    off_out[dx] = (uint32_t)(r2 * 128 + ((r2 & 7) << 4));
  }
  const int T = P.total_tiles;
  int i = 0;
  // Outer loops over the tap sets (level, class): `set` is a loop counter (uniform); this CTA's tiles arrive in
  // set order because tiles are numbered set-major.
  for (int l = 0; l < P.num_levels; ++l)
    for (int cc = 0; cc < P.class_count; ++cc) {
      const int set = l * P.class_count + cc;
      const int set_end = P.lv[l].tile_begin + (cc + 1) * P.lv[l].tiles_per_class;
      for (; 2 * (i * P.num_pairs + cx.pair) < T && min(2 * (i * P.num_pairs + cx.pair) + cx.rank, T - 1) < set_end;
           ++i) {
#pragma unroll 1
        for (int sub = 0; sub < kNumSubs; ++sub) {  // uniform counter; this warp takes sub % 4 == myk
          if ((sub & 3) != myk) continue;
          const uint32_t gq = (uint32_t)i * kNumChunks + (sub >> 1);  // q box (32 channels) of this sub-chunk
          const int qs = gq % kQStages, as_ = sub & 3;                // kNumSubs % kAStages == 0
          const uint32_t qph = (gq / kQStages) & 1, aph = ((uint32_t)i * 2 + (sub >> 2)) & 1;
          mbar_wait(bar0 + 8u * qs, qph);                                   // q_full
          mbar_wait(bar0 + 8u * (2 * kQStages + kAStages + as_), aph ^ 1);  // a_empty
          tc_fence_after();
          const uint32_t qt = cx.sbase + kOffQ + qs * kQStageStride;  // shared-window address: LDS, not generic LD
          const uint32_t tcol = trow + as_ * kAStageCols;
#pragma unroll(kStencilUnroll)
          for (int j4 = 0; j4 < 4; ++j4) {  // 4 channels per step
            {
              const int jj = (sub & 1) * 4 + j4;  // 16-byte channel group inside the q box
              const float* tp = &P.taps[set][0][sub * kSub + j4 * 4];
              const uint32_t jx = (uint32_t)jj << 4;
              const float4 k13l = *reinterpret_cast<const float4*>(tp + 1 * kC);
              const float4 k13c = *reinterpret_cast<const float4*>(tp + 2 * kC);
              const float4 k13r = *reinterpret_cast<const float4*>(tp + 3 * kC);
              uint32_t shi[4], slo[4], qhi[4], qlo[4];
              float4 qc4;
              float2 t3[3][2];
              float2 t_own[2], t_out[2];
#pragma unroll
              for (int rr = 0; rr < 2; ++rr) {   // rr = 0: the lane's own row, 1: the row on the far side
                const float4 ql = lds4s(qt + ((rr ? off_out[0] : off_own[0]) ^ jx));
                const float4 qm = lds4s(qt + ((rr ? off_out[1] : off_own[1]) ^ jx));
                const float4 qr = lds4s(qt + ((rr ? off_out[2] : off_own[2]) ^ jx));
                if (rr == 0) qc4 = qm;
                const float2 v0 = relu2(__ffma2_rn(make_float2(k13r.x, k13r.y), make_float2(qr.x, qr.y),
                                                   __ffma2_rn(make_float2(k13l.x, k13l.y), make_float2(ql.x, ql.y),
                                                              __fmul2_rn(make_float2(k13c.x, k13c.y), make_float2(qm.x, qm.y)))));
                const float2 v1 = relu2(__ffma2_rn(make_float2(k13r.z, k13r.w), make_float2(qr.z, qr.w),
                                                   __ffma2_rn(make_float2(k13l.z, k13l.w), make_float2(ql.z, ql.w),
                                                              __fmul2_rn(make_float2(k13c.z, k13c.w), make_float2(qm.z, qm.w)))));
                if (rr == 0) {
                  t_own[0] = v0;
                  t_own[1] = v1;
                } else {
                  t_out[0] = v0;
                  t_out[1] = v1;
                }
              }
#pragma unroll
              for (int h = 0; h < 2; ++h) {
                const float2 t_x = make_float2(__shfl_xor_sync(0xffffffffu, t_own[h].x, 16), __shfl_xor_sync(0xffffffffu, t_own[h].y, 16));
                t3[0][h] = upper ? t_out[h] : t_x;
                t3[1][h] = t_own[h];
                t3[2][h] = upper ? t_x : t_out[h];
              }
              const float4 c11 = *reinterpret_cast<const float4*>(tp + 7 * kC);
              const float4 k31u = *reinterpret_cast<const float4*>(tp + 4 * kC);
              const float4 k31c = *reinterpret_cast<const float4*>(tp + 5 * kC);
              const float4 k31d = *reinterpret_cast<const float4*>(tp + 6 * kC);
#pragma unroll
              for (int h = 0; h < 2; ++h) {
                const float2 k1 = h ? make_float2(c11.z, c11.w) : make_float2(c11.x, c11.y);
                const float2 ku = h ? make_float2(k31u.z, k31u.w) : make_float2(k31u.x, k31u.y);
                const float2 kc = h ? make_float2(k31c.z, k31c.w) : make_float2(k31c.x, k31c.y);
                const float2 kd = h ? make_float2(k31d.z, k31d.w) : make_float2(k31d.x, k31d.y);
                const float2 qc = h ? make_float2(qc4.z, qc4.w) : make_float2(qc4.x, qc4.y);
                const float2 bv = relu2(__ffma2_rn(kd, t3[2][h], __ffma2_rn(ku, t3[0][h], __fmul2_rn(kc, t3[1][h]))));
                // a = relu(k11 * relu(k11 * q)) == c11 * relu(q) with c11 = k11 > 0 ? k11^2 : 0 (row 7 of the set)
                const float2 sv = __fadd2_rn(__ffma2_rn(k1, relu2(qc), bv), qc);
                split2(sv, shi[2 * h], shi[2 * h + 1], slo[2 * h], slo[2 * h + 1]);
                split2(qc, qhi[2 * h], qhi[2 * h + 1], qlo[2 * h], qlo[2 * h + 1]);
              }
              tmem_st4(tcol + j4 * 4, shi);
              tmem_st4(tcol + kSub + j4 * 4, slo);
              tmem_st4(tcol + 2 * kSub + j4 * 4, qhi);
              tmem_st4(tcol + 3 * kSub + j4 * 4, qlo);
            }
          }
          tmem_wait_st();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            mbar_arrive(bar0 + 8u * (kQStages + qs));       // q_empty
            mbar_arrive_remote(a_full_leader + 8u * as_);   // a_full (leader CTA)
          }
        }
      }
    }
}

__global__ void __launch_bounds__(kThreads, 1) correlate_tc_kernel(const __grid_constant__ Params P) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const uint32_t sbase = smem_u32(smem);
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  // rank inside the CTA pair; == %cluster_ctarank for cluster dims (2,1,1), but written from blockIdx so that ptxas
  // can prove it warp-uniform (an inline-asm special-register read is opaque to its uniformity analysis)
  const uint32_t rank = blockIdx.x & 1;
  const int pair = blockIdx.x >> 1;

  // barrier addresses
  const uint32_t bar0 = sbase + kOffBars;
  auto q_full = [&](int s) { return bar0 + 8u * s; };
  auto q_empty = [&](int s) { return bar0 + 8u * (kQStages + s); };
  auto a_full = [&](int s) { return bar0 + 8u * (2 * kQStages + s); };
  auto a_empty = [&](int s) { return bar0 + 8u * (2 * kQStages + kAStages + s); };
  auto acc_full = [&](int s) { return bar0 + 8u * (2 * kQStages + 2 * kAStages + s); };
  auto acc_empty = [&](int s) { return bar0 + 8u * (2 * kQStages + 2 * kAStages + kAccStages + s); };

  if (tid == 0) {
    for (int s = 0; s < kQStages; ++s) {
      mbar_init(q_full(s), 1);
      mbar_init(q_empty(s), kStencilWarps / 2);  // the 8 warps that read a q box
    }
    for (int s = 0; s < kAStages; ++s) {
      mbar_init(a_full(s), 2 * 4);  // one warp per TMEM quadrant, both CTAs (used in the leader only)
      mbar_init(a_empty(s), 1);
    }
    for (int s = 0; s < kAccStages; ++s) {
      mbar_init(acc_full(s), 1);
      mbar_init(acc_empty(s), 8);  // 4 epilogue warps x 2 CTAs (leader only)
    }
    *reinterpret_cast<volatile uint32_t*>(smem + kOffFlag) = 0;
    fence_barrier_init();
  }
  if (warp == kWarpAlloc) {
    tmem_alloc<2>(sbase + kOffTmemPtr, kTmemCols);
    tmem_relinquish<2>();
  }
  if (warp == kWarpTma && lane == 0) {
    for (int l = 0; l < P.num_levels; ++l) {
      tma_prefetch_desc(&P.in_map[l]);
      tma_prefetch_desc(&P.out_map[l]);
    }
  }
  // resident weights: this CTA's 64 rows of W3, split into tf32 hi / lo, K-major SW128 chunks
  {
    const float* wsrc = P.w3 + (size_t)rank * kBHalfRows * 256;
    for (int i = tid; i < (int)kBHalfRows * 64; i += kThreads) {  // float4 index: 64 per row
      int r = i >> 6, c = (i & 63) << 2;
      float4 v = ldg4(wsrc + (size_t)r * 256 + c);
      float x[4] = {v.x, v.y, v.z, v.w};
      uint32_t hi[4], lo[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint32_t h;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(h) : "f"(x[j]));
        hi[j] = h;
        lo[j] = __float_as_uint(x[j] - __uint_as_float(h));
      }
      uint32_t off = (uint32_t)(c >> 5) * kBChunkBytes + sw128_offset(r, c & 31);
      *reinterpret_cast<uint4*>(smem + kOffBHi + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
      *reinterpret_cast<uint4*>(smem + kOffBLo + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    }
    if (tid < kC) reinterpret_cast<float*>(smem + kOffBias)[tid] = P.b3[tid];
  }
  fence_proxy_async_smem();
  tc_fence_before();
  cluster_sync();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem + kOffTmemPtr);

  // static schedule: iteration i of pair k handles tiles 2*(i*num_pairs + k) + rank
  const int T = P.total_tiles;
  auto tile_of = [&](int i) { return 2 * (i * P.num_pairs + pair) + (int)rank; };
  auto iter_valid = [&](int i) { return 2 * (i * P.num_pairs + pair) < T; };

  if (warp == kWarpTma) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      uint32_t g = 0;
      for (int i = 0; iter_valid(i); ++i) {
        int t = min(tile_of(i), T - 1);
        TileCoord tcd = decode_tile(P, t);
        int b = tcd.b;
        for (int ch = 0; ch < kNumChunks; ++ch, ++g) {
          int s = g % kQStages;
          uint32_t ph = (g / kQStages) & 1;
          mbar_wait(q_empty(s), ph ^ 1);
          mbar_arrive_expect_tx(q_full(s), kQStageBytes);
          tma_load_4d(sbase + kOffQ + s * kQStageStride, &P.in_map[tcd.level], q_full(s), ch * kChunk, tcd.x0 - 1,
                      tcd.y0 - 1, b);
        }
      }
    }
  } else if (warp == kWarpMma) {
    // ------------------------------------------------------------------ MMA issuer (leader CTA, one thread)
    if (rank == 0) {
      const uint32_t idesc = idesc_tf32(256, 128);
      const uint64_t bhi0 = smem_desc_k_sw128(sbase + kOffBHi);
      const uint64_t blo0 = smem_desc_k_sw128(sbase + kOffBLo);
      // A watcher thread (warp kWarpAlloc) does all the barrier waiting and publishes the number of sub-chunks whose
      // operands are in place through one shared-memory word; this warp only polls that word.  The whole warp runs
      // the loop converged and one elected lane issues, so that every tcgen05.mma operand is a warp-uniform value
      // in a uniform register (inside an `if (lane == 0)` region ptxas wraps each MMA in a broadcast-and-retry loop
      // whose latency exceeds the 64 cycles of the MMA itself).
      int n_iter = 0;
      for (int i = 0; iter_valid(i); ++i) ++n_iter;
      const uint32_t total = (uint32_t)n_iter * kNumSubs;
      const uint32_t flag = sbase + kOffFlag;
      uint32_t upto = 0;
      for (uint32_t g = 0; g < total; ++g) {
        while (upto <= g) {
          uint32_t v;
          asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(v) : "r"(flag) : "memory");
          upto = __shfl_sync(0xffffffffu, v, 0);
        }
        tc_fence_after();
        const int sub = g % kNumSubs, s = g % kAStages;
        const int as_ = (g / kNumSubs) % kAccStages;
        const uint32_t d = tmem_base + kColAcc + as_ * 128;
        const uint32_t a0 = tmem_base + kColA + s * kAStageCols;
        if (elect_one()) {
#pragma unroll
          for (int half = 0; half < 2; ++half) {
#pragma unroll
            for (int ks = 0; ks < kSub / 8; ++ks) {
              const uint32_t ah = a0 + half * 2 * kSub + ks * 8, al = ah + kSub;
              const uint64_t boff =
                  (uint64_t)(((half * 4 + (sub >> 1)) * kBChunkBytes + (sub & 1) * kSub * 4 + ks * 32) >> 4);
              const uint32_t acc = (sub | half | ks) ? 1u : 0u;
              mma_tf32_ts<2>(d, ah, bhi0 + boff, idesc, acc);
              mma_tf32_ts<2>(d, al, bhi0 + boff, idesc, 1u);
              mma_tf32_ts<2>(d, ah, blo0 + boff, idesc, 1u);
            }
          }
          mma_commit_pair(a_empty(s), 3);
          if (sub == kNumSubs - 1) mma_commit_pair(acc_full(as_), 3);
        }
        __syncwarp();
      }
    }
  } else if (warp == kWarpAlloc) {
    // ------------------------------------------------------------------ barrier watcher of the MMA thread (leader)
    if (rank == 0 && lane == 0) {
      int n_iter = 0;
      for (int i = 0; iter_valid(i); ++i) ++n_iter;
      const uint32_t total = (uint32_t)n_iter * kNumSubs;
      const uint32_t flag = sbase + kOffFlag;
      for (uint32_t g = 0; g < total; ++g) {
        if (g % kNumSubs == 0) {  // first sub-chunk of a tile: its accumulator must have been drained
          const uint32_t it = g / kNumSubs;
          mbar_wait(acc_empty(it % kAccStages), ((it / kAccStages) & 1) ^ 1);
        }
        mbar_wait(a_full(g % kAStages), (g / kAStages) & 1);
        asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"(flag), "r"(g + 1) : "memory");
      }
    }
  } else if (warp >= kWarpEpi0 && warp < kWarpEpi0 + 4) {
    // ------------------------------------------------------------------ epilogue
    const int qd = warp & 3;
    const int m = qd * 32 + lane;  // pixel row of the tile == TMEM lane
    const uint32_t acc_empty_leader = map_to_cta(acc_empty(0), 0);
    const bool issuer = (warp == kWarpEpi0 && lane == 0);
    for (int i = 0; iter_valid(i); ++i) {
      int t = tile_of(i);
      bool do_store = t < T;
      TileCoord tcd = decode_tile(P, min(t, T - 1));
      const int pg = tcd.b * P.num_classes + P.class_begin + tcd.cc;
      int as_ = i % kAccStages;
      uint32_t aph = (i / kAccStages) & 1;
      mbar_wait(acc_full(as_), aph);
      tc_fence_after();
      const uint32_t trow = tmem_base + ((uint32_t)(qd * 32) << 16) + kColAcc + as_ * 128;
      const bool px_valid = do_store && tcd.y0 + (m >> 4) < P.lv[tcd.level].H && tcd.x0 + (m & 15) < P.lv[tcd.level].W;
      float vmax = 0.f;
#pragma unroll 1
      for (int j = 0; j < 4; ++j) {
        uint32_t v[32];
        tmem_ld32(trow + j * 32, v);
        tmem_wait_ld();
        if (j == 3) {  // accumulator fully read: hand it back to the MMA warp
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_remote(acc_empty_leader + 8u * as_);
        }
        if (issuer) tma_store_wait_read<0>();  // staging tile free again
        named_bar_sync(1, 128);
#pragma unroll
        for (int c4 = 0; c4 < 8; ++c4) {
          const float4 bb = lds4s(sbase + kOffBias + (j * 32 + c4 * 4) * 4);
          float4 o;
          o.x = fmaxf(__uint_as_float(v[c4 * 4 + 0]) + bb.x, 0.f);
          o.y = fmaxf(__uint_as_float(v[c4 * 4 + 1]) + bb.y, 0.f);
          o.z = fmaxf(__uint_as_float(v[c4 * 4 + 2]) + bb.z, 0.f);
          o.w = fmaxf(__uint_as_float(v[c4 * 4 + 3]) + bb.w, 0.f);
          vmax = fmaxf(fmaxf(vmax, fmaxf(o.x, o.y)), fmaxf(o.z, o.w));
          sts4s(sbase + kOffOut + (m >> 3) * 1024 + (m & 7) * 128 + ((c4 ^ (m & 7)) << 4), o);
        }
        fence_proxy_async_smem();
        named_bar_sync(1, 128);
        if (issuer && do_store) {
          tma_store_4d(&P.out_map[tcd.level], sbase + kOffOut, j * 32, tcd.x0, tcd.y0, pg);
          tma_store_commit();
        }
      }
      // max of this problem's output (>= 0 after the ReLU) = the operand bound the tower convolution needs
      // (fod_conv2d_nhwc x_amax, per image): one atomic per warp and tile, no extra pass over the maps
      if (P.attn_amax[tcd.level]) {
        const uint32_t wmax = __reduce_max_sync(0xffffffffu, __float_as_uint(px_valid ? vmax : 0.f));
        if (lane == 0 && wmax) atomicMax(reinterpret_cast<unsigned int*>(P.attn_amax[tcd.level] + pg), wmax);
      }
    }
    if (issuer) tma_store_wait<0>();
  } else if (warp >= kWarpSten0) {
    // ------------------------------------------------------------------ stencil: build A in tensor memory
    StencilCtx cx;
    cx.smem = smem;
    cx.sbase = sbase;
    cx.tmem_base = tmem_base;
    cx.bar0 = bar0;
    cx.pair = pair;
    cx.rank = (int)rank;
    stencil_role(P, cx, warp);
  }
  // ---------------------------------------------------------------------- teardown
  __syncwarp();
  tc_fence_before();
  cluster_sync();
  if (warp == kWarpAlloc) tmem_dealloc<2>(tmem_base, kTmemCols);
}

}  // namespace ctc
}  // namespace fod

using namespace fod;

extern "C" int fod_correlate_levels(const float* const* q, const float* const* taps, const fod_level_t* levels,
                                    int num_levels, const float* w3, const float* b3, float* const* attn,
                                    float* const* attn_amax, int batch, int num_classes, fod_stream_t stream) {
  FOD_REQUIRE(q && taps && levels && w3 && b3 && attn, "fod_correlate_levels: null pointer");
  FOD_REQUIRE(num_levels >= 1 && num_levels <= FOD_MAX_LEVELS, "fod_correlate_levels: 1..%d levels", FOD_MAX_LEVELS);
  FOD_REQUIRE(batch >= 0 && num_classes >= 0, "fod_correlate_levels: bad sizes");
  FOD_REQUIRE((((uintptr_t)w3 | (uintptr_t)b3) & 15) == 0, "fod_correlate_levels: weights must be 16-byte aligned");
  if ((long)batch * num_classes == 0) return FOD_OK;
  FOD_REQUIRE((long)batch * num_classes < (1L << 24), "fod_correlate_levels: too many problems");
  ctc::Params prm;
  memset(&prm, 0, sizeof(prm));
  for (int l = 0; l < num_levels; ++l) {
    const int H = levels[l].height, W = levels[l].width;
    FOD_REQUIRE(H > 0 && W > 0 && q[l] && attn[l] && taps[l], "fod_correlate_levels: level %d invalid", l);
    prm.attn_amax[l] = attn_amax ? attn_amax[l] : nullptr;
    FOD_REQUIRE((((uintptr_t)q[l] | (uintptr_t)attn[l]) & 15) == 0,
                "fod_correlate_levels: level %d pointers must be 16-byte aligned", l);
    int rc = make_nhwc_map(&prm.in_map[l], q[l], batch, H, W, kC, kC, ctc::kChunk, ctc::kHaloW, ctc::kHaloH, 1,
                           CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc != FOD_OK) return rc;
    rc = make_nhwc_map(&prm.out_map[l], attn[l], batch * num_classes, H, W, kC, kC, ctc::kChunk, ctc::kTileW, ctc::kTileH, 1,
                       CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc != FOD_OK) return rc;
  }
  prm.w3 = w3;
  prm.b3 = b3;
  prm.num_levels = num_levels;
  prm.num_classes = num_classes;
  int dev = 0, sms = 0;
  FOD_CUDA_CALL(cudaGetDevice(&dev));
  FOD_CUDA_CALL(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int max_pairs = sms / 2 > 0 ? sms / 2 : 1;
  FOD_CUDA_CALL(cudaFuncSetAttribute(ctc::correlate_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)ctc::kSmemAlloc));
  // The taps ride in the launch parameters (ctc::Params::taps, kMaxTapSets sets): classes are processed in groups that
  // fit, one persistent launch per group.  Nothing outside the launch is written: the call is re-entrant.
  const int group = ctc::kMaxTapSets / num_levels;
  for (int c0 = 0; c0 < num_classes; c0 += group) {
    const int cn = num_classes - c0 < group ? num_classes - c0 : group;
    long tiles = 0;
    for (int l = 0; l < num_levels; ++l) {
      ctc::Level& L = prm.lv[l];
      L.H = levels[l].height;
      L.W = levels[l].width;
      L.tiles_x = (L.W + ctc::kTileW - 1) / ctc::kTileW;
      L.tiles_per_problem = L.tiles_x * ((L.H + ctc::kTileH - 1) / ctc::kTileH);
      L.tiles_per_class = batch * L.tiles_per_problem;
      L.tile_begin = (int)tiles;
      tiles += (long)cn * L.tiles_per_class;
      FOD_REQUIRE(tiles < (1L << 30), "fod_correlate_levels: too many tiles");
      for (int cc = 0; cc < cn; ++cc) {   // set = l * cn + cc
        const float* src = taps[l] + (size_t)(c0 + cc) * 7 * kC;
        float(*dst)[kC] = prm.taps[l * cn + cc];
        memcpy(dst, src, sizeof(float) * 7 * kC);
        for (int ch = 0; ch < kC; ++ch) dst[7][ch] = src[ch] > 0.f ? src[ch] * src[ch] : 0.f;
      }
    }
    prm.class_begin = c0;
    prm.class_count = cn;
    prm.total_tiles = (int)tiles;
    const int need_pairs = (int)((tiles + 1) / 2);
    prm.num_pairs = need_pairs < max_pairs ? need_pairs : max_pairs;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * prm.num_pairs);
    cfg.blockDim = dim3(ctc::kThreads);
    cfg.dynamicSmemBytes = ctc::kSmemAlloc;
    cfg.stream = as_stream(stream);
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, ctc::correlate_tc_kernel, prm);
    if (e != cudaSuccess) {
      set_error("fod_correlate_levels: launch failed: %s", cudaGetErrorString(e));
      return FOD_ERR_CUDA;
    }
  }
  return FOD_OK;
}
