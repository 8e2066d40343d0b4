// R2+R3 on the 5th-generation tensor cores: folded relation head (one [rows x 8192] . [8192 x 128] contraction per
// ROI row), per-class bias, ReLU, cls_score / bbox_pred, softmax and apply_deltas
// (fsod_roi_heads.py:482-520, custom_fast_rcnn.py:160-170, d2 box_regression.py:77-115).
//
// Design (B200, sm_100a) - the same skeleton as correlate_tc.cu:
//   * work unit = 128 consecutive ROI rows of one problem; CTA pairs (cluster of 2, cta_group::2) cover two units
//     per MMA (M = 256) and split the 128 rows of the folded weight matrix between them (N = 2 x 64).
//   * K = 8192 is streamed in 32-wide chunks by TMA: the pooled rows (A, fp32, 128-byte swizzle) and the pre-split
//     fp16 hi / lo planes of the folded weights (B, 64-byte swizzle) land in shared-memory rings (6 stages each).
//   * fp32 accuracy on 16-bit tensor-core inputs, the arithmetic of conv_tc.cu: every operand is scaled by a power of
//     two that puts its tensor's largest magnitude into [2^13, 2^14) and split, x * 2^e = hi + lo (two fp16, 22
//     significant bits); a product is hi.hi + lo.hi + hi.lo on kind::f16 MMAs (K = 16 per instruction: half the
//     tensor time of the 3xTF32 scheme this kernel used in round 1), the exact scales are undone in the epilogue.
//   * 8 converter warps (one ROI row per lane = TMEM lane) read their row of the A chunk (conflict-free LDS.128),
//     scale and split it and write the packed fp16 pairs into TENSOR MEMORY; the MMA reads A from tensor memory and
//     only the weights from shared memory.
//   * accumulators (2 x 128 columns) are double buffered; the 4 epilogue warps own one ROI row per lane, so the
//     six output dot products, the softmax and the box decoding need no cross-lane traffic.
#include <cuda_fp16.h>

#include "pair.cuh"
#include "split_format.cuh"

namespace fod {

using namespace tc;

namespace rtc {

constexpr int kK = 64 * kC;          // 8192
constexpr int kChunk = 32;           // K per pipeline stage
constexpr int kNumChunks = kK / kChunk;  // 256
constexpr int kStages = 6;           // A ring, B ring and TMEM A ring
constexpr int kAccStages = 2;
// The tensor core adds into its fp32 accumulator with round-toward-zero (measured, tools/tc_probe.cu acc: the
// relative bias grows by ~1.7e-8 per accumulated MMA).  1536 MMAs per output (K = 8192 / 16, 3 products) would leave
// a 2.6e-5 bias, so the K loop is cut into kParts partial sums of 96 MMAs each (bias ~1.6e-6, the chain length of the
// correlation kernel); the partials are added in IEEE fp32 by the epilogue warps into a running sum held in
// shared memory.
constexpr int kParts = 16;
constexpr int kChunksPerPart = kNumChunks / kParts;  // 16 chunks x 6 MMAs
constexpr uint32_t kABytes = 128 * 128;       // 128 rows x 32 fp32
constexpr uint32_t kBHalfRows = 64;
constexpr uint32_t kBPlaneBytes = kBHalfRows * 64;   // 4096: hi or lo fp16 plane of one chunk (64-byte rows)
constexpr uint32_t kBBytes = 2 * kBPlaneBytes;

constexpr uint32_t kOffA = 0;
constexpr uint32_t kOffB = kOffA + kStages * kABytes;
constexpr uint32_t kOffSum = kOffB + kStages * kBBytes;     // running sum [32 col groups][128 rows] x 16 B
constexpr uint32_t kOffBias = kOffSum + 128 * kC * 4;       // 2 x [128] fp32
constexpr uint32_t kOffWout = kOffBias + 2 * kC * 4;        // [6][128] + [6] (+pad) fp32
constexpr int kMaxProblems = 2047;
constexpr uint32_t kOffPref = kOffWout + (6 * kC + 8) * 4;  // int32[P + 1]: exclusive prefix of units per problem
constexpr uint32_t kOffBars = kOffPref + (kMaxProblems + 1) * 4;
constexpr uint32_t kNumBars = 5 * kStages + 2 * kAccStages;
constexpr uint32_t kOffTmemPtr = kOffBars + kNumBars * 8;
constexpr uint32_t kOffFlag = kOffTmemPtr + 8;   // chunks released to the MMA thread by its barrier watcher
constexpr uint32_t kSmemBytes = kOffTmemPtr + 16;
constexpr uint32_t kSmemAlloc = kSmemBytes + 1024;

// Converter warps: 4 TMEM quadrants x 2 halves of the 32-wide K chunk.  One chunk costs a warp ~900 cycles (two mbarrier
// waits of ~250 cycles each, the split, tcgen05.st), the 6 MMAs of a chunk 384; a second set of 8 warps taking alternate
// chunks measured neutral (119 vs 120 us)
constexpr int kConvWarps = 8;
constexpr int kWarpTma = 0, kWarpMma = 1, kWarpAlloc = 2, kWarpTmaB = 3, kWarpEpi0 = 4, kWarpConv0 = 8;
constexpr int kThreads = (kWarpConv0 + kConvWarps) * 32;  // 512

constexpr uint32_t kTmemCols = 512;
constexpr uint32_t kAStageCols = 32; // [hi: 16 columns of packed fp16 pairs | lo: 16]
constexpr uint32_t kColA = 0;        // 6 stages x 32
constexpr uint32_t kColAcc = 256;    // 2 stages x 128

constexpr float kScaleClamp = 4.135166556742356f;  // log(1000/16), d2 box_regression.py:13

struct Params {
  CUtensorMap a_map;    // pooled, tiled [P*units*256*128][32] (pooled_row in roi.cu), box 32 x 128 (one contiguous 16 KB A tile)
  CUtensorMap whi_map;  // w_fold fp16 hi plane [128][8192], box 32 x 64
  CUtensorMap wlo_map;  // w_fold fp16 lo plane
  const float* x_amax;    // [n_amax] bounds of max|pooled| (= of the feature maps); their maximum fixes the A scale
  const float* w_inv;     // 1 / weight scale (tail of the packed weights)
  int n_amax;
  int amax_stride;        // 0: n_amax scalars (one scale per call); B: x_amax is [n_amax][B], a unit is scaled with column
                          // (problem / classes) - the bounds of ITS image, so batch mates do not influence a result
  const float* bias_cls;  // [C][128]
  const float* rois;      // [P][roi_cap][4]
  const int32_t* roi_count;
  float* det_boxes;
  float* det_scores;
  float* logits;
  float* deltas;
  const float* w_out;     // [6][128]
  const float* b_out;     // [6]
  float reg_w[4];
  int num_problems, classes, roi_cap, tiles_per_problem, num_pairs;
};

struct Slot {
  int p, r0, rows;  // rows = valid ROI rows in this unit (0 = padding unit of the last pair)
};

// Units (128-row tiles that contain at least one ROI) are numbered densely over the problems; pref[p] = number of
// units in problems < p (shared memory, built at kernel start from roi_count).
__device__ __forceinline__ Slot decode_unit(const Params& P, const int* pref, int t) {
  Slot s;
  s.p = 0;
  s.r0 = 0;
  s.rows = 0;
  if (t < pref[P.num_problems]) {
    int lo = 0, hi = P.num_problems - 1;  // largest p with pref[p] <= t
    while (lo < hi) {
      int mid = (lo + hi + 1) >> 1;
      if (pref[mid] <= t) lo = mid; else hi = mid - 1;
    }
    s.p = lo;
    s.r0 = (t - pref[lo]) * 128;
    int cnt = P.roi_count ? min(__ldg(P.roi_count + lo), P.roi_cap) : P.roi_cap;
    s.rows = min(128, cnt - s.r0);
  }
  return s;
}

__global__ void __launch_bounds__(kThreads, 1) relation_tc_kernel(const __grid_constant__ Params P) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const uint32_t sbase = smem_u32(smem);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = blockIdx.x & 1;  // == %cluster_ctarank for cluster dims (2,1,1)
  const int pair = blockIdx.x >> 1;
  float xs = 1.f, xs_inv = 1.f;   // operand scale 2^e of the pooled rows (converters) and its inverse (epilogue)
  auto image_scale = [&](int img) { pow2_scale(image_bound(P.x_amax, P.n_amax, P.amax_stride, img), xs, xs_inv); };
  image_scale(0);

  const uint32_t bar0 = sbase + kOffBars;
  auto a_full = [&](int s) { return bar0 + 8u * s; };                       // TMA -> converters (A chunk landed)
  auto a_empty = [&](int s) { return bar0 + 8u * (kStages + s); };          // converters -> TMA
  auto b_full = [&](int s) { return bar0 + 8u * (2 * kStages + s); };       // TMA of both CTAs -> MMA (leader)
  auto ready = [&](int s) { return bar0 + 8u * (3 * kStages + s); };        // converters of both CTAs -> MMA (leader)
  auto st_free = [&](int s) { return bar0 + 8u * (4 * kStages + s); };      // MMA commit -> TMEM A stage + B stage free
  auto acc_full = [&](int s) { return bar0 + 8u * (5 * kStages + s); };
  auto acc_empty = [&](int s) { return bar0 + 8u * (5 * kStages + kAccStages + s); };

  if (tid == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(a_full(s), 1);
      mbar_init(a_empty(s), kConvWarps);
      mbar_init(b_full(s), 1);  // leader only: armed by the leader's producer for the bytes of both CTAs
      mbar_init(ready(s), 2 * kConvWarps + 1);  // converter warps of both CTAs + the weight producer's expect_tx
      mbar_init(st_free(s), 1);
    }
    for (int s = 0; s < kAccStages; ++s) {
      mbar_init(acc_full(s), 1);
      mbar_init(acc_empty(s), 8);  // 4 epilogue warps x 2 CTAs
    }
    *reinterpret_cast<volatile uint32_t*>(smem + kOffFlag) = 0;
    fence_barrier_init();
  }
  int* pref = reinterpret_cast<int*>(smem + kOffPref);
  const uint32_t tmem_base = pair_setup(smem + kOffTmemPtr, warp, kWarpAlloc, kTmemCols, [&] {
    if (warp == kWarpTma && lane == 0) {
      tma_prefetch_desc(&P.a_map);
      tma_prefetch_desc(&P.whi_map);
      tma_prefetch_desc(&P.wlo_map);
    }
    for (int i = tid; i < 6 * kC + 6; i += kThreads)
      reinterpret_cast<float*>(smem + kOffWout)[i] = i < 6 * kC ? P.w_out[i] : P.b_out[i - 6 * kC];
    if (warp == kWarpTmaB) {  // exclusive prefix sum of the unit counts, one warp, 32 problems per step
      int carry = 0;
      for (int base = 0; base < P.num_problems; base += 32) {
        const int p = base + lane;
        int v = 0;
        if (p < P.num_problems) {
          const int cnt = P.roi_count ? min(__ldg(P.roi_count + p), P.roi_cap) : P.roi_cap;
          v = (max(cnt, 0) + 127) >> 7;
        }
        int inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int n = __shfl_up_sync(0xffffffffu, inc, o);
          if (lane >= o) inc += n;
        }
        if (p < P.num_problems) pref[p] = carry + inc - v;
        carry += __shfl_sync(0xffffffffu, inc, 31);
      }
      if (lane == 0) pref[P.num_problems] = carry;
    }
  });

  // Static schedule over the dense unit list: iteration i of pair k owns units 2*(i*num_pairs+k) and +1.
  const int total_units = pref[P.num_problems];
  auto slot_of = [&](int i, int r) { return 2 * (i * P.num_pairs + pair) + r; };
  auto in_range = [&](int i) { return slot_of(i, 0) < total_units; };

  if (warp == kWarpTma) {
    // ------------------------------------------------------------------ TMA producer, A operand (pooled rows)
    if (lane == 0) {
      uint32_t g = 0;
      for (int i = 0; in_range(i); ++i) {
        const Slot me = decode_unit(P, pref, slot_of(i, rank));
        const int tile0 = (me.p * P.tiles_per_problem + (me.r0 >> 7)) * kNumChunks;  // first A tile of this unit
        for (int kc = 0; kc < kNumChunks; ++kc, ++g) {
          const uint32_t s = ring_stage(g, kStages);
          mbar_wait(a_empty(s), ring_phase(g, kStages) ^ 1);
          mbar_arrive_expect_tx(a_full(s), kABytes);
          tma_load_2d(sbase + kOffA + s * kABytes, &P.a_map, a_full(s), 0, (tile0 + kc) * 128);
        }
      }
    }
  } else if (warp == kWarpTmaB) {
    // ------------------------------------------------------------------ TMA producer, B operand (weights); its own
    // thread so that a late st_free never delays the A stream and vice versa
    if (lane == 0) {
      // An mbarrier wait costs ~250 cycles even when its phase completed long ago, and the MMA warp's watcher is the
      // only thread that waits once per chunk: the weight bytes of both CTAs therefore complete the SAME barrier as
      // the converter warps' arrivals (ready), one wait per chunk instead of two.
      const uint32_t b_full_leader = map_to_cta(ready(0), 0);
      uint32_t g = 0;
      for (int i = 0; in_range(i); ++i) {
        for (int kc = 0; kc < kNumChunks; ++kc, ++g) {
          const uint32_t s = ring_stage(g, kStages);
          // each CTA loads its 64 rows; both CTAs' bytes complete on the LEADER's barrier
          mbar_wait(st_free(s), ring_phase(g, kStages) ^ 1);
          if (rank == 0) mbar_arrive_expect_tx(ready(s), 2 * kBBytes);
          tma_load_2d_2sm(sbase + kOffB + s * kBBytes, &P.whi_map, b_full_leader + 8u * s, kc * kChunk, rank * kBHalfRows);
          tma_load_2d_2sm(sbase + kOffB + s * kBBytes + kBPlaneBytes, &P.wlo_map, b_full_leader + 8u * s, kc * kChunk,
                          rank * kBHalfRows);
        }
      }
    }
  } else if (warp == kWarpMma) {
    if (rank == 0) {
      const uint32_t idesc = idesc_f16(256, 128);
      // The watcher thread (warp kWarpAlloc) publishes the number of chunks whose operands are in place; this warp only
      // polls that word.  The whole warp runs the loop converged and one elected lane issues, so that every tcgen05.mma
      // operand is a warp-uniform value in a uniform register (inside an `if (lane == 0)` region ptxas wraps each MMA in
      // a broadcast-and-retry loop whose latency exceeds the 64 cycles of the MMA itself).
      int n_iter = 0;
      for (int i = 0; in_range(i); ++i) ++n_iter;
      const uint32_t total = (uint32_t)n_iter * kNumChunks;
      uint32_t upto = 0;
      for (uint32_t g = 0; g < total; ++g) {
        flag_wait(sbase + kOffFlag, upto, g);
        tc_fence_after();
        const uint32_t s = ring_stage(g, kStages), as_ = ring_stage(g / kChunksPerPart, kAccStages);
        const bool first = (g % kChunksPerPart) == 0, last = (g % kChunksPerPart) == kChunksPerPart - 1;
        const uint32_t d = tmem_base + kColAcc + as_ * 128;
        const uint32_t a0 = tmem_base + kColA + s * kAStageCols;
        const uint64_t bhi = smem_desc_k_sw64(sbase + kOffB + s * kBBytes);
        const uint64_t blo = smem_desc_k_sw64(sbase + kOffB + s * kBBytes + kBPlaneBytes);
        if (elect_one()) {
#pragma unroll
          for (int ks = 0; ks < 2; ++ks) {  // K = 16 fp16 per MMA: 8 packed columns of A, 32 bytes of a B row
            const uint32_t ah = a0 + ks * 8, al = ah + 16;
            const uint64_t boff = (uint64_t)((ks * 32) >> 4);
            mma_f16_ts<2>(d, ah, bhi + boff, idesc, (!first || ks) ? 1u : 0u);
            mma_f16_ts<2>(d, al, bhi + boff, idesc, 1u);
            mma_f16_ts<2>(d, ah, blo + boff, idesc, 1u);
          }
          mma_commit_pair(st_free(s), 3);
          if (last) mma_commit_pair(acc_full(as_), 3);
        }
        __syncwarp();
      }
    }
  } else if (warp == kWarpAlloc) {
    // ------------------------------------------------------------------ barrier watcher of the MMA thread (leader)
    if (rank == 0 && lane == 0) {
      int n_iter = 0;
      for (int i = 0; in_range(i); ++i) ++n_iter;
      const uint32_t total = (uint32_t)n_iter * kNumChunks;
      for (uint32_t g = 0; g < total; ++g) {
        // A chunk of both CTAs is in tensor memory and the weight chunks have landed
        mbar_wait(ready(ring_stage(g, kStages)), ring_phase(g, kStages));
        if (g % kChunksPerPart == 0) {  // first chunk of a partial sum: its accumulator must have been drained
          const uint32_t gp = g / kChunksPerPart;
          mbar_wait(acc_empty(ring_stage(gp, kAccStages)), ring_phase(gp, kAccStages) ^ 1);
        }
        flag_publish(sbase + kOffFlag, g + 1);
      }
    }
  } else if (warp >= kWarpEpi0 && warp < kWarpEpi0 + 4) {
    // ------------------------------------------------------------------ epilogue: one ROI row per lane
    const int qd = warp & 3;
    const int m = qd * 32 + lane;
    const uint32_t acc_empty_leader = map_to_cta(acc_empty(0), 0);
    uint32_t gp = 0;
    const float w_inv = __ldg(P.w_inv);
    float rescale = xs_inv * w_inv;   // undoes the two power-of-two operand scales (exact)
    const uint32_t sum_s = sbase + kOffSum + (uint32_t)m * 16;  // + col_group * 2048: lanes = consecutive 16 B
    for (int i = 0; in_range(i); ++i) {
      const Slot me = decode_unit(P, pref, slot_of(i, rank));
      if (P.amax_stride) {
        image_scale(me.p / P.classes);
        rescale = xs_inv * w_inv;
      }
      // per-class folded bias of this unit -> shared memory (read back as broadcast)
      const int c = me.p % P.classes;
      const uint32_t bias_s = sbase + kOffBias;
      named_bar_sync(1, 128);  // previous unit's readers of the bias buffer are done
      if (warp == kWarpEpi0) {
        const float4 bv = ldg4(P.bias_cls + (size_t)c * kC + lane * 4);
        sts4s(bias_s + lane * 16, bv);
      }
      named_bar_sync(1, 128);
      float out[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
      for (int part = 0; part < kParts; ++part, ++gp) {
        const uint32_t as_ = ring_stage(gp, kAccStages);
        mbar_wait(acc_full(as_), ring_phase(gp, kAccStages));
        tc_fence_after();
        const uint32_t trow = tmem_base + ((uint32_t)(qd * 32) << 16) + kColAcc + as_ * 128;
#pragma unroll 1
        for (int j = 0; j < 4; ++j) {
          uint32_t v[32];
          tmem_ld32(trow + j * 32, v);
          tmem_wait_ld();
          if (j == 3) acc_release(acc_empty_leader + 8u * as_, lane);   // accumulator fully read
#pragma unroll
          for (int c4 = 0; c4 < 8; ++c4) {
            const uint32_t sa = sum_s + (uint32_t)(j * 8 + c4) * 2048;
            float4 x = make_float4(__uint_as_float(v[c4 * 4 + 0]), __uint_as_float(v[c4 * 4 + 1]),
                                   __uint_as_float(v[c4 * 4 + 2]), __uint_as_float(v[c4 * 4 + 3]));
            if (part > 0) {
              const float4 r = lds4s(sa);
              x.x += r.x; x.y += r.y; x.z += r.z; x.w += r.w;
            }
            if (part < kParts - 1) {
              sts4s(sa, x);
            } else {
              const float4 bb = lds4s(bias_s + (j * 32 + c4 * 4) * 4);
              const float f0 = fmaxf(fmaf(x.x, rescale, bb.x), 0.f), f1 = fmaxf(fmaf(x.y, rescale, bb.y), 0.f);
              const float f2 = fmaxf(fmaf(x.z, rescale, bb.z), 0.f), f3 = fmaxf(fmaf(x.w, rescale, bb.w), 0.f);
#pragma unroll
              for (int o = 0; o < 6; ++o) {
                const float4 w = lds4s(sbase + kOffWout + (o * kC + j * 32 + c4 * 4) * 4);
                out[o] = fmaf(f3, w.w, fmaf(f2, w.z, fmaf(f1, w.y, fmaf(f0, w.x, out[o]))));
              }
            }
          }
        }
      }
      if (m < me.rows) {
        const size_t row = (size_t)me.p * P.roi_cap + me.r0 + m;
        const float* bo = reinterpret_cast<const float*>(smem + kOffWout) + 6 * kC;
        const float l0 = out[0] + bo[0], l1 = out[1] + bo[1];
        const float d0 = out[2] + bo[2], d1 = out[3] + bo[3], d2 = out[4] + bo[4], d3 = out[5] + bo[5];
        if (P.logits) {
          P.logits[row * 2] = l0;
          P.logits[row * 2 + 1] = l1;
        }
        if (P.deltas) *reinterpret_cast<float4*>(P.deltas + row * 4) = make_float4(d0, d1, d2, d3);
        // softmax over (fg, bg) -> fg probability (custom_fast_rcnn.py:169)
        const float mx = fmaxf(l0, l1);
        const float e0 = expf(l0 - mx), e1 = expf(l1 - mx);
        P.det_scores[row] = e0 / (e0 + e1);
        // apply_deltas (box_regression.py:87-115); clipping happens in fod_final_detect
        const float4 bx = *reinterpret_cast<const float4*>(P.rois + row * 4);
        const float w = bx.z - bx.x, h = bx.w - bx.y;
        const float cx = bx.x + 0.5f * w, cy = bx.y + 0.5f * h;
        const float dx = d0 / P.reg_w[0], dy = d1 / P.reg_w[1];
        const float dw = fminf(d2 / P.reg_w[2], kScaleClamp), dh = fminf(d3 / P.reg_w[3], kScaleClamp);
        const float pcx = __fadd_rn(__fmul_rn(dx, w), cx), pcy = __fadd_rn(__fmul_rn(dy, h), cy);
        const float pw = __fmul_rn(expf(dw), w), ph = __fmul_rn(expf(dh), h);
        const float x1 = __fsub_rn(pcx, __fmul_rn(0.5f, pw)), y1 = __fsub_rn(pcy, __fmul_rn(0.5f, ph));
        const float x2 = __fadd_rn(pcx, __fmul_rn(0.5f, pw)), y2 = __fadd_rn(pcy, __fmul_rn(0.5f, ph));
        *reinterpret_cast<float4*>(P.det_boxes + row * 4) = make_float4(x1, y1, x2, y2);
      }
    }
  } else if (warp >= kWarpConv0) {
    // ------------------------------------------------------------------ converters: A chunk smem -> tf32 hi/lo in TMEM
    const int wc = warp - kWarpConv0;
    const int qd = wc & 3, half = wc >> 2;
    const int m = qd * 32 + lane;
    const uint32_t ready_leader = map_to_cta(ready(0), 0);
    const uint32_t trow = tmem_base + ((uint32_t)(qd * 32) << 16) + kColA + half * 8;
    const uint32_t arow = (uint32_t)(m * 128);
    uint32_t g = 0;
    for (int i = 0; in_range(i); ++i) {
      if (P.amax_stride) image_scale(decode_unit(P, pref, slot_of(i, rank)).p / P.classes);
      for (int kc = 0; kc < kNumChunks; ++kc, ++g) {
        const uint32_t s = ring_stage(g, kStages), ph = ring_phase(g, kStages);
        mbar_wait(a_full(s), ph);
        const uint32_t at = sbase + kOffA + s * kABytes + arow;
        float4 x[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) x[j] = lds4s(at + ((((half * 4 + j) ^ (m & 7)) & 7) << 4));
        uint32_t hi[8], lo[8];   // this warp's 16 K values of the chunk as packed fp16 pairs
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          split_f16x2(x[j].x * xs, x[j].y * xs, hi[2 * j + 0], lo[2 * j + 0]);
          split_f16x2(x[j].z * xs, x[j].w * xs, hi[2 * j + 1], lo[2 * j + 1]);
        }
        mbar_wait(st_free(s), ph ^ 1);  // the MMAs that read this TMEM stage have completed
        tc_fence_after();
        tmem_st8(trow + s * kAStageCols, hi);
        tmem_st8(trow + s * kAStageCols + 16, lo);
        tmem_wait_st();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          mbar_arrive(a_empty(s));
          mbar_arrive_remote(ready_leader + 8u * s);
        }
      }
    }
  }
  pair_teardown(warp, kWarpAlloc, tmem_base, kTmemCols);
}

}  // namespace rtc
}  // namespace fod

using namespace fod;

extern "C" int fod_relation_head(const float* pooled, const float* x_amax, int n_amax, int amax_per_image,
                                 const float* w_fold_packed,
                                 const float* bias_cls, const float* w_out, const float* b_out, const float* rois,
                                 const int32_t* roi_count, int num_problems, int problems_per_image, int roi_cap,
                                 const float* reg_weights, float* det_boxes, float* det_scores, float* logits, float* deltas,
                                 fod_stream_t stream) {
  FOD_REQUIRE(pooled && x_amax && w_fold_packed && bias_cls && w_out && b_out && rois && reg_weights && det_boxes && det_scores,
              "fod_relation_head: null pointer");
  FOD_REQUIRE(n_amax >= 1 && n_amax <= 8, "fod_relation_head: 1..8 operand bounds");
  FOD_REQUIRE(num_problems >= 0 && problems_per_image > 0 && roi_cap > 0, "fod_relation_head: bad sizes");
  FOD_REQUIRE(num_problems % problems_per_image == 0, "fod_relation_head: num_problems not a multiple of classes");
  FOD_REQUIRE(num_problems <= rtc::kMaxProblems, "fod_relation_head: more than %d problems per call", rtc::kMaxProblems);
  FOD_REQUIRE((((uintptr_t)pooled | (uintptr_t)w_fold_packed | (uintptr_t)bias_cls | (uintptr_t)rois | (uintptr_t)det_boxes |
                (uintptr_t)deltas) & 15) == 0, "fod_relation_head: pointers must be 16-byte aligned");
  if (num_problems == 0) return FOD_OK;
  rtc::Params prm;
  memset(&prm, 0, sizeof(prm));
  const long units = (long)num_problems * ((roi_cap + 127) / 128);
  FOD_REQUIRE(units * rtc::kNumChunks * 128 < (1L << 31), "fod_relation_head: pooled buffer too large for one call");
  int rc = make_matrix_map(&prm.a_map, pooled, units * rtc::kNumChunks * 128, rtc::kChunk, rtc::kChunk, 128);
  if (rc != FOD_OK) return rc;
  // packed weights = fod_conv2d_pack_weights of the folded matrix seen as a 1x1 convolution [128][8192][1][1]:
  // fp16 hi plane [128][8192], lo plane, then {1/scale, scale, max|w|, 0}
  const __half* whi = reinterpret_cast<const __half*>(w_fold_packed);
  rc = make_matrix_map_f16(&prm.whi_map, whi, kC, rtc::kK, rtc::kChunk, rtc::kBHalfRows);
  if (rc != FOD_OK) return rc;
  rc = make_matrix_map_f16(&prm.wlo_map, whi + (size_t)kC * rtc::kK, kC, rtc::kK, rtc::kChunk, rtc::kBHalfRows);
  if (rc != FOD_OK) return rc;
  prm.w_inv = w_fold_packed + (size_t)kC * rtc::kK;   // two fp16 planes = kC * kK floats
  prm.x_amax = x_amax;
  prm.n_amax = n_amax;
  prm.amax_stride = amax_per_image ? num_problems / problems_per_image : 0;
  prm.bias_cls = bias_cls;
  prm.rois = rois;
  prm.roi_count = roi_count;
  prm.det_boxes = det_boxes;
  prm.det_scores = det_scores;
  prm.logits = logits;
  prm.deltas = deltas;
  prm.w_out = w_out;
  prm.b_out = b_out;
  for (int i = 0; i < 4; ++i) prm.reg_w[i] = reg_weights[i];
  prm.num_problems = num_problems;
  prm.classes = problems_per_image;
  prm.roi_cap = roi_cap;
  prm.tiles_per_problem = (roi_cap + 127) / 128;
  const int total_slots = num_problems * prm.tiles_per_problem;   // the most units the ROI counts can make
  rc = pair_count((total_slots + 1) / 2, &prm.num_pairs);
  if (rc != FOD_OK) return rc;
  void* args[] = {&prm};
  return launch_clusters((const void*)rtc::relation_tc_kernel, args, prm.num_pairs, 2, rtc::kThreads, rtc::kSmemAlloc,
                         stream, "fod_relation_head");
}
