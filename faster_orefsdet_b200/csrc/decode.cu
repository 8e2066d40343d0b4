// D1+D2+D3: heat-map sigmoid -> candidate threshold -> per-level radix-select top-k ->
// box decode -> dense level-major candidate list.  The keys of a level live in shared memory of
// the CTA that selects it; its offset into the level-major list is the number of survivors of the
// lower levels, which it recounts itself (a read of 4 bytes per pixel, no cross-CTA dependency).
// Two CTAs per problem: one for level 0 (three quarters of the pixels of a stride-8/16/32 pyramid)
// and one that walks the remaining levels, so a batch of 64 problems is ONE wave of 128 CTAs.
// Tap mode (the folded 3x3 output convolution) first forms the keys of every pixel in a wide
// kernel over all SMs - nine L1-friendly reads per pixel - and the selecting CTAs read those.
//
// Selection: key = fp32 bits of p (positive floats order like their bit patterns),
// 0 for non-candidates.  An MSB-first 8-bit radix select (warp-aggregated shared
// atomics into per-warp histograms) finds the k-th largest key T and how many
// elements equal to T are needed; one ordered block scan then emits the survivors
// in ascending location order: all keys > T plus the first `need` keys == T.
#include "common.cuh"

namespace fod {

constexpr int kDecThreads = 1024;
constexpr int kDecWarps = kDecThreads / 32;
constexpr int kMaxLevelPixels = 40960;  // 160 KB of keys

struct DecodeParams {
  const float* hm[FOD_MAX_LEVELS];
  const float* reg[FOD_MAX_LEVELS];
  int H[FOD_MAX_LEVELS], W[FOD_MAX_LEVELS], stride[FOD_MAX_LEVELS];
  int hm_ps[FOD_MAX_LEVELS], reg_ps[FOD_MAX_LEVELS];   // pixel strides in floats (1 / 4 = dense)
  // tap mode (fod_decode_topk_taps): hm[l] points at G[P][H][W][tap_ps], the products of the 3x3 output convolution's
  // taps (tap = ky*3 + kx) with the tower output at pixel p: column tap = heat-map, column 12 + tap*4 + j = regression
  // output j (l, t, r, b).  The convolution at pixel (y, x) is bias + sum over taps of G[(y+ky-1, x+kx-1)][column].
  // The nine heat-map products of a pixel sit in its first 36 bytes, and each of them is wanted by a different
  // neighbouring output pixel - the L1 serves that reuse, L2 sees two sectors per pixel instead of nine; the four
  // regression products of one tap are one aligned 16-byte read, nine of them per emitted candidate.
  int taps;            // 0: hm / reg maps, 9: tap products
  const uint32_t* keys;   // tap mode: [P][key_stride] keys of all levels (decode_keys_kernel), level l at key_off[l]
  int key_off[FOD_MAX_LEVELS], key_stride;
  float bias[5];       // agn_hm.bias, bbox_pred.bias (tap mode)
  int num_levels;
  int hm_is_logit, reg_channels_last, reg_activate;
  float reg_scale[FOD_MAX_LEVELS];   // reg_activate: reg = relu(reg_scale[l] * raw) (Scale + ReLU of CenterNetHead)
  float thresh;
  int pre_topk, cand_cap;
};

// heat-map logit of the 3x3 output convolution at pixel (y, x) from the per-tap products (zero padding)
__device__ __forceinline__ float tap_sum(const float* __restrict__ G, int ps, int H, int W, int y, int x, float bias) {
  float acc = 0.f;
#pragma unroll
  for (int ky = 0; ky < 3; ++ky) {
    const int yy = y + ky - 1;
    if (yy < 0 || yy >= H) continue;
#pragma unroll
    for (int kx = 0; kx < 3; ++kx) {
      const int xx = x + kx - 1;
      if (xx < 0 || xx >= W) continue;
      acc += __ldg(G + ((size_t)yy * W + xx) * ps + (ky * 3 + kx));
    }
  }
  return acc + bias;
}
// the four regression outputs at pixel (y, x): the same sums (same order per output), four at a time
__device__ __forceinline__ float4 tap_sum_reg(const float* __restrict__ G, int ps, int H, int W, int y, int x, const float* bias) {
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int ky = 0; ky < 3; ++ky) {
    const int yy = y + ky - 1;
    if (yy < 0 || yy >= H) continue;
#pragma unroll
    for (int kx = 0; kx < 3; ++kx) {
      const int xx = x + kx - 1;
      if (xx < 0 || xx >= W) continue;
      const float4 v = ldg4(G + ((size_t)yy * W + xx) * ps + 12 + (ky * 3 + kx) * 4);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
  }
  return make_float4(acc.x + bias[1], acc.y + bias[2], acc.z + bias[3], acc.w + bias[4]);
}

// tap mode, step 1: the key of every pixel of every level (fp32 bits of sigmoid(heat-map) above the threshold, else 0);
// consecutive threads take consecutive pixels, so the nine products a pixel contributes are read by neighbouring
// threads of the same CTA and come out of the L1
__global__ void __launch_bounds__(256)
decode_keys_kernel(DecodeParams prm, uint32_t* __restrict__ keys_out) {
  const int idx = blockIdx.x * 256 + threadIdx.x, p = blockIdx.y;
  if (idx >= prm.key_stride) return;
  int l = 0;
  while (l + 1 < prm.num_levels && idx >= prm.key_off[l + 1]) ++l;
  const int i = idx - prm.key_off[l], H = prm.H[l], W = prm.W[l], hps = prm.hm_ps[l];
  const float v = tap_sum(prm.hm[l] + (size_t)p * H * W * hps, hps, H, W, i / W, i % W, prm.bias[0]);
  const float pr = 1.0f / (1.0f + expf(-v));
  keys_out[(size_t)p * prm.key_stride + idx] = (pr > prm.thresh) ? __float_as_uint(pr) : 0u;
}

__global__ void __launch_bounds__(kDecThreads, 1)
decode_topk_kernel(DecodeParams prm, float* __restrict__ boxes, float* __restrict__ scores, int64_t* __restrict__ loc,
                   int32_t* __restrict__ level_count, int32_t* __restrict__ cand_count, uint32_t* __restrict__ status) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint32_t* keys = reinterpret_cast<uint32_t*>(smem_raw);
  __shared__ int hist[kDecWarps][256];
  __shared__ int warp_sums[kDecWarps + 1];
  __shared__ int sh[2];
  const int roles = min(prm.num_levels, 2);
  const int p = blockIdx.x / roles, role = blockIdx.x - p * roles;
  const int l_begin = role == 0 ? 0 : 1, l_end = (role == 0 && roles == 2) ? 1 : prm.num_levels;
  const int tid = threadIdx.x;
  auto block_sum = [&](int local) { return block_reduce(local, warp_sums, [](int a, int b) { return a + b; }); };
  // key of pixel i of level ll: fp32 bits of the probability if it passes the threshold, else 0
  auto key_of = [&](int ll, int i) -> uint32_t {
    if (prm.taps) return __ldg(prm.keys + (size_t)p * prm.key_stride + prm.key_off[ll] + i);
    const float v = __ldg(prm.hm[ll] + ((size_t)p * prm.H[ll] * prm.W[ll] + i) * prm.hm_ps[ll]);
    const float pr = prm.hm_is_logit ? 1.0f / (1.0f + expf(-v)) : v;
    return (pr > prm.thresh) ? __float_as_uint(pr) : 0u;
  };
  // survivors of the levels below this CTA's first one (the predicate their own CTA evaluates)
  int out_base = 0;
  for (int ll = 0; ll < l_begin; ++ll) {
    const int nn = prm.H[ll] * prm.W[ll];
    int local = 0;
    for (int i = tid; i < nn; i += kDecThreads) local += (key_of(ll, i) != 0u);
    out_base += min(block_sum(local), prm.pre_topk);
  }
  for (int l = l_begin; l < l_end; ++l) {
    const int H = prm.H[l], W = prm.W[l], n = H * W, stride = prm.stride[l];
    const int hps = prm.hm_ps[l], rps = prm.reg_ps[l];
    const float* hm = prm.hm[l] + (size_t)p * n * hps;
    // ---- pass 0: keys + candidate count
    int local = 0;
    for (int i = tid; i < n; i += kDecThreads) {
      const uint32_t k = key_of(l, i);
      keys[i] = k;
      local += (k != 0u);
    }
    const int cnt = block_sum(local);
    uint32_t T = 0u;   // select keys > T plus the first `need` keys == T
    int need = 0;
    if (cnt > prm.pre_topk) T = radix_select([&](int i) { return keys[i]; }, n, prm.pre_topk, hist, sh, need);
    // ---- ordered emission
    const int nsel = min(cnt, prm.pre_topk);
    if (out_base + nsel > prm.cand_cap && tid == 0) atomicOr(status, FOD_STATUS_CAND_OVERFLOW);
    const float half = (float)(stride / 2);
    const float fstride = (float)stride;
    int gt_before = 0, eq_before = 0;
    for (int i0 = 0; i0 < n; i0 += kDecThreads) {
      int i = i0 + tid;
      uint32_t k = (i < n) ? keys[i] : 0u;
      int is_gt = (k > T) ? 1 : 0;
      int is_eq = (T != 0u && k == T) ? 1 : 0;
      // both counts in one scan: a level has fewer than 2^16 pixels (kMaxLevelPixels)
      int tot;
      const int excl = block_exclusive_scan(is_gt | (is_eq << 16), warp_sums, tot);
      int gt_pos = gt_before + (excl & 0xffff);
      int eq_pos = eq_before + (excl >> 16);
      bool sel = is_gt || (is_eq && eq_pos < need);
      if (sel) {
        int o = out_base + gt_pos + min(eq_pos, need);
        if (o < prm.cand_cap) {
          int y = i / W, xx = i - y * W;
          float gx = __fadd_rn((float)(xx * stride), half);
          float gy = __fadd_rn((float)(y * stride), half);
          float r0, r1, r2, r3;
          if (prm.taps) {
            const float4 r = tap_sum_reg(hm, hps, H, W, y, xx, prm.bias);
            r0 = r.x; r1 = r.y; r2 = r.z; r3 = r.w;
          } else if (prm.reg_channels_last) {
            const float* rp = prm.reg[l] + ((size_t)p * n + i) * rps;
            if ((reinterpret_cast<uintptr_t>(rp) & 15) == 0) {
              float4 r = ldg4(rp);
              r0 = r.x; r1 = r.y; r2 = r.z; r3 = r.w;
            } else {       // a channel slice of a wider NHWC buffer (the fused agn_hm | bbox_pred convolution output)
              r0 = __ldg(rp); r1 = __ldg(rp + 1); r2 = __ldg(rp + 2); r3 = __ldg(rp + 3);
            }
          } else {
            const float* rp = prm.reg[l] + (size_t)p * 4 * n + i;
            r0 = __ldg(rp); r1 = __ldg(rp + n); r2 = __ldg(rp + 2 * (size_t)n); r3 = __ldg(rp + 3 * (size_t)n);
          }
          if (prm.reg_activate) {   // F.relu(scale * x), centernet_head.py:157-160 (one rounded product, then max)
            const float sc = prm.reg_scale[l];
            r0 = fmaxf(__fmul_rn(r0, sc), 0.f);
            r1 = fmaxf(__fmul_rn(r1, sc), 0.f);
            r2 = fmaxf(__fmul_rn(r2, sc), 0.f);
            r3 = fmaxf(__fmul_rn(r3, sc), 0.f);
          }
          float x1 = __fsub_rn(gx, __fmul_rn(r0, fstride));
          float y1 = __fsub_rn(gy, __fmul_rn(r1, fstride));
          float x2 = __fadd_rn(gx, __fmul_rn(r2, fstride));
          float y2 = __fadd_rn(gy, __fmul_rn(r3, fstride));
          x2 = fmaxf(x2, __fadd_rn(x1, 0.01f));
          y2 = fmaxf(y2, __fadd_rn(y1, 0.01f));
          size_t ob = (size_t)p * prm.cand_cap + o;
          *reinterpret_cast<float4*>(boxes + ob * 4) = make_float4(x1, y1, x2, y2);
          scores[ob] = __fsqrt_rn(__uint_as_float(k));
          loc[ob] = i;
        }
      }
      gt_before += tot & 0xffff;
      eq_before += tot >> 16;
    }
    if (tid == 0) level_count[p * prm.num_levels + l] = nsel;
    if (tid == 0 && l == prm.num_levels - 1) cand_count[p] = min(out_base + nsel, prm.cand_cap);
    out_base += nsel;
    __syncthreads();   // keys / histograms are reused by the next level
  }
}

}  // namespace fod

using namespace fod;

static int decode_launch(const float* const* hm, const float* const* reg, const fod_level_t* levels, int num_levels,
                         int num_problems, int hm_is_logit, int reg_channels_last, const int* hm_pixel_stride,
                         const int* reg_pixel_stride, const float* reg_scale, int taps, const float* bias5,
                         float score_thresh, int pre_topk, int cand_cap, float* boxes, float* scores, int64_t* loc,
                         int32_t* level_count, int32_t* cand_count, uint32_t* status, void* workspace, fod_stream_t stream) {
  FOD_REQUIRE(hm && levels && boxes && scores && loc && level_count && cand_count && status && (taps || reg) &&
                  (!taps || workspace),
              "fod_decode_topk: null pointer");
  FOD_REQUIRE(num_levels >= 1 && num_levels <= FOD_MAX_LEVELS, "fod_decode_topk: num_levels %d out of range", num_levels);
  FOD_REQUIRE(num_problems >= 0 && pre_topk > 0 && cand_cap >= num_levels * pre_topk,
              "fod_decode_topk: cand_cap %d < num_levels*pre_topk %d", cand_cap, num_levels * pre_topk);
  FOD_REQUIRE(score_thresh >= 0.f, "fod_decode_topk: score_thresh must be >= 0");
  if (num_problems == 0) return FOD_OK;
  DecodeParams prm;
  int maxpix = 0;
  for (int l = 0; l < num_levels; ++l) {
    FOD_REQUIRE(hm[l] && (taps || reg[l]), "fod_decode_topk: null level pointer");
    FOD_REQUIRE(levels[l].height > 0 && levels[l].width > 0 && levels[l].stride > 0, "fod_decode_topk: bad level %d", l);
    prm.hm[l] = hm[l];
    prm.reg[l] = taps ? nullptr : reg[l];
    prm.H[l] = levels[l].height;
    prm.W[l] = levels[l].width;
    prm.stride[l] = levels[l].stride;
    prm.hm_ps[l] = hm_pixel_stride ? hm_pixel_stride[l] : (taps ? 48 : 1);
    prm.reg_ps[l] = reg_pixel_stride ? reg_pixel_stride[l] : 4;
    FOD_REQUIRE(prm.hm_ps[l] >= (taps ? 48 : 1) && (!taps || prm.hm_ps[l] % 4 == 0) && prm.reg_ps[l] >= 4, "fod_decode_topk: bad pixel stride at level %d", l);
    FOD_REQUIRE(!reg_pixel_stride || reg_channels_last, "fod_decode_topk: reg_pixel_stride needs the channels-last layout");
    int px = levels[l].height * levels[l].width;
    if (px > maxpix) maxpix = px;
  }
  if (maxpix > kMaxLevelPixels) {
    set_error("fod_decode_topk: level with %d pixels exceeds the in-smem limit %d", maxpix, kMaxLevelPixels);
    return FOD_ERR_CAPACITY;
  }
  prm.num_levels = num_levels;
  prm.hm_is_logit = hm_is_logit;
  prm.reg_channels_last = reg_channels_last;
  prm.reg_activate = reg_scale ? 1 : 0;
  for (int l = 0; l < FOD_MAX_LEVELS; ++l) prm.reg_scale[l] = (reg_scale && l < num_levels) ? reg_scale[l] : 1.f;
  prm.taps = taps;
  prm.keys = static_cast<const uint32_t*>(workspace);
  prm.key_stride = 0;
  for (int l = 0; l < FOD_MAX_LEVELS; ++l) {
    prm.key_off[l] = prm.key_stride;
    if (l < num_levels) prm.key_stride += levels[l].height * levels[l].width;
  }
  for (int i = 0; i < 5; ++i) prm.bias[i] = bias5 ? bias5[i] : 0.f;
  prm.thresh = score_thresh;
  prm.pre_topk = pre_topk;
  prm.cand_cap = cand_cap;
  FOD_REQUIRE((long)num_problems * num_levels < (1L << 30), "fod_decode_topk: too many problems");
  size_t smem = (size_t)maxpix * sizeof(uint32_t);
  FOD_CUDA_CALL(cudaFuncSetAttribute(decode_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  if (taps) {
    decode_keys_kernel<<<dim3((unsigned)((prm.key_stride + 255) / 256), (unsigned)num_problems), 256, 0, as_stream(stream)>>>(
        prm, static_cast<uint32_t*>(workspace));
    FOD_CUDA_LAUNCH_CHECK("fod_decode_topk_taps (keys)");
  }
  const int roles = num_levels < 2 ? num_levels : 2;
  decode_topk_kernel<<<num_problems * roles, kDecThreads, smem, as_stream(stream)>>>(prm, boxes, scores, loc, level_count,
                                                                                     cand_count, status);
  FOD_CUDA_LAUNCH_CHECK("fod_decode_topk");
  return FOD_OK;
}

extern "C" int fod_decode_topk(const float* const* hm, const float* const* reg, const fod_level_t* levels,
                               int num_levels, int num_problems, int hm_is_logit, int reg_channels_last,
                               const int* hm_pixel_stride, const int* reg_pixel_stride, const float* reg_scale,
                               float score_thresh, int pre_topk, int cand_cap, float* boxes, float* scores,
                               int64_t* loc, int32_t* level_count, int32_t* cand_count, uint32_t* status,
                               fod_stream_t stream) {
  return decode_launch(hm, reg, levels, num_levels, num_problems, hm_is_logit, reg_channels_last, hm_pixel_stride,
                       reg_pixel_stride, reg_scale, 0, nullptr, score_thresh, pre_topk, cand_cap, boxes, scores, loc,
                       level_count, cand_count, status, nullptr, stream);
}

extern "C" int fod_decode_topk_taps(const float* const* taps, const int* tap_pixel_stride, const float* bias5,
                                    const fod_level_t* levels, int num_levels, int num_problems, const float* reg_scale,
                                    float score_thresh, int pre_topk, int cand_cap, float* boxes, float* scores,
                                    int64_t* loc, int32_t* level_count, int32_t* cand_count, uint32_t* status,
                                    void* workspace, fod_stream_t stream) {
  FOD_REQUIRE(bias5, "fod_decode_topk_taps: null bias");
  return decode_launch(taps, nullptr, levels, num_levels, num_problems, 1, 1, tap_pixel_stride, nullptr, reg_scale, 9, bias5,
                       score_thresh, pre_topk, cand_cap, boxes, scores, loc, level_count, cand_count, status, workspace, stream);
}

extern "C" size_t fod_decode_topk_taps_workspace_bytes(const fod_level_t* levels, int num_levels, int num_problems) {
  size_t px = 0;
  for (int l = 0; levels && l < num_levels && l < FOD_MAX_LEVELS; ++l) px += (size_t)levels[l].height * levels[l].width;
  return px * (size_t)(num_problems > 0 ? num_problems : 0) * sizeof(uint32_t);
}
