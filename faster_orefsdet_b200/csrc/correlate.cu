// Q1 (support taps); Q2+Q3 (correlation + 1x1 relation conv) live in correlate_tc.cu.
#include "common.cuh"

namespace fod {

// ------------------------------------------------------------------------------------------------
// Q1: adaptive average pools (1,1), (1,3), (3,1) of the prototype.
// PyTorch adaptive pooling bins: start = floor(i*n/out), end = ceil((i+1)*n/out).
// ------------------------------------------------------------------------------------------------
__global__ void support_taps_kernel(const float* __restrict__ proto, int h, int w, float* __restrict__ taps) {
  const int c = blockIdx.x;          // class
  const int ch = threadIdx.x;        // channel 0..127
  const float* P = proto + (size_t)c * h * w * kC;
  float col[3] = {0.f, 0.f, 0.f}, row[3] = {0.f, 0.f, 0.f}, all = 0.f;
  int cs[3], ce[3], rs[3], re[3];
  for (int i = 0; i < 3; ++i) {
    cs[i] = (i * w) / 3;
    ce[i] = ((i + 1) * w + 2) / 3;
    rs[i] = (i * h) / 3;
    re[i] = ((i + 1) * h + 2) / 3;
  }
  for (int y = 0; y < h; ++y)
    for (int x = 0; x < w; ++x) {
      float v = P[((size_t)y * w + x) * kC + ch];
      all += v;
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        if (x >= cs[i] && x < ce[i]) col[i] += v;
        if (y >= rs[i] && y < re[i]) row[i] += v;
      }
    }
  float* T = taps + (size_t)c * 7 * kC;
  T[0 * kC + ch] = all / (float)(h * w);
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    T[(1 + i) * kC + ch] = col[i] / (float)(h * (ce[i] - cs[i]));
    T[(4 + i) * kC + ch] = row[i] / (float)(w * (re[i] - rs[i]));
  }
}

}  // namespace fod

using namespace fod;

extern "C" int fod_support_taps(const float* proto, int num_classes, int h, int w, float* taps, fod_stream_t stream) {
  FOD_REQUIRE(proto && taps, "fod_support_taps: null pointer");
  FOD_REQUIRE(num_classes >= 0 && h > 0 && w > 0, "fod_support_taps: bad sizes");
  if (num_classes == 0) return FOD_OK;
  support_taps_kernel<<<num_classes, kC, 0, as_stream(stream)>>>(proto, h, w, taps);
  FOD_CUDA_LAUNCH_CHECK("fod_support_taps");
  return FOD_OK;
}
