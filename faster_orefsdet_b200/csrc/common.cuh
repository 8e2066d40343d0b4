// Shared helpers for the fod_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/fod_b200.h"

namespace fod {

constexpr int kC = FOD_CHANNELS;  // 128 channels everywhere on this path

void set_error(const char* fmt, ...);

#define FOD_REQUIRE(cond, ...)      \
  do {                              \
    if (!(cond)) {                  \
      fod::set_error(__VA_ARGS__);  \
      return FOD_ERR_BAD_ARG;       \
    }                               \
  } while (0)

#define FOD_CUDA_LAUNCH_CHECK(name)                                                   \
  do {                                                                                \
    cudaError_t e__ = cudaGetLastError();                                             \
    if (e__ != cudaSuccess) {                                                         \
      fod::set_error("%s: launch failed: %s", name, cudaGetErrorString(e__));         \
      return FOD_ERR_CUDA;                                                            \
    }                                                                                 \
  } while (0)

#define FOD_CUDA_CALL(expr)                                                           \
  do {                                                                                \
    cudaError_t e__ = (expr);                                                         \
    if (e__ != cudaSuccess) {                                                         \
      fod::set_error("%s failed: %s", #expr, cudaGetErrorString(e__));                \
      return FOD_ERR_CUDA;                                                            \
    }                                                                                 \
  } while (0)

inline cudaStream_t as_stream(fod_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

// Order-preserving map float -> uint32 (ascending float == ascending uint).
__device__ __forceinline__ uint32_t float_to_ordered(float f) {
  uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// IoU test with the exact arithmetic of torchvision's CPU nms kernel
// (torchvision/csrc/ops/cpu/nms_kernel.cpp): every operation a separately rounded
// fp32 op (no FMA contraction), the ratio compared against the double threshold.
// thr_f is the smallest float whose double value exceeds the double threshold, so
// `ovr >= thr_f`  <=>  `(double)ovr > thr`.
__device__ __forceinline__ bool iou_exceeds(const float4 a, float area_a, const float4 b, float area_b, float thr_f) {
  float xx1 = fmaxf(a.x, b.x), yy1 = fmaxf(a.y, b.y);
  float xx2 = fminf(a.z, b.z), yy2 = fminf(a.w, b.w);
  float w = fmaxf(0.f, __fsub_rn(xx2, xx1));
  float h = fmaxf(0.f, __fsub_rn(yy2, yy1));
  float inter = __fmul_rn(w, h);
  float uni = __fsub_rn(__fadd_rn(area_a, area_b), inter);
  // Same decision as the exact quotient below, without the division in the clear cases: for uni > 0 and thr > 0
  // the rounded quotient is >= thr iff inter/uni is, up to half an ulp; a 1e-6 relative margin around thr*uni is
  // hundreds of ulps wide, everything inside it takes the exact path.  (Most pairs do not overlap at all.)
  if (uni > 0.f && thr_f > 0.f) {
    const float t = __fmul_rn(thr_f, uni);
    if (inter > __fmul_rn(t, 1.000001f)) return true;
    if (inter < __fmul_rn(t, 0.999999f)) return false;
  }
  float ovr = __fdiv_rn(inter, uni);
  return ovr >= thr_f;  // false for NaN, like `ovr > thr`
}

__device__ __forceinline__ float box_area(const float4 b) { return __fmul_rn(__fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y)); }

float iou_threshold_as_float(double thr);

// Block primitives of a 1024-thread CTA (32 warps); every thread of the CTA calls them.  Each ends with a barrier, after
// which `sh` may be used again.
//
// op-reduction of one value per thread (op = a + b or fmaxf(a, b)); the result in every thread.  sh: __shared__ T[32]
template <class T, class Op>
__device__ inline T block_reduce(T v, T* sh, Op op) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = op(v, __shfl_xor_sync(0xffffffffu, v, o));
  if (lane == 0) sh[warp] = v;
  __syncthreads();
  if (warp == 0) {
    v = sh[lane];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = op(v, __shfl_xor_sync(0xffffffffu, v, o));
    if (lane == 0) sh[0] = v;
  }
  __syncthreads();
  const T r = sh[0];
  __syncthreads();
  return r;
}

// Exclusive prefix sum of one int per thread in thread order; `total` gets the sum over the CTA.  sh: __shared__ int[33]
__device__ inline int block_exclusive_scan(int v, int* sh, int& total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) sh[warp] = x;
  __syncthreads();
  if (warp == 0) {
    const int w = sh[lane];
    int xs = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, xs, o);
      if (lane >= o) xs += y;
    }
    sh[lane] = xs - w;
    if (lane == 31) sh[32] = xs;
  }
  __syncthreads();
  const int res = sh[warp] + x - v;
  total = sh[32];
  __syncthreads();
  return res;
}

// Radix select of a 1024-thread CTA: the k-th largest of the n keys key_at(0..n-1) (k <= n) as T, and in `need` how many
// keys equal to T belong to the k largest.  MSB-first, 8 bits per pass; warp-aggregated shared atomics into per-warp
// histograms hist[32][256]; sh: __shared__ int[2].  Every thread of the CTA calls it and gets the same (T, need).
template <class KeyAt>
__device__ inline uint32_t radix_select(KeyAt key_at, int n, int k, int (*hist)[256], int* sh, int& need) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int kWarps = 32;
  uint32_t prefix = 0u, mask = 0u;
  int remaining = k;
  for (int shift = 24; shift >= 0; shift -= 8) {
    for (int i = tid; i < kWarps * 256; i += 1024) (&hist[0][0])[i] = 0;
    __syncthreads();
    for (int i0 = 0; i0 < n; i0 += 1024) {
      int i = i0 + tid;
      bool act = false;
      int bin = 0;
      if (i < n) {
        uint32_t key = key_at(i);
        act = (key & mask) == prefix;
        bin = (key >> shift) & 255;
      }
      unsigned am = __ballot_sync(0xffffffffu, act);
      if (act) {
        unsigned peers = __match_any_sync(am, bin);
        if (lane == __ffs(peers) - 1) hist[warp][bin] += __popc(peers);
      }
      __syncwarp();
    }
    __syncthreads();
    // column sums over the per-warp histograms, then a top-down scan by warp 0
    if (tid < 256) {
      int sum = 0;
#pragma unroll 8
      for (int w = 0; w < kWarps; ++w) sum += hist[w][tid];
      hist[0][tid] = sum;
    }
    __syncthreads();
    if (warp == 0) {
      // lane handles bins [lane*8, lane*8+8); suffix sums from the top
      int c[8], tot = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        c[j] = hist[0][lane * 8 + j];
        tot += c[j];
      }
      int x = tot;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        int y = __shfl_down_sync(0xffffffffu, x, o);
        if (lane + o < 32) x += y;
      }
      const int above = x - tot;  // elements in lanes above this one
      // the digit d is the highest bin with (count of bins >= d) >= remaining
      if (above < remaining && above + tot >= remaining) {
        int acc = above;
        for (int j = 7; j >= 0; --j) {
          if (acc + c[j] >= remaining) {
            sh[0] = lane * 8 + j;
            sh[1] = remaining - acc;
            break;
          }
          acc += c[j];
        }
      }
    }
    __syncthreads();
    prefix |= (uint32_t)sh[0] << shift;
    mask |= 255u << shift;
    remaining = sh[1];
    __syncthreads();
  }
  need = remaining;
  return prefix;
}

// Launches `kernel` on `clusters` clusters of `cluster_size` CTAs of `threads` threads with `smem_bytes` of dynamic
// shared memory (also set as the kernel's limit).  args[i] points at a local of exactly the type of parameter i; `name`
// prefixes the error message
inline int launch_clusters(const void* kernel, void** args, int clusters, int cluster_size, int threads, size_t smem_bytes,
                           fod_stream_t stream, const char* name) {
  FOD_CUDA_CALL(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)clusters * (unsigned)cluster_size);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem_bytes;
  cfg.stream = as_stream(stream);
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = (unsigned)cluster_size;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  const cudaError_t e = cudaLaunchKernelExC(&cfg, kernel, args);
  if (e != cudaSuccess) {
    set_error("%s: launch failed: %s", name, cudaGetErrorString(e));
    return FOD_ERR_CUDA;
  }
  return FOD_OK;
}

}  // namespace fod
