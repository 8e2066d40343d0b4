// Probe for the fp16-split variant of the tensor-core GEMM: tcgen05.mma kind::f16 with A in tensor memory (packed
// half2 per 32-bit column), B in shared memory (fp16, K-major, 64-byte swizzle, loaded by TMA).  x = hi + lo with
// hi = fp16(x * 2^e), lo = fp16(x * 2^e - hi): three products hi.hi + lo.hi + hi.lo, fp32 accumulation.
// `ss` mode: the same products with A in shared memory instead (K-major, 128-byte swizzle, per 128-byte row
// [16 hi | 16 lo | 16 hi | 16 lo] as the split hand-off stores it, the layout the shared-memory A convolution reads):
// D must equal the tensor-memory result bit for bit at A start offsets of 0, 2048 and 4096 bytes (a tap row of the
// convolution's stride-1 boxes), and both paths are timed.
// Development tool:  f16_probe [N] [ss]   (nvcc -gencode arch=compute_100a,code=sm_100a tools/f16_probe.cu csrc/tmap.cu csrc/api.cu)
#include <cuda_fp16.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <vector>

#include "../faster_orefsdet_b200/csrc/common.cuh"
#include "../faster_orefsdet_b200/csrc/tc05.cuh"

using namespace fod;
using namespace fod::tc;

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %d\n", cudaGetErrorString(e), __LINE__); exit(2); } } while (0)

constexpr int K = 32;

struct P { CUtensorMap bhi, blo; };

// ss: A from shared memory, rows starting `dy` * 16 rows (dy * 2048 bytes) into a 160-row swizzled buffer
__global__ void __launch_bounds__(128, 1) probe(const __grid_constant__ P p, const float* __restrict__ X, float xs, float* __restrict__ out,
                                                int N, int repeat, int ss, int dy) {
  extern __shared__ __align__(1024) uint8_t raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) & ~uintptr_t(1023));
  __shared__ uint64_t bar, bar2;
  __shared__ uint32_t tb;
  const int tid = threadIdx.x, warp = tid >> 5;
  const uint32_t sb = smem_u32(smem), plane = (uint32_t)N * 64;
  if (warp == 0) { tmem_alloc<1>(smem_u32(&tb), 512); tmem_relinquish<1>(); }
  if (tid == 0) {
    mbar_init(smem_u32(&bar), 1); mbar_init(smem_u32(&bar2), 1); fence_barrier_init();
    mbar_arrive_expect_tx(smem_u32(&bar2), 2 * plane);
    tma_load_2d(sb, &p.bhi, smem_u32(&bar2), 0, 0);
    tma_load_2d(sb + plane, &p.blo, smem_u32(&bar2), 0, 0);
  }
  tc_fence_before(); __syncthreads(); tc_fence_after();
  const uint32_t t0 = tb;
  // A row tid: packed half2 columns: hi at [0,16), lo at [16,32)
  uint32_t vh[16], vl[16];
  for (int j = 0; j < 16; ++j) {
    float a = X[tid * K + 2 * j] * xs, b = X[tid * K + 2 * j + 1] * xs;
    __half2 h = __floats2half2_rn(a, b);
    float2 hf = __half22float2(h);
    __half2 l = __floats2half2_rn(a - hf.x, b - hf.y);
    vh[j] = *reinterpret_cast<uint32_t*>(&h);
    vl[j] = *reinterpret_cast<uint32_t*>(&l);
  }
  const uint32_t ta = t0 + ((uint32_t)(warp * 32) << 16);
  tmem_st16(ta, vh); tmem_st16(ta + 16, vl); tmem_wait_st();
  const uint32_t sa = sb + (2 * plane + 1023) / 1024 * 1024;   // A buffer (ss)
  {
    const uint32_t r = (uint32_t)(tid + 16 * dy), row = sa + r * 128;
    const uint32_t* src[8] = {vh, vh + 4, vl, vl + 4, vh + 8, vh + 12, vl + 8, vl + 12};   // 16-byte chunks of the row
    for (uint32_t c = 0; c < 8; ++c)
      asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(row + ((c ^ (r & 7)) << 4)), "r"(src[c][0]), "r"(src[c][1]),
                   "r"(src[c][2]), "r"(src[c][3]) : "memory");
    fence_proxy_async_smem();
  }
  tc_fence_before(); __syncthreads(); tc_fence_after();
  mbar_wait(smem_u32(&bar2), 0);
  long long t_start = clock64();
  if (warp == 0) {
    const uint32_t idesc = idesc_f16(128, N), d = t0 + 64;
    const uint64_t bh = smem_desc_k_sw64(sb), bl = smem_desc_k_sw64(sb + plane);
    for (int rep = 0; rep < repeat; ++rep) {
      if (elect_one()) {
        if (ss) {
          const uint64_t a = smem_desc_k_sw128(sa + (uint32_t)dy * 2048);
#pragma unroll
          for (int ks = 0; ks < 2; ++ks) {   // hi at +64 ks bytes, lo at +64 ks + 32
            const uint64_t bo = (uint64_t)((ks * 32) >> 4), ah = a + (uint64_t)(ks * 4), al = ah + 2;
            mma_f16_ss<1>(d, ah, bh + bo, idesc, (rep | ks) ? 1u : 0u);
            mma_f16_ss<1>(d, al, bh + bo, idesc, 1u);
            mma_f16_ss<1>(d, ah, bl + bo, idesc, 1u);
          }
        } else {
#pragma unroll
          for (int ks = 0; ks < 2; ++ks) {
            const uint64_t bo = (uint64_t)((ks * 32) >> 4);
            mma_f16_ts<1>(d, t0 + ks * 8, bh + bo, idesc, (rep | ks) ? 1u : 0u);
            mma_f16_ts<1>(d, t0 + 16 + ks * 8, bh + bo, idesc, 1u);
            mma_f16_ts<1>(d, t0 + ks * 8, bl + bo, idesc, 1u);
          }
        }
      }
      __syncwarp();
    }
    if (elect_one()) mma_commit(smem_u32(&bar));
  }
  mbar_wait(smem_u32(&bar), 0);
  tc_fence_after();
  if (tid == 0 && repeat > 1)
    printf("  %s: %d MMAs (M=128 N=%d K=16 f16) in %lld cycles = %.1f cycles/MMA\n", ss ? "SS" : "TS", repeat * 6, N, clock64() - t_start,
           double(clock64() - t_start) / (repeat * 6));
  for (int c0 = 0; c0 < N; c0 += 32) {
    uint32_t v[32];
    tmem_ld32(t0 + ((uint32_t)(warp * 32) << 16) + 64 + c0, v);
    tmem_wait_ld();
    for (int j = 0; j < 32; ++j) out[tid * N + c0 + j] = __uint_as_float(v[j]);
  }
  tc_fence_before(); __syncthreads();
  if (warp == 0) tmem_dealloc<1>(t0, 512);
}

int main(int argc, char** argv) {
  const int N = argc > 1 ? atoi(argv[1]) : 128;
  const bool ss = argc > 2 && !strcmp(argv[2], "ss");
  std::vector<float> X(128 * K), W(N * K);
  srand(1);
  for (auto& v : X) v = (rand() / (float)RAND_MAX - 0.3f) * 37.f;
  for (auto& v : W) v = (rand() / (float)RAND_MAX - 0.5f) * 0.21f;
  float ax = 0, aw = 0;
  for (auto v : X) ax = fmaxf(ax, fabsf(v));
  for (auto v : W) aw = fmaxf(aw, fabsf(v));
  const float xs = exp2f(13 - ceilf(log2f(ax))), ws = exp2f(13 - ceilf(log2f(aw)));
  std::vector<__half> whi(N * K), wlo(N * K);
  for (int i = 0; i < N * K; ++i) {
    float s = W[i] * ws;
    whi[i] = __float2half_rn(s);
    wlo[i] = __float2half_rn(s - __half2float(whi[i]));
  }
  float *dX, *dO; __half *dhi, *dlo;
  CK(cudaMalloc(&dX, X.size() * 4)); CK(cudaMalloc(&dO, 128 * N * 4)); CK(cudaMalloc(&dhi, N * K * 2)); CK(cudaMalloc(&dlo, N * K * 2));
  CK(cudaMemcpy(dX, X.data(), X.size() * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dhi, whi.data(), N * K * 2, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dlo, wlo.data(), N * K * 2, cudaMemcpyHostToDevice));
  P p;
  PFN_encodeTiled enc = get_encode_tiled();
  for (int i = 0; i < 2; ++i) {
    cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)N};
    cuuint64_t strides[1] = {(cuuint64_t)K * 2};
    cuuint32_t box[2] = {32, (cuuint32_t)N};
    cuuint32_t es[2] = {1, 1};
    CUresult r = enc(i ? &p.blo : &p.bhi, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, i ? (void*)dlo : (void*)dhi, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { printf("encode failed %d\n", (int)r); return 2; }
  }
  const int smem = (2 * N * 64 + 1023) / 1024 * 1024 + 160 * 128 + 2048;
  CK(cudaFuncSetAttribute(probe, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  if (ss) {   // D of the SS path at each A start offset against the TS path, bit for bit; then both timed
    std::vector<float> Ots(128 * N), Oss(128 * N);
    probe<<<1, 128, smem>>>(p, dX, xs, dO, N, 1, 0, 0);
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(Ots.data(), dO, Ots.size() * 4, cudaMemcpyDeviceToHost));
    for (int dy = 0; dy < 3; ++dy) {
      probe<<<1, 128, smem>>>(p, dX, xs, dO, N, 1, 1, dy);
      CK(cudaDeviceSynchronize());
      CK(cudaMemcpy(Oss.data(), dO, Oss.size() * 4, cudaMemcpyDeviceToHost));
      int ndiff = 0, cmin = N, cmax = -1;
      double dmax = 0, ref = 0;
      for (int i = 0; i < 128 * N; ++i) {
        ref = fmax(ref, fabs(Ots[i]));
        if (memcmp(&Oss[i], &Ots[i], 4)) {
          ++ndiff;
          cmin = i % N < cmin ? i % N : cmin;
          cmax = i % N > cmax ? i % N : cmax;
          dmax = fmax(dmax, fabs((double)Oss[i] - Ots[i]));
        }
      }
      if (!ndiff) printf("N=%d SS, A at +%d bytes: D equals the TS result bitwise\n", N, dy * 2048);
      else printf("N=%d SS, A at +%d bytes: D differs from the TS result in %d of %d elements (columns %d..%d), by up to %.3e "
                  "of max|D| %.3e\n", N, dy * 2048, ndiff, 128 * N, cmin, cmax, dmax / ref, ref);
    }
    for (int mode = 0; mode < 2; ++mode) {
      probe<<<1, 128, smem>>>(p, dX, xs, dO, N, 2000, mode, 0);
      CK(cudaDeviceSynchronize());
    }
    return 0;
  }
  for (int repeat : {1, 2000}) {
    probe<<<1, 128, smem>>>(p, dX, xs, dO, N, repeat, 0, 0);
    CK(cudaDeviceSynchronize());
    if (repeat > 1) break;
    std::vector<float> O(128 * N);
    CK(cudaMemcpy(O.data(), dO, O.size() * 4, cudaMemcpyDeviceToHost));
    double maxerr = 0, maxref = 0;
    for (int m = 0; m < 128; ++m)
      for (int n = 0; n < N; ++n) {
        double ref = 0;
        for (int k = 0; k < K; ++k) ref += (double)X[m * K + k] * W[n * K + k];
        double got = (double)O[m * N + n] / ((double)xs * ws);
        maxerr = fmax(maxerr, fabs(got - ref));
        maxref = fmax(maxref, fabs(ref));
      }
    printf("N=%d scales 2^%g 2^%g: max abs err %.3e  max |ref| %.3e  rel %.3e -> %s\n", N, log2(xs), log2(ws), maxerr, maxref,
           maxerr / maxref, maxerr / maxref < 3e-6 ? "OK" : "FAIL");
  }
  return 0;
}
