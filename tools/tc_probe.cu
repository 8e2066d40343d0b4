// Hardware probe for the tcgen05 / TMEM / TMA building blocks used by the fod_b200 tensor-core kernels.
// Development tool (not part of the library): each mode checks one mechanism against a CPU fp64 result.
//   tc_probe g1ts | g1ss | g2ts | g2ss | tma
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "../faster_orefsdet_b200/csrc/common.cuh"
#include "../faster_orefsdet_b200/csrc/tc05.cuh"

using namespace fod;
using namespace fod::tc;

#define CK(x)                                                                          \
  do {                                                                                 \
    cudaError_t e = (x);                                                               \
    if (e != cudaSuccess) {                                                            \
      printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e), __FILE__, __LINE__);   \
      exit(2);                                                                         \
    }                                                                                  \
  } while (0)

constexpr int K = 64;    // two 32-wide K chunks
#ifndef PROBE_NT
#define PROBE_NT 128
#endif
constexpr int NT = PROBE_NT;  // total N

// G = cta group (1 or 2), TS = A from tensor memory (else shared memory), NPROD = 1 (plain tf32) or 3 (3xTF32)
template <int G, bool TS, int NPROD>
__global__ void __launch_bounds__(128, 1) gemm_probe(const float* __restrict__ X, const float* __restrict__ W,
                                                     float* __restrict__ out, int repeat) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_base_s;
  constexpr int NB = NT / G;  // B rows held by this CTA
  // layout: B_hi [2 chunks][NB rows][128 B], B_lo same, then (SS) A_hi [2][128][128B], A_lo
  uint8_t* b_hi = smem;
  uint8_t* b_lo = b_hi + 2 * NB * 128;
  uint8_t* a_hi = b_lo + 2 * NB * 128;
  uint8_t* a_lo = a_hi + 2 * 128 * 128;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = (G == 2) ? cluster_ctarank() : 0;

  if (warp == 0) {
    tmem_alloc<G>(smem_u32(&tmem_base_s), 256);
    tmem_relinquish<G>();
  }
  if (tid == 0) {
    mbar_init(smem_u32(&bar), 1);
    fence_barrier_init();
  }
  // B: rows n = rank*NB + r
  for (int i = tid; i < NB * K; i += 128) {
    int r = i / K, c = i % K;
    uint32_t hi, lo;
    split_tf32(W[(size_t)(rank * NB + r) * K + c], hi, lo);
    uint32_t off = (c >> 5) * NB * 128 + sw128_offset(r, c & 31);
    *reinterpret_cast<uint32_t*>(b_hi + off) = hi;
    *reinterpret_cast<uint32_t*>(b_lo + off) = lo;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;
  // A: row m = rank*128 + tid
  const float* xr = X + (size_t)(rank * 128 + tid) * K;
  if (TS) {
    // columns [0,64) hi, [64,128) lo ; accumulator at column 128
#pragma unroll
    for (int c0 = 0; c0 < K; c0 += 16) {
      uint32_t vh[16], vl[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) split_tf32(xr[c0 + j], vh[j], vl[j]);
      uint32_t ta = tmem_base + ((uint32_t)(warp * 32) << 16);
      tmem_st16(ta + c0, vh);
      tmem_st16(ta + 64 + c0, vl);
    }
    tmem_wait_st();
  } else {
    for (int c = 0; c < K; ++c) {
      uint32_t hi, lo;
      split_tf32(xr[c], hi, lo);
      uint32_t off = (c >> 5) * 128 * 128 + sw128_offset(tid, c & 31);
      *reinterpret_cast<uint32_t*>(a_hi + off) = hi;
      *reinterpret_cast<uint32_t*>(a_lo + off) = lo;
    }
  }
  fence_proxy_async_smem();
  tc_fence_before();
  if (G == 2) cluster_sync(); else __syncthreads();
  tc_fence_after();

  long long t_start = clock64();
  if (rank == 0 && tid == 0) {
    const uint32_t idesc = idesc_tf32(128 * G, NT);
    const uint32_t d = tmem_base + 128;
    uint32_t acc = 0;
    for (int rep = 0; rep < (repeat < 0 ? -repeat : repeat); ++rep)  // repeat > 1: accumulate the same product again (accumulator rounding probe)
    for (int kc = 0; kc < 2; ++kc)
      for (int ks = 0; ks < 4; ++ks) {
        uint64_t bh = smem_desc_k_sw128(smem_u32(b_hi) + kc * NB * 128 + ks * 32);
        uint64_t bl = smem_desc_k_sw128(smem_u32(b_lo) + kc * NB * 128 + ks * 32);
        if (TS) {
          uint32_t ah = tmem_base + kc * 32 + ks * 8, al = ah + 64;
          mma_tf32_ts<G>(d, ah, bh, idesc, acc);
          acc = 1;
          if (NPROD == 3) {
            mma_tf32_ts<G>(d, al, bh, idesc, 1);
            mma_tf32_ts<G>(d, ah, bl, idesc, 1);
          }
        } else {
          uint64_t ah = smem_desc_k_sw128(smem_u32(a_hi) + kc * 128 * 128 + ks * 32);
          uint64_t al = smem_desc_k_sw128(smem_u32(a_lo) + kc * 128 * 128 + ks * 32);
          mma_tf32_ss<G>(d, ah, bh, idesc, acc);
          acc = 1;
          if (NPROD == 3) {
            mma_tf32_ss<G>(d, al, bh, idesc, 1);
            mma_tf32_ss<G>(d, ah, bl, idesc, 1);
          }
        }
      }
    if (G == 2) mma_commit_pair(smem_u32(&bar), 3); else mma_commit(smem_u32(&bar));
  }
  if (repeat < 0 && warp > 0) {  // contention probe: keep storing to unused TMEM columns while the MMAs run
    uint32_t z[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) z[j] = j;
    long long t0 = clock64();
    const int nst = 2000;
    for (int it = 0; it < nst; ++it) {
      tmem_st16(tmem_base + ((uint32_t)(warp * 32) << 16) + 256 - 64 + (it & 3) * 16, z);
      tmem_wait_st();
    }
    if (lane == 0 && rank == 0)
      printf("  warp %d: %d x (tcgen05.st.x16 + wait::st) in %lld cycles = %.1f cycles each\n", warp, nst, clock64() - t0,
             double(clock64() - t0) / nst);
  }
  mbar_wait(smem_u32(&bar), 0);
  tc_fence_after();
  if (repeat < 0) repeat = -repeat;
  if (rank == 0 && tid == 0 && repeat > 1)
    printf("  G=%d %s prod=%d: %d MMAs (M=%d N=%d K=8) in %lld cycles = %.1f cycles/MMA\n", G, TS ? "TS" : "SS", NPROD,
           repeat * 8 * NPROD, 128 * G, NT, clock64() - t_start, double(clock64() - t_start) / (repeat * 8 * NPROD));
  float* orow = out + (size_t)(rank * 128 + tid) * NT;
#pragma unroll
  for (int c0 = 0; c0 < NT; c0 += 32) {
    uint32_t v[32];
    tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + 128 + c0, v);
    tmem_wait_ld();
#pragma unroll
    for (int j = 0; j < 32; ++j) orow[c0 + j] = __uint_as_float(v[j]);
  }
  tc_fence_before();
  if (G == 2) cluster_sync(); else __syncthreads();
  if (warp == 0) tmem_dealloc<G>(tmem_base, 256);
}

template <int G, bool TS, int NPROD>
static int run_gemm(const char* name, int repeat = 1) {
  const int M = 128 * G;
  std::vector<float> X((size_t)M * K), W((size_t)NT * K), out((size_t)M * NT);
  srand(1234);
  for (auto& v : X) v = (float)rand() / RAND_MAX * 2.f - 1.f;
  for (auto& v : W) v = (float)rand() / RAND_MAX * 2.f - 1.f;
  float *dX, *dW, *dO;
  CK(cudaMalloc(&dX, X.size() * 4));
  CK(cudaMalloc(&dW, W.size() * 4));
  CK(cudaMalloc(&dO, out.size() * 4));
  CK(cudaMemcpy(dX, X.data(), X.size() * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dW, W.data(), W.size() * 4, cudaMemcpyHostToDevice));
  CK(cudaMemset(dO, 0xff, out.size() * 4));
  size_t smem = 1024 + 4 * (NT / G) * 128 + 4 * 128 * 128;
  auto kern = gemm_probe<G, TS, NPROD>;
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(G);
  cfg.blockDim = dim3(128);
  cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = G;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  CK(cudaLaunchKernelEx(&cfg, kern, (const float*)dX, (const float*)dW, dO, repeat));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(out.data(), dO, out.size() * 4, cudaMemcpyDeviceToHost));
  double maxerr = 0, maxref = 0;
  for (int m = 0; m < M; ++m)
    for (int n = 0; n < NT; ++n) {
      double r = 0;
      for (int k = 0; k < K; ++k) r += (double)X[(size_t)m * K + k] * W[(size_t)n * K + k];
      r *= abs(repeat);
      maxerr = fmax(maxerr, fabs(r - out[(size_t)m * NT + n]));
      maxref = fmax(maxref, fabs(r));
    }
  double sum_signed = 0;
  for (int m = 0; m < M; ++m)
    for (int n = 0; n < NT; ++n) {
      double r = 0;
      for (int k = 0; k < K; ++k) r += (double)X[(size_t)m * K + k] * W[(size_t)n * K + k];
      r *= repeat;
      sum_signed += (out[(size_t)m * NT + n] - r) / (fabs(r) + 1e-3);
    }
  printf("repeat=%d mean signed rel err (sign-normalised: err*sign(ref)) ", repeat);
  {
    double s2 = 0;
    for (int m = 0; m < M; ++m)
      for (int n = 0; n < NT; ++n) {
        double r = 0;
        for (int k = 0; k < K; ++k) r += (double)X[(size_t)m * K + k] * W[(size_t)n * K + k];
        r *= repeat;
        s2 += (out[(size_t)m * NT + n] - r) * (r > 0 ? 1 : -1) / (fabs(r) + 1e-3);
      }
    printf("%.3e\n", s2 / (M * NT));
  }
  printf("%s G=%d %s prod=%d: max abs err %.3e (max |ref| %.3f) rel %.3e -> %s\n", name, G, TS ? "TS" : "SS", NPROD,
         maxerr, maxref, maxerr / maxref, (maxerr / maxref < (NPROD == 3 ? 2e-6 : 2e-3)) ? "OK" : "FAIL");
  return 0;
}

// TMA: load a [10][18][32ch] halo box with negative origin (zero fill) from an NHWC map, dump smem; then
// store an [8][16][32ch] box from swizzled smem.
__global__ void tma_probe(const __grid_constant__ CUtensorMap in_map, const __grid_constant__ CUtensorMap out_map,
                          float* __restrict__ dump, int y0, int x0, int c0, int n) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ uint64_t bar;
  if (threadIdx.x == 0) {
    mbar_init(smem_u32(&bar), 1);
    fence_barrier_init();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    mbar_arrive_expect_tx(smem_u32(&bar), 180 * 128);
    tma_load_4d(smem_u32(smem), &in_map, smem_u32(&bar), c0, x0 - 1, y0 - 1, n);
  }
  mbar_wait(smem_u32(&bar), 0);
  // de-swizzle into dump [180][32]
  for (int i = threadIdx.x; i < 180 * 32; i += blockDim.x) {
    int r = i / 32, c = i % 32;
    dump[i] = *reinterpret_cast<float*>(smem + sw128_offset(r, c));
  }
  __syncthreads();
  // staging tile for the store: pixel (ty,tx) row = ty*16+tx, value = centre of the halo tile + 1000
  uint8_t* st = smem + 24 * 1024;
  for (int i = threadIdx.x; i < 128 * 32; i += blockDim.x) {
    int r = i / 32, c = i % 32, ty = r / 16, tx = r % 16;
    float v = *reinterpret_cast<float*>(smem + sw128_offset((ty + 1) * 18 + tx + 1, c)) + 1000.f;
    *reinterpret_cast<float*>(st + sw128_offset(r, c)) = v;
  }
  fence_proxy_async_smem();
  __syncthreads();
  if (threadIdx.x == 0) {
    tma_store_4d(&out_map, smem_u32(st), c0, x0, y0, n);
    tma_store_commit();
    tma_store_wait<0>();
  }
}

static int run_tma() {
  const int N = 2, H = 20, W = 20, C = 128;
  std::vector<float> in((size_t)N * H * W * C), out(in.size(), -1.f), dump(180 * 32);
  for (size_t i = 0; i < in.size(); ++i) in[i] = (float)(i % 9973) + 1.f;
  float *dI, *dO, *dD;
  CK(cudaMalloc(&dI, in.size() * 4));
  CK(cudaMalloc(&dO, in.size() * 4));
  CK(cudaMalloc(&dD, dump.size() * 4));
  CK(cudaMemcpy(dI, in.data(), in.size() * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dO, out.data(), in.size() * 4, cudaMemcpyHostToDevice));
  CUtensorMap im, om;
  if (make_nhwc_map(&im, dI, N, H, W, C, C, 32, 18, 10, 1, CU_TENSOR_MAP_SWIZZLE_128B) ||
      make_nhwc_map(&om, dO, N, H, W, C, C, 32, 16, 8, 1, CU_TENSOR_MAP_SWIZZLE_128B)) {
    char buf[256];
    fod_last_error(buf, sizeof buf);
    printf("tensor map: %s\n", buf);
    return 1;
  }
  int bad_total = 0;
  const int cases[3][4] = {{0, 0, 0, 0}, {16, 16, 32, 1}, {8, 16, 96, 1}};  // y0, x0, c0, n
  for (auto& cs : cases) {
    int y0 = cs[0], x0 = cs[1], c0 = cs[2], n = cs[3];
    CK(cudaFuncSetAttribute(tma_probe, cudaFuncAttributeMaxDynamicSharedMemorySize, 48 * 1024));
    tma_probe<<<1, 128, 48 * 1024>>>(im, om, dD, y0, x0, c0, n);
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(dump.data(), dD, dump.size() * 4, cudaMemcpyDeviceToHost));
    int bad = 0;
    for (int r = 0; r < 180; ++r)
      for (int c = 0; c < 32; ++c) {
        int yy = y0 - 1 + r / 18, xx = x0 - 1 + r % 18;
        float ref = (yy < 0 || yy >= H || xx < 0 || xx >= W) ? 0.f : in[(((size_t)n * H + yy) * W + xx) * C + c0 + c];
        if (dump[r * 32 + c] != ref) ++bad;
      }
    printf("tma load  (y0=%d x0=%d c0=%d n=%d): %d mismatches\n", y0, x0, c0, n, bad);
    bad_total += bad;
  }
  CK(cudaMemcpy(out.data(), dO, in.size() * 4, cudaMemcpyDeviceToHost));
  int bad = 0;
  for (int n = 0; n < N; ++n)
    for (int y = 0; y < H; ++y)
      for (int x = 0; x < W; ++x)
        for (int c = 0; c < C; ++c) {
          float ref = -1.f;
          for (auto& cs : cases)
            if (n == cs[3] && y >= cs[0] && y < cs[0] + 8 && x >= cs[1] && x < cs[1] + 16 && c >= cs[2] && c < cs[2] + 32)
              ref = in[(((size_t)n * H + y) * W + x) * C + c] + 1000.f;
          if (out[(((size_t)n * H + y) * W + x) * C + c] != ref) ++bad;
        }
  printf("tma store: %d mismatches -> %s\n", bad, (bad + bad_total) ? "FAIL" : "OK");
  return 0;
}

int main(int argc, char** argv) {
  const char* mode = argc > 1 ? argv[1] : "g1ts";
  if (!strcmp(mode, "g1ts")) { run_gemm<1, true, 1>(mode); return run_gemm<1, true, 3>(mode); }
  if (!strcmp(mode, "g1ss")) { run_gemm<1, false, 1>(mode); return run_gemm<1, false, 3>(mode); }
  if (!strcmp(mode, "g2ts")) { run_gemm<2, true, 1>(mode); return run_gemm<2, true, 3>(mode); }
  if (!strcmp(mode, "g2ss")) { run_gemm<2, false, 1>(mode); return run_gemm<2, false, 3>(mode); }
  if (!strcmp(mode, "acc")) {  // accumulator rounding: error growth with the number of accumulations
    for (int r : {1, 16, 128, 1024}) run_gemm<1, true, 3>(mode, r);
    return 0;
  }
  if (!strcmp(mode, "contend")) {  // MMA chain while other warps store to tensor memory
    run_gemm<1, true, 3>(mode, -512);
    run_gemm<2, true, 3>(mode, -512);
    run_gemm<2, true, 3>(mode, -16);
    return 0;
  }
  if (!strcmp(mode, "rate")) {  // MMA issue rate
    run_gemm<1, true, 3>(mode, 512);
    run_gemm<1, false, 3>(mode, 512);
    run_gemm<2, true, 3>(mode, 512);
    run_gemm<2, false, 3>(mode, 512);
    run_gemm<2, true, 1>(mode, 512);
    return 0;
  }
  if (!strcmp(mode, "tma")) return run_tma();
  printf("unknown mode\n");
  return 1;
}
