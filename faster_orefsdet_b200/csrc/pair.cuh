// The rules every CTA-pair tensor-core kernel keeps (conv_tc.cu: conv_tc_kernel_tmem / conv_tc_kernel_smem,
// correlate_tc.cu: correlate_tc_kernel, relation_tc.cu: relation_tc_kernel).  Two CTAs form a cluster and share one
// cta_group::2 MMA issued by the leader (rank 0); the MMA warp walks its rings by a running index, a watcher thread does
// all the barrier waiting for it, and the epilogue warps of both CTAs hand every accumulator stage back to the leader.
// A copy of one of these rules that drifts from the others hangs the pair, so each is written once, here.  The host
// launches them through launch_clusters (common.cuh) with a cluster size of 2.
#pragma once
#include "common.cuh"
#include "tc05.cuh"

namespace fod {
namespace tc {

// Stage and phase parity of the g-th use of an n-stage ring; the next stage after s
__device__ __forceinline__ uint32_t ring_stage(uint32_t g, uint32_t n) { return g % n; }
__device__ __forceinline__ uint32_t ring_phase(uint32_t g, uint32_t n) { return (g / n) & 1u; }
__device__ __forceinline__ uint32_t ring_next(uint32_t s, uint32_t n) { return s + 1 == n ? 0u : s + 1; }

// Watcher -> MMA warp: the number of chunks whose operands are in place (an mbarrier wait costs ~200 cycles even on a
// long-completed phase, so only the watcher waits on barriers).  The MMA warp polls converged; lane 0's load decides.
__device__ __forceinline__ void flag_publish(uint32_t flag, uint32_t n) {
  asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"(flag), "r"(n) : "memory");
}
__device__ __forceinline__ void flag_wait(uint32_t flag, uint32_t& upto, uint32_t g) {
  while (upto <= g) {
    uint32_t v;
    asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(v) : "r"(flag) : "memory");
    upto = __shfl_sync(0xffffffffu, v, 0);
  }
}

// Both CTAs allocate the pair's `cols` columns of tensor memory (warp alloc_warp writes the base to tmem_ptr), run
// `work` (whatever else must be in place before the pair starts), then barrier initialisation, allocation and that work
// become visible to both CTAs.  Returns the tensor-memory base.
template <class Work>
__device__ __forceinline__ uint32_t pair_setup(uint8_t* tmem_ptr, int warp, int alloc_warp, uint32_t cols, Work&& work) {
  if (warp == alloc_warp) {
    tmem_alloc<2>(smem_u32(tmem_ptr), cols);
    tmem_relinquish<2>();
  }
  work();
  tc_fence_before();
  cluster_sync();
  tc_fence_after();
  return *reinterpret_cast<volatile uint32_t*>(tmem_ptr);
}
// No CTA of the pair frees the tensor memory before both have finished with it
__device__ __forceinline__ void pair_teardown(int warp, int alloc_warp, uint32_t tmem_base, uint32_t cols) {
  __syncwarp();
  tc_fence_before();
  cluster_sync();
  if (warp == alloc_warp) tmem_dealloc<2>(tmem_base, cols);
}

// An epilogue warp has read its columns of an accumulator stage: one arrival on that stage's barrier `empty` of the
// leader CTA (a shared::cluster address) hands them back to the MMA warp
__device__ __forceinline__ void acc_release(uint32_t empty, int lane) {
  tc_fence_before();
  __syncwarp();
  if (lane == 0) mbar_arrive_remote(empty);
}

// Bound of max|x| that the operand scale of image n comes from: the maximum over the n_amax rows of column n of
// x_amax [n_amax][stride], or over the n_amax scalars when stride is 0 (one bound for the whole batch, any n)
__device__ __forceinline__ float image_bound(const float* x_amax, int n_amax, int stride, int n) {
  float amax = 0.f;
  const float* col = x_amax + (stride ? n : 0);
  const int step = stride ? stride : 1;
#pragma unroll 4
  for (int i = 0; i < n_amax; ++i) amax = fmaxf(amax, __ldg(col + (size_t)i * step));
  return amax;
}

}  // namespace tc

// CTA pairs for `units` pair units: one pair per two SMs, at least one, and no more than there are units
inline int pair_count(long units, int* pairs) {
  int dev = 0, sms = 0;
  FOD_CUDA_CALL(cudaGetDevice(&dev));
  FOD_CUDA_CALL(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int max_pairs = sms / 2 > 0 ? sms / 2 : 1;
  *pairs = units < max_pairs ? (int)units : max_pairs;
  return FOD_OK;
}

}  // namespace fod
