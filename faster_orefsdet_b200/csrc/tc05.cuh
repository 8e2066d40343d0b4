// Thin inline-PTX layer over the Blackwell (sm_100a) async machinery used by the
// tensor-core kernels of this library: mbarrier, TMA (cp.async.bulk.tensor),
// tensor memory (tcgen05.alloc/ld/st) and the 5th-generation MMA (tcgen05.mma,
// kind::tf32) with its commit/fence protocol.  No CUTLASS, no libcuda link: the
// one driver entry point needed on the host (cuTensorMapEncodeTiled) is resolved
// through cudaGetDriverEntryPoint.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace fod {
namespace tc {

// ------------------------------------------------------------------------------------------------
// addresses
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// shared::cta address of this CTA -> shared::cluster address of the same offset in CTA `rank`
__device__ __forceinline__ uint32_t map_to_cta(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}

// ------------------------------------------------------------------------------------------------
// mbarrier
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// arrive on a barrier of another (or this) CTA of the cluster; `bar` is a shared::cluster address.  No cluster-scope
// release (no memory barrier): for hand-offs whose payload is not generic memory (tensor memory made visible by
// tcgen05.wait + tcgen05.fence::before_thread_sync)
__device__ __forceinline__ void mbar_arrive_remote(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Wait for the phase with the given parity.  A protocol bug would otherwise hang the GPU until the
// watchdog; after ~2^26 failed probes (seconds) the kernel traps instead so the host sees an error.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 26)) __trap();
  }
}

// generic-proxy writes (st.shared) -> visible to the async proxy (TMA store, tcgen05.mma operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------
// TMA
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
// cta_group::2 form: the bytes complete on an mbarrier of the PEER (leader) CTA; `bar` is a shared::cluster address
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_2sm(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2,
                                                int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ------------------------------------------------------------------------------------------------
// tensor memory
// ------------------------------------------------------------------------------------------------
template <int kCtaGroup>
__device__ __forceinline__ void tmem_alloc(uint32_t smem_result_addr, uint32_t ncols) {
  if constexpr (kCtaGroup == 1)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_result_addr), "r"(ncols)
                 : "memory");
  else
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_result_addr), "r"(ncols)
                 : "memory");
}
template <int kCtaGroup>
__device__ __forceinline__ void tmem_relinquish() {
  if constexpr (kCtaGroup == 1)
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  else
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int kCtaGroup>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  if constexpr (kCtaGroup == 1)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
  else
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// 32 lanes x 32-bit, 32 consecutive columns: thread t of the warp <-> TMEM lane (quadrant base + t)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint32_t (&v)[4]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]),
               "r"(v[3])
               : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(v[0]),
               "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
      "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}

// ------------------------------------------------------------------------------------------------
// tcgen05.mma, kind::tf32
// ------------------------------------------------------------------------------------------------
// Shared-memory operand descriptor, K-major, 128-byte swizzle: rows of 128 bytes (32 fp32 of K), 8 rows form
// one 1024-byte swizzle atom (16-byte chunk j of row r is stored at chunk j ^ (r & 7)), atoms stacked along
// M/N every 1024 bytes (SBO).  The tile base must be 1024-byte aligned; K advances inside the 128-byte row by
// adding the byte offset to the start address.
__device__ __forceinline__ uint64_t smem_desc_k_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);        // start address  [0,14)
  d |= (uint64_t)1 << 16;                          // leading byte offset (unused with swizzle) [16,30)
  d |= (uint64_t)(1024 >> 4) << 32;                // stride byte offset: 8 rows * 128 B       [32,46)
  d |= (uint64_t)1 << 46;                          // descriptor version (Blackwell)           [46,48)
  d |= (uint64_t)2 << 61;                          // SWIZZLE_128B                             [61,64)
  return d;
}
// Instruction descriptor: D fp32, A/B tf32, both K-major, dense.  M in {64,128,256}, N multiple of 8/16.
__host__ __device__ constexpr uint32_t idesc_tf32(int M, int N) {
  return (1u << 4)                       // D format  F32
         | (2u << 7)                     // A format  TF32
         | (2u << 10)                    // B format  TF32
         | (0u << 15) | (0u << 16)       // A, B K-major
         | ((uint32_t)(N >> 3) << 17)    // N / 8
         | ((uint32_t)(M >> 4) << 24);   // M / 16
}
// ---- kind::f16 (fp16 operands, fp32 accumulation): K = 16 per instruction.  Measured (tools/f16_probe.cu): 64 cycles
// at N = 128 and 32 cycles at N = 64, where kind::tf32 (K = 8) needs 64 and 45.
__host__ __device__ constexpr uint32_t idesc_f16(int M, int N) {
  return (1u << 4)                       // D format  F32
         | (0u << 7) | (0u << 10)        // A, B format F16
         | (0u << 15) | (0u << 16)       // A, B K-major
         | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// Shared-memory operand descriptor, K-major, 64-byte swizzle: rows of 64 bytes (32 fp16 of K), 8 rows per 512-byte atom.
__device__ __forceinline__ uint64_t smem_desc_k_sw64(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(512 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)4 << 61;                // SWIZZLE_64B
  return d;
}
// D[tmem] (+)= A[tmem] * B[smem]^T, A: lane = row, each 32-bit column holds two consecutive fp16 of K (low half first)
template <int kCtaGroup>
__device__ __forceinline__ void mma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  if constexpr (kCtaGroup == 1)
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
        "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
  else
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
        "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// D[tmem] (+)= A[smem] * B[smem]^T, fp16 operands
template <int kCtaGroup>
__device__ __forceinline__ void mma_f16_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  if constexpr (kCtaGroup == 1)
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
  else
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// D[tmem] (+)= A[smem] * B[smem]^T
template <int kCtaGroup>
__device__ __forceinline__ void mma_tf32_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  if constexpr (kCtaGroup == 1)
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
  else
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]^T   (A: lane = row, one fp32 per column along K)
template <int kCtaGroup>
__device__ __forceinline__ void mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  if constexpr (kCtaGroup == 1)
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
        "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
  else
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
        "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Make an mbarrier track completion of all tcgen05.mma issued so far by this thread (implies
// tcgen05.fence::before_thread_sync).  cta_group::2: multicast to the same barrier offset in the CTAs of `mask`.
__device__ __forceinline__ void mma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mma_commit_pair(uint32_t bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"(mask)
               : "memory");
}

// ------------------------------------------------------------------------------------------------
// 3xTF32 operand split: x = hi + lo, hi = x rounded to nearest tf32 (integer add of half an ulp, then mask;
// the tensor core reads only the top 19 bits of each 32-bit operand), lo = x - hi (exact in fp32, |lo| <=
// 2^-11 |x|, sign random).  The hardware truncates lo to tf32: error <= 2^-21 |x| with random sign, so it does
// not accumulate coherently along K (a truncated hi would make every lo positive and the error a bias that
// grows linearly with K: measured 1e-4 absolute at K = 8192).  A*B ~= Ahi*Bhi + Alo*Bhi + Ahi*Blo.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = (__float_as_uint(x) + 0x1000u) & 0xFFFFE000u;
  lo = __float_as_uint(x - __uint_as_float(hi));
}

// explicit shared-window accesses (a generic pointer would compile to LD/ST with address-space resolution)
__device__ __forceinline__ float4 lds4s(uint32_t saddr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
  return v;
}
__device__ __forceinline__ void sts4s(uint32_t saddr, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(saddr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// byte offset of fp32 element (row r, column c) inside a K-major SW128 tile (c in [0,32))
__device__ __forceinline__ uint32_t sw128_offset(int r, int c) {
  return (uint32_t)((r >> 3) * 1024 + (r & 7) * 128 + ((((c >> 2) ^ (r & 7)) & 7) << 4) + ((c & 3) << 2));
}

}  // namespace tc

// ------------------------------------------------------------------------------------------------
// host: tensor-map encoding without linking libcuda
// ------------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
PFN_encodeTiled get_encode_tiled();

// fp32 NHWC map [N][H][W][C] whose pixels lie pixel_stride floats apart (>= C: a channel slice of a wider map) -> 4-D
// tensor map (dims innermost first: C, W, H, N), box (bc, bw, bh, 1), element strides (1, estride, estride, 1);
// out-of-bounds elements read as zero / are not written.  CU_TENSOR_MAP_SWIZZLE_128B needs bc * 4 == 128; with
// CU_TENSOR_MAP_SWIZZLE_NONE the box lands in shared memory as a dense [bh][bw][bc] array (bc * 4 a multiple of 16).
int make_nhwc_map(CUtensorMap* out, const float* base, int N, int H, int W, int C, long pixel_stride, int bc, int bw, int bh,
                  int estride, CUtensorMapSwizzle swizzle);
// fp32 row-major matrix [rows][cols] -> 2-D tensor map, box (box_cols, box_rows), 128-byte swizzle
// (box_cols * 4 must be 128), rows beyond the matrix read as zero.
int make_matrix_map(CUtensorMap* out, const float* base, long rows, long cols, int box_cols, int box_rows);
// fp16 row-major matrix [rows][cols] -> 2-D tensor map, box (box_cols, box_rows), 64-byte swizzle (box_cols * 2 must be 64)
int make_matrix_map_f16(CUtensorMap* out, const void* base, long rows, long cols, int box_cols, int box_rows);

}  // namespace fod
