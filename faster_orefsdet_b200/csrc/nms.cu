// Greedy NMS kernels: one problem per CTA or per thread-block CLUSTER, everything resident in shared memory.
//
//   sort   : bitonic sort of 64-bit keys (~ordered(score) << 32 | row) -> stable score-descending order (lower input
//            row first among equal scores); the boxes are then gathered in sorted order (sort_and_gather).
//   sweep  : blocked greedy suppression, 64 sorted boxes per step:
//              1. 64x64 IoU bit matrix of the chunk, stored by COLUMN (warp ballots),
//              2. the chunk is resolved by ONE WARP with a fixed-point iteration on the column masks
//                 (kept_j = alive_j and no kept_i, i < j, overlaps j: converges to the greedy answer in
//                 (longest suppression chain + 1) ballot rounds instead of one serial step per survivor),
//              3. the chunk's survivors suppress every later box (all threads; G = 1..32 lanes share a box, more
//                 the fewer boxes are alive).
//            Only survivors ever test later boxes, so the work is kept*n/2 IoU
//            pairs instead of n^2/2, and no n x n mask goes through HBM.
//            The sweep stops as soon as the caller's top-k is decided.
//   cluster: the kernel is instruction bound on one SM (profiles/r1_ncu_v5_summary.md: 59 % issue-active on 64 of
//            148 SMs), so a problem may be spread over S = 1, 2 or 4 CTAs of a cluster.  Every CTA holds the sorted boxes
//            and resolves every chunk redundantly (identical results by construction); step 3 is split: CTA r owns
//            the suppression words w with w % S == r.  After each pair of chunks the owners of the next pair's four
//            words push them into every peer's shared memory (st.shared::cluster) and the cluster barriers once.
//
// IoU arithmetic is bit-identical to torchvision's CPU kernel (common.cuh).
#include "common.cuh"
#include "tc05.cuh"

namespace fod {

#ifdef FOD_NMS_PROF
__device__ long long g_nms_prof[16];
#define PROF_DECL long long prof_acc[16] = {0}
#define PROF_T(var) long long var = clock64()
#define PROF_ADD(slot, t0) prof_acc[slot] += clock64() - (t0)
#define PROF_CNT(slot, v) prof_acc[slot] += (v)
#define PROF_FLUSH(lo, hi) do { if (threadIdx.x == 0 && blockIdx.x == 0) for (int i_ = lo; i_ < hi; ++i_) g_nms_prof[i_] += prof_acc[i_]; } while (0)
#else
#define PROF_DECL
#define PROF_T(var)
#define PROF_ADD(slot, t0)
#define PROF_CNT(slot, v)
#define PROF_FLUSH(lo, hi)
#endif

constexpr int kNmsThreads = 1024;
constexpr int kChunk = 64;
constexpr int kPreRead = 3;      // list passes a thread may hold in registers (suppression pass of greedy_sweep)
constexpr int kMaxCluster = 4;   // measured: 8 CTAs per problem are slower than 4 (cluster barrier + the redundant sort / resolve)

struct NmsSmem {
  unsigned long long* keys;     // [npad] sort keys (sort_key), ~0 padding
  float4* box;                  // [ncap] sorted boxes (clipped / class-offset as the kernel needs)
  float4* kbox;                 // [128] survivors of the chunk pair being applied
  uint32_t* colmask;            // [2 buffers][lo 64 | hi 64]: bit i of word j: chunk box i (i < j) overlaps chunk box j
  float* karea;                 // [128]
  uint32_t* suppressed;         // [nms_words(ncap)]; a CTA of a cluster keeps only its own words up to date
  uint32_t* chunk_sup;          // [2 parities][4 + 2]: suppression words of the chunk pair being resolved (pushed by their
                                // owners), then the pair's two cross words (second chunk suppressed by the first one's survivors)
  int* scalars;                 // [8]
  uint16_t* kept;               // [ncap + 128] sorted ranks of survivors, growing from the front ...
  uint16_t* alist_top;          // ... and, from the END of the same array downwards (entry e at alist_top[-e]), this CTA's
                                // boxes that are still alive and not yet resolved (any order).  While a pair of chunks is
                                // being resolved the list still holds the pair's own <= 128 boxes: survivors + listed
                                // <= n + 128, which is the size of the array.
};

__host__ __device__ constexpr int next_pow2(int n) {
  int p = 1;
  while (p < n) p <<= 1;
  return p;
}

__host__ __device__ constexpr size_t nms_words(int ncap) { return (size_t)(ncap + 31) / 32 + 4; }   // 4 spare (zero) words

// The layout of NmsSmem for up to ncap rows: where each array starts when the first starts at `base`, and where the
// last one (with 64 bytes of slack) ends.  Walked with a pointer by carve and with a byte offset by nms_smem_bytes.
template <class T>
struct NmsArrays {
  T keys, box, kbox, colmask, karea, suppressed, chunk_sup, scalars, kept, end;
};
template <class T>
__host__ __device__ constexpr NmsArrays<T> nms_arrays(T base, int ncap) {
  NmsArrays<T> a{};
  a.keys = base;
  base += (size_t)next_pow2(ncap < 64 ? 64 : ncap) * 8;
  a.box = base;
  base += (size_t)ncap * 16;
  a.kbox = base;
  base += 128 * 16;
  a.colmask = base;
  base += 2 * 128 * 4;
  a.karea = base;
  base += 128 * 4;
  a.suppressed = base;
  base += nms_words(ncap) * 4;
  a.chunk_sup = base;
  base += 48;
  a.scalars = base;
  base += 32;
  a.kept = base;
  base += (size_t)(ncap + 2 * kChunk) * 2 + 64;
  a.end = base;
  return a;
}

__host__ __device__ constexpr size_t nms_smem_bytes(int ncap) { return nms_arrays<size_t>(0, ncap).end; }
// Every entry point rejects more than FOD_NMS_MAX_BOXES rows, and the size grows with the row count
static_assert(nms_smem_bytes(FOD_NMS_MAX_BOXES) <= 227 * 1024, "the largest NMS problem must fit in shared memory");

__device__ inline NmsSmem carve(unsigned char* base, int ncap) {
  const NmsArrays<unsigned char*> a = nms_arrays(base, ncap);
  NmsSmem s;
  s.keys = reinterpret_cast<unsigned long long*>(a.keys);
  s.box = reinterpret_cast<float4*>(a.box);
  s.kbox = reinterpret_cast<float4*>(a.kbox);
  s.colmask = reinterpret_cast<uint32_t*>(a.colmask);
  s.karea = reinterpret_cast<float*>(a.karea);
  s.suppressed = reinterpret_cast<uint32_t*>(a.suppressed);
  s.chunk_sup = reinterpret_cast<uint32_t*>(a.chunk_sup);
  s.scalars = reinterpret_cast<int*>(a.scalars);
  s.kept = reinterpret_cast<uint16_t*>(a.kept);
  s.alist_top = s.kept + (ncap + 2 * kChunk - 1);
  return s;
}

// Sort key of input row `row`: ascending keys = descending scores, lower row first among equal scores
__device__ __forceinline__ unsigned long long sort_key(float score, int row) {
  return ((unsigned long long)(~float_to_ordered(score)) << 32) | (unsigned)row;
}
// Input row of sorted rank r
__device__ __forceinline__ int row_of(const NmsSmem& s, int r) { return (int)(s.keys[r] & 0xffffffffu); }

// One compare-exchange step of the bitonic network on E consecutive keys per thread held in registers (thread t owns
// the global indices E*t .. E*t+E-1): partner distance j < 32*E, so the partner sits in this thread or in another lane
// of the warp (two 32-bit shuffles per key).
template <int E>
__device__ __forceinline__ void bitonic_reg_step(unsigned long long (&v)[E], int k, int j, int g0) {
  if (j < E) {
#pragma unroll
    for (int e = 0; e < E; ++e) {
      if ((e & j) == 0 && (e | j) < E) {
        const bool up = ((g0 + e) & k) == 0;
        const unsigned long long a = v[e], b = v[e | j];
        if ((a > b) == up) {
          v[e] = b;
          v[e | j] = a;
        }
      }
    }
  } else {
    const int lj = j / E;   // lane distance
#pragma unroll
    for (int e = 0; e < E; ++e) {
      const unsigned long long a = v[e];
      const uint32_t plo = __shfl_xor_sync(0xffffffffu, (uint32_t)a, lj);
      const uint32_t phi = __shfl_xor_sync(0xffffffffu, (uint32_t)(a >> 32), lj);
      const unsigned long long b = ((unsigned long long)phi << 32) | plo;
      const int g = g0 + e;
      const bool keep_min = ((g & j) == 0) == ((g & k) == 0);
      v[e] = keep_min ? (a < b ? a : b) : (a > b ? a : b);
    }
  }
}

// One compare-exchange step (k, j) of the bitonic network on keys[0..npad) in shared memory, by the whole CTA; ends with
// a barrier
__device__ inline void bitonic_smem_step(unsigned long long* keys, int npad, int k, int j) {
  for (int t = threadIdx.x; t < (npad >> 1); t += blockDim.x) {
    const int i = 2 * t - (t & (j - 1)), l = i + j;
    const unsigned long long a = keys[i], b = keys[l];
    if ((a > b) == ((i & k) == 0)) {
      keys[i] = b;
      keys[l] = a;
    }
  }
  __syncthreads();
}

template <int E>
__device__ inline void bitonic_sort_reg(unsigned long long* keys, int npad) {
  // npad == E * blockDim.x.  Stages with partner distance >= 32*E go through shared memory, the rest stay in registers.
  const int t = threadIdx.x, g0 = E * t;
  unsigned long long v[E];
#pragma unroll
  for (int e = 0; e < E; ++e) v[e] = keys[g0 + e];
  const int warp_span = 32 * E;
  // k <= warp_span: entirely inside a warp
  for (int k = 2; k <= warp_span; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) bitonic_reg_step<E>(v, k, j, g0);
  for (int k = warp_span * 2; k <= npad; k <<= 1) {
#pragma unroll
    for (int e = 0; e < E; ++e) keys[g0 + e] = v[e];
    __syncthreads();
    for (int j = k >> 1; j >= warp_span; j >>= 1) bitonic_smem_step(keys, npad, k, j);
#pragma unroll
    for (int e = 0; e < E; ++e) v[e] = keys[g0 + e];
    for (int j = warp_span >> 1; j > 0; j >>= 1) bitonic_reg_step<E>(v, k, j, g0);
  }
#pragma unroll
  for (int e = 0; e < E; ++e) keys[g0 + e] = v[e];
  __syncthreads();
}

// keys[0..npad) ascending.  Called by the whole CTA (blockDim.x == kNmsThreads).
__device__ inline void bitonic_sort(unsigned long long* keys, int npad) {
  if (npad == 2 * kNmsThreads) return bitonic_sort_reg<2>(keys, npad);
  if (npad == 4 * kNmsThreads) return bitonic_sort_reg<4>(keys, npad);
  if (npad == 8 * kNmsThreads) return bitonic_sort_reg<8>(keys, npad);
  for (int k = 2; k <= npad; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) bitonic_smem_step(keys, npad, k, j);
}

// The prologue of every NMS kernel: keys[0..n) hold sort_key of the rows and are visible to the CTA.  Pads the keys to
// npad, sorts them and fills s.box[r] = box_of(row_of(s, r)) for every sorted rank r < n.
template <class BoxFn>
__device__ inline void sort_and_gather(const NmsSmem& s, int n, BoxFn box_of) {
  const int npad = next_pow2(max(n, 64));
  for (int i = n + threadIdx.x; i < npad; i += blockDim.x) s.keys[i] = ~0ull;
  __syncthreads();
  bitonic_sort(s.keys, npad);
  for (int r = threadIdx.x; r < n; r += blockDim.x) s.box[r] = box_of(row_of(s, r));
  __syncthreads();
}

// barrier over the CTA (S == 1) or over the whole cluster, with release / acquire of shared-memory writes
__device__ __forceinline__ void sync_group(int S) {
  if (S > 1) tc::cluster_sync();
  else __syncthreads();
}
__device__ __forceinline__ void st_cluster_u32(uint32_t cluster_addr, uint32_t v) {
  asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(cluster_addr), "r"(v) : "memory");
}

// Greedy sweep over s.box[0..n) (sorted).  score_of_rank(r) gives the score of sorted rank r.
// Stops early once `limit` survivors exist and (if keep_ties) no later box can tie the limit-th score.
// S = CTAs per problem (cluster size), rank = this CTA's rank in the cluster: every CTA calls with identical data and
// gets the same survivor list in s.kept; the return value is its length.
//
// Per pair of chunks: [resolve the first: one warp] sync [bit matrix of the second + its boxes against the first one's
// survivors: all warps] sync [resolve the second: one warp] sync [bit matrix of the next pair's first chunk + suppression
// of later boxes by the pair's survivors: all warps] sync [exchange of the next pair's suppression words: cluster only].  A warp that runs alone is latency bound (~5 cycles
// per dependent instruction), so the resolve step works on 32-bit halves and everything that does not depend on it is
// moved into the all-warps phase.
template <typename ScoreFn>
__device__ inline int greedy_sweep(const NmsSmem& s, int n, float thr_f, int limit, bool keep_ties, ScoreFn score_of_rank,
                                   const int S, const int rank) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nwords = (n + 31) >> 5;
  const int nchunks = (n + kChunk - 1) / kChunk;
  PROF_DECL;
  for (int w = tid; w < nwords + 4; w += blockDim.x) s.suppressed[w] = 0;
  if (tid < 4) s.chunk_sup[tid] = 0;  // pair 0 (parity 0) starts with nothing suppressed; parity 1 is always pushed
  // this CTA's boxes: ranks j whose word (j >> 5) is congruent to `rank` modulo S; all alive at the start
  for (int q = tid;; q += blockDim.x) {
    const int j = (rank + (q >> 5) * S) * 32 + (q & 31);
    if (j >= n) break;      // (only the last word of the list is partial, so the valid q form a prefix)
    s.alist_top[-q] = (uint16_t)j;
  }
  if (tid == 0) {
    const int full_words = n >> 5, tail = n & 31;      // words 0..full_words-1 are complete
    int my_n = (full_words > rank ? (full_words - rank + S - 1) / S : 0) * 32;
    if (tail && full_words % S == rank) my_n += tail;
    s.scalars[0] = 0;  // kept count
    s.scalars[1] = 0;
    s.scalars[3] = my_n;
    s.scalars[4] = 0;
  }
  // IoU bit matrix of chunk c2 by column into buffer (c2 & 1): warp w handles columns 2w and 2w+1, lanes are the rows
  // i < j.  Columns already known to be suppressed are skipped (their mask is never looked at).
  auto build_colmask = [&](int c2) {
    const int base2 = c2 * kChunk, m2 = min(kChunk, n - base2);
    uint32_t* clo = s.colmask + (c2 & 1) * 128;
    uint32_t* chi = clo + 64;
#pragma unroll
    for (int rr = 0; rr < 2; ++rr) {
      const int j = warp * 2 + rr;
      unsigned lo = 0, hi = 0;
      if (j < m2 && !((s.suppressed[(base2 + j) >> 5] >> ((base2 + j) & 31)) & 1u)) {
        const float4 bj = s.box[base2 + j];
        const float aj = box_area(bj);
        bool p0 = false, p1 = false;
        if (lane < j) {
          const float4 bi = s.box[base2 + lane];
          p0 = iou_exceeds(bi, box_area(bi), bj, aj, thr_f);
        }
        lo = __ballot_sync(0xffffffffu, p0);
        if (j > 32) {
          if (lane + 32 < j) {
            const float4 bi = s.box[base2 + lane + 32];
            p1 = iou_exceeds(bi, box_area(bi), bj, aj, thr_f);
          }
          hi = __ballot_sync(0xffffffffu, p1);
        }
      }
      if (lane == 0) {
        clo[j] = lo;
        chi[j] = hi;
      }
    }
  };
  __syncthreads();
  build_colmask(0);
  sync_group(S);  // also: every CTA of the cluster is running before anyone writes into a peer's shared memory
  // 2. resolution of chunk c by one warp: fixed point of kept_j = alive_j && !(colmask_j & kept), 32-bit halves.  The
  //    chunk's survivors are appended to s.kept and to the pair's survivor boxes from slot `kofs` on.  (warp 0 only)
  auto resolve = [&](int c, uint32_t suplo, uint32_t suphi, int kofs) {
    const int base = c * kChunk;
    const int m = min(kChunk, n - base);
    const uint32_t validlo = m >= 32 ? 0xffffffffu : ((1u << m) - 1u);
    const uint32_t validhi = m == 64 ? 0xffffffffu : (m > 32 ? ((1u << (m - 32)) - 1u) : 0u);
    const uint32_t alo = validlo & ~suplo, ahi = validhi & ~suphi;
    const uint32_t* clo = s.colmask + (c & 1) * 128;
    const uint32_t c0 = clo[lane], c1l = clo[lane + 32], c1h = clo[64 + lane + 32];
    const bool a0 = (alo >> lane) & 1u, a1 = (ahi >> lane) & 1u;
    uint32_t klo = alo, khi = ahi;
    for (int it = 0; it < kChunk; ++it) {
      const uint32_t nlo = __ballot_sync(0xffffffffu, a0 && !(c0 & klo));
      const uint32_t nhi = __ballot_sync(0xffffffffu, a1 && !((c1l & klo) | (c1h & khi)));
      PROF_CNT(10, 1);
      if (nlo == klo && nhi == khi) break;
      klo = nlo;
      khi = nhi;
    }
    int cnt = s.scalars[0];
    const uint32_t lt = (1u << lane) - 1u;
    const int nklo = __popc(klo);
    if ((klo >> lane) & 1u) {
      const int pos = __popc(klo & lt);
      const float4 b = s.box[base + lane];
      s.kept[cnt + pos] = (uint16_t)(base + lane);
      s.kbox[kofs + pos] = b;
      s.karea[kofs + pos] = box_area(b);
    }
    if ((khi >> lane) & 1u) {
      const int pos = nklo + __popc(khi & lt);
      const float4 b = s.box[base + lane + 32];
      s.kept[cnt + pos] = (uint16_t)(base + lane + 32);
      s.kbox[kofs + pos] = b;
      s.karea[kofs + pos] = box_area(b);
    }
    const int nk = nklo + __popc(khi);
    cnt += nk;
    __syncwarp();
    if (lane == 0) {
      s.scalars[0] = cnt;
      s.scalars[2] = kofs + nk;   // survivors of the pair so far
      // early stop: the top-`limit` survivors are decided
      int stop = 0;
      if (limit > 0 && cnt >= limit && base + kChunk < n) {
        if (!keep_ties) {
          stop = 1;
        } else {
          float sl = score_of_rank(s.kept[limit - 1]);
          if (score_of_rank(base + kChunk) < sl) stop = 1;
        }
      }
      s.scalars[1] = stop;
    }
  };
  // Chunks are taken in PAIRS: the second chunk of a pair gets the first one's suppression from a direct 64 x nk test
  // (two boxes per warp, redundantly in every CTA of a cluster), so the expensive pass over all later boxes - whose cost
  // is mostly its fixed per-warp skeleton, see profiles/r2_ncu_summary.md - runs once per 128 candidates.
  for (int c = 0; c < nchunks; c += 2) {
    const int base = c * kChunk;
    const int par = (c >> 1) & 1;
    uint32_t* csup = s.chunk_sup + par * 6;   // [0..1] chunk c, [2..3] chunk c + 1, [4..5] cross words of chunk c + 1
    PROF_T(t2);
    if (warp == 0) {
      if (lane < 2) csup[4 + lane] = 0;
      resolve(c, S > 1 ? csup[0] : s.suppressed[base >> 5], S > 1 ? csup[1] : s.suppressed[(base >> 5) + 1], 0);
      if (lane == 0) s.scalars[4] = 0;   // survivor counter of the pair's compaction pass
    }
    __syncthreads();
    if (s.scalars[1] || c + 1 == nchunks) break;  // same decision in every CTA of the cluster (identical data)
    {
      // 1'. bit matrix of the pair's second chunk, and its boxes against the first chunk's survivors
      build_colmask(c + 1);
      const int nk0 = s.scalars[2];
      const int base1 = base + kChunk, m1 = min(kChunk, n - base1);
#pragma unroll
      for (int rr = 0; rr < 2; ++rr) {
        const int j = warp * 2 + rr;
        bool hit = false;
        if (j < m1) {
          const float4 bj = s.box[base1 + j];
          const float aj = box_area(bj);
          for (int k = lane; k < nk0; k += 32) hit = hit || iou_exceeds(s.kbox[k], s.karea[k], bj, aj, thr_f);
        }
        if (__any_sync(0xffffffffu, hit) && lane == 0) atomicOr(&csup[4 + (j >> 5)], 1u << (j & 31));
      }
    }
    __syncthreads();
    if (warp == 0) {
      const int w1 = (base + kChunk) >> 5;
      resolve(c + 1, (S > 1 ? csup[2] : s.suppressed[w1]) | csup[4], (S > 1 ? csup[3] : s.suppressed[w1 + 1]) | csup[5], s.scalars[2]);
    }
    __syncthreads();
    PROF_ADD(2, t2);
    PROF_T(t3);
    if (s.scalars[1] || c + 2 >= nchunks) break;
    const int nk = s.scalars[2];
    // 1'. the next pair's first bit matrix (independent of the suppression state, so it shares this all-warps phase)
    build_colmask(c + 2);
    PROF_ADD(14, t3);
    // 3. survivors of this pair suppress later boxes.  This CTA owns the words w with w % S == rank and keeps a list
    //    of its boxes that are alive and beyond the resolved chunks; one pass tests every listed box against the
    //    pair's survivors (G lanes share a box and split the survivor list) and compacts the list in place, so the
    //    work follows the number of boxes still alive, not the number of candidates.
    if (nk > 0) {   // (a pair without survivors changes nothing; its own entries are dropped by the next pass)
      const int lim = base + 2 * kChunk;
      const int nal = s.scalars[3];
      int lg = 0;
      while (lg < 5 && (nal << (lg + 1)) <= kNmsThreads) ++lg;
      const int G = 1 << lg, per_pass = kNmsThreads >> lg;
      const int sub = tid & (G - 1), grp = tid >> lg;
      const unsigned gmask = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << (lane & ~(G - 1)));
      // suppression test of list entry j against the pair's survivors (the G lanes of a group split them)
      auto test = [&](int j, bool live) {
        bool hit = false;
        if (live) {
          const float4 bj = s.box[j];
          const float aj = box_area(bj);
          for (int k = sub; k < nk; k += G) {
            if (iou_exceeds(s.kbox[k], s.karea[k], bj, aj, thr_f)) {
              hit = true;
              break;
            }
          }
        }
        return (__ballot_sync(0xffffffffu, hit) & gmask) != 0u;
      };
      if (nal <= kPreRead * per_pass) {
        // The usual case: every thread fetches its entries of all passes first, so after ONE barrier the compaction may
        // write anywhere in the list; a warp then runs its passes back to back and claims its output slots with one
        // atomic (the order of the list is irrelevant: it is a set).
        int js[kPreRead];
#pragma unroll
        for (int q = 0; q < kPreRead; ++q) {
          const int e = q * per_pass + grp;
          js[q] = e < nal ? (int)s.alist_top[-e] : -1;
        }
        __syncthreads();
        unsigned survbits = 0;   // bit q: entry q of this thread survives (set in the group's first lane only)
        int wtot = 0;
        const int wfirst = (warp * 32) >> lg;   // this warp's first entry of pass 0: a warp without entries skips the pass
#pragma unroll
        for (int q = 0; q < kPreRead; ++q) {
          if (q * per_pass + wfirst < nal) {   // uniform over the warp
            const int j = js[q];
            const bool live = j >= lim;
            const bool dead = test(j, live);
            if (live && dead && sub == 0) atomicOr(&s.suppressed[j >> 5], 1u << (j & 31));
            const bool surv = live && !dead && sub == 0;
            survbits |= (surv ? 1u : 0u) << q;
            wtot += __popc(__ballot_sync(0xffffffffu, surv));
          }
        }
        int wbase = 0;
        if (lane == 0 && wtot) wbase = atomicAdd(&s.scalars[4], wtot);
        wbase = __shfl_sync(0xffffffffu, wbase, 0);
#pragma unroll
        for (int q = 0; q < kPreRead; ++q) {
          if (q * per_pass + wfirst < nal) {
            const bool surv = (survbits >> q) & 1u;
            const unsigned sm = __ballot_sync(0xffffffffu, surv);
            if (surv) s.alist_top[-(wbase + __popc(sm & ((1u << lane) - 1u)))] = (uint16_t)js[q];
            wbase += __popc(sm);
          }
        }
      } else {
        for (int e0 = 0; e0 < nal; e0 += per_pass) {
          const int e = e0 + grp;
          const int j = e < nal ? (int)s.alist_top[-e] : -1;
          const bool live = j >= lim;
          const bool dead = test(j, live);
          if (live && dead && sub == 0) atomicOr(&s.suppressed[j >> 5], 1u << (j & 31));
          const bool surv = live && !dead && sub == 0;
          const unsigned sm = __ballot_sync(0xffffffffu, surv);
          int wbase = 0;
          if (lane == 0 && sm) wbase = atomicAdd(&s.scalars[4], __popc(sm));
          wbase = __shfl_sync(0xffffffffu, wbase, 0);
          __syncthreads();  // every entry of this pass has been read; the writes stay below the next pass's entries
          if (surv) s.alist_top[-(wbase + __popc(sm & ((1u << lane) - 1u)))] = (uint16_t)j;
        }
      }
    }
    PROF_ADD(15, t3);
    __syncthreads();
    PROF_ADD(3, t3);
    PROF_T(t4);
    if (tid == 0 && nk > 0) s.scalars[3] = s.scalars[4];
    if (S > 1) {
      // hand the next pair's four suppression words to every CTA (parity-alternating slots: the peers may still be
      // reading this pair's slots)
      const int first_word = (base + 2 * kChunk) >> 5;
      if (tid < 4 * S) {
        const int wsel = tid / S, dst = tid - wsel * S;
        const int w = first_word + wsel;
        if (w % S == rank)   // (zero beyond the list: the array has spare words)
          st_cluster_u32(tc::map_to_cta(tc::smem_u32(&s.chunk_sup[(par ^ 1) * 6 + wsel]), (uint32_t)dst), s.suppressed[w]);
      }
      tc::cluster_sync();
    }
    PROF_ADD(4, t4);
    PROF_ADD(5, t2);
    PROF_CNT(9, 1);
  }
  __syncthreads();
  PROF_FLUSH(0, 6);
  PROF_FLUSH(9, 16);
  return s.scalars[0];
}

// ------------------------------------------------------------------------------------------------
// N0: proposals
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kNmsThreads, 1)
nms_proposals_kernel(const float* __restrict__ boxes, const float* __restrict__ scores, const int32_t* __restrict__ count,
                     int cand_cap, float thr_f, int post_topk, int roi_cap, int64_t* __restrict__ keep,
                     float* __restrict__ out_boxes, float* __restrict__ out_scores, int32_t* __restrict__ out_count,
                     uint32_t* __restrict__ status, const int S) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int p = blockIdx.x / S, rank = blockIdx.x - p * S;   // S consecutive CTAs = one cluster = one problem
  const int tid = threadIdx.x;
  int n = count ? count[p] : cand_cap;
  n = max(0, min(n, cand_cap));
  PROF_DECL;
  PROF_T(tk0);
  NmsSmem s = carve(smem_raw, cand_cap);
  const float* pb = boxes + (size_t)p * cand_cap * 4;
  const float* ps = scores + (size_t)p * cand_cap;
  for (int i = tid; i < n; i += blockDim.x) s.keys[i] = sort_key(ps[i], i);
  sort_and_gather(s, n, [&](int row) { return *reinterpret_cast<const float4*>(pb + (size_t)row * 4); });
  // row_of written out: through the call this kernel compiles differently (6344 instead of 6328 SASS instructions,
  // CUDA 12.9), and the one-warp resolve that reads this score was 1 % slower (B200, 1000 W)
  auto score_of_rank = [&](int r) { return ps[(int)(s.keys[r] & 0xffffffffu)]; };
  PROF_ADD(6, tk0);
  PROF_T(tk1);
  int kept = greedy_sweep(s, n, thr_f, post_topk, true, score_of_rank, S, rank);
  PROF_ADD(7, tk1);
  PROF_CNT(8, kept);
  PROF_FLUSH(6, 9);
  int m = kept;
  if (post_topk > 0 && kept > post_topk) {
    // keep every survivor whose score >= the post_topk-th best (fsod_rpn.py:1198-1206)
    float sl = score_of_rank(s.kept[post_topk - 1]);
    if (tid == 0) s.scalars[4] = kept;
    __syncthreads();
    for (int i = post_topk + tid; i < kept; i += blockDim.x) {
      // first position whose score drops below sl
      bool below = score_of_rank(s.kept[i]) < sl;
      bool prev_below = score_of_rank(s.kept[i - 1]) < sl;
      if (below && !prev_below) s.scalars[4] = i;
    }
    __syncthreads();
    m = s.scalars[4];
  }
  if (rank != 0) return;   // every CTA of the cluster holds the same result; the first one writes it
  if (m > roi_cap) {
    if (tid == 0) atomicOr(status, FOD_STATUS_PROPOSAL_OVERFLOW);
    m = roi_cap;
  }
  for (int i = tid; i < m; i += blockDim.x) {
    int r = s.kept[i];
    int idx = row_of(s, r);
    keep[(size_t)p * roi_cap + i] = idx;
    *reinterpret_cast<float4*>(out_boxes + ((size_t)p * roi_cap + i) * 4) = s.box[r];
    out_scores[(size_t)p * roi_cap + i] = ps[idx];
  }
  if (tid == 0) out_count[p] = m;
}

// ------------------------------------------------------------------------------------------------
// R4 / N1 / O1: final class-wise NMS + postprocess, one CTA per image
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float4 clip_box(float4 b, float w, float h) {
  return make_float4(fminf(fmaxf(b.x, 0.f), w), fminf(fmaxf(b.y, 0.f), h), fminf(fmaxf(b.z, 0.f), w),
                     fminf(fmaxf(b.w, 0.f), h));
}

__device__ __forceinline__ float max_coord(float4 b) { return fmaxf(fmaxf(b.x, b.y), fmaxf(b.z, b.w)); }

// Class offset step of torchvision's coordinate trick (boxes.py batched_nms): boxes.max() + 1 over the CTA, from each
// thread's maximum over its boxes.  sh: __shared__ float[32]
__device__ inline float coord_step(float lmax, float* sh) {
  return __fadd_rn(block_reduce(lmax, sh, [](float a, float b) { return fmaxf(a, b); }), 1.0f);
}

// box + cls * coord_step on every coordinate, each operation separately rounded like the fp32 tensor ops it restates
__device__ __forceinline__ float4 offset_box(float4 b, float cls, float coord_step) {
  const float off = __fmul_rn(cls, coord_step);
  return make_float4(__fadd_rn(b.x, off), __fadd_rn(b.y, off), __fadd_rn(b.z, off), __fadd_rn(b.w, off));
}

__global__ void __launch_bounds__(kNmsThreads, 1)
final_detect_kernel(const float* __restrict__ det_boxes, const float* __restrict__ det_scores,
                    const int32_t* __restrict__ roi_count, int C, int roi_cap, int ncap, float score_thresh, float thr_f,
                    int max_det, const int32_t* __restrict__ image_hw, const int32_t* __restrict__ out_hw,
                    float* __restrict__ out_boxes, float* __restrict__ out_scores, int64_t* __restrict__ out_classes,
                    int64_t* __restrict__ out_rows, int32_t* __restrict__ out_count, uint32_t* __restrict__ status,
                    const int S) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ int sh_scan[33];
  __shared__ float sh_max[32];
  const int b = blockIdx.x / S, rank = blockIdx.x - b * S;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  NmsSmem s = carve(smem_raw, ncap);
  const size_t img_row0 = (size_t)b * C * roi_cap;
  const float* ib = det_boxes + img_row0 * 4;
  const float* is = det_scores + img_row0;
  const int total_rows = C * roi_cap;
  const int ih = image_hw[b * 2], iw = image_hw[b * 2 + 1];
  const float fw = (float)iw, fh = (float)ih;
  // 1. compaction of valid rows in class-major order (d2 fast_rcnn.py:137-155)
  int n = 0;
  float lmax = -INFINITY;
  for (int start = 0; start < total_rows; start += blockDim.x) {
    int row = start + tid;
    bool ok = false;
    float sc = 0.f;
    if (row < total_rows) {
      int c = row / roi_cap, r = row - c * roi_cap;
      int cnt = roi_count ? min(roi_count[b * C + c], roi_cap) : roi_cap;
      if (r < cnt) {
        sc = is[row];
        float4 bx = *reinterpret_cast<const float4*>(ib + (size_t)row * 4);
        bool fin = isfinite(bx.x) && isfinite(bx.y) && isfinite(bx.z) && isfinite(bx.w) && isfinite(sc);
        ok = fin && (sc > score_thresh);
        if (ok) lmax = fmaxf(lmax, max_coord(clip_box(bx, fw, fh)));
      }
    }
    int tot;
    const int i = n + block_exclusive_scan(ok ? 1 : 0, sh_scan, tot);
    if (ok && i < ncap) s.keys[i] = sort_key(sc, row);
    n += tot;
  }
  if (n > ncap) {
    if (tid == 0 && rank == 0) atomicOr(status, FOD_STATUS_DET_OVERFLOW);
    n = ncap;
  }
  // 2. max coordinate (torchvision boxes.py batched_nms: boxes.max()); 3. sort, gather clipped class-offset boxes
  const float step = coord_step(lmax, sh_max);
  sort_and_gather(s, n, [&](int row) {
    const float4 bx = clip_box(*reinterpret_cast<const float4*>(ib + (size_t)row * 4), fw, fh);
    return offset_box(bx, (float)(row / roi_cap), step);
  });
  auto score_of_rank = [&](int r) { return is[row_of(s, r)]; };
  int kept = greedy_sweep(s, n, thr_f, max_det, false, score_of_rank, S, rank);
  if (max_det >= 0) kept = min(kept, max_det);
  // 4. detector_postprocess on the survivors (d2 postprocessing.py:42-59), order preserved.
  const int oh = out_hw ? out_hw[b * 2] : ih, ow = out_hw ? out_hw[b * 2 + 1] : iw;
  const float sx = (float)((double)ow / (double)iw), sy = (float)((double)oh / (double)ih);
  if (warp == 0 && rank == 0) {
    int written = 0;
    for (int i0 = 0; i0 < kept; i0 += 32) {
      int i = i0 + lane;
      bool ok = false;
      float4 bx = make_float4(0, 0, 0, 0);
      int row = 0;
      if (i < kept) {
        row = row_of(s, s.kept[i]);
        bx = clip_box(*reinterpret_cast<const float4*>(ib + (size_t)row * 4), fw, fh);
        bx.x = fminf(fmaxf(__fmul_rn(bx.x, sx), 0.f), (float)ow);
        bx.z = fminf(fmaxf(__fmul_rn(bx.z, sx), 0.f), (float)ow);
        bx.y = fminf(fmaxf(__fmul_rn(bx.y, sy), 0.f), (float)oh);
        bx.w = fminf(fmaxf(__fmul_rn(bx.w, sy), 0.f), (float)oh);
        ok = (__fsub_rn(bx.z, bx.x) > 0.f) && (__fsub_rn(bx.w, bx.y) > 0.f);
      }
      unsigned m = __ballot_sync(0xffffffffu, ok);
      if (ok) {
        int o = written + __popc(m & ((1u << lane) - 1u));
        size_t base = (size_t)b * max_det + o;
        *reinterpret_cast<float4*>(out_boxes + base * 4) = bx;
        out_scores[base] = is[row];
        out_classes[base] = row / roi_cap;
        if (out_rows) out_rows[base] = row;
      }
      written += __popc(m);
    }
    if (lane == 0) out_count[b] = written;
  }
}

// Generic single-problem batched_nms (operator boundary).
__global__ void __launch_bounds__(kNmsThreads, 1)
batched_nms_kernel(const float* __restrict__ boxes, const float* __restrict__ scores, const int64_t* __restrict__ idxs,
                   int n, float thr_f, int64_t* __restrict__ keep, int32_t* __restrict__ keep_count, const int S) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ float sh_max[32];
  const int tid = threadIdx.x;
  const int rank = blockIdx.x;   // one problem = one cluster of S CTAs
  NmsSmem s = carve(smem_raw, n);
  float lmax = -INFINITY;
  for (int i = tid; i < n; i += blockDim.x) {
    s.keys[i] = sort_key(scores[i], i);
    lmax = fmaxf(lmax, max_coord(*reinterpret_cast<const float4*>(boxes + (size_t)i * 4)));
  }
  const float step = coord_step(lmax, sh_max);
  sort_and_gather(s, n, [&](int i) {
    const float4 bx = *reinterpret_cast<const float4*>(boxes + (size_t)i * 4);
    return idxs ? offset_box(bx, (float)idxs[i], step) : bx;
  });
  auto score_of_rank = [&](int r) { return scores[row_of(s, r)]; };
  int kept = greedy_sweep(s, n, thr_f, 0, false, score_of_rank, S, rank);
  if (rank != 0) return;
  for (int i = tid; i < kept; i += blockDim.x) keep[i] = row_of(s, s.kept[i]);
  if (tid == 0) *keep_count = kept;
}

// ------------------------------------------------------------------------------------------------
// N2: RPN proposals (find_top_rpn_proposals, d2!/modeling/proposal_generator/proposal_utils.py:19-119)
//   rpn_keys_kernel   : the selection key of every anchor of every level (wide, over all SMs)
//   rpn_select_kernel : one CTA per (problem, level): radix select of the level's top k, then the k anchors in ascending
//                       anchor order are decoded, filtered and clipped into the level's k candidate slots
//   rpn_nms_kernel    : one cluster per problem: the surviving candidates through sort_and_gather + greedy_sweep
// ------------------------------------------------------------------------------------------------
struct RpnParams {
  const float* map[FOD_MAX_LEVELS];       // [P][H][W][ps]: logit of anchor a in channel a, delta j in channel A + 4a + j
  const float* anchors[FOD_MAX_LEVELS];   // [H*W*A][4]
  const int32_t* image_hw;                // [P][2]
  int pixels[FOD_MAX_LEVELS], ps[FOD_MAX_LEVELS];
  int key_off[FOD_MAX_LEVELS + 1];        // first key of level l in a problem's key row; key_off[L] = anchors per problem
  int sel_off[FOD_MAX_LEVELS + 1];        // first candidate slot of level l; sel_off[L] = candidate slots per problem
  int num_levels, A, pre_topk;
  float inv_w[4];                         // 1 / BBOX_REG_WEIGHTS, rounded to fp32 like ATen's tensor / python-float
  float scale_clamp;                      // log(1000 / 16) as fp32 (box_regression.py _DEFAULT_SCALE_CLAMP)
  float min_size;
};

// Selection key: ascending key = ascending logit in the order of torch.sort, i.e. -0.0 equal to +0.0 and every NaN
// above +inf
__device__ __forceinline__ uint32_t rpn_key(float v) {
  if (isnan(v)) return 0xffffffffu;
  return float_to_ordered(v == 0.f ? 0.f : v);
}

// level of entry i of a row laid out by `off` (constant indices only: the parameter array stays in the constant bank)
__device__ __forceinline__ int rpn_level_of(const int (&off)[FOD_MAX_LEVELS + 1], int L, int i) {
  int l = 0;
#pragma unroll
  for (int j = 1; j < FOD_MAX_LEVELS; ++j) l += (j < L && i >= off[j]) ? 1 : 0;
  return l;
}

__global__ void __launch_bounds__(256) rpn_keys_kernel(RpnParams prm, uint32_t* __restrict__ keys) {
  const int idx = blockIdx.x * 256 + threadIdx.x, p = blockIdx.y;
  const int total = prm.key_off[prm.num_levels];
  if (idx >= total) return;
  const int l = rpn_level_of(prm.key_off, prm.num_levels, idx);
  const int i = idx - prm.key_off[l], pix = i / prm.A, a = i - pix * prm.A;
  const float v = __ldg(prm.map[l] + ((size_t)p * prm.pixels[l] + pix) * prm.ps[l] + a);
  keys[(size_t)p * total + idx] = rpn_key(v);
}

// Box2BoxTransform.apply_deltas (box_regression.py:77-115) of one anchor, with the roundings of its separate fp32 ATen ops
__device__ __forceinline__ float4 rpn_decode(float4 an, float d0, float d1, float d2, float d3, const float* inv_w,
                                             float clamp) {
  const float w = __fsub_rn(an.z, an.x), h = __fsub_rn(an.w, an.y);
  const float cx = __fadd_rn(an.x, __fmul_rn(0.5f, w)), cy = __fadd_rn(an.y, __fmul_rn(0.5f, h));
  const float dx = __fmul_rn(d0, inv_w[0]), dy = __fmul_rn(d1, inv_w[1]);
  float dw = __fmul_rn(d2, inv_w[2]), dh = __fmul_rn(d3, inv_w[3]);
  dw = isnan(dw) ? dw : fminf(dw, clamp);      // torch.clamp(max=) lets NaN through
  dh = isnan(dh) ? dh : fminf(dh, clamp);
  const float pcx = __fadd_rn(__fmul_rn(dx, w), cx), pcy = __fadd_rn(__fmul_rn(dy, h), cy);
  const float pw = __fmul_rn(expf(dw), w), ph = __fmul_rn(expf(dh), h);
  const float hw = __fmul_rn(0.5f, pw), hh = __fmul_rn(0.5f, ph);
  return make_float4(__fsub_rn(pcx, hw), __fsub_rn(pcy, hh), __fadd_rn(pcx, hw), __fadd_rn(pcy, hh));
}

// A candidate slot whose logit is NaN holds a dropped row (non-finite box or logit, or empty after the clip)
__global__ void __launch_bounds__(1024, 1)
rpn_select_kernel(RpnParams prm, const uint32_t* __restrict__ keys, float4* __restrict__ cand_box,
                  float* __restrict__ cand_logit) {
  __shared__ int hist[32][256];
  __shared__ int scan_sh[33];
  __shared__ int sh[2];
  const int L = prm.num_levels;
  const int p = blockIdx.x / L, l = blockIdx.x - p * L;
  const int tid = threadIdx.x;
  const int A = prm.A, n = prm.key_off[l + 1] - prm.key_off[l], k = min(n, prm.pre_topk);
  const uint32_t* lk = keys + (size_t)p * prm.key_off[L] + prm.key_off[l];
  // keys > T, plus the first `need` keys == T (a stable descending sort takes the lowest anchor indices first)
  uint32_t T = 0u;
  int need = 0;
  if (n > k) T = radix_select([&](int i) { return __ldg(lk + i); }, n, k, hist, sh, need);
  const float fh = (float)prm.image_hw[2 * p], fw = (float)prm.image_hw[2 * p + 1];
  const float* map = prm.map[l] + (size_t)p * prm.pixels[l] * prm.ps[l];
  const float4* anc = reinterpret_cast<const float4*>(prm.anchors[l]);
  float4* ob = cand_box + (size_t)p * prm.sel_off[L] + prm.sel_off[l];
  float* ol = cand_logit + (size_t)p * prm.sel_off[L] + prm.sel_off[l];
  int gt_before = 0, eq_before = 0;
  for (int i0 = 0; i0 < n; i0 += 1024) {
    const int i = i0 + tid;
    const uint32_t key = i < n ? __ldg(lk + i) : 0u;
    const int is_gt = i < n && key > T, is_eq = i < n && need > 0 && key == T;
    int tot;   // both counts of the 1024 keys of this step in one scan (each <= 1024)
    const int excl = block_exclusive_scan(is_gt | (is_eq << 16), scan_sh, tot);
    const int gt_pos = gt_before + (excl & 0xffff), eq_pos = eq_before + (excl >> 16);
    if (is_gt || (is_eq && eq_pos < need)) {
      const int o = gt_pos + min(eq_pos, need);
      const int pix = i / A, a = i - pix * A;
      const float* px = map + (size_t)pix * prm.ps[l];
      const float logit = __ldg(px + a);
      const float* d = px + A + 4 * a;
      const float4 b = rpn_decode(__ldg(anc + i), __ldg(d), __ldg(d + 1), __ldg(d + 2), __ldg(d + 3), prm.inv_w,
                                     prm.scale_clamp);
      bool ok = isfinite(b.x) && isfinite(b.y) && isfinite(b.z) && isfinite(b.w) && isfinite(logit);
      const float4 c = clip_box(b, fw, fh);                                 // Boxes.clip
      ok = ok && __fsub_rn(c.z, c.x) > prm.min_size && __fsub_rn(c.w, c.y) > prm.min_size;   // Boxes.nonempty
      ob[o] = c;
      ol[o] = ok ? logit : __int_as_float(0x7fffffff);
    }
    gt_before += tot & 0xffff;
    eq_before += tot >> 16;
  }
}

__global__ void __launch_bounds__(kNmsThreads, 1)
rpn_nms_kernel(RpnParams prm, const float4* __restrict__ cand_box, const float* __restrict__ cand_logit, float thr_f,
               int post_topk, float* __restrict__ out_boxes, float* __restrict__ out_logits, int32_t* __restrict__ out_count,
               const int S) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ float sh_max[32];
  const int L = prm.num_levels, cap = prm.sel_off[L];
  const int p = blockIdx.x / S, rank = blockIdx.x - p * S;
  const int tid = threadIdx.x;
  NmsSmem s = carve(smem_raw, cap);
  const float4* pb = cand_box + (size_t)p * cap;
  const float* pl = cand_logit + (size_t)p * cap;
  if (tid == 0) s.scalars[0] = 0;
  __syncthreads();
  // the surviving candidates as sort keys (any order: the slot index breaks ties), and their largest coordinate
  float lmax = -INFINITY;
  for (int i = tid; i < cap; i += blockDim.x) {
    const float sc = pl[i];
    if (!isnan(sc)) {
      s.keys[atomicAdd(&s.scalars[0], 1)] = sort_key(sc, i);
      lmax = fmaxf(lmax, max_coord(pb[i]));
    }
  }
  __syncthreads();
  const int n = s.scalars[0];
  if (n == 0) {   // (the same in every CTA of the cluster)
    if (rank == 0 && tid == 0) out_count[p] = 0;
    return;
  }
  // batched_nms over the levels: torchvision's coordinate trick, as fod_batched_nms with idxs = level
  const float step = L > 1 ? coord_step(lmax, sh_max) : 0.f;
  sort_and_gather(s, n, [&](int i) {
    return L > 1 ? offset_box(pb[i], (float)rpn_level_of(prm.sel_off, L, i), step) : pb[i];
  });
  auto score_of_rank = [&](int r) { return pl[row_of(s, r)]; };
  const int m = min(greedy_sweep(s, n, thr_f, post_topk, false, score_of_rank, S, rank), post_topk);
  if (rank != 0) return;
  for (int i = tid; i < m; i += blockDim.x) {
    const int row = row_of(s, s.kept[i]);
    *reinterpret_cast<float4*>(out_boxes + ((size_t)p * post_topk + i) * 4) = pb[row];
    out_logits[(size_t)p * post_topk + i] = pl[row];
  }
  if (tid == 0) out_count[p] = m;
}

// CTAs per problem: the largest power of two <= kMaxCluster that keeps problems * S within the SM count.
static int pick_cluster(long problems) {
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  int S = 1, smax = kMaxCluster;
  if (const char* e = getenv("FOD_NMS_MAX_CLUSTER")) smax = atoi(e) > 0 ? atoi(e) : smax;   // development knob
  while (S * 2 <= smax && problems * (S * 2) <= sms) S *= 2;
  return S;
}

}  // namespace fod

#ifdef FOD_NMS_PROF
extern "C" int fod_nms_prof(long long* out16, int reset) {
  if (reset) {
    long long z[16] = {0};
    cudaMemcpyToSymbol(fod::g_nms_prof, z, sizeof(z));
  } else {
    cudaMemcpyFromSymbol(out16, fod::g_nms_prof, sizeof(long long) * 16);
  }
  return 0;
}
#endif

using namespace fod;

extern "C" int fod_nms_proposals(const float* boxes, const float* scores, const int32_t* count, int num_problems,
                                 int cand_cap, double iou_thresh, int post_topk, int roi_cap, int64_t* keep,
                                 float* out_boxes, float* out_scores, int32_t* out_count, uint32_t* status,
                                 fod_stream_t stream) {
  FOD_REQUIRE(boxes && scores && keep && out_boxes && out_scores && out_count && status, "fod_nms_proposals: null pointer");
  FOD_REQUIRE(num_problems >= 0 && cand_cap > 0 && roi_cap > 0, "fod_nms_proposals: bad sizes");
  if (cand_cap > FOD_NMS_MAX_BOXES) {
    set_error("fod_nms_proposals: cand_cap %d > %d", cand_cap, FOD_NMS_MAX_BOXES);
    return FOD_ERR_CAPACITY;
  }
  if (num_problems == 0) return FOD_OK;
  float thr_f = iou_threshold_as_float(iou_thresh);
  int S = pick_cluster(num_problems);
  void* args[] = {&boxes, &scores, &count, &cand_cap, &thr_f, &post_topk, &roi_cap, &keep, &out_boxes, &out_scores,
                  &out_count, &status, &S};
  return launch_clusters((const void*)nms_proposals_kernel, args, num_problems, S, kNmsThreads, nms_smem_bytes(cand_cap),
                         stream, "fod_nms_proposals");
}

extern "C" int fod_final_detect(const float* det_boxes, const float* det_scores, const int32_t* roi_count, int batch,
                                int problems_per_image, int roi_cap, float score_thresh, double iou_thresh, int max_det,
                                const int32_t* image_hw, const int32_t* out_hw, float* out_boxes, float* out_scores,
                                int64_t* out_classes, int64_t* out_rows, int32_t* out_count, uint32_t* status,
                                fod_stream_t stream) {
  FOD_REQUIRE(det_boxes && det_scores && image_hw && out_boxes && out_scores && out_classes && out_count && status,
              "fod_final_detect: null pointer");
  FOD_REQUIRE(batch >= 0 && problems_per_image > 0 && roi_cap > 0 && max_det > 0, "fod_final_detect: bad sizes");
  if (batch == 0) return FOD_OK;
  long rows = (long)problems_per_image * roi_cap;
  int ncap = (int)(rows < FOD_NMS_MAX_BOXES ? rows : FOD_NMS_MAX_BOXES);
  float thr_f = iou_threshold_as_float(iou_thresh);
  // rows per image decide how far a problem is spread: a few hundred rows are a handful of chunks, not worth a cluster
  int S = rows > 1024 ? pick_cluster(batch) : 1;
  void* args[] = {&det_boxes, &det_scores, &roi_count, &problems_per_image, &roi_cap, &ncap, &score_thresh, &thr_f,
                  &max_det, &image_hw, &out_hw, &out_boxes, &out_scores, &out_classes, &out_rows, &out_count, &status, &S};
  return launch_clusters((const void*)final_detect_kernel, args, batch, S, kNmsThreads, nms_smem_bytes(ncap), stream,
                         "fod_final_detect");
}

extern "C" int fod_batched_nms(const float* boxes, const float* scores, const int64_t* idxs, int n, double iou_thresh,
                               int64_t* keep, int32_t* keep_count, fod_stream_t stream) {
  FOD_REQUIRE(keep_count, "fod_batched_nms: null keep_count");
  FOD_REQUIRE(n >= 0, "fod_batched_nms: negative n");
  if (n > FOD_NMS_MAX_BOXES) {
    set_error("fod_batched_nms: n %d > %d", n, FOD_NMS_MAX_BOXES);
    return FOD_ERR_CAPACITY;
  }
  if (n == 0) {
    FOD_CUDA_CALL(cudaMemsetAsync(keep_count, 0, sizeof(int32_t), as_stream(stream)));
    return FOD_OK;
  }
  FOD_REQUIRE(boxes && scores && keep, "fod_batched_nms: null pointer");
  float thr_f = iou_threshold_as_float(iou_thresh);
  int S = n > 512 ? pick_cluster(1) : 1;
  void* args[] = {&boxes, &scores, &idxs, &n, &thr_f, &keep, &keep_count, &S};
  return launch_clusters((const void*)batched_nms_kernel, args, 1, S, kNmsThreads, nms_smem_bytes(n), stream,
                         "fod_batched_nms");
}

// Level geometry of fod_rpn_proposals: key and candidate-slot offsets; false if an anchor count overflows int
static bool rpn_geometry(const fod_level_t* levels, int num_levels, int num_anchors, int pre_topk, int* key_off, int* sel_off) {
  long keys = 0, sel = 0;
  for (int l = 0; l < num_levels; ++l) {
    key_off[l] = (int)keys;
    sel_off[l] = (int)sel;
    const long n = (long)levels[l].height * levels[l].width * num_anchors;
    keys += n;
    sel += n < pre_topk ? n : pre_topk;
    if (keys >= (1L << 30)) return false;
  }
  key_off[num_levels] = (int)keys;
  sel_off[num_levels] = (int)sel;
  return true;
}

static size_t align16(size_t b) { return (b + 15) & ~(size_t)15; }

// workspace: candidate boxes [P][slots] float4 | candidate logits [P][slots] | keys [P][anchors] uint32
extern "C" size_t fod_rpn_proposals_workspace_bytes(const fod_level_t* levels, int num_levels, int num_problems,
                                                   int num_anchors, int pre_topk) {
  int key_off[FOD_MAX_LEVELS + 1], sel_off[FOD_MAX_LEVELS + 1];
  if (!levels || num_levels < 1 || num_levels > FOD_MAX_LEVELS || num_problems <= 0 || num_anchors <= 0 || pre_topk <= 0 ||
      !rpn_geometry(levels, num_levels, num_anchors, pre_topk, key_off, sel_off))
    return 0;
  const size_t P = (size_t)num_problems, slots = (size_t)sel_off[num_levels];
  return P * slots * 16 + align16(P * slots * 4) + P * (size_t)key_off[num_levels] * 4;
}

extern "C" int fod_rpn_proposals(const float* const* maps, const int* pixel_stride, const float* const* anchors,
                                 const fod_level_t* levels, int num_levels, int num_problems, int num_anchors,
                                 const int32_t* image_hw, int pre_topk, const float* box_weights, float min_size,
                                 double iou_thresh, int post_topk, float* out_boxes, float* out_logits, int32_t* out_count,
                                 void* workspace, fod_stream_t stream) {
  FOD_REQUIRE(maps && pixel_stride && anchors && levels && image_hw && box_weights && out_boxes && out_logits && out_count &&
                  workspace,
              "fod_rpn_proposals: null pointer");
  FOD_REQUIRE(num_levels >= 1 && num_levels <= FOD_MAX_LEVELS, "fod_rpn_proposals: num_levels %d out of range", num_levels);
  FOD_REQUIRE(num_problems >= 0 && num_anchors > 0 && pre_topk > 0 && post_topk > 0, "fod_rpn_proposals: bad sizes");
  FOD_REQUIRE((reinterpret_cast<uintptr_t>(out_boxes) & 15) == 0 && (reinterpret_cast<uintptr_t>(workspace) & 15) == 0,
              "fod_rpn_proposals: out_boxes and workspace must be 16-byte aligned");
  RpnParams prm = {};
  for (int l = 0; l < num_levels; ++l) {
    FOD_REQUIRE(maps[l] && anchors[l] && (reinterpret_cast<uintptr_t>(anchors[l]) & 15) == 0,
                "fod_rpn_proposals: null or misaligned level pointer");
    FOD_REQUIRE(levels[l].height > 0 && levels[l].width > 0, "fod_rpn_proposals: bad level %d", l);
    FOD_REQUIRE(pixel_stride[l] >= 5 * num_anchors, "fod_rpn_proposals: pixel stride %d < 5 * %d channels at level %d",
                pixel_stride[l], num_anchors, l);
    prm.map[l] = maps[l];
    prm.anchors[l] = anchors[l];
    prm.pixels[l] = levels[l].height * levels[l].width;
    prm.ps[l] = pixel_stride[l];
  }
  if (!rpn_geometry(levels, num_levels, num_anchors, pre_topk, prm.key_off, prm.sel_off)) {
    set_error("fod_rpn_proposals: more than 2^30 anchors per problem");
    return FOD_ERR_CAPACITY;
  }
  const int slots = prm.sel_off[num_levels];
  if (slots > FOD_NMS_MAX_BOXES) {
    set_error("fod_rpn_proposals: %d candidates per problem > %d", slots, FOD_NMS_MAX_BOXES);
    return FOD_ERR_CAPACITY;
  }
  if (num_problems == 0) return FOD_OK;
  prm.image_hw = image_hw;
  prm.num_levels = num_levels;
  prm.A = num_anchors;
  prm.pre_topk = pre_topk;
  for (int j = 0; j < 4; ++j) prm.inv_w[j] = 1.0f / (float)box_weights[j];
  prm.scale_clamp = (float)log(1000.0 / 16);
  prm.min_size = min_size;
  const size_t P = (size_t)num_problems;
  float4* cand_box = static_cast<float4*>(workspace);
  float* cand_logit = reinterpret_cast<float*>(cand_box + P * slots);
  uint32_t* keys = reinterpret_cast<uint32_t*>(reinterpret_cast<unsigned char*>(cand_logit) + align16(P * slots * 4));
  const cudaStream_t st = as_stream(stream);
  rpn_keys_kernel<<<dim3((unsigned)((prm.key_off[num_levels] + 255) / 256), (unsigned)num_problems), 256, 0, st>>>(prm, keys);
  FOD_CUDA_LAUNCH_CHECK("fod_rpn_proposals (keys)");
  rpn_select_kernel<<<num_problems * num_levels, 1024, 0, st>>>(prm, keys, cand_box, cand_logit);
  FOD_CUDA_LAUNCH_CHECK("fod_rpn_proposals (select)");
  float thr_f = iou_threshold_as_float(iou_thresh);
  int S = slots > 512 ? pick_cluster(num_problems) : 1;
  const float4* cb = cand_box;
  const float* cl = cand_logit;
  void* args[] = {&prm, &cb, &cl, &thr_f, &post_topk, &out_boxes, &out_logits, &out_count, &S};
  return launch_clusters((const void*)rpn_nms_kernel, args, num_problems, S, kNmsThreads, nms_smem_bytes(slots), stream,
                         "fod_rpn_proposals");
}
