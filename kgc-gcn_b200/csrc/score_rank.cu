// K6: fused 1-N scoring + rank count on the 5th-generation tensor cores (tcgen05 + TMEM + TMA).
//
// Replaces reference model.py:177-178 (X @ all_ent^T + bias) and main.py:122-126 (filter, double
// argsort) for evaluation: for every query q the kernel counts the entities whose logit beats the
// target's, without ever writing the [B, N] score matrix.
//
//   s[q, j] = sum_k Q[q, k] * E[j, k]      bf16 operands (K padded to kpad = 16 * ksteps), fp32 accumulate
//   Q[q, d..d+2] = 1, E[j, d..d+2] = bf16 hi / mid / lo split of bias[j]  -> s includes the bias
//   count_gt[q] += #{ j : s[q, j] >  thr[q] },  count_eq[q] += #{ j : s[q, j] == thr[q] }
//
// One persistent CTA per SM, 12 warps, warp-specialised:
//   warp 0   TMA producer: the CTA's two 128-query A tiles once per work item, then a 6-deep ring of
//            B stages (128 entities x 64 K, 16 KB, 128-byte swizzle)
//   warp 1   MMA issuer (one thread): tcgen05.mma cta_group::1 kind::f16, M = 128, N = 128, K = 16;
//            every B stage feeds BOTH A tiles, so each byte of the entity table pulled through L2
//            does 2 x 128 rows of work (halves L2 -> SM traffic, the limiter for a K = 208 GEMM)
//   warp 2   TMEM allocator (512 columns: 2 accumulator stages x 2 A tiles x 128 fp32 columns)
//   warps 4-11  epilogue: tcgen05.ld 32x32b.x32 -> compare against the row's threshold -> integer
//            counters in registers; MMA of stage s+1 overlaps the epilogue of stage s
// Work item = (pair of query tiles, chunk of entity tiles); consecutive items share the entity chunk so
// concurrently running CTAs hit the same B tiles in L2.  Integer atomics publish the counts (exact).
//
// kgc_score_pairs runs the same MMA sequence on gathered (query row, entity row) pairs and returns the
// diagonal: the target score thr[q] and the scores of the filtered positives come from the SAME
// instruction path as the sweep, so the filter correction is bit-consistent.
//
// K6k (kgc_score_topk): the same sweep whose epilogue keeps each query's best K in {16, 32} (score, id) keys of a work
// item, skipping its exclusion list; topk_merge_kernel reduces the per-item lists.  kgc_topk_dense makes the same
// selection over dense fp32 logits (exact mode) with the same list, exclusion cursor, partial layout and merge.
// kgc_topk_merge combines finished results of disjoint entity ranges (shards) with the same list and output loop.
#include <cuda.h>

#include <cstdlib>
#include <cuda_bf16.h>

#include "common.cuh"

namespace kgc {
namespace {

constexpr int kBlockM = 128;             // queries per A tile (UMMA M)
constexpr int kBlockN = 128;             // entities per B tile (UMMA N)
constexpr int kBlockK = 64;              // bf16 elements per K block = one 128-byte swizzle row
constexpr int kUmmaK = 16;
constexpr int kMaxKBlocks = 4;           // kpad <= 256
constexpr int kMTiles = 2;
constexpr int kStagesB = 6;
constexpr int kAccStages = 2;
constexpr int kTileBytes = kBlockM * kBlockK * 2;       // 16 KB (A K-block and B stage alike)
constexpr int kThreads = 384;
constexpr int kEpiWarp0 = 4;
constexpr int kTmemCols = 512;
constexpr int kSmemA = kMTiles * kMaxKBlocks * kTileBytes;              // 128 KB
constexpr int kSmemB = kStagesB * kTileBytes;                           //  96 KB
constexpr int kSmemBar = 256;
constexpr int kSmemBytes = kSmemA + kSmemB + kSmemBar + 1024;           // + alignment slack

// ------------------------------------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// One lane of a fully converged warp (PTX elect.sync).  The surrounding code stays warp-uniform, so ptxas keeps the
// shared-memory / instruction descriptors in UNIFORM registers; running the whole role under `if (lane == 0)` makes
// them per-thread values and every tcgen05.mma then pays a chain of R2UR moves (~120 cycles per MMA, measured).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n"
      ".reg .b32 rx;\n"
      ".reg .pred px;\n"
      "elect.sync rx|px, 0xFFFFFFFF;\n"
      "@px mov.s32 %0, 1;\n"
      "}"
      : "+r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// the same load delivered to the same shared-memory offset (and the same mbarrier offset) of every CTA in cta_mask
__device__ __forceinline__ void tma_load_2d_mc(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1,
                                               uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%4, %5}], "
      "[%2], %3;" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "h"(cta_mask), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {          // every thread of every CTA of the cluster
  asm volatile("barrier.cluster.arrive.release.aligned;\n"
               "barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, bf16 x bf16 -> fp32, issued by ONE thread for the CTA
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
// all tcgen05.mma issued so far by this thread arrive on the mbarrier when they complete
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// the same arrival on the mbarrier at this offset in every CTA of cta_mask (the B stage is shared by a CTA pair)
__device__ __forceinline__ void umma_commit_mc(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(cta_mask)
               : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor: K-major tile, 128-byte swizzle, rows of 128 B, 8-row atoms 1024 B apart.
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);     // start address  [0,14)
  d |= (uint64_t)0 << 16;                          // leading byte offset (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;                // stride byte offset [32,46): 8 rows * 128 B
  d |= (uint64_t)1 << 46;                          // descriptor version (sm_100)
  d |= (uint64_t)2 << 61;                          // layout type: SWIZZLE_128B
  return d;
}
// Instruction descriptor, kind::f16: D = f32, A = B = bf16, both K-major, N >> 3 at [17,23), M >> 4 at [24,29)
constexpr uint32_t kInstrDesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(kBlockN >> 3) << 17) |
                                ((uint32_t)(kBlockM >> 4) << 24);

struct SharedLayout {
  uint8_t* a;            // [kMTiles][kMaxKBlocks][16 KB]
  uint8_t* b;            // [kStagesB][16 KB]
  uint64_t* full;        // [kStagesB]
  uint64_t* empty;       // [kStagesB]
  uint64_t* a_full;      // [1]
  uint64_t* a_empty;     // [1]
  uint64_t* acc_full;    // [kAccStages]
  uint64_t* acc_empty;   // [kAccStages]
  uint32_t* tmem_slot;
};
__device__ __forceinline__ SharedLayout carve(uint8_t* raw) {
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(raw) + 1023) & ~uintptr_t(1023));
  SharedLayout s;
  s.a = base;
  s.b = base + kSmemA;
  uint64_t* bars = reinterpret_cast<uint64_t*>(base + kSmemA + kSmemB);
  s.full = bars;
  s.empty = bars + kStagesB;
  s.a_full = bars + 2 * kStagesB;
  s.a_empty = s.a_full + 1;
  s.acc_full = s.a_empty + 1;
  s.acc_empty = s.acc_full + kAccStages;
  s.tmem_slot = reinterpret_cast<uint32_t*>(s.acc_empty + kAccStages);
  return s;
}

struct ScoreParams {
  int64_t n_queries;      // B (valid A rows)
  int64_t n_entities;     // N (valid B rows)
  int32_t ksteps;         // kpad / 16
  int32_t n_kblocks;      // ceil(kpad / 64)
  int32_t n_mp;           // number of query-tile pairs (sweep) / pair tiles (pairs mode)
  int32_t n_tiles;        // entity tiles
  int32_t chunk_tiles;    // entity tiles per work item
  int32_t n_items;
  const float* thr;       // [B]
  int32_t* count_gt;      // [B]
  int32_t* count_eq;      // [B] or nullptr
  float* pair_out;        // pairs mode: [n_pairs]
  int64_t n_pairs;
  const int64_t* excl_ptr;   // top-k mode: exclusion CSR [B + 1] / [nnz], ascending per row (nullptr: no filter)
  const int32_t* excl_idx;
  uint64_t* topk_part;       // top-k mode: [n_chunks, B, K] sorted keys of every work item
  uint32_t* topk_floor;      // top-k mode: [B] order-preserving bits of the best K-th score a finished item found (0: none)
};

// ------------------------------------------------------------------------------------------------ top-k selection (K6k)
// An entry is one 64-bit key: the score's order-preserving bits in the high word, ~id in the low word, so that ONE unsigned
// compare orders by (score descending, id ascending).  -0.0 is mapped to +0.0 first (the float compares treat them as
// equal).  The empty entry is the key of (-inf, id -1): its low word is 0, which no real id (< 2^31) produces.
__device__ __forceinline__ uint64_t topk_key(float s, int32_t id) {
  uint32_t u = __float_as_uint(s);
  if (u == 0x80000000u) u = 0u;
  const uint32_t ord = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return ((uint64_t)ord << 32) | (uint32_t)~id;
}
__device__ __forceinline__ float topk_key_score(uint64_t key) {
  const uint32_t ord = (uint32_t)(key >> 32);
  return __uint_as_float((ord & 0x80000000u) ? (ord & 0x7FFFFFFFu) : ~ord);
}
__device__ __forceinline__ int32_t topk_key_id(uint64_t key) { return (int32_t)~(uint32_t)key; }

// Register-resident list of the K largest keys seen, sorted descending.  Every index is a compile-time constant after
// unrolling: one dynamic index would move the whole list to local memory.
template <int K>
struct TopList {
  uint64_t key[K];
  float thr;              // insert test s > thr: max(score of key[K - 1], floor); -inf while the list is not full
  float floor;            // candidates at or below it cannot reach the final top K (-inf: no bound known)

  __device__ __forceinline__ void init(bool active) {
#pragma unroll
    for (int i = 0; i < K; ++i) key[i] = topk_key(__int_as_float(0xff800000), -1);
    floor = __int_as_float(0xff800000);
    thr = __int_as_float(active ? 0xff800000 : 0x7f800000);    // +inf: an inactive row never inserts
  }
  // c > key[K - 1]: compare-and-shift, the last entry falls off
  __device__ __forceinline__ void insert(uint64_t c) {
#pragma unroll
    for (int i = K - 1; i > 0; --i) key[i] = c > key[i - 1] ? key[i - 1] : (c > key[i] ? c : key[i]);
    key[0] = c > key[0] ? c : key[0];
    thr = fmaxf(topk_key_score(key[K - 1]), floor);
  }
  // Another list of the same query already holds K real entries scoring >= s_K (its K-th): a candidate below s_K has K
  // better keys elsewhere and cannot be in the final top K; one AT s_K still may (lower id), hence the next float down.
  __device__ __forceinline__ void set_floor(uint32_t ord) {
    if (ord == 0u) return;
    floor = nextafterf(topk_key_score((uint64_t)ord << 32), __int_as_float(0xff800000));
    thr = fmaxf(thr, floor);
  }
  __device__ __forceinline__ bool full() const { return (uint32_t)key[K - 1] != 0u; }
};

// Walks one row's ascending exclusion list alongside ascending candidate ids; ids outside the list's range and duplicates
// are harmless.  Only candidates that beat the list's K-th entry ask, and most of them find nxt > id without a load.
struct ExclCursor {
  const int32_t* idx;
  int64_t cur, end;
  int32_t nxt;            // idx[cur], or INT_MAX past the end

  __device__ __forceinline__ void init(const int64_t* ptr, const int32_t* idx_, int64_t q, int64_t first_id) {
    idx = idx_;
    cur = end = 0;
    nxt = 0x7FFFFFFF;
    if (ptr == nullptr) return;
    int64_t lo = __ldg(ptr + q), hi = __ldg(ptr + q + 1);
    end = hi;
    while (lo < hi) {                                            // first entry >= first_id
      const int64_t mid = (lo + hi) >> 1;
      if ((int64_t)__ldg(idx + mid) < first_id) lo = mid + 1; else hi = mid;
    }
    cur = lo;
    if (cur < end) nxt = __ldg(idx + cur);
  }
  __device__ __forceinline__ bool excluded(int32_t id) {
    while (nxt < id) nxt = (++cur < end) ? __ldg(idx + cur) : 0x7FFFFFFF;
    return nxt == id;
  }
};

// The one selection step every top-k path uses: ids arrive ascending per list, so a candidate that only ties the K-th
// entry loses to it (lower id first) and the strict float compare is the whole test on the common path.
template <int K>
__device__ __forceinline__ void topk_offer(TopList<K>& L, ExclCursor& X, float s, int32_t id) {
  if (s > L.thr && !X.excluded(id)) L.insert(topk_key(s, id));
}

// kCluster: launched as clusters of TWO CTAs that sweep the same entity tiles for different query tiles.  Each CTA of the
// pair fetches HALF of every B stage (64 entity rows) and the TMA multicasts it into both CTAs' shared memory: every byte
// of the entity table crosses L2 -> SM once per 512 queries instead of once per 256.  (Measured: no gain - the sweep is
// not bound by the 4.3 TB/s it pulls out of L2; opt-in.)  A stage's `full` barrier collects both halves (its own TMA and
// the peer's), its `empty` barrier the retired MMAs of BOTH CTAs (tcgen05.commit multicast) - a slot is rewritten by the
// peer's TMA as well.
//
// kTopK (K6k, 16 or 32): instead of counting, every epilogue thread keeps its query row's kTopK best (score, id) keys of the
// work item in registers (TopList) and writes them to P.topk_part[chunk, q, :]; topk_merge_kernel reduces the chunks.
template <bool kPairs, bool kCountEq, bool kCluster, int kTopK = 0>
__global__ void __launch_bounds__(kThreads, 1)
score_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
             const __grid_constant__ CUtensorMap map_bh, const ScoreParams P) {
  extern __shared__ uint8_t smem_raw[];
  const SharedLayout S = carve(smem_raw);
  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
  constexpr int kNumM = kPairs ? 1 : kMTiles;
  static_assert(!(kPairs && kCluster), "pairs mode runs single CTAs");
  static_assert(kTopK == 0 || (!kPairs && !kCountEq && !kCluster), "top-k mode is a single-CTA sweep");
  const uint32_t cta_rank = kCluster ? cluster_ctarank() : 0u;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
    for (int i = 0; i < kStagesB; ++i) {
      mbar_init(S.full + i, 1);
      mbar_init(S.empty + i, kCluster ? 2 : 1);
    }
    mbar_init(S.a_full, 1);
    mbar_init(S.a_empty, 1);
    for (int i = 0; i < kAccStages; ++i) {
      mbar_init(S.acc_full + i, 1);
      mbar_init(S.acc_empty + i, 4 * kNumM);      // one arrival per epilogue warp
    }
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 2) tmem_alloc(S.tmem_slot, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (kCluster) cluster_sync_all();                            // the peer's barriers exist before anything targets them
  const uint32_t tmem_base = *S.tmem_slot;

  if (warp == 0) {
    // ================================================================== TMA producer
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0, a_phase = 0;
      for (int item = blockIdx.x; item < P.n_items; item += gridDim.x) {
        const int chunk = item / P.n_mp, mp = item % P.n_mp;
        const int t0 = kPairs ? mp : chunk * P.chunk_tiles;
        const int t1 = kPairs ? mp + 1 : min(t0 + P.chunk_tiles, P.n_tiles);
        mbar_wait(S.a_empty, a_phase ^ 1);                     // previous item's MMAs have finished reading A
        mbar_expect_tx(S.a_full, kNumM * P.n_kblocks * kTileBytes);
        for (int m = 0; m < kNumM; ++m)
          for (int kb = 0; kb < P.n_kblocks; ++kb)
            tma_load_2d(S.a + (m * kMaxKBlocks + kb) * kTileBytes, &map_a, S.a_full, kb * kBlockK,
                        (mp * kNumM + m) * kBlockM);
        a_phase ^= 1;
        for (int t = t0; t < t1; ++t) {
          for (int kb = 0; kb < P.n_kblocks; ++kb) {
            mbar_wait(S.empty + stage, phase ^ 1);
            mbar_expect_tx(S.full + stage, kTileBytes);
            if (kCluster)                                          // my half of the stage, into both CTAs
              tma_load_2d_mc(S.b + stage * kTileBytes + cta_rank * (kTileBytes / 2), &map_bh, S.full + stage, kb * kBlockK,
                             t * kBlockN + (int)cta_rank * (kBlockN / 2), (uint16_t)3);
            else
              tma_load_2d(S.b + stage * kTileBytes, &map_b, S.full + stage, kb * kBlockK, t * kBlockN);
            if (++stage == kStagesB) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================================================================== MMA issuer (warp-uniform loop, one elected lane issues)
    {
      int stage = 0, acc = 0;
      uint32_t phase = 0, acc_phase = 0, a_phase = 0;
      const uint32_t a_base = smem_u32(S.a), b_base = smem_u32(S.b);
      for (int item = blockIdx.x; item < P.n_items; item += gridDim.x) {
        const int chunk = item / P.n_mp, mp = item % P.n_mp;
        const int t0 = kPairs ? mp : chunk * P.chunk_tiles;
        const int t1 = kPairs ? mp + 1 : min(t0 + P.chunk_tiles, P.n_tiles);
        mbar_wait(S.a_full, a_phase);
        a_phase ^= 1;
        tc_fence_after();
        for (int t = t0; t < t1; ++t) {
          mbar_wait(S.acc_empty + acc, acc_phase ^ 1);         // epilogue has drained this accumulator stage
          tc_fence_after();
          for (int kb = 0; kb < P.n_kblocks; ++kb) {
            mbar_wait(S.full + stage, phase);
            tc_fence_after();
            const int nk = min(kBlockK / kUmmaK, P.ksteps - kb * (kBlockK / kUmmaK));
            const uint64_t bdesc = make_sw128_desc(b_base + stage * kTileBytes);
            const uint64_t adesc0 = make_sw128_desc(a_base + kb * kTileBytes);
            const uint64_t adesc1 = make_sw128_desc(a_base + (kMaxKBlocks + kb) * kTileBytes);
            const uint32_t d0 = tmem_base + acc * (kMTiles * kBlockN);
            if (elect_one()) {
              // straight-line issue: with a runtime trip count the loop carried three R2UR moves and ~20 uniform-datapath
              // instructions per pair of MMAs (SASS) - about the 64 cycles the tensor pipe needs for one of them
#pragma unroll
              for (int k = 0; k < kBlockK / kUmmaK; ++k) {
                if (k < nk) {
                  // + k * 32 bytes along K inside the swizzle row: descriptor start address is in 16-byte units
                  const uint32_t accum = (k != 0 || kb != 0) ? 1u : 0u;
                  umma_bf16(d0, adesc0 + 2 * k, bdesc + 2 * k, kInstrDesc, accum);
                  if (kNumM == 2) umma_bf16(d0 + kBlockN, adesc1 + 2 * k, bdesc + 2 * k, kInstrDesc, accum);
                }
              }
              if (kCluster) umma_commit_mc(S.empty + stage, (uint16_t)3);   // ... in BOTH CTAs: the slot is shared
              else umma_commit(S.empty + stage);               // B stage is free once these MMAs retire
              if (kb == P.n_kblocks - 1) {
                umma_commit(S.acc_full + acc);                 // accumulators of this entity tile are complete
                if (t == t1 - 1) umma_commit(S.a_empty);       // A tiles may be overwritten
              }
            }
            __syncwarp();
            if (++stage == kStagesB) { stage = 0; phase ^= 1; }
          }
          if (++acc == kAccStages) { acc = 0; acc_phase ^= 1; }
        }
      }
    }
  } else if (kTopK != 0 && warp >= kEpiWarp0) {
    // ================================================================== top-k epilogue (TMEM -> registers -> sorted list)
    // Single-buffered tcgen05.ld: the second 32-register buffer of the counting epilogue would not fit next to a K = 32
    // list (64 registers) under the 168-register budget of 384 threads; the loads stay hidden behind the next tile's MMAs.
    constexpr int K = kTopK > 0 ? kTopK : 1;
    const int m = (warp - kEpiWarp0) / 4;
    const int quarter = warp % 4;
    const int row = quarter * 32 + lane;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int item = blockIdx.x; item < P.n_items; item += gridDim.x) {
      const int chunk = item / P.n_mp, mp = item % P.n_mp;
      const int t0 = chunk * P.chunk_tiles;
      const int t1 = min(t0 + P.chunk_tiles, P.n_tiles);
      const int64_t q = (int64_t)(mp * kNumM + m) * kBlockM + row;
      const bool active = q < P.n_queries;
      TopList<K> L;
      L.init(active);
      // items of other entity chunks that already finished bound this query's K-th score from below: without that bound
      // every item starts empty and pays ~K ln(entities / K) inserts per row, serialised over the warp's 32 rows
      if (active) L.set_floor(*reinterpret_cast<volatile uint32_t*>(P.topk_floor + q));
      ExclCursor X;
      X.init(active ? P.excl_ptr : nullptr, P.excl_idx, q, (int64_t)t0 * kBlockN);
      for (int t = t0; t < t1; ++t) {
        mbar_wait(S.acc_full + acc, acc_phase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * (kMTiles * kBlockN) + m * kBlockN;
        const int valid = (int)min((int64_t)kBlockN, P.n_entities - (int64_t)t * kBlockN);
#pragma unroll 1
        for (int c = 0; c < kBlockN / 32; ++c) {
          uint32_t v[32];
          __syncwarp();                                        // tcgen05.ld is .aligned: the insert path diverges
          tmem_ld32(taddr + c * 32, v);
          tmem_ld_wait();
          if (valid < kBlockN) {
#pragma unroll
            for (int j = 0; j < 32; ++j)                     // entity rows past N are zero-filled by TMA: never insert
              if (c * 32 + j >= valid) v[j] = 0xff800000u;
          }
          // common path: the block's maximum against the K-th score (a tree: no 32-long dependent chain)
          float mx[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) mx[j] = fmaxf(__uint_as_float(v[j]), __uint_as_float(v[j + 16]));
#pragma unroll
          for (int w = 8; w > 0; w >>= 1)
#pragma unroll
            for (int j = 0; j < w; ++j) mx[j] = fmaxf(mx[j], mx[j + w]);
          if (mx[0] > L.thr) {
            const int32_t id0 = t * kBlockN + c * 32;
#pragma unroll
            for (int j = 0; j < 32; ++j) topk_offer(L, X, __uint_as_float(v[j]), id0 + j);
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(S.acc_empty + acc);
        if (++acc == kAccStages) { acc = 0; acc_phase ^= 1; }
      }
      if (active) {
        uint4* dst = reinterpret_cast<uint4*>(P.topk_part + ((int64_t)chunk * P.n_queries + q) * K);
#pragma unroll
        for (int i = 0; i < K; i += 2)
          dst[i / 2] = make_uint4((uint32_t)L.key[i], (uint32_t)(L.key[i] >> 32), (uint32_t)L.key[i + 1],
                                  (uint32_t)(L.key[i + 1] >> 32));
        // integer max: the merged result does not depend on which items saw the bound (every final entry survives it)
        if (L.full()) atomicMax(P.topk_floor + q, (uint32_t)(L.key[K - 1] >> 32));
      }
    }
  } else if (warp >= kEpiWarp0 && (warp - kEpiWarp0) / 4 < kNumM) {
    // ================================================================== epilogue (TMEM -> registers -> counters)
    const int m = (warp - kEpiWarp0) / 4;
    const int quarter = warp % 4;                              // TMEM lane quarter this warp may access
    const int row = quarter * 32 + lane;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int item = blockIdx.x; item < P.n_items; item += gridDim.x) {
      const int chunk = item / P.n_mp, mp = item % P.n_mp;
      const int t0 = kPairs ? mp : chunk * P.chunk_tiles;
      const int t1 = kPairs ? mp + 1 : min(t0 + P.chunk_tiles, P.n_tiles);
      const int64_t q = (int64_t)(mp * kNumM + m) * kBlockM + row;
      float thr = __int_as_float(0x7f800000);                  // +inf: rows past the end never count
      if (!kPairs && q < P.n_queries) thr = __ldg(P.thr + q);
      int gt = 0, eq = 0;
      float diag = 0.f;
      for (int t = t0; t < t1; ++t) {
        mbar_wait(S.acc_full + acc, acc_phase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * (kMTiles * kBlockN) + m * kBlockN;
        const int valid = (int)min((int64_t)kBlockN, P.n_entities - (int64_t)t * kBlockN);
        uint32_t v[2][32];
        tmem_ld32(taddr, v[0]);
#pragma unroll
        for (int c = 0; c < kBlockN / 32; ++c) {
          tmem_ld_wait();
          if (c + 1 < kBlockN / 32) tmem_ld32(taddr + (c + 1) * 32, v[(c + 1) & 1]);
          if (kPairs) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (c * 32 + j == row) diag = __uint_as_float(v[c & 1][j]);
          } else if (valid == kBlockN) {
            // four independent counters: one counter made a serial chain of 128 dependent (add, select) pairs per tile -
            // about as long as the tile's MMAs
            int g4[4] = {0, 0, 0, 0}, e4[4] = {0, 0, 0, 0};
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const float s = __uint_as_float(v[c & 1][j]);
              if (s > thr) ++g4[j & 3];
              if (kCountEq && s == thr) ++e4[j & 3];
            }
            gt += (g4[0] + g4[1]) + (g4[2] + g4[3]);
            if (kCountEq) eq += (e4[0] + e4[1]) + (e4[2] + e4[3]);
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const float s = __uint_as_float(v[c & 1][j]);
              const bool in = c * 32 + j < valid;              // entity rows past N are zero-filled by TMA: skip
              gt += (in && s > thr) ? 1 : 0;
              if (kCountEq) eq += (in && s == thr) ? 1 : 0;
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(S.acc_empty + acc);
        if (++acc == kAccStages) { acc = 0; acc_phase ^= 1; }
      }
      if (kPairs) {
        if (q < P.n_pairs) P.pair_out[q] = diag;
      } else if (q < P.n_queries) {
        if (gt) atomicAdd(P.count_gt + q, gt);                 // integer atomics: exact, order-independent
        if (kCountEq && eq) atomicAdd(P.count_eq + q, eq);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (kCluster) cluster_sync_all();                            // no CTA leaves while the peer may still write or signal into it
  if (warp == 2) tmem_dealloc(tmem_base, kTmemCols);
}

// ------------------------------------------------------------------------------------------------ packing / gather / finalize
__device__ __forceinline__ uint16_t bf16_bits(float f) { return __bfloat16_as_ushort(__float2bfloat16_rn(f)); }

// entity row j: [bf16(all_ent[j, 0..d)), hi, mid, lo of bias[j], zeros]  (bias = hi + mid + lo to ~2^-24)
__global__ void pack_entities_kernel(const float* __restrict__ ent, const float* __restrict__ bias, int64_t n, int d,
                                     int kpad, uint16_t* __restrict__ out) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n * kpad) return;
  const int64_t r = i / kpad;
  const int c = (int)(i % kpad);
  uint16_t v = 0;
  if (c < d) {
    v = bf16_bits(ent[r * d + c]);
  } else if (c < d + 3) {
    const float b = bias ? bias[r] : 0.f;
    const float hi = __bfloat162float(__float2bfloat16_rn(b));
    const float r1 = b - hi;
    const float mid = __bfloat162float(__float2bfloat16_rn(r1));
    const float lo = r1 - mid;
    v = bf16_bits(c == d ? hi : (c == d + 1 ? mid : lo));
  }
  out[i] = v;
}
__global__ void pack_queries_kernel(const float* __restrict__ xq, int64_t b, int d, int kpad, uint16_t* __restrict__ out) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= b * kpad) return;
  const int64_t r = i / kpad;
  const int c = (int)(i % kpad);
  uint16_t v = 0;
  if (c < d) v = bf16_bits(xq[r * d + c]);
  else if (c < d + 3) v = 0x3F80;   // 1.0 in bf16: picks up the three bias columns
  out[i] = v;
}
// rows of 16-byte chunks: out[p, :] = table[idx[p], :]
__global__ void gather_rows_kernel(const uint4* __restrict__ table, const int32_t* __restrict__ idx, int64_t n_pairs,
                                   int chunks, uint4* __restrict__ out) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n_pairs * chunks) return;
  const int64_t p = i / chunks;
  const int c = (int)(i % chunks);
  out[i] = __ldg(table + (int64_t)idx[p] * chunks + c);
}

// rank[q] = 1 + gt[q] - #{filtered j != o : s_j > thr};  eq likewise (minus the target itself)
__global__ void rank_finalize_kernel(const int32_t* __restrict__ count_gt, const int32_t* __restrict__ count_eq,
                                     const float* __restrict__ thr, const float* __restrict__ s_filt,
                                     const int64_t* __restrict__ filt_ptr, const int32_t* __restrict__ filt_idx,
                                     const int64_t* __restrict__ obj, int64_t b, int32_t* __restrict__ ranks,
                                     int32_t* __restrict__ eq_out) {
  const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (q >= b) return;
  int gt = count_gt[q];
  int eq = count_eq ? count_eq[q] - 1 : 0;       // the sweep also met the target itself (s == thr)
  const float t = thr[q];
  const int32_t o = (int32_t)obj[q];
  for (int64_t k = filt_ptr[q]; k < filt_ptr[q + 1]; ++k) {
    if (filt_idx[k] == o) continue;
    const float s = s_filt[k];
    gt -= (s > t) ? 1 : 0;
    eq -= (s == t) ? 1 : 0;
  }
  ranks[q] = 1 + gt;
  if (eq_out) eq_out[q] = eq;
}
// Exact-mode counts over DENSE fp32 logits z[B, ld] (kgc_score_1n_logits): gt[q] += #{j < n : z[q, j] > thr[q]}, eq likewise.
// grid = (column chunks, queries); integer partial sums -> one integer atomic per CTA (order-independent).
constexpr int kDenseThreads = 256, kDenseCols = 8 * kDenseThreads;
__global__ void __launch_bounds__(kDenseThreads)
rank_count_dense_kernel(const float* __restrict__ z, int64_t ld, int64_t n, const float* __restrict__ thr,
                        int32_t* __restrict__ count_gt, int32_t* __restrict__ count_eq) {
  const int64_t q = blockIdx.y;
  const float t = thr[q];
  const float* row = z + q * ld;
  int gt = 0, eq = 0;
  const int64_t c0 = (int64_t)blockIdx.x * kDenseCols;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int64_t c = c0 + i * kDenseThreads + threadIdx.x;
    if (c < n) {
      const float s = __ldg(row + c);
      gt += s > t ? 1 : 0;
      eq += s == t ? 1 : 0;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    gt += __shfl_xor_sync(0xFFFFFFFFu, gt, o);
    eq += __shfl_xor_sync(0xFFFFFFFFu, eq, o);
  }
  __shared__ int sg[kDenseThreads / 32], se[kDenseThreads / 32];
  if (threadIdx.x % 32 == 0) { sg[threadIdx.x / 32] = gt; se[threadIdx.x / 32] = eq; }
  __syncthreads();
  if (threadIdx.x == 0) {
    int g = 0, e = 0;
    for (int w = 0; w < kDenseThreads / 32; ++w) { g += sg[w]; e += se[w]; }
    if (g) atomicAdd(count_gt + q, g);
    if (count_eq != nullptr && e) atomicAdd(count_eq + q, e);
  }
}

// Exact-mode top-k over DENSE fp32 logits: grid = (column chunks of kTopkDenseCols, queries).  Thread t offers columns
// c0 + t, c0 + t + 256, ... (ascending ids) to its own TopList, then the block folds the 256 lists pairwise through shared
// memory (each fold keeps the top K of two lists; keys are unique, so the result does not depend on the order) and writes
// one list per chunk: the same [n_chunks, B, K] partials as the tcgen05 sweep, reduced by the same merge kernel.
constexpr int kTopkDenseThreads = 256, kTopkDensePerThread = 64;
constexpr int kTopkDenseCols = kTopkDenseThreads * kTopkDensePerThread;
// Folds a list of `len` keys, sorted descending, into L: key(i) yields the i-th key.
template <int K, class KeyAt>
__device__ __forceinline__ void topk_fold_keys(TopList<K>& L, int len, KeyAt key) {
  for (int i = 0; i < len; ++i) {
    const uint64_t c = key(i);
    if (!(c > L.key[K - 1])) break;
    L.insert(c);
  }
}
template <int K>
__device__ __forceinline__ void topk_fold(TopList<K>& L, const uint64_t* list) {    // list: K keys, sorted descending
  topk_fold_keys(L, K, [list](int i) { return list[i]; });
}
template <int K>
__global__ void __launch_bounds__(kTopkDenseThreads)
topk_dense_kernel(const float* __restrict__ z, int64_t ld, int64_t n, int64_t b, const int64_t* __restrict__ excl_ptr,
                  const int32_t* __restrict__ excl_idx, uint64_t* __restrict__ part) {
  const int64_t q = blockIdx.y;
  const float* row = z + q * ld;
  const int64_t c0 = (int64_t)blockIdx.x * kTopkDenseCols + threadIdx.x;
  TopList<K> L;
  L.init(true);
  ExclCursor X;
  X.init(excl_ptr, excl_idx, q, c0);
#pragma unroll 4
  for (int i = 0; i < kTopkDensePerThread; ++i) {
    const int64_t c = c0 + (int64_t)i * kTopkDenseThreads;
    if (c < n) topk_offer(L, X, __ldg(row + c), (int32_t)c);
  }
  __shared__ __align__(16) uint64_t sm[kTopkDenseThreads / 2 * K];
  for (int half = kTopkDenseThreads / 2; half > 0; half >>= 1) {
    __syncthreads();
    if (threadIdx.x >= half && threadIdx.x < 2 * half) {
#pragma unroll
      for (int i = 0; i < K; ++i) sm[(threadIdx.x - half) * K + i] = L.key[i];
    }
    __syncthreads();
    if (threadIdx.x < half) topk_fold(L, sm + threadIdx.x * K);
  }
  if (threadIdx.x == 0) {
    uint64_t* dst = part + ((int64_t)blockIdx.x * b + q) * K;
#pragma unroll
    for (int i = 0; i < K; ++i) dst[i] = L.key[i];
  }
}

// The first k entries of a finished list: scores (padding -inf), ids (padding -1), count of real entries.
template <int K>
__device__ __forceinline__ void topk_store(const TopList<K>& L, int64_t q, int k, float* __restrict__ top_s,
                                           int32_t* __restrict__ top_id, int32_t* __restrict__ count) {
  int cnt = 0;
#pragma unroll
  for (int i = 0; i < K; ++i) {
    if (i < k) {
      top_s[q * k + i] = topk_key_score(L.key[i]);
      top_id[q * k + i] = topk_key_id(L.key[i]);
      cnt += (uint32_t)L.key[i] != 0u ? 1 : 0;
    }
  }
  count[q] = cnt;
}

// Final [k] per query from the [n_chunks, B, K] partial lists; one thread per query, chunks in order, keys unique ->
// deterministic for any chunk count.  Output: scores (padding -inf), ids (padding -1), count of real entries.
template <int K>
__global__ void topk_merge_kernel(const uint64_t* __restrict__ part, int64_t n_chunks, int64_t b, int k,
                                  float* __restrict__ top_s, int32_t* __restrict__ top_id, int32_t* __restrict__ count) {
  const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (q >= b) return;
  TopList<K> L;
  L.init(true);
  for (int64_t c = 0; c < n_chunks; ++c) topk_fold(L, part + (c * b + q) * K);
  topk_store(L, q, k, top_s, top_id, count);
}

// Cross-shard merge (kgc_topk_merge): the same fold and output over n_lists finished [b, k] results (float scores, int32
// ids, id < 0 padding), keys built as the lists are read.  Ids are disjoint across lists, so keys are unique and the
// result does not depend on the list order.
template <int K>
__global__ void topk_merge_lists_kernel(const float* __restrict__ part_s, const int32_t* __restrict__ part_id,
                                        int64_t n_lists, int64_t b, int k, float* __restrict__ top_s,
                                        int32_t* __restrict__ top_id, int32_t* __restrict__ count) {
  const int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (q >= b) return;
  TopList<K> L;
  L.init(true);
  for (int64_t l = 0; l < n_lists; ++l) {
    const float* s = part_s + (l * b + q) * k;
    const int32_t* id = part_id + (l * b + q) * k;
    topk_fold_keys(L, k, [s, id](int i) {
      const int32_t e = __ldg(id + i);
      return e < 0 ? topk_key(__int_as_float(0xff800000), -1) : topk_key(__ldg(s + i), e);
    });
  }
  topk_store(L, q, k, top_s, top_id, count);
}

// sums13 = {count, sum rank, sum 1/rank, hits@1..10}; one block, fixed order -> deterministic
__global__ void rank_sums_kernel(const int32_t* __restrict__ ranks, int64_t b, double* __restrict__ sums13) {
  __shared__ double sm[13][256];
  double acc[13];
  for (int i = 0; i < 13; ++i) acc[i] = 0;
  for (int64_t q = threadIdx.x; q < b; q += 256) {
    const int r = ranks[q];
    acc[0] += 1.0;
    acc[1] += (double)r;
    acc[2] += (double)(1.0f / (float)r);       // main.py:131 divides in fp32
    for (int k = 1; k <= 10; ++k) acc[2 + k] += (r <= k) ? 1.0 : 0.0;
  }
  for (int i = 0; i < 13; ++i) sm[i][threadIdx.x] = acc[i];
  __syncthreads();
  if (threadIdx.x < 13) {
    double s = 0;
    for (int k = 0; k < 256; ++k) s += sm[threadIdx.x][k];
    sums13[threadIdx.x] = s;
  }
}

// ------------------------------------------------------------------------------------------------ host helpers
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int get_encode_fn(EncodeTiledFn* out) {
  ensure_thread_context();
  static EncodeTiledFn cached = nullptr;
  if (!cached) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    KGC_CUDA_TRY(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    KGC_REQUIRE(qres == cudaDriverEntryPointSuccess && fn != nullptr, "cuTensorMapEncodeTiled not available");
    cached = reinterpret_cast<EncodeTiledFn>(fn);
  }
  *out = cached;
  return 0;
}

// bf16 [rows, kpad] row-major -> boxes of 64 (K) x 128 (rows), 128-byte swizzle, zero fill out of bounds
int make_map(CUtensorMap* map, const void* base, int64_t rows, int kpad, int box_rows = kBlockM) {
  EncodeTiledFn enc;
  if (get_encode_fn(&enc)) return 1;
  KGC_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15) == 0, "bf16 table must be 16-byte aligned");
  cuuint64_t dims[2] = {(cuuint64_t)kpad, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)kpad * 2};
  cuuint32_t box[2] = {(cuuint32_t)kBlockK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  KGC_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")");
  return 0;
}

inline int check_kpad(int kpad) { return (kpad < 16 || kpad % 16 != 0 || kpad > kMaxKBlocks * kBlockK) ? 1 : 0; }

// Work items of the sweep: P.n_mp (query-tile pairs, set by the caller), n_tiles, chunk_tiles and n_items.  Entity
// chunks: enough work items to balance 148 persistent CTAs, chunk small enough to stay in L2 (<= ~48 MB of bf16 rows) so
// that the CTAs sweeping one chunk share its tiles.  kgc_score_rank, kgc_score_topk and its workspace size all use it.
void plan_chunks(ScoreParams& P, int64_t n, int kpad) {
  P.n_tiles = (int32_t)ceil_div(n, kBlockN);
  const int64_t max_chunk_tiles = (int64_t)(48 << 20) / ((int64_t)kBlockN * kpad * 2);
  int best_chunks = 1;
  double best_cost = 1e30;
  for (int c = 1; c <= 4096 && c <= P.n_tiles; ++c) {
    const int64_t ct = ceil_div(P.n_tiles, c);
    if (ct > max_chunk_tiles && c < P.n_tiles) continue;
    const int64_t items = (int64_t)P.n_mp * c;
    const int64_t waves = ceil_div(items, kNumSMs);
    // cost ~ time of the slowest CTA: waves * (tiles per item + A-load overhead of ~2 tiles)
    const double cost = (double)waves * (double)(ct + 2);
    if (cost < best_cost) { best_cost = cost; best_chunks = c; }
  }
  P.chunk_tiles = (int32_t)ceil_div(P.n_tiles, best_chunks);
  P.n_items = P.n_mp * (int32_t)ceil_div(P.n_tiles, P.chunk_tiles);
}

constexpr int kTopkMax = 32;              // the largest register list that fits the sweep's epilogue without spilling
inline int topk_list_len(int k) { return k <= 16 ? 16 : 32; }

// chunks of the top-k sweep for (b, n, kpad): the leading dimension of its partial lists
int64_t topk_sweep_chunks(int64_t b, int64_t n, int kpad) {
  ScoreParams P = {};
  P.n_mp = (int32_t)ceil_div(b, kMTiles * kBlockM);
  plan_chunks(P, n, kpad);
  return ceil_div(P.n_tiles, P.chunk_tiles);
}

template <int K>
int launch_topk_sweep(const CUtensorMap& ma, const CUtensorMap& mb, const ScoreParams& P, cudaStream_t st) {
  auto kern = score_kernel<false, false, false, K>;
  static SmemAttrCache attr;
  KGC_CUDA_TRY(attr.ensure(kern, (size_t)kSmemBytes));
  const int grid = P.n_items < kNumSMs ? P.n_items : kNumSMs;
  kern<<<grid, kThreads, kSmemBytes, st>>>(ma, mb, mb, P);
  KGC_LAUNCH_CHECK();
  return 0;
}

template <int K>
int launch_topk_merge(const uint64_t* part, int64_t n_chunks, int64_t b, int k, float* top_s, int32_t* top_id,
                      int32_t* count, cudaStream_t st) {
  topk_merge_kernel<K><<<(unsigned)ceil_div(b, 128), 128, 0, st>>>(part, n_chunks, b, k, top_s, top_id, count);
  KGC_LAUNCH_CHECK();
  return 0;
}

template <bool kPairs, bool kCountEq>
int launch_score(const CUtensorMap& ma, const CUtensorMap& mb, const ScoreParams& P, cudaStream_t st) {
  auto kern = score_kernel<kPairs, kCountEq, false>;
  static SmemAttrCache attr;                           // one per <kPairs, kCountEq> instantiation
  KGC_CUDA_TRY(attr.ensure(kern, (size_t)kSmemBytes));
  const int grid = P.n_items < kNumSMs ? P.n_items : kNumSMs;
  kern<<<grid, kThreads, kSmemBytes, st>>>(ma, mb, mb, P);
  KGC_LAUNCH_CHECK();
  return 0;
}

// sweep as clusters of two CTAs (see score_kernel): n_items and the grid are even, item 2i / 2i + 1 share an entity chunk
template <bool kCountEq>
int launch_score_pairs_of_ctas(const CUtensorMap& ma, const CUtensorMap& mb, const CUtensorMap& mbh, const ScoreParams& P,
                               cudaStream_t st) {
  auto kern = score_kernel<false, kCountEq, true>;
  static SmemAttrCache attr;
  KGC_CUDA_TRY(attr.ensure(kern, (size_t)kSmemBytes));
  int grid = P.n_items < kNumSMs ? P.n_items : kNumSMs;
  grid &= ~1;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = kSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  KGC_CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, ma, mb, mbh, P));
  return 0;
}

}  // namespace
}  // namespace kgc

using namespace kgc;

extern "C" int32_t kgc_score_kpad(int32_t d) {
  if (d <= 0 || d + 3 > kMaxKBlocks * kBlockK) return -1;
  return (d + 3 + 15) / 16 * 16;
}

extern "C" int kgc_score_pack_entities(const float* all_ent, const float* bias, int64_t n, int32_t d, uint16_t* e_bf16,
                                       void* stream) {
  const int kpad = kgc_score_kpad(d);
  KGC_REQUIRE(kpad > 0, "d + 3 must be <= 256");
  if (n == 0) return 0;
  pack_entities_kernel<<<(unsigned)ceil_div(n * kpad, 256), 256, 0, as_stream(stream)>>>(all_ent, bias, n, d, kpad, e_bf16);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_score_pack_queries(const float* xq, int64_t b, int32_t d, uint16_t* q_bf16, void* stream) {
  const int kpad = kgc_score_kpad(d);
  KGC_REQUIRE(kpad > 0, "d + 3 must be <= 256");
  if (b == 0) return 0;
  pack_queries_kernel<<<(unsigned)ceil_div(b * kpad, 256), 256, 0, as_stream(stream)>>>(xq, b, d, kpad, q_bf16);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" size_t kgc_score_pairs_workspace_bytes(int64_t n_pairs, int32_t kpad) {
  const int64_t padded = ceil_div(n_pairs > 0 ? n_pairs : 1, kBlockM) * kBlockM;
  return (size_t)padded * kpad * 2 * 2;       // gathered query rows + gathered entity rows
}

extern "C" int kgc_score_pairs(const uint16_t* q_bf16, const uint16_t* e_bf16, const int32_t* pair_q,
                               const int32_t* pair_e, int64_t n_pairs, int32_t kpad, float* s_out, void* workspace,
                               size_t workspace_bytes, void* stream) {
  KGC_REQUIRE(check_kpad(kpad) == 0, "kpad must be a multiple of 16 in [16, 256]");
  if (n_pairs == 0) return 0;
  KGC_REQUIRE(workspace && workspace_bytes >= kgc_score_pairs_workspace_bytes(n_pairs, kpad), "workspace too small");
  cudaStream_t st = as_stream(stream);
  const int64_t padded = ceil_div(n_pairs, kBlockM) * kBlockM;
  uint16_t* ga = static_cast<uint16_t*>(workspace);
  uint16_t* gb = ga + padded * kpad;
  const int chunks = kpad * 2 / 16;
  const unsigned grid = (unsigned)ceil_div(n_pairs * chunks, 256);
  gather_rows_kernel<<<grid, 256, 0, st>>>((const uint4*)q_bf16, pair_q, n_pairs, chunks, (uint4*)ga);
  KGC_LAUNCH_CHECK();
  gather_rows_kernel<<<grid, 256, 0, st>>>((const uint4*)e_bf16, pair_e, n_pairs, chunks, (uint4*)gb);
  KGC_LAUNCH_CHECK();
  CUtensorMap ma, mb;
  if (make_map(&ma, ga, n_pairs, kpad) || make_map(&mb, gb, n_pairs, kpad)) return 1;
  ScoreParams P = {};
  P.n_queries = n_pairs;
  P.n_entities = n_pairs;
  P.ksteps = kpad / kUmmaK;
  P.n_kblocks = (kpad + kBlockK - 1) / kBlockK;
  P.n_mp = (int32_t)(padded / kBlockM);
  P.n_tiles = P.n_mp;
  P.chunk_tiles = 1;
  P.n_items = P.n_mp;
  P.pair_out = s_out;
  P.n_pairs = n_pairs;
  return launch_score<true, false>(ma, mb, P, st);
}

extern "C" int kgc_score_rank(const uint16_t* q_bf16, const uint16_t* e_bf16, int64_t b, int64_t n, int32_t kpad,
                              const float* thr, int32_t* count_gt, int32_t* count_eq, void* stream) {
  KGC_REQUIRE(check_kpad(kpad) == 0, "kpad must be a multiple of 16 in [16, 256]");
  KGC_REQUIRE(b > 0 && n > 0 && b < (int64_t(1) << 30) && n < (int64_t(1) << 31), "bad sizes");
  cudaStream_t st = as_stream(stream);
  CUtensorMap ma, mb;
  if (make_map(&ma, q_bf16, b, kpad) || make_map(&mb, e_bf16, n, kpad)) return 1;
  ScoreParams P = {};
  P.n_queries = b;
  P.n_entities = n;
  P.ksteps = kpad / kUmmaK;
  P.n_kblocks = (kpad + kBlockK - 1) / kBlockK;
  P.n_mp = (int32_t)ceil_div(b, kMTiles * kBlockM);
  // CTA pairs that share their B stages (TMA multicast), KGC_SCORE_CLUSTER=1.  Built to test whether the sweep is bound by
  // L2 -> SM traffic: it is not - 104.4 ms against 104.7 ms with single CTAs (65,536 x 4.59 M, B200 under its power cap) -
  // so single CTAs stay the default.  The pair needs an even number of query-tile pairs (a padding pair has no valid
  // query: its rows never count)
  static const bool cluster_ok = [] { const char* e = getenv("KGC_SCORE_CLUSTER"); return e && e[0] == '1'; }();
  const bool cluster = cluster_ok && P.n_mp >= 2;
  if (cluster) P.n_mp = (P.n_mp + 1) & ~1;
  plan_chunks(P, n, kpad);
  P.thr = thr;
  P.count_gt = count_gt;
  P.count_eq = count_eq;
  if (cluster) {
    CUtensorMap mbh;
    if (make_map(&mbh, e_bf16, n, kpad, kBlockN / 2)) return 1;
    if (count_eq) return launch_score_pairs_of_ctas<true>(ma, mb, mbh, P, st);
    return launch_score_pairs_of_ctas<false>(ma, mb, mbh, P, st);
  }
  if (count_eq) return launch_score<false, true>(ma, mb, P, st);
  return launch_score<false, false>(ma, mb, P, st);
}

extern "C" size_t kgc_score_topk_workspace_bytes(int64_t b, int64_t n, int32_t kpad, int32_t k) {
  if (b <= 0 || n <= 0 || check_kpad(kpad) || k < 1 || k > kTopkMax) return 0;
  // [n_chunks, b, K] partial lists, then the [b] per-query score floors
  return (size_t)topk_sweep_chunks(b, n, kpad) * (size_t)b * topk_list_len(k) * sizeof(uint64_t) + (size_t)b * sizeof(uint32_t);
}

extern "C" int kgc_score_topk(const uint16_t* q_bf16, const uint16_t* e_bf16, int64_t b, int64_t n, int32_t kpad,
                              const int64_t* excl_ptr, const int32_t* excl_idx, int32_t k, float* top_s, int32_t* top_id,
                              int32_t* count, void* workspace, size_t workspace_bytes, void* stream) {
  KGC_REQUIRE(check_kpad(kpad) == 0, "kpad must be a multiple of 16 in [16, 256]");
  KGC_REQUIRE(b > 0 && n > 0 && b < (int64_t(1) << 30) && n < (int64_t(1) << 31), "bad sizes");
  KGC_REQUIRE(k >= 1 && k <= kTopkMax, "k must be in [1, 32]");
  KGC_REQUIRE((excl_ptr == nullptr) == (excl_idx == nullptr), "excl_ptr and excl_idx go together");
  KGC_REQUIRE(top_s && top_id && count, "null output");
  KGC_REQUIRE(workspace && workspace_bytes >= kgc_score_topk_workspace_bytes(b, n, kpad, k), "workspace too small");
  cudaStream_t st = as_stream(stream);
  CUtensorMap ma, mb;
  if (make_map(&ma, q_bf16, b, kpad) || make_map(&mb, e_bf16, n, kpad)) return 1;
  ScoreParams P = {};
  P.n_queries = b;
  P.n_entities = n;
  P.ksteps = kpad / kUmmaK;
  P.n_kblocks = (kpad + kBlockK - 1) / kBlockK;
  P.n_mp = (int32_t)ceil_div(b, kMTiles * kBlockM);
  plan_chunks(P, n, kpad);
  P.excl_ptr = excl_ptr;
  P.excl_idx = excl_idx;
  P.topk_part = static_cast<uint64_t*>(workspace);
  const int64_t n_chunks = ceil_div(P.n_tiles, P.chunk_tiles);
  P.topk_floor = reinterpret_cast<uint32_t*>(P.topk_part + n_chunks * b * topk_list_len(k));
  KGC_CUDA_TRY(cudaMemsetAsync(P.topk_floor, 0, (size_t)b * sizeof(uint32_t), st));
  if (topk_list_len(k) == 16) {
    if (launch_topk_sweep<16>(ma, mb, P, st)) return 1;
    return launch_topk_merge<16>(P.topk_part, n_chunks, b, k, top_s, top_id, count, st);
  }
  if (launch_topk_sweep<32>(ma, mb, P, st)) return 1;
  return launch_topk_merge<32>(P.topk_part, n_chunks, b, k, top_s, top_id, count, st);
}

extern "C" int kgc_topk_merge(const float* part_s, const int32_t* part_id, int64_t n_lists, int64_t b, int32_t k,
                              float* top_s, int32_t* top_id, int32_t* count, void* stream) {
  KGC_REQUIRE(n_lists >= 1 && b > 0 && b < (int64_t(1) << 31), "bad sizes (n_lists >= 1, 0 < b < 2^31)");
  KGC_REQUIRE(k >= 1 && k <= kTopkMax, "k must be in [1, 32]");
  KGC_REQUIRE(part_s && part_id, "null input");
  KGC_REQUIRE(top_s && top_id && count, "null output");
  cudaStream_t st = as_stream(stream);
  const unsigned grid = (unsigned)ceil_div(b, 128);
  if (topk_list_len(k) == 16)
    topk_merge_lists_kernel<16><<<grid, 128, 0, st>>>(part_s, part_id, n_lists, b, k, top_s, top_id, count);
  else
    topk_merge_lists_kernel<32><<<grid, 128, 0, st>>>(part_s, part_id, n_lists, b, k, top_s, top_id, count);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" size_t kgc_topk_dense_workspace_bytes(int64_t b, int64_t n, int32_t k) {
  if (b <= 0 || n <= 0 || k < 1 || k > kTopkMax) return 0;
  return (size_t)ceil_div(n, kTopkDenseCols) * (size_t)b * topk_list_len(k) * sizeof(uint64_t);
}

extern "C" int kgc_topk_dense(const float* logits, int64_t ld, int64_t n, int64_t b, const int64_t* excl_ptr,
                              const int32_t* excl_idx, int32_t k, float* top_s, int32_t* top_id, int32_t* count,
                              void* workspace, size_t workspace_bytes, void* stream) {
  KGC_REQUIRE(logits && b > 0 && n > 0 && n < (int64_t(1) << 31) && ld >= n && b <= 65535,
              "bad sizes (at most 65,535 queries per call)");
  KGC_REQUIRE(k >= 1 && k <= kTopkMax, "k must be in [1, 32]");
  KGC_REQUIRE((excl_ptr == nullptr) == (excl_idx == nullptr), "excl_ptr and excl_idx go together");
  KGC_REQUIRE(top_s && top_id && count, "null output");
  KGC_REQUIRE(workspace && workspace_bytes >= kgc_topk_dense_workspace_bytes(b, n, k), "workspace too small");
  cudaStream_t st = as_stream(stream);
  uint64_t* part = static_cast<uint64_t*>(workspace);
  const int64_t n_chunks = ceil_div(n, kTopkDenseCols);
  const dim3 grid((unsigned)n_chunks, (unsigned)b);
  if (topk_list_len(k) == 16) {
    topk_dense_kernel<16><<<grid, kTopkDenseThreads, 0, st>>>(logits, ld, n, b, excl_ptr, excl_idx, part);
    KGC_LAUNCH_CHECK();
    return launch_topk_merge<16>(part, n_chunks, b, k, top_s, top_id, count, st);
  }
  topk_dense_kernel<32><<<grid, kTopkDenseThreads, 0, st>>>(logits, ld, n, b, excl_ptr, excl_idx, part);
  KGC_LAUNCH_CHECK();
  return launch_topk_merge<32>(part, n_chunks, b, k, top_s, top_id, count, st);
}

extern "C" int kgc_rank_count_dense(const float* logits, int64_t ld, int64_t n_ent, int64_t b, const float* thr,
                                    int32_t* count_gt, int32_t* count_eq, void* stream) {
  if (b == 0 || n_ent == 0) return 0;
  KGC_REQUIRE(logits && thr && count_gt && ld >= n_ent && b <= 65535, "bad arguments (at most 65,535 queries per call)");
  rank_count_dense_kernel<<<dim3((unsigned)ceil_div(n_ent, kDenseCols), (unsigned)b), kDenseThreads, 0, as_stream(stream)>>>(
      logits, ld, n_ent, thr, count_gt, count_eq);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_rank_finalize(const int32_t* count_gt, const int32_t* count_eq, const float* thr, const float* s_filt,
                                 const int64_t* filt_ptr, const int32_t* filt_idx, const int64_t* obj, int64_t b,
                                 int32_t* ranks, int32_t* eq_out, double* sums13, void* stream) {
  if (b == 0) return 0;
  cudaStream_t st = as_stream(stream);
  rank_finalize_kernel<<<(unsigned)ceil_div(b, 256), 256, 0, st>>>(count_gt, count_eq, thr, s_filt, filt_ptr, filt_idx, obj,
                                                                  b, ranks, eq_out);
  KGC_LAUNCH_CHECK();
  if (sums13) {
    rank_sums_kernel<<<1, 256, 0, st>>>(ranks, b, sums13);
    KGC_LAUNCH_CHECK();
  }
  return 0;
}
