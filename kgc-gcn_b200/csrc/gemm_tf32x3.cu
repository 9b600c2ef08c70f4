// Dense transforms of the layer on the 5th-generation tensor cores with fp32-grade accuracy ("3xTF32").
//
// The reference multiplies in plain fp32 (torch default, TF32 off): res_h = agg_h @ W_h, g_h = d_res_h @ W_h^T
// (model.py:116 and its autograd).  Nine such N x 100 x 200 GEMMs are half of a training step when left to the
// fp32 SIMT path (profiles/r01_launches_conv_step.md).  Here every fp32 operand is split into two TF32 numbers,
//   v = hi + lo,   hi = v rounded to the nearest TF32 (cvt.rna.tf32.f32),  lo = v - hi (exact in fp32, |lo| <= 2^-11 |v|)
// rounded to TF32 in turn, and C = A_lo B_hi + A_hi B_lo + A_hi B_hi is accumulated in fp32 in TMEM by tcgen05.mma
// kind::tf32: the dropped term A_lo B_lo and the rounding of lo are both <= 2^-22 relative, i.e. fp32-level.
//
//   C[M, N] = A[M, K] @ Bt[N, K]^T        A row-major fp32 (streamed), Bt = the small operand, pre-split and packed
//
// Measured limits (round 1, tests/gemm_timeline.py + ncu): the kernel is bound by the SHARED-MEMORY port, not by the
// tensor pipe: SS-mode MMAs re-read the A tile three times per k-step, the splitter moves 3x the tile bytes and the
// epilogue transposes through shared memory - about 600 KB of shared-memory traffic per 128 x 80 output tile
// (~4,700 cycles at 128 B/cycle).  Next step: A_hi / A_lo in TMEM (tcgen05.st by the splitter, TS-mode MMA).
//
// Persistent CTAs; a CTA owns one column tile of C (NT <= 112 columns) and keeps the hi / lo tiles of Bt for it
// resident in shared memory; warp roles:
//   warp 0      TMA producer: Bt tiles once, then raw fp32 A tiles (128 rows x 32 K, 128-byte swizzle) into a 4-6 deep ring
//   warps 2-9   splitter: raw tile -> hi (in place) + lo tile (element-wise on the swizzled bytes, layout-agnostic),
//               fence.proxy.async, then hand the stage to the MMA warp
//   warp 1      one thread issues 3 tcgen05.mma (M = 128, N = NT, K = 8) per 8-wide k-step
//   warps 10-13 epilogue: tcgen05.ld -> 32x32 transpose through shared memory -> coalesced 128-byte row segments of C
//   warp 14     TMEM allocator (2 accumulator stages)
#include <cuda.h>

#include <cstdlib>
#include "common.cuh"

namespace kgc {
namespace {

constexpr int kBM = 128;                  // rows of A / C per tile (UMMA M)
constexpr int kBK = 32;                   // fp32 elements per K block = one 128-byte swizzle row
constexpr int kUK = 8;                    // K per tf32 MMA
constexpr int kMaxKB = 8;                 // K <= 256
constexpr int kMaxStages = 8;             // raw A ring (TMA targets)
constexpr int kAStages = 4;               // TMEM stages of the split A operand: 32 hi + 32 lo columns each
constexpr int kAccCols = 256;             // two fp32 accumulator stages of 128 columns
constexpr int kTmemColsTS = kAccCols + kAStages * 64;   // 512: the whole tensor memory of the SM
constexpr int kTileA = kBM * kBK * 4;     // 16 KB
constexpr int kThreadsG = 480;            // 15 warps: TMA, MMA, 8 splitters, 4 epilogue, TMEM allocator
constexpr int kSplitWarps = 8;
constexpr int kBBudget = 116 * 1024;      // resident hi + lo tiles of Bt (the rest of shared memory is the A ring:
                                          // the ring must cover TMA latency + split + MMA, ~6 K-blocks in flight)
constexpr int kTmemColsG = 256;
constexpr int kEpiBuf = 32 * 128;          // one epilogue buffer: a TMA-store box of 32 rows x 32 fp32 columns
constexpr int kEpiStage = 4 * 2 * kEpiBuf; // 4 epilogue warps, double buffered (32 KB)

__device__ __forceinline__ uint32_t s_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mb_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(s_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mb_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(s_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mb_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(s_u32(bar)) : "memory");
}
__device__ __forceinline__ void mb_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(s_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          s_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(s_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_3d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          s_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(s_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(map)),
               "r"(s_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, const void* smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(map)),
               "r"(s_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
// TS form: the A operand (128 rows x 8 TF32) is read from tensor memory, [lane 0.., column a_tmem..a_tmem+7]
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n"
      "}" ::"r"(tmem_d),
      "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(acc)
      : "memory");
}
__device__ __forceinline__ void tmem_st16_g(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
      "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
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
// Round to the nearest TF32 (10-bit mantissa, ties away from zero = cvt.rna.tf32.f32), result in fp32 bits.  Done with
// two integer instructions: cvt.rna runs on the quarter-rate conversion pipe (16 lanes / clock / SM), which made the
// splitter warps the bottleneck of both GEMM kernels (measured: ~512 cycles per 128 x 32 tile for the cvt alone).
__device__ __forceinline__ uint32_t tf32_rn(float v) { return (__float_as_uint(v) + 0x1000u) & 0xFFFFE000u; }
__device__ __forceinline__ void split_tf32(uint32_t v, uint32_t& hi, uint32_t& lo) {
  hi = tf32_rn(__uint_as_float(v));
  lo = tf32_rn(__uint_as_float(v) - __uint_as_float(hi));
}
__device__ __forceinline__ void umma_commit_g(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(s_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32_g(uint32_t taddr, uint32_t (&v)[32]) {
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
// K-major tile, 128-byte swizzle (rows of 32 fp32), 8-row atoms 1024 B apart
__device__ __forceinline__ uint64_t sw128_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

constexpr int kMaxBatch = 3;               // problems of one launch (same shapes, different operands): in / out / loop halves
struct GemmMaps {
  CUtensorMap a[kMaxBatch], bhi[kMaxBatch], blo[kMaxBatch], c[kMaxBatch], c16[kMaxBatch];
};

struct GemmParams {
  int64_t M;
  int32_t n_prob;
  int32_t N, K;
  int32_t n_kb, ksteps, NT, n_ntiles, n_mtiles, stages;
  float* C;
  int64_t ldc;
  const float* row_bias;   // optional: C[m, n] = f(acc + row_bias[m])
  int32_t act;             // 0: identity, 1: logistic sigmoid
  int32_t trans_c;         // store C transposed: Ct[n, m] (the tensor maps then describe Ct)
  int32_t trans_a;         // A is given transposed, At[K, M] row-major (M % 32 == 0): tiles land as [m group][k][32 m]
  // optional dropout of the streamed operand while it is split (backward of the layer tail): keep[m * keep_pitch + c] holds
  // the keep flags of columns 4c..4c+3 of row m, low nibble for problem 0, high nibble for problem 1; problem 2 is taken
  // as it is.  A kept element is multiplied by keep_scale = 1 / (1 - p), a dropped one becomes 0.
  const uint8_t* keep;
  int32_t keep_pitch;
  float keep_scale;
  long long* dbg;     // optional timeline of CTA 0: [role][event] clock64 stamps (debug aid)
};

__global__ void __launch_bounds__(kThreadsG, 1)
gemm_tf32x3_kernel(const __grid_constant__ GemmMaps maps, const GemmParams P) {
  extern __shared__ uint8_t smem_raw[];
  if (P.dbg != nullptr && threadIdx.x == 0) {                      // debug aid: launch-to-exit envelope over all CTAs (ns)
    long long g;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(g));
    atomicMin(reinterpret_cast<long long*>(P.dbg) + 8 * 64 + 0, g);
    if (blockIdx.x == 0) { P.dbg[8 * 64 + 2] = g; P.dbg[8 * 64 + 3] = clock64(); }
  }
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
  const int tile_b = P.NT * kBK * 4;                               // bytes of one Bt K-block tile (NT rows x 128 B)
  const int tile_b_al = (tile_b + 1023) & ~1023;                   // keep every tile 1024-byte aligned (swizzle atoms)
  uint8_t* s_bhi = base;                                           // [n_kb][tile_b_al]
  uint8_t* s_blo = s_bhi + P.n_kb * tile_b_al;
  const int kStages = P.stages;
  uint8_t* s_a = s_blo + P.n_kb * tile_b_al;                       // [stages][16 KB] raw fp32 tiles (TMA targets)
  uint8_t* s_stage = s_a + kStages * kTileA;                       // [4 epilogue warps][2 buffers][32 x 32 floats]
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_stage + kEpiStage);
  uint64_t* b_full = bars;
  uint64_t* raw_full = bars + 1;                                   // [kMaxStages] TMA landed
  uint64_t* raw_empty = raw_full + kMaxStages;                     // [kMaxStages] splitters have read the raw stage
  uint64_t* split_full = raw_empty + kMaxStages;                   // [kAStages] hi / lo of a K block are in TMEM
  uint64_t* split_empty = split_full + kAStages;                   // [kAStages] MMAs done with the TMEM A stage
  uint64_t* acc_full = split_empty + kAStages;                     // [2]
  uint64_t* acc_empty = acc_full + 2;                              // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

  if (warp == 0 && lane == 0) {
    mb_init(b_full, 1);
    for (int i = 0; i < kStages; ++i) {
      mb_init(raw_full + i, 1);
      mb_init(raw_empty + i, kSplitWarps);
    }
    for (int i = 0; i < kAStages; ++i) {
      mb_init(split_full + i, kSplitWarps);
      mb_init(split_empty + i, 1);
    }
    for (int i = 0; i < 2; ++i) {
      mb_init(acc_full + i, 1);
      mb_init(acc_empty + i, 4);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 14) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s_u32(tmem_slot)), "r"(kTmemColsTS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_a = tmem_base + kAccCols;                    // A stages: [kAStages][hi 32 columns | lo 32 columns]
  const bool dbg_on = P.dbg != nullptr && blockIdx.x == 0;
  int dbg_n = 0;
#define KGC_DBG(role) do { if (dbg_on && dbg_n < 64) P.dbg[(role) * 64 + dbg_n++] = clock64(); } while (0)

  // work: this CTA owns column tile nt of problem prob and the row tiles mt = first, first + step, ...
  const int groups = P.n_prob * P.n_ntiles;                        // host launches a multiple of groups CTAs
  const int prob = (blockIdx.x % groups) / P.n_ntiles;
  const int nt = blockIdx.x % P.n_ntiles;
  const int first = blockIdx.x / groups;
  const int step = gridDim.x / groups;
  const CUtensorMap* map_a = &maps.a[prob];
  const CUtensorMap* map_bhi = &maps.bhi[prob];
  const CUtensorMap* map_blo = &maps.blo[prob];
  const CUtensorMap* map_c = &maps.c[prob];
  const CUtensorMap* map_c16 = &maps.c16[prob];

  if (warp == 0) {
    if (lane == 0) {
      mb_expect_tx(b_full, 2u * P.n_kb * tile_b);
      for (int kb = 0; kb < P.n_kb; ++kb) {
        tma_2d(s_bhi + kb * tile_b_al, map_bhi, b_full, kb * kBK, nt * P.NT);
        tma_2d(s_blo + kb * tile_b_al, map_blo, b_full, kb * kBK, nt * P.NT);
      }
      int stage = 0;
      uint32_t phase = 0;
      for (int mt = first; mt < P.n_mtiles; mt += step) {
        for (int kb = 0; kb < P.n_kb; ++kb) {
          mb_wait(raw_empty + stage, phase ^ 1);
          KGC_DBG(0);
          mb_expect_tx(raw_full + stage, kTileA);
          if (P.trans_a) tma_3d(s_a + stage * kTileA, map_a, raw_full + stage, 0, kb * kBK, mt * (kBM / 32));
          else tma_2d(s_a + stage * kTileA, map_a, raw_full + stage, kb * kBK, mt * kBM);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp >= 2 && warp < 2 + kSplitWarps) {
    // ================================================================== splitter: raw row -> (hi, lo) in TENSOR MEMORY
    // A warp can only touch the TMEM lanes of its quarter (warp % 4); two warps share a quarter and take 16 of the 32
    // K columns each.  Thread = row r of the tile: its 128-byte row sits at r * 128 with the 16-byte chunks XOR-ed by
    // r % 8 (TMA 128-byte swizzle) - 8 consecutive rows hit 8 different chunks, so the LDS.128 are conflict-free.
    const int quarter = warp % 4, half = (warp - 2) / 4;
    const int r = quarter * 32 + lane;
    int stage = 0, ts = 0;
    uint32_t phase = 0, tphase = 0;
    // dropout of the streamed operand (P.keep): the 64 keep bytes of this thread's row cover all K blocks of a tile; they
    // are loaded ONE TILE AHEAD (a global load inside the per-K-block chain costs its full latency every block: measured
    // +2.2 ms per launch at the Wikidata5M shape) and this thread's word of a K block is picked with a select chain
    // (a runtime index into the register array would send it to local memory)
    const bool masked = P.keep != nullptr && prob < 2 && !P.trans_a;
    uint32_t kcur[kMaxKB], knxt[kMaxKB];
#pragma unroll
    for (int j = 0; j < kMaxKB; ++j) kcur[j] = knxt[j] = 0u;
    auto load_keep = [&](int mt_, uint32_t (&w)[kMaxKB]) {
      const int64_t grow = (int64_t)mt_ * kBM + r;
      if (mt_ < P.n_mtiles && grow < P.M) {
        const uint4* kp = reinterpret_cast<const uint4*>(P.keep + grow * P.keep_pitch);
#pragma unroll
        for (int q = 0; q < kMaxKB / 2; ++q) {                     // 16 bytes = K blocks 2q, 2q + 1: words (kb, half 0), (kb, half 1)
          const uint4 t4 = __ldg(kp + q);
          w[2 * q] = half ? t4.y : t4.x;
          w[2 * q + 1] = half ? t4.w : t4.z;
        }
      }
    };
    if (masked) load_keep(first, knxt);
    for (int mt = first; mt < P.n_mtiles; mt += step) {
      if (masked) {
#pragma unroll
        for (int j = 0; j < kMaxKB; ++j) kcur[j] = knxt[j];
        load_keep(mt + step, knxt);
      }
      for (int kb = 0; kb < P.n_kb; ++kb) {
        uint32_t kw = 0;                                           // keep flags of this thread's 16 columns (4 bytes)
        if (masked) {
#pragma unroll
          for (int j = 0; j < kMaxKB; ++j)
            if (kb == j) kw = kcur[j];
          if (prob == 1) kw >>= 4;
        }
        mb_wait(raw_full + stage, phase);
        if (warp == 2 && lane == 0) KGC_DBG(1);
        uint32_t h[16], l[16];
        if (P.trans_a) {
          // At tile: box (32 m, 32 k) per m group = quarter; this thread's row m = lane is a COLUMN of the box: k-th
          // value at row k, 16-byte chunk (lane / 4) ^ (k % 8) - the 32 lanes of a warp hit 32 different banks
          const uint8_t* col = s_a + stage * kTileA + quarter * 4096 + ((lane & 3) << 2);
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const int kk = half * 16 + i;
            const uint32_t v = *reinterpret_cast<const uint32_t*>(col + kk * 128 + (((lane >> 2) ^ (kk & 7)) << 4));
            split_tf32(v, h[i], l[i]);
          }
        } else {
          const uint8_t* row = s_a + stage * kTileA + r * 128;
          uint4 v[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) v[i] = *reinterpret_cast<const uint4*>(row + (((half * 4 + i) ^ (r & 7)) << 4));
          if (masked) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const uint32_t nb = kw >> (8 * i);
              v[i].x = (nb & 1u) ? __float_as_uint(__uint_as_float(v[i].x) * P.keep_scale) : 0u;
              v[i].y = (nb & 2u) ? __float_as_uint(__uint_as_float(v[i].y) * P.keep_scale) : 0u;
              v[i].z = (nb & 4u) ? __float_as_uint(__uint_as_float(v[i].z) * P.keep_scale) : 0u;
              v[i].w = (nb & 8u) ? __float_as_uint(__uint_as_float(v[i].w) * P.keep_scale) : 0u;
            }
          }
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            // hi = nearest TF32, lo = nearest TF32 of (v - hi): measurably tighter than truncation at K = 200
            split_tf32(v[i].x, h[4 * i + 0], l[4 * i + 0]);
            split_tf32(v[i].y, h[4 * i + 1], l[4 * i + 1]);
            split_tf32(v[i].z, h[4 * i + 2], l[4 * i + 2]);
            split_tf32(v[i].w, h[4 * i + 3], l[4 * i + 3]);
          }
        }
        __syncwarp();
        if (lane == 0) mb_arrive(raw_empty + stage);               // the raw tile is in registers: hand the stage back to TMA
        mb_wait(split_empty + ts, tphase ^ 1);                     // the MMAs that read this TMEM stage have retired
        if (warp == 2 && lane == 0) KGC_DBG(2);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t taddr = tmem_a + ((uint32_t)(quarter * 32) << 16) + ts * 64 + half * 16;
        tmem_st16_g(taddr, h);
        tmem_st16_g(taddr + 32, l);
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) mb_arrive(split_full + ts);
        if (warp == 2 && lane == 0) KGC_DBG(3);
        if (++stage == kStages) { stage = 0; phase ^= 1; }
        if (++ts == kAStages) { ts = 0; tphase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ================================================================== MMA issuer (warp-uniform loop, one elected lane issues)
    {
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(P.NT >> 3) << 17) | ((uint32_t)(kBM >> 4) << 24);
      int ts = 0, acc = 0;
      uint32_t tphase = 0, acc_phase = 0;
      mb_wait(b_full, 0);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      for (int mt = first; mt < P.n_mtiles; mt += step) {
        mb_wait(acc_empty + acc, acc_phase ^ 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t d_addr = tmem_base + acc * (kAccCols / 2);
        for (int kb = 0; kb < P.n_kb; ++kb) {
          mb_wait(split_full + ts, tphase);
          if (lane == 0) KGC_DBG(4);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const int nk = min(kBK / kUK, P.ksteps - kb * (kBK / kUK));
          const uint32_t a_hi = tmem_a + ts * 64, a_lo = a_hi + 32;            // TS mode: the A operand is read from TMEM
          const uint64_t b_hi = sw128_desc(s_u32(s_bhi + kb * tile_b_al));
          const uint64_t b_lo = sw128_desc(s_u32(s_blo + kb * tile_b_al));
          if (elect_one()) {
            // straight-line issue (a runtime trip count makes the loop carry R2UR moves and ~20 uniform-datapath
            // instructions per step: measured on the K6 scorer, +6%)
#pragma unroll
            for (int k = 0; k < kBK / kUK; ++k) {                  // + 8 TMEM columns / + 32 bytes (2 descriptor units) along K
              if (k < nk) {
                umma_tf32_ts(d_addr, a_lo + 8 * k, b_hi + 2 * k, idesc, (k != 0 || kb != 0) ? 1u : 0u);    // small terms first
                umma_tf32_ts(d_addr, a_hi + 8 * k, b_lo + 2 * k, idesc, 1u);
                umma_tf32_ts(d_addr, a_hi + 8 * k, b_hi + 2 * k, idesc, 1u);
              }
            }
            umma_commit_g(split_empty + ts);
            if (kb == P.n_kb - 1) umma_commit_g(acc_full + acc);
          }
          __syncwarp();
          if (lane == 0) KGC_DBG(5);
          if (++ts == kAStages) { ts = 0; tphase ^= 1; }
        }
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp >= 10 && warp <= 13) {
    // ================================================================== epilogue: TMEM -> swizzled smem boxes -> TMA store
    // A thread owns a TMEM lane (= a row of C).  Storing rows straight from registers (or 128-byte row segments after
    // a shared-memory transpose) keeps the LSU busy for ~1,400 cycles per 32 x 32 block (measured); instead each warp
    // lays its 32 x 32 block out as a TMA box (128-byte rows, 128-byte swizzle: conflict-free 16-byte stores; a
    // 16-column tail of the tile uses a 64-byte-swizzled box) and one lane hands it to the TMA engine, which also
    // clips rows >= M and columns >= N.  Wide rows matter: the engine retires one row request at a time.
    const int quarter = warp % 4;
    uint8_t* stg = s_stage + (warp - 10) * (2 * kEpiBuf);          // two buffers of one box
    const int64_t row_q = quarter * 32;
    int acc = 0, buf = 0;
    uint32_t acc_phase = 0;
    for (int mt = first; mt < P.n_mtiles; mt += step) {
      mb_wait(acc_full + acc, acc_phase);
      if (warp == 10 && lane == 0) KGC_DBG(6);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const int64_t m0 = (int64_t)mt * kBM + row_q;
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * (kAccCols / 2);
      for (int c0 = 0; c0 < P.NT; c0 += 32) {
        uint32_t v[32];
        tmem_ld32_g(taddr + c0, v);                                // columns past NT belong to the allocation: never stored
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        if (c0 + 32 >= P.NT) {                                     // last read of this accumulator: give it back to the MMA warp
          asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
          __syncwarp();
          if (lane == 0) mb_arrive(acc_empty + acc);
        }
        // the TMA store that read this buffer two blocks ago must have drained it (bulk groups are per thread: lane 0)
        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
        __syncwarp();
        uint8_t* bb = stg + buf * kEpiBuf;
        const bool wide = c0 + 32 <= P.NT;                         // 32-column box (128-byte rows), else the 16-column tail box
        if (P.row_bias != nullptr) {                               // 1-N scoring: + bias[entity], logistic sigmoid (model.py:178-179)
          const float bv = m0 + lane < P.M ? P.row_bias[m0 + lane] : 0.f;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float z = __uint_as_float(v[j]) + bv;
            v[j] = __float_as_uint(P.act == 1 ? 1.f / (1.f + expf(-z)) : z);
          }
        }
        if (P.trans_c) {
          // transposed block: element (row = lane, column j) -> box row j, 4-byte slot lane (bank = a permutation of lane)
#pragma unroll
          for (int j = 0; j < 32; ++j)
            *reinterpret_cast<uint32_t*>(bb + j * 128 + ((((lane >> 2) ^ (j & 7)) << 4) | ((lane & 3) << 2))) = v[j];
        } else if (wide) {
          uint8_t* bx = bb + lane * 128;
          const int sw = lane & 7;
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<uint4*>(bx + ((q ^ sw) << 4)) = make_uint4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
        } else {
          uint8_t* bx = bb + lane * 64;
          const int sw = (lane >> 1) & 3;
#pragma unroll
          for (int q = 0; q < 4; ++q)
            *reinterpret_cast<uint4*>(bx + ((q ^ sw) << 4)) = make_uint4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) {
          const int col = nt * P.NT + c0;
          if (m0 < P.M && col < P.N) {
            if (P.trans_c) tma_store_2d(wide ? map_c : map_c16, bb, (int)m0, col);     // Ct: inner coordinate = row of C
            else tma_store_2d(wide ? map_c : map_c16, bb, col, (int)m0);
          }
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        buf ^= 1;
      }
      if (warp == 10 && lane == 0) KGC_DBG(7);
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // all stores complete before the CTA exits
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (P.dbg != nullptr && threadIdx.x == 0) {
    long long g;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(g));
    atomicMax(reinterpret_cast<long long*>(P.dbg) + 8 * 64 + 1, g);
    if (blockIdx.x == 0) { P.dbg[8 * 64 + 4] = g; P.dbg[8 * 64 + 5] = clock64(); }
  }
  if (warp == 14) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemColsTS) : "memory");
  }
}

// Bt_hi / Bt_lo [n_pad, k_pad] from B viewed as element (k, n) = B[k * sk + n * sn]; zero padded
__global__ void pack_b_kernel(const float* __restrict__ B, int64_t sk, int64_t sn, int N, int K, int n_pad, int k_pad,
                              float* __restrict__ hi, float* __restrict__ lo) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_pad * k_pad) return;
  const int n = i / k_pad, k = i % k_pad;
  float v = 0.f;
  if (n < N && k < K) v = B[(int64_t)k * sk + (int64_t)n * sn];
  uint32_t h, l;
  split_tf32(__float_as_uint(v), h, l);
  hi[i] = __uint_as_float(h);
  lo[i] = __uint_as_float(l);
}

// ---------------------------------------------------------------------------------------------------------------
// Parameter-side work of one MGCNConv step, batched.  The layer's small operands (three [D, Dout] weights, the relation
// table, two [1, D] self-loop vectors) need ~20 tiny tensor operations per step in the reference formulation
// (model.py:86, 92-94, 107 and their autograd); each costs a launch (~2 us inside a CUDA graph) for a few KB of work.
struct PrepArgs {
  const float *rels, *loop_rel, *loop_edge, *w0, *w1, *w2, *w_rel;   // w0..2: in, out, loop (no array: a runtime index
                                                                     // into a by-value parameter forces a local-memory copy)
  int n_rels, D, Dout;
  int n_pad_f, k_pad_f, n_pad_b, k_pad_b;                         // packed layouts of W (N = Dout, K = D) and W^T (N = D, K = Dout)
  float *relp, *all_rel, *packed_f, *packed_b;
};

__global__ void __launch_bounds__(256) conv_prep_kernel(const PrepArgs a) {
  const int T = a.n_rels + 1;
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int n0 = T * a.D, n1 = T * a.Dout, nf = a.n_pad_f * a.k_pad_f, nb = a.n_pad_b * a.k_pad_b;
  if (i < n0) {                                                   // relp = cat(rels, loop_rel)   (model.py:86)
    const int t = i / a.D, c = i % a.D;
    a.relp[i] = t < a.n_rels ? a.rels[i] : a.loop_rel[c];
    return;
  }
  i -= n0;
  if (i < n1) {                                                   // all_rel = relp @ w_rel        (model.py:107)
    const int t = i / a.Dout, o = i % a.Dout;
    const float* r = t < a.n_rels ? a.rels + (int64_t)t * a.D : a.loop_rel;
    float acc = 0.f;
#pragma unroll 25
    for (int c = 0; c < a.D; ++c) acc = fmaf(r[c], a.w_rel[(int64_t)c * a.Dout + o], acc);   // unrolled: 25 loads in flight
    a.all_rel[i] = acc;
    return;
  }
  i -= n1;
  if (i < 3 * nf) {                                               // Bt[n, k] = W_h[k, n]  (x loop_rel[k] loop_edge[k] for the self-loop)
    // consecutive threads take consecutive n: coalesced reads of the row-major weight (the strided 4-byte writes are cheap)
    const int h = i / nf, j0 = i % nf, k = j0 / a.n_pad_f, n = j0 % a.n_pad_f, j = n * a.k_pad_f + k;
    float v = 0.f;
    if (n < a.Dout && k < a.D) {
      const float* wh = h == 0 ? a.w0 : (h == 1 ? a.w1 : a.w2);
      v = wh[(int64_t)k * a.Dout + n];
      if (h == 2) v *= a.loop_rel[k] * a.loop_edge[k];
    }
    uint32_t hi, lo;
    split_tf32(__float_as_uint(v), hi, lo);
    float* dst = a.packed_f + (int64_t)h * 2 * nf;
    dst[j] = __uint_as_float(hi);
    dst[nf + j] = __uint_as_float(lo);
    return;
  }
  i -= 3 * nf;
  if (i < 4 * nb) {                                               // Bt[n, k] = W_h^T[k, n] = W_h[n, k]; h = 3: the relation transform
    const int h = i / nb, j = i % nb, n = j / a.k_pad_b, k = j % a.k_pad_b;
    float v = 0.f;
    if (n < a.D && k < a.Dout) {
      const float* wh = h == 0 ? a.w0 : (h == 1 ? a.w1 : (h == 2 ? a.w2 : a.w_rel));
      v = wh[(int64_t)n * a.Dout + k];
      if (h == 2) v *= a.loop_rel[n] * a.loop_edge[n];
    }
    uint32_t hi, lo;
    split_tf32(__float_as_uint(v), hi, lo);
    float* dst = a.packed_b + (int64_t)h * 2 * nb;
    dst[j] = __uint_as_float(hi);
    dst[nb + j] = __uint_as_float(lo);
  }
}

struct ParamGradArgs {
  const float *m_loop, *w_loop, *loop_rel, *loop_edge, *relp, *w_rel, *g_rel, *d_relp;
  int n_rels, D, Dout;
  float *d_w_loop, *d_loop_rel, *d_loop_edge, *d_rels, *d_w_rel;
};

__global__ void __launch_bounds__(256) conv_param_grads_kernel(const ParamGradArgs a) {
  const int T = a.n_rels + 1;
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int nw = a.D * a.Dout;
  if (i < nw) {                                                   // d_w_loop = diag(loop_rel . loop_edge) m_loop
    const int c = i / a.Dout;
    a.d_w_loop[i] = a.loop_rel[c] * a.loop_edge[c] * a.m_loop[i];
    return;
  }
  i -= nw;
  if (i < nw) {                                                   // d_w_rel = relp^T @ [g_rel; 0]
    const int c = i / a.Dout, o = i % a.Dout;
    float acc = 0.f;
    if (a.g_rel != nullptr) {
#pragma unroll 8
      for (int t = 0; t < a.n_rels; ++t) acc = fmaf(a.relp[(int64_t)t * a.D + c], a.g_rel[(int64_t)t * a.Dout + o], acc);
    }
    a.d_w_rel[i] = acc;
    return;
  }
  i -= nw;
  // one WARP per (t, c): the lanes stride over Dout (coalesced rows of g_rel / w_rel / m_loop / w_loop), fixed shuffle tree
  const int pair = i / 32, lane = i % 32;
  if (pair < T * a.D) {                                           // d_relp + [g_rel; 0] @ w_rel^T; last row -> the self-loop vectors
    const int t = pair / a.D, c = pair % a.D;
    const float* u = t < a.n_rels ? a.g_rel + (int64_t)t * a.Dout : a.m_loop + (int64_t)c * a.Dout;
    const float* w = t < a.n_rels ? a.w_rel + (int64_t)c * a.Dout : a.w_loop + (int64_t)c * a.Dout;
    float acc = 0.f;
    if (t == a.n_rels || a.g_rel != nullptr)
      for (int o = lane; o < a.Dout; o += 32) acc = fmaf(u[o], w[o], acc);
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, s);
    if (lane == 0) {
      const float val = a.d_relp[pair];
      if (t < a.n_rels) {
        a.d_rels[pair] = val + acc;
      } else {                                                    // acc = d_v[c] = sum_o m_loop[c, o] w_loop[c, o]
        a.d_loop_edge[c] = acc * a.loop_rel[c];
        a.d_loop_rel[c] = acc * a.loop_edge[c] + val;
      }
    }
  }
}

// The same gradients when the two products over the relation rows - d_w_rel = relp^T [g_rel; 0] and rel_add = g_rel w_rel^T -
// were computed by K4c / K4b (at 1,644 relation rows the loops above are 0.29 ms of serial work per thread).
__global__ void __launch_bounds__(256) conv_param_grads2_kernel(const ParamGradArgs a, const float* __restrict__ rel_add) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int nw = a.D * a.Dout;
  if (i < nw) {
    const int c = i / a.Dout;
    a.d_w_loop[i] = a.loop_rel[c] * a.loop_edge[c] * a.m_loop[i];
    return;
  }
  i -= nw;
  const int n_el = a.n_rels * a.D, n_el_pad = (n_el + 31) & ~31;  // the warps of the last region must be whole hardware warps
  if (i < n_el_pad) {
    if (i < n_el) a.d_rels[i] = a.d_relp[i] + rel_add[i];
    return;
  }
  i -= n_el_pad;
  const int c = i / 32, lane = i % 32;
  if (c < a.D) {                                                  // self-loop row: d_v[c] = sum_o m_loop[c, o] w_loop[c, o]
    const float* u = a.m_loop + (int64_t)c * a.Dout;
    const float* w = a.w_loop + (int64_t)c * a.Dout;
    float acc = 0.f;
    for (int o = lane; o < a.Dout; o += 32) acc = fmaf(u[o], w[o], acc);
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, s);
    if (lane == 0) {
      a.d_loop_edge[c] = acc * a.loop_rel[c];
      a.d_loop_rel[c] = acc * a.loop_edge[c] + a.d_relp[(int64_t)a.n_rels * a.D + c];
    }
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
int encode_fn(EncodeTiledFn* out) {
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
// fp32 [rows, cols] with row pitch `pitch` floats -> boxes of 32 (K) x box_rows, 128-byte swizzle, zero fill
int make_map_f32(CUtensorMap* map, const void* ptr, int64_t rows, int64_t cols, int64_t pitch, int box_rows,
                 CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B, int box_cols = kBK) {
  EncodeTiledFn enc;
  if (encode_fn(&enc)) return 1;
  KGC_REQUIRE((reinterpret_cast<uintptr_t>(ptr) & 15) == 0 && (pitch * 4) % 16 == 0, "operand must be 16-byte aligned with a 16-byte pitch");
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)pitch * 4};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  KGC_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")");
  return 0;
}

// 32-column groups of fp32 [rows, cols] fetched by ONE box: dims (32 columns, rows, groups), group stride 128 B;
// the box takes 32 rows x box_groups groups and lands as [group][row][32 columns]
int make_map_f32_groups(CUtensorMap* map, const void* ptr, int64_t rows, int groups, int64_t pitch, int box_groups,
                        CUtensorMapSwizzle swizzle) {
  EncodeTiledFn enc;
  if (encode_fn(&enc)) return 1;
  KGC_REQUIRE((reinterpret_cast<uintptr_t>(ptr) & 15) == 0 && (pitch * 4) % 16 == 0, "operand must be 16-byte aligned with a 16-byte pitch");
  cuuint64_t dims[3] = {32, (cuuint64_t)rows, (cuuint64_t)groups};
  cuuint64_t strides[2] = {(cuuint64_t)pitch * 4, 128};
  cuuint32_t box[3] = {32, 32, (cuuint32_t)box_groups};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  KGC_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (grouped operand) failed (" + std::to_string((int)r) + ")");
  return 0;
}
int make_map_f32_mn_groups(CUtensorMap* map, const void* ptr, int64_t rows, int groups, int64_t pitch) {
  return make_map_f32_groups(map, ptr, rows, groups, pitch, groups, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B);
}

// partial sums [parts][rows][cols] fp32 -> boxes of 32 columns x 32 rows of one part, 128-byte swizzle (TMA stores clip)
int make_map_f32_parts(CUtensorMap* map, const void* ptr, int64_t parts, int64_t rows, int64_t cols) {
  EncodeTiledFn enc;
  if (encode_fn(&enc)) return 1;
  KGC_REQUIRE((reinterpret_cast<uintptr_t>(ptr) & 15) == 0 && cols % 4 == 0, "partials must be 16-byte aligned with a 16-byte pitch");
  cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)parts};
  cuuint64_t strides[2] = {(cuuint64_t)cols * 4, (cuuint64_t)rows * cols * 4};
  cuuint32_t box[3] = {32, 32, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  KGC_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")");
  return 0;
}

struct Tiling {
  int n_kb, k_pad, ksteps, NT, n_ntiles, n_pad;
};
int make_tiling(int N, int K, Tiling* t) {
  if (N <= 0 || K <= 0 || K > kMaxKB * kBK || N > 1024) return 1;
  t->n_kb = (K + kBK - 1) / kBK;
  t->k_pad = t->n_kb * kBK;
  t->ksteps = (K + kUK - 1) / kUK;
  int nt_max = kBBudget / (2 * t->n_kb * kBK * 4);
  nt_max = nt_max / 16 * 16;
  if (nt_max > 128) nt_max = 128;
  if (nt_max < 16) return 1;
  t->n_ntiles = (N + nt_max - 1) / nt_max;
  t->NT = ((N + t->n_ntiles - 1) / t->n_ntiles + 15) / 16 * 16;
  t->n_pad = t->NT * t->n_ntiles;
  return 0;
}


// ================================================================================================================
// Weight-gradient reduction on the tensor cores:  C[Ka, Nb] = A[M, Ka]^T @ B[M, Nb]  (contraction over the node rows)
//
// Both operands are MN-major for the MMA (the contraction index m is the SLOW index of both row-major arrays): a TMA
// box of 32 columns x 32 rows lands as 32 swizzled 128-byte rows = eight 4-row K atoms of an MN-major
// SWIZZLE_128B_BASE32B operand; the boxes of consecutive 32-column groups sit kTnBox bytes apart (leading byte offset),
// 4-row atoms 512 bytes apart (stride byte offset).  One tcgen05.mma kind::tf32 consumes 8 rows (K = 8 = two atoms).  Both operands are streamed, so both are split
// (hi in place, lo into a second ring) by the splitter warps; D[128 x 208] stays in TMEM for the CTA's whole row slab
// and is written once as a partial; partials are added in CTA order by gemm_tn_partials_reduce (deterministic).
constexpr int kTnRows = 32;                      // node rows per K block
constexpr int kTnBox = kTnRows * 128;            // one 32-column x 32-row box: 4 KB
constexpr int kTnStages = 3;
constexpr int kTnLoStages = 2;
constexpr int kTnMaxGb = 7;                      // 32-column groups of B: Nb <= 224

struct GemmTnMaps {                              // per problem of a batched launch
  CUtensorMap a[kMaxBatch], b[kMaxBatch], a3[kMaxBatch], b3[kMaxBatch], p[kMaxBatch];
};

struct GemmTnParams {
  int64_t M;
  int64_t m_prob[kMaxBatch];                     // rows of each problem (<= M; fewer for a compacted plane): slabs past them
                                                 // have no CTA work and no partial
  int32_t n_prob, n_slabs;                       // CTA = (problem, row slab); partial[problem][slab][Ka][Nb]
  int32_t Ka, Nb, ga, gb, n_pad;                 // ga / gb = 32-column groups of A / B; n_pad = MMA N (multiple of 16)
  int32_t ga_full, gb_full;                      // groups that lie completely inside the operand (fetched by one 3-D TMA)
  int32_t kmajor;                                // split-K product of K-major operands (see kgc_gemm_nt_splitk)
  int64_t rows_per_cta;
  float* partial;                                // [grid][Ka][Nb]
  const uint8_t* keep;                           // optional dropout of the B operand while it is split (see GemmParams::keep)
  int32_t keep_pitch;
  float keep_scale;
  long long* dbg;                                // optional timeline of CTA 0 (debug aid, see kgc_gemm_set_debug)
};

// MN-major TF32 operands have ONE legal shared-memory layout on sm_100: 128-byte swizzle with 32-byte atoms
// (UMMA layout type SWIZZLE_128B_BASE32B, TMA CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B): rows of 128 B (32 MN elements),
// 4-row K atoms (32-byte chunks XOR-ed with row % 4), atoms 512 B apart along K, MN groups kTnBox apart.
__device__ __forceinline__ uint64_t sw128_mn_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);            // start address
  d |= (uint64_t)(kTnBox >> 4) << 16;                     // leading byte offset: next 32-element MN group
  d |= (uint64_t)(512 >> 4) << 32;                        // stride byte offset: next 4-row K atom
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)1 << 61;                                 // SWIZZLE_128B_BASE32B
  return d;
}

__global__ void __launch_bounds__(kThreadsG, 1)
gemm_tn_tc_kernel(const __grid_constant__ GemmTnMaps maps, const GemmTnParams P) {
  extern __shared__ uint8_t smem_raw[];
  const int prob = blockIdx.x % P.n_prob, slab = blockIdx.x / P.n_prob;
  const int64_t Mp = prob == 0 ? P.m_prob[0] : (prob == 1 ? P.m_prob[1] : P.m_prob[2]);
  const int64_t m0 = slab * P.rows_per_cta;
  if (m0 >= Mp && Mp < P.M) return;                                // a slab past a shorter problem's rows: not reduced
  if (P.dbg != nullptr && threadIdx.x == 0) {                      // debug aid: launch-to-exit envelope over all CTAs (ns)
    long long g;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(g));
    atomicMin(reinterpret_cast<long long*>(P.dbg) + 8 * 64 + 0, g);
    if (blockIdx.x == 0) { P.dbg[8 * 64 + 2] = g; P.dbg[8 * 64 + 3] = clock64(); }
  }
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
  const int stage_bytes = (P.ga + P.gb) * kTnBox;          // A boxes then B boxes
  uint8_t* s_raw = base;                                   // [kTnStages][stage_bytes]  raw -> hi (in place)
  uint8_t* s_lo = s_raw + kTnStages * stage_bytes;         // [kTnLoStages][stage_bytes]
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_lo + kTnLoStages * stage_bytes);
  uint64_t* raw_full = bars;                               // [kTnStages]
  uint64_t* split_full = raw_full + kTnStages;             // [kTnStages]
  uint64_t* empty = split_full + kTnStages;                // [kTnStages]
  uint64_t* lo_empty = empty + kTnStages;                  // [kTnLoStages]
  uint64_t* acc_full = lo_empty + kTnLoStages;             // [1]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < kTnStages; ++i) {
      mb_init(raw_full + i, 1);
      mb_init(split_full + i, kSplitWarps);
      mb_init(empty + i, 1);
    }
    for (int i = 0; i < kTnLoStages; ++i) mb_init(lo_empty + i, 1);
    mb_init(acc_full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 14) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s_u32(tmem_slot)), "r"(kTmemColsG)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  const bool dbg_on = P.dbg != nullptr && blockIdx.x == 0;
  int dbg_n = 0;

  const CUtensorMap* map_a = &maps.a[prob];
  const CUtensorMap* map_b = &maps.b[prob];
  const CUtensorMap* map_a3 = &maps.a3[prob];
  const CUtensorMap* map_b3 = &maps.b3[prob];
  const CUtensorMap* map_p = &maps.p[prob];
  const int64_t m1 = m0 + P.rows_per_cta < Mp ? m0 + P.rows_per_cta : Mp;
  const int n_kb = m1 > m0 ? (int)((m1 - m0 + kTnRows - 1) / kTnRows) : 0;

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int kb = 0; kb < n_kb; ++kb) {
        mb_wait(empty + stage, phase ^ 1);
        KGC_DBG(0);
        uint8_t* dst = s_raw + stage * stage_bytes;
        const int row = (int)(m0 + (int64_t)kb * kTnRows);
        if (P.kmajor) {
          // K-major operands A[Ka, K], Bt[Nb, K]: a K block is 32 contraction COLUMNS; A lands as 128 rows x 128 B,
          // Bt as n_pad rows x 128 B (128-byte swizzle), rows past Ka / Nb and columns past K zero-filled by TMA
          mb_expect_tx(raw_full + stage, (uint32_t)(kTileA + P.n_pad * 128));
          tma_2d(dst, map_a, raw_full + stage, row, 0);
          tma_2d(dst + kTileA, map_b, raw_full + stage, row, 0);
          if (++stage == kTnStages) { stage = 0; phase ^= 1; }
          continue;
        }
        mb_expect_tx(raw_full + stage, (uint32_t)stage_bytes);
        // rows past m1 belong to the next CTA's slab: they are masked out by the splitter (zeroed), rows past M are
        // zero-filled by TMA
        // one instruction fetches all the complete 32-column groups of an operand (a TMA issue costs ~170 cycles of the
        // producer thread); the ragged last group and the all-padding groups go through the zero-filling 2-D map
        if (P.ga_full > 0) tma_3d(dst, map_a3, raw_full + stage, 0, row, 0);
        for (int g = P.ga_full; g < P.ga; ++g) tma_2d(dst + g * kTnBox, map_a, raw_full + stage, g * 32, row);
        if (P.gb_full > 0) tma_3d(dst + P.ga * kTnBox, map_b3, raw_full + stage, 0, row, 0);
        for (int g = P.gb_full; g < P.gb; ++g) tma_2d(dst + (P.ga + g) * kTnBox, map_b, raw_full + stage, g * 32, row);
        if (++stage == kTnStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp >= 2 && warp < 2 + kSplitWarps) {
    const int t = threadIdx.x - 64;
    constexpr int kSplitThreads = kSplitWarps * 32;
    int stage = 0, ls = 0;
    uint32_t phase = 0, lphase = 0;
    const int n_vec = stage_bytes / 16;
    const bool masked = P.keep != nullptr && prob < 2 && !P.kmajor;
    const int brow_t = (t & 255) >> 3;                                            // this thread's row inside every box
    const int c16_t = ((((t & 7) >> 1) ^ (brow_t & 3)) << 1) | (t & 1);           // ... and its 16-byte column chunk
    uint32_t nbn[kTnMaxGb];
#pragma unroll
    for (int g = 0; g < kTnMaxGb; ++g) nbn[g] = 0u;
    if (masked && n_kb > 0 && m0 + brow_t < m1) {
      const uint8_t* kp = P.keep + (m0 + brow_t) * P.keep_pitch + c16_t;
#pragma unroll
      for (int g = 0; g < kTnMaxGb; ++g)
        if (g < P.gb) nbn[g] = (uint32_t)__ldg(kp + g * 8);
    }
    for (int kb = 0; kb < n_kb; ++kb) {
      mb_wait(raw_full + stage, phase);
      if (t == 0) KGC_DBG(1);
      mb_wait(lo_empty + ls, lphase ^ 1);
      if (t == 0) KGC_DBG(2);
      uint4* hi = reinterpret_cast<uint4*>(s_raw + stage * stage_bytes);
      uint4* lo = reinterpret_cast<uint4*>(s_lo + ls * stage_bytes);
      // rows of this K block that lie past the CTA's slab must not contribute: a 16-byte vector v of a box belongs to
      // box row (v % 256) / 8  (32 rows x 8 vectors per box; the swizzle permutes vectors only inside a row)
      const int rows_valid = P.kmajor ? kTnRows : (int)min((int64_t)kTnRows, m1 - (m0 + (int64_t)kb * kTnRows));
      if (masked) {
        // B operand = the upstream plane, dropped while it is split.  With 256 splitter threads the k-th trip of a thread
        // handles box k: boxes 0..3 = A, box 4 + g = 32-column group g of B; the thread's position inside a box is fixed:
        // row brow = t / 8, and (un-swizzling: the 32-byte chunks of a 128-byte row are XOR-ed with row % 4, layout
        // SWIZZLE_128B_BASE32B; the 16-byte half is kept) 16-byte column chunk c16 -> ONE keep byte per trip.  The bytes
        // of the NEXT K block are loaded before this one is processed (see the K4b splitter).
        uint32_t nbc[kTnMaxGb];
#pragma unroll
        for (int g = 0; g < kTnMaxGb; ++g) nbc[g] = nbn[g];
        if (kb + 1 < n_kb) {
          const uint8_t* kp = P.keep + (m0 + (int64_t)(kb + 1) * kTnRows + brow_t) * P.keep_pitch + c16_t;
          const bool ok = m0 + (int64_t)(kb + 1) * kTnRows + brow_t < m1;
#pragma unroll
          for (int g = 0; g < kTnMaxGb; ++g) nbn[g] = (ok && g < P.gb) ? (uint32_t)__ldg(kp + g * 8) : 0u;
        }
#pragma unroll
        for (int k = 0; k < 4 + kTnMaxGb; ++k) {
          if (k < 4 + P.gb) {
            const int v = t + k * kSplitThreads;
            uint4 x = hi[v];
            if (brow_t >= rows_valid) x = make_uint4(0u, 0u, 0u, 0u);
            else if (k >= 4) {
              uint32_t nb = nbc[k >= 4 ? k - 4 : 0];
              if (prob == 1) nb >>= 4;
              x.x = (nb & 1u) ? __float_as_uint(__uint_as_float(x.x) * P.keep_scale) : 0u;
              x.y = (nb & 2u) ? __float_as_uint(__uint_as_float(x.y) * P.keep_scale) : 0u;
              x.z = (nb & 4u) ? __float_as_uint(__uint_as_float(x.z) * P.keep_scale) : 0u;
              x.w = (nb & 8u) ? __float_as_uint(__uint_as_float(x.w) * P.keep_scale) : 0u;
            }
            uint4 h, l;
            split_tf32(x.x, h.x, l.x);
            split_tf32(x.y, h.y, l.y);
            split_tf32(x.z, h.z, l.z);
            split_tf32(x.w, h.w, l.w);
            hi[v] = h;
            lo[v] = l;
          }
        }
      } else
      for (int v = t; v < n_vec; v += kSplitThreads) {
        uint4 x = hi[v];
        if (((v & 255) >> 3) >= rows_valid) x = make_uint4(0u, 0u, 0u, 0u);
        uint4 h, l;
        split_tf32(x.x, h.x, l.x);
        split_tf32(x.y, h.y, l.y);
        split_tf32(x.z, h.z, l.z);
        split_tf32(x.w, h.w, l.w);
        hi[v] = h;
        lo[v] = l;
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncwarp();
      if (lane == 0) mb_arrive(split_full + stage);
      if (t == 0) KGC_DBG(3);
      if (++stage == kTnStages) { stage = 0; phase ^= 1; }
      if (++ls == kTnLoStages) { ls = 0; lphase ^= 1; }
    }
  } else if (warp == 1) {
    // MN-major A and B (bits 15, 16), TF32 operands, fp32 accumulate, M = 128, N = n_pad
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(P.n_pad >> 3) << 17) |
                           ((uint32_t)(kBM >> 4) << 24);
    int stage = 0, ls = 0;
    uint32_t phase = 0;
    for (int kb = 0; kb < n_kb; ++kb) {
      mb_wait(split_full + stage, phase);
      if (lane == 0) KGC_DBG(4);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t hi_a = s_u32(s_raw + stage * stage_bytes), hi_b = hi_a + P.ga * kTnBox;
      const uint32_t lo_a = s_u32(s_lo + ls * stage_bytes), lo_b = lo_a + P.ga * kTnBox;
      if (P.kmajor) {
        const uint32_t idesc_k = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(P.n_pad >> 3) << 17) | ((uint32_t)(kBM >> 4) << 24);
        const uint64_t a_hi = sw128_desc(hi_a), a_lo = sw128_desc(lo_a);
        const uint64_t b_hi = sw128_desc(hi_a + kTileA), b_lo = sw128_desc(lo_a + kTileA);
        if (elect_one()) {
          for (int k = 0; k < kTnRows / kUK; ++k) {
            umma_tf32(tmem_base, a_lo + 2 * k, b_hi + 2 * k, idesc_k, (kb | k) != 0 ? 1u : 0u);
            umma_tf32(tmem_base, a_hi + 2 * k, b_lo + 2 * k, idesc_k, 1u);
            umma_tf32(tmem_base, a_hi + 2 * k, b_hi + 2 * k, idesc_k, 1u);
          }
          umma_commit_g(empty + stage);
          umma_commit_g(lo_empty + ls);
          if (kb == n_kb - 1) umma_commit_g(acc_full);
        }
      } else if (elect_one()) {
        for (int k = 0; k < kTnRows / kUK; ++k) {                  // 8 node rows per MMA: the next 8-row K group is 1024 B on
          const uint32_t off = k * 1024;
          umma_tf32(tmem_base, sw128_mn_desc(lo_a + off), sw128_mn_desc(hi_b + off), idesc, (kb | k) != 0 ? 1u : 0u);
          umma_tf32(tmem_base, sw128_mn_desc(hi_a + off), sw128_mn_desc(lo_b + off), idesc, 1u);
          umma_tf32(tmem_base, sw128_mn_desc(hi_a + off), sw128_mn_desc(hi_b + off), idesc, 1u);
        }
        umma_commit_g(empty + stage);
        umma_commit_g(lo_empty + ls);
        if (kb == n_kb - 1) umma_commit_g(acc_full);
      }
      __syncwarp();
      if (lane == 0) KGC_DBG(5);
      if (++stage == kTnStages) { stage = 0; phase ^= 1; }
      if (++ls == kTnLoStages) ls = 0;
    }
  } else if (warp >= 10 && warp <= 13) {
    // epilogue: D row i (TMEM lane) -> partial[cta][i][0..Nb).  One 4-byte store per thread would touch 32 sectors
    // per instruction (rows are Nb * 4 bytes apart); instead each warp lays a 32 x 32 block out as a 128-byte-swizzled
    // box in the (now idle) pipeline stages and one lane issues a TMA store, clipped at Ka rows / Nb columns.
    const int quarter = warp % 4;
    const int i = quarter * 32 + lane;
    float* out = P.partial + (((int64_t)prob * P.n_slabs + slab) * P.Ka + i) * P.Nb;
    if (n_kb > 0) {
      mb_wait(acc_full, 0);                                        // every MMA has retired: shared memory is free
      if (warp == 10 && lane == 0) KGC_DBG(6);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16);
      uint8_t* stg = s_raw + (warp - 10) * (2 * kEpiBuf);
      int buf = 0;
      for (int c0 = 0; c0 < P.n_pad; c0 += 32) {
        uint32_t v[32];
        tmem_ld32_g(taddr + c0, v);
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
        __syncwarp();
        uint8_t* bb = stg + buf * kEpiBuf;
        uint8_t* bx = bb + lane * 128;
        const int sw = lane & 7;
#pragma unroll
        for (int q = 0; q < 8; ++q)
          *reinterpret_cast<uint4*>(bx + ((q ^ sw) << 4)) = make_uint4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) {
          if (c0 < P.Nb && quarter * 32 < P.Ka) tma_store_3d(map_p, bb, c0, quarter * 32, slab);
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        buf ^= 1;
      }
      if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
      if (warp == 10 && lane == 0) KGC_DBG(7);
    } else if (i < P.Ka) {
      for (int j = 0; j < P.Nb; ++j) out[j] = 0.f;
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (P.dbg != nullptr && threadIdx.x == 0) {
    long long g;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(g));
    atomicMax(reinterpret_cast<long long*>(P.dbg) + 8 * 64 + 1, g);
    if (blockIdx.x == 0) { P.dbg[8 * 64 + 4] = g; P.dbg[8 * 64 + 5] = clock64(); }
  }
  if (warp == 14) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemColsG) : "memory");
  }
}

// C[e] = sum over the CTA partials in a FIXED order: 8 part-lanes per element, then their sums in lane order; the
// partials (up to thousands at 4.6 M rows) are added in double precision and rounded once
struct TnOut {
  float* c[kMaxBatch];
  int32_t n_parts[kMaxBatch];                    // partials of each problem (its slabs; the stride is n_parts of the launch)
};
__global__ void __launch_bounds__(256)
gemm_tn_partials_reduce(const float* __restrict__ partial_all, int n_parts, int n_elem, const TnOut outs) {
  __shared__ double sm[8][33];
  const float* partial = partial_all + (int64_t)blockIdx.y * n_parts * n_elem;      // blockIdx.y = problem of the batch
  float* C = blockIdx.y == 0 ? outs.c[0] : (blockIdx.y == 1 ? outs.c[1] : outs.c[2]);   // no runtime index into a parameter
  const int n_parts_p = blockIdx.y == 0 ? outs.n_parts[0] : (blockIdx.y == 1 ? outs.n_parts[1] : outs.n_parts[2]);
  const int e = blockIdx.x * 32 + threadIdx.x;
  double s = 0.0;
  if (e < n_elem) {
    int g = threadIdx.y;
    for (; g + 24 < n_parts_p; g += 32) {                      // four independent loads in flight, added in part order
      const float v0 = partial[(int64_t)g * n_elem + e], v1 = partial[(int64_t)(g + 8) * n_elem + e];
      const float v2 = partial[(int64_t)(g + 16) * n_elem + e], v3 = partial[(int64_t)(g + 24) * n_elem + e];
      s += (double)v0; s += (double)v1; s += (double)v2; s += (double)v3;
    }
    for (; g < n_parts_p; g += 8) s += (double)partial[(int64_t)g * n_elem + e];
  }
  sm[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0 && e < n_elem) {
    double t = sm[0][threadIdx.x];
#pragma unroll
    for (int k = 1; k < 8; ++k) t += sm[k][threadIdx.x];
    C[e] = (float)t;
  }
}

// fp32 [rows, cols] -> boxes of 32 columns x 32 rows (MN-major operand tiles), 128-byte swizzle, zero fill
int make_map_f32_mn(CUtensorMap* map, const void* ptr, int64_t rows, int64_t cols, int64_t pitch) {
  return make_map_f32(map, ptr, rows, cols, pitch, kTnRows, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B);
}

}  // namespace
}  // namespace kgc

using namespace kgc;

static long long* g_gemm_dbg = nullptr;

extern "C" int kgc_conv_prep(const float* rels, int32_t n_rels, const float* loop_rel, const float* loop_edge, const float* w_in,
                             const float* w_out, const float* w_loop, const float* w_rel, int32_t D, int32_t Dout, float* relp,
                             float* all_rel, float* packed_fwd, float* packed_bwd, void* stream) {
  Tiling tf, tb;
  KGC_REQUIRE(make_tiling(Dout, D, &tf) == 0 && make_tiling(D, Dout, &tb) == 0, "unsupported layer width (<= 256)");
  KGC_REQUIRE(n_rels >= 0 && rels && loop_rel && loop_edge && w_in && w_out && w_loop && w_rel && relp && all_rel && packed_fwd && packed_bwd,
              "null buffer");
  PrepArgs a;
  a.rels = rels; a.loop_rel = loop_rel; a.loop_edge = loop_edge; a.w0 = w_in; a.w1 = w_out; a.w2 = w_loop; a.w_rel = w_rel;
  a.n_rels = n_rels; a.D = D; a.Dout = Dout;
  a.n_pad_f = tf.n_pad; a.k_pad_f = tf.k_pad; a.n_pad_b = tb.n_pad; a.k_pad_b = tb.k_pad;
  a.relp = relp; a.all_rel = all_rel; a.packed_f = packed_fwd; a.packed_b = packed_bwd;
  const int64_t total = (int64_t)(n_rels + 1) * (D + Dout) + 3 * (int64_t)tf.n_pad * tf.k_pad + 4 * (int64_t)tb.n_pad * tb.k_pad;
  conv_prep_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, as_stream(stream)>>>(a);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_conv_param_grads(const float* m_loop, const float* w_loop, const float* loop_rel, const float* loop_edge,
                                    const float* relp, const float* w_rel, const float* g_rel, const float* d_relp,
                                    int32_t n_rels, int32_t D, int32_t Dout, float* d_w_loop, float* d_loop_rel,
                                    float* d_loop_edge, float* d_rels, float* d_w_rel, const float* rel_add, void* stream) {
  KGC_REQUIRE(m_loop && w_loop && loop_rel && loop_edge && relp && w_rel && d_relp && d_w_loop && d_loop_rel && d_loop_edge && d_rels && d_w_rel,
              "null buffer");
  ParamGradArgs a;
  a.m_loop = m_loop; a.w_loop = w_loop; a.loop_rel = loop_rel; a.loop_edge = loop_edge; a.relp = relp; a.w_rel = w_rel;
  a.g_rel = g_rel; a.d_relp = d_relp; a.n_rels = n_rels; a.D = D; a.Dout = Dout;
  a.d_w_loop = d_w_loop; a.d_loop_rel = d_loop_rel; a.d_loop_edge = d_loop_edge; a.d_rels = d_rels; a.d_w_rel = d_w_rel;
  if (rel_add != nullptr) {                                       // d_w_rel and rel_add = g_rel w_rel^T come from the GEMM kernels
    KGC_REQUIRE((D * Dout) % 32 == 0, "D * Dout must be a multiple of 32");
    const int64_t total2 = (int64_t)D * Dout + (((int64_t)n_rels * D + 31) & ~31ll) + (int64_t)D * 32;
    conv_param_grads2_kernel<<<(unsigned)ceil_div(total2, 256), 256, 0, as_stream(stream)>>>(a, rel_add);
    KGC_LAUNCH_CHECK();
    return 0;
  }
  const int64_t total = 2 * (int64_t)D * Dout + (int64_t)(n_rels + 1) * D * 32;
  conv_param_grads_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, as_stream(stream)>>>(a);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" size_t kgc_gemm_packed_b_bytes(int32_t N, int32_t K) {
  Tiling t;
  if (make_tiling(N, K, &t)) return 0;
  return (size_t)2 * t.n_pad * t.k_pad * sizeof(float);
}

extern "C" int kgc_gemm_pack_b(const float* B, int64_t stride_k, int64_t stride_n, int32_t N, int32_t K, float* packed,
                               void* stream) {
  Tiling t;
  KGC_REQUIRE(make_tiling(N, K, &t) == 0, "unsupported GEMM shape (K <= 256, N <= 1024)");
  const int total = t.n_pad * t.k_pad;
  pack_b_kernel<<<(total + 255) / 256, 256, 0, as_stream(stream)>>>(B, stride_k, stride_n, N, K, t.n_pad, t.k_pad, packed,
                                                                    packed + total);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" void kgc_gemm_set_debug(long long* buf) { g_gemm_dbg = buf; }   // device buffer of 9 * 64 int64, or NULL

// C_i[M, N] = f(A_i[M, K] @ Bt_i^T + row_bias) (trans_c = 0) or Ct_i[N, M] = the same, stored transposed (trans_c = 1),
// i < n_prob problems of identical shape in ONE launch: the CTAs are dealt to (problem, column tile) groups, so a batch
// fills the 148 SMs with whole row-tile rounds where a single N x 100 x 200 product leaves a 14% tail
static int launch_gemm_nt(int n_prob, const float* const* A, int64_t M, int32_t K, int64_t lda, const float* const* packed_b,
                          int32_t N, float* const* C, int64_t ldc, const float* row_bias, int32_t act, int32_t trans_c,
                          int32_t trans_a, void* stream, const uint8_t* keep = nullptr, int32_t keep_pitch = 0,
                          float keep_scale = 1.f) {
  Tiling t;
  KGC_REQUIRE(n_prob >= 1 && n_prob <= kMaxBatch, "1..3 problems per launch");
  KGC_REQUIRE(make_tiling(N, K, &t) == 0, "unsupported GEMM shape (K <= 256, N <= 1024)");
  KGC_REQUIRE(M > 0 && lda >= (trans_a ? M : (int64_t)K) && ldc >= (trans_c ? M : (int64_t)N), "bad leading dimensions");
  KGC_REQUIRE(!trans_a || M % 32 == 0, "a transposed A operand needs M % 32 == 0");
  KGC_REQUIRE(ldc % 4 == 0, "C needs a 16-byte row pitch (TMA store)");
  GemmMaps maps;
  const int total = t.n_pad * t.k_pad;
  for (int i = 0; i < kMaxBatch; ++i) {
    const int j = i < n_prob ? i : 0;          // unused slots repeat problem 0 (never dereferenced)
    KGC_REQUIRE((reinterpret_cast<uintptr_t>(C[j]) & 15) == 0, "C must be 16-byte aligned (TMA store)");
    if (trans_c) {     // Ct[N, M]: boxes of 32 rows of C (inner) x 32 / 16 columns of C
      if (make_map_f32(&maps.c[i], C[j], N, M, ldc, 32, CU_TENSOR_MAP_SWIZZLE_128B, 32)) return 1;
      if (make_map_f32(&maps.c16[i], C[j], N, M, ldc, 16, CU_TENSOR_MAP_SWIZZLE_128B, 32)) return 1;
    } else {
      if (make_map_f32(&maps.c[i], C[j], M, N, ldc, 32, CU_TENSOR_MAP_SWIZZLE_128B, 32)) return 1;
      if (make_map_f32(&maps.c16[i], C[j], M, N, ldc, 32, CU_TENSOR_MAP_SWIZZLE_64B, 16)) return 1;
    }
    if (trans_a) {     // At[K, M]: dims (32 m, K, M / 32 groups), one box = 4 groups x 32 k
      if (make_map_f32_groups(&maps.a[i], A[j], K, (int)(M / 32), lda, kBM / 32, CU_TENSOR_MAP_SWIZZLE_128B)) return 1;
    } else if (make_map_f32(&maps.a[i], A[j], M, K, lda, kBM)) {
      return 1;
    }
    if (make_map_f32(&maps.bhi[i], packed_b[j], t.n_pad, t.k_pad, t.k_pad, t.NT)) return 1;
    if (make_map_f32(&maps.blo[i], packed_b[j] + total, t.n_pad, t.k_pad, t.k_pad, t.NT)) return 1;
  }
  GemmParams P;
  P.M = M; P.N = N; P.K = K; P.n_prob = n_prob;
  P.n_kb = t.n_kb; P.ksteps = t.ksteps; P.NT = t.NT; P.n_ntiles = t.n_ntiles;
  P.n_mtiles = (int32_t)ceil_div(M, kBM);
  P.C = C[0]; P.ldc = ldc; P.row_bias = row_bias; P.act = act; P.trans_c = trans_c; P.trans_a = trans_a; P.dbg = g_gemm_dbg;
  KGC_REQUIRE(keep == nullptr || (!trans_a && keep_pitch % 16 == 0 && keep_pitch >= 8 * kMaxKB && (reinterpret_cast<uintptr_t>(keep) & 15) == 0),
              "keep flags: one byte per 4 columns, 16-byte aligned rows of at least 64 bytes");
  P.keep = keep; P.keep_pitch = keep_pitch; P.keep_scale = keep_scale;
  const int tile_b_al = (t.NT * kBK * 4 + 1023) & ~1023;
  const size_t fixed = (size_t)2 * t.n_kb * tile_b_al + kEpiStage + 512 + 1024;
  int stages = (int)((226 * 1024 - fixed) / kTileA);
  if (stages > kMaxStages) stages = kMaxStages;
  KGC_REQUIRE(stages >= 2, "shared-memory plan does not fit");
  P.stages = stages;
  const size_t smem = fixed + (size_t)stages * kTileA;
  static SmemAttrCache attr;
  KGC_CUDA_TRY(attr.ensure(gemm_tf32x3_kernel, smem));
  // a multiple of (problems x column tiles) CTAs, at most one per SM, never more row-tile owners than row tiles
  const int groups = n_prob * t.n_ntiles;
  int per = kNumSMs / groups;
  if (per > P.n_mtiles) per = P.n_mtiles;
  if (per < 1) per = 1;
  gemm_tf32x3_kernel<<<per * groups, kThreadsG, smem, as_stream(stream)>>>(maps, P);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_gemm_nt(const float* A, int64_t M, int32_t K, int64_t lda, const float* packed_b, int32_t N, float* C,
                           int64_t ldc, void* stream) {
  return launch_gemm_nt(1, &A, M, K, lda, &packed_b, N, &C, ldc, nullptr, 0, 0, 0, stream);
}

extern "C" int kgc_gemm_nt_batch(int32_t n_prob, const float* const* A, int64_t M, int32_t K, int64_t lda,
                                 const float* const* packed_b, int32_t N, float* const* C, int64_t ldc, void* stream) {
  KGC_REQUIRE(A && packed_b && C, "null pointer table");
  return launch_gemm_nt(n_prob, A, M, K, lda, packed_b, N, C, ldc, nullptr, 0, 0, 0, stream);
}

// Ct[N, M] = (A @ Bt^T)^T with A given transposed, At[K, M] row-major: the long dimension M is contiguous in BOTH the
// streamed operand and the result (a [K, M] weight or activation matrix and a gradient of the same shape)
extern "C" int kgc_gemm_nt_batch_masked(int32_t n_prob, const float* const* A, int64_t M, int32_t K, int64_t lda,
                                        const float* const* packed_b, int32_t N, float* const* C, int64_t ldc,
                                        const uint8_t* keep, int32_t keep_pitch, float keep_scale, void* stream) {
  KGC_REQUIRE(A && packed_b && C, "null pointer table");
  return launch_gemm_nt(n_prob, A, M, K, lda, packed_b, N, C, ldc, nullptr, 0, 0, 0, stream, keep, keep_pitch, keep_scale);
}

extern "C" int kgc_gemm_nt_trans(const float* At, int64_t M, int32_t K, int64_t ldat, const float* packed_b, int32_t N,
                                 float* Ct, int64_t ldct, void* stream) {
  return launch_gemm_nt(1, &At, M, K, ldat, &packed_b, N, &Ct, ldct, nullptr, 0, 1, 1, stream);
}

// pred[b, n] = sigmoid(X[b, :] . E[n, :] + bias[n]): the entity table is the streamed operand, the queries the packed
// small one, the epilogue adds the entity bias, applies the sigmoid and stores the block transposed into pred[B, N]
extern "C" int kgc_score_1n_fwd(const float* ent, int64_t n_ent, int32_t D, int64_t ld_ent, const float* packed_x, int32_t B,
                                const float* bias, float* pred, int64_t ld_pred, void* stream) {
  KGC_REQUIRE(bias != nullptr, "bias is required");
  return launch_gemm_nt(1, &ent, n_ent, D, ld_ent, &packed_x, B, &pred, ld_pred, bias, 1, 1, 0, stream);
}

// Rows a CTA accumulates into ONE fp32 TMEM partial.  The tensor core's fp32 accumulation error grows about linearly with
// the length of the dependent MMA chain (measured on the weight gradients of the Wikidata5M shape, 4.6 M rows, whose sums
// cancel heavily; max-norm-relative error against float64): one slab per SM = 31 k rows per partial -> 7.4e-4; 4,096 rows
// -> 5.7e-5; the WN18RR shape's 836 rows -> 1.0e-5.  Slabs of <= 1,024 rows, partials added in double precision by the
// reduce kernel.  Beyond one wave every extra CTA costs its set-up and epilogue (~4 us per 1.2 MB slab) and 80 KB of partial.
constexpr int64_t kTnMaxSlabRows = 1024;

static int64_t tn_max_slab_rows() {
  static int64_t rows = 0;
  if (rows == 0) {
    const char* e = getenv("KGC_TN_SLAB_ROWS");            // measurement aid (profiles/r02_k4c_slabs.md)
    rows = e != nullptr && atoll(e) >= 64 ? atoll(e) : kTnMaxSlabRows;
  }
  return rows;
}

static int64_t tn_slabs(int64_t M, int n_prob) {
  const int64_t per_wave = kNumSMs / n_prob > 0 ? kNumSMs / n_prob : 1;
  int64_t slabs = ceil_div(M, (int64_t)2 * kTnRows);        // at least two K blocks per CTA
  if (slabs > per_wave) slabs = per_wave;
  const int64_t need = ceil_div(M, tn_max_slab_rows());
  if (slabs < need) slabs = ceil_div(need, per_wave) * per_wave;      // whole waves
  return slabs < 1 ? 1 : slabs;
}

// Entity-major form for the fused loss: predT[n, b] = sigmoid(E[n, :] . X[b, :] + bias[n]), rows of ld_t >= B floats - the
// kernel's natural orientation (contiguous 128-byte row pieces 4 B bytes apart instead of 4 N bytes apart)
extern "C" int kgc_score_1n_fwd_t(const float* ent, int64_t n_ent, int32_t D, int64_t ld_ent, const float* packed_x, int32_t B,
                                  const float* bias, float* pred_t, int64_t ld_t, void* stream) {
  KGC_REQUIRE(bias != nullptr, "bias is required");
  return launch_gemm_nt(1, &ent, n_ent, D, ld_ent, &packed_x, B, &pred_t, ld_t, bias, 1, 0, 0, stream);
}

// The same product WITHOUT the sigmoid: logit[b, n] = X[b, :] . E[n, :] + bias[n] (fp32-grade, 3xTF32) - the exact-mode
// evaluation scorer (scoring.filtered_rank(precision='fp32')) ranks on these where bf16-rounded operands could move a rank
extern "C" int kgc_score_1n_logits(const float* ent, int64_t n_ent, int32_t D, int64_t ld_ent, const float* packed_x, int32_t B,
                                   const float* bias, float* logits, int64_t ld_logits, void* stream) {
  KGC_REQUIRE(bias != nullptr, "bias is required");
  return launch_gemm_nt(1, &ent, n_ent, D, ld_ent, &packed_x, B, &logits, ld_logits, bias, 0, 1, 0, stream);
}

extern "C" size_t kgc_gemm_tn_tc_workspace_bytes(int64_t M, int32_t Ka, int32_t Nb) {
  int64_t parts = kNumSMs;                                  // covers 1..3 problems of one launch
  for (int n = 1; n <= kMaxBatch; ++n) {
    const int64_t s = tn_slabs(M > 0 ? M : 1, n) * n;
    if (s > parts) parts = s;
  }
  return (size_t)parts * Ka * Nb * sizeof(float);
}

// C[Ka, Nb] = A[M, Ka]^T @ B[M, Nb] on the tensor cores (3xTF32).  Ka <= 128, Nb <= 224, multiples of 4.
// m_prob (optional): rows of each problem, <= M.  The row slabs are those of M rows for every problem, so a problem of M rows
// gets the same partials, in the same order, as in a launch where every problem has M rows.
static int launch_gemm_tn_tc(int n_prob, const float* const* A, int64_t lda, const float* const* B, int64_t ldb, int64_t M,
                             int32_t Ka, int32_t Nb, float* const* C, void* workspace, size_t workspace_bytes, int32_t kmajor,
                             void* stream, const uint8_t* keep = nullptr, int32_t keep_pitch = 0, float keep_scale = 1.f,
                             const int64_t* m_prob = nullptr) {
  KGC_REQUIRE(n_prob >= 1 && n_prob <= kMaxBatch, "1..3 problems per launch");
  KGC_REQUIRE(M > 0 && Ka > 0 && Nb > 0 && Ka <= 128 && Nb <= 224, "supported: Ka <= 128, Nb <= 224");
  KGC_REQUIRE(Nb % 4 == 0 && lda % 4 == 0 && ldb % 4 == 0 && (kmajor || Ka % 4 == 0), "dimensions and leading dimensions must be multiples of 4");
  KGC_REQUIRE(workspace && workspace_bytes >= kgc_gemm_tn_tc_workspace_bytes(M, Ka, Nb), "workspace too small");
  GemmTnParams P;
  P.n_pad = (Nb + 15) / 16 * 16;
  P.kmajor = kmajor;
  P.M = M; P.Ka = Ka; P.Nb = Nb; P.n_prob = n_prob;
  P.ga = 4;                                   // the MMA always reads M = 128 rows of D: 4 groups (columns past Ka are zero-filled)
  P.gb = (P.n_pad + 31) / 32;
  int slabs = (int)tn_slabs(M, n_prob);       // one wave of CTAs, more when a slab would exceed kTnMaxSlabRows rows
  P.rows_per_cta = ceil_div(ceil_div(M, slabs), kTnRows) * kTnRows;     // slabs start on K-block boundaries
  slabs = (int)ceil_div(M, P.rows_per_cta);
  P.n_slabs = slabs;
  TnOut outs;
  for (int i = 0; i < kMaxBatch; ++i) {
    const int64_t m = (m_prob != nullptr && i < n_prob) ? m_prob[i] : M;
    KGC_REQUIRE(m >= 0 && m <= M, "rows of a problem must lie in [0, M]");
    P.m_prob[i] = m;
    outs.n_parts[i] = (int)ceil_div(m, P.rows_per_cta);
  }
  P.partial = static_cast<float*>(workspace);
  P.dbg = g_gemm_dbg;
  KGC_REQUIRE(keep == nullptr || (!kmajor && keep_pitch >= 8 * P.gb), "keep flags: one byte per 4 columns of B, rows that cover the padded width");
  P.keep = keep; P.keep_pitch = keep_pitch; P.keep_scale = keep_scale;
  P.ga_full = kmajor ? 0 : Ka / 32;
  P.gb_full = kmajor ? 0 : Nb / 32;
  GemmTnMaps maps;
  for (int i = 0; i < kMaxBatch; ++i) {
    const int j = i < n_prob ? i : 0;          // unused slots repeat problem 0 (never dereferenced)
    outs.c[i] = C[j];
    // a problem without rows still gets valid maps (never read): one row of its operands
    const int64_t Mi = P.m_prob[j] > 0 ? P.m_prob[j] : 1;
    if (kmajor) {      // A[Ka, M], Bt[Nb, M] with the contraction index M contiguous
      if (make_map_f32(&maps.a[i], A[j], Ka, Mi, lda, kBM) || make_map_f32(&maps.b[i], B[j], Nb, Mi, ldb, P.n_pad)) return 1;
    } else if (make_map_f32_mn(&maps.a[i], A[j], Mi, Ka, lda) || make_map_f32_mn(&maps.b[i], B[j], Mi, Nb, ldb)) {
      return 1;
    }
    maps.a3[i] = maps.a[i]; maps.b3[i] = maps.b[i];                      // placeholders when an operand has no complete group
    if (P.ga_full > 0 && make_map_f32_mn_groups(&maps.a3[i], A[j], Mi, P.ga_full, lda)) return 1;
    if (P.gb_full > 0 && make_map_f32_mn_groups(&maps.b3[i], B[j], Mi, P.gb_full, ldb)) return 1;
    if (make_map_f32_parts(&maps.p[i], P.partial + (int64_t)j * slabs * Ka * Nb, slabs, Ka, Nb)) return 1;
  }
  const size_t stage = (size_t)(P.ga + P.gb) * kTnBox;
  const size_t smem = (kTnStages + kTnLoStages) * stage + 512 + 1024;
  KGC_REQUIRE(smem <= 227 * 1024, "shared-memory plan does not fit");
  static SmemAttrCache attr;
  KGC_CUDA_TRY(attr.ensure(gemm_tn_tc_kernel, smem));
  cudaStream_t st = as_stream(stream);
  gemm_tn_tc_kernel<<<slabs * n_prob, kThreadsG, smem, st>>>(maps, P);
  KGC_LAUNCH_CHECK();
  gemm_tn_partials_reduce<<<dim3((Ka * Nb + 31) / 32, n_prob), dim3(32, 8), 0, st>>>(P.partial, slabs, Ka * Nb, outs);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_gemm_tn_tc(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t M, int32_t Ka, int32_t Nb,
                              float* C, void* workspace, size_t workspace_bytes, void* stream) {
  return launch_gemm_tn_tc(1, &A, lda, &B, ldb, M, Ka, Nb, &C, workspace, workspace_bytes, 0, stream);
}

extern "C" int kgc_gemm_tn_tc_batch(int32_t n_prob, const float* const* A, int64_t lda, const float* const* B, int64_t ldb,
                                    int64_t M, int32_t Ka, int32_t Nb, float* const* C, void* workspace,
                                    size_t workspace_bytes, void* stream) {
  KGC_REQUIRE(A && B && C, "null pointer table");
  return launch_gemm_tn_tc(n_prob, A, lda, B, ldb, M, Ka, Nb, C, workspace, workspace_bytes, 0, stream);
}

// the same with rows[i] <= M rows for problem i (the layer's compacted planes): problems of M rows keep their bits
extern "C" int kgc_gemm_tn_tc_batch_rows(int32_t n_prob, const float* const* A, int64_t lda, const float* const* B, int64_t ldb,
                                         const int64_t* rows, int64_t M, int32_t Ka, int32_t Nb, float* const* C, void* workspace,
                                         size_t workspace_bytes, void* stream) {
  KGC_REQUIRE(A && B && C && rows, "null pointer table");
  return launch_gemm_tn_tc(n_prob, A, lda, B, ldb, M, Ka, Nb, C, workspace, workspace_bytes, 0, stream, nullptr, 0, 1.f, rows);
}

extern "C" int kgc_gemm_tn_tc_batch_masked(int32_t n_prob, const float* const* A, int64_t lda, const float* const* B, int64_t ldb,
                                           int64_t M, int32_t Ka, int32_t Nb, float* const* C, void* workspace,
                                           size_t workspace_bytes, const uint8_t* keep, int32_t keep_pitch, float keep_scale,
                                           void* stream) {
  KGC_REQUIRE(A && B && C, "null pointer table");
  return launch_gemm_tn_tc(n_prob, A, lda, B, ldb, M, Ka, Nb, C, workspace, workspace_bytes, 0, stream, keep, keep_pitch,
                           keep_scale);
}

// C[Ma, Nb] = A[Ma, K] @ Bt[Nb, K]^T with a LONG contraction (K >> Ma, Nb): the K range is cut into per-CTA slabs, both
// operands are streamed K-major, partial products stay in TMEM and are added in CTA order.  Ma <= 128, Nb <= 224.
extern "C" int kgc_gemm_nt_splitk(const float* A, int64_t lda, const float* Bt, int64_t ldb, int64_t K, int32_t Ma, int32_t Nb,
                                  float* C, void* workspace, size_t workspace_bytes, void* stream) {
  return launch_gemm_tn_tc(1, &A, lda, &Bt, ldb, K, Ma, Nb, &C, workspace, workspace_bytes, 1, stream);
}
