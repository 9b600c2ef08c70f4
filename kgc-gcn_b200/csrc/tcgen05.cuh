// The PTX layer of the tensor-core kernels (K4b / K4c / K6t in gemm_tf32x3.cu, K6 / K6k in score_rank.cu): mbarriers,
// fences, TMA, tensor memory, tcgen05.mma and its shared-memory descriptor, plus the host-side tensor-map encoding.
// What belongs to one kernel (instruction descriptors, tile layouts, the TF32 split) stays in its file.
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace kgc {
namespace {

// ------------------------------------------------------------------------------------------------ shared memory, mbarriers
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

// ------------------------------------------------------------------------------------------------ fences
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

// ------------------------------------------------------------------------------------------------ TMA
// loads complete_tx on `bar`; stores join the issuing thread's bulk group (bulk_commit_group / bulk_wait_group*)
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(map)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, const void* smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(map)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// at most N committed groups still READ their shared-memory source (the buffers of older ones may be reused)
template <int N>
__device__ __forceinline__ void bulk_wait_group_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
// at most N committed groups still pending (0: every store has completed)
template <int N>
__device__ __forceinline__ void bulk_wait_group() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

// ------------------------------------------------------------------------------------------------ tensor memory
// one warp allocates `cols` columns (a power of two >= 32) and writes the base address to *slot; the CTA then gives up
// its allocation permit (one allocation per CTA)
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// 32 lanes x 32 consecutive 32-bit columns: v[j] = column taddr + j of this thread's lane (complete after tmem_ld_wait)
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
// 32 lanes x 16 consecutive 32-bit columns from v[0..16) of each thread (complete after tmem_st_wait)
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
      "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------ tcgen05.mma (one thread issues for the CTA)
// D[tmem] (+)= A[smem] * B[smem]^T, kind::tf32 (fp32 accumulate); acc = 0 overwrites D
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
// kind::f16 (the instruction descriptor selects bf16 or fp16 operands), fp32 accumulate
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

}  // namespace

// ------------------------------------------------------------------------------------------------ host: tensor maps
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// Tiled map of a `rank`-dimensional array: dims innermost first, strides = byte strides of dims 1.., box in elements, element
// strides 1, L2 promotion of 256 B, out-of-bounds elements zero-filled by loads and clipped by stores.  TMA needs a 16-byte
// aligned base and 16-byte multiples as strides.
inline int encode_tiled(CUtensorMap* map, CUtensorMapDataType dtype, cuuint32_t rank, const void* base, const cuuint64_t* dims,
                        const cuuint64_t* strides, const cuuint32_t* box, CUtensorMapSwizzle swizzle) {
  ensure_thread_context();
  static EncodeTiledFn enc = nullptr;                    // one lookup per process (an inline function's static)
  if (!enc) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    KGC_CUDA_TRY(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    KGC_REQUIRE(qres == cudaDriverEntryPointSuccess && fn != nullptr, "cuTensorMapEncodeTiled not available");
    enc = reinterpret_cast<EncodeTiledFn>(fn);
  }
  bool aligned = (reinterpret_cast<uintptr_t>(base) & 15) == 0;
  for (cuuint32_t i = 0; i + 1 < rank; ++i) aligned = aligned && strides[i] % 16 == 0;
  KGC_REQUIRE(aligned, "a TMA operand needs a 16-byte aligned base and 16-byte multiples as row / plane pitches");
  const cuuint32_t estr[3] = {1, 1, 1};
  const CUresult r = enc(map, dtype, rank, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  KGC_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")");
  return 0;
}

}  // namespace kgc
