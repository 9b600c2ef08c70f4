// K2 / K3: relation-aware aggregation, forward and backward (HBM-bound segment reductions).
//
// Reference arithmetic replaced (model.py:111-118 + PyG aggr='add', model.py:50,99-100):
//   m_e = (x[src_e] * rel[type_e] * edge_emb[e]) @ W * norm_e ;  out[dst] += m_e
// restated as aggregate-then-transform (the matmul is linear, SURVEY.md fact 8):
//   agg[dst] = sum_e norm_e * x[src_e] (.) rel[type_e] (.) ee[e]      (this file)
//   res      = agg @ W                                                   (dense GEMM, host side)
//
// Streaming design: the sorted edge records are cut into CHUNKS of 32 consecutive records, one warp per chunk whatever
// the row boundaries (every warp has the same amount of work, no per-row launch overhead); lane l owns float4 columns
// l and l + 32 of a row (the second only for D > 128), so a 400-byte row is one fully coalesced 25-lane request; a row
// that lies inside one chunk is written straight to the output; the (at most two) rows a chunk shares with its
// neighbours go to CARRY rows, which kgc_rows_reduce adds in a fixed order.  No float atomics anywhere: results are
// bit-reproducible run to run.
//
// Why agg_kernel looks as it does (profiles/r01_agg_variants.md has the measurements and the rejected variants):
//   * the kernel is bound by the latency of each warp's serial instruction stream and of its row loads, not by DRAM
//     bandwidth.  So it keeps instructions per edge low: the 32 edges of a full chunk are fully unrolled (shuffle lanes
//     and batch slots are compile-time, no per-edge bounds checks) and addresses are 32-bit float4 indices (one IMAD +
//     one IMAD.WIDE per load; the launcher checks that every table fits).
//   * loads go in BATCHES: all row loads of KU edges, then all their arithmetic.  A warp has six scoreboard slots; a
//     continuous ring of loads (edge e + P issued as soon as edge e is consumed) shares them between the load being waited
//     for and the loads behind it and ran slower than batches despite fewer instructions.
//   * batches are as large as fit the register budget of 3 CTAs per SM (one column per lane) or 2 (two columns) without
//     spills: more resident warps hide more load latency than longer batches.

#include "common.cuh"

namespace kgc {
namespace {

constexpr int kGroup = 8;          // kgc_rows_reduce: lanes per partial-row group
constexpr int kThreads = 256;
constexpr int kMaxNF = 8;          // kgc_rows_reduce: D <= 8 * 8 * 4 = 256
constexpr int kChunk = KGC_CHUNK_EDGES;
constexpr int kWarpsPerBlock = kThreads / 32;
constexpr uint32_t kRowMask = 0x3FFFFFFFu, kFirst = 0x40000000u, kLast = 0x80000000u;

__device__ __forceinline__ float4 mul3s(float s, const float4& a, const float4& b, const float4& c) {
  // s * ((a*b)*c), the reference's product order (model.py:115) followed by the norm (model.py:118)
  return make_float4(s * ((a.x * b.x) * c.x), s * ((a.y * b.y) * c.y), s * ((a.z * b.z) * c.z),
                     s * ((a.w * b.w) * c.w));
}
__device__ __forceinline__ void add4(float4& acc, const float4& v) {
  acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
}
__device__ __forceinline__ float4 mul4(const float4& a, const float4& b) {
  return make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w);
}
__device__ __forceinline__ float4 scale4(float s, const float4& a) {
  return make_float4(s * a.x, s * a.y, s * a.z, s * a.w);
}

enum Mode { kFwd = 0, kBwdSrc = 1, kBwdRel = 2 };

struct StreamArgs {
  const float4* x;            // node rows (global ids)
  const float4* rel;          // relation rows (fwd, bwd_src)
  const float4* ee;           // edge-embedding rows (global edge ids of this rank)
  const float4* g3;           // bwd: [2, n_dst_rows, D] upstream planes
  const float4* addend;       // bwd_src: self-loop term added on rows finished inside a chunk (or null)
  const kgc_edge_rec_t* rec;
  const uint32_t* rowflags;   // row | first << 30 | last << 31 per sorted record
  const kgc_chunk_t* chunks;
  float4* out_final;
  float4* carry;
  float4* d_ee;               // bwd_src: per-edge output
  int64_t n_rec;
  int64_t plane;              // n_dst_rows * D4 (bwd)
  int32_t n_edges_in;         // records with eid >= n_edges_in belong to the out half (bwd)
  int32_t D4;
  int64_t max_rows;           // known bound on the row indices of g3 / outputs (guard of the 32-bit float4 indices)
};

// One warp walks one chunk of kChunk (= 32) sorted records.  Lane l first loads record cb + l (one coalesced request for
// the whole chunk); every edge's record is then broadcast with warp shuffles, so all gather addresses of the chunk are
// known after a single memory round trip.  NC = float4 columns per lane (1: D <= 128, 2: D <= 256).
template <int MODE, int KU, int MINB, int NC>
__global__ void __launch_bounds__(kThreads, MINB)
agg_kernel(const StreamArgs A) {
  // Full unroll in every mode.  The d_x / d_ee pass has ~110 instructions per edge: unrolling all 32 makes a 56 KB loop
  // body and ncu shows 6.5 stall cycles per issued instruction waiting for the instruction cache ("no instruction"; 0.4
  // in the two smaller kernels).  Bodies of 32 / 16 / 8 edges (1, 2 or 4 trips per chunk) measured 11.69 / 11.63 /
  // 11.60 ms at the Wikidata5M shape and 47.4 / 48.7 / 49.4 us at the WN18RR shape - the fetch stalls are not on the
  // critical path of a DRAM-latency-bound kernel, so the partial unrolls were removed.
  static_assert(kChunk == 32, "one record per lane");
  constexpr bool kHasC = MODE != kFwd;        // third gathered operand
  constexpr bool kHasR = MODE != kBwdRel;     // relation row
  const int lane = threadIdx.x % 32;
  // PERSISTENT warps: the grid fills the GPU once and every warp walks chunks w, w + W, w + 2W, ... (W = warps of the
  // grid), fetching the records of its next chunk while it processes the current one
  const int warp = __shfl_sync(0xffffffffu, (int)threadIdx.x / 32, 0);          // warp-uniform for the compiler
  const int64_t n_chunks = (A.n_rec + kChunk - 1) / kChunk;
  const int64_t stride = (int64_t)gridDim.x * kWarpsPerBlock;
  int64_t chunk = blockIdx.x * (int64_t)kWarpsPerBlock + warp;
  if (chunk >= n_chunks) return;
  const uint32_t D4 = (uint32_t)A.D4;
  auto active = [&](int f) { return lane + 32 * f < (int)D4; };                  // column f of this lane exists
  auto col = [&](int f) -> uint32_t { return active(f) ? lane + 32 * f : 0; };
  const float4* __restrict__ ee = A.ee;
  const float4* __restrict__ xs = A.x;
  const float4* __restrict__ rel = A.rel;
  const float4* __restrict__ g3 = A.g3;
  const uint32_t plane = (uint32_t)A.plane;
  const uint32_t n_in = (uint32_t)A.n_edges_in;
  auto rec_index = [&](int64_t ch) {
    const int64_t b = ch * kChunk;
    const int n = (int)(b + kChunk < A.n_rec ? kChunk : A.n_rec - b);
    return b + (lane < n ? lane : n - 1);
  };
  int2 slots_n = __ldg(reinterpret_cast<const int2*>(A.chunks + chunk));
  int4 rec_n = ld_rec(A.rec + rec_index(chunk));
  uint32_t flag_n = __ldg(A.rowflags + rec_index(chunk));

  float4 va[KU][NC], vb[KU][NC], vc[kHasC ? KU : 1][NC], vr[kHasR ? KU : 1][NC];
  int4 rec;
  uint32_t flag;
  float4 acc[NC];
  bool started_here;
  int2 slots;
  float4* const out_final = A.out_final;
  float4* const carry = A.carry;
  float4* const d_ee = A.d_ee;
  const float4* const addend = A.addend;
  // the relation row and every gathered row of edge e into batch slot u
  auto issue = [&](int u, int e) {
    const uint32_t eid = (uint32_t)__shfl_sync(0xffffffffu, rec.x, e);
    const uint32_t ra = (uint32_t)__shfl_sync(0xffffffffu, rec.y, e);
    const uint32_t rb = (uint32_t)__shfl_sync(0xffffffffu, rec.z, e);
    if (MODE == kFwd) {
#pragma unroll
      for (int f = 0; f < NC; ++f) {
        if (active(f)) {
          va[u][f] = ld_stream(ee + (eid * D4 + col(f)));
          vb[u][f] = __ldg(xs + (ra * D4 + col(f)));
          vr[kHasR ? u : 0][f] = __ldg(rel + (rb * D4 + col(f)));
        }
      }
    } else if (MODE == kBwdSrc) {
      const uint32_t erow = __shfl_sync(0xffffffffu, flag, e) & kRowMask;
#pragma unroll
      for (int f = 0; f < NC; ++f) {
        if (active(f)) {
          va[u][f] = ld_stream(ee + (eid * D4 + col(f)));
          vb[u][f] = __ldg(g3 + ((eid >= n_in ? plane : 0u) + ra * D4 + col(f)));
          vc[kHasC ? u : 0][f] = __ldg(xs + (erow * D4 + col(f)));
          vr[kHasR ? u : 0][f] = __ldg(rel + (rb * D4 + col(f)));
        }
      }
    } else {
#pragma unroll
      for (int f = 0; f < NC; ++f) {
        if (active(f)) {
          va[u][f] = ld_stream(ee + (eid * D4 + col(f)));
          vb[u][f] = __ldg(g3 + ((eid >= n_in ? plane : 0u) + rb * D4 + col(f)));
          vc[kHasC ? u : 0][f] = __ldg(xs + (ra * D4 + col(f)));
        }
      }
    }
  };
  // `last` = this record closes its row (rows are contiguous, so the next record opens one: the accumulator is cleared
  // here and no per-edge "first" test is needed)
  auto consume = [&](int u, int e, bool last) {
    const float nrm = __int_as_float(__shfl_sync(0xffffffffu, rec.w, e));
    if (MODE == kFwd) {
#pragma unroll
      for (int f = 0; f < NC; ++f) add4(acc[f], mul3s(nrm, vb[u][f], vr[kHasR ? u : 0][f], va[u][f]));
    } else if (MODE == kBwdSrc) {
      const uint32_t eid = (uint32_t)__shfl_sync(0xffffffffu, rec.x, e);
#pragma unroll
      for (int f = 0; f < NC; ++f) {
        const float4 pe = scale4(nrm, mul4(vb[u][f], vr[kHasR ? u : 0][f]));
        if (active(f)) st_stream(d_ee + (eid * D4 + col(f)), mul4(pe, vc[kHasC ? u : 0][f]));
        add4(acc[f], mul4(pe, va[u][f]));
      }
    } else {
#pragma unroll
      for (int f = 0; f < NC; ++f) add4(acc[f], mul3s(nrm, vb[u][f], vc[kHasC ? u : 0][f], va[u][f]));
    }
    if (last) {
      const uint32_t row = __shfl_sync(0xffffffffu, flag, e) & kRowMask;
#pragma unroll
      for (int f = 0; f < NC; ++f) {
        float4* out = started_here ? out_final + (row * D4 + col(f)) : carry + ((uint32_t)slots.x * D4 + col(f));
        if (active(f)) {
          float4 v = acc[f];
          if (MODE == kBwdSrc && started_here && addend != nullptr) add4(v, __ldg(addend + (row * D4 + col(f))));
          *out = v;
        }
        acc[f] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
      started_here = true;
    }
  };

  while (chunk < n_chunks) {
    const int64_t next = chunk + stride;
    const int64_t cb = chunk * kChunk;
    const int cnt = (int)(cb + kChunk < A.n_rec ? kChunk : A.n_rec - cb);
    slots = slots_n;
    rec = rec_n;
    flag = flag_n;
    if (next < n_chunks) {                                         // records of the next chunk: in flight during this one
      slots_n = __ldg(reinterpret_cast<const int2*>(A.chunks + next));
      rec_n = ld_rec(A.rec + rec_index(next));
      flag_n = __ldg(A.rowflags + rec_index(next));
    }
#pragma unroll
    for (int f = 0; f < NC; ++f) acc[f] = make_float4(0.f, 0.f, 0.f, 0.f);
    const uint32_t valid = cnt == kChunk ? 0xffffffffu : ((1u << cnt) - 1u);
    const uint32_t last_mask = __ballot_sync(0xffffffffu, (flag & kLast) != 0) & valid;
    started_here = (__shfl_sync(0xffffffffu, flag, 0) & kFirst) != 0;
    if (cnt == kChunk) {
#pragma unroll
      for (int base = 0; base < kChunk; base += KU) {
#pragma unroll
        for (int u = 0; u < KU; ++u)
          if (base + u < kChunk) issue(u, base + u);
#pragma unroll
        for (int u = 0; u < KU; ++u)
          if (base + u < kChunk) consume(u, base + u, (last_mask >> (base + u)) & 1u);
      }
    } else {                                                     // the stream's last, partial chunk
      for (int e = 0; e < cnt; ++e) {
        issue(0, e);
        consume(0, e, (last_mask >> e) & 1u);
      }
    }
    if (!((last_mask >> (cnt - 1)) & 1u)) {                      // the row continues in the next chunk
#pragma unroll
      for (int f = 0; f < NC; ++f)
        if (active(f)) carry[(uint32_t)slots.y * D4 + col(f)] = acc[f];
    }
    chunk = next;
  }
}

// out[rows[i]] = addend ? addend[rows[i]] : 0   (rows without any edge record)
__global__ void rows_fill_kernel(const int32_t* __restrict__ rows, int64_t n_rows, const float4* __restrict__ addend,
                                 float4* __restrict__ out, int D4) {
  const int64_t i = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / 32;
  const int lane = threadIdx.x % 32;
  if (i >= n_rows) return;
  const int64_t r = rows[i];
  for (int c = lane; c < D4; c += 32)
    out[r * D4 + c] = addend ? __ldg(addend + r * D4 + c) : make_float4(0.f, 0.f, 0.f, 0.f);
}

// ------------------------------------------------------------------------------------------------ fix-up levels
// One 512-thread block per item: 64 groups of 8 lanes stride over the item's carry / partial rows (4 rows in flight
// per group), the 4 groups of a warp are combined with shuffles, the 32 warp sums through shared memory - always in the
// same order, so the result is deterministic.  Fan-in up to 2048 rows per item: a 38k-edge hub row (1,187 carry rows)
// is ONE item and one launch; a 9M-edge hub needs two levels.  The first n_large items of a level get a block each;
// the (thousands of) small items - rows that merely straddle a chunk boundary - get one 8-lane group each.
constexpr int kRedThreads = 512;
constexpr int kRedGroups = kRedThreads / kGroup;     // 64

template <int NF>
__global__ void __launch_bounds__(kRedThreads)
rows_reduce_kernel(const float4* __restrict__ part_in, const kgc_item_t* __restrict__ items, int64_t n_items,
                   int64_t n_large, float4* __restrict__ out_final, float4* __restrict__ out_part,
                   const float4* __restrict__ addend, int D4) {
  __shared__ float4 sm[kRedThreads / 32][NF * kGroup];
  const int grp = threadIdx.x / kGroup, g = threadIdx.x % kGroup, warp = threadIdx.x / 32, lane = threadIdx.x % 32;
  if ((int64_t)blockIdx.x >= n_large) {
    // small items (a row that merely straddles one or two chunk boundaries: 2-16 carry rows): one 8-lane group each
    const int64_t item = n_large + ((int64_t)blockIdx.x - n_large) * kRedGroups + grp;
    if (item >= n_items) return;
    const int4 it = __ldg(reinterpret_cast<const int4*>(items + item));
    float4 acc[NF];
#pragma unroll
    for (int f = 0; f < NF; ++f) acc[f] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int r = it.x; r < it.y; ++r) {
#pragma unroll
      for (int f = 0; f < NF; ++f) {
        const int c = g + f * kGroup;
        if (c < D4) add4(acc[f], __ldg(part_in + (int64_t)r * D4 + c));
      }
    }
    const bool final_row = (it.w & 1) != 0;
    float4* out = (final_row ? out_final : out_part) + (int64_t)it.z * D4;
#pragma unroll
    for (int f = 0; f < NF; ++f) {
      const int c = g + f * kGroup;
      if (c < D4) {
        float4 v = acc[f];
        if (final_row && addend != nullptr) add4(v, __ldg(addend + (int64_t)it.z * D4 + c));
        out[c] = v;
      }
    }
    return;
  }
  const int4 it = __ldg(reinterpret_cast<const int4*>(items + blockIdx.x));
  float4 acc[NF];
#pragma unroll
  for (int f = 0; f < NF; ++f) acc[f] = make_float4(0.f, 0.f, 0.f, 0.f);
  int r = it.x + grp;
  for (; r + 3 * kRedGroups < it.y; r += 4 * kRedGroups) {      // 4 independent rows in flight, added in row order
    float4 v[4][NF];
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int f = 0; f < NF; ++f) {
        const int c = g + f * kGroup;
        if (c < D4) v[u][f] = __ldg(part_in + (int64_t)(r + u * kRedGroups) * D4 + c);
      }
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int f = 0; f < NF; ++f) {
        const int c = g + f * kGroup;
        if (c < D4) add4(acc[f], v[u][f]);
      }
  }
  for (; r < it.y; r += kRedGroups) {
#pragma unroll
    for (int f = 0; f < NF; ++f) {
      const int c = g + f * kGroup;
      if (c < D4) add4(acc[f], __ldg(part_in + (int64_t)r * D4 + c));
    }
  }
  // the 4 groups of a warp hold the same columns: (g0 + g1) + (g2 + g3), fixed order
#pragma unroll
  for (int f = 0; f < NF; ++f) {
    float4 t;
    t.x = __shfl_xor_sync(0xffffffffu, acc[f].x, 8); t.y = __shfl_xor_sync(0xffffffffu, acc[f].y, 8);
    t.z = __shfl_xor_sync(0xffffffffu, acc[f].z, 8); t.w = __shfl_xor_sync(0xffffffffu, acc[f].w, 8);
    add4(acc[f], t);
    t.x = __shfl_xor_sync(0xffffffffu, acc[f].x, 16); t.y = __shfl_xor_sync(0xffffffffu, acc[f].y, 16);
    t.z = __shfl_xor_sync(0xffffffffu, acc[f].z, 16); t.w = __shfl_xor_sync(0xffffffffu, acc[f].w, 16);
    add4(acc[f], t);
    if (lane < kGroup) sm[warp][g + f * kGroup] = acc[f];
  }
  __syncthreads();
  if (warp == 0 && lane < kGroup) {
    const bool final_row = (it.w & 1) != 0;
    float4* out = (final_row ? out_final : out_part) + (int64_t)it.z * D4;
#pragma unroll
    for (int f = 0; f < NF; ++f) {
      const int c = g + f * kGroup;
      if (c < D4) {
        float4 v = sm[0][c];
        for (int k = 1; k < kRedThreads / 32; ++k) add4(v, sm[k][c]);
        if (final_row && addend != nullptr) add4(v, __ldg(addend + (int64_t)it.z * D4 + c));
        out[c] = v;
      }
    }
  }
}

inline int check_dim(int32_t D, int* D4, int* NF) {
  if (D <= 0 || D % 4 != 0 || D > kMaxNF * kGroup * 4) return 1;
  *D4 = D / 4;
  *NF = (*D4 + kGroup - 1) / kGroup;
  return 0;
}

#define KGC_DISPATCH_NF(NFV, ...)                         \
  switch (NFV) {                                          \
    case 1: { constexpr int NF = 1; __VA_ARGS__; } break; \
    case 2: { constexpr int NF = 2; __VA_ARGS__; } break; \
    case 3: { constexpr int NF = 3; __VA_ARGS__; } break; \
    case 4: { constexpr int NF = 4; __VA_ARGS__; } break; \
    case 5: { constexpr int NF = 5; __VA_ARGS__; } break; \
    case 6: { constexpr int NF = 6; __VA_ARGS__; } break; \
    case 7: { constexpr int NF = 7; __VA_ARGS__; } break; \
    default: { constexpr int NF = 8; __VA_ARGS__; } break; \
  }

// agg_kernel configuration: edges per batch (kAggKU[NC - 1][MODE]) and CTAs per SM, the largest batches that compile
// without spills.  One column per lane (measured on B200 at the WN18RR / FB15k-237 shapes, profiles/r01_agg_variants.md):
// fwd 4, bwd_src 3, bwd_rel 4 edges at 3 CTAs (80 registers); 2 CTAs x 8 edges and 4 CTAs x 2-3 edges were 10-20% slower.
// Two columns per lane: fwd 4, bwd_src 2, bwd_rel 3 edges at 2 CTAs (128 registers; profiles/r12_one_agg_kernel_ptxas_sass.md).
constexpr int kAggKU[2][3] = {{4, 3, 4}, {4, 2, 3}};

template <int MODE, int NC>
void launch_agg(const StreamArgs& A, int64_t blocks, cudaStream_t st) {
  constexpr int minb = NC == 1 ? 3 : 2;
  if (blocks > (int64_t)minb * kNumSMs) blocks = (int64_t)minb * kNumSMs;   // persistent grid
  agg_kernel<MODE, kAggKU[NC - 1][MODE], minb, NC><<<(unsigned)blocks, kThreads, 0, st>>>(A);
}

template <int MODE>
int launch_stream(const StreamArgs& A, cudaStream_t st) {
  if (A.n_rec == 0) return 0;
  // 32-bit float4 indices: edge ids are < n_rec, node / output rows < max_rows (the host checks the node table)
  KGC_REQUIRE((uint64_t)A.n_rec * A.D4 < (1ull << 32) && (uint64_t)A.max_rows * A.D4 < (1ull << 32),
              "tables of 2^32 float4 or more are not supported (32-bit float4 indices)");
  const int64_t blocks = ceil_div(ceil_div(A.n_rec, kChunk), kWarpsPerBlock);
  if (A.D4 <= 32)                                                 // D <= 128: one float4 column per lane
    launch_agg<MODE, 1>(A, blocks, st);
  else
    launch_agg<MODE, 2>(A, blocks, st);
  KGC_LAUNCH_CHECK();
  return 0;
}

}  // namespace
}  // namespace kgc

using namespace kgc;

extern "C" int kgc_agg_fwd(const float* x, const float* rel, int64_t n_types, const float* ee,
                           const kgc_edge_rec_t* rec_dst, const uint32_t* rowflags, const kgc_chunk_t* chunks,
                           int64_t n_rec, float* out_final, float* carry, int32_t D, void* stream) {
  int D4, nf;
  KGC_REQUIRE(check_dim(D, &D4, &nf) == 0, "D must be a multiple of 4 and <= 256");
  StreamArgs A = {};
  (void)n_types;
  A.x = (const float4*)x; A.rel = (const float4*)rel; A.ee = (const float4*)ee;
  A.rec = rec_dst; A.rowflags = rowflags; A.chunks = chunks;
  A.out_final = (float4*)out_final; A.carry = (float4*)carry;
  A.n_rec = n_rec; A.D4 = D4;
  return launch_stream<kFwd>(A, as_stream(stream));
}

extern "C" int kgc_agg_bwd_src(const float* x, const float* rel, int64_t n_types, const float* ee, const float* g3,
                               const kgc_edge_rec_t* rec_src, const uint32_t* rowflags, const kgc_chunk_t* chunks,
                               int64_t n_rec, int64_t n_dst_rows, int64_t n_edges_in, const float* loop_addend,
                               float* d_ee, float* dx_final, float* carry, int32_t D, void* stream) {
  int D4, nf;
  KGC_REQUIRE(check_dim(D, &D4, &nf) == 0, "D must be a multiple of 4 and <= 256");
  StreamArgs A = {};
  (void)n_types;
  A.max_rows = 3 * n_dst_rows;
  A.x = (const float4*)x; A.rel = (const float4*)rel; A.ee = (const float4*)ee; A.g3 = (const float4*)g3;
  A.addend = (const float4*)loop_addend;
  A.rec = rec_src; A.rowflags = rowflags; A.chunks = chunks;
  A.out_final = (float4*)dx_final; A.carry = (float4*)carry; A.d_ee = (float4*)d_ee;
  A.n_rec = n_rec; A.plane = n_dst_rows * (int64_t)D4; A.n_edges_in = (int32_t)n_edges_in; A.D4 = D4;
  return launch_stream<kBwdSrc>(A, as_stream(stream));
}

extern "C" int kgc_agg_bwd_rel(const float* x, const float* ee, const float* g3, const kgc_edge_rec_t* rec_type,
                               const uint32_t* rowflags, const kgc_chunk_t* chunks, int64_t n_rec, int64_t n_dst_rows,
                               int64_t n_edges_in, float* drel_final, float* carry, int32_t D, void* stream) {
  int D4, nf;
  KGC_REQUIRE(check_dim(D, &D4, &nf) == 0, "D must be a multiple of 4 and <= 256");
  StreamArgs A = {};
  A.max_rows = 3 * n_dst_rows;
  A.x = (const float4*)x; A.ee = (const float4*)ee; A.g3 = (const float4*)g3;
  A.rec = rec_type; A.rowflags = rowflags; A.chunks = chunks;
  A.out_final = (float4*)drel_final; A.carry = (float4*)carry;
  A.n_rec = n_rec; A.plane = n_dst_rows * (int64_t)D4; A.n_edges_in = (int32_t)n_edges_in; A.D4 = D4;
  return launch_stream<kBwdRel>(A, as_stream(stream));
}

__global__ void block_sum_kernel(const float4* __restrict__ in, int64_t n_blocks, int64_t n4, float4* __restrict__ out) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n4) return;
  float4 acc = __ldg(in + i);
  for (int64_t b = 1; b < n_blocks; ++b) add4(acc, __ldg(in + b * n4 + i));
  out[i] = acc;
}

extern "C" int kgc_block_sum(const float* in, int64_t n_blocks, int64_t n, float* out, void* stream) {
  KGC_REQUIRE(in && out && n_blocks >= 1 && n > 0 && n % 4 == 0, "bad arguments");
  block_sum_kernel<<<(unsigned)ceil_div(n / 4, 256), 256, 0, as_stream(stream)>>>((const float4*)in, n_blocks, n / 4,
                                                                               (float4*)out);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_rows_fill(const int32_t* rows, int64_t n_rows, const float* addend, float* out, int32_t D,
                             void* stream) {
  int D4, nf;
  KGC_REQUIRE(check_dim(D, &D4, &nf) == 0, "D must be a multiple of 4 and <= 256");
  if (n_rows == 0) return 0;
  rows_fill_kernel<<<(unsigned)ceil_div(n_rows * 32, 256), 256, 0, as_stream(stream)>>>(rows, n_rows, (const float4*)addend,
                                                                                   (float4*)out, D4);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_rows_reduce(const float* part_in, const kgc_item_t* items, int64_t n_items, int64_t n_large,
                               float* out_final, float* out_part, const float* addend, int32_t D, void* stream) {
  int D4, nf;
  KGC_REQUIRE(check_dim(D, &D4, &nf) == 0, "D must be a multiple of 4 and <= 256");
  KGC_REQUIRE(n_large >= 0 && n_large <= n_items, "n_large must lie in [0, n_items]");
  if (n_items == 0) return 0;
  const unsigned grid = (unsigned)(n_large + ceil_div(n_items - n_large, kRedGroups));
  KGC_DISPATCH_NF(nf, (rows_reduce_kernel<NF><<<grid, kRedThreads, 0, as_stream(stream)>>>(
                          (const float4*)part_in, items, n_items, n_large, (float4*)out_final, (float4*)out_part,
                          (const float4*)addend, D4)));
  KGC_LAUNCH_CHECK();
  return 0;
}
