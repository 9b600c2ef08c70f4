// K2 / K3: relation-aware aggregation, forward and backward (HBM-bound segment reductions).
//
// Reference arithmetic replaced (model.py:111-118 + PyG aggr='add', model.py:50,99-100):
//   m_e = (x[src_e] * rel[type_e] * edge_emb[e]) @ W * norm_e ;  out[dst] += m_e
// restated as aggregate-then-transform (the matmul is linear, SURVEY.md fact 8):
//   agg[dst] = sum_e norm_e * x[src_e] (.) rel[type_e] (.) ee[e]      (this file)
//   res      = agg @ W                                                   (dense GEMM, host side)
//
// Streaming design: the sorted edge records are cut into CHUNKS of 32 consecutive records, one warp per chunk whatever
// the row boundaries (every warp has the same amount of work, no per-row launch overhead); lane l owns float4 column l
// of a row, so a 400-byte row is one fully coalesced 25-lane request; a row that lies inside one chunk is written
// straight to the output; the (at most two) rows a chunk shares with its neighbours go to CARRY rows, which
// kgc_rows_reduce adds in a fixed order.  No float atomics anywhere: results are bit-reproducible run to run.
//
// Two kernels implement it.  agg_lean_kernel (D <= 128, the product path at the reference's D = 100) and
// agg_stream_kernel (the earlier version, kept for 128 < D <= 256: two float4 columns per lane).
//
// History of the measurements that shaped agg_lean_kernel (profiles/r01_agg_variants.md has every number):
//   * agg_stream_kernel reached 0.53 / 0.53 / 0.47 of the measured HBM peak (fwd / bwd_src / bwd_rel, WN18RR shape) and
//     looked latency-bound: every unit below 45% busy, same time for sequential and for random row order
//     (tests/gather_probe.py), no gain from more loads in flight.  Rejected on the way: per-row bulk async copies
//     (UBLKCP, 0.2-0.3 - the copy engine retires ~one 400-byte request per 30 cycles per SM), a per-warp cp.async ring
//     (0.29 / 0.37 / 0.23), double-buffered register batches (no change), L2 prefetch of the next chunk (worse), records
//     broadcast from shared memory (spills), one-warp CTAs, dynamic chunk claiming (same).
//   * ncu source-level sampling then showed WHY: 75 warp instructions per edge, only 28% of the stall samples on the first
//     use of a loaded row, the other 72% spread evenly over ~700 SASS instructions (fixed-latency waits, shuffles, branch
//     bookkeeping, per-edge bounds checks, 64-bit address arithmetic) at 3.5 warps per scheduler.  The kernel was bound by
//     the serial instruction latency of each warp, not by memory.
//   * a continuous register ring (edge e + P issued as soon as edge e is consumed) cut the instruction count to 47 per
//     edge but ran SLOWER (45 / 88 / 63 us): a warp has six scoreboard slots, the load being waited for shares its slot
//     with loads issued after it, and the ring degenerates (long-scoreboard stall 3 -> 12 cycles per issue).  Batches -
//     all loads of kU edges, then all their arithmetic - are the structure the scoreboards reward.
//   * agg_lean_kernel: 42 instructions per edge, batches of 3-4 edges at 3 CTAs per SM (80 registers, no spills):
//     35.8 / 64.6 / 39.9 us -> 26.6 / 47.1 / 28.8 us = 0.70 / 0.73 / 0.65 of the measured peak, bit-identical outputs.
//     Relation rows staged in shared memory and grids balanced to equal chunks per warp changed nothing measurable.
//     ncu of the kept kernel: DRAM 47%, L1TEX 62%, 19 resident warps per SM, long-scoreboard 9 cycles per issue - it is
//     now memory-latency-bound; the torch copy of the same bytes, timed the same way, reaches 0.77-0.79.

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

// agg_stream_kernel (128 < D <= 256).  One warp walks one chunk of kChunk (= 32) sorted records.  Lane l first loads record cb + l (one coalesced
// 512-byte + 128-byte request for the whole chunk); every edge's record is then broadcast with warp shuffles,
// so all gather addresses of the chunk are known after a single memory round trip.  kU edges are in flight per
// trip: phase 1 issues their DRAM / L2 row loads (edge embedding + the gathered operand), phase 2 consumes them
// in record order with the L1-resident operands (relation row, and the source row in the backward pass).
template <int MODE> struct Unroll { static constexpr int value = 8; };
template <> struct Unroll<kBwdRel> { static constexpr int value = 4; };      // three DRAM/L2 operands per edge
template <> struct Unroll<kBwdSrc> { static constexpr int value = 6; };      // ee, g[dst] and x[src] per edge

template <int MODE, int NF>
__global__ void __launch_bounds__(kThreads, 2)
agg_stream_kernel(const StreamArgs A) {
  constexpr int kU = Unroll<MODE>::value;
  static_assert(kChunk == 32, "one record per lane");
  // PERSISTENT warps: the grid fills the GPU once (2 CTAs per SM) and every warp walks chunks w, w + W, w + 2W, ...
  // (W = warps of the grid), fetching the records of its next chunk while it processes the current one.  One warp per
  // chunk with a one-shot grid paid a record round trip per chunk with nothing else in flight (fwd 37.4 -> 34.9 us).
  // Claiming chunks dynamically from an atomic work counter instead of the static stride measured the same (35.2 us).
  const int lane = threadIdx.x % 32;
  const int64_t n_chunks = (A.n_rec + kChunk - 1) / kChunk;
  const int64_t stride = (int64_t)gridDim.x * kWarpsPerBlock;
  int64_t chunk = blockIdx.x * (int64_t)kWarpsPerBlock + threadIdx.x / 32;
  if (chunk >= n_chunks) return;
  const int D4 = A.D4;
  bool active[NF];
#pragma unroll
  for (int f = 0; f < NF; ++f) active[f] = lane + f * 32 < D4;
  auto rec_index = [&](int64_t ch) {
    const int64_t b = ch * kChunk;
    const int n = (int)(b + kChunk < A.n_rec ? kChunk : A.n_rec - b);
    return b + (lane < n ? lane : n - 1);
  };
  int2 slots_n = __ldg(reinterpret_cast<const int2*>(A.chunks + chunk));
  int4 myrec_n = ld_rec(A.rec + rec_index(chunk));
  uint32_t myflag_n = __ldg(A.rowflags + rec_index(chunk));
 while (chunk < n_chunks) {
  const int64_t next = chunk + stride;
  const int64_t cb = chunk * kChunk;
  const int cnt = (int)(cb + kChunk < A.n_rec ? kChunk : A.n_rec - cb);
  const int2 slots = slots_n;
  const int4 myrec = myrec_n;
  const uint32_t myflag = myflag_n;
  if (next < n_chunks) {                                         // records of the next chunk: in flight during this one
    slots_n = __ldg(reinterpret_cast<const int2*>(A.chunks + next));
    myrec_n = ld_rec(A.rec + rec_index(next));
    myflag_n = __ldg(A.rowflags + rec_index(next));
  }

  float4 acc[NF];
#pragma unroll
  for (int f = 0; f < NF; ++f) acc[f] = make_float4(0.f, 0.f, 0.f, 0.f);
  bool started_here = (__shfl_sync(0xffffffffu, myflag, 0) & kFirst) != 0;
  bool open_row = false;

  for (int base = 0; base < cnt; base += kU) {
    float4 va[kU][NF], vb[kU][NF], vc[kU][MODE == kFwd ? 1 : NF];
    // ---- phase 1: the long-latency row loads of kU edges
#pragma unroll
    for (int u = 0; u < kU; ++u) {
      const int e = base + u < cnt ? base + u : cnt - 1;          // clamped: a duplicate load, never consumed
      const uint32_t eid = (uint32_t)__shfl_sync(0xffffffffu, myrec.x, e);
      const uint32_t ra = (uint32_t)__shfl_sync(0xffffffffu, myrec.y, e);
      const uint32_t rb = (uint32_t)__shfl_sync(0xffffffffu, myrec.z, e);
      const uint32_t erow = __shfl_sync(0xffffffffu, myflag, e) & kRowMask;
#pragma unroll
      for (int f = 0; f < NF; ++f) {
        const int c = lane + f * 32;
        if (active[f]) {
          va[u][f] = ld_stream(A.ee + (uint64_t)eid * D4 + c);
          if (MODE == kFwd) {
            vb[u][f] = __ldg(A.x + (uint64_t)ra * D4 + c);
          } else if (MODE == kBwdSrc) {
            vb[u][f] = __ldg(A.g3 + ((int)eid >= A.n_edges_in ? A.plane : 0) + (uint64_t)ra * D4 + c);
            vc[u][f] = __ldg(A.x + (uint64_t)erow * D4 + c);                 // x[src]: one miss per row, then L1
          } else {
            vb[u][f] = __ldg(A.g3 + ((int)eid >= A.n_edges_in ? A.plane : 0) + (uint64_t)rb * D4 + c);
            vc[u][f] = __ldg(A.x + (uint64_t)ra * D4 + c);
          }
        }
      }
    }
    // ---- phase 2: consume in record order
#pragma unroll
    for (int u = 0; u < kU; ++u) {
      if (base + u < cnt) {                                      // warp-uniform
        const int e = base + u;
        const uint32_t flags = __shfl_sync(0xffffffffu, myflag, e);
        const float nrm = __int_as_float(__shfl_sync(0xffffffffu, myrec.w, e));
        const int64_t row = flags & kRowMask;
        // shuffles stay outside the lane predicate: every lane of the warp must take part
        const uint32_t rb = (uint32_t)__shfl_sync(0xffffffffu, myrec.z, e);
        const uint32_t eid = (uint32_t)__shfl_sync(0xffffffffu, myrec.x, e);
        (void)rb; (void)eid;
        if (flags & kFirst) {
#pragma unroll
          for (int f = 0; f < NF; ++f) acc[f] = make_float4(0.f, 0.f, 0.f, 0.f);
          started_here = true;
        }
        open_row = true;
#pragma unroll
        for (int f = 0; f < NF; ++f) {
          const int c = lane + f * 32;
          if (active[f]) {
            if (MODE == kFwd) {
              add4(acc[f], mul3s(nrm, vb[u][f], __ldg(A.rel + (uint64_t)rb * D4 + c), va[u][f]));
            } else if (MODE == kBwdSrc) {
              const float4 pe = scale4(nrm, mul4(vb[u][f], __ldg(A.rel + (uint64_t)rb * D4 + c)));   // norm * g[dst] * rel
              st_stream(A.d_ee + (uint64_t)eid * D4 + c, mul4(pe, vc[u][f]));                           // * x[src]
              add4(acc[f], mul4(pe, va[u][f]));
            } else {
              add4(acc[f], mul3s(nrm, vb[u][f], vc[u][f], va[u][f]));                                   // norm * g * x * ee
            }
          }
        }
        if (flags & kLast) {                                     // the row ends here
          float4* out = started_here ? A.out_final + row * D4 : A.carry + (int64_t)slots.x * D4;
#pragma unroll
          for (int f = 0; f < NF; ++f) {
            const int c = lane + f * 32;
            if (active[f]) {
              float4 v = acc[f];
              if (MODE == kBwdSrc && started_here && A.addend != nullptr) add4(v, __ldg(A.addend + row * D4 + c));
              out[c] = v;
            }
          }
          open_row = false;
        }
      }
    }
  }
  if (open_row) {                                                // the row continues in the next chunk
    float4* out = A.carry + (int64_t)slots.y * D4;
#pragma unroll
    for (int f = 0; f < NF; ++f) {
      const int c = lane + f * 32;
      if (active[f]) out[c] = acc[f];
    }
  }
  chunk = next;
 }   // persistent chunk loop
}

// ---------------------------------------------------------------------------------------------- lean variant
// Same chunks / carry protocol / arithmetic as agg_stream_kernel.  ncu of that kernel (profiles/r01_ncu_agg_lean.md):
// 75 warp instructions per edge, 72% of the stall samples spread evenly over them (fixed-latency waits, shuffles,
// branch bookkeeping) and only 28% on the first use of a loaded row - instruction-latency-bound at 14 warps per SM.
// This version (i) fully unrolls the 32 edges of a FULL chunk (shuffle lanes and batch slots are compile-time, no
// per-edge bounds checks; the stream's single partial chunk takes a plain loop), (ii) issues ALL row loads of a batch,
// the relation row included, in the load phase, so the consume phase is pure arithmetic, (iii) forms addresses from
// 32-bit float4 indices (one IMAD + one IMAD.WIDE per load), (iv) runs at 3-4 CTAs per SM with small batches.
template <int MODE, int KU, int MINB>
__global__ void __launch_bounds__(kThreads, MINB)
agg_lean_kernel(const StreamArgs A) {
  // Full unroll in every mode.  The d_x / d_ee pass has ~110 instructions per edge: unrolling all 32 makes a 56 KB loop
  // body and ncu shows 6.5 stall cycles per issued instruction waiting for the instruction cache ("no instruction"; 0.4
  // in the two smaller kernels).  Bodies of 32 / 16 / 8 edges (1, 2 or 4 trips per chunk) measured 11.69 / 11.63 /
  // 11.60 ms at the Wikidata5M shape and 47.4 / 48.7 / 49.4 us at the WN18RR shape - the fetch stalls are not on the
  // critical path of a DRAM-latency-bound kernel, so the partial unrolls were removed.
  static_assert(kChunk == 32, "one record per lane");
  constexpr bool kHasC = MODE != kFwd;        // third gathered operand
  constexpr bool kHasR = MODE != kBwdRel;     // relation row
  const int lane = threadIdx.x % 32;
  const int warp = __shfl_sync(0xffffffffu, (int)threadIdx.x / 32, 0);          // warp-uniform for the compiler
  const int64_t n_chunks = (A.n_rec + kChunk - 1) / kChunk;
  const int64_t stride = (int64_t)gridDim.x * kWarpsPerBlock;
  int64_t chunk = blockIdx.x * (int64_t)kWarpsPerBlock + warp;
  if (chunk >= n_chunks) return;
  const uint32_t D4 = (uint32_t)A.D4;
  const bool act = lane < (int)D4;
  const uint32_t c = act ? lane : 0;
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

  float4 va[KU], vb[KU], vc[kHasC ? KU : 1], vr[kHasR ? KU : 1];
  int4 rec;
  uint32_t flag;
  float4 acc;
  bool started_here;
  int2 slots;
  float4* const out_final = A.out_final;
  float4* const carry = A.carry;
  float4* const d_ee = A.d_ee;
  const float4* const addend = A.addend;
  auto issue = [&](int u, int e) {
    const uint32_t eid = (uint32_t)__shfl_sync(0xffffffffu, rec.x, e);
    const uint32_t ra = (uint32_t)__shfl_sync(0xffffffffu, rec.y, e);
    const uint32_t rb = (uint32_t)__shfl_sync(0xffffffffu, rec.z, e);
    if (MODE == kFwd) {
      if (act) {
        va[u] = ld_stream(ee + (eid * D4 + c));
        vb[u] = __ldg(xs + (ra * D4 + c));
        vr[kHasR ? u : 0] = __ldg(rel + (rb * D4 + c));
      }
    } else if (MODE == kBwdSrc) {
      const uint32_t erow = __shfl_sync(0xffffffffu, flag, e) & kRowMask;
      if (act) {
        va[u] = ld_stream(ee + (eid * D4 + c));
        vb[u] = __ldg(g3 + ((eid >= n_in ? plane : 0u) + ra * D4 + c));
        vc[kHasC ? u : 0] = __ldg(xs + (erow * D4 + c));
        vr[kHasR ? u : 0] = __ldg(rel + (rb * D4 + c));
      }
    } else {
      if (act) {
        va[u] = ld_stream(ee + (eid * D4 + c));
        vb[u] = __ldg(g3 + ((eid >= n_in ? plane : 0u) + rb * D4 + c));
        vc[kHasC ? u : 0] = __ldg(xs + (ra * D4 + c));
      }
    }
  };
  // `last` = this record closes its row (rows are contiguous, so the next record opens one: the accumulator is cleared
  // here and no per-edge "first" test is needed)
  auto consume = [&](int u, int e, bool last) {
    const float nrm = __int_as_float(__shfl_sync(0xffffffffu, rec.w, e));
    const float4 rv = vr[kHasR ? u : 0];
    if (MODE == kFwd) {
      add4(acc, mul3s(nrm, vb[u], rv, va[u]));
    } else if (MODE == kBwdSrc) {
      const uint32_t eid = (uint32_t)__shfl_sync(0xffffffffu, rec.x, e);
      const float4 pe = scale4(nrm, mul4(vb[u], rv));
      if (act) st_stream(d_ee + (eid * D4 + c), mul4(pe, vc[kHasC ? u : 0]));
      add4(acc, mul4(pe, va[u]));
    } else {
      add4(acc, mul3s(nrm, vb[u], vc[kHasC ? u : 0], va[u]));
    }
    if (last) {
      const uint32_t row = __shfl_sync(0xffffffffu, flag, e) & kRowMask;
      float4* out = started_here ? out_final + (row * D4 + c) : carry + ((uint32_t)slots.x * D4 + c);
      if (act) {
        float4 v = acc;
        if (MODE == kBwdSrc && started_here && addend != nullptr) add4(v, __ldg(addend + (row * D4 + c)));
        *out = v;
      }
      acc = make_float4(0.f, 0.f, 0.f, 0.f);
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
    acc = make_float4(0.f, 0.f, 0.f, 0.f);
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
      if (act) carry[(uint32_t)slots.y * D4 + c] = acc;
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

// Lean kernel configuration (edges per batch, CTAs per SM), measured on B200 at the WN18RR / FB15k-237 shapes
// (history in profiles/r01_agg_variants.md): fwd 4 x 3, bwd_src 3 x 3, bwd_rel 4 x 3 - the largest
// batches that fit 80 registers without spills; 2 CTAs x 8 edges and 4 CTAs x 2-3 edges were 10-20% slower.
template <int MODE> struct LeanCfg { static constexpr int ku = 4, minb = 3; };
template <> struct LeanCfg<kBwdSrc> { static constexpr int ku = 3, minb = 3; };

template <int MODE>
int launch_stream(const StreamArgs& A, cudaStream_t st) {
  if (A.n_rec == 0) return 0;
  const int64_t n_chunks = ceil_div(A.n_rec, kChunk);
  int64_t blocks = ceil_div(n_chunks, kWarpsPerBlock);
  if (A.D4 <= 32) {                                               // D <= 128: one float4 column per lane
    // 32-bit float4 indices: edge ids are < n_rec, node / output rows < max_rows (the host checks the node table)
    KGC_REQUIRE((uint64_t)A.n_rec * A.D4 < (1ull << 32) && (uint64_t)A.max_rows * A.D4 < (1ull << 32),
                "tables of 2^32 float4 or more are not supported (32-bit float4 indices)");
    constexpr int minb = LeanCfg<MODE>::minb;
    if (blocks > (int64_t)minb * kNumSMs) blocks = (int64_t)minb * kNumSMs;   // persistent grid
    agg_lean_kernel<MODE, LeanCfg<MODE>::ku, minb><<<(unsigned)blocks, kThreads, 0, st>>>(A);
  } else {
    if (blocks > 2 * kNumSMs) blocks = 2 * kNumSMs;               // persistent: 2 resident CTAs per SM (__launch_bounds__)
    agg_stream_kernel<MODE, 2><<<(unsigned)blocks, kThreads, 0, st>>>(A);
  }
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
