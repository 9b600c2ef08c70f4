// K5: label / batch builder (and the negative-sampler extension).
// Replaces KBDataset.__getitem__ / get_label / collate_fn (reference data_loader.py:25-51): the dense
// multi-hot [B,N] label is written straight into device memory from the query->objects CSR, so the
// per-query Python loop and the B*N*4-byte host-to-device copy of every step disappear.
#include "common.cuh"

namespace kgc {
namespace {

constexpr int kThreads = 256;

// One block row per query: fill label[b,:] with `add`, then overwrite the positives with `pos`.
// The fill is the HBM-bound part (B*N*4 bytes written once, 128-bit stores); positives are a
// handful of scattered 4-byte stores issued after a block barrier so they win over the fill.
__global__ void __launch_bounds__(kThreads)
label_build_kernel(const int64_t* __restrict__ qid, const int64_t* __restrict__ triples,
                   const int64_t* __restrict__ ptr, const int32_t* __restrict__ idx, int64_t n_entity, float pos,
                   float add, int64_t* __restrict__ triple_out, float* __restrict__ label) {
  const int64_t b = blockIdx.y;
  const int64_t q = qid[b];
  float* row = label + b * n_entity;
  // this block's slice of the row
  const int64_t per = (n_entity + gridDim.x - 1) / gridDim.x;
  const int64_t lo = blockIdx.x * per, hi = lo + per < n_entity ? lo + per : n_entity;
  // 128-bit body where the row slice is 16-byte aligned, scalar head / tail otherwise
  const uintptr_t addr = reinterpret_cast<uintptr_t>(row + lo);
  const int64_t head = ((16 - (addr & 15)) & 15) / 4;
  const int64_t body_lo = lo + head < hi ? lo + head : hi;
  const int64_t n4 = (hi - body_lo) / 4;
  for (int64_t k = lo + threadIdx.x; k < body_lo; k += kThreads) row[k] = add;
  float4* row4 = reinterpret_cast<float4*>(row + body_lo);
  const float4 v = make_float4(add, add, add, add);
  for (int64_t k = threadIdx.x; k < n4; k += kThreads) row4[k] = v;
  for (int64_t k = body_lo + n4 * 4 + threadIdx.x; k < hi; k += kThreads) row[k] = add;
  __syncthreads();
  for (int64_t k = ptr[q] + threadIdx.x; k < ptr[q + 1]; k += kThreads) {
    const int64_t j = idx[k];
    if (j >= lo && j < hi) row[j] = pos;
  }
  if (blockIdx.x == 0 && threadIdx.x < 3) triple_out[b * 3 + threadIdx.x] = triples[q * 3 + threadIdx.x];
}

__device__ __forceinline__ bool is_positive(const int32_t* idx, int64_t lo, int64_t hi, int32_t v) {
  while (lo < hi) {   // idx is ascending within a query
    const int64_t mid = (lo + hi) >> 1;
    const int32_t m = idx[mid];
    if (m == v) return true;
    if (m < v) lo = mid + 1; else hi = mid;
  }
  return false;
}

__global__ void neg_sample_kernel(const int64_t* __restrict__ qid, int64_t B, const int64_t* __restrict__ ptr,
                                  const int32_t* __restrict__ idx, int64_t n_entity,
                                  const uint32_t* __restrict__ draws, int k, int tries, int32_t* __restrict__ neg) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= B * k) return;
  const int64_t q = qid[t / k];
  const int64_t lo = ptr[q], hi = ptr[q + 1];
  int32_t out = -1;
  for (int a = 0; a < tries; ++a) {
    const uint32_t u = draws[t * tries + a];
    const int32_t cand = (int32_t)(((uint64_t)u * (uint64_t)n_entity) >> 32);
    if (!is_positive(idx, lo, hi, cand)) { out = cand; break; }
  }
  neg[t] = out;
}

// Positive sampler (extension, companion of the negative sampler): slot j of query qid[b] is the
// ((u * len) >> 32)-th entry of the query's object list - sampling with replacement; -1 for a query without objects.
__global__ void pos_sample_kernel(const int64_t* __restrict__ qid, int64_t B, const int64_t* __restrict__ ptr,
                                  const int32_t* __restrict__ idx, const uint32_t* __restrict__ draws, int p,
                                  int32_t* __restrict__ out) {
  const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (t >= B * p) return;
  const int64_t q = qid[t / p];
  const int64_t lo = ptr[q], len = ptr[q + 1] - lo;
  out[t] = len > 0 ? idx[lo + (int64_t)(((uint64_t)draws[t] * (uint64_t)len) >> 32)] : -1;
}

// Edge sampler (extension, no reference counterpart): triple t_j = (draws[j] * E) >> 32 contributes its in-half edge t_j to
// column j and its out-half edge t_j + E to column m + j of the sampled sub-graph - the layout MGCNConv expects (in half
// first).  A pure function of the caller's draws (sampling with replacement).
__global__ void edge_sample_kernel(const int64_t* __restrict__ src, const int64_t* __restrict__ dst,
                                   const int64_t* __restrict__ type, int64_t n_triples, const uint32_t* __restrict__ draws,
                                   int64_t m, int64_t* __restrict__ sub_src, int64_t* __restrict__ sub_dst,
                                   int64_t* __restrict__ sub_type, int64_t* __restrict__ eids) {
  const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (j >= 2 * m) return;
  const int64_t t = (int64_t)(((uint64_t)draws[j < m ? j : j - m] * (uint64_t)n_triples) >> 32);
  const int64_t e = j < m ? t : t + n_triples;
  sub_src[j] = src[e];
  sub_dst[j] = dst[e];
  sub_type[j] = type[e];
  eids[j] = e;
}

}  // namespace
}  // namespace kgc

using namespace kgc;

extern "C" int kgc_edge_sample(const int64_t* src, const int64_t* dst, const int64_t* type, int64_t n_triples,
                               const uint32_t* draws, int64_t m, int64_t* sub_src, int64_t* sub_dst, int64_t* sub_type,
                               int64_t* eids, void* stream) {
  KGC_REQUIRE(n_triples > 0 && n_triples < (1ll << 31) && m >= 0, "bad sizes");
  if (m == 0) return 0;
  KGC_REQUIRE(src && dst && type && draws && sub_src && sub_dst && sub_type && eids, "null buffer");
  edge_sample_kernel<<<(unsigned)ceil_div(2 * m, kThreads), kThreads, 0, as_stream(stream)>>>(src, dst, type, n_triples, draws,
                                                                                         m, sub_src, sub_dst, sub_type, eids);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_label_build(const int64_t* qid, int64_t B, const int64_t* triples, const int64_t* ptr,
                               const int32_t* idx, int64_t n_entity, float pos, float add, int64_t* triple_out,
                               float* label, void* stream) {
  KGC_REQUIRE(B >= 0 && n_entity > 0, "bad sizes");
  if (B == 0) return 0;
  KGC_REQUIRE(B <= 65535, "batch too large for one launch (<= 65535 queries)");
  // enough column blocks that B * gx >= 4 waves of 148 SMs, at least 4096 floats per block
  int64_t gx = ceil_div(4 * kNumSMs, B);
  const int64_t max_gx = ceil_div(n_entity, 4096);
  if (gx > max_gx) gx = max_gx;
  if (gx < 1) gx = 1;
  dim3 grid((unsigned)gx, (unsigned)B);
  label_build_kernel<<<grid, kThreads, 0, as_stream(stream)>>>(qid, triples, ptr, idx, n_entity, pos, add, triple_out,
                                                              label);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_neg_sample(const int64_t* qid, int64_t B, const int64_t* ptr, const int32_t* idx, int64_t n_entity,
                              const uint32_t* draws, int32_t k, int32_t tries, int32_t* neg, void* stream) {
  KGC_REQUIRE(B >= 0 && k > 0 && tries > 0 && n_entity > 0, "bad sizes");
  if (B == 0) return 0;
  neg_sample_kernel<<<(unsigned)ceil_div(B * k, kThreads), kThreads, 0, as_stream(stream)>>>(qid, B, ptr, idx, n_entity,
                                                                                         draws, k, tries, neg);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_pos_sample(const int64_t* qid, int64_t B, const int64_t* ptr, const int32_t* idx, const uint32_t* draws,
                              int32_t p, int32_t* out, void* stream) {
  KGC_REQUIRE(B >= 0 && p > 0, "bad sizes");
  if (B == 0) return 0;
  KGC_REQUIRE(qid && ptr && idx && draws && out, "null buffer");
  pos_sample_kernel<<<(unsigned)ceil_div(B * p, kThreads), kThreads, 0, as_stream(stream)>>>(qid, B, ptr, idx, draws, p, out);
  KGC_LAUNCH_CHECK();
  return 0;
}
