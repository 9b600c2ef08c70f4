// K4: layer tail - dropout combine, /3, BatchNorm1d over the node rows, tanh - and its backward.
// Replaces reference model.py:103-106.  Elementwise + column reductions over [n_rows, Dout]; the
// column statistics are accumulated in fp64 per thread, reduced per block in a fixed order and
// finalised by one small kernel, so the result is deterministic and accurate (no atomics).
#include "common.cuh"

namespace kgc {
namespace {

constexpr int kThreads = 256;
constexpr int kMaxBlocks = 4 * kNumSMs;

struct Stripe {
  int64_t row_beg, row_end;
};
__device__ __forceinline__ Stripe block_stripe(int64_t n_rows) {
  const int64_t per = (n_rows + gridDim.x - 1) / gridDim.x;
  Stripe s;
  s.row_beg = blockIdx.x * per;
  s.row_end = s.row_beg + per < n_rows ? s.row_beg + per : n_rows;
  return s;
}

__device__ __forceinline__ float4 mask4(const uint8_t* m, int64_t idx4, float s) {
  const uchar4 v = *reinterpret_cast<const uchar4*>(m + idx4 * 4);
  return make_float4(v.x ? s : 0.f, v.y ? s : 0.f, v.z ? s : 0.f, v.w ? s : 0.f);
}

constexpr int kKeepPitch = 64;            // bytes per row of the packed keep flags: one byte per float4 column (Dout <= 256)
__device__ __forceinline__ uint32_t nibble(const float4& m) {
  return (m.x != 0.f ? 1u : 0u) | (m.y != 0.f ? 2u : 0u) | (m.z != 0.f ? 4u : 0u) | (m.w != 0.f ? 8u : 0u);
}

__device__ __forceinline__ float4 keep4(const float4& g, uint32_t nb, float s) {
  return make_float4((nb & 1u) ? g.x * s : 0.f, (nb & 2u) ? g.y * s : 0.f, (nb & 4u) ? g.z * s : 0.f, (nb & 8u) ? g.w * s : 0.f);
}

struct DropCfg {
  const uint8_t* mask_in;     // injected keep masks (tests / replay of recorded draws) ...
  const uint8_t* mask_out;
  const int64_t* seed;        // ... or a device-resident seed for the counter-based generator (NULL = no dropout)
  uint32_t drop_thr;
  float keep_scale;
};
__device__ __forceinline__ float4 drop_scale4(const DropCfg& d, int plane, int64_t i) {
  const uint8_t* m = plane == 0 ? d.mask_in : d.mask_out;
  if (m != nullptr) return mask4(m, i, d.keep_scale);
  if (d.seed != nullptr) return philox_mask4(i, (uint32_t)plane, (uint64_t)__ldg(d.seed), d.drop_thr, d.keep_scale);
  return make_float4(1.f, 1.f, 1.f, 1.f);
}

// Sum the per-thread double4 accumulators of the RL row-lanes of a block, in lane order, and store
// them as partials[block][which][col].
__device__ __forceinline__ void block_store_partials(double4 a, double4 b, int rl, int c, int RL, int Do4,
                                                     double* partials, double4* sm) {
  // sm holds 2 * RL * Do4 double4
  const bool active = rl < RL;
  if (active) {
    sm[(0 * RL + rl) * Do4 + c] = a;
    sm[(1 * RL + rl) * Do4 + c] = b;
  }
  __syncthreads();
  if (active && rl == 0) {
    double4 sa = sm[c], sb = sm[RL * Do4 + c];
    for (int k = 1; k < RL; ++k) {
      const double4 ta = sm[(0 * RL + k) * Do4 + c], tb = sm[(1 * RL + k) * Do4 + c];
      sa.x += ta.x; sa.y += ta.y; sa.z += ta.z; sa.w += ta.w;
      sb.x += tb.x; sb.y += tb.y; sb.z += tb.z; sb.w += tb.w;
    }
    double4* out = reinterpret_cast<double4*>(partials) + (int64_t)blockIdx.x * 2 * Do4;
    out[c] = sa;
    out[Do4 + c] = sb;
  }
}

// Compacted in / out planes (the layer's sparse halves): plane h holds only the rows with at least one edge, slot[h][r] =
// the compact row of node row r or -1 (an empty row, whose value is exactly 0).  slot[h] == NULL: plane h is dense.
struct PlaneRows {
  const int32_t* slot[2];
  const float4* rows[2];
};
__device__ __forceinline__ float4 plane_value(const float4* __restrict__ dense, const PlaneRows& pr, int h, int64_t r,
                                              int64_t i, int c, int Do4) {
  if (pr.slot[h] == nullptr) return __ldg(dense + i);
  const int32_t s = __ldg(pr.slot[h] + r);
  return s >= 0 ? __ldg(pr.rows[h] + (int64_t)s * Do4 + c) : make_float4(0.f, 0.f, 0.f, 0.f);
}

__global__ void __launch_bounds__(kThreads)
tail_fwd_kernel(const float4* __restrict__ res3, const PlaneRows pr, const DropCfg drop, const float4* __restrict__ bias,
                int64_t n_rows, int Do4, float4* __restrict__ pre, double* __restrict__ partials,
                uint8_t* __restrict__ keep) {
  extern __shared__ double4 sm[];
  const int RL = kThreads / Do4;
  const int rl = threadIdx.x / Do4, c = threadIdx.x % Do4;
  const Stripe s = block_stripe(n_rows);
  const int64_t plane = n_rows * (int64_t)Do4;
  double4 sum = make_double4(0, 0, 0, 0), sq = make_double4(0, 0, 0, 0);
  if (rl < RL) {
    const float4 bv = bias ? __ldg(bias + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    for (int64_t r = s.row_beg + rl; r < s.row_end; r += RL) {
      const int64_t i = r * Do4 + c;
      float4 a = plane_value(res3, pr, 0, r, i, c, Do4), b = plane_value(res3 + plane, pr, 1, r, i, c, Do4);
      const float4 l = __ldg(res3 + 2 * plane + i);
      uint32_t kb = 0;
      { const float4 m = drop_scale4(drop, 0, i); a.x *= m.x; a.y *= m.y; a.z *= m.z; a.w *= m.w; kb |= nibble(m); }
      { const float4 m = drop_scale4(drop, 1, i); b.x *= m.x; b.y *= m.y; b.z *= m.z; b.w *= m.w; kb |= nibble(m) << 4; }
      // the keep flags of the four columns, both planes, in one byte: the backward GEMMs apply them to the single
      // upstream plane while they split it (kgc_gemm_nt_batch / kgc_gemm_tn_tc_batch), nothing is regenerated or stored
      // per plane
      if (keep != nullptr) keep[r * kKeepPitch + c] = (uint8_t)kb;
      float4 o;   // (drop(in) + drop(out) + loop) / 3 [+ bias]   (model.py:103-105)
      o.x = (a.x + b.x + l.x) / 3.0f + bv.x;
      o.y = (a.y + b.y + l.y) / 3.0f + bv.y;
      o.z = (a.z + b.z + l.z) / 3.0f + bv.z;
      o.w = (a.w + b.w + l.w) / 3.0f + bv.w;
      pre[i] = o;
      sum.x += o.x; sum.y += o.y; sum.z += o.z; sum.w += o.w;
      sq.x += (double)o.x * o.x; sq.y += (double)o.y * o.y; sq.z += (double)o.z * o.z; sq.w += (double)o.w * o.w;
    }
  }
  block_store_partials(sum, sq, rl, c, RL, Do4, partials, sm);
}

// Column finalisers: one block per 8 columns; 32 row-lanes stride over the per-block partials, then the
// 32 lane sums are added in lane order - fixed order, deterministic, and ~100x less serial than one
// thread per column.
constexpr int kFinCols = 2, kFinLanes = 128;     // 100 blocks of 256 threads for Dout = 200

__device__ __forceinline__ void reduce_partials(const double* __restrict__ partials, int64_t n_blocks, int Dout,
                                                int c, int lane, double (*sm)[kFinLanes][kFinCols], double* s_out,
                                                double* q_out) {
  double s = 0, q = 0;
  if (c < Dout) {
    for (int64_t b = lane; b < n_blocks; b += kFinLanes) {
      s += partials[(b * 2 + 0) * Dout + c];
      q += partials[(b * 2 + 1) * Dout + c];
    }
  }
  const int cc = threadIdx.x % kFinCols;
  sm[0][lane][cc] = s;
  sm[1][lane][cc] = q;
  __syncthreads();
  if (lane == 0) {
    s = sm[0][0][cc];
    q = sm[1][0][cc];
    for (int k = 1; k < kFinLanes; ++k) {
      s += sm[0][k][cc];
      q += sm[1][k][cc];
    }
  }
  *s_out = s;
  *q_out = q;
}

// sums[0][c] = sum over blocks of partial 0, sums[1][c] = of partial 1 (fp64, fixed order)
__global__ void __launch_bounds__(kFinCols * kFinLanes)
colsum_finalize_kernel(const double* __restrict__ partials, int64_t n_blocks, int Dout, double* __restrict__ sums) {
  __shared__ double sm[2][kFinLanes][kFinCols];
  const int c = blockIdx.x * kFinCols + threadIdx.x % kFinCols, lane = threadIdx.x / kFinCols;
  double s = 0, q = 0;
  reduce_partials(partials, n_blocks, Dout, c, lane, sm, &s, &q);
  if (lane != 0 || c >= Dout) return;
  sums[c] = s;
  sums[Dout + c] = q;
}

// the same reduction, with a float copy of the sums (the backward hands d_beta / d_gamma to autograd in fp32)
__global__ void __launch_bounds__(kFinCols * kFinLanes)
colsum_finalize2_kernel(const double* __restrict__ partials, int64_t n_blocks, int Dout, double* __restrict__ sums,
                        float* __restrict__ sums32) {
  __shared__ double sm[2][kFinLanes][kFinCols];
  const int c = blockIdx.x * kFinCols + threadIdx.x % kFinCols, lane = threadIdx.x / kFinCols;
  double s = 0, q = 0;
  reduce_partials(partials, n_blocks, Dout, c, lane, sm, &s, &q);
  if (lane != 0 || c >= Dout) return;
  sums[c] = s;
  sums[Dout + c] = q;
  sums32[c] = (float)s;
  sums32[Dout + c] = (float)q;
}

// single-GPU training: partials -> sums -> batch statistics -> nn.BatchNorm1d's running-statistics update, one launch
__global__ void __launch_bounds__(kFinCols * kFinLanes)
colstats_finalize_kernel(const double* __restrict__ partials, int64_t n_blocks, int64_t n_rows, int Dout, float eps,
                         float momentum, float* __restrict__ rmean, float* __restrict__ rvar,
                         int64_t* __restrict__ n_tracked, double* __restrict__ sums, float* __restrict__ stats) {
  __shared__ double sm[2][kFinLanes][kFinCols];
  const int c = blockIdx.x * kFinCols + threadIdx.x % kFinCols, lane = threadIdx.x / kFinCols;
  double s = 0, q = 0;
  reduce_partials(partials, n_blocks, Dout, c, lane, sm, &s, &q);
  if (blockIdx.x == 0 && threadIdx.x == 0 && n_tracked != nullptr) *n_tracked += 1;
  if (lane != 0 || c >= Dout) return;
  if (sums != nullptr) {
    sums[c] = s;
    sums[Dout + c] = q;
  }
  const double mean = s / (double)n_rows;
  double var = q / (double)n_rows - mean * mean;
  if (var < 0) var = 0;
  const float meanf = (float)mean, varf = (float)var;
  stats[c] = meanf;
  stats[Dout + c] = varf;
  stats[2 * Dout + c] = (float)(1.0 / sqrt(var + (double)eps));
  if (rmean != nullptr && rvar != nullptr) {        // momentum update with the UNBIASED variance (torch semantics, fp32)
    const float unbias = (float)n_rows / (float)(n_rows > 1 ? n_rows - 1 : 1);
    rmean[c] = rmean[c] * (1.f - momentum) + momentum * meanf;
    rvar[c] = rvar[c] * (1.f - momentum) + (momentum * unbias) * varf;
  }
}

// stats[0] = mean, stats[1] = biased variance, stats[2] = 1/sqrt(var + eps)
__global__ void colstats_from_sums_kernel(const double* __restrict__ sums, int64_t n_rows, int Dout, float eps,
                                          int training, const float* __restrict__ rmean,
                                          const float* __restrict__ rvar, float* __restrict__ stats) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= Dout) return;
  double mean, var;
  if (training) {
    mean = sums[c] / (double)n_rows;
    var = sums[Dout + c] / (double)n_rows - mean * mean;
    if (var < 0) var = 0;
  } else {
    mean = rmean[c];
    var = rvar[c];
  }
  stats[c] = (float)mean;
  stats[Dout + c] = (float)var;
  stats[2 * Dout + c] = (float)(1.0 / sqrt(var + (double)eps));
}

// Optional dropout of the OUTPUT (MGCN.encode applies F.dropout(all_ent, gcn_drop) right after the layer, model.py:34: a
// read + write + mask pass over [N, Dout] each way): the same Philox stream as the tail's own masks, plane 2; the keep
// flags go to out_keep (low nibble of byte c of a row = columns 4c..4c+3) for the backward.
struct OutDrop {
  const int64_t* seed;        // NULL: no output dropout
  uint32_t drop_thr;
  float keep_scale;
  uint8_t* keep;              // written by the forward / read by the backward
};

__global__ void __launch_bounds__(kThreads)
tail_apply_kernel(const float4* __restrict__ pre, const float4* __restrict__ stats, const float4* __restrict__ gamma,
                  const float4* __restrict__ beta, int64_t n4, int Do4, float4* __restrict__ all_ent, const OutDrop od) {
  const int64_t i = blockIdx.x * (int64_t)kThreads + threadIdx.x;
  if (i >= n4) return;
  const int c = (int)(i % Do4);
  const float4 v = __ldg(pre + i), m = __ldg(stats + c), rs = __ldg(stats + 2 * Do4 + c);
  const float4 ga = __ldg(gamma + c), be = __ldg(beta + c);
  float4 o;   // tanh(BatchNorm(out))   (model.py:106)
  o.x = tanhf((v.x - m.x) * rs.x * ga.x + be.x);
  o.y = tanhf((v.y - m.y) * rs.y * ga.y + be.y);
  o.z = tanhf((v.z - m.z) * rs.z * ga.z + be.z);
  o.w = tanhf((v.w - m.w) * rs.w * ga.w + be.w);
  if (od.seed != nullptr) {
    const float4 k = philox_mask4(i, 2u, (uint64_t)__ldg(od.seed), od.drop_thr, od.keep_scale);
    o.x *= k.x; o.y *= k.y; o.z *= k.z; o.w *= k.w;
    od.keep[(i / Do4) * kKeepPitch + c] = (uint8_t)nibble(k);
  }
  all_ent[i] = o;
}

__global__ void __launch_bounds__(kThreads)
tail_bwd_reduce_kernel(const float4* __restrict__ g_ent, const float4* __restrict__ pre, const float4* __restrict__ stats,
                       const float4* __restrict__ gamma, const float4* __restrict__ beta, int64_t n_rows, int Do4,
                       double* __restrict__ partials, const uint8_t* __restrict__ out_keep, float out_scale) {
  extern __shared__ double4 sm[];
  const int RL = kThreads / Do4;
  const int rl = threadIdx.x / Do4, c = threadIdx.x % Do4;
  const Stripe s = block_stripe(n_rows);
  double4 s1 = make_double4(0, 0, 0, 0), s2 = make_double4(0, 0, 0, 0);
  if (rl < RL) {
    // all_ent = tanh(BatchNorm(pre)) is recomputed from pre (one plane less to read; the tail is HBM-bound)
    const float4 m = __ldg(stats + c), rs = __ldg(stats + 2 * Do4 + c), ga = __ldg(gamma + c), be = __ldg(beta + c);
    for (int64_t r = s.row_beg + rl; r < s.row_end; r += RL) {
      const int64_t i = r * Do4 + c;
      float4 g = __ldg(g_ent + i);
      const float4 v = __ldg(pre + i);
      if (out_keep != nullptr) g = keep4(g, out_keep[r * kKeepPitch + c], out_scale);
      const float4 xh = make_float4((v.x - m.x) * rs.x, (v.y - m.y) * rs.y, (v.z - m.z) * rs.z, (v.w - m.w) * rs.w);
      const float4 t = make_float4(tanhf(xh.x * ga.x + be.x), tanhf(xh.y * ga.y + be.y), tanhf(xh.z * ga.z + be.z),
                                   tanhf(xh.w * ga.w + be.w));
      const float dzx = g.x * (1.f - t.x * t.x), dzy = g.y * (1.f - t.y * t.y);
      const float dzz = g.z * (1.f - t.z * t.z), dzw = g.w * (1.f - t.w * t.w);
      s1.x += dzx; s1.y += dzy; s1.z += dzz; s1.w += dzw;
      s2.x += (double)dzx * xh.x;
      s2.y += (double)dzy * xh.y;
      s2.z += (double)dzz * xh.z;
      s2.w += (double)dzw * xh.w;
    }
  }
  block_store_partials(s1, s2, rl, c, RL, Do4, partials, sm);
}

__global__ void __launch_bounds__(kThreads)
tail_bwd_apply_kernel(const float4* __restrict__ g_ent, const float4* __restrict__ pre, const float4* __restrict__ stats,
                      const float4* __restrict__ gamma, const float4* __restrict__ beta, const double* __restrict__ sums,
                      int training, int64_t n_rows, int64_t n_rows_global, int Do4, float4* __restrict__ d_out,
                      const uint8_t* __restrict__ keep, float keep_scale, float4* __restrict__ d_res_in,
                      float4* __restrict__ d_res_out, const int32_t* __restrict__ slot_in,
                      const int32_t* __restrict__ slot_out, const uint8_t* __restrict__ out_keep, float out_scale) {
  const int64_t n4 = n_rows * (int64_t)Do4;
  const int64_t i = blockIdx.x * (int64_t)kThreads + threadIdx.x;
  if (i >= n4) return;
  const int c = (int)(i % Do4);
  float4 g = __ldg(g_ent + i);
  const float4 v = __ldg(pre + i);
  if (out_keep != nullptr) g = keep4(g, out_keep[(i / Do4) * kKeepPitch + c], out_scale);
  const float4 m = __ldg(stats + c), rs = __ldg(stats + 2 * Do4 + c), ga = __ldg(gamma + c), be = __ldg(beta + c);
  const float4 xh = make_float4((v.x - m.x) * rs.x, (v.y - m.y) * rs.y, (v.z - m.z) * rs.z, (v.w - m.w) * rs.w);
  const float4 t = make_float4(tanhf(xh.x * ga.x + be.x), tanhf(xh.y * ga.y + be.y), tanhf(xh.z * ga.z + be.z),
                               tanhf(xh.w * ga.w + be.w));
  float4 dz = make_float4(g.x * (1.f - t.x * t.x), g.y * (1.f - t.y * t.y), g.z * (1.f - t.z * t.z),
                          g.w * (1.f - t.w * t.w));
  float4 dp;
  if (training) {   // BatchNorm backward with batch statistics
    const float inv_n = 1.0f / (float)n_rows_global;
    const double* sp = sums + 4 * c;
    const double* sq = sums + 4 * (Do4 + c);
    const float4 s1 = make_float4((float)sp[0], (float)sp[1], (float)sp[2], (float)sp[3]);
    const float4 s2 = make_float4((float)sq[0], (float)sq[1], (float)sq[2], (float)sq[3]);
    dp.x = ga.x * rs.x * (dz.x - s1.x * inv_n - xh.x * s2.x * inv_n);
    dp.y = ga.y * rs.y * (dz.y - s1.y * inv_n - xh.y * s2.y * inv_n);
    dp.z = ga.z * rs.z * (dz.z - s1.z * inv_n - xh.z * s2.z * inv_n);
    dp.w = ga.w * rs.w * (dz.w - s1.w * inv_n - xh.w * s2.w * inv_n);
  } else {
    dp = make_float4(ga.x * rs.x * dz.x, ga.y * rs.y * dz.y, ga.z * rs.z * dz.z, ga.w * rs.w * dz.w);
  }
  // ONE upstream plane: d out / 3.  The self-loop transform takes it as it is; the in / out halves are this plane times
  // their keep flags x 1 / (1 - p), applied by the GEMM kernels while they split the operand (tail_fwd's packed flags)
  const float4 third = make_float4(dp.x / 3.0f, dp.y / 3.0f, dp.z / 3.0f, dp.w / 3.0f);
  d_out[i] = third;
  if (d_res_in != nullptr) {
    // three-plane form: the dropped in / out planes are written here (tail_fwd's keep flags, nothing regenerated) and the
    // GEMMs stream them as they are - their operand splitters are the busier side of those kernels.  A compacted plane
    // (slot != NULL) receives only the rows that have edges, at their compact row
    const int64_t r = i / Do4;
    const uint32_t kb = keep != nullptr ? keep[r * kKeepPitch + c] : 0xFFu;
    const float s = keep != nullptr ? keep_scale : 1.f;
    const int64_t o_in = slot_in == nullptr ? i : (int64_t)__ldg(slot_in + r) * Do4 + c;
    const int64_t o_out = slot_out == nullptr ? i : (int64_t)__ldg(slot_out + r) * Do4 + c;
    if (o_in >= 0)
      d_res_in[o_in] = make_float4((kb & 1u) ? third.x * s : 0.f, (kb & 2u) ? third.y * s : 0.f,
                                   (kb & 4u) ? third.z * s : 0.f, (kb & 8u) ? third.w * s : 0.f);
    if (o_out >= 0)
      d_res_out[o_out] = make_float4((kb & 16u) ? third.x * s : 0.f, (kb & 32u) ? third.y * s : 0.f,
                                     (kb & 64u) ? third.z * s : 0.f, (kb & 128u) ? third.w * s : 0.f);
  }
}

// dst[dst_rows[j]] = src[src_rows[j]] for j < n (rows of D floats; a NULL row list is the identity): the gather of the
// occupied rows of an aggregation plane into its compact block, and the scatter of the compact upstream rows back
__global__ void __launch_bounds__(kThreads)
rows_copy_kernel(const float4* __restrict__ src, int64_t ld_src, const int32_t* __restrict__ src_rows, float4* __restrict__ dst,
                 int64_t ld_dst, const int32_t* __restrict__ dst_rows, int64_t n4, int D4) {
  const int64_t i = blockIdx.x * (int64_t)kThreads + threadIdx.x;
  if (i >= n4) return;
  const int64_t j = i / D4;
  const int c = (int)(i % D4);
  const int64_t rs = src_rows != nullptr ? (int64_t)__ldg(src_rows + j) : j;
  const int64_t rd = dst_rows != nullptr ? (int64_t)__ldg(dst_rows + j) : j;
  dst[rd * ld_dst + c] = __ldg(src + rs * ld_src + c);
}

inline int check_dout(int32_t Dout) { return (Dout <= 0 || Dout % 4 != 0 || Dout > 1024) ? 1 : 0; }
inline size_t partial_smem(int Do4) { return size_t(2) * (kThreads / Do4) * Do4 * sizeof(double4); }

}  // namespace
}  // namespace kgc

using namespace kgc;

extern "C" int64_t kgc_tail_num_blocks(int64_t n_rows) {
  int64_t nb = ceil_div(n_rows > 0 ? n_rows : 1, 32);
  return nb < kMaxBlocks ? nb : kMaxBlocks;
}

static DropCfg make_drop(const uint8_t* mask_in, const uint8_t* mask_out, const int64_t* seed, float drop_p, float keep_scale) {
  DropCfg d;
  d.mask_in = mask_in;
  d.mask_out = mask_out;
  d.seed = (seed != nullptr && drop_p > 0.f) ? seed : nullptr;
  const double thr = (double)drop_p * 4294967296.0;
  d.drop_thr = thr >= 4294967295.0 ? 0xFFFFFFFFu : (uint32_t)thr;
  d.keep_scale = keep_scale;
  return d;
}

// one float4 of keep flags per thread: exactly the mask the tail kernels regenerate from (seed, plane)
__global__ void dropout_mask_kernel(const int64_t* __restrict__ seed, uint32_t plane, uint32_t drop_thr, int64_t n4,
                                    uchar4* __restrict__ out) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n4) return;
  const float4 m = philox_mask4(i, plane, (uint64_t)__ldg(seed), drop_thr, 1.0f);
  out[i] = make_uchar4(m.x != 0.f, m.y != 0.f, m.z != 0.f, m.w != 0.f);
}

extern "C" int kgc_dropout_mask(const int64_t* seed, int32_t plane, float drop_p, int64_t n_elem, uint8_t* mask, void* stream) {
  KGC_REQUIRE(seed != nullptr && n_elem % 4 == 0 && plane >= 0, "bad arguments");
  const DropCfg d = make_drop(nullptr, nullptr, seed, drop_p, 1.0f);
  const int64_t n4 = n_elem / 4;
  if (n4 == 0) return 0;
  dropout_mask_kernel<<<(unsigned)ceil_div(n4, kThreads), kThreads, 0, as_stream(stream)>>>(seed, (uint32_t)plane, d.drop_thr,
                                                                                     n4, (uchar4*)mask);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int32_t kgc_keep_pitch() { return kKeepPitch; }

extern "C" int kgc_tail_fwd_rows(const float* res3, const int32_t* slot_in, const float* rows_in, const int32_t* slot_out,
                                 const float* rows_out, const uint8_t* mask_in, const uint8_t* mask_out, const int64_t* seed,
                                 float drop_p, float keep_scale, const float* bias, int64_t n_rows, int32_t Dout, float* pre,
                                 double* partials, uint8_t* keep, void* stream) {
  KGC_REQUIRE(check_dout(Dout) == 0, "Dout must be a multiple of 4 and <= 1024");
  KGC_REQUIRE(keep == nullptr || Dout <= 4 * kKeepPitch, "packed keep flags need Dout <= 256");
  KGC_REQUIRE(n_rows > 0, "n_rows must be positive");
  KGC_REQUIRE((slot_in == nullptr || rows_in != nullptr) && (slot_out == nullptr || rows_out != nullptr),
              "a compacted plane needs its rows");
  const int Do4 = Dout / 4;
  const size_t smem = partial_smem(Do4);   // <= 16 KB
  PlaneRows pr;
  pr.slot[0] = slot_in;
  pr.slot[1] = slot_out;
  pr.rows[0] = (const float4*)rows_in;
  pr.rows[1] = (const float4*)rows_out;
  tail_fwd_kernel<<<(unsigned)kgc_tail_num_blocks(n_rows), kThreads, smem, as_stream(stream)>>>(
      (const float4*)res3, pr, make_drop(mask_in, mask_out, seed, drop_p, keep_scale), (const float4*)bias, n_rows, Do4,
      (float4*)pre, partials, keep);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_tail_fwd(const float* res3, const uint8_t* mask_in, const uint8_t* mask_out, const int64_t* seed,
                            float drop_p, float keep_scale, const float* bias, int64_t n_rows, int32_t Dout, float* pre,
                            double* partials, uint8_t* keep, void* stream) {
  return kgc_tail_fwd_rows(res3, nullptr, nullptr, nullptr, nullptr, mask_in, mask_out, seed, drop_p, keep_scale, bias, n_rows,
                           Dout, pre, partials, keep, stream);
}

extern "C" int kgc_rows_copy(const float* src, int64_t ld_src, const int32_t* src_rows, float* dst, int64_t ld_dst,
                             const int32_t* dst_rows, int64_t n, int32_t D, void* stream) {
  KGC_REQUIRE(D > 0 && D % 4 == 0 && ld_src % 4 == 0 && ld_dst % 4 == 0 && n >= 0, "rows of a multiple of 4 floats");
  KGC_REQUIRE(n == 0 || (src != nullptr && dst != nullptr), "null buffer");
  const int64_t n4 = n * (D / 4);
  if (n4 == 0) return 0;
  rows_copy_kernel<<<(unsigned)ceil_div(n4, kThreads), kThreads, 0, as_stream(stream)>>>(
      (const float4*)src, ld_src / 4, src_rows, (float4*)dst, ld_dst / 4, dst_rows, n4, D / 4);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_colsum_finalize(const double* partials, int64_t n_blocks, int32_t Dout, double* sums, void* stream) {
  KGC_REQUIRE(check_dout(Dout) == 0, "Dout must be a multiple of 4 and <= 1024");
  colsum_finalize_kernel<<<(unsigned)ceil_div(Dout, kFinCols), kFinCols * kFinLanes, 0, as_stream(stream)>>>(
      partials, n_blocks, Dout, sums);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_colsum_finalize2(const double* partials, int64_t n_blocks, int32_t Dout, double* sums, float* sums32,
                                    void* stream) {
  KGC_REQUIRE(check_dout(Dout) == 0, "Dout must be a multiple of 4 and <= 1024");
  KGC_REQUIRE(partials && sums && sums32 && n_blocks > 0, "null buffer");
  colsum_finalize2_kernel<<<(unsigned)ceil_div(Dout, kFinCols), kFinCols * kFinLanes, 0, as_stream(stream)>>>(
      partials, n_blocks, Dout, sums, sums32);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_colstats_finalize(const double* partials, int64_t n_blocks, int64_t n_rows, int32_t Dout, float eps,
                                     float momentum, float* running_mean, float* running_var,
                                     int64_t* num_batches_tracked, double* sums, float* stats, void* stream) {
  KGC_REQUIRE(check_dout(Dout) == 0, "Dout must be a multiple of 4 and <= 1024");
  KGC_REQUIRE(partials && stats && n_blocks > 0 && n_rows > 0, "null buffer");
  KGC_REQUIRE((running_mean == nullptr) == (running_var == nullptr), "running_mean and running_var come together");
  colstats_finalize_kernel<<<(unsigned)ceil_div(Dout, kFinCols), kFinCols * kFinLanes, 0, as_stream(stream)>>>(
      partials, n_blocks, n_rows, Dout, eps, momentum, running_mean, running_var, num_batches_tracked, sums, stats);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_colstats_from_sums(const double* sums, int64_t n_rows, int32_t Dout, float eps, int32_t training,
                                      const float* running_mean, const float* running_var, float* stats, void* stream) {
  KGC_REQUIRE(check_dout(Dout) == 0, "Dout must be a multiple of 4 and <= 1024");
  KGC_REQUIRE(training || (running_mean && running_var), "eval mode needs running statistics");
  KGC_REQUIRE(!training || sums, "training mode needs the column sums");
  colstats_from_sums_kernel<<<(unsigned)ceil_div(Dout, 128), 128, 0, as_stream(stream)>>>(
      sums, n_rows, Dout, eps, training, running_mean, running_var, stats);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_tail_apply(const float* pre, const float* stats, const float* gamma, const float* beta,
                              int64_t n_rows, int32_t Dout, float* all_ent, const int64_t* out_seed, float out_drop_p,
                              uint8_t* out_keep, void* stream) {
  KGC_REQUIRE(check_dout(Dout) == 0, "Dout must be a multiple of 4 and <= 1024");
  const int Do4 = Dout / 4;
  const int64_t n4 = n_rows * Do4;
  OutDrop od;
  od.seed = (out_seed != nullptr && out_drop_p > 0.f) ? out_seed : nullptr;
  KGC_REQUIRE(od.seed == nullptr || (out_keep != nullptr && Dout <= 4 * kKeepPitch && out_drop_p < 1.f),
              "output dropout needs a keep-flag buffer, Dout <= 256 and p < 1");
  const DropCfg d = make_drop(nullptr, nullptr, out_seed, out_drop_p, 1.f);
  od.drop_thr = d.drop_thr;
  od.keep_scale = 1.f / (1.f - out_drop_p);
  od.keep = out_keep;
  tail_apply_kernel<<<(unsigned)ceil_div(n4, kThreads), kThreads, 0, as_stream(stream)>>>(
      (const float4*)pre, (const float4*)stats, (const float4*)gamma, (const float4*)beta, n4, Do4, (float4*)all_ent, od);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_tail_bwd_reduce(const float* g_ent, const float* pre, const float* stats, const float* gamma,
                                   const float* beta, int64_t n_rows, int32_t Dout, double* partials, const uint8_t* out_keep,
                                   float out_scale, void* stream) {
  KGC_REQUIRE(check_dout(Dout) == 0, "Dout must be a multiple of 4 and <= 1024");
  const int Do4 = Dout / 4;
  const size_t smem = partial_smem(Do4);   // <= 16 KB
  tail_bwd_reduce_kernel<<<(unsigned)kgc_tail_num_blocks(n_rows), kThreads, smem, as_stream(stream)>>>(
      (const float4*)g_ent, (const float4*)pre, (const float4*)stats, (const float4*)gamma, (const float4*)beta, n_rows, Do4,
      partials, out_keep, out_scale);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_tail_bwd_apply_rows(const float* g_ent, const float* pre, const float* stats, const float* gamma,
                                       const float* beta, const double* sums, int32_t training, int64_t n_rows,
                                       int64_t n_rows_global, int32_t Dout, float* d_out, const uint8_t* keep, float keep_scale,
                                       float* d_res_in, const int32_t* slot_in, float* d_res_out, const int32_t* slot_out,
                                       const uint8_t* out_keep, float out_scale, void* stream) {
  KGC_REQUIRE(check_dout(Dout) == 0, "Dout must be a multiple of 4 and <= 1024");
  KGC_REQUIRE((d_res_in == nullptr) == (d_res_out == nullptr), "the in and out planes come together");
  const int Do4 = Dout / 4;
  const int64_t n4 = n_rows * Do4;
  tail_bwd_apply_kernel<<<(unsigned)ceil_div(n4, kThreads), kThreads, 0, as_stream(stream)>>>(
      (const float4*)g_ent, (const float4*)pre, (const float4*)stats, (const float4*)gamma, (const float4*)beta, sums,
      training, n_rows, n_rows_global, Do4, (float4*)d_out, keep, keep_scale, (float4*)d_res_in, (float4*)d_res_out, slot_in,
      slot_out, out_keep, out_scale);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_tail_bwd_apply(const float* g_ent, const float* pre, const float* stats, const float* gamma,
                                  const float* beta, const double* sums, int32_t training, int64_t n_rows,
                                  int64_t n_rows_global, int32_t Dout, float* d_out, const uint8_t* keep, float keep_scale,
                                  float* d_res2, const uint8_t* out_keep, float out_scale, void* stream) {
  return kgc_tail_bwd_apply_rows(g_ent, pre, stats, gamma, beta, sums, training, n_rows, n_rows_global, Dout, d_out, keep,
                                 keep_scale, d_res2, nullptr, d_res2 != nullptr ? d_res2 + n_rows * Dout : nullptr, nullptr,
                                 out_keep, out_scale, stream);
}
