// Training-time 1-N scoring, backward through the sigmoid (autograd of reference model.py:177-179).
//
// The forward (kgc_score_1n_fwd, gemm_tf32x3.cu) produced pred[B, N] = sigmoid(X E^T + bias).  The two gradient GEMMs
// that follow contract over the batch (d_E = d_logit^T X) and over the entities (d_X = d_logit E); both tensor-core
// kernels stream their big operand row-major with the ENTITY index as the row, so this kernel writes the logit gradient
// transposed, d_logitT[N, ldt], in the same pass that applies p (1 - p) and reduces the bias gradient:
//   d_logitT[n, b] = d_pred[b, n] * pred[b, n] * (1 - pred[b, n]),     d_bias[n] = sum_b d_logitT[n, b]
// One CTA owns 32 entities and walks the batch in tiles of 32 queries: coalesced 128-byte reads along n, a padded
// shared-memory transpose, coalesced 128-byte writes along b.  The bias sum is a fixed shuffle tree per tile, tiles added
// in order: deterministic, no atomics.
#include "bce.cuh"
#include "common.cuh"

namespace kgc {
namespace {

constexpr int kThreadsST = 256;

__global__ void __launch_bounds__(kThreadsST)
score_1n_bwd_logit_kernel(const float* __restrict__ d_pred, int64_t ld_dp, const float* __restrict__ pred, int64_t ld_p,
                          int64_t n_ent, int B, int ldt, float* __restrict__ d_logitT, float* __restrict__ d_bias) {
  __shared__ float tile[32][33];
  const int lane = threadIdx.x % 32, warp = threadIdx.x / 32;      // 8 warps x 4 rows
  const int64_t n0 = (int64_t)blockIdx.x * 32;
  float bias_acc[4] = {0.f, 0.f, 0.f, 0.f};                         // lane 0 of each warp: rows warp * 4 + i
  for (int b0 = 0; b0 < ldt; b0 += 32) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int b = b0 + warp * 4 + i;
      const int64_t n = n0 + lane;
      float g = 0.f;
      if (b < B && n < n_ent) {
        const float p = pred[(int64_t)b * ld_p + n];
        g = d_pred[(int64_t)b * ld_dp + n] * p * (1.f - p);
      }
      tile[warp * 4 + i][lane] = g;
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = warp * 4 + i;                                   // entity n0 + r, query b0 + lane
      const float g = tile[lane][r];
      if (n0 + r < n_ent && b0 + lane < ldt) d_logitT[(n0 + r) * ldt + b0 + lane] = g;   // pad columns [B, ldt) get zeros
      float s = g;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
      bias_acc[i] += s;
    }
    __syncthreads();
  }
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (n0 + warp * 4 + i < n_ent) d_bias[n0 + warp * 4 + i] = bias_acc[i];
  }
}

// ---- N1 (SURVEY.md 8(f)): BCE against SPARSE positives fused with the backward through the sigmoid ----------------
// The reference builds a dense multi-hot label [B, N] per batch (data_loader.py:34-43), copies it to the device and runs
// BCELoss over it (model.py:42-44).  Here the label exists only as one bit per (entity, query): label_mask_t_kernel sets the
// bits of the batch's positives (integer atomicOr: order-independent), and bce_1n_t_kernel walks pred once, producing the
// summed loss AND the logit gradient AND the bias gradient - the dense label, the BCE forward and the BCE backward passes
// over [B, N] disappear.  Arithmetic follows ATen's kernels:
//   loss term   = (y - 1) * max(log1p(-p), -100) - y * max(log(p), -100)
//   d_pred      = (p - y) / max((1 - p) * p, 1e-12) * (1 / (B N))          (mean reduction, unit upstream)
//   d_logit     = d_pred * p * (1 - p)                                     (as score_1n_bwd_logit_kernel)
// with y = pos on the batch's positives and add elsewhere (the two values kgc_label_build writes).
//
// Everything is ENTITY-MAJOR.  A batch-major pred [B, N] has rows 4 N bytes apart: the scorer's transposed TMA stores and a
// loss kernel's reads touch it in 128-byte pieces, one per DRAM page - 3.4 ms each at N = 4.6 M (1.4-1.8 TB/s).  The
// scorer instead stores its natural orientation predT [N, ldt] (rows of 4 B bytes, contiguous), the label bits are kept
// per entity (maskT [N, ceil(B / 32)]), and bce_1n_t_kernel is a plain row-wise pass that overwrites predT with the logit
// gradient IN PLACE - no transpose, no second [B, N]-sized buffer.
__global__ void __launch_bounds__(kThreadsST)
label_mask_t_kernel(const int64_t* __restrict__ qid, const int64_t* __restrict__ ptr, const int32_t* __restrict__ idx,
                    int64_t n_entity, int wb, uint32_t* __restrict__ mask_t) {
  const int64_t b = blockIdx.x;
  const int64_t q = qid[b];
  for (int64_t k = ptr[q] + threadIdx.x; k < ptr[q + 1]; k += kThreadsST) {
    const int64_t j = idx[k];
    if (j >= 0 && j < n_entity) atomicOr(mask_t + j * wb + (b >> 5), 1u << (b & 31));
  }
}

// one warp per entity row (grid-stride, fixed assignment: deterministic); a lane owns the float4 columns lane, lane + 32, ...
__global__ void __launch_bounds__(kThreadsST)
bce_1n_t_kernel(float* __restrict__ pred_t, const uint32_t* __restrict__ mask_t, int wb, int64_t n_ent, int B, int ldt,
                float pos, float add, float inv_count, float* __restrict__ d_bias, double* __restrict__ loss_partial) {
  __shared__ double warp_loss[kThreadsST / 32];
  const int lane = threadIdx.x % 32, warp = threadIdx.x / 32;
  const int64_t n_warps = (int64_t)gridDim.x * (kThreadsST / 32);
  double loss = 0.0;
  for (int64_t n = (int64_t)blockIdx.x * (kThreadsST / 32) + warp; n < n_ent; n += n_warps) {
    float4* row = reinterpret_cast<float4*>(pred_t + n * ldt);
    float bsum = 0.f;
    for (int c = lane; c * 4 < ldt; c += 32) {
      float4 v = row[c];
      const uint32_t w = __ldg(mask_t + n * wb + ((4 * c) >> 5)) >> ((4 * c) & 31);
      float* e = reinterpret_cast<float*>(&v);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float g = 0.f;
        if (4 * c + j < B) {
          const float p = e[j];
          const float y = ((w >> j) & 1u) ? pos : add;
          loss += (double)bce_loss_term(p, y);
          g = bce_logit_grad(p, y, inv_count);
        }
        e[j] = g;                                                   // pad columns [B, ldt) get zeros
        bsum += g;
      }
      row[c] = v;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) bsum += __shfl_xor_sync(0xFFFFFFFFu, bsum, o);
    if (lane == 0) d_bias[n] = bsum;
  }
  const double s = cta_sum(warp_sum(loss), warp_loss, lane, warp);
  if (threadIdx.x == 0) loss_partial[blockIdx.x] = s;
}

// mean over B * N elements: one CTA adds the per-CTA partials in a fixed order (thread t takes t, t + 256, ...; then a tree)
__global__ void __launch_bounds__(kThreadsST)
bce_1n_finalize_kernel(const double* __restrict__ partial, int64_t n_partial, double inv_count, float* __restrict__ loss) {
  __shared__ double sh[kThreadsST];
  const double s = cta_sum_partials(partial, n_partial, sh);
  if (threadIdx.x == 0) loss[0] = (float)(s * inv_count);
}

// ---- the same loss on an ENTITY-SHARDED table (several GPUs, MGCN.shard): rank r holds the rows of the entities it owns,
// in its own row order.  The label bits of a shard are those of kgc_label_mask_t_build with entity j moved to its local
// row row_of[j] (-1: another rank owns j).  The loss pass is bce_1n_t_kernel itself, with the divisor of the whole table
// (B * n_total): each of the shard's gradient rows is bit-identical to that row of the unsharded pass.  The shard's loss is
// returned as a plain fp64 sum (the ranks add their sums; the caller divides).
__global__ void __launch_bounds__(kThreadsST)
label_mask_t_rows_kernel(const int64_t* __restrict__ qid, const int64_t* __restrict__ ptr, const int32_t* __restrict__ idx,
                         const int32_t* __restrict__ row_of, int64_t n_rows, int wb, uint32_t* __restrict__ mask_t) {
  const int64_t b = blockIdx.x;
  const int64_t q = qid[b];
  for (int64_t k = ptr[q] + threadIdx.x; k < ptr[q + 1]; k += kThreadsST) {
    const int64_t j = idx[k];
    if (j < 0) continue;
    const int64_t r = row_of[j];
    if (r >= 0 && r < n_rows) atomicOr(mask_t + r * wb + (b >> 5), 1u << (b & 31));
  }
}

// the shard's loss: the per-CTA partials added in bce_1n_finalize_kernel's order, not scaled
__global__ void __launch_bounds__(kThreadsST)
bce_1n_sum_kernel(const double* __restrict__ partial, int64_t n_partial, double* __restrict__ loss_sum) {
  __shared__ double sh[kThreadsST];
  const double s = cta_sum_partials(partial, n_partial, sh);
  if (threadIdx.x == 0) loss_sum[0] = s;
}

}  // namespace
}  // namespace kgc

using namespace kgc;

extern "C" int kgc_score_1n_bwd_logit(const float* d_pred, int64_t ld_dp, const float* pred, int64_t ld_p, int64_t n_ent,
                                      int32_t B, int32_t ldt, float* d_logitT, float* d_bias, void* stream) {
  KGC_REQUIRE(n_ent > 0 && B > 0 && ldt >= B && ld_dp >= n_ent && ld_p >= n_ent, "bad sizes");
  KGC_REQUIRE(d_pred && pred && d_logitT && d_bias, "null buffer");
  score_1n_bwd_logit_kernel<<<(unsigned)ceil_div(n_ent, 32), kThreadsST, 0, as_stream(stream)>>>(
      d_pred, ld_dp, pred, ld_p, n_ent, B, ldt, d_logitT, d_bias);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int64_t kgc_bce_1n_t_blocks(int64_t n_ent) {
  const int64_t b = ceil_div(n_ent > 0 ? n_ent : 1, kThreadsST / 32);
  return b < 8 * kNumSMs ? b : 8 * kNumSMs;
}

extern "C" int kgc_label_mask_t_build(const int64_t* qid, int64_t B, const int64_t* ptr, const int32_t* idx, int64_t n_entity,
                                      uint32_t* mask_t, void* stream) {
  KGC_REQUIRE(B >= 0 && n_entity > 0, "bad sizes");
  if (B == 0) return 0;
  KGC_REQUIRE(qid && ptr && idx && mask_t, "null buffer");
  const int wb = (int)ceil_div(B, 32);
  KGC_CUDA_TRY(cudaMemsetAsync(mask_t, 0, (size_t)(n_entity * wb) * sizeof(uint32_t), as_stream(stream)));
  label_mask_t_kernel<<<(unsigned)B, kThreadsST, 0, as_stream(stream)>>>(qid, ptr, idx, n_entity, wb, mask_t);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_bce_1n_bwd_logit_t(float* pred_t, const uint32_t* mask_t, int64_t n_ent, int32_t B, int32_t ldt, float pos,
                                      float add, float* d_bias, double* loss_partial, float* loss, void* stream) {
  KGC_REQUIRE(n_ent > 0 && B > 0 && ldt >= B && ldt % 4 == 0, "bad sizes (ldt a multiple of 4)");
  KGC_REQUIRE(pred_t && mask_t && d_bias && loss_partial && loss, "null buffer");
  KGC_REQUIRE((reinterpret_cast<uintptr_t>(pred_t) & 15) == 0, "pred_t must be 16-byte aligned");
  const int64_t blocks = kgc_bce_1n_t_blocks(n_ent);
  const double count = (double)B * (double)n_ent;
  bce_1n_t_kernel<<<(unsigned)blocks, kThreadsST, 0, as_stream(stream)>>>(pred_t, mask_t, (int)ceil_div(B, 32), n_ent, B, ldt, pos,
                                                                       add, (float)(1.0 / count), d_bias, loss_partial);
  KGC_LAUNCH_CHECK();
  bce_1n_finalize_kernel<<<1, kThreadsST, 0, as_stream(stream)>>>(loss_partial, blocks, 1.0 / count, loss);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_label_mask_t_build_rows(const int64_t* qid, int64_t B, const int64_t* ptr, const int32_t* idx,
                                           const int32_t* row_of, int64_t n_rows, uint32_t* mask_t, void* stream) {
  KGC_REQUIRE(B >= 0 && n_rows >= 0, "bad sizes");
  if (B == 0 || n_rows == 0) return 0;
  KGC_REQUIRE(qid && ptr && idx && row_of && mask_t, "null buffer");
  const int wb = (int)ceil_div(B, 32);
  KGC_CUDA_TRY(cudaMemsetAsync(mask_t, 0, (size_t)(n_rows * wb) * sizeof(uint32_t), as_stream(stream)));
  label_mask_t_rows_kernel<<<(unsigned)B, kThreadsST, 0, as_stream(stream)>>>(qid, ptr, idx, row_of, n_rows, wb, mask_t);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_bce_1n_bwd_logit_t_shard(float* pred_t, const uint32_t* mask_t, int64_t n_rows, int32_t B, int32_t ldt,
                                            float pos, float add, int64_t n_total, float* d_bias, double* loss_partial,
                                            double* loss_sum, void* stream) {
  KGC_REQUIRE(n_rows >= 0 && n_total > 0 && n_rows <= n_total && B > 0 && ldt >= B && ldt % 4 == 0,
              "bad sizes (0 <= n_rows <= n_total, ldt a multiple of 4)");
  KGC_REQUIRE(loss_partial && loss_sum, "null buffer");
  KGC_REQUIRE(n_rows == 0 || (pred_t && mask_t && d_bias), "null buffer");
  KGC_REQUIRE((reinterpret_cast<uintptr_t>(pred_t) & 15) == 0, "pred_t must be 16-byte aligned");
  const int64_t blocks = kgc_bce_1n_t_blocks(n_rows);
  const double count = (double)B * (double)n_total;                 // the unsharded call's divisor, formed the same way
  bce_1n_t_kernel<<<(unsigned)blocks, kThreadsST, 0, as_stream(stream)>>>(pred_t, mask_t, (int)ceil_div(B, 32), n_rows, B, ldt,
                                                                       pos, add, (float)(1.0 / count), d_bias, loss_partial);
  KGC_LAUNCH_CHECK();
  bce_1n_sum_kernel<<<1, kThreadsST, 0, as_stream(stream)>>>(loss_partial, blocks, loss_sum);
  KGC_LAUNCH_CHECK();
  return 0;
}
