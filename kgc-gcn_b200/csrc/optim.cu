// K9: gradient-norm clipping + Adam in two passes over the parameters (the optimiser half of the reference's training step).
// Replaces main.py:68-71 - nn.utils.clip_grad_norm_(model.parameters(), clip_grad) followed by torch.optim.Adam.step()
// (main.py:217) - for fp32 parameters: 29.4 M of them at the WN18RR shape (edge embeddings 17.4 M, fc weight 7.8 M, entity
// embeddings 4.1 M).  torch runs four multi-tensor launches for the clip (norms, norm of norms, scale in place: reads the
// gradients twice and rewrites them) and two for the fused Adam: 340 us per step.  Here: pass 1 reads the gradients once
// (squared-norm partials, fp64, fixed order), a one-block kernel turns them into the clip coefficient, advances the step
// counter and forms the bias corrections, pass 2 applies coef * g inside the Adam update (the clipped gradient is never
// written back).  Everything the step needs lives in device memory (lr included), so a CUDA graph of the step stays valid
// when the host changes the learning rate.
//
// Arithmetic (torch.optim.Adam, amsgrad = False, maximize = False, L2 weight decay added to the gradient):
//   g' = coef * g + wd * p;  m = m + (1 - b1) (g' - m);  v = b2 v + (1 - b2) g'^2
//   p -= (lr / (1 - b1^t)) * m / (sqrt(v) / sqrt(1 - b2^t) + eps),   coef = min(1, max_norm / (||g||_2 + 1e-6))
#include "common.cuh"

namespace kgc {
namespace {

constexpr int kThreadsOpt = 256;
constexpr int kChunkOpt = 16384;       // elements per CTA work item (64 float4 per thread)

// hyper[0..5] = lr, beta1, beta2, eps, weight_decay, max_norm (<= 0: no clipping); state[0] = step (as double),
// state[1] = coef, state[2] = lr / (1 - b1^t), state[3] = 1 / sqrt(1 - b2^t), state[4] = total gradient norm
__global__ void __launch_bounds__(kThreadsOpt)
adam_prepare_kernel(const double* __restrict__ partials, int64_t n_partials, const float* __restrict__ hyper,
                    double* __restrict__ state) {
  __shared__ double sm[kThreadsOpt / 32];
  double d = 0.0;
  for (int64_t i = threadIdx.x; i < n_partials; i += kThreadsOpt) d += partials[i];     // fixed order per thread
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
  if (threadIdx.x % 32 == 0) sm[threadIdx.x / 32] = d;
  __syncthreads();
  if (threadIdx.x != 0) return;
  double s = 0.0;
  for (int w = 0; w < kThreadsOpt / 32; ++w) s += sm[w];
  const double norm = sqrt(s);
  const double max_norm = (double)hyper[5];
  double coef = 1.0;
  if (max_norm > 0.0) {
    coef = max_norm / (norm + 1e-6);
    if (coef > 1.0) coef = 1.0;
  }
  const double t = state[0] + 1.0;
  state[0] = t;
  state[1] = coef;
  state[2] = (double)hyper[0] / (1.0 - pow((double)hyper[1], t));
  state[3] = 1.0 / sqrt(1.0 - pow((double)hyper[2], t));
  state[4] = norm;
}

// The fp64 sum of the squares of g[0, n) in a fixed order (per-thread fp32, warp tree, warps in order): thread 0 returns it.
__device__ __forceinline__ double chunk_sqnorm(const float* g, int n, double (&sm)[kThreadsOpt / 32]) {
  float acc = 0.f;                                   // <= 64 squares per thread before the fp64 tree
  if ((reinterpret_cast<uintptr_t>(g) & 15) == 0) {
    const float4* g4 = reinterpret_cast<const float4*>(g);
    for (int i = threadIdx.x; i < n / 4; i += kThreadsOpt) {
      const float4 v = __ldg(g4 + i);
      acc += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
    }
    for (int i = (n / 4) * 4 + threadIdx.x; i < n; i += kThreadsOpt) acc += g[i] * g[i];
  } else {
    for (int i = threadIdx.x; i < n; i += kThreadsOpt) acc += g[i] * g[i];
  }
  double d = (double)acc;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
  if (threadIdx.x % 32 == 0) sm[threadIdx.x / 32] = d;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x == 0)
    for (int w = 0; w < kThreadsOpt / 32; ++w) s += sm[w];
  return s;
}

// work item i covers elements [items[i].y, items[i].y + items[i].z) of tensor items[i].x
__global__ void __launch_bounds__(kThreadsOpt)
grad_sqnorm_kernel(const kgc_opt_tensor_t* __restrict__ tensors, const int4* __restrict__ items, double* __restrict__ partials) {
  __shared__ double sm[kThreadsOpt / 32];
  const int4 it = __ldg(items + blockIdx.x);
  const double s = chunk_sqnorm(tensors[it.x].grad + (int64_t)it.y * kChunkOpt, it.z, sm);
  if (threadIdx.x == 0) partials[blockIdx.x] = s;
}

// the same, except that an item with items[i].w != 0 adds 0: a tensor another rank counts (sharded models, kgc_clip_adam_sqnorm)
__global__ void __launch_bounds__(kThreadsOpt)
grad_sqnorm_flagged_kernel(const kgc_opt_tensor_t* __restrict__ tensors, const int4* __restrict__ items,
                           double* __restrict__ partials) {
  __shared__ double sm[kThreadsOpt / 32];
  const int4 it = __ldg(items + blockIdx.x);
  if (it.w != 0) {
    if (threadIdx.x == 0) partials[blockIdx.x] = 0.0;
    return;
  }
  const double s = chunk_sqnorm(tensors[it.x].grad + (int64_t)it.y * kChunkOpt, it.z, sm);
  if (threadIdx.x == 0) partials[blockIdx.x] = s;
}

// sqnorm[0] = the partials added in adam_prepare_kernel's order: on one rank without flags, sqrt(sqnorm[0]) is the norm
// kgc_clip_adam_step computes, bit for bit
__global__ void __launch_bounds__(kThreadsOpt)
sqnorm_sum_kernel(const double* __restrict__ partials, int64_t n_partials, double* __restrict__ sqnorm) {
  __shared__ double sm[kThreadsOpt / 32];
  double d = 0.0;
  for (int64_t i = threadIdx.x; i < n_partials; i += kThreadsOpt) d += partials[i];     // fixed order per thread
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
  if (threadIdx.x % 32 == 0) sm[threadIdx.x / 32] = d;
  __syncthreads();
  if (threadIdx.x != 0) return;
  double s = 0.0;
  for (int w = 0; w < kThreadsOpt / 32; ++w) s += sm[w];
  sqnorm[0] = s;
}

__device__ __forceinline__ void adam1(float& p, float g, float& m, float& v, float coef, float wd, float b1c, float b2,
                                      float b2c, float step_size, float inv_bc2_sqrt, float eps) {
  float gg = g * coef;
  if (wd != 0.f) gg = fmaf(wd, p, gg);
  m = fmaf(b1c, gg - m, m);                        // lerp(m, g, 1 - beta1)
  v = fmaf(b2c * gg, gg, b2 * v);
  const float denom = sqrtf(v) * inv_bc2_sqrt + eps;
  p -= step_size * (m / denom);
}

__global__ void __launch_bounds__(kThreadsOpt)
adam_update_kernel(const kgc_opt_tensor_t* __restrict__ tensors, const int4* __restrict__ items, const float* __restrict__ hyper,
                   const double* __restrict__ state) {
  const int4 it = __ldg(items + blockIdx.x);
  const kgc_opt_tensor_t T = tensors[it.x];
  const int64_t off = (int64_t)it.y * kChunkOpt;
  const int n = it.z;
  const float b1 = hyper[1], b2 = hyper[2], eps = hyper[3], wd = hyper[4];
  const float coef = (float)state[1], step_size = (float)state[2], inv_bc2_sqrt = (float)state[3];
  const float b1c = 1.f - b1, b2c = 1.f - b2;
  float* p = T.param + off;
  const float* g = T.grad + off;
  float* m = T.exp_avg + off;
  float* v = T.exp_avg_sq + off;
  const bool vec = ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(m) |
                     reinterpret_cast<uintptr_t>(v)) & 15) == 0;
  if (vec) {
    float4* p4 = reinterpret_cast<float4*>(p);
    const float4* g4 = reinterpret_cast<const float4*>(g);
    float4* m4 = reinterpret_cast<float4*>(m);
    float4* v4 = reinterpret_cast<float4*>(v);
    for (int i = threadIdx.x; i < n / 4; i += kThreadsOpt) {
      float4 pp = p4[i], mm = m4[i], vv = v4[i];
      const float4 gg = ld_stream(g4 + i);
      adam1(pp.x, gg.x, mm.x, vv.x, coef, wd, b1c, b2, b2c, step_size, inv_bc2_sqrt, eps);
      adam1(pp.y, gg.y, mm.y, vv.y, coef, wd, b1c, b2, b2c, step_size, inv_bc2_sqrt, eps);
      adam1(pp.z, gg.z, mm.z, vv.z, coef, wd, b1c, b2, b2c, step_size, inv_bc2_sqrt, eps);
      adam1(pp.w, gg.w, mm.w, vv.w, coef, wd, b1c, b2, b2c, step_size, inv_bc2_sqrt, eps);
      p4[i] = pp; m4[i] = mm; v4[i] = vv;
    }
    for (int i = (n / 4) * 4 + threadIdx.x; i < n; i += kThreadsOpt)
      adam1(p[i], g[i], m[i], v[i], coef, wd, b1c, b2, b2c, step_size, inv_bc2_sqrt, eps);
  } else {
    for (int i = threadIdx.x; i < n; i += kThreadsOpt)
      adam1(p[i], g[i], m[i], v[i], coef, wd, b1c, b2, b2c, step_size, inv_bc2_sqrt, eps);
  }
}

}  // namespace
}  // namespace kgc

using namespace kgc;

extern "C" int32_t kgc_opt_chunk_elems(void) { return kChunkOpt; }

extern "C" int kgc_clip_adam_step(const kgc_opt_tensor_t* tensors, const int32_t* items, int64_t n_items,
                                  const float* hyper, double* state, double* partials, void* stream) {
  KGC_REQUIRE(tensors != nullptr && items != nullptr && hyper != nullptr && state != nullptr && partials != nullptr,
              "null argument");
  if (n_items == 0) return 0;
  KGC_REQUIRE(n_items < (1ll << 31), "too many work items");
  cudaStream_t st = as_stream(stream);
  const int4* it4 = reinterpret_cast<const int4*>(items);
  grad_sqnorm_kernel<<<(unsigned)n_items, kThreadsOpt, 0, st>>>(tensors, it4, partials);
  KGC_LAUNCH_CHECK();
  adam_prepare_kernel<<<1, kThreadsOpt, 0, st>>>(partials, n_items, hyper, state);
  KGC_LAUNCH_CHECK();
  adam_update_kernel<<<(unsigned)n_items, kThreadsOpt, 0, st>>>(tensors, it4, hyper, state);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_clip_adam_sqnorm(const kgc_opt_tensor_t* tensors, const int32_t* items, int64_t n_items, double* partials,
                                    double* sqnorm, void* stream) {
  KGC_REQUIRE(tensors != nullptr && items != nullptr && partials != nullptr && sqnorm != nullptr, "null argument");
  KGC_REQUIRE(n_items >= 0 && n_items < (1ll << 31), "bad number of work items");
  cudaStream_t st = as_stream(stream);
  if (n_items == 0) {
    KGC_CUDA_TRY(cudaMemsetAsync(sqnorm, 0, sizeof(double), st));
    return 0;
  }
  grad_sqnorm_flagged_kernel<<<(unsigned)n_items, kThreadsOpt, 0, st>>>(tensors, reinterpret_cast<const int4*>(items), partials);
  KGC_LAUNCH_CHECK();
  sqnorm_sum_kernel<<<1, kThreadsOpt, 0, st>>>(partials, n_items, sqnorm);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_clip_adam_apply(const kgc_opt_tensor_t* tensors, const int32_t* items, int64_t n_items, const float* hyper,
                                   double* state, const double* sqnorm, void* stream) {
  KGC_REQUIRE(tensors != nullptr && items != nullptr && hyper != nullptr && state != nullptr && sqnorm != nullptr,
              "null argument");
  if (n_items == 0) return 0;
  KGC_REQUIRE(n_items < (1ll << 31), "too many work items");
  cudaStream_t st = as_stream(stream);
  const int4* it4 = reinterpret_cast<const int4*>(items);
  adam_prepare_kernel<<<1, kThreadsOpt, 0, st>>>(sqnorm, 1, hyper, state);      // the norm of ONE partial: sqrt(*sqnorm)
  KGC_LAUNCH_CHECK();
  adam_update_kernel<<<(unsigned)n_items, kThreadsOpt, 0, st>>>(tensors, it4, hyper, state);
  KGC_LAUNCH_CHECK();
  return 0;
}
