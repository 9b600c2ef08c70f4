// ATen's binary cross-entropy and the fixed-order loss reductions of the training objectives: the 1-N loss
// (score_train.cu) and the sampled 1-vs-k losses (score_sampled.cu) share one definition, so they stay bit-compatible.
#pragma once
#include "common.cuh"

namespace kgc {

// One element of ATen's BCE (log clamped at -100) at probability p and label y:
//   (y - 1) * max(log1p(-p), -100) - y * max(log(p), -100)
__device__ __forceinline__ float bce_loss_term(float p, float y) {
  const float lp = fmaxf(logf(p), -100.f), l1p = fmaxf(log1pf(-p), -100.f);
  return (y - 1.f) * l1p - y * lp;
}

// The logit gradient of c times that element: ATen's d_pred = (p - y) / max((1 - p) p, 1e-12), times c, times the
// sigmoid's p (1 - p), multiplied left to right.
__device__ __forceinline__ float bce_logit_grad(float p, float y, float c) {
  return (p - y) / fmaxf((1.f - p) * p, 1e-12f) * c * p * (1.f - p);
}

// The sum of v over the warp's 32 lanes in a fixed xor-shuffle tree: every lane ends with the same bits.
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
  return v;
}

// The CTA's sum of a warp-uniform v: lane 0 of each warp parks it in sh[warp] (shared memory, one double per warp),
// then thread 0 adds the warps in warp order.  The result is meaningful in thread 0 only.  lane and warp come from the
// kernel: a read of threadIdx.x in an inlined helper does not carry the kernel's __launch_bounds__ range, and the
// kernel's index arithmetic and registers change with it.
template <int kWarps>
__device__ __forceinline__ double cta_sum(double v, double (&sh)[kWarps], int lane, int warp) {
  if (lane == 0) sh[warp] = v;
  __syncthreads();
  double s = 0.0;
  if (lane == 0 && warp == 0)
    for (int w = 0; w < kWarps; ++w) s += sh[w];
  return s;
}

// The sum of partial[0, n) by one CTA of kThreads threads in a fixed order: thread t adds t, t + kThreads, ..., then a
// tree over sh (shared memory, one double per thread).  The result is meaningful in thread 0 only.
template <int kThreads>
__device__ __forceinline__ double cta_sum_partials(const double* __restrict__ partial, int64_t n, double (&sh)[kThreads]) {
  double s = 0.0;
  for (int64_t i = threadIdx.x; i < n; i += kThreads) s += partial[i];
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int o = kThreads / 2; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
    __syncthreads();
  }
  return sh[0];
}

}  // namespace kgc
