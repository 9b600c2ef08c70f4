// K6s: sampled (1-vs-k) scoring fused with the BCE loss - the negative-sampled training objective (extension: the reference
// trains 1-N only).  Each query b scores C chosen candidates cand[b, 0..C): the first n_pos are its positives (label pos),
// the rest negatives (label add); an id outside [0, N) is an empty slot (no loss, no gradient).  The cost is B x C
// gathered rows, independent of N, so the batch can grow far beyond what the 1-N objective's [N, B] tiles allow.
//
// Forward (one pass): logit = <x[b], E[cand]> + bias[cand] in fp32 (warp_dot), p = sigmoid, then ATen's BCE as
// kgc_bce_1n_bwd_logit_t (bce.cuh) with the VALID-slot count as the mean's divisor: g = bce_logit_grad(p, y, 1 / count)
// (unit upstream gradient) and, while the candidate row is still in registers, d_x[b] += g * E[cand] in slot order.  A
// warp owns one query: the x row lives in registers, a candidate row is one coalesced request of 4 D bytes (800 at
// D = 200), and the rows of a batch of kRowsInFlight slots are all loaded before the first is consumed (the lesson of
// agg_kernel, DESIGN section 4).
//
// Table backward: d_E[n] = sum over the slots s with cand[s] = n of g[s] * (scale x[b(s)]) and d_bias[n] = scale sum g[s],
// dense [N, D] / [N] with zeros elsewhere (the encoder's backward takes a dense upstream).  Duplicate candidates are the
// normal case (across queries and within one), so instead of float atomics the (entity, slot) pairs are stable-sorted by
// entity (CUB radix sort, as K1) and one warp per distinct entity adds its slots in slot order: deterministic.
//
// kgc_sampled_adv_fwd is the self-adversarial forward (Sun et al. 2019): each query's negatives are weighted by a softmax
// of their own logits at a temperature, computed online in the same single pass (sampled_adv_fwd_kernel).  Its g is a
// logit gradient like any other, so the table backward above serves both.
#include <cmath>

#include <cub/device/device_radix_sort.cuh>

#include "bce.cuh"
#include "common.cuh"

namespace kgc {
namespace {

constexpr int kThreadsSS = 256;
constexpr int kWarpsSS = kThreadsSS / 32;
constexpr int kRowsInFlight = 8;          // candidate (or query) rows a warp loads before consuming the first
constexpr unsigned kFull = 0xFFFFFFFFu;

__device__ __forceinline__ bool slot_valid(int32_t e, int64_t n_ent) { return e >= 0 && e < n_ent; }

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

__device__ __forceinline__ void fma4(float s, const float4& a, float4& acc) {
  acc.x = fmaf(s, a.x, acc.x);
  acc.y = fmaf(s, a.y, acc.y);
  acc.z = fmaf(s, a.z, acc.z);
  acc.w = fmaf(s, a.w, acc.w);
}

// <x, r> in fp32: a per-lane FMA chain over the lane's float4 columns, then a fixed xor-shuffle tree (every lane ends
// with the same bits)
template <int NV>
__device__ __forceinline__ float warp_dot(const float4 (&xr)[NV], const float4 (&r)[NV]) {
  float s = 0.f;
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    s = fmaf(xr[v].x, r[v].x, s);
    s = fmaf(xr[v].y, r[v].y, s);
    s = fmaf(xr[v].z, r[v].z, s);
    s = fmaf(xr[v].w, r[v].w, s);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(kFull, s, o);
  return s;
}

// number of valid slots (integer sum: the order of the atomics does not matter)
__global__ void __launch_bounds__(kThreadsSS)
count_valid_kernel(const int32_t* __restrict__ cand, int64_t n_slots, int64_t n_ent, int32_t* __restrict__ count) {
  int c = 0;
  for (int64_t i = (int64_t)blockIdx.x * kThreadsSS + threadIdx.x; i < n_slots; i += (int64_t)gridDim.x * kThreadsSS)
    c += slot_valid(cand[i], n_ent) ? 1 : 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(kFull, c, o);
  if ((threadIdx.x & 31) == 0 && c != 0) atomicAdd(count, c);
}

template <int NV>    // float4 columns per lane: D <= 128 * NV
__global__ void __launch_bounds__(kThreadsSS)
sampled_bce_fwd_kernel(const float* __restrict__ x, int64_t B, int D4, const float* __restrict__ ent, int64_t ld_ent,
                       int64_t n_ent, const float* __restrict__ bias, const int32_t* __restrict__ cand, int C, int n_pos,
                       float pos, float add, const int32_t* __restrict__ count, float* __restrict__ g_out,
                       float* __restrict__ d_x, double* __restrict__ loss_partial) {
  __shared__ double warp_loss[kWarpsSS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t b = (int64_t)blockIdx.x * kWarpsSS + warp;
  const int n_valid = *count;
  const float inv_count = n_valid > 0 ? (float)(1.0 / (double)n_valid) : 0.f;
  double loss = 0.0;                                             // the same value in every lane
  if (b < B) {
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 xr[NV], acc[NV];
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const int c4 = lane + 32 * v;
      xr[v] = c4 < D4 ? ldg4(x + b * 4 * D4 + 4 * c4) : zero;
      acc[v] = zero;
    }
    const int32_t* cb = cand + b * C;
    for (int c0 = 0; c0 < C; c0 += kRowsInFlight) {
      const int32_t mine = (lane < kRowsInFlight && c0 + lane < C) ? cb[c0 + lane] : -1;
      int32_t e[kRowsInFlight];
      float4 r[kRowsInFlight][NV];
      float bi[kRowsInFlight];
#pragma unroll
      for (int u = 0; u < kRowsInFlight; ++u) {
        e[u] = __shfl_sync(kFull, mine, u);
        if (!slot_valid(e[u], n_ent)) e[u] = -1;
      }
#pragma unroll
      for (int u = 0; u < kRowsInFlight; ++u) {                  // every row load of the batch before any is consumed
#pragma unroll
        for (int v = 0; v < NV; ++v) {
          const int c4 = lane + 32 * v;
          r[u][v] = (e[u] >= 0 && c4 < D4) ? ldg4(ent + (int64_t)e[u] * ld_ent + 4 * c4) : zero;
        }
        bi[u] = e[u] >= 0 ? __ldg(bias + e[u]) : 0.f;
      }
      float g_mine = 0.f;
#pragma unroll
      for (int u = 0; u < kRowsInFlight; ++u) {
        const float s = warp_dot(xr, r[u]);
        float g = 0.f;
        if (e[u] >= 0) {
          const float z = s + bi[u];
          const float p = 1.f / (1.f + expf(-z));                 // the 1-N scorer's epilogue sigmoid
          const float y = c0 + u < n_pos ? pos : add;
          loss += (double)bce_loss_term(p, y);
          g = bce_logit_grad(p, y, inv_count);
#pragma unroll
          for (int v = 0; v < NV; ++v) fma4(g, r[u][v], acc[v]);
        }
        if (lane == u) g_mine = g;
      }
      if (lane < kRowsInFlight && c0 + lane < C) g_out[b * C + c0 + lane] = g_mine;   // 0 on empty slots
    }
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const int c4 = lane + 32 * v;
      if (c4 < D4) *reinterpret_cast<float4*>(d_x + b * 4 * D4 + 4 * c4) = acc[v];
    }
  }
  const double s = cta_sum(loss, warp_loss, lane, warp);
  if (threadIdx.x == 0) loss_partial[blockIdx.x] = s;
}

// mean over the valid slots: one CTA adds the per-CTA partials in a fixed order (0 when no slot is valid)
__global__ void __launch_bounds__(kThreadsSS)
sampled_bce_finalize_kernel(const double* __restrict__ partial, int64_t n_partial, const int32_t* __restrict__ count,
                            float* __restrict__ loss) {
  __shared__ double sh[kThreadsSS];
  const double s = cta_sum_partials(partial, n_partial, sh);
  if (threadIdx.x == 0) loss[0] = *count > 0 ? (float)(s / (double)*count) : 0.f;
}

// Self-adversarial variant (RotatE's negative weighting).  Q+ / Q- = the queries with at least one valid positive /
// negative slot (integer sums: the order of the atomics does not matter).  One warp per query, grid-stride.
__global__ void __launch_bounds__(kThreadsSS)
count_adv_kernel(const int32_t* __restrict__ cand, int64_t B, int C, int n_pos, int64_t n_ent, int32_t* __restrict__ counts) {
  const int lane = threadIdx.x & 31;
  int qp = 0, qn = 0;
  for (int64_t b = ((int64_t)blockIdx.x * kThreadsSS + threadIdx.x) >> 5; b < B; b += ((int64_t)gridDim.x * kThreadsSS) >> 5) {
    bool hp = false, hn = false;
    for (int c = lane; c < C; c += 32)
      if (slot_valid(cand[b * C + c], n_ent)) (c < n_pos ? hp : hn) = true;
    qp += __any_sync(kFull, hp) ? 1 : 0;
    qn += __any_sync(kFull, hn) ? 1 : 0;
  }
  if (lane == 0 && qp != 0) atomicAdd(counts, qp);
  if (lane == 0 && qn != 0) atomicAdd(counts + 1, qn);
}

// The loss of sampled_bce_fwd_kernel with the negatives of query b weighted by w = softmax over its valid negative slots
// of (alpha z) (constants: no gradient through them), the two halves averaged over the queries that have them:
//   L = 1/2 (1/Q+) sum_b (1/|P_b|) sum_{P_b} l(z, pos) + 1/2 (1/Q-) sum_b sum_{Q_b} w l(z, add)
// Same row traffic as sampled_bce_fwd_kernel (every candidate row read once, kRowsInFlight in flight).  The softmax is
// taken online: a warp-uniform running max m of alpha z, sum S of exp(alpha z - m) and negative d_x accumulator, the
// latter two rescaled when a batch raises m.  The main loop parks each slot's logit in g; once the query's last row is
// done one pass over its C slots turns the logits into the final coefficients and the loss terms (recomputed from the
// parked logit with the same formulas).  d_x = acc_pos / (2 Q+ |P_b|) + acc_neg / (2 Q- S).
// loss_partial: [gridDim.x] positive-half sums, then [gridDim.x] negative-half sums (per query already divided by
// |P_b| / S); sampled_adv_finalize_kernel divides by 2 Q+ / 2 Q-.
template <int NV>    // float4 columns per lane: D <= 128 * NV
__global__ void __launch_bounds__(kThreadsSS)
sampled_adv_fwd_kernel(const float* __restrict__ x, int64_t B, int D4, const float* __restrict__ ent, int64_t ld_ent,
                       int64_t n_ent, const float* __restrict__ bias, const int32_t* __restrict__ cand, int C, int n_pos,
                       float pos, float add, float alpha, const int32_t* __restrict__ counts, float* g_out,
                       float* __restrict__ d_x, double* __restrict__ loss_partial) {
  __shared__ double warp_loss[2][kWarpsSS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t b = (int64_t)blockIdx.x * kWarpsSS + warp;
  const int q_pos = counts[0], q_neg = counts[1];
  double loss_p = 0.0, loss_n = 0.0;                             // this query's two halves, the same value in every lane
  if (b < B) {
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 xr[NV], acc_p[NV], acc_n[NV];
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const int c4 = lane + 32 * v;
      xr[v] = c4 < D4 ? ldg4(x + b * 4 * D4 + 4 * c4) : zero;
      acc_p[v] = zero;
      acc_n[v] = zero;
    }
    const int32_t* cb = cand + b * C;
    float* gb = g_out + b * C;
    float m = -INFINITY, S = 0.f;                                // warp-uniform running max of alpha z and sum
    int n_p = 0;                                                 // |P_b|
    for (int c0 = 0; c0 < C; c0 += kRowsInFlight) {
      const int32_t mine = (lane < kRowsInFlight && c0 + lane < C) ? cb[c0 + lane] : -1;
      int32_t e[kRowsInFlight];
      float4 r[kRowsInFlight][NV];
      float bi[kRowsInFlight];
#pragma unroll
      for (int u = 0; u < kRowsInFlight; ++u) {
        e[u] = __shfl_sync(kFull, mine, u);
        if (!slot_valid(e[u], n_ent)) e[u] = -1;
      }
#pragma unroll
      for (int u = 0; u < kRowsInFlight; ++u) {                  // every row load of the batch before any is consumed
#pragma unroll
        for (int v = 0; v < NV; ++v) {
          const int c4 = lane + 32 * v;
          r[u][v] = (e[u] >= 0 && c4 < D4) ? ldg4(ent + (int64_t)e[u] * ld_ent + 4 * c4) : zero;
        }
        bi[u] = e[u] >= 0 ? __ldg(bias + e[u]) : 0.f;
      }
      float z[kRowsInFlight];
      float m_new = m;
#pragma unroll
      for (int u = 0; u < kRowsInFlight; ++u) {
        z[u] = warp_dot(xr, r[u]) + bi[u];
        if (e[u] >= 0 && c0 + u >= n_pos) m_new = fmaxf(m_new, alpha * z[u]);
      }
      if (m_new > m) {                                           // rescale what was summed under the old max
        const float sc = expf(m - m_new);
        S *= sc;
#pragma unroll
        for (int v = 0; v < NV; ++v) {
          acc_n[v].x *= sc;
          acc_n[v].y *= sc;
          acc_n[v].z *= sc;
          acc_n[v].w *= sc;
        }
        m = m_new;
      }
      float z_mine = 0.f;
#pragma unroll
      for (int u = 0; u < kRowsInFlight; ++u) {
        if (e[u] >= 0) {
          const float p = 1.f / (1.f + expf(-z[u]));
          if (c0 + u < n_pos) {
            ++n_p;
#pragma unroll
            for (int v = 0; v < NV; ++v) fma4(bce_logit_grad(p, pos, 1.f), r[u][v], acc_p[v]);
          } else {
            const float w = expf(alpha * z[u] - m);
            S += w;
#pragma unroll
            for (int v = 0; v < NV; ++v) fma4(bce_logit_grad(p, add, w), r[u][v], acc_n[v]);
          }
        }
        if (lane == u) z_mine = z[u];
      }
      if (lane < kRowsInFlight && c0 + lane < C) gb[c0 + lane] = z_mine;
    }
    __syncwarp();                                                // the parked logits are visible to every lane
    const float cp = n_p > 0 ? (float)(1.0 / (2.0 * (double)q_pos * (double)n_p)) : 0.f;
    const float cn = S > 0.f ? (float)(1.0 / (2.0 * (double)q_neg * (double)S)) : 0.f;
    double lp = 0.0, ln = 0.0;
    for (int c = lane; c < C; c += 32) {
      float gv = 0.f;                                            // 0 on empty slots
      if (slot_valid(cb[c], n_ent)) {
        const float zc = gb[c];
        const float p = 1.f / (1.f + expf(-zc));
        const float y = c < n_pos ? pos : add;
        const float term = bce_loss_term(p, y);
        if (c < n_pos) {
          lp += (double)term;
          gv = bce_logit_grad(p, y, cp);
        } else {
          const float w = expf(alpha * zc - m);
          ln += (double)w * (double)term;
          gv = bce_logit_grad(p, y, w * cn);
        }
      }
      gb[c] = gv;
    }
    lp = warp_sum(lp);
    ln = warp_sum(ln);
    loss_p = n_p > 0 ? lp / (double)n_p : 0.0;
    loss_n = S > 0.f ? ln / (double)S : 0.0;
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const int c4 = lane + 32 * v;
      if (c4 < D4) {
        const float4 o = make_float4(fmaf(cn, acc_n[v].x, cp * acc_p[v].x), fmaf(cn, acc_n[v].y, cp * acc_p[v].y),
                                     fmaf(cn, acc_n[v].z, cp * acc_p[v].z), fmaf(cn, acc_n[v].w, cp * acc_p[v].w));
        *reinterpret_cast<float4*>(d_x + b * 4 * D4 + 4 * c4) = o;
      }
    }
  }
  const double sp = cta_sum(loss_p, warp_loss[0], lane, warp);
  const double sn = cta_sum(loss_n, warp_loss[1], lane, warp);
  if (threadIdx.x == 0) {
    loss_partial[blockIdx.x] = sp;
    loss_partial[gridDim.x + blockIdx.x] = sn;
  }
}

// L = sum_pos / (2 Q+) + sum_neg / (2 Q-): each half's per-CTA partials added by one CTA in a fixed order (a half whose
// count is 0 adds 0)
__global__ void __launch_bounds__(kThreadsSS)
sampled_adv_finalize_kernel(const double* __restrict__ partial, int64_t n_partial, const int32_t* __restrict__ counts,
                            float* __restrict__ loss) {
  __shared__ double sh[2][kThreadsSS];
  const double sp = cta_sum_partials(partial, n_partial, sh[0]);
  const double sn = cta_sum_partials(partial + n_partial, n_partial, sh[1]);
  if (threadIdx.x == 0) {
    const double lp = counts[0] > 0 ? sp / (2.0 * (double)counts[0]) : 0.0;
    const double ln = counts[1] > 0 ? sn / (2.0 * (double)counts[1]) : 0.0;
    loss[0] = (float)(lp + ln);
  }
}

// sort keys: the entity, or N for an empty slot (sorts after every entity); values: the slot
__global__ void __launch_bounds__(kThreadsSS)
slot_keys_kernel(const int32_t* __restrict__ cand, int64_t n_slots, int64_t n_ent, int32_t* __restrict__ keys,
                 int32_t* __restrict__ slots) {
  const int64_t i = (int64_t)blockIdx.x * kThreadsSS + threadIdx.x;
  if (i >= n_slots) return;
  const int32_t e = cand[i];
  keys[i] = slot_valid(e, n_ent) ? e : (int32_t)n_ent;
  slots[i] = (int32_t)i;
}

// A warp looks at 32 sorted positions and takes every run of one entity that STARTS there (the run may extend past them),
// so each distinct entity is owned by exactly one warp.  The run's slots come in ascending slot order (stable sort) and
// are added in that order: d_E[n] = sum g[s] * (scale * x[b(s)]), d_bias[n] = scale * sum g[s].
template <int NV>
__global__ void __launch_bounds__(kThreadsSS)
table_grad_kernel(const int32_t* __restrict__ keys, const int32_t* __restrict__ slots, int64_t n_slots, int64_t n_ent,
                  const float* __restrict__ x, int D4, int C, const float* __restrict__ g, const float* __restrict__ scale,
                  float* __restrict__ d_ent, int64_t ld_d, float* __restrict__ d_bias) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t base = ((int64_t)blockIdx.x * kWarpsSS + warp) * 32;
  if (base >= n_slots) return;
  const int64_t i = base + lane;
  const int32_t key = i < n_slots ? keys[i] : (int32_t)n_ent;
  const int32_t prev = (i > 0 && i < n_slots) ? keys[i - 1] : -1;
  uint32_t heads = __ballot_sync(kFull, key < n_ent && key != prev);
  const float sc = *scale;
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  while (heads) {
    const int h = __ffs(heads) - 1;
    heads &= heads - 1;
    const int32_t n = __shfl_sync(kFull, key, h);
    float4 acc[NV];
#pragma unroll
    for (int v = 0; v < NV; ++v) acc[v] = zero;
    float bsum = 0.f;
    for (int64_t j0 = base + h;; j0 += 32) {
      const int64_t j = j0 + lane;
      const bool in = j < n_slots && keys[j] == n;
      const int n_in = __popc(__ballot_sync(kFull, in));       // the run covers lanes [0, n_in): keys are sorted
      const int32_t slot = in ? slots[j] : 0;
      const float gs = in ? g[slot] : 0.f;
      for (int u0 = 0; u0 < n_in; u0 += kRowsInFlight) {
        float4 xr[kRowsInFlight][NV];
        float gu[kRowsInFlight];
#pragma unroll
        for (int u = 0; u < kRowsInFlight; ++u) {              // every row load of the batch before any is consumed
          const int k = u0 + u;
          const int32_t sl = __shfl_sync(kFull, slot, k & 31);
          gu[u] = __shfl_sync(kFull, gs, k & 31);
          const int64_t b = sl / C;
#pragma unroll
          for (int v = 0; v < NV; ++v) {
            const int c4 = lane + 32 * v;
            xr[u][v] = (k < n_in && c4 < D4) ? ldg4(x + b * 4 * D4 + 4 * c4) : zero;
          }
        }
#pragma unroll
        for (int u = 0; u < kRowsInFlight; ++u) {
          if (u0 + u < n_in) {
            bsum += gu[u];
#pragma unroll
            for (int v = 0; v < NV; ++v) {
              const float4 xs = make_float4(sc * xr[u][v].x, sc * xr[u][v].y, sc * xr[u][v].z, sc * xr[u][v].w);
              fma4(gu[u], xs, acc[v]);
            }
          }
        }
      }
      if (n_in < 32) break;
    }
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const int c4 = lane + 32 * v;
      if (c4 < D4) *reinterpret_cast<float4*>(d_ent + (int64_t)n * ld_d + 4 * c4) = acc[v];
    }
    if (lane == 0) d_bias[n] = bsum * sc;
  }
}

size_t align_up(size_t v) { return (v + 255) / 256 * 256; }

int key_bits(int64_t n_ent) {        // bits that hold 0 .. n_ent (the empty-slot key)
  int bits = 1;
  while ((int64_t{1} << bits) <= n_ent) ++bits;
  return bits;
}

cudaError_t sort_temp_bytes(int64_t n_slots, int64_t n_ent, size_t* out) {
  return cub::DeviceRadixSort::SortPairs(nullptr, *out, (const int32_t*)nullptr, (int32_t*)nullptr,
                                         (const int32_t*)nullptr, (int32_t*)nullptr, (int)n_slots, 0, key_bits(n_ent));
}

bool shapes_ok(int64_t B, int32_t D, int32_t C, int64_t n_ent) {
  return B > 0 && C > 0 && D > 0 && D <= 256 && D % 4 == 0 && n_ent > 0 && n_ent < (int64_t{1} << 31) - 1 &&
         B * (int64_t)C < (int64_t{1} << 31);
}

// the requirements kgc_sampled_bce_fwd and kgc_sampled_adv_fwd share: the failed one's message, or nullptr
const char* check_fwd_args(const float* x, int64_t B, int32_t D, const float* ent, int64_t n_ent, int64_t ld_ent,
                           const float* bias, const int32_t* cand, int32_t C, int32_t n_pos, const float* g, const float* d_x,
                           const int32_t* counts, const double* loss_partial, const float* loss) {
  if (!shapes_ok(B, D, C, n_ent)) return "bad sizes (B, C > 0, B * C < 2^31, 0 < D <= 256, D % 4 == 0, 0 < N < 2^31 - 1)";
  if (n_pos < 0 || n_pos > C) return "n_pos must lie in [0, C]";
  if (ld_ent < D || ld_ent % 4 != 0) return "entity rows need ld_ent >= D and a 16-byte pitch";
  if (!(x && ent && bias && cand && g && d_x && counts && loss_partial && loss)) return "null buffer";
  if (((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(ent) | reinterpret_cast<uintptr_t>(d_x)) & 15) != 0)
    return "x, all_ent and d_x must be 16-byte aligned";
  return nullptr;
}

// the instantiation of a row kernel for D = 4 * D4: one float4 column per lane up to D = 128, two up to 256
template <typename Kernel>
Kernel for_width(int D4, Kernel nv1, Kernel nv2) { return D4 <= 32 ? nv1 : nv2; }

}  // namespace
}  // namespace kgc

using namespace kgc;

extern "C" int64_t kgc_sampled_bce_fwd_blocks(int64_t B) { return ceil_div(B > 0 ? B : 1, kWarpsSS); }

extern "C" int kgc_sampled_bce_fwd(const float* x, int64_t B, int32_t D, const float* ent, int64_t n_ent, int64_t ld_ent,
                                   const float* bias, const int32_t* cand, int32_t C, int32_t n_pos, float pos, float add,
                                   float* g, float* d_x, int32_t* count, double* loss_partial, float* loss, void* stream) {
  if (const char* err = check_fwd_args(x, B, D, ent, n_ent, ld_ent, bias, cand, C, n_pos, g, d_x, count, loss_partial, loss))
    return fail(__func__, err);
  cudaStream_t s = as_stream(stream);
  const int64_t n_slots = B * C;
  KGC_CUDA_TRY(cudaMemsetAsync(count, 0, sizeof(int32_t), s));
  const int64_t cblocks = ceil_div(n_slots, kThreadsSS) < 4 * kNumSMs ? ceil_div(n_slots, kThreadsSS) : 4 * kNumSMs;
  count_valid_kernel<<<(unsigned)cblocks, kThreadsSS, 0, s>>>(cand, n_slots, n_ent, count);
  KGC_LAUNCH_CHECK();
  const int64_t blocks = kgc_sampled_bce_fwd_blocks(B);
  const int D4 = D / 4;
  const auto fwd = for_width(D4, sampled_bce_fwd_kernel<1>, sampled_bce_fwd_kernel<2>);
  fwd<<<(unsigned)blocks, kThreadsSS, 0, s>>>(x, B, D4, ent, ld_ent, n_ent, bias, cand, C, n_pos, pos, add, count, g, d_x,
                                              loss_partial);
  KGC_LAUNCH_CHECK();
  sampled_bce_finalize_kernel<<<1, kThreadsSS, 0, s>>>(loss_partial, blocks, count, loss);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_sampled_adv_fwd(const float* x, int64_t B, int32_t D, const float* ent, int64_t n_ent, int64_t ld_ent,
                                   const float* bias, const int32_t* cand, int32_t C, int32_t n_pos, float pos, float add,
                                   float temperature, float* g, float* d_x, int32_t* counts, double* loss_partial, float* loss,
                                   void* stream) {
  if (const char* err = check_fwd_args(x, B, D, ent, n_ent, ld_ent, bias, cand, C, n_pos, g, d_x, counts, loss_partial, loss))
    return fail(__func__, err);
  KGC_REQUIRE(std::isfinite(temperature) && temperature >= 0.f, "the adversarial temperature must be finite and >= 0");
  cudaStream_t s = as_stream(stream);
  KGC_CUDA_TRY(cudaMemsetAsync(counts, 0, 2 * sizeof(int32_t), s));
  const int64_t blocks = kgc_sampled_bce_fwd_blocks(B);
  const int64_t cblocks = blocks < 4 * kNumSMs ? blocks : 4 * kNumSMs;
  count_adv_kernel<<<(unsigned)cblocks, kThreadsSS, 0, s>>>(cand, B, C, n_pos, n_ent, counts);
  KGC_LAUNCH_CHECK();
  const int D4 = D / 4;
  const auto fwd = for_width(D4, sampled_adv_fwd_kernel<1>, sampled_adv_fwd_kernel<2>);
  fwd<<<(unsigned)blocks, kThreadsSS, 0, s>>>(x, B, D4, ent, ld_ent, n_ent, bias, cand, C, n_pos, pos, add, temperature, counts,
                                              g, d_x, loss_partial);
  KGC_LAUNCH_CHECK();
  sampled_adv_finalize_kernel<<<1, kThreadsSS, 0, s>>>(loss_partial, blocks, counts, loss);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" size_t kgc_sampled_bce_bwd_table_workspace_bytes(int64_t n_slots, int64_t n_ent) {
  if (n_slots <= 0 || n_slots >= (int64_t{1} << 31) || n_ent <= 0 || n_ent >= (int64_t{1} << 31) - 1) return 0;
  size_t temp = 0;
  if (sort_temp_bytes(n_slots, n_ent, &temp) != cudaSuccess) return 0;
  return 4 * align_up((size_t)n_slots * sizeof(int32_t)) + align_up(temp);
}

extern "C" int kgc_sampled_bce_bwd_table(const float* x, int64_t B, int32_t D, const int32_t* cand, int32_t C, const float* g,
                                         const float* scale, int64_t n_ent, float* d_ent, int64_t ld_d, float* d_bias,
                                         void* workspace, size_t workspace_bytes, void* stream) {
  KGC_REQUIRE(shapes_ok(B, D, C, n_ent), "bad sizes (B, C > 0, B * C < 2^31, 0 < D <= 256, D % 4 == 0, 0 < N < 2^31 - 1)");
  KGC_REQUIRE(ld_d >= D && ld_d % 4 == 0, "d_ent rows need ld_d >= D and a 16-byte pitch");
  KGC_REQUIRE(x && cand && g && scale && d_ent && d_bias && workspace, "null buffer");
  KGC_REQUIRE(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(d_ent) | reinterpret_cast<uintptr_t>(workspace)) & 15) == 0,
              "x, d_ent and the workspace must be 16-byte aligned");
  const int64_t n_slots = B * C;
  const size_t need = kgc_sampled_bce_bwd_table_workspace_bytes(n_slots, n_ent);
  KGC_REQUIRE(need > 0 && workspace_bytes >= need, "workspace too small (kgc_sampled_bce_bwd_table_workspace_bytes)");
  cudaStream_t s = as_stream(stream);
  const size_t arr = align_up((size_t)n_slots * sizeof(int32_t));
  uint8_t* w = static_cast<uint8_t*>(workspace);
  int32_t* keys_in = reinterpret_cast<int32_t*>(w);
  int32_t* keys_out = reinterpret_cast<int32_t*>(w + arr);
  int32_t* slots_in = reinterpret_cast<int32_t*>(w + 2 * arr);
  int32_t* slots_out = reinterpret_cast<int32_t*>(w + 3 * arr);
  void* temp = w + 4 * arr;
  size_t temp_bytes = workspace_bytes - 4 * arr;
  // rows no slot touches stay zero
  KGC_CUDA_TRY(cudaMemset2DAsync(d_ent, (size_t)ld_d * sizeof(float), 0, (size_t)D * sizeof(float), (size_t)n_ent, s));
  KGC_CUDA_TRY(cudaMemsetAsync(d_bias, 0, (size_t)n_ent * sizeof(float), s));
  slot_keys_kernel<<<(unsigned)ceil_div(n_slots, kThreadsSS), kThreadsSS, 0, s>>>(cand, n_slots, n_ent, keys_in, slots_in);
  KGC_LAUNCH_CHECK();
  KGC_CUDA_TRY(cub::DeviceRadixSort::SortPairs(temp, temp_bytes, keys_in, keys_out, slots_in, slots_out, (int)n_slots, 0,
                                               key_bits(n_ent), s));
  const unsigned blocks = (unsigned)ceil_div(ceil_div(n_slots, 32), kWarpsSS);
  const int D4 = D / 4;
  const auto grad = for_width(D4, table_grad_kernel<1>, table_grad_kernel<2>);
  grad<<<blocks, kThreadsSS, 0, s>>>(keys_out, slots_out, n_slots, n_ent, x, D4, C, g, scale, d_ent, ld_d, d_bias);
  KGC_LAUNCH_CHECK();
  return 0;
}
