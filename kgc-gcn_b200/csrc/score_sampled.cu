// K6s: sampled (1-vs-k) scoring fused with the training loss - the negative-sampled objective (extension: the reference
// trains 1-N only).  Each query b scores C chosen candidates cand[b, 0..C): the first n_pos are its positives, the rest
// negatives; an id outside [0, N) is an empty slot (no loss, no gradient).  The cost is B x C gathered rows, independent
// of N, so the batch can grow far beyond what the 1-N objective's [N, B] tiles allow.
//
// Forward (one pass, sampled_fwd_kernel): a warp owns one query, the x row lives in registers, a candidate row is one
// coalesced request of 4 D bytes (800 at D = 200), and the rows of a batch of kRowsInFlight slots are all loaded before
// the first is consumed (the lesson of agg_kernel, DESIGN section 4).  logit = <x[b], E[cand]> + bias[cand] in fp32
// (warp_dot).  What the loss does with a batch of logits and rows, and after the query's last row, is a policy type:
//   BceLoss  ATen's BCE (kgc_sampled_bce_fwd): p = sigmoid, labels pos / add, the valid-slot count as the mean's divisor,
//            g = bce_logit_grad(p, y, 1 / count) and d_x[b] += g * E[cand] in slot order while the row is in registers;
//   AdvLoss  self-adversarial BCE (kgc_sampled_adv_fwd, Sun et al. 2019): the negatives weighted by a softmax of their
//            own logits at a temperature, computed online;
//   CeLoss   softmax cross-entropy of each positive against its query's negatives (kgc_sampled_ce_fwd).
// The three entries run one launcher: zero the counts, count_kernel (what the loss divides by), the forward, and
// sampled_finalize_kernel (the per-CTA loss partials added in a fixed order).
//
// Table backward: d_E[n] = sum over the slots s with cand[s] = n of g[s] * (scale x[b(s)]) and d_bias[n] = scale sum g[s],
// dense [N, D] / [N] with zeros elsewhere (the encoder's backward takes a dense upstream).  Every loss's g is a logit
// gradient, so one backward serves all three.  Duplicate candidates are the normal case (across queries and within one),
// so instead of float atomics the (entity, slot) pairs are stable-sorted by entity (CUB radix sort, as K1) and one warp
// per distinct entity adds its slots in slot order: deterministic.
#include <cmath>
#include <type_traits>

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

// Online softmax: when a batch raises the warp-uniform running max m to m_new, rescale the sum S and the accumulator
// summed under the old max
template <int NV>
__device__ __forceinline__ void raise_max(float m_new, float& m, float& S, float4 (&acc)[NV]) {
  if (m_new > m) {
    const float sc = expf(m - m_new);
    S *= sc;
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      acc[v].x *= sc;
      acc[v].y *= sc;
      acc[v].z *= sc;
      acc[v].w *= sc;
    }
    m = m_new;
  }
}

// The forward's operands, the same for the three losses.  counts: what the loss divides by (count_kernel);
// loss_partial: Loss::kHalves x gridDim.x per-CTA sums.
struct SampledArgs {
  const float* x;             // [B, 4 * D4]
  int64_t B;
  int D4;
  const float* ent;           // [n_ent] rows of pitch ld_ent
  int64_t ld_ent;
  int64_t n_ent;
  const float* bias;          // [n_ent]
  const int32_t* cand;        // [B, C]
  int C;
  int n_pos;
  float pos, add;             // BceLoss, AdvLoss: the labels
  float alpha;                // AdvLoss: the temperature
  float eps;                  // CeLoss: the label smoothing
  int32_t* counts;
  float* g;                   // [B, C]
  float* d_x;                 // [B, 4 * D4]
  double* loss_partial;
};

// A loss policy supplies, for sampled_fwd_kernel and the launcher:
//   kHalves      the number of counts and of per-CTA loss sums (1, or 2 for the self-adversarial loss's two halves);
//   kMinBlocks   the CTAs an SM the forward is compiled for (__launch_bounds__), at NV = 1 and 2: without a bound
//                ptxas gives the NV = 2 loops 148 to 168 registers (one CTA an SM) and the NV = 1 BCE loop 108 (two);
//   tally        what count_kernel adds for a query with n_p valid positive and n_q valid negative slots;
//   State<NV>    the per-query state: batch() takes a batch's logits z and rows and leaves in z the values to park in
//                g; finish() runs after the query's last row and gives d_x[b] and the query's loss halves.

// Plain BCE: L = mean over the valid slots of ATen's BCE; counts[0] = the valid slots
struct BceLoss {
  static constexpr int kHalves = 1, kMinBlocks[2] = {3, 2};   // 80 and 128 registers, no spills
  __device__ static void tally(int n_p, int n_q, int (&t)[2]) { t[0] += n_p + n_q; }

  template <int NV>
  struct State {
    float4 acc[NV];
    float inv_count;
    double loss = 0.0;                                           // the same value in every lane

    __device__ explicit State(const SampledArgs& a) {
      const int n_valid = *a.counts;
      inv_count = n_valid > 0 ? (float)(1.0 / (double)n_valid) : 0.f;
#pragma unroll
      for (int v = 0; v < NV; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    }

    __device__ void batch(const SampledArgs& a, int c0, const int32_t (&e)[kRowsInFlight],
                          const float4 (&r)[kRowsInFlight][NV], float (&z)[kRowsInFlight]) {
#pragma unroll
      for (int u = 0; u < kRowsInFlight; ++u) {
        float g = 0.f;                                           // 0 on empty slots
        if (e[u] >= 0) {
          const float p = 1.f / (1.f + expf(-z[u]));              // the 1-N scorer's epilogue sigmoid
          const float y = c0 + u < a.n_pos ? a.pos : a.add;
          loss += (double)bce_loss_term(p, y);
          g = bce_logit_grad(p, y, inv_count);
#pragma unroll
          for (int v = 0; v < NV; ++v) fma4(g, r[u][v], acc[v]);
        }
        z[u] = g;
      }
    }

    __device__ void finish(const SampledArgs&, const int32_t*, float*, int, float4 (&o)[NV], double (&l)[kHalves]) {
#pragma unroll
      for (int v = 0; v < NV; ++v) o[v] = acc[v];
      l[0] = loss;
    }
  };
};

// Self-adversarial BCE (RotatE's negative weighting): the negatives of query b weighted by w = softmax over its valid
// negative slots of (alpha z) (constants: no gradient through them), the two halves averaged over the queries that have
// them:
//   L = 1/2 (1/Q+) sum_b (1/|P_b|) sum_{P_b} l(z, pos) + 1/2 (1/Q-) sum_b sum_{Q_b} w l(z, add)
// counts = Q+, Q- (the queries with at least one valid positive / negative slot).  The softmax is taken online: a
// warp-uniform running max m of alpha z, sum S of exp(alpha z - m) and negative d_x accumulator.  The logits are parked
// in g; after the query's last row one pass over its C slots turns them into the final coefficients and the loss terms
// (recomputed from the parked logit with the same formulas).  d_x = acc_pos / (2 Q+ |P_b|) + acc_neg / (2 Q- S).  The
// loss halves are per query already divided by |P_b| / S; sampled_finalize_kernel divides by 2 Q+ / 2 Q-.
struct AdvLoss {
  static constexpr int kHalves = 2, kMinBlocks[2] = {2, 2};
  __device__ static void tally(int n_p, int n_q, int (&t)[2]) {
    t[0] += n_p > 0 ? 1 : 0;
    t[1] += n_q > 0 ? 1 : 0;
  }

  template <int NV>
  struct State {
    float4 acc_p[NV], acc_n[NV];
    float m = -INFINITY, S = 0.f;                                // warp-uniform running max of alpha z and sum
    int n_p = 0;                                                 // |P_b|

    __device__ explicit State(const SampledArgs&) {
#pragma unroll
      for (int v = 0; v < NV; ++v) acc_p[v] = acc_n[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    }

    __device__ void batch(const SampledArgs& a, int c0, const int32_t (&e)[kRowsInFlight],
                          const float4 (&r)[kRowsInFlight][NV], float (&z)[kRowsInFlight]) {
      float m_new = m;
#pragma unroll
      for (int u = 0; u < kRowsInFlight; ++u)
        if (e[u] >= 0 && c0 + u >= a.n_pos) m_new = fmaxf(m_new, a.alpha * z[u]);
      raise_max(m_new, m, S, acc_n);
#pragma unroll
      for (int u = 0; u < kRowsInFlight; ++u) {
        if (e[u] >= 0) {
          const float p = 1.f / (1.f + expf(-z[u]));
          if (c0 + u < a.n_pos) {
            ++n_p;
#pragma unroll
            for (int v = 0; v < NV; ++v) fma4(bce_logit_grad(p, a.pos, 1.f), r[u][v], acc_p[v]);
          } else {
            const float w = expf(a.alpha * z[u] - m);
            S += w;
#pragma unroll
            for (int v = 0; v < NV; ++v) fma4(bce_logit_grad(p, a.add, w), r[u][v], acc_n[v]);
          }
        }
      }
    }

    __device__ void finish(const SampledArgs& a, const int32_t* cb, float* gb, int lane, float4 (&o)[NV],
                           double (&l)[kHalves]) {
      __syncwarp();                                              // the parked logits are visible to every lane
      const int q_pos = a.counts[0], q_neg = a.counts[1];
      const float cp = n_p > 0 ? (float)(1.0 / (2.0 * (double)q_pos * (double)n_p)) : 0.f;
      const float cn = S > 0.f ? (float)(1.0 / (2.0 * (double)q_neg * (double)S)) : 0.f;
      double lp = 0.0, ln = 0.0;
      for (int c = lane; c < a.C; c += 32) {
        float gv = 0.f;                                          // 0 on empty slots
        if (slot_valid(cb[c], a.n_ent)) {
          const float zc = gb[c];
          const float p = 1.f / (1.f + expf(-zc));
          const float y = c < a.n_pos ? a.pos : a.add;
          const float term = bce_loss_term(p, y);
          if (c < a.n_pos) {
            lp += (double)term;
            gv = bce_logit_grad(p, y, cp);
          } else {
            const float w = expf(a.alpha * zc - m);
            ln += (double)w * (double)term;
            gv = bce_logit_grad(p, y, w * cn);
          }
        }
        gb[c] = gv;
      }
      lp = warp_sum(lp);
      ln = warp_sum(ln);
      l[0] = n_p > 0 ? lp / (double)n_p : 0.0;
      l[1] = S > 0.f ? ln / (double)S : 0.0;
#pragma unroll
      for (int v = 0; v < NV; ++v)
        o[v] = make_float4(fmaf(cn, acc_n[v].x, cp * acc_p[v].x), fmaf(cn, acc_n[v].y, cp * acc_p[v].y),
                           fmaf(cn, acc_n[v].z, cp * acc_p[v].z), fmaf(cn, acc_n[v].w, cp * acc_p[v].w));
    }
  };
};

// Softmax cross-entropy: each valid positive slot p of query b against the valid negative slots Q_b of that query,
// K_b = 1 + |Q_b| classes (other positives are not in p's denominator):
//   l_p = (1 - eps) (LSE_p - z_p) + eps (LSE_p - (z_p + sum_{Q_b} z_q) / K_b),  LSE_p = log(e^{z_p} + sum_{Q_b} e^{z_q})
// and L = (1 / P) sum l_p, counts[0] = P the valid positive slots.  Online over the negatives: a warp-uniform running
// max m over their logits, S = sum e^{z_q - m} and acc_w = sum e^{z_q - m} E[q]; with eps > 0 also the plain sum
// acc_1 = sum E[q].  The logits are parked in g.  After the query's last row a pass over its negative slots gives |Q_b|
// and Z = sum z_q from the parked logits, and one over its positive slots gives, from the final S, the negatives'
// softmax mass under p, 1 - softmax_p(p), the loss term and r_p = softmax_p(q) e^{m - z_q} (the same for every q), all
// against max(m, z_p) so that no exponent is positive; then
//   g_p = (eps |Q_b| / K_b - (1 - softmax_p(p))) / P,   g_q = (e^{z_q - m} R - |P_b| eps / K_b) / P,  R = sum_{P_b} r_p
// and d_x = (R acc_w - |P_b| eps / K_b acc_1) / P + sum_{P_b} g_p E[p]: the positive rows (n_pos of the C) are read a
// second time.  A positive without a valid negative has softmax_p(p) = 1 and |Q_b| = 0, so 0 loss and 0 gradient; a
// query without a valid positive has R = |P_b| = 0.  (Two CTAs an SM at NV = 1 too: in the 80 registers of three ptxas
// spills a row offset.)
struct CeLoss {
  static constexpr int kHalves = 1, kMinBlocks[2] = {2, 2};
  __device__ static void tally(int n_p, int, int (&t)[2]) { t[0] += n_p; }

  template <int NV>
  struct State {
    float4 acc_w[NV], acc_1[NV];
    float m = -INFINITY, S = 0.f;                                // warp-uniform

    __device__ explicit State(const SampledArgs&) {
#pragma unroll
      for (int v = 0; v < NV; ++v) acc_w[v] = acc_1[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    }

    __device__ void batch(const SampledArgs& a, int c0, const int32_t (&e)[kRowsInFlight],
                          const float4 (&r)[kRowsInFlight][NV], float (&z)[kRowsInFlight]) {
      float m_new = m;
#pragma unroll
      for (int u = 0; u < kRowsInFlight; ++u)
        if (e[u] >= 0 && c0 + u >= a.n_pos) m_new = fmaxf(m_new, z[u]);
      raise_max(m_new, m, S, acc_w);
#pragma unroll
      for (int u = 0; u < kRowsInFlight; ++u) {
        if (e[u] >= 0 && c0 + u >= a.n_pos) {
          const float w = expf(z[u] - m);
          S += w;
#pragma unroll
          for (int v = 0; v < NV; ++v) fma4(w, r[u][v], acc_w[v]);
          if (a.eps > 0.f) {
#pragma unroll
            for (int v = 0; v < NV; ++v) fma4(1.f, r[u][v], acc_1[v]);
          }
        }
      }
    }

    __device__ void finish(const SampledArgs& a, const int32_t* cb, float* gb, int lane, float4 (&o)[NV],
                           double (&l)[kHalves]) {
      __syncwarp();                                              // the parked logits are visible to every lane
      const float eps = a.eps;
      int n_q = 0;                                               // |Q_b| and the sum Z of its logits, from the parked ones
      double Z = 0.0;
      for (int c = a.n_pos + lane; c < a.C; c += 32) {
        if (slot_valid(cb[c], a.n_ent)) {
          ++n_q;
          Z += (double)gb[c];
        }
      }
      n_q = __reduce_add_sync(kFull, n_q);
      Z = warp_sum(Z);
      const int n_valid = *a.counts;                             // read here: one register less across the row loop
      const float inv_p = n_valid > 0 ? (float)(1.0 / (double)n_valid) : 0.f;
      const float inv_k = 1.f / (float)(1 + n_q);
      const float eps_pos = eps * (float)n_q * inv_k;            // eps (1 - 1 / K_b)
      float R = 0.f;
      double lsum = 0.0;
      int n_p = 0;                                               // |P_b|
      for (int c = lane; c < a.n_pos; c += 32) {
        float gv = 0.f;                                          // 0 on empty slots
        if (slot_valid(cb[c], a.n_ent)) {
          const float zp = gb[c];
          float q_mass, rp, lse_z;                               // 1 - softmax_p(p), r_p, LSE_p - z_p
          if (zp >= m) {                                         // also every positive of a query without negatives
            const float em = expf(m - zp);
            const float t = S * em;
            q_mass = t / (1.f + t);
            rp = em / (1.f + t);
            lse_z = log1pf(t);
          } else {
            const float ep = expf(zp - m);
            q_mass = S / (ep + S);
            rp = 1.f / (ep + S);
            lse_z = (m - zp) + logf(ep + S);
          }
          ++n_p;
          R += rp;
          lsum += (double)lse_z + (double)eps * ((double)n_q * (double)zp - Z) / (double)(1 + n_q);
          gv = (eps_pos - q_mass) * inv_p;
        }
        gb[c] = gv;
      }
      R = (float)warp_sum((double)R);
      l[0] = warp_sum(lsum);
      n_p = __reduce_add_sync(kFull, n_p);
      const float eps_neg = (float)n_p * eps * inv_k;            // |P_b| eps / K_b
      for (int c = a.n_pos + lane; c < a.C; c += 32) {
        float gv = 0.f;
        if (slot_valid(cb[c], a.n_ent)) gv = (expf(gb[c] - m) * R - eps_neg) * inv_p;
        gb[c] = gv;
      }
      const float cw = R * inv_p, c1 = -eps_neg * inv_p;
#pragma unroll
      for (int v = 0; v < NV; ++v)
        o[v] = make_float4(fmaf(cw, acc_w[v].x, c1 * acc_1[v].x), fmaf(cw, acc_w[v].y, c1 * acc_1[v].y),
                           fmaf(cw, acc_w[v].z, c1 * acc_1[v].z), fmaf(cw, acc_w[v].w, c1 * acc_1[v].w));
      __syncwarp();                                              // the positives' final g is visible to every lane
      for (int c = 0; c < a.n_pos; ++c) {                        // the positive rows again, in slot order
        const int32_t ep = cb[c];
        if (!slot_valid(ep, a.n_ent)) continue;
        const float gp = gb[c];
#pragma unroll
        for (int v = 0; v < NV; ++v) {
          const int c4 = lane + 32 * v;
          if (c4 < a.D4) fma4(gp, ldg4(a.ent + (int64_t)ep * a.ld_ent + 4 * c4), o[v]);
        }
      }
    }
  };
};

// |P_b| and |Q_b|, query b's valid positive and negative slots (one warp per query, grid-stride), added into the counts
// the loss divides by (integer sums: the order of the atomics does not matter)
template <class Loss>
__global__ void __launch_bounds__(kThreadsSS)
count_kernel(const int32_t* __restrict__ cand, int64_t B, int C, int n_pos, int64_t n_ent, int32_t* __restrict__ counts) {
  const int lane = threadIdx.x & 31;
  int t[2] = {0, 0};
  for (int64_t b = ((int64_t)blockIdx.x * kThreadsSS + threadIdx.x) >> 5; b < B; b += ((int64_t)gridDim.x * kThreadsSS) >> 5) {
    int n_p = 0, n_q = 0;
    for (int c = lane; c < C; c += 32)
      if (slot_valid(cand[b * C + c], n_ent)) ++(c < n_pos ? n_p : n_q);
    Loss::tally(__reduce_add_sync(kFull, n_p), __reduce_add_sync(kFull, n_q), t);
  }
#pragma unroll
  for (int h = 0; h < Loss::kHalves; ++h)
    if (lane == 0 && t[h] != 0) atomicAdd(counts + h, t[h]);
}

// One warp per query b: the x row, the candidate loop (a batch of kRowsInFlight ids, their rows and biases loaded before
// any is consumed, the logits, the Loss's batch step, the values it parks stored to g), the Loss's finish, d_x[b], and
// the CTA's loss partials (Loss::kHalves sums, each in warp order).
template <class Loss, int NV>    // float4 columns per lane: D <= 128 * NV
__global__ void __launch_bounds__(kThreadsSS, Loss::kMinBlocks[NV - 1])
sampled_fwd_kernel(const SampledArgs a) {
  constexpr int H = Loss::kHalves;
  __shared__ double warp_loss[H][kWarpsSS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t b = (int64_t)blockIdx.x * kWarpsSS + warp;
  double loss[H] = {};                                           // this query's loss halves, the same value in every lane
  if (b < a.B) {
    const int D4 = a.D4;
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 xr[NV];
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const int c4 = lane + 32 * v;
      xr[v] = c4 < D4 ? ldg4(a.x + b * 4 * D4 + 4 * c4) : zero;
    }
    typename Loss::template State<NV> st(a);
    const int32_t* cb = a.cand + b * a.C;
    float* gb = a.g + b * a.C;
    for (int c0 = 0; c0 < a.C; c0 += kRowsInFlight) {
      const int32_t mine = (lane < kRowsInFlight && c0 + lane < a.C) ? cb[c0 + lane] : -1;
      int32_t e[kRowsInFlight];
      float4 r[kRowsInFlight][NV];
      float bi[kRowsInFlight];
#pragma unroll
      for (int u = 0; u < kRowsInFlight; ++u) {
        e[u] = __shfl_sync(kFull, mine, u);
        if (!slot_valid(e[u], a.n_ent)) e[u] = -1;
      }
#pragma unroll
      for (int u = 0; u < kRowsInFlight; ++u) {                  // every row load of the batch before any is consumed
#pragma unroll
        for (int v = 0; v < NV; ++v) {
          const int c4 = lane + 32 * v;
          r[u][v] = (e[u] >= 0 && c4 < D4) ? ldg4(a.ent + (int64_t)e[u] * a.ld_ent + 4 * c4) : zero;
        }
        bi[u] = e[u] >= 0 ? __ldg(a.bias + e[u]) : 0.f;
      }
      float z[kRowsInFlight];
#pragma unroll
      for (int u = 0; u < kRowsInFlight; ++u) z[u] = warp_dot(xr, r[u]) + bi[u];
      st.batch(a, c0, e, r, z);
      float park = 0.f;
#pragma unroll
      for (int u = 0; u < kRowsInFlight; ++u)
        if (lane == u) park = z[u];
      if (lane < kRowsInFlight && c0 + lane < a.C) gb[c0 + lane] = park;
    }
    float4 o[NV];
    st.finish(a, cb, gb, lane, o, loss);
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const int c4 = lane + 32 * v;
      if (c4 < D4) *reinterpret_cast<float4*>(a.d_x + b * 4 * D4 + 4 * c4) = o[v];
    }
  }
  double s[H];
#pragma unroll
  for (int h = 0; h < H; ++h) s[h] = cta_sum(loss[h], warp_loss[h], lane, warp);
  if (threadIdx.x == 0) {
#pragma unroll
    for (int h = 0; h < H; ++h) a.loss_partial[h * gridDim.x + blockIdx.x] = s[h];
  }
}

// The loss from the per-CTA partials, each half added by one CTA in a fixed order; a zero count gives 0.
//   one half: sum / counts[0];   two halves (self-adversarial): sum_pos / (2 Q+) + sum_neg / (2 Q-)
template <int H>
__global__ void __launch_bounds__(kThreadsSS)
sampled_finalize_kernel(const double* __restrict__ partial, int64_t n_partial, const int32_t* __restrict__ counts,
                        float* __restrict__ loss) {
  __shared__ double sh[H][kThreadsSS];
  double s[H];
#pragma unroll
  for (int h = 0; h < H; ++h) s[h] = cta_sum_partials(partial + h * n_partial, n_partial, sh[h]);
  if (threadIdx.x == 0) {
    if constexpr (H == 1) {
      loss[0] = counts[0] > 0 ? (float)(s[0] / (double)counts[0]) : 0.f;
    } else {
      const double lp = counts[0] > 0 ? s[0] / (2.0 * (double)counts[0]) : 0.0;
      const double ln = counts[1] > 0 ? s[1] / (2.0 * (double)counts[1]) : 0.0;
      loss[0] = (float)(lp + ln);
    }
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

// the requirements the three sampled forwards share: the failed one's message, or nullptr
const char* check_fwd_args(const SampledArgs& a, int32_t D, const float* loss) {
  if (!shapes_ok(a.B, D, a.C, a.n_ent)) return "bad sizes (B, C > 0, B * C < 2^31, 0 < D <= 256, D % 4 == 0, 0 < N < 2^31 - 1)";
  if (a.n_pos < 0 || a.n_pos > a.C) return "n_pos must lie in [0, C]";
  if (a.ld_ent < D || a.ld_ent % 4 != 0) return "entity rows need ld_ent >= D and a 16-byte pitch";
  if (!(a.x && a.ent && a.bias && a.cand && a.g && a.d_x && a.counts && a.loss_partial && loss)) return "null buffer";
  if (((reinterpret_cast<uintptr_t>(a.x) | reinterpret_cast<uintptr_t>(a.ent) | reinterpret_cast<uintptr_t>(a.d_x)) & 15) != 0)
    return "x, all_ent and d_x must be 16-byte aligned";
  return nullptr;
}

// the instantiation of a row kernel for D = 4 * D4: one float4 column per lane up to D = 128, two up to 256
template <typename Kernel>
Kernel for_width(int D4, Kernel nv1, Kernel nv2) { return D4 <= 32 ? nv1 : nv2; }

// the sampled forward of one loss: zero its counts, count them, one pass over the rows, the loss from the partials
template <class Loss>
cudaError_t launch_sampled_fwd(const SampledArgs& a, float* loss, cudaStream_t s) {
  cudaError_t err = cudaMemsetAsync(a.counts, 0, Loss::kHalves * sizeof(int32_t), s);
  if (err != cudaSuccess) return err;
  const int64_t blocks = kgc_sampled_bce_fwd_blocks(a.B);
  const int64_t cblocks = blocks < 4 * kNumSMs ? blocks : 4 * kNumSMs;
  count_kernel<Loss><<<(unsigned)cblocks, kThreadsSS, 0, s>>>(a.cand, a.B, a.C, a.n_pos, a.n_ent,
                                                              a.counts);
  if ((err = cudaGetLastError()) != cudaSuccess) return err;
  const auto fwd = for_width(a.D4, sampled_fwd_kernel<Loss, 1>, sampled_fwd_kernel<Loss, 2>);
  fwd<<<(unsigned)blocks, kThreadsSS, 0, s>>>(a);
  if ((err = cudaGetLastError()) != cudaSuccess) return err;
  sampled_finalize_kernel<Loss::kHalves><<<1, kThreadsSS, 0, s>>>(a.loss_partial, blocks, a.counts, loss);
  return cudaGetLastError();
}

// ---- Shared negatives: every query of the batch scores the same k rows E_S = ent[shared] ----------------------------
// The candidate layout is cand[b] = [pos_cand[b] | shared with query b's known objects set to -1], the loss is the
// per-query one above on that matrix.  The k x B logits of the shared part come from the tensor-core scorer
// (kgc_score_1n_logits_t, entity-major logitT[j, b]); the filter is a bit per (slot, query) in the same orientation; the
// n_pos positive rows of each query are gathered by a warp as in sampled_fwd_kernel.  A CTA of the loss pass owns 32
// queries (lane = query, so a row of the tile is one coalesced 128-byte piece and a mask word serves the whole warp)
// and its 16 warps share the k rows.

constexpr int kWarpsSh = 16;                      // warps of a shared loss CTA (32 queries: two each for the positives)
constexpr int kThreadsSh = 32 * kWarpsSh;
constexpr int kRowsSh = 8;                        // tile rows a warp loads before consuming the first

// The operands of the shared pass.  nq [B]: query b's valid unfiltered shared slots (shared_count_kernel);
// loss_partial: Loss::kHalves x gridDim.x sums; bias_partial [gridDim.x, k]: each CTA's sum of g over its 32 queries.
struct SharedArgs {
  float* logit_t;             // [k, ldt]: logits in, the logit gradient out
  int64_t ldt;
  const uint32_t* mask_t;     // [k, W]
  int64_t W;
  const int32_t* shared;      // [k]
  int k;
  const float* x;             // [B, 4 * D4]
  int64_t B;
  int D4;
  const float* ent;           // rows of pitch ld_ent
  int64_t ld_ent;
  int64_t n_ent;
  const float* bias;
  const int32_t* pos_cand;    // [B, n_pos]
  int n_pos;
  float pos, add, alpha, eps;
  float* g_pos;               // [B, n_pos]
  float* d_x;                 // [B, 4 * D4]: the positives' part
  int32_t* counts;
  int32_t* nq;
  double* loss_partial;
  float* bias_partial;
};

// is slot j of the shared tile a valid negative of lane `lane`'s query (b < B)
__device__ __forceinline__ bool shared_ok(const SharedArgs& a, int j, bool in_batch, int lane) {
  return in_batch && slot_valid(__ldg(a.shared + j), a.n_ent) &&
         ((__ldg(a.mask_t + (int64_t)j * a.W + blockIdx.x) >> lane) & 1u) == 0u;
}

// The filter bits: one warp per query b, its lanes over the query's known objects; each object is looked up in the
// shared ids sorted by id and every slot of its run gets bit (b & 31) of word (b >> 5).  Integer ORs only.
__global__ void __launch_bounds__(kThreadsSS)
shared_mask_kernel(const int32_t* __restrict__ ids, int k, const int64_t* __restrict__ qid, int64_t B,
                   const int64_t* __restrict__ ptr, const int32_t* __restrict__ idx, int64_t n_ent, const int32_t* __restrict__ slots,
                   uint32_t* __restrict__ mask_t, int64_t W) {
  const int lane = threadIdx.x & 31;
  const int64_t b = (int64_t)blockIdx.x * kWarpsSS + (threadIdx.x >> 5);
  if (b >= B) return;
  const int64_t q = qid[b];
  const uint32_t bit = 1u << (b & 31);
  for (int64_t i = ptr[q] + lane; i < ptr[q + 1]; i += 32) {
    const int32_t o = idx[i];
    if (!slot_valid(o, n_ent)) continue;
    int lo = 0, hi = k;                                          // the first position with ids[pos] >= o
    while (lo < hi) {
      const int mid = (lo + hi) >> 1;
      if (ids[mid] < o) lo = mid + 1; else hi = mid;
    }
    for (int j = lo; j < k && ids[j] == o; ++j) atomicOr(mask_t + (int64_t)slots[j] * W + (b >> 5), bit);
  }
}

// ent rows and biases of the shared ids (zeros for an id outside [0, n_ent)): E_S [k, D] contiguous, b_S [k]
__global__ void __launch_bounds__(kThreadsSS)
shared_rows_kernel(const float* __restrict__ ent, int64_t ld_ent, const float* __restrict__ bias, int64_t n_ent,
                   const int32_t* __restrict__ shared, int k, int D4, float* __restrict__ rows, float* __restrict__ row_bias) {
  const int64_t i = (int64_t)blockIdx.x * kThreadsSS + threadIdx.x;
  if (i >= (int64_t)k * D4) return;
  const int j = (int)(i / D4), c4 = (int)(i % D4);
  const int32_t e = shared[j];
  const bool ok = slot_valid(e, n_ent);
  *reinterpret_cast<float4*>(rows + 4 * i) = ok ? ldg4(ent + (int64_t)e * ld_ent + 4 * c4) : make_float4(0.f, 0.f, 0.f, 0.f);
  if (c4 == 0) row_bias[j] = ok ? bias[e] : 0.f;
}

// |P_b| and |Q_b| of the broadcast matrix: a CTA owns the 32 queries of one mask word column, its warps share the k
// rows (lane = query), the warps' counts are added in shared memory; nq[b] = |Q_b| for the pass, the Loss's tally into
// the counts (integer sums)
template <class Loss>
__global__ void __launch_bounds__(kThreadsSS)
shared_count_kernel(const SharedArgs a) {
  __shared__ int sh[kWarpsSS][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t b = (int64_t)blockIdx.x * 32 + lane;
  int n = 0;
  for (int j = warp; j < a.k; j += kWarpsSS) n += shared_ok(a, j, b < a.B, lane) ? 1 : 0;
  sh[warp][lane] = n;
  __syncthreads();
  if (warp != 0) return;
  int n_q = 0, n_p = 0;
  for (int w = 0; w < kWarpsSS; ++w) n_q += sh[w][lane];
  int t[2] = {0, 0};
  if (b < a.B) {
    for (int c = 0; c < a.n_pos; ++c) n_p += slot_valid(a.pos_cand[b * a.n_pos + c], a.n_ent) ? 1 : 0;
    a.nq[b] = n_q;
    Loss::tally(n_p, n_q, t);
  }
#pragma unroll
  for (int h = 0; h < Loss::kHalves; ++h) {
    const int s = __reduce_add_sync(kFull, t[h]);
    if (lane == 0 && s != 0) atomicAdd(a.counts + h, s);
  }
}

// The shared loss pass, one CTA per 32 queries b0 + lane:
//   A (AdvLoss, CeLoss)  per query the online max m and sum S of exp(v - m) over its valid negatives (v = alpha z / z),
//                        and for CeLoss the sum Z of their logits, each warp over its rows, the warps merged in order;
//   B                    warp w gathers the positive rows of queries b0 + w and b0 + w + 16: their logits, gradients g_pos, loss terms and
//                        d_x[b] = sum g_pos E[p] in slot order (CeLoss: also R = sum r_p, as CeLoss::State::finish);
//   C                    each warp over its rows again: the negatives' gradient (over the logit in place), loss terms,
//                        and the row's sum of g over the 32 queries into bias_partial.
// The per-slot arithmetic is that of the per-query policies above.
template <class Loss, int NV>
__global__ void __launch_bounds__(kThreadsSh, 1)
shared_loss_kernel(const SharedArgs a) {
  constexpr int H = Loss::kHalves;
  constexpr bool kAdv = std::is_same<Loss, AdvLoss>::value, kCe = std::is_same<Loss, CeLoss>::value;
  __shared__ float sh_m[kWarpsSh][32], sh_s[kWarpsSh][32];
  __shared__ double sh_z[kWarpsSh][32];
  __shared__ float q_m[32], q_s[32], q_c[32], q_r[32];          // per query: max, sum, negative coefficient, R
  __shared__ double warp_loss[H][kWarpsSh];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t b0 = (int64_t)blockIdx.x * 32, b = b0 + lane;
  const bool in_batch = b < a.B, in_tile = b < a.ldt;
  double loss[H] = {};
  if constexpr (kAdv || kCe) {
    float m = -INFINITY, S = 0.f;
    double Z = 0.0;
    for (int j0 = warp; j0 < a.k; j0 += kWarpsSh * kRowsSh) {
      float z[kRowsSh];
      bool ok[kRowsSh];
#pragma unroll
      for (int u = 0; u < kRowsSh; ++u) {                        // every load of the batch before any is consumed
        const int j = j0 + u * kWarpsSh;
        ok[u] = j < a.k && shared_ok(a, j, in_batch, lane);
        z[u] = ok[u] ? a.logit_t[(int64_t)j * a.ldt + b] : 0.f;
      }
#pragma unroll
      for (int u = 0; u < kRowsSh; ++u) {
        if (!ok[u]) continue;
        const float v = kAdv ? a.alpha * z[u] : z[u];
        if (v > m) {
          S = S * expf(m - v) + 1.f;
          m = v;
        } else {
          S += expf(v - m);
        }
        if (kCe) Z += (double)z[u];
      }
    }
    sh_m[warp][lane] = m;
    sh_s[warp][lane] = S;
    sh_z[warp][lane] = Z;
    __syncthreads();
    if (warp == 0) {
      float M = -INFINITY;
      for (int w = 0; w < kWarpsSh; ++w) M = fmaxf(M, sh_m[w][lane]);
      float St = 0.f;
      double Zt = 0.0;
      for (int w = 0; w < kWarpsSh; ++w) {
        if (sh_s[w][lane] > 0.f) St += sh_s[w][lane] * expf(sh_m[w][lane] - M);
        Zt += sh_z[w][lane];
      }
      q_m[lane] = M;
      q_s[lane] = St;
      sh_z[0][lane] = Zt;
    }
    __syncthreads();
  }
  for (int qw = warp; qw < 32; qw += kWarpsSh) {                 // B: the positives of query b0 + qw
    const int64_t bq = b0 + qw;
    if (bq < a.B) {
      const int D4 = a.D4;
      const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
      float4 acc[NV];
#pragma unroll
      for (int v = 0; v < NV; ++v) acc[v] = zero;
      const int32_t* pc = a.pos_cand + bq * a.n_pos;
      int n_p = 0;
      for (int c = lane; c < a.n_pos; c += 32) n_p += slot_valid(pc[c], a.n_ent) ? 1 : 0;
      n_p = __reduce_add_sync(kFull, n_p);
      const int n_q = a.nq[bq];
      // CeLoss's per-query constants (CeLoss::State::finish)
      const float inv_p = a.counts[0] > 0 ? (float)(1.0 / (double)a.counts[0]) : 0.f;
      float cp = 0.f;                                            // the positives' coefficient of BCE / AdvLoss
      if (kAdv) cp = n_p > 0 ? (float)(1.0 / (2.0 * (double)a.counts[0] * (double)n_p)) : 0.f;
      else if (!kCe) cp = inv_p;                                 // BceLoss: 1 / the valid slots
      float R = 0.f;
      double lsum = 0.0;
      for (int c = 0; c < a.n_pos; ++c) {
        const int32_t e = pc[c];
        float gv = 0.f;
        if (slot_valid(e, a.n_ent)) {
          float4 r[NV];
          float dot = 0.f;                                       // warp_dot with the x columns held one at a time
#pragma unroll
          for (int v = 0; v < NV; ++v) {
            const int c4 = lane + 32 * v;
            r[v] = c4 < D4 ? ldg4(a.ent + (int64_t)e * a.ld_ent + 4 * c4) : zero;
            const float4 xv = c4 < D4 ? ldg4(a.x + bq * 4 * D4 + 4 * c4) : zero;
            dot = fmaf(xv.x, r[v].x, dot);
            dot = fmaf(xv.y, r[v].y, dot);
            dot = fmaf(xv.z, r[v].z, dot);
            dot = fmaf(xv.w, r[v].w, dot);
          }
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(kFull, dot, o);
          const float zp = dot + __ldg(a.bias + e);
          if constexpr (kCe) {
            const float m = q_m[qw], S = q_s[qw];
            float q_mass, rp, lse_z;
            if (zp >= m) {
              const float em = expf(m - zp);
              const float t = S * em;
              q_mass = t / (1.f + t);
              rp = em / (1.f + t);
              lse_z = log1pf(t);
            } else {
              const float ep = expf(zp - m);
              q_mass = S / (ep + S);
              rp = 1.f / (ep + S);
              lse_z = (m - zp) + logf(ep + S);
            }
            R += rp;
            lsum += (double)lse_z + (double)a.eps * ((double)n_q * (double)zp - sh_z[0][qw]) / (double)(1 + n_q);
            gv = (a.eps * (float)n_q * (1.f / (float)(1 + n_q)) - q_mass) * inv_p;    // eps (1 - 1 / K_b) - ...
          } else {
            const float p = 1.f / (1.f + expf(-zp));
            lsum += (double)bce_loss_term(p, a.pos);
            gv = bce_logit_grad(p, a.pos, cp);
          }
#pragma unroll
          for (int v = 0; v < NV; ++v) fma4(gv, r[v], acc[v]);
        }
        if (lane == 0) a.g_pos[bq * a.n_pos + c] = gv;
      }
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        const int c4 = lane + 32 * v;
        if (c4 < D4) *reinterpret_cast<float4*>(a.d_x + bq * 4 * D4 + 4 * c4) = acc[v];
      }
      if (lane == 0) loss[0] += kAdv ? (n_p > 0 ? lsum / (double)n_p : 0.0) : lsum;
      if (lane == 0) {                                           // the negatives' coefficients of this query
        if (kAdv) {
          q_c[qw] = q_s[qw] > 0.f ? (float)(1.0 / (2.0 * (double)a.counts[1] * (double)q_s[qw])) : 0.f;
        } else if (kCe) {
          q_r[qw] = R * inv_p;
          q_c[qw] = (float)n_p * a.eps * (1.f / (float)(1 + n_q)) * inv_p;    // |P_b| eps / K_b / P
        } else {
          q_c[qw] = inv_p;
        }
      }
    }
  }
  __syncthreads();
  {                                                              // C: the negatives' gradient over the logit tile
    const float c_neg = in_batch ? q_c[lane] : 0.f;
    const float m = (kAdv || kCe) && in_batch ? q_m[lane] : 0.f;
    const float r_q = kCe && in_batch ? q_r[lane] : 0.f;
    double ln = 0.0;
    for (int j0 = warp; j0 < a.k; j0 += kWarpsSh * kRowsSh) {
      float z[kRowsSh];
      bool ok[kRowsSh];
#pragma unroll
      for (int u = 0; u < kRowsSh; ++u) {
        const int j = j0 + u * kWarpsSh;
        ok[u] = j < a.k && shared_ok(a, j, in_batch, lane);
        z[u] = ok[u] ? a.logit_t[(int64_t)j * a.ldt + b] : 0.f;
      }
#pragma unroll
      for (int u = 0; u < kRowsSh; ++u) {
        const int j = j0 + u * kWarpsSh;
        if (j >= a.k) break;
        float gv = 0.f;                                          // 0 on filtered and empty slots
        if (ok[u]) {
          if constexpr (kCe) {
            gv = expf(z[u] - m) * r_q - c_neg;
          } else {
            const float p = 1.f / (1.f + expf(-z[u]));
            const float term = bce_loss_term(p, a.add);
            if constexpr (kAdv) {
              const float w = expf(a.alpha * z[u] - m);
              ln += (double)w * (double)term;
              gv = bce_logit_grad(p, a.add, w * c_neg);
            } else {
              loss[0] += (double)term;
              gv = bce_logit_grad(p, a.add, c_neg);
            }
          }
        }
        if (in_tile) a.logit_t[(int64_t)j * a.ldt + b] = gv;
        const float gs = (float)warp_sum((double)gv);
        if (lane == 0) a.bias_partial[(int64_t)blockIdx.x * a.k + j] = gs;
      }
    }
    if constexpr (kAdv) loss[1] = in_batch && q_s[lane] > 0.f ? ln / (double)q_s[lane] : 0.0;
  }
  double s[H];
#pragma unroll
  for (int h = 0; h < H; ++h) s[h] = cta_sum(warp_sum(loss[h]), warp_loss[h], lane, warp);
  if (threadIdx.x == 0) {
#pragma unroll
    for (int h = 0; h < H; ++h) a.loss_partial[h * gridDim.x + blockIdx.x] = s[h];
  }
}

// d_bias_s[j] = sum over the CTAs of the pass of bias_partial[c, j], in CTA order
__global__ void __launch_bounds__(kThreadsSS)
shared_bias_kernel(const float* __restrict__ bias_partial, int64_t n_cta, int k, float* __restrict__ d_bias_s) {
  const int64_t j = (int64_t)blockIdx.x * kThreadsSS + threadIdx.x;
  if (j >= k) return;
  float s = 0.f;
  for (int64_t c = 0; c < n_cta; ++c) s += bias_partial[c * k + j];
  d_bias_s[j] = s;
}

// d_ent[n] += scale * sum over the shared slots j with shared[j] = n of d_rows[j], d_bias[n] likewise: a warp per 32
// sorted positions takes every run of one id that starts there and adds its slots in slot order
template <int NV>
__global__ void __launch_bounds__(kThreadsSS)
shared_table_kernel(const int32_t* __restrict__ ids, const int32_t* __restrict__ slots, int k, int64_t n_ent,
                    const float* __restrict__ d_rows, int64_t ld_rows, const float* __restrict__ d_row_bias, int D4,
                    const float* __restrict__ scale, float* __restrict__ d_ent, int64_t ld_d, float* __restrict__ d_bias) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t base = ((int64_t)blockIdx.x * kWarpsSS + warp) * 32;
  if (base >= k) return;
  const int64_t i = base + lane;
  const int32_t key = i < k ? ids[i] : (int32_t)n_ent;
  const int32_t prev = (i > 0 && i < k) ? ids[i - 1] : -1;
  uint32_t heads = __ballot_sync(kFull, slot_valid(key, n_ent) && key != prev);
  const float sc = *scale;
  while (heads) {
    const int h = __ffs(heads) - 1;
    heads &= heads - 1;
    const int32_t n = __shfl_sync(kFull, key, h);
    float4 acc[NV];
#pragma unroll
    for (int v = 0; v < NV; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
    float bsum = 0.f;
    for (int64_t j = base + h; j < k && ids[j] == n; ++j) {
      const int32_t sl = slots[j];
#pragma unroll
      for (int v = 0; v < NV; ++v) {
        const int c4 = lane + 32 * v;
        if (c4 < D4) {
          const float4 r = ldg4(d_rows + (int64_t)sl * ld_rows + 4 * c4);
          acc[v].x += r.x;
          acc[v].y += r.y;
          acc[v].z += r.z;
          acc[v].w += r.w;
        }
      }
      bsum += d_row_bias[sl];
    }
#pragma unroll
    for (int v = 0; v < NV; ++v) {
      const int c4 = lane + 32 * v;
      if (c4 < D4) {
        float4* o = reinterpret_cast<float4*>(d_ent + (int64_t)n * ld_d + 4 * c4);
        float4 t = *o;
        t.x = fmaf(sc, acc[v].x, t.x);
        t.y = fmaf(sc, acc[v].y, t.y);
        t.z = fmaf(sc, acc[v].z, t.z);
        t.w = fmaf(sc, acc[v].w, t.w);
        *o = t;
      }
    }
    if (lane == 0) d_bias[n] = fmaf(sc, bsum, d_bias[n]);
  }
}

// the shared loss of one policy: zero its counts, count them, the pass, the shared slots' d_bias, the loss
template <class Loss>
cudaError_t launch_shared_loss(const SharedArgs& a, float* d_bias_s, float* loss, cudaStream_t s) {
  cudaError_t err = cudaMemsetAsync(a.counts, 0, Loss::kHalves * sizeof(int32_t), s);
  if (err != cudaSuccess) return err;
  const int64_t blocks = kgc_shared_loss_blocks(a.B);
  shared_count_kernel<Loss><<<(unsigned)blocks, kThreadsSS, 0, s>>>(a);
  if ((err = cudaGetLastError()) != cudaSuccess) return err;
  const auto pass = for_width(a.D4, shared_loss_kernel<Loss, 1>, shared_loss_kernel<Loss, 2>);
  pass<<<(unsigned)blocks, kThreadsSh, 0, s>>>(a);
  if ((err = cudaGetLastError()) != cudaSuccess) return err;
  shared_bias_kernel<<<(unsigned)ceil_div(a.k, kThreadsSS), kThreadsSS, 0, s>>>(a.bias_partial, blocks, a.k, d_bias_s);
  if ((err = cudaGetLastError()) != cudaSuccess) return err;
  sampled_finalize_kernel<Loss::kHalves><<<1, kThreadsSS, 0, s>>>(a.loss_partial, blocks, a.counts, loss);
  return cudaGetLastError();
}

// workspace of the shared loss: counts (2), nq [B], loss partials (2 x blocks doubles), bias partials [blocks, k]
struct SharedWs {
  size_t counts, nq, loss_partial, bias_partial, total;
  SharedWs(int64_t B, int64_t k) {
    const int64_t blocks = ceil_div(B, 32);
    counts = 0;
    nq = align_up(2 * sizeof(int32_t));
    loss_partial = nq + align_up((size_t)B * sizeof(int32_t));
    bias_partial = loss_partial + align_up((size_t)2 * blocks * sizeof(double));
    total = bias_partial + align_up((size_t)blocks * k * sizeof(float));
  }
};

}  // namespace
}  // namespace kgc

using namespace kgc;

extern "C" int64_t kgc_sampled_bce_fwd_blocks(int64_t B) { return ceil_div(B > 0 ? B : 1, kWarpsSS); }

extern "C" int kgc_sampled_bce_fwd(const float* x, int64_t B, int32_t D, const float* ent, int64_t n_ent, int64_t ld_ent,
                                   const float* bias, const int32_t* cand, int32_t C, int32_t n_pos, float pos, float add,
                                   float* g, float* d_x, int32_t* count, double* loss_partial, float* loss, void* stream) {
  const SampledArgs a{x, B, D / 4, ent, ld_ent, n_ent, bias, cand, C, n_pos, pos, add, 0.f, 0.f, count, g, d_x, loss_partial};
  if (const char* err = check_fwd_args(a, D, loss)) return fail(__func__, err);
  KGC_CUDA_TRY(launch_sampled_fwd<BceLoss>(a, loss, as_stream(stream)));
  return 0;
}

extern "C" int kgc_sampled_adv_fwd(const float* x, int64_t B, int32_t D, const float* ent, int64_t n_ent, int64_t ld_ent,
                                   const float* bias, const int32_t* cand, int32_t C, int32_t n_pos, float pos, float add,
                                   float temperature, float* g, float* d_x, int32_t* counts, double* loss_partial, float* loss,
                                   void* stream) {
  const SampledArgs a{x, B, D / 4, ent, ld_ent, n_ent, bias, cand, C, n_pos, pos, add, temperature, 0.f, counts, g, d_x,
                      loss_partial};
  if (const char* err = check_fwd_args(a, D, loss)) return fail(__func__, err);
  KGC_REQUIRE(std::isfinite(temperature) && temperature >= 0.f, "the adversarial temperature must be finite and >= 0");
  KGC_CUDA_TRY(launch_sampled_fwd<AdvLoss>(a, loss, as_stream(stream)));
  return 0;
}

extern "C" int kgc_sampled_ce_fwd(const float* x, int64_t B, int32_t D, const float* ent, int64_t n_ent, int64_t ld_ent,
                                  const float* bias, const int32_t* cand, int32_t C, int32_t n_pos, float label_smoothing,
                                  float* g, float* d_x, int32_t* count, double* loss_partial, float* loss, void* stream) {
  const SampledArgs a{x, B, D / 4, ent, ld_ent, n_ent, bias, cand, C, n_pos, 0.f, 0.f, 0.f, label_smoothing, count, g, d_x,
                      loss_partial};
  if (const char* err = check_fwd_args(a, D, loss)) return fail(__func__, err);
  KGC_REQUIRE(label_smoothing >= 0.f && label_smoothing <= 1.f, "the label smoothing must be a number in [0, 1]");
  KGC_CUDA_TRY(launch_sampled_fwd<CeLoss>(a, loss, as_stream(stream)));
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

extern "C" size_t kgc_shared_mask_workspace_bytes(int32_t k, int64_t n_ent) {
  if (k <= 0 || n_ent <= 0 || n_ent >= (int64_t{1} << 31) - 1) return 0;
  size_t temp = 0;
  if (sort_temp_bytes(k, n_ent, &temp) != cudaSuccess) return 0;
  return 2 * align_up((size_t)k * sizeof(int32_t)) + align_up(temp);
}

extern "C" int kgc_shared_mask_build(const int32_t* shared, int32_t k, const int64_t* qid, int64_t B, const int64_t* ptr,
                                     const int32_t* idx, int64_t n_ent, uint32_t* mask_t, int32_t* sorted_ids,
                                     int32_t* sorted_slots, void* workspace, size_t workspace_bytes, void* stream) {
  KGC_REQUIRE(k > 0 && B > 0 && n_ent > 0 && n_ent < (int64_t{1} << 31) - 1, "bad sizes (k, B > 0, 0 < N < 2^31 - 1)");
  KGC_REQUIRE(shared && qid && ptr && idx && mask_t && sorted_ids && sorted_slots && workspace, "null buffer");
  const size_t need = kgc_shared_mask_workspace_bytes(k, n_ent);
  KGC_REQUIRE(need > 0 && workspace_bytes >= need, "workspace too small (kgc_shared_mask_workspace_bytes)");
  cudaStream_t s = as_stream(stream);
  const size_t arr = align_up((size_t)k * sizeof(int32_t));
  uint8_t* w = static_cast<uint8_t*>(workspace);
  int32_t* keys_in = reinterpret_cast<int32_t*>(w);
  int32_t* slots_in = reinterpret_cast<int32_t*>(w + arr);
  const int64_t W = ceil_div(B, 32);
  KGC_CUDA_TRY(cudaMemsetAsync(mask_t, 0, (size_t)k * W * sizeof(uint32_t), s));
  slot_keys_kernel<<<(unsigned)ceil_div(k, kThreadsSS), kThreadsSS, 0, s>>>(shared, k, n_ent, keys_in, slots_in);
  KGC_LAUNCH_CHECK();
  size_t temp_bytes = workspace_bytes - 2 * arr;
  KGC_CUDA_TRY(cub::DeviceRadixSort::SortPairs(w + 2 * arr, temp_bytes, keys_in, sorted_ids, slots_in, sorted_slots, (int)k,
                                               0, key_bits(n_ent), s));
  shared_mask_kernel<<<(unsigned)ceil_div(B, kWarpsSS), kThreadsSS, 0, s>>>(sorted_ids, k, qid, B, ptr, idx, n_ent,
                                                                            sorted_slots, mask_t, W);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int kgc_shared_rows(const float* ent, int64_t n_ent, int32_t D, int64_t ld_ent, const float* bias,
                               const int32_t* shared, int32_t k, float* rows, float* row_bias, void* stream) {
  KGC_REQUIRE(k > 0 && n_ent > 0 && D > 0 && D % 4 == 0 && ld_ent >= D && ld_ent % 4 == 0, "bad sizes");
  KGC_REQUIRE(ent && bias && shared && rows && row_bias, "null buffer");
  KGC_REQUIRE(((reinterpret_cast<uintptr_t>(ent) | reinterpret_cast<uintptr_t>(rows)) & 15) == 0,
              "all_ent and rows must be 16-byte aligned");
  const int64_t n4 = (int64_t)k * (D / 4);
  shared_rows_kernel<<<(unsigned)ceil_div(n4, kThreadsSS), kThreadsSS, 0, as_stream(stream)>>>(
      ent, ld_ent, bias, n_ent, shared, k, D / 4, rows, row_bias);
  KGC_LAUNCH_CHECK();
  return 0;
}

extern "C" int64_t kgc_shared_loss_blocks(int64_t B) { return ceil_div(B > 0 ? B : 1, 32); }

extern "C" size_t kgc_shared_loss_workspace_bytes(int64_t B, int32_t k) {
  if (B <= 0 || k <= 0) return 0;
  return SharedWs(B, k).total;
}

namespace kgc {
namespace {

template <class Loss>
int shared_loss_entry(const char* fn, float* logit_t, int64_t ldt, const uint32_t* mask_t, const int32_t* shared, int32_t k,
                      const float* x, int64_t B, int32_t D, const float* ent, int64_t n_ent, int64_t ld_ent,
                      const float* bias, const int32_t* pos_cand, int32_t n_pos, float pos, float add, float alpha,
                      float eps, float* g_pos, float* d_x, float* d_bias_s, float* loss, void* workspace,
                      size_t workspace_bytes, void* stream) {
  if (!(k > 0 && n_pos > 0 && B > 0 && B * (int64_t)k < (int64_t{1} << 31) && D > 0 && D <= 256 && D % 4 == 0 &&
        n_ent > 0 && n_ent < (int64_t{1} << 31) - 1 && ldt >= B && ld_ent >= D && ld_ent % 4 == 0))
    return fail(fn, "bad sizes (k, n_pos, B > 0, B * k < 2^31, 0 < D <= 256, D % 4 == 0, ldt >= B, ld_ent >= D, "
                    "ld_ent % 4 == 0)");
  if (!(logit_t && mask_t && shared && x && ent && bias && pos_cand && g_pos && d_x && d_bias_s && loss && workspace))
    return fail(fn, "null buffer");
  if (((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(ent) | reinterpret_cast<uintptr_t>(d_x)) & 15) != 0)
    return fail(fn, "x, all_ent and d_x must be 16-byte aligned");
  const SharedWs ws(B, k);
  if (workspace_bytes < ws.total) return fail(fn, "workspace too small (kgc_shared_loss_workspace_bytes)");
  uint8_t* w = static_cast<uint8_t*>(workspace);
  const SharedArgs a{logit_t, ldt, mask_t, ceil_div(B, 32), shared, k, x, B, D / 4, ent, ld_ent, n_ent, bias, pos_cand,
                     n_pos, pos, add, alpha, eps, g_pos, d_x,
                     reinterpret_cast<int32_t*>(w + ws.counts), reinterpret_cast<int32_t*>(w + ws.nq),
                     reinterpret_cast<double*>(w + ws.loss_partial), reinterpret_cast<float*>(w + ws.bias_partial)};
  const cudaError_t err = launch_shared_loss<Loss>(a, d_bias_s, loss, as_stream(stream));
  if (err != cudaSuccess) return fail(fn, std::string("launch -> ") + cudaGetErrorString(err));
  return 0;
}

}  // namespace
}  // namespace kgc

extern "C" int kgc_shared_bce_loss(float* logit_t, int64_t ldt, const uint32_t* mask_t, const int32_t* shared, int32_t k,
                                   const float* x, int64_t B, int32_t D, const float* ent, int64_t n_ent, int64_t ld_ent,
                                   const float* bias, const int32_t* pos_cand, int32_t n_pos, float pos, float add,
                                   float* g_pos, float* d_x, float* d_bias_s, float* loss, void* workspace,
                                   size_t workspace_bytes, void* stream) {
  return shared_loss_entry<BceLoss>(__func__, logit_t, ldt, mask_t, shared, k, x, B, D, ent, n_ent, ld_ent, bias, pos_cand,
                                    n_pos, pos, add, 0.f, 0.f, g_pos, d_x, d_bias_s, loss, workspace, workspace_bytes,
                                    stream);
}

extern "C" int kgc_shared_adv_loss(float* logit_t, int64_t ldt, const uint32_t* mask_t, const int32_t* shared, int32_t k,
                                   const float* x, int64_t B, int32_t D, const float* ent, int64_t n_ent, int64_t ld_ent,
                                   const float* bias, const int32_t* pos_cand, int32_t n_pos, float pos, float add,
                                   float temperature, float* g_pos, float* d_x, float* d_bias_s, float* loss,
                                   void* workspace, size_t workspace_bytes, void* stream) {
  KGC_REQUIRE(std::isfinite(temperature) && temperature >= 0.f, "the adversarial temperature must be finite and >= 0");
  return shared_loss_entry<AdvLoss>(__func__, logit_t, ldt, mask_t, shared, k, x, B, D, ent, n_ent, ld_ent, bias, pos_cand,
                                    n_pos, pos, add, temperature, 0.f, g_pos, d_x, d_bias_s, loss, workspace,
                                    workspace_bytes, stream);
}

extern "C" int kgc_shared_ce_loss(float* logit_t, int64_t ldt, const uint32_t* mask_t, const int32_t* shared, int32_t k,
                                  const float* x, int64_t B, int32_t D, const float* ent, int64_t n_ent, int64_t ld_ent,
                                  const float* bias, const int32_t* pos_cand, int32_t n_pos, float label_smoothing,
                                  float* g_pos, float* d_x, float* d_bias_s, float* loss, void* workspace,
                                  size_t workspace_bytes, void* stream) {
  KGC_REQUIRE(label_smoothing >= 0.f && label_smoothing <= 1.f, "the label smoothing must be a number in [0, 1]");
  return shared_loss_entry<CeLoss>(__func__, logit_t, ldt, mask_t, shared, k, x, B, D, ent, n_ent, ld_ent, bias, pos_cand,
                                   n_pos, 0.f, 0.f, 0.f, label_smoothing, g_pos, d_x, d_bias_s, loss, workspace,
                                   workspace_bytes, stream);
}

extern "C" int kgc_shared_bwd_table(const int32_t* sorted_ids, const int32_t* sorted_slots, int32_t k, int64_t n_ent,
                                    int32_t D, const float* d_rows, int64_t ld_rows, const float* d_row_bias,
                                    const float* scale, float* d_ent, int64_t ld_d, float* d_bias, void* stream) {
  KGC_REQUIRE(k > 0 && n_ent > 0 && n_ent < (int64_t{1} << 31) - 1 && D > 0 && D <= 256 && D % 4 == 0, "bad sizes");
  KGC_REQUIRE(ld_rows >= D && ld_rows % 4 == 0 && ld_d >= D && ld_d % 4 == 0, "rows need a 16-byte pitch of >= D floats");
  KGC_REQUIRE(sorted_ids && sorted_slots && d_rows && d_row_bias && scale && d_ent && d_bias, "null buffer");
  KGC_REQUIRE(((reinterpret_cast<uintptr_t>(d_rows) | reinterpret_cast<uintptr_t>(d_ent)) & 15) == 0,
              "d_rows and d_ent must be 16-byte aligned");
  const unsigned blocks = (unsigned)ceil_div(ceil_div(k, 32), kWarpsSS);
  const int D4 = D / 4;
  const auto add = for_width(D4, shared_table_kernel<1>, shared_table_kernel<2>);
  add<<<blocks, kThreadsSS, 0, as_stream(stream)>>>(sorted_ids, sorted_slots, k, n_ent, d_rows, ld_rows, d_row_bias, D4,
                                                    scale, d_ent, ld_d, d_bias);
  KGC_LAUNCH_CHECK();
  return 0;
}
