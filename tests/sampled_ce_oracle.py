"""Float64 restatement of the negative-sampled softmax cross-entropy (kgc_sampled_ce_fwd, score_sampled_ce).
tests/test_sampled_ce_cpu.py pins it to torch.nn.functional.cross_entropy + autograd on per-positive logit rows;
tests/test_gpu_sampled_ce.py holds the kernels to it."""
import torch


def sampled_ce(x, all_ent, bias, cand, n_pos, eps=0.0):
    """Query b scores z = <x[b], all_ent[c]> + bias[c] for its candidates cand[b, :] (positives in the first ``n_pos``
    columns, negatives after them; ids outside [0, N) are empty slots).  With P_b / Q_b its valid positive / negative
    slots, K_b = 1 + |Q_b| and LSE_p = log(exp(z_p) + sum_{Q_b} exp(z_q)):

        l_p = (1 - eps) (LSE_p - z_p) + eps (LSE_p - (z_p + sum_{Q_b} z_q) / K_b),   L = (1/P) sum_b sum_{P_b} l_p

    with P the number of valid positive slots (L = 0 when P = 0).  The logit gradient is (softmax_p(p) - (1 - eps) -
    eps / K_b) / P on a positive slot and sum_{P_b} (softmax_p(q) - eps / K_b) / P on a negative one.  Returns (loss,
    g [B, C], d_x, d_all_ent, d_bias) for a unit upstream gradient, in float64."""
    x, ent, bias = (torch.as_tensor(t).double().cpu() for t in (x, all_ent, bias))
    cand = torch.as_tensor(cand).long().cpu()
    B, C = cand.shape
    N = ent.shape[0]
    valid = (cand >= 0) & (cand < N)
    c = torch.where(valid, cand, torch.zeros_like(cand))
    z = (x[:, None, :] * ent[c]).sum(-1) + bias[c]
    is_pos = torch.zeros((B, C), dtype=torch.bool)
    is_pos[:, :n_pos] = True
    vp, vn = valid & is_pos, valid & ~is_pos
    n_q = vn.sum(1).double()
    k_b = 1.0 + n_q
    P = int(vp.sum())
    zn = torch.where(vn, z, torch.full_like(z, -float('inf')))
    lse_q = torch.logsumexp(zn, 1)                                     # -inf for a query without valid negatives
    lse = torch.logaddexp(z, lse_q[:, None])                           # LSE_p for every slot taken as a positive
    z_sum = torch.where(vn, z, torch.zeros_like(z)).sum(1)
    l = (1.0 - eps) * (lse - z) + eps * (lse - (z + z_sum[:, None]) / k_b[:, None])
    inv_p = 1.0 / P if P else 0.0
    loss = torch.where(vp, l, torch.zeros_like(l)).sum() * inv_p
    # softmax_p(p) - (1 - eps) - eps / K_b written as eps |Q_b| / K_b - (1 - softmax_p(p)): exactly 0 without negatives
    g_pos = (eps * n_q[:, None] / k_b[:, None] + torch.expm1(z - lse)) * inv_p
    # softmax_p(q) = exp(z_q - LSE_p), summed over the valid positives p of the query
    lse_p = torch.where(vp, lse, torch.full_like(lse, float('inf')))[:, :n_pos]          # [B, n_pos]
    soft = torch.exp(z[:, None, :] - lse_p[:, :, None]).sum(1) if n_pos else torch.zeros_like(z)
    g_neg = (soft - vp.sum(1).double()[:, None] * eps / k_b[:, None]) * inv_p
    g = torch.where(vp, g_pos, torch.where(vn, g_neg, torch.zeros_like(z)))
    d_x = (g[:, :, None] * ent[c]).sum(1)
    d_ent = torch.zeros_like(ent).index_add_(0, c.reshape(-1), (g[:, :, None] * x[:, None, :]).reshape(B * C, -1))
    d_bias = torch.zeros((N,), dtype=torch.float64).index_add_(0, c.reshape(-1), g.reshape(-1))
    return loss, g, d_x, d_ent, d_bias
