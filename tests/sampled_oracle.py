"""Float64 restatements of the negative-sampled training objectives (extensions without a reference counterpart: the
reference trains 1-N only): the positive sampler and the three sampled losses.  tests/test_sampled_cpu.py,
test_sampled_adv_cpu.py and test_sampled_ce_cpu.py pin them to torch (BCELoss, RotatE's formula, cross_entropy) +
autograd; the GPU tests hold the kernels (kgc_pos_sample, kgc_sampled_bce_fwd, kgc_sampled_adv_fwd, kgc_sampled_ce_fwd,
kgc_sampled_bce_bwd_table) to them.

Each loss returns (loss, g [B, C] logit gradient, d_x, d_all_ent, d_bias) for a unit upstream gradient, in float64.
Query b scores z = <x[b], all_ent[c]> + bias[c] for its candidates cand[b, :]: positives in the first ``n_pos`` columns,
negatives after them; ids outside [0, N) are empty slots (no loss, no gradient)."""
import numpy as np
import torch


def pos_sample(label_lists, qid, draws):
    """Restatement of kgc_pos_sample: out[b, j] = label_lists[qid[b]][(draws[b, j] * len) >> 32] (sampling with
    replacement), -1 for a query without objects."""
    d = np.asarray(draws).astype(np.uint64)
    B, P = d.shape
    out = np.full((B, P), -1, dtype=np.int32)
    for b in range(B):
        lst = list(label_lists[int(qid[b])])
        if lst:
            for j in range(P):
                out[b, j] = int(lst[int((d[b, j] * np.uint64(len(lst))) >> np.uint64(32))])
    return out


def _logits(x, all_ent, bias, cand, n_pos):
    """The shared front: float64 operands, the valid mask, the ids with empty slots clamped to 0, the logits z [B, C] and
    the positive-column mask."""
    x, ent, bias = (torch.as_tensor(t).double().cpu() for t in (x, all_ent, bias))
    cand = torch.as_tensor(cand).long().cpu()
    B, C = cand.shape
    N = ent.shape[0]
    valid = (cand >= 0) & (cand < N)
    c = torch.where(valid, cand, torch.zeros_like(cand))
    z = (x[:, None, :] * ent[c]).sum(-1) + bias[c]
    is_pos = torch.zeros((B, C), dtype=torch.bool)
    is_pos[:, :n_pos] = True
    return x, ent, valid, c, z, is_pos


def _grads(g, x, ent, c):
    """The shared tail: d_x, d_all_ent and d_bias from the logit gradient g (zero on empty slots)."""
    B, C = c.shape
    d_x = (g[:, :, None] * ent[c]).sum(1)
    d_ent = torch.zeros_like(ent).index_add_(0, c.reshape(-1), (g[:, :, None] * x[:, None, :]).reshape(B * C, -1))
    d_bias = torch.zeros((ent.shape[0],), dtype=torch.float64).index_add_(0, c.reshape(-1), g.reshape(-1))
    return d_x, d_ent, d_bias


def sampled_bce(x, all_ent, bias, cand, n_pos, pos=1.0, add=0.0):
    """Mean BCE over the valid slots of p = sigmoid(z), label ``pos`` in the first ``n_pos`` columns and ``add`` after
    them.  ATen's elementwise formulas (logs clamped at -100, the gradient's denominator at 1e-12).  Loss 0 and zero
    gradients without a valid slot."""
    x, ent, valid, c, z, is_pos = _logits(x, all_ent, bias, cand, n_pos)
    p = torch.sigmoid(z)
    y = torch.where(is_pos, torch.tensor(float(pos), dtype=torch.float64), torch.tensor(float(add), dtype=torch.float64))
    count = int(valid.sum())
    g = torch.zeros_like(z)
    loss = torch.zeros((), dtype=torch.float64)
    if count:
        term = (y - 1.0) * torch.log1p(-p).clamp_min(-100.0) - y * torch.log(p).clamp_min(-100.0)
        loss = term[valid].sum() / count
        d_pred = (p - y) / ((1.0 - p) * p).clamp_min(1e-12) / count
        g = torch.where(valid, d_pred * p * (1.0 - p), g)
    return (loss, g) + _grads(g, x, ent, c)


def sampled_adv(x, all_ent, bias, cand, n_pos, alpha, pos=1.0, add=0.0):
    """Self-adversarial BCE (kgc_sampled_adv_fwd, score_sampled_bce(..., adversarial_temperature=alpha)).  With P_b / Q_b
    query b's valid positive / negative slots, l ATen's BCE term (logs clamped at -100) of p = sigmoid(z) and
    w = softmax over Q_b of (alpha z), a constant:

        L = 1/2 (1/Q+) sum_{b: P_b} (1/|P_b|) sum_{P_b} l(z, pos) + 1/2 (1/Q-) sum_{b: Q_b} sum_{Q_b} w l(z, add)

    where Q+ / Q- count the queries with a non-empty P_b / Q_b; a half with a zero count is 0.  The logit gradient is
    g = c (p - y) / max((1 - p) p, 1e-12) p (1 - p) with c = 1 / (2 Q+ |P_b|) on a positive slot and w / (2 Q-) on a
    negative one."""
    x, ent, valid, c, z, is_pos = _logits(x, all_ent, bias, cand, n_pos)
    p = torch.sigmoid(z)
    y = torch.where(is_pos, torch.tensor(float(pos), dtype=torch.float64), torch.tensor(float(add), dtype=torch.float64))
    vp, vn = valid & is_pos, valid & ~is_pos
    n_p, n_n = vp.sum(1), vn.sum(1)
    q_pos, q_neg = int((n_p > 0).sum()), int((n_n > 0).sum())
    # softmax over each query's valid negatives (rows without any get all-zero weights)
    a = torch.where(vn, float(alpha) * z, torch.tensor(-float('inf'), dtype=torch.float64))
    m = a.max(1, keepdim=True).values
    e = torch.where(vn, torch.exp(a - torch.where(torch.isfinite(m), m, torch.zeros_like(m))), torch.zeros_like(z))
    s = e.sum(1, keepdim=True)
    w = torch.where(s > 0, e / torch.where(s > 0, s, torch.ones_like(s)), torch.zeros_like(e))
    coef = torch.zeros_like(z)
    if q_pos:
        coef = torch.where(vp, 1.0 / (2.0 * q_pos * n_p.clamp_min(1).double())[:, None], coef)
    if q_neg:
        coef = torch.where(vn, w / (2.0 * q_neg), coef)
    term = (y - 1.0) * torch.log1p(-p).clamp_min(-100.0) - y * torch.log(p).clamp_min(-100.0)
    loss = (coef * torch.where(valid, term, torch.zeros_like(term))).sum()
    g = torch.where(valid, coef * (p - y) / ((1.0 - p) * p).clamp_min(1e-12) * p * (1.0 - p), torch.zeros_like(z))
    return (loss, g) + _grads(g, x, ent, c)


def sampled_ce(x, all_ent, bias, cand, n_pos, eps=0.0):
    """Softmax cross-entropy (kgc_sampled_ce_fwd, score_sampled_ce).  With P_b / Q_b query b's valid positive / negative
    slots, K_b = 1 + |Q_b| and LSE_p = log(exp(z_p) + sum_{Q_b} exp(z_q)):

        l_p = (1 - eps) (LSE_p - z_p) + eps (LSE_p - (z_p + sum_{Q_b} z_q) / K_b),   L = (1/P) sum_b sum_{P_b} l_p

    with P the number of valid positive slots (L = 0 when P = 0).  The logit gradient is (softmax_p(p) - (1 - eps) -
    eps / K_b) / P on a positive slot and sum_{P_b} (softmax_p(q) - eps / K_b) / P on a negative one."""
    x, ent, valid, c, z, is_pos = _logits(x, all_ent, bias, cand, n_pos)
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
    return (loss, g) + _grads(g, x, ent, c)
