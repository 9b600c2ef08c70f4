"""Float64 restatement of the self-adversarial negative-sampled objective (kgc_sampled_adv_fwd, score_sampled_bce(...,
adversarial_temperature=alpha)).  tests/test_sampled_adv_cpu.py pins it to torch.nn.BCELoss + autograd and to RotatE's
logsigmoid formula; tests/test_gpu_sampled_adv.py holds the kernels to it."""
import torch


def sampled_adv(x, all_ent, bias, cand, n_pos, alpha, pos=1.0, add=0.0):
    """Query b scores p = sigmoid(z), z = <x[b], all_ent[c]> + bias[c], for its candidates cand[b, :] (label ``pos`` in the
    first ``n_pos`` columns, ``add`` after them; ids outside [0, N) are empty slots).  With P_b / Q_b its valid positive /
    negative slots, l ATen's BCE term (logs clamped at -100) and w = softmax over Q_b of (alpha z), a constant:

        L = 1/2 (1/Q+) sum_{b: P_b} (1/|P_b|) sum_{P_b} l(z, pos) + 1/2 (1/Q-) sum_{b: Q_b} sum_{Q_b} w l(z, add)

    where Q+ / Q- count the queries with a non-empty P_b / Q_b; a half with a zero count is 0.  The logit gradient is
    g = c (p - y) / max((1 - p) p, 1e-12) p (1 - p) with c = 1 / (2 Q+ |P_b|) on a positive slot and w / (2 Q-) on a
    negative one.  Returns (loss, g [B, C], d_x, d_all_ent, d_bias) for a unit upstream gradient, in float64."""
    x, ent, bias = (torch.as_tensor(t).double().cpu() for t in (x, all_ent, bias))
    cand = torch.as_tensor(cand).long().cpu()
    B, C = cand.shape
    N = ent.shape[0]
    valid = (cand >= 0) & (cand < N)
    c = torch.where(valid, cand, torch.zeros_like(cand))
    z = (x[:, None, :] * ent[c]).sum(-1) + bias[c]
    p = torch.sigmoid(z)
    is_pos = torch.zeros((B, C), dtype=torch.bool)
    is_pos[:, :n_pos] = True
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
    coef = torch.zeros((B, C), dtype=torch.float64)
    if q_pos:
        coef = torch.where(vp, 1.0 / (2.0 * q_pos * n_p.clamp_min(1).double())[:, None], coef)
    if q_neg:
        coef = torch.where(vn, w / (2.0 * q_neg), coef)
    term = (y - 1.0) * torch.log1p(-p).clamp_min(-100.0) - y * torch.log(p).clamp_min(-100.0)
    loss = (coef * torch.where(valid, term, torch.zeros_like(term))).sum()
    g = torch.where(valid, coef * (p - y) / ((1.0 - p) * p).clamp_min(1e-12) * p * (1.0 - p), torch.zeros_like(z))
    d_x = (g[:, :, None] * ent[c]).sum(1)
    d_ent = torch.zeros_like(ent).index_add_(0, c.reshape(-1), (g[:, :, None] * x[:, None, :]).reshape(B * C, -1))
    d_bias = torch.zeros((N,), dtype=torch.float64).index_add_(0, c.reshape(-1), g.reshape(-1))
    return loss, g, d_x, d_ent, d_bias
