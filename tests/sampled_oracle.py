"""Float64 restatements of the negative-sampled training objective (extensions without a reference counterpart: the
reference trains 1-N only).  tests/test_sampled_cpu.py pins them to torch.nn.BCELoss + autograd; the GPU tests hold the
kernels (kgc_pos_sample, kgc_sampled_bce_fwd / kgc_sampled_bce_bwd_table) to them."""
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


def sampled_bce(x, all_ent, bias, cand, n_pos, pos=1.0, add=0.0):
    """Mean BCE over the valid slots of p[b, c] = sigmoid(<x[b], all_ent[cand[b, c]]> + bias[cand[b, c]]), label ``pos``
    in the first ``n_pos`` columns and ``add`` after them; ids outside [0, N) are empty slots.  ATen's elementwise
    formulas (logs clamped at -100, the gradient's denominator at 1e-12), in float64.  Returns (loss, g [B, C] logit
    gradient, d_x, d_all_ent, d_bias) for a unit upstream gradient; loss 0 and zero gradients without a valid slot."""
    x, ent, bias = (torch.as_tensor(t).double().cpu() for t in (x, all_ent, bias))
    cand = torch.as_tensor(cand).long().cpu()
    B, C = cand.shape
    N = ent.shape[0]
    valid = (cand >= 0) & (cand < N)
    c = torch.where(valid, cand, torch.zeros_like(cand))
    z = (x[:, None, :] * ent[c]).sum(-1) + bias[c]
    p = torch.sigmoid(z)
    y = torch.full((B, C), float(add), dtype=torch.float64)
    y[:, :n_pos] = float(pos)
    count = int(valid.sum())
    g = torch.zeros((B, C), dtype=torch.float64)
    loss = torch.zeros((), dtype=torch.float64)
    if count:
        term = (y - 1.0) * torch.log1p(-p).clamp_min(-100.0) - y * torch.log(p).clamp_min(-100.0)
        loss = term[valid].sum() / count
        d_pred = (p - y) / ((1.0 - p) * p).clamp_min(1e-12) / count
        g = torch.where(valid, d_pred * p * (1.0 - p), g)
    d_x = (g[:, :, None] * ent[c]).sum(1)
    d_ent = torch.zeros_like(ent).index_add_(0, c.reshape(-1), (g[:, :, None] * x[:, None, :]).reshape(B * C, -1))
    d_bias = torch.zeros((N,), dtype=torch.float64).index_add_(0, c.reshape(-1), g.reshape(-1))
    return loss, g, d_x, d_ent, d_bias
