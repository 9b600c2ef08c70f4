"""Self-adversarial negative sampling, host side: the float64 restatement of tests/sampled_oracle.py against
torch.nn.BCELoss(weight=...) + autograd on the gathered probabilities and against RotatE's logsigmoid formula, its bridge
to the plain sampled objective at alpha = 0, and the argument checks of the Python surface (no GPU needed)."""
import numpy as np
import pytest
import torch

import sampled_oracle as so


def _weighted_bce_autograd(x, ent, bias, cand, n_pos, alpha, pos, add):
    """torch.nn.BCELoss(weight=c, reduction='sum') over the valid slots' probabilities, gradients by autograd, float64.
    c = 1 / (2 Q+ |P_b|) on a positive slot and w / (2 Q-) on a negative one, w = softmax over the query's valid negatives
    of alpha times the detached logits."""
    x, ent, bias = (t.clone().double().requires_grad_(True) for t in (x, ent, bias))
    cand = torch.as_tensor(cand).long()
    B, C = cand.shape
    valid = (cand >= 0) & (cand < ent.shape[0])
    b_idx, j_idx = torch.nonzero(valid, as_tuple=True)
    ids = cand[b_idx, j_idx]
    z = (x[b_idx] * ent[ids]).sum(1) + bias[ids]
    is_pos = j_idx < n_pos
    zd = z.detach()
    weight = torch.zeros_like(zd)
    q_pos = len(set(b_idx[is_pos].tolist()))
    q_neg = len(set(b_idx[~is_pos].tolist()))
    for b in range(B):
        sel_p = (b_idx == b) & is_pos
        sel_n = (b_idx == b) & ~is_pos
        if sel_p.any():
            weight[sel_p] = 1.0 / (2.0 * q_pos * int(sel_p.sum()))
        if sel_n.any():
            weight[sel_n] = torch.softmax(alpha * zd[sel_n], 0) / (2.0 * q_neg)
    target = torch.where(is_pos, torch.tensor(float(pos), dtype=torch.float64), torch.tensor(float(add), dtype=torch.float64))
    loss = torch.nn.BCELoss(weight=weight, reduction='sum')(torch.sigmoid(z), target)
    loss.backward()
    return loss.detach(), x.grad, ent.grad, bias.grad


def _case(B, C, N, D, n_pos, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, D, generator=g)
    ent = torch.randn(N, D, generator=g) * (1.0 / D ** 0.5)
    bias = torch.randn(N, generator=g) * 0.1
    cand = torch.randint(0, N, (B, C), generator=g)
    cand[0, 0] = -1                                       # an empty positive slot
    cand[1, :n_pos] = -1                                  # a query without positives
    cand[2, n_pos:] = -1                                  # a query whose negative slots are all empty
    cand[3, :] = cand[3, 0]                               # one entity in every slot of a query
    cand[4, -1] = -1                                      # an empty negative slot
    return x, ent, bias, cand


@pytest.mark.parametrize('alpha', [0.0, 0.5, 1.0, 4.0])
@pytest.mark.parametrize('B,C,N,D,n_pos,smooth,seed', [
    (7, 9, 50, 8, 1, 0.0, 0),       # duplicates within and across queries
    (6, 70, 13, 4, 3, 0.1, 1),      # N < C: every query repeats entities; label smoothing
    (16, 6, 1000, 20, 3, 0.0, 2),
])
def test_sampled_adv_oracle_matches_weighted_bceloss(B, C, N, D, n_pos, smooth, seed, alpha):
    x, ent, bias, cand = _case(B, C, N, D, n_pos, seed)
    pos, add = (float(np.float32(1.0 - smooth) + np.float32(1.0 / N)), float(np.float32(1.0 / N))) if smooth else (1.0, 0.0)
    loss, gl, d_x, d_ent, d_bias = so.sampled_adv(x, ent, bias, cand, n_pos, alpha, pos, add)
    r_loss, r_x, r_ent, r_bias = _weighted_bce_autograd(x, ent, bias, cand, n_pos, alpha, pos, add)
    assert abs(float(loss) - float(r_loss)) <= 1e-12 * abs(float(r_loss))
    for got, ref in ((d_x, r_x), (d_ent, r_ent), (d_bias, r_bias)):
        assert float((got - ref).abs().max()) <= 1e-12 * float(ref.abs().max())
    assert float(gl[cand < 0].abs().max()) == 0.0
    assert float(gl[1].abs().max()) > 0.0 and float(gl[2].abs().max()) > 0.0     # each keeps its other half
    c = cand.clamp_min(0).long()
    assert torch.allclose((gl[:, :, None] * ent.double()[c]).sum(1), d_x, rtol=0, atol=1e-15)


@pytest.mark.parametrize('alpha', [0.0, 0.5, 1.0, 4.0])
def test_sampled_adv_oracle_is_rotate_formula(alpha):
    """pos = 1, add = 0, one positive, no empty slot, unsaturated logits: RotatE's self-adversarial loss
    (-logsigmoid(z_pos).mean() - (softmax(alpha z_neg).detach() * logsigmoid(-z_neg)).sum(1).mean()) / 2."""
    B, C, N, D = 12, 17, 40, 16
    g = torch.Generator().manual_seed(9)
    x = torch.randn(B, D, generator=g)
    ent = torch.randn(N, D, generator=g) * (1.0 / D ** 0.5)
    bias = torch.randn(N, generator=g) * 0.1
    cand = torch.randint(0, N, (B, C), generator=g)
    loss, _, d_x, d_ent, d_bias = so.sampled_adv(x, ent, bias, cand, 1, alpha)
    xd, ed, bd = (t.clone().double().requires_grad_(True) for t in (x, ent, bias))
    z = (xd[:, None, :] * ed[cand]).sum(-1) + bd[cand]
    assert float(z.detach().abs().max()) < 10.0
    zp, zn = z[:, 0], z[:, 1:]
    w = torch.softmax(alpha * zn.detach(), 1)
    ref = (-torch.nn.functional.logsigmoid(zp).mean() - (w * torch.nn.functional.logsigmoid(-zn)).sum(1).mean()) / 2
    ref.backward()
    assert abs(float(loss) - float(ref)) <= 1e-12 * abs(float(ref))
    for got, r in ((d_x, xd.grad), (d_ent, ed.grad), (d_bias, bd.grad)):
        assert float((got - r).abs().max()) <= 1e-12 * float(r.abs().max())


def test_sampled_adv_oracle_without_valid_slots():
    loss, gl, d_x, d_ent, d_bias = so.sampled_adv(torch.ones(2, 4), torch.ones(3, 4), torch.zeros(3),
                                                  torch.full((2, 5), -1), 1, 1.0)
    assert float(loss) == 0.0 and float(gl.abs().sum()) == 0.0
    assert float(d_x.abs().sum()) == 0.0 and float(d_ent.abs().sum()) == 0.0 and float(d_bias.abs().sum()) == 0.0


@pytest.mark.parametrize('n_pos', [1, 3])
def test_sampled_adv_oracle_alpha_zero_bridge(n_pos):
    """alpha = 0 with the same numbers of valid positives and negatives in every query: the mean of the two plain sampled
    losses, 1/2 (sampled_bce(cand[:, :P], P) + sampled_bce(cand[:, P:], 0)), and the same for every gradient."""
    B, C, N, D = 9, 14, 30, 8
    g = torch.Generator().manual_seed(4 + n_pos)
    x = torch.randn(B, D, generator=g)
    ent = torch.randn(N, D, generator=g) * 0.4
    bias = torch.randn(N, generator=g) * 0.1
    cand = torch.randint(0, N, (B, C), generator=g)
    cand[:, n_pos - 1] = -1                               # one empty positive and one empty negative slot per query
    cand[:, C - 2] = -1
    pos, add = 0.93, 0.01
    got = so.sampled_adv(x, ent, bias, cand, n_pos, 0.0, pos, add)
    a = so.sampled_bce(x, ent, bias, cand[:, :n_pos], n_pos, pos, add)
    b = so.sampled_bce(x, ent, bias, cand[:, n_pos:], 0, pos, add)
    assert abs(float(got[0]) - 0.5 * float(a[0] + b[0])) <= 1e-12 * abs(float(got[0]))
    assert float((got[1] - 0.5 * torch.cat([a[1], b[1]], 1)).abs().max()) <= 1e-12 * float(got[1].abs().max())
    for i in (2, 3, 4):
        ref = 0.5 * (a[i] + b[i])
        assert float((got[i] - ref).abs().max()) <= 1e-12 * float(ref.abs().max())


@pytest.mark.parametrize('alpha', [-0.5, float('nan'), float('inf'), True, '1.0', torch.tensor(1.0)])
def test_score_sampled_bce_adversarial_temperature_errors(alpha):
    """A negative, non-finite, bool or non-number temperature is a ValueError raised before any device work (the
    tensors here are on the CPU, which would otherwise be a RuntimeError)."""
    import kgc_gcn_b200 as k
    x, ent, bias = torch.zeros(3, 8), torch.zeros(10, 8), torch.zeros(10)
    cand = torch.zeros(3, 4, dtype=torch.int32)
    with pytest.raises(ValueError):
        k.score_sampled_bce(x, ent, bias, cand, 1, adversarial_temperature=alpha)


def test_score_sampled_bce_adversarial_temperature_accepted():
    import kgc_gcn_b200 as k
    x, ent, bias = torch.zeros(3, 8), torch.zeros(10, 8), torch.zeros(10)
    cand = torch.zeros(3, 4, dtype=torch.int32)
    for alpha in (0, 0.0, 1, 2.5, np.float32(0.5)):
        with pytest.raises(RuntimeError):                                 # past the check: CPU tensors, no fallback
            k.score_sampled_bce(x, ent, bias, cand, 1, adversarial_temperature=alpha)


def test_graphed_step_adversarial_temperature_errors():
    import kgc_gcn_b200 as k
    kb = k.KBDataset([{'triple': (0, 0, -1), 'label': [1, 2]}], 5, None, training=True)
    with pytest.raises(ValueError):
        k.GraphedTrainStep(None, None, None, kb, 4, adversarial_temperature=1.0)                 # without negatives=
    with pytest.raises(ValueError):
        k.GraphedTrainStep(None, None, None, kb, 4, fused_loss=True, adversarial_temperature=1.0)
    for alpha in (-1.0, float('nan'), True):
        with pytest.raises(ValueError):
            k.GraphedTrainStep(None, None, None, kb, 4, negatives=8, adversarial_temperature=alpha)
