"""Negative-sampled softmax cross-entropy, host side: the float64 restatement of tests/sampled_oracle.py against
torch.nn.functional.cross_entropy(label_smoothing=eps) + autograd on explicitly built per-positive logit rows, and the
argument checks of the Python surface (no GPU needed)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import sampled_oracle as so


def _cross_entropy_autograd(x, ent, bias, cand, n_pos, eps):
    """For each valid positive slot p of query b the row [z_p, z_q for the valid negative slots q of b] with target 0,
    F.cross_entropy(label_smoothing=eps) summed over the rows and divided by their number; gradients by autograd."""
    x, ent, bias = (t.clone().double().requires_grad_(True) for t in (x, ent, bias))
    cand = torch.as_tensor(cand).long()
    B, C = cand.shape
    N = ent.shape[0]
    total, rows = x.sum() * 0.0, 0
    for b in range(B):
        ids = cand[b]
        ok = (ids >= 0) & (ids < N)
        safe = torch.where(ok, ids, torch.zeros_like(ids))
        zb = (x[b][None, :] * ent[safe]).sum(1) + bias[safe]
        neg = [j for j in range(n_pos, C) if ok[j]]
        for p in range(n_pos):
            if not ok[p]:
                continue
            row = torch.cat([zb[p:p + 1], zb[neg]])
            total = total + F.cross_entropy(row[None], torch.zeros(1, dtype=torch.long), label_smoothing=eps,
                                            reduction='sum')
            rows += 1
    loss = total / rows if rows else total
    loss.backward()
    return loss.detach(), x.grad, ent.grad, bias.grad


def _case(B, C, N, D, n_pos, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, D, generator=g)
    ent = torch.randn(N, D, generator=g) * (scale / D ** 0.5)
    bias = torch.randn(N, generator=g) * 0.1
    cand = torch.randint(0, N, (B, C), generator=g)
    cand[0, 0] = -1                                       # an empty positive slot
    cand[1, :n_pos] = -1                                  # a query without positives
    cand[2, n_pos:] = -1                                  # a query whose negative slots are all empty
    cand[3, :] = cand[3, 0]                               # one entity in every slot of a query
    cand[4, -1] = N + 3                                   # an id past the table: an empty negative slot
    return x, ent, bias, cand


@pytest.mark.parametrize('eps', [0.0, 0.1])
@pytest.mark.parametrize('B,C,N,D,n_pos,seed,scale', [
    (7, 9, 50, 8, 1, 0, 1.0),       # duplicates within and across queries
    (6, 70, 13, 4, 3, 1, 1.0),      # N < C: every query repeats entities; n_pos > 1
    (16, 6, 1000, 20, 3, 2, 1.0),
    (9, 12, 40, 16, 2, 3, 60.0),    # logits in the hundreds
])
def test_sampled_ce_oracle_matches_cross_entropy(B, C, N, D, n_pos, seed, scale, eps):
    x, ent, bias, cand = _case(B, C, N, D, n_pos, seed, scale)
    loss, gl, d_x, d_ent, d_bias = so.sampled_ce(x, ent, bias, cand, n_pos, eps)
    r_loss, r_x, r_ent, r_bias = _cross_entropy_autograd(x, ent, bias, cand, n_pos, eps)
    assert abs(float(loss) - float(r_loss)) <= 1e-12 * abs(float(r_loss))
    for got, ref in ((d_x, r_x), (d_ent, r_ent), (d_bias, r_bias)):
        assert float((got - ref).abs().max()) <= 1e-12 * float(ref.abs().max())
    empty = (cand < 0) | (cand >= N)
    assert float(gl[empty].abs().max()) == 0.0
    assert float(gl[1].abs().max()) == 0.0                # no positive: the query adds nothing
    assert float(gl[2].abs().max()) == 0.0                # positives without negatives: 0 loss and 0 gradient
    c = cand.clamp(0, N - 1).long()
    assert torch.allclose((gl[:, :, None] * ent.double()[c]).sum(1), d_x, rtol=0, atol=1e-12 * float(d_x.abs().max()))


def test_sampled_ce_oracle_positive_without_negatives_adds_nothing():
    """A batch whose only valid positive has no valid negative: the loss is 0 and so is every gradient; with one more
    query that has both, the loss is that query's term over P = 2."""
    x, ent, bias = torch.randn(2, 4), torch.randn(6, 4), torch.randn(6)
    cand = torch.tensor([[1, -1, -1], [2, 3, 4]])
    for eps in (0.0, 0.1):
        loss, gl, d_x, _, _ = so.sampled_ce(x[:1], ent, bias, cand[:1], 1, eps)
        assert float(loss) == 0.0 and float(gl.abs().sum()) == 0.0 and float(d_x.abs().sum()) == 0.0
        both = so.sampled_ce(x, ent, bias, cand, 1, eps)[0]
        one = so.sampled_ce(x[1:], ent, bias, cand[1:], 1, eps)[0]
        assert abs(float(both) - 0.5 * float(one)) <= 1e-15 * abs(float(one))


def test_sampled_ce_oracle_without_valid_slots():
    loss, gl, d_x, d_ent, d_bias = so.sampled_ce(torch.ones(2, 4), torch.ones(3, 4), torch.zeros(3),
                                                 torch.full((2, 5), -1), 1, 0.1)
    assert float(loss) == 0.0 and float(gl.abs().sum()) == 0.0
    assert float(d_x.abs().sum()) == 0.0 and float(d_ent.abs().sum()) == 0.0 and float(d_bias.abs().sum()) == 0.0


def _cpu_args():
    return torch.zeros(3, 8), torch.zeros(10, 8), torch.zeros(10), torch.zeros(3, 4, dtype=torch.int32)


@pytest.mark.parametrize('eps', [-0.1, 1.5, float('nan'), float('inf'), True, '0.1', torch.tensor(0.1)])
def test_score_sampled_ce_label_smoothing_errors(eps):
    """A label smoothing outside [0, 1], non-finite, bool or not a number is a ValueError raised before any device work
    (the tensors here are on the CPU, which would otherwise be a RuntimeError)."""
    import kgc_gcn_b200 as k
    x, ent, bias, cand = _cpu_args()
    with pytest.raises(ValueError):
        k.score_sampled_ce(x, ent, bias, cand, 1, label_smoothing=eps)


def test_score_sampled_ce_argument_errors():
    """The argument rules of score_sampled_bce: shapes, n_pos in [0, C], int32 candidates."""
    import kgc_gcn_b200 as k
    x, ent, bias, cand = _cpu_args()
    for args in ((x[0], ent, bias, cand, 1), (x, ent[:, :4], bias, cand, 1), (x, ent, bias, cand, 5),
                 (x, ent, bias, cand, -1), (x, ent, bias, cand, True), (x, ent, bias, cand.long(), 1),
                 (x[:, :6], ent[:, :6], bias, cand, 1)):
        with pytest.raises(ValueError):
            k.score_sampled_ce(*args)


def test_score_sampled_ce_accepted_arguments_reach_the_device_check():
    import kgc_gcn_b200 as k
    x, ent, bias, cand = _cpu_args()
    for eps in (0, 0.0, 0.1, 1, np.float32(0.5)):
        with pytest.raises(RuntimeError):                                 # past the checks: CPU tensors, no fallback
            k.score_sampled_ce(x, ent, bias, cand, 1, label_smoothing=eps)


def test_loss_sampled_criterion_errors():
    """MGCN.loss_sampled rejects a temperature with 'ce', a label smoothing with 'bce' and an unknown criterion before
    it touches the model, the dataset or a device."""
    import kgc_gcn_b200 as k
    m = k.MGCN.__new__(k.MGCN)
    for kw in (dict(criterion='ce', adversarial_temperature=1.0), dict(label_smoothing=0.1),
               dict(criterion='bce', label_smoothing=0.1), dict(criterion='softmax'), dict(criterion=None),
               dict(criterion='ce', label_smoothing=2.0)):
        with pytest.raises(ValueError):
            m.loss_sampled([0], None, None, 4, **kw)


def test_graphed_step_criterion_errors():
    import kgc_gcn_b200 as k
    kb = k.KBDataset([{'triple': (0, 0, -1), 'label': [1, 2]}], 5, None, training=True)
    for kw in (dict(criterion='ce'),                                                   # without negatives=
               dict(criterion='ce', fused_loss=True),
               dict(negatives=8, criterion='ce', adversarial_temperature=1.0),
               dict(negatives=8, label_smoothing=0.1),                                  # smoothing with 'bce'
               dict(negatives=8, criterion='kl'),
               dict(negatives=8, criterion='ce', label_smoothing=-0.5),
               dict(negatives=8, criterion='ce', label_smoothing=float('nan'))):
        with pytest.raises(ValueError):
            k.GraphedTrainStep(None, None, None, kb, 4, **kw)
