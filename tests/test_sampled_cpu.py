"""Negative-sampled training, host side: the float64 restatements of tests/sampled_oracle.py against torch.nn.BCELoss +
autograd on the gathered probabilities, and the argument checks of the Python surface (no GPU needed)."""
import numpy as np
import pytest
import torch

import sampled_oracle as so


def _bce_autograd(x, ent, bias, cand, n_pos, pos, add):
    """torch.nn.BCELoss (mean) over the valid slots' probabilities, gradients by autograd, float64."""
    x, ent, bias = (t.clone().double().requires_grad_(True) for t in (x, ent, bias))
    cand = torch.as_tensor(cand).long()
    B, C = cand.shape
    valid = (cand >= 0) & (cand < ent.shape[0])
    col = torch.arange(C).expand(B, C)
    b_idx, e_idx = torch.nonzero(valid, as_tuple=True)
    ids = cand[b_idx, e_idx]
    prob = torch.sigmoid((x[b_idx] * ent[ids]).sum(1) + bias[ids])
    target = torch.where(col[b_idx, e_idx] < n_pos, torch.tensor(float(pos), dtype=torch.float64),
                         torch.tensor(float(add), dtype=torch.float64))
    loss = torch.nn.BCELoss()(prob, target)
    loss.backward()
    return loss.detach(), x.grad, ent.grad, bias.grad


@pytest.mark.parametrize('B,C,N,D,n_pos,smooth,seed', [
    (7, 9, 50, 8, 1, 0.0, 0),       # duplicates within and across queries
    (5, 70, 13, 4, 3, 0.1, 1),      # N < C: every query repeats entities; label smoothing
    (16, 6, 1000, 20, 2, 0.0, 2),
])
def test_sampled_bce_oracle_matches_bceloss(B, C, N, D, n_pos, smooth, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, D, generator=g)
    ent = torch.randn(N, D, generator=g) * 0.5
    bias = torch.randn(N, generator=g) * 0.1
    cand = torch.randint(0, N, (B, C), generator=g)
    cand[0, 0] = -1                                       # an empty positive slot
    cand[1, :n_pos] = -1                                  # a query without positives
    cand[2, C - 1] = -1                                   # an empty negative slot
    cand[3, :] = cand[3, 0]                               # one entity in every slot of a query
    pos, add = (float(np.float32(1.0 - smooth) + np.float32(1.0 / N)), float(np.float32(1.0 / N))) if smooth else (1.0, 0.0)
    loss, gl, d_x, d_ent, d_bias = so.sampled_bce(x, ent, bias, cand, n_pos, pos, add)
    r_loss, r_x, r_ent, r_bias = _bce_autograd(x, ent, bias, cand, n_pos, pos, add)
    assert abs(float(loss) - float(r_loss)) <= 1e-12 * abs(float(r_loss))
    for got, ref in ((d_x, r_x), (d_ent, r_ent), (d_bias, r_bias)):
        assert float((got - ref).abs().max()) <= 1e-12 * float(ref.abs().max())
    assert float(gl[cand < 0].abs().max()) == 0.0
    # the logit gradient is what the parameter gradients are built from
    c = cand.clamp_min(0).long()
    assert torch.allclose((gl[:, :, None] * ent.double()[c]).sum(1), d_x, rtol=0, atol=1e-15)


def test_sampled_bce_oracle_without_valid_slots():
    loss, gl, d_x, d_ent, d_bias = so.sampled_bce(torch.ones(2, 4), torch.ones(3, 4), torch.zeros(3),
                                                  torch.full((2, 5), -1), 1)
    assert float(loss) == 0.0 and float(gl.abs().sum()) == 0.0
    assert float(d_x.abs().sum()) == 0.0 and float(d_ent.abs().sum()) == 0.0 and float(d_bias.abs().sum()) == 0.0


def test_pos_sample_oracle():
    """Slot j is list[(u * len) >> 32]: u = 0 takes the first object, u = 2^32 - 1 the last; -1 for an empty list."""
    lists = [[3, 8, 9], [], [5]]
    draws = np.array([[0, 2 ** 32 - 1, 2 ** 31], [7, 7, 7], [123, 2 ** 32 - 1, 0]], dtype=np.uint64)
    out = so.pos_sample(lists, np.array([0, 1, 2]), draws)
    np.testing.assert_array_equal(out, [[3, 9, 8], [-1, -1, -1], [5, 5, 5]])
    rng = np.random.default_rng(0)
    big = [sorted(set(rng.integers(0, 100, 20).tolist())) for _ in range(4)]
    d = rng.integers(0, 2 ** 32, (4, 1000), dtype=np.uint64)
    out = so.pos_sample(big, np.arange(4), d)
    for b in range(4):
        assert set(out[b].tolist()) <= set(big[b])
        assert len(set(out[b].tolist())) == len(big[b])        # 1,000 draws reach every object of a 20-entry list


def test_score_sampled_bce_argument_errors():
    import kgc_gcn_b200 as k
    x, ent, bias = torch.zeros(3, 8), torch.zeros(10, 8), torch.zeros(10)
    cand = torch.zeros(3, 4, dtype=torch.int32)
    with pytest.raises(ValueError):
        k.score_sampled_bce(x, ent, bias, cand[:2], 1)                  # B mismatch
    with pytest.raises(ValueError):
        k.score_sampled_bce(x, ent[:, :4], bias, cand, 1)               # D mismatch
    with pytest.raises(ValueError):
        k.score_sampled_bce(x, ent, bias[:9], cand, 1)                  # bias length
    with pytest.raises(ValueError):
        k.score_sampled_bce(x[:, :6], ent[:, :6], bias, cand, 1)        # D % 4 != 0
    with pytest.raises(ValueError):
        k.score_sampled_bce(torch.zeros(3, 260), torch.zeros(10, 260), bias, cand, 1)   # D > 256
    with pytest.raises(ValueError):
        k.score_sampled_bce(x, ent, bias, cand, 5)                      # n_pos > C
    with pytest.raises(ValueError):
        k.score_sampled_bce(x, ent, bias, cand, -1)
    with pytest.raises(ValueError):
        k.score_sampled_bce(x, ent, bias, cand.long(), 1)               # int32 ids only
    with pytest.raises(ValueError):
        k.score_sampled_bce(x, ent, bias, cand.view(-1), 1)
    with pytest.raises(RuntimeError):
        k.score_sampled_bce(x, ent, bias, cand, 1)                      # CPU tensors: no fallback


def test_sampler_and_step_argument_errors():
    import kgc_gcn_b200 as k
    kb = k.KBDataset([{'triple': (0, 0, -1), 'label': [1, 2]}], 5, None, training=True)
    with pytest.raises(ValueError):
        kb.positives([0], 0)
    with pytest.raises(RuntimeError):
        kb.positives([0], 2, device='cpu')
    with pytest.raises(ValueError):
        k.GraphedTrainStep(None, None, None, kb, 4, negatives=8, fused_loss=True)
    with pytest.raises(ValueError):
        k.GraphedTrainStep(None, None, None, kb, 4, negatives=0)
