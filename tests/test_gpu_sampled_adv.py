"""Self-adversarial negative sampling on the GPU: kgc_sampled_adv_fwd + the shared table backward against the float64
restatement of tests/sampled_adv_oracle.py, its bridge to the plain sampled objective at alpha = 0, the hardest-negative
limit, MGCN.loss_sampled(adversarial_temperature=...) and GraphedTrainStep(negatives=k, adversarial_temperature=...)
on data/Toy."""
import copy
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import mgcn_oracle as orc
import sampled_adv_oracle as sa
import sampled_oracle as so

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def k():
    import kgc_gcn_b200
    assert torch.cuda.is_available()
    kgc_gcn_b200._lib.lib()
    return kgc_gcn_b200


def _case(B, C, N, D, n_pos, strided, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, D, generator=g)
    ent = torch.randn(N, D, generator=g) * (1.0 / D ** 0.5)       # logits of order 1: alpha * max|z| stays moderate
    bias = torch.randn(N, generator=g) * 0.1
    cand = torch.randint(0, N, (B, C), generator=g, dtype=torch.int32)
    cand[0, 0] = -1                                       # empty positive slot
    cand[1, :n_pos] = -1                                  # a query without positives
    cand[2, n_pos:] = -1                                  # a query whose negative slots are all empty
    cand[3, :] = cand[3, 0]                               # one entity in every slot
    cand[4, C - 1] = -1                                   # empty negative slot
    cand[5:, 0] = cand[6, 0]                              # an entity shared by many queries
    ent_d = ent.cuda()
    if strided:                                           # rows inside a wider table (pitch D + 12)
        wide = torch.full((N, D + 12), float('nan'), device='cuda')
        wide[:, :D] = ent_d
        ent_d = wide[:, :D]
    return x, ent, bias, cand, ent_d


def _max_logit(x, ent, bias, cand):
    c = cand.clamp_min(0).long()
    return float(((x.double()[:, None, :] * ent.double()[c]).sum(-1) + bias.double()[c]).abs().max())


def _run(k, x, ent_d, bias, cand, n_pos, pos, add, alpha, strided, upstream=2.5):
    xg = x.cuda().requires_grad_(True)
    eg = ent_d.detach() if strided else ent_d.detach().clone()
    eg.requires_grad_(True)
    bg = bias.cuda().requires_grad_(True)
    loss = k.score_sampled_bce(xg, eg, bg, cand.cuda(), n_pos, pos, add, adversarial_temperature=alpha)
    (loss * upstream).backward()
    torch.cuda.synchronize()
    return [loss.detach().cpu(), xg.grad.cpu(), eg.grad.cpu(), bg.grad.cpu()]


@pytest.mark.parametrize('alpha', [0.0, 0.5, 1.0, 4.0])
@pytest.mark.parametrize('B,C,N,D,n_pos,strided,smooth', [
    (96, 65, 50, 200, 1, False, 0.0),      # k = 64 negatives over 50 entities: heavy duplicates
    (40, 19, 3000, 200, 3, True, 0.1),     # n_pos > 1, strided all_ent, label smoothing
    (70, 33, 400, 100, 2, False, 0.0),
    (37, 12, 90, 4, 1, True, 0.0),
])
def test_sampled_adv_matches_float64(k, B, C, N, D, n_pos, strided, smooth, alpha):
    """Loss within 1e-6 relative, d_x / d_all_ent / d_bias within 1e-5 of their max-norm against float64; the upstream
    scalar is applied; two runs bit-identical."""
    x, ent, bias, cand, ent_d = _case(B, C, N, D, n_pos, strided, B + C + N + D)
    assert alpha * _max_logit(x, ent, bias, cand) <= 24.0
    pos, add = (float(np.float32(1.0 - smooth) + np.float32(1.0 / N)), float(np.float32(1.0 / N))) if smooth else (1.0, 0.0)
    outs = [_run(k, x, ent_d, bias, cand, n_pos, pos, add, alpha, strided) for _ in range(2)]
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    loss, d_x, d_ent, d_bias = outs[0]
    r_loss, _, r_x, r_ent, r_bias = sa.sampled_adv(x, ent, bias, cand, n_pos, alpha, pos, add)
    assert abs(float(loss) - float(r_loss)) <= 1e-6 * abs(float(r_loss)), (float(loss), float(r_loss))
    for got, ref, name in ((d_x, 2.5 * r_x, 'd_x'), (d_ent, 2.5 * r_ent, 'd_ent'), (d_bias, 2.5 * r_bias, 'd_bias')):
        err = float((got.double() - ref).abs().max()) / float(ref.abs().max())
        assert err <= 1e-5, (name, err)
    untouched = torch.ones(N, dtype=torch.bool)
    untouched[cand[cand >= 0].long()] = False
    assert float(d_ent[untouched].abs().sum()) == 0.0 and float(d_bias[untouched].abs().sum()) == 0.0


@pytest.mark.parametrize('alpha', [0.0, 1.0])
def test_sampled_adv_logit_gradient_and_counts_through_the_c_abi(k, alpha):
    """kgc_sampled_adv_fwd's g [B, C] (0 on empty slots) against float64, and counts = (Q+, Q-)."""
    B, C, N, D, n_pos = 50, 21, 60, 200, 2
    x, ent, bias, cand, _ = _case(B, C, N, D, n_pos, False, 7)
    cand[7, :] = -1                                       # a query without any valid slot
    L, p = k._lib, k._lib.ptr
    xd, ed, bd, cd = x.cuda(), ent.cuda(), bias.cuda(), cand.cuda()
    g = torch.full((B, C), float('nan'), device='cuda')
    d_x = torch.empty((B, D), device='cuda')
    counts = torch.full((2,), -7, dtype=torch.int32, device='cuda')
    partial = torch.empty((2 * int(L.lib().kgc_sampled_bce_fwd_blocks(B)),), dtype=torch.float64, device='cuda')
    loss = torch.empty((1,), device='cuda')
    L.call('kgc_sampled_adv_fwd', p(xd), B, D, p(ed), N, D, p(bd), p(cd), C, n_pos, 1.0, 0.0, alpha, p(g), p(d_x), p(counts),
           p(partial), p(loss), L.stream())
    torch.cuda.synchronize()
    valid = cand >= 0
    assert counts.cpu().tolist() == [int(valid[:, :n_pos].any(1).sum()), int(valid[:, n_pos:].any(1).sum())]
    r_loss, r_g, r_x, _, _ = sa.sampled_adv(x, ent, bias, cand, n_pos, alpha)
    assert float((g.cpu().double() - r_g).abs().max()) <= 1e-5 * float(r_g.abs().max())
    assert float(g.cpu()[~valid].abs().sum()) == 0.0
    assert float((d_x.cpu().double() - r_x).abs().max()) <= 1e-5 * float(r_x.abs().max())
    assert abs(float(loss) - float(r_loss)) <= 1e-6 * abs(float(r_loss))


def test_sampled_adv_c_abi_rejects_bad_temperature(k):
    L, p = k._lib, k._lib.ptr
    B, C, N, D = 4, 3, 10, 8
    t = {n: torch.zeros(s, device='cuda') for n, s in (('x', (B, D)), ('e', (N, D)), ('b', (N,)), ('g', (B, C)), ('dx', (B, D)))}
    cand = torch.zeros((B, C), dtype=torch.int32, device='cuda')
    counts = torch.zeros((2,), dtype=torch.int32, device='cuda')
    partial = torch.zeros((2 * int(L.lib().kgc_sampled_bce_fwd_blocks(B)),), dtype=torch.float64, device='cuda')
    loss = torch.zeros((1,), device='cuda')
    for alpha in (-1.0, float('nan'), float('inf')):
        with pytest.raises(RuntimeError):
            L.call('kgc_sampled_adv_fwd', p(t['x']), B, D, p(t['e']), N, D, p(t['b']), p(cand), C, 1, 1.0, 0.0, alpha,
                   p(t['g']), p(t['dx']), p(counts), p(partial), p(loss), L.stream())


@pytest.mark.parametrize('n_pos', [1, 3])
def test_sampled_adv_alpha_zero_bridge(k, n_pos):
    """alpha = 0 with the same numbers of valid positives and negatives in every query equals 1/2 of the two plain
    sampled losses over the positive and the negative columns (loss within 1e-6, gradients within 1e-5 of their
    max-norm)."""
    B, C, N, D = 64, 40, 500, 200
    x, ent, bias, _, _ = _case(B, C, N, D, n_pos, False, 21 + n_pos)
    g = torch.Generator().manual_seed(5)
    cand = torch.randint(0, N, (B, C), generator=g, dtype=torch.int32)
    cand[:, n_pos - 1] = -1                               # one empty positive and one empty negative slot per query
    cand[:, C - 2] = -1
    cand_d = cand.cuda()
    pos, add = 0.93, 0.01
    res = {}
    for name in ('adv', 'plain'):
        xg, eg, bg = (t.cuda().requires_grad_(True) for t in (x, ent, bias))
        if name == 'adv':
            loss = k.score_sampled_bce(xg, eg, bg, cand_d, n_pos, pos, add, adversarial_temperature=0.0)
        else:
            loss = 0.5 * (k.score_sampled_bce(xg, eg, bg, cand_d[:, :n_pos].contiguous(), n_pos, pos, add)
                          + k.score_sampled_bce(xg, eg, bg, cand_d[:, n_pos:].contiguous(), 0, pos, add))
        loss.backward()
        res[name] = (float(loss), xg.grad, eg.grad, bg.grad)
    a, b = res['adv'], res['plain']
    assert abs(a[0] - b[0]) <= 1e-6 * abs(b[0]), (a[0], b[0])
    for ga, gb, name in zip(a[1:], b[1:], ('d_x', 'd_ent', 'd_bias')):
        err = float((ga - gb).abs().max()) / float(gb.abs().max())
        assert err <= 1e-5, (name, err)


def test_sampled_adv_hardest_negative(k):
    """alpha = 50 with entity logits at least 1 apart: every other negative's weight is below e^-50, so the negative half
    is the mean over the queries of the top negative's BCE term, and the logit gradient sits on the top negative's slots.
    The logits stay in [-3, 2], away from the fp32 saturation of the BCE terms."""
    B, C, N, D = 30, 17, 6, 4
    x = torch.zeros(B, D)
    x[:, 0] = 1.0
    ent = torch.zeros(N, D)
    ent[:, 0] = torch.randperm(N, generator=torch.Generator().manual_seed(2)).float() - 3.0     # z = ent[:, 0]
    bias = torch.zeros(N)
    cand = torch.randint(0, N, (B, C), generator=torch.Generator().manual_seed(3), dtype=torch.int32)
    xg, eg, bg = x.cuda(), ent.cuda(), bias.cuda()
    loss = k.score_sampled_bce(xg, eg, bg, cand.cuda(), 1, adversarial_temperature=50.0)
    z = ent[:, 0].double()[cand.long()]
    top = z[:, 1:].max(1).values
    ref = 0.5 * float((-torch.nn.functional.logsigmoid(z[:, 0])).mean() + (-torch.nn.functional.logsigmoid(-top)).mean())
    assert abs(float(loss) - ref) <= 1e-6 * abs(ref), (float(loss), ref)
    _, r_g, _, _, _ = sa.sampled_adv(x, ent, bias, cand, 1, 50.0)
    L, p = k._lib, k._lib.ptr
    g = torch.empty((B, C), device='cuda')
    counts = torch.empty((2,), dtype=torch.int32, device='cuda')
    partial = torch.empty((2 * int(L.lib().kgc_sampled_bce_fwd_blocks(B)),), dtype=torch.float64, device='cuda')
    L.call('kgc_sampled_adv_fwd', p(xg), B, D, p(eg), N, D, p(bg), p(cand.cuda()), C, 1, 1.0, 0.0, 50.0, p(g),
           p(torch.empty((B, D), device='cuda')), p(counts), p(partial), p(torch.empty((1,), device='cuda')), L.stream())
    g = g.cpu().double()
    is_top = z == top[:, None]
    is_top[:, 0] = False
    assert float(g[:, 1:][~is_top[:, 1:]].abs().max()) <= 1e-12
    # the top slots of a query share sigmoid(top) / (2 B) (duplicates split it)
    top_sum = (g * is_top).sum(1)
    assert float((top_sum - torch.sigmoid(top) / (2 * B)).abs().max()) <= 1e-5 * float(top_sum.abs().max())
    assert float((g - r_g).abs().max()) <= 1e-5 * float(r_g.abs().max())


def _params(**kw):
    base = dict(gcn_in_dim=20, gcn_out_dim=200, gcn_drop=0.0, hidden_drop=0.0, feat_drop=0.0, k_w=10, k_h=20,
                num_filter=2, kernel_size=7, bias=False, lbl_smooth=0.0, batch_size=128)
    base.update(kw)
    return SimpleNamespace(**base)


@pytest.fixture(scope='module')
def toy(golden_dir, k):
    cwd = os.getcwd()
    os.chdir(golden_dir)
    try:
        dl = k.DataLoader('Toy', _params())
    finally:
        os.chdir(cwd)
    dl.graph.to('cuda')
    z = np.load(os.path.join(golden_dir, 'toy_model.npz'))
    m = k.MGCN(dl.num_entity, dl.num_relation, dl.num_edge, _params())
    m.load_state_dict({kk[3:]: torch.from_numpy(z[kk]) for kk in z.files if kk.startswith('sd.')}, strict=True)
    m.conv1.drop.p = 0.0
    return dl, m.cuda()


def _adv_coefficients(z, valid, n_pos, alpha):
    """BCELoss weights of the objective from the float64 logits z [B, C] of the candidate slots (detached)."""
    B, C = valid.shape
    is_pos = torch.zeros_like(valid)
    is_pos[:, :n_pos] = True
    vp, vn = valid & is_pos, valid & ~is_pos
    q_pos, q_neg = int(vp.any(1).sum()), int(vn.any(1).sum())
    coef = torch.zeros((B, C), dtype=torch.float64, device=z.device)
    for b in range(B):
        if vp[b].any():
            coef[b, vp[b]] = 1.0 / (2.0 * q_pos * int(vp[b].sum()))
        if vn[b].any():
            coef[b, vn[b]] = torch.softmax(alpha * z[b, vn[b]], 0) / (2.0 * q_neg)
    return coef


def test_loss_sampled_adversarial_matches_dense_route_toy(k, toy):
    """MGCN.loss_sampled(adversarial_temperature=1) == BCELoss(weight=c, reduction='sum') on model(src, rel,
    graph).gather(1, cand) over the valid slots, with the weights from float64 logits of the model's own query rows and
    entity table (detached) and cand = [positives | negatives] as the oracle samplers give them for the same draws: loss
    within 1e-6, every parameter gradient at the bar of test_loss_sampled_matches_dense_route_toy."""
    dl, m0 = toy
    ds = dl._get_dataset('train', _params())
    N = ds.num_entity
    qid = np.arange(1, len(ds))                           # the Toy training set has 17 queries
    B, P, K, TR = len(qid), 2, 9, 3
    alpha = 1.0
    rng = np.random.default_rng(1)
    pd = rng.integers(0, 2 ** 32, (B, P), dtype=np.uint64)
    nd = rng.integers(0, 2 ** 32, (B, K, TR), dtype=np.uint64)
    lists = [ds.idx[ds.ptr[q]:ds.ptr[q + 1]].tolist() for q in range(len(ds))]
    cand = np.concatenate([so.pos_sample(lists, qid, pd), orc.neg_sample(lists, qid, N, nd)], 1)
    pos, add = ds.label_values()
    grads, losses = {}, {}
    for mode in ('dense', 'sampled'):
        m = copy.deepcopy(m0).train()
        m.conv1.drop.p = 0.0
        if mode == 'dense':
            trip = torch.from_numpy(ds.triples[qid]).cuda()
            c = torch.from_numpy(cand).long().cuda()
            valid = c >= 0
            with torch.no_grad():
                all_ent, all_rel = m.encode(dl.graph)
                xq = m.conv2.query(all_ent.index_select(0, trip[:, 0]), all_rel.index_select(0, trip[:, 1]))
                z = (xq.double() @ all_ent.double().t() + m.conv2.bias.double()).gather(1, c.clamp_min(0))
            coef = _adv_coefficients(z, valid, P, alpha)
            pred = m(trip[:, 0], trip[:, 1], dl.graph)
            target = torch.full(c.shape, add, device='cuda')
            target[:, :P] = pos
            loss = torch.nn.BCELoss(weight=coef[valid].float(), reduction='sum')(pred.gather(1, c.clamp_min(0))[valid],
                                                                                 target[valid])
        else:
            draws = (torch.from_numpy(pd.astype(np.int64)), torch.from_numpy(nd.astype(np.int64)))
            loss = m.loss_sampled(qid, ds, dl.graph, K, n_pos=P, tries=TR, draws=draws, adversarial_temperature=alpha)
        loss.backward()
        losses[mode] = float(loss.item())
        grads[mode] = {n: p.grad.detach().clone() for n, p in m.named_parameters() if p.grad is not None}
    assert abs(losses['dense'] - losses['sampled']) <= 1e-6 * abs(losses['dense']), losses
    assert grads['dense'].keys() == grads['sampled'].keys()
    top = max(float(g.abs().max()) for g in grads['dense'].values())
    for n, g in grads['dense'].items():
        assert float((g - grads['sampled'][n]).abs().max()) <= 1e-5 * float(g.abs().max()) + 1e-6 * top, n


def test_graphed_train_step_adversarial_matches_eager_toy(k, toy):
    """GraphedTrainStep(negatives=k, adversarial_temperature=1): each replay equals the eager
    loss_sampled(adversarial_temperature=1) step on the same draws and query ids; a ragged last batch runs eagerly."""
    dl, m0 = toy
    ds = dl._get_dataset('train', _params())
    qids = [list(range(0, 16)), list(range(1, 17)), list(range(0, 16)), list(range(16, 0, -1))]     # 17 Toy queries
    K, alpha = 12, 1.0
    m_g, m_e = copy.deepcopy(m0).train(), copy.deepcopy(m0).train()
    opt_g = k.ClipAdam(m_g.parameters(), lr=1e-2, max_norm=1.0)
    opt_e = k.ClipAdam(m_e.parameters(), lr=1e-2, max_norm=1.0)
    gen = torch.Generator(device='cuda').manual_seed(11)
    step = k.GraphedTrainStep(m_g, opt_g, dl.graph, ds, 16, warmup=0, negatives=K, generator=gen,
                              adversarial_temperature=alpha)
    for q in qids:
        lg = float(step(q).item())
        draws = (step.pos_draws.clone(), step.neg_draws.clone())
        opt_e.zero_grad(set_to_none=True)
        le = m_e.loss_sampled(q, ds, dl.graph, K, draws=draws, adversarial_temperature=alpha)
        le.backward()
        opt_e.step()
        assert abs(lg - float(le)) <= 1e-5 * max(1.0, abs(float(le))), (lg, float(le))
    for (n, a), b in zip(m_g.named_parameters(), m_e.parameters()):
        assert float((a - b).abs().max()) <= 1e-5 * max(1.0, float(b.abs().max())), n
    ragged = float(step(list(range(3, 13))).item())
    assert np.isfinite(ragged) and ragged > 0.0
