"""Negative-sampled (1-vs-k) training on the GPU: the positive sampler, the fused sampled scoring + BCE kernels (K6s)
against the float64 restatements of tests/sampled_oracle.py, the bridge to the 1-N objective, MGCN.loss_sampled and
GraphedTrainStep(negatives=k) on data/Toy, and ConvE's fc layer above 128 queries."""
import copy
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import mgcn_oracle as orc
import sampled_oracle as so

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def k():
    import kgc_gcn_b200
    assert torch.cuda.is_available()
    kgc_gcn_b200._lib.lib()
    return kgc_gcn_b200


def test_positives_match_oracle(k):
    """KBDataset.positives is bit-exact against the restatement for the caller's draws (empty lists give -1) and only
    ever returns known objects when it draws from torch's generator."""
    rng = np.random.default_rng(5)
    N, Q, P = 1000, 80, 7
    qs = [{'triple': (0, 0, -1), 'label': sorted(set(rng.integers(0, N, int(rng.integers(0, 12))).tolist()))}
          for _ in range(Q)]
    qs[3]['label'] = []
    kb = k.KBDataset(qs, N, None, training=True)
    qid = rng.permutation(Q)[:41]
    qid[0] = 3
    draws = rng.integers(0, 2 ** 32, (41, P), dtype=np.uint64)
    draws[1, 0], draws[1, 1] = 0, 2 ** 32 - 1
    got = kb.positives(qid, P, draws=torch.from_numpy(draws.astype(np.int64))).cpu().numpy()
    np.testing.assert_array_equal(got, so.pos_sample([q['label'] for q in qs], qid, draws))
    drawn = kb.positives(qid, P).cpu().numpy()
    for b in range(41):
        lst = qs[int(qid[b])]['label']
        assert set(drawn[b].tolist()) <= (set(lst) if lst else {-1})


def _case(B, C, N, D, n_pos, strided, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, D, generator=g)
    ent = torch.randn(N, D, generator=g) * (2.0 / D ** 0.5)
    bias = torch.randn(N, generator=g) * 0.1
    cand = torch.randint(0, N, (B, C), generator=g, dtype=torch.int32)
    cand[0, 0] = -1                                       # empty positive slot
    cand[1, :n_pos] = -1                                  # a query without positives
    cand[2, C - 1] = -1                                   # empty negative slot
    cand[3, :] = cand[3, 0]                               # one entity in every slot
    cand[4:, 0] = cand[5, 0]                              # an entity shared by many queries
    ent_d = ent.cuda()
    if strided:                                           # rows inside a wider table (pitch D + 12)
        wide = torch.full((N, D + 12), float('nan'), device='cuda')
        wide[:, :D] = ent_d
        ent_d = wide[:, :D]
    return x, ent, bias, cand, ent_d


@pytest.mark.parametrize('B,C,N,D,n_pos,strided,smooth', [
    (96, 65, 50, 200, 1, False, 0.0),      # k = 64 negatives over 50 entities: heavy duplicates
    (40, 19, 3000, 200, 3, True, 0.1),     # n_pos > 1, strided all_ent, label smoothing
    (70, 33, 400, 100, 2, False, 0.0),
    (37, 12, 90, 4, 1, True, 0.0),
])
def test_sampled_bce_matches_float64(k, B, C, N, D, n_pos, strided, smooth):
    """Loss within 1e-6 relative, d_x / d_all_ent / d_bias (and the logit gradient) within 1e-5 of their max-norm
    against float64; the upstream scalar is applied; two runs bit-identical."""
    x, ent, bias, cand, ent_d = _case(B, C, N, D, n_pos, strided, B + C + N + D)
    pos, add = (float(np.float32(1.0 - smooth) + np.float32(1.0 / N)), float(np.float32(1.0 / N))) if smooth else (1.0, 0.0)
    outs = []
    for _ in range(2):
        xg = x.cuda().requires_grad_(True)
        eg = ent_d.detach().clone() if not strided else ent_d.detach()
        eg.requires_grad_(True)
        bg = bias.cuda().requires_grad_(True)
        loss = k.score_sampled_bce(xg, eg, bg, cand.cuda(), n_pos, pos, add)
        (loss * 2.5).backward()
        torch.cuda.synchronize()
        outs.append([loss.detach().cpu(), xg.grad.cpu(), eg.grad.cpu(), bg.grad.cpu()])
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    loss, d_x, d_ent, d_bias = outs[0]
    r_loss, r_g, r_x, r_ent, r_bias = so.sampled_bce(x, ent, bias, cand, n_pos, pos, add)
    assert abs(float(loss) - float(r_loss)) <= 1e-6 * abs(float(r_loss)), (float(loss), float(r_loss))
    for got, ref, name in ((d_x, 2.5 * r_x, 'd_x'), (d_ent, 2.5 * r_ent, 'd_ent'), (d_bias, 2.5 * r_bias, 'd_bias')):
        err = float((got.double() - ref).abs().max()) / float(ref.abs().max())
        assert err <= 1e-5, (name, err)
    assert tuple(d_ent.shape) == (N, D)
    untouched = torch.ones(N, dtype=torch.bool)
    untouched[cand[cand >= 0].long()] = False
    assert float(d_ent[untouched].abs().sum()) == 0.0 and float(d_bias[untouched].abs().sum()) == 0.0


def test_sampled_bce_logit_gradient_through_the_c_abi(k):
    """kgc_sampled_bce_fwd's g [B, C] and valid-slot count against float64 (0 on empty slots)."""
    B, C, N, D, n_pos = 50, 21, 60, 200, 2
    x, ent, bias, cand, _ = _case(B, C, N, D, n_pos, False, 7)
    L, p = k._lib, k._lib.ptr
    xd, ed, bd, cd = x.cuda(), ent.cuda(), bias.cuda(), cand.cuda()
    g = torch.full((B, C), float('nan'), device='cuda')
    d_x = torch.empty((B, D), device='cuda')
    count = torch.full((1,), -7, dtype=torch.int32, device='cuda')
    partial = torch.empty((int(L.lib().kgc_sampled_bce_fwd_blocks(B)),), dtype=torch.float64, device='cuda')
    loss = torch.empty((1,), device='cuda')
    L.call('kgc_sampled_bce_fwd', p(xd), B, D, p(ed), N, D, p(bd), p(cd), C, n_pos, 1.0, 0.0, p(g), p(d_x), p(count),
           p(partial), p(loss), L.stream())
    torch.cuda.synchronize()
    assert int(count) == int((cand >= 0).sum())
    _, r_g, _, _, _ = so.sampled_bce(x, ent, bias, cand, n_pos)
    assert float((g.cpu().double() - r_g).abs().max()) <= 1e-5 * float(r_g.abs().max())
    assert float(g.cpu()[cand < 0].abs().sum()) == 0.0


def test_sampled_bce_equals_1n_when_every_entity_is_a_candidate(k):
    """Bridge to the existing objective: with each query's candidates = its one positive + every other entity,
    score_sampled_bce is score_1n_bce (loss within 1e-6, gradients within 1e-5 of their max-norm)."""
    from kgc_gcn_b200.scoring import score_1n_bce
    B, N, D = 48, 1000, 200
    g = torch.Generator().manual_seed(3)
    x = torch.randn(B, D, generator=g).cuda()
    ent = (torch.randn(N, D, generator=g) * 0.14).cuda()
    bias = (torch.randn(N, generator=g) * 0.1).cuda()
    obj = torch.randint(0, N, (B,), generator=g)
    rest = torch.arange(N).expand(B, N)
    others = rest[rest != obj[:, None]].view(B, N - 1)
    cand = torch.cat([obj[:, None], others], 1).to(torch.int32).cuda()
    ptr = torch.arange(B + 1, dtype=torch.int64).cuda()
    idx = obj.to(torch.int32).cuda()
    qid = torch.arange(B, dtype=torch.int64).cuda()
    res = {}
    for name in ('sampled', '1n'):
        xg, eg, bg = (t.clone().requires_grad_(True) for t in (x, ent, bias))
        if name == 'sampled':
            loss = k.score_sampled_bce(xg, eg, bg, cand, 1)
        else:
            loss = score_1n_bce(xg, eg, bg, qid, ptr, idx)
        loss.backward()
        res[name] = (float(loss), xg.grad, eg.grad, bg.grad)
    a, b = res['sampled'], res['1n']
    assert abs(a[0] - b[0]) <= 1e-6 * abs(b[0]), (a[0], b[0])
    for ga, gb, name in zip(a[1:], b[1:], ('d_x', 'd_ent', 'd_bias')):
        err = float((ga - gb).abs().max()) / float(gb.abs().max())
        assert err <= 1e-5, (name, err)


def test_score_sampled_bce_rejects_bad_ids(k):
    x, ent, bias = torch.zeros(3, 8, device='cuda'), torch.zeros(10, 8, device='cuda'), torch.zeros(10, device='cuda')
    cand = torch.zeros(3, 4, dtype=torch.int32, device='cuda')
    cand[2, 3] = 10
    with pytest.raises(ValueError):
        k.score_sampled_bce(x, ent, bias, cand, 1)
    with pytest.raises(RuntimeError):
        k.score_sampled_bce(x, ent.cpu(), bias, cand, 1)


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


def test_loss_sampled_matches_dense_route_toy(k, toy):
    """MGCN.loss_sampled == BCELoss(model(src, rel, graph).gather(1, cand), target) over the valid slots, with cand =
    [positives | negatives] as the oracle samplers give them for the same draws: loss within 1e-6, every parameter gradient
    at the bar of test_loss_sparse_matches_dense_route.  (No label smoothing here: at N = 7 the smoothed positive label is
    0.9 + 1/7 > 1, which torch's BCELoss refuses; smoothing is covered against float64 above.)"""
    dl, m0 = toy
    ds = dl._get_dataset('train', _params())
    N = ds.num_entity
    qid = np.arange(1, len(ds))                           # the Toy training set has 17 queries
    B, P, K, TR = len(qid), 2, 9, 3
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
            pred = m(trip[:, 0], trip[:, 1], dl.graph)
            c = torch.from_numpy(cand).long().cuda()
            valid = c >= 0
            target = torch.full(c.shape, add, device='cuda')
            target[:, :P] = pos
            loss = torch.nn.BCELoss()(pred.gather(1, c.clamp_min(0))[valid], target[valid])
        else:
            draws = (torch.from_numpy(pd.astype(np.int64)), torch.from_numpy(nd.astype(np.int64)))
            loss = m.loss_sampled(qid, ds, dl.graph, K, n_pos=P, tries=TR, draws=draws)
        loss.backward()
        losses[mode] = float(loss.item())
        grads[mode] = {n: p.grad.detach().clone() for n, p in m.named_parameters() if p.grad is not None}
    assert abs(losses['dense'] - losses['sampled']) <= 1e-6 * abs(losses['dense']), losses
    assert grads['dense'].keys() == grads['sampled'].keys()
    top = max(float(g.abs().max()) for g in grads['dense'].values())
    for n, g in grads['dense'].items():
        assert float((g - grads['sampled'][n]).abs().max()) <= 1e-5 * float(g.abs().max()) + 1e-6 * top, n


def test_graphed_train_step_negatives_matches_eager_toy(k, toy):
    """GraphedTrainStep(negatives=k): each replay equals the eager loss_sampled step on the same draws and query ids;
    a ragged last batch runs eagerly."""
    dl, m0 = toy
    ds = dl._get_dataset('train', _params())
    qids = [list(range(0, 16)), list(range(1, 17)), list(range(0, 16)), list(range(16, 0, -1))]     # 17 Toy queries
    K = 12
    m_g, m_e = copy.deepcopy(m0).train(), copy.deepcopy(m0).train()
    opt_g = k.ClipAdam(m_g.parameters(), lr=1e-2, max_norm=1.0)
    opt_e = k.ClipAdam(m_e.parameters(), lr=1e-2, max_norm=1.0)
    gen = torch.Generator(device='cuda').manual_seed(11)
    step = k.GraphedTrainStep(m_g, opt_g, dl.graph, ds, 16, warmup=0, negatives=K, generator=gen)
    for q in qids:
        lg = float(step(q).item())
        draws = (step.pos_draws.clone(), step.neg_draws.clone())
        opt_e.zero_grad(set_to_none=True)
        le = m_e.loss_sampled(q, ds, dl.graph, K, draws=draws)
        le.backward()
        opt_e.step()
        assert abs(lg - float(le)) <= 1e-5 * max(1.0, abs(float(le))), (lg, float(le))
    for (n, a), b in zip(m_g.named_parameters(), m_e.parameters()):
        assert float((a - b).abs().max()) <= 1e-5 * max(1.0, float(b.abs().max())), n
    ragged = float(step(list(range(3, 13))).item())
    assert np.isfinite(ragged) and ragged > 0.0


@pytest.mark.parametrize('B', [129, 512, 4096])
def test_linear_tc_above_128_rows(k, B):
    """ConvE's fc layer at B > 128 (tiles of 128 rows, d_W in 256-row chunks added in order) within the bar of
    test_linear_tc_fc_layer against float64; deterministic."""
    F, O = 39200, 200
    g = torch.Generator().manual_seed(B)
    x = torch.randn(B, F, generator=g).cuda().requires_grad_(True)
    w = (torch.randn(O, F, generator=g) * 0.01).cuda().requires_grad_(True)
    b = (torch.randn(O, generator=g) * 0.1).cuda().requires_grad_(True)
    dy = torch.randn(B, O, generator=g).cuda()
    assert k.linear_tc_supported(x, w)
    y = k.linear_tc(x, w, b)
    y.backward(dy)
    xd, wd, bd = (t.detach().double().requires_grad_(True) for t in (x, w, b))
    (xd @ wd.t() + bd).backward(dy.double())
    yd = xd.detach() @ wd.detach().t() + bd.detach()
    for got, ref, name in ((y.detach(), yd, 'y'), (x.grad, xd.grad, 'dx'), (w.grad, wd.grad, 'dw'), (b.grad, bd.grad, 'db')):
        err = float((got.double() - ref).abs().max()) / float(ref.abs().max())
        assert err <= 4e-6, (name, err)
    x2, w2, b2 = (t.detach().clone().requires_grad_(True) for t in (x, w, b))
    y2 = k.linear_tc(x2, w2, b2)
    y2.backward(dy)
    assert torch.equal(y2, y) and torch.equal(x2.grad, x.grad) and torch.equal(w2.grad, w.grad)


@pytest.mark.parametrize('B', [77, 128])
def test_linear_tc_up_to_128_rows_is_one_launch_each(k, B):
    """Up to 128 rows linear_tc is the single split-K forward and the two single transposed-operand launches it always
    was: bit-identical to calling those kernels directly."""
    F, O = 39200, 200
    g = torch.Generator().manual_seed(B + 1)
    x = torch.randn(B, F, generator=g).cuda().requires_grad_(True)
    w = (torch.randn(O, F, generator=g) * 0.01).cuda().requires_grad_(True)
    dy = torch.randn(B, O, generator=g).cuda()
    y = k.linear_tc(x, w)
    y.backward(dy)
    y0 = k.gemm_nt_splitk(x.detach(), w.detach(), torch.empty((B, O), device='cuda'))
    dx0 = k.gemm_nt_trans(w.detach(), dy.t(), torch.empty_like(x))
    dw0 = k.gemm_nt_trans(x.detach(), dy, torch.empty_like(w))
    assert torch.equal(y, y0) and torch.equal(x.grad, dx0) and torch.equal(w.grad, dw0)
