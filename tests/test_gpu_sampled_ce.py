"""Negative-sampled softmax cross-entropy on the GPU: kgc_sampled_ce_fwd + the shared table backward against the float64
restatement of tests/sampled_oracle.py, at ordinary and at large logits, its bridge to the 1vsAll cross-entropy,
MGCN.loss_sampled(criterion='ce') and GraphedTrainStep(negatives=k, criterion='ce') on data/Toy."""
import copy
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import mgcn_oracle as orc
import sampled_oracle as so

pytestmark = pytest.mark.gpu

SHAPES = [
    (96, 65, 50, 200, 1, False),       # k = 64 negatives over 50 entities: heavy duplicates
    (40, 19, 3000, 200, 3, True),      # n_pos > 1, strided all_ent
    (70, 33, 400, 100, 2, False),
    (37, 12, 90, 4, 1, True),
]


@pytest.fixture(scope='module')
def k():
    import kgc_gcn_b200
    assert torch.cuda.is_available()
    kgc_gcn_b200._lib.lib()
    return kgc_gcn_b200


def _slots(cand, n_pos):
    C = cand.shape[1]
    cand[0, 0] = -1                                       # empty positive slot
    cand[1, :n_pos] = -1                                  # a query without positives
    cand[2, n_pos:] = -1                                  # a query whose negative slots are all empty
    cand[3, :] = cand[3, 0]                               # one entity in every slot
    cand[4, C - 1] = -1                                   # empty negative slot
    cand[5:, 0] = cand[6, 0]                              # an entity shared by many queries
    return cand


def _case(B, C, N, D, n_pos, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, D, generator=g)
    ent = torch.randn(N, D, generator=g) * (1.0 / D ** 0.5)
    bias = torch.randn(N, generator=g) * 0.1
    cand = _slots(torch.randint(0, N, (B, C), generator=g, dtype=torch.int32), n_pos)
    return x, ent, bias, cand


def _large_case(B, C, N, D, n_pos, seed):
    """Integer-valued x, rows and bias (every logit exact in fp32) with logits of standard deviation ~75, so |z| reaches
    ~300; query 7's positive sits 450 above 0 and query 8's 450 below (zero rows, bias +-450), far from all negatives."""
    g = torch.Generator().manual_seed(seed)
    a = int(round((3.0 * 75.0 ** 2 / (4.0 * D)) ** 0.5))            # Var(x) = 4; Var(ent) = a (a + 1) / 3
    x = torch.randint(-3, 4, (B, D), generator=g).float()
    ent = torch.randint(-a, a + 1, (N, D), generator=g).float()
    bias = torch.randint(-2, 3, (N,), generator=g).float()
    cand = _slots(torch.randint(0, N - 2, (B, C), generator=g, dtype=torch.int32), n_pos)
    ent[N - 2:] = 0.0
    bias[N - 2], bias[N - 1] = 450.0, -450.0
    cand[7, 0], cand[8, 0] = N - 2, N - 1
    return x, ent, bias, cand


def _device_table(ent, strided):
    ent_d = ent.cuda()
    if strided:                                           # rows inside a wider table (pitch D + 12)
        wide = torch.full((ent.shape[0], ent.shape[1] + 12), float('nan'), device='cuda')
        wide[:, :ent.shape[1]] = ent_d
        ent_d = wide[:, :ent.shape[1]]
    return ent_d


def _run(k, x, ent_d, bias, cand, n_pos, eps, strided, upstream=2.5):
    xg = x.cuda().requires_grad_(True)
    eg = ent_d.detach() if strided else ent_d.detach().clone()
    eg.requires_grad_(True)
    bg = bias.cuda().requires_grad_(True)
    loss = k.score_sampled_ce(xg, eg, bg, cand.cuda(), n_pos, label_smoothing=eps)
    (loss * upstream).backward()
    torch.cuda.synchronize()
    return [loss.detach().cpu(), xg.grad.cpu(), eg.grad.cpu(), bg.grad.cpu()]


def _check(k, x, ent, bias, cand, n_pos, eps, strided):
    """Loss within 1e-6 relative, d_x / d_all_ent / d_bias within 1e-5 of their max-norm against float64 with the upstream
    scalar applied; two runs bit-identical; rows no slot names get exactly 0."""
    N = ent.shape[0]
    ent_d = _device_table(ent, strided)
    outs = [_run(k, x, ent_d, bias, cand, n_pos, eps, strided) for _ in range(2)]
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    loss, d_x, d_ent, d_bias = outs[0]
    for t in outs[0]:
        assert bool(torch.isfinite(t).all())
    r_loss, _, r_x, r_ent, r_bias = so.sampled_ce(x, ent, bias, cand, n_pos, eps)
    assert abs(float(loss) - float(r_loss)) <= 1e-6 * abs(float(r_loss)), (float(loss), float(r_loss))
    for got, ref, name in ((d_x, 2.5 * r_x, 'd_x'), (d_ent, 2.5 * r_ent, 'd_ent'), (d_bias, 2.5 * r_bias, 'd_bias')):
        err = float((got.double() - ref).abs().max()) / float(ref.abs().max())
        assert err <= 1e-5, (name, err)
    untouched = torch.ones(N, dtype=torch.bool)
    untouched[cand[cand >= 0].long()] = False
    assert float(d_ent[untouched].abs().sum()) == 0.0 and float(d_bias[untouched].abs().sum()) == 0.0


@pytest.mark.parametrize('eps', [0.0, 0.1])
@pytest.mark.parametrize('B,C,N,D,n_pos,strided', SHAPES)
def test_sampled_ce_matches_float64(k, B, C, N, D, n_pos, strided, eps):
    x, ent, bias, cand = _case(B, C, N, D, n_pos, B + C + N + D)
    _check(k, x, ent, bias, cand, n_pos, eps, strided)


@pytest.mark.parametrize('eps', [0.0, 0.1])
@pytest.mark.parametrize('B,C,N,D,n_pos,strided', SHAPES)
def test_sampled_ce_large_logits_match_float64(k, B, C, N, D, n_pos, strided, eps):
    x, ent, bias, cand = _large_case(B, C, N, D, n_pos, 3 * B + C)
    c = cand.clamp_min(0).long()
    z = (x.double()[:, None, :] * ent.double()[c]).sum(-1) + bias.double()[c]
    neg = z[:, n_pos:].masked_fill(cand[:, n_pos:] < 0, -float('inf')).max(1).values
    assert float(z[cand >= 0].abs().max()) >= 300.0
    assert float(z[7, 0] - neg[7]) >= 100.0 and float(neg[8] - z[8, 0]) >= 100.0
    _check(k, x, ent, bias, cand, n_pos, eps, strided)


@pytest.mark.parametrize('eps', [0.0, 0.1])
def test_sampled_ce_logit_gradient_through_the_c_abi(k, eps):
    """kgc_sampled_ce_fwd's g [B, C] (0 on empty slots), d_x, loss and count = P against float64."""
    B, C, N, D, n_pos = 50, 21, 60, 200, 2
    x, ent, bias, cand = _case(B, C, N, D, n_pos, 7)
    cand[9, :] = -1                                       # a query without any valid slot
    L, p = k._lib, k._lib.ptr
    xd, ed, bd, cd = x.cuda(), ent.cuda(), bias.cuda(), cand.cuda()
    g = torch.full((B, C), float('nan'), device='cuda')
    d_x = torch.empty((B, D), device='cuda')
    count = torch.full((1,), -7, dtype=torch.int32, device='cuda')
    partial = torch.empty((int(L.lib().kgc_sampled_bce_fwd_blocks(B)),), dtype=torch.float64, device='cuda')
    loss = torch.empty((1,), device='cuda')
    L.call('kgc_sampled_ce_fwd', p(xd), B, D, p(ed), N, D, p(bd), p(cd), C, n_pos, eps, p(g), p(d_x), p(count),
           p(partial), p(loss), L.stream())
    torch.cuda.synchronize()
    valid = cand >= 0
    assert int(count) == int(valid[:, :n_pos].sum())
    r_loss, r_g, r_x, _, _ = so.sampled_ce(x, ent, bias, cand, n_pos, eps)
    assert float((g.cpu().double() - r_g).abs().max()) <= 1e-5 * float(r_g.abs().max())
    assert float(g.cpu()[~valid].abs().sum()) == 0.0
    assert float(g.cpu()[2].abs().sum()) == 0.0           # positives without negatives
    assert float((d_x.cpu().double() - r_x).abs().max()) <= 1e-5 * float(r_x.abs().max())
    assert abs(float(loss) - float(r_loss)) <= 1e-6 * abs(float(r_loss))


def test_sampled_ce_c_abi_rejects_bad_arguments(k):
    L, p = k._lib, k._lib.ptr
    B, C, N, D = 4, 3, 10, 8
    t = {n: torch.zeros(s, device='cuda') for n, s in (('x', (B, D)), ('e', (N, D)), ('b', (N,)), ('g', (B, C)), ('dx', (B, D)))}
    cand = torch.zeros((B, C), dtype=torch.int32, device='cuda')
    count = torch.zeros((1,), dtype=torch.int32, device='cuda')
    partial = torch.zeros((int(L.lib().kgc_sampled_bce_fwd_blocks(B)),), dtype=torch.float64, device='cuda')
    loss = torch.zeros((1,), device='cuda')

    def call(n_pos, eps):
        L.call('kgc_sampled_ce_fwd', p(t['x']), B, D, p(t['e']), N, D, p(t['b']), p(cand), C, n_pos, eps, p(t['g']),
               p(t['dx']), p(count), p(partial), p(loss), L.stream())
    for eps in (-0.1, 1.5, float('nan'), float('inf')):
        with pytest.raises(RuntimeError, match='label smoothing'):
            call(1, eps)
    for n_pos in (-1, C + 1):
        with pytest.raises(RuntimeError, match='n_pos'):
            call(n_pos, 0.1)
    call(C, 1.0)                                          # the ends of both ranges are taken
    call(0, 0.0)
    torch.cuda.synchronize()
    assert float(loss) == 0.0                             # no positive slot: P = 0


@pytest.mark.parametrize('eps', [0.0, 0.1])
def test_sampled_ce_one_vs_all_bridge(k, eps):
    """cand[b] = [o_b, every entity but o_b]: the loss is F.cross_entropy(x @ E^T + bias, o, label_smoothing=eps) in
    float64 (within 1e-6), and so are the gradients (within 1e-5 of their max-norm)."""
    B, N, D = 16, 3001, 200
    g = torch.Generator().manual_seed(31)
    x = torch.randn(B, D, generator=g)
    ent = torch.randn(N, D, generator=g) * (2.0 / D ** 0.5)
    bias = torch.randn(N, generator=g) * 0.1
    o = torch.randint(0, N, (B,), generator=g)
    ids = torch.arange(N).expand(B, N)
    rest = ids[ids != o[:, None]].view(B, N - 1)
    cand = torch.cat([o[:, None], rest], 1).to(torch.int32)
    xg, eg, bg = (t.cuda().requires_grad_(True) for t in (x, ent, bias))
    loss = k.score_sampled_ce(xg, eg, bg, cand.cuda(), 1, label_smoothing=eps)
    loss.backward()
    xr, er, br = (t.double().requires_grad_(True) for t in (x, ent, bias))
    ref = F.cross_entropy(xr @ er.t() + br, o, label_smoothing=eps)
    ref.backward()
    assert abs(float(loss) - float(ref)) <= 1e-6 * abs(float(ref)), (float(loss), float(ref))
    for got, r, name in ((xg.grad, xr.grad, 'd_x'), (eg.grad, er.grad, 'd_ent'), (bg.grad, br.grad, 'd_bias')):
        err = float((got.cpu().double() - r).abs().max()) / float(r.abs().max())
        assert err <= 1e-5, (name, err)


def _params(**kw):
    base = dict(gcn_in_dim=20, gcn_out_dim=200, gcn_drop=0.0, hidden_drop=0.0, feat_drop=0.0, k_w=10, k_h=20,
                num_filter=2, kernel_size=7, bias=False, lbl_smooth=0.1, batch_size=128)
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


@pytest.mark.parametrize('eps', [0.0, 0.1])
def test_loss_sampled_ce_matches_dense_route_toy(k, toy, eps):
    """MGCN.loss_sampled(criterion='ce') == F.cross_entropy(label_smoothing=eps) over the rows [z_p, z_negatives] of the
    dense route's logits (encode, ConvE's query, addmm with the entity table) gathered at cand = [positives | negatives]
    as the oracle samplers give them for the same draws: loss within 1e-6, every parameter gradient at the bar of
    test_loss_sampled_matches_dense_route_toy.  The dataset's lbl_smooth (0.1 here) does not enter."""
    dl, m0 = toy
    ds = dl._get_dataset('train', _params())
    N = ds.num_entity
    qid = np.arange(1, len(ds))                           # the Toy training set has 17 queries
    B, P, K, TR = len(qid), 2, 9, 3
    rng = np.random.default_rng(2)
    pd = rng.integers(0, 2 ** 32, (B, P), dtype=np.uint64)
    nd = rng.integers(0, 2 ** 32, (B, K, TR), dtype=np.uint64)
    lists = [ds.idx[ds.ptr[q]:ds.ptr[q + 1]].tolist() for q in range(len(ds))]
    cand = np.concatenate([so.pos_sample(lists, qid, pd), orc.neg_sample(lists, qid, N, nd)], 1)
    grads, losses = {}, {}
    for mode in ('dense', 'sampled'):
        m = copy.deepcopy(m0).train()
        m.conv1.drop.p = 0.0
        if mode == 'dense':
            trip = torch.from_numpy(ds.triples[qid]).cuda()
            c = torch.from_numpy(cand).long().cuda()
            all_ent, all_rel = m.encode(dl.graph)
            xq = m.conv2.query(all_ent.index_select(0, trip[:, 0]), all_rel.index_select(0, trip[:, 1]))
            z = torch.addmm(m.conv2.bias, xq, all_ent.t()).gather(1, c.clamp_min(0))
            total, rows = 0.0, 0
            for b in range(B):
                neg = [j for j in range(P, P + K) if c[b, j] >= 0]
                for p in range(P):
                    if c[b, p] < 0:
                        continue
                    row = torch.cat([z[b, p:p + 1], z[b, neg]])
                    total = total + F.cross_entropy(row[None], torch.zeros(1, dtype=torch.long, device='cuda'),
                                                    label_smoothing=eps, reduction='sum')
                    rows += 1
            loss = total / rows
        else:
            draws = (torch.from_numpy(pd.astype(np.int64)), torch.from_numpy(nd.astype(np.int64)))
            loss = m.loss_sampled(qid, ds, dl.graph, K, n_pos=P, tries=TR, draws=draws, criterion='ce',
                                  label_smoothing=eps)
        loss.backward()
        losses[mode] = float(loss.item())
        grads[mode] = {n: p.grad.detach().clone() for n, p in m.named_parameters() if p.grad is not None}
    assert abs(losses['dense'] - losses['sampled']) <= 1e-6 * abs(losses['dense']), losses
    assert grads['dense'].keys() == grads['sampled'].keys()
    top = max(float(g.abs().max()) for g in grads['dense'].values())
    for n, g in grads['dense'].items():
        assert float((g - grads['sampled'][n]).abs().max()) <= 1e-5 * float(g.abs().max()) + 1e-6 * top, n


def test_graphed_train_step_ce_matches_eager_toy(k, toy):
    """GraphedTrainStep(negatives=k, criterion='ce', label_smoothing=0.1): each replay equals the eager
    loss_sampled(criterion='ce', label_smoothing=0.1) step on the same draws and query ids; a ragged last batch runs
    eagerly."""
    dl, m0 = toy
    ds = dl._get_dataset('train', _params())
    qids = [list(range(0, 16)), list(range(1, 17)), list(range(0, 16)), list(range(16, 0, -1))]     # 17 Toy queries
    K, eps = 12, 0.1
    m_g, m_e = copy.deepcopy(m0).train(), copy.deepcopy(m0).train()
    opt_g = k.ClipAdam(m_g.parameters(), lr=1e-2, max_norm=1.0)
    opt_e = k.ClipAdam(m_e.parameters(), lr=1e-2, max_norm=1.0)
    gen = torch.Generator(device='cuda').manual_seed(11)
    step = k.GraphedTrainStep(m_g, opt_g, dl.graph, ds, 16, warmup=0, negatives=K, generator=gen, criterion='ce',
                              label_smoothing=eps)
    for q in qids:
        lg = float(step(q).item())
        draws = (step.pos_draws.clone(), step.neg_draws.clone())
        opt_e.zero_grad(set_to_none=True)
        le = m_e.loss_sampled(q, ds, dl.graph, K, draws=draws, criterion='ce', label_smoothing=eps)
        le.backward()
        opt_e.step()
        assert abs(lg - float(le)) <= 1e-5 * max(1.0, abs(float(le))), (lg, float(le))
    for (n, a), b in zip(m_g.named_parameters(), m_e.parameters()):
        assert float((a - b).abs().max()) <= 1e-5 * max(1.0, float(b.abs().max())), n
    ragged = float(step(list(range(3, 13))).item())
    assert np.isfinite(ragged) and ragged > 0.0
