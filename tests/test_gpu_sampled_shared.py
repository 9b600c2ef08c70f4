"""Batch-shared negatives for the sampled 1-vs-k losses on the GPU: score_shared_bce (plain and self-adversarial) and
score_shared_ce against the float64 restatement of tests/sampled_oracle.py on the broadcast candidate matrix
[pos_cand[b] | shared with query b's known objects set to -1], against the per-query kernels on the same matrix, the
filter mask through the C ABI, determinism, MGCN.loss_sampled(shared_negatives=True) and the graphed step on data/Toy."""
import copy
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import sampled_oracle as so

pytestmark = pytest.mark.gpu

# B, k, N, D, n_pos
SHAPES = [
    (96, 64, 50, 200, 1),          # heavy duplicates in shared
    (300, 200, 400, 100, 3),       # B over two query tiles (not a multiple of one), k not a multiple of 128, n_pos > 1
    (70, 130, 3000, 200, 2),
]
LOSSES = [('bce', None), ('bce', 0.0), ('bce', 1.0), ('bce', 4.0), ('ce', 0.0), ('ce', 0.1)]


@pytest.fixture(scope='module')
def k():
    import kgc_gcn_b200
    assert torch.cuda.is_available()
    kgc_gcn_b200._lib.lib()
    return kgc_gcn_b200


def _csr(lists):
    ptr = np.zeros(len(lists) + 1, dtype=np.int64)
    ptr[1:] = np.cumsum([len(l) for l in lists])
    idx = np.concatenate([np.asarray(l, dtype=np.int32) for l in lists]) if ptr[-1] else np.zeros(0, np.int32)
    return torch.from_numpy(ptr), torch.from_numpy(idx)


def _case(B, K, N, D, n_pos, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, D, generator=g) * scale
    ent = torch.randn(N, D, generator=g) * (1.0 / D ** 0.5)
    bias = torch.randn(N, generator=g) * 0.1
    shared = torch.randint(0, N, (K,), generator=g, dtype=torch.int32)
    n_q = B + 5
    rng = np.random.default_rng(seed)
    lists = [sorted(set(rng.integers(0, N, int(rng.integers(0, 6))).tolist())) for _ in range(n_q)]
    sh = shared.tolist()
    lists[3] = sorted(set(lists[3]) | set(sh[:5]))        # shared ids that are known objects of some queries
    lists[4] = sorted(set(sh))                            # a query whose shared negatives are all filtered
    qid = torch.from_numpy(rng.integers(0, n_q, B)).long()
    qid[0], qid[1] = 3, 4
    ptr, idx = _csr(lists)
    pos = torch.randint(0, N, (B, n_pos), generator=g, dtype=torch.int32)
    pos[2, :] = -1                                        # a query without positives
    pos[5, 0] = -1
    return x, ent, bias, pos, shared, qid, ptr, idx


def _oracle(kind, opt, x, ent, bias, cand, n_pos):
    if kind == 'ce':
        return so.sampled_ce(x, ent, bias, cand, n_pos, opt)
    if opt is None:
        return so.sampled_bce(x, ent, bias, cand, n_pos, 1.0, 0.0)
    return so.sampled_adv(x, ent, bias, cand, n_pos, opt, 1.0, 0.0)


def _run_shared(k, kind, opt, x, ent, bias, pos, shared, qid, ptr, idx, upstream=2.5):
    xg, eg, bg = (t.cuda().requires_grad_(True) for t in (x, ent, bias))
    args = (xg, eg, bg, pos.cuda(), shared.cuda(), qid.cuda(), ptr.cuda(), idx.cuda())
    if kind == 'ce':
        loss = k.score_shared_ce(*args, label_smoothing=opt)
    else:
        loss = k.score_shared_bce(*args, adversarial_temperature=opt)
    (loss * upstream).backward()
    torch.cuda.synchronize()
    return [loss.detach().cpu(), xg.grad.cpu(), eg.grad.cpu(), bg.grad.cpu()]


def _run_per_query(k, kind, opt, x, ent, bias, cand, n_pos, upstream=2.5):
    xg, eg, bg = (t.cuda().requires_grad_(True) for t in (x, ent, bias))
    if kind == 'ce':
        loss = k.score_sampled_ce(xg, eg, bg, cand.cuda(), n_pos, label_smoothing=opt)
    else:
        loss = k.score_sampled_bce(xg, eg, bg, cand.cuda(), n_pos, adversarial_temperature=opt)
    (loss * upstream).backward()
    torch.cuda.synchronize()
    return [loss.detach().cpu(), xg.grad.cpu(), eg.grad.cpu(), bg.grad.cpu()]


def _close(got, ref, upstream=2.5):
    loss, d_x, d_ent, d_bias = got
    r_loss, r_x, r_ent, r_bias = ref
    assert abs(float(loss) - float(r_loss)) <= 1e-6 * abs(float(r_loss)), (float(loss), float(r_loss))
    for g, r, name in ((d_x, upstream * r_x, 'd_x'), (d_ent, upstream * r_ent, 'd_ent'), (d_bias, upstream * r_bias, 'd_bias')):
        err = float((g.double() - r.double()).abs().max()) / float(r.double().abs().max())
        assert err <= 1e-5, (name, err)


def _check(k, kind, opt, case):
    x, ent, bias, pos, shared, qid, ptr, idx = case
    n_pos = pos.shape[1]
    cand = k.scoring.shared_candidates(pos, shared, qid, ptr, idx)
    runs = [_run_shared(k, kind, opt, *case) for _ in range(2)]
    for a, b in zip(*runs):
        assert torch.equal(a, b)                          # repeat calls are bit-identical
    for t in runs[0]:
        assert bool(torch.isfinite(t).all())
    r_loss, _, r_x, r_ent, r_bias = _oracle(kind, opt, x, ent, bias, cand, n_pos)
    _close(runs[0], (r_loss, r_x, r_ent, r_bias))
    return cand


@pytest.mark.parametrize('kind,opt', LOSSES)
@pytest.mark.parametrize('B,K,N,D,n_pos', SHAPES)
def test_shared_matches_float64(k, B, K, N, D, n_pos, kind, opt):
    cand = _check(k, kind, opt, _case(B, K, N, D, n_pos, B + K + N + D))
    assert bool((cand[1, n_pos:] == -1).all())            # the all-filtered query
    assert bool((cand[0, n_pos:] == -1).any())


@pytest.mark.parametrize('opt', [0.0, 0.1])
def test_shared_ce_large_logits_match_float64(k, opt):
    """Logits beyond 300 in magnitude: the log-sum-exp runs against each query's max.  Integer-valued x, rows and bias,
    so every logit is exact in fp32 and under the 3xTF32 split."""
    case = list(_case(40, 96, 500, 200, 1, 77))
    g = torch.Generator().manual_seed(78)
    a = int(round((3.0 * 75.0 ** 2 / (4.0 * 200)) ** 0.5))            # logits of standard deviation ~75
    case[0] = torch.randint(-3, 4, (40, 200), generator=g).float()
    case[1] = torch.randint(-a, a + 1, (500, 200), generator=g).float()
    case[2] = torch.randint(-3, 4, (500,), generator=g).float()
    x, ent, bias = case[:3]
    assert float((x.double() @ ent.double().t()).abs().max()) > 300.0
    _check(k, 'ce', opt, case)


@pytest.mark.parametrize('kind,opt', LOSSES)
def test_shared_matches_per_query_kernels(k, kind, opt):
    """B = 2,048, k = 3,000, N = 200,003, D = 200: the shared path against the per-query kernels on the broadcast matrix.
    Both sides round the logits in fp32 (differently), and the adversarial weights amplify that by alpha |z|: x is scaled
    so that alpha max|z| stays below 24, as in the per-query parity tests."""
    case = _case(2048, 3000, 200003, 200, 1, 5, scale=0.5)
    x, ent, bias, pos, shared, qid, ptr, idx = case
    cand = k.scoring.shared_candidates(pos.cuda(), shared.cuda(), qid.cuda(), ptr.cuda(), idx.cuda())
    got = _run_shared(k, kind, opt, *case)
    ref = _run_per_query(k, kind, opt, x, ent, bias, cand, 1)
    _close(got, [ref[0]] + [t / 2.5 for t in ref[1:]])


def test_shared_mask_is_bit_exact(k):
    """kgc_shared_mask_build's bits and sorted pairs against numpy."""
    B, K, N = 77, 150, 60
    _, _, _, _, shared, qid, ptr, idx = _case(B, K, N, 8, 1, 3)
    L, p = k._lib, k._lib.ptr
    W = (B + 31) // 32
    mask = torch.full((K, W), -1, dtype=torch.int32, device='cuda')
    ids = torch.empty((K,), dtype=torch.int32, device='cuda')
    slots = torch.empty((K,), dtype=torch.int32, device='cuda')
    nb = int(L.lib().kgc_shared_mask_workspace_bytes(K, N))
    ws = torch.empty((nb,), dtype=torch.uint8, device='cuda')
    sd, qd, pd, idd = shared.cuda(), qid.cuda(), ptr.cuda(), idx.cuda()
    L.call('kgc_shared_mask_build', p(sd), K, p(qd), B, p(pd), p(idd), N, p(mask), p(ids), p(slots), p(ws), nb, L.stream())
    torch.cuda.synchronize()
    ref = np.zeros((K, W), dtype=np.uint32)
    sh, pn, ix = shared.numpy(), ptr.numpy(), idx.numpy()
    for b in range(B):
        known = set(ix[pn[qid[b]]:pn[qid[b] + 1]].tolist())
        for j in range(K):
            if int(sh[j]) in known:
                ref[j, b >> 5] |= np.uint32(1 << (b & 31))
    assert np.array_equal(mask.cpu().numpy().view(np.uint32), ref)
    order = np.argsort(sh, kind='stable')
    assert np.array_equal(ids.cpu().numpy(), sh[order]) and np.array_equal(slots.cpu().numpy(), order)


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


@pytest.mark.parametrize('criterion,opt', [('bce', None), ('bce', 1.0), ('ce', 0.1)])
def test_loss_sampled_shared_matches_per_query_route_toy(k, toy, criterion, opt):
    """MGCN.loss_sampled(shared_negatives=True) on the 7-entity Toy graph equals the per-query kernels on the broadcast
    candidates built from the same draws: loss within 1e-6, every parameter gradient at the loss_sampled bars."""
    dl, m0 = toy
    ds = dl._get_dataset('train', _params())
    qid = np.arange(1, len(ds))
    B, P, K = len(qid), 2, 9
    rng = np.random.default_rng(4)
    pd = torch.from_numpy(rng.integers(0, 2 ** 32, (B, P), dtype=np.uint64).astype(np.int64))
    nd = torch.from_numpy(rng.integers(0, 2 ** 32, (K,), dtype=np.uint64).astype(np.int64))
    kw = dict(criterion=criterion, adversarial_temperature=opt) if criterion == 'bce' else dict(criterion='ce',
                                                                                                 label_smoothing=opt)
    grads, losses = {}, {}
    for mode in ('per_query', 'shared'):
        m = copy.deepcopy(m0).train()
        m.conv1.drop.p = 0.0
        if mode == 'shared':
            loss = m.loss_sampled(qid, ds, dl.graph, K, n_pos=P, draws=(pd, nd), shared_negatives=True, **kw)
        else:
            dev = 'cuda'
            triples, ptr, idx = ds.device_csr(dev)
            q = torch.from_numpy(qid).long().cuda()
            pos = ds.positives(q, P, draws=pd, device=dev)
            shared = ds.shared_negatives(K, draws=nd, device=dev)
            cand = k.scoring.shared_candidates(pos, shared, q, ptr, idx)
            assert bool((cand[:, P:] == -1).any())             # filtering happens on Toy
            _, x, all_ent = m._train_queries(q, triples, dl.graph)
            if criterion == 'ce':
                loss = k.score_sampled_ce(x, all_ent, m.conv2.bias, cand, P, label_smoothing=opt)
            else:
                pv, av = ds.label_values()
                loss = k.score_sampled_bce(x, all_ent, m.conv2.bias, cand, P, pv, av, adversarial_temperature=opt)
        loss.backward()
        losses[mode] = float(loss.item())
        grads[mode] = {n: p.grad.detach().clone() for n, p in m.named_parameters() if p.grad is not None}
    assert abs(losses['per_query'] - losses['shared']) <= 1e-6 * abs(losses['per_query']), losses
    assert grads['per_query'].keys() == grads['shared'].keys()
    top = max(float(g.abs().max()) for g in grads['per_query'].values())
    for n, g in grads['per_query'].items():
        assert float((g - grads['shared'][n]).abs().max()) <= 1e-5 * float(g.abs().max()) + 1e-6 * top, n


@pytest.mark.parametrize('criterion,opt', [('bce', None), ('bce', 1.0), ('ce', 0.1)])
def test_graphed_train_step_shared_matches_eager_toy(k, toy, criterion, opt):
    """GraphedTrainStep(negatives=k, shared_negatives=True): each replay equals the eager step on the same draws (the
    static neg_draws buffer is [k])."""
    dl, m0 = toy
    ds = dl._get_dataset('train', _params())
    qids = [list(range(0, 16)), list(range(1, 17)), list(range(0, 16)), list(range(16, 0, -1))]
    K = 12
    kw = dict(criterion=criterion, adversarial_temperature=opt) if criterion == 'bce' else dict(criterion='ce',
                                                                                                 label_smoothing=opt)
    m_g, m_e = copy.deepcopy(m0).train(), copy.deepcopy(m0).train()
    opt_g = k.ClipAdam(m_g.parameters(), lr=1e-2, max_norm=1.0)
    opt_e = k.ClipAdam(m_e.parameters(), lr=1e-2, max_norm=1.0)
    gen = torch.Generator(device='cuda').manual_seed(11)
    step = k.GraphedTrainStep(m_g, opt_g, dl.graph, ds, 16, warmup=0, negatives=K, generator=gen, shared_negatives=True,
                              **kw)
    assert tuple(step.neg_draws.shape) == (K,)
    for q in qids:
        lg = float(step(q).item())
        draws = (step.pos_draws.clone(), step.neg_draws.clone())
        opt_e.zero_grad(set_to_none=True)
        le = m_e.loss_sampled(q, ds, dl.graph, K, draws=draws, shared_negatives=True, **kw)
        le.backward()
        opt_e.step()
        assert abs(lg - float(le)) <= 1e-5 * max(1.0, abs(float(le))), (lg, float(le))
    for (n, a), b in zip(m_g.named_parameters(), m_e.parameters()):
        assert float((a - b).abs().max()) <= 1e-5 * max(1.0, float(b.abs().max())), n
