"""N1 (SURVEY.md 8(f)): training loss against sparse positives - kgc_label_mask_t_build + kgc_bce_1n_bwd_logit_t through the
C ABI against the oracle restatement (which tests/test_oracle_golden.py pins to the reference's dense-label BCELoss path), and
MGCN.loss_sparse / GraphedTrainStep(fused_loss=True) against the dense route on data/Toy.

First B200 run: 7 passed (gpurun_out/pytest_n1.log, end of round 1); the fused step is opt-in (fused_loss=True) until it
has been timed."""
import copy
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import mgcn_oracle as orc

pytestmark = pytest.mark.gpu


def _csr(n_query, n_entity, rng, hub=None):
    sizes = rng.integers(0, 6, n_query)
    if hub is not None:
        sizes[hub] = min(n_entity, 700)                      # a hub query: more positives than one CTA pass of 256 threads
    ptr = np.zeros(n_query + 1, dtype=np.int64)
    idx = []
    for q in range(n_query):
        idx.extend(sorted(rng.choice(n_entity, size=int(sizes[q]), replace=False).tolist()))
        ptr[q + 1] = len(idx)
    return ptr, np.asarray(idx, dtype=np.int32)


@pytest.mark.parametrize('B,N,smooth', [(128, 40943, 0.1), (16, 7, 0.0), (37, 1000, 0.1), (1, 33, 0.0), (130, 4097, 0.0)])
def test_sparse_bce_t_kernels_match_oracle(B, N, smooth):
    """Bit-exact label bits; loss within 2e-6 relative, logit / bias gradients within 2e-6 of max|gradient| of the oracle
    evaluated in float64 on the same float32 pred (the kernel's float32 logs vs float64 logs); pad columns zeroed;
    two runs bit-identical."""
    import kgc_gcn_b200 as k
    L = k._lib
    rng = np.random.default_rng(B * 7 + N)
    Q = B + 5
    ptr, idx = _csr(Q, N, rng, hub=2 if N >= 700 else None)
    qid = rng.permutation(Q)[:B].astype(np.int64)
    if N >= 700:
        qid[0] = 2
    pos, add = (float(np.float32(np.float32(1.0 - smooth) + np.float32(1.0 / N))), float(np.float32(1.0 / N))) if smooth else (1.0, 0.0)
    z = torch.randn((B, N), generator=torch.Generator().manual_seed(B + N)) * 3.0
    z[0, 0] = 30.0
    z[B - 1, N - 1] = -110.0                                 # saturated: the clamps of torch's BCE
    pred = torch.sigmoid(z)
    ldt = (B + 3) // 4 * 4
    dev = dict(device='cuda')
    qid_d, ptr_d, idx_d = (torch.from_numpy(a).cuda() for a in (qid, ptr, idx))
    p = L.ptr
    # entity-major: bits per entity, the loss pass overwrites predT [N, ldt] in place
    outs = []
    for _ in range(2):
        mask_t = torch.full((N, (B + 31) // 32), -1, dtype=torch.int32, **dev)       # the call zeroes it
        buf = torch.full((N, ldt), float('nan'), **dev)
        buf[:, :B] = pred.t().cuda()
        d_bias = torch.full((N,), float('nan'), **dev)
        partial = torch.empty((int(L.lib().kgc_bce_1n_t_blocks(N)),), dtype=torch.float64, **dev)
        loss = torch.empty((1,), **dev)
        L.call('kgc_label_mask_t_build', p(qid_d), B, p(ptr_d), p(idx_d), N, p(mask_t), L.stream())
        L.call('kgc_bce_1n_bwd_logit_t', p(buf), p(mask_t), N, B, ldt, pos, add, p(d_bias), p(partial), p(loss), L.stream())
        torch.cuda.synchronize()
        outs.append((mask_t.cpu(), buf.cpu(), d_bias.cpu(), loss.cpu()))
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    mask_t, buf, d_bias, loss = outs[0]
    bits = orc.label_mask(ptr, idx, qid, N)                                          # [B, words] bits over entities
    dense = ((bits[:, np.arange(N) >> 5] >> (np.arange(N) & 31).astype(np.uint32)) & 1).astype(bool)     # [B, N]
    got_t = mask_t.numpy().view(np.uint32)
    dense_t = ((got_t[:, np.arange(B) >> 5] >> (np.arange(B) & 31).astype(np.uint32)) & 1).astype(bool)  # [N, B]
    assert np.array_equal(dense_t, dense.T)
    o_loss, o_dl, o_db = orc.bce_1n_sparse(pred.double(), ptr, idx, qid, pos, add)
    assert abs(float(loss) - float(o_loss)) <= 2e-6 * abs(float(o_loss))
    scale = float(o_dl.abs().max())
    assert float((buf[:, :B].double() - o_dl.t()).abs().max()) <= 2e-6 * scale
    assert float(buf[:, B:].abs().sum()) == 0.0
    assert float((d_bias.double() - o_db).abs().max()) <= 2e-6 * scale * max(1.0, B ** 0.5)

def _params(**kw):
    base = dict(gcn_in_dim=20, gcn_out_dim=200, gcn_drop=0.0, hidden_drop=0.0, feat_drop=0.0, k_w=10, k_h=20,
                num_filter=2, kernel_size=7, bias=False, lbl_smooth=0.0, batch_size=128)
    base.update(kw)
    return SimpleNamespace(**base)


@pytest.fixture(scope='module')
def toy(golden_dir):
    import kgc_gcn_b200 as k
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
    return k, dl, m.cuda()


def test_loss_sparse_matches_dense_route(toy):
    """MGCN.loss_sparse == loss(forward(...), K5 label): value within 1e-6, every parameter gradient within 1e-5 of its
    max-norm + 1e-6 of the largest gradient (two fp32 evaluation orders of the same formulas)."""
    k, dl, m0 = toy
    ds = dl._get_dataset('train', _params())
    qid = list(range(1, 17))
    grads, losses = {}, {}
    for mode in ('dense', 'sparse'):
        m = copy.deepcopy(m0).train()
        m.conv1.drop.p = 0.0
        if mode == 'dense':
            trip, lab = ds.build_batch(qid, 'cuda')
            loss = m.loss(m(trip[:, 0], trip[:, 1], dl.graph), lab)
        else:
            loss = m.loss_sparse(qid, ds, dl.graph)
        loss.backward()
        losses[mode] = float(loss.item())
        grads[mode] = {n: p.grad.detach().clone() for n, p in m.named_parameters() if p.grad is not None}
    assert abs(losses['dense'] - losses['sparse']) <= 1e-6 * abs(losses['dense']), losses
    assert grads['dense'].keys() == grads['sparse'].keys()
    top = max(float(g.abs().max()) for g in grads['dense'].values())
    for n, g in grads['dense'].items():               # parameters whose true gradient is zero hold rounding noise: 1e-6 of the largest
        assert float((g - grads['sparse'][n]).abs().max()) <= 1e-5 * float(g.abs().max()) + 1e-6 * top, n


def test_graphed_train_step_fused_loss(toy):
    """GraphedTrainStep(fused_loss=True) follows the dense-label graph step loss for loss."""
    k, dl, m0 = toy
    ds = dl._get_dataset('train', _params())
    qids = [list(range(0, 16)), list(range(1, 17)), list(range(0, 16))]
    losses = {}
    for fused in (False, True):
        torch.manual_seed(3)
        m = copy.deepcopy(m0).train()
        m.conv1.drop.p = 0.0
        opt = k.ClipAdam(m.parameters(), lr=1e-2, max_norm=1.0)
        step = k.GraphedTrainStep(m, opt, dl.graph, ds, 16, warmup=0, fused_loss=fused)
        losses[fused] = [float(step(q).item()) for q in qids]
    for a, b in zip(losses[False], losses[True]):
        assert abs(a - b) <= 1e-5 * max(1.0, abs(a)), losses
