"""GPU parity tests of the graph-convolution path (K1-K4) against the oracle and the golden fixtures
produced by the unmodified reference.  Everything goes through the C ABI (ctypes -> libkgc_b200.so).

Tolerances (BASELINE.json north_star: "fp32 embeddings within rtol 1e-5"; SURVEY.md fact 9: judged
against the reference's float64 run, because two fp32 evaluations differ from each other by more):
    elementwise |ours - truth| <= 1e-5 * |truth| + 1e-5 * max|truth|
Integer structures (permutations, row pointers, degrees) are bit-exact.
"""
import os

import numpy as np
import pytest
import torch

import mgcn_oracle as orc

pytestmark = pytest.mark.gpu

RTOL = 1e-5


def close(ours, truth, name, rtol=RTOL):
    ours = ours.detach().double().cpu().numpy() if torch.is_tensor(ours) else np.asarray(ours, dtype=np.float64)
    truth = np.asarray(truth, dtype=np.float64)
    assert ours.shape == truth.shape, (name, ours.shape, truth.shape)
    scale = max(float(np.abs(truth).max()), 1e-30)
    err = np.abs(ours - truth)
    bound = rtol * np.abs(truth) + rtol * scale
    worst = float((err - bound).max())
    assert worst <= 0, '{}: max err {:.3e} (scale {:.3e}), max-norm-relative {:.3e}'.format(
        name, float(err.max()), scale, float(err.max()) / scale)


@pytest.fixture(scope='module')
def k():
    import kgc_gcn_b200
    assert torch.cuda.is_available()
    kgc_gcn_b200._lib.lib()
    return kgc_gcn_b200


def make_conv(k, z, d_in, d_out, R, p_drop):
    conv = k.MGCNConv(d_in, d_out, 2 * R, dropout=p_drop).cuda()
    with torch.no_grad():
        for name in ('loop_weight', 'in_weight', 'out_weight', 'rels_weight', 'loop_rel', 'loop_edge'):
            getattr(conv, name).copy_(torch.from_numpy(z['w.' + name]))
        conv.ent_bn.weight.copy_(torch.from_numpy(z['w.ent_bn.weight']))
        conv.ent_bn.bias.copy_(torch.from_numpy(z['w.ent_bn.bias']))
        conv.ent_bn.running_mean.copy_(torch.from_numpy(z['w.ent_bn.running_mean']))
        conv.ent_bn.running_var.copy_(torch.from_numpy(z['w.ent_bn.running_var']))
    return conv


def run_case(k, z, masks=None, training=True):
    d_in, d_out = z['x'].shape[1], z['g_ent'].shape[1]
    R = int(z['R'])
    conv = make_conv(k, z, d_in, d_out, R, 0.1 if masks is not None else 0.0)
    conv.train(training)
    if masks is not None:
        conv.set_dropout_masks(torch.from_numpy(masks[0]), torch.from_numpy(masks[1]))
    dev = 'cuda'
    x = torch.from_numpy(z['x']).to(dev).requires_grad_(True)
    ee = torch.from_numpy(z['edge_embs']).to(dev).requires_grad_(True)
    rl = torch.from_numpy(z['rels']).to(dev).requires_grad_(True)
    ei = torch.from_numpy(z['edge_index']).to(dev)
    et = torch.from_numpy(z['edge_type']).to(dev)
    ent, rel = conv(x, ei, et, None, ee, rl)
    torch.autograd.backward([ent, rel], [torch.from_numpy(z['g_ent']).to(dev), torch.from_numpy(z['g_rel']).to(dev)])
    grads = {'x': x.grad, 'edge_embs': ee.grad, 'rels': rl.grad, 'w.ent_bn.weight': conv.ent_bn.weight.grad,
             'w.ent_bn.bias': conv.ent_bn.bias.grad}
    for name in ('loop_weight', 'in_weight', 'out_weight', 'rels_weight', 'loop_rel', 'loop_edge'):
        grads['w.' + name] = getattr(conv, name).grad
    return conv, ent, rel, grads


@pytest.mark.parametrize('name', ['conv_toy_small', 'conv_toy_eval', 'conv_toy_full', 'conv_synth_hub'])
def test_conv_golden(k, golden_dir, name):
    z = np.load(os.path.join(golden_dir, name + '.npz'))
    conv, ent, rel, grads = run_case(k, z, training=bool(z['training']))
    close(ent, z['all_ent.f64'], 'all_ent')
    close(rel, z['all_rel.f64'], 'all_rel')
    for key, g in grads.items():
        close(g, z['grad.{}.f64'.format(key)], 'grad ' + key)
    if bool(z['training']):
        close(conv.ent_bn.running_mean, z['bn.running_mean_after'], 'running_mean')
        close(conv.ent_bn.running_var, z['bn.running_var_after'], 'running_var')
        assert int(conv.ent_bn.num_batches_tracked) == 1


def test_conv_golden_dropout_masks(k, golden_dir):
    """The reference's own Bernoulli draws (replayed by oracle/make_golden.py) injected as keep masks."""
    z = np.load(os.path.join(golden_dir, 'conv_synth_masks.npz'))
    _, ent, rel, grads = run_case(k, z, masks=(z['mask_in'], z['mask_out']))
    close(ent, z['all_ent.f64'], 'all_ent')
    close(rel, z['all_rel.f64'], 'all_rel')
    for key, g in grads.items():
        close(g, z['grad.{}.f64'.format(key)], 'grad ' + key)


def synth_case(N, R, E, d_in, d_out, seed):
    tri = orc.synthetic_triples(N, R, E, seed)
    g = orc.build_graph(tri, N, R)
    p = orc.conv_params(N, R, E, d_in, d_out, seed=seed)
    gen = torch.Generator().manual_seed(seed + 1)
    z = {'x': p['x'].numpy(), 'rels': p['rels'].numpy(), 'edge_embs': p['edge_embs'].numpy(), 'R': R,
         'edge_index': g['edge_index'], 'edge_type': g['edge_attr'][0],
         'g_ent': torch.randn(N, d_out, generator=gen).numpy(), 'g_rel': torch.randn(2 * R, d_out, generator=gen).numpy()}
    for kk, v in p['w'].items():
        z['w.' + kk] = v.numpy()
    return z, p


@pytest.mark.parametrize('shape', [(3000, 7, 9000, 100, 200, 31), (500, 40, 4000, 36, 24, 32), (64, 2, 70000, 8, 12, 33)])
def test_conv_vs_oracle_f64(k, shape):
    """Mid-size synthetic graphs with Zipf hubs (multi-level reductions: one dst row holds ~44% of the edges)
    against the oracle evaluated in float64 on the same inputs."""
    N, R, E, d_in, d_out, seed = shape
    z, p = synth_case(N, R, E, d_in, d_out, seed)
    dt = torch.float64
    w64 = {kk: v.to(dt) for kk, v in p['w'].items()}
    ent64, rel64, g64, _ = orc.conv_fwd_bwd(p['x'].to(dt), torch.from_numpy(z['edge_index']),
                                            torch.from_numpy(z['edge_type']), p['edge_embs'].to(dt), p['rels'].to(dt),
                                            w64, torch.from_numpy(z['g_ent']), torch.from_numpy(z['g_rel']))
    _, ent, rel, grads = run_case(k, z)
    close(ent, ent64.numpy(), 'all_ent')
    close(rel, rel64.numpy(), 'all_rel')
    names = {'x': 'entity_embedding', 'edge_embs': 'edge_embeddings', 'rels': 'relation_embedding'}
    for key, g in grads.items():
        ok = names.get(key, 'conv1.' + key[2:])
        close(g, g64[ok].numpy(), 'grad ' + key)


def test_conv_deterministic(k):
    z, _ = synth_case(2000, 5, 12000, 100, 200, 41)
    outs = []
    for _ in range(2):
        _, ent, rel, grads = run_case(k, z)
        outs.append([ent, rel] + [grads[kk] for kk in sorted(grads)])
    for a, b in zip(*outs):
        assert torch.equal(a, b)          # bit-identical: fixed reduction order, no float atomics


def test_csr_build_bit_exact(k):
    N, R, E = 1500, 9, 20000
    tri = orc.synthetic_triples(N, R, E, 51)
    g = orc.build_graph(tri, N, R)
    ei = torch.from_numpy(g['edge_index']).cuda()
    et = torch.from_numpy(g['edge_attr'][0]).cuda()
    plan = k.GraphPlan(ei, et, N, 2 * R + 1)
    src, dst, typ = g['edge_index'][0], g['edge_index'][1], g['edge_attr'][0]
    for key, perm_t, ptr_t, rows in ((dst, plan.perm_dst, plan.rowptr_dst, N), (src, plan.perm_src, plan.rowptr_src, N),
                                     (typ, plan.perm_type, plan.rowptr_type, 2 * R + 1)):
        perm, rowptr = orc.stable_csr(key, rows)
        np.testing.assert_array_equal(perm_t.cpu().numpy(), perm)
        np.testing.assert_array_equal(ptr_t.cpu().numpy(), rowptr)
    perm, rowptr = orc.stable_csr(dst, N)
    mid = rowptr[:-1] + np.bincount(dst[:E], minlength=N)
    np.testing.assert_array_equal(plan.rowmid_dst.cpu().numpy(), mid)
    deg = np.stack([orc.half_degree(g['edge_index'][:, :E], N), orc.half_degree(g['edge_index'][:, E:], N)])
    np.testing.assert_array_equal(plan.deg.cpu().numpy(), deg)
    norm = torch.cat([orc.compute_norm(g['edge_index'][:, :E], N), orc.compute_norm(g['edge_index'][:, E:], N)]).numpy()
    np.testing.assert_allclose(plan.norm.cpu().numpy(), norm, rtol=3e-7, atol=0)
    assert ((plan.norm.cpu().numpy() == 0) == (norm == 0)).all()
    rec = plan.rec_dst.cpu().numpy()
    np.testing.assert_array_equal(rec[:, 0], perm)
    np.testing.assert_array_equal(rec[:, 1], src[perm])
    np.testing.assert_array_equal(rec[:, 2], typ[perm])
    np.testing.assert_array_equal(rec[:, 3].view(np.float32), plan.norm.cpu().numpy()[perm])


def test_output_dropout_inside_the_tail(k):
    """MGCNConv(..., _out_drop=p) (what MGCN.encode uses for F.dropout(all_ent, gcn_drop), model.py:34): the output equals
    the undropped output x the Philox mask of plane 2 x 1/(1-p) bit for bit, and every gradient equals autograd through
    that explicit product (the layer's own dropout replayed with injected masks so both runs draw the same)."""
    z, masks = synth_case(1200, 4, 7000, 100, 200, 47), None
    z = z[0]
    d_in, d_out, R = z['x'].shape[1], z['g_ent'].shape[1], int(z['R'])
    rng = np.random.default_rng(3)
    m_in = torch.from_numpy((rng.random((z['x'].shape[0], d_out)) > 0.1).astype(np.uint8))
    m_out = torch.from_numpy((rng.random((z['x'].shape[0], d_out)) > 0.1).astype(np.uint8))
    p_out = 0.3
    res = {}
    for fused in (True, False):
        conv = make_conv(k, z, d_in, d_out, R, 0.1).train()
        conv.set_dropout_masks(m_in, m_out)
        x = torch.from_numpy(z['x']).cuda().requires_grad_(True)
        ee = torch.from_numpy(z['edge_embs']).cuda().requires_grad_(True)
        rl = torch.from_numpy(z['rels']).cuda().requires_grad_(True)
        ei, et = torch.from_numpy(z['edge_index']).cuda(), torch.from_numpy(z['edge_type']).cuda()
        g_ent, g_rel = torch.from_numpy(z['g_ent']).cuda(), torch.from_numpy(z['g_rel']).cuda()
        if fused:
            ent, rel = conv(x, ei, et, None, ee, rl, _out_drop=p_out)
            seed = conv._last_out_seed.clone()
        else:
            ent0, rel = conv(x, ei, et, None, ee, rl)
            mask = torch.empty(ent0.shape, dtype=torch.uint8, device='cuda')
            k._lib.call('kgc_dropout_mask', k._lib.ptr(seed), 2, p_out, mask.numel(), k._lib.ptr(mask), k._lib.stream())
            assert 0.6 < float(mask.float().mean()) < 0.8
            ent = ent0 * (mask.float() * np.float32(1.0 / (1.0 - p_out)))
        torch.autograd.backward([ent, rel], [g_ent, g_rel])
        res[fused] = [ent.detach(), rel.detach(), x.grad, ee.grad, rl.grad] + [p_.grad for p_ in conv.parameters()]
    assert torch.equal(res[True][0], res[False][0]) and torch.equal(res[True][1], res[False][1])
    for a, b in zip(res[True][2:], res[False][2:]):
        assert float((a - b).abs().max()) <= 2e-6 * float(b.abs().max()) + 1e-12


def test_hybrid_partition_on_device(k):
    """partition.partition_edges_hybrid_device (torch ops on the GPU) == partition_edges_hybrid (numpy), every field, for
    2 / 3 / 8 ranks on a hub-heavy graph whose node count is not a multiple of the rank count."""
    from kgc_gcn_b200.partition import partition_edges_hybrid, partition_edges_hybrid_device
    N, R, E = 30001, 7, 160000
    tri = orc.synthetic_triples(N, R, E, 4)
    g = orc.build_graph(tri, N, R)
    ei, et = g['edge_index'], g['edge_attr'][0]
    ei_d, et_d = torch.from_numpy(ei).cuda(), torch.from_numpy(et).cuda()
    for world in (2, 3, 8):
        for rank in (0, world - 1):
            a = partition_edges_hybrid(ei, et, N, world, rank)
            b = partition_edges_hybrid_device(ei_d, et_d, N, world, rank)
            assert set(a) == set(b)
            for key in a:
                got = b[key].cpu().numpy() if torch.is_tensor(b[key]) else b[key]
                assert np.array_equal(np.asarray(a[key]), np.asarray(got)), (world, rank, key)


def test_stream_plan_on_device(k):
    """kgc_stream_plan_flags + the device-side slot numbering (plan.build_stream_plan_device) against the numpy
    restatement (plan.build_stream_plan): rowflags, chunk carry slots, carry count, empty rows and fix-up levels bit for
    bit - random segment sets with empty segments, rows spanning many chunks, a partial last chunk; then the three
    schedules of a whole GraphPlan against the numpy schedules of its row pointers."""
    from kgc_gcn_b200.plan import StreamPlan, build_stream_plan, build_stream_plan_device
    rng = np.random.default_rng(21)
    for trial in range(6):
        n_seg = int(rng.integers(1, 400))
        length = rng.integers(0, 6, n_seg) * (rng.random(n_seg) < 0.7)
        hubs = rng.integers(0, n_seg, 3)
        length[hubs] += rng.integers(40, 5000, 3)                       # rows that span many chunks (several fix-up levels)
        if trial == 0:
            length[:] = 0
            length[n_seg // 2] = 7
        end = np.cumsum(length)
        beg = end - length
        row = rng.permutation(n_seg + 50)[:n_seg]
        n_rec = int(end[-1])
        want = build_stream_plan(beg, end, row, n_rec, fan_in=64)
        dev_args = [torch.from_numpy(a.astype(np.int32)).cuda() for a in (beg, end, row)]
        got = build_stream_plan_device(*dev_args, n_rec, fan_in=64)
        np.testing.assert_array_equal(got['rowflags'].cpu().numpy().view(np.uint32), want['rowflags'])
        np.testing.assert_array_equal(got['chunks'].cpu().numpy(), want['chunks'])
        assert got['n_carry'] == want['n_carry']
        np.testing.assert_array_equal(got['fill_rows'], want['fill_rows'])
        assert len(got['levels']) == len(want['levels'])
        for (ia, pa), (ib, pb) in zip(got['levels'], want['levels']):
            np.testing.assert_array_equal(ia, ib)
            assert pa == pb
    N, R, E = 3000, 7, 40000
    tri = orc.synthetic_triples(N, R, E, 5)
    g = orc.build_graph(tri, N, R)
    ei, et = torch.from_numpy(g['edge_index']).cuda(), torch.from_numpy(g['edge_attr'][0]).cuda()
    plan = k.GraphPlan(ei, et, N, 2 * R + 1, type_block_rows=512)
    rp_dst, rm_dst, rp_src, rp_typ = (t.cpu().numpy().astype(np.int64)
                                      for t in (plan.rowptr_dst, plan.rowmid_dst, plan.rowptr_src, plan.rowptr_type))
    Nd, n2, dev = plan.num_dst_rows, plan.num_edges2, plan.device
    # forward: records [rowptr[i], rowmid[i]) reduce into row i (in half), [rowmid[i], rowptr[i+1]) into row Nd + i (out half)
    drows = np.arange(Nd, dtype=np.int64)
    fb = np.stack([rp_dst[:-1], rm_dst], 1).reshape(-1)
    fe = np.stack([rm_dst, rp_dst[1:]], 1).reshape(-1)
    fr = np.stack([drows, drows + Nd], 1).reshape(-1)
    host = {'fwd': StreamPlan(build_stream_plan(fb, fe, fr, n2), n2, dev, prefill_ranges=[(0, Nd), (Nd, 2 * Nd)]),
            'bwd_src': StreamPlan(build_stream_plan(rp_src[:-1], rp_src[1:], np.arange(N, dtype=np.int64), n2), n2, dev),
            'bwd_rel': StreamPlan(build_stream_plan(rp_typ[:-1], rp_typ[1:], np.arange(plan.num_type_rows, dtype=np.int64),
                                                    n2), n2, dev)}
    for name in ('fwd', 'bwd_src', 'bwd_rel'):
        a, b = host[name], getattr(plan, name)
        assert torch.equal(a.rowflags, b.rowflags) and torch.equal(a.chunks, b.chunks) and a.n_carry == b.n_carry
        assert len(a.levels) == len(b.levels) and a.prefill == b.prefill
        for la, lb in zip(a.levels, b.levels):
            assert torch.equal(la[0], lb[0]) and la[1:] == lb[1:]


def test_type_sort_blocked_by_subject(k, monkeypatch):
    """The d_rel pass blocked by subject row (kgc_csr_build type_block_rows): the permutation is the stable sort by
    (block of the subject, type) bit for bit; the layer's outputs and gradients with the blocked pass equal the plain
    pass (d_rel within float tolerance: the partial rows are added block by block; everything else bit for bit)."""
    N, R, E = 1500, 9, 20000
    tri = orc.synthetic_triples(N, R, E, 51)
    g = orc.build_graph(tri, N, R)
    ei = torch.from_numpy(g['edge_index']).cuda()
    et = torch.from_numpy(g['edge_attr'][0]).cuda()
    T, BR = 2 * R + 1, 256
    plan = k.GraphPlan(ei, et, N, T, type_block_rows=BR)
    src, dst, typ = g['edge_index'][0], g['edge_index'][1], g['edge_attr'][0]
    subj = np.concatenate([src[:E], dst[E:]])
    n_blocks = -(-N // BR)
    assert plan.num_type_blocks == n_blocks and plan.num_type_rows == n_blocks * T
    perm, rowptr = orc.stable_csr((subj // BR) * T + typ, n_blocks * T)
    np.testing.assert_array_equal(plan.perm_type.cpu().numpy(), perm)
    np.testing.assert_array_equal(plan.rowptr_type.cpu().numpy(), rowptr)
    rec = plan.rec_type.cpu().numpy()
    np.testing.assert_array_equal(rec[:, 0], perm)
    np.testing.assert_array_equal(rec[:, 1], src[perm])
    np.testing.assert_array_equal(rec[:, 2], dst[perm])
    # the other two sorts are untouched
    for key, perm_t in ((dst, plan.perm_dst), (src, plan.perm_src)):
        np.testing.assert_array_equal(perm_t.cpu().numpy(), orc.stable_csr(key, N)[0])
    z, _ = synth_case(2000, 5, 12000, 100, 200, 43)
    res = {}
    # N = 2,000 rows: the default block of 65,536 rows leaves the type sort plain (N < 4 blocks), 128 rows block it
    for br in (k.plan.TYPE_BLOCK_ROWS, 128):
        monkeypatch.setattr(k.plan, 'TYPE_BLOCK_ROWS', br)
        k.plan._PLAN_CACHE.clear()
        _, ent, rel, grads = run_case(k, z)
        res[br] = (ent, rel, grads)
    k.plan._PLAN_CACHE.clear()
    plain, blocked = res.values()
    assert torch.equal(plain[0], blocked[0]) and torch.equal(plain[1], blocked[1])
    for name in plain[2]:
        a, b = plain[2][name], blocked[2][name]
        if torch.equal(a, b):
            continue
        assert name in ('rels', 'w.loop_rel'), name
        assert float((a - b).abs().max()) <= 2e-6 * float(a.abs().max()) + 1e-12, name


def test_csr_toy_known_answers(k, golden_dir):
    import json
    with open(os.path.join(golden_dir, 'toy_loader.json')) as f:
        toy = json.load(f)
    ei = torch.tensor(toy['edge_index']).cuda()
    et = torch.tensor(toy['edge_attr'][0]).cuda()
    plan = k.GraphPlan(ei, et, 7, 11)
    n = plan.norm.cpu().numpy()
    np.testing.assert_allclose(n[:10], [.40825, .28868, .40825, 0, 0, 0, 0, .70711, 0, 0], atol=2e-5)   # SURVEY App. B
    np.testing.assert_allclose(n[10:], [0, 0, 0, 0, 0, 0, .40825, .70711, .57735, .70711], atol=2e-5)
    conv = k.MGCNConv(4, 4, 10).cuda()
    np.testing.assert_array_equal(conv.compute_norm(ei[:, :10], 7).cpu().numpy(), n[:10])


def test_csr_rejects_bad_ids(k):
    ei = torch.tensor([[0, 1, 2, 9], [1, 2, 0, 0]]).cuda()
    et = torch.tensor([0, 0, 1, 1]).cuda()
    with pytest.raises(RuntimeError, match='out of range'):
        k.GraphPlan(ei, et, 3, 3)


def test_label_build_bit_exact(k, golden_dir, toy_dir):
    ds = orc.load_dataset(toy_dir)
    prm = type('P', (), {'lbl_smooth': 0.1})()
    z = np.load(os.path.join(golden_dir, 'toy_batches.npz'))
    kb = k.KBDataset(ds['queries']['train'], 7, prm, training=True)
    trip, lab = kb.build_batch(np.arange(len(kb)), 'cuda')
    np.testing.assert_array_equal(trip.cpu().numpy(), z['train_triple'])
    np.testing.assert_array_equal(lab.cpu().numpy(), z['train_label'])       # incl. the 0.9 + 1/7 > 1 quirk
    kb = k.KBDataset(ds['queries']['valid_tail'], 7, prm, training=False)
    trip, lab = kb.build_batch(np.arange(len(kb)), 'cuda')
    np.testing.assert_array_equal(trip.cpu().numpy(), z['valid_tail_triple'])
    np.testing.assert_array_equal(lab.cpu().numpy(), z['valid_tail_label'])
    # ragged / larger: N not a multiple of 4, empty label lists, random order
    rng = np.random.default_rng(0)
    N, Q = 10007, 300
    qs = [{'triple': (int(rng.integers(N)), 1, -1), 'label': sorted(set(rng.integers(0, N, rng.integers(0, 40)).tolist()))}
          for _ in range(Q)]
    kb = k.KBDataset(qs, N, prm, training=True)
    qid = rng.permutation(Q)[:131]
    trip, lab = kb.build_batch(qid, 'cuda')
    t0, l0 = orc.make_batch(qs, qid, N, lbl_smooth=0.1, training=True)
    np.testing.assert_array_equal(trip.cpu().numpy(), t0)
    np.testing.assert_array_equal(lab.cpu().numpy(), l0)


def test_samplers_through_the_python_api(k):
    """KBDataset.negatives / DataLoader.sample_edges (extensions, parity unpinned): bit-exact against the oracle's
    restatements for the caller's draws; negatives never hit a known object; the sampled sub-graph convolves."""
    rng = np.random.default_rng(11)
    N, Q, K, TR = 97, 60, 5, 3
    qs = [{'triple': (0, 0, -1), 'label': sorted(set(rng.integers(0, N, 30).tolist()))} for _ in range(Q)]
    kb = k.KBDataset(qs, N, None)
    qid = rng.permutation(Q)[:23]
    draws = rng.integers(0, 2 ** 32, (23, K, TR), dtype=np.uint64)
    neg = kb.negatives(qid, K, draws=torch.from_numpy(draws.astype(np.int64)), tries=TR)
    exp = orc.neg_sample([q['label'] for q in qs], qid, N, draws)
    np.testing.assert_array_equal(neg.cpu().numpy(), exp)
    drawn = kb.negatives(qid, K, tries=8).cpu().numpy()                  # draws from torch's generator
    for b in range(23):
        assert not (set(drawn[b][drawn[b] >= 0].tolist()) & set(qs[int(qid[b])]['label']))
    # edge sampler on a synthetic graph
    Ng, R, E = 500, 4, 3000
    tri = orc.synthetic_triples(Ng, R, E, 9)
    g = orc.build_graph(tri, Ng, R)
    dl = k.DataLoader.__new__(k.DataLoader)
    dl.num_edge, dl.num_relation = E, R
    dl.graph = k.GraphData(edge_index=torch.from_numpy(g['edge_index']).cuda(),
                                       edge_attr=torch.from_numpy(g['edge_attr']).cuda())
    dl.graph.entity, dl.graph.num_nodes = torch.arange(Ng).cuda(), Ng
    ed = rng.integers(0, 2 ** 32, 700, dtype=np.uint64)
    sub = dl.sample_edges(700, draws=torch.from_numpy(ed.astype(np.int64)))
    ei, et, cols = orc.edge_sample(g['edge_index'], g['edge_attr'][0], E, ed)
    np.testing.assert_array_equal(sub.edge_index.cpu().numpy(), ei)
    np.testing.assert_array_equal(sub.edge_attr[0].cpu().numpy(), et)
    np.testing.assert_array_equal(sub.edge_attr[1].cpu().numpy(), cols)
    assert (sub.edge_attr[0][:700] < R).all() and (sub.edge_attr[0][700:] >= R).all()       # in half first, then reverses
    p = orc.conv_params(Ng, R, E, 100, 200, seed=1)
    conv = k.MGCNConv(100, 200, 2 * R).cuda().train()
    x = p['x'].cuda().requires_grad_(True)
    ee = p['edge_embs'].cuda()[sub.edge_attr[1]].requires_grad_(True)
    ent, rel = conv(x, sub.edge_index, sub.edge_attr[0], None, ee, p['rels'].cuda())
    ent.sum().backward()
    assert torch.isfinite(ent).all() and torch.isfinite(x.grad).all() and ent.shape == (Ng, 200)


def test_neg_sampler_matches_restatement(k):
    """Extension without a reference counterpart (parity unpinned): checked against its own restatement."""
    import ctypes
    rng = np.random.default_rng(5)
    N, Q, K, TR = 50, 40, 6, 4
    qs = [{'triple': (0, 0, -1), 'label': sorted(set(rng.integers(0, N, 25).tolist()))} for _ in range(Q)]
    kb = k.KBDataset(qs, N, None)
    _, ptr, idx = kb.device_csr(torch.device('cuda'))
    qid = torch.from_numpy(rng.permutation(Q)[:17].astype(np.int64)).cuda()
    draws = torch.from_numpy(rng.integers(0, 2 ** 32, (17, K, TR), dtype=np.uint64).astype(np.uint32).view(np.int32)).cuda()
    neg = torch.empty((17, K), dtype=torch.int32, device='cuda')
    L = k._lib
    L.call('kgc_neg_sample', L.ptr(qid), 17, L.ptr(ptr), L.ptr(idx), N, L.ptr(draws), K, TR, L.ptr(neg), L.stream())
    d = draws.cpu().numpy().view(np.uint32).astype(np.uint64)
    exp = np.full((17, K), -1, dtype=np.int32)
    for b in range(17):
        pos = set(qs[int(qid[b])]['label'])
        for j in range(K):
            for a in range(TR):
                c = int((d[b, j, a] * np.uint64(N)) >> np.uint64(32))
                if c not in pos:
                    exp[b, j] = c
                    break
    np.testing.assert_array_equal(neg.cpu().numpy(), exp)


def test_state_dict_names(k):
    prm = type('P', (), dict(gcn_in_dim=8, gcn_out_dim=200, gcn_drop=0.3, hidden_drop=0.3, feat_drop=0.3, k_w=10, k_h=20,
                             num_filter=2, kernel_size=7, bias=False))()
    m = k.MGCN(7, 5, 10, prm)
    keys = set(m.state_dict().keys())
    expect = {'entity_embedding', 'relation_embedding', 'edge_embeddings', 'conv1.loop_weight', 'conv1.in_weight',
              'conv1.out_weight', 'conv1.rels_weight', 'conv1.loop_rel', 'conv1.loop_edge', 'conv2.bias',
              'conv2.conv_e.weight', 'conv2.fc.weight', 'conv2.fc.bias'}
    for bn in ('conv1.ent_bn', 'conv2.bn0', 'conv2.bn1', 'conv2.bn2'):
        expect |= {bn + s for s in ('.weight', '.bias', '.running_mean', '.running_var', '.num_batches_tracked')}
    assert keys == expect


@pytest.mark.parametrize('M,K,N', [(1000, 100, 200), (40943, 200, 100), (5, 12, 20), (129, 36, 24), (300, 256, 17)])
def test_gemm_tf32x3_fp32_grade(k, M, K, N):
    """K4b: the 3xTF32 tensor-core GEMM is as close to the exact product as a plain fp32 GEMM is."""
    g = torch.Generator().manual_seed(M + K + N)
    a = torch.randn(M, K, generator=g)
    b = torch.randn(K, N, generator=g) * 0.1
    truth = (a.double() @ b.double())
    scale = float(truth.abs().max())
    out = torch.full((M, N), float('nan'), device='cuda')
    k.gemm_nt(a.cuda(), b.cuda(), out)
    err = float((out.cpu().double() - truth).abs().max()) / scale
    err_fp32 = float(((a @ b).double() - truth).abs().max()) / scale
    print('gemm_tf32x3 M={} K={} N={}: err {:.2e} (fp32 GEMM {:.2e})'.format(M, K, N, err, err_fp32))
    assert err <= max(4 * err_fp32, 2e-6), (err, err_fp32)
    # transposed small operand (strided view) and a row-strided A / C, as the layer uses them
    bt = (torch.randn(N, K, generator=g) * 0.1)
    big = torch.randn(M, K + 4, generator=g).cuda()
    a2 = big[:, :K]
    out2 = torch.full((M, N + 4), float('nan'), device='cuda')
    k.gemm_nt(a2, bt.cuda().t(), out2[:, :N])
    truth2 = a2.cpu().double() @ bt.double().t()
    assert float((out2[:, :N].cpu().double() - truth2).abs().max()) / float(truth2.abs().max()) <= 2e-6
    assert torch.isnan(out2[:, N:]).all()                        # nothing written outside the N valid columns


@pytest.mark.parametrize('M,Ka,Nb', [(40943, 100, 200), (1000, 12, 20), (77, 128, 256), (3, 4, 8), (5000, 128, 224), (33, 100, 200)])
def test_gemm_tn_weight_gradient(k, M, Ka, Nb):
    """K4c: C = A^T @ B over the node rows, fp32, deterministic."""
    g = torch.Generator().manual_seed(M + Ka)
    a = torch.randn(M, Ka, generator=g)
    b = torch.randn(M, Nb, generator=g)
    truth = a.double().t() @ b.double()
    scale = float(truth.abs().max())
    err_fp32 = float(((a.t() @ b).double() - truth).abs().max()) / scale
    for tc in (False, True):              # register-tiled fp32 kernel, then the tensor-core (3xTF32, MN-major) kernel
        out = torch.full((Ka, Nb), float('nan'), device='cuda')
        k.gemm_tn(a.cuda(), b.cuda(), out, tensor_cores=tc)
        err = float((out.cpu().double() - truth).abs().max()) / scale
        print('gemm_tn tc={} M={} Ka={} Nb={}: err {:.2e} (fp32 GEMM {:.2e})'.format(tc, M, Ka, Nb, err, err_fp32))
        assert err <= max(6 * err_fp32, 3e-6)
        out2 = torch.empty(Ka, Nb, device='cuda')
        k.gemm_tn(a.cuda(), b.cuda(), out2, tensor_cores=tc)
        assert torch.equal(out, out2)


def test_in_kernel_dropout_matches_its_own_masks(k):
    """K4 Philox dropout: a training step with the in-kernel generator equals, bit for bit, the same step with the
    masks that generator produces injected explicitly; the keep rate is 1 - p; seeds change every step."""
    z, _ = synth_case(1500, 4, 6000, 100, 200, 61)
    d_in, d_out, R = 100, 200, 4
    conv = make_conv(k, z, d_in, d_out, R, 0.1).train()
    torch.manual_seed(7)
    dev = 'cuda'

    def run(masks):
        x = torch.from_numpy(z['x']).to(dev).requires_grad_(True)
        ee = torch.from_numpy(z['edge_embs']).to(dev).requires_grad_(True)
        rl = torch.from_numpy(z['rels']).to(dev).requires_grad_(True)
        conv.set_dropout_masks(*masks) if masks else conv.set_dropout_masks(None, None)
        conv.zero_grad()
        ent, rel = conv(x, torch.from_numpy(z['edge_index']).to(dev), torch.from_numpy(z['edge_type']).to(dev), None, ee, rl)
        torch.autograd.backward([ent, rel], [torch.from_numpy(z['g_ent']).to(dev), torch.from_numpy(z['g_rel']).to(dev)])
        return [ent, rel, x.grad, ee.grad, rl.grad, conv.in_weight.grad.clone(), conv.out_weight.grad.clone()]
    a = run(None)
    seed1 = conv._last_seed.clone()
    m_in, m_out = conv.dropout_masks(seed1, 1500)
    keep = float(m_in.float().mean())
    assert abs(keep - 0.9) < 0.005 and not torch.equal(m_in, m_out)
    b = run((m_in, m_out))
    for u, v in zip(a, b):
        assert torch.equal(u, v)
    run(None)
    assert int(conv._last_seed) != int(seed1)
    assert '_drop_seed' not in conv.state_dict()


def test_conv_full_wn18rr_shape_vs_oracle_f64(k):
    """BASELINE.json configs[1] at FULL size (40,943 entities, 11 relations, 86,835 triples, Zipf objects): outputs and
    every gradient against the oracle's float64 run on the same inputs."""
    z, p = synth_case(40943, 11, 86835, 100, 200, 0)
    dt = torch.float64
    w64 = {kk: v.to(dt) for kk, v in p['w'].items()}
    ent64, rel64, g64, _ = orc.conv_fwd_bwd(p['x'].to(dt), torch.from_numpy(z['edge_index']),
                                            torch.from_numpy(z['edge_type']), p['edge_embs'].to(dt), p['rels'].to(dt),
                                            w64, torch.from_numpy(z['g_ent']), torch.from_numpy(z['g_rel']))
    _, ent, rel, grads = run_case(k, z)
    close(ent, ent64.numpy(), 'all_ent')
    close(rel, rel64.numpy(), 'all_rel')
    names = {'x': 'entity_embedding', 'edge_embs': 'edge_embeddings', 'rels': 'relation_embedding'}
    for key, g in grads.items():
        close(g, g64[names.get(key, 'conv1.' + key[2:])].numpy(), 'grad ' + key, rtol=2e-5)


def test_conv_edge_cases(k):
    """Edgeless graph, wide rows (D > 128: the two-float4-per-lane instantiation), a single node."""
    # (a) no edges at all: the layer reduces to the self-loop branch
    N, R, d_in, d_out = 50, 2, 100, 200
    p = orc.conv_params(N, R, 0, d_in, d_out, seed=5)
    conv = k.MGCNConv(d_in, d_out, 2 * R, dropout=0.0).cuda().train()
    with torch.no_grad():
        for name in ('loop_weight', 'in_weight', 'out_weight', 'rels_weight', 'loop_rel', 'loop_edge'):
            getattr(conv, name).copy_(p['w'][name])
    ei = torch.zeros((2, 0), dtype=torch.int64, device='cuda')
    et = torch.zeros((0,), dtype=torch.int64, device='cuda')
    x = p['x'].cuda().requires_grad_(True)
    ee = torch.zeros((0, d_in), device='cuda', requires_grad=True)
    ent, rel = conv(x, ei, et, None, ee, p['rels'].cuda())
    w64 = {kk: v.double() for kk, v in p['w'].items()}
    ent64, rel64, _ = orc.conv_forward(p['x'].double(), ei.cpu(), et.cpu(), torch.zeros(0, d_in).double(), p['rels'].double(),
                                       w64, training=True)
    close(ent, ent64.numpy(), 'edgeless all_ent')
    ent.sum().backward()
    assert x.grad is not None and torch.isfinite(x.grad).all()
    # (b) D = 160 (> 128) and Dout = 72 with hubs
    z, p2 = synth_case(300, 3, 2500, 160, 72, 77)
    dt = torch.float64
    w64 = {kk: v.to(dt) for kk, v in p2['w'].items()}
    e64, r64, g64, _ = orc.conv_fwd_bwd(p2['x'].to(dt), torch.from_numpy(z['edge_index']), torch.from_numpy(z['edge_type']),
                                        p2['edge_embs'].to(dt), p2['rels'].to(dt), w64, torch.from_numpy(z['g_ent']),
                                        torch.from_numpy(z['g_rel']))
    _, ent, rel, grads = run_case(k, z)
    close(ent, e64.numpy(), 'wide all_ent')
    close(grads['x'], g64['entity_embedding'].numpy(), 'wide d_x')
    close(grads['edge_embs'], g64['edge_embeddings'].numpy(), 'wide d_ee')
    close(grads['rels'], g64['relation_embedding'].numpy(), 'wide d_rel')


def test_conv_linearity_and_determinism_at_fb15k237_shape(k):
    """Size-independent properties at BASELINE.json configs[2] size (14,541 entities, 237 relations, 272,115 triples):
    the aggregation is linear in the edge embeddings (agg(2 ee) = 2 agg(ee) exactly: scaling by 2 is exact in fp32) and two
    runs are bit-identical."""
    N, R, E, D = 14541, 237, 272115, 100
    tri = orc.synthetic_triples(N, R, E, 1)
    g = orc.build_graph(tri, N, R)
    ei, et = torch.from_numpy(g['edge_index']).cuda(), torch.from_numpy(g['edge_attr'][0]).cuda()
    plan = k.get_plan(ei, et, N, 2 * R + 1)
    gen = torch.Generator().manual_seed(2)
    x = torch.randn(N, D, generator=gen).cuda()
    rel = torch.randn(2 * R + 1, D, generator=gen).cuda()
    ee = torch.randn(2 * E, D, generator=gen).cuda()
    L = k._lib
    p, st = L.ptr, L.stream

    def agg(eet):
        out = torch.empty((2, N, D), device='cuda')

        def level0(sp, out_final, carry):
            L.call('kgc_agg_fwd', p(x), p(rel), rel.shape[0], p(eet), p(plan.rec_dst), p(sp.rowflags), p(sp.chunks), sp.n_rec,
                   p(out_final), p(carry), D, st())
        plan.run_reduction(plan.fwd, level0, out, D, tag='t')
        return out
    a1, a2, a3 = agg(ee), agg(ee), agg(ee * 2)
    assert torch.equal(a1, a2)
    assert torch.equal(a3, a1 * 2)
    # row sums against a float64 scatter of the same per-edge messages (checksum of the whole output)
    src, dst, typ = g['edge_index'][0], g['edge_index'][1], g['edge_attr'][0]
    norm = plan.norm.double()
    msg = norm[:, None] * x.double()[torch.from_numpy(src).cuda()] * rel.double()[torch.from_numpy(typ).cuda()] * ee.double()
    ref = torch.zeros((2 * N, D), dtype=torch.float64, device='cuda')
    rows = torch.from_numpy(dst).cuda() + (torch.arange(2 * E, device='cuda') >= E) * N
    ref.index_add_(0, rows, msg)
    close(a1.reshape(2 * N, D), ref.cpu().numpy(), 'fb15k237 agg', rtol=2e-5)


@pytest.mark.parametrize('B,F,O', [(128, 39200, 200), (77, 4096, 200), (5, 8192, 32), (128, 5024, 100)])
def test_linear_tc_fc_layer(k, B, F, O):
    """ConvE's fc layer (model.py:173) on the 3xTF32 kernels: split-K forward, transposed-operand backward; fp32 accuracy
    against the fp64 evaluation, deterministic."""
    g = torch.Generator().manual_seed(B + F + O)
    x = (torch.randn(B, F, generator=g)).cuda().requires_grad_(True)
    w = (torch.randn(O, F, generator=g) * 0.01).cuda().requires_grad_(True)
    b = (torch.randn(O, generator=g) * 0.1).cuda().requires_grad_(True)
    dy = torch.randn(B, O, generator=g).cuda()
    assert k.linear_tc_supported(x, w)
    y = k.linear_tc(x, w, b)
    y.backward(dy)
    xd, wd, bd = (t.detach().double().requires_grad_(True) for t in (x, w, b))
    yd = xd @ wd.t() + bd
    yd.backward(dy.double())
    y32 = (x.detach() @ w.detach().t() + b.detach())
    for got, ref, ref32, name in ((y.detach(), yd.detach(), y32, 'y'), (x.grad, xd.grad, None, 'dx'), (w.grad, wd.grad, None, 'dw'),
                                  (b.grad, bd.grad, None, 'db')):
        scale = float(ref.abs().max())
        err = float((got.double() - ref).abs().max()) / scale
        err32 = float((ref32.double() - ref).abs().max()) / scale if ref32 is not None else float('nan')
        print('linear_tc B={} F={} O={} {}: err {:.2e} (fp32 GEMM {:.2e})'.format(B, F, O, name, err, err32))
        assert err <= 4e-6, (name, err)
    x2, w2, b2 = (t.detach().clone().requires_grad_(True) for t in (x, w, b))
    y2 = k.linear_tc(x2, w2, b2)
    y2.backward(dy)
    assert torch.equal(y2, y) and torch.equal(x2.grad, x.grad) and torch.equal(w2.grad, w.grad)


def test_gemm_batches_match_single_launches(k):
    """The batched K4b / K4c launches give bit-identical K4b results and fp32-accurate, deterministic K4c results; K4c with
    rows = M for every problem gives the bits of the launch without rows."""
    from kgc_gcn_b200.conv import gemm_nt_batch, gemm_tn_batch, _pack_b
    g = torch.Generator().manual_seed(5)
    M, K, N = 5000, 100, 200
    a = [torch.randn(M, K, generator=g).cuda() for _ in range(3)]
    w = [(torch.randn(K, N, generator=g) * 0.1).cuda() for _ in range(3)]
    single = [k.gemm_nt(a[i], w[i], torch.empty(M, N, device='cuda')) for i in range(3)]
    for n in (2, 3):
        outs = [torch.full((M, N), float('nan'), device='cuda') for _ in range(n)]
        gemm_nt_batch(a[:n], [_pack_b(w[i]) for i in range(n)], outs)
        for i in range(n):
            assert torch.equal(outs[i], single[i])
    b = [torch.randn(M, N, generator=g).cuda() for _ in range(3)]
    for n in (1, 2, 3):
        outs = [torch.full((K, N), float('nan'), device='cuda') for _ in range(n)]
        gemm_tn_batch(a[:n], b[:n], outs)
        outs2 = [torch.empty((K, N), device='cuda') for _ in range(n)]
        gemm_tn_batch(a[:n], b[:n], outs2)
        outs3 = [torch.empty((K, N), device='cuda') for _ in range(n)]
        gemm_tn_batch(a[:n], b[:n], outs3, rows=[M] * n)        # every problem of full height: the bits of rows=None
        for i in range(n):
            truth = a[i].double().t() @ b[i].double()
            assert float((outs[i].double() - truth).abs().max()) / float(truth.abs().max()) <= 3e-6
            assert torch.equal(outs[i], outs2[i])
            assert torch.equal(outs[i], outs3[i])


@pytest.mark.parametrize('workload', ['wn18rr', 'fb15k237', 'wikidata5m'])
def test_layer_parity_at_baseline_shapes(k, workload):
    """The WHOLE layer - forward outputs and every gradient - at BASELINE.json's full shapes (configs[1..3]) against the
    float64 restatement of the reference (oracle.conv_fwd_bwd_big: edge-chunked, pinned on the CPU to the reference-order
    oracle), run on the same GPU as the checker.  Dropout p = 0.1 with injected keep masks.  Uses bench.py's own case
    builder and parity routine, so the number bench.py prints under `parity` is this one.  Bar: max-norm-relative error
    below 2e-5 for every tensor (two fp32 evaluations of the reference differ by 5e-6 .. 1e-4, SURVEY.md fact 9)."""
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location('kgc_bench', os.path.join(root, 'bench.py'))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    if workload == 'wikidata5m' and torch.cuda.get_device_properties(0).total_memory < 120 * (1 << 30):
        pytest.skip('needs a 180 GB B200')
    case = bench.LayerCase(k, orc, workload, torch.device('cuda', 0))
    try:
        par = bench.parity_vs_float64(case, orc)
        print(workload, {n: float('{:.2e}'.format(v)) for n, v in par['per_tensor'].items()})
        assert par['ok'], par
        # determinism at full size: a second step with the same masks gives the same bits
        m_in, m_out = case.masks(case.node_ids)
        case.conv.set_dropout_masks(m_in, m_out)
        ent1, _ = case.step()
        g1 = {n: v.clone() for n, v in case.grads().items()}
        ent1 = ent1.clone()
        ent2, _ = case.step()
        assert torch.equal(ent1, ent2)
        for n, v in case.grads().items():
            assert torch.equal(g1[n], v), n
    finally:
        del case
        k.plan._PLAN_CACHE.clear()
        torch.cuda.empty_cache()
