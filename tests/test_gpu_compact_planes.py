"""The single-GPU layer on compacted halves (plan.compact_halves): the occupied-row tables of the plan, and the layer's
outputs and gradients on the compact path against the dense path (bit for bit, apart from the weight gradient of a
compacted half, which sums fewer rows) and against the float64 oracle, in eager steps and graph replays."""
import numpy as np
import pytest
import torch

import mgcn_oracle as orc

pytestmark = pytest.mark.gpu

RTOL = 1e-5
D_IN, D_OUT = 100, 200


@pytest.fixture(scope='module')
def k():
    import kgc_gcn_b200
    assert torch.cuda.is_available()
    kgc_gcn_b200._lib.lib()
    return kgc_gcn_b200


def force(monkeypatch, k, mode):
    """'dense': no half compacted; 'sparse': the halves with at most half of their rows occupied; 'all': both halves."""
    monkeypatch.setattr(k.plan, 'COMPACT_MIN_PLANE_BYTES', -1)
    monkeypatch.setattr(k.plan, 'COMPACT_MAX_OCCUPANCY', {'dense': -1.0, 'sparse': 0.5, 'all': 1.0}[mode])
    monkeypatch.setenv('KGC_TAIL_PLANES', '3')          # the compact path always writes three planes: compare like with like


def graph(kind, N=3000, R=7, E=9000, seed=61):
    if kind == 'empty':
        return np.zeros((2, 0), dtype=np.int64), np.zeros((0,), dtype=np.int64), N, R, 0
    tri = orc.synthetic_triples(N, R, E, seed, uniform_obj=(kind == 'dense'))
    if kind == 'out_sparse':                            # objects <-> subjects: the out half carries the Zipf objects
        tri = np.ascontiguousarray(tri[:, ::-1])
    g = orc.build_graph(tri, N, R)
    return g['edge_index'], g['edge_attr'][0], N, R, E


def inputs(N, R, E, seed=5):
    p = orc.conv_params(N, R, E, D_IN, D_OUT, seed=seed)
    gen = torch.Generator().manual_seed(seed + 1)
    return p, torch.randn(N, D_OUT, generator=gen), torch.randn(2 * R, D_OUT, generator=gen)


def run(k, ei, et, p, g_ent, g_rel, R, dropout=0.1, out_drop=0.0, training=True):
    torch.manual_seed(0)                                # the same first dropout seed for every run
    conv = k.MGCNConv(D_IN, D_OUT, 2 * R, dropout=dropout).cuda().train(training)
    with torch.no_grad():
        for name in ('loop_weight', 'in_weight', 'out_weight', 'rels_weight', 'loop_rel', 'loop_edge'):
            getattr(conv, name).copy_(p['w'][name])
    x = p['x'].cuda().requires_grad_(True)
    ee = p['edge_embs'].cuda().requires_grad_(True)
    rl = p['rels'].cuda().requires_grad_(True)
    ent, rel = conv(x, torch.from_numpy(ei).cuda(), torch.from_numpy(et).cuda(), None, ee, rl, _out_drop=out_drop)
    torch.autograd.backward([ent, rel], [g_ent.cuda(), g_rel.cuda()])
    out = {'all_ent': ent.detach(), 'all_rel': rel.detach(), 'd_x': x.grad, 'd_ee': ee.grad, 'd_rel': rl.grad,
           'running_mean': conv.ent_bn.running_mean.clone(), 'running_var': conv.ent_bn.running_var.clone()}
    for name, prm in conv.named_parameters():
        out['d_' + name] = prm.grad
    return out


def rel_err(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max()) / max(float(b.abs().max()), 1e-30)


def test_rows_and_slots_match_the_edges(k):
    for kind in ('in_sparse', 'out_sparse', 'dense', 'empty'):
        ei, et, N, R, E = graph(kind)
        plan = k.plan.GraphPlan(torch.from_numpy(ei).cuda(), torch.from_numpy(et).cuda(), N, 2 * R + 1)
        dst = ei[1]
        for h, half in enumerate((dst[:E], dst[E:])):
            rows = np.unique(half).astype(np.int32)
            assert plan.n_c[h] == rows.size
            assert plan.rows[h].dtype == torch.int32 and np.array_equal(plan.rows[h].cpu().numpy(), rows)
            slot = np.full(N, -1, dtype=np.int32)
            slot[rows] = np.arange(rows.size, dtype=np.int32)
            assert plan.slot[h].dtype == torch.int32 and np.array_equal(plan.slot[h].cpu().numpy(), slot)


def test_compaction_rule(k):
    ei, et, N, R, E = graph('in_sparse')
    plan = k.plan.GraphPlan(torch.from_numpy(ei).cuda(), torch.from_numpy(et).cuda(), N, 2 * R + 1)
    assert plan.n_c[0] < 0.5 * N and plan.n_c[1] == N        # Zipf objects: sparse in half; every entity is a subject
    assert plan.compact_halves(4 * D_OUT) == (False, False)   # 2.4 MB planes: served from L2, never compacted
    big = (k.plan.COMPACT_MIN_PLANE_BYTES // (4 * D_OUT)) + 1
    assert 4 * D_OUT * big > k.plan.COMPACT_MIN_PLANE_BYTES
    # the rule as the plan applies it at a plane beyond L2 (same occupancy)
    rows = plan.num_dst_rows
    try:
        plan.num_dst_rows = big
        plan.n_c = [int(plan.n_c[0] * big / rows), big]
        assert plan.compact_halves(4 * D_OUT) == (True, False)
    finally:
        plan.num_dst_rows = rows


@pytest.mark.parametrize('kind,modes', [('in_sparse', ('sparse', 'all')), ('out_sparse', ('sparse', 'all')),
                                        ('dense', ('all',)), ('empty', ('all',))])
def test_compact_layer_is_the_dense_layer(k, monkeypatch, kind, modes):
    ei, et, N, R, E = graph(kind)
    p, g_ent, g_rel = inputs(N, R, E)
    for dropout, out_drop, training in ((0.1, 0.0, True), (0.1, 0.2, True), (0.0, 0.0, False)):
        force(monkeypatch, k, 'dense')
        want = run(k, ei, et, p, g_ent, g_rel, R, dropout, out_drop, training)
        for mode in modes:
            force(monkeypatch, k, mode)
            plan = k.get_plan(torch.from_numpy(ei).cuda(), torch.from_numpy(et).cuda(), N, 2 * R + 1)
            comp = plan.compact_halves(4 * D_OUT)
            assert any(comp)
            got = run(k, ei, et, p, g_ent, g_rel, R, dropout, out_drop, training)
            loose = {'d_in_weight'} if comp[0] else set()
            loose |= {'d_out_weight'} if comp[1] else set()
            for name, w in want.items():
                if name in loose:
                    assert rel_err(got[name], w) <= 1e-6, (kind, mode, name, rel_err(got[name], w))
                else:
                    assert torch.equal(got[name], w), (kind, mode, name, dropout, out_drop, training)


@pytest.mark.parametrize('kind', ['in_sparse', 'out_sparse'])
def test_compact_layer_vs_oracle_f64(k, monkeypatch, kind):
    ei, et, N, R, E = graph(kind)
    p, g_ent, g_rel = inputs(N, R, E)
    force(monkeypatch, k, 'all')
    got = run(k, ei, et, p, g_ent, g_rel, R, dropout=0.0)
    dt = torch.float64
    w64 = {kk: v.to(dt) for kk, v in p['w'].items()}
    ent64, rel64, g64, _ = orc.conv_fwd_bwd(p['x'].to(dt), torch.from_numpy(ei), torch.from_numpy(et), p['edge_embs'].to(dt),
                                            p['rels'].to(dt), w64, g_ent, g_rel)
    pairs = {'all_ent': ent64, 'all_rel': rel64, 'd_x': g64['entity_embedding'], 'd_ee': g64['edge_embeddings'],
             'd_rel': g64['relation_embedding']}
    for name in ('loop_weight', 'in_weight', 'out_weight', 'rels_weight', 'loop_rel', 'loop_edge'):
        pairs['d_' + name] = g64['conv1.' + name]
    for name, truth in pairs.items():
        assert rel_err(got[name].cpu(), truth) <= 2 * RTOL, (kind, name, rel_err(got[name].cpu(), truth))


def test_compact_layer_graph_replay(k, monkeypatch):
    """The compact path captured in a CUDA graph: replays give the eager step's outputs and gradients bit for bit."""
    ei, et, N, R, E = graph('in_sparse')
    p, g_ent, g_rel = inputs(N, R, E)
    force(monkeypatch, k, 'sparse')
    conv = k.MGCNConv(D_IN, D_OUT, 2 * R, dropout=0.0).cuda().train()
    with torch.no_grad():
        for name in ('loop_weight', 'in_weight', 'out_weight', 'rels_weight', 'loop_rel', 'loop_edge'):
            getattr(conv, name).copy_(p['w'][name])
    x = p['x'].cuda().requires_grad_(True)
    ee = p['edge_embs'].cuda().requires_grad_(True)
    rl = p['rels'].cuda().requires_grad_(True)
    ei_d, et_d, ge, gr = torch.from_numpy(ei).cuda(), torch.from_numpy(et).cuda(), g_ent.cuda(), g_rel.cuda()
    leaves = [x, ee, rl] + list(conv.parameters())
    assert k.get_plan(ei_d, et_d, N, 2 * R + 1).compact_halves(4 * D_OUT) == (True, False)

    def step():
        for t in leaves:
            t.grad = None
        ent, rel = conv(x, ei_d, et_d, None, ee, rl)
        torch.autograd.backward([ent, rel], [ge, gr])
        return ent, rel
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            ent, rel = step()
        want = [ent.clone(), rel.clone()] + [t.grad.clone() for t in leaves]
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    # nothing of the eager autograd graphs may outlive them: their gradient accumulators belong to another stream
    del ent, rel
    g = torch.cuda.CUDAGraph()
    for t in leaves:
        t.grad = None
    with torch.cuda.graph(g):
        ent_g, rel_g = step()
    for _ in range(3):
        g.replay()
        torch.cuda.synchronize()
        got = [ent_g, rel_g] + [t.grad for t in leaves]
        for a, b in zip(got, want):
            assert torch.equal(a, b)
