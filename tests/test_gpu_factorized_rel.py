"""The d_rel pass factorized by (object, type) group (plan.GroupedPlan): the numpy restatement of the grouped streams and of
the factorization (CPU), the device tables against the restatement bit for bit, the grouped kernels against the plain ones
through the C ABI, and the grouped layer against the float64 oracle and the plain layer."""
import numpy as np
import pytest
import torch

import mgcn_oracle as orc


@pytest.fixture(scope='module')
def k():
    import kgc_gcn_b200
    assert torch.cuda.is_available()
    kgc_gcn_b200._lib.lib()
    return kgc_gcn_b200


def plan_mod():
    import importlib
    return importlib.import_module('kgc_gcn_b200.plan')


def graph(kind, seed=3):
    """(edge_index [2, 2E], edge_type [2E], N, R) of the test graphs."""
    rng = np.random.default_rng(seed)
    if kind == 'toy':
        tri = np.array([[0, 0, 1], [2, 0, 1], [3, 1, 1], [1, 1, 0], [4, 0, 1], [0, 1, 2], [2, 1, 2]], dtype=np.int64)
        N, R = 6, 3                                    # entity 5 has no edge, type 2 has no edge
    elif kind == 'zipf':
        N, R = 700, 6
        tri = orc.synthetic_triples(N, R, 5000, seed)
    elif kind == 'zipf_many_types':
        N, R = 900, 40
        tri = orc.synthetic_triples(N, R, 7001, seed)  # 2E = 14,002 records: a partial last chunk
    elif kind == 'never_subject':
        N, R = 300, 4
        tri = orc.synthetic_triples(N, R, 2000, seed)
        tri = tri[tri[:, 0] != 7]                      # entity 7 is never a subject
        tri = tri[tri[:, 2] != 7]
    elif kind == 'hub':
        # one (object, type) group of 70,000 edges: 2,188 chunks, two fix-up levels
        N, R = 5000, 3
        hub = np.stack([rng.integers(1, N, 70000), np.zeros(70000, np.int64), np.zeros(70000, np.int64)], 1)
        tri = np.concatenate([hub, orc.synthetic_triples(N, R, 3000, seed)])
    elif kind == 'singletons':
        N, R = 400, 5                                  # every (object, type) pair once: no grouping
        o = rng.permutation(N)[:300]
        tri = np.stack([rng.integers(0, N, 300), rng.integers(0, R, 300), o], 1)
    else:
        raise ValueError(kind)
    g = orc.build_graph(np.ascontiguousarray(tri), N, R)
    return g['edge_index'], g['edge_attr'][0], N, R


def csr(key, n_rows):
    perm = np.argsort(key, kind='stable')
    return perm, np.searchsorted(key[perm], np.arange(n_rows + 1))


def grouped_host(ei, et, N, R):
    """The two grouped streams of GroupedPlan restated in numpy from the edge list (CSR by dst / src, stable)."""
    P = plan_mod()
    T = 2 * R + 1
    n2 = et.shape[0]
    n_in = n2 // 2
    src, dst = ei[0], ei[1]
    pd, rpd = csr(dst, N)
    f = P.build_grouped_stream(dst[pd], pd < n_in, et[pd], rpd, T, N, 2 * N)
    ps, rps = csr(src, N)
    s = P.build_grouped_stream(src[ps], ps >= n_in, et[ps], rps, T, 0, N)
    return (pd, f), (ps, s)


KINDS = ['toy', 'zipf', 'zipf_many_types', 'never_subject', 'hub', 'singletons']


@pytest.mark.parametrize('kind', KINDS)
def test_grouped_stream_restatement(kind):
    """CPU: the numpy restatement puts each row's plain records first (in CSR order), then one run per (row, type) group of
    the grouped half in (row, type) order; the segments tile the records and give every row one plain segment."""
    ei, et, N, R = graph(kind)
    T = 2 * R + 1
    n_in = et.shape[0] // 2
    eids = np.arange(et.shape[0])
    fwd, src = grouped_host(ei, et, N, R)
    # forward: rows of dst, in half grouped, plain rows N + dst, groups from 2 N; src: rows of src, out half grouped, plain
    # rows src, groups from N
    for (perm, g), grouped_half, row_of, base, gbase in ((fwd, eids < n_in, ei[1], N, 2 * N),
                                                         (src, eids >= n_in, ei[0], 0, N)):
        pos = perm[g['order']]                          # edge id of every re-sorted record
        assert np.array_equal(np.sort(g['order']), eids)
        beg, end, row = g['seg_beg'], g['seg_end'], g['seg_row']
        assert beg[0] == 0 and end[-1] == et.shape[0] and np.array_equal(beg[1:], end[:-1]) and (end >= beg).all()
        plain = row < gbase
        assert np.array_equal(np.sort(row[plain]), base + np.arange(N))
        assert np.array_equal(row[~plain] - gbase, np.arange(int((~plain).sum())))
        for b, e, r in zip(beg, end, row):
            recs = pos[b:e]
            if r < gbase:                               # plain: the row's plain-half edges in ascending edge id
                assert np.array_equal(recs, np.flatnonzero((row_of == r - base) & ~grouped_half))
            else:
                i = int(r - gbase)
                assert e > b and (row_of[recs] == g['grp_row'][i]).all() and (et[recs] == g['grp_type'][i]).all()
                assert grouped_half[recs].all() and (np.diff(recs) > 0).all()
        keys = g['grp_row'] * (T + 1) + g['grp_type']
        assert (np.diff(keys) > 0).all()
        sp = plan_mod().build_stream_plan(beg, end, row, et.shape[0])
        assert sp['rowflags'].shape[0] == et.shape[0]


@pytest.mark.parametrize('kind', ['toy', 'zipf', 'never_subject', 'hub'])
def test_factorization_float64(kind):
    """CPU, float64: agg_in, the out half's d_x term and d_rel computed from the group rows P / Q equal the per-edge sums."""
    ei, et, N, R = graph(kind)
    T, D = 2 * R + 1, 8
    rng = np.random.default_rng(1)
    n2 = et.shape[0]
    n_in = n2 // 2
    x, ee, rel = rng.standard_normal((N, D)), rng.standard_normal((n2, D)), rng.standard_normal((T, D))
    g_in, g_out, nrm = rng.standard_normal((N, D)), rng.standard_normal((N, D)), rng.random(n2)
    src, dst = ei[0], ei[1]
    (pd, f), (ps, s) = grouped_host(ei, et, N, R)
    # group rows from the streams: P over the forward stream's group segments, Q over the src stream's
    P = np.zeros((f['grp_row'].shape[0], D))
    for b, e, r in zip(f['seg_beg'], f['seg_end'], f['seg_row']):
        if r >= 2 * N:
            eids = pd[f['order'][b:e]]
            P[r - 2 * N] = (nrm[eids, None] * x[src[eids]] * ee[eids]).sum(0)
    Q = np.zeros((s['grp_row'].shape[0], D))
    for b, e, r in zip(s['seg_beg'], s['seg_end'], s['seg_row']):
        if r >= N:
            eids = ps[s['order'][b:e]]
            Q[r - N] = (nrm[eids, None] * g_out[dst[eids]] * ee[eids]).sum(0)
    ii, oo = np.arange(n_in), np.arange(n_in, n2)
    agg_in = np.zeros((N, D))
    np.add.at(agg_in, dst[ii], nrm[ii, None] * x[src[ii]] * rel[et[ii]] * ee[ii])
    got = np.zeros((N, D))
    np.add.at(got, f['grp_row'], rel[f['grp_type']] * P)
    np.testing.assert_allclose(got, agg_in, rtol=1e-12, atol=1e-12)
    dx_out = np.zeros((N, D))
    np.add.at(dx_out, src[oo], nrm[oo, None] * g_out[dst[oo]] * rel[et[oo]] * ee[oo])
    got = np.zeros((N, D))
    np.add.at(got, s['grp_row'], rel[s['grp_type']] * Q)
    np.testing.assert_allclose(got, dx_out, rtol=1e-12, atol=1e-12)
    d_rel = np.zeros((T, D))
    np.add.at(d_rel, et[ii], nrm[ii, None] * g_in[dst[ii]] * x[src[ii]] * ee[ii])
    np.add.at(d_rel, et[oo], nrm[oo, None] * g_out[dst[oo]] * x[src[oo]] * ee[oo])
    got = np.zeros((T, D))
    np.add.at(got, f['grp_type'], g_in[f['grp_row']] * P)
    np.add.at(got, s['grp_type'], x[s['grp_row']] * Q)
    np.testing.assert_allclose(got, d_rel, rtol=1e-12, atol=1e-12)


def test_group_reduce_schedule():
    """CPU: the group-reduce levels (fan-in 32, then 2,048) sum every segment exactly once; empty segments give a final
    item of their own."""
    P = plan_mod()
    rng = np.random.default_rng(0)
    lens = np.concatenate([rng.integers(0, 40, 300), [0, 70000, 33, 0]])
    end = np.cumsum(lens)
    beg = end - lens
    levels = P.build_levels(beg, end, np.arange(lens.shape[0]), P.GROUP_FAN_IN, P.CHUNK1)
    assert len(levels) == 3 and (levels[0][0][:, 1] - levels[0][0][:, 0]).max() <= P.GROUP_FAN_IN
    vals = rng.standard_normal(int(end[-1]))
    prev = None
    out = np.full(lens.shape[0], np.nan)
    for li, (items, n_part) in enumerate(levels):
        part = np.zeros(n_part)
        for b, e, o, fl in items:
            v = (vals if li == 0 else prev)[b:e].sum()
            if fl & 1:
                out[o] = v
            else:
                part[o] = v
        prev = part
    np.testing.assert_allclose(out, np.add.reduceat(np.append(vals, 0), beg) * (lens > 0), rtol=1e-12, atol=1e-9)


# ---------------------------------------------------------------------------------------------------------------- GPU
def device_plan(k, ei, et, N, R):
    return k.plan.GraphPlan(torch.from_numpy(ei).cuda(), torch.from_numpy(et).cuda(), N, 2 * R + 1)


@pytest.mark.gpu
@pytest.mark.parametrize('kind', ['toy', 'zipf', 'zipf_many_types', 'never_subject', 'hub'])
def test_grouped_plan_tables_on_device(k, monkeypatch, kind):
    """GroupedPlan's streams and tables equal the numpy restatement bit for bit (records, rowflags, chunks, fix-up items,
    source rows, group tables and their by-type order)."""
    monkeypatch.setattr(k.plan, 'GROUP_MAX_SHARE', 1.0)
    monkeypatch.setattr(k.plan, 'GROUP_MIN_EDGES', 0)
    ei, et, N, R = graph(kind)
    T = 2 * R + 1
    n_in = et.shape[0] // 2
    plan = device_plan(k, ei, et, N, R)
    grp = plan.grouped
    assert grp is not None
    (pd, f), (ps, s) = grouped_host(ei, et, N, R)
    rec_dst, rec_src = plan.rec_dst.cpu().numpy(), plan.rec_src.cpu().numpy()
    want_f = rec_dst[f['order']].copy()
    want_f[want_f[:, 0] < n_in, 2] = T - 1
    assert np.array_equal(grp.rec_f.cpu().numpy(), want_f)
    assert np.array_equal(grp.rec_s.cpu().numpy(), rec_src[s['order']])
    assert np.array_equal(grp.xrow_s.cpu().numpy(), ei[0][ps][s['order']])
    for g, sp_dev, prefill in ((f, grp.fwd, [(N, 2 * N)]), (s, grp.src, None)):
        want = k.plan.StreamPlan(k.plan.build_stream_plan(g['seg_beg'], g['seg_end'], g['seg_row'], et.shape[0]),
                                 et.shape[0], 'cuda', prefill_ranges=prefill)
        assert torch.equal(sp_dev.rowflags, want.rowflags) and torch.equal(sp_dev.chunks, want.chunks)
        assert sp_dev.n_carry == want.n_carry and sp_dev.prefill == want.prefill and len(sp_dev.levels) == len(want.levels)
        for la, lb in zip(sp_dev.levels, want.levels):
            assert torch.equal(la[0], lb[0]) and la[1:] == lb[1:]
    if kind == 'hub':
        assert len(grp.fwd.levels) == 2
    for name, key in (('grp_in_row', f['grp_row']), ('grp_in_type', f['grp_type']), ('grp_out_row', s['grp_row']),
                      ('grp_out_type', s['grp_type'])):
        assert np.array_equal(getattr(grp, name), key), name
    o_in = np.argsort(f['grp_type'], kind='stable')
    assert np.array_equal(grp.drel_in.prow.cpu().numpy(), o_in)
    assert np.array_equal(grp.drel_in.mrow.cpu().numpy(), f['grp_row'][o_in])
    assert grp.n_in_rows == plan.n_c[0]


def rel_err(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max()) / max(float(b.abs().max()), 1e-30)


@pytest.mark.gpu
@pytest.mark.parametrize('kind,D', [('zipf', 100), ('hub', 100), ('zipf_many_types', 200), ('never_subject', 36)])
def test_grouped_kernels_against_plain(k, monkeypatch, kind, D):
    """Through the C ABI on identical inputs: the grouped d_x pass gives d_ee bit for bit as kgc_agg_bwd_src, d_x and d_rel
    within 1e-6 of the plain passes; agg_in from the group rows within 1e-6 of the plain forward."""
    monkeypatch.setattr(k.plan, 'GROUP_MAX_SHARE', 1.0)
    monkeypatch.setattr(k.plan, 'GROUP_MIN_EDGES', 0)
    ei, et, N, R = graph(kind)
    T = 2 * R + 1
    plan = device_plan(k, ei, et, N, R)
    grp = plan.grouped
    L = k._lib
    p, st = L.ptr, L.stream
    gen = torch.Generator().manual_seed(4)
    n2 = et.shape[0]
    x = torch.randn(N, D, generator=gen).cuda()
    rel = torch.randn(T, D, generator=gen).cuda()
    rel[T - 1] = 0.5                                    # the self-loop row is never read by an edge
    ee = torch.randn(n2, D, generator=gen).cuda()
    g3 = torch.randn(3, N, D, generator=gen).cuda()
    # forward: plain agg_in vs group rows + kgc_group_reduce
    agg = torch.empty((2, N, D), device='cuda')
    plan.run_reduction(plan.fwd, lambda sp, o, c: L.call('kgc_agg_fwd', p(x), p(rel), T, p(ee), p(plan.rec_dst), p(sp.rowflags),
                                                          p(sp.chunks), sp.n_rec, p(o), p(c), D, st()), agg, D, tag='t')
    rel_f = torch.cat([rel[:T - 1], torch.ones((1, D), device='cuda')], 0)
    agg_g = torch.empty((2 * N + grp.n_in, D), device='cuda')
    plan.run_reduction(grp.fwd, lambda sp, o, c: L.call('kgc_agg_fwd', p(x), p(rel_f), T, p(ee), p(grp.rec_f), p(sp.rowflags),
                                                         p(sp.chunks), sp.n_rec, p(o), p(c), D, st()), agg_g, D, tag='tg')
    # the out half: same records in the same order, at other positions of the stream (other chunk boundaries, carry sums)
    assert rel_err(agg_g[N:2 * N], agg[1]) <= 1e-6
    agg_in = torch.zeros((N, D), device='cuda')
    grp.agg_in.run(plan, agg_g[2 * N:], rel, agg_in, D, tag='tgi')
    assert rel_err(agg_in, agg[0]) <= 1e-6
    agg_c = torch.empty((grp.n_in_rows, D), device='cuda')
    grp.agg_in_c.run(plan, agg_g[2 * N:], rel, agg_c, D, tag='tgc')
    assert torch.equal(agg_c, agg_in[plan.rows[0].long()])
    # backward: d_ee / d_x / d_rel
    d_ee, d_x = torch.empty_like(ee), torch.empty((N, D), device='cuda')
    plan.run_reduction(plan.bwd_src, lambda sp, o, c: L.call(
        'kgc_agg_bwd_src', p(x), p(rel), T, p(ee), p(g3), p(plan.rec_src), p(sp.rowflags), p(sp.chunks), sp.n_rec, N, n2 // 2,
        p(g3[2]), p(d_ee), p(o), p(c), D, st()), d_x, D, addend=g3[2], tag='ts')
    d_rel = torch.empty((T, D), device='cuda')
    plan.run_rel_reduction(lambda sp, o, c: L.call('kgc_agg_bwd_rel', p(x), p(ee), p(g3), p(plan.rec_type), p(sp.rowflags),
                                                    p(sp.chunks), sp.n_rec, N, n2 // 2, p(o), p(c), D, st()), d_rel, D, tag='tr')
    addend = torch.cat([g3[2], torch.zeros((grp.n_out, D), device='cuda')], 0)
    d_ee_g = torch.empty_like(ee)
    dxq = torch.empty((N + grp.n_out, D), device='cuda')
    plan.run_reduction(grp.src, lambda sp, o, c: L.call(
        'kgc_agg_bwd_src_grouped', p(x), p(rel), T, p(ee), p(g3), p(grp.rec_s), p(sp.rowflags), p(grp.xrow_s), p(sp.chunks),
        sp.n_rec, N, n2 // 2, grp.n_out, p(addend), p(d_ee_g), p(o), p(c), D, st()), dxq, D, addend=addend, tag='tsg')
    grp.dx.run(plan, dxq[N:], rel, dxq[:N], D, accumulate=True, tag='tgx')
    d_rel_g = torch.full((T, D), float('nan'), device='cuda')
    grp.drel_in.run(plan, agg_g[2 * N:], g3[0], d_rel_g, D, tag='tgri')
    grp.drel_out.run(plan, dxq[N:], x, d_rel_g, D, accumulate=True, tag='tgro')
    torch.cuda.synchronize()
    assert torch.equal(d_ee_g, d_ee)
    assert rel_err(dxq[:N], d_x) <= 1e-6, rel_err(dxq[:N], d_x)
    assert rel_err(d_rel_g, d_rel) <= 1e-6, rel_err(d_rel_g, d_rel)
    assert not bool(d_rel_g[T - 1].any())              # the self-loop type has no edge: written as zero


def run_layer(k, ei, et, p, g_ent, g_rel, R, d_in, d_out, dropout=0.0, masks=None):
    torch.manual_seed(0)
    conv = k.MGCNConv(d_in, d_out, 2 * R, dropout=dropout).cuda().train()
    with torch.no_grad():
        for name in ('loop_weight', 'in_weight', 'out_weight', 'rels_weight', 'loop_rel', 'loop_edge'):
            getattr(conv, name).copy_(p['w'][name])
    if masks is not None:
        conv.set_dropout_masks(torch.from_numpy(masks[0]), torch.from_numpy(masks[1]))
    x = p['x'].cuda().requires_grad_(True)
    ee = p['edge_embs'].cuda().requires_grad_(True)
    rl = p['rels'].cuda().requires_grad_(True)
    ent, rel = conv(x, torch.from_numpy(ei).cuda(), torch.from_numpy(et).cuda(), None, ee, rl)
    torch.autograd.backward([ent, rel], [g_ent.cuda(), g_rel.cuda()])
    out = {'all_ent': ent.detach(), 'all_rel': rel.detach(), 'd_x': x.grad, 'd_ee': ee.grad, 'd_rel': rl.grad}
    for name, prm in conv.named_parameters():
        out['d_' + name] = prm.grad
    return out


def force(monkeypatch, k, grouped, compact):
    k.plan._PLAN_CACHE.clear()
    monkeypatch.setattr(k.plan, 'GROUP_MAX_SHARE', 1.0 if grouped else -1.0)
    monkeypatch.setattr(k.plan, 'GROUP_MIN_EDGES', 0 if grouped else 1 << 62)
    monkeypatch.setattr(k.plan, 'COMPACT_MIN_PLANE_BYTES', -1 if compact else 1 << 62)


@pytest.mark.gpu
@pytest.mark.parametrize('d_in,compact,drop', [(100, False, None), (100, True, None), (200, False, 'masks'),
                                               (200, True, 'masks'), (100, True, 'kernel')])
def test_grouped_layer_vs_oracle_f64(k, monkeypatch, d_in, compact, drop):
    """The grouped layer against the float64 oracle at the 2e-5 bar, with and without compacted halves, with injected keep
    masks; with in-kernel dropout it agrees with the plain layer (same Philox draws)."""
    N, R, E, d_out = 3000, 7, 9000, 200
    tri = orc.synthetic_triples(N, R, E, 61)
    g = orc.build_graph(tri, N, R)
    ei, et = g['edge_index'], g['edge_attr'][0]
    p = orc.conv_params(N, R, E, d_in, d_out, seed=5)
    gen = torch.Generator().manual_seed(6)
    g_ent, g_rel = torch.randn(N, d_out, generator=gen), torch.randn(2 * R, d_out, generator=gen)
    masks = None
    if drop == 'masks':
        rng = np.random.default_rng(9)
        masks = ((rng.random((N, d_out)) >= 0.1).astype(np.uint8), (rng.random((N, d_out)) >= 0.1).astype(np.uint8))
    dropout = 0.0 if drop is None else 0.1
    force(monkeypatch, k, True, compact)
    plan = k.get_plan(torch.from_numpy(ei).cuda(), torch.from_numpy(et).cuda(), N, 2 * R + 1)
    assert plan.grouped is not None and plan.compact_halves(4 * d_out)[0] == compact
    got = run_layer(k, ei, et, p, g_ent, g_rel, R, d_in, d_out, dropout, masks)
    force(monkeypatch, k, False, compact)
    assert k.get_plan(torch.from_numpy(ei).cuda(), torch.from_numpy(et).cuda(), N, 2 * R + 1).grouped is None
    plain = run_layer(k, ei, et, p, g_ent, g_rel, R, d_in, d_out, dropout, masks)
    k.plan._PLAN_CACHE.clear()
    for name, w in plain.items():
        if name == 'd_ee':
            continue
        assert rel_err(got[name], w) <= 2e-6, (name, rel_err(got[name], w))
    assert rel_err(got['d_ee'], plain['d_ee']) <= 2e-6
    if drop == 'kernel':
        return
    dt = torch.float64
    w64 = {kk: v.to(dt) for kk, v in p['w'].items()}
    m64 = (None, None) if masks is None else (torch.from_numpy(masks[0]).to(dt), torch.from_numpy(masks[1]).to(dt))
    ent64, rel64, g64, _ = orc.conv_fwd_bwd(p['x'].to(dt), torch.from_numpy(ei), torch.from_numpy(et), p['edge_embs'].to(dt),
                                            p['rels'].to(dt), w64, g_ent, g_rel, mask_in=m64[0], mask_out=m64[1])
    pairs = {'all_ent': ent64, 'all_rel': rel64, 'd_x': g64['entity_embedding'], 'd_ee': g64['edge_embeddings'],
             'd_rel': g64['relation_embedding']}
    for name in ('loop_weight', 'in_weight', 'out_weight', 'rels_weight', 'loop_rel', 'loop_edge'):
        pairs['d_' + name] = g64['conv1.' + name]
    for name, truth in pairs.items():
        assert rel_err(got[name].cpu(), truth) <= 2e-5, (name, rel_err(got[name].cpu(), truth))


@pytest.mark.gpu
def test_grouped_layer_deterministic_and_graph_replay(k, monkeypatch):
    """Two grouped steps are bit-identical, and a CUDA-graph replay of the step equals the eager step."""
    N, R, E, d_in, d_out = 3000, 7, 9000, 100, 200
    tri = orc.synthetic_triples(N, R, E, 62)
    g = orc.build_graph(tri, N, R)
    ei, et = g['edge_index'], g['edge_attr'][0]
    p = orc.conv_params(N, R, E, d_in, d_out, seed=7)
    gen = torch.Generator().manual_seed(8)
    ge, gr = torch.randn(N, d_out, generator=gen).cuda(), torch.randn(2 * R, d_out, generator=gen).cuda()
    force(monkeypatch, k, True, True)
    conv = k.MGCNConv(d_in, d_out, 2 * R, dropout=0.0).cuda().train()
    with torch.no_grad():
        for name in ('loop_weight', 'in_weight', 'out_weight', 'rels_weight', 'loop_rel', 'loop_edge'):
            getattr(conv, name).copy_(p['w'][name])
    x = p['x'].cuda().requires_grad_(True)
    ee = p['edge_embs'].cuda().requires_grad_(True)
    rl = p['rels'].cuda().requires_grad_(True)
    ei_d, et_d = torch.from_numpy(ei).cuda(), torch.from_numpy(et).cuda()
    leaves = [x, ee, rl] + list(conv.parameters())
    assert k.get_plan(ei_d, et_d, N, 2 * R + 1).grouped is not None

    def step():
        for t in leaves:
            t.grad = None
        ent, rel = conv(x, ei_d, et_d, None, ee, rl)
        torch.autograd.backward([ent, rel], [ge, gr])
        return ent, rel
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        outs = []
        for _ in range(2):
            ent, rel = step()
            outs.append([ent.clone(), rel.clone()] + [t.grad.clone() for t in leaves])
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    want = outs[1]
    del ent, rel
    graph_ = torch.cuda.CUDAGraph()
    for t in leaves:
        t.grad = None
    with torch.cuda.graph(graph_):
        ent_g, rel_g = step()
    for _ in range(2):
        graph_.replay()
        torch.cuda.synchronize()
        for a, b in zip([ent_g, rel_g] + [t.grad for t in leaves], want):
            assert torch.equal(a, b)
    k.plan._PLAN_CACHE.clear()


@pytest.mark.gpu
def test_singleton_groups_take_the_plain_path(k, monkeypatch):
    """A graph whose (object, type) pairs are all distinct has nothing to factor: the plan keeps the plain streams."""
    monkeypatch.setattr(k.plan, 'GROUP_MIN_EDGES', 0)
    ei, et, N, R = graph('singletons')
    assert device_plan(k, ei, et, N, R).grouped is None


@pytest.mark.gpu
def test_small_bench_shapes_keep_the_plain_path(k, monkeypatch):
    """The WN18RR / FB15k-237 shapes are below GROUP_MIN_EDGES and keep the plain path; their groups would qualify (4.8 % /
    9.8 % of the edges per half)."""
    for N, R, E, seed in ((40943, 11, 86835, 0), (14541, 237, 272115, 1)):
        g = orc.build_graph(orc.synthetic_triples(N, R, E, seed), N, R)
        assert device_plan(k, g['edge_index'], g['edge_attr'][0], N, R).grouped is None
        monkeypatch.setattr(k.plan, 'GROUP_MIN_EDGES', 0)
        plan = device_plan(k, g['edge_index'], g['edge_attr'][0], N, R)
        assert plan.grouped is not None and plan.grouped.n_in <= 0.1 * E and plan.grouped.n_out == plan.grouped.n_in
        monkeypatch.undo()


@pytest.mark.gpu
def test_empty_graph_grouped(k, monkeypatch):
    """No edges at all with the grouped path forced: every group reduction has only empty items and writes zeros, so the
    layer equals the plain layer bit for bit."""
    N, R, d_in, d_out = 50, 2, 100, 200
    p = orc.conv_params(N, R, 0, d_in, d_out, seed=5)
    ei, et = np.zeros((2, 0), dtype=np.int64), np.zeros((0,), dtype=np.int64)
    gen = torch.Generator().manual_seed(6)
    g_ent, g_rel = torch.randn(N, d_out, generator=gen), torch.randn(2 * R, d_out, generator=gen)
    res = {}
    for grouped in (True, False):
        force(monkeypatch, k, grouped, True)
        assert (k.get_plan(torch.from_numpy(ei).cuda(), torch.from_numpy(et).cuda(), N, 2 * R + 1).grouped is not None) == grouped
        res[grouped] = run_layer(k, ei, et, p, g_ent, g_rel, R, d_in, d_out)
    k.plan._PLAN_CACHE.clear()
    for name, v in res[False].items():
        assert torch.equal(res[True][name], v), name
