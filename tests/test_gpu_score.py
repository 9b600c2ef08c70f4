"""GPU parity tests of the fused scoring + filtered-rank path (K6, tcgen05/TMA) through the C ABI.

Bit-exact gate: integer rank counts given identical scores.  Inputs made of small integers are exactly
representable in bf16 and their dot products are exact in fp32 whatever the accumulation order, so the
tensor-core scores equal the oracle's and count_gt / count_eq / ranks must match bit for bit (ties are
frequent with integer scores, which exercises the == path).
Tolerance gate (bf16 operands): scores within 2^-7 relative of the fp32 product, and rank counts inside
the interval the oracle gives when the target margin is widened by that tolerance.
"""
import json
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import mgcn_oracle as orc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def k():
    import kgc_gcn_b200
    kgc_gcn_b200._lib.lib()
    return kgc_gcn_b200


def int_case(B, N, d, seed, nfilt=3):
    g = torch.Generator().manual_seed(seed)
    xq = torch.randint(-3, 4, (B, d), generator=g).float()
    tab = torch.randint(-3, 4, (N, d), generator=g).float()
    bias = torch.randint(-2, 3, (N,), generator=g).float()
    obj = torch.randint(0, N, (B,), generator=g)
    lens = torch.randint(0, 2 * nfilt + 1, (B,), generator=g).tolist()
    lists = []
    for q in range(B):          # sorted, unique; the target is in the list for half of the queries (as the reference's labels are)
        cand = set(torch.randperm(N, generator=g)[:min(lens[q], N)].tolist())
        if q % 2 == 0:
            cand.add(int(obj[q]))
        lists.append(sorted(cand))
    fptr = np.zeros(B + 1, dtype=np.int64)
    np.cumsum([len(x) for x in lists], out=fptr[1:])
    fidx = np.asarray([v for x in lists for v in x], dtype=np.int32)
    return xq, tab, bias, obj, fptr, fidx


def run_rank(k, xq, tab, bias, obj, fptr, fidx, count_eq=True):
    return k.filtered_rank(xq.cuda(), tab.cuda(), None if bias is None else bias.cuda(), obj.cuda(),
                           torch.from_numpy(fptr).cuda(), torch.from_numpy(fidx).cuda(), count_eq=count_eq)


@pytest.mark.parametrize('B,N,d', [(96, 400, 200), (300, 1000, 200), (1, 127, 200), (129, 129, 100), (257, 5000, 61),
                                   (640, 20000, 200)])
def test_rank_counts_bit_exact(k, B, N, d):
    xq, tab, bias, obj, fptr, fidx = int_case(B, N, d, seed=B + N)
    scores = (xq.double() @ tab.double().t() + bias.double()).numpy()
    gt, eq = orc.rank_counts(scores, fptr, fidx, obj.numpy())
    out = run_rank(k, xq, tab, bias, obj, fptr, fidx)
    np.testing.assert_array_equal(out['thr'].cpu().numpy(), scores[np.arange(B), obj.numpy()].astype(np.float32))
    np.testing.assert_array_equal(out['count_gt'].cpu().numpy(), gt)
    np.testing.assert_array_equal(out['count_eq'].cpu().numpy(), eq)
    np.testing.assert_array_equal(out['ranks'].cpu().numpy(), 1 + gt)
    sums = orc.metric_sums(1 + gt)
    got = dict(zip(k.scoring.SUM_KEYS, out['sums'].cpu().tolist()))
    for key, v in sums.items():
        assert abs(got[key] - v) <= 1e-4 * max(1.0, abs(v)), key
    # the reference's own dense formulation lands inside [1 + gt, 1 + gt + eq] (ties are implementation-defined there)
    lab = torch.zeros(B, N)
    for q in range(B):
        lab[q, torch.from_numpy(fidx[fptr[q]:fptr[q + 1]]).long()] = 1
    ref = orc.filtered_ranks_dense(torch.from_numpy(scores).float(), lab, obj).numpy()
    assert ((ref >= 1 + gt) & (ref <= 1 + gt + eq)).all()


def test_gt_only_variant_matches(k):
    xq, tab, bias, obj, fptr, fidx = int_case(200, 3000, 200, seed=5)
    a = run_rank(k, xq, tab, bias, obj, fptr, fidx, count_eq=True)
    b = run_rank(k, xq, tab, bias, obj, fptr, fidx, count_eq=False)
    assert torch.equal(a['ranks'], b['ranks'])


def test_pair_scores_exact_and_bias_split(k):
    g = torch.Generator().manual_seed(3)
    B, N, d = 200, 333, 200
    xq = torch.randint(-3, 4, (B, d), generator=g).float()
    tab = torch.randint(-3, 4, (N, d), generator=g).float()
    bias = torch.randn(N, generator=g) * 3                      # arbitrary fp32 bias: hi + mid + lo split must be exact
    table = k.EntityTable(tab.cuda(), bias.cuda())
    q16 = k.pack_queries(xq.cuda())
    pq = torch.randint(0, B, (1000,), generator=g).int()
    pe = torch.randint(0, N, (1000,), generator=g).int()
    s = k.pair_scores(q16, table, pq.cuda(), pe.cuda()).cpu()
    dots = (xq[pq.long()].double() * tab[pe.long()].double()).sum(1)
    ref = (dots + bias[pe.long()].double())
    # the dot is an exact integer; the three bias pieces add in fp32: error <= a few ulp of the sum
    assert float((s.double() - ref).abs().max()) <= 4e-7 * float(ref.abs().max())


def test_rank_random_floats_within_tolerance(k):
    g = torch.Generator().manual_seed(9)
    B, N, d = 512, 30000, 200
    xq = torch.randn(B, d, generator=g).abs()
    tab = torch.rand(N, d, generator=g) * 2 - 1
    bias = torch.randn(N, generator=g) * 0.1
    obj = torch.randint(0, N, (B,), generator=g)
    fptr = np.arange(0, 4 * B + 1, 4, dtype=np.int64)
    fidx = np.sort(torch.randint(0, N, (B, 4), generator=g).numpy().astype(np.int32), axis=1).reshape(-1)
    out = run_rank(k, xq, tab, bias, obj, fptr, fidx)
    x16, t16 = xq.bfloat16().double(), tab.bfloat16().double()
    scores = (x16 @ t16.t() + bias.double()).numpy()               # exact product of the bf16-rounded operands
    so = scores[np.arange(B), obj.numpy()]
    thr = out['thr'].cpu().double().numpy()
    tol = 2e-6 * np.abs(scores).max()                               # fp32 accumulation of 203 terms
    assert np.abs(thr - so).max() <= tol
    # operands rounded to bf16: scores within 2^-7 relative of the fp32 ones (stated tolerance of the bf16 path)
    full = (xq.double() @ tab.double().t() + bias.double()).numpy()
    assert np.abs(scores - full).max() <= 2.0 ** -7 * np.abs(full).max()
    keep = np.ones((B, N), dtype=bool)
    for q in range(B):
        keep[q, fidx[fptr[q]:fptr[q + 1]]] = False
        keep[q, obj[q]] = False
    lo = ((scores > (so + tol)[:, None]) & keep).sum(1)
    hi = ((scores > (so - tol)[:, None]) & keep).sum(1)
    gt = out['count_gt'].cpu().numpy()
    assert ((gt >= lo) & (gt <= hi)).all()
    assert (gt == ((scores > so[:, None]) & keep).sum(1)).mean() > 0.97


def test_full_sweep_properties_at_scale(k):
    """Size-independent properties at a BASELINE-like size (16k queries x 1M entities, d = 200):
    thr = -inf counts every entity exactly once for every query, thr = +inf counts none, and the
    integer-input counts equal an exact fp32 matmul of the same integers."""
    g = torch.Generator().manual_seed(1)
    B, N, d = 16384, 1000003, 200
    xq = torch.randint(-2, 3, (B, d), generator=g).float().cuda()
    tab = torch.randint(-2, 3, (N, d), generator=g, dtype=torch.int8).float().cuda()
    table = k.EntityTable(tab, None)
    q16 = k.pack_queries(xq)
    L = k._lib
    for thr_val, expect in ((-float('inf'), N), (float('inf'), 0)):
        thr = torch.full((B,), thr_val, device='cuda')
        gt = torch.zeros(B, dtype=torch.int32, device='cuda')
        L.call('kgc_score_rank', L.ptr(q16), L.ptr(table.data), B, N, table.kpad, L.ptr(thr), L.ptr(gt), None, L.stream())
        assert int(gt.min()) == expect and int(gt.max()) == expect
    thr = torch.randint(-20, 21, (B,), generator=g).float().cuda()
    gt = torch.zeros(B, dtype=torch.int32, device='cuda')
    eq = torch.zeros(B, dtype=torch.int32, device='cuda')
    L.call('kgc_score_rank', L.ptr(q16), L.ptr(table.data), B, N, table.kpad, L.ptr(thr), L.ptr(gt), L.ptr(eq), L.stream())
    ref_gt = torch.zeros(B, dtype=torch.int64, device='cuda')
    ref_eq = torch.zeros(B, dtype=torch.int64, device='cuda')
    for lo in range(0, N, 65536):                                # exact: small integers, |sum| < 2^24
        s = xq[:2048] @ tab[lo:lo + 65536].t()
        ref_gt[:2048] += (s > thr[:2048, None]).sum(1)
        ref_eq[:2048] += (s == thr[:2048, None]).sum(1)
    assert torch.equal(gt[:2048].long(), ref_gt[:2048]) and torch.equal(eq[:2048].long(), ref_eq[:2048])


def test_toy_predict_identical_metrics(k, golden_dir):
    """BASELINE.json north_star: bf16 scoring 'with identical MRR/hits@k on data/Toy' - our predict()/evaluate()
    against the sums the reference's own predict()/evaluate() produced for the same state dict."""
    prm = SimpleNamespace(gcn_in_dim=20, gcn_out_dim=200, gcn_drop=0.0, hidden_drop=0.0, feat_drop=0.0, k_w=10, k_h=20,
                          num_filter=2, kernel_size=7, bias=False, lbl_smooth=0.0, batch_size=128, device='cuda')
    cwd = os.getcwd()
    os.chdir(golden_dir)
    try:
        dl = k.DataLoader('Toy', prm)
    finally:
        os.chdir(cwd)
    dl.graph.to('cuda')
    z = np.load(os.path.join(golden_dir, 'toy_model.npz'))
    m = k.MGCN(dl.num_entity, dl.num_relation, dl.num_edge, prm)
    m.load_state_dict({kk[3:]: torch.from_numpy(z[kk]) for kk in z.files if kk.startswith('sd.')})
    m = m.cuda()
    with open(os.path.join(golden_dir, 'toy_metrics.json')) as f:
        gold = json.load(f)
    torch.manual_seed(5)
    iters = dl.get_data_loaders(4, 0, prm)
    for mode in ('tail', 'head'):
        res = k.predict(m, iters, dl.graph, 'valid', 'cuda', mode=mode + '_batch')
        for key, v in gold[mode].items():
            assert abs(res[key] - v) <= 1e-4 * max(1.0, abs(v)), (mode, key, res[key], v)
    ev = k.evaluate(m, iters, dl.graph, prm, 'valid')
    for key, v in gold['evaluate'].items():
        assert abs(float(ev[key]) - v) < 1e-5, (key, ev[key], v)
    # and through MGCN.rank for one explicit batch
    trip = torch.from_numpy(z['eval.tail.triple']).cuda()
    ds = dl._get_dataset('valid_tail', prm)
    _, fptr, fidx = ds.sparse_batch(np.arange(len(ds)))
    with torch.no_grad():
        m.eval()
        out = m.rank(trip[:, 0], trip[:, 1], trip[:, 2], torch.from_numpy(fptr).cuda(), torch.from_numpy(fidx).cuda(), dl.graph,
                     count_eq=True)
    lab = torch.from_numpy(np.stack([orc.make_label(q['label'], 7) for q in dl.triplets['valid_tail']]))
    ref = orc.filtered_ranks_dense(torch.from_numpy(z['eval.tail.score.f32']), lab, trip[:, 2].cpu()).numpy()
    np.testing.assert_array_equal(out['ranks'].cpu().numpy(), ref)


@pytest.mark.parametrize('B,N,D', [(128, 40943, 200), (77, 1001, 200), (5, 14, 32), (256, 3000, 100), (1, 130, 8), (300, 2000, 200), (600, 777, 64)])
def test_score_1n_training_path(k, B, N, D):
    """K6t: dense sigmoid scores (model.py:177-179) and their autograd on the 3xTF32 tensor-core kernels agree with the
    fp64 evaluation of the same expression to fp32 accuracy; nothing is written outside [B, N]."""
    from kgc_gcn_b200.scoring import score_1n, score_1n_supported
    g = torch.Generator().manual_seed(B * 7 + N)
    x = (torch.randn(B, D, generator=g) * 0.3).cuda().requires_grad_(True)
    ent = (torch.randn(N, D, generator=g) * 0.3).cuda().requires_grad_(True)
    bias = (torch.randn(N, generator=g) * 0.1).cuda().requires_grad_(True)
    label = (torch.rand(B, N, generator=g) < 0.01).float().cuda()
    assert score_1n_supported(x, ent)
    pred = score_1n(x, ent, bias)
    assert pred.shape == (B, N)
    loss = torch.nn.functional.binary_cross_entropy(pred, label)
    loss.backward()
    xd, ed, bd = (t.detach().double().requires_grad_(True) for t in (x, ent, bias))
    pred_ref = torch.sigmoid(xd @ ed.t() + bd)
    loss_ref = torch.nn.functional.binary_cross_entropy(pred_ref, label.double())
    loss_ref.backward()
    # fp32 tolerance: sigmoid output <= 1 -> absolute 2e-6; gradients relative to their largest entry
    assert float((pred.detach().double() - pred_ref.detach()).abs().max()) <= 2e-6
    assert abs(float(loss.detach()) - float(loss_ref.detach())) <= 2e-6 * max(1.0, abs(float(loss_ref.detach())))
    for got, ref, name in ((x.grad, xd.grad, 'x'), (ent.grad, ed.grad, 'ent'), (bias.grad, bd.grad, 'bias')):
        scale = float(ref.abs().max())
        err = float((got.double() - ref).abs().max())
        print('score_1n B={} N={} D={} d_{}: err {:.2e} / scale {:.2e}'.format(B, N, D, name, err, scale))
        assert err <= 2e-5 * scale + 1e-9, (name, err, scale)
    # deterministic
    x2, e2, b2 = (t.detach().clone().requires_grad_(True) for t in (x, ent, bias))
    torch.nn.functional.binary_cross_entropy(score_1n(x2, e2, b2), label).backward()
    assert torch.equal(x2.grad, x.grad) and torch.equal(e2.grad, ent.grad) and torch.equal(b2.grad, bias.grad)


def test_filtered_rank_exact_mode(k):
    """precision='fp32' (exact mode): ranks computed from fp32-grade dense logits (what the reference ranks, main.py:121-126)
    at a realistic entity count with CLOSELY spaced logits.  Against float64 scores every rank must lie in the interval
    allowed by an fp32-sized error band (1e-5 of the score scale) - where bf16-rounded operands (2^-7 relative) move ranks;
    on integer-valued inputs (exact in every precision) the two precisions agree bit for bit."""
    g = torch.Generator().manual_seed(11)
    B, N, d = 300, 40943, 200
    xq = torch.randn(B, d, generator=g).abs().cuda()
    tab = (torch.rand(N, d, generator=g) * 2 - 1).cuda()
    bias = (torch.randn(N, generator=g) * 0.1).cuda()
    obj = torch.randint(0, N, (B,), generator=g).cuda()
    fptr = torch.arange(0, 3 * B + 1, 3, dtype=torch.int64).cuda()
    fidx = torch.randint(0, N, (B, 3), generator=g).sort(1).values.reshape(-1).to(torch.int32).cuda()
    s64 = xq.double() @ tab.double().t() + bias.double()
    thr = s64[torch.arange(B, device='cuda'), obj]
    keep = torch.ones((B, N), dtype=torch.bool, device='cuda')
    keep[torch.arange(B, device='cuda').repeat_interleave(3), fidx.long()] = False
    keep[torch.arange(B, device='cuda'), obj] = False
    band = 1e-5 * float(s64.abs().max())
    lo = ((s64 > (thr + band)[:, None]) & keep).sum(1)
    hi = ((s64 > (thr - band)[:, None]) & keep).sum(1)
    exact = k.filtered_rank(xq, tab, bias, obj, fptr, fidx, count_eq=True, precision='fp32')
    r = exact['ranks'].long() - 1
    assert bool(((r >= lo) & (r <= hi)).all()), 'fp32-mode ranks outside the fp32 error band'
    gt64 = ((s64 > thr[:, None]) & keep).sum(1)
    fast = k.filtered_rank(xq, tab, bias, obj, fptr, fidx, count_eq=True)
    moved_fast = int((fast['ranks'].long() - 1 != gt64).sum())
    moved_exact = int((r != gt64).sum())
    print('ranks that differ from the float64 ranking: bf16 sweep {} / {}, fp32 mode {} / {}'.format(moved_fast, B, moved_exact, B))
    assert moved_exact <= moved_fast and moved_exact <= B // 50
    assert float((exact['thr'].double() - thr).abs().max()) <= 2e-6 * float(s64.abs().max())
    # integer-valued inputs: both precisions are exact, so they must agree bit for bit (incl. ties)
    xi = torch.randint(-3, 4, (B, d), generator=g).float().cuda()
    ti = torch.randint(-3, 4, (N, d), generator=g).float().cuda()
    bi = torch.randint(-2, 3, (N,), generator=g).float().cuda()
    a = k.filtered_rank(xi, ti, bi, obj, fptr, fidx, count_eq=True)
    b = k.filtered_rank(xi, ti, bi, obj, fptr, fidx, count_eq=True, precision='fp32')
    assert torch.equal(a['ranks'], b['ranks']) and torch.equal(a['count_eq'], b['count_eq']) and torch.equal(a['thr'], b['thr'])
    assert int(a['count_eq'].sum()) > 0                      # the integer case does contain ties
    from kgc_gcn_b200.scoring import tie_adjusted_sums
    opt = tie_adjusted_sums(a['ranks'], a['count_eq'], 'optimistic')
    assert torch.allclose(opt, a['sums'], rtol=1e-12, atol=1e-9)
    pes, mean = tie_adjusted_sums(a['ranks'], a['count_eq'], 'pessimistic'), tie_adjusted_sums(a['ranks'], a['count_eq'], 'mean')
    assert float(pes[1]) > float(mean[1]) > float(opt[1]) and float(pes[2]) < float(mean[2]) < float(opt[2])


def _restated_evaluate(data_dir, sd, prm):
    """evaluate() of main.py:80-135 on the valid split, restated by the oracle in float64 on the CPU (GCN + ConvE eval
    forward, sigmoid scores, the reference's dense filtered rank on float32 scores, its sums and rounding) - the same
    functions tests/test_oracle_golden.py holds to the reference's own predict() / evaluate() output stored in
    tests/golden (toy_model.npz, toy_metrics.json, rank_case.npz).  ``sd``: a state dict with the reference's names."""
    ds = orc.load_dataset(data_dir)
    N = ds['num_entity']
    g = orc.build_graph(ds['triples']['train'], N, ds['num_relation'])
    sd = {kk: v.detach().cpu().double() for kk, v in sd.items() if v.is_floating_point()}
    w = {kk[len('conv1.'):]: v for kk, v in sd.items() if kk.startswith('conv1.')}
    dec = {kk[len('conv2.'):]: v for kk, v in sd.items() if kk.startswith('conv2.')}
    ent, rel, _ = orc.conv_forward(sd['entity_embedding'], torch.from_numpy(g['edge_index']), torch.from_numpy(g['edge_attr'][0]),
                                   sd['edge_embeddings'], sd['relation_embedding'], w, training=False)
    sums = {}
    for mode in ('tail', 'head'):
        qs = ds['queries']['valid_' + mode]
        trip = torch.tensor([q['triple'] for q in qs], dtype=torch.long)
        sc = orc.score_tail(orc.conve_front(ent[trip[:, 0]], rel[trip[:, 1]], dec, prm.k_w, prm.k_h), ent, dec['bias'])
        lab = torch.from_numpy(np.stack([orc.make_label(q['label'], N) for q in qs]))
        sums[mode] = orc.metric_sums(orc.filtered_ranks_dense(sc.float(), lab, trip[:, 2]).numpy())
    return g, orc.combine_metrics(sums['tail'], sums['head'])


def test_predict_against_the_reference_at_realistic_size(k, tmp_path):
    """Our predict() / evaluate() on a synthetic data set of realistic size (8,000 entities, 24,000 training triples, 400
    validation triples) written as text files, with a seeded state dict spread so that the scores are not at their xavier
    init: MR / MRR / hits@k of the exact mode (precision='fp32') must equal, to the 5 places evaluate() rounds to unless a
    rank sits on an fp32 tie, (a) the float64 restatement of the reference's evaluate() that the golden fixtures pin
    (_restated_evaluate), and (b) when oracle/_ref is built (KGC_REFERENCE_DIR), the reference's OWN predict() / evaluate()
    (main.py:80-135, run on the CPU through oracle/shims) on the same state dict.  The bf16 sweep is reported next to it."""
    import build_ref
    ref = build_ref.load_reference()
    N, R, E = 8000, 12, 24000
    tri = orc.synthetic_triples(N, R, E + 800, 21)
    root = tmp_path / 'data' / 'Synth'
    root.mkdir(parents=True)
    for name, rows in (('train', tri[:E]), ('valid', tri[E:E + 400]), ('test', tri[E + 400:])):
        (root / (name + '.txt')).write_text('\n'.join('e{} r{} e{}'.format(s, r, o) for s, r, o in rows.tolist()) + '\n')
    prm = SimpleNamespace(gcn_in_dim=100, gcn_out_dim=200, gcn_drop=0.3, hidden_drop=0.3, feat_drop=0.3, k_w=10, k_h=20,
                          num_filter=32, kernel_size=7, bias=False, lbl_smooth=0.1, batch_size=128, device='cuda')
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        dl = k.DataLoader('Synth', prm)
        rdl = ref[1].DataLoader('Synth', prm) if ref is not None else None
    finally:
        os.chdir(cwd)
    torch.manual_seed(3)
    if ref is not None:
        assert dl.num_entity == rdl.num_entity and dl.num_edge == rdl.num_edge
        src = ref[0].MGCN(rdl.num_entity, rdl.num_relation, rdl.num_edge, prm)
    else:
        src = k.MGCN(dl.num_entity, dl.num_relation, dl.num_edge, prm)
    with torch.no_grad():                                    # spread the scores: a trained model is not at its xavier init
        src.conv2.bias.normal_(0, 0.5)
        src.entity_embedding.mul_(30.0)
    src.eval()
    m = k.MGCN(dl.num_entity, dl.num_relation, dl.num_edge, prm)
    m.load_state_dict(src.state_dict(), strict=True)
    m = m.cuda()
    g, restated = _restated_evaluate(str(root), src.state_dict(), prm)
    assert np.array_equal(g['edge_index'], dl.graph.edge_index.cpu().numpy())      # same entity / relation ids
    dl.graph.to('cuda')
    compare = {'restated reference (float64 oracle)': restated}
    if ref is not None:
        prm_cpu = SimpleNamespace(**dict(vars(prm), device='cpu'))
        torch.manual_seed(4)
        compare['reference'] = ref[2].evaluate(src, rdl.get_data_loaders(128, 0, prm_cpu), rdl.graph, prm_cpu, 'valid')
    iters = dl.get_data_loaders(128, 0, prm)
    ours = {p_: k.evaluate(m, iters, dl.graph, prm, 'valid', precision=p_) for p_ in ('fp32', 'bf16')}
    print(compare, 'fp32 mode', ours['fp32'], 'bf16 sweep', ours['bf16'])
    # the GCN / ConvE front end run with different summation orders on both sides (1e-6-level differences in the logits),
    # so a handful of near-tied ranks may differ by one place: MR within 0.05%, MRR / hits within 2.5e-3 (1 of 800 queries = 1.25e-3)
    for what, want in compare.items():
        assert set(want) == {'mr', 'mrr', 'hits@1', 'hits@3', 'hits@10'}, what
        for key, v in want.items():
            tol = 5e-4 * abs(v) if key == 'mr' else 2.5e-3
            assert abs(float(ours['fp32'][key]) - float(v)) <= tol, (what, key, ours['fp32'][key], v)
