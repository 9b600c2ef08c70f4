"""Filtered top-k entity prediction (K6k): ``topk`` / ``MGCN.topk`` on the fused tcgen05 sweep (bf16) and on the fp32-grade
dense logits (exact mode), and ``DataLoader.known_objects``.

The rule in both precisions: the eligible entities of a query (not in its exclusion list) sorted by (logit descending,
entity id ascending), the first k, padded with (-inf, -1).  On small-integer inputs every score is exact in bf16 and in
fp32, so both precisions must equal the numpy reference bit for bit, ties included.
"""
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import mgcn_oracle as orc

gpu = pytest.mark.gpu
KS = (1, 5, 10, 16, 17, 32)


@pytest.fixture(scope='module')
def k():
    import kgc_gcn_b200
    kgc_gcn_b200._lib.lib()
    return kgc_gcn_b200


def int_operands(B, N, d, seed):
    g = torch.Generator().manual_seed(seed)
    xq = torch.randint(-3, 4, (B, d), generator=g).float()
    tab = torch.randint(-3, 4, (N, d), generator=g).float()
    bias = torch.randint(-2, 3, (N,), generator=g).float()
    return xq, tab, bias


def csr(lists):
    ptr = np.zeros(len(lists) + 1, dtype=np.int64)
    np.cumsum([len(x) for x in lists], out=ptr[1:])
    idx = np.asarray([v for x in lists for v in x], dtype=np.int32)
    return ptr, idx


def exclusion_lists(B, N, mode, seed):
    """'none': no filter; 'random': sorted lists of up to 12 ids with duplicates and ids outside [0, N); 'few': every
    third row leaves only q % 4 entities eligible (the rest random), so that rows come back padded."""
    if mode == 'none':
        return None, None
    rng = np.random.default_rng(seed)
    lists = []
    for q in range(B):
        if mode == 'few' and q % 3 == 0:
            keep = rng.choice(N, size=q % 4, replace=False)
            lst = np.setdiff1d(np.arange(N), keep).tolist()
        else:
            lst = rng.integers(0, N, size=int(rng.integers(0, 13))).tolist()
            if q % 5 == 1 and lst:
                lst += lst[:2]                                   # duplicates
            if q % 7 == 2:
                lst += [-3, N, N + 5]                            # ignored: outside [0, N)
        lists.append(sorted(lst))
    return csr(lists)


def reference_order(scores, ptr, idx, kmax=32):
    """numpy: per row, the first kmax eligible ids of the stable sort by (-score, id)."""
    B, N = scores.shape
    out = []
    for q in range(B):
        keep = np.ones(N, dtype=bool)
        if ptr is not None:
            ex = idx[ptr[q]:ptr[q + 1]].astype(np.int64)
            keep[ex[(ex >= 0) & (ex < N)]] = False
        ids = np.nonzero(keep)[0]
        out.append(ids[np.lexsort((ids, -scores[q, ids]))][:kmax])
    return out


def reference_topk(scores, ptr, idx, kk, order=None):
    """(scores [B, kk] float32, ids [B, kk] int64, count [B] int32) with (-inf, -1) padding."""
    order = reference_order(scores, ptr, idx, kk) if order is None else order
    B = scores.shape[0]
    s_out = np.full((B, kk), -np.inf, dtype=np.float32)
    i_out = np.full((B, kk), -1, dtype=np.int64)
    cnt = np.zeros(B, dtype=np.int32)
    for q in range(B):
        o = order[q][:kk]
        s_out[q, :len(o)] = scores[q, o]
        i_out[q, :len(o)] = o
        cnt[q] = len(o)
    return s_out, i_out, cnt


def run(k, xq, tab, bias, kk, ptr, idx, precision, table=None):
    cu = lambda a: None if a is None else torch.from_numpy(a).cuda()          # noqa: E731
    return k.topk(xq.cuda(), None if tab is None else tab.cuda(), None if bias is None else bias.cuda(), kk, cu(ptr),
                  cu(idx), table=table, precision=precision)


def assert_equal_reference(out, ref, what):
    s, i, c = ref
    np.testing.assert_array_equal(out['count'].cpu().numpy(), c, err_msg=what)
    np.testing.assert_array_equal(out['ids'].cpu().numpy(), i, err_msg=what)
    np.testing.assert_array_equal(out['scores'].cpu().numpy(), s, err_msg=what)


@gpu
@pytest.mark.parametrize('B,N,d', [(1, 127, 200), (96, 129, 200), (129, 1000, 200), (300, 20000, 200), (640, 1000, 200),
                                   (640, 129, 200), (96, 20000, 61)])
def test_topk_bit_exact_integer_inputs(k, B, N, d):
    xq, tab, bias = int_operands(B, N, d, seed=B * 31 + N + d)
    scores = (xq.double() @ tab.double().t() + bias.double()).numpy()
    table = k.EntityTable(tab.cuda(), bias.cuda())
    for mode in ('none', 'random', 'few'):
        ptr, idx = exclusion_lists(B, N, mode, seed=B + N)
        order = reference_order(scores, ptr, idx)
        for kk in KS:
            ref = reference_topk(scores, ptr, idx, kk, order)
            for precision in ('bf16', 'fp32'):
                out = run(k, xq, tab, bias, kk, ptr, idx, precision, table=table if precision == 'bf16' else None)
                assert out['scores'].shape == (B, kk) and out['ids'].dtype == torch.int64 and out['count'].dtype == torch.int32
                assert_equal_reference(out, ref, '{} k={} {}'.format(mode, kk, precision))
            if mode == 'few' and kk == 32:
                assert (ref[2] < kk).any()                       # padded rows were exercised


@gpu
def test_topk_adversarial_orders(k):
    """bias[j] = j with zero operands: every entity beats the list and inserts.  All scores equal: the k lowest eligible
    ids.  A -0.0 / +0.0 mix: the zeros tie and go by id."""
    B, N, d = 130, 50000, 200
    xq = torch.zeros(B, d)
    tab = torch.zeros(N, d)
    for name, bias in (('increasing', torch.arange(N, dtype=torch.float32)),
                       ('equal', torch.full((N,), 3.0)),
                       ('signed zeros', torch.tensor([(-0.0, 0.0, 1.0, -0.0, 0.0, -1.0, -0.0)[j % 7] for j in range(N)]))):
        scores = bias.double().numpy()[None, :].repeat(B, 0)
        for mode in ('none', 'random'):
            ptr, idx = exclusion_lists(B, N, mode, seed=7)
            for kk in (10, 32):
                ref = reference_topk(scores, ptr, idx, kk)
                for precision in ('bf16', 'fp32'):
                    out = run(k, xq, tab, bias, kk, ptr, idx, precision)
                    assert_equal_reference(out, ref, '{} {} k={} {}'.format(name, mode, kk, precision))
                    if name == 'signed zeros':
                        assert not torch.signbit(out['scores'][out['scores'] == 0]).any()


def random_case(B, N, d, seed, n_excl=4):
    g = torch.Generator().manual_seed(seed)
    xq = torch.randn(B, d, generator=g).abs()
    tab = torch.rand(N, d, generator=g) * 2 - 1
    bias = torch.randn(N, generator=g) * 0.1
    ptr = np.arange(0, n_excl * B + 1, n_excl, dtype=np.int64)
    idx = np.sort(torch.randint(0, N, (B, n_excl), generator=g).numpy().astype(np.int32), axis=1).reshape(-1)
    return xq, tab, bias, ptr, idx


def band_checks(s64, ptr, idx, ids, kk, band):
    """Every returned id scores within ``band`` of the float64 k-th eligible score or above it; every eligible id that
    beats the k-th score by more than ``band`` is returned.  Returns the number of rows whose id set differs from float64."""
    B, N = s64.shape
    moved = 0
    for q in range(B):
        keep = np.ones(N, dtype=bool)
        keep[idx[ptr[q]:ptr[q + 1]]] = False
        got = ids[q]
        assert keep[got].all()
        elig = np.nonzero(keep)[0]
        order = elig[np.lexsort((elig, -s64[q, elig]))]
        kth = s64[q, order[kk - 1]]
        assert (s64[q, got] >= kth - band).all(), q
        must = elig[s64[q, elig] > kth + band]
        assert np.isin(must, got).all(), q
        moved += int(set(got.tolist()) != set(order[:kk].tolist()))
    return moved


@gpu
def test_topk_consistent_with_kernel_scores(k):
    """bf16 sweep, random floats: returned scores are kgc_score_pairs' scores bit for bit; kgc_score_rank with the k-th
    score as threshold (corrected for the exclusions) puts fewer than k eligible entities strictly above it and at least k
    at or above it; against float64 every id lies within the bf16 band of the k-th score."""
    B, N, d, kk = 300, 30000, 200, 10
    xq, tab, bias, ptr, idx = random_case(B, N, d, seed=9)
    table = k.EntityTable(tab.cuda(), bias.cuda())
    out = run(k, xq, tab, bias, kk, ptr, idx, 'bf16', table=table)
    assert bool((out['count'] == kk).all())
    q16 = k.pack_queries(xq.cuda())
    rows = torch.arange(B, dtype=torch.int32).repeat_interleave(kk).cuda()
    s_pair = k.pair_scores(q16, table, rows, out['ids'].reshape(-1).to(torch.int32).contiguous())
    assert torch.equal(s_pair.view(B, kk), out['scores'])
    L = k._lib
    thr = out['scores'][:, kk - 1].contiguous()
    gt = torch.zeros(B, dtype=torch.int32, device='cuda')
    eq = torch.zeros(B, dtype=torch.int32, device='cuda')
    L.call('kgc_score_rank', L.ptr(q16), L.ptr(table.data), B, N, table.kpad, L.ptr(thr), L.ptr(gt), L.ptr(eq), L.stream())
    uniq = [np.unique(idx[ptr[q]:ptr[q + 1]]) for q in range(B)]      # a duplicate exclusion is one entity
    er = torch.cat([torch.full((len(u),), q, dtype=torch.int32) for q, u in enumerate(uniq)]).cuda()
    ei = torch.from_numpy(np.concatenate(uniq).astype(np.int32)).cuda()
    s_ex = k.pair_scores(q16, table, er, ei)
    ex_gt = torch.zeros(B, dtype=torch.int64, device='cuda').index_add_(0, er.long(), (s_ex > thr[er.long()]).long())
    ex_ge = torch.zeros(B, dtype=torch.int64, device='cuda').index_add_(0, er.long(), (s_ex >= thr[er.long()]).long())
    assert bool(((gt.long() - ex_gt) < kk).all())
    assert bool(((gt.long() + eq.long() - ex_ge) >= kk).all())
    full = (xq.double() @ tab.double().t() + bias.double()).numpy()
    band = 2.0 ** -7 * np.abs(full).max()
    # each score is within the band of float64 (test_rank_random_floats_within_tolerance), so two scores move by 2 bands
    band_checks(full, ptr, idx, out['ids'].cpu().numpy(), kk, 2 * band)


@gpu
def test_topk_exact_mode_random_floats(k):
    """precision='fp32': scores within 4e-6 max|s| of float64, ids consistent with float64 within an fp32-sized band, and
    no more rows whose id set differs from the float64 answer than the bf16 sweep has.  The score bar is twice the 2e-6 of
    the exact-mode rank test: the top k are the extreme logits, where all 200 products share a sign and the 3xTF32 split
    error of kgc_score_1n_logits adds up instead of cancelling (2.1e-6 max|s| measured on a B200 for this case)."""
    B, N, d, kk = 300, 40943, 200, 10
    xq, tab, bias, ptr, idx = random_case(B, N, d, seed=11, n_excl=3)
    s64 = (xq.double() @ tab.double().t() + bias.double()).numpy()
    scale = np.abs(s64).max()
    exact = run(k, xq, tab, bias, kk, ptr, idx, 'fp32')
    ids = exact['ids'].cpu().numpy()
    got = s64[np.arange(B)[:, None], ids]
    err = np.abs(exact['scores'].cpu().double().numpy() - got).max()
    print('fp32 mode: top-{} scores within {:.2e} max|s| of float64'.format(kk, err / scale))
    assert err <= 4e-6 * scale
    moved_exact = band_checks(s64, ptr, idx, ids, kk, 2e-5 * scale)
    fast = run(k, xq, tab, bias, kk, ptr, idx, 'bf16')
    moved_fast = band_checks(s64, ptr, idx, fast['ids'].cpu().numpy(), kk, 2 * 2.0 ** -7 * scale)
    print('rows whose top-{} set differs from float64: bf16 sweep {} / {}, fp32 mode {} / {}'.format(
        kk, moved_fast, B, moved_exact, B))
    assert moved_exact <= moved_fast


@gpu
def test_topk_at_scale_many_chunks(k):
    """2,048 integer queries against 1,000,003 entities (many work items per query, a large merge) against a chunked torch
    matmul + stable sort, with 4 exclusions per query."""
    g = torch.Generator().manual_seed(1)
    B, N, d = 2048, 1000003, 200
    xq = torch.randint(-2, 3, (B, d), generator=g).float().cuda()
    tab = torch.randint(-2, 3, (N, d), generator=g, dtype=torch.int8).float().cuda()
    bias = torch.randint(-2, 3, (N,), generator=g).float().cuda()
    ex = torch.randint(0, N, (B, 4), generator=g).sort(1).values.cuda()
    ptr = torch.arange(0, 4 * B + 1, 4, dtype=torch.int64).cuda()
    idx = ex.reshape(-1).to(torch.int32).contiguous()
    table = k.EntityTable(tab, bias)
    for kk in (10, 32):
        best_s = torch.empty((B, 0), device='cuda')
        best_i = torch.empty((B, 0), dtype=torch.int64, device='cuda')
        for lo in range(0, N, 65536):                            # exact: small integers
            s = xq @ tab[lo:lo + 65536].t() + bias[lo:lo + 65536]
            hit = (ex >= lo) & (ex < lo + s.shape[1])
            s[torch.arange(B, device='cuda')[:, None].expand_as(ex)[hit], (ex - lo)[hit]] = -float('inf')
            cs, ci = torch.sort(s, dim=1, descending=True, stable=True)
            # earlier chunks first: among equal scores the lower id keeps the earlier position
            best_s = torch.cat([best_s, cs[:, :kk]], 1)
            best_i = torch.cat([best_i, ci[:, :kk] + lo], 1)
            best_s, o = torch.sort(best_s, dim=1, descending=True, stable=True)
            best_i = best_i.gather(1, o)
            best_s, best_i = best_s[:, :kk], best_i[:, :kk]
        for precision in ('bf16', 'fp32'):
            out = k.topk(xq, tab, bias, kk, ptr, idx, table=table if precision == 'bf16' else None, precision=precision)
            assert torch.equal(out['ids'], best_i), (kk, precision)
            assert torch.equal(out['scores'], best_s), (kk, precision)
            assert bool((out['count'] == kk).all())


@gpu
def test_topk_deterministic(k):
    B, N, d = 640, 50000, 200
    xq, tab, bias, ptr, idx = random_case(B, N, d, seed=5)
    for precision, kk in (('bf16', 10), ('bf16', 32), ('fp32', 17)):
        a = run(k, xq, tab, bias, kk, ptr, idx, precision)
        b = run(k, xq, tab, bias, kk, ptr, idx, precision)
        assert all(torch.equal(a[key], b[key]) for key in ('scores', 'ids', 'count')), precision


def _toy_loader(k, golden_dir, native=True):
    prm = SimpleNamespace(gcn_in_dim=20, gcn_out_dim=200, gcn_drop=0.0, hidden_drop=0.0, feat_drop=0.0, k_w=10, k_h=20,
                          num_filter=2, kernel_size=7, bias=False, lbl_smooth=0.0, batch_size=128, device='cuda',
                          native_ingest=native)
    cwd = os.getcwd()
    os.chdir(golden_dir)
    try:
        return k.DataLoader('Toy', prm), prm
    finally:
        os.chdir(cwd)


@gpu
def test_toy_model_topk_matches_oracle_logits(k, golden_dir):
    """MGCN.topk on the stored Toy model: ids in the order of the float64 oracle logits wherever neighbouring logits differ
    by more than 1e-5 relative, with and without the known-facts filter, in both precisions."""
    dl, prm = _toy_loader(k, golden_dir)
    dl.graph.to('cuda')
    z = np.load(os.path.join(golden_dir, 'toy_model.npz'))
    sd = {kk[3:]: torch.from_numpy(z[kk]) for kk in z.files if kk.startswith('sd.')}
    m = k.MGCN(dl.num_entity, dl.num_relation, dl.num_edge, prm)
    m.load_state_dict(sd)
    m = m.cuda().eval()
    sd64 = {kk: v.double() for kk, v in sd.items() if v.is_floating_point()}
    w = {kk[len('conv1.'):]: v for kk, v in sd64.items() if kk.startswith('conv1.')}
    dec = {kk[len('conv2.'):]: v for kk, v in sd64.items() if kk.startswith('conv2.')}
    ei, ea = dl.graph.edge_index.cpu(), dl.graph.edge_attr.cpu()
    ent, rel, _ = orc.conv_forward(sd64['entity_embedding'], ei, ea[0], sd64['edge_embeddings'], sd64['relation_embedding'],
                                   w, training=False)
    N = dl.num_entity
    trip = np.concatenate([dl._get_dataset(s, prm).triples for s in ('valid_tail', 'valid_head', 'test_tail')])
    src, rel_ = torch.from_numpy(trip[:, 0]), torch.from_numpy(trip[:, 1])
    logits = orc.score_tail(orc.conve_front(ent[src], rel[rel_], dec, prm.k_w, prm.k_h), ent, dec['bias'], sigmoid=False).numpy()
    kk = min(10, N)
    for exclude in (None, dl.known_objects(src, rel_)):
        ptr, idx = (None, None) if exclude is None else (exclude[0].cpu().numpy(), exclude[1].cpu().numpy())
        _, ref_i, ref_c = reference_topk(logits, ptr, idx, kk)
        for precision in ('bf16', 'fp32'):
            with torch.no_grad():
                out = m.topk(src.cuda(), rel_.cuda(), dl.graph, k=kk, exclude=exclude, precision=precision)
            ids, cnt = out['ids'].cpu().numpy(), out['count'].cpu().numpy()
            np.testing.assert_array_equal(cnt, ref_c)
            for q in range(len(trip)):
                ls = logits[q, ref_i[q, :ref_c[q]]]
                for i in range(ref_c[q]):
                    # the position is determined when the logit is separated from both neighbours (and from the first
                    # entity left out, for the last place)
                    nb = [ls[i - 1]] if i > 0 else []
                    nb += [ls[i + 1]] if i + 1 < ref_c[q] else []
                    if i + 1 == ref_c[q]:
                        rest = np.ones(N, dtype=bool)
                        rest[ref_i[q, :ref_c[q]]] = False
                        if ptr is not None:
                            rest[idx[ptr[q]:ptr[q + 1]]] = False
                        if rest.any():
                            nb.append(logits[q, rest].max())
                    if all(abs(ls[i] - v) > 1e-5 * max(abs(ls[i]), abs(v)) for v in nb):
                        assert ids[q, i] == ref_i[q, i], (precision, exclude is None, q, i)


def _synth_text(root, N=300, R=6, E=1500, seed=4):
    tri = orc.synthetic_triples(N, R, E + 200, seed)
    d = os.path.join(root, 'data', 'Synth')
    os.makedirs(d, exist_ok=True)
    for name, rows in (('train', tri[:E]), ('valid', tri[E:E + 100]), ('test', tri[E + 100:])):
        with open(os.path.join(d, name + '.txt'), 'w') as f:
            f.write('\n'.join('e{} r{} e{}'.format(s, r, o) for s, r, o in rows.tolist()) + '\n')
    return root


def test_known_objects_is_the_all_split_filter(k, golden_dir, tmp_path):
    """CPU: for every valid / test query (s, r, o) - tail and head direction - known_objects(s, r) is the query's label
    list (the reference's all-split filter), on both loader paths; an (s, r) that occurs nowhere gives an empty row."""
    roots = {'Toy': golden_dir, 'Synth': _synth_text(str(tmp_path))}
    for name, root in roots.items():
        for native in (True, False):
            prm = SimpleNamespace(native_ingest=native, lbl_smooth=0.0)
            cwd = os.getcwd()
            os.chdir(root)
            try:
                dl = k.DataLoader(name, prm)
            finally:
                os.chdir(cwd)
            for key in ('valid_tail', 'valid_head', 'test_tail', 'test_head'):
                qs = dl.triplets[key]
                trip = np.asarray([q['triple'] for q in qs], dtype=np.int64).reshape(-1, 3)
                ptr, idx = dl.known_objects(torch.from_numpy(trip[:, 0]), trip[:, 1])
                assert ptr.dtype == torch.int64 and idx.dtype == torch.int32 and ptr.device == dl.graph.device
                ptr, idx = ptr.numpy(), idx.numpy()
                assert len(ptr) == len(qs) + 1
                for q, item in enumerate(qs):
                    assert idx[ptr[q]:ptr[q + 1]].tolist() == sorted(item['label']), (name, native, key, q)
            # an unknown pair: relation id beyond any triple's relation for entity 0 in both directions
            ptr, idx = dl.known_objects([0, dl.num_entity - 1], [2 * dl.num_relation - 1, 0])
            assert ptr[0] == 0 and int(ptr[-1]) == len(idx)


@gpu
def test_topk_argument_errors(k):
    xq, tab, bias = int_operands(4, 200, 200, seed=1)
    xq, tab, bias = xq.cuda(), tab.cuda(), bias.cuda()
    ptr = torch.tensor([0, 2, 3, 3, 5], dtype=torch.int64).cuda()
    idx = torch.tensor([1, 7, 4, 9, 11], dtype=torch.int32).cuda()
    k.topk(xq, tab, bias, 3, ptr, idx)
    for bad_k in (0, 33, -1, 2.0):
        with pytest.raises(ValueError):
            k.topk(xq, tab, bias, bad_k, ptr, idx)
    with pytest.raises(ValueError):                                  # row 0 unsorted
        k.topk(xq, tab, bias, 3, ptr, torch.tensor([7, 1, 4, 9, 11], dtype=torch.int32).cuda())
    with pytest.raises(ValueError):                                  # wrong length
        k.topk(xq, tab, bias, 3, ptr[:-1].contiguous(), idx)
    with pytest.raises(ValueError):                                  # decreasing ptr
        k.topk(xq, tab, bias, 3, torch.tensor([0, 3, 2, 3, 5], dtype=torch.int64).cuda(), idx)
    with pytest.raises(ValueError):
        k.topk(xq, tab, bias, 3, ptr, None)
    with pytest.raises(ValueError):
        k.topk(xq, tab, bias, 3, precision='fp16')
    with pytest.raises(RuntimeError):
        k.topk(xq.cpu(), tab.cpu(), bias.cpu(), 3)
    with pytest.raises(RuntimeError):
        k.topk(xq, tab, bias, 3, ptr.cpu(), idx.cpu())
    # rows that cross a row boundary downwards are fine: [9, 11] after [4]
    out = k.topk(xq, tab, bias, 3, ptr, idx)
    assert out['ids'].shape == (4, 3)
