"""CPU tests of the host logic: reduction plan scheduling, loader, epoch permutation, C-ABI exports.
No kernel is launched here (there is no GPU in the authoring container and no CPU fallback)."""
import ctypes
import json
import os
import re
from types import SimpleNamespace

import numpy as np
import pytest
import torch

import mgcn_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def simulate(levels, values, n_out):
    """Execute a reduction plan in numpy: what kgc_agg_fwd (level 0) + kgc_rows_reduce (levels >= 1) do."""
    out = np.full(n_out, np.nan)
    cur = values
    for items, n_part in levels:
        part = np.full(n_part, np.nan)
        for beg, end, o, flags in items.tolist():
            s = cur[beg:end].sum()
            if flags & 1:
                assert o == flags >> 1
                out[o] = s
            else:
                part[o] = s
        cur = part
    return out


@pytest.mark.parametrize('seed', [0, 1, 2])
def test_build_levels_exact(seed):
    from kgc_gcn_b200 import build_levels
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, 5, 400)
    lens[7], lens[100], lens[399] = 70000, 33, 1025 * 32 + 1      # hubs -> 3 levels
    ptr = np.concatenate([[0], np.cumsum(lens)])
    rows = rng.permutation(400)
    levels = build_levels(ptr[:-1], ptr[1:], rows, 32, 1024)
    assert len(levels) >= 2 and levels[-1][1] == 0
    vals = rng.integers(-5, 6, ptr[-1]).astype(np.float64)
    out = simulate(levels, vals, 400)
    exp = np.array([vals[ptr[i]:ptr[i + 1]].sum() for i in range(400)])
    np.testing.assert_array_equal(out[rows], exp)
    for items, _ in levels[:1]:
        assert (items[:, 1] - items[:, 0]).max() <= 32
    for items, _ in levels[1:]:
        assert (items[:, 1] - items[:, 0]).max() <= 1024


def test_build_levels_empty_rows_write_zero():
    from kgc_gcn_b200 import build_levels
    levels = build_levels(np.array([0, 0, 2]), np.array([0, 2, 2]), np.array([0, 1, 2]))
    assert len(levels) == 1
    assert levels[0][0].tolist() == [[0, 0, 0, 1], [0, 2, 1, 3], [2, 2, 2, 5]]


def simulate_stream(sp, values, n_out, chunk=32):
    """What kgc_agg_* (one warp per chunk) + kgc_rows_fill + kgc_rows_reduce do, in numpy."""
    out = np.full(n_out, np.nan)
    carry = np.full(max(sp['n_carry'], 1), np.nan)
    flags = sp['rowflags']
    n_rec = flags.shape[0]
    for c in range(sp['chunks'].shape[0]):
        head, tail = sp['chunks'][c]
        cb, ce = c * chunk, min((c + 1) * chunk, n_rec)
        started = bool(flags[cb] & (1 << 30))
        acc, open_row = 0.0, False
        for p in range(cb, ce):
            row = int(flags[p] & 0x3FFFFFFF)
            if flags[p] & (1 << 30):
                acc, started = 0.0, True
            open_row = True
            acc += values[p]
            if flags[p] & (1 << 31):
                if started:
                    assert np.isnan(out[row])
                    out[row] = acc
                else:
                    assert head >= 0 and np.isnan(carry[head])
                    carry[head] = acc
                open_row = False
        if open_row:
            assert tail >= 0 and np.isnan(carry[tail])
            carry[tail] = acc
    for r in sp['fill_rows']:
        assert np.isnan(out[r])
        out[r] = 0.0
    cur = carry
    for items, n_part in sp['levels']:
        part = np.full(n_part, np.nan)
        for beg, end, o, fl in items.tolist():
            s = cur[beg:end].sum()
            assert not np.isnan(s)
            if fl & 1:
                assert np.isnan(out[o])
                out[o] = s
            else:
                part[o] = s
        cur = part
    return out


@pytest.mark.parametrize('seed', [0, 1, 2, 3])
def test_stream_plan_exact(seed):
    """Every output row is produced exactly once and equals the segment sum, whatever the chunk alignment."""
    from kgc_gcn_b200 import build_stream_plan
    rng = np.random.default_rng(seed)
    S = 300
    lens = rng.integers(0, 6, S)
    lens[5], lens[100], lens[S - 1] = 40000, 33, 2048 * 32 * 3 + 7   # hubs: one and two fix-up levels
    if seed == 3:
        lens[:] = 0
        lens[17] = 5                                                   # almost everything empty
    ptr = np.concatenate([[0], np.cumsum(lens)])
    rows = rng.permutation(S)
    n_rec = int(ptr[-1])
    sp = build_stream_plan(ptr[:-1], ptr[1:], rows, n_rec)
    vals = rng.integers(-5, 6, n_rec).astype(np.float64)
    out = simulate_stream(sp, vals, S)
    exp = np.array([vals[ptr[i]:ptr[i + 1]].sum() for i in range(S)])
    np.testing.assert_array_equal(out[rows], exp)
    assert sp['chunks'].shape == (-(-n_rec // 32), 2)
    for items, _ in sp['levels']:
        assert (items[:, 1] - items[:, 0]).max() <= 2048


def test_stream_plan_forward_layout():
    """Two planes interleaved in record order (in half then out half of every dst row), as GraphPlan builds it."""
    from kgc_gcn_b200 import build_stream_plan
    rowptr = np.array([0, 3, 3, 70, 71])
    rowmid = np.array([1, 3, 40, 70])
    fb = np.stack([rowptr[:-1], rowmid], 1).reshape(-1)
    fe = np.stack([rowmid, rowptr[1:]], 1).reshape(-1)
    fr = np.stack([np.arange(4), np.arange(4) + 4], 1).reshape(-1)
    sp = build_stream_plan(fb, fe, fr, 71)
    vals = np.arange(71, dtype=np.float64)
    out = simulate_stream(sp, vals, 8)
    exp = np.zeros(8)
    for i in range(4):
        exp[i] = vals[rowptr[i]:rowmid[i]].sum()
        exp[4 + i] = vals[rowmid[i]:rowptr[i + 1]].sum()
    np.testing.assert_array_equal(out, exp)
    assert sorted(sp['fill_rows'].tolist()) == [1, 3, 5]


def params(**kw):
    base = dict(gcn_in_dim=20, gcn_out_dim=200, gcn_drop=0.0, hidden_drop=0.0, feat_drop=0.0, k_w=10, k_h=20,
                num_filter=2, kernel_size=7, bias=False, lbl_smooth=0.1, batch_size=128)
    base.update(kw)
    return SimpleNamespace(**base)


@pytest.fixture()
def toy_loader(golden_dir):
    import kgc_gcn_b200 as k
    cwd = os.getcwd()
    os.chdir(golden_dir)
    try:
        yield k.DataLoader('Toy', params())
    finally:
        os.chdir(cwd)


def test_loader_host_side(toy_loader, golden_dir):
    dl = toy_loader
    with open(os.path.join(golden_dir, 'toy_loader.json')) as f:
        gold = json.load(f)
    assert dl.entity2id == gold['entity2id'] and dl.relation2id == gold['relation2id']
    assert dl.graph.edge_index.tolist() == gold['edge_index']
    assert dl.graph.edge_attr.tolist() == gold['edge_attr']
    et, eid = dl.graph.edge_attr                      # unpackable like model.py:26
    assert eid.tolist() == list(range(20))
    np.testing.assert_array_equal(dl.graph.edge_norm.numpy(), np.asarray(gold['edge_norm'], dtype=np.float32))
    for key in gold['triplets']:
        got = [{'triple': list(q['triple']), 'label': sorted(q['label'])} for q in dl.triplets[key]]
        assert got == gold['triplets'][key]
    assert dl.graph.to('cpu') is dl.graph              # in-place .to (main.py:206 ignores the return value)


def test_dataset_csr_and_label_values(toy_loader):
    import kgc_gcn_b200 as k
    dl = toy_loader
    ds = dl._get_dataset('train', params())
    assert len(ds) == 17
    assert ds.ptr.tolist()[:4] == [0, 3, 4, 5] and ds.idx.tolist()[:5] == [1, 2, 3, 0, 0]
    pos, add = ds.label_values()
    ref = orc.make_label([2], 7, 0.1, True)
    assert np.float32(pos) == ref[2] and np.float32(add) == ref[0] and pos > 1.0      # the reference's quirk
    assert dl._get_dataset('valid_tail', params()).label_values() == (1.0, 0.0)
    trip, fptr, fidx = ds.sparse_batch([9, 0])
    assert trip.tolist() == [[6, 8, -1], [0, 0, -1]] and fptr.tolist() == [0, 2, 5] and fidx.tolist() == [0, 2, 1, 2, 3]
    with pytest.raises(ValueError):
        dl._get_dataset('bogus', params())
    with pytest.raises(RuntimeError, match='GPU only'):
        ds.build_batch([0, 1], 'cpu')                  # no CPU fallback


def test_epoch_permutation_matches_torch_dataloader():
    """Under the same torch.manual_seed the batch order equals the order of the reference's shuffle=True torch DataLoaders
    (data_loader.py:169-176) - a REAL DataLoader, whose iterator draws a base seed before the sampler draws its own - over
    several epochs, with and without worker processes."""
    from kgc_gcn_b200 import epoch_permutation
    n = 17
    for workers in (0, 2):
        dl = torch.utils.data.DataLoader(list(range(n)), batch_size=4, shuffle=True, num_workers=workers)
        torch.manual_seed(123)
        ref = [[int(v) for b in dl for v in b] for _ in range(3)]
        torch.manual_seed(123)
        got = [epoch_permutation(n).tolist() for _ in range(3)]
        assert got == ref, workers
    assert sorted(got[0]) == list(range(n))


def test_batch_iterator_lengths(toy_loader):
    dl = toy_loader
    it = dl.get_data_loaders(4, 0, params())
    assert len(it['train']) == 5 and len(it['valid_head']) == 2
    sizes = [len(b) for b in it['train'].batches()]
    assert sizes == [4, 4, 4, 4, 1]


def test_state_dict_names():
    import kgc_gcn_b200 as k
    m = k.MGCN(7, 5, 10, params(gcn_in_dim=8))
    keys = set(m.state_dict().keys())
    expect = {'entity_embedding', 'relation_embedding', 'edge_embeddings', 'conv1.loop_weight', 'conv1.in_weight',
              'conv1.out_weight', 'conv1.rels_weight', 'conv1.loop_rel', 'conv1.loop_edge', 'conv2.bias',
              'conv2.conv_e.weight', 'conv2.fc.weight', 'conv2.fc.bias'}
    for bn in ('conv1.ent_bn', 'conv2.bn0', 'conv2.bn1', 'conv2.bn2'):
        expect |= {bn + s for s in ('.weight', '.bias', '.running_mean', '.running_var', '.num_batches_tracked')}
    assert keys == expect
    assert m.entity_embedding.shape == (7, 8) and m.relation_embedding.shape == (10, 8)
    assert m.edge_embeddings.shape == (20, 8) and m.conv2.fc.weight.shape == (200, 14 * 14 * 2)


def test_arange_check_is_cached_per_owner_tensor(monkeypatch):
    """MGCN skips the identity gathers of model.py:29-30 when the index is arange; the (synchronising) check runs once per
    index tensor - also for ``edge_type, edge_ids = data.edge_attr`` (model.py:26), which makes a new view object per call -
    and again for a different tensor, whatever its address."""
    import kgc_gcn_b200 as k
    m = k.MGCN(7, 5, 10, params())
    evaluations = [0]
    real = torch.arange

    def counting(*a, **kw):
        evaluations[0] += 1
        return real(*a, **kw)
    attr = torch.stack([torch.zeros(20, dtype=torch.int64), real(20)])
    monkeypatch.setattr(torch, 'arange', counting)
    for _ in range(4):
        _, edge_ids = attr
        assert m._is_arange(edge_ids, 20)
    assert evaluations[0] == 1
    del attr, edge_ids
    for _ in range(3):                                  # new tensors (the allocator may hand out the old address again)
        _, edge_ids = torch.stack([torch.zeros(20, dtype=torch.int64), real(20).flip(0)])
        assert not m._is_arange(edge_ids, 20)
    assert not m._is_arange(real(5), 20) and m._is_arange(real(7), 7)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, 'kgc-gcn_b200')
    for fn in os.listdir(pkg):
        if fn.endswith('.py'):
            src = open(os.path.join(pkg, fn)).read()
            assert 'mgcn_oracle' not in src and 'oracle' not in re.findall(r'^\s*(?:from|import)\s+(\w+)', src, re.M), fn


def test_c_abi_exports_every_declared_symbol():
    """libkgc_b200.so loads and exports every function include/kgc_b200.h declares (no compute calls here)."""
    import kgc_gcn_b200 as k
    hdr = open(os.path.join(ROOT, 'include', 'kgc_b200.h')).read()
    hdr = re.sub(r'/\*.*?\*/', '', hdr, flags=re.S)
    declared = set(re.findall(r'\b(kgc_[a-z0-9_]+)\s*\(', hdr))
    assert len(declared) >= 17
    h = ctypes.CDLL(k._lib.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(h, name), 'missing export ' + name
    assert declared == set(k._lib.SIGNATURES), declared ^ set(k._lib.SIGNATURES)
    assert k._lib.lib().kgc_abi_version() == 1


def test_cpu_tensors_fail_loudly():
    import kgc_gcn_b200 as k
    conv = k.MGCNConv(8, 8, 4)
    ei = torch.tensor([[0, 1], [1, 0]])
    with pytest.raises(RuntimeError, match='CUDA'):
        conv(torch.zeros(2, 8), ei, torch.tensor([0, 2]), None, torch.zeros(2, 8), torch.zeros(4, 8))
    # the sampler extensions: GPU only, no CPU fallback either
    kb = k.KBDataset([{'triple': (0, 0, -1), 'label': [1, 2]}], 5, None)
    with pytest.raises(RuntimeError, match='GPU only'):
        kb.negatives([0], 2, device='cpu')
    dl = k.DataLoader.__new__(k.DataLoader)
    dl.num_edge, dl.num_relation = 1, 2
    dl.graph = k.GraphData(edge_index=ei, edge_attr=torch.tensor([[0, 2], [0, 1]]))
    with pytest.raises(RuntimeError, match='GPU only'):
        dl.sample_edges(1)


def test_uint32_draws_as_int32_bits():
    """data_loader._u32_bits: the samplers take uint32 draws as any integer tensor; the C ABI reads int32 bit patterns."""
    from kgc_gcn_b200.data_loader import _u32_bits
    vals = [0, 1, 2 ** 31 - 1, 2 ** 31, 2 ** 32 - 1, 2 ** 32 + 5]
    got = _u32_bits(torch.tensor(vals, dtype=torch.int64))
    assert got.dtype == torch.int32
    assert (got.numpy().view(np.uint32) == np.array([v % 2 ** 32 for v in vals], dtype=np.uint32)).all()
    same = torch.tensor([-1, 7], dtype=torch.int32)
    assert _u32_bits(same) is same or torch.equal(_u32_bits(same), same)


def _write_dataset(root, name, files):
    d = os.path.join(root, 'data', name)
    os.makedirs(d, exist_ok=True)
    for split, text in files.items():
        with open(os.path.join(d, split + '.txt'), 'wb') as f:
            f.write(text.encode('utf-8'))


def _load(root, name, native):
    import kgc_gcn_b200 as k
    cwd = os.getcwd()
    os.chdir(root)
    try:
        return k.DataLoader(name, params(native_ingest=native))
    finally:
        os.chdir(cwd)


def _same_loader(a, b):
    assert a.entity2id == b.entity2id and a.relation2id == b.relation2id
    assert list(a.entity2id) == list(b.entity2id) and list(a.relation2id) == list(b.relation2id)     # insertion order too
    assert (a.num_entity, a.num_relation, a.num_edge) == (b.num_entity, b.num_relation, b.num_edge)
    assert torch.equal(a.graph.edge_index, b.graph.edge_index) and torch.equal(a.graph.edge_attr, b.graph.edge_attr)
    assert torch.equal(a.graph.edge_norm, b.graph.edge_norm) and torch.equal(a.graph.entity, b.graph.entity)
    assert sorted(a.triplets.keys()) == sorted(b.triplets.keys())
    for key in b.triplets:
        qa, qb = a._get_dataset(key, params()), b._get_dataset(key, params())
        np.testing.assert_array_equal(qa.triples, qb.triples)
        np.testing.assert_array_equal(qa.ptr, qb.ptr)
        np.testing.assert_array_equal(qa.idx, qb.idx)
        assert [(tuple(q['triple']), sorted(q['label'])) for q in a.triplets[key]] == \
            [(tuple(q['triple']), sorted(q['label'])) for q in b.triplets[key]]
        assert all(('sub_samp' in q) == (key == 'train') for q in a.triplets[key])
        # sparse (CSR) batches for the fused scorer: same slices, and the group-indirect valid / test sets of the native
        # ingest serve them without expanding a per-query copy of every filter list
        fresh = a._get_dataset(key, params())
        rng = np.random.default_rng(len(qb))
        for _ in range(3):
            qid = rng.integers(0, len(qb), size=min(5, len(qb)))
            for x, y in zip(fresh.sparse_batch(qid), qb.sparse_batch(qid)):
                np.testing.assert_array_equal(x, y)
                assert x.dtype == y.dtype
        if getattr(fresh, '_lazy', None) is not None and key != 'train':
            assert fresh._ptr is None and fresh._lazy.qg is not None


def test_native_ingest_matches_python_passes(tmp_path, golden_dir):
    """N4 (csrc/ingest.cu) against the Python restatement of data_loader.py:64-111 on Toy and on random text with duplicate
    lines, blank lines, tabs / runs of spaces, CRLF and lone CR line ends, entities and relations that first appear in the
    valid / test files, and no trailing newline."""
    from kgc_gcn_b200.data_loader import LazyTriplets
    a, b = _load(golden_dir, 'Toy', True), _load(golden_dir, 'Toy', False)
    assert isinstance(a.triplets, LazyTriplets) and not isinstance(b.triplets, LazyTriplets)
    _same_loader(a, b)
    rng = np.random.default_rng(3)
    for case in range(4):
        n_ent, n_rel = int(rng.integers(5, 60)), int(rng.integers(1, 7))
        seps = [' ', '\t', '  ', ' \t ']
        ends = ['\n', '\r\n', '\n\n', '\r', '\n \n']

        def lines(n, lo_e, lo_r):
            out = []
            for _ in range(n):
                s, o = rng.integers(lo_e, n_ent, 2)
                r = rng.integers(lo_r, n_rel)
                sep = seps[int(rng.integers(len(seps)))]
                row = sep.join(['e%d' % s, 'rel_%d' % r, 'e%d' % o])
                out.append(('  ' if rng.random() < 0.2 else '') + row + ends[int(rng.integers(len(ends)))])
                if rng.random() < 0.15:
                    out.append(out[-1])                               # duplicate line
            return ''.join(out)
        files = {'train': lines(int(rng.integers(20, 200)), n_ent // 3, n_rel // 2),
                 'valid': lines(int(rng.integers(1, 40)), 0, 0), 'test': lines(int(rng.integers(1, 40)), 0, 0).rstrip()}
        _write_dataset(str(tmp_path), 'rand%d' % case, files)
        _same_loader(_load(str(tmp_path), 'rand%d' % case, True), _load(str(tmp_path), 'rand%d' % case, False))


def test_native_ingest_failures_and_fallbacks(tmp_path):
    """The reference's own failures stay: a line without three tokens raises ValueError, a token that only matches
    case-insensitively KeyError (data_loader.py:69-71 lower-cases, :83-85 does not).  Text the native parser does not
    reproduce exactly (non-ASCII tokens, relation names ending in _reverse) goes through the Python passes."""
    from kgc_gcn_b200.data_loader import LazyTriplets, native_ingest
    root = str(tmp_path)
    ok = 'a r b\nb r c\n'
    _write_dataset(root, 'short', {'train': 'a r b\nb r\n', 'valid': ok, 'test': ok})
    _write_dataset(root, 'case', {'train': 'a r b\nB r c\n', 'valid': ok, 'test': ok})
    _write_dataset(root, 'uni', {'train': 'a r b\nécole r c\n', 'valid': ok, 'test': ok})
    _write_dataset(root, 'rev', {'train': 'a r b\nb r_reverse c\n', 'valid': ok, 'test': ok})
    for native in (True, False):
        with pytest.raises(ValueError):
            _load(root, 'short', native)
        with pytest.raises(KeyError) as err:
            _load(root, 'case', native)
        assert 'B' in str(err.value)
    with pytest.raises(OSError):
        native_ingest(os.path.join(root, 'data', 'missing'))
    for name in ('uni', 'rev'):
        assert native_ingest(os.path.join(root, 'data', name)) is None
        dl = _load(root, name, True)
        assert not isinstance(dl.triplets, LazyTriplets)
        _same_loader(dl, _load(root, name, False))


def test_native_ingest_long_tokens_and_first_keyerror(tmp_path):
    """Tokens longer than the 16 bytes a hash slot stores inline (same 16-byte prefix, same length, differing only in the
    tail; a 16-byte token next to its 17-byte extension) keep distinct ids; the KeyError names the FIRST case-mismatched
    token in the reference's look-up order (train before valid before test; subject, relation, object within a line), and a
    malformed line anywhere wins over it (the vocabulary pass fails first, data_loader.py:64-71)."""
    root = str(tmp_path)
    pre = 'x' * 16
    names = [pre, pre + 'a', pre + 'b', pre + 'ab', pre + 'ba', 'x' * 15, 'y' * 40, 'y' * 39 + 'z']
    rng = np.random.default_rng(11)
    def lines(n):
        return ''.join('%s rel_%s_%d %s\n' % (names[rng.integers(len(names))], 'q' * 20, rng.integers(3), names[rng.integers(len(names))])
                       for _ in range(n))
    _write_dataset(root, 'long', {'train': lines(60), 'valid': lines(10), 'test': lines(10)})
    a = _load(root, 'long', True)
    _same_loader(a, _load(root, 'long', False))
    assert a.num_entity == len(set(names)) and a.num_relation == 3
    ok = 'a r b\nb r c\n'
    cases = {'k_rel': ({'train': 'a r b\nb R C\n', 'valid': ok, 'test': ok}, 'R'),
             'k_obj': ({'train': 'a r b\nb r C\nA r b\n', 'valid': ok, 'test': ok}, 'C'),
             'k_valid': ({'train': ok, 'valid': 'a r b\nb r Cc\n', 'test': 'Zz r b\n'}, 'Cc'),
             'k_long': ({'train': 'a r b\n' + pre + 'Tail r b\n', 'valid': ok, 'test': ok}, pre + 'Tail')}
    for name, (files, token) in cases.items():
        _write_dataset(root, name, files)
        for native in (True, False):
            with pytest.raises(KeyError) as err:
                _load(root, name, native)
            assert err.value.args[0] == token, (name, native, err.value.args)
    _write_dataset(root, 'k_short', {'train': 'A r b\n', 'valid': ok, 'test': 'a r\n'})
    for native in (True, False):
        with pytest.raises(ValueError):
            _load(root, 'k_short', native)


def test_gather_segments_edge_cases():
    from kgc_gcn_b200.data_loader import _gather_segments
    ptr = np.asarray([0, 0, 3, 3, 4], dtype=np.int64)          # rows of length 0, 3, 0, 1
    idx = np.asarray([7, 8, 9, 5], dtype=np.int32)
    p, v = _gather_segments(ptr, idx, [])
    assert p.tolist() == [0] and v.shape == (0,)
    p, v = _gather_segments(ptr, idx, [0, 2])
    assert p.tolist() == [0, 0, 0] and v.shape == (0,)
    p, v = _gather_segments(ptr, idx, [3, 1, 1, 0])
    assert p.tolist() == [0, 1, 4, 7, 7] and v.tolist() == [5, 7, 8, 9, 7, 8, 9] and v.dtype == np.int32


def test_checkpoint_interchanges_with_the_reference(tmp_path):
    """utils.save_checkpoint / load_checkpoint (reference utils.py:121-155): same files both ways - what ours writes the
    reference's own loader reads (oracle/_ref, when built) and vice versa; a stored checkpoint of the same state still loads,
    and both it and a fresh one load through the reference loader's own steps; best.ckpt follows is_best; the returned
    measure; a missing file raises; last.ckpt is replaced atomically."""
    import sys
    import kgc_gcn_b200 as k
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import build_ref
    ref = build_ref.load_reference()
    torch.manual_seed(3)
    model = torch.nn.Sequential(torch.nn.Linear(7, 5), torch.nn.BatchNorm1d(5))
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    model(torch.randn(4, 7)).sum().backward()
    opt.step()
    state = {'epoch': 3, 'state_dict': model.state_dict(), 'optim_dict': opt.state_dict(), 'measure': {'mrr': 0.25}}
    d = str(tmp_path / 'ckpt')
    k.save_checkpoint(state, False, d)
    assert os.path.exists(os.path.join(d, 'last.ckpt')) and not os.path.exists(os.path.join(d, 'best.ckpt'))
    k.save_checkpoint(state, True, d)
    assert os.path.samefile(os.path.join(d, 'last.ckpt'), os.path.join(d, 'best.ckpt'))       # a link, not a second copy
    state2 = dict(state, epoch=4)
    k.save_checkpoint(state2, False, d)                                  # best.ckpt keeps the epoch-3 file
    assert torch.load(os.path.join(d, 'best.ckpt'), weights_only=False)['epoch'] == 3
    assert torch.load(os.path.join(d, 'last.ckpt'), weights_only=False)['epoch'] == 4
    assert not [f for f in os.listdir(d) if f.endswith('.tmp')]

    def fresh():
        m = torch.nn.Sequential(torch.nn.Linear(7, 5), torch.nn.BatchNorm1d(5))
        return m, torch.optim.Adam(m.parameters(), lr=1e-3)

    def same(m, o):
        for a, b in zip(m.state_dict().values(), model.state_dict().values()):
            assert torch.equal(a, b)
        sa, sb = o.state_dict()['state'], opt.state_dict()['state']
        assert sa.keys() == sb.keys() and all(torch.equal(sa[i]['exp_avg'], sb[i]['exp_avg']) for i in sa)

    m, o = fresh()
    assert k.load_checkpoint(os.path.join(d, 'last.ckpt'), m, o) == {'mrr': 0.25}
    same(m, o)
    with pytest.raises(FileNotFoundError):
        k.load_checkpoint(os.path.join(d, 'nope.ckpt'), m)

    def close(m, o):                                  # same state, computed on another machine (last-bit differences)
        for a, b in zip(m.state_dict().values(), model.state_dict().values()):
            assert torch.allclose(a.float(), b.float(), rtol=1e-5, atol=1e-6)
        sa, sb = o.state_dict()['state'], opt.state_dict()['state']
        assert sa.keys() == sb.keys() and all(torch.allclose(sa[i]['exp_avg'], sb[i]['exp_avg'], rtol=1e-5, atol=1e-7) for i in sa)

    # tests/golden/ckpt_linear_bn_adam.ckpt: this same state (epoch 3) as save_checkpoint wrote it when the file was stored -
    # ours must keep reading it; and that file and the one written above load the way the reference's load_checkpoint
    # reads a checkpoint (utils.py:139-155: torch.load, then load_state_dict of 'state_dict' and of 'optim_dict')
    golden = os.path.join(ROOT, 'tests', 'golden', 'ckpt_linear_bn_adam.ckpt')
    m, o = fresh()
    assert k.load_checkpoint(golden, m, o) == {'mrr': 0.25}
    close(m, o)
    for path in (golden, os.path.join(d, 'best.ckpt')):
        ckpt = torch.load(path, map_location='cpu')
        m, o = fresh()
        m.load_state_dict(ckpt['state_dict'])
        o.load_state_dict(ckpt['optim_dict'])
        assert ckpt['epoch'] == 3 and ckpt.get('measure') == {'mrr': 0.25}
        close(m, o)
    if ref is None:                                   # the reference's own utils.py: only where KGC_REFERENCE_DIR built it
        return
    ref_utils = sys.modules['utils']
    m, o = fresh()
    assert ref_utils.load_checkpoint(os.path.join(d, 'best.ckpt'), m, o) == {'mrr': 0.25}     # ours -> reference
    same(m, o)
    d2 = str(tmp_path / 'ckpt_ref')
    ref_utils.save_checkpoint(state, True, d2)                                                # reference -> ours
    m, o = fresh()
    assert k.load_checkpoint(os.path.join(d2, 'best.ckpt'), m, o) == {'mrr': 0.25}
    same(m, o)


def test_rows_and_table_gradient_matches_autograd():
    """model._RowsAndTable: (table[idx], table) whose backward adds the rows' gradient INTO the dense table gradient - same
    gradients as index_select + plain use of the table, with duplicate indices, with and without a dense gradient."""
    from kgc_gcn_b200.model import _RowsAndTable
    torch.manual_seed(0)
    t = torch.randn(50, 8, dtype=torch.float64, requires_grad=True)
    idx = torch.tensor([3, 7, 3, 49, 0, 7, 7])
    w1, w2 = torch.randn(7, 8, dtype=torch.float64), torch.randn(50, 8, dtype=torch.float64)
    for use_table in (True, False):
        r, tt = _RowsAndTable.apply(t, idx)
        ((r * w1).sum() + ((tt * w2).sum() if use_table else 0)).backward()
        got, t.grad = t.grad.clone(), None
        ((t.index_select(0, idx) * w1).sum() + ((t * w2).sum() if use_table else 0)).backward()
        want, t.grad = t.grad.clone(), None
        assert torch.allclose(got, want, rtol=0, atol=1e-14)


def test_stream_plan_prefill_of_mostly_empty_planes():
    """plan.StreamPlan(prefill_ranges=...): a plane that is >= 3/4 rows without records (and large) is zero-filled by a
    memset - its empty rows leave the fix-up items - while a dense plane keeps its few empty rows as items; small plans
    never pre-fill.  Host logic only (CPU tensors)."""
    from kgc_gcn_b200.plan import build_stream_plan, StreamPlan
    rng = np.random.default_rng(0)
    Nd = 400000
    deg = np.zeros(2 * Nd, dtype=np.int64)
    deg[rng.choice(Nd, 20000, replace=False)] = rng.integers(1, 50, 20000)        # plane 0: 95% of the rows are empty
    deg[Nd:] = rng.integers(1, 5, Nd)                                             # plane 1: dense ...
    hole = Nd + rng.choice(Nd, 1000, replace=False)
    deg[hole] = 0                                                                 # ... but for 1,000 empty rows
    end = np.cumsum(deg)
    beg = end - deg
    sp = build_stream_plan(beg, end, np.arange(2 * Nd), int(end[-1]))
    n_empty = int((deg == 0).sum())
    assert sp['fill_rows'].shape[0] == n_empty
    plain = StreamPlan(sp, int(end[-1]), 'cpu')
    pre = StreamPlan(sp, int(end[-1]), 'cpu', prefill_ranges=[(0, Nd), (Nd, 2 * Nd)])
    assert plain.prefill == [] and pre.prefill == [(0, Nd)]
    items_plain = sum(l[1] for l in plain.levels)
    items_pre = sum(l[1] for l in pre.levels)
    assert items_plain - items_pre == int((deg[:Nd] == 0).sum())                  # plane 0's empty rows left the items
    first = pre.levels[0][0].numpy()
    empties = first[(first[:, 0] == 0) & (first[:, 1] == 0) & ((first[:, 3] & 1) == 1)]
    assert sorted(empties[:, 2].tolist()) == sorted(hole.tolist())                # plane 1's empty rows are still items
    small = build_stream_plan(beg[:2000], np.minimum(end[:2000], end[1999]), np.arange(2000), int(end[1999]))
    assert StreamPlan(small, int(end[1999]), 'cpu', prefill_ranges=[(0, 1000), (1000, 2000)]).prefill == []
