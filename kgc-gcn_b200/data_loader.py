"""DataLoader / KBDataset: drop-in mirrors of the reference data layer (data_loader.py:17-192).

Host side (Python, as in the reference): vocabulary + id assignment, (s, r) -> objects grouping, query
lists, the bi-directional edge list.  Device side: the per-step work - epoch permutation, the dense
multi-hot [B, N] label with the reference's label smoothing, the [B, 3] triple gather - runs in K5
(kgc_label_build) straight into device memory from a query -> objects CSR, replacing the per-query
Python loop of KBDataset.get_label and the B*N*4-byte host-to-device copy of every step.
Sparse (CSR) batches for the fused scorer are offered next to the dense reference-compatible ones.
"""
import logging
import os
from collections import OrderedDict, defaultdict

import numpy as np
import torch

from . import _lib


class GraphData(object):
    """Stand-in for torch_geometric.data.Data as the reference uses it (data_loader.py:151-155):
    tensor attributes ``edge_index``, ``edge_attr`` (unpackable as edge_type, edge_ids - model.py:26),
    ``entity``, ``edge_norm``, plus ``num_nodes``; ``.to(device)`` moves them IN PLACE because
    main.py:206 ignores the return value."""

    def __init__(self, edge_index=None, edge_attr=None, **kwargs):
        self.edge_index, self.edge_attr = edge_index, edge_attr
        for k, v in kwargs.items():
            setattr(self, k, v)

    def to(self, device):
        for k, v in list(self.__dict__.items()):
            if torch.is_tensor(v):
                setattr(self, k, v.to(device))
        return self

    @property
    def device(self):
        return self.edge_index.device


def _u32_bits(draws):
    """uint32 draws as the int32 bit patterns the C ABI reads (int32 / uint32 tensors are taken as they are, wider
    integer tensors are reduced modulo 2^32)."""
    if draws.dtype == torch.int32:
        return draws.contiguous()
    if draws.dtype == torch.uint32:
        return draws.contiguous().view(torch.int32)
    d = draws.to(torch.int64) & 0xFFFFFFFF
    return torch.where(d >= (1 << 31), d - (1 << 32), d).to(torch.int32).contiguous()


def _gather_segments(ptr, idx, rows):
    """Concatenation of idx[ptr[r]:ptr[r + 1]] for r in rows -> (new_ptr [len(rows) + 1], values), vectorised."""
    rows = np.asarray(rows, dtype=np.int64)
    lens = ptr[rows + 1] - ptr[rows]
    out_ptr = np.zeros(rows.shape[0] + 1, dtype=np.int64)
    np.cumsum(lens, out=out_ptr[1:])
    total = int(out_ptr[-1])
    if total == 0:
        return out_ptr, idx[:0]
    pos = np.arange(total, dtype=np.int64) - np.repeat(out_ptr[:-1], lens) + np.repeat(ptr[rows], lens)
    return out_ptr, idx[pos]


class QuerySet(object):
    """One query set as the native ingest delivers it: triples [Q, 3] int64 and the sorted unique objects of the queries
    as CSR.  Train: ``gptr`` / ``gidx`` are per query (``qg`` None).  Valid / test: they hold every referenced (s, r) group
    ONCE and ``qg`` [Q] maps a query to its group - a hub group is the filter of thousands of queries; the per-query
    ``ptr`` / ``idx`` form is expanded only when somebody asks for it (dense label batches).
    ``as_list()`` gives the reference's list of dicts (data_loader.py:98-111)."""

    def __init__(self, triples, gptr, gidx, train, qg=None):
        self.triples, self.gptr, self.gidx, self.train, self.qg = triples, gptr, gidx, train, qg
        self._flat = None

    def __len__(self):
        return int(self.triples.shape[0])

    def segments(self, qid):
        """(ptr [len(qid) + 1], idx) of the queries ``qid`` without expanding the whole set."""
        qid = np.asarray(qid, dtype=np.int64)
        return _gather_segments(self.gptr, self.gidx, qid if self.qg is None else self.qg[qid])

    @property
    def flat(self):
        """Per-query (ptr, idx) of the whole set."""
        if self._flat is None:
            self._flat = (self.gptr, self.gidx) if self.qg is None else self.segments(np.arange(len(self)))
        return self._flat

    def as_list(self):
        out = []
        ptr, idx = self.flat
        trip, ptr, idx = self.triples.tolist(), ptr.tolist(), idx.tolist()
        for q, t in enumerate(trip):
            d = {'triple': tuple(t), 'label': idx[ptr[q]:ptr[q + 1]]}
            if self.train:
                d['sub_samp'] = 1
            out.append(d)
        return out


class LazyTriplets(dict):
    """``DataLoader.triplets`` when the data came through the native ingest: the five query sets as QuerySet objects,
    turned into the reference's lists of dicts on first access of a key."""

    def __init__(self, sets):
        super(LazyTriplets, self).__init__()
        self._sets = sets
        for k in sets:
            dict.__setitem__(self, k, None)

    def __getitem__(self, key):
        v = dict.__getitem__(self, key)
        if v is None:
            v = self._sets[key].as_list()
            dict.__setitem__(self, key, v)
        return v

    def query_set(self, key):
        return self._sets[key]


def native_ingest(data_dir):
    """N4 (csrc/ingest.cu): the two text passes of the reference loader in C++.  Returns a dict of numpy arrays and token
    lists, or None when the text is outside what the native parser reproduces exactly (non-ASCII tokens, relation names
    ending in ``_reverse``).  Malformed lines raise ValueError, tokens that only match case-insensitively KeyError - the
    reference's own failures."""
    import ctypes
    h = _lib.lib()
    handle = ctypes.c_void_p()
    rc = h.kgc_ingest_open(os.fsencode(data_dir), ctypes.byref(handle))
    if rc != 0:
        msg = h.kgc_last_error().decode(errors='replace')
        if rc == 2:
            return None
        if rc == 1:
            raise ValueError(msg)
        if rc == 4:
            raise KeyError(msg)
        raise OSError(msg)
    try:
        def arr(array, n, dtype):
            a = np.empty(n, dtype=dtype)
            if h.kgc_ingest_copy(handle, array, a.ctypes.data_as(ctypes.c_void_p), a.nbytes) != 0:
                raise RuntimeError(h.kgc_last_error().decode())
            return a
        cnt = lambda what: int(h.kgc_ingest_count(handle, what))      # noqa: E731
        def names(array):                      # one blob instead of one call per token
            blob = arr(array, (cnt(array),), np.uint8).tobytes().decode('ascii')
            return blob.split('\n')[:-1] if blob else []
        out = {'entities': names(5), 'relations': names(6)}
        assert len(out['entities']) == cnt(0) and len(out['relations']) == cnt(1)
        for k, split in enumerate(('train', 'valid', 'test')):
            out[split] = arr(2 + k, (cnt(2 + k), 3), np.int64)
        for q, name in enumerate(('train', 'valid_tail', 'valid_head', 'test_tail', 'test_head')):
            nq, nnz, rows = cnt(10 + 2 * q), cnt(11 + 2 * q), cnt(20 + q)
            out['q_' + name] = QuerySet(arr(10 + 3 * q, (nq, 3), np.int64), arr(11 + 3 * q, (rows + 1,), np.int64),
                                        arr(12 + 3 * q, (nnz,), np.int32), train=(q == 0),
                                        qg=None if q == 0 else arr(30 + q, (nq,), np.int32))
        return out
    finally:
        h.kgc_ingest_close(handle)


class KBDataset(object):
    """Query set in CSR form.  ``triplets`` is the reference's list of {'triple': (s, r, o), 'label': [objs]}."""

    def __init__(self, triplets, num_entity, params, training=False):
        self.num_entity = int(num_entity)
        self.params = params
        self.training = training
        if isinstance(triplets, QuerySet):                       # CSR arrays straight from the native ingest (N4)
            self._triplets = None
            self._lazy = triplets
            self.triples = triplets.triples
            self._ptr = self._idx = None                           # per-query form: expanded on first use
        else:
            self._triplets = triplets
            self._lazy = None
            q = len(triplets)
            self.triples = np.asarray([t['triple'] for t in triplets], dtype=np.int64).reshape(q, 3)
            self._ptr = np.zeros(q + 1, dtype=np.int64)
            idx = []
            for i, t in enumerate(triplets):
                objs = sorted(int(o) for o in t['label'])
                idx.extend(objs)
                self._ptr[i + 1] = len(idx)
            self._idx = np.asarray(idx, dtype=np.int32)
        self._dev = {}

    @property
    def ptr(self):
        if self._ptr is None:
            self._ptr, self._idx = self._lazy.flat
        return self._ptr

    @property
    def idx(self):
        if self._idx is None:
            self._ptr, self._idx = self._lazy.flat
        return self._idx

    @property
    def triplets(self):
        """The reference's list of {'triple': ..., 'label': [...]} (materialised on first use when the data came as CSR)."""
        if self._triplets is None:
            self._triplets = self._lazy.as_list()
        return self._triplets

    def label_values(self):
        """(pos, add): label = add everywhere, pos on the positives.  Training with lbl_smooth != 0 gives
        (1 - ls) * y + 1 / N (data_loader.py:41-43 - note 1/N, not ls/N), evaluated in float32 like numpy does."""
        ls = float(getattr(self.params, 'lbl_smooth', 0.0) or 0.0)
        if self.training and ls != 0.0:
            add = np.float32(1.0 / self.num_entity)
            pos = np.float32(np.float32(1.0 - ls) * np.float32(1.0) + add)
            return float(pos), float(add)
        return 1.0, 0.0

    def device_csr(self, device):
        key = str(device)
        if key not in self._dev:
            self._dev[key] = tuple(torch.from_numpy(a).to(device) for a in (self.triples, self.ptr, self.idx))
        return self._dev[key]

    def build_batch(self, qid, device):
        """K5: (triple[B,3] int64, label[B,N] float32) on ``device`` for the query ids ``qid``."""
        device = torch.device(device)
        if device.type != 'cuda':
            raise RuntimeError('label/batch build runs on the GPU only (no CPU fallback); move the graph with '
                               'graph.to("cuda") before get_data_loaders')
        triples, ptr, idx = self.device_csr(device)
        qid = torch.as_tensor(qid, dtype=torch.int64).to(device, non_blocking=True)
        b = int(qid.numel())
        triple = torch.empty((b, 3), dtype=torch.int64, device=device)
        label = torch.empty((b, self.num_entity), dtype=torch.float32, device=device)
        pos, add = self.label_values()
        p = _lib.ptr
        with torch.cuda.device(device):
            _lib.call('kgc_label_build', p(qid), b, p(triples), p(ptr), p(idx), self.num_entity, pos, add, p(triple),
                      p(label), _lib.stream())
        return triple, label

    def negatives(self, qid, k, draws=None, tries=4, device='cuda', generator=None):
        """GPU negative sampler (extension: the reference trains 1-N and ships no sampler, SURVEY.md fact 2).  ``k``
        entities per query of ``qid`` that are NOT among the query's known objects -> int32 [B, k] on ``device``; -1 where
        all ``tries`` candidates of a slot collided.  A pure function of ``draws`` (uint32 [B, k, tries], candidate =
        (u * N) >> 32); when omitted they come from torch's generator (``generator`` or the global one on the device)."""
        device = torch.device(device)
        if device.type != 'cuda':
            raise RuntimeError('the negative sampler runs on the GPU only (no CPU fallback)')
        _, ptr, idx = self.device_csr(device)
        qid = torch.as_tensor(qid, dtype=torch.int64).to(device)
        b = int(qid.numel())
        if draws is None:
            draws = torch.randint(0, 1 << 32, (b, int(k), int(tries)), dtype=torch.int64, device=device, generator=generator)
        draws = torch.as_tensor(draws).to(device)
        if tuple(draws.shape) != (b, int(k), int(tries)):
            raise ValueError('draws must be [len(qid), k, tries]')
        d32 = _u32_bits(draws)
        neg = torch.empty((b, int(k)), dtype=torch.int32, device=device)
        p = _lib.ptr
        with torch.cuda.device(device):
            _lib.call('kgc_neg_sample', p(qid), b, p(ptr), p(idx), self.num_entity, p(d32), int(k), int(tries), p(neg), _lib.stream())
        return neg

    def positives(self, qid, p, draws=None, device='cuda', generator=None):
        """GPU positive sampler, the companion of ``negatives``: ``p`` of each query's known objects, drawn with replacement
        from its object list (the training queries are (s, r, -1): the objects come from the lists, not the triple) ->
        int32 [B, p] on ``device``; -1 for a query without objects.  A pure function of ``draws`` (uint32 [B, p], slot =
        list[(u * len) >> 32]); when omitted they come from torch's generator (``generator`` or the global one)."""
        if isinstance(p, bool) or int(p) != p or p < 1:
            raise ValueError('p must be a positive integer, got {!r}'.format(p))
        device = torch.device(device)
        if device.type != 'cuda':
            raise RuntimeError('the positive sampler runs on the GPU only (no CPU fallback)')
        _, ptr, idx = self.device_csr(device)
        qid = torch.as_tensor(qid, dtype=torch.int64).to(device)
        b = int(qid.numel())
        if draws is None:
            draws = torch.randint(0, 1 << 32, (b, int(p)), dtype=torch.int64, device=device, generator=generator)
        draws = torch.as_tensor(draws).to(device)
        if tuple(draws.shape) != (b, int(p)):
            raise ValueError('draws must be [len(qid), p]')
        d32 = _u32_bits(draws)
        out = torch.empty((b, int(p)), dtype=torch.int32, device=device)
        with torch.cuda.device(device):
            _lib.call('kgc_pos_sample', _lib.ptr(qid), b, _lib.ptr(ptr), _lib.ptr(idx), _lib.ptr(d32), int(p), _lib.ptr(out),
                      _lib.stream())
        return out

    def sparse_batch(self, qid):
        """Host CSR slice for the fused scorer: (triple[B,3], filt_ptr[B+1] int64, filt_idx[nnz] int32), numpy."""
        qid = np.asarray(qid, dtype=np.int64)
        if self._lazy is not None and self._ptr is None:           # group-indirect sets: no per-query copy of hub lists
            fptr, fidx = self._lazy.segments(qid)
        else:
            fptr, fidx = _gather_segments(self.ptr, self.idx, qid)
        return self.triples[qid], fptr, fidx.astype(np.int32)

    def collate_fn(self, batch):
        return torch.stack([b[0] for b in batch], dim=0), torch.stack([b[1] for b in batch], dim=0)

    def __len__(self):
        return int(self.triples.shape[0])

    def __getitem__(self, idx):
        raise RuntimeError('KBDataset is batch-built on the GPU; iterate the loaders from get_data_loaders() '
                           'or call build_batch(qid, device)')


def epoch_permutation(n, shuffle=True):
    """Order of one epoch.  Restates what iterating the reference's shuffle=True torch DataLoaders does to the global torch
    generator (data_loader.py:169-176): ``iter(DataLoader)`` first draws its ``_base_seed`` (one int64, consumed whatever
    num_workers is), then RandomSampler draws one int64 seed and runs torch.randperm under a fresh generator seeded with
    it - so under the same torch.manual_seed the batches of every epoch come out in the reference's order
    (tests/test_host_cpu.py compares with a real torch DataLoader)."""
    if not shuffle:
        return np.arange(n, dtype=np.int64)
    torch.empty((), dtype=torch.int64).random_()                  # DataLoader.__iter__: _base_seed (drawn and not used here)
    seed = int(torch.empty((), dtype=torch.int64).random_().item())
    gen = torch.Generator()
    gen.manual_seed(seed)
    return torch.randperm(n, generator=gen).numpy()


class BatchIterator(object):
    """Re-iterable, has len(); yields (triple[B,3] int64, label[B,N] float32) like the reference's torch
    DataLoader (data_loader.py:180-192) but already on the graph's device."""

    def __init__(self, dataset, batch_size, shuffle=True, drop_last=False, device='cuda'):
        self.dataset, self.batch_size, self.shuffle, self.drop_last = dataset, int(batch_size), shuffle, drop_last
        self.device = torch.device(device)

    def __len__(self):
        n = len(self.dataset)
        return n // self.batch_size if self.drop_last else (n + self.batch_size - 1) // self.batch_size

    def batches(self):
        """Query-id batches of one epoch (host integers)."""
        perm = epoch_permutation(len(self.dataset), self.shuffle)
        for i in range(len(self)):
            yield perm[i * self.batch_size:(i + 1) * self.batch_size]

    def __iter__(self):
        for qid in self.batches():
            yield self.dataset.build_batch(qid, self.device)

    def sparse(self):
        """Same epoch order, CSR labels on the device: (triple, filt_ptr, filt_idx) for MGCN.rank / predict."""
        for qid in self.batches():
            trip, fptr, fidx = self.dataset.sparse_batch(qid)
            yield (torch.from_numpy(trip).to(self.device), torch.from_numpy(fptr).to(self.device),
                   torch.from_numpy(fidx).to(self.device))


class DataLoader(object):

    def __init__(self, dataset, params):
        self.data_dir = os.path.join('data', dataset)
        self.params = params
        self.graph = self._load_data()

    def _load_data(self):
        native = native_ingest(self.data_dir) if getattr(self.params, 'native_ingest', True) else None
        if native is not None:                 # N4: both text passes in C++, query sets as CSR arrays
            n_rel = len(native['relations'])
            self.entity2id = {name: i for i, name in enumerate(native['entities'])}
            self.relation2id = {name: i for i, name in enumerate(native['relations'])}
            self.relation2id.update({name + '_reverse': i + n_rel for i, name in enumerate(native['relations'])})
            self.num_entity, self.num_relation = len(native['entities']), n_rel
            self.num_edge = int(native['train'].shape[0])
            self._split_triples = {split: native[split] for split in ('train', 'valid', 'test')}
            self.triplets = LazyTriplets({k: native['q_' + k] for k in ('train', 'valid_tail', 'valid_head', 'test_tail',
                                                                          'test_head')})
            graph = self._build_graph(np.arange(self.num_entity, dtype=np.int64), native['train'], bi_direction=True)
            logging.info('entity={}, relation={}, train_triplets={}, valid_triplets={}, test_triplets={}'.format(
                self.num_entity, self.num_relation, native['train'].shape[0], native['valid'].shape[0], native['test'].shape[0]))
            return graph
        # pass 1 (data_loader.py:64-74): ids in first-appearance order over train, valid, test; tokens lower-cased
        ent2id, rel2id = OrderedDict(), OrderedDict()
        splits = ('train', 'valid', 'test')
        for split in splits:
            with open(os.path.join(self.data_dir, split + '.txt'), 'r') as f:
                for line in f:
                    if not line.strip():
                        continue
                    sub, rel, obj = (tok.lower() for tok in line.strip().split())
                    ent2id.setdefault(sub, len(ent2id))
                    rel2id.setdefault(rel, len(rel2id))
                    ent2id.setdefault(obj, len(ent2id))
        n_rel = len(rel2id)
        for name, idx in list(rel2id.items()):
            rel2id[name + '_reverse'] = idx + n_rel
        self.entity2id, self.relation2id = dict(ent2id), dict(rel2id)
        self.num_entity, self.num_relation = len(ent2id), n_rel

        # pass 2 (data_loader.py:80-96): tokens NOT lower-cased here - a mixed-case dataset raises KeyError
        # exactly as the reference does; (s, r) -> {o} in both directions, snapshot after the train split
        data = {}
        known = defaultdict(set)
        known_train = None
        for split in splits:
            rows = []
            with open(os.path.join(self.data_dir, split + '.txt'), 'r') as f:
                for line in f:
                    if not line.strip():
                        continue
                    head, relation, tail = line.strip().split()
                    s, r, o = self.entity2id[head], self.relation2id[relation], self.entity2id[tail]
                    rows.append((s, r, o))
                    known[(s, r)].add(o)
                    known[(o, r + n_rel)].add(s)
            data[split] = rows
            if split == 'train':
                known_train = OrderedDict((k, sorted(v)) for k, v in known.items())
        known_all = {k: sorted(v) for k, v in known.items()}
        self.num_edge = len(data['train'])
        self._split_triples = {split: np.asarray(data[split], dtype=np.int64).reshape(-1, 3) for split in splits}

        # query lists (data_loader.py:98-111)
        trip = {'train': [{'triple': (s, r, -1), 'label': objs, 'sub_samp': 1} for (s, r), objs in known_train.items()]}
        for split in ('valid', 'test'):
            tails, heads = [], []
            for s, r, o in data[split]:
                tails.append({'triple': (s, r, o), 'label': known_all[(s, r)]})
                heads.append({'triple': (o, r + n_rel, s), 'label': known_all[(o, r + n_rel)]})
            trip[split + '_tail'], trip[split + '_head'] = tails, heads
        self.triplets = trip

        graph = self._build_graph(np.arange(self.num_entity, dtype=np.int64),
                                  np.asarray(data['train'], dtype=np.int64).reshape(-1, 3), bi_direction=True)
        logging.info('entity={}, relation={}, train_triplets={}, valid_triplets={}, test_triplets={}'.format(
            self.num_entity, self.num_relation, len(data['train']), len(data['valid']), len(data['test'])))
        return graph

    def _edge_normal(self, edge_type, edge_index, num_entity):
        """1 / in-degree(dst), inf -> 0 (data_loader.py:122-130).  Kept for API compatibility only: the
        convolution never reads it (SURVEY.md fact 6)."""
        dst = np.asarray(edge_index[1], dtype=np.int64)
        deg = np.bincount(dst, minlength=num_entity).astype(np.float32)
        with np.errstate(divide='ignore'):
            norm = (np.float32(1.0) / deg[dst]).astype(np.float32)
        norm[np.isinf(norm)] = 0
        return torch.from_numpy(norm)

    def _build_graph(self, graph_nodes, triplets, bi_direction=True):
        """Bi-directional edge list (data_loader.py:132-157): columns 0..E-1 = (s -> o, r), E..2E-1 = (o -> s, r + R)."""
        src, rel, dst = triplets.transpose()
        if bi_direction is True:
            src, dst = np.concatenate((src, dst)), np.concatenate((dst, src))
            rel = np.concatenate((rel, rel + self.num_relation))
        edge_index = np.stack((src, dst))
        edge_attr = np.stack((rel, np.arange(edge_index.shape[1])))
        data = GraphData(edge_index=torch.from_numpy(edge_index), edge_attr=torch.from_numpy(edge_attr))
        data.entity = torch.from_numpy(graph_nodes)
        data.num_nodes = len(graph_nodes)
        data.edge_norm = self._edge_normal(rel, edge_index, len(graph_nodes))
        return data

    def sample_edges(self, m, draws=None, generator=None):
        """GPU edge sampler (extension without a reference counterpart: the reference convolves over the full edge list every
        step, main.py:61).  ``m`` training triples drawn with replacement -> a GraphData in the reference's layout
        (edge_index [2, 2m]: the m sampled edges, then their reverses; edge_attr = [types; columns of the full edge list],
        i.e. ``edge_attr[1]`` indexes ``edge_embeddings`` as in model.py:30) on the graph's device.  A pure function of
        ``draws`` (uint32 [m], triple = (u * E) >> 32); when omitted they come from torch's generator."""
        g = self.graph
        dev = g.edge_index.device
        if dev.type != 'cuda':
            raise RuntimeError('the edge sampler runs on the GPU only (no CPU fallback); move the graph with graph.to("cuda")')
        m = int(m)
        if draws is None:
            draws = torch.randint(0, 1 << 32, (m,), dtype=torch.int64, device=dev, generator=generator)
        draws = torch.as_tensor(draws).to(dev)
        if tuple(draws.shape) != (m,):
            raise ValueError('draws must be [m]')
        d32 = _u32_bits(draws)
        ei = g.edge_index.contiguous()
        et = g.edge_attr[0].contiguous()
        sub = torch.empty((4, 2 * m), dtype=torch.int64, device=dev)
        p = _lib.ptr
        with torch.cuda.device(dev):
            _lib.call('kgc_edge_sample', p(ei[0]), p(ei[1]), p(et), self.num_edge, p(d32), m, p(sub[0]), p(sub[1]), p(sub[2]),
                      p(sub[3]), _lib.stream())
        data = GraphData(edge_index=sub[:2], edge_attr=sub[2:])
        data.entity, data.num_nodes = g.entity, g.num_nodes
        return data

    def known_objects(self, src, rel):
        """Exclusion CSR for arbitrary queries (src[q], rel[q], ?): (ptr [B+1] int64, idx int32) on the graph's device, row q
        = the sorted objects o with (src[q], rel[q], o) in train, valid or test; a reverse relation r + R gives the subjects s
        of (s, r, src[q]) (the reference's all-split filter, data_loader.py:80-96).  For ``MGCN.topk(..., exclude=...)``."""
        if getattr(self, '_known', None) is None:
            n_rel2 = 2 * self.num_relation
            t = np.concatenate([self._split_triples[s] for s in ('train', 'valid', 'test')]).reshape(-1, 3)
            keys = np.concatenate([t[:, 0] * n_rel2 + t[:, 1], t[:, 2] * n_rel2 + t[:, 1] + self.num_relation])
            objs = np.concatenate([t[:, 2], t[:, 0]])
            order = np.lexsort((objs, keys))
            keys, objs = keys[order], objs[order]
            if keys.size:
                first = np.ones(keys.size, dtype=bool)
                first[1:] = (keys[1:] != keys[:-1]) | (objs[1:] != objs[:-1])
                keys, objs = keys[first], objs[first]
            ukeys, start = np.unique(keys, return_index=True)
            gptr = np.append(start, keys.size).astype(np.int64)
            self._known = (ukeys, gptr, objs.astype(np.int32))
        ukeys, gptr, gidx = self._known
        src = np.asarray(src.cpu() if torch.is_tensor(src) else src, dtype=np.int64).reshape(-1)
        rel = np.asarray(rel.cpu() if torch.is_tensor(rel) else rel, dtype=np.int64).reshape(-1)
        q = src * (2 * self.num_relation) + rel
        pos = np.minimum(np.searchsorted(ukeys, q), max(ukeys.size - 1, 0))
        found = ukeys.size > 0
        found = (ukeys[pos] == q) if found else np.zeros(q.shape, dtype=bool)
        # unknown (s, r): an empty row, read from the empty group appended at the end
        groups = np.where(found, pos, ukeys.size)
        ptr, idx = _gather_segments(np.append(gptr, gptr[-1]), gidx, groups)
        dev = self.graph.device
        return torch.from_numpy(ptr).to(dev), torch.from_numpy(np.ascontiguousarray(idx, dtype=np.int32)).to(dev)

    def _queries(self, key):
        t = self.triplets
        return t.query_set(key) if isinstance(t, LazyTriplets) else t[key]

    def _get_dataset(self, data_type, params):
        if data_type == 'train':
            return KBDataset(self._queries('train'), len(self.entity2id), params, training=True)
        elif data_type in ['valid_head', 'valid_tail', 'test_head', 'test_tail']:
            return KBDataset(self._queries(data_type), len(self.entity2id), params)
        else:
            raise ValueError('Unkown data type')

    def _create_data_loader(self, dataset, batch_size, num_workers, shuffle, drop_last=False):
        # num_workers is accepted for signature compatibility; batches are built by one CUDA kernel per step
        return BatchIterator(dataset, batch_size, shuffle=shuffle, drop_last=drop_last, device=self.graph.device)

    def get_data_loaders(self, batch_size, num_workers, params):
        marks = ['train', 'valid_head', 'valid_tail', 'test_head', 'test_tail']
        return {mark: self._create_data_loader(self._get_dataset(mark, params), batch_size=batch_size,
                                               num_workers=num_workers, shuffle=True, drop_last=False)
                for mark in marks}
