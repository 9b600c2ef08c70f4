"""MGCN and ConvE: drop-in mirrors of the reference classes (model.py:10-44, 130-181).

Same constructors, forward signatures, parameter / state-dict names (SURVEY.md 8(b)), so a checkpoint
written by the reference loads here and vice versa.  The encoder is the CUDA MGCNConv; the ConvE front
end (bn0 -> 7x7 conv -> bn1 -> relu -> fc -> bn2 -> relu, model.py:161-175) is SURVEY.md "next" row N2: bn0 / bn1 (K7),
the convolution (K8) and the fc layer (3xTF32 tensor-core GEMMs) run on our kernels, bn2 on torch; the 1-N scoring tail of ``forward`` (which must return the dense [B,N] matrix to stay
call-compatible) and its autograd run on the 3xTF32 tensor-core kernels (K6t, scoring.score_1n); ``rank`` uses the
fused tensor-core scoring + ranking kernel (K6).
"""
import weakref

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib
from .conv import MGCNConv, get_param, linear_tc, linear_tc_supported


class _BnReluDropFn(torch.autograd.Function):
    """dropout(relu(batch_norm(x))) over [B, C, H, W] (model.py:168-170) on the K7 kernels."""

    @staticmethod
    def forward(ctx, x, gamma, beta, running_mean, running_var, eps, momentum, training, drop_p, seed, relu):
        x_ = _lib.require_cuda(x.detach(), torch.float32, 'x')
        B, C = int(x_.shape[0]), int(x_.shape[1])
        HW = int(x_.shape[2] * x_.shape[3])
        p = _lib.ptr
        partials = torch.empty((int(_lib.lib().kgc_bn2d_partials_bytes(C)) // 8,), dtype=torch.float64, device=x.device)
        stats = torch.empty((2, C), dtype=torch.float32, device=x.device)
        y = torch.empty_like(x_)
        _lib.call('kgc_bn2d_relu_drop_fwd', p(x_), B, C, HW, p(gamma.detach()), p(beta.detach()), p(running_mean),
                  p(running_var), float(eps), float(momentum), int(training), int(relu), p(seed), float(drop_p), p(partials),
                  p(stats), p(y), _lib.stream())
        ctx.save_for_backward(x_, gamma.detach(), beta.detach(), stats, seed if seed is not None else torch.empty(0))
        ctx.cfg = (bool(training), float(drop_p), seed is not None, int(relu))
        return y

    @staticmethod
    def backward(ctx, dy):
        x, gamma, beta, stats, seed = ctx.saved_tensors
        training, drop_p, has_seed, relu = ctx.cfg
        B, C = int(x.shape[0]), int(x.shape[1])
        HW = int(x.shape[2] * x.shape[3])
        dy = dy.contiguous()
        p = _lib.ptr
        partials = torch.empty((int(_lib.lib().kgc_bn2d_partials_bytes(C)) // 8,), dtype=torch.float64, device=x.device)
        sums = torch.empty((2, C), dtype=torch.float32, device=x.device)
        dx = torch.empty_like(x)
        _lib.call('kgc_bn2d_relu_drop_bwd', p(dy), p(x), B, C, HW, p(gamma), p(beta), p(stats), int(training), relu,
                  p(seed) if has_seed else None, drop_p, p(partials), p(sums), p(dx), _lib.stream())
        return dx, sums[1], sums[0], None, None, None, None, None, None, None, None


class _Conv1chFn(torch.autograd.Function):
    """nn.Conv2d(1, F, (K, K)) forward / backward (model.py:166) on the K8 direct-convolution kernels."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        x_ = _lib.require_cuda(x.detach(), torch.float32, 'x').contiguous()
        w_ = weight.detach().contiguous()
        B, H, W = int(x_.shape[0]), int(x_.shape[2]), int(x_.shape[3])
        F_, K = int(w_.shape[0]), int(w_.shape[2])
        y = torch.empty((B, F_, H - K + 1, W - K + 1), dtype=torch.float32, device=x.device)
        p = _lib.ptr
        _lib.call('kgc_conv1ch_fwd', p(x_), p(w_), p(bias.detach().contiguous()) if bias is not None else None, B, F_, K, H, W,
                  p(y), _lib.stream())
        ctx.save_for_backward(x_, w_)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        x, w = ctx.saved_tensors
        dy = dy.contiguous()
        B, H, W = int(x.shape[0]), int(x.shape[2]), int(x.shape[3])
        F_, K = int(w.shape[0]), int(w.shape[2])
        p = _lib.ptr
        dx = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        dw = torch.empty_like(w) if ctx.needs_input_grad[1] else None
        ws = torch.empty((int(_lib.lib().kgc_conv1ch_bwd_workspace_bytes(B, F_, K)) // 4,), dtype=torch.float32, device=x.device)
        _lib.call('kgc_conv1ch_bwd', p(dy), p(x), p(w), B, F_, K, H, W, p(dx), p(dw), p(ws), _lib.stream())
        db = dy.sum((0, 2, 3)) if ctx.has_bias and ctx.needs_input_grad[2] else None
        return dx, dw, db


class ConvE(nn.Module):

    def __init__(self, params, num_entities):
        super(ConvE, self).__init__()
        self.params = params
        self.bn0 = nn.BatchNorm2d(1)
        self.bn1 = nn.BatchNorm2d(params.num_filter)
        self.bn2 = nn.BatchNorm1d(params.gcn_out_dim)
        self.hidden_drop = nn.Dropout(params.hidden_drop)
        self.feature_drop = nn.Dropout(params.feat_drop)
        self.conv_e = nn.Conv2d(in_channels=1, out_channels=params.num_filter,
                                kernel_size=(params.kernel_size, params.kernel_size), stride=1, padding=0,
                                bias=params.bias)
        flat_sz_h = int(2 * params.k_w) - params.kernel_size + 1
        flat_sz_w = params.k_h - params.kernel_size + 1
        self.flat_sz = flat_sz_h * flat_sz_w * params.num_filter
        self.fc = nn.Linear(self.flat_sz, params.gcn_out_dim)
        self.register_parameter('bias', nn.Parameter(torch.zeros(num_entities)))
        # dropout stream of the K7 kernel (device-resident counter, not part of the state dict)
        self.register_buffer('_drop_seed', torch.zeros(1, dtype=torch.int64), persistent=False)
        self._drop_seeded = False

    @staticmethod
    def _k7_ok(x, bn, p=0.0):
        return (x.is_cuda and x.dtype == torch.float32 and (x.shape[2] * x.shape[3]) % 4 == 0 and bn.affine
                and bn.track_running_stats and bn.momentum is not None and 0.0 <= p < 1.0)

    def _bn0(self, x):
        """model.py:165 - the ONE-channel BatchNorm2d over the input image (cuDNN: one CTA, 27 us forward + 50 us backward
        for 51,200 values) - on the K7 kernels."""
        bn = self.bn0
        if not self._k7_ok(x, bn):
            _lib.library_path('ConvE.bn0', 'K7 takes CUDA fp32 maps with H * W % 4 == 0 and an affine BatchNorm with running '
                                           'statistics and a fixed momentum')
            return bn(x)
        if self.training:
            bn.num_batches_tracked.add_(1)
        return _BnReluDropFn.apply(x.contiguous(), bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.eps, bn.momentum,
                                   self.training, 0.0, None, 0)

    def _bn1_relu_drop(self, x):
        """model.py:168-170 - bn1, relu, feature dropout - on the K7 kernels where they apply (GPU, fp32, H * W % 4 == 0,
        BatchNorm with running statistics and a fixed momentum); the torch / cuDNN modules otherwise."""
        bn, p = self.bn1, self.feature_drop.p
        if not self._k7_ok(x, bn, p):
            _lib.library_path('ConvE.bn1', 'K7 takes CUDA fp32 maps with H * W % 4 == 0 and an affine BatchNorm with running '
                                           'statistics and a fixed momentum')
            return self.feature_drop(F.relu(bn(x)))
        seed = None
        if self.training and p > 0.0:
            if not self._drop_seeded:
                self._drop_seed.fill_(int(torch.randint(0, 2 ** 62, (1,)).item()))
                self._drop_seeded = True
            self._drop_seed.add_(0x9E3779B97F4A7C15 & 0x7FFFFFFFFFFFFFFF)     # new stream every step (device op: graph-capturable)
            seed = self._drop_seed.clone()
        if self.training:
            bn.num_batches_tracked.add_(1)
        return _BnReluDropFn.apply(x.contiguous(), bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.eps, bn.momentum,
                                   self.training, p, seed, 1)

    def _conv(self, x):
        """model.py:166 - the one-input-channel k x k convolution - on the K8 kernels for the shapes they take (GPU, fp32,
        stride 1, no padding, W = 20, k in {3, 5, 7}); the torch / cuDNN module otherwise."""
        c = self.conv_e
        if (x.is_cuda and x.dtype == torch.float32 and c.in_channels == 1 and c.kernel_size[0] == c.kernel_size[1]
                and c.stride == (1, 1) and c.padding == (0, 0) and c.dilation == (1, 1) and c.groups == 1
                and _lib.lib().kgc_conv1ch_supported(c.out_channels, c.kernel_size[0], x.shape[2], x.shape[3])):
            return _Conv1chFn.apply(x, c.weight, c.bias)
        _lib.library_path('ConvE.conv_e', 'K8 takes CUDA fp32, one input channel, stride 1, no padding, W = 20, k in {3, 5, 7}')
        return c(x)

    def query(self, src_emb, rel_emb):
        """Front end: (src_emb, rel_emb) -> query matrix X[B, Dout] (model.py:161-175)."""
        d = self.params.gcn_out_dim
        stack_inp = torch.cat([src_emb.view(-1, 1, d), rel_emb.view(-1, 1, d)], dim=1)
        x = torch.transpose(stack_inp, 2, 1).reshape(-1, 1, 2 * self.params.k_w, self.params.k_h)
        x = self._bn0(x)
        x = self._conv(x)
        x = self._bn1_relu_drop(x)
        x = x.view(-1, self.flat_sz)
        # model.py:173: the 39,200 -> 200 fc layer; fp32-grade tensor-core kernels for the shapes they take
        if linear_tc_supported(x, self.fc.weight):
            x = linear_tc(x, self.fc.weight, self.fc.bias)
        else:
            _lib.library_path('ConvE.fc', 'the tensor-core fc kernels take CUDA fp32, out <= 224, flat % 32 == 0, flat >= 4096')
            x = self.fc(x)
        x = self.hidden_drop(x)
        return F.relu(self.bn2(x))

    def forward(self, src_emb, rel_emb, all_ent):
        x = self.query(src_emb, rel_emb)
        # model.py:177-179: mm, += bias, sigmoid - on the tensor-core scorer (K6t) for the shapes it takes
        from .scoring import score_1n, score_1n_supported
        if score_1n_supported(x, all_ent):
            return score_1n(x, all_ent, self.bias)
        _lib.library_path('ConvE 1-N scoring', 'K6t takes CUDA fp32 with Dout <= 224, Dout % 4 == 0 and 16-byte aligned entity rows')
        return torch.sigmoid(torch.addmm(self.bias, x, all_ent.transpose(1, 0)))


class _RowsAndTable(torch.autograd.Function):
    """(table[idx], table) for a table that is ALSO consumed whole by the scorer (model.py:36-40: ``src_emb =
    index_select(all_ent, 0, src)`` next to ``conv2(src_emb, rel_emb, all_ent)``).  Plain autograd turns the gradient of
    the few selected rows into a dense zero table + index_add and then adds that table to the scorer's dense gradient:
    two extra passes over [N, Dout] per step (3.7 GB each way at the Wikidata5M shape).  Here the rows' gradient is added
    INTO the scorer's dense gradient.  Duplicate indices are summed by a [B, B] equality matrix product first, so every
    duplicate writes the same total: deterministic, no atomics."""

    @staticmethod
    def forward(ctx, table, idx):
        ctx.save_for_backward(idx)
        ctx.shape = table.shape
        return table.index_select(0, idx), table.detach().view_as(table)

    @staticmethod
    def backward(ctx, d_rows, d_table):
        (idx,) = ctx.saved_tensors
        if d_table is None:
            d_table = torch.zeros(ctx.shape, dtype=d_rows.dtype, device=d_rows.device)
        elif not d_table.is_contiguous():
            d_table = d_table.contiguous()
        if d_rows is not None:
            same = (idx[:, None] == idx[None, :]).to(d_rows.dtype)            # rows of one entity share one total
            total = same @ d_rows
            d_table.index_copy_(0, idx, d_table.index_select(0, idx) + total)
        return d_table, None


class MGCN(nn.Module):

    def __init__(self, num_entities, num_relations, num_edges, params):
        super(MGCN, self).__init__()
        self.params = params
        self.entity_embedding = get_param((num_entities, params.gcn_in_dim))
        self.relation_embedding = get_param((2 * num_relations, params.gcn_in_dim))
        self.edge_embeddings = get_param((2 * num_edges, params.gcn_in_dim))
        self.conv1 = MGCNConv(params.gcn_in_dim, params.gcn_out_dim, num_relations * 2)
        self.conv2 = ConvE(params, num_entities)
        self.loss_fn = nn.BCELoss()
        self._arange_cache = {}

    def __getstate__(self):
        state = self.__dict__.copy()
        state['_arange_cache'] = {}                      # weak references do not pickle; the cache refills on first use
        return state

    def _is_arange(self, idx, n):
        """data.entity / edge_ids are arange in every graph the reference builds (data_loader.py:145-153);
        the identity gathers of model.py:29-30 are then skipped (they copy 16 MB + 70 MB per WN18RR step).
        The check costs one device sync, so it is cached on the identity + version of the index tensor."""
        key = (idx.data_ptr(), idx._version, idx.numel(), n, str(idx.device))
        # ``edge_type, edge_ids = data.edge_attr`` (model.py:26) makes a NEW view object per call: the owner of the memory is
        # the view's base.  While that object is alive the address cannot have been recycled for another tensor.
        owner = idx._base if idx._base is not None else idx
        hit = self._arange_cache.get(key)
        if hit is not None and hit[1]() is owner:
            return hit[0]
        ok = idx.numel() == n and bool((idx == torch.arange(n, device=idx.device)).all())
        if len(self._arange_cache) > 16:
            self._arange_cache.clear()
        self._arange_cache[key] = (ok, weakref.ref(owner))
        return ok

    def encode(self, data):
        """GCN encoder (model.py:25-34): returns (all_ent after gcn_drop, all_rel)."""
        entity, edge_index, edge_norm = data.entity, data.edge_index, data.edge_norm
        edge_type, edge_ids = data.edge_attr
        ent = self.entity_embedding
        if not self._is_arange(entity, ent.size(0)):
            ent = torch.index_select(ent, 0, entity)
        edge = self.edge_embeddings
        if not self._is_arange(edge_ids, edge.size(0)):
            edge = torch.index_select(edge, 0, edge_ids)
        p = float(self.params.gcn_drop)
        if self.training and 0.0 < p < 1.0 and isinstance(self.conv1, MGCNConv) and self.conv1.out_channels <= 256:
            # model.py:34 inside the layer's last kernel: no read + write + mask pass over [N, Dout] (2.9 ms per step each
            # way at the Wikidata5M shape); the undropped all_ent is not needed by anything downstream
            return self.conv1(ent, edge_index, edge_type, edge_norm, edge, self.relation_embedding, _out_drop=p)
        all_ent, all_rel = self.conv1(ent, edge_index, edge_type, edge_norm, edge, self.relation_embedding)
        all_ent = F.dropout(all_ent, p=self.params.gcn_drop, training=self.training)
        return all_ent, all_rel

    @staticmethod
    def _rows(all_ent, idx):
        """(all_ent[idx], all_ent) with the rows' gradient folded into the table's (see _RowsAndTable)."""
        if all_ent.requires_grad and all_ent.is_cuda and idx.numel() <= 4096:
            return _RowsAndTable.apply(all_ent, idx)
        return torch.index_select(all_ent, 0, idx), all_ent

    def forward(self, src, rel, data):
        all_ent, all_rel = self.encode(data)
        src_emb, all_ent = self._rows(all_ent, src)
        rel_emb = torch.index_select(all_rel, 0, rel)
        return self.conv2(src_emb, rel_emb, all_ent)

    def loss(self, pred, label):
        return self.loss_fn(pred, label)

    def loss_sparse(self, qid, dataset, data):
        """``loss(forward(src, rel, data), label)`` for the training queries ``qid`` of ``dataset`` (a KBDataset) without the
        dense [B, N] label or the BCE tensors (SURVEY.md 8(f) N1): src / rel are the queries' triples and the label is read
        as sparse positives from the dataset's CSR with its ``label_values()`` (label smoothing as data_loader.py:41-43).
        Same value and gradients as the dense route within fp32 rounding (tests/test_gpu_zz_loss.py)."""
        from .scoring import score_1n_bce, score_1n_supported
        dev = self.entity_embedding.device
        triples, ptr, idx = dataset.device_csr(dev)
        qid = torch.as_tensor(qid, dtype=torch.int64).to(dev, non_blocking=True)
        trip = torch.index_select(triples, 0, qid)
        all_ent, all_rel = self.encode(data)
        src_emb, all_ent = self._rows(all_ent, trip[:, 0])
        x = self.conv2.query(src_emb, torch.index_select(all_rel, 0, trip[:, 1]))
        if not score_1n_supported(x, all_ent):
            raise RuntimeError('loss_sparse: shape not taken by the tensor-core scorer (Dout <= 224, Dout % 4 == 0); '
                               'use loss(forward(...), label)')
        pos, add = dataset.label_values()
        return score_1n_bce(x, all_ent, self.conv2.bias, qid, ptr, idx, pos, add)

    def loss_sampled(self, qid, dataset, data, k, n_pos=1, tries=4, draws=None, generator=None, adversarial_temperature=None):
        """Negative-sampled (1-vs-k) training loss for the training queries ``qid`` of ``dataset`` (a KBDataset): each query
        scores ``n_pos`` of its known objects (``dataset.positives``) and ``k`` entities that are not (``dataset.negatives``,
        ``tries`` draws per slot) - candidates [pos | neg] - through ``scoring.score_sampled_bce`` with the dataset's
        ``label_values()``.  Unlike ``loss_sparse`` the cost of the scoring does not grow with N, so the batch can be large.
        ``draws = (pos_draws [B, n_pos], neg_draws [B, k, tries])`` (uint32 values) makes the call a pure function of them;
        otherwise they come from torch's generator (``generator`` or the global one), positives first.
        ``adversarial_temperature=alpha`` weights each query's negatives by softmax(alpha * logit) (self-adversarial
        negative sampling, see ``scoring.score_sampled_bce``); None: the plain mean over the valid slots."""
        from .scoring import check_adversarial_temperature, score_sampled_bce
        check_adversarial_temperature(adversarial_temperature)
        dev = self.entity_embedding.device
        triples, _, _ = dataset.device_csr(dev)
        qid = torch.as_tensor(qid, dtype=torch.int64).to(dev, non_blocking=True)
        pos_draws, neg_draws = draws if draws is not None else (None, None)
        cand = torch.cat([dataset.positives(qid, n_pos, draws=pos_draws, device=dev, generator=generator),
                          dataset.negatives(qid, k, draws=neg_draws, tries=tries, device=dev, generator=generator)], 1)
        trip = torch.index_select(triples, 0, qid)
        all_ent, all_rel = self.encode(data)
        src_emb, all_ent = self._rows(all_ent, trip[:, 0])
        x = self.conv2.query(src_emb, torch.index_select(all_rel, 0, trip[:, 1]))
        pos, add = dataset.label_values()
        return score_sampled_bce(x, all_ent, self.conv2.bias, cand, n_pos, pos, add,
                                 adversarial_temperature=adversarial_temperature)

    def rank(self, src, rel, obj, filt_ptr, filt_idx, data, count_eq=False):
        """Filtered rank of obj among all entities for the queries (src, rel) without materialising the
        [B, N] scores (K6): what main.py:121-126 computes from model(sub, rel, graph)."""
        from .scoring import filtered_rank
        all_ent, all_rel = self.encode(data)
        xq = self.conv2.query(torch.index_select(all_ent, 0, src), torch.index_select(all_rel, 0, rel))
        return filtered_rank(xq, all_ent, self.conv2.bias, obj, filt_ptr, filt_idx, count_eq=count_eq)

    def topk(self, src, rel, data, k=10, exclude=None, precision='bf16', table=None, n_offset=0, group=None):
        """The k most likely objects of the queries (src, rel, ?) without materialising the [B, N] scores (K6k):
        ``scoring.topk`` on the ConvE query.  ``exclude``: (ptr, idx) CSR of entities to leave out per query, e.g.
        ``DataLoader.known_objects(src, rel)`` for the known facts; None keeps every entity.

        Entity-sharded, as ``scoring.topk``: ``table`` is this rank's bf16 shard of the encoded entities, rows
        ``n_offset .. n_offset + table.n`` (with precision='fp32' the same rows of the fp32 encoding are scored).  With a
        ``group`` and no ``table``, the ranks split the entities into even ranges (rank r: rows r * ceil(N / world) ...).
        Every rank of the group returns the unsharded answer."""
        from .scoring import topk
        all_ent, all_rel = self.encode(data)
        xq = self.conv2.query(torch.index_select(all_ent, 0, src), torch.index_select(all_rel, 0, rel))
        ptr, idx = exclude if exclude is not None else (None, None)
        ent, bias = all_ent, self.conv2.bias
        if n_offset != 0 and table is None:
            raise ValueError('n_offset names the first row of a table shard: pass table= as well')
        if table is not None or group is not None:
            if table is not None:
                lo, hi = n_offset, n_offset + table.n
            else:
                import torch.distributed as dist
                n, world = int(all_ent.shape[0]), dist.get_world_size(group)
                per = -(-n // world)
                lo = min(dist.get_rank(group) * per, n)
                hi = min(lo + per, n)
            n_offset = lo
            ent, bias = all_ent[lo:hi], (bias[lo:hi] if bias is not None else None)
        return topk(xq, ent, bias, k, ptr, idx, table=table, precision=precision, n_offset=n_offset, group=group)
