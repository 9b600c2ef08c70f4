"""Fused 1-N scoring + filtered ranking (K6) and the reference-facing evaluation helpers.

Replaces ConvE's scoring tail (model.py:177-179) + predict's filter / double argsort (main.py:117-133)
for evaluation.  The [B, N] score matrix is never written: a tcgen05 / TMA kernel sweeps the bf16 entity
table once per pair of 128-query tiles and counts, per query, the entities whose logit beats the target's.

Tie semantics (SURVEY.md section 7): rank = 1 + count_gt on the LOGIT (sigmoid is monotone but saturates
in fp32, which manufactures ties the reference then breaks arbitrarily); count_eq is reported so that
callers can check reference_rank in [1 + gt, 1 + gt + eq].
"""
import math
import numbers

import torch

from . import _lib
from .conv import _pack_b


class _Score1N(torch.autograd.Function):
    """pred[B, N] = sigmoid(x @ all_ent^T + bias) with its autograd on the tensor-core kernels (K6t): the training-time
    scoring tail of model.py:177-179."""

    @staticmethod
    def forward(ctx, x, all_ent, bias):
        x = _lib.require_cuda(x.detach(), torch.float32, 'x')
        ent = _lib.require_cuda(all_ent.detach(), torch.float32, 'all_ent')
        bias_ = _lib.require_cuda(bias.detach(), torch.float32, 'bias')
        B, D = int(x.shape[0]), int(x.shape[1])
        N = int(ent.shape[0])
        ldp = (N + 3) // 4 * 4
        p = _lib.ptr
        packed = _pack_b(x.t())                         # the queries are the small operand: [K = D, N = B]
        buf = torch.empty((B, ldp), dtype=torch.float32, device=x.device)
        _lib.call('kgc_score_1n_fwd', p(ent), N, D, ent.stride(0), p(packed), B, p(bias_), p(buf), ldp, _lib.stream())
        pred = buf[:, :N]
        ctx.save_for_backward(x, ent, pred)
        return pred

    @staticmethod
    def backward(ctx, d_pred):
        from .conv import gemm_nt, gemm_tn
        x, ent, pred = ctx.saved_tensors
        B, D = int(x.shape[0]), int(x.shape[1])
        N = int(ent.shape[0])
        if d_pred.stride(1) != 1:
            d_pred = d_pred.contiguous()
        ldt = (B + 3) // 4 * 4
        d_logit_t = torch.empty((N, ldt), dtype=torch.float32, device=x.device)
        d_bias = torch.empty((N,), dtype=torch.float32, device=x.device)
        p = _lib.ptr
        _lib.call('kgc_score_1n_bwd_logit', p(d_pred), d_pred.stride(0), p(pred), pred.stride(0), N, B, ldt,
                  p(d_logit_t), p(d_bias), _lib.stream())
        d_x = d_ent = None
        if ctx.needs_input_grad[0]:
            d_x = gemm_tn(d_logit_t, ent, torch.empty((ldt, D), dtype=torch.float32, device=x.device))[:B]
        if ctx.needs_input_grad[1]:
            d_ent = gemm_nt(d_logit_t[:, :B], x, torch.empty((N, D), dtype=torch.float32, device=x.device))
        return d_x, d_ent, (d_bias if ctx.needs_input_grad[2] else None)


B_TILE = 256      # queries per K6t launch (the packed query operand of one launch); larger batches run tile by tile


def score_1n_supported(x, all_ent):
    """Shapes the tensor-core training scorer takes (the caller reports anything else through _lib.library_path).  Any batch
    size: batches above B_TILE queries are scored tile by tile."""
    return (x.is_cuda and x.dtype == torch.float32 and all_ent.dtype == torch.float32 and x.dim() == 2
            and x.shape[0] > 0 and x.shape[1] <= 224 and x.shape[1] % 4 == 0
            and all_ent.stride(1) == 1 and all_ent.stride(0) % 4 == 0 and all_ent.data_ptr() % 16 == 0)


def score_1n(x, all_ent, bias):
    """sigmoid(x @ all_ent^T + bias) [B, N] (model.py:177-179), differentiable."""
    if x.shape[0] <= B_TILE:
        return _Score1N.apply(x, all_ent, bias)
    return torch.cat([_Score1N.apply(x[i:i + B_TILE], all_ent, bias) for i in range(0, x.shape[0], B_TILE)], 0)


class _Score1NBCE(torch.autograd.Function):
    """loss = BCELoss(sigmoid(x @ all_ent^T + bias), label) with the label given as SPARSE positives (SURVEY.md 8(f) N1):
    model.py:177-179 + model.py:42-44 + the label build of data_loader.py:34-43 in one differentiable call.  The forward
    runs the K6t scorer, sets one bit per positive and makes ONE pass over pred that yields the mean loss, the logit
    gradient (transposed) and the bias gradient for a unit upstream gradient; the backward scales by the upstream scalar
    and runs the two gradient GEMMs.  The dense label and the BCE forward / backward tensors are never built."""

    @staticmethod
    def forward(ctx, x, all_ent, bias, qid, ptr, idx, pos, add):
        x = _lib.require_cuda(x.detach(), torch.float32, 'x')
        ent = _lib.require_cuda(all_ent.detach(), torch.float32, 'all_ent')
        bias_ = _lib.require_cuda(bias.detach(), torch.float32, 'bias')
        qid = _lib.require_cuda(qid, torch.int64, 'qid')
        ptr = _lib.require_cuda(ptr, torch.int64, 'ptr')
        idx = _lib.require_cuda(idx, torch.int32, 'idx')
        B, D = int(x.shape[0]), int(x.shape[1])
        N = int(ent.shape[0])
        if int(qid.numel()) != B:
            raise ValueError('qid has {} entries for {} queries'.format(int(qid.numel()), B))
        ldt = (B + 3) // 4 * 4
        p, dev = _lib.ptr, x.device
        packed = _pack_b(x.t())
        # entity-major throughout: the scorer stores predT [N, ldt] (its natural orientation), the positives are bits per
        # entity, and the loss pass overwrites predT with the logit gradient in place (the [N, ldt] operand of both
        # gradient GEMMs) - no [B, N]-pitched buffer, no transpose
        d_logit_t = torch.empty((N, ldt), dtype=torch.float32, device=dev)
        _lib.call('kgc_score_1n_fwd_t', p(ent), N, D, ent.stride(0), p(packed), B, p(bias_), p(d_logit_t), ldt, _lib.stream())
        mask_t = torch.empty((N, (B + 31) // 32), dtype=torch.int32, device=dev)          # uint32 bits; zeroed by the call
        _lib.call('kgc_label_mask_t_build', p(qid), B, p(ptr), p(idx), N, p(mask_t), _lib.stream())
        d_bias = torch.empty((N,), dtype=torch.float32, device=dev)
        partial = torch.empty((int(_lib.lib().kgc_bce_1n_t_blocks(N)),), dtype=torch.float64, device=dev)
        loss = torch.empty((1,), dtype=torch.float32, device=dev)
        _lib.call('kgc_bce_1n_bwd_logit_t', p(d_logit_t), p(mask_t), N, B, ldt, float(pos), float(add), p(d_bias),
                  p(partial), p(loss), _lib.stream())
        ctx.save_for_backward(x, ent, d_logit_t, d_bias)
        return loss[0]

    @staticmethod
    def backward(ctx, g):
        from .conv import gemm_nt, gemm_tn
        x, ent, d_logit_t, d_bias = ctx.saved_tensors
        B, D = int(x.shape[0]), int(x.shape[1])
        N, ldt = int(ent.shape[0]), int(d_logit_t.shape[1])
        d_x = d_ent = None
        if ctx.needs_input_grad[0]:
            d_x = gemm_tn(d_logit_t, ent, torch.empty((ldt, D), dtype=torch.float32, device=x.device))[:B] * g
        if ctx.needs_input_grad[1]:                      # the upstream scalar rides on the small operand
            d_ent = gemm_nt(d_logit_t[:, :B], (x * g).contiguous(), torch.empty((N, D), dtype=torch.float32, device=x.device))
        return d_x, d_ent, (d_bias * g if ctx.needs_input_grad[2] else None), None, None, None, None, None


def score_1n_bce(x, all_ent, bias, qid, ptr, idx, pos=1.0, add=0.0):
    """Mean BCE of sigmoid(x @ all_ent^T + bias) against the labels of queries ``qid`` (device int64 [B]) given as the
    query -> objects CSR (``ptr`` int64, ``idx`` int32, on the device): label = ``pos`` on the positives, ``add`` elsewhere
    (``KBDataset.label_values()``).  Differentiable in x, all_ent and bias; same shapes as ``score_1n_supported``."""
    B = int(x.shape[0])
    if B <= B_TILE:
        return _Score1NBCE.apply(x, all_ent, bias, qid, ptr, idx, pos, add)
    total = None
    for i in range(0, B, B_TILE):                       # mean over B * N = tile means weighted by their share of the batch
        part = _Score1NBCE.apply(x[i:i + B_TILE], all_ent, bias, qid[i:i + B_TILE], ptr, idx, pos, add)
        part = part * (float(min(B_TILE, B - i)) / B)
        total = part if total is None else total + part
    return total


class _Score1NBCEShard(torch.autograd.Function):
    """``score_1n_bce`` on an entity-sharded table (``MGCN.shard``): this rank holds the rows ``ent`` / ``bias`` of the
    entities it owns, and every rank scores the same B queries x.  Per tile of B_TILE queries the scorer runs on the local
    rows, the positives set their bits in the local rows (``row_of``) and the shard loss pass writes the logit gradient with
    the divisor of the whole table (B_tile * n_total) and the shard's fp64 loss sum.  The ranks add the loss sums (ONE
    all-reduce); in the backward they add the partial d_x [B, D] (ONE all-reduce), while d_ent and d_bias stay local."""

    @staticmethod
    def forward(ctx, x, all_ent, bias, qid, ptr, idx, row_of, n_total, coll, pos, add):
        x = _lib.require_cuda(x.detach(), torch.float32, 'x')
        ent = _lib.require_cuda(all_ent.detach(), torch.float32, 'all_ent')
        bias_ = _lib.require_cuda(bias.detach(), torch.float32, 'bias')
        qid = _lib.require_cuda(qid, torch.int64, 'qid')
        ptr = _lib.require_cuda(ptr, torch.int64, 'ptr')
        idx = _lib.require_cuda(idx, torch.int32, 'idx')
        row_of = _lib.require_cuda(row_of, torch.int32, 'row_of')
        B, D = int(x.shape[0]), int(x.shape[1])
        Nl = int(ent.shape[0])
        if int(qid.numel()) != B:
            raise ValueError('qid has {} entries for {} queries'.format(int(qid.numel()), B))
        p, dev = _lib.ptr, x.device
        tiles = [(i, min(B_TILE, B - i)) for i in range(0, B, B_TILE)]
        sums = torch.zeros(((len(tiles) + 1) // 2 * 2,), dtype=torch.float64, device=dev)     # 16-byte all-reduce payload
        d_logit, d_bias = [], []
        for t, (i, bt) in enumerate(tiles):
            ldt = (bt + 3) // 4 * 4
            d_logit_t = torch.empty((Nl, ldt), dtype=torch.float32, device=dev)
            _lib.call('kgc_score_1n_fwd_t', p(ent), Nl, D, ent.stride(0), p(_pack_b(x[i:i + bt].t())), bt, p(bias_), p(d_logit_t),
                      ldt, _lib.stream())
            mask_t = torch.empty((Nl, (bt + 31) // 32), dtype=torch.int32, device=dev)
            _lib.call('kgc_label_mask_t_build_rows', p(qid[i:i + bt]), bt, p(ptr), p(idx), p(row_of), Nl, p(mask_t), _lib.stream())
            db = torch.empty((Nl,), dtype=torch.float32, device=dev)
            partial = torch.empty((int(_lib.lib().kgc_bce_1n_t_blocks(Nl)),), dtype=torch.float64, device=dev)
            _lib.call('kgc_bce_1n_bwd_logit_t_shard', p(d_logit_t), p(mask_t), Nl, bt, ldt, float(pos), float(add), int(n_total),
                      p(db), p(partial), p(sums[t:t + 1]), _lib.stream())
            d_logit.append(d_logit_t)
            d_bias.append(db)
        coll.all_reduce(sums, 'bce_1n_loss')
        # score_1n_bce's value: per tile the mean over bt * N, weighted by the tile's share of the batch
        loss = None
        for t, (i, bt) in enumerate(tiles):
            part = sums[t] * (1.0 / (float(bt) * float(n_total)))
            if len(tiles) > 1:
                part = part * (float(bt) / B)
            loss = part if loss is None else loss + part
        ctx.save_for_backward(x, ent, *d_logit, *d_bias)
        ctx.tiles, ctx.coll = tiles, coll
        return loss.to(torch.float32)

    @staticmethod
    def backward(ctx, g):
        from .conv import gemm_nt, gemm_tn
        x, ent = ctx.saved_tensors[:2]
        T = len(ctx.tiles)
        d_logit, d_bias_t = ctx.saved_tensors[2:2 + T], ctx.saved_tensors[2 + T:]
        B, D = int(x.shape[0]), int(x.shape[1])
        Nl = int(ent.shape[0])
        gs = [g if T == 1 else g * (float(bt) / B) for _, bt in ctx.tiles]
        d_x = torch.empty((B, D), dtype=torch.float32, device=x.device)
        for (i, bt), dl, gt in zip(ctx.tiles, d_logit, gs):
            d_x[i:i + bt] = gemm_tn(dl, ent, torch.empty((dl.shape[1], D), dtype=torch.float32, device=x.device))[:bt] * gt
        ctx.coll.all_reduce(d_x, 'bce_1n_dx')                 # every rank's entities contribute to every query's d_x
        d_ent = d_bias = None
        if ctx.needs_input_grad[1]:
            for (i, bt), dl, gt in zip(ctx.tiles, d_logit, gs):
                part = gemm_nt(dl[:, :bt], (x[i:i + bt] * gt).contiguous(), torch.empty((Nl, D), dtype=torch.float32,
                                                                                       device=x.device))
                d_ent = part if d_ent is None else d_ent + part
        if ctx.needs_input_grad[2]:
            for db, gt in zip(d_bias_t, gs):
                d_bias = db * gt if d_bias is None else d_bias + db * gt
        return d_x, d_ent, d_bias, None, None, None, None, None, None, None, None


def score_1n_bce_shard(x, all_ent, bias, qid, ptr, idx, row_of, n_total, coll, pos=1.0, add=0.0):
    """``score_1n_bce`` over all ``n_total`` entities when this rank holds only the rows of the entities it owns:
    ``all_ent`` / ``bias`` are those rows, ``row_of`` [n_total] int32 maps a global entity id to its local row (-1: another
    rank's), ``coll`` is the partition's exchange (``GraphPartition.collectives``).  Every rank passes the same x and qid and
    gets the same loss; the gradients of x are summed over the ranks, those of all_ent and bias are the local rows'.
    Batches above B_TILE queries are scored tile by tile as ``score_1n_bce`` does."""
    if not score_1n_supported(x, all_ent):
        raise RuntimeError('score_1n_bce_shard: shape not taken by the tensor-core scorer (Dout <= 224, Dout % 4 == 0)')
    return _Score1NBCEShard.apply(x, all_ent, bias, qid, ptr, idx, row_of, int(n_total), coll, pos, add)


# each sampled loss: its C forward and its number of halves (int32 counts, and fp64 loss partials per forward CTA)
_SAMPLED_FWD = {'bce': ('kgc_sampled_bce_fwd', 1), 'adv': ('kgc_sampled_adv_fwd', 2), 'ce': ('kgc_sampled_ce_fwd', 1)}


class _ScoreSampled(torch.autograd.Function):
    """loss = the sampled 1-vs-k loss ``kind`` (K6s): 'bce' the mean BCE of sigmoid(<x[b], all_ent[cand[b, c]]> +
    bias[cand[b, c]]) over the valid slots, 'adv' the self-adversarial loss of ``score_sampled_bce`` and 'ce' the softmax
    cross-entropy of ``score_sampled_ce``; ``scalars`` are that entry's own ((pos, add), (pos, add, temperature) or
    (label_smoothing,)).  The forward makes one pass that yields the loss, the logit gradient g [B, C] and d_x for a unit
    upstream gradient; the backward, the same for every loss, scales d_x and builds the dense table gradient by sorting
    the (entity, slot) pairs (no float atomics).  The entity rows are taken with their row pitch, so they may sit in a
    wider table."""

    @staticmethod
    def forward(ctx, x, all_ent, bias, cand, n_pos, kind, scalars):
        x = _lib.require_cuda(x.detach(), torch.float32, 'x')
        ent = all_ent.detach()
        if ent.dtype != torch.float32:
            raise TypeError('all_ent must be torch.float32, got {}'.format(ent.dtype))
        if ent.stride(1) != 1 or ent.stride(0) % 4 != 0 or ent.data_ptr() % 16 != 0:
            ent = ent.clone(memory_format=torch.contiguous_format)
        bias_ = _lib.require_cuda(bias.detach(), torch.float32, 'bias')
        cand = _lib.require_cuda(cand, torch.int32, 'cand')
        B, D, C, N = int(x.shape[0]), int(x.shape[1]), int(cand.shape[1]), int(ent.shape[0])
        dev, p = x.device, _lib.ptr
        fn, halves = _SAMPLED_FWD[kind]
        g = torch.empty((B, C), dtype=torch.float32, device=dev)
        d_x = torch.empty((B, D), dtype=torch.float32, device=dev)
        counts = torch.empty((halves,), dtype=torch.int32, device=dev)
        partial = torch.empty((halves * int(_lib.lib().kgc_sampled_bce_fwd_blocks(B)),), dtype=torch.float64, device=dev)
        loss = torch.empty((1,), dtype=torch.float32, device=dev)
        _lib.call(fn, p(x), B, D, p(ent), N, ent.stride(0), p(bias_), p(cand), C, int(n_pos), *(float(v) for v in scalars),
                  p(g), p(d_x), p(counts), p(partial), p(loss), _lib.stream())
        ctx.save_for_backward(x, cand, g, d_x)
        ctx.n_ent = N
        return loss[0]

    @staticmethod
    def backward(ctx, d_loss):
        x, cand, g, d_x = ctx.saved_tensors
        B, D, C, N = int(x.shape[0]), int(x.shape[1]), int(cand.shape[1]), ctx.n_ent
        d_ent = d_bias = None
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            dev, p = x.device, _lib.ptr
            scale = d_loss.reshape(1).to(torch.float32).contiguous()
            d_ent = torch.empty((N, D), dtype=torch.float32, device=dev)
            d_bias = torch.empty((N,), dtype=torch.float32, device=dev)
            ws_bytes = int(_lib.lib().kgc_sampled_bce_bwd_table_workspace_bytes(B * C, N))
            ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
            _lib.call('kgc_sampled_bce_bwd_table', p(x), B, D, p(cand), C, p(g), p(scale), N, p(d_ent), D, p(d_bias), p(ws),
                      ws_bytes, _lib.stream())
        return (d_x * d_loss if ctx.needs_input_grad[0] else None, d_ent if ctx.needs_input_grad[1] else None,
                d_bias if ctx.needs_input_grad[2] else None, None, None, None, None)


def check_adversarial_temperature(temperature):
    """``temperature`` as a float: None stays None; anything but a finite real number >= 0 is a ValueError."""
    if temperature is None:
        return None
    if isinstance(temperature, bool) or not isinstance(temperature, numbers.Real) or not math.isfinite(temperature) \
            or temperature < 0:
        raise ValueError('adversarial_temperature must be a finite number >= 0 (or None), got {!r}'.format(temperature))
    return float(temperature)


def score_sampled_bce(x, all_ent, bias, cand, n_pos, pos=1.0, add=0.0, adversarial_temperature=None):
    """Negative-sampled (1-vs-k) BCE: query b of ``x`` [B, D] scores only its candidates ``cand`` [B, C] (int32 entity ids;
    the first ``n_pos`` columns are positives with label ``pos``, the rest negatives with label ``add``, e.g.
    ``KBDataset.label_values()``; -1 marks an empty slot, which adds neither loss nor gradient).  Returns the mean BCE of
    sigmoid(<x[b], all_ent[c]> + bias[c]) over the valid slots (0 when there are none), differentiable in ``x``,
    ``all_ent`` and ``bias``.  The cost is B x C gathered rows, independent of N.  D % 4 == 0, D <= 256; deterministic and graph-capturable.

    ``adversarial_temperature=alpha`` (a finite number >= 0) selects self-adversarial negative sampling (Sun et al. 2019,
    RotatE): query b's valid negatives are weighted by w = softmax(alpha * logit) over them, a constant (no gradient flows
    through the weights), and the loss is 1/2 (mean over the queries with a valid positive of the mean BCE of its valid
    positives) + 1/2 (mean over the queries with a valid negative of the w-weighted BCE sum of its valid negatives); a half
    without such queries adds 0.  alpha = 0 weights a query's negatives uniformly; a large alpha approaches the hardest
    negative.  Same single pass, same row traffic and the same backward as the plain objective.  None (default): the plain
    mean over the valid slots."""
    temperature = check_adversarial_temperature(adversarial_temperature)
    _check_sampled_args('score_sampled_bce', x, all_ent, bias, cand, n_pos)
    if temperature is None:
        return _ScoreSampled.apply(x, all_ent, bias, cand, int(n_pos), 'bce', (pos, add))
    return _ScoreSampled.apply(x, all_ent, bias, cand, int(n_pos), 'adv', (pos, add, temperature))


def check_label_smoothing(label_smoothing):
    """``label_smoothing`` as a float: anything but a finite real number in [0, 1] is a ValueError."""
    if isinstance(label_smoothing, bool) or not isinstance(label_smoothing, numbers.Real) \
            or not (0.0 <= label_smoothing <= 1.0):
        raise ValueError('label_smoothing must be a finite number in [0, 1], got {!r}'.format(label_smoothing))
    return float(label_smoothing)


def check_sampled_criterion(criterion, adversarial_temperature, label_smoothing):
    """The loss options of the sampled objective (``MGCN.loss_sampled``, ``GraphedTrainStep``), checked together:
    ``criterion`` 'bce' (``score_sampled_bce``, optionally self-adversarial) or 'ce' (``score_sampled_ce``, optionally
    label-smoothed).  Returns (temperature or None, label smoothing as a float); a combination that one criterion does not
    take is a ValueError."""
    if criterion not in ('bce', 'ce'):
        raise ValueError("criterion must be 'bce' or 'ce', got {!r}".format(criterion))
    temperature = check_adversarial_temperature(adversarial_temperature)
    eps = check_label_smoothing(label_smoothing)
    if criterion == 'ce' and temperature is not None:
        raise ValueError("adversarial_temperature weights the BCE negatives: it does not combine with criterion='ce'")
    if criterion == 'bce' and eps != 0.0:
        raise ValueError("label_smoothing is the cross-entropy's (criterion='ce'); the BCE criterion takes the dataset's "
                         "label values")
    return temperature, eps


def score_sampled_ce(x, all_ent, bias, cand, n_pos, label_smoothing=0.0):
    """Negative-sampled (1-vs-k) softmax cross-entropy (InfoNCE; LibKGE's ``kl``, PyKEEN's ``CrossEntropyLoss``): query b
    of ``x`` [B, D] scores its candidates ``cand`` [B, C] (int32 entity ids, the first ``n_pos`` columns positives, the
    rest negatives; an id outside [0, N) is an empty slot), z = <x[b], all_ent[c]> + bias[c].  Each valid positive p is
    classified against the query's valid negatives Q_b: the row [z_p, z_{Q_b}] with target 0 (the other positives are not
    in its denominator; duplicate entities count as separate classes), and the loss is
    ``F.cross_entropy(row, 0, label_smoothing=eps)`` averaged over the valid positive slots of the batch (0 when there are
    none).  A positive without a valid negative adds 0 loss and 0 gradient.  ``label_smoothing`` eps in [0, 1] is the
    cross-entropy's own; the dataset's BCE label values do not enter.  Differentiable in ``x``, ``all_ent`` and
    ``bias``; the log-sum-exp runs against a running max, so logits of any size are safe.  Same argument rules, single
    pass over the candidate rows (the positive rows are read twice) and table backward as ``score_sampled_bce``;
    deterministic and graph-capturable."""
    eps = check_label_smoothing(label_smoothing)
    _check_sampled_args('score_sampled_ce', x, all_ent, bias, cand, n_pos)
    return _ScoreSampled.apply(x, all_ent, bias, cand, int(n_pos), 'ce', (eps,))


def _check_sampled_args(fn, x, all_ent, bias, cand, n_pos):
    """The shapes, dtypes and devices the sampled forwards take (``fn`` names the caller in the messages)."""
    if x.dim() != 2 or all_ent.dim() != 2 or bias.dim() != 1 or cand.dim() != 2:
        raise ValueError('{} takes x [B, D], all_ent [N, D], bias [N] and cand [B, C]'.format(fn))
    B, D = int(x.shape[0]), int(x.shape[1])
    N, C = int(all_ent.shape[0]), int(cand.shape[1])
    if int(all_ent.shape[1]) != D or int(bias.shape[0]) != N or int(cand.shape[0]) != B:
        raise ValueError('shape mismatch: x {}, all_ent {}, bias {}, cand {}'.format(
            tuple(x.shape), tuple(all_ent.shape), tuple(bias.shape), tuple(cand.shape)))
    if B < 1 or C < 1 or N < 1 or D < 4 or D > 256 or D % 4 != 0:
        raise ValueError('{} needs B, C, N >= 1 and D % 4 == 0, D <= 256 (got B={}, C={}, N={}, D={})'.format(
            fn, B, C, N, D))
    if isinstance(n_pos, bool) or int(n_pos) != n_pos or not 0 <= n_pos <= C:
        raise ValueError('n_pos must be an integer in [0, C = {}], got {!r}'.format(C, n_pos))
    if cand.dtype != torch.int32:
        raise ValueError('cand must be torch.int32, got {}'.format(cand.dtype))
    if B * C >= 2 ** 31 or N >= 2 ** 31 - 1:
        raise ValueError('{} takes B * C < 2^31 slots and N < 2^31 - 1 entities'.format(fn))
    for t, name in ((x, 'x'), (all_ent, 'all_ent'), (bias, 'bias'), (cand, 'cand')):
        if not t.is_cuda:
            raise RuntimeError('{} must be a CUDA tensor: the M-GCN hot path runs on the GPU only (no CPU fallback)'.format(name))
    if not torch.cuda.is_current_stream_capturing() and bool((cand >= N).any()):
        # (not checked while a CUDA graph is captured: the check reads back; the kernels treat such ids as empty slots)
        raise ValueError('cand holds entity ids >= N = {}'.format(N))


# each shared loss: its C pass
_SHARED_LOSS = {'bce': 'kgc_shared_bce_loss', 'adv': 'kgc_shared_adv_loss', 'ce': 'kgc_shared_ce_loss'}


class _ScoreShared(torch.autograd.Function):
    """The sampled loss ``kind`` of ``_ScoreSampled`` on the broadcast candidates [pos_cand[b] | shared, filtered by query
    b's known objects], with the shared part on the tensor cores: the k gathered rows E_S are scored against the batch
    tile by tile (entity-major logitT [k, ldb], kgc_score_1n_logits_t), the loss pass overwrites the tile with the logit
    gradient and yields the positives' gradient g_pos and d_x part.  The backward scales by the upstream scalar: d_x =
    g_T^T E_S + the positives' part, d_E_S = the per-tile g_T x products added in tile order, and the table gradient is
    the positives' (kgc_sampled_bce_bwd_table, which zero-fills) plus the shared rows added through the sorted ids."""

    @staticmethod
    def forward(ctx, x, all_ent, bias, pos_cand, shared, qid, ptr, idx, kind, scalars):
        x = _lib.require_cuda(x.detach(), torch.float32, 'x').contiguous()
        ent = all_ent.detach()
        if ent.dtype != torch.float32:
            raise TypeError('all_ent must be torch.float32, got {}'.format(ent.dtype))
        if ent.stride(1) != 1 or ent.stride(0) % 4 != 0 or ent.data_ptr() % 16 != 0:
            ent = ent.clone(memory_format=torch.contiguous_format)
        bias_ = _lib.require_cuda(bias.detach(), torch.float32, 'bias').contiguous()
        pos_cand = _lib.require_cuda(pos_cand, torch.int32, 'pos_cand').contiguous()
        shared = _lib.require_cuda(shared, torch.int32, 'shared').contiguous()
        qid = _lib.require_cuda(qid, torch.int64, 'qid').contiguous()
        ptr = _lib.require_cuda(ptr, torch.int64, 'ptr')
        idx = _lib.require_cuda(idx, torch.int32, 'idx')
        B, D, N = int(x.shape[0]), int(x.shape[1]), int(ent.shape[0])
        n_pos, k = int(pos_cand.shape[1]), int(shared.numel())
        dev, p, lib = x.device, _lib.ptr, _lib.lib()
        ldb = (B + 31) // 32 * 32                       # a whole 32-query group per column block of the loss pass
        rows = torch.empty((k, D), dtype=torch.float32, device=dev)
        row_bias = torch.empty((k,), dtype=torch.float32, device=dev)
        _lib.call('kgc_shared_rows', p(ent), N, D, ent.stride(0), p(bias_), p(shared), k, p(rows), p(row_bias), _lib.stream())
        logit_t = torch.empty((k, ldb), dtype=torch.float32, device=dev)
        for i in range(0, B, B_TILE):
            bt = min(B_TILE, B - i)
            _lib.call('kgc_score_1n_logits_t', p(rows), k, D, D, p(_pack_b(x[i:i + bt].t())), bt, p(row_bias),
                      p(logit_t[:, i:]), ldb, _lib.stream())
        mask_t = torch.empty((k, ldb // 32), dtype=torch.int32, device=dev)
        ids = torch.empty((k,), dtype=torch.int32, device=dev)
        slots = torch.empty((k,), dtype=torch.int32, device=dev)
        ws_bytes = int(lib.kgc_shared_mask_workspace_bytes(k, N))
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
        _lib.call('kgc_shared_mask_build', p(shared), k, p(qid), B, p(ptr), p(idx), N, p(mask_t), p(ids), p(slots), p(ws),
                  ws_bytes, _lib.stream())
        g_pos = torch.empty((B, n_pos), dtype=torch.float32, device=dev)
        d_x = torch.empty((B, D), dtype=torch.float32, device=dev)
        d_bias_s = torch.empty((k,), dtype=torch.float32, device=dev)
        loss = torch.empty((1,), dtype=torch.float32, device=dev)
        ws_bytes = int(lib.kgc_shared_loss_workspace_bytes(B, k))
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
        _lib.call(_SHARED_LOSS[kind], p(logit_t), ldb, p(mask_t), p(shared), k, p(x), B, D, p(ent), N, ent.stride(0),
                  p(bias_), p(pos_cand), n_pos, *(float(v) for v in scalars), p(g_pos), p(d_x), p(d_bias_s), p(loss), p(ws),
                  ws_bytes, _lib.stream())
        ctx.save_for_backward(x, rows, logit_t, pos_cand, g_pos, d_x, d_bias_s, ids, slots)
        ctx.n_ent = N
        return loss[0]

    @staticmethod
    def backward(ctx, d_loss):
        from .conv import gemm_nt, gemm_tn
        x, rows, g_t, pos_cand, g_pos, d_x_pos, d_bias_s, ids, slots = ctx.saved_tensors
        B, D, N = int(x.shape[0]), int(x.shape[1]), ctx.n_ent
        k, ldb, n_pos = int(rows.shape[0]), int(g_t.shape[1]), int(pos_cand.shape[1])
        dev, p = x.device, _lib.ptr
        d_x = d_ent = d_bias = None
        if ctx.needs_input_grad[0]:
            d_x = (gemm_tn(g_t, rows, torch.empty((ldb, D), dtype=torch.float32, device=dev))[:B] + d_x_pos) * d_loss
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
            scale = d_loss.reshape(1).to(torch.float32).contiguous()
            d_rows = torch.empty((k, D), dtype=torch.float32, device=dev)
            part = torch.empty((k, D), dtype=torch.float32, device=dev) if B > B_TILE else None
            for i in range(0, B, B_TILE):               # the tiles' products added in tile order
                bt = min(B_TILE, B - i)
                gemm_nt(g_t[:, i:i + bt], x[i:i + bt], d_rows if i == 0 else part)
                if i > 0:
                    d_rows += part
            d_ent = torch.empty((N, D), dtype=torch.float32, device=dev)
            d_bias = torch.empty((N,), dtype=torch.float32, device=dev)
            ws_bytes = int(_lib.lib().kgc_sampled_bce_bwd_table_workspace_bytes(B * n_pos, N))
            ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
            _lib.call('kgc_sampled_bce_bwd_table', p(x), B, D, p(pos_cand), n_pos, p(g_pos), p(scale), N, p(d_ent), D,
                      p(d_bias), p(ws), ws_bytes, _lib.stream())
            _lib.call('kgc_shared_bwd_table', p(ids), p(slots), k, N, D, p(d_rows), D, p(d_bias_s), p(scale), p(d_ent), D,
                      p(d_bias), _lib.stream())
        return (d_x, d_ent if ctx.needs_input_grad[1] else None, d_bias if ctx.needs_input_grad[2] else None,
                None, None, None, None, None, None, None)


def score_shared_bce(x, all_ent, bias, pos_cand, shared, qid, ptr, idx, pos=1.0, add=0.0, adversarial_temperature=None):
    """``score_sampled_bce`` with batch-shared negatives: query b of ``x`` [B, D] scores its positives ``pos_cand``
    [B, n_pos] (int32, -1 an empty slot, e.g. ``KBDataset.positives``) and the ``k`` entities ``shared`` (int32 [k], e.g.
    ``KBDataset.shared_negatives``) that every query shares, each with the entries that are known objects of query
    ``qid[b]`` (the query -> objects CSR ``ptr`` int64 / ``idx`` int32 that ``score_1n_bce`` takes) left out.  The value
    and the gradients are exactly those of ``score_sampled_bce`` on the candidates [pos_cand[b] | shared with the known
    objects of qid[b] set to -1] (duplicates in ``shared`` count as separate slots; a filtered entry is an empty slot of
    that query only).  The k x B logits are one dense product on the tensor cores, so each shared row is read once per
    batch instead of once per query: thousands of negatives per query cost about what the per-query path pays for
    hundreds.  D % 4 == 0, D <= 224; deterministic and graph-capturable."""
    temperature = check_adversarial_temperature(adversarial_temperature)
    _check_shared_args('score_shared_bce', x, all_ent, bias, pos_cand, shared, qid, ptr, idx)
    if temperature is None:
        return _ScoreShared.apply(x, all_ent, bias, pos_cand, shared, qid, ptr, idx, 'bce', (pos, add))
    return _ScoreShared.apply(x, all_ent, bias, pos_cand, shared, qid, ptr, idx, 'adv', (pos, add, temperature))


def score_shared_ce(x, all_ent, bias, pos_cand, shared, qid, ptr, idx, label_smoothing=0.0):
    """``score_sampled_ce`` with batch-shared negatives: each valid positive of ``pos_cand`` [B, n_pos] is classified
    against the ``shared`` [k] entities that are not known objects of its query (see ``score_shared_bce`` for the
    candidate layout and the arguments).  The value and gradients are those of ``score_sampled_ce`` on the broadcast
    candidates; the log-sum-exp runs against each query's max, so logits of any size are safe."""
    eps = check_label_smoothing(label_smoothing)
    _check_shared_args('score_shared_ce', x, all_ent, bias, pos_cand, shared, qid, ptr, idx)
    return _ScoreShared.apply(x, all_ent, bias, pos_cand, shared, qid, ptr, idx, 'ce', (eps,))


def shared_candidates(pos_cand, shared, qid, ptr, idx):
    """The broadcast candidate matrix that defines the shared losses: int32 [B, n_pos + k], row b = [pos_cand[b] | shared
    with every entry that is a known object of query qid[b] set to -1] (torch ops, any device: a reference, not the
    training path)."""
    pos_cand = torch.as_tensor(pos_cand).to(torch.int32)
    shared = torch.as_tensor(shared, device=pos_cand.device).to(torch.int32).reshape(-1)
    qid = torch.as_tensor(qid, device=pos_cand.device).to(torch.int64).reshape(-1)
    ptr = torch.as_tensor(ptr, device=pos_cand.device).to(torch.int64)
    idx = torch.as_tensor(idx, device=pos_cand.device).to(torch.int64)
    B, k = int(pos_cand.shape[0]), int(shared.numel())
    lens = ptr[qid + 1] - ptr[qid]
    rows = torch.repeat_interleave(torch.arange(B, device=pos_cand.device), lens)
    starts = torch.repeat_interleave(ptr[qid], lens)
    offs = torch.arange(int(lens.sum()), device=pos_cand.device) - torch.repeat_interleave(torch.cumsum(lens, 0) - lens, lens)
    known = torch.zeros((B, k), dtype=torch.int32, device=pos_cand.device)
    objs = idx[starts + offs]
    known.index_add_(0, rows, (objs[:, None] == shared[None, :].to(torch.int64)).to(torch.int32))    # [nnz, k] hits
    neg = torch.where(known > 0, torch.full_like(shared, -1)[None, :].expand(B, k), shared[None, :].expand(B, k))
    return torch.cat([pos_cand, neg], 1)


def _check_shared_args(fn, x, all_ent, bias, pos_cand, shared, qid, ptr, idx):
    """The shapes, dtypes and devices the shared-negative losses take (``fn`` names the caller in the messages)."""
    if x.dim() != 2 or all_ent.dim() != 2 or bias.dim() != 1 or pos_cand.dim() != 2 or shared.dim() != 1:
        raise ValueError('{} takes x [B, D], all_ent [N, D], bias [N], pos_cand [B, n_pos] and shared [k]'.format(fn))
    B, D = int(x.shape[0]), int(x.shape[1])
    N, n_pos, k = int(all_ent.shape[0]), int(pos_cand.shape[1]), int(shared.shape[0])
    if int(all_ent.shape[1]) != D or int(bias.shape[0]) != N or int(pos_cand.shape[0]) != B or qid.dim() != 1 \
            or int(qid.shape[0]) != B:
        raise ValueError('shape mismatch: x {}, all_ent {}, bias {}, pos_cand {}, qid {}'.format(
            tuple(x.shape), tuple(all_ent.shape), tuple(bias.shape), tuple(pos_cand.shape), tuple(qid.shape)))
    if B < 1 or N < 1 or D < 4 or D > 224 or D % 4 != 0:
        raise ValueError('{} needs B, N >= 1 and D % 4 == 0, D <= 224 (got B={}, N={}, D={})'.format(fn, B, N, D))
    if k < 1 or n_pos < 1:
        raise ValueError('{} needs k >= 1 shared negatives and n_pos >= 1 positive columns (got k={}, n_pos={})'.format(
            fn, k, n_pos))
    if pos_cand.dtype != torch.int32 or shared.dtype != torch.int32 or idx.dtype != torch.int32:
        raise ValueError('pos_cand, shared and idx must be torch.int32, got {}, {}, {}'.format(
            pos_cand.dtype, shared.dtype, idx.dtype))
    if qid.dtype != torch.int64 or ptr.dtype != torch.int64:
        raise ValueError('qid and ptr must be torch.int64, got {}, {}'.format(qid.dtype, ptr.dtype))
    if B * k >= 2 ** 31 or B * n_pos >= 2 ** 31 or N >= 2 ** 31 - 1:
        raise ValueError('{} takes B * k < 2^31 slots and N < 2^31 - 1 entities'.format(fn))
    for t, name in ((x, 'x'), (all_ent, 'all_ent'), (bias, 'bias'), (pos_cand, 'pos_cand'), (shared, 'shared'),
                    (qid, 'qid'), (ptr, 'ptr'), (idx, 'idx')):
        if not t.is_cuda:
            raise RuntimeError('{} must be a CUDA tensor: the M-GCN hot path runs on the GPU only (no CPU fallback)'.format(name))
    if not torch.cuda.is_current_stream_capturing():
        # (not checked while a CUDA graph is captured: the checks read back; the kernels treat such ids as empty slots)
        if bool(((shared < 0) | (shared >= N)).any()):
            raise ValueError('shared holds entity ids outside [0, N = {})'.format(N))
        if bool((pos_cand >= N).any()):
            raise ValueError('pos_cand holds entity ids >= N = {}'.format(N))


def score_kpad(d):
    kpad = int(_lib.lib().kgc_score_kpad(int(d)))
    if kpad < 0:
        raise ValueError('scoring dimension {} too large (d + 3 <= 256)'.format(d))
    return kpad


class EntityTable(object):
    """bf16 copy of all_ent [N, d] with the decoder bias folded into three extra K columns (pitch kpad)."""

    def __init__(self, all_ent, bias=None):
        all_ent = _lib.require_cuda(all_ent.detach(), torch.float32, 'all_ent')
        self.n, self.d = int(all_ent.shape[0]), int(all_ent.shape[1])
        self.kpad = score_kpad(self.d)
        if bias is not None:
            bias = _lib.require_cuda(bias.detach(), torch.float32, 'bias')
        self.data = torch.empty((self.n, self.kpad), dtype=torch.bfloat16, device=all_ent.device)
        _lib.call('kgc_score_pack_entities', _lib.ptr(all_ent), _lib.ptr(bias), self.n, self.d, _lib.ptr(self.data),
                  _lib.stream())


def pack_queries(xq):
    xq = _lib.require_cuda(xq.detach(), torch.float32, 'xq')
    b, d = int(xq.shape[0]), int(xq.shape[1])
    out = torch.empty((b, score_kpad(d)), dtype=torch.bfloat16, device=xq.device)
    _lib.call('kgc_score_pack_queries', _lib.ptr(xq), b, d, _lib.ptr(out), _lib.stream())
    return out


def pair_scores(q_bf16, table, pair_q, pair_e):
    """s[p] = <Q[pair_q[p]], E[pair_e[p]]> (+ bias) through the same tcgen05 path as the sweep."""
    n_pairs = int(pair_q.numel())
    out = torch.empty((n_pairs,), dtype=torch.float32, device=q_bf16.device)
    if n_pairs == 0:
        return out
    ws_bytes = int(_lib.lib().kgc_score_pairs_workspace_bytes(n_pairs, table.kpad))
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=q_bf16.device)
    p = _lib.ptr
    _lib.call('kgc_score_pairs', p(q_bf16), p(table.data), p(pair_q), p(pair_e), n_pairs, table.kpad, p(out), p(ws),
              ws_bytes, _lib.stream())
    return out


def dense_logits(xq, all_ent, bias):
    """logits[B, N] = xq @ all_ent^T + bias on the fp32-grade tensor-core kernel (3xTF32, K6t without the sigmoid)."""
    xq = _lib.require_cuda(xq.detach(), torch.float32, 'xq')
    ent = _lib.require_cuda(all_ent.detach(), torch.float32, 'all_ent')
    bias = _lib.require_cuda(bias.detach(), torch.float32, 'bias')
    B, D, N = int(xq.shape[0]), int(xq.shape[1]), int(ent.shape[0])
    if not score_1n_supported(xq, ent) or B > B_TILE:
        raise ValueError('dense_logits: at most {} queries per call, Dout <= 224, Dout % 4 == 0'.format(B_TILE))
    ldp = (N + 3) // 4 * 4
    p = _lib.ptr
    packed = _pack_b(xq.t())
    buf = torch.empty((B, ldp), dtype=torch.float32, device=xq.device)
    _lib.call('kgc_score_1n_logits', p(ent), N, D, ent.stride(0), p(packed), B, p(bias), p(buf), ldp, _lib.stream())
    return buf, ldp


def _filtered_rank_fp32(xq, all_ent, bias, obj, filt_ptr, filt_idx, want_eq):
    """Exact-mode core: fp32-grade dense logits tile by tile (the matrix the reference materialises, main.py:121), integer
    counts over them, target / filter logits read from the SAME matrix (bit-consistent with the counts)."""
    dev, b, n = xq.device, int(xq.shape[0]), int(all_ent.shape[0])
    gt = torch.zeros((b,), dtype=torch.int32, device=dev)
    eq = torch.zeros((b,), dtype=torch.int32, device=dev) if want_eq else None
    thr = torch.empty((b,), dtype=torch.float32, device=dev)
    s_filt = torch.empty((int(filt_idx.numel()),), dtype=torch.float32, device=dev)
    lens = filt_ptr[1:] - filt_ptr[:-1]
    rows_of = torch.repeat_interleave(torch.arange(b, device=dev), lens)
    fp = filt_ptr.tolist() if b <= 4096 else None
    p = _lib.ptr
    for i in range(0, b, B_TILE):
        j = min(i + B_TILE, b)
        z, ld = dense_logits(xq[i:j], all_ent, bias)
        thr[i:j] = z[torch.arange(j - i, device=dev), obj[i:j]]
        a, e = (fp[i], fp[j]) if fp is not None else (int(filt_ptr[i]), int(filt_ptr[j]))
        if e > a:
            s_filt[a:e] = z[rows_of[a:e] - i, filt_idx[a:e].long()]
        _lib.call('kgc_rank_count_dense', p(z), ld, n, j - i, p(thr[i:j]), p(gt[i:j]), p(eq[i:j]) if eq is not None else None,
                  _lib.stream())
    return thr, s_filt, gt, eq


def filtered_rank(xq, all_ent, bias, obj, filt_ptr, filt_idx, count_eq=False, table=None, n_offset=0, group=None,
                  precision='bf16'):
    """Filtered rank of obj[q] among all entities for every query row of ``xq`` [B, d].

    filt_ptr [B+1] int64 / filt_idx [nnz] int32: the known positives of each query (CSR, the all-split filter
    of data_loader.py:108-110; may or may not contain the target).  Returns a dict with ranks [B] int32,
    count_gt [B] int32 (already filter-corrected), count_eq (if asked), thr [B] (target logits) and
    sums [13] float64 = {count, sum rank, sum 1/rank, hits@1..10} (main.py:128-133).

    ``precision='bf16'`` (default): the fused tcgen05 sweep K6 - operands rounded to bf16 (logits within 2^-7 relative of
    fp32), the [B, N] matrix never written; the throughput path.  ``precision='fp32'``: exact mode - fp32-grade (3xTF32)
    dense logits tile by tile + integer counts over them: what the reference ranks (fp32 scores, main.py:121-126), for
    evaluations whose metrics must not depend on bf16 rounding of near-tied candidates (needs ``all_ent`` / ``bias``).

    Entity-sharded use (one process per GPU, bf16 path): pass this rank's ``table`` shard (rows n_offset .. n_offset+n)
    and the process ``group``; target / filter logits are computed by the owning rank and summed (each entry
    is non-zero on exactly one rank, so the sum is exact), integer counts are all-reduced (bit-exact).
    """
    dev = xq.device
    b = int(xq.shape[0])
    obj = _lib.require_cuda(obj, torch.int64, 'obj')
    filt_ptr = _lib.require_cuda(filt_ptr, torch.int64, 'filt_ptr')
    filt_idx = _lib.require_cuda(filt_idx, torch.int32, 'filt_idx')
    p = _lib.ptr
    if precision == 'fp32':
        if group is not None or all_ent is None or bias is None:
            raise ValueError("precision='fp32' takes the unsharded fp32 all_ent / bias")
        thr, s_filt, gt, eq = _filtered_rank_fp32(xq, all_ent, bias, obj, filt_ptr, filt_idx, count_eq)
    elif precision == 'bf16':
        if table is None:
            table = EntityTable(all_ent, bias)
        q_bf16 = pack_queries(xq)
        # (query, entity) pairs whose logits are needed exactly: the targets, then every filtered positive
        lens = (filt_ptr[1:] - filt_ptr[:-1])
        rows = torch.arange(b, device=dev, dtype=torch.int32)
        pair_q = torch.cat([rows, torch.repeat_interleave(rows, lens)])
        pair_e = torch.cat([obj.to(torch.int32), filt_idx])
        if group is None:
            s_pairs = pair_scores(q_bf16, table, pair_q, pair_e)
        else:
            import torch.distributed as dist
            local = (pair_e >= n_offset) & (pair_e < n_offset + table.n)
            sel = torch.nonzero(local).squeeze(1)
            s_pairs = torch.zeros((pair_q.numel(),), dtype=torch.float32, device=dev)
            s_pairs[sel] = pair_scores(q_bf16, table, pair_q[sel].contiguous(), (pair_e[sel] - n_offset).contiguous())
            dist.all_reduce(s_pairs, group=group)
        thr = s_pairs[:b].contiguous()
        s_filt = s_pairs[b:].contiguous()
        gt = torch.zeros((b,), dtype=torch.int32, device=dev)
        eq = torch.zeros((b,), dtype=torch.int32, device=dev) if count_eq else None
        _lib.call('kgc_score_rank', p(q_bf16), p(table.data), b, table.n, table.kpad, p(thr), p(gt), p(eq), _lib.stream())
        if group is not None:
            import torch.distributed as dist
            dist.all_reduce(gt, group=group)
            if eq is not None:
                dist.all_reduce(eq, group=group)
    else:
        raise ValueError("precision must be 'bf16' or 'fp32'")
    ranks = torch.empty((b,), dtype=torch.int32, device=dev)
    eq_out = torch.empty((b,), dtype=torch.int32, device=dev) if count_eq else None
    sums = torch.empty((13,), dtype=torch.float64, device=dev)
    _lib.call('kgc_rank_finalize', p(gt), p(eq), p(thr), p(s_filt), p(filt_ptr), p(filt_idx), p(obj), b, p(ranks),
              p(eq_out), p(sums), _lib.stream())
    out = {'ranks': ranks, 'count_gt': ranks - 1, 'thr': thr, 'sums': sums}
    if count_eq:
        out['count_eq'] = eq_out
    return out


TOPK_MAX = 32      # the largest list the fused sweep keeps in registers (K6k)


def _check_exclusions(b, excl_ptr, excl_idx):
    """Device copies of the exclusion CSR after checking its shape: ``ptr`` [b+1] non-decreasing within [0, nnz], every
    row sorted ascending (what the kernels' forward cursor relies on).  (None, None) when no filter is given."""
    if excl_ptr is None and excl_idx is None:
        return None, None
    if excl_ptr is None or excl_idx is None:
        raise ValueError('excl_ptr and excl_idx go together')
    ptr = _lib.require_cuda(excl_ptr, torch.int64, 'excl_ptr')
    idx = _lib.require_cuda(excl_idx, torch.int32, 'excl_idx')
    if ptr.dim() != 1 or int(ptr.numel()) != b + 1:
        raise ValueError('excl_ptr must have B + 1 = {} entries, got {}'.format(b + 1, tuple(ptr.shape)))
    nnz = int(idx.numel())
    bad = (ptr[1:] < ptr[:-1]).any() | (ptr[0] < 0) | (ptr[-1] > nnz)
    if nnz > 1:
        # pair (p, p + 1) decreasing inside one row: rows end where the next one starts
        dec = idx[1:] < idx[:-1]
        cut = ptr[1:-1] - 1
        dec[cut[(cut >= 0) & (cut < nnz - 1)]] = False
        pos = torch.arange(nnz - 1, device=idx.device)
        bad = bad | (dec & (pos >= ptr[0]) & (pos + 1 < ptr[-1])).any()
    if bool(bad):
        raise ValueError('malformed exclusion CSR: excl_ptr must be non-decreasing within [0, len(excl_idx)] and every '
                         'row of excl_idx sorted ascending')
    return (ptr, idx) if nnz > 0 else (None, None)


def _check_k(k):
    if isinstance(k, bool) or not isinstance(k, int) or not 1 <= k <= TOPK_MAX:
        raise ValueError('k must be an integer in [1, {}], got {!r}'.format(TOPK_MAX, k))


def topk(xq, all_ent, bias, k, excl_ptr=None, excl_idx=None, table=None, precision='bf16', n_offset=0, group=None):
    """The ``k`` best entities for every query row of ``xq`` [B, d] against ``all_ent`` [N, d] (+ ``bias`` [N]), leaving out
    each query's exclusion list (the known positives: ``excl_ptr`` [B+1] int64 / ``excl_idx`` int32 CSR, rows sorted
    ascending, e.g. ``DataLoader.known_objects``; None: no filter).

    Order: logit descending, then entity id ascending (-0.0 == +0.0).  Returns {'scores': [B, k] float32 logits, 'ids':
    [B, k] int64, 'count': [B] int32 real entries}; rows with fewer than k eligible entities are padded with (-inf, -1).
    1 <= k <= 32.  Deterministic.

    ``precision='bf16'`` (default): the fused tcgen05 sweep (K6k) on the bf16 entity table - ``table=`` reuses an
    ``EntityTable`` - without writing the [B, N] logits; scores are bit-identical to ``pair_scores``.  ``precision='fp32'``:
    the same selection over fp32-grade dense logits (3xTF32), 256 queries at a time, as in ``filtered_rank``'s exact mode.

    Entity-sharded use, as in ``filtered_rank``: the local rows (``table``, or ``all_ent`` / ``bias`` in fp32) are the
    global entities ``n_offset .. n_offset + n``; the queries and the exclusion CSR are replicated and given in global ids.
    Without ``group`` the result is this slice's top k in global ids (``merge_topk`` combines slices).  With the process
    ``group`` every rank sweeps its rows, the [B, k] results are all-gathered and merged (``merge_topk``) on every rank:
    every rank returns the answer of the unsharded call, bit for bit.  The ranks' row ranges must be disjoint and every
    rank must pass the same B and k (checked: ValueError).  A rank may own no rows."""
    _check_k(k)
    if precision not in ('bf16', 'fp32'):
        raise ValueError("precision must be 'bf16' or 'fp32'")
    if isinstance(n_offset, bool) or not isinstance(n_offset, int) or n_offset < 0:
        raise ValueError('n_offset must be a non-negative integer, got {!r}'.format(n_offset))
    xq = _lib.require_cuda(xq.detach(), torch.float32, 'xq')
    dev, b = xq.device, int(xq.shape[0])
    ptr, idx = _check_exclusions(b, excl_ptr, excl_idx)
    if n_offset == 0 and group is None:
        scores, ids, count = _topk_rows(xq, all_ent, bias, k, ptr, idx, table, precision)
        return {'scores': scores, 'ids': ids.long(), 'count': count}
    if precision == 'bf16' and table is not None:
        n = table.n
    elif all_ent is not None:
        n = int(all_ent.shape[0])
    else:
        raise ValueError("topk takes this shard's rows: table= (bf16) or all_ent (fp32)")
    if n_offset + n >= 2 ** 31:
        raise ValueError('global entity ids must stay below 2^31 (n_offset + n = {})'.format(n_offset + n))
    if group is not None:
        _check_shards(dev, b, k, n_offset, n, group)
    if n > 0 and b > 0:
        if idx is not None:
            # local ids: the shift keeps every row sorted; ids outside [0, n) match no row (clamped into int32 range)
            idx = (idx.long() - n_offset).clamp_(-1, n).to(torch.int32)
        scores, ids, count = _topk_rows(xq, all_ent, bias, k, ptr, idx, table, precision)
        ids = torch.where(ids >= 0, ids + n_offset, ids)
    else:                                  # no rows here: all padding, no launch (the kernels take n > 0 only)
        scores = torch.full((b, k), -float('inf'), dtype=torch.float32, device=dev)
        ids = torch.full((b, k), -1, dtype=torch.int32, device=dev)
        count = torch.zeros((b,), dtype=torch.int32, device=dev)
    if group is None:
        return {'scores': scores, 'ids': ids.long(), 'count': count}
    import torch.distributed as dist
    world = dist.get_world_size(group)
    all_s = torch.empty((world * b, k), dtype=torch.float32, device=dev)
    all_i = torch.empty((world * b, k), dtype=torch.int32, device=dev)
    dist.all_gather_into_tensor(all_s, scores, group=group)
    dist.all_gather_into_tensor(all_i, ids, group=group)
    return merge_topk(all_s.view(world, b, k), all_i.view(world, b, k))


def _check_shards(dev, b, k, n_offset, n, group):
    """One all-gather of (n_offset, n, B, k): every rank raises the same ValueError when the ranks disagree on B or k or
    their row ranges overlap (overlapping shards would return an entity twice)."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    meta = torch.tensor([n_offset, n, b, k], dtype=torch.int64, device=dev)
    every = torch.empty((world, 4), dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(every, meta, group=group)
    every = every.tolist()
    if any(r[2] != b or r[3] != k for r in every):
        raise ValueError('topk with a group: every rank must pass the same B and k, got (B, k) = {}'.format(
            [(r[2], r[3]) for r in every]))
    spans = sorted((r[0], r[0] + r[1]) for r in every if r[1] > 0)
    for (_, hi), (lo, _) in zip(spans, spans[1:]):
        if lo < hi:
            raise ValueError('topk with a group: the ranks\' row ranges overlap: {}'.format(
                [(r[0], r[0] + r[1]) for r in every]))


def _topk_rows(xq, all_ent, bias, k, ptr, idx, table, precision):
    """(scores [B, k], ids [B, k] int32 local, count [B]) over the rows of ``table`` (bf16) or ``all_ent`` (fp32)."""
    dev, b = xq.device, int(xq.shape[0])
    scores = torch.empty((b, k), dtype=torch.float32, device=dev)
    ids = torch.empty((b, k), dtype=torch.int32, device=dev)
    count = torch.empty((b,), dtype=torch.int32, device=dev)
    p = _lib.ptr
    if precision == 'bf16':
        if table is None:
            table = EntityTable(all_ent, bias)
        if b > 0:
            q_bf16 = pack_queries(xq)
            ws_bytes = int(_lib.lib().kgc_score_topk_workspace_bytes(b, table.n, table.kpad, k))
            ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
            _lib.call('kgc_score_topk', p(q_bf16), p(table.data), b, table.n, table.kpad, p(ptr), p(idx), k, p(scores),
                      p(ids), p(count), p(ws), ws_bytes, _lib.stream())
    else:
        if all_ent is None:
            raise ValueError("precision='fp32' takes the fp32 all_ent (and bias)")
        ent = _lib.require_cuda(all_ent.detach(), torch.float32, 'all_ent')
        n, d = int(ent.shape[0]), int(ent.shape[1])
        bias = (torch.zeros((n,), dtype=torch.float32, device=dev) if bias is None
                else _lib.require_cuda(bias.detach(), torch.float32, 'bias'))
        if d % 4 != 0:       # the 3xTF32 scorer takes d % 4 == 0; zero columns leave every logit unchanged
            pad = 4 - d % 4
            xq = torch.nn.functional.pad(xq, (0, pad))
            ent = torch.nn.functional.pad(ent, (0, pad))
        ws_bytes = int(_lib.lib().kgc_topk_dense_workspace_bytes(min(b, B_TILE), n, k))
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
        for i in range(0, b, B_TILE):
            j = min(i + B_TILE, b)
            z, ld = dense_logits(xq[i:j], ent, bias)
            _lib.call('kgc_topk_dense', p(z), ld, n, j - i, p(ptr[i:]) if ptr is not None else None, p(idx), k,
                      p(scores[i:j]), p(ids[i:j]), p(count[i:j]), p(ws), ws_bytes, _lib.stream())
    return scores, ids, count


def merge_topk(scores, ids, k=None):
    """The ``k`` best entries of the union of S finished top-k results (``kgc_topk_merge``): ``scores`` [S, B, k_in] float32
    and ``ids`` [S, B, k_in] int32 or int64 (< 0: padding), every row sorted as ``topk`` returns it, ids disjoint across
    the S results - e.g. ``topk`` of disjoint entity ranges, one per shard or per slice of a table streamed through
    ``topk(..., n_offset=lo)``.  ``k`` (default k_in, at most 32): a smaller k reads the first k entries of every row, a
    larger one pads every row with (-inf, -1).  Returns the dict ``topk`` returns, ordered and padded the same way; the
    result does not depend on the order of the S results.  With k <= k_in it equals ``topk`` over the union of the ranges."""
    scores = _lib.require_cuda(scores.detach(), torch.float32, 'scores')
    if not (torch.is_tensor(ids) and ids.is_cuda):
        raise RuntimeError('ids must be a CUDA tensor: the M-GCN hot path runs on the GPU only (no CPU fallback)')
    if scores.dim() != 3 or tuple(ids.shape) != tuple(scores.shape) or scores.shape[0] < 1 or scores.shape[2] < 1:
        raise ValueError('scores and ids must both be [S, B, k] with S >= 1 and k >= 1, got {} and {}'.format(
            tuple(scores.shape), tuple(ids.shape)))
    if ids.dtype == torch.int64:
        if ids.numel() and int(ids.max()) >= 2 ** 31:
            raise ValueError('ids must be below 2^31')
        ids = ids.clamp(min=-1).to(torch.int32)
    ids = _lib.require_cuda(ids, torch.int32, 'ids')
    n_lists, b, k_in = (int(v) for v in scores.shape)
    k = k_in if k is None else k
    _check_k(k)
    if k < k_in:
        scores, ids = scores[:, :, :k].contiguous(), ids[:, :, :k].contiguous()
    elif k > k_in:
        scores = torch.nn.functional.pad(scores, (0, k - k_in), value=-float('inf'))
        ids = torch.nn.functional.pad(ids, (0, k - k_in), value=-1)
    dev = scores.device
    top_s = torch.empty((b, k), dtype=torch.float32, device=dev)
    top_id = torch.empty((b, k), dtype=torch.int32, device=dev)
    count = torch.empty((b,), dtype=torch.int32, device=dev)
    if b > 0:
        p = _lib.ptr
        _lib.call('kgc_topk_merge', p(scores), p(ids), n_lists, b, k, p(top_s), p(top_id), p(count), _lib.stream())
    return {'scores': top_s, 'ids': top_id.long(), 'count': count}


def tie_adjusted_sums(ranks, count_eq, ties):
    """sums13 under a tie policy: 'optimistic' rank = 1 + gt (what kgc_rank_finalize gives), 'pessimistic' = 1 + gt + eq,
    'mean' = 1 + gt + eq / 2 (the expectation of the reference's arbitrary tie order, main.py:126)."""
    r = ranks.to(torch.float64)
    if ties == 'pessimistic':
        r = r + count_eq.to(torch.float64)
    elif ties == 'mean':
        r = r + 0.5 * count_eq.to(torch.float64)
    elif ties != 'optimistic':
        raise ValueError("ties must be 'optimistic', 'mean' or 'pessimistic'")
    parts = [torch.tensor(float(r.numel()), dtype=torch.float64, device=r.device), r.sum(),
             (1.0 / r.to(torch.float32)).to(torch.float64).sum()]
    parts += [(r <= k).to(torch.float64).sum() for k in range(1, 11)]
    return torch.stack(parts)


SUM_KEYS = ['count', 'mr', 'mrr'] + ['hits@{}'.format(k) for k in range(1, 11)]


def predict(model, data_iters, graph, data_type, device, mode='tail_batch', precision='bf16', ties='optimistic'):
    """Drop-in for main.py:105-135: same signature and result dict (count, mr, mrr, hits@1..10 sums).
    The encoder runs ONCE per call (in eval mode all_ent / all_rel do not depend on the batch: SURVEY.md
    "next" row N3, results identical); every batch then goes through the fused scorer.

    ``precision='fp32'`` ranks fp32-grade logits (exact mode, see filtered_rank) instead of bf16-rounded ones.  ``ties``:
    how candidates whose logit EQUALS the target's are counted - the reference's double argsort breaks ties arbitrarily
    (main.py:126); 'optimistic' (1 + #greater, default), 'mean' or 'pessimistic'.  The number of tied candidates met is
    returned under 'ties' (0 on tie-free data: then all three policies and the reference agree); a warning is issued once
    when ties occur under the optimistic policy, because a degenerate constant-score model would otherwise score MRR = 1."""
    model.eval()
    with torch.no_grad():
        all_ent, all_rel = model.encode(graph)
        table = EntityTable(all_ent, model.conv2.bias) if precision == 'bf16' else None
        total = torch.zeros((13,), dtype=torch.float64, device=all_ent.device)
        n_tied = torch.zeros((), dtype=torch.int64, device=all_ent.device)
        for trip, fptr, fidx in data_iters['{}_{}'.format(data_type, mode.split('_')[0])].sparse():
            sub, rel, obj = trip[:, 0], trip[:, 1], trip[:, 2]
            xq = model.conv2.query(all_ent.index_select(0, sub), all_rel.index_select(0, rel))
            out = filtered_rank(xq, all_ent, model.conv2.bias, obj, fptr, fidx, count_eq=True, table=table, precision=precision)
            n_tied += out['count_eq'].sum()
            total += out['sums'] if ties == 'optimistic' else tie_adjusted_sums(out['ranks'], out['count_eq'], ties)
        total = total.cpu().tolist()
        n_tied = int(n_tied)
    if n_tied and ties == 'optimistic':
        import warnings
        warnings.warn('kgc_gcn_b200.predict: {} candidates tie with their query\'s target logit; ranks are 1 + #greater '
                      '(optimistic). Pass ties="mean" or "pessimistic" for a tie-aware evaluation.'.format(n_tied), RuntimeWarning)
    res = {k: float(v) for k, v in zip(SUM_KEYS, total)}
    res['ties'] = n_tied
    return res


def evaluate(model, data_iters, graph, params, data_type, mark='Val', hits=(1, 3, 10), precision=None, ties=None):
    """Drop-in for main.py:80-102: (tail + head) / (2 * count), rounded to 5 places.  ``precision`` / ``ties`` as in predict
    (defaults: ``params.eval_precision`` / ``params.eval_ties`` when set, else 'bf16' / 'optimistic')."""
    import logging
    import numpy as np
    precision = precision or getattr(params, 'eval_precision', 'bf16')
    ties = ties or getattr(params, 'eval_ties', 'optimistic')
    tail = predict(model, data_iters, graph, data_type, params.device, mode='tail_batch', precision=precision, ties=ties)
    head = predict(model, data_iters, graph, data_type, params.device, mode='head_batch', precision=precision, ties=ties)
    count = float(tail['count'])
    results = {'mr': np.round((tail['mr'] + head['mr']) / (2 * count), 5),
               'mrr': np.round((tail['mrr'] + head['mrr']) / (2 * count), 5)}
    for k in hits:
        key = 'hits@{}'.format(k)
        results[key] = np.round((tail[key] + head[key]) / (2 * count), 5)
    logging.info('- {} metrics: {}  '.format(mark, '; '.join('{}: {:05.3f}'.format(k, v) for k, v in results.items())))
    return results
