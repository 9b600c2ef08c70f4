"""Graph plan: sorted CSRs (K1, built by the CUDA library) + the work-item tables that drive the
deterministic segmented reductions of K2/K3.

The plan is built once per graph (the reference re-derives degrees, norms and gather/scatter
indices on every step: model.py:96-101) and cached on the identity of the edge tensors.
"""
import numpy as np
import torch

from . import _lib

TYPE_BLOCK_ROWS = 65536   # subject rows per block of the blocked d_rel pass (GraphPlan.type_block_rows)
CHUNK0 = 32      # build_levels default fan-in of the first level
CHUNK1 = 2048    # carry / partial rows per item on the fix-up levels (one 1024-thread block): a 38k-edge hub row
                 # (1,187 carry rows) is one item and ONE launch; a 9M-edge hub needs two levels


def build_levels(seg_beg, seg_end, seg_row, chunk0=CHUNK0, chunk1=CHUNK1):
    """Host-side scheduling (pure integer numpy): split every segment [beg,end) into items of at most
    ``chunk`` entries.  A segment that fits one item writes its final row directly; longer segments
    write one partial row per item and become segments of the next level (over partial rows) until
    one item remains.  Returns [(items int32 [n,4] = (beg, end, out, flags), n_partial_rows), ...];
    flags = (final_row << 1) | is_final, out = final row (is_final) or partial slot."""
    levels = []
    beg = np.asarray(seg_beg, dtype=np.int64)
    end = np.asarray(seg_end, dtype=np.int64)
    row = np.asarray(seg_row, dtype=np.int64)
    chunk = chunk0
    while True:
        length = end - beg
        nch = np.maximum(1, -(-length // chunk))
        total = int(nch.sum())
        seg = np.repeat(np.arange(beg.shape[0], dtype=np.int64), nch)
        first = np.cumsum(nch) - nch
        k = np.arange(total, dtype=np.int64) - first[seg]
        ibeg = beg[seg] + k * chunk
        iend = np.minimum(ibeg + chunk, end[seg])
        final = nch[seg] == 1
        slot = np.cumsum(~final) - 1
        out = np.where(final, row[seg], slot)
        flags = (row[seg] << 1) | final.astype(np.int64)
        assert total < 2 ** 31 and (flags < 2 ** 31).all()
        items = np.stack([ibeg, iend, out, flags], 1).astype(np.int32)
        n_part = int((~final).sum())
        levels.append((items, n_part))
        if n_part == 0:
            return levels
        multi = nch > 1
        pfirst = np.cumsum(np.where(multi, nch, 0)) - np.where(multi, nch, 0)
        beg, end, row = pfirst[multi], (pfirst + nch)[multi], row[multi]
        chunk = chunk1


# Compacted halves of the single-GPU layer (conv._ConvFn): a half whose destination rows are mostly empty - a knowledge
# graph's in half, whose rows are the objects of the training triples: 1.1 % of the rows at the Wikidata5M shape - runs its
# dense transforms, tail and weight gradient on its occupied rows only.  A half is compacted when at most this share of its
# rows has an edge ...
COMPACT_MAX_OCCUPANCY = 0.5
# ... and its [rows, Dout] plane is larger than L2 (126 MB): below that the planes are served from L2 and the two row copies
# and the extra launches of the compact path are a larger share of what they save (tests/compact_planes_time.py times both
# paths at the bench shapes)
COMPACT_MIN_PLANE_BYTES = 128 << 20

# Relation gradient factorized by (object, type) group (GroupedPlan): the single-GPU layer takes the grouped streams when in
# both halves the groups - (dst, type) pairs of the in half, (src, type) pairs of the out half - number at most this share of
# the half's edges.  A knowledge graph's objects are hubs (Wikidata5M shape: 3.2 % of the in-half edges), so the d_rel pass,
# a second full read of the edge-embedding table, becomes a reduction over group rows
GROUP_MAX_SHARE = 0.25
# ... and the graph has at least this many directed edges.  Below it the d_rel pass is served largely from L2 and the step is
# bound by launches, which the grouped path adds (tests/factorized_rel_time.py on one B200: WN18RR shape, 173,670 edges,
# 0.383 -> 0.416 ms; FB15k-237 shape, 544,230 edges, 0.413 -> 0.433 ms; Wikidata5M shape, 41.2 M edges, 41.1 -> 38.4 ms)
GROUP_MIN_EDGES = 1 << 22
GROUP_FAN_IN = 32  # entries per first-level item of kgc_group_reduce (one warp, one entry index per lane)

SMALL_ITEM = 16   # fix-up items with at most this many rows are summed by one 8-lane group instead of a whole block
CHUNK_EDGES = 32  # KGC_CHUNK_EDGES: sorted records per streaming chunk (one warp)


def build_grouped_stream(rec_row, rec_grouped, rec_type, rowptr, n_types, plain_base, group_base):
    """Host-side restatement (numpy) of one grouped stream of GroupedPlan.

    The records of a row-sorted CSR (record p belongs to row rec_row[p]; row r holds [rowptr[r], rowptr[r+1])) are
    re-sorted stably by (row, 0) for the records of the PLAIN half and (row, 1 + type) for those of the GROUPED half
    (rec_grouped), so every row keeps its plain records first, in their order, followed by one run per (row, type) group.
    Segments, in record order: one per row for its plain records (output row plain_base + row; empty when it has none) and one
    per group (output row group_base + group id, ids in (row, type) order).  Returns dict with
      order     [n_rec] int64   CSR position of every re-sorted record
      seg_beg / seg_end / seg_row  int64   the segments (for build_stream_plan)
      grp_row / grp_type           int64   row and type of every group"""
    rec_row = np.asarray(rec_row, dtype=np.int64)
    rowptr = np.asarray(rowptr, dtype=np.int64)
    T1 = int(n_types) + 1
    n_rec, n_rows = rec_row.shape[0], rowptr.shape[0] - 1
    key = rec_row * T1 + np.where(np.asarray(rec_grouped, dtype=bool), np.asarray(rec_type, dtype=np.int64) + 1, 0)
    order = np.argsort(key, kind='stable')
    skey = key[order]
    brk = np.flatnonzero(np.diff(skey)) + 1
    beg = np.concatenate([np.zeros(min(n_rec, 1), dtype=np.int64), brk])
    end = np.concatenate([brk, np.full(min(n_rec, 1), n_rec, dtype=np.int64)])
    ukey = skey[beg]
    is_grp = ukey % T1 != 0
    row = np.where(is_grp, group_base + np.cumsum(is_grp) - 1, plain_base + ukey // T1)
    has_plain = np.zeros(n_rows, dtype=bool)
    has_plain[ukey[~is_grp] // T1] = True
    miss = np.flatnonzero(~has_plain)                  # rows without plain records: an empty segment where their records begin
    allkey = np.concatenate([ukey, miss * T1])
    o = np.argsort(allkey, kind='stable')              # the keys are distinct
    return {'order': order, 'seg_beg': np.concatenate([beg, rowptr[miss]])[o],
            'seg_end': np.concatenate([end, rowptr[miss]])[o], 'seg_row': np.concatenate([row, plain_base + miss])[o],
            'grp_row': ukey[is_grp] // T1, 'grp_type': ukey[is_grp] % T1 - 1}


def build_grouped_stream_device(rec_row, rec_grouped, rec_type, rowptr, n_types, plain_base, group_base):
    """build_grouped_stream with torch ops on the device (int64 CUDA tensors in, the same dict of int64 CUDA tensors out;
    bit-identical, tests/test_gpu_factorized_rel.py)."""
    dev = rec_row.device
    T1 = int(n_types) + 1
    n_rows = rowptr.numel() - 1
    key = rec_row * T1 + torch.where(rec_grouped, rec_type + 1, torch.zeros_like(rec_type))
    skey, order = torch.sort(key, stable=True)
    del key
    ukey, cnt = torch.unique_consecutive(skey, return_counts=True)
    del skey
    end = torch.cumsum(cnt, 0)
    beg = end - cnt
    is_grp = ukey % T1 != 0
    row = torch.where(is_grp, group_base + torch.cumsum(is_grp, 0) - 1, plain_base + torch.div(ukey, T1, rounding_mode='floor'))
    has_plain = torch.zeros((n_rows,), dtype=torch.bool, device=dev)
    has_plain[torch.div(ukey[~is_grp], T1, rounding_mode='floor')] = True
    miss = torch.nonzero(~has_plain).view(-1)
    o = torch.argsort(torch.cat([ukey, miss * T1]))
    rp = rowptr.to(torch.int64)
    gk = ukey[is_grp]
    return {'order': order, 'seg_beg': torch.cat([beg, rp[miss]])[o], 'seg_end': torch.cat([end, rp[miss]])[o],
            'seg_row': torch.cat([row, plain_base + miss])[o], 'grp_row': torch.div(gk, T1, rounding_mode='floor'),
            'grp_type': gk % T1 - 1}


def group_segments(keys, n_out=None):
    """Segments of a key-sorted group table: (beg, end, key) of every distinct key, or - n_out given - of every key in
    [0, n_out) (empty segments for the keys without groups)."""
    keys = np.asarray(keys, dtype=np.int64)
    if n_out is None:
        u, first = np.unique(keys, return_index=True)
        return first, np.append(first[1:], keys.shape[0]), u
    ptr = np.searchsorted(keys, np.arange(n_out + 1, dtype=np.int64))
    return ptr[:-1], ptr[1:], np.arange(n_out, dtype=np.int64)


def _fixup_levels(levels, device):
    """Device copies of build_levels tables for kgc_rows_reduce: hub rows first (a block each), then the many small items
    (an 8-lane group each).  [(items, n_items, n_part, n_large)]"""
    out = []
    for it, n_part in levels:
        large = (it[:, 1] - it[:, 0]) > SMALL_ITEM
        order = np.concatenate([np.nonzero(large)[0], np.nonzero(~large)[0]])
        out.append((torch.from_numpy(np.ascontiguousarray(it[order])).to(device), int(it.shape[0]), n_part, int(large.sum())))
    return out


class GroupReduce(object):
    """Schedule of one deterministic reduction over group rows (kgc_group_reduce + kgc_rows_reduce levels):
    out[seg_row[s]] (= or +=) sum over i in [seg_beg[s], seg_end[s]), ascending, of mult[mrow[i]] (.) part[prow[i] or i]."""

    def __init__(self, seg_beg, seg_end, seg_row, mrow, prow, device):
        levels = build_levels(seg_beg, seg_end, seg_row, GROUP_FAN_IN, CHUNK1)
        it0, self.n_part0 = levels[0]
        assert (it0[:, 1] - it0[:, 0]).max(initial=0) <= GROUP_FAN_IN
        self.items0, self.n_items0 = torch.from_numpy(np.ascontiguousarray(it0)).to(device), int(it0.shape[0])
        self.levels = _fixup_levels(levels[1:], device)
        self.mrow = torch.from_numpy(np.asarray(mrow, dtype=np.int32)).to(device)
        self.prow = None if prow is None else torch.from_numpy(np.asarray(prow, dtype=np.int32)).to(device)

    def run(self, plan, part, mult, out, D, accumulate=False, tag='g'):
        p = _lib.ptr
        prev = plan.scratch(tag + 'part0', (self.n_part0, D)) if self.n_part0 else None
        _lib.call('kgc_group_reduce', p(part), p(self.prow), p(mult), p(self.mrow), p(self.items0), self.n_items0, p(out), p(prev),
                  int(accumulate), D, _lib.stream())
        for li, (items, n_items, n_part, n_large) in enumerate(self.levels):
            nxt = plan.scratch('{}part{}'.format(tag, li + 1), (n_part, D)) if n_part else None
            _lib.call('kgc_rows_reduce', p(prev), p(items), n_items, n_large, p(out), p(nxt), p(out) if accumulate else None, D,
                      _lib.stream())
            prev = nxt


class GroupedPlan(object):
    """The single-GPU layer's streams and group tables for the d_rel pass factorized by (object, type) group.

    Edge e = s -> o of type t (in half; its reverse o -> s of type t + R is in the out half):
      agg_in[o]    = sum_t rel[t] (.) P[o,t],   P[o,t] = sum_{e in (o,t)} n_e x[s_e] (.) ee[e]      (forward stream)
      d_x[o]      += sum_t rel[t] (.) Q[o,t],   Q[o,t] = sum_{e in (o,t)} n_e g_out[s_e] (.) ee[e]  (src stream)
      d_rel[t]     = sum_o g_in[o] (.) P[o,t]  (in types),   sum_o x[o] (.) Q[o,t]  (out types)
    fwd: the dst-sorted records, each row's out-half records first (output row Nd + row), then its in-half records as one
      run per (row, type) group (output row 2 Nd + group); their type field is the index of a row of ones appended to the
      relation rows, so kgc_agg_fwd writes P.  rec_f, fwd (StreamPlan), n_in groups: grp_in_row / grp_in_type.
    src: the src-sorted records, each row's in-half records first (output row = row), then its out-half records as one run
      per (row, type) group (output row N + group): kgc_agg_bwd_src_grouped writes d_x without the out half, and Q.
      rec_s, xrow_s (source row per record), src (StreamPlan), n_out groups: grp_out_row / grp_out_type.
    Device memory: two record arrays (16 B per edge each), two rowflags arrays and xrow_s (4 B per edge each) - 44 B per
    directed edge, 1.8 GB at the Wikidata5M shape - next to the plain streams, which bench.py and the partitioned layer keep."""

    def __init__(self, plan, edge_index, n_in_groups_max, n_out_groups_max):
        dev, Nd, N, T = plan.device, plan.num_dst_rows, plan.num_nodes, plan.num_types
        n2, n_in = plan.num_edges2, plan.num_edges_in
        self.ones_row = T - 1          # kgc_agg_fwd reads cat(rels, ones): row T - 1 of it is the row of ones
        self.qualifies = False
        # ---- forward stream: dst-sorted, in half grouped
        eid = plan.rec_dst[:, 0].to(torch.int64)
        g = build_grouped_stream_device(edge_index[1][eid], eid < n_in, plan.rec_dst[:, 2].to(torch.int64),
                                        plan.rowptr_dst, T, Nd, 2 * Nd)
        self.n_in = int(g['grp_row'].numel())
        if self.n_in > n_in_groups_max:
            return
        rec = plan.rec_dst[g['order']]
        rec[:, 2] = torch.where(rec[:, 0] < n_in, torch.full_like(rec[:, 2], self.ones_row), rec[:, 2])
        self.rec_f = rec
        del g['order'], rec, eid
        i32 = lambda t: t.to(torch.int32).contiguous()
        sp = build_stream_plan_device(i32(g['seg_beg']), i32(g['seg_end']), i32(g['seg_row']), n2)
        self.fwd = StreamPlan(sp, n2, dev, prefill_ranges=[(Nd, 2 * Nd)])
        grp_in_row, grp_in_type = g['grp_row'].cpu().numpy(), g['grp_type'].cpu().numpy()
        del g, sp
        # ---- src stream: src-sorted, out half grouped
        eid = plan.rec_src[:, 0].to(torch.int64)
        src = edge_index[0][eid]
        g = build_grouped_stream_device(src, eid >= n_in, plan.rec_src[:, 2].to(torch.int64), plan.rowptr_src, T, 0, N)
        self.n_out = int(g['grp_row'].numel())
        if self.n_out > n_out_groups_max:
            del self.rec_f, self.fwd
            return
        self.rec_s = plan.rec_src[g['order']].contiguous()
        self.xrow_s = src[g['order']].to(torch.int32)
        del src, eid
        sp = build_stream_plan_device(i32(g['seg_beg']), i32(g['seg_end']), i32(g['seg_row']), n2)
        self.src = StreamPlan(sp, n2, dev)
        grp_out_row, grp_out_type = g['grp_row'].cpu().numpy(), g['grp_type'].cpu().numpy()
        del g, sp
        self.grp_in_row, self.grp_in_type, self.grp_out_row, self.grp_out_type = grp_in_row, grp_in_type, grp_out_row, grp_out_type
        # ---- group reductions
        # agg_in from P: one segment per occupied in-half row (plan.rows[0], ascending = the groups' row order), written to
        # the compacted rows (row j) or to the plane (row rows[0][j])
        b, e, r = group_segments(grp_in_row)
        self.agg_in_c = GroupReduce(b, e, np.arange(r.shape[0]), grp_in_type, None, dev)
        self.agg_in = GroupReduce(b, e, r, grp_in_type, None, dev)
        self.n_in_rows = int(r.shape[0])
        # d_x += rel (.) Q, on the rows that have out-half groups
        b, e, r = group_segments(grp_out_row)
        self.dx = GroupReduce(b, e, r, grp_out_type, None, dev)
        # d_rel: every type row from P (types without in-half groups, the self-loop type among them, become 0), then the
        # types of the out-half groups add their sum from Q; the groups of a type in their (row) order
        o_in = np.argsort(grp_in_type, kind='stable')
        b, e, r = group_segments(grp_in_type[o_in], T)
        self.drel_in = GroupReduce(b, e, r, grp_in_row[o_in], o_in, dev)
        o_out = np.argsort(grp_out_type, kind='stable')
        b, e, r = group_segments(grp_out_type[o_out])
        self.drel_out = GroupReduce(b, e, r, grp_out_row[o_out], o_out, dev)
        self.qualifies = True


def build_stream_plan(seg_beg, seg_end, seg_row, n_rec, chunk=CHUNK_EDGES, fan_in=CHUNK1):
    """Host-side scheduling of one streaming aggregation (pure integer numpy).

    The segments [seg_beg, seg_end) tile the sorted record array in order (empty segments allowed); segment s
    reduces into output row seg_row[s].  Returns dict with
      rowflags [n_rec] uint32   row | first-record-of-segment << 30 | last-record-of-segment << 31
      chunks   [n_chunks, 2] int32  (head_slot, tail_slot) carry rows of every chunk of ``chunk`` records, -1 if unused
      n_carry                   number of carry rows
      fill_rows [k] int32       output rows of the empty segments (written by kgc_rows_fill)
      levels                    build_levels() tables that reduce the carry rows of the rows spanning several chunks
    A row's carry rows get consecutive slot numbers in chunk order, so each spanning row is one contiguous
    segment of the carry array."""
    beg = np.asarray(seg_beg, dtype=np.int64)
    end = np.asarray(seg_end, dtype=np.int64)
    row = np.asarray(seg_row, dtype=np.int64)
    assert row.size == 0 or int(row.max()) < (1 << 30)
    length = end - beg
    nz = length > 0
    rec_seg = np.repeat(np.arange(beg.shape[0], dtype=np.int64), length)
    assert rec_seg.shape[0] == n_rec
    flags = row[rec_seg].astype(np.uint32)
    flags[beg[nz]] |= np.uint32(1 << 30)
    flags[end[nz] - 1] |= np.uint32(1 << 31)
    n_chunks = -(-n_rec // chunk) if n_rec else 0
    cb = np.arange(n_chunks, dtype=np.int64) * chunk
    ce = np.minimum(cb + chunk, n_rec)
    if n_chunks:
        lead = rec_seg[cb]                               # segment of the chunk's first record
        trail = rec_seg[ce - 1]                          # ... and of its last record
        needs_head = (beg[lead] < cb) & (end[lead] <= ce)    # began earlier and ends inside this chunk
        needs_tail = end[trail] > ce                         # still open at the end of the chunk
    else:
        needs_head = needs_tail = np.zeros(0, dtype=bool)
    inter = np.stack([needs_head, needs_tail], 1).reshape(-1)
    slot = np.cumsum(inter) - 1
    slots = np.where(inter, slot, -1).reshape(-1, 2).astype(np.int32)
    n_carry = int(inter.sum())
    # rows spanning several chunks: carry rows tail(c_first) .. head(c_last), consecutive by construction
    c_first = beg // chunk
    c_last = (end - 1) // chunk
    span = nz & (c_last > c_first)
    s_beg = slots[c_first[span], 1].astype(np.int64)
    s_end = slots[c_last[span], 0].astype(np.int64) + 1
    assert (s_end - s_beg == (c_last - c_first)[span] + 1).all()
    levels = build_levels(s_beg, s_end, row[span], fan_in, fan_in) if span.any() else []
    return {'rowflags': flags, 'chunks': slots, 'n_carry': n_carry, 'fill_rows': row[~nz].astype(np.int32),
            'levels': levels}


def build_stream_plan_device(seg_beg, seg_end, seg_row, n_rec, chunk=CHUNK_EDGES, fan_in=CHUNK1):
    """The same schedule as build_stream_plan with the O(n_rec) part on the GPU (kgc_stream_plan_flags: row + first / last
    flags per record by binary search over the segment starts, head / tail carry flags per chunk); slot numbers are a prefix
    sum on the device; only the rows that span chunks (a few per mille of the records) come to the host for the fix-up
    levels.  ``seg_*``: int32 CUDA tensors.  Returns the build_stream_plan dict with ``rowflags`` / ``chunks`` as CUDA tensors
    (int32 views) - bit-identical contents (tests/test_gpu_conv.py::test_stream_plan_on_device)."""
    dev = seg_beg.device
    n_seg = int(seg_beg.numel())
    n_chunks = -(-n_rec // chunk) if n_rec else 0
    rowflags = torch.empty((n_rec,), dtype=torch.int32, device=dev)
    inter = torch.zeros((2 * n_chunks,), dtype=torch.int32, device=dev)
    if n_rec:
        rec_seg = torch.empty((n_rec,), dtype=torch.int32, device=dev)
        _lib.call('kgc_stream_plan_flags', _lib.ptr(seg_beg), _lib.ptr(seg_end), _lib.ptr(seg_row), n_seg, n_rec, chunk,
                  _lib.ptr(rowflags), _lib.ptr(rec_seg), _lib.ptr(inter), _lib.stream())
        del rec_seg
    slot = torch.cumsum(inter, 0, dtype=torch.int64) - 1
    slots = torch.where(inter != 0, slot, torch.full_like(slot, -1)).to(torch.int32).view(-1, 2).contiguous()
    n_carry = int(inter.sum())
    beg, end = seg_beg.to(torch.int64), seg_end.to(torch.int64)
    nz = end > beg
    c_first = torch.div(beg, chunk, rounding_mode='floor')
    c_last = torch.div(end - 1, chunk, rounding_mode='floor')
    span = nz & (c_last > c_first)
    fill_rows = seg_row[~nz].to(torch.int32).cpu().numpy()
    if bool(span.any()):
        s_beg = slots[c_first[span], 1].to(torch.int64)
        s_end = slots[c_last[span], 0].to(torch.int64) + 1
        host = torch.stack([s_beg, s_end, seg_row[span].to(torch.int64)]).cpu().numpy()
        levels = build_levels(host[0], host[1], host[2], fan_in, fan_in)
    else:
        levels = []
    return {'rowflags': rowflags, 'chunks': slots, 'n_carry': n_carry, 'fill_rows': fill_rows, 'levels': levels}


class StreamPlan(object):
    """Device copy of one streaming-aggregation schedule (see build_stream_plan)."""

    def __init__(self, sp, n_rec, device, prefill_ranges=None):
        self.n_rec = int(n_rec)
        if torch.is_tensor(sp['rowflags']):                         # built on the device (build_stream_plan_device)
            self.rowflags, self.chunks = sp['rowflags'], sp['chunks']
        else:
            self.rowflags = torch.from_numpy(sp['rowflags'].view(np.int32)).to(device)
            self.chunks = torch.from_numpy(np.ascontiguousarray(sp['chunks'])).to(device)
        self.n_carry = sp['n_carry']
        self.fill_rows = torch.from_numpy(sp['fill_rows']).to(device)
        self.n_fill = int(sp['fill_rows'].shape[0])
        self.levels = []
        levels = list(sp['levels'])
        # Rows without records.  A knowledge graph's in-half plane is mostly such rows (few entities are ever an object:
        # 4.4 M of 4.6 M rows at the Wikidata5M shape): when a contiguous row range is >= 3/4 empty and large, the range
        # is zero-filled by one memset before the streaming kernel (0.3 ms) instead of one 8-lane work item per row (0.87 ms);
        # the remaining empty rows ride in the first fix-up launch as before
        self.prefill = []
        fr_all = sp['fill_rows'].astype(np.int64)
        for lo, hi in (prefill_ranges or ()):
            inside = (fr_all >= lo) & (fr_all < hi)
            n_in = int(inside.sum())
            if n_in >= (1 << 18) and n_in >= 0.75 * (hi - lo):
                self.prefill.append((int(lo), int(hi)))
                fr_all = fr_all[~inside]
        if self.prefill:
            sp = dict(sp, fill_rows=fr_all.astype(np.int32))
            self.n_fill = int(fr_all.shape[0])
        if self.n_fill:
            # rows without any record ride along in the first fix-up launch as EMPTY final items (out = addend or 0):
            # one launch less per aggregation than a separate kgc_rows_fill
            fr = sp['fill_rows'].astype(np.int64)
            empty = np.stack([np.zeros_like(fr), np.zeros_like(fr), fr, (fr << 1) | 1], 1).astype(np.int32)
            if levels:
                levels[0] = (np.concatenate([levels[0][0], empty], 0), levels[0][1])
            else:
                levels = [(empty, 0)]
            self.n_fill = 0
        self.levels = _fixup_levels(levels, device)


class GraphPlan(object):
    """Sorted CSRs + reduction plans of one (edge_index, edge_type) pair.

    Attributes mirror include/kgc_b200.h: deg[2,N] int32, norm[2E] f32, perm_{dst,src,type}[2E] int32,
    rowptr_{dst,src}[N+1], rowptr_type[T+1], rowmid_dst[N], rec_{dst,src,type}[2E,4] int32 (bit view).
    """

    def __init__(self, edge_index, edge_type, num_nodes, num_types, n_edges_in=None, n_dst_rows=None, dst_offset=0,
                 deg=None, type_block_rows=None):
        """Single GPU: edge_index [2, 2E] with the in half first (defaults).  Partitioned (SURVEY.md 8(e)): only the
        edges this rank owns, ``n_edges_in`` in-half edges first, src = global ids, dst = LOCAL row ids in
        [0, n_dst_rows) (global id = dst + dst_offset) and ``deg`` = the GLOBAL per-half degrees [2, num_nodes] int32."""
        edge_index = _lib.require_cuda(edge_index, torch.int64, 'edge_index')
        edge_type = _lib.require_cuda(edge_type, torch.int64, 'edge_type')
        if edge_index.dim() != 2 or edge_index.size(0) != 2 or edge_index.size(1) != edge_type.numel():
            raise ValueError('edge_index must be [2, 2E] and edge_type [2E]')
        n2 = int(edge_type.numel())
        if n_edges_in is None:
            if n2 % 2 != 0:
                raise ValueError('the edge list must hold an in half and an out half of equal size (model.py:84-90)')
            n_edges_in = n2 // 2
        dev = edge_index.device
        N, T = int(num_nodes), int(num_types)
        Nd = N if n_dst_rows is None else int(n_dst_rows)
        self.device, self.num_nodes, self.num_types, self.num_edges2 = dev, N, T, n2
        self.num_dst_rows, self.dst_offset, self.num_edges_in = Nd, int(dst_offset), int(n_edges_in)
        i32 = dict(dtype=torch.int32, device=dev)
        if deg is None:
            self.deg = torch.empty((2, N), **i32)
        else:
            self.deg = _lib.require_cuda(deg, torch.int32, 'deg')
            if tuple(self.deg.shape) != (2, N):
                raise ValueError('deg must be [2, num_nodes]')
        self.norm = torch.empty((n2,), dtype=torch.float32, device=dev)
        self.perm_dst, self.perm_src, self.perm_type = (torch.empty((n2,), **i32) for _ in range(3))
        self.rowptr_dst, self.rowptr_src = torch.empty((Nd + 1,), **i32), torch.empty((N + 1,), **i32)
        # the d_rel pass blocked by subject row (kgc_csr_build): node tables far beyond L2 only.  65,536 rows = 26 MB of x
        # + 26 MB of g per block at D = 100; type_block_rows overrides (0 = plain type sort)
        if type_block_rows is None:
            type_block_rows = TYPE_BLOCK_ROWS if N >= 4 * TYPE_BLOCK_ROWS else 0
        self.type_block_rows = int(type_block_rows)
        Tr = int(_lib.lib().kgc_csr_type_rows(N, T, self.type_block_rows))
        self.num_type_rows, self.num_type_blocks = Tr, Tr // T
        self.rowptr_type = torch.empty((Tr + 1,), **i32)
        self.rowmid_dst = torch.empty((Nd,), **i32)
        self.rec_dst, self.rec_src, self.rec_type = (torch.empty((n2, 4), **i32) for _ in range(3))
        h = _lib.lib()
        ws_bytes = int(h.kgc_csr_workspace_bytes(n2, N, Tr))
        if ws_bytes == 0:
            raise RuntimeError('kgc_csr_workspace_bytes failed: ' + h.kgc_last_error().decode())
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
        src, dst = edge_index[0].contiguous(), edge_index[1].contiguous()
        p = _lib.ptr
        _lib.call('kgc_csr_build', p(src), p(dst), p(edge_type), n2, self.num_edges_in, N, Nd, self.dst_offset, T,
                  0 if deg is None else 1, p(self.deg), p(self.norm),
                  p(self.perm_dst), p(self.rowptr_dst), p(self.rowmid_dst), p(self.rec_dst),
                  p(self.perm_src), p(self.rowptr_src), p(self.rec_src),
                  p(self.perm_type), p(self.rowptr_type), p(self.rec_type), self.type_block_rows, p(ws), ws_bytes, _lib.stream())
        del ws
        # ---- reduction plans: the per-record / per-chunk tables are built on the device from the row pointers
        # (build_stream_plan is the numpy restatement of the same tables, the tested reference)
        # forward: records of dst row i = [rowptr[i], rowmid[i]) (in half, output row i) then [rowmid[i], rowptr[i+1])
        # (out half, output row Nd + i): 2 * Nd segments in record order
        rp, rm = self.rowptr_dst, self.rowmid_dst
        drows = torch.arange(Nd, dtype=torch.int32, device=dev)
        fb = torch.stack([rp[:-1], rm], 1).reshape(-1).contiguous()
        fe = torch.stack([rm, rp[1:]], 1).reshape(-1).contiguous()
        fr = torch.stack([drows, drows + Nd], 1).reshape(-1).contiguous()
        sp_f = build_stream_plan_device(fb, fe, fr, n2)
        del fb, fe, fr
        sp_s = build_stream_plan_device(self.rowptr_src[:-1].contiguous(), self.rowptr_src[1:].contiguous(),
                                        torch.arange(N, dtype=torch.int32, device=dev), n2)
        sp_r = build_stream_plan_device(self.rowptr_type[:-1].contiguous(), self.rowptr_type[1:].contiguous(),
                                        torch.arange(Tr, dtype=torch.int32, device=dev), n2)
        self.fwd = StreamPlan(sp_f, n2, dev, prefill_ranges=[(0, Nd), (Nd, 2 * Nd)])     # per plane; no addend in the forward
        self.bwd_src = StreamPlan(sp_s, n2, dev)
        self.bwd_rel = StreamPlan(sp_r, n2, dev)
        self._scratch = {}
        # occupied destination rows of each half (single-GPU plans only): rows[h] int32 ascending, the rows with at least one
        # record in half h; slot[h] int32 [Nd], the compact index of every row or -1; n_c[h] = their count (host int)
        self.rows = self.slot = self.n_c = None
        if n_dst_rows is None and deg is None and self.dst_offset == 0:
            rp, rm = self.rowptr_dst.to(torch.int64), self.rowmid_dst.to(torch.int64)
            self.rows, self.slot, self.n_c = [], [], []
            for cnt in (rm - rp[:-1], rp[1:] - rm):
                rows = torch.nonzero(cnt > 0).view(-1)
                slot = torch.full((Nd,), -1, **i32)
                slot[rows] = torch.arange(rows.numel(), **i32)
                self.rows.append(rows.to(torch.int32))
                self.slot.append(slot)
                self.n_c.append(int(rows.numel()))
        # the d_rel pass factorized by (object, type) group (GroupedPlan): single GPU, large graph, both halves hub-heavy enough
        self.grouped = None
        if self.rows is not None and n2 >= GROUP_MIN_EDGES:
            g = GroupedPlan(self, edge_index, GROUP_MAX_SHARE * self.num_edges_in, GROUP_MAX_SHARE * (n2 - self.num_edges_in))
            self.grouped = g if g.qualifies else None

    def compact_halves(self, row_bytes):
        """(in, out): whether the single-GPU layer runs that half on its occupied rows, for planes of ``row_bytes`` per row
        (see COMPACT_MAX_OCCUPANCY / COMPACT_MIN_PLANE_BYTES; the same rule for both halves)."""
        if self.rows is None:
            return (False, False)
        Nd = self.num_dst_rows
        large = Nd * row_bytes > COMPACT_MIN_PLANE_BYTES
        return tuple(bool(large and n <= COMPACT_MAX_OCCUPANCY * Nd) for n in self.n_c)

    def side_stream(self):
        """A second stream of this device for work that is off the step's critical path (created once per plan)."""
        if getattr(self, '_side', None) is None:
            self._side = torch.cuda.Stream(device=self.device)
        return self._side

    def scratch(self, name, shape, dtype=torch.float32, zeros=False):
        """Reusable device workspace (caller-allocated, as the C ABI requires); ``zeros``: zero-filled when it is allocated."""
        key = (name, tuple(shape), dtype)
        t = self._scratch.get(key)
        if t is None:
            t = (torch.zeros if zeros else torch.empty)(shape, dtype=dtype, device=self.device)
            self._scratch[key] = t
        return t

    def run_rel_reduction(self, level0, d_relp, D, tag='r'):
        """The d_rel pass: the type-sorted reduction into d_relp [num_types, D]; when the sort is blocked by subject row the
        pass yields one partial row per (block, type) and kgc_block_sum adds the blocks in ascending order."""
        if self.num_type_blocks == 1:
            return self.run_reduction(self.bwd_rel, level0, d_relp, D, tag=tag)
        part = self.scratch(tag + 'blocks', (self.num_type_rows, D))
        self.run_reduction(self.bwd_rel, level0, part, D, tag=tag)
        _lib.call('kgc_block_sum', _lib.ptr(part), self.num_type_blocks, self.num_types * D, _lib.ptr(d_relp), _lib.stream())

    def run_reduction(self, sp, level0, out_final, D, addend=None, tag='', skip_prefill=()):
        """Launch the streaming kernel through ``level0(sp, out_final, carry)``, fill the rows without records and
        reduce the carry rows of chunk-spanning rows through kgc_rows_reduce (fixed order, deterministic).
        ``skip_prefill``: pre-filled row ranges the caller never reads (their rows without records stay unwritten)."""
        carry = self.scratch(tag + 'carry', (max(sp.n_carry, 1), D))
        if addend is None:
            for lo, hi in getattr(sp, 'prefill', ()):
                if (lo, hi) not in skip_prefill:
                    out_final.view(-1, D)[lo:hi].zero_()
        elif getattr(sp, 'prefill', ()):
            raise ValueError('a pre-filled plan cannot take an addend')
        level0(sp, out_final, carry)
        if sp.n_fill:
            _lib.call('kgc_rows_fill', _lib.ptr(sp.fill_rows), sp.n_fill, _lib.ptr(addend), _lib.ptr(out_final), D,
                      _lib.stream())
        prev = carry
        for li, (items, n_items, n_part, n_large) in enumerate(sp.levels):
            part = self.scratch('{}part{}'.format(tag, li), (n_part, D)) if n_part else None
            _lib.call('kgc_rows_reduce', _lib.ptr(prev), _lib.ptr(items), n_items, n_large, _lib.ptr(out_final),
                      _lib.ptr(part), _lib.ptr(addend), D, _lib.stream())
            prev = part


_PLAN_CACHE = {}
_PLAN_CACHE_MAX = 8


def get_plan(edge_index, edge_type, num_nodes, num_types):
    """Plans are cached on the identity + version of the edge tensors (the graph is static across steps,
    main.py:61,121)."""
    key = (edge_index.data_ptr(), edge_type.data_ptr(), edge_index._version, edge_type._version,
           tuple(edge_index.shape), tuple(edge_index.stride()), int(num_nodes), int(num_types), str(edge_index.device))
    plan = _PLAN_CACHE.get(key)
    if plan is None:
        if len(_PLAN_CACHE) >= _PLAN_CACHE_MAX:
            _PLAN_CACHE.pop(next(iter(_PLAN_CACHE)))
        plan = GraphPlan(edge_index, edge_type, num_nodes, num_types)
        plan._keepalive = (edge_index, edge_type)     # pins the addresses the key refers to
        _PLAN_CACHE[key] = plan
    return plan
