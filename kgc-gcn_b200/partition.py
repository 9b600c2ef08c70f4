"""Destination partition of the graph for one-process-per-GPU runs (SURVEY.md 8(e)).

Every directed edge (its edge_embeddings row and optimiser state) belongs to ONE rank, normally the rank that owns its
DESTINATION node; entity_embedding rows belong to the owner of the node.  The forward needs the source rows of the owned
edges (all-gather of x), the backward returns source-row gradients to their owners (reduce-scatter of d_x).

Two ways of choosing the owners:
  * ``balance='range'``  - ``world`` equal contiguous node ranges (the plain reading of "range-partitioned by destination").
    On hub-heavy graphs (the Zipf workloads of SURVEY.md 8(d), real KGs) the rank that holds the hubs owns most edges:
    with the WN18RR-shape generator rank 0 of 2 owns 75% of the edges, rank 0 of 8 owns 56%.
  * ``balance='edges'`` (default) - the same machinery after a node RENUMBERING: nodes are dealt to ranks by decreasing
    in-degree, the heaviest to the least-loaded rank (equal node counts, near-equal edge counts), and the few HUB rows
    whose in-degree alone exceeds half a rank's share are SPLIT: their incoming edges are dealt round-robin to all
    ranks, every rank accumulates them into a private virtual row, and the virtual rows are summed across ranks (one small all-reduce of
    [2, n_hub, D]) into the hub's real row; the backward broadcasts the hub rows' upstream gradient the same way.
    In the renumbered id space rank r owns the contiguous block [r B, (r + 1) B), B = nodes per rank + n_hub (the last
    n_hub rows of a block are the virtual rows), so the range machinery (K1 with dst_offset, all-gather, reduce-scatter)
    is used unchanged.
"""
import numpy as np
import torch

from .plan import GraphPlan


def _half_degrees(ei, E, num_nodes):
    return np.stack([np.bincount(ei[0, :E], minlength=num_nodes), np.bincount(ei[0, E:], minlength=num_nodes)]).astype(np.int32)


def partition_edges(edge_index, edge_type, num_nodes, world, rank):
    """Range partition, pure host integer logic (numpy): which edges rank ``rank`` owns and their local numbering.

    Returns dict(lo, hi, owned_eids [n_local] int64 (in-half edges first, ascending), n_edges_in,
    src (global ids), dst (local row ids), type, deg [2, N] int32 = GLOBAL per-half out-degree by src
    (model.py:73-75), padded to world * per columns).  Blocks are ``per = ceil(num_nodes / world)`` rows wide (equal
    all-gather blocks); when ``num_nodes`` is not a multiple of ``world`` the last block(s) end in rows that do not exist:
    no edge refers to them and the layer never touches them (``hi - lo`` real rows, possibly fewer than ``per``)."""
    ei = np.asarray(edge_index, dtype=np.int64)
    et = np.asarray(edge_type, dtype=np.int64)
    n2 = ei.shape[1]
    if n2 % 2 != 0:
        raise ValueError('edge list must hold an in half and an out half of equal size')
    E = n2 // 2
    per = -(-num_nodes // world)
    lo, hi = min(rank * per, num_nodes), min((rank + 1) * per, num_nodes)
    dst = ei[1]
    owned = np.nonzero((dst >= lo) & (dst < hi))[0]          # ascending: in-half edges (< E) come first
    n_in = int(np.searchsorted(owned, E))
    return {'lo': lo, 'hi': hi, 'per': per, 'owned_eids': owned, 'n_edges_in': n_in, 'src': ei[0, owned],
            'dst': dst[owned] - lo, 'type': et[owned], 'deg': _half_degrees(ei, E, world * per)}


def balanced_assignment(edge_index, num_nodes, world, hub_fraction=0.5, max_hubs=64, n_greedy=8192, weights=None):
    """Edge-balanced node -> (rank, local row) assignment and the hub rows to split; identical on every rank.

    Returns dict(owner [N], slot [N], hubs [n_hub] (node ids, decreasing in-degree), n_loc).  A node is a split hub when
    its in-degree (edges of both halves that point to it) exceeds ``hub_fraction`` of a rank's mean edge count - no
    assignment of whole rows could balance such a row (splitting costs two small all-reduces per step, so rows that can
    be balanced whole are).  The ``n_greedy`` heaviest remaining nodes go, one by one, to the least-loaded rank
    (LPT); the light tail is dealt in snake order, the lightest nodes filling the ranks that took few heavy ones.
    Rank r ends with ``count[r]`` = N // world (+ 1 for the first N % world ranks) nodes; ``n_loc`` = the largest count is
    the row stride of a rank's block, so ranks with one node less carry one row that does not exist (never referenced)."""
    ei = np.asarray(edge_index, dtype=np.int64)
    n2 = ei.shape[1]
    base, rem = divmod(num_nodes, world)
    cap_all = base + (np.arange(world, dtype=np.int64) < rem)  # nodes per rank
    n_loc = int(cap_all.max())
    # ``weights``: the load a node brings to its owner (default: its in-degree = the edges that point to it); with explicit
    # weights no row is split
    indeg = np.bincount(ei[1], minlength=num_nodes).astype(np.int64) if weights is None else np.asarray(weights, dtype=np.int64)
    hubs = np.zeros((0,), dtype=np.int64)
    if world > 1 and weights is None:
        thr = max(1.0, hub_fraction * n2 / world)
        cand = np.nonzero(indeg > thr)[0]
        cand = cand[np.argsort(-indeg[cand], kind='stable')]
        hubs = cand[:max_hubs]
    w = indeg.copy()
    w[hubs] = 0                                               # their edges are dealt to every rank
    order = np.argsort(-w, kind='stable')
    owner = np.empty(num_nodes, dtype=np.int64)
    k = min(num_nodes, n_greedy)
    load = np.zeros(world, dtype=np.int64)
    count = np.zeros(world, dtype=np.int64)
    for v in order[:k]:                                        # LPT over the heavy head
        free = count < cap_all
        r = int(np.argmin(np.where(free, load, np.iinfo(np.int64).max)))
        owner[v] = r
        load[r] += w[v]
        count[r] += 1
    rest = order[k:]
    cap = cap_all - count
    m = int(cap.min())
    j = np.arange(m * world, dtype=np.int64)
    rnd, pos = j // world, j % world
    owner[rest[:m * world]] = np.where(rnd % 2 == 0, pos, world - 1 - pos)    # snake: 0..W-1, W-1..0, ...
    owner[rest[m * world:]] = np.repeat(np.arange(world, dtype=np.int64), cap - m)   # the lightest nodes fill the gaps
    slot = np.empty(num_nodes, dtype=np.int64)
    by_rank = np.argsort(owner[order], kind='stable')          # per rank, nodes in decreasing weight
    slot[order[by_rank]] = np.arange(num_nodes, dtype=np.int64) - np.repeat(np.cumsum(cap_all) - cap_all, cap_all)
    return {'owner': owner, 'slot': slot, 'hubs': hubs, 'n_loc': n_loc, 'count': cap_all}


def partition_edges_balanced(edge_index, edge_type, num_nodes, world, rank, hub_fraction=0.5, max_hubs=64):
    """Edge-balanced partition with split hub rows (module docstring), pure host integer logic (numpy).

    Returns dict(n_loc (row stride of the real rows: the largest node count of any rank), n_hub, block = n_loc + n_hub,
    owned_nodes [n_real <= n_loc] (global ids in local-row order; n_real = N // world or that + 1), hubs [n_hub],
    hub_owner [n_hub], hub_row [n_hub] (local row of the hub at its owner), owned_eids (ascending, in half first),
    n_edges_in, newid [N] (node -> renumbered id = owner * block + local row), halo_rows [n_halo] (ascending renumbered ids
    of the REMOTE rows this rank's edges read), src (COMPACT ids: [0, block) = own rows, block + i = halo_rows[i]), dst
    (local rows, virtual rows are n_loc + h), type, deg [2, block + n_halo] (global per-half degrees by compact id),
    n_halo_max (largest halo of any rank: size of the symmetric tables), peer_idx [world, n_real] int32 (compact row of this
    rank's node v in rank r's table, -1 when r's edges never read v: the partial gradients the owner has to add))."""
    ei = np.asarray(edge_index, dtype=np.int64)
    et = np.asarray(edge_type, dtype=np.int64)
    n2 = ei.shape[1]
    if n2 % 2 != 0:
        raise ValueError('edge list must hold an in half and an out half of equal size')
    E = n2 // 2
    a = balanced_assignment(ei, num_nodes, world, hub_fraction, max_hubs)
    owner, slot, hubs, n_loc = a['owner'], a['slot'], a['hubs'], a['n_loc']
    n_hub = int(hubs.shape[0])
    block = n_loc + n_hub
    newid = owner * block + slot
    dst = ei[1]
    edge_rank = owner[dst]
    dst_new = newid[dst]
    for h, v in enumerate(hubs):                               # deal the hub's incoming edges round-robin, in edge order
        e = np.nonzero(dst == v)[0]
        r = np.arange(e.shape[0], dtype=np.int64) % world
        edge_rank[e] = r
        dst_new[e] = r * block + n_loc + h
    owned = np.nonzero(edge_rank == rank)[0]
    n_in = int(np.searchsorted(owned, E))
    deg = _half_degrees(ei, E, num_nodes)
    deg_ext = np.zeros((2, world * block), dtype=np.int32)
    deg_ext[:, newid] = deg
    for h, v in enumerate(hubs):
        deg_ext[:, np.arange(world) * block + n_loc + h] = deg[:, v][:, None]
    mine = np.nonzero(owner == rank)[0]
    owned_nodes = mine[np.argsort(slot[mine], kind='stable')]
    # halo bookkeeping of the peer-memory exchange (K10): the remote rows this rank's records reference, and for each of
    # its own rows the set of ranks whose edges reference it (bit r = rank r leaves a partial gradient for the row)
    src_new = newid[ei[0]]
    touch = np.zeros(world * block, dtype=np.uint64)
    for r in range(world):
        seen = np.zeros(world * block, dtype=bool)
        seen[src_new[edge_rank == r]] = True                   # boolean scatter: no sort of the 2E source ids
        touch[seen] |= np.uint64(1 << r)
    # COMPACT numbering of this rank's node table: [0, block) = its own rows (real + virtual), then only the remote rows
    # its edges read (ascending renumbered id) - every per-rank structure is O(own rows + halo), not O(all nodes)
    ids = np.arange(world * block, dtype=np.int64)
    n_real = int(a['count'][rank])                             # this rank's real rows (n_loc or n_loc - 1)
    peer_idx = np.full((world, n_real), -1, dtype=np.int32)    # row of MY node v in rank r's partial table, -1: untouched
    n_halo_all = np.zeros(world, dtype=np.int64)
    halo_rows = None
    for r in range(world):
        bit = ((touch >> np.uint64(r)) & np.uint64(1)).astype(bool)
        remote = bit & ((ids < r * block) | (ids >= (r + 1) * block))
        hr = np.nonzero(remote)[0]
        n_halo_all[r] = hr.shape[0]
        pos = np.full(world * block, -1, dtype=np.int64)
        pos[hr] = block + np.arange(hr.shape[0], dtype=np.int64)
        pos[r * block:(r + 1) * block] = np.where(bit[r * block:(r + 1) * block], np.arange(block, dtype=np.int64), -1)
        peer_idx[r] = pos[rank * block:rank * block + n_real]
        if r == rank:
            halo_rows = hr
            cmap = pos.copy()
            cmap[r * block:(r + 1) * block] = np.arange(block, dtype=np.int64)
    n_halo = int(halo_rows.shape[0])
    comp_ids = np.concatenate([np.arange(rank * block, (rank + 1) * block, dtype=np.int64), halo_rows])
    return {'n_loc': n_loc, 'n_real': n_real, 'n_hub': n_hub, 'block': block, 'owned_nodes': owned_nodes, 'hubs': hubs,
            'hub_owner': owner[hubs], 'hub_row': slot[hubs], 'owned_eids': owned, 'n_edges_in': n_in,
            'src': cmap[newid[ei[0, owned]]], 'dst': dst_new[owned] - rank * block, 'type': et[owned],
            'deg': np.ascontiguousarray(deg_ext[:, comp_ids]), 'newid': newid, 'halo_rows': halo_rows.astype(np.int32),
            'n_halo': n_halo, 'n_halo_max': int(n_halo_all.max()), 'peer_idx': peer_idx}


def partition_edges_hybrid(edge_index, edge_type, num_nodes, world, rank):
    """Hybrid cut (degree-based edge placement), pure host integer logic (numpy).

    The destination partition moves one x row in and one d_x row out per DISTINCT remote source of a rank's edges; on a
    hub-heavy graph almost every source of an edge that points to a hub is remote (Wikidata5M shape, 8 ranks: 1.75 M halo
    rows per rank, 700 MB each way per step).  Here an edge lives with the owner of its LOWER-degree endpoint (its
    anchor; ties go to the destination, so a graph without skew degenerates to the destination partition): the
    high-degree endpoint is the remote one, and there are few distinct high-degree nodes.  A rank therefore holds
      * edges whose destination is its own row and whose source may be remote      (as in the destination partition), and
      * edges whose SOURCE is its own row and whose destination is remote: their messages are accumulated into a private
        partial row per remote destination, and the owner of the destination adds the partial rows of all ranks in rank
        order (forward); the upstream gradient rows of those destinations are pulled from their owners (backward).
    Both roles share one compact numbering of a rank's node table: [0, n_loc) = its own rows, n_loc + i = remote[i]
    (ascending renumbered id of every remote node its edges touch as source or destination).  Nodes are dealt to ranks
    by decreasing anchored-edge count (LPT head, snake tail): equal node counts, near-equal edge counts, no split rows.

    Returns dict(n_loc, n_real, n_hub = 0, block = n_loc, owned_nodes, owned_eids (ascending, in half first), n_edges_in,
    newid [N] (= owner * n_loc + local row), halo_rows [n_remote] int32 (the remote list), n_halo, n_halo_max, n_remote_all
    [world], src / dst (compact ids), type, deg [2, n_loc + n_remote], peer_idx [world, n_real] int32 (row of this rank's
    node v in rank r's table when r's edges read it as a SOURCE, else -1; r = rank: v), peer_dst_idx [world, n_real]
    (the same for r's edges that point to v: where r keeps its partial aggregate of v))."""
    ei = np.asarray(edge_index, dtype=np.int64)
    et = np.asarray(edge_type, dtype=np.int64)
    n2 = ei.shape[1]
    if n2 % 2 != 0:
        raise ValueError('edge list must hold an in half and an out half of equal size')
    E = n2 // 2
    src, dst = ei[0], ei[1]
    tot = np.bincount(src, minlength=num_nodes) + np.bincount(dst, minlength=num_nodes)
    anchor = np.where(tot[src] < tot[dst], src, dst)
    w = np.bincount(anchor, minlength=num_nodes).astype(np.int64)
    a = balanced_assignment(ei, num_nodes, world, weights=w)
    owner, slot, n_loc = a['owner'], a['slot'], a['n_loc']
    block = n_loc
    newid = owner * block + slot
    edge_rank = owner[anchor]
    owned = np.nonzero(edge_rank == rank)[0]
    n_in = int(np.searchsorted(owned, E))
    src_new, dst_new = newid[src], newid[dst]
    n_real = int(a['count'][rank])
    mine = np.nonzero(owner == rank)[0]
    owned_nodes = mine[np.argsort(slot[mine], kind='stable')]
    my_ids = np.arange(rank * block, rank * block + n_real, dtype=np.int64)
    ids = np.arange(world * block, dtype=np.int64)
    peer_src = np.full((world, n_real), -1, dtype=np.int32)
    peer_dst = np.full((world, n_real), -1, dtype=np.int32)
    n_remote_all = np.zeros(world, dtype=np.int64)
    remote_mine = cmap = None
    for r in range(world):
        sel = edge_rank == r
        seen_s = np.zeros(world * block, dtype=bool)
        seen_d = np.zeros(world * block, dtype=bool)
        seen_s[src_new[sel]] = True
        seen_d[dst_new[sel]] = True
        outside = (ids < r * block) | (ids >= (r + 1) * block)
        remote = np.nonzero((seen_s | seen_d) & outside)[0]
        n_remote_all[r] = remote.shape[0]
        pos = np.full(world * block, -1, dtype=np.int64)
        pos[remote] = block + np.arange(remote.shape[0], dtype=np.int64)
        if r == rank:
            peer_src[r] = peer_dst[r] = np.arange(n_real, dtype=np.int32)       # its own partial rows
            remote_mine = remote
            cmap = pos
            cmap[r * block:(r + 1) * block] = np.arange(block, dtype=np.int64)
        else:
            peer_src[r] = np.where(seen_s[my_ids], pos[my_ids], -1)
            peer_dst[r] = np.where(seen_d[my_ids], pos[my_ids], -1)
    deg = _half_degrees(ei, E, num_nodes)
    deg_ext = np.zeros((2, world * block), dtype=np.int32)
    deg_ext[:, newid] = deg
    comp_ids = np.concatenate([np.arange(rank * block, (rank + 1) * block, dtype=np.int64), remote_mine])
    return {'n_loc': n_loc, 'n_real': n_real, 'n_hub': 0, 'block': block, 'owned_nodes': owned_nodes,
            'hubs': np.zeros((0,), dtype=np.int64), 'owned_eids': owned, 'n_edges_in': n_in,
            'src': cmap[src_new[owned]], 'dst': cmap[dst_new[owned]], 'type': et[owned],
            'deg': np.ascontiguousarray(deg_ext[:, comp_ids]), 'newid': newid, 'halo_rows': remote_mine.astype(np.int32),
            'n_halo': int(remote_mine.shape[0]), 'n_halo_max': int(n_remote_all.max()), 'n_remote_all': n_remote_all,
            'peer_idx': peer_src, 'peer_dst_idx': peer_dst}


def _balanced_assignment_t(w, num_nodes, world, n_greedy=8192):
    """balanced_assignment(weights=w) with torch tensors on w's device (the O(N) parts; the LPT loop over the n_greedy
    heaviest nodes runs on the host over copies of their weights).  Same integers as the numpy function."""
    dev = w.device
    base, rem = divmod(num_nodes, world)
    cap_all = base + (torch.arange(world, dtype=torch.int64) < rem).to(torch.int64)          # host
    n_loc = int(cap_all.max())
    order = torch.sort(-w, stable=True).indices
    k = min(num_nodes, n_greedy)
    head = order[:k].cpu().numpy()
    w_head = w[order[:k]].cpu().numpy()
    cap_np = cap_all.numpy()
    load = np.zeros(world, dtype=np.int64)
    count = np.zeros(world, dtype=np.int64)
    own_head = np.empty(k, dtype=np.int64)
    big = np.iinfo(np.int64).max
    for i in range(k):                                        # LPT over the heavy head
        r = int(np.argmin(np.where(count < cap_np, load, big)))
        own_head[i] = r
        load[r] += w_head[i]
        count[r] += 1
    owner = torch.empty(num_nodes, dtype=torch.int64, device=dev)
    owner[order[:k]] = torch.from_numpy(own_head).to(dev)
    rest = order[k:]
    cap = cap_np - count
    m = int(cap.min())
    j = torch.arange(m * world, dtype=torch.int64, device=dev)
    rnd, pos = torch.div(j, world, rounding_mode='floor'), j % world
    owner[rest[:m * world]] = torch.where(rnd % 2 == 0, pos, world - 1 - pos)    # snake: 0..W-1, W-1..0, ...
    owner[rest[m * world:]] = torch.repeat_interleave(torch.arange(world, dtype=torch.int64, device=dev),
                                                      torch.from_numpy(cap - m).to(dev))
    slot = torch.empty(num_nodes, dtype=torch.int64, device=dev)
    by_rank = torch.sort(owner[order], stable=True).indices    # per rank, nodes in decreasing weight
    first = (torch.cumsum(cap_all, 0) - cap_all).to(dev)
    slot[order[by_rank]] = torch.arange(num_nodes, dtype=torch.int64, device=dev) - torch.repeat_interleave(first, cap_all.to(dev))
    return {'owner': owner, 'slot': slot, 'n_loc': n_loc, 'count': cap_np}


def partition_edges_hybrid_device(edge_index, edge_type, num_nodes, world, rank):
    """partition_edges_hybrid on the device of ``edge_index`` (torch ops: histograms, stable sorts, boolean scatters; the
    numpy function needs ~8 s per rank at the Wikidata5M shape, all of it host work outside every timed region).  Returns the
    same dict with torch tensors on that device in place of the numpy arrays ('count' / 'n_remote_all' stay host arrays);
    bit-identical contents (tests/test_gpu_conv.py::test_hybrid_partition_on_device)."""
    ei = edge_index.to(torch.int64)
    et = edge_type.to(torch.int64)
    dev = ei.device
    n2 = int(ei.shape[1])
    if n2 % 2 != 0:
        raise ValueError('edge list must hold an in half and an out half of equal size')
    E = n2 // 2
    src, dst = ei[0], ei[1]
    tot = torch.bincount(src, minlength=num_nodes) + torch.bincount(dst, minlength=num_nodes)
    anchor = torch.where(tot[src] < tot[dst], src, dst)
    w = torch.bincount(anchor, minlength=num_nodes)
    a = _balanced_assignment_t(w, num_nodes, world)
    owner, slot, n_loc = a['owner'], a['slot'], a['n_loc']
    block = n_loc
    newid = owner * block + slot
    edge_rank = owner[anchor]
    owned = torch.nonzero(edge_rank == rank).squeeze(1)
    n_in = int(torch.searchsorted(owned, torch.tensor([E], device=dev, dtype=torch.int64)))
    src_new, dst_new = newid[src], newid[dst]
    n_real = int(a['count'][rank])
    mine = torch.nonzero(owner == rank).squeeze(1)
    owned_nodes = mine[torch.sort(slot[mine], stable=True).indices]
    my_ids = torch.arange(rank * block, rank * block + n_real, dtype=torch.int64, device=dev)
    ids = torch.arange(world * block, dtype=torch.int64, device=dev)
    peer_src = torch.full((world, n_real), -1, dtype=torch.int32, device=dev)
    peer_dst = torch.full((world, n_real), -1, dtype=torch.int32, device=dev)
    n_remote_all = np.zeros(world, dtype=np.int64)
    remote_mine = cmap = None
    for r in range(world):
        sel = edge_rank == r
        seen_s = torch.zeros(world * block, dtype=torch.bool, device=dev)
        seen_d = torch.zeros(world * block, dtype=torch.bool, device=dev)
        seen_s[src_new[sel]] = True
        seen_d[dst_new[sel]] = True
        outside = (ids < r * block) | (ids >= (r + 1) * block)
        remote = torch.nonzero((seen_s | seen_d) & outside).squeeze(1)
        n_remote_all[r] = int(remote.numel())
        pos = torch.full((world * block,), -1, dtype=torch.int64, device=dev)
        pos[remote] = block + torch.arange(remote.numel(), dtype=torch.int64, device=dev)
        if r == rank:
            own = torch.arange(n_real, dtype=torch.int32, device=dev)
            peer_src[r], peer_dst[r] = own, own
            remote_mine = remote
            cmap = pos
            cmap[r * block:(r + 1) * block] = torch.arange(block, dtype=torch.int64, device=dev)
        else:
            peer_src[r] = torch.where(seen_s[my_ids], pos[my_ids], torch.full_like(my_ids, -1)).to(torch.int32)
            peer_dst[r] = torch.where(seen_d[my_ids], pos[my_ids], torch.full_like(my_ids, -1)).to(torch.int32)
    deg = torch.stack([torch.bincount(src[:E], minlength=num_nodes), torch.bincount(src[E:], minlength=num_nodes)]).to(torch.int32)
    deg_ext = torch.zeros((2, world * block), dtype=torch.int32, device=dev)
    deg_ext[:, newid] = deg
    comp_ids = torch.cat([torch.arange(rank * block, (rank + 1) * block, dtype=torch.int64, device=dev), remote_mine])
    return {'n_loc': n_loc, 'n_real': n_real, 'n_hub': 0, 'block': block, 'owned_nodes': owned_nodes,
            'hubs': np.zeros((0,), dtype=np.int64), 'owned_eids': owned, 'n_edges_in': n_in,
            'src': cmap[src_new[owned]], 'dst': cmap[dst_new[owned]], 'type': et[owned],
            'deg': deg_ext[:, comp_ids].contiguous(), 'newid': newid, 'halo_rows': remote_mine.to(torch.int32),
            'n_halo': int(remote_mine.numel()), 'n_halo_max': int(n_remote_all.max()), 'n_remote_all': n_remote_all,
            'peer_idx': peer_src, 'peer_dst_idx': peer_dst}


def sparse_peer_table(peer, rank):
    """[world, n_real] table of partial-row positions (-1: none) -> (rows [n_list] int32: the own rows some OTHER rank holds
    a partial row for, idx [world, n_list] int32: the table restricted to them, this rank's own line set to -1)."""
    peer = np.asarray(peer)
    others = peer.copy()
    others[rank] = -1
    rows = np.nonzero((others >= 0).any(0))[0].astype(np.int32)
    return torch.from_numpy(rows), torch.from_numpy(np.ascontiguousarray(others[:, rows]).astype(np.int32))


def halo_pull_order(halo_rows, block, rank, world, trip=8):
    """The sequence in which kgc_p2p_halo_gather pulls the positions of ``halo_rows`` (ascending renumbered ids, i.e.
    ascending owner): trips of ``trip`` consecutive positions are dealt to the owners in turn - first trip of owner
    rank + 1, of rank + 2, ..., then their second trips, ... - so that every reader spreads over all owners from the first
    trip on and no owner's NVLink egress is shared by all readers at once.  Pure host integer logic; a permutation."""
    hr = np.asarray(halo_rows, dtype=np.int64)
    n = int(hr.shape[0])
    if n == 0:
        return np.zeros((0,), dtype=np.int32)
    n_trips = -(-n // trip)
    first = np.arange(n_trips, dtype=np.int64) * trip
    owner = hr[first] // block                                  # a trip belongs to the owner of its first row
    turn = (owner - rank - 1) % world                           # 0 for the owner right behind this rank
    start = np.searchsorted(owner, owner, side='left')          # first trip of that owner (owners ascend)
    k = np.arange(n_trips, dtype=np.int64) - start              # number of the trip within its owner
    trips = np.lexsort((turn, k))                               # by k, then by turn
    pos = (first[trips][:, None] + np.arange(trip, dtype=np.int64)[None, :]).reshape(-1)
    return pos[pos < n].astype(np.int32)


class GraphPartition(object):
    """This rank's share of the graph + its GraphPlan (built by K1 with the global degrees).

    ``owned_nodes`` [n_real]: global ids of this rank's node rows in local-row order (shard x / masks / upstream gradients
    with it); ``owned_eids``: global ids of the edges it owns (shard edge_embeddings with it).  ``n_loc`` = the row stride
    of a block (largest node count of any rank; ``n_real`` is n_loc or, when num_nodes is not a multiple of the number of
    ranks, one less: the missing row is never referenced), virtual hub rows are local rows n_loc .. n_loc + n_hub."""

    def __init__(self, edge_index, edge_type, num_nodes, num_types, world, rank, device, group=None, balance='edges',
                 hub_fraction=0.1, p2p='auto'):
        ei = edge_index.cpu().numpy() if torch.is_tensor(edge_index) else edge_index
        et = edge_type.cpu().numpy() if torch.is_tensor(edge_type) else edge_type
        self.world, self.rank, self.group, self.num_nodes = int(world), int(rank), group, int(num_nodes)
        self.balance = balance
        self.device = torch.device(device)
        self._p2p_mode, self._p2p = p2p, {}
        if balance == 'range':
            info = partition_edges(ei, et, num_nodes, world, rank)
            self.lo, self.hi = info['lo'], info['hi']
            self.n_loc, self.n_hub, self.block, self.n_real = info['per'], 0, info['per'], self.hi - self.lo
            self.owned_nodes = torch.arange(self.lo, self.hi, dtype=torch.int64, device=device)
            ext_nodes, offset = world * info['per'], rank * info['per']      # gathered layout: equal blocks of `per` rows
            self.hub_idx_mine = self.hub_rows_mine = None
        elif balance == 'edges':
            info = partition_edges_balanced(ei, et, num_nodes, world, rank, hub_fraction=hub_fraction)
            self.lo = self.hi = None
            self.n_loc, self.n_hub, self.block, self.n_real = info['n_loc'], info['n_hub'], info['block'], info['n_real']
            self.owned_nodes = torch.from_numpy(info['owned_nodes']).to(device)
            ext_nodes, offset = self.block + info['n_halo'], 0      # compact node table: own rows, then the halo
            mine = np.nonzero(info['hub_owner'] == rank)[0]
            self.hub_idx_mine = torch.from_numpy(mine.astype(np.int64)).to(device)           # which hubs this rank owns
            self.hub_rows_mine = torch.from_numpy(info['hub_row'][mine].astype(np.int64)).to(device)   # their local rows
            self.hubs = info['hubs']
            self.halo_rows = torch.from_numpy(info['halo_rows']).to(device)
            self.halo_rows64 = self.halo_rows.to(torch.int64)
            self.halo_order = torch.from_numpy(halo_pull_order(info['halo_rows'], self.block, rank, world)).to(device)
            self.n_halo, self.n_halo_max = info['n_halo'], info['n_halo_max']
            self.peer_idx = torch.from_numpy(info['peer_idx']).to(device)
        elif balance == 'hybrid':
            # an edge lives with its lower-degree endpoint (partition_edges_hybrid): remote rows are few; they are read as
            # sources AND written as destinations (partial aggregates the owners add up), one compact numbering for both.
            # On a CUDA device the partition itself is computed there (the same integers as the numpy version)
            if self.device.type == 'cuda':
                ei_d = (edge_index if torch.is_tensor(edge_index) else torch.from_numpy(np.asarray(edge_index))).to(self.device)
                et_d = (edge_type if torch.is_tensor(edge_type) else torch.from_numpy(np.asarray(edge_type))).to(self.device)
                info = partition_edges_hybrid_device(ei_d, et_d, num_nodes, world, rank)
                del ei_d, et_d
            else:
                info = partition_edges_hybrid(ei, et, num_nodes, world, rank)
            tt = lambda a: (a if torch.is_tensor(a) else torch.from_numpy(np.asarray(a))).to(device)      # noqa: E731
            nn_ = lambda a: a.cpu().numpy() if torch.is_tensor(a) else np.asarray(a)                       # noqa: E731
            self.lo = self.hi = None
            self.n_loc, self.n_hub, self.block, self.n_real = info['n_loc'], 0, info['block'], info['n_real']
            self.owned_nodes = tt(info['owned_nodes'])
            ext_nodes, offset = self.block + info['n_halo'], 0
            self.hub_idx_mine = self.hub_rows_mine = None
            self.hubs = info['hubs']
            self.halo_rows = tt(info['halo_rows'])
            self.halo_rows64 = self.halo_rows.to(torch.int64)
            self.halo_order = torch.from_numpy(halo_pull_order(nn_(info['halo_rows']), self.block, rank, world)).to(device)
            self.n_halo, self.n_halo_max = info['n_halo'], info['n_halo_max']
            self.n_remote_all = [int(v) for v in info['n_remote_all']]
            self.peer_idx = tt(info['peer_idx'])
            self.peer_dst_idx = tt(info['peer_dst_idx'])
            # only the rows OTHER ranks contributed to take part in the two reductions: (row list, [world, n_list] index
            # table with -1 in this rank's own line - its own value is already in place)
            self.sparse_src = tuple(t.to(device) for t in sparse_peer_table(nn_(info['peer_idx']), rank))
            self.sparse_dst = tuple(t.to(device) for t in sparse_peer_table(nn_(info['peer_dst_idx']), rank))
            info = dict(info, owned_eids=tt(info['owned_eids']), src=tt(info['src']), dst=tt(info['dst']), type=tt(info['type']),
                        deg=tt(info['deg']))
        else:
            raise ValueError("balance must be 'hybrid', 'edges' or 'range'")
        self.hybrid = balance == 'hybrid'
        as_t = lambda a: (a if torch.is_tensor(a) else torch.from_numpy(a)).to(device)                     # noqa: E731
        self.owned_eids = as_t(info['owned_eids'])
        self.n_edges_in = info['n_edges_in']
        self.edge_index = torch.stack([as_t(info['src']), as_t(info['dst'])])
        self.edge_type = as_t(info['type'])
        self.plan = GraphPlan(self.edge_index, self.edge_type, ext_nodes, num_types, n_edges_in=self.n_edges_in,
                              n_dst_rows=ext_nodes if self.hybrid else self.block, dst_offset=offset,
                              deg=as_t(info['deg']))

    def collectives(self, D=None):
        """The exchanges of this partition (conv._Collectives) for feature width ``D``.  ``D=None``: those of a width
        already in use (the first peer-memory context created, e.g. by the layer's forward), NCCL when there is none."""
        from .conv import _Collectives
        ctx = next((c for c in self._p2p.values() if c is not None), None) if D is None else self.p2p(D)
        return _Collectives(self.group, self.world, self.num_nodes, self.n_hub, self.hub_idx_mine, self.hub_rows_mine, ctx,
                            self.rank, getattr(self, 'halo_rows64', None), self.n_loc)

    def row_of(self):
        """[num_nodes] int32 on the device: the local row of every node this rank owns (``owned_nodes`` order), -1 for
        the nodes of other ranks."""
        if getattr(self, '_row_of', None) is None:
            r = torch.full((self.num_nodes,), -1, dtype=torch.int32, device=self.device)
            r[self.owned_nodes] = torch.arange(self.owned_nodes.numel(), dtype=torch.int32, device=self.device)
            self._row_of = r
        return self._row_of

    # ------------------------------------------------------------------ peer-memory halo exchange (K10)
    def p2p(self, D):
        """Symmetric buffers + peer pointer tables of the halo exchange for feature width ``D`` (allocated and rendezvoused
        at first use - a collective call), or None when the exchange runs on NCCL: range partitions, CPU / gloo groups,
        ``p2p=False``, or a torch build / topology without symmetric memory (``p2p='auto'`` falls back silently,
        ``p2p=True`` raises)."""
        if D in self._p2p:
            return self._p2p[D]
        ctx = None
        if self.hybrid and not self._p2p_mode:
            raise RuntimeError("balance='hybrid' exchanges partial aggregates over peer memory (K10): it needs p2p")
        if self._p2p_mode and self.balance in ('edges', 'hybrid') and self.world > 1 and self.world <= 8 and self.device.type == 'cuda':
            err = None
            try:
                ctx = _P2PContext(self, D)
            except Exception as exc:                            # pragma: no cover (depends on the box)
                err, ctx = exc, None
            # all ranks or none - and every rank reaches this all-reduce, whatever happened on it
            ok = torch.tensor([1 if ctx is not None else 0], device=self.device)
            import torch.distributed as dist
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)
            if int(ok) == 0:
                ctx = None
                if self._p2p_mode is True or self.hybrid:
                    raise RuntimeError('peer-memory exchange (symmetric memory) is not available on every rank'
                                       + ('' if err is None else ': {!r}'.format(err)))
        elif self.hybrid:
            raise RuntimeError("balance='hybrid' needs 2..8 CUDA ranks with peer memory")
        self._p2p[D] = ctx
        return ctx


class _P2PContext(object):
    """Symmetric memory of one partition and feature width: the gathered node table, the partial d_x table, the staging
    slots of the small all-reduces and the barrier flags, with the device arrays of peer pointers the K10 kernels take."""

    STAGE_BYTES = 4 << 20

    def __init__(self, part, D):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        group = part.group if part.group is not None else dist.group.WORLD
        dev, W, B = part.device, part.world, part.block
        self.rank, self.world, self.block, self.D = part.rank, W, B, D
        rows = B + part.n_halo_max                                              # same size on every rank (symmetric)
        self.table = symm.empty((rows, D), dtype=torch.float32, device=dev)     # own block, then the pulled halo rows
        self.partial = symm.empty((rows, D), dtype=torch.float32, device=dev)   # this rank's partial d_x, same numbering
        self.flags = symm.empty((64,), dtype=torch.int32, device=dev)
        self.flags2 = symm.empty((64,), dtype=torch.int32, device=dev)          # second barrier channel (exchange stream)
        self.stage = symm.empty((self.STAGE_BYTES,), dtype=torch.uint8, device=dev)  # slots of the one-shot all-reduces
        self.table.zero_(); self.partial.zero_(); self.flags.zero_(); self.flags2.zero_(); self.stage.zero_()
        self._h_table = symm.rendezvous(self.table, group)
        self._h_partial = symm.rendezvous(self.partial, group)
        self._h_flags = symm.rendezvous(self.flags, group)
        self._h_flags2 = symm.rendezvous(self.flags2, group)
        self._h_stage = symm.rendezvous(self.stage, group)
        self.table_ptrs, self.partial_ptrs, self.flag_ptrs, self.stage_ptrs = (
            int(h.buffer_ptrs_dev) for h in (self._h_table, self._h_partial, self._h_flags, self._h_stage))
        self.flag2_ptrs = int(self._h_flags2.buffer_ptrs_dev)
        self.hybrid = bool(getattr(part, 'hybrid', False))
        if self.hybrid:
            # partial aggregates [2, rows_r, D] and upstream gradient planes [3, rows_r, D] of every rank, rows_r = its own
            # rows + ITS remote rows (plane stride differs per rank: per-plane peer pointer tables)
            self.agg_buf = symm.empty((2 * rows * D,), dtype=torch.float32, device=dev)
            self.g3_buf = symm.empty((3 * rows * D,), dtype=torch.float32, device=dev)
            self.agg_buf.zero_(); self.g3_buf.zero_()
            self._h_agg = symm.rendezvous(self.agg_buf, group)
            self._h_g3 = symm.rendezvous(self.g3_buf, group)
            rows_r = [B + n for n in part.n_remote_all]
            self.rows_mine = rows_r[part.rank]
            mk = lambda h_, plane: torch.tensor([int(p) + plane * rows_r[r] * D * 4 for r, p in enumerate(h_.buffer_ptrs)],   # noqa: E731
                                                dtype=torch.int64, device=dev)
            self.agg_plane_ptrs = [mk(self._h_agg, h) for h in (0, 1)]
            self.g3_plane_ptrs = [mk(self._h_g3, h) for h in (0, 1)]
            self.sparse_src, self.sparse_dst = part.sparse_src, part.sparse_dst
        self._slots, self._stage_used = {}, 0
        self.epoch = torch.zeros((1,), dtype=torch.int32, device=dev)
        self.epoch2 = torch.zeros((1,), dtype=torch.int32, device=dev)
        self.exchange_stream = torch.cuda.Stream(device=dev)     # halo pulls next to rank-local kernels of the main stream
        self.halo_order = getattr(part, 'halo_order', None)
        self.error = torch.zeros((1,), dtype=torch.int32, device=dev)
        self.halo_rows, self.peer_idx = part.halo_rows, part.peer_idx
        torch.cuda.synchronize(dev)
        dist.barrier(group=group)                               # every rank's buffers are zeroed before anyone pulls

    def barrier(self, channel=0):
        """Flag barrier on the current stream.  Barriers of ONE channel must be ordered by stream dependencies (they share an
        epoch counter); channel 1 belongs to the exchange stream's backward pulls, which run next to the main stream's
        one-shot all-reduces (channel 0)."""
        import ctypes
        from . import _lib
        flags, epoch = (self.flag_ptrs, self.epoch) if channel == 0 else (self.flag2_ptrs, self.epoch2)
        _lib.call('kgc_p2p_barrier', ctypes.c_void_p(flags), self.rank, self.world, _lib.ptr(epoch),
                  _lib.ptr(self.error), _lib.stream())

    def gather(self, x_local, fence=False):
        """x rows of this rank -> its block of the table; barrier; pull the remote rows this rank's edges read.
        ``fence``: barrier BEFORE the rows are overwritten as well - needed when nothing else synchronises the ranks between
        two gathers (evaluation-mode forwards: no BatchNorm all-reduce, no backward), so that no peer is still pulling the
        previous contents."""
        import ctypes
        from . import _lib
        n = x_local.shape[0]
        if fence:
            self.barrier()
        self.table[:n].copy_(x_local)
        self.barrier()
        _lib.call('kgc_p2p_halo_gather', ctypes.c_void_p(self.table_ptrs), self.rank, _lib.ptr(self.halo_rows),
                  _lib.ptr(self.halo_order), self.halo_rows.numel(), self.block, self.D, _lib.stream())
        return self.table

    def reduce(self, addend, n_rows, out=None, channel=0):
        """barrier; d_x of this rank's rows = addend + the partials of the ranks that touched them, in rank order."""
        import ctypes
        from . import _lib
        if out is None:
            out = torch.empty((n_rows, self.D), dtype=torch.float32, device=self.table.device)
        self.barrier(channel)
        _lib.call('kgc_p2p_halo_reduce', ctypes.c_void_p(self.partial_ptrs), self.world, _lib.ptr(self.peer_idx), None,
                  n_rows, _lib.ptr(addend), _lib.ptr(out), self.D, _lib.stream())
        return out

    # ---- hybrid cut: partial aggregates to their owners (forward), upstream gradient rows to the ranks that need them (backward)
    def g3_planes(self):
        """This rank's [3, rows, D] upstream-gradient planes in symmetric memory (rows = own + remote rows; peers read the
        own rows of planes 0 / 1).  Rows of plane 2 behind the real rows are zero and stay zero (the self-loop addend)."""
        return self.g3_buf[:3 * self.rows_mine * self.D].view(3, self.rows_mine, self.D)

    def _reduce_sparse(self, ptr_table, sparse, local, channel):
        """Remote rows of ``local`` [rows, D] -> this rank's symmetric copy (what the owners read); barrier; own rows that
        other ranks hold partial rows for += those rows, in rank order, in place."""
        import ctypes
        from . import _lib
        rows, idx = sparse
        if rows.numel():
            _lib.call('kgc_p2p_halo_reduce', ctypes.c_void_p(ptr_table), self.world, _lib.ptr(idx), _lib.ptr(rows), rows.numel(),
                      _lib.ptr(local), _lib.ptr(local), self.D, _lib.stream())

    def reduce_agg(self, agg):
        """Forward of the hybrid cut: agg [2, rows, D] (rank-local).  The partial aggregates of the remote destinations go
        to symmetric memory, the ranks meet, and every owner adds the partial rows the others hold for its rows."""
        B, R, D = self.block, self.rows_mine, self.D
        sym = self.agg_buf[:2 * R * D].view(2, R, D)
        sym[:, B:].copy_(agg[:, B:])
        self.barrier()
        for h in (0, 1):
            self._reduce_sparse(self.agg_plane_ptrs[h].data_ptr(), self.sparse_dst, agg[h], 0)

    def reduce_dx(self, d_x_full, channel=1):
        """Backward of the hybrid cut: d_x_full [rows, D] (rank-local; own rows complete but for the other ranks' partial rows)."""
        B, R = self.block, self.rows_mine
        self.partial[B:R].copy_(d_x_full[B:R])
        self.barrier(channel)
        self._reduce_sparse(self.partial_ptrs, self.sparse_src, d_x_full, channel)

    def gather_g(self):
        """barrier; rows of the remote destinations of planes 0 / 1 of g3 <- their owners' rows."""
        import ctypes
        from . import _lib
        self.barrier()
        for h in (0, 1):
            _lib.call('kgc_p2p_halo_gather', ctypes.c_void_p(self.g3_plane_ptrs[h].data_ptr()), self.rank, _lib.ptr(self.halo_rows),
                      _lib.ptr(self.halo_order), self.halo_rows.numel(), self.block, self.D, _lib.stream())

    def all_reduce(self, t, tag):
        """In-place sum of a small contiguous fp32 / fp64 tensor over the ranks (one kernel: stage, flag barrier, add in rank
        order).  ``tag`` names the call site: every site owns a staging slot, so a slot is rewritten only a full step later.
        Returns False (caller falls back to NCCL) when the tensor does not fit the kernel's constraints."""
        import ctypes
        from . import _lib
        nbytes = t.numel() * t.element_size()
        if t.dtype not in (torch.float32, torch.float64) or not t.is_contiguous() or nbytes % 16 or t.data_ptr() % 16 \
                or nbytes == 0 or nbytes > (1 << 20):
            return False
        key = (tag, nbytes, t.dtype)
        off = self._slots.get(key)
        if off is None:
            off = self._stage_used
            if off + nbytes > self.STAGE_BYTES:
                return False
            self._slots[key] = off
            self._stage_used = (off + nbytes + 255) // 256 * 256
        _lib.call('kgc_p2p_allreduce', ctypes.c_void_p(self.stage_ptrs), off, ctypes.c_void_p(self.flag_ptrs), self.rank,
                  self.world, _lib.ptr(self.epoch), _lib.ptr(self.error), _lib.ptr(t), _lib.ptr(t), nbytes,
                  1 if t.dtype == torch.float64 else 0, _lib.stream())
        return True

    def check(self):
        """The barrier has no data-path time-out (ranks may skew freely); its ~2-minute watchdog for a vanished peer sets
        the error word and traps, so a failure surfaces as a CUDA error on the next synchronising call.  This reads the
        error word for callers that want the explicit message."""
        if int(self.error) != 0:
            raise RuntimeError('kgc_p2p_barrier: a peer rank did not arrive within the watchdog period')
