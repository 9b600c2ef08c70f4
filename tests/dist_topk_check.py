"""Multi-GPU check of entity-sharded top-k, launched by tests/test_gpu_topk_shard.py as
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port P tests/dist_topk_check.py
One process per GPU (NCCL).  Every rank compares ``topk(..., group=WORLD)`` with the unsharded call (bit for bit, both
precisions): range shards of an N that is not a multiple of the rank count, shards with the last rank owning no rows,
and ``MGCN.topk`` with a group on the stored Toy model.  Overlapping ranges and ranks that disagree on B raise
ValueError on every rank."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'oracle'))
sys.path.insert(0, HERE)
import kgc_gcn_b200 as k                                                      # noqa: E402
from test_gpu_topk import _toy_loader, exclusion_lists, int_operands, random_case   # noqa: E402


def same(a, b, what):
    for key in ('count', 'ids', 'scores'):
        assert a[key].dtype == b[key].dtype and torch.equal(a[key], b[key]), (what, key)


def main():
    rank, world = int(os.environ['RANK']), int(os.environ['WORLD_SIZE'])
    dev = torch.device('cuda', int(os.environ.get('LOCAL_RANK', rank)))
    torch.cuda.set_device(dev)
    dist.init_process_group('nccl', device_id=dev)
    W = dist.group.WORLD
    cu = lambda a: None if a is None else torch.from_numpy(a).to(dev)          # noqa: E731
    B, N, d = 300, 5000 * world + 3, 200                                      # N NOT a multiple of the rank count
    per = -(-N // world)
    even = [(min(r * per, N), min((r + 1) * per, N)) for r in range(world)]
    # the last rank owns no rows; the others split N unevenly
    cut = [0] + [(N * (r + 1)) // (world - 1) + (7 if r + 1 < world - 1 else 0) for r in range(world - 1)]
    last_empty = [(cut[r], cut[r + 1]) for r in range(world - 1)] + [(N, N)]
    layouts = [('even', even)] + ([('last rank empty', last_empty)] if world > 1 else [])
    cases = 0
    xi, ti, bi = int_operands(B, N, d, seed=5)
    xf, tf, bf, pf, jf = random_case(B, N, d, seed=7)
    inputs = [('int', xi, ti, bi, {m: exclusion_lists(B, N, m, seed=6) for m in ('none', 'random', 'few')}),
              ('float', xf, tf, bf, {'random': (pf, jf)})]
    for name, xq, tab, bias, filters in inputs:
        xq, tab, bias = xq.to(dev), tab.to(dev), bias.to(dev)
        table = k.EntityTable(tab, bias)
        for mode, (ptr, idx) in filters.items():
            for kk in (1, 10, 17, 32):
                for precision in ('bf16', 'fp32'):
                    whole = k.topk(xq, tab, bias, kk, cu(ptr), cu(idx), table=table if precision == 'bf16' else None,
                                   precision=precision)
                    for layout, spans in layouts:
                        lo, hi = spans[rank]
                        shard = k.EntityTable(tab[lo:hi], bias[lo:hi]) if precision == 'bf16' and hi > lo else None
                        got = k.topk(xq, tab[lo:hi], bias[lo:hi], kk, cu(ptr), cu(idx), table=shard, precision=precision,
                                     n_offset=lo, group=W)
                        same(got, whole, (name, mode, kk, precision, layout, rank))
                        cases += 1

    # argument checks that need a group: every rank raises, none hangs
    xq, tab, bias = (t.to(dev) for t in int_operands(8, 600, d, seed=9))
    for bad in ('overlap', 'B') if world > 1 else ():
        try:
            if bad == 'overlap':                                           # every rank claims all rows
                k.topk(xq, tab, bias, 5, n_offset=0 if rank == 0 else 1, group=W)
            else:
                k.topk(xq[:8 - (rank % 2)], tab[rank * 300:(rank + 1) * 300], bias[rank * 300:(rank + 1) * 300], 5,
                       n_offset=rank * 300, group=W)
            raise AssertionError('no ValueError for ' + bad)
        except ValueError:
            pass

    # MGCN.topk with a group on the stored Toy model (its reference widths run some torch library ops)
    os.environ['KGC_STRICT'] = '0'
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    dl, prm = _toy_loader(k, os.path.join(HERE, 'golden'))
    dl.graph.to(dev)
    z = np.load(os.path.join(HERE, 'golden', 'toy_model.npz'))
    m = k.MGCN(dl.num_entity, dl.num_relation, dl.num_edge, prm)
    m.load_state_dict({kk[3:]: torch.from_numpy(z[kk]) for kk in z.files if kk.startswith('sd.')})
    m = m.to(dev).eval()
    trip = np.concatenate([dl._get_dataset(s, prm).triples for s in ('valid_tail', 'valid_head', 'test_tail')])
    src, rel = torch.from_numpy(trip[:, 0]).to(dev), torch.from_numpy(trip[:, 1]).to(dev)
    excl = tuple(t.to(dev) for t in dl.known_objects(src.cpu(), rel.cpu()))
    ne = dl.num_entity
    lo, hi = min(rank * -(-ne // world), ne), min((rank + 1) * -(-ne // world), ne)
    assert hi > lo
    with torch.no_grad():
        all_ent, _ = m.encode(dl.graph)
        shard = k.EntityTable(all_ent[lo:hi], m.conv2.bias[lo:hi])
        for precision in ('bf16', 'fp32'):
            for exclude in (None, excl):
                what = ('toy', precision, exclude is None)
                whole = m.topk(src, rel, dl.graph, k=10, exclude=exclude, precision=precision)
                # the model's own even split, then this rank's table shard (fp32: the same rows of the fp32 encoding)
                same(m.topk(src, rel, dl.graph, k=10, exclude=exclude, precision=precision, group=W), whole, what)
                same(m.topk(src, rel, dl.graph, k=10, exclude=exclude, precision=precision, table=shard, n_offset=lo,
                            group=W), whole, what + ('table',))
                cases += 2
    dist.barrier()
    if rank == 0:
        print('DIST_TOPK_OK', {'world': world, 'N': N, 'cases': cases})
    dist.destroy_process_group()


if __name__ == '__main__':
    main()
