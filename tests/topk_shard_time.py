"""Debug aid (not a test): CUDA-event timing of entity-sharded filtered top-k at the Wikidata5M shape of bench.py's aux
leg - B = 65,536 queries, N = 4,594,485 entities, d = 200, the same seeded inputs, 4 exclusions per query - with the
entity table range-sharded as bench.py's aux_filtered_rank shards it (shard r of W: rows r * ceil(N / W) ...).

One process per GPU, W = the number of processes:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node W tests/topk_shard_time.py [--reps 5]

Every rank runs topk(..., n_offset=lo, group=WORLD), also at W = 1 (a one-rank gather and merge).  For k = 10 and 32,
rank 0 prints, with the GPU names and power limits:
  - sweep_ms: kgc_score_topk on this rank's shard (its own score floor), median of --reps, max over ranks;
  - gather_merge_ms: all-gather of the [B, k] results + kgc_topk_merge, median, max over ranks;
  - call_ms / queries_per_s: the whole topk(..., group) call (packing, checks, sweep, gather, merge), max over ranks;
  - rank_ms: kgc_score_rank on the same shard and queries, for reference;
and asserts that on the first 2,048 queries the sharded call equals the unsharded one on the whole table, bit for bit.

One GPU, the shards of every W in --shards swept one after another (no process group):

    python tests/topk_shard_time.py --shards 1,2,4,8 [--reps 5]

A shard's sweep does not communicate, so the largest of its W shard times is the per-rank sweep time of W GPUs (up to
the spread between cards).  It reports that, kgc_score_rank on the same shard, kgc_topk_merge over W lists, and the
local topk(..., n_offset=lo) call of the largest shard; the all-gather between GPUs is not part of it.  The merged result
of every W must equal the W = 1 sweep on all 65,536 queries, bit for bit (asserted).
"""
import argparse
import json
import os
import subprocess
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np                  # noqa: E402
import torch                        # noqa: E402
import torch.distributed as dist    # noqa: E402

import kgc_gcn_b200 as k                 # noqa: E402
from bench import _mix32, synth_rows     # noqa: E402


def gpu_info():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i',
                          str(torch.cuda.current_device())], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return out.stdout.strip()


def timed(fn, reps, sync_ranks=True):
    """Median CUDA-event time of fn over reps, all ranks starting together; max over ranks."""
    ms = []
    for _ in range(reps):
        if sync_ranks:
            dist.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    t = torch.tensor([float(np.median(ms))], dtype=torch.float64, device='cuda')
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t[0])


def inputs(dev):
    B, N, d = 65536, 4594485, 200
    qid = torch.arange(B, dtype=torch.int64, device=dev)
    xq = synth_rows(qid, d, 1.7, 31).abs_()
    fptr = torch.arange(0, 4 * B + 1, 4, device=dev, dtype=torch.int64)
    fidx = (_mix32(torch.arange(4 * B, dtype=torch.int64, device=dev) + 4099) % N).view(B, 4).sort(1).values.reshape(-1).to(torch.int32)
    return B, N, d, xq, fptr, fidx


def shard_table(lo, hi, d, dev):
    rows = torch.arange(lo, hi, dtype=torch.int64, device=dev)
    return k.EntityTable(synth_rows(rows, d, 1.0, 32), synth_rows(rows, 1, 0.1, 33).view(-1))


def event_ms(fn, reps):
    """Median CUDA-event time of fn over reps (after one untimed call)."""
    fn()
    ms = []
    for _ in range(reps):
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return float(np.median(ms))


def one_gpu(args):
    """The shards of every W in --shards, swept one after another on this GPU."""
    L = k._lib
    dev = torch.device('cuda')
    B, N, d, xq, fptr, fidx = inputs(dev)
    q16 = k.pack_queries(xq)
    res = {'gpu': gpu_info(), 'B': B, 'N': N, 'd': d, 'exclusions_per_query': 4, 'reps': args.reps}
    ref = {}
    for W in [int(w) for w in args.shards.split(',')]:
        per = -(-N // W)
        shards = [(min(r * per, N), min((r + 1) * per, N)) for r in range(W)]
        t = {'rank_ms': [], 'k10': [], 'k32': [], 'call_k10': []}
        lists = {10: ([], []), 32: ([], [])}
        for lo, hi in shards:
            table = shard_table(lo, hi, d, dev)
            lidx = (fidx.long() - lo).clamp_(-1, hi - lo).to(torch.int32)
            thr = torch.zeros(B, device=dev)
            gt = torch.zeros(B, dtype=torch.int32, device=dev)
            t['rank_ms'].append(event_ms(lambda: L.call('kgc_score_rank', L.ptr(q16), L.ptr(table.data), B, table.n,
                                                        table.kpad, L.ptr(thr), L.ptr(gt), None, L.stream()), args.reps))
            for kk in (10, 32):
                s = torch.empty((B, kk), device=dev)
                i = torch.empty((B, kk), dtype=torch.int32, device=dev)
                c = torch.empty((B,), dtype=torch.int32, device=dev)
                wsb = int(L.lib().kgc_score_topk_workspace_bytes(B, table.n, table.kpad, kk))
                ws = torch.empty((wsb,), dtype=torch.uint8, device=dev)
                t['k{}'.format(kk)].append(event_ms(lambda: L.call(
                    'kgc_score_topk', L.ptr(q16), L.ptr(table.data), B, table.n, table.kpad, L.ptr(fptr), L.ptr(lidx), kk,
                    L.ptr(s), L.ptr(i), L.ptr(c), L.ptr(ws), wsb, L.stream()), args.reps))
                del ws
                lists[kk][0].append(s)
                lists[kk][1].append(torch.where(i >= 0, i + lo, i))
            t['call_k10'].append(event_ms(lambda: k.topk(xq, None, None, 10, fptr, fidx, table=table, n_offset=lo),
                                          args.reps))
            del table
            torch.cuda.empty_cache()
        e = {'rows_per_shard': per, 'rank_ms': max(t['rank_ms']), 'shard_call_k10_ms': max(t['call_k10'])}
        for kk in (10, 32):
            S, I = torch.stack(lists[kk][0]), torch.stack(lists[kk][1])
            e['k{}'.format(kk)] = {'sweep_ms': max(t['k{}'.format(kk)]), 'sweep_ms_per_shard': t['k{}'.format(kk)],
                                   'merge_ms': event_ms(lambda: k.merge_topk(S, I), args.reps)}
            e['k{}'.format(kk)]['sweep_over_rank'] = e['k{}'.format(kk)]['sweep_ms'] / e['rank_ms']
            got = k.merge_topk(S, I)
            if W == 1:
                ref[kk] = got
            elif kk in ref:
                e['k{}'.format(kk)]['equals_unsharded_all_queries'] = all(torch.equal(got[key], ref[kk][key])
                                                                         for key in ('scores', 'ids', 'count'))
                assert e['k{}'.format(kk)]['equals_unsharded_all_queries'], (W, kk)
        res['W{}'.format(W)] = e
        print(json.dumps({'W': W, **e}), flush=True)
    for W in [int(w) for w in args.shards.split(',')]:
        for kk in (10, 32):
            if 'W1' in res:
                res['W{}'.format(W)]['k{}'.format(kk)]['speedup_vs_W1'] = \
                    res['W1']['k{}'.format(kk)]['sweep_ms'] / res['W{}'.format(W)]['k{}'.format(kk)]['sweep_ms']
    print(json.dumps(res), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--shards', default=None, help='one GPU, no process group: e.g. 1,2,4,8')
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'needs a GPU'
    if args.shards is not None:
        return one_gpu(args)
    rank, world = int(os.environ['RANK']), int(os.environ['WORLD_SIZE'])
    dev = torch.device('cuda', int(os.environ.get('LOCAL_RANK', rank)))
    torch.cuda.set_device(dev)
    dist.init_process_group('nccl', device_id=dev)
    W = dist.group.WORLD
    L = k._lib
    B, N, d, xq, fptr, fidx = inputs(dev)
    per = -(-N // world)
    lo, hi = min(rank * per, N), min((rank + 1) * per, N)
    table = shard_table(lo, hi, d, dev)
    q16 = k.pack_queries(xq)
    lidx = (fidx.long() - lo).clamp_(-1, hi - lo).to(torch.int32)         # this shard's exclusions, as topk passes them
    gpus = [None] * world
    dist.all_gather_object(gpus, gpu_info())
    res = {'gpus': gpus, 'world': world, 'B': B, 'N': N, 'd': d, 'rows_per_rank': per, 'exclusions_per_query': 4,
           'reps': args.reps}

    def rank_sweep():
        thr = torch.zeros(B, device=dev)
        gt = torch.zeros(B, dtype=torch.int32, device=dev)
        return lambda: L.call('kgc_score_rank', L.ptr(q16), L.ptr(table.data), B, table.n, table.kpad, L.ptr(thr),
                              L.ptr(gt), None, L.stream())
    rk = rank_sweep()
    rk()
    res['rank_ms'] = timed(rk, args.reps)
    for kk in (10, 32):
        s = torch.empty((B, kk), device=dev)
        i = torch.empty((B, kk), dtype=torch.int32, device=dev)
        c = torch.empty((B,), dtype=torch.int32, device=dev)
        wsb = int(L.lib().kgc_score_topk_workspace_bytes(B, table.n, table.kpad, kk))
        ws = torch.empty((wsb,), dtype=torch.uint8, device=dev)

        def sweep():
            L.call('kgc_score_topk', L.ptr(q16), L.ptr(table.data), B, table.n, table.kpad, L.ptr(fptr), L.ptr(lidx), kk,
                   L.ptr(s), L.ptr(i), L.ptr(c), L.ptr(ws), wsb, L.stream())
        sweep()
        gs = torch.empty((world * B, kk), device=dev)
        gi = torch.empty((world * B, kk), dtype=torch.int32, device=dev)

        def gather_merge():
            dist.all_gather_into_tensor(gs, s, group=W)
            dist.all_gather_into_tensor(gi, i, group=W)
            return k.merge_topk(gs.view(world, B, kk), gi.view(world, B, kk))
        gather_merge()

        def call():
            return k.topk(xq, None, None, kk, fptr, fidx, table=table, n_offset=lo, group=W)
        call()
        e = {'sweep_ms': timed(sweep, args.reps), 'gather_merge_ms': timed(gather_merge, args.reps),
             'call_ms': timed(call, args.reps)}
        e['queries_per_s'] = B / (e['call_ms'] * 1e-3)
        e['sweep_over_rank'] = e['sweep_ms'] / res['rank_ms']
        res['k{}'.format(kk)] = e
        del ws
        if rank == 0:
            print(json.dumps({'k': kk, **e}), flush=True)

    # sharded == unsharded on the first 2,048 queries: every rank builds the whole table once
    nq = 2048
    del q16
    torch.cuda.empty_cache()
    full = shard_table(0, N, d, dev)
    xs, fp, fi = xq[:nq].contiguous(), fptr[:nq + 1].contiguous(), fidx[:4 * nq].contiguous()
    ok = True
    for kk in (10, 32):
        one = k.topk(xs, None, None, kk, fp, fi, table=full)
        sh = k.topk(xs, None, None, kk, fp, fi, table=table, n_offset=lo, group=W)
        ok = ok and all(torch.equal(one[key], sh[key]) for key in ('scores', 'ids', 'count'))
    t = torch.tensor([1 if ok else 0], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    res['sharded_equals_unsharded_2048'] = bool(int(t[0]))
    if rank == 0:
        print(json.dumps(res), flush=True)
    assert res['sharded_equals_unsharded_2048'], 'sharded top-k differs from the unsharded call'
    dist.destroy_process_group()


if __name__ == '__main__':
    main()
