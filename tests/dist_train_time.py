"""Time the sharded training step (MGCN.shard + GraphedTrainStep(fused_loss=True)) at the Wikidata5M shape:
    python -m torch.distributed.run --nnodes=1 --nproc-per-node W tests/dist_train_time.py [--steps 20] [--warmup 3]
bench.py's seeded graph generator, B = 128, host query ids in and loss.item() out (the scope of bench.py's N = 1 e2e).
Every rank builds only its shard of the entity and edge tables (a pure function of row id and seed), so the full tables
are never materialised.  W = 1: the sharded step runs eagerly (peer memory, which the capture needs, takes two or more
ranks), next to the single-GPU GraphedTrainStep(fused_loss=True).  Prints one JSON line on rank 0: ms per step, peak
device memory per rank, the card and its power limit."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.distributed as dist
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'oracle'))
sys.dont_write_bytecode = True
import mgcn_oracle as orc          # noqa: E402
import kgc_gcn_b200 as k           # noqa: E402
import bench                       # noqa: E402


def template(N, R, E, prm):
    """An MGCN of N entities and 2E edges whose three big tables are zero-stride views (no memory): shard() copies only
    this rank's rows of them.  The small parameters get their usual random initialisation (torch.manual_seed first)."""
    m = k.MGCN(1, R, 1, prm)
    m.entity_embedding = nn.Parameter(torch.zeros((1, prm.gcn_in_dim)).expand(N, prm.gcn_in_dim))
    m.edge_embeddings = nn.Parameter(torch.zeros((1, prm.gcn_in_dim)).expand(2 * E, prm.gcn_in_dim))
    m.conv2.bias = nn.Parameter(torch.zeros((1,)).expand(N))
    return m


def timed(fn, batches, warm):
    ms, n = 0.0, 0
    for i, q in enumerate(batches):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn(q)
        b.record()
        torch.cuda.synchronize()
        if i >= warm:
            ms += a.elapsed_time(b)
            n += 1
    return ms / max(n, 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--workload', default='wikidata5m')
    args = ap.parse_args()
    rank, world = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1))
    dev = torch.device('cuda', int(os.environ.get('LOCAL_RANK', rank)))
    torch.cuda.set_device(dev)
    dist.init_process_group('nccl', device_id=dev)
    N, R, E, seed = bench.WORKLOADS[args.workload]
    B = bench.BATCH
    prm = bench.params_ns()
    tri = orc.synthetic_triples(N, R, E, seed)
    g = orc.build_graph(tri, N, R)
    ds = k.KBDataset(bench.synthetic_query_set(k, tri, R), N, prm, training=True)
    rng = np.random.default_rng(0)                                 # the same batches on every rank
    batches = [rng.choice(len(ds), B, replace=False) for _ in range(args.warmup + args.steps)]
    out = {'workload': args.workload + '_shape', 'n_gpus': world, 'batch': B, 'steps': args.steps, 'warmup': args.warmup}

    # ---- the single-GPU step of bench.py's N = 1 e2e, in the same run
    if world == 1:
        graph = k.GraphData(edge_index=torch.from_numpy(g['edge_index']), edge_attr=torch.from_numpy(g['edge_attr']))
        graph.entity = torch.from_numpy(g['entity'])
        graph.edge_norm = torch.from_numpy(g['edge_norm'])
        graph.num_nodes = N
        graph.to(dev)
        torch.manual_seed(0)
        with torch.device(dev):
            model = k.MGCN(N, R, E, prm)
        model.train()
        opt = k.ClipAdam(model.parameters(), lr=1e-3, max_norm=1.0)
        step = k.GraphedTrainStep(model, opt, graph, ds, B, fused_loss=True)
        torch.cuda.reset_peak_memory_stats(dev)
        out['single_gpu_graphed_ms'] = timed(lambda q: step(q).item(), batches, args.warmup)
        out['single_gpu_peak_gb'] = torch.cuda.max_memory_allocated(dev) / 1e9
        del model, opt, step, graph
        k.plan._PLAN_CACHE.clear()
        torch.cuda.empty_cache()

    # ---- the sharded model
    part = k.GraphPartition(g['edge_index'], g['edge_attr'][0], N, 2 * R + 1, world, rank, dev,
                            balance='hybrid' if world > 1 else 'edges', p2p='auto' if world > 1 else False)
    del g, tri
    torch.manual_seed(0)
    sh = template(N, R, E, prm).shard(part).train()
    with torch.no_grad():
        sh.entity_embedding.copy_(bench.synth_rows(part.owned_nodes, prm.gcn_in_dim, bench.xavier_bound(N, prm.gcn_in_dim), 11))
        sh.edge_embeddings.copy_(bench.synth_rows(part.owned_eids, prm.gcn_in_dim, bench.xavier_bound(2 * E, prm.gcn_in_dim), 12))
    opt = k.ClipAdam(sh.parameters(), lr=1e-3, max_norm=1.0, partition=part, sharded=sh.sharded_parameters())
    torch.cuda.reset_peak_memory_stats(dev)
    if world > 1:
        step = k.GraphedTrainStep(sh, opt, None, ds, B, fused_loss=True)
        ms = timed(lambda q: step(q).item(), batches, args.warmup)
        out['sharded_scope'] = 'GraphedTrainStep(fused_loss=True) on the sharded model (hybrid cut, peer memory): one graph replay per step'
    else:
        def eager(q):
            opt.zero_grad(set_to_none=True)
            loss = sh.loss_sparse(q, ds)
            loss.backward()
            opt.step()
            loss.item()
        out['sharded_scope'] = 'sharded model on one rank, eager loss_sparse / backward / ClipAdam.step (no graph capture without peer memory)'
        try:
            ms = timed(eager, batches, args.warmup)
        except Exception as exc:                                   # reported, not hidden: the line says what failed
            ms, out['sharded_error'] = None, repr(exc)[:300]
    peak = torch.tensor([torch.cuda.max_memory_allocated(dev) / 1e9], dtype=torch.float64, device=dev)
    peaks = [torch.zeros_like(peak) for _ in range(world)]
    dist.all_gather(peaks, peak)
    out['sharded_ms'] = ms
    out['peak_gb_per_rank'] = [round(float(p), 2) for p in peaks]
    if rank == 0:
        try:
            card = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader',
                                   '-i', str(dev.index)], stdout=subprocess.PIPE, text=True, timeout=30).stdout.strip()
        except (OSError, subprocess.TimeoutExpired):
            card = 'unknown'
        out['card'] = card
        print(json.dumps(out), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == '__main__':
    main()
