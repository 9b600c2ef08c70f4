"""Timing script (not a test): negative-sampled training at the Wikidata5M shape of bench.py (N = 4,594,485 entities,
822 relations, 20,614,279 triples, d = 200, the same seeded synthetic graph).

    python tests/sampled_loss_time.py [--reps 10] [--steps 10] [--batches 128,1024,4096] [--k 256]

Reports, with the GPU name and power limit read in the same run:
  - kernel times (CUDA events, median of --reps) of kgc_sampled_bce_fwd and kgc_sampled_bce_bwd_table at B = 4,096,
    k = 256 negatives + 1 positive, D = 200, each next to its algorithmic bytes over 6,539 GB/s (the copy rate measured
    on a B200, DESIGN section 4); the 3.7 GB entity table exceeds L2, so the gathered rows come from HBM;
  - the whole GraphedTrainStep(negatives=k) step (host ids in, loss out) at each batch size: ms/step, training
    queries/s and peak device memory, next to the fused 1-N step (GraphedTrainStep(fused_loss=True)) at B = 128.
"""
import argparse
import json
import os
import subprocess
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'oracle'))
import numpy as np       # noqa: E402
import torch             # noqa: E402

import kgc_gcn_b200 as k                                                                # noqa: E402
from bench import WORKLOADS, _mix32, params_ns, synth_rows, synthetic_query_set         # noqa: E402

COPY_GBS = 6539.0


def gpu_info():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv'],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return out.stdout.strip()


def median_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def kernel_times(N, B, C, D, reps):
    L, p, dev = k._lib, k._lib.ptr, torch.device('cuda')
    rows = torch.arange(N, dtype=torch.int64, device=dev)
    ent = synth_rows(rows, D, 1.0 / D ** 0.5, 41)
    bias = synth_rows(rows, 1, 0.1, 42).view(-1)
    x = synth_rows(torch.arange(B, dtype=torch.int64, device=dev), D, 1.0, 43)
    cand = (_mix32(torch.arange(B * C, dtype=torch.int64, device=dev) + 977) % N).to(torch.int32).view(B, C)
    g = torch.empty((B, C), device=dev)
    d_x = torch.empty((B, D), device=dev)
    count = torch.empty((1,), dtype=torch.int32, device=dev)
    partial = torch.empty((int(L.lib().kgc_sampled_bce_fwd_blocks(B)),), dtype=torch.float64, device=dev)
    loss = torch.empty((1,), device=dev)
    scale = torch.ones((1,), device=dev)
    d_ent = torch.empty((N, D), device=dev)
    d_bias = torch.empty((N,), device=dev)
    ws_bytes = int(L.lib().kgc_sampled_bce_bwd_table_workspace_bytes(B * C, N))
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)

    def fwd():
        L.call('kgc_sampled_bce_fwd', p(x), B, D, p(ent), N, D, p(bias), p(cand), C, 1, 1.0, 0.0, p(g), p(d_x), p(count),
               p(partial), p(loss), L.stream())

    def bwd():
        L.call('kgc_sampled_bce_bwd_table', p(x), B, D, p(cand), C, p(g), p(scale), N, p(d_ent), D, p(d_bias), p(ws), ws_bytes,
               L.stream())
    slots = B * C
    # forward: every slot reads its id, entity row and bias and writes g; x read and d_x written once
    fwd_bytes = slots * (4 + 4 * D + 4 + 4) + 2 * B * D * 4
    # table backward: the dense table and bias written once, every slot reads id, g and its query row
    bwd_bytes = N * (D + 1) * 4 + slots * (4 + 4 + 4 * D)
    out = {}
    for name, fn, nbytes in (('fwd', fwd, fwd_bytes), ('bwd_table', bwd, bwd_bytes)):
        ms = median_ms(fn, reps)
        out[name] = {'ms': round(ms, 4), 'bytes': nbytes, 'GB/s': round(nbytes / ms / 1e6, 1),
                     'copy_rate_ms': round(nbytes / COPY_GBS / 1e6, 4), 'of_copy_rate': round(nbytes / COPY_GBS / 1e6 / ms, 3)}
    del ent, d_ent, ws
    torch.cuda.empty_cache()
    return out


def step_times(orc, batches, k_neg, steps, warm):
    N, R, E, seed = WORKLOADS['wikidata5m']
    dev = torch.device('cuda')
    tri = orc.synthetic_triples(N, R, E, seed)
    g = orc.build_graph(tri, N, R)
    prm = params_ns()
    graph = k.GraphData(edge_index=torch.from_numpy(g['edge_index']), edge_attr=torch.from_numpy(g['edge_attr']))
    graph.entity = torch.from_numpy(g['entity'])
    graph.edge_norm = torch.from_numpy(g['edge_norm'])
    graph.num_nodes = N
    graph.to(dev)
    ds = k.KBDataset(synthetic_query_set(k, tri, R), N, prm, training=True)
    rng = np.random.default_rng(0)
    res = []
    for mode, B in [('fused_1n', 128)] + [('sampled', b) for b in batches]:
        torch.manual_seed(0)
        with torch.device(dev):
            model = k.MGCN(N, R, E, prm)
        model.train()
        opt = k.ClipAdam(model.parameters(), lr=1e-3, max_norm=1.0)
        gen = torch.Generator(device=dev).manual_seed(1)
        if mode == 'fused_1n':
            step = k.GraphedTrainStep(model, opt, graph, ds, B, fused_loss=True)
        else:
            step = k.GraphedTrainStep(model, opt, graph, ds, B, negatives=k_neg, generator=gen)
        torch.cuda.reset_peak_memory_stats()
        ms, losses = [], []
        for i in range(warm + steps):
            qid = rng.integers(0, len(ds), B)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            losses.append(float(step(qid).item()))
            b.record()
            torch.cuda.synchronize()
            if i >= warm:
                ms.append(a.elapsed_time(b))
        m = float(np.mean(ms))
        row = {'mode': mode, 'B': B, 'k': k_neg if mode == 'sampled' else None, 'ms_per_step': round(m, 2),
               'ms_min': round(float(min(ms)), 2), 'queries_per_s': round(B / m * 1e3, 1),
               'peak_mem_GB': round(torch.cuda.max_memory_allocated() / 1e9, 2), 'steps': len(ms),
               'loss_first_last': [round(losses[0], 6), round(losses[-1], 6)]}
        print(json.dumps(row), flush=True)
        res.append(row)
        del model, opt, step
        k.plan._PLAN_CACHE.clear()
        torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--batches', default='128,1024,4096')
    ap.add_argument('--k', type=int, default=256)
    ap.add_argument('--no-steps', action='store_true', help='kernel times only')
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'needs a GPU'
    print(gpu_info(), flush=True)
    import mgcn_oracle as orc
    N = WORKLOADS['wikidata5m'][0]
    kt = kernel_times(N, 4096, args.k + 1, 200, args.reps)
    print(json.dumps({'kernels': kt, 'B': 4096, 'C': args.k + 1, 'D': 200, 'N': N}), flush=True)
    if not args.no_steps:
        step_times(orc, [int(b) for b in args.batches.split(',')], args.k, args.steps, args.warmup)


if __name__ == '__main__':
    main()
