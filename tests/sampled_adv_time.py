"""Timing script (not a test): self-adversarial negative sampling next to the plain sampled objective at the Wikidata5M
shape of bench.py (N = 4,594,485 entities, d = 200, the same seeded synthetic graph as tests/sampled_loss_time.py).

    python tests/sampled_adv_time.py [--reps 10] [--steps 10] [--B 4096] [--k 256] [--alpha 1.0]

Reports, with the GPU name and power limit read in the same run:
  - kernel times (CUDA events, median of --reps) of kgc_sampled_bce_fwd and kgc_sampled_adv_fwd at B = 4,096, k = 256
    negatives + 1 positive, D = 200, the two launched alternately in the same loop, each next to its algorithmic bytes
    over 6,539 GB/s (the copy rate measured on a B200, DESIGN section 4); the 3.7 GB entity table exceeds L2;
  - the whole GraphedTrainStep(negatives=k) step (host ids in, loss out) at B = 4,096 without and with
    adversarial_temperature=alpha, run plain / adversarial / plain / adversarial to show the spread.
"""
import argparse
import json
import os
import sys

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
import numpy as np       # noqa: E402
import torch             # noqa: E402

from sampled_loss_time import COPY_GBS, gpu_info, k          # noqa: E402  (puts the repository and oracle/ on sys.path)
from bench import WORKLOADS, _mix32, params_ns, synth_rows, synthetic_query_set         # noqa: E402


def kernel_times(N, B, C, D, reps, alpha):
    L, p, dev = k._lib, k._lib.ptr, torch.device('cuda')
    rows = torch.arange(N, dtype=torch.int64, device=dev)
    ent = synth_rows(rows, D, 1.0 / D ** 0.5, 41)
    bias = synth_rows(rows, 1, 0.1, 42).view(-1)
    x = synth_rows(torch.arange(B, dtype=torch.int64, device=dev), D, 1.0, 43)
    cand = (_mix32(torch.arange(B * C, dtype=torch.int64, device=dev) + 977) % N).to(torch.int32).view(B, C)
    g = torch.empty((B, C), device=dev)
    d_x = torch.empty((B, D), device=dev)
    counts = torch.empty((2,), dtype=torch.int32, device=dev)
    partial = torch.empty((2 * int(L.lib().kgc_sampled_bce_fwd_blocks(B)),), dtype=torch.float64, device=dev)
    loss = torch.empty((1,), device=dev)

    def plain():
        L.call('kgc_sampled_bce_fwd', p(x), B, D, p(ent), N, D, p(bias), p(cand), C, 1, 1.0, 0.0, p(g), p(d_x), p(counts),
               p(partial), p(loss), L.stream())

    def adv():
        L.call('kgc_sampled_adv_fwd', p(x), B, D, p(ent), N, D, p(bias), p(cand), C, 1, 1.0, 0.0, alpha, p(g), p(d_x),
               p(counts), p(partial), p(loss), L.stream())
    slots = B * C
    # every slot reads its id, entity row and bias and writes g; x read and d_x written once.  The adversarial pass also
    # re-reads each slot's id and parked logit once (8 bytes a slot, from L2 in practice); they are not counted.
    nbytes = slots * (4 + 4 * D + 4 + 4) + 2 * B * D * 4
    fns = (('kgc_sampled_bce_fwd', plain), ('kgc_sampled_adv_fwd', adv))
    for _, fn in fns:
        fn()
    torch.cuda.synchronize()
    ts = {name: [] for name, _ in fns}
    for _ in range(reps):
        for name, fn in fns:                          # alternated: both see the same clocks and neighbours
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts[name].append(a.elapsed_time(b))
    out = {}
    for name, _ in fns:
        ms = float(np.median(ts[name]))
        out[name] = {'ms': round(ms, 4), 'ms_min': round(float(min(ts[name])), 4), 'ms_max': round(float(max(ts[name])), 4),
                     'bytes': nbytes, 'GB/s': round(nbytes / ms / 1e6, 1), 'of_copy_rate': round(nbytes / COPY_GBS / 1e6 / ms, 3)}
    del ent
    torch.cuda.empty_cache()
    return out


def step_times(B, k_neg, alpha, steps, warm):
    import mgcn_oracle as orc
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
    res = []
    for temp in (None, alpha, None, alpha):
        rng = np.random.default_rng(0)
        torch.manual_seed(0)
        with torch.device(dev):
            model = k.MGCN(N, R, E, prm)
        model.train()
        opt = k.ClipAdam(model.parameters(), lr=1e-3, max_norm=1.0)
        gen = torch.Generator(device=dev).manual_seed(1)
        step = k.GraphedTrainStep(model, opt, graph, ds, B, negatives=k_neg, generator=gen, adversarial_temperature=temp)
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
        row = {'mode': 'sampled' if temp is None else 'sampled_adv', 'adversarial_temperature': temp, 'B': B, 'k': k_neg,
               'ms_per_step': round(m, 2), 'ms_min': round(float(min(ms)), 2), 'queries_per_s': round(B / m * 1e3, 1),
               'steps': len(ms), 'loss_first_last': [round(losses[0], 6), round(losses[-1], 6)]}
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
    ap.add_argument('--B', type=int, default=4096)
    ap.add_argument('--k', type=int, default=256)
    ap.add_argument('--alpha', type=float, default=1.0)
    ap.add_argument('--no-steps', action='store_true', help='kernel times only')
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'needs a GPU'
    print(gpu_info(), flush=True)
    N = WORKLOADS['wikidata5m'][0]
    kt = kernel_times(N, args.B, args.k + 1, 200, args.reps, args.alpha)
    print(json.dumps({'kernels': kt, 'B': args.B, 'C': args.k + 1, 'D': 200, 'N': N, 'alpha': args.alpha}), flush=True)
    if not args.no_steps:
        step_times(args.B, args.k, args.alpha, args.steps, args.warmup)


if __name__ == '__main__':
    main()
