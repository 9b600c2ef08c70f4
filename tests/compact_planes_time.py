"""Timing script (not a test): the single-GPU layer with its sparse in half compacted (plan.compact_halves) next to the
dense path, on bench.py's seeded synthetic graphs.

    python tests/compact_planes_time.py [--reps 10] [--steps 10] [--workloads wikidata5m,wn18rr,fb15k237]

Reports, with the GPU name and power limit read in the same run:
  - at the Wikidata5M shape (N = 4,594,485, D = 100 -> 200), kernel times (CUDA events, median of --reps, L2 flushed
    before every launch) of each piece the compaction changes, dense and compact launched alternately in the same loop:
    the in-plane prefill memset, K4b forward, kgc_tail_fwd, kgc_tail_bwd_apply, K4b backward, K4c and the row copies;
  - the whole layer step (forward + backward, CUDA graph replays, L2 flushed between them) per workload, dense and
    compact alternately (dense / compact / dense / compact).  At the WN18RR and FB15k-237 shapes the compaction is
    forced past its plane-size rule, which is what sets that rule.
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

from sampled_loss_time import gpu_info, k          # noqa: E402  (puts the repository and oracle/ on sys.path)
from bench import D_IN, D_OUT, Flusher, LayerCase, oracle, synth_rows      # noqa: E402

conv_mod = k.conv


def timed(pairs, reps, flush):
    """pairs: [(name, fn)], launched in turn every repetition; -> {name: median ms}."""
    for _, fn in pairs:
        fn()
    torch.cuda.synchronize()
    ts = {name: [] for name, _ in pairs}
    for _ in range(reps):
        for name, fn in pairs:
            flush()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts[name].append(a.elapsed_time(b))
    return {name: {'ms': round(float(np.median(v)), 4), 'ms_min': round(float(min(v)), 4), 'ms_max': round(float(max(v)), 4)}
            for name, v in ts.items()}


def kernel_times(case, reps, flush):
    L, p, st = k._lib, k._lib.ptr, k._lib.stream
    N, D, Do, dev = case.N, D_IN, D_OUT, case.dev
    plan = k.get_plan(case.ei, case.et, N, 2 * case.R + 1)
    n_c, rows, slot = plan.n_c[0], plan.rows[0], plan.slot[0]
    ids = torch.arange(N, dtype=torch.int64, device=dev)
    x = case.x.detach()
    agg = synth_rows(torch.arange(2 * N, dtype=torch.int64, device=dev), D, 0.1, 31).view(2, N, D)
    w = [synth_rows(torch.arange(D, dtype=torch.int64, device=dev) + 1000 * i, Do, 0.1, 32) for i in range(3)]
    wt = [t.t().contiguous() for t in w]
    pf = [conv_mod._pack_b(t) for t in w]                 # [D, Dout] operands of the forward
    pb = [conv_mod._pack_b(t) for t in wt]                # [Dout, D] operands of the backward
    res3 = torch.empty((3, N, Do), device=dev)
    agg_c = torch.empty((n_c, D), device=dev)
    res_c = torch.empty((n_c, Do), device=dev)
    pre = torch.empty((N, Do), device=dev)
    nb = int(L.lib().kgc_tail_num_blocks(N))
    partials = torch.empty((nb, 2, Do), dtype=torch.float64, device=dev)
    keep = torch.empty((N, int(L.lib().kgc_keep_pitch())), dtype=torch.uint8, device=dev)
    seed = torch.tensor([12345], dtype=torch.int64, device=dev)
    g_ent = case.g_ent
    stats = torch.ones((3, Do), device=dev)
    gamma, beta = torch.ones(Do, device=dev), torch.zeros(Do, device=dev)
    sums = torch.zeros((2, Do), dtype=torch.float64, device=dev)
    d_out = torch.empty((N, Do), device=dev)
    d_res2 = torch.empty((2, N, Do), device=dev)
    d_res_c = torch.empty((n_c, Do), device=dev)
    g3 = torch.empty((3, N, D), device=dev)
    g3_c = torch.empty((n_c, D), device=dev)
    dw = torch.empty((3, D, Do), device=dev)
    scale = 1.0 / 0.9
    del ids

    def tail_fwd(rows_on):
        if rows_on:
            L.call('kgc_tail_fwd_rows', p(res3), p(slot), p(res_c), None, None, None, None, p(seed), 0.1, scale, None, N, Do,
                   p(pre), p(partials), p(keep), st())
        else:
            L.call('kgc_tail_fwd', p(res3), None, None, p(seed), 0.1, scale, None, N, Do, p(pre), p(partials), p(keep), st())

    def tail_bwd(rows_on):
        L.call('kgc_tail_bwd_apply_rows', p(g_ent), p(pre), p(stats), p(gamma), p(beta), p(sums), 1, N, N, Do, p(d_out), p(keep),
               scale, p(d_res_c if rows_on else d_res2[0]), p(slot) if rows_on else None, p(d_res2[1]), None, None, 1.0, st())

    out = {'N': N, 'n_c_in': n_c, 'D': D, 'Dout': Do}
    out['prefill_memset_in_plane'] = timed([('dense', lambda: agg[0].zero_())], reps, flush)['dense']
    out['k4b_fwd'] = timed([
        ('dense_batch3', lambda: conv_mod.gemm_nt_batch([agg[0], agg[1], x], pf, [res3[0], res3[1], res3[2]])),
        ('compact_gather', lambda: conv_mod.rows_copy(agg[0], rows, agg_c, None, n_c)),
        ('compact_gemm_nc', lambda: conv_mod.gemm_nt(agg_c, None, res_c, packed=pf[0])),
        ('compact_batch2', lambda: conv_mod.gemm_nt_batch([agg[1], x], pf[1:], [res3[1], res3[2]]))], reps, flush)
    out['tail_fwd'] = timed([('dense', lambda: tail_fwd(False)), ('compact', lambda: tail_fwd(True))], reps, flush)
    out['tail_bwd_apply'] = timed([('dense', lambda: tail_bwd(False)), ('compact', lambda: tail_bwd(True))], reps, flush)
    out['k4b_bwd'] = timed([
        ('dense_batch3', lambda: conv_mod.gemm_nt_batch([d_res2[0], d_res2[1], d_out], pb, [g3[0], g3[1], g3[2]])),
        ('compact_gemm_nc', lambda: conv_mod.gemm_nt(d_res_c, None, g3_c, packed=pb[0])),
        ('compact_scatter', lambda: conv_mod.rows_copy(g3_c, None, g3[0], rows, n_c)),
        ('compact_batch2', lambda: conv_mod.gemm_nt_batch([d_res2[1], d_out], pb[1:], [g3[1], g3[2]]))], reps, flush)
    out['k4c'] = timed([
        ('dense_batch3', lambda: conv_mod.gemm_tn_batch([agg[0], agg[1], x], [d_res2[0], d_res2[1], d_out], [dw[0], dw[1], dw[2]])),
        ('compact_rows', lambda: conv_mod.gemm_tn_batch_rows([agg_c, agg[1], x], [d_res_c, d_res2[1], d_out], [dw[0], dw[1], dw[2]],
                                                             [n_c, N, N]))], reps, flush)
    for key in ('k4b_fwd', 'k4b_bwd'):
        v = out[key]
        v['compact_total_ms'] = round(sum(t['ms'] for n_, t in v.items() if n_.startswith('compact')), 4)
    return out


def step_times(case, steps, warm, flush, force):
    """Graph-replayed layer steps, dense and compact alternately; ``force``: compact past the plane-size rule."""
    res = {}
    graphs = {}
    saved = (k.plan.COMPACT_MIN_PLANE_BYTES, k.plan.COMPACT_MAX_OCCUPANCY)
    for mode in ('dense', 'compact'):
        k.plan.COMPACT_MIN_PLANE_BYTES, k.plan.COMPACT_MAX_OCCUPANCY = \
            (saved[0], -1.0) if mode == 'dense' else ((-1 if force else saved[0]), saved[1])
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    case.step()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            plan = k.get_plan(case.ei, case.et, case.N, 2 * case.R + 1)
            comp = plan.compact_halves(4 * D_OUT)
            k._lib.LAUNCHES = 0
            case.step()
            launches = k._lib.LAUNCHES
            g = torch.cuda.CUDAGraph()
            for t in case.leaves:
                t.grad = None
            with torch.cuda.graph(g):
                case.step()
            graphs[mode] = g
            res[mode] = {'compacted': comp, 'n_c': plan.n_c, 'launches_per_step': launches, 'ms': []}
        finally:
            k.plan.COMPACT_MIN_PLANE_BYTES, k.plan.COMPACT_MAX_OCCUPANCY = saved
    for _ in range(2):
        for mode in ('dense', 'compact'):
            g = graphs[mode]
            for _ in range(warm):
                g.replay()
            torch.cuda.synchronize()
            ts = []
            for _ in range(steps):
                flush()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                g.replay()
                b.record()
                torch.cuda.synchronize()
                ts.append(a.elapsed_time(b))
            res[mode]['ms'].append(round(float(np.mean(ts)), 4))
    del graphs
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--workloads', default='wikidata5m,wn18rr,fb15k237')
    ap.add_argument('--no-kernels', action='store_true')
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'needs a GPU'
    print(gpu_info(), flush=True)
    orc = oracle()
    dev = torch.device('cuda')
    flush = Flusher(dev)
    for wl in args.workloads.split(','):
        case = LayerCase(k, orc, wl, dev)
        if wl == 'wikidata5m' and not args.no_kernels:
            print(json.dumps({'workload': wl, 'kernels': kernel_times(case, args.reps, flush)}), flush=True)
            torch.cuda.empty_cache()
        st = step_times(case, args.steps, args.warmup, flush, force=(wl != 'wikidata5m'))
        print(json.dumps({'workload': wl, 'layer_step': st, 'compaction_forced': wl != 'wikidata5m'}), flush=True)
        del case
        k.plan._PLAN_CACHE.clear()
        torch.cuda.empty_cache()


if __name__ == '__main__':
    main()
