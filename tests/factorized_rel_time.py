"""Timing script (not a test): the single-GPU layer with the d_rel pass factorized by (object, type) group (plan.GroupedPlan)
next to the plain path, on bench.py's seeded synthetic graphs.

    python tests/factorized_rel_time.py [--reps 10] [--steps 10] [--workloads wikidata5m,wn18rr,fb15k237]

Reports, with the GPU name and power limit read in the same run:
  - at the Wikidata5M shape (N = 4,594,485, 2E = 41,228,558, D = 100), times (CUDA events, median of --reps, L2 flushed
    before every launch) of the aggregation pieces, plain and grouped launched alternately in the same loop: the forward
    pass, the d_x / d_ee pass and the d_rel pass of the plain path; the grouped forward pass, agg_in from the group rows,
    the grouped d_x / d_ee pass, d_x += rel (.) Q and the two d_rel reductions of the grouped path.  Every pass includes
    its fix-up levels;
  - the whole layer step (forward + backward, CUDA graph replays, L2 flushed between them) per workload, plain and grouped
    alternately (plain / grouped / plain / grouped).
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

from sampled_time import gpu_info, k               # noqa: E402  (puts the repository and oracle/ on sys.path)
from bench import D_IN, Flusher, LayerCase, oracle, synth_rows      # noqa: E402
from compact_planes_time import timed               # noqa: E402


def kernel_times(case, reps, flush):
    L, p, st = k._lib, k._lib.ptr, k._lib.stream
    N, D, dev = case.N, D_IN, case.dev
    T = 2 * case.R + 1
    plan = k.get_plan(case.ei, case.et, N, T)
    grp = plan.grouped
    assert grp is not None, 'the Wikidata5M-shape graph should take the grouped path'
    n2, n_in = plan.num_edges2, plan.num_edges_in
    x, ee = case.x.detach(), case.ee.detach()
    relp = torch.cat([case.rl.detach(), case.conv.loop_rel.detach()], 0).contiguous()
    rel_f = torch.cat([case.rl.detach(), torch.ones((1, D), device=dev)], 0).contiguous()
    g3_all = torch.zeros((3 * N + grp.n_out, D), device=dev)
    g3_all[:3 * N] = synth_rows(torch.arange(3 * N, dtype=torch.int64, device=dev), D, 1.0, 21)
    g3 = g3_all[:3 * N].view(3, N, D)
    agg = torch.empty((2, N, D), device=dev)
    agg_g = torch.empty((2 * N + grp.n_in, D), device=dev)
    agg_c = torch.empty((grp.n_in_rows, D), device=dev)
    d_ee, d_x = torch.empty_like(ee), torch.empty((N, D), device=dev)
    dxq = torch.empty((N + grp.n_out, D), device=dev)
    d_rel = torch.empty((T, D), device=dev)

    def plain_fwd():
        plan.run_reduction(plan.fwd, lambda sp, o, c: L.call('kgc_agg_fwd', p(x), p(relp), T, p(ee), p(plan.rec_dst), p(sp.rowflags),
                                                              p(sp.chunks), sp.n_rec, p(o), p(c), D, st()),
                           agg, D, tag='kf', skip_prefill=[(0, N)])

    def plain_src():
        plan.run_reduction(plan.bwd_src, lambda sp, o, c: L.call(
            'kgc_agg_bwd_src', p(x), p(relp), T, p(ee), p(g3), p(plan.rec_src), p(sp.rowflags), p(sp.chunks), sp.n_rec, N, n_in,
            p(g3[2]), p(d_ee), p(o), p(c), D, st()), d_x, D, addend=g3[2], tag='ks')

    def plain_rel():
        plan.run_rel_reduction(lambda sp, o, c: L.call('kgc_agg_bwd_rel', p(x), p(ee), p(g3), p(plan.rec_type), p(sp.rowflags),
                                                        p(sp.chunks), sp.n_rec, N, n_in, p(o), p(c), D, st()), d_rel, D, tag='kr')

    def grp_fwd():
        plan.run_reduction(grp.fwd, lambda sp, o, c: L.call('kgc_agg_fwd', p(x), p(rel_f), T, p(ee), p(grp.rec_f), p(sp.rowflags),
                                                             p(sp.chunks), sp.n_rec, p(o), p(c), D, st()),
                           agg_g, D, tag='kfg')

    def grp_src():
        plan.run_reduction(grp.src, lambda sp, o, c: L.call(
            'kgc_agg_bwd_src_grouped', p(x), p(relp), T, p(ee), p(g3), p(grp.rec_s), p(sp.rowflags), p(grp.xrow_s), p(sp.chunks),
            sp.n_rec, N, n_in, grp.n_out, p(g3_all[2 * N:]), p(d_ee), p(o), p(c), D, st()), dxq, D, addend=g3_all[2 * N:], tag='ksg')

    def grp_rel():
        grp.drel_in.run(plan, agg_g[2 * N:], g3[0], d_rel, D, tag='kgri')
        grp.drel_out.run(plan, dxq[N:], x, d_rel, D, accumulate=True, tag='kgro')
    out = {'N': N, 'n_edges2': n2, 'D': D, 'groups_in': grp.n_in, 'groups_out': grp.n_out, 'rows_in': grp.n_in_rows}
    out['fwd'] = timed([('plain', plain_fwd), ('grouped', grp_fwd),
                        ('grouped_agg_in', lambda: grp.agg_in_c.run(plan, agg_g[2 * N:], relp, agg_c, D, tag='kgi'))], reps, flush)
    out['bwd_dx'] = timed([('plain', plain_src), ('grouped', grp_src),
                           ('grouped_dx_from_groups', lambda: grp.dx.run(plan, dxq[N:], relp, dxq[:N], D, accumulate=True,
                                                                         tag='kgx'))], reps, flush)
    out['bwd_drel'] = timed([('plain', plain_rel), ('grouped', grp_rel)], reps, flush)
    out['plain_total_ms'] = round(out['fwd']['plain']['ms'] + out['bwd_dx']['plain']['ms'] + out['bwd_drel']['plain']['ms'], 4)
    out['grouped_total_ms'] = round(out['fwd']['grouped']['ms'] + out['fwd']['grouped_agg_in']['ms'] + out['bwd_dx']['grouped']['ms']
                                    + out['bwd_dx']['grouped_dx_from_groups']['ms'] + out['bwd_drel']['grouped']['ms'], 4)
    return out


def step_times(case, steps, warm, flush):
    """Graph-replayed layer steps, plain and grouped alternately (each mode on a plan of its own, kept alive while its graph
    is replayed)."""
    res, graphs, plans = {}, {}, {}
    saved = k.plan.GROUP_MAX_SHARE, k.plan.GROUP_MIN_EDGES
    for mode in ('plain', 'grouped'):
        # the grouped arm ignores the size rule (GROUP_MIN_EDGES): at the two small shapes it is what sets that rule
        k.plan.GROUP_MAX_SHARE, k.plan.GROUP_MIN_EDGES = (-1.0, saved[1]) if mode == 'plain' else (saved[0], 0)
        k.plan._PLAN_CACHE.clear()
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    case.step()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            plans[mode] = plan = k.get_plan(case.ei, case.et, case.N, 2 * case.R + 1)
            k._lib.LAUNCHES = 0
            case.step()
            launches = k._lib.LAUNCHES
            g = torch.cuda.CUDAGraph()
            for t in case.leaves:
                t.grad = None
            with torch.cuda.graph(g):
                case.step()
            graphs[mode] = g
            res[mode] = {'grouped': plan.grouped is not None, 'launches_per_step': launches, 'ms': []}
        finally:
            k.plan.GROUP_MAX_SHARE, k.plan.GROUP_MIN_EDGES = saved
    for _ in range(2):
        for mode in ('plain', 'grouped'):
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
    del graphs, plans
    k.plan._PLAN_CACHE.clear()
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
        st = step_times(case, args.steps, args.warmup, flush)
        print(json.dumps({'workload': wl, 'layer_step': st}), flush=True)
        del case
        k.plan._PLAN_CACHE.clear()
        torch.cuda.empty_cache()


if __name__ == '__main__':
    main()
