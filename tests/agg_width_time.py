"""The level-0 aggregation kernels (kgc_agg_fwd / _bwd_src / _bwd_rel) at layer widths the benchmark does not run: each
launched alone through the C ABI at the FB15k-237 and Wikidata5M graph shapes, CUDA events, L2 flushed before every
launch (bench.Flusher).  Several builds of the library are loaded side by side and timed alternately in one process, so
an A/B of two builds shares the graph, the inputs and the GPU's state:

    python tests/agg_width_time.py [--libs A.so,B.so] [--widths 200,256] [--workloads fb15k237,wikidata5m] [--rounds 3]

One line per workload, width and library: the median ms of each kernel over all rounds, the range of the per-round
medians, and a checksum of everything the three kernels wrote (equal checksums: the same bits)."""
import argparse
import ctypes
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import kgc_gcn_b200 as k  # noqa: E402

KERNELS = ('kgc_agg_fwd', 'kgc_agg_bwd_src', 'kgc_agg_bwd_rel')


def load(path):
    h = ctypes.CDLL(os.path.abspath(path))
    for name in KERNELS + ('kgc_last_error',):
        res, args = k._lib.SIGNATURES[name]
        getattr(h, name).restype, getattr(h, name).argtypes = res, args
    return h


def checksum(ts):
    """Position-weighted sums of the int32 bit patterns (wrapping int64), chunked to bound the temporaries."""
    s = 0
    for t in ts:
        v = t.reshape(-1).view(torch.int32)
        for a in range(0, v.numel(), 1 << 27):
            c = v[a:a + (1 << 27)].to(torch.int64)
            w = torch.arange(a, a + c.numel(), dtype=torch.int64, device=c.device) * 2654435761 + 97
            s = (s * 1000003 + int((c * w).sum())) & ((1 << 64) - 1)
    return '%016x' % s


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--libs', default=k._lib.LIB_PATH, help='comma-separated library paths, timed alternately')
    ap.add_argument('--widths', default='200,256')
    ap.add_argument('--workloads', default='fb15k237,wikidata5m')
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--iters', type=int, default=10)
    a = ap.parse_args()
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    libs = [(p, load(p)) for p in a.libs.split(',')]
    print('gpu:', torch.cuda.get_device_name(dev), '| libs:', [p for p, _ in libs])
    flush = bench.Flusher(dev)
    orc = bench.oracle()
    for wl in a.workloads.split(','):
        N, R, E, seed = bench.WORKLOADS[wl]
        T = 2 * R + 1
        g = orc.build_graph(orc.synthetic_triples(N, R, E, seed), N, R)
        plan = k.get_plan(torch.from_numpy(g['edge_index']).to(dev), torch.from_numpy(g['edge_attr'][0]).to(dev), N, T)
        sf, ss, sr = plan.fwd, plan.bwd_src, plan.bwd_rel
        for D in [int(w) for w in a.widths.split(',')]:
            ar = lambda n: torch.arange(n, dtype=torch.int64, device=dev)      # noqa: E731
            x = bench.synth_rows(ar(N), D, bench.xavier_bound(N, D), 11)
            ee = bench.synth_rows(ar(2 * E), D, bench.xavier_bound(2 * E, D), 12)
            relp = bench.synth_rows(ar(T), D, bench.xavier_bound(T, D), 16)
            g3 = bench.synth_rows(ar(3 * N), D, 1.0, 21).view(3, N, D)
            agg, d_x = torch.empty((2, N, D), device=dev), torch.empty((N, D), device=dev)
            d_ee, d_rel = torch.empty_like(ee), torch.empty((plan.num_type_rows, D), device=dev)
            carry = [torch.empty((max(s.n_carry, 1), D), device=dev) for s in (sf, ss, sr)]
            outs = [agg, d_x, d_ee, d_rel] + carry
            p, st = k._lib.ptr, k._lib.stream

            def launches(h):
                def call(name, *args):
                    if getattr(h, name)(*args) != 0:
                        raise RuntimeError('{} failed: {}'.format(name, h.kgc_last_error().decode()))
                return [
                    lambda: call('kgc_agg_fwd', p(x), p(relp), T, p(ee), p(plan.rec_dst), p(sf.rowflags), p(sf.chunks),
                                 sf.n_rec, p(agg), p(carry[0]), D, st()),
                    lambda: call('kgc_agg_bwd_src', p(x), p(relp), T, p(ee), p(g3), p(plan.rec_src), p(ss.rowflags),
                                 p(ss.chunks), ss.n_rec, N, E, p(g3[2]), p(d_ee), p(d_x), p(carry[1]), D, st()),
                    lambda: call('kgc_agg_bwd_rel', p(x), p(ee), p(g3), p(plan.rec_type), p(sr.rowflags), p(sr.chunks),
                                 sr.n_rec, N, E, p(d_rel), p(carry[2]), D, st())]
            fns = {path: launches(h) for path, h in libs}
            sums = {}
            for path, _ in libs:                     # every output zeroed, then written once by this library
                for t in outs:
                    t.zero_()
                for fn in fns[path]:
                    fn()
                sums[path] = checksum(outs)
            ms = {(path, i): [] for path, _ in libs for i in range(3)}
            for _ in range(a.rounds):
                for path, _ in libs:
                    for i, fn in enumerate(fns[path]):
                        fn()
                        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                              for _ in range(a.iters)]
                        for e0, e1 in ev:
                            flush()
                            e0.record()
                            fn()
                            e1.record()
                        torch.cuda.synchronize()
                        ms[(path, i)].append([e0.elapsed_time(e1) for e0, e1 in ev])
            for path, _ in libs:
                cols = []
                for i, name in enumerate(KERNELS):
                    per_round = [float(np.median(r)) for r in ms[(path, i)]]
                    cols.append('{} {:.4f} ({:.4f}-{:.4f})'.format(name[8:], float(np.median(sum(ms[(path, i)], []))),
                                                                   min(per_round), max(per_round)))
                print('{} D={} {}: {} | checksum {}'.format(wl, D, path, ' '.join(cols), sums[path]), flush=True)
            del x, ee, relp, g3, agg, d_x, d_ee, d_rel, carry, outs, fns
            torch.cuda.empty_cache()
        k.plan._PLAN_CACHE.clear()
        torch.cuda.empty_cache()


if __name__ == '__main__':
    main()
