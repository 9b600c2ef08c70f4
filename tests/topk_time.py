"""Debug aid (not a test): CUDA-event timing of filtered top-k prediction (K6k) at the Wikidata5M shape of bench.py's aux
leg - B = 65,536 queries, N = 4,594,485 entities, d = 200, the same seeded inputs, 4 exclusions per query.

    python tests/topk_time.py [--reps 5]

Reports, with the GPU name and power limit:
  - kernel time of kgc_score_topk (k = 10, k = 32) next to kgc_score_rank on the same packed operands: the three are
    alternated and the median of --reps repetitions is taken (the operands, 1.9 GB of bf16 entity rows, exceed L2);
  - the whole topk() call (query packing, checks, sweep, merge) in queries/s;
  - the adversarial order: scores = bias[j] = j (zero embeddings), so that every entity beats every list and inserts;
  - the exact mode (precision='fp32') at B = 1,024.
"""
import argparse
import json
import os
import subprocess
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np       # noqa: E402
import torch             # noqa: E402

import kgc_gcn_b200 as k                 # noqa: E402
from bench import _mix32, synth_rows     # noqa: E402


def gpu_info():
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv'],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return out.stdout.strip()


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'needs a GPU'
    print(gpu_info(), flush=True)
    L = k._lib
    dev = torch.device('cuda')
    B, N, d = 65536, 4594485, 200
    qid = torch.arange(B, dtype=torch.int64, device=dev)
    xq = synth_rows(qid, d, 1.7, 31).abs_()
    fptr = torch.arange(0, 4 * B + 1, 4, device=dev, dtype=torch.int64)
    fidx = (_mix32(torch.arange(4 * B, dtype=torch.int64, device=dev) + 4099) % N).view(B, 4).sort(1).values.reshape(-1).to(torch.int32)
    rows = torch.arange(N, dtype=torch.int64, device=dev)
    tab = synth_rows(rows, d, 1.0, 32)
    bias = synth_rows(rows, 1, 0.1, 33).view(-1)
    table = k.EntityTable(tab, bias)
    q16 = k.pack_queries(xq)
    res = {'gpu': gpu_info().splitlines()[-1], 'B': B, 'N': N, 'd': d, 'exclusions_per_query': 4, 'reps': args.reps}

    def topk_kernel(tb, kk, ptr=fptr, idx=fidx):
        out = {'s': torch.empty((B, kk), device=dev), 'i': torch.empty((B, kk), dtype=torch.int32, device=dev),
               'c': torch.empty((B,), dtype=torch.int32, device=dev)}
        wsb = int(L.lib().kgc_score_topk_workspace_bytes(B, tb.n, tb.kpad, kk))
        ws = torch.empty((wsb,), dtype=torch.uint8, device=dev)

        def go():
            L.call('kgc_score_topk', L.ptr(q16), L.ptr(tb.data), B, tb.n, tb.kpad, L.ptr(ptr), L.ptr(idx), kk, L.ptr(out['s']),
                   L.ptr(out['i']), L.ptr(out['c']), L.ptr(ws), wsb, L.stream())
        return go, out, wsb

    top10, out10, ws10 = topk_kernel(table, 10)
    top32, _, ws32 = topk_kernel(table, 32)
    top10()
    thr = out10['s'][:, 9].contiguous()
    gt = torch.zeros(B, dtype=torch.int32, device=dev)

    def rank():
        L.call('kgc_score_rank', L.ptr(q16), L.ptr(table.data), B, table.n, table.kpad, L.ptr(thr), L.ptr(gt), None, L.stream())
    for fn in (rank, top10, top32):
        fn()
    torch.cuda.synchronize()
    t = {'rank': [], 'topk10': [], 'topk32': []}
    for _ in range(args.reps):
        for name, fn in (('rank', rank), ('topk10', top10), ('topk32', top32)):
            t[name].append(event_ms(fn))
    med = {n: float(np.median(v)) for n, v in t.items()}
    flops = 2.0 * B * N * d
    res['kernel_ms_median'] = med
    res['kernel_ms_all'] = t
    res['topk10_over_rank'] = med['topk10'] / med['rank']
    res['topk32_over_rank'] = med['topk32'] / med['rank']
    res['tflops_unpadded'] = {n: flops / (v * 1e-3) / 1e12 for n, v in med.items()}
    res['workspace_mb'] = {'k10': ws10 / 2 ** 20, 'k32': ws32 / 2 ** 20}
    print(json.dumps({'kernels': med}), flush=True)

    # the whole public call: packing, CSR checks, sweep, merge
    def whole():
        return k.topk(xq, None, None, 10, fptr, fidx, table=table)
    whole()
    torch.cuda.synchronize()
    ms = [event_ms(whole) for _ in range(3)]
    res['topk_call_ms'] = float(np.median(ms))
    res['topk_call_queries_per_s'] = B / (res['topk_call_ms'] * 1e-3)
    print(json.dumps({'topk_call_ms': res['topk_call_ms']}), flush=True)

    # adversarial: zero embeddings, bias[j] = j -> every entity beats the current K-th key and inserts
    del table
    torch.cuda.empty_cache()
    adv = k.EntityTable(torch.zeros((N, d), device=dev), rows.to(torch.float32))
    a10, a_out, _ = topk_kernel(adv, 10)
    a32, _, _ = topk_kernel(adv, 32)
    a10()
    torch.cuda.synchronize()
    ok = bool((a_out['i'][:, 0] >= N - 5).all())        # the highest ids not excluded
    ta = {'adversarial_topk10': [], 'adversarial_topk32': []}
    for _ in range(max(3, args.reps // 2)):
        ta['adversarial_topk10'].append(event_ms(a10))
        ta['adversarial_topk32'].append(event_ms(a32))
    res['adversarial_kernel_ms_median'] = {n: float(np.median(v)) for n, v in ta.items()}
    res['adversarial_top1_is_highest_id'] = ok
    print(json.dumps(res['adversarial_kernel_ms_median']), flush=True)
    del adv
    torch.cuda.empty_cache()

    # exact mode at B = 1,024 (fp32-grade dense logits, 256 queries per tile)
    nb = 1024
    xs, fp, fi = xq[:nb].contiguous(), fptr[:nb + 1].contiguous(), fidx[:4 * nb].contiguous()

    def exact():
        return k.topk(xs, tab, bias, 10, fp, fi, precision='fp32')
    exact()
    torch.cuda.synchronize()
    ms = [event_ms(exact) for _ in range(3)]
    res['fp32_B'] = nb
    res['fp32_call_ms'] = float(np.median(ms))
    res['fp32_queries_per_s'] = nb / (res['fp32_call_ms'] * 1e-3)
    print(json.dumps(res), flush=True)


if __name__ == '__main__':
    main()
