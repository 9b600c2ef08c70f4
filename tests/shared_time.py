"""CUDA-event medians of the sampled losses' forward + backward at B = 4,096, D = 200, N = 4,594,485 (the Wikidata5M
shape): per-query negatives (score_sampled_bce / _ce on [B, 1 + k] candidates) against batch-shared ones
(score_shared_bce / _ce) at k = 256 and 4,096, launched alternately.  Prints the GPU name and power limit first.

    python tests/shared_time.py [--reps 20] [--out profiles/r16_shared_time.log]
"""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import kgc_gcn_b200 as k   # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       stdout=subprocess.PIPE, text=True)
    say('gpu: ' + q.stdout.strip())
    B, D, N = 4096, 200, 4594485
    g = torch.Generator(device='cuda').manual_seed(0)
    x = torch.randn(B, D, device='cuda', generator=g).requires_grad_(True)
    ent = (torch.randn(N, D, device='cuda', generator=g) * D ** -0.5).requires_grad_(True)
    bias = (torch.randn(N, device='cuda', generator=g) * 0.1).requires_grad_(True)
    n_q = 4 * B
    lens = torch.randint(0, 8, (n_q,), device='cuda', generator=g)
    ptr = torch.zeros(n_q + 1, dtype=torch.int64, device='cuda')
    ptr[1:] = torch.cumsum(lens, 0)
    idx = torch.randint(0, N, (int(ptr[-1]),), device='cuda', generator=g).to(torch.int32)
    qid = torch.randperm(n_q, device='cuda', generator=g)[:B]
    pos = torch.randint(0, N, (B, 1), device='cuda', generator=g).to(torch.int32)
    for kk in (256, 4096):
        shared = torch.randint(0, N, (kk,), device='cuda', generator=g).to(torch.int32)
        cand = torch.cat([pos, torch.randint(0, N, (B, kk), device='cuda', generator=g).to(torch.int32)], 1)
        for crit in ('bce', 'ce'):
            if crit == 'bce':
                per_q = lambda: k.score_sampled_bce(x, ent, bias, cand, 1)           # noqa: E731
                sh = lambda: k.score_shared_bce(x, ent, bias, pos, shared, qid, ptr, idx)   # noqa: E731
            else:
                per_q = lambda: k.score_sampled_ce(x, ent, bias, cand, 1)            # noqa: E731
                sh = lambda: k.score_shared_ce(x, ent, bias, pos, shared, qid, ptr, idx)    # noqa: E731
            ts = {'per_query': [], 'shared': []}
            for r in range(a.reps + 2):
                for name, fn in (('per_query', per_q), ('shared', sh)):
                    x.grad = ent.grad = bias.grad = None
                    torch.cuda.synchronize()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    fn().backward()
                    e1.record()
                    torch.cuda.synchronize()
                    if r >= 2:
                        ts[name].append(e0.elapsed_time(e1))
            med = {n: sorted(v)[len(v) // 2] for n, v in ts.items()}
            say('B={} k={} D={} N={} {}: fwd+bwd median per_query {:.3f} ms  shared {:.3f} ms  ({} reps, alternating)'.format(
                B, kk, D, N, crit, med['per_query'], med['shared'], a.reps))
    if a.out:
        os.makedirs(os.path.dirname(a.out), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write('\n'.join(lines) + '\n')


if __name__ == '__main__':
    main()
