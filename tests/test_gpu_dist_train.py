"""Multi-GPU training of M-GCN (MGCN.shard): the shard kernels of the 1-N loss and the split ClipAdam step on one GPU, and
the sharded training step on two GPUs against the single-GPU model (tests/dist_train_check.py, skipped on a 1-GPU box)."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import kgc_gcn_b200 as k          # noqa: E402

pytestmark = pytest.mark.gpu
N_ROWS, B = 50003, 300            # a prime row count; two 256-query tiles of the scorer


def _csr(rng, n_query, n):
    """Query -> objects CSR (ascending objects per query, 0 to 40 of them, some queries empty)."""
    lens = rng.integers(0, 41, n_query)
    lens[::17] = 0
    ptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    idx = np.concatenate([np.sort(rng.choice(n, int(m), replace=False)) for m in lens]).astype(np.int32)
    return ptr, idx


def _shards(rng, n, n_shards):
    """Uneven random split of [0, n): per shard the global ids in local-row order, and row_of [n] int32."""
    owner = rng.choice(n_shards, n, p=np.arange(1, n_shards + 1) / (n_shards * (n_shards + 1) / 2))
    row_of = np.full(n, -1, dtype=np.int32)
    ids = []
    for s in range(n_shards):
        mine = rng.permutation(np.nonzero(owner == s)[0])
        row_of[mine] = np.arange(mine.shape[0], dtype=np.int32)
        ids.append(mine)
    return ids, owner, row_of


def _mask_numpy(qid, ptr, idx, rows, n_rows, Bq):
    wb = (Bq + 31) // 32
    m = np.zeros((n_rows, wb), dtype=np.uint32)
    for b, q in enumerate(qid):
        for j in idx[ptr[q]:ptr[q + 1]]:
            r = rows[j]
            if r >= 0:
                m[r, b >> 5] |= np.uint32(1 << (b & 31))
    return m.view(np.int32)


@pytest.mark.parametrize('n_shards', [1, 2, 3, 4])
@pytest.mark.parametrize('smooth', [False, True])
def test_shard_mask_and_loss_pass_match_the_unsharded_call(n_shards, smooth):
    dev = torch.device('cuda')
    rng = np.random.default_rng(10 * n_shards + int(smooth))
    ptr, idx = _csr(rng, 700, N_ROWS)
    qid = rng.integers(0, 700, B).astype(np.int64)
    ids, owner, row_of = _shards(rng, N_ROWS, n_shards)
    pos, add = ((np.float32(0.9) + np.float32(1.0 / N_ROWS)), np.float32(1.0 / N_ROWS)) if smooth else (1.0, 0.0)
    ldt = (B + 3) // 4 * 4
    g = torch.Generator().manual_seed(n_shards)
    pred = torch.rand((N_ROWS, ldt), generator=g, dtype=torch.float64)
    pred[::97] = pred[::97] ** 40                                  # probabilities near 0 and 1 (the clamped logs)
    pred[1::89] = 1.0 - pred[1::89] ** 40
    pred = pred.float().clamp(1e-30, 1.0 - 2 ** -24).to(dev)
    p = k._lib.ptr
    d_qid, d_ptr, d_idx = (torch.from_numpy(a).to(dev) for a in (qid, ptr, idx))
    st = k._lib.stream()

    whole = pred.clone()
    mask = torch.empty((N_ROWS, (B + 31) // 32), dtype=torch.int32, device=dev)
    k._lib.call('kgc_label_mask_t_build', p(d_qid), B, p(d_ptr), p(d_idx), N_ROWS, p(mask), st)
    d_bias = torch.empty((N_ROWS,), dtype=torch.float32, device=dev)
    part_w = torch.empty((int(k._lib.lib().kgc_bce_1n_t_blocks(N_ROWS)),), dtype=torch.float64, device=dev)
    loss = torch.empty((1,), dtype=torch.float32, device=dev)
    k._lib.call('kgc_bce_1n_bwd_logit_t', p(whole), p(mask), N_ROWS, B, ldt, float(pos), float(add), p(d_bias), p(part_w),
                p(loss), st)
    total = 0.0
    for s in range(n_shards):
        gid = torch.from_numpy(ids[s]).to(dev)
        n = int(gid.numel())
        rows = np.where(owner == s, row_of, -1).astype(np.int32)   # this shard's map: -1 for the other shards' entities
        m_s = torch.full((n, (B + 31) // 32), -1, dtype=torch.int32, device=dev)           # the call zeroes it
        k._lib.call('kgc_label_mask_t_build_rows', p(d_qid), B, p(d_ptr), p(d_idx), p(torch.from_numpy(rows).to(dev)), n,
                    p(m_s), st)
        want = _mask_numpy(qid, ptr, idx, rows, n, B)
        assert np.array_equal(m_s.cpu().numpy(), want)
        pred_s = pred.index_select(0, gid).contiguous()
        db_s = torch.empty((n,), dtype=torch.float32, device=dev)
        part_s = torch.empty((int(k._lib.lib().kgc_bce_1n_t_blocks(n)),), dtype=torch.float64, device=dev)
        ls = torch.empty((1,), dtype=torch.float64, device=dev)
        k._lib.call('kgc_bce_1n_bwd_logit_t_shard', p(pred_s), p(m_s), n, B, ldt, float(pos), float(add), N_ROWS, p(db_s),
                    p(part_s), p(ls), st)
        assert torch.equal(pred_s, whole.index_select(0, gid)), 'logit gradient rows of shard %d' % s
        assert torch.equal(db_s, d_bias.index_select(0, gid)), 'd_bias of shard %d' % s
        total += float(ls)
    ref = float(part_w.sum())                                      # the unsharded fp64 sum: loss * B * N before rounding
    assert abs(total - ref) <= 1e-12 * abs(ref)
    assert abs(np.float32(total / (B * N_ROWS)) - float(loss)) <= 1e-6 * abs(float(loss))


def _opt_tables(tensors, dev, flags=None):
    """kgc_opt_tensor_t table [n, 4] int64 and work items [n_items, 4] int32 over (param, grad, m, v) tuples."""
    chunk = int(k._lib.lib().kgc_opt_chunk_elems())
    table = torch.tensor([[t.data_ptr() for t in ts] for ts in tensors], dtype=torch.int64, device=dev)
    items = []
    for i, ts in enumerate(tensors):
        n = ts[0].numel()
        for c in range((n + chunk - 1) // chunk):
            items.append((i, c, min(chunk, n - c * chunk), 0 if flags is None else flags[i]))
    return table, torch.tensor(items, dtype=torch.int32, device=dev)


def _ulp_dist(a, b):
    ia = a.view(torch.int32).to(torch.int64)
    ib = b.view(torch.int32).to(torch.int64)
    ia = torch.where(ia < 0, -(ia & 0x7FFFFFFF), ia)
    ib = torch.where(ib < 0, -(ib & 0x7FFFFFFF), ib)
    return int((ia - ib).abs().max())


@pytest.mark.parametrize('n_shards', [1, 2, 3, 4])
@pytest.mark.parametrize('clipping', [False, True])
def test_split_clip_adam_equals_the_whole_step(n_shards, clipping):
    """One sharded table (rows split unevenly) and two replicated tensors, counted on 'rank' 0 only, against
    kgc_clip_adam_step on the whole model; three steps."""
    dev = torch.device('cuda')
    rng = np.random.default_rng(n_shards)
    g = torch.Generator().manual_seed(7 + n_shards)
    shapes = {'table': (50003, 20), 'w': (333, 77), 'b': (1001,)}
    full = {n: torch.randn(s, generator=g).to(dev) for n, s in shapes.items()}
    grads = [{n: torch.randn(s, generator=g).to(dev) * 0.01 for n, s in shapes.items()} for _ in range(3)]
    ids, _, _ = _shards(rng, 50003, n_shards)
    sq = sum(float((gr[n].double() ** 2).sum()) for gr in grads[:1] for n in shapes) ** 0.5
    max_norm = sq * 0.25 if clipping else sq * 100.0
    hyper = torch.tensor([1e-2, 0.9, 0.999, 1e-8, 1e-4, max_norm], dtype=torch.float32, device=dev)
    p = k._lib.ptr
    st = k._lib.stream()

    # the whole model
    W = {n: (full[n].clone(), torch.empty_like(full[n]), torch.zeros_like(full[n]), torch.zeros_like(full[n])) for n in shapes}
    state_w = torch.zeros((5,), dtype=torch.float64, device=dev)
    # the whole model again, stepped by sqnorm + apply without flags: equal to the step bit for bit, norm included
    W2 = {n: tuple(t.clone() for t in W[n]) for n in shapes}
    state_w2 = torch.zeros((5,), dtype=torch.float64, device=dev)
    # the shards: rank s holds its rows of the table and a copy of the replicated tensors
    R = []
    for s in range(n_shards):
        gid = torch.from_numpy(ids[s]).to(dev)
        r = {'table': (full['table'][gid].clone(),) + tuple(torch.zeros((gid.numel(), 20), device=dev) for _ in range(3))}
        for n in ('w', 'b'):
            r[n] = (full[n].clone(), torch.empty_like(full[n]), torch.zeros_like(full[n]), torch.zeros_like(full[n]))
        R.append((gid, r, torch.zeros((5,), dtype=torch.float64, device=dev)))
    for step in range(3):
        for n in shapes:
            W[n][1].copy_(grads[step][n])
        tab, it = _opt_tables([W[n] for n in shapes], dev)
        partials = torch.empty((it.shape[0],), dtype=torch.float64, device=dev)
        k._lib.call('kgc_clip_adam_step', p(tab), p(it), it.shape[0], p(hyper), p(state_w), p(partials), st)
        for n in shapes:
            W2[n][1].copy_(grads[step][n])
        tab2, it2 = _opt_tables([W2[n] for n in shapes], dev)
        sq2 = torch.empty((2,), dtype=torch.float64, device=dev)
        k._lib.call('kgc_clip_adam_sqnorm', p(tab2), p(it2), it2.shape[0], p(partials), p(sq2), st)
        k._lib.call('kgc_clip_adam_apply', p(tab2), p(it2), it2.shape[0], p(hyper), p(state_w2), p(sq2), st)
        assert torch.equal(state_w2, state_w)
        for n in shapes:
            for j in (0, 2, 3):
                assert torch.equal(W2[n][j], W[n][j])
        sqs, tabs = [], []
        for s, (gid, r, _) in enumerate(R):
            r['table'][1].copy_(grads[step]['table'][gid])
            for n in ('w', 'b'):
                r[n][1].copy_(grads[step][n])
            tab_s, it_s = _opt_tables([r[n] for n in shapes], dev, flags=[0, int(s != 0), int(s != 0)])
            part_s = torch.empty((it_s.shape[0],), dtype=torch.float64, device=dev)
            sqn = torch.empty((2,), dtype=torch.float64, device=dev)
            k._lib.call('kgc_clip_adam_sqnorm', p(tab_s), p(it_s), it_s.shape[0], p(part_s), p(sqn), st)
            sqs.append(sqn)
            tabs.append((tab_s, it_s))
        glob = sqs[0].clone()
        for sqn in sqs[1:]:
            glob += sqn                                            # the all-reduce, in rank order
        for (gid, r, state_s), (tab_s, it_s) in zip(R, tabs):
            k._lib.call('kgc_clip_adam_apply', p(tab_s), p(it_s), it_s.shape[0], p(hyper), p(state_s), p(glob.clone()), st)
        torch.cuda.synchronize()
        for gid, r, state_s in R:
            # the shards' rows sit in another order, so the fp32 per-thread sums of the chunks differ in rounding
            assert abs(float(state_s[4]) - float(state_w[4])) <= 1e-7 * float(state_w[4])
            assert (float(state_s[1]) < 1.0) == clipping
            for n in shapes:
                got = r[n]
                want = [t[gid] for t in W[n]] if n == 'table' else W[n]
                for j in (0, 2, 3):                                 # parameter, exp_avg, exp_avg_sq
                    if clipping:
                        assert _ulp_dist(got[j], want[j]) <= 2, (n, j, step)
                    else:
                        assert torch.equal(got[j], want[j]), (n, j, step)


def test_split_clip_adam_argument_checks():
    p = k._lib.ptr
    with pytest.raises(RuntimeError, match='null argument'):
        k._lib.call('kgc_clip_adam_sqnorm', None, None, 1, None, None, k._lib.stream())
    with pytest.raises(RuntimeError, match='bad sizes'):
        t = torch.zeros((4,), device='cuda')
        k._lib.call('kgc_bce_1n_bwd_logit_t_shard', p(t), p(t), 5, 4, 4, 1.0, 0.0, 4, p(t), p(t), p(t), k._lib.stream())


def _launch(n_proc, script, marker):
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(n_proc), '--master-addr',
           '127.0.0.1', '--master-port', str(port), os.path.join(ROOT, 'tests', script)]
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1200)
    assert p.returncode == 0 and marker in p.stdout, p.stdout[-6000:]


def test_one_rank_sharded_model_matches_mgcn():
    """The sharded model's code path on one rank (NCCL, edge-balanced partition): loss, gradients, norm, full_state_dict."""
    _launch(1, 'dist_train_check.py', 'DIST_TRAIN_OK')


def test_two_gpu_sharded_training_step():
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    _launch(2, 'dist_train_check.py', 'DIST_TRAIN_OK')
