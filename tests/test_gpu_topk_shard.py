"""Entity-sharded filtered top-k: ``topk(..., n_offset=lo)`` on slices of the entity table, ``merge_topk`` /
``kgc_topk_merge``, and ``topk(..., group=...)`` in one process (the two-process run is tests/dist_topk_check.py).

The bar: sweeping disjoint slices and merging them gives the unsharded call's scores, ids and counts bit for bit, in
both precisions.  In bf16 a logit is one packed query row against one packed entity row; in fp32 it is one 3xTF32 row
against one column in a fixed K order; neither depends on where the row sits in the table.
"""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch

from test_gpu_topk import csr, exclusion_lists, int_operands, random_case, reference_topk

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def k():
    import kgc_gcn_b200
    kgc_gcn_b200._lib.lib()
    return kgc_gcn_b200


def straddle_lists(B, N, cuts, seed):
    """Every row excludes ids on both sides of a shard boundary (plus a few random ones and ids outside [0, N))."""
    rng = np.random.default_rng(seed)
    lists = []
    for q in range(B):
        c = cuts[q % len(cuts)]
        lst = [c - 2, c - 1, c, c + 1] + rng.integers(0, N, size=3).tolist() + ([-1, N] if q % 4 == 0 else [])
        lists.append(sorted(v for v in lst if -1 <= v <= N))
    return csr(lists)


def sharded(k, xq, tab, bias, kk, ptr, idx, precision, bounds):
    """topk of every slice [bounds[i], bounds[i + 1]) with global ids, merged with merge_topk."""
    cu = lambda a: None if a is None else torch.from_numpy(a).cuda()          # noqa: E731
    parts = []
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        table = k.EntityTable(tab[lo:hi], bias[lo:hi]) if precision == 'bf16' and hi > lo else None
        out = k.topk(xq, tab[lo:hi], bias[lo:hi], kk, cu(ptr), cu(idx), table=table, precision=precision, n_offset=lo)
        if hi == lo:
            assert bool((out['count'] == 0).all()) and bool((out['ids'] == -1).all())
        else:
            assert bool(((out['ids'] == -1) | ((out['ids'] >= lo) & (out['ids'] < hi))).all())
        parts.append(out)
    return k.merge_topk(torch.stack([o['scores'] for o in parts]), torch.stack([o['ids'] for o in parts]))


def assert_same(a, b, what):
    for key in ('count', 'ids', 'scores'):
        assert a[key].dtype == b[key].dtype and a[key].shape == b[key].shape, (what, key)
        assert torch.equal(a[key], b[key]), (what, key)


def splits(N, kk):
    """1 to 5 pieces; boundaries off the 128-row tiles; one piece smaller than k; one empty piece (not at row 0: a slice
    at offset 0 is the plain unsharded call, which takes N > 0)."""
    small = max(kk - 1, 1)
    return [[0, N], [0, 7001 % N, N], [0, 300, 300 + small, N],
            [0, 129, 129, N // 3, 2 * N // 3 + 5, N], [0, N // 2 + 3, N // 2 + 3, N]]


@gpu
@pytest.mark.parametrize('B,N,d', [(300, 20000, 200), (130, 1000, 61)])
def test_shard_merge_bit_exact_integer_inputs(k, B, N, d):
    """Small-integer operands: many exact ties, also across boundaries (the lower id wins); the merge must also equal
    the numpy reference."""
    xq, tab, bias = (t.cuda() for t in int_operands(B, N, d, seed=B + N + d))
    scores = (xq.double() @ tab.double().t() + bias.double()).cpu().numpy()
    table = k.EntityTable(tab, bias)
    cuts = sorted({c for s in splits(N, 32) for c in s[1:-1]})
    modes = {m: exclusion_lists(B, N, m, seed=N + d) for m in ('none', 'random', 'few')}
    modes['straddle'] = straddle_lists(B, N, cuts, seed=3)
    for mode, (ptr, idx) in modes.items():
        cu = lambda a: None if a is None else torch.from_numpy(a).cuda()      # noqa: E731
        for kk in (1, 10, 16, 17, 32):
            ref = reference_topk(scores, ptr, idx, kk)
            for precision in ('bf16', 'fp32'):
                whole = k.topk(xq, tab, bias, kk, cu(ptr), cu(idx), table=table if precision == 'bf16' else None,
                               precision=precision)
                np.testing.assert_array_equal(whole['ids'].cpu().numpy(), ref[1])
                for bounds in splits(N, kk):
                    got = sharded(k, xq, tab, bias, kk, ptr, idx, precision, bounds)
                    assert_same(got, whole, (mode, kk, precision, bounds))
            if mode == 'few':
                assert (ref[2] < 32).any()                            # rows with fewer than k eligible entities


@gpu
def test_shard_merge_bit_exact_random_floats(k):
    B, N, d = 300, 30011, 200
    xq, tab, bias, ptr, idx = random_case(B, N, d, seed=21)
    xq, tab, bias = xq.cuda(), tab.cuda(), bias.cuda()
    table = k.EntityTable(tab, bias)
    for kk in (1, 10, 32):
        for precision in ('bf16', 'fp32'):
            whole = k.topk(xq, tab, bias, kk, torch.from_numpy(ptr).cuda(), torch.from_numpy(idx).cuda(),
                           table=table if precision == 'bf16' else None, precision=precision)
            for bounds in splits(N, kk):
                assert_same(sharded(k, xq, tab, bias, kk, ptr, idx, precision, bounds), whole, (kk, precision, bounds))


def numpy_merge(s, i, kk):
    """Union of the real entries of every list, sorted by (logit descending, id ascending), -0.0 == +0.0."""
    S, B, _ = s.shape
    out_s = np.full((B, kk), -np.inf, dtype=np.float32)
    out_i = np.full((B, kk), -1, dtype=np.int64)
    cnt = np.zeros(B, dtype=np.int32)
    for q in range(B):
        real = i[:, q, :] >= 0
        ss, ii = s[:, q, :][real], i[:, q, :][real].astype(np.int64)
        o = np.lexsort((ii, -ss.astype(np.float64)))[:kk]
        out_s[q, :len(o)] = ss[o] + np.float32(0.0)                       # -0.0 comes back as +0.0
        out_i[q, :len(o)] = ii[o]
        cnt[q] = len(o)
    return out_s, out_i, cnt


def sorted_lists(rng, S, B, kin, values):
    """S lists per row over disjoint ids, each of random fill (0 .. kin real entries), sorted as topk returns them."""
    s = np.full((S, B, kin), -np.inf, dtype=np.float32)
    i = np.full((S, B, kin), -1, dtype=np.int32)
    for q in range(B):
        ids = rng.permutation(S * kin * 4)[:S * kin].reshape(S, kin)
        for l in range(S):
            fill = int(rng.integers(0, kin + 1)) if q % 5 else (0 if l == 0 else kin)
            sc = rng.choice(values, size=fill).astype(np.float32)
            o = np.lexsort((ids[l, :fill], -sc.astype(np.float64)))
            s[l, q, :fill], i[l, q, :fill] = sc[o], ids[l, :fill][o]
    return s, i


@gpu
def test_merge_topk_against_numpy(k):
    # hand-made: a cross-list tie goes by id, -0.0 ties +0.0, an all-padding list, lists of different fill
    ninf = -np.inf
    s = np.array([[[3.0, 2.0, 2.0, -0.0]], [[3.0, 2.0, 0.0, ninf]], [[ninf, ninf, ninf, ninf]]], dtype=np.float32)
    i = np.array([[[7, 1, 9, 5]], [[2, 4, 3, -1]], [[-1, -1, -1, -1]]], dtype=np.int32)
    out = k.merge_topk(torch.from_numpy(s).cuda(), torch.from_numpy(i).cuda())
    assert out['ids'].tolist() == [[2, 7, 1, 4]] and out['scores'].tolist() == [[3.0, 3.0, 2.0, 2.0]]
    assert out['count'].tolist() == [4] and out['ids'].dtype == torch.int64
    out = k.merge_topk(torch.from_numpy(s).cuda(), torch.from_numpy(i).cuda(), k=9)
    assert out['ids'].tolist() == [[2, 7, 1, 4, 9, 3, 5, -1, -1]] and out['count'].tolist() == [7]
    assert not torch.signbit(out['scores'][0, 5:7]).any()                 # the zeros come back as +0.0
    assert out['scores'][0, 7:].tolist() == [ninf, ninf]
    one = k.merge_topk(torch.from_numpy(s[2:]).cuda(), torch.from_numpy(i[2:]).cuda())
    assert one['count'].tolist() == [0] and one['ids'].tolist() == [[-1] * 4]

    rng = np.random.default_rng(0)
    values = np.array([-2.0, -1.0, -0.0, 0.0, 1.0, 1.5, 2.0, np.float32(1e-3), -np.inf], dtype=np.float32)
    for S, B, kin in ((1, 40, 1), (2, 300, 10), (3, 257, 16), (5, 130, 17), (8, 200, 32)):
        s, i = sorted_lists(rng, S, B, kin, values)
        ts, ti = torch.from_numpy(s).cuda(), torch.from_numpy(i).cuda()
        for kk in sorted({1, kin, min(kin + 5, 32), max(kin - 3, 1)}):
            # reading only the first kk entries of every list: the reference sees the same truncated lists
            ref = numpy_merge(s[:, :, :kk], i[:, :, :kk], kk)
            out = k.merge_topk(ts, ti, k=kk)
            np.testing.assert_array_equal(out['count'].cpu().numpy(), ref[2], err_msg=str((S, kin, kk)))
            np.testing.assert_array_equal(out['ids'].cpu().numpy(), ref[1], err_msg=str((S, kin, kk)))
            np.testing.assert_array_equal(out['scores'].cpu().numpy(), ref[0], err_msg=str((S, kin, kk)))
            assert not torch.signbit(out['scores'][out['scores'] == 0]).any()
            perm = torch.from_numpy(rng.permutation(S)).cuda()               # the list order does not matter
            assert_same(k.merge_topk(ts[perm], ti[perm].long(), k=kk), out, (S, kin, kk))


@gpu
def test_shard_arguments(k):
    s = torch.zeros((2, 3, 4), device='cuda')
    i = torch.zeros((2, 3, 4), dtype=torch.int32, device='cuda')
    for bad in ((s, i[:, :, :3]), (s[0], i[0]), (s[:0], i[:0]), (s.double(), i)):
        with pytest.raises((ValueError, TypeError)):
            k.merge_topk(*bad)
    for kk in (0, 33, 2.0):
        with pytest.raises(ValueError):
            k.merge_topk(s, i, k=kk)
    with pytest.raises(ValueError):                                       # k_in > 32 without a smaller k
        k.merge_topk(torch.zeros((1, 3, 33), device='cuda'), torch.zeros((1, 3, 33), dtype=torch.int32, device='cuda'))
    with pytest.raises(ValueError):
        k.merge_topk(s, torch.full((2, 3, 4), 2 ** 31, dtype=torch.int64, device='cuda'))
    with pytest.raises(RuntimeError):
        k.merge_topk(s.cpu(), i.cpu())
    xq, tab, bias = (t.cuda() for t in int_operands(4, 300, 200, seed=2))
    for off in (-1, 1.5, True):
        with pytest.raises(ValueError):
            k.topk(xq, tab, bias, 3, n_offset=off)
    with pytest.raises(ValueError):                                       # ids past 2^31
        k.topk(xq, tab, bias, 3, n_offset=2 ** 31 - 100)
    with pytest.raises(ValueError):                                       # no rows given
        k.topk(xq, None, None, 3, n_offset=5)
    # zero queries: empty results, no launch
    e = k.merge_topk(torch.zeros((2, 0, 4), device='cuda'), torch.zeros((2, 0, 4), dtype=torch.int32, device='cuda'))
    assert e['ids'].shape == (0, 4) and e['count'].shape == (0,)


def test_topk_merge_abi_rejects_bad_arguments():
    """CPU: the C entry refuses bad sizes and null pointers before it touches the device."""
    import kgc_gcn_b200 as k
    h = k._lib.lib()
    buf = (ctypes.c_char * 4096)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    ok = (p, p, 2, 3, 4, p, p, p, None)
    for pos, val in ((2, 0), (3, 0), (3, -1), (4, 0), (4, 33), (0, None), (1, None), (5, None), (6, None), (7, None)):
        args = list(ok)
        args[pos] = val
        assert h.kgc_topk_merge(*args) != 0, (pos, val)
        assert b'' != h.kgc_last_error()


@gpu
def test_shard_merge_at_scale(k):
    """2,048 integer queries x 1,000,003 entities in 4 uneven shards against the unsharded call, both precisions."""
    g = torch.Generator().manual_seed(3)
    B, N, d = 2048, 1000003, 200
    xq = torch.randint(-2, 3, (B, d), generator=g).float().cuda()
    tab = torch.randint(-2, 3, (N, d), generator=g, dtype=torch.int8).float().cuda()
    bias = torch.randint(-2, 3, (N,), generator=g).float().cuda()
    ex = torch.randint(0, N, (B, 4), generator=g).sort(1).values
    ptr = np.arange(0, 4 * B + 1, 4, dtype=np.int64)
    idx = ex.reshape(-1).numpy().astype(np.int32)
    bounds = [0, 250001, 500000, 749999, N]
    table = k.EntityTable(tab, bias)
    for kk in (10, 32):
        for precision in ('bf16', 'fp32'):
            whole = k.topk(xq, tab, bias, kk, torch.from_numpy(ptr).cuda(), torch.from_numpy(idx).cuda(),
                           table=table if precision == 'bf16' else None, precision=precision)
            assert bool((whole['count'] == kk).all())
            assert_same(sharded(k, xq, tab, bias, kk, ptr, idx, precision, bounds), whole, (kk, precision))


@gpu
def test_group_of_one_process(k):
    """topk(..., group=...) in a one-rank NCCL group: the gather / merge path equals the plain call."""
    import torch.distributed as dist
    if dist.is_initialized():
        pytest.skip('a process group is already initialised')
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    dist.init_process_group('nccl', init_method='tcp://127.0.0.1:{}'.format(port), rank=0, world_size=1,
                            device_id=torch.device('cuda', torch.cuda.current_device()))
    try:
        B, N, d = 300, 5003, 200
        xq, tab, bias = (t.cuda() for t in int_operands(B, N, d, seed=8))
        ptr, idx = (torch.from_numpy(a).cuda() for a in exclusion_lists(B, N, 'few', seed=8))
        for precision in ('bf16', 'fp32'):
            for kk in (10, 32):
                whole = k.topk(xq, tab, bias, kk, ptr, idx, precision=precision)
                assert_same(k.topk(xq, tab, bias, kk, ptr, idx, precision=precision, group=dist.group.WORLD), whole,
                            (precision, kk))
                # this rank's rows are [7, N + 7) of a larger table: the ids move, nothing else
                got = k.topk(xq, tab, bias, kk, ptr, (idx.long() + 7).int(), precision=precision, n_offset=7,
                             group=dist.group.WORLD)
                assert torch.equal(got['ids'], torch.where(whole['ids'] >= 0, whole['ids'] + 7, whole['ids']))
                assert torch.equal(got['scores'], whole['scores']) and torch.equal(got['count'], whole['count'])
    finally:
        dist.destroy_process_group()


@gpu
def test_two_gpu_sharded_topk():
    """tests/dist_topk_check.py on two processes, one GPU each (skipped on a 1-GPU box)."""
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr', '127.0.0.1',
           '--master-port', str(port), os.path.join(ROOT, 'tests', 'dist_topk_check.py')]
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert p.returncode == 0 and 'DIST_TOPK_OK' in p.stdout, p.stdout[-4000:]
