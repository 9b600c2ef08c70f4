"""bench.py --dump-outputs on the GPU: what it writes is the last timed step's outputs and gradients (checked against the
float64 oracle run with that step's own dropout draws), as float32 .npy files within 64 MB; two runs with the same
arguments write the same arrays (the inputs are seeded); --steps is the number of steps the timed loop ran."""
import importlib.util
import json
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAST = ['--workload', 'wn18rr', '--no-extras', '--no-aux', '--no-e2e', '--no-cpu-baseline', '--no-parity']


def _bench_module():
    spec = importlib.util.spec_from_file_location('kgc_bench', os.path.join(ROOT, 'bench.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _bench(out_dir, steps):
    p = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', str(steps), '--warmup', '2',
                        '--dump-outputs', str(out_dir)] + FAST,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-4000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_dump_outputs_is_reproducible(tmp_path):
    a, b = tmp_path / 'a', tmp_path / 'b'
    line = _bench(a, 3)
    assert line['steps'] == 3 and line['timed_steps'] == 3                      # timed_steps: iterations of the timed loop
    assert _bench(b, 4)['timed_steps'] == 4
    names = sorted(os.listdir(a))
    assert names == sorted(os.listdir(b))
    want = {'all_ent', 'all_rel', 'd_x', 'd_ee', 'd_rel', 'd_loop_weight', 'd_in_weight', 'd_out_weight', 'd_rels_weight',
            'd_loop_rel', 'd_loop_edge', 'd_ent_bn_weight', 'd_ent_bn_bias'}
    assert want <= {n[:-len('.npy')] for n in names} and all(n.endswith('.npy') for n in names)
    assert sum(os.path.getsize(a / n) for n in names) <= 64 << 20
    R, rows = 11, 16384               # bench.WORKLOADS['wn18rr'] (40,943 entities, 2 x 86,835 edges: both sampled), DUMP_MAX_ROWS
    shapes = {'all_ent': (rows, 200), 'all_rel': (2 * R, 200), 'd_x': (rows, 100), 'd_ee': (rows, 100), 'd_rel': (2 * R, 100)}
    for n in names:
        x = np.load(a / n)
        assert x.dtype == np.float32 and np.isfinite(x).all(), n
        if n[:-4] in shapes:
            assert x.shape == shapes[n[:-4]], n
    # runs 3 and 4 steps long end on different dropout draws: the outputs differ, the dropout-free all_rel does not
    assert np.allclose(np.load(a / 'all_rel.npy'), np.load(b / 'all_rel.npy'), rtol=1e-6, atol=0)
    assert not np.allclose(np.load(a / 'all_ent.npy'), np.load(b / 'all_ent.npy'))
    c = tmp_path / 'c'
    _bench(c, 3)
    for n in names:
        x, y = np.load(a / n), np.load(c / n)
        scale = float(np.abs(y).max()) or 1.0
        assert x.shape == y.shape and float(np.abs(x - y).max()) <= 1e-5 * scale, n     # same inputs; only summation order may differ


def test_dump_is_the_last_timed_step(tmp_path):
    """In process: bench_layer's dump equals the float64 oracle (oracle.conv_fwd_bwd_big) of the LAST timed step - its
    dropout keep masks regenerated from that step's seed - on the same sampled rows; another step's draws or gradients
    accumulated over steps would be off by far more than the fp32 tolerance."""
    bench = _bench_module()
    import kgc_gcn_b200 as k
    k._lib.lib()
    orc = bench.oracle()
    dev = torch.device('cuda', 0)
    args = SimpleNamespace(steps=3, warmup=2, no_graph=False, no_parity=True)
    res, case = bench.bench_layer(k, orc, 'wn18rr', dev, args, bench.Flusher(dev), with_roofline=False, dump_dir=str(tmp_path))
    assert res['timed_steps'] == 3 and res['launch'] == 'cuda_graph'
    conv = case.conv
    m_in, m_out = conv.dropout_masks(conv._last_seed, case.N)                 # the graph replay rewrites _last_seed
    w = {n: getattr(conv, n).detach() for n in ('loop_weight', 'in_weight', 'out_weight', 'rels_weight', 'loop_rel', 'loop_edge')}
    w['ent_bn.weight'], w['ent_bn.bias'] = conv.ent_bn.weight.detach(), conv.ent_bn.bias.detach()
    truth = orc.conv_fwd_bwd_big(case.x.detach(), case.ei, case.et, case.ee.detach(), case.rl.detach(), w, case.g_ent, case.g_rel,
                                 mask_in=m_in, mask_out=m_out, drop_p=0.1, d_ee_check=case.ee.grad)
    assert truth['d_ee_max_abs_err'] <= bench.PARITY_TOL * truth['d_ee_max_abs']

    def sample(t):
        rows = torch.randperm(t.size(0), generator=torch.Generator().manual_seed(0))[:bench.DUMP_MAX_ROWS].sort().values
        return t[rows.to(t.device)]
    want = {'all_ent': sample(truth['all_ent']), 'all_rel': truth['all_rel'], 'd_x': sample(truth['entity_embedding']),
            'd_rel': truth['relation_embedding']}
    for n in ('loop_weight', 'in_weight', 'out_weight', 'rels_weight', 'loop_rel', 'loop_edge', 'ent_bn.weight', 'ent_bn.bias'):
        want['d_' + n.replace('.', '_')] = truth['conv1.' + n]
    for n, v in want.items():
        got = torch.from_numpy(np.load(tmp_path / (n + '.npy'))).double()
        v = v.detach().double().cpu().reshape(got.shape)
        err = float((got - v).abs().max()) / (float(v.abs().max()) + 1e-300)
        assert err < bench.PARITY_TOL, (n, err)
    # d_ee: the dumped rows are the rows of the gradient the oracle checked above
    assert torch.equal(torch.from_numpy(np.load(tmp_path / 'd_ee.npy')), sample(case.ee.grad).cpu())
