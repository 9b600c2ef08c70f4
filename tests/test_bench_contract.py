"""bench.py contract checks that need no GPU: the algorithmic-byte model against SURVEY.md 8(d)'s totals, and the reference
arm (the reference's layer and training step on the host cores, bounded sample) printing ONE JSON line with the contract's
keys - alone on rank 0 when launched with WORLD_SIZE > 1."""
import importlib.util
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location('kgc_bench', os.path.join(ROOT, 'bench.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_algorithmic_bytes_match_survey_totals():
    b = _bench()
    want = {'wn18rr': (121.0e6, 206.5e6), 'fb15k237': (242.0e6, 465.6e6), 'wikidata5m': (22.5e9, 40.8e9)}   # SURVEY.md 8(d)
    for name, (fwd_w, bwd_w) in want.items():
        n, r, e, _ = b.WORKLOADS[name]
        fwd, bwd = b.algorithmic_bytes(n, r, e)
        assert abs(fwd - fwd_w) <= 0.005 * fwd_w and abs(bwd - bwd_w) <= 0.005 * bwd_w, (name, fwd, bwd)
    n, r, e, _ = b.WORKLOADS['wn18rr']
    assert round(sum(b.algorithmic_bytes(n, r, e)) / (2 * e)) == 1886            # bytes per directed edge


def _run_reference(env_extra):
    env = dict(os.environ, **env_extra)
    p = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0'],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600, env=env, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    return [ln for ln in p.stdout.splitlines() if ln.strip()]


def test_reference_arm_prints_one_contract_line():
    lines = _run_reference({'RANK': '0', 'WORLD_SIZE': '1'})
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['metric'] == 'edges/sec GCN fwd+bwd' and d['unit'] == 'edges/s'
    assert d['n_gpus'] == 1 and d['steps'] == 1 and d['higher_is_better'] is True and d['gpu_launches'] == 0
    assert d['timed_steps'] == 1 and d['e2e']['steps'] == 1
    # the default workload is the GPU arm's (Wikidata5M shape); the CPU runs a bounded sample of it and says which
    assert d['config']['workload'] == 'wikidata5m_shape' and 'divided by 64' in d['config']['sample']
    e_sample = 20614279 // 64
    assert d['value'] > 0 and abs(d['value'] - 2 * e_sample / (d['ms_per_step'] * 1e-3)) <= 1e-6 * d['value']
    cb = d['cpu_baseline']
    assert cb['kind'] in ('reference', 'port') and cb['cores'] >= 1 and cb['value'] == d['value'] and 'divided by 64' in cb['sample']
    # same scopes as the GPU arm: value = the layer's forward + backward, e2e = the whole training step (slower)
    e = d['e2e']
    assert e['unit'] == 'edges/s' and e['h2d_bytes_per_step'] == 0 and e['d2h_bytes_per_step'] == 0
    assert 0 < e['value'] < d['value'] and abs(e['value'] - 2 * e_sample / (e['ms_per_step'] * 1e-3)) <= 1e-6 * e['value']


def test_reference_bytecode_is_the_reference():
    """oracle/_ref (built by oracle/build_ref.py from the reference checkout KGC_REFERENCE_DIR names) imports as the
    reference's own modules; the port and the unmodified reference give the same layer outputs on a small graph (the golden
    fixtures pin the same thing; this checks the artefact bench.py --impl reference actually runs)."""
    import pytest
    import torch
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import build_ref
    if os.environ.get('KGC_REFERENCE_DIR'):
        assert build_ref.build_ref()
    ref = build_ref.load_reference()
    if ref is None:
        pytest.skip('oracle/_ref was not built (set KGC_REFERENCE_DIR to a checkout of the reference)')
    import mgcn_oracle as orc
    ref_model = ref[0]
    N, R, E = 50, 3, 200
    tri = orc.synthetic_triples(N, R, E, 1)
    g = orc.build_graph(tri, N, R)
    torch.manual_seed(0)
    conv = ref_model.MGCNConv(8, 12, 2 * R, dropout=0.0).double()
    p = orc.conv_params(N, R, E, 8, 12, seed=2)
    ei, et = torch.from_numpy(g['edge_index']), torch.from_numpy(g['edge_attr'][0])
    ent, rel = conv(p['x'].double(), ei, et, None, p['edge_embs'].double(), p['rels'].double())
    w = {k: getattr(conv, k).detach() for k in ('loop_weight', 'in_weight', 'out_weight', 'rels_weight', 'loop_rel', 'loop_edge')}
    w.update({'ent_bn.weight': conv.ent_bn.weight.detach(), 'ent_bn.bias': conv.ent_bn.bias.detach(),
              'ent_bn.running_mean': torch.zeros(12).double(), 'ent_bn.running_var': torch.ones(12).double()})
    ent_o, rel_o, _ = orc.conv_forward(p['x'].double(), ei, et, p['edge_embs'].double(), p['rels'].double(), w, training=True)
    assert float((ent.detach() - ent_o).abs().max()) < 1e-12 and float((rel.detach() - rel_o).abs().max()) < 1e-12


def test_reference_arm_other_ranks_exit_quietly():
    assert _run_reference({'RANK': '1', 'WORLD_SIZE': '2', 'LOCAL_RANK': '1'}) == []


@pytest.mark.parametrize('extra', [['--steps', '0'], ['--impl', 'reference', '--dump-outputs', 'out'],
                                   ['--dump-outputs', 'out', '--gpus', '2']])
def test_bad_arguments_are_refused_before_any_work(extra, tmp_path):
    """--steps below 1, and --dump-outputs where there is no single-GPU timed layer step to dump, end with a usage error."""
    env = dict(os.environ, RANK='0', WORLD_SIZE='2' if '--gpus' in extra else '1')
    p = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + extra, stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                       text=True, timeout=120, env=env, cwd=str(tmp_path))
    assert p.returncode == 2 and p.stdout == '' and 'error' in p.stderr
    assert not os.path.exists(str(tmp_path / 'out'))
