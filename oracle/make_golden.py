"""Generate tests/golden/* by running the UNMODIFIED reference.  TEST INFRASTRUCTURE ONLY.

Needs a checkout of the reference (weilonghu/KGC-GCN), which is not part of this repository:
    KGC_REFERENCE_DIR=<checkout> python oracle/make_golden.py
The reference modules are imported from where they lie through ``oracle/shims`` (four
stand-ins for its absent third-party imports); nothing is copied.  The fixtures are small
(< 2 MB in total), committed, and are what pins ``oracle/mgcn_oracle.py`` and the CUDA path.
"""
import json
import os
import sys
from types import SimpleNamespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.environ.get('KGC_REFERENCE_DIR')
if not REF or not os.path.isfile(os.path.join(REF, 'model.py')):
    sys.exit('oracle/make_golden.py runs the reference: set KGC_REFERENCE_DIR to a checkout of weilonghu/KGC-GCN')
OUT = os.path.join(ROOT, 'tests', 'golden')

sys.path.insert(0, os.path.join(HERE, 'shims'))
sys.path.insert(0, REF)
sys.path.insert(0, HERE)
os.chdir(REF)                     # the reference resolves data/<ds> relative to the cwd (data_loader.py:57)

import data_loader as ref_dl      # noqa: E402  (the reference)
import model as ref_model         # noqa: E402  (the reference)
import main as ref_main           # noqa: E402  (the reference)
import mgcn_oracle as orc         # noqa: E402


def params(**kw):
    base = dict(gcn_in_dim=100, gcn_out_dim=200, gcn_drop=0.3, hidden_drop=0.3, feat_drop=0.3, k_w=10, k_h=20,
                num_filter=200, kernel_size=7, bias=False, lbl_smooth=0.1, batch_size=128)
    base.update(kw)
    return SimpleNamespace(**base)


def npy(t):
    return t.detach().cpu().numpy()


# ---------------------------------------------------------------- A. Toy loader known-answers
def toy_loader():
    dl = ref_dl.DataLoader('Toy', params())
    g = dl.graph
    trip = {k: [{'triple': [int(a) for a in q['triple']], 'label': sorted(int(a) for a in q['label'])} for q in v]
            for k, v in dl.triplets.items()}
    blob = {
        'entity2id': dl.entity2id, 'relation2id': dl.relation2id,
        'num_entity': dl.num_entity, 'num_relation': dl.num_relation, 'num_edge': dl.num_edge,
        'edge_index': g.edge_index.tolist(), 'edge_attr': g.edge_attr.tolist(), 'entity': g.entity.tolist(),
        'edge_norm': [float(v) for v in g.edge_norm.tolist()], 'num_nodes': int(g.num_nodes),
        'triplets': trip,
    }
    # one collated training batch in list order (ls = 0.1: the reference's > 1 label quirk included) and one eval batch
    ds_tr = dl._get_dataset('train', params())
    tr = ds_tr.collate_fn([ds_tr[i] for i in range(len(ds_tr))])
    ds_ev = dl._get_dataset('valid_tail', params())
    ev = ds_ev.collate_fn([ds_ev[i] for i in range(len(ds_ev))])
    np.savez_compressed(os.path.join(OUT, 'toy_batches.npz'), train_triple=npy(tr[0]), train_label=npy(tr[1]),
                        valid_tail_triple=npy(ev[0]), valid_tail_label=npy(ev[1]))
    with open(os.path.join(OUT, 'toy_loader.json'), 'w') as f:
        json.dump(blob, f, indent=1, sort_keys=True)
    return dl


# ---------------------------------------------------------------- B/D. convolution fixtures
def conv_case(name, edge_index, edge_type, N, R, d_in, d_out, seed, with_masks=False, training=True):
    E = edge_type.numel() // 2
    p = orc.conv_params(N, R, E, d_in, d_out, seed=seed)
    gsd = torch.Generator().manual_seed(seed + 1)
    g_ent = torch.randn(N, d_out, generator=gsd)
    g_rel = torch.randn(2 * R, d_out, generator=gsd)
    gamma = torch.rand(d_out, generator=gsd) + 0.5
    beta = torch.randn(d_out, generator=gsd) * 0.1
    rmean = torch.randn(d_out, generator=gsd) * 0.01
    rvar = torch.rand(d_out, generator=gsd) * 0.01 + 0.001
    out = {'edge_index': npy(edge_index), 'edge_type': npy(edge_type), 'N': N, 'R': R,
           'x': npy(p['x']), 'rels': npy(p['rels']), 'edge_embs': npy(p['edge_embs']),
           'g_ent': npy(g_ent), 'g_rel': npy(g_rel), 'training': int(training)}
    for k, v in p['w'].items():
        out['w.' + k] = npy(v)
    out['w.ent_bn.weight'], out['w.ent_bn.bias'] = npy(gamma), npy(beta)
    out['w.ent_bn.running_mean'], out['w.ent_bn.running_var'] = npy(rmean), npy(rvar)

    for dt, tag in ((torch.float64, 'f64'), (torch.float32, 'f32')):
        conv = ref_model.MGCNConv(d_in, d_out, 2 * R, dropout=0.1 if with_masks else 0.0)
        with torch.no_grad():
            for k in ('loop_weight', 'in_weight', 'out_weight', 'rels_weight', 'loop_rel', 'loop_edge'):
                getattr(conv, k).copy_(p['w'][k])
            conv.ent_bn.weight.copy_(gamma)
            conv.ent_bn.bias.copy_(beta)
            conv.ent_bn.running_mean.copy_(rmean)
            conv.ent_bn.running_var.copy_(rvar)
        conv = conv.to(dt)
        conv.train(training)
        x = p['x'].to(dt).requires_grad_(True)
        ee = p['edge_embs'].to(dt).requires_grad_(True)
        rl = p['rels'].to(dt).requires_grad_(True)
        if with_masks:
            # nn.Dropout draws one Bernoulli tensor per call from the global CPU generator; replay the two
            # draws (in_res, then out_res - model.py:103) ahead of time to learn the masks the reference will use.
            torch.manual_seed(seed + 7)
            ones = torch.ones(N, d_out, dtype=dt)
            m_in = torch.nn.functional.dropout(ones, 0.1, True) != 0
            m_out = torch.nn.functional.dropout(ones, 0.1, True) != 0
            torch.manual_seed(seed + 7)
            if tag == 'f64':
                out['mask_in'], out['mask_out'] = npy(m_in).astype(np.uint8), npy(m_out).astype(np.uint8)
            else:
                # the f32 draw consumes the generator differently; store its masks separately
                out['mask_in_f32'], out['mask_out_f32'] = npy(m_in).astype(np.uint8), npy(m_out).astype(np.uint8)
        all_ent, all_rel = conv(x, edge_index, edge_type, None, ee, rl)
        torch.autograd.backward([all_ent, all_rel], [g_ent.to(dt), g_rel.to(dt)])
        out['all_ent.' + tag], out['all_rel.' + tag] = npy(all_ent), npy(all_rel)
        if tag == 'f64':
            out['bn.running_mean_after'] = npy(conv.ent_bn.running_mean)
            out['bn.running_var_after'] = npy(conv.ent_bn.running_var)
        grads = {'x': x.grad, 'edge_embs': ee.grad, 'rels': rl.grad}
        for k in ('loop_weight', 'in_weight', 'out_weight', 'rels_weight', 'loop_rel', 'loop_edge'):
            grads['w.' + k] = getattr(conv, k).grad
        grads['w.ent_bn.weight'], grads['w.ent_bn.bias'] = conv.ent_bn.weight.grad, conv.ent_bn.bias.grad
        for k, v in grads.items():
            out['grad.{}.{}'.format(k, tag)] = npy(v)
        n_in = conv.compute_norm(edge_index[:, :E], N)
        n_out = conv.compute_norm(edge_index[:, E:], N)
        out['norm_in'], out['norm_out'] = npy(n_in), npy(n_out)
    np.savez_compressed(os.path.join(OUT, name + '.npz'), **out)


def synth_graph(N, R, E, seed):
    tri = orc.synthetic_triples(N, R, E, seed)
    g = orc.build_graph(tri, N, R)
    return torch.from_numpy(g['edge_index']), torch.from_numpy(g['edge_attr'][0])


# ---------------------------------------------------------------- C. whole model + predict on Toy
def toy_model(dl):
    prm = params(gcn_in_dim=20, num_filter=2, gcn_drop=0.0, hidden_drop=0.0, feat_drop=0.0, lbl_smooth=0.0)
    torch.manual_seed(1234)
    m = ref_model.MGCN(dl.num_entity, dl.num_relation, dl.num_edge, prm)
    m.conv1.drop.p = 0.0              # MGCNConv's dropout is a ctor default (model.py:49), not a flag
    with torch.no_grad():             # non-trivial BN state and decoder bias so the eval path is exercised
        g = torch.Generator().manual_seed(99)
        m.conv2.bias.copy_(torch.randn(dl.num_entity, generator=g) * 0.1)
        for bn in (m.conv1.ent_bn, m.conv2.bn0, m.conv2.bn1, m.conv2.bn2):
            bn.running_mean.copy_(torch.randn(bn.running_mean.shape, generator=g) * 0.05)
            bn.running_var.copy_(torch.rand(bn.running_var.shape, generator=g) * 0.5 + 0.5)
            bn.weight.copy_(torch.rand(bn.weight.shape, generator=g) + 0.5)
            bn.bias.copy_(torch.randn(bn.bias.shape, generator=g) * 0.1)
    sd = {k: npy(v) for k, v in m.state_dict().items()}
    out = {'sd.' + k: v for k, v in sd.items()}
    graph = dl.graph

    # eval-mode forward on every valid_tail / valid_head query, in list order, float32 and float64
    for mode in ('tail', 'head'):
        qs = dl.triplets['valid_' + mode]
        trip = torch.tensor([q['triple'] for q in qs], dtype=torch.long)
        out['eval.{}.triple'.format(mode)] = npy(trip)
        for dt, tag in ((torch.float32, 'f32'), (torch.float64, 'f64')):
            mm = m.double() if dt == torch.float64 else m.float()
            mm.eval()
            with torch.no_grad():
                sc = mm(trip[:, 0], trip[:, 1], graph)
            out['eval.{}.score.{}'.format(mode, tag)] = npy(sc)
        m.float()

    # the reference's own predict()/evaluate() (main.py:80-135) with batch size 4 (shuffled order is irrelevant to sums)
    torch.manual_seed(5)
    iters = dl.get_data_loaders(4, 0, prm)
    m.float()
    res_t = ref_main.predict(m, iters, graph, 'valid', torch.device('cpu'), mode='tail_batch')
    res_h = ref_main.predict(m, iters, graph, 'valid', torch.device('cpu'), mode='head_batch')
    ev = ref_main.evaluate(m, iters, graph, SimpleNamespace(device=torch.device('cpu')), 'valid')
    metrics = {'tail': {k: float(v) for k, v in res_t.items()}, 'head': {k: float(v) for k, v in res_h.items()},
               'evaluate': {k: float(v) for k, v in ev.items()}}

    # train-mode step (all dropout off): loss + every parameter gradient, float64
    md = m.double()
    md.train()
    qs = dl.triplets['train']
    trip = torch.tensor([q['triple'] for q in qs], dtype=torch.long)
    lab = torch.stack([torch.from_numpy(orc.make_label(q['label'], dl.num_entity)) for q in qs]).double()
    md.zero_grad()
    pred = md(trip[:, 0], trip[:, 1], graph)
    loss = md.loss(pred, lab)
    loss.backward()
    out['train.triple'], out['train.label'] = npy(trip), npy(lab).astype(np.float32)
    out['train.pred.f64'] = npy(pred)
    out['train.loss.f64'] = np.asarray(loss.item())
    for k, v in md.named_parameters():
        out['train.grad.' + k] = npy(v.grad)
    m.float()
    np.savez_compressed(os.path.join(OUT, 'toy_model.npz'), **out)
    with open(os.path.join(OUT, 'toy_metrics.json'), 'w') as f:
        json.dump(metrics, f, indent=1, sort_keys=True)


# ---------------------------------------------------------------- E. filtered-rank fixture (reference formulation)
def rank_case():
    g = torch.Generator().manual_seed(11)
    B, N = 24, 97
    pred = torch.sigmoid(torch.randn(B, N, generator=g) * 3)
    label = (torch.rand(B, N, generator=g) < 0.06).float()
    obj = torch.randint(0, N, (B,), generator=g)
    label[torch.arange(B), obj] = 1.0
    # reference lines main.py:122-126 verbatim semantics through its own predict() body is not callable in isolation;
    # run them through the oracle restatement AND through the reference predict() with a stub model below.

    class Stub(torch.nn.Module):
        def forward(self, sub, rel, graph):
            return pred[sub]

    trip = torch.stack([torch.arange(B), torch.zeros(B, dtype=torch.long), obj], 1)
    iters = {'valid_tail': [(trip, label)]}
    res = ref_main.predict(Stub(), iters, None, 'valid', torch.device('cpu'), mode='tail_batch')
    np.savez_compressed(os.path.join(OUT, 'rank_case.npz'), pred=npy(pred), label=npy(label), obj=npy(obj),
                        **{'res.' + k: np.asarray(float(v)) for k, v in res.items()})


if __name__ == '__main__':
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(1)
    dl = toy_loader()
    g = dl.graph
    et = g.edge_attr[0]
    conv_case('conv_toy_small', g.edge_index, et, dl.num_entity, dl.num_relation, 12, 20, seed=3)
    conv_case('conv_toy_eval', g.edge_index, et, dl.num_entity, dl.num_relation, 12, 20, seed=4, training=False)
    conv_case('conv_toy_full', g.edge_index, et, dl.num_entity, dl.num_relation, 100, 200, seed=5)
    ei, ety = synth_graph(60, 3, 240, seed=21)
    conv_case('conv_synth_hub', ei, ety, 60, 3, 12, 20, seed=6)
    conv_case('conv_synth_masks', ei, ety, 60, 3, 12, 20, seed=8, with_masks=True)
    toy_model(dl)
    rank_case()
    print('golden fixtures written to', OUT)
    for fn in sorted(os.listdir(OUT)):
        print('  {:28s} {:9d} B'.format(fn, os.path.getsize(os.path.join(OUT, fn))))
