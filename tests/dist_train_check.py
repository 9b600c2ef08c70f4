"""Multi-GPU check of the sharded training step, launched by tests/test_gpu_dist_train.py as
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port P tests/dist_train_check.py
One process per GPU.  Every rank also runs the single-GPU MGCN on the whole graph.  (1) Without dropout, on the hybrid cut
(peer memory) and on the edge-balanced partition over NCCL: one eager sharded loss_sparse against MGCN.loss_sparse (loss,
every parameter gradient, ClipAdam's gradient norm); on peer memory also 5 graphed steps against 5 single-GPU graphed
steps.  (2) With every dropout on (hybrid cut): replicated parameters stay bit-equal across ranks, graph replays equal eager
steps on the same dropout streams, two runs are bit-identical, and full_state_dict() loads into a single-GPU MGCN.
(3) The sampled objectives, unequal query ids and graph capture on NCCL are rejected."""
import copy
import os
import sys
from types import SimpleNamespace

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'oracle'))
import mgcn_oracle as orc          # noqa: E402  (synthetic inputs only)
import kgc_gcn_b200 as k           # noqa: E402
from bench import synthetic_query_set   # noqa: E402

B, STEPS = 128, 5
# gradients that are zero in exact arithmetic: the BatchNorm that follows (bn1 after the bias-free convolution, bn2 after fc,
# in training mode) removes any scale / shift of its input, so only rounding noise is left; they are compared against the
# gradient scale of the weight they feed instead of their own
STRUCTURAL_ZERO = {'conv2.bn0.weight': 'conv2.conv_e.weight', 'conv2.bn0.bias': 'conv2.conv_e.weight',
                   'conv2.fc.bias': 'conv2.fc.weight'}


def params(drop):
    return SimpleNamespace(gcn_in_dim=100, gcn_out_dim=200, gcn_drop=drop, hidden_drop=drop, feat_drop=drop, k_w=10, k_h=20,
                           num_filter=200, kernel_size=7, bias=False, lbl_smooth=0.1, batch_size=B)


def rel(a, b):
    return abs(a - b) / max(abs(b), 1e-30)


def same_on_all_ranks(t):
    r = t.detach().clone()
    dist.broadcast(r, src=0)
    return torch.equal(r, t.detach())


def seed_modules(model):
    return [m for m in model.modules() if hasattr(m, '_drop_seed')]


def one_rank_checks(report, part, N, R, E, qs, batches, host_model, sharded):
    """One rank: eager steps with every dropout on, full_state_dict and the rejections that do not need peer memory."""
    prm = params(0.3)
    ds = k.KBDataset(qs, N, prm, training=True)
    sh, opt = sharded(host_model(prm, 0.1), part)
    losses = []
    for q in batches:
        opt.zero_grad(set_to_none=True)
        loss = sh.loss_sparse(q, ds)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert all(np.isfinite(losses)), losses
    sd = sh.full_state_dict()
    single = k.MGCN(N, R, E, prm)
    single.load_state_dict(sd, strict=True)
    assert torch.equal(single.entity_embedding.detach()[part.owned_nodes.cpu()], sh.entity_embedding.detach().cpu())
    assert torch.equal(single.edge_embeddings.detach()[part.owned_eids.cpu()], sh.edge_embeddings.detach().cpu())
    try:
        k.GraphedTrainStep(sh, opt, None, ds, B, negatives=16)
        raise AssertionError('negatives= on a sharded model was not rejected')
    except ValueError as exc:
        assert 'sampled' in str(exc), exc
    dist.barrier()
    print('DIST_TRAIN_OK', {t: {kk: float('{:.2e}'.format(v)) for kk, v in e.items()} for t, e in report.items()},
          'losses', losses)
    dist.destroy_process_group()


def main():
    rank, world = int(os.environ['RANK']), int(os.environ['WORLD_SIZE'])
    dev = torch.device('cuda', int(os.environ.get('LOCAL_RANK', rank)))
    torch.cuda.set_device(dev)
    dist.init_process_group('nccl', device_id=dev)
    N, R, E = 3000 * world + 1, 6, 9000 * world
    tri = orc.synthetic_triples(N, R, E, 77)
    g = orc.build_graph(tri, N, R)
    graph = k.GraphData(edge_index=torch.from_numpy(g['edge_index']), edge_attr=torch.from_numpy(g['edge_attr']))
    graph.entity = torch.from_numpy(g['entity'])
    graph.edge_norm = torch.from_numpy(g['edge_norm'])
    graph.num_nodes = N
    graph.to(dev)
    qs = synthetic_query_set(k, tri, R)
    batches = [np.random.default_rng(100 + i).choice(len(qs), B, replace=False) for i in range(STEPS)]
    report = {}

    def host_model(prm, layer_drop):
        torch.manual_seed(0)
        m = k.MGCN(N, R, E, prm)                                   # on the host: only shards go to the device
        m.conv1.drop.p = layer_drop
        return m.train()

    def sharded(host, part, seed=1):
        torch.manual_seed(seed)                                    # the same dropout streams on every rank
        sh = host.shard(part).train()
        opt = k.ClipAdam(sh.parameters(), lr=1e-3, max_norm=1.0, partition=part, sharded=sh.sharded_parameters())
        return sh, opt

    # ---- (1) no dropout: against the single-GPU model
    prm = params(0.0)
    ds = k.KBDataset(qs, N, prm, training=True)
    # one rank: the edge-balanced partition over NCCL only (peer memory, and so the hybrid cut and graph capture, needs two)
    configs = (('hybrid', 'auto'), ('edges', False)) if world > 1 else (('edges', False),)
    for balance, p2p in configs:
        tag = '{}/{}'.format(balance, 'p2p' if p2p else 'nccl')
        part = k.GraphPartition(g['edge_index'], g['edge_attr'][0], N, 2 * R + 1, world, rank, dev, balance=balance, p2p=p2p)
        host = host_model(prm, 0.0)
        ref = copy.deepcopy(host).to(dev).train()
        sh, opt = sharded(host, part)
        opt_ref = k.ClipAdam(ref.parameters(), lr=1e-3, max_norm=1.0)
        loss_ref = ref.loss_sparse(batches[0], ds, graph)
        loss_ref.backward()
        loss = sh.loss_sparse(batches[0], ds)
        loss.backward()
        e = {'loss': rel(loss.item(), loss_ref.item())}
        assert e['loss'] < 1e-6, (tag, e)
        ref_p = dict(ref.named_parameters())
        owned = {'entity_embedding': part.owned_nodes, 'conv2.bias': part.owned_nodes, 'edge_embeddings': part.owned_eids}
        for name, prm_ in sh.named_parameters():
            want = ref_p[name].grad
            if name in owned:
                err = float((prm_.grad - want[owned[name]]).abs().max()) / (float(want.abs().max()) + 1e-30)
            else:
                scale = ref_p[STRUCTURAL_ZERO[name]].grad if name in STRUCTURAL_ZERO else want
                err = float((prm_.grad - want).abs().max()) / (float(scale.abs().max()) + 1e-30)
                assert same_on_all_ranks(prm_.grad), (tag, name, 'replicated gradient differs across ranks')
            assert err < 2e-5, (tag, name, err)
            e['d_' + name] = err
        opt.step()
        opt_ref.step()
        e['grad_norm'] = rel(float(opt.last_grad_norm), float(opt_ref.last_grad_norm))
        assert e['grad_norm'] < 1e-6, (tag, e)
        if p2p:
            host = host_model(prm, 0.0)
            ref = copy.deepcopy(host).to(dev).train()
            sh, opt = sharded(host, part)
            step_ref = k.GraphedTrainStep(ref, k.ClipAdam(ref.parameters(), lr=1e-3, max_norm=1.0), graph, ds, B,
                                          fused_loss=True)
            step = k.GraphedTrainStep(sh, opt, None, ds, B, fused_loss=True)
            for i, q in enumerate(batches):
                a, b = float(step(q).item()), float(step_ref(q).item())
                e['graphed_%d' % i] = rel(a, b)
                assert e['graphed_%d' % i] < 1e-4, (tag, i, a, b)
            del step, step_ref
        else:
            try:
                k.GraphedTrainStep(sh, opt, None, ds, B, fused_loss=True)
                raise AssertionError('capture on NCCL was not rejected')
            except ValueError as exc:
                assert 'NCCL' in str(exc), exc
        report[tag] = e
        del ref, sh, opt, opt_ref
        torch.cuda.empty_cache()

    if world == 1:
        one_rank_checks(report, part, N, R, E, qs, batches, host_model, sharded)
        return

    # ---- (2) every dropout on, hybrid cut on peer memory
    prm = params(0.3)
    ds = k.KBDataset(qs, N, prm, training=True)
    part = k.GraphPartition(g['edge_index'], g['edge_attr'][0], N, 2 * R + 1, world, rank, dev, balance='hybrid')

    def graphed_run():
        sh, opt = sharded(host_model(prm, 0.1), part)
        step = k.GraphedTrainStep(sh, opt, None, ds, B, fused_loss=True)
        losses = [step(q).item() for q in batches]
        return losses, sh, opt, step

    losses1, sh1, opt1, step1 = graphed_run()
    for name, prm_ in sh1.named_parameters():
        if all(prm_ is not t for t in sh1.sharded_parameters()):
            assert same_on_all_ranks(prm_), ('replicated parameter differs across ranks', name)
    for name, buf in sh1.named_buffers():
        assert same_on_all_ranks(buf), ('replicated buffer differs across ranks', name)
    del step1
    losses2, sh2, opt2, step2 = graphed_run()
    assert losses1 == losses2, (losses1, losses2)
    for (n1, a), (_, b) in zip(sh1.state_dict().items(), sh2.state_dict().items()):
        assert torch.equal(a, b), ('two runs differ', n1)

    # graph replays against eager steps: a second sharded model takes the graphed model's state after its first step and
    # its dropout streams before every replay (ConvE's torch-generator dropout is off here: its stream is the generator's)
    prm_e = params(0.3)
    prm_e.hidden_drop = 0.0
    ds_e = k.KBDataset(qs, N, prm_e, training=True)
    sh_g, opt_g = sharded(host_model(prm_e, 0.1), part)
    sh_e, opt_e = sharded(host_model(prm_e, 0.1), part)
    step_g = k.GraphedTrainStep(sh_g, opt_g, None, ds_e, B, fused_loss=True)
    step_g(batches[0])
    sh_e.load_state_dict(sh_g.state_dict())
    opt_e.load_state_dict(opt_g.state_dict())
    for q in batches[1:]:
        seeds = [m._drop_seed.clone() for m in seed_modules(sh_g)]
        lg = step_g(q).item()
        for m, s in zip(seed_modules(sh_e), seeds):
            m._drop_seed.copy_(s)
            m._drop_seeded = True
        opt_e.zero_grad(set_to_none=True)
        le = sh_e.loss_sparse(q, ds_e)
        le.backward()
        opt_e.step()
        assert lg == le.item(), (lg, le.item())
    for (n1, a), (_, b) in zip(sh_g.state_dict().items(), sh_e.state_dict().items()):
        assert torch.equal(a, b), ('graph replay differs from the eager step', n1)
    del step_g

    sd = sh1.full_state_dict()
    if rank == 0:
        single = k.MGCN(N, R, E, prm)
        single.load_state_dict(sd, strict=True)
        assert torch.equal(single.entity_embedding.detach()[part.owned_nodes.cpu()], sh1.entity_embedding.detach().cpu())
        assert torch.equal(single.conv2.fc.weight.detach(), sh1.conv2.fc.weight.detach().cpu())
    else:
        assert sd is None

    # ---- (3) rejections
    try:
        k.GraphedTrainStep(sh1, opt1, None, ds, B, negatives=16)
        raise AssertionError('negatives= on a sharded model was not rejected')
    except ValueError as exc:
        assert 'sampled' in str(exc), exc
    try:
        sh1.loss_sampled(batches[0], ds, None, 16)
        raise AssertionError('loss_sampled on a sharded model was not rejected')
    except ValueError as exc:
        assert 'sampled' in str(exc), exc
    step = k.GraphedTrainStep(sh1, opt1, None, ds, B, fused_loss=True)
    try:
        step(batches[rank])
        raise AssertionError('unequal query ids were not rejected')
    except ValueError as exc:
        assert 'same query ids' in str(exc), exc
    ctx = part.p2p(100)
    ctx.check()
    dist.barrier()
    if rank == 0:
        print('DIST_TRAIN_OK', {t: {kk: float('{:.2e}'.format(v)) for kk, v in e.items()} for t, e in report.items()},
              'losses', losses1)
    dist.destroy_process_group()


if __name__ == '__main__':
    main()
