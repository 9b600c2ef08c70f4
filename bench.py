"""bench.py - headline benchmark of the M-GCN hot path on B200 (contract: see the task brief / DESIGN.md section 6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload wn18rr|fb15k237|wikidata5m]
                    [--dump-outputs DIR]

Metric (BASELINE.json): edges/sec of the relation-aware graph convolution, forward + backward, where an "edge" is one
directed edge of edge_index (2E per pass; SURVEY.md 8(d)).  ONE JSON line on stdout.

Workload.  N = 1: the Wikidata5M-shape graph (the largest configuration of BASELINE.json that fits one B200 and the one
its HBM target is about); the WN18RR and FB15k-237 shapes are measured in the same run and reported under ``workloads``.
N > 1: STRONG scaling of the same Wikidata5M-shape graph over the dst-partitioned layer (SURVEY.md 8(e)); every rank also
runs the single-GPU layer on the whole graph once, outside the timed region, and the line carries the parity of the
partitioned outputs and gradients against it (rc != 0 when it fails).  ``KGC_BENCH_WEAK=1`` keeps round 1's weak-scaling
mode (N x the named shape).

  value        MGCNConv.forward + backward with every input resident in HBM (CUDA-event time, L2 flushed between steps,
               dropout p = 0.1 drawn inside the timed region, one CUDA-graph replay per step)
  e2e          the same metric through the reference-facing API for a whole training step (host query ids -> model ->
               loss -> backward -> clip -> Adam -> loss.item()), host<->device copies inside the timed region
  roofline     the dominant aggregation kernel timed alone: SURVEY.md 8(d) algorithmic bytes / CUDA-event time vs the
               measured HBM peak; ``passes`` = the whole forward / backward aggregation (every launch, fix-ups included)
               against 8(d)'s per-pass bytes; ``traffic`` from the committed ncu capture (profiles/r02_ncu_traffic.json)
  parity       max-norm-relative error of every output and gradient against the float64 restatement of the reference
               (oracle.conv_fwd_bwd_big, run on the same GPU as the CHECKER, outside every timed region)
  cpu_baseline the reference's own layer on the host cores (oracle/_ref = the unmodified reference when it was built,
               else the pinned port), on a bounded sample of the workload
  aux          filtered-rank queries/sec of the fused tcgen05 scorer (second half of BASELINE.json's metric); N > 1: the
               entity table sharded over the ranks, integer counts all-reduced, sharded == unsharded asserted in-run
`--impl reference` times the reference's CPU implementation of the same two scopes (layer fwd+bwd = value, full training
step = e2e) on a bounded sample of the same workload; rank 0 only.
`--dump-outputs DIR` (N = 1) writes what the last timed layer step computed to DIR/<name>.npy (see dump_outputs), so that
two builds can be compared output for output.  bench.py writes nothing into the source tree.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True         # the source tree may be read-only; nothing is cached in it

WORKLOADS = {
    # name: (N entities, R relations, E train triples, synthetic seed)        SURVEY.md 8(d)
    'wn18rr': (40943, 11, 86835, 0),
    'fb15k237': (14541, 237, 272115, 1),
    'wikidata5m': (4594485, 822, 20614279, 2),
}
D_IN, D_OUT, BATCH = 100, 200, 128
# the reference's formulation needs ~80 GB of host RAM at the Wikidata5M shape (SURVEY.md 8(d)); its CPU legs run on the
# same generator with the node and triple counts divided by this factor (relations kept) and say so in `sample`
CPU_SAMPLE_DIV = {'wn18rr': 1, 'fb15k237': 1, 'wikidata5m': 64}
PARITY_TOL = 2e-5          # max-norm-relative, fp32 kernels vs float64 truth (tests/test_gpu_conv.py uses the same bar)


def params_ns():
    from types import SimpleNamespace
    return SimpleNamespace(gcn_in_dim=D_IN, gcn_out_dim=D_OUT, gcn_drop=0.3, hidden_drop=0.3, feat_drop=0.3, k_w=10,
                           k_h=20, num_filter=200, kernel_size=7, bias=False, lbl_smooth=0.1, batch_size=BATCH)


def oracle():
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import mgcn_oracle
    return mgcn_oracle


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return p, float(p['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    # B200_PROFILING.md fallbacks
    return {'bf16_tflops': 1600.0, 'bf16_tflops_sustained': 1400.0}, 6650.0, 'fallback (B200_PROFILING.md)'


def ncu_traffic(workload, kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture of this bench
    command (profiles/r02_ncu_traffic.json, written by profiles/summarize_traffic.py); None when not captured."""
    path = os.path.join(ROOT, 'profiles', 'r02_ncu_traffic.json')
    try:
        with open(path) as f:
            return json.load(f).get(workload, {}).get(kernel)
    except (OSError, ValueError):
        return None


def algorithmic_bytes(N, R, E, D=D_IN):
    """SURVEY.md 8(d): compulsory traffic, each tensor once, fp32, int32 indices."""
    T = 2 * R + 1
    fwd = 2 * E * (4 * D + 12) + 2 * N * (4 * D + 4) + N * 4 * D + T * 4 * D
    bwd = 2 * E * (8 * D + 12) + 2 * N * 4 * D + N * 4 * D + N * 4 * D + 2 * T * 4 * D
    return fwd, bwd


# ------------------------------------------------------------------------------------------------ synthetic tensors
_M32 = 0xFFFFFFFF


def _mix32(h):
    """lowbias32 on int64 tensors holding values in [0, 2^32) (products wrap in two's complement; the low 32 bits are exact)."""
    h = ((h ^ (h >> 16)) * 0x7FEB352D) & _M32
    h = ((h ^ (h >> 15)) * 0x846CA68B) & _M32
    return h ^ (h >> 16)


def synth_rows(row_ids, D, bound, seed, chunk=1 << 20):
    """[len(row_ids), D] float32 uniform in [-bound, bound): a pure function of (seed, row id, column), so that every rank
    of a partitioned run can build exactly its rows of a tensor that is never materialised whole on the host (the
    Wikidata5M-shape edge table is 16.5 GB).  ``row_ids``: int64 tensor on the target device."""
    n = int(row_ids.numel())
    out = torch.empty((n, D), dtype=torch.float32, device=row_ids.device)
    cols = torch.arange(D, dtype=torch.int64, device=row_ids.device)
    salt = _mix32(torch.tensor([(seed * 0x9E3779B1 + 0x85EBCA6B) & _M32], dtype=torch.int64, device=row_ids.device))
    for a in range(0, n, chunk):
        idx = row_ids[a:a + chunk, None] * D + cols
        h = _mix32((idx & _M32) ^ _mix32(((idx >> 32) + salt) & _M32))
        out[a:a + chunk] = (h.to(torch.float32) * (2.0 / 4294967296.0) - 1.0) * bound
    return out


def xavier_bound(rows, cols):
    return float(np.sqrt(6.0 / (rows + cols)))


def small_weights(R, seed=0):
    """The replicated parameters of MGCNConv (utils.get_param: xavier-uniform), CPU generator."""
    g = torch.Generator().manual_seed(seed)

    def xav(shape):
        return torch.empty(*shape).uniform_(-xavier_bound(*shape), xavier_bound(*shape), generator=g)
    w = {name: xav((D_IN, D_OUT)) for name in ('loop_weight', 'in_weight', 'out_weight', 'rels_weight')}
    w['loop_rel'], w['loop_edge'] = xav((1, D_IN)), xav((1, D_IN))
    w['rels'] = xav((2 * R, D_IN))
    w['g_rel'] = torch.randn(2 * R, D_OUT, generator=g)
    return w


class ClockSampler(object):
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe).  In-process NVML (a 5 ms
    poll on a thread: a 100 ms timed region on 8 ranks still gets samples); `nvidia-smi -lms 100` when NVML cannot be loaded."""
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
    NAMES = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']

    def __init__(self, index):
        self.rows, self.proc, self.index, self.thread, self.stop, self.source = [], None, index, None, False, None

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:                                               # the CUDA device's own UUID: immune to CUDA_VISIBLE_DEVICES renumbering
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            return pynvml, pynvml.nvmlDeviceGetHandleByUUID(('GPU-' + uuid).encode())
        except Exception:
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.index)

    def _poll(self, nv, h):
        bits = [(nv.nvmlClocksEventReasonHwSlowdown, 0), (nv.nvmlClocksEventReasonHwThermalSlowdown, 1),
                (nv.nvmlClocksEventReasonSwThermalSlowdown, 2), (nv.nvmlClocksEventReasonSwPowerCap, 3)]
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        while True:
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                self.rows.append([str(sm), str(mx), ''] + ['Active' if r & b else 'Not Active' for b, _ in bits])
            except Exception:
                pass
            if self.stop:
                break
            time.sleep(0.005)

    def __enter__(self):
        try:
            nv, h = self._nvml_handle()
            self.thread = threading.Thread(target=self._poll, args=(nv, h), daemon=True)
            self.thread.start()
            self.source = 'nvml'
            return self
        except Exception:
            self.thread = None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
            self.source = 'nvidia-smi'
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def __exit__(self, *a):
        if self.source == 'nvml':
            self.stop = True
            self.thread.join(timeout=1.0)
        elif self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        for r in list(self.rows):
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(self.NAMES, r[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable'], 'samples': 0}
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(max(mx)), 'reasons': sorted(reasons), 'samples': len(sm),
                'source': self.source}


def synthetic_query_set(k, tri, R):
    """(s, r) -> objects grouping of the train triples in both directions (data_loader.py:86-102) as the CSR query set the
    loader's native ingest produces - vectorised (the Wikidata5M shape has 41 M (query, object) pairs)."""
    s, r, o = tri[:, 0], tri[:, 1], tri[:, 2]
    keys = np.concatenate([s * (2 * R) + r, o * (2 * R) + (r + R)])
    objs = np.concatenate([o, s])
    order = np.lexsort((objs, keys))
    keys, objs = keys[order], objs[order]
    keep = np.ones(keys.shape[0], dtype=bool)
    keep[1:] = (keys[1:] != keys[:-1]) | (objs[1:] != objs[:-1])
    keys, objs = keys[keep], objs[keep]
    first = np.ones(keys.shape[0], dtype=bool)
    first[1:] = keys[1:] != keys[:-1]
    starts = np.nonzero(first)[0]
    ptr = np.concatenate([starts, [keys.shape[0]]]).astype(np.int64)
    qk = keys[starts]
    triples = np.stack([qk // (2 * R), qk % (2 * R), np.full_like(qk, -1)], 1).astype(np.int64)
    from kgc_gcn_b200.data_loader import QuerySet
    return QuerySet(triples, ptr, objs.astype(np.int32), train=True)


# ------------------------------------------------------------------------------------------------ CPU arms
def cpu_sample_shape(workload):
    N, R, E, seed = WORKLOADS[workload]
    div = CPU_SAMPLE_DIV[workload]
    return max(N // div, 64), R, max(E // div, 256), seed, div


def _sample_note(workload, N, R, E, div):
    if div == 1:
        return 'whole {}-shape graph (N={}, R={}, E={})'.format(workload, N, R, E)
    return ('{}-shape generator with nodes and triples divided by {} (N={}, R={}, E={}): the reference formulation needs '
            '~80 GB of host RAM at the full shape'.format(workload, div, N, R, E))


def reference_cpu_legs(workload, steps, warmup, budget_s, want_step=True):
    """The reference's CPU implementation of the path on a bounded sample of ``workload``: (a) MGCNConv forward +
    backward (model.py:82-118 + autograd; the scope of `value`), (b) the whole training step (main.py:57-71 incl. the
    host label build of data_loader.py:34-51; the scope of `e2e`).  Runs the UNMODIFIED reference from oracle/_ref
    (byte-compiled by oracle/build_ref.py) through oracle/shims when present (kind = "reference"), else the pinned port
    oracle/mgcn_oracle.py (kind = "port").  Returns dict(kind, cores, N, R, E, div, layer_s, step_s, n_layer, n_step)."""
    orc = oracle()
    import build_ref
    ref = build_ref.load_reference()
    torch.set_num_threads(os.cpu_count() or 1)
    N, R, E, seed, div = cpu_sample_shape(workload)
    torch.manual_seed(0)
    tri = orc.synthetic_triples(N, R, E, seed)
    g = orc.build_graph(tri, N, R)
    prm = params_ns()
    ei, ea = torch.from_numpy(g['edge_index']), torch.from_numpy(g['edge_attr'])
    gen = torch.Generator().manual_seed(1)
    g_ent, g_rel = torch.randn(N, D_OUT, generator=gen), torch.randn(2 * R, D_OUT, generator=gen)
    if ref is not None:
        ref_model, ref_dl, _ = ref
        from torch_geometric.data import Data                       # oracle/shims
        data = Data(edge_index=ei, edge_attr=ea)
        data.entity, data.num_nodes, data.edge_norm = torch.arange(N), N, torch.from_numpy(g['edge_norm'])
        model = ref_model.MGCN(N, R, E, prm)
        queries = synthetic_queries_list(tri, R)
        ds = ref_dl.KBDataset(queries, N, prm, training=True)

        def layer():
            for p_ in model.parameters():
                p_.grad = None
            ent, rel = model.conv1(model.entity_embedding, data.edge_index, ea[0], data.edge_norm, model.edge_embeddings,
                                   model.relation_embedding)
            torch.autograd.backward([ent, rel], [g_ent, g_rel])

        def batch(qid):
            return ds.collate_fn([ds[int(i)] for i in qid])

        def fwd(trip):
            return model(trip[:, 0], trip[:, 1], data)
        loss_fn = model.loss
    else:
        model = orc.OracleMGCN(N, R, E, prm)
        queries = synthetic_queries_list(tri, R)
        w = {name: getattr(model.conv1, name) for name in ('loop_weight', 'in_weight', 'out_weight', 'rels_weight',
                                                           'loop_rel', 'loop_edge')}
        w.update({'ent_bn.weight': model.conv1.ent_bn.weight, 'ent_bn.bias': model.conv1.ent_bn.bias,
                  'ent_bn.running_mean': model.conv1.ent_bn.running_mean, 'ent_bn.running_var': model.conv1.ent_bn.running_var})

        def layer():
            m_in = torch.empty(N, D_OUT).bernoulli_(0.9)
            m_out = torch.empty(N, D_OUT).bernoulli_(0.9)
            orc.conv_fwd_bwd(model.entity_embedding.detach(), ei, ea[0], model.edge_embeddings.detach(),
                             model.relation_embedding.detach(), {k_: v.detach() for k_, v in w.items()}, g_ent, g_rel,
                             mask_in=m_in, mask_out=m_out)

        def batch(qid):
            trip, lab = orc.make_batch(queries, qid, N, prm.lbl_smooth, True)
            return torch.from_numpy(trip), torch.from_numpy(lab)

        def fwd(trip):
            return model(trip[:, 0], trip[:, 1], ei, ea[0])
        loss_fn = torch.nn.functional.binary_cross_entropy
    model.train()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    rng = np.random.default_rng(0)

    def train_step():
        qid = rng.integers(0, len(queries), BATCH)
        trip, lab = batch(qid)                                      # KBDataset + collate (data_loader.py:25-51)
        opt.zero_grad()
        loss = loss_fn(fwd(trip), lab)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
        opt.step()
        return loss.item()

    def timed(fn, n_warm, n_steps, budget):
        times, t_end = [], time.time() + (budget if budget is not None else float('inf'))
        for i in range(n_warm + n_steps):
            t0 = time.perf_counter()
            fn()
            if i >= n_warm:
                times.append(time.perf_counter() - t0)
            if len(times) >= 2 and time.time() > t_end:
                break
        return times
    # at least one untimed call per leg: the first one pays for first-touch allocation and thread-pool start-up, which
    # would otherwise make the layer alone (timed first) look slower than the training step that contains it
    warmup = max(1, warmup)
    lt = timed(layer, warmup, steps, budget_s)
    st = timed(train_step, warmup, steps, budget_s) if want_step else []
    return {'kind': 'reference' if ref is not None else 'port', 'cores': torch.get_num_threads(), 'N': N, 'R': R, 'E': E,
            'div': div, 'layer_s': float(np.mean(lt)), 'n_layer': len(lt),
            'step_s': float(np.mean(st)) if st else None, 'n_step': len(st)}


def synthetic_queries_list(tri, R):
    """The reference's list-of-dicts query form (data_loader.py:98-102) for the CPU legs (small samples only)."""
    from collections import OrderedDict
    known = OrderedDict()
    for s, r, o in tri.tolist():
        known.setdefault((s, r), set()).add(o)
        known.setdefault((o, r + R), set()).add(s)
    return [{'triple': (s, r, -1), 'label': sorted(v), 'sub_samp': 1} for (s, r), v in known.items()]


def cpu_baseline_entry(legs, workload):
    impl = 'the UNMODIFIED reference (oracle/_ref bytecode of model.py through oracle/shims)' if legs['kind'] == 'reference' \
        else 'oracle port (oracle/mgcn_oracle.py, reference op order)'
    return {'value': 2 * legs['E'] / legs['layer_s'], 'unit': 'edges/s', 'cores': legs['cores'], 'kind': legs['kind'],
            'sample': '{}: MGCNConv forward + backward, fp32, dropout p=0.1 drawn per step, mean of {} steps, {:.3f} s/step; {}'
                      .format(impl, legs['n_layer'], legs['layer_s'], _sample_note(workload, legs['N'], legs['R'], legs['E'], legs['div']))}


def run_reference(args, rank, world):
    """Reference arm (rank 0 only): value = the reference's layer fwd+bwd on the host cores - the SAME scope as our
    `value`; e2e.value = its whole training step - the same scope as our `e2e`."""
    if rank != 0:
        return
    workload = args.workload or 'wikidata5m'
    legs = reference_cpu_legs(workload, args.steps, args.warmup, budget_s=None)
    N, R, E, _ = WORKLOADS[workload]
    val = 2 * legs['E'] / legs['layer_s']
    e2e_val = 2 * legs['E'] / legs['step_s']
    base = cpu_baseline_entry(legs, workload)
    line = {
        'impl': 'reference', 'metric': 'edges/sec GCN fwd+bwd', 'value': val, 'unit': 'edges/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'timed_steps': legs['n_layer'], 'warmup': max(1, args.warmup), 'ms_per_step': 1e3 * legs['layer_s'],
        'higher_is_better': True,
        'scaling': 'strong' if (world > 1 and not os.environ.get('KGC_BENCH_WEAK')) else 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': workload + '_shape', 'N': N, 'R': R, 'E': E, 'd_in': D_IN, 'd_out': D_OUT, 'batch': BATCH,
                   'scope': 'value = MGCNConv forward + backward on the host CPU (same scope as the GPU arm\'s value); '
                            'e2e = full training step on the host CPU (same scope as the GPU arm\'s e2e)',
                   'sample': _sample_note(workload, legs['N'], legs['R'], legs['E'], legs['div'])},
        'cpu_baseline': base,
        'e2e': {'value': e2e_val, 'unit': 'edges/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0,
                'ms_per_step': 1e3 * legs['step_s'], 'steps': legs['n_step'],
                'scope': 'label build (data_loader.py:34-51), model forward, BCE, backward, clip_grad_norm_, Adam, loss.item() '
                         '(main.py:57-71) on the host CPU'},
        'gpu_launches': 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------------ our arm
def time_kernel(fn, flush, iters=20, warm=3):
    for _ in range(warm):
        fn()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for a, b in ev:
        flush()
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    return float(np.mean([a.elapsed_time(b) for a, b in ev]))


class Flusher(object):
    def __init__(self, dev):
        self.buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        self.src = torch.zeros(64 << 20, dtype=torch.float32, device=dev)

    def __call__(self):
        # write a buffer larger than L2 (126 MB), then stream a second one through it so that the dirty lines are
        # written back BEFORE the timed region starts (otherwise their eviction is charged to the timed kernel)
        self.buf.zero_()
        self.src.sum()


class LayerCase(object):
    """One workload on this rank: graph, parameters (device-generated), the layer and a fwd+bwd step."""

    def __init__(self, k, orc, workload, dev, world=1, rank=0, scale=1):
        self.k, self.workload, self.dev, self.world, self.rank = k, workload, dev, world, rank
        N1, R, E1, seed = WORKLOADS[workload]
        self.N, self.R, self.E = N1 * scale, R, E1 * scale
        N, E = self.N, self.E
        t0 = time.time()
        self.tri = orc.synthetic_triples(N, R, E, seed)
        self.g = orc.build_graph(self.tri, N, R)
        self.w = small_weights(R)
        torch.manual_seed(0)
        self.conv = self.make_conv()
        self.g_rel = self.w['g_rel'].to(dev)
        self.rl = self.w['rels'].to(dev).requires_grad_(True)
        if world == 1:
            self.part = None
            self.ei = torch.from_numpy(self.g['edge_index']).to(dev)
            self.et = torch.from_numpy(self.g['edge_attr'][0]).to(dev)
            self.node_ids = torch.arange(N, dtype=torch.int64, device=dev)
            self.edge_ids = torch.arange(2 * E, dtype=torch.int64, device=dev)
        else:
            p2p_on = os.environ.get('KGC_P2P', '1') != '0'
            balance = os.environ.get('KGC_BALANCE', 'hybrid' if p2p_on else 'edges')
            self.part = k.GraphPartition(self.g['edge_index'], self.g['edge_attr'][0], N, 2 * R + 1, world, rank, dev,
                                         balance=balance, p2p='auto' if p2p_on else False)
            if balance == 'hybrid':
                try:                                       # peer memory is decided collectively: all ranks or none
                    self.part.p2p(D_IN)
                except RuntimeError as exc:
                    sys.stderr.write('hybrid cut unavailable ({}): destination partition instead\n'.format(exc))
                    self.part = k.GraphPartition(self.g['edge_index'], self.g['edge_attr'][0], N, 2 * R + 1, world, rank, dev,
                                                 balance='edges', p2p='auto')
            self.node_ids, self.edge_ids = self.part.owned_nodes, self.part.owned_eids
        self.x = self.rows('x', self.node_ids).requires_grad_(True)
        self.ee = self.rows('ee', self.edge_ids).requires_grad_(True)
        self.g_ent = self.rows('g_ent', self.node_ids)
        self.leaves = [self.x, self.ee, self.rl] + list(self.conv.parameters())
        self.setup_s = time.time() - t0

    def rows(self, what, ids):
        """Rows ``ids`` of the synthetic tensors: entity / edge embeddings at their xavier bound (utils.py:113-118), the
        upstream gradient of all_ent uniform with unit variance."""
        if what == 'x':
            return synth_rows(ids, D_IN, xavier_bound(self.N, D_IN), 11)
        if what == 'ee':
            return synth_rows(ids, D_IN, xavier_bound(2 * self.E, D_IN), 12)
        return synth_rows(ids, D_OUT, float(np.sqrt(3.0)), 13)

    def masks(self, ids):
        """Keep masks [len(ids), Dout] uint8 (p = 0.1) as a function of the node id: the partitioned and the single-GPU
        layer replay the same draws in the parity check."""
        u_in, u_out = synth_rows(ids, D_OUT, 1.0, 14), synth_rows(ids, D_OUT, 1.0, 15)
        return (u_in > -0.8).to(torch.uint8), (u_out > -0.8).to(torch.uint8)

    def make_conv(self):
        conv = self.k.MGCNConv(D_IN, D_OUT, 2 * self.R).to(self.dev)      # dropout p = 0.1, the reference default (model.py:49)
        with torch.no_grad():
            for name in ('loop_weight', 'in_weight', 'out_weight', 'rels_weight', 'loop_rel', 'loop_edge'):
                getattr(conv, name).copy_(self.w[name])
        return conv.train()

    def step(self):
        for t in self.leaves:
            t.grad = None
        if self.part is None:
            ent, rel = self.conv(self.x, self.ei, self.et, None, self.ee, self.rl)
        else:
            ent, rel = self.conv.forward_partitioned(self.x, self.part, self.ee, self.rl)
        torch.autograd.backward([ent, rel], [self.g_ent, self.g_rel])
        return ent, rel

    def grads(self):
        c = self.conv
        return {'d_x': self.x.grad, 'd_ee': self.ee.grad, 'd_rel': self.rl.grad, 'd_loop_weight': c.loop_weight.grad,
                'd_in_weight': c.in_weight.grad, 'd_out_weight': c.out_weight.grad, 'd_rels_weight': c.rels_weight.grad,
                'd_loop_rel': c.loop_rel.grad, 'd_loop_edge': c.loop_edge.grad, 'd_gamma': c.ent_bn.weight.grad}


def rel_err(a, b, chunk=1 << 26):
    """max |a - b| / max |b|, both maxima in float64, evaluated in slices of <= 64 Mi elements (the operands are up to
    16 GB at the Wikidata5M shape: whole-tensor float64 copies do not fit next to the layer's own buffers)."""
    a, b = a.detach().reshape(-1), b.detach().reshape(-1)
    num = den = 0.0
    for i in range(0, max(a.numel(), 1), chunk):
        bb = b[i:i + chunk].to(torch.float64)
        if bb.numel() == 0:
            break
        num = max(num, float((a[i:i + chunk].to(torch.float64) - bb).abs().max()))
        den = max(den, float(bb.abs().max()))
    return num / (den + 1e-300)


def parity_vs_float64(case, orc):
    """Single GPU: our fp32 layer (injected dropout masks) against oracle.conv_fwd_bwd_big in float64 on the same GPU."""
    m_in, m_out = case.masks(case.node_ids)
    case.conv.set_dropout_masks(m_in, m_out)
    try:
        ent, rel = case.step()
    finally:
        case.conv.set_dropout_masks(None, None)
    w = {name: getattr(case.conv, name).detach() for name in ('loop_weight', 'in_weight', 'out_weight', 'rels_weight',
                                                              'loop_rel', 'loop_edge')}
    w['ent_bn.weight'], w['ent_bn.bias'] = case.conv.ent_bn.weight.detach(), case.conv.ent_bn.bias.detach()
    truth = orc.conv_fwd_bwd_big(case.x.detach(), case.ei, case.et, case.ee.detach(), case.rl.detach(), w, case.g_ent, case.g_rel,
                                 mask_in=m_in, mask_out=m_out, drop_p=0.1, d_ee_check=case.ee.grad)
    g = case.grads()
    names = {'d_x': 'entity_embedding', 'd_rel': 'relation_embedding', 'd_loop_weight': 'conv1.loop_weight',
             'd_in_weight': 'conv1.in_weight', 'd_out_weight': 'conv1.out_weight', 'd_rels_weight': 'conv1.rels_weight',
             'd_loop_rel': 'conv1.loop_rel', 'd_loop_edge': 'conv1.loop_edge', 'd_gamma': 'conv1.ent_bn.weight'}
    errs = {'all_ent': rel_err(ent, truth['all_ent']), 'all_rel': rel_err(rel, truth['all_rel']),
            'd_ee': truth['d_ee_max_abs_err'] / (truth['d_ee_max_abs'] + 1e-300)}
    for ours, theirs in names.items():
        errs[ours] = rel_err(g[ours], truth[theirs])
    del truth
    torch.cuda.empty_cache()
    worst = max(errs.values())
    return {'vs': 'float64 restatement of the reference (oracle.conv_fwd_bwd_big) on the same inputs and dropout masks',
            'max_rel_err': worst, 'tol': PARITY_TOL, 'ok': bool(worst < PARITY_TOL), 'per_tensor': errs}


def parity_vs_single_gpu(case, dist):
    """N > 1: every rank runs the single-GPU layer on the WHOLE graph (same kernels, one GPU) and compares its own rows of
    the partitioned outputs and gradients with it; the replicated gradients must be bit-equal on every rank."""
    k, dev = case.k, case.dev
    m_in, m_out = case.masks(case.node_ids)
    case.conv.set_dropout_masks(m_in, m_out)
    try:
        ent_l, rel_l = case.step()
    finally:
        case.conv.set_dropout_masks(None, None)
    got = {kk: v.detach() for kk, v in case.grads().items()}      # the leaves' .grad tensors themselves (no second copy)
    got['all_ent'], got['all_rel'] = ent_l.detach(), rel_l.detach()
    del ent_l, rel_l
    for t_ in case.leaves:
        t_.grad = None
    k.plan._PLAN_CACHE.clear()
    torch.cuda.empty_cache()
    # bit-equality of the replicated tensors across ranks: all-gather an integer checksum
    rep = [n for n in got if n not in ('d_x', 'd_ee', 'all_ent')]
    sums = torch.stack([got[n].contiguous().view(torch.int32).to(torch.int64).sum() for n in rep])
    allsums = [torch.empty_like(sums) for _ in range(case.world)]
    dist.all_gather(allsums, sums)
    bit_equal = all(bool(torch.equal(s, allsums[0])) for s in allsums)
    # the single-GPU answer
    N, E = case.N, case.E
    all_nodes = torch.arange(N, dtype=torch.int64, device=dev)
    ref_conv = case.make_conv()
    fm_in, fm_out = case.masks(all_nodes)
    ref_conv.set_dropout_masks(fm_in, fm_out)
    x = case.rows('x', all_nodes).requires_grad_(True)
    ee = case.rows('ee', torch.arange(2 * E, dtype=torch.int64, device=dev)).requires_grad_(True)
    rl = case.w['rels'].to(dev).requires_grad_(True)
    ei = torch.from_numpy(case.g['edge_index']).to(dev)
    et = torch.from_numpy(case.g['edge_attr'][0]).to(dev)
    ent, rel = ref_conv(x, ei, et, None, ee, rl)
    torch.autograd.backward([ent, rel], [case.rows('g_ent', all_nodes), case.g_rel])
    ref_conv.set_dropout_masks(None, None)
    del fm_in, fm_out, ei, et
    k.plan._PLAN_CACHE.clear()                       # the whole-graph plan and its scratch planes (tens of GB at this shape)
    torch.cuda.empty_cache()
    own, oe = case.node_ids, case.edge_ids
    want = {'all_ent': lambda: ent[own], 'all_rel': lambda: rel, 'd_x': lambda: x.grad[own], 'd_ee': lambda: ee.grad[oe],
            'd_rel': lambda: rl.grad, 'd_loop_weight': lambda: ref_conv.loop_weight.grad,
            'd_in_weight': lambda: ref_conv.in_weight.grad, 'd_out_weight': lambda: ref_conv.out_weight.grad,
            'd_rels_weight': lambda: ref_conv.rels_weight.grad, 'd_loop_rel': lambda: ref_conv.loop_rel.grad,
            'd_loop_edge': lambda: ref_conv.loop_edge.grad, 'd_gamma': lambda: ref_conv.ent_bn.weight.grad}
    errs = {}
    for n in want:                                   # one tensor at a time: the row selections are copies of up to 8 GB
        errs[n] = rel_err(got.pop(n), want[n]())
    del want, ent, rel, x, ee, ref_conv, got
    torch.cuda.empty_cache()
    t = torch.tensor([max(errs.values())], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    worst = float(t[0])
    return {'vs': 'the single-GPU layer on the whole graph (run by every rank, same inputs and dropout masks), own rows',
            'max_rel_err': worst, 'tol': PARITY_TOL, 'ranks_bit_equal': bool(bit_equal),
            'ok': bool(worst < PARITY_TOL and bit_equal), 'per_tensor_rank0': errs}


def capture_and_time(case, args, dist, flush, clocks_index):
    """Warm-up, CUDA-graph capture of the fwd+bwd step, K timed replays (L2 flushed between them), max over ranks."""
    k = case.k
    L = k._lib
    launch_mode, graph = 'eager', None
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            case.step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    L.LAUNCHES = 0
    case.step()
    launches_per_step = L.LAUNCHES
    last = {}                                        # (all_ent, all_rel) of the latest step; a replay rewrites them in place

    def run_step():
        last.pop('out', None)                        # eager: do not hold the previous step's outputs through this one
        last['out'] = case.step()
    if not args.no_graph:
        try:
            graph = torch.cuda.CUDAGraph()
            for t in case.leaves:
                t.grad = None
            with torch.cuda.graph(graph):
                last['out'] = case.step()
            run_step = graph.replay
            launch_mode = 'cuda_graph'
        except Exception as exc:                      # pragma: no cover
            sys.stderr.write('graph capture failed, timing eager launches: {}\n'.format(exc))
            torch.cuda.synchronize()
    for _ in range(max(3, args.warmup)):
        run_step()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    timed_steps = 0
    with ClockSampler(clocks_index) as clocks:
        for a, b in ev:
            flush()
            a.record()
            run_step()
            b.record()
            timed_steps += 1
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
    total_ms = float(sum(a.elapsed_time(b) for a, b in ev))
    if dist is not None:
        t = torch.tensor([total_ms], device=case.dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t[0])
    return {'total_ms': total_ms, 'timed_steps': timed_steps, 'launch_mode': launch_mode, 'launches_per_step': launches_per_step,
            'clocks': clocks.summary(), 'graph': graph, 'outputs': last['out']}


def kernel_rooflines(case, flush):
    """The aggregation kernels alone through the C ABI (CUDA events on the launch stream, L2 flushed before every launch)
    and the whole forward / backward aggregation passes (every launch, fix-up levels included).  Fractions are against
    SURVEY.md 8(d)'s ALGORITHMIC bytes (each tensor once) and the measured HBM peak; ``kernel_bytes`` is what the kernel
    has to move in the implemented two-pass backward (the type-sorted pass re-reads the edge table)."""
    k = case.k
    L = k._lib
    p, st = L.ptr, L.stream
    N, R, E, D, T = case.N, case.R, case.E, D_IN, 2 * case.R + 1
    plan = k.get_plan(case.ei, case.et, N, T)
    conv, dev = case.conv, case.dev
    relp = torch.cat([case.rl.detach(), conv.loop_rel.detach()], 0).contiguous()
    xd, eed = case.x.detach(), case.ee.detach()
    agg = torch.empty((2, N, D), device=dev)
    g3 = synth_rows(torch.arange(3 * N, dtype=torch.int64, device=dev), D, 1.0, 21).view(3, N, D)
    d_ee, d_x, d_rel = torch.empty_like(eed), torch.empty((N, D), device=dev), torch.empty((plan.num_type_rows, D), device=dev)
    d_rel_sum = torch.empty((T, D), device=dev)
    sf, ss, sr = plan.fwd, plan.bwd_src, plan.bwd_rel

    def l0_fwd(sp, out_final, carry):
        L.call('kgc_agg_fwd', p(xd), p(relp), T, p(eed), p(plan.rec_dst), p(sp.rowflags), p(sp.chunks), sp.n_rec, p(out_final),
               p(carry), D, st())

    def l0_src(sp, out_final, carry):
        L.call('kgc_agg_bwd_src', p(xd), p(relp), T, p(eed), p(g3), p(plan.rec_src), p(sp.rowflags), p(sp.chunks), sp.n_rec, N, E,
               p(g3[2]), p(d_ee), p(out_final), p(carry), D, st())

    def l0_rel(sp, out_final, carry):
        L.call('kgc_agg_bwd_rel', p(xd), p(eed), p(g3), p(plan.rec_type), p(sp.rowflags), p(sp.chunks), sp.n_rec, N, E,
               p(out_final), p(carry), D, st())
    carry = {n_: torch.empty((max(s_.n_carry, 1), D), device=dev) for n_, s_ in (('f', sf), ('s', ss), ('r', sr))}
    fns = {'agg_fwd': lambda: l0_fwd(sf, agg, carry['f']), 'agg_bwd_src': lambda: l0_src(ss, d_x, carry['s']),
           'agg_bwd_rel': lambda: l0_rel(sr, d_rel, carry['r'])}

    def pass_fwd():
        plan.run_reduction(sf, l0_fwd, agg, D, tag='rf_f')

    def pass_bwd():
        plan.run_reduction(ss, l0_src, d_x, D, addend=g3[2], tag='rf_s')
        plan.run_rel_reduction(l0_rel, d_rel_sum, D, tag='rf_r')
    row = 4 * D
    fwd_b, bwd_b = algorithmic_bytes(N, R, E)
    n_ch = (2 * E + 31) // 32
    survey = {'agg_fwd': fwd_b, 'agg_bwd_src': bwd_b - T * row, 'agg_bwd_rel': T * row}
    moved = {   # what each kernel has to read / write in the implemented design: edge stream + 20 B of record per edge + dense operands once
        'agg_fwd': 2 * E * (row + 20) + N * row + T * row + 2 * N * row + 8 * n_ch,
        'agg_bwd_src': 2 * E * (2 * row + 20) + N * row + 3 * N * row + T * row + N * row + 8 * n_ch,
        'agg_bwd_rel': 2 * E * (row + 20) + N * row + 2 * N * row + T * row + 8 * n_ch,
    }
    _, peak, peak_src = measured_peaks()
    iters = 20 if 2 * E < 5000000 else 5
    out = {}
    cp_dst = torch.empty_like(eed)
    ms_cp = time_kernel(lambda: cp_dst.copy_(eed), flush, iters=iters)
    cp_bytes = 2 * eed.numel() * 4
    out['copy_same_size_reference'] = {'ms': ms_cp, 'bytes': cp_bytes, 'achieved_gbs': cp_bytes / (ms_cp * 1e-3) / 1e9,
                                       'frac': cp_bytes / (ms_cp * 1e-3) / 1e9 / peak,
                                       'note': 'torch copy of the edge-embedding table, timed the same way: what a plain '
                                               'streaming kernel of this size reaches (launch latency + tail included)'}
    del cp_dst
    for name, fn in fns.items():
        ms = time_kernel(fn, flush, iters=iters)
        out[name] = {'ms': ms, 'survey_bytes': survey[name], 'frac_survey': survey[name] / (ms * 1e-3) / 1e9 / peak,
                     'kernel_bytes': moved[name], 'frac_kernel': moved[name] / (ms * 1e-3) / 1e9 / peak,
                     'traffic_ncu': ncu_traffic(case.workload, name)}
    ms_f, ms_b = time_kernel(pass_fwd, flush, iters=iters), time_kernel(pass_bwd, flush, iters=iters)
    passes = {
        'fwd': {'ms': ms_f, 'survey_bytes': fwd_b, 'frac': fwd_b / (ms_f * 1e-3) / 1e9 / peak},
        'bwd': {'ms': ms_b, 'survey_bytes': bwd_b, 'frac': bwd_b / (ms_b * 1e-3) / 1e9 / peak},
        'fwd_bwd': {'ms': ms_f + ms_b, 'survey_bytes': fwd_b + bwd_b, 'frac': (fwd_b + bwd_b) / ((ms_f + ms_b) * 1e-3) / 1e9 / peak},
        'note': 'every launch of the pass (level-0 kernel + fix-up levels; backward = src-sorted pass + type-sorted pass) '
                'against SURVEY.md 8(d) bytes of the pass',
    }
    top = max(fns, key=lambda n_: out[n_]['ms'])
    roof = {'kernel': top, 'bound': 'hbm', 'achieved': survey[top] / (out[top]['ms'] * 1e-3) / 1e9, 'peak': peak, 'unit': 'GB/s',
            'frac': out[top]['frac_survey'], 'traffic': out[top]['traffic_ncu'], 'peak_source': peak_src,
            'algorithmic_bytes': survey[top], 'ms': out[top]['ms'], 'passes': passes,
            'how': 'kernel launched alone through the C ABI, CUDA events on the launch stream, L2 flushed before each launch; '
                   'achieved = SURVEY.md 8(d) algorithmic bytes of the tensors this kernel is responsible for / time'}
    return roof, out


DUMP_MAX_ROWS = 16384      # row sample of every output with more rows: ~29 MB in all at the Wikidata5M shape


def dump_outputs(case, ent, rel, out_dir):
    """What the last timed step handed its caller, as ``out_dir/<name>.npy`` (float32): the layer's outputs all_ent /
    all_rel and the gradient of every input and parameter (d_x, d_ee, d_rel, d_<parameter>).  A tensor with more than
    DUMP_MAX_ROWS rows is cut to that many rows, drawn by torch.randperm from a generator seeded with 0 (the same rows
    for every tensor of the same height), in increasing row order.  The inputs are pure functions of the workload's
    seeds, so two builds run with the same arguments can be compared array for array."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {'all_ent': ent, 'all_rel': rel, 'd_x': case.x.grad, 'd_ee': case.ee.grad, 'd_rel': case.rl.grad}
    for name, prm in case.conv.named_parameters():
        arrays['d_' + name.replace('.', '_')] = prm.grad
    for name, t in arrays.items():
        if t is None:
            raise RuntimeError('--dump-outputs: the timed step produced no {}'.format(name))
        t = t.detach()
        if t.dim() > 0 and t.size(0) > DUMP_MAX_ROWS:
            rows = torch.randperm(t.size(0), generator=torch.Generator().manual_seed(0))[:DUMP_MAX_ROWS].sort().values
            t = t[rows.to(t.device)]
        np.save(os.path.join(out_dir, name + '.npy'), t.to(torch.float32).cpu().numpy())
    sys.stderr.write('--dump-outputs: {} arrays of the last timed step written to {}\n'.format(len(arrays), out_dir))


def bench_layer(k, orc, workload, dev, args, flush, with_roofline=True, dump_dir=None):
    """value / parity / rooflines of one workload on ONE GPU; ``dump_dir``: write the last timed step's outputs there."""
    case = LayerCase(k, orc, workload, dev)
    res = {'N': case.N, 'R': case.R, 'E': case.E, 'setup_s': case.setup_s}
    torch.cuda.synchronize()
    t0 = time.time()
    k.get_plan(case.ei, case.et, case.N, 2 * case.R + 1)          # K1 (three sorted CSRs) + the streaming schedules: once per graph
    torch.cuda.synchronize()
    res['plan_build_s'] = time.time() - t0
    if not args.no_parity:
        try:
            res['parity'] = parity_vs_float64(case, orc)
        except Exception as exc:                       # pragma: no cover
            res['parity'] = {'ok': False, 'error': repr(exc)}
            torch.cuda.empty_cache()
    t = capture_and_time(case, args, None, flush, dev.index or 0)
    if dump_dir is not None:
        dump_outputs(case, *t['outputs'], dump_dir)
    t['outputs'] = None
    ms = t['total_ms'] / t['timed_steps']
    fwd_b, bwd_b = algorithmic_bytes(case.N, case.R, case.E)
    _, peak, peak_src = measured_peaks()
    res.update({'value': 2 * case.E / (ms * 1e-3), 'ms_per_step': ms, 'timed_steps': t['timed_steps'], 'launch': t['launch_mode'],
                'launches_per_step': t['launches_per_step'], 'clocks': t['clocks'],
                'step_hbm': {'algorithmic_bytes_fwd_bwd': fwd_b + bwd_b, 'achieved_gbs': (fwd_b + bwd_b) / (ms * 1e-3) / 1e9,
                             'frac_of_peak': (fwd_b + bwd_b) / (ms * 1e-3) / 1e9 / peak, 'peak_gbs': peak, 'peak_source': peak_src,
                             'note': 'whole layer incl. the dense GEMMs and the BN/tanh tail, SURVEY.md 8(d) bytes'}})
    t['graph'] = None
    if with_roofline:
        try:
            res['roofline'], res['kernels'] = kernel_rooflines(case, flush)
        except Exception as exc:                       # pragma: no cover
            res['roofline'], res['kernels'] = None, {'error': repr(exc)}
    return res, case


def run_ours(args, rank, world, local_rank):
    import kgc_gcn_b200 as k
    k._lib.lib()
    orc = oracle()                       # synthetic-workload generators, the float64 parity checker, the cpu_baseline leg
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=dev)
    flush = Flusher(dev)
    weak = bool(os.environ.get('KGC_BENCH_WEAK'))
    workload = args.workload or ('wn18rr' if (weak and world > 1) else 'wikidata5m')
    peaks, peak, peak_src = measured_peaks()
    N1, R, E1, _ = WORKLOADS[workload]
    line = {'metric': 'edges/sec GCN fwd+bwd', 'unit': 'edges/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': max(3, args.warmup), 'higher_is_better': True, 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic'}
    rc = 0
    if world == 1:
        res, case = bench_layer(k, orc, workload, dev, args, flush, dump_dir=args.dump_outputs)
        value, ms = res['value'], res['ms_per_step']
        N, E = case.N, case.E
        line.update({'value': value, 'ms_per_step': ms, 'timed_steps': res['timed_steps'], 'scaling': 'weak',
                     'gpu_launches': res['launches_per_step'] * res['timed_steps'],
                     'plan_build_s': res.get('plan_build_s'),
                     'clocks': res['clocks'], 'roofline': res.get('roofline'), 'kernels': res.get('kernels'),
                     'step_hbm': res['step_hbm'], 'parity': res.get('parity')})
        launch_mode, par = res['launch'], 'single GPU'
        tri, g = case.tri, case.g
        del case, res
        k.plan._PLAN_CACHE.clear()                   # the plan's scratch planes (tens of GB at the Wikidata5M shape)
        torch.cuda.empty_cache()
        if line['parity'] is not None and not line['parity'].get('ok', False):
            rc = 3
        # ---- e2e: the whole training step through the reference-facing API, host ids in, loss out
        if args.no_e2e:
            e2e = {'ms_total': float('nan'), 'steps': 0, 'h2d': 0, 'd2h': 0, 'scope': 'skipped'}
        else:
            try:
                e2e = e2e_train_step(k, tri, g, N, R, E, dev, args)
                e2e['workload'] = workload + '_shape'
            except Exception as exc:                  # pragma: no cover - keep the headline line if the e2e leg fails
                sys.stderr.write('e2e leg failed at the {} shape: {!r}\n'.format(workload, exc))
                e2e = {'ms_total': float('nan'), 'steps': 0, 'h2d': 0, 'd2h': 0, 'scope': 'failed: {!r}'.format(exc)}
                k.plan._PLAN_CACHE.clear()
                torch.cuda.empty_cache()
        del tri, g
    else:
        scale = world if weak else 1
        case = LayerCase(k, orc, workload, dev, world, rank, scale=scale)
        N, E = case.N, case.E
        parity = None
        if not args.no_parity and not weak:
            parity = parity_vs_single_gpu(case, dist)
            if not parity['ok']:
                rc = 3
        t = capture_and_time(case, args, dist, flush, local_rank)
        ms = t['total_ms'] / t['timed_steps']
        value = 2 * E / (ms * 1e-3)                      # E counts every rank's triples
        launch_mode = t['launch_mode']
        part = case.part
        p2p = part.p2p(D_IN)
        if getattr(part, 'hybrid', False):
            par = ('hybrid cut over {} GPUs: an edge lives with the owner of its lower-degree endpoint (largest edge share {:.3f}x the '
                   'mean, {} remote rows of {} on rank 0); x rows in, partial aggregates to their owners, upstream rows in, partial '
                   'd_x to their owners: pulls over NVLink peer memory (K10); BN sums, replicated grads: one-shot peer-memory kernel'
                   .format(world, float(part.owned_eids.numel()) * world / (2 * E), part.n_halo, N))
        else:
            par = ('edge-balanced dst partition over {} GPUs ({} split hub rows, largest edge share {:.3f}x the mean); halo exchange of '
                   'x / d_x: {}; all-reduce of hub rows, BN sums, replicated grads: {}'
                   .format(world, part.n_hub, float(part.owned_eids.numel()) * world / (2 * E),
                           'pulls over NVLink peer memory (K10)' if p2p is not None else 'NCCL all-gather / reduce-scatter',
                           'one-shot peer-memory kernel (K10)' if p2p is not None else 'NCCL'))
        if p2p is not None:
            p2p.check()
        line.update({'value': value, 'ms_per_step': ms, 'timed_steps': t['timed_steps'], 'scaling': 'weak' if weak else 'strong',
                     'gpu_launches': t['launches_per_step'] * t['timed_steps'], 'clocks': t['clocks'], 'parity': parity,
                     'roofline': None, 'kernels': None,
                     'step_hbm': {'note': 'per-kernel rooflines are measured at N = 1 (same kernels on every rank)'}})
        if args.no_e2e:
            e2e = {'ms_total': float('nan'), 'steps': 0, 'h2d': 0, 'd2h': 0, 'scope': 'skipped'}
        else:
            try:
                e2e = e2e_partitioned_step(k, case, args, dist)
            except Exception as exc:                  # pragma: no cover
                sys.stderr.write('partitioned e2e leg failed: {!r}\n'.format(exc))
                e2e = {'ms_total': float('nan'), 'steps': 0, 'h2d': 0, 'd2h': 0, 'scope': 'failed: {!r}'.format(exc)}
        tm = torch.tensor([e2e['ms_total']], device=dev, dtype=torch.float64)
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        e2e['ms_total'] = float(tm[0])
        # release the CUDA graph (it may hold captured NCCL kernels) before the communicator goes away
        t['graph'] = None
        del case
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        dist.barrier()
    e2e_value = 2 * E * e2e['steps'] / (e2e['ms_total'] * 1e-3) if e2e['steps'] else None
    line['config'] = {'workload': workload + '_shape' + (' x{} (one shape-sized partition per GPU)'.format(world) if (weak and world > 1) else ''),
                      'N': N, 'R': R, 'E': E, 'directed_edges': 2 * E, 'd_in': D_IN, 'd_out': D_OUT,
                      'dropout': 'p=0.1 keep masks drawn inside the timed region (training mode)',
                      'l2': 'flushed between steps (256 MiB memset + 256 MiB read, outside the timed events)',
                      'launch': launch_mode, 'parallelism': par}
    line['e2e'] = {'value': e2e_value, 'unit': 'edges/s', 'h2d_bytes_per_step': e2e['h2d'], 'd2h_bytes_per_step': e2e['d2h'],
                   'ms_per_step': e2e['ms_total'] / e2e['steps'] if e2e['steps'] else None, 'scope': e2e['scope']}
    for extra in ('eager_ms_per_step', 'dense_label_ms_per_step', 'fused_loss_ms_per_step', 'workload'):
        if e2e.get(extra) is not None:
            line['e2e'][extra] = e2e[extra]
    # ---- second half of the metric: filtered-rank queries/s (every N: the entity table is sharded over the ranks)
    if not args.no_aux:
        try:
            line['aux'] = aux_filtered_rank(k, dev, args, world, rank, dist)
            if line['aux'].get('sharded_equals_unsharded') is False:
                rc = 4
        except Exception as exc:                       # pragma: no cover
            line['aux'] = {'error': repr(exc)}
            torch.cuda.empty_cache()
    if rank != 0:
        shutdown(dist)
        sys.exit(rc)
    # ---- the other single-GPU shapes of BASELINE.json, same run (N = 1 only)
    if world == 1 and not args.workload and not args.no_extras:
        line['workloads'] = {}
        for extra in ('wn18rr', 'fb15k237'):
            try:
                res, c = bench_layer(k, orc, extra, dev, args, flush)
                del c
                k.plan._PLAN_CACHE.clear()
                res.pop('kernels', None)
                line['workloads'][extra + '_shape'] = res
                if res.get('parity') is not None and not res['parity'].get('ok', False):
                    rc = 3
            except Exception as exc:                   # pragma: no cover
                line['workloads'][extra + '_shape'] = {'error': repr(exc)}
            torch.cuda.empty_cache()
    if not args.no_cpu_baseline:
        legs = reference_cpu_legs(workload, steps=8, warmup=1, budget_s=12.0, want_step=False)
        line['cpu_baseline'] = cpu_baseline_entry(legs, workload)
    emit(line)
    shutdown(dist)
    sys.exit(rc)


def shutdown(dist):
    """Tear the process group down; a watchdog ends the process if NCCL teardown stalls (the JSON line is already out)."""
    if dist is None:
        return
    sys.stdout.flush()
    timer = threading.Timer(20.0, lambda: os._exit(0))
    timer.daemon = True
    timer.start()
    try:
        dist.destroy_process_group()
    finally:
        timer.cancel()


def e2e_train_step(k, tri, g, N, R, E, dev, args):
    """Whole training step through the public API, host ids in, loss out: GraphedTrainStep(fused_loss=True) - one CUDA-graph
    replay per step (host query ids through a pinned staging buffer -> MGCN encoder + ConvE -> 1-N scores -> BCE against the
    sparse positives -> backward -> ClipAdam -> loss.item()).  On the small shapes the dense-label graph step and the plain
    eager loop of the reference's main.py are timed as well and reported next to it."""
    prm = params_ns()
    graph = k.GraphData(edge_index=torch.from_numpy(g['edge_index']), edge_attr=torch.from_numpy(g['edge_attr']))
    graph.entity = torch.from_numpy(g['entity'])
    graph.edge_norm = torch.from_numpy(g['edge_norm'])
    graph.num_nodes = N
    graph.to(dev)
    ds = k.KBDataset(synthetic_query_set(k, tri, R), N, prm, training=True)
    loader = k.BatchIterator(ds, BATCH, shuffle=True, device=dev)
    steps, warm = args.steps, max(3, args.warmup)
    big = N * BATCH * 4 > (1 << 30)                       # a dense [B, N] fp32 tensor above 1 GiB: only the fused loss is timed
    modes = ('graph_fused',) if big else ('graph_fused', 'graph', 'eager')
    out = {}
    for mode in modes:
        torch.manual_seed(0)
        with torch.device(dev):                           # parameters are created on the GPU (the edge table alone is 16.5 GB at the Wikidata5M shape)
            model = k.MGCN(N, R, E, prm)
        model.train()
        opt = k.ClipAdam(model.parameters(), lr=1e-3, max_norm=1.0)          # clip_grad_norm_ + Adam (K9), main.py:68-71
        batches = loader.batches()
        step = k.GraphedTrainStep(model, opt, graph, ds, BATCH, fused_loss=(mode == 'graph_fused')) if mode != 'eager' else None
        ms, n = 0.0, 0
        try:
            for i in range(warm + steps):
                qid = next(batches)
                while len(qid) != BATCH:
                    qid = next(batches)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                if step is not None:
                    step(qid).item()                                          # H2D: query ids; D2H: the loss
                else:
                    trip, lab = ds.build_batch(qid, dev)
                    opt.zero_grad()
                    pred = model(trip[:, 0], trip[:, 1], graph)
                    loss = model.loss(pred, lab)
                    loss.backward()
                    opt.step()                                                # clips inside (max_norm = 1.0)
                    loss.item()
                b.record()
                torch.cuda.synchronize()
                if i >= warm:
                    ms += a.elapsed_time(b)
                    n += 1
            out[mode] = (ms, n)
        except Exception as exc:                                              # pragma: no cover
            sys.stderr.write('e2e mode {} failed: {!r}\n'.format(mode, exc))
            torch.cuda.synchronize()
        del model, opt, step
        k.plan._PLAN_CACHE.clear()
        torch.cuda.empty_cache()
    per = {m: v[0] / v[1] for m, v in out.items() if v[1]}
    if 'graph_fused' not in per:
        raise RuntimeError('the graph-captured training step did not run')
    res = {'ms_total': out['graph_fused'][0], 'steps': out['graph_fused'][1], 'h2d': BATCH * 8, 'd2h': 4,
           'scope': 'full training step through the public API (GraphedTrainStep(fused_loss=True), one CUDA-graph replay per step): '
                    'host query ids (pinned staging buffer) -> MGCN encoder + ConvE -> 1-N scores -> BCE against the sparse positives '
                    'fused with the logit gradient (N1) -> backward -> ClipAdam (gradient-norm clip + Adam, K9) -> loss.item()',
           'fused_loss_ms_per_step': per.get('graph_fused'), 'dense_label_ms_per_step': per.get('graph'),
           'eager_ms_per_step': per.get('eager')}
    return res


def e2e_partitioned_step(k, case, args, dist):
    """N > 1: the partitioned encoder step through forward_partitioned with the batch coming from pinned host memory every
    step (H2D) and the scalar loss read back (D2H).  The decoder is NOT in this number: the loss is a stand-in (mean of the
    batch's entity and relation rows, summed over ranks) - compare it with the N = 1 `value`, not with the N = 1 e2e."""
    steps, warm = args.steps, max(3, args.warmup)
    dev, part, conv, N, R = case.dev, case.part, case.conv, case.N, case.R
    rng = np.random.default_rng(0)
    host = torch.empty((BATCH, 2), dtype=torch.int64).pin_memory()
    local_row = torch.full((N,), -1, dtype=torch.int64, device=dev)
    local_row[part.owned_nodes] = torch.arange(part.n_real, device=dev)
    ms, n = 0.0, 0
    for i in range(warm + steps):
        host[:, 0] = torch.from_numpy(rng.integers(0, N, BATCH))
        host[:, 1] = torch.from_numpy(rng.integers(0, 2 * R, BATCH))
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        batch = host.to(dev, non_blocking=True)
        for t in case.leaves:
            t.grad = None
        ent, rel = conv.forward_partitioned(case.x, part, case.ee, case.rl)
        rows = local_row[batch[:, 0]]                    # -1: the entity lives on another rank
        mine = rows >= 0
        loss = (ent[rows.clamp_min(0)].mean(1) * mine).sum() + rel[batch[:, 1]].mean() / part.world
        loss.backward()
        tot = loss.detach().clone()
        dist.all_reduce(tot)
        tot.item()
        b.record()
        torch.cuda.synchronize()
        if i >= warm:
            ms += a.elapsed_time(b)
            n += 1
    return {'ms_total': ms, 'steps': n, 'h2d': BATCH * 16, 'd2h': 4,
            'scope': 'ENCODER ONLY (not the N = 1 e2e scope): batch ids from pinned host memory -> forward_partitioned -> stand-in '
                     'scalar loss -> backward -> loss.item(), eager launches'}


def aux_filtered_rank(k, dev, args, world, rank, dist):
    """Second half of BASELINE.json's metric: filtered-rank queries/sec of the fused tcgen05 scorer, B = 65,536 queries,
    d = 200 against N entities (SURVEY.md 8(d): X = |N(0,1)|-like, E ~ U(-1,1), bias ~ 0.1 U, 4 filtered positives per query).
    N > 1: rows of the entity table range-sharded over the ranks, queries replicated, target / filter logits computed by
    the owning rank and summed (exact), int32 counts all-reduced; the first 2,048 queries are also ranked against the whole
    table on every rank and the sharded ranks must equal them bit for bit."""
    L = k._lib
    peaks, _, _ = measured_peaks()
    sizes = [4594485] if not args.aux_full else [1000000, 2000000, 4594485]
    B, d = 65536, D_OUT
    out = []
    equal = None
    for N in sizes:
        qid = torch.arange(B, dtype=torch.int64, device=dev)
        xq = synth_rows(qid, d, 1.7, 31).abs_()
        obj = (_mix32(qid + 977) % N).to(torch.int64)
        fptr = torch.arange(0, 4 * B + 1, 4, device=dev, dtype=torch.int64)
        fidx = (_mix32(torch.arange(4 * B, dtype=torch.int64, device=dev) + 4099) % N).view(B, 4).sort(1).values.reshape(-1).to(torch.int32)
        per = -(-N // world)
        lo, hi = min(rank * per, N), min((rank + 1) * per, N)
        rows = torch.arange(lo, hi, dtype=torch.int64, device=dev)
        tab = synth_rows(rows, d, 1.0, 32)
        bias = synth_rows(rows, 1, 0.1, 33).view(-1)
        table = k.EntityTable(tab, bias)
        del tab
        grp = None if world == 1 else dist.group.WORLD

        def whole():
            return k.filtered_rank(xq, None, None, obj, fptr, fidx, table=table, n_offset=lo, group=grp)
        for _ in range(2):
            res = whole()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        reps = 3
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for a, b_ in ev:
            a.record()
            res = whole()
            b_.record()
        torch.cuda.synchronize()
        ms_whole = float(np.mean([a.elapsed_time(b_) for a, b_ in ev]))
        # the sweep kernel alone (dominant): packed operands resident, thresholds given
        q16 = k.pack_queries(xq)
        thr = res['thr']
        gt = torch.zeros(B, dtype=torch.int32, device=dev)

        def sweep():
            L.call('kgc_score_rank', L.ptr(q16), L.ptr(table.data), B, table.n, table.kpad, L.ptr(thr), L.ptr(gt), None, L.stream())
        ms_sweep = time_kernel(sweep, lambda: None, iters=3, warm=1)
        if dist is not None:
            t = torch.tensor([ms_whole, ms_sweep], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_whole, ms_sweep = float(t[0]), float(t[1])
        flops = 2.0 * B * N * d                                  # whole job, un-padded K
        tf = flops / (ms_sweep * 1e-3) / 1e12
        entry = {'B': B, 'N': N, 'd': d, 'queries_per_s': B / (ms_whole * 1e-3), 'ms_whole_call': ms_whole,
                 'ms_sweep_kernel': ms_sweep, 'sweep_tflops_unpadded_all_gpus': tf,
                 'frac_of_bf16_sustained': tf / world / peaks['bf16_tflops_sustained'],
                 'frac_of_bf16_burst': tf / world / peaks['bf16_tflops'], 'mean_rank': float(res['sums'][1] / res['sums'][0])}
        if world > 1 and N == sizes[-1]:
            # sharded == unsharded on a slice: every rank builds the whole table once and ranks 2,048 queries against it
            nq = 2048
            full = k.EntityTable(synth_rows(torch.arange(N, dtype=torch.int64, device=dev), d, 1.0, 32),
                                 synth_rows(torch.arange(N, dtype=torch.int64, device=dev), 1, 0.1, 33).view(-1))
            f2 = fptr[:nq + 1].contiguous()
            one = k.filtered_rank(xq[:nq].contiguous(), None, None, obj[:nq].contiguous(), f2, fidx[:4 * nq].contiguous(),
                                  count_eq=True, table=full)
            sh = k.filtered_rank(xq[:nq].contiguous(), None, None, obj[:nq].contiguous(), f2, fidx[:4 * nq].contiguous(),
                                 count_eq=True, table=table, n_offset=lo, group=grp)
            ok = torch.equal(one['ranks'], sh['ranks']) and torch.equal(one['count_eq'], sh['count_eq']) and \
                torch.equal(one['thr'], sh['thr'])
            t = torch.tensor([1 if ok else 0], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            equal = bool(int(t[0]))
            del full
        out.append(entry)
        del table, xq, q16
        torch.cuda.empty_cache()
    res = {'metric': 'filtered-rank queries/sec (fused tcgen05 scoring, bf16 operands, fp32 accumulate)', 'unit': 'queries/s',
           'value': out[-1]['queries_per_s'], 'n_gpus': world, 'sweeps': out,
           'sharding': 'single GPU' if world == 1 else 'entity rows range-sharded over {} GPUs, queries replicated, int32 counts all-reduced (NCCL)'.format(world),
           'roofline': {'bound': 'tensor', 'achieved': out[-1]['sweep_tflops_unpadded_all_gpus'] / world,
                        'peak': peaks['bf16_tflops_sustained'], 'unit': 'TFLOP/s per GPU', 'frac': out[-1]['frac_of_bf16_sustained'],
                        'note': 'un-padded flops 2*B*N*200 / (sweep-kernel CUDA-event time, max over ranks) / GPUs vs measured sustained cuBLAS bf16'}}
    if equal is not None:
        res['sharded_equals_unsharded'] = equal
    return res


_REAL_STDOUT = None


def guard_stdout():
    """Everything libraries print on fd 1 (NCCL prints its version there) goes to stderr; the ONE JSON line is written
    to the saved descriptor by emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    data = (json.dumps(line) + '\n').encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default=None, choices=sorted(WORKLOADS),
                    help='default: wikidata5m (+ wn18rr and fb15k237 as extra entries at N = 1)')
    ap.add_argument('--no-graph', action='store_true')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-aux', action='store_true', help='skip the filtered-rank scoring sweep')
    ap.add_argument('--aux-full', action='store_true', help='scoring sweep at N = 1M, 2M and 4,594,485')
    ap.add_argument('--no-e2e', action='store_true', help='profiling runs only: skip the end-to-end leg')
    ap.add_argument('--no-parity', action='store_true', help='profiling runs only: skip the parity check')
    ap.add_argument('--no-extras', action='store_true', help='N = 1: skip the WN18RR / FB15k-237 entries')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='N = 1, --impl ours: write the outputs and gradients of the last timed layer step to DIR/<name>.npy '
                         '(float32; tensors taller than {} rows as a seeded row sample)'.format(DUMP_MAX_ROWS))
    args = ap.parse_args()
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs is not None and (args.impl != 'ours' or world > 1):
        ap.error('--dump-outputs needs --impl ours on one GPU (WORLD_SIZE=1)')
    guard_stdout()
    if args.impl == 'reference':
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == '__main__':
    main()
