"""Graph-captured training step: the reference's inner loop (main.py:57-71) as ONE CUDA graph replay.

The reference issues ~200 small operations per step from Python; on a B200 the step is then bound by the host, not the
GPU.  ``GraphedTrainStep`` captures forward + BCE loss + backward + gradient clipping + Adam into a CUDA graph over static
input buffers; per step the host only hands over the batch's query ids (K5 builds the batch straight into the static
buffers), replays the graph and reads the loss back.  Numerics are those of the eager step (same kernels, same order).
"""
import torch

from . import _lib


class GraphedTrainStep(object):
    """step = GraphedTrainStep(model, optimizer, graph, dataset, batch_size); loss = step(qid).

    ``optimizer`` must be capturable (``kgc_gcn_b200.ClipAdam(..., max_norm=clip_grad)``, which also does the gradient
    clipping, or ``torch.optim.Adam(..., capturable=True)``); ``dataset`` is the KBDataset of the
    training queries; batches whose size differs from ``batch_size`` (the last one of an epoch) run eagerly.
    ``fused_loss=True`` (opt-in) trains through ``MGCN.loss_sparse``: the label stays a sparse list of positives and the
    dense [B, N] label, its build and the BCE tensors drop out of the step (SURVEY.md 8(f) N1).
    ``negatives=k`` trains the negative-sampled objective instead (``MGCN.loss_sampled``: ``n_pos`` positives and k
    negatives per query, ``tries`` draws per negative): its cost does not grow with N, so ``batch_size`` can be in the
    thousands.  Each step draws the samplers' uint32 inputs from ``generator`` (or torch's global one) into static device
    buffers (``pos_draws`` [B, n_pos], ``neg_draws`` [B, k, tries]) before the replay; the graph itself holds no RNG, so
    a replay equals the eager ``loss_sampled`` step on the same draws.  ``adversarial_temperature=alpha`` (with
    ``negatives=k`` only) trains with self-adversarial negative weights (``MGCN.loss_sampled``); the graph holds alpha as
    a constant."""

    def __init__(self, model, optimizer, graph, dataset, batch_size, clip_grad=1.0, warmup=3, fused_loss=False,
                 negatives=None, n_pos=1, tries=4, generator=None, adversarial_temperature=None):
        from .scoring import check_adversarial_temperature
        adversarial_temperature = check_adversarial_temperature(adversarial_temperature)
        if adversarial_temperature is not None and negatives is None:
            raise ValueError('adversarial_temperature weights the sampled negatives: it needs negatives=k')
        if negatives is not None:
            if fused_loss:
                raise ValueError('negatives= and fused_loss=True are two different objectives: pass one of them')
            if int(negatives) < 1 or int(n_pos) < 1 or int(tries) < 1:
                raise ValueError('negatives, n_pos and tries must be positive')
        self.model, self.opt, self.graph_data, self.ds = model, optimizer, graph, dataset
        self.clip, self.B = float(clip_grad), int(batch_size)
        dev = graph.edge_index.device
        if dev.type != 'cuda':
            raise RuntimeError('GraphedTrainStep runs on the GPU only')
        self.dev = dev
        self.params = [p for p in model.parameters() if p.requires_grad]
        self.trip = torch.zeros((self.B, 3), dtype=torch.int64, device=dev)
        self.fused_loss = bool(fused_loss)
        self.negatives = None if negatives is None else int(negatives)
        self.n_pos, self.tries, self.generator = int(n_pos), int(tries), generator
        self.adversarial_temperature = adversarial_temperature
        self.pos_draws = self.neg_draws = None
        if self.negatives is not None:
            self.pos_draws = torch.zeros((self.B, self.n_pos), dtype=torch.int64, device=dev)
            self.neg_draws = torch.zeros((self.B, self.negatives, self.tries), dtype=torch.int64, device=dev)
        self.label = None if (self.fused_loss or self.negatives is not None) else \
            torch.zeros((self.B, dataset.num_entity), dtype=torch.float32, device=dev)
        self.qid = torch.zeros((self.B,), dtype=torch.int64, device=dev)
        self._opt_clips = bool(getattr(optimizer, 'param_groups', None)) and \
            all(g.get('max_norm') for g in optimizer.param_groups)
        # pinned staging buffer of the batch's query ids (the only per-step host -> device traffic) and the event that says
        # the previous step's copy has left it
        try:
            self._pin = torch.empty((self.B,), dtype=torch.int64, pin_memory=True)
            self._pin_done = torch.cuda.Event()
        except RuntimeError:                          # no pinned memory to be had: stage from pageable memory
            self._pin = self._pin_done = None
        self.loss = None
        self.cuda_graph = None
        self._warmup = int(warmup)

    def _fill(self, qid):
        """Host ids -> static device buffers (H2D of B int64), then K5 into the static triple / label buffers."""
        host = torch.as_tensor(qid, dtype=torch.int64)
        if self._pin is not None and not host.is_cuda:
            self._pin_done.synchronize()
            self._pin.copy_(host)
            self.qid.copy_(self._pin, non_blocking=True)
            self._pin_done.record()
        else:
            self.qid.copy_(host, non_blocking=True)
        if self.negatives is not None:               # fresh sampler inputs, drawn outside the graph (positives first)
            self.pos_draws.random_(0, 1 << 32, generator=self.generator)
            self.neg_draws.random_(0, 1 << 32, generator=self.generator)
            return
        if self.fused_loss:                           # the graph reads the triples and the positives through qid
            return
        triples, ptr, idx = self.ds.device_csr(self.dev)
        pos, add = self.ds.label_values()
        p = _lib.ptr
        _lib.call('kgc_label_build', p(self.qid), self.B, p(triples), p(ptr), p(idx), self.ds.num_entity, pos, add,
                  p(self.trip), p(self.label), _lib.stream())

    def _body(self, trip, label, qid=None, draws=None):
        if self.negatives is not None:
            loss = self.model.loss_sampled(qid, self.ds, self.graph_data, self.negatives, n_pos=self.n_pos, tries=self.tries,
                                           draws=draws, generator=self.generator,
                                           adversarial_temperature=self.adversarial_temperature)
        elif qid is not None:
            loss = self.model.loss_sparse(qid, self.ds, self.graph_data)
        else:
            pred = self.model(trip[:, 0], trip[:, 1], self.graph_data)
            loss = self.model.loss(pred, label)
        loss.backward()
        if not self._opt_clips:                       # ClipAdam(max_norm=...) clips inside its step (K9)
            torch.nn.utils.clip_grad_norm_(self.params, self.clip)
        self.opt.step()
        return loss.detach()

    def _capture(self):
        self.model.train()
        # warm-up iterations (allocator, cuBLAS / cuDNN handles, lazy optimiser state) must not change the training
        # trajectory: parameters, buffers and optimiser state are restored afterwards
        fresh = len(self.opt.state) == 0
        if hasattr(self.opt, '_sync_steps'):         # ClipAdam: eager steps taken so far -> state[p]['step'] before the snapshot
            self.opt._sync_steps()
        # a fresh optimiser warms up with lr = 0: the parameters then stay bit-identical without a second copy of the model
        # (the edge table alone is 16.5 GB at the Wikidata5M shape) and the moments are zeroed afterwards; an optimiser
        # that already holds state gets parameters and state snapshotted and restored
        saved_p = None if fresh else [p.detach().clone() for p in self.params]
        saved_lr = [g['lr'] for g in self.opt.param_groups]
        if fresh:
            for g in self.opt.param_groups:
                g['lr'] = 0.0
        # the non-persistent dropout-stream buffers (_drop_seed) are NOT restored: they were drawn from torch's generator
        # during the first warm-up forward and keep advancing (restoring them would pin the stream to seed 0)
        named_b = [(n, b) for n, b in self.model.named_buffers() if not n.endswith('_drop_seed')]
        saved_b = [b.detach().clone() for _, b in named_b]
        saved_s = None if fresh else [[v.detach().clone() if torch.is_tensor(v) else v for v in st.values()]
                                      for st in self.opt.state.values()]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(max(self._warmup, 1)):
                self.opt.zero_grad(set_to_none=True)
                self._body(self.trip, self.label, *self._graph_inputs())
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        for g, lr in zip(self.opt.param_groups, saved_lr):
            g['lr'] = lr
        with torch.no_grad():
            if saved_p is not None:
                for p, sp in zip(self.params, saved_p):
                    p.copy_(sp)
            for (_, b), sb in zip(named_b, saved_b):
                b.copy_(sb)
            for i, st in enumerate(self.opt.state.values()):
                for j, (key, v) in enumerate(st.items()):
                    if torch.is_tensor(v):
                        v.zero_() if fresh else v.copy_(saved_s[i][j])
        del saved_p, saved_b, saved_s
        self.opt.zero_grad(set_to_none=True)
        torch.cuda.empty_cache()                      # the warm-up's activations go back to the driver before the graph pool grows
        if hasattr(self.opt, 'prepare'):             # ClipAdam: device-side step counter (from the restored state) / hyper-parameters
            self.opt.prepare(from_state=True)
        self.cuda_graph = torch.cuda.CUDAGraph()
        self.opt.zero_grad(set_to_none=True)
        with torch.cuda.graph(self.cuda_graph):
            self.loss = self._body(self.trip, self.label, *self._graph_inputs())

    def _graph_inputs(self):
        """(qid, draws) arguments of the captured body: the static buffers the objective reads."""
        if self.negatives is not None:
            return self.qid, (self.pos_draws, self.neg_draws)
        return (self.qid if self.fused_loss else None), None

    def __call__(self, qid):
        if len(qid) != self.B:                       # ragged last batch: the eager path (same arithmetic)
            self.opt.zero_grad(set_to_none=True)
            if self.fused_loss or self.negatives is not None:
                return self._body(None, None, torch.as_tensor(qid, dtype=torch.int64).to(self.dev))
            trip, label = self.ds.build_batch(qid, self.dev)
            return self._body(trip, label)
        self._fill(qid)
        if hasattr(self.opt, 'sync_hyper'):
            self.opt.sync_hyper()                    # a scheduler may have changed the learning rate (device-side copy)
        if self.cuda_graph is None:
            self._capture()                          # capture records the step; nothing has been executed for this batch yet
        self.cuda_graph.replay()
        return self.loss
