"""ClipAdam: the optimiser half of the reference's training step (main.py:68-71, 217) on the K9 kernels.

The reference runs ``nn.utils.clip_grad_norm_(model.parameters(), clip_grad)`` and then ``torch.optim.Adam.step()``.
``ClipAdam(params, lr=..., weight_decay=..., max_norm=clip_grad)`` does both in ``step()``: one pass over the gradients
for the norm, one fused update pass that applies the clip coefficient in flight (the ``.grad`` tensors are left as the
backward wrote them).  State keys (``step``, ``exp_avg``, ``exp_avg_sq``) and ``state_dict()`` layout are
``torch.optim.Adam``'s, so checkpoints written by the reference (utils.py:121-155, ``optim_dict``) load and vice versa.
The learning rate, step counter and bias corrections live in device memory: a CUDA graph of the step stays valid when a
scheduler changes ``param_group['lr']`` (call ``sync_hyper()`` - ``step()`` does outside graph capture).
GPU only, fp32 parameters, one parameter group when clipping (the norm is taken over the group, as the reference's is
over all parameters).

A model sharded over several GPUs (``MGCN.shard``) passes ``partition=`` (its GraphPartition) and ``sharded=`` (its
sharded parameters, ``model.sharded_parameters()``): the norm is then that of the whole model - every rank's sharded
parameters plus the replicated ones counted on rank 0, summed over the ranks in one all-reduce of the partition's
exchange (peer memory when it has it, NCCL otherwise) - and every rank applies the same coefficient.
"""
import torch

from . import _lib


class ClipAdam(torch.optim.Optimizer):

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, max_norm=None, partition=None,
                 sharded=()):
        if lr < 0.0 or eps < 0.0 or not 0.0 <= betas[0] < 1.0 or not 0.0 <= betas[1] < 1.0 or weight_decay < 0.0:
            raise ValueError('invalid Adam hyper-parameters')
        defaults = dict(lr=lr, betas=tuple(betas), eps=eps, weight_decay=weight_decay, max_norm=max_norm,
                        amsgrad=False, maximize=False, foreach=None, capturable=True, differentiable=False, fused=None,
                        decoupled_weight_decay=False)
        super(ClipAdam, self).__init__(params, defaults)
        if len(self.param_groups) > 1 and any(g.get('max_norm') for g in self.param_groups):
            raise ValueError('ClipAdam clips over one parameter group (the reference passes model.parameters())')
        if partition is None and len(tuple(sharded)):
            raise ValueError('sharded= names the parameters a partition splits: pass partition= as well')
        if partition is not None and len(self.param_groups) > 1:
            raise ValueError('ClipAdam over a sharded model takes one parameter group')
        self.partition = partition
        self._sharded = set(id(p) for p in sharded)
        self._coll = None
        self._dev = {}            # group index -> device-side buffers
        self.last_grad_norm = None

    # ------------------------------------------------------------------ device-side bookkeeping of one group
    def _group_state(self, gi, group, params):
        key = tuple(id(p) for p in params)
        st = self._dev.get(gi)
        if st is not None and st['key'] == key:
            return st
        dev = params[0].device
        chunk = int(_lib.lib().kgc_opt_chunk_elems())
        items = []
        for t, p in enumerate(params):
            n = p.numel()
            # a replicated tensor of a sharded model enters the norm on rank 0 only
            skip = int(self.partition is not None and self.partition.rank != 0 and id(p) not in self._sharded)
            for c in range((n + chunk - 1) // chunk):
                items.append((t, c, min(chunk, n - c * chunk), skip))
        step0 = 0.0
        for p in params:
            s = self.state[p]
            if len(s) == 0:
                s['step'] = torch.zeros((), dtype=torch.float32, device=dev)
                s['exp_avg'] = torch.zeros_like(p, memory_format=torch.preserve_format)
                s['exp_avg_sq'] = torch.zeros_like(p, memory_format=torch.preserve_format)
            step0 = max(step0, float(s['step']))
        if st is not None:                   # the set of parameters with gradients changed: keep counting from the device
            step0 = max(step0, float(st['state'][0]))
        st = {
            'key': key,
            'items': torch.tensor(items, dtype=torch.int32, device=dev).reshape(-1, 4),
            'n_items': len(items),
            'partials': torch.empty((max(len(items), 1),), dtype=torch.float64, device=dev),
            'sqnorm': torch.zeros((2,), dtype=torch.float64, device=dev),      # [0]: squared norm; 16-byte all-reduce payload
            'state': torch.tensor([step0, 1.0, 0.0, 0.0, 0.0], dtype=torch.float64, device=dev),
            'hyper': torch.zeros((6,), dtype=torch.float32, device=dev),
            'hyper_host': None,
            'table': torch.zeros((len(params), 4), dtype=torch.int64, device=dev),
            'pinned': [],          # host copies of the pointer table referenced by captured memcpy nodes
            'pinned_next': torch.zeros((len(params), 4), dtype=torch.int64).pin_memory(),
        }
        self._dev[gi] = st
        return st

    def _sync_steps(self):
        """Live device-side step counter -> ``state[p]['step']`` (what torch.optim.Adam keeps per parameter)."""
        for gi, group in enumerate(self.param_groups):
            st = self._dev.get(gi)
            if st is None:
                continue
            step = st['state'][0].to(torch.float32)
            for p in group['params']:
                if p in self.state and 'step' in self.state[p]:
                    self.state[p]['step'].copy_(step)

    def prepare(self, from_state=False):
        """Build the device-side state for every parameter that requires a gradient and push the hyper-parameters and the
        step count - call before capturing ``step()`` into a CUDA graph.  The count continues from the live device counter
        (eager steps taken so far); ``from_state=True`` takes it from ``state[p]['step']`` instead (a caller that has just
        restored the optimiser state, e.g. GraphedTrainStep after its warm-up)."""
        if not from_state:
            self._sync_steps()
        for gi, group in enumerate(self.param_groups):
            params = [p for p in group['params'] if p.requires_grad]
            if params:
                old = self._dev.pop(gi, None)
                st = self._group_state(gi, group, params)
                if old is not None:
                    st['pinned'] = old['pinned']          # still referenced by graphs captured earlier
        self.sync_hyper()

    def sync_hyper(self):
        """Host -> device copy of (lr, betas, eps, weight_decay, max_norm) where they changed (not capturable)."""
        for gi, group in enumerate(self.param_groups):
            st = self._dev.get(gi)
            if st is None:
                continue
            h = (float(group['lr']), float(group['betas'][0]), float(group['betas'][1]), float(group['eps']),
                 float(group['weight_decay']), float(group.get('max_norm') or 0.0))
            if st['hyper_host'] != h:
                st['hyper'].copy_(torch.tensor(h, dtype=torch.float32))
                st['hyper_host'] = h

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        capturing = torch.cuda.is_current_stream_capturing()
        for gi, group in enumerate(self.param_groups):
            params = [p for p in group['params'] if p.grad is not None]
            if not params:
                continue
            for p in params:
                if not p.is_cuda or p.dtype != torch.float32 or p.grad.is_sparse:
                    raise RuntimeError('ClipAdam: dense fp32 CUDA parameters only (no CPU fallback)')
            st = self._group_state(gi, group, params)
            if not capturing:
                self.sync_hyper()
            elif st['hyper_host'] is None:
                raise RuntimeError('ClipAdam: call prepare() before capturing step() into a CUDA graph')
            grads = [p.grad if p.grad.is_contiguous() else p.grad.contiguous() for p in params]
            host = torch.zeros((len(params), 4), dtype=torch.int64)
            for i, (p, g) in enumerate(zip(params, grads)):
                s = self.state[p]
                if not p.is_contiguous():
                    raise RuntimeError('ClipAdam: parameters must be contiguous')
                host[i, 0], host[i, 1] = p.data_ptr(), g.data_ptr()
                host[i, 2], host[i, 3] = s['exp_avg'].data_ptr(), s['exp_avg_sq'].data_ptr()
            if capturing:                     # a memcpy node that re-reads this pinned buffer at every replay: keep it alive
                pinned = st['pinned_next']
                if pinned is None:
                    raise RuntimeError('ClipAdam: call prepare() before every CUDA-graph capture of step()')
                pinned.copy_(host)
                st['pinned'].append(pinned)
                st['pinned_next'] = None
                st['table'].copy_(pinned, non_blocking=True)
            else:                             # gradients are re-allocated by every backward: refresh the table (32 B / tensor)
                st['table'].copy_(host)
            if self.partition is None:
                _lib.call('kgc_clip_adam_step', _lib.ptr(st['table']), _lib.ptr(st['items']), st['n_items'],
                          _lib.ptr(st['hyper']), _lib.ptr(st['state']), _lib.ptr(st['partials']), _lib.stream())
            else:
                _lib.call('kgc_clip_adam_sqnorm', _lib.ptr(st['table']), _lib.ptr(st['items']), st['n_items'],
                          _lib.ptr(st['partials']), _lib.ptr(st['sqnorm']), _lib.stream())
                if self._coll is None:                # the exchange of the model's forward (it ran before this step)
                    self._coll = self.partition.collectives()
                self._coll.all_reduce(st['sqnorm'], 'clip_sqnorm')
                _lib.call('kgc_clip_adam_apply', _lib.ptr(st['table']), _lib.ptr(st['items']), st['n_items'],
                          _lib.ptr(st['hyper']), _lib.ptr(st['state']), _lib.ptr(st['sqnorm']), _lib.stream())
            self.last_grad_norm = st['state'][4]
        return loss

    # ------------------------------------------------------------------ torch.optim.Adam-compatible checkpoints
    def state_dict(self):
        self._sync_steps()
        return super(ClipAdam, self).state_dict()

    def load_state_dict(self, state_dict):
        keep = [g.get('max_norm') for g in self.param_groups]
        super(ClipAdam, self).load_state_dict(state_dict)
        for g, m in zip(self.param_groups, keep):          # a torch.optim.Adam checkpoint has no max_norm: keep ours
            g.setdefault('max_norm', m)
        self._dev = {}                      # rebuilt (with the loaded step count) by the next step()
