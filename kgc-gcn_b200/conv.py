"""MGCNConv: the relation-aware graph convolution (reference model.py:47-127), B200 path.

Same constructor, parameter names, forward signature and return values as the reference class; the arithmetic runs in
libkgc_b200.so: K1 (sorted CSRs, norms, schedules), K2 / K3 (streaming aggregation, forward and backward), K4b / K4c (the
dense transforms on tcgen05 with fp32-grade accuracy, 3xTF32), K4 (dropout, /3, BatchNorm1d, tanh), K0 (parameter-side
kernels):

    agg_h[i]  = sum_{e in half h, dst_e = i} norm_e * x[src_e] (.) rel+[type_e] (.) ee[e]     K2
    res_h     = agg_h @ W_h ; res_loop = x @ (diag(loop_rel (.) loop_edge) W_loop)               K4b
    all_ent   = tanh(BN((drop(res_in) + drop(res_out) + res_loop) / 3 [+ bias]))                  K4
    all_rel   = (rel+ @ W_rel)[:-1]                                                              K0

(aggregate-then-transform is exact algebra because the message transform is linear, SURVEY.md fact 8).
Backward is hand-derived (SURVEY.md Appendix A) and runs K3 / K4-backward / K4b / K4c; it is deterministic.
``forward_partitioned`` is the same layer on a partitioned graph (partition.py): one process per GPU, exchanges over
NVLink peer memory (K10).
"""
import ctypes

import torch
import torch.nn as nn

from . import _lib
from .plan import get_plan

# The backward's upstream planes of the in / out halves = d_out x keep flags x 1 / (1 - p): either written by the tail
# kernel as two more planes, or applied by the GEMMs while they split the ONE plane.  Measured (graph-timed layer step,
# B200): Wikidata5M shape 49.7 vs 50.5 ms, WN18RR 0.387 vs 0.400 ms - the operand splitters are the busier side of K4b /
# K4c (+1.9 / +1.0 ms against -2.5 ms of tail traffic) - but FB15k-237 0.462 vs 0.411 ms: when the planes stay in L2 the
# extra writes are what costs.  So the three planes are written when together they exceed this size.
TAIL_MASKED_MAX_BYTES = 48 << 20
# ... and whenever the layer is wider than the masked K4c launch (gemm_tn_batch with keep flags) takes: d_in <= 128, d_out <= 224.
GEMM_TN_TC_MAX_KA, GEMM_TN_TC_MAX_NB = 128, 224


def get_param(shape):
    """utils.get_param (reference utils.py:113-118): xavier-uniform Parameter."""
    param = nn.Parameter(torch.empty(*shape))
    nn.init.xavier_uniform_(param.data)
    return param


def _mm(a, b, out):
    return torch.mm(a, b, out=out)


def _workspace(plan, name, nbytes, device):
    """A float32 buffer of nbytes: the plan's scratch buffer ``name`` when there is a plan (the same memory on every step, as
    a captured CUDA graph needs), else a new tensor."""
    if plan is not None:
        return plan.scratch(name, (nbytes // 4,))
    return torch.empty((nbytes // 4,), dtype=torch.float32, device=device)


def _ptr_array(ts):
    return (ctypes.c_void_p * len(ts))(*[t.data_ptr() for t in ts])


def _pack_b(b_kn, plan=None, name=None):
    """The small operand of K4b, b_kn[K, N] (any strided view: a weight, its transpose, a query block), split into hi / lo
    TF32 and packed by kgc_gemm_pack_b into a workspace buffer (see _workspace)."""
    K, N = b_kn.shape
    nbytes = int(_lib.lib().kgc_gemm_packed_b_bytes(N, K))
    if nbytes == 0:
        raise ValueError('unsupported small operand K={} N={} (K <= 256, N <= 1024)'.format(K, N))
    packed = _workspace(plan, name, nbytes, b_kn.device)
    _lib.call('kgc_gemm_pack_b', _lib.ptr(b_kn), b_kn.stride(0), b_kn.stride(1), N, K, _lib.ptr(packed), _lib.stream())
    return packed


def gemm_nt(a, b_kn, out, plan=None, tag='b', packed=None):
    """out[M, N] = a[M, K] @ b_kn[K, N] on the tensor cores with fp32-grade accuracy (K4b, 3xTF32).
    ``a`` and ``out`` are row-major (possibly row-strided views); ``b_kn`` is any strided [K, N] view of the small
    operand (a weight or its transpose): it is split and packed per call (a few KB)."""
    M, K = a.shape
    N = out.shape[1]
    if a.stride(1) != 1 or out.stride(1) != 1:
        raise ValueError('gemm_nt needs unit inner strides')
    if packed is None:                                  # ``packed``: the operand already split by kgc_conv_prep / _pack_b
        if tuple(b_kn.shape) != (K, N):
            raise ValueError('gemm_nt: b_kn must be [K, N] = [{}, {}]'.format(K, N))
        packed = _pack_b(b_kn, plan, 'gemm_pack_' + tag)
    # C is written by TMA stores: 16-byte aligned rows; an odd pitch goes through a padded buffer
    dst = out if (out.data_ptr() % 16 == 0 and out.stride(0) % 4 == 0) else \
        torch.empty((M, (N + 3) // 4 * 4), dtype=torch.float32, device=a.device)[:, :N]
    gemm_nt_batch([a], [packed], [dst])
    if dst is not out:
        out.copy_(dst)
    return out


def gemm_nt_batch(a_list, packed_list, out_list, keep=None, keep_scale=1.0):
    """Up to three products out_i = a_i @ B_i of identical shape in ONE launch (K4b); ``packed_list`` holds the split small
    operands (kgc_conv_prep / _pack_b).  ``keep`` (uint8 [M, pitch], kgc_tail_fwd's packed keep flags): dropout of the
    streamed operand while it is split - problem 0 by the low nibbles, problem 1 by the high nibbles, problem 2 as it is."""
    M, K = a_list[0].shape
    N = out_list[0].shape[1]
    lda, ldc = a_list[0].stride(0), out_list[0].stride(0)
    for a, o in zip(a_list, out_list):
        if a.shape != (M, K) or o.shape != (M, N) or a.stride() != (lda, 1) or o.stride() != (ldc, 1):
            raise ValueError('gemm_nt_batch needs operands of identical shape and strides')
    _lib.call('kgc_gemm_nt_batch', len(a_list), _ptr_array(a_list), M, K, lda, _ptr_array(packed_list), N, _ptr_array(out_list),
              ldc, _lib.ptr(keep), 0 if keep is None else keep.stride(0), float(keep_scale), _lib.stream())
    return out_list


def _gemm_tn_tc(a_list, b_list, out_list, M, plan, rows=None, keep=None, keep_scale=1.0):
    """One kgc_gemm_tn_tc_batch launch on operands the caller has checked."""
    n = len(a_list)
    Ka, Nb = a_list[0].shape[1], b_list[0].shape[1]
    nbytes = int(_lib.lib().kgc_gemm_tn_tc_workspace_bytes(M, Ka, Nb))
    ws = _workspace(plan, 'kgc_gemm_tn_tc_ws', nbytes, a_list[0].device)
    _lib.call('kgc_gemm_tn_tc_batch', n, _ptr_array(a_list), a_list[0].stride(0), _ptr_array(b_list), b_list[0].stride(0),
              None if rows is None else (ctypes.c_int64 * n)(*rows), M, Ka, Nb, _ptr_array(out_list), _lib.ptr(ws), nbytes,
              _lib.ptr(keep), 0 if keep is None else keep.stride(0), float(keep_scale), _lib.stream())


def gemm_tn_batch(a_list, b_list, out_list, plan=None, keep=None, keep_scale=1.0, rows=None):
    """Up to three weight-gradient reductions out_i = a_i^T @ b_i of identical shape in ONE launch (K4c on the tensor
    cores; Ka <= 128, Nb <= 224 - wider shapes go through gemm_tn one by one).  ``keep``: the b operands dropped while they
    are split, as in gemm_nt_batch.  ``rows``: rows[i] <= M leading rows of problem i (M = the operands' row count): the
    problems of M rows get exactly the bits they get without ``rows``; a shorter problem (a compacted plane) sums only the
    slabs its rows fill."""
    M = max(a.shape[0] for a in a_list)
    Ka, Nb = a_list[0].shape[1], b_list[0].shape[1]
    lda, ldb = a_list[0].stride(0), b_list[0].stride(0)
    fits = all(a.shape[1] == Ka and b.shape[1] == Nb and a.stride() == (lda, 1) and b.stride() == (ldb, 1) and o.is_contiguous()
               for a, b, o in zip(a_list, b_list, out_list))
    if rows is None:
        fits = fits and all(a.shape[0] == M and b.shape[0] == M for a, b in zip(a_list, b_list))
    elif not fits or max(rows) != M or any(a.shape[0] < r or b.shape[0] < r for a, b, r in zip(a_list, b_list, rows)):
        raise ValueError('gemm_tn_batch with rows needs operands of identical widths and strides and rows <= their heights')
    if not fits or Ka > GEMM_TN_TC_MAX_KA or Nb > GEMM_TN_TC_MAX_NB:    # one gemm_tn per problem
        if keep is not None:
            raise ValueError('gemm_tn_batch: the masked form needs Ka <= 128, Nb <= 224 and operands of identical shape')
        for i, (a, b, o) in enumerate(zip(a_list, b_list, out_list)):
            r = a.shape[0] if rows is None else rows[i]
            if r:
                gemm_tn(a[:r], b[:r], o, plan)
            else:
                o.zero_()
        return out_list
    _gemm_tn_tc(a_list, b_list, out_list, M, plan, rows, keep, keep_scale)
    return out_list


def rows_copy(src, src_rows, dst, dst_rows, n):
    """dst[dst_rows[j]] = src[src_rows[j]] for j < n (row lists int32 or None = the identity; one launch, none for n = 0)."""
    _lib.call('kgc_rows_copy', _lib.ptr(src), src.stride(0), _lib.ptr(src_rows), _lib.ptr(dst), dst.stride(0), _lib.ptr(dst_rows),
              int(n), src.shape[1], _lib.stream())


def gemm_nt_trans(a_t, b_kn, out_t):
    """out_t[N, M] = (a_t[K, M]^T @ b_kn[K, N])^T: K4b with the streamed operand and the result transposed in memory, so
    that the long dimension M is contiguous in both (M % 32 == 0, K <= 256)."""
    K, M = a_t.shape
    N = b_kn.shape[1]
    if a_t.stride(1) != 1 or out_t.stride(1) != 1 or out_t.shape != (N, M):
        raise ValueError('gemm_nt_trans needs unit inner strides and out_t of shape [N, M]')
    p = _lib.ptr
    _lib.call('kgc_gemm_nt_trans', p(a_t), M, K, a_t.stride(0), p(_pack_b(b_kn)), N, p(out_t), out_t.stride(0), _lib.stream())
    return out_t


def gemm_nt_splitk(a, bt, out):
    """out[Ma, Nb] = a[Ma, K] @ bt[Nb, K]^T for a long contraction K (split over the CTAs; Ma <= 128, Nb <= 224)."""
    Ma, K = a.shape
    Nb = bt.shape[0]
    if a.stride(1) != 1 or bt.stride(1) != 1 or not out.is_contiguous():
        raise ValueError('gemm_nt_splitk needs unit inner strides and a contiguous output')
    nbytes = int(_lib.lib().kgc_gemm_tn_tc_workspace_bytes(K, Ma, Nb))
    ws = torch.empty((nbytes // 4,), dtype=torch.float32, device=a.device)
    p = _lib.ptr
    _lib.call('kgc_gemm_nt_splitk', p(a), a.stride(0), p(bt), bt.stride(0), K, Ma, Nb, p(out), p(ws), nbytes, _lib.stream())
    return out


LINEAR_ROWS = 128       # rows of x per split-K forward / d_x launch (the kernels' Ma <= 128)
LINEAR_DW_ROWS = 256    # rows of the d_W contraction per launch (K <= 256); partials added in chunk order


class _LinearFn(torch.autograd.Function):
    """y = x @ W^T + b for a wide input (ConvE's fc, model.py:173: 39,200 -> 200) on the 3xTF32 tensor-core kernels:
    split-K forward, transposed-operand kernels for d_W and d_x.  Any batch: the forward and d_x run tile by tile over 128
    rows, d_W sums chunks of 256 rows in order (deterministic); up to 128 rows it is one launch each."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        x_, w_ = x.detach(), weight.detach()
        B = x_.shape[0]
        y = torch.empty((B, w_.shape[0]), dtype=torch.float32, device=x.device)
        for i in range(0, B, LINEAR_ROWS):
            gemm_nt_splitk(x_[i:i + LINEAR_ROWS], w_, y[i:i + LINEAR_ROWS])
        if bias is not None:
            y += bias.detach()
        ctx.save_for_backward(x_, w_)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        x, w = ctx.saved_tensors
        dy = dy.contiguous()
        dx = dw = db = None
        B = x.shape[0]
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            for i in range(0, B, LINEAR_ROWS):                          # d_x[B, F] = d_y @ W
                gemm_nt_trans(w, dy[i:i + LINEAR_ROWS].t(), dx[i:i + LINEAR_ROWS])
        if ctx.needs_input_grad[1]:
            dw = gemm_nt_trans(x[:LINEAR_DW_ROWS], dy[:LINEAR_DW_ROWS], torch.empty_like(w))   # d_W[O, F] = d_y^T @ x
            if B > LINEAR_DW_ROWS:
                part = torch.empty_like(w)
                for i in range(LINEAR_DW_ROWS, B, LINEAR_DW_ROWS):
                    dw += gemm_nt_trans(x[i:i + LINEAR_DW_ROWS], dy[i:i + LINEAR_DW_ROWS], part)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            db = dy.sum(0)
        return dx, dw, db


def linear_tc_supported(x, weight):
    B, F = x.shape
    O = weight.shape[0]
    return (x.is_cuda and x.dtype == torch.float32 and weight.dtype == torch.float32 and x.is_contiguous()
            and weight.is_contiguous() and B > 0 and O <= 224 and O % 4 == 0 and F % 32 == 0 and F >= 4096
            and x.data_ptr() % 16 == 0 and weight.data_ptr() % 16 == 0)


def linear_tc(x, weight, bias=None):
    """Differentiable y = x @ weight^T + bias on the tensor-core kernels (see linear_tc_supported for the shapes); any
    number of rows (tiles of 128)."""
    return _LinearFn.apply(x, weight, bias)


def gemm_tn(a, b, out, plan=None, tensor_cores=True):
    """out[Ka, Nb] = a[M, Ka]^T @ b[M, Nb] (K4c): the weight-gradient reduction over the node rows.  Tensor-core path
    (3xTF32, MN-major operands) for Ka <= 128, Nb <= 224; register-tiled fp32 FMA kernel for wider outputs.  Both add
    their per-CTA partials in a fixed order (deterministic)."""
    M, Ka = a.shape
    Nb = b.shape[1]
    if a.stride(1) != 1 or b.stride(1) != 1 or not out.is_contiguous():
        raise ValueError('gemm_tn needs unit inner strides and a contiguous output')
    if Nb > 256:
        raise ValueError('gemm_tn supports Nb <= 256')
    for i0 in range(0, Ka, 128):                       # wider A: one call per block of 128 columns (= 128 contiguous rows of out)
        kb = min(128, Ka - i0)
        a_blk, out_blk = a[:, i0:i0 + kb], out[i0:i0 + kb]
        if tensor_cores and Nb <= 224:
            _gemm_tn_tc([a_blk], [b], [out_blk], M, plan)
        else:
            nbytes = int(_lib.lib().kgc_gemm_tn_workspace_bytes(M, kb, Nb))
            ws = _workspace(plan, 'kgc_gemm_tn_ws', nbytes, a.device)
            p = _lib.ptr
            _lib.call('kgc_gemm_tn', p(a_blk), a.stride(0), p(b), b.stride(0), M, kb, Nb, p(out_blk), p(ws), nbytes, _lib.stream())
    return out


class _Done(object):
    """Stand-in for an async work handle whose work is already ordered on the current stream."""

    def wait(self):
        return None


class _StreamJoin(object):
    """Work handle of kernels issued on another CUDA stream: wait() makes the current stream wait for them."""

    def __init__(self, stream):
        self.stream = stream

    def wait(self):
        torch.cuda.current_stream().wait_stream(self.stream)


class _Collectives(object):
    """The four exchanges of the dst-partitioned layer (SURVEY.md 8(e)); ``None`` context = single GPU."""

    def __init__(self, group, world, n_global, n_hub=0, hub_idx_mine=None, hub_rows_mine=None, p2p=None, rank=0,
                 halo_rows=None, n_loc=None):
        self.group, self.world, self.n_global, self.rank = group, int(world), int(n_global), int(rank)
        # row stride of a rank's block of real rows (None: the caller's x has exactly that many rows).  When the node count
        # is not a multiple of the number of ranks some ranks hold n_loc - 1 real rows; rows n_real .. n_loc do not exist
        self.n_loc = None if n_loc is None else int(n_loc)
        self.p2p = p2p          # partition._P2PContext: halo exchange over NVLink peer memory (K10) instead of NCCL
        # edge-balanced partitions number a rank's node table COMPACTLY: its own block, then the remote rows it reads
        # (halo_rows = their ids in the gathered layout); None = range partition (table = all rows, global ids)
        self.halo_rows = halo_rows
        # split hub rows of an edge-balanced partition (partition.py): every rank accumulates a share of a hub's incoming
        # edges into a private virtual row (local rows n_loc .. n_loc + n_hub); hub_idx_mine / hub_rows_mine = the hubs this
        # rank owns and their real local rows
        self.n_hub, self.hub_idx_mine, self.hub_rows_mine = int(n_hub), hub_idx_mine, hub_rows_mine

    def sum_hub_rows(self, planes, n_loc):
        """planes [P, n_loc + n_hub, D]: virtual rows summed over ranks, result added into the owners' real rows."""
        if self.n_hub == 0:
            return
        buf = planes[:, n_loc:, :].contiguous()
        self.all_reduce(buf, 'hub_f')
        if self.hub_idx_mine.numel():
            planes[:, self.hub_rows_mine, :] = buf[:, self.hub_idx_mine, :]

    def spread_hub_rows(self, planes, n_planes, n_loc):
        """The inverse for the backward: every rank's virtual rows receive planes[:n_planes] of the hubs' real rows."""
        if self.n_hub == 0:
            return
        buf = torch.zeros((n_planes, self.n_hub, planes.shape[2]), dtype=planes.dtype, device=planes.device)
        if self.hub_idx_mine.numel():
            buf[:, self.hub_idx_mine, :] = planes[:n_planes, self.hub_rows_mine, :]
        self.all_reduce(buf, 'hub_b')                          # every entry is non-zero on one rank: exact
        planes[:n_planes, n_loc:, :] = buf

    def all_gather_rows(self, x_local, async_op=False):
        import torch.distributed as dist
        out = torch.empty((self.world * x_local.shape[0],) + tuple(x_local.shape[1:]), dtype=x_local.dtype,
                          device=x_local.device)
        work = dist.all_gather_into_tensor(out, x_local.contiguous(), group=self.group, async_op=async_op)
        return (out, work) if async_op else out

    def gather_compact(self, x_blk):
        """Library path of the compact node table: all-gather every block, keep own block + the halo rows."""
        full = self.all_gather_rows(x_blk)
        return torch.cat([x_blk, full.index_select(0, self.halo_rows)], 0)

    def reduce_compact(self, partial, block):
        """Library path back: compact partial d_x -> dense gathered layout -> reduce-scatter -> this rank's block."""
        full = partial.new_zeros((self.world * block, partial.shape[1]))
        full[self.rank * block:(self.rank + 1) * block] = partial[:block]
        full[self.halo_rows] = partial[block:block + self.halo_rows.numel()]
        return self.reduce_scatter_rows(full)

    def reduce_scatter_rows(self, full, async_op=False):
        import torch.distributed as dist
        rows = full.shape[0] // self.world
        if dist.get_backend(self.group) == 'gloo':       # gloo (CPU tests of the host logic) has no reduce-scatter
            dist.all_reduce(full, group=self.group)
            r = dist.get_rank(self.group)
            out = full[r * rows:(r + 1) * rows].clone()
            return (out, None) if async_op else out
        out = torch.empty((rows,) + tuple(full.shape[1:]), dtype=full.dtype, device=full.device)
        work = dist.reduce_scatter_tensor(out, full.contiguous(), group=self.group, async_op=async_op)
        return (out, work) if async_op else out

    def all_reduce(self, t, tag=None):
        """Sum over the ranks, in place.  With the peer-memory context and a call-site ``tag``: the one-shot K10 kernel
        (stage + flag barrier + add in rank order, ~1 launch instead of an NCCL ring); otherwise NCCL / gloo."""
        if self.p2p is not None and tag is not None and self.p2p.all_reduce(t, tag):
            return t
        import torch.distributed as dist
        dist.all_reduce(t, group=self.group)
        return t


class _ConvFn(torch.autograd.Function):

    @staticmethod
    def forward(ctx, x, rels, ee, w_in, w_out, w_loop, w_rel, loop_rel, loop_edge, gamma, beta, bias,
                plan, mask_in, mask_out, keep_scale, training, running_mean, running_var, eps, coll, seed, drop_p,
                bn_track=None, out_drop=None):
        # x: this rank's node rows [Nl, D] (all rows on one GPU); ee: the rows of the edges this rank owns
        Nl, D = x.shape
        Dout = w_in.shape[1]
        p, st = _lib.ptr, _lib.stream
        x = _lib.require_cuda(x, torch.float32, 'x')
        ee = _lib.require_cuda(ee, torch.float32, 'edge_embs')
        n_global = Nl if coll is None else coll.n_global
        n_hub = 0 if coll is None else coll.n_hub           # virtual rows of split hubs follow the block of real rows
        n_loc = Nl if coll is None or coll.n_loc is None else coll.n_loc      # block stride: Nl or Nl + 1 (uneven counts)
        if not 0 <= n_loc - Nl <= 1:
            raise ValueError('x has {} rows, the partition expects {} or {}'.format(Nl, n_loc, n_loc - 1))
        Nb = n_loc + n_hub
        compact = coll is not None and coll.halo_rows is not None
        n_table = Nl if coll is None else (Nb + coll.halo_rows.numel() if compact else Nb * coll.world)
        # hybrid cut (partition.partition_edges_hybrid): remote rows are destinations too - every table row can be written
        hybrid = coll is not None and coll.p2p is not None and coll.p2p.hybrid
        n_dst = n_table if hybrid else Nb
        if ee.shape[0] != plan.num_edges2 or n_dst != plan.num_dst_rows or plan.num_nodes != n_table:
            raise ValueError('edge_embs / x do not match the graph plan')
        T = rels.shape[0] + 1
        if T != plan.num_types:
            raise ValueError('rels_embs rows + 1 must equal the number of edge types of the plan')
        # K0: cat(rels, loop_rel) (model.py:86), relp @ w_rel (model.py:107) and the TF32 packs of the six small GEMM
        # operands of this step (forward and backward) in one launch
        nf = int(_lib.lib().kgc_gemm_packed_b_bytes(Dout, D)) // 4
        nbk = int(_lib.lib().kgc_gemm_packed_b_bytes(D, Dout)) // 4
        if nf == 0 or nbk == 0:
            raise ValueError('unsupported layer width {} -> {} (<= 256)'.format(D, Dout))
        relp = torch.empty((T, D), dtype=torch.float32, device=x.device)
        all_rel_pad = torch.empty((T, Dout), dtype=torch.float32, device=x.device)
        packed_f = torch.empty((3, nf), dtype=torch.float32, device=x.device)
        packed_b = torch.empty((4, nbk), dtype=torch.float32, device=x.device)
        rels_c, wts = rels.detach().contiguous(), [w.detach().contiguous() for w in (w_in, w_out, w_loop, w_rel)]
        # ... on a side stream: the aggregation below reads the relation rows straight from `rels` (real edges never carry
        # the self-loop type), so K0 leaves the critical path; the main stream joins before the first dense transform
        main, side = torch.cuda.current_stream(), plan.side_stream()
        side.wait_stream(main)
        with torch.cuda.stream(side):
            _lib.call('kgc_conv_prep', p(rels_c), T - 1, p(loop_rel.detach()), p(loop_edge.detach()), p(wts[0]), p(wts[1]),
                      p(wts[2]), p(wts[3]), D, Dout, p(relp), p(all_rel_pad), p(packed_f), p(packed_b), st())
        # halo exchange: every rank needs the source rows of its edges (all-gather of the row partition); it runs on
        # NCCL's stream while this rank's self-loop transform (which only needs its own rows) runs here
        gather = None
        if coll is None:
            x_full = x
        elif coll.p2p is not None:
            # K10: publish this rank's rows, barrier, pull exactly the remote rows its records reference (peer loads) - on the
            # exchange stream, next to K0 and the self-loop transform of this rank's own rows (NVLink-bound vs tensor-bound)
            ex = coll.p2p.exchange_stream
            ex.wait_stream(main)
            with torch.cuda.stream(ex):
                x_full = coll.p2p.gather(x, fence=not training)
            gather = _StreamJoin(ex)
        elif compact:                                               # library fallback of the compact table
            x_blk = x if Nb == Nl else torch.cat([x, x.new_zeros((Nb - Nl, D))], 0)
            x_full, gather = coll.gather_compact(x_blk), _Done()
        else:
            x_full, gather = coll.all_gather_rows(x if Nb == Nl else torch.cat([x, x.new_zeros((Nb - Nl, D))], 0),
                                                  async_op=True)

        res3 = plan.scratch('res3', (3, Nl, Dout))
        if gather is not None:                                      # self-loop: (x . lr . le) @ W = x @ (diag(lr . le) W)
            main.wait_stream(side)
            gemm_nt(x, None, res3[2], packed=packed_f[2])          # overlaps the all-gather
            gather.wait()
        if max(x_full.shape[0], 3 * n_dst, ee.shape[0]) * (D // 4) >= 1 << 32:      # K2/K3 use 32-bit float4 indices
            raise ValueError('kgc_gcn_b200: node / edge tables of 2^32 float4 elements or more are not supported')
        agg_c, res_c = [None, None], [None, None]                   # compacted halves: [n_c, D] rows and their transforms
        # one GPU: a half whose rows are mostly without edges (plan.compact_halves) runs its dense transform, its share of the
        # tail and its weight gradient on its occupied rows only (plan.rows / plan.slot); its other rows are never read, so
        # the aggregation does not zero-fill them
        comp = plan.compact_halves(4 * Dout) if coll is None else (False, False)
        # one GPU, hub-heavy graph (plan.grouped, GroupedPlan): the in half is aggregated per (object, type) group into the
        # rows P behind the two planes, without the relation factor (its records name a row of ones), and agg_in = sum_t
        # rel[t] (.) P[o, t] follows; the backward reuses P for d_rel
        grp = plan.grouped if coll is None else None
        agg_all = torch.empty((2 * n_dst + (grp.n_in if grp is not None else 0), D), dtype=torch.float32, device=x.device)
        agg = agg_all[:2 * n_dst].view(2, n_dst, D)
        if grp is None:
            def level0(sp, out_final, carry):
                _lib.call('kgc_agg_fwd', p(x_full), p(rels_c), T - 1, p(ee), p(plan.rec_dst), p(sp.rowflags), p(sp.chunks),
                          sp.n_rec, p(out_final), p(carry), D, st())
            plan.run_reduction(plan.fwd, level0, agg, D, tag='f',
                               skip_prefill=[(h * n_dst, (h + 1) * n_dst) for h in (0, 1) if comp[h]])
        else:
            rel_f = torch.cat([rels_c, rels_c.new_ones((1, D))], 0)      # row T - 1 = grp.ones_row

            def level0(sp, out_final, carry):
                _lib.call('kgc_agg_fwd', p(x_full), p(rel_f), T, p(ee), p(grp.rec_f), p(sp.rowflags), p(sp.chunks), sp.n_rec,
                          p(out_final), p(carry), D, st())
            plan.run_reduction(grp.fwd, level0, agg_all, D, tag='fg', skip_prefill=[(n_dst, 2 * n_dst)] if comp[1] else ())
            P = agg_all[2 * n_dst:]
            if comp[0]:                                             # agg_in straight into the compacted rows
                agg_c[0] = torch.empty((max(plan.n_c[0], 1), D), dtype=torch.float32, device=x.device)
                grp.agg_in_c.run(plan, P, rels_c, agg_c[0], D, tag='gi')
            else:
                agg[0].zero_()
                grp.agg_in.run(plan, P, rels_c, agg[0], D, tag='gi')
        if gather is None:
            main.wait_stream(side)                                  # K0's operand packs are needed from here on

        if hybrid:
            coll.p2p.reduce_agg(agg)                                # K10: the owners add the partial rows of the other ranks (rank order)
        if gather is not None:
            coll.sum_hub_rows(agg, n_loc)
            gemm_nt_batch([agg[0, :Nl], agg[1, :Nl]], [packed_f[0], packed_f[1]], [res3[0], res3[1]])
        elif not any(comp):                                         # the three transforms of the step in one launch
            gemm_nt_batch([agg[0], agg[1], x], [packed_f[0], packed_f[1], packed_f[2]], [res3[0], res3[1], res3[2]])
        else:
            # a compacted half: its occupied rows gathered into [n_c, D] and transformed on their own (a launch of n_c rows;
            # sharing the batched launch would leave its CTAs idle), the dense planes in one launch
            dense = [h for h in (0, 1) if not comp[h]]
            for h in (0, 1):
                if comp[h]:
                    n_c = plan.n_c[h]
                    res_c[h] = plan.scratch('res_c%d' % h, (max(n_c, 1), Dout))
                    if agg_c[h] is None:
                        agg_c[h] = torch.empty((max(n_c, 1), D), dtype=torch.float32, device=x.device)
                        if n_c:
                            rows_copy(agg[h], plan.rows[h], agg_c[h], None, n_c)
                    if n_c:
                        gemm_nt(agg_c[h][:n_c], None, res_c[h][:n_c], packed=packed_f[h])
            gemm_nt_batch([agg[h] for h in dense] + [x], [packed_f[h] for h in dense] + [packed_f[2]],
                          [res3[h] for h in dense] + [res3[2]])

        nb = int(_lib.lib().kgc_tail_num_blocks(Nl))
        partials = plan.scratch('colpart', (nb, 2, Dout), torch.float64)
        sums = torch.empty((2, Dout), dtype=torch.float64, device=x.device)
        pre = torch.empty((Nl, Dout), dtype=torch.float32, device=x.device)
        stats = torch.empty((3, Dout), dtype=torch.float32, device=x.device)
        all_ent = torch.empty((Nl, Dout), dtype=torch.float32, device=x.device)
        # keep flags of the two dropped planes, one byte per four columns: the backward GEMMs apply them while they split the
        # ONE upstream plane (no masked planes are written, nothing is regenerated)
        dropping = (mask_in is not None or seed is not None) and drop_p > 0.0
        keep = torch.empty((Nl, int(_lib.lib().kgc_keep_pitch())), dtype=torch.uint8, device=x.device) if dropping else None
        _lib.call('kgc_tail_fwd', p(res3), p(plan.slot[0]) if comp[0] else None, p(res_c[0]), p(plan.slot[1]) if comp[1] else None,
                  p(res_c[1]), p(mask_in), p(mask_out), p(seed), float(drop_p), float(keep_scale), p(bias), Nl, Dout, p(pre),
                  p(partials), p(keep), st())
        if training and coll is None:
            # one GPU: column sums -> batch statistics -> nn.BatchNorm1d's running-statistics bookkeeping in ONE launch
            # (bn_track = (momentum, num_batches_tracked) when the module tracks running statistics)
            mom, nbt = bn_track if bn_track is not None else (0.0, None)
            _lib.call('kgc_colstats_finalize', p(partials), nb, n_global, Dout, float(eps), float(mom),
                      p(running_mean) if bn_track is not None else None, p(running_var) if bn_track is not None else None,
                      p(nbt), None, p(stats), st())
        else:
            if training:
                _lib.call('kgc_colsum_finalize', p(partials), nb, Dout, p(sums), st())
                coll.all_reduce(sums, 'bn_f')                        # BatchNorm statistics over ALL node rows
            _lib.call('kgc_colstats_from_sums', p(sums), n_global, Dout, float(eps), int(training), p(running_mean),
                      p(running_var), p(stats), st())
        # out_drop = (p, seed): MGCN.encode's F.dropout(all_ent, gcn_drop) (model.py:34) in the same pass
        out_p, out_seed = out_drop if out_drop is not None else (0.0, None)
        out_keep = torch.empty((Nl, int(_lib.lib().kgc_keep_pitch())), dtype=torch.uint8, device=x.device) if out_seed is not None else None
        _lib.call('kgc_tail_apply', p(pre), p(stats), p(gamma), p(beta), Nl, Dout, p(all_ent), p(out_seed), float(out_p),
                  p(out_keep), st())
        ctx.out_scale = 1.0 / (1.0 - float(out_p)) if out_seed is not None else 1.0
        all_rel = all_rel_pad[:-1]

        ctx.plan, ctx.training, ctx.keep_scale, ctx.has_bias, ctx.coll = plan, bool(training), float(keep_scale), \
            bias is not None, coll
        ctx.drop_p = float(drop_p)
        ctx.comp, ctx.grp = comp, grp
        ctx.save_for_backward(x, x_full, relp, ee, w_in, w_out, w_loop, w_rel, loop_rel, loop_edge, gamma, beta, agg_all, pre,
                              all_ent, stats, keep, packed_b, out_keep, agg_c[0], agg_c[1])
        ctx.mark_non_differentiable(stats)
        return all_ent, all_rel, stats

    @staticmethod
    def backward(ctx, g_ent, g_rel, _g_stats):
        (x, x_full, relp, ee, w_in, w_out, w_loop, w_rel, loop_rel, loop_edge, gamma, beta, agg_all, pre, all_ent, stats, keep,
         packed_b, out_keep, agg_c0, agg_c1) = ctx.saved_tensors
        plan, coll, comp, grp = ctx.plan, ctx.coll, ctx.comp, ctx.grp
        agg = agg_all[:2 * plan.num_dst_rows].view(2, plan.num_dst_rows, -1)
        Nl, D = x.shape
        n_global = Nl if coll is None else coll.n_global      # BatchNorm rows (real nodes of all ranks)
        n_hub = 0 if coll is None else coll.n_hub
        n_loc = Nl if coll is None or coll.n_loc is None else coll.n_loc
        Nb = n_loc + n_hub
        Dout = w_in.shape[1]
        T = relp.shape[0]
        p, st = _lib.ptr, _lib.stream
        dev = x.device
        if g_ent is None:
            g_ent = torch.zeros_like(all_ent)
        g_ent = g_ent.contiguous()

        # ---- K4 backward: tanh, BatchNorm, /3, dropout
        nb = int(_lib.lib().kgc_tail_num_blocks(Nl))
        partials = plan.scratch('colpart', (nb, 2, Dout), torch.float64)
        sums = torch.empty((2, Dout), dtype=torch.float64, device=dev)
        d_out = plan.scratch('d_out', (Nl, Dout))          # ONE upstream plane (d out / 3); the GEMMs apply the keep flags
        _lib.call('kgc_tail_bwd_reduce', p(g_ent), p(pre), p(stats), p(gamma), p(beta), Nl, Dout, p(partials), p(out_keep),
                  ctx.out_scale, st())
        if coll is None:
            sums32 = torch.empty((2, Dout), dtype=torch.float32, device=dev)
            _lib.call('kgc_colsum_finalize2', p(partials), nb, Dout, p(sums), p(sums32), st())
        else:
            _lib.call('kgc_colsum_finalize', p(partials), nb, Dout, p(sums), st())
            coll.all_reduce(sums, 'bn_b')
            sums32 = sums.float()
        # the in / out halves' upstream planes: three planes or one masked plane by size and width (TAIL_MASKED_MAX_BYTES,
        # GEMM_TN_TC_MAX_*).  A compacted half always takes the three-plane form: its upstream rows are written compact, [n_c, Dout].
        three = 3 * Nl * Dout * 4 > TAIL_MASKED_MAX_BYTES or D > GEMM_TN_TC_MAX_KA or Dout > GEMM_TN_TC_MAX_NB or any(comp)
        d_res = [(plan.scratch('d_res_c%d' % h, (max(plan.n_c[h], 1), Dout)) if comp[h] else plan.scratch('d_res2_%d' % h, (Nl, Dout)))
                 if three else None for h in (0, 1)]
        _lib.call('kgc_tail_bwd_apply', p(g_ent), p(pre), p(stats), p(gamma), p(beta), p(sums), int(ctx.training), Nl,
                  n_global, Dout, p(d_out), p(keep), ctx.keep_scale, p(d_res[0]), p(plan.slot[0]) if comp[0] else None,
                  p(d_res[1]), p(plan.slot[1]) if comp[1] else None, p(out_keep), ctx.out_scale, st())
        ups = [d_res[0], d_res[1], d_out] if three else [d_out, d_out, d_out]
        gkeep = None if three else keep
        d_beta, d_gamma = sums32[0], sums32[1]

        # replicated-parameter gradients: one flat buffer so that a partitioned run needs ONE all-reduce
        flat = torch.empty((3 * D * Dout + T * D + (Dout if ctx.has_bias else 0),), dtype=torch.float32, device=dev)
        d_w_in, d_w_out, m_loop = (flat[k * D * Dout:(k + 1) * D * Dout].view(D, Dout) for k in range(3))
        d_relp = flat[3 * D * Dout:3 * D * Dout + T * D].view(T, D)
        # weight-gradient reductions over the node rows (K4c on the tensor cores, deterministic).  Nothing on the d_x / d_ee /
        # d_rel chain below needs them: on one GPU they run on the side stream next to that chain (a K4c CTA leaves room for
        # one aggregation CTA per SM) and the main stream joins before the parameter-gradient kernel
        main, side = torch.cuda.current_stream(), plan.side_stream()
        side.wait_stream(main)
        with torch.cuda.stream(side):
            agg_c = (agg_c0, agg_c1)                            # a compacted half sums its n_c rows
            gemm_tn_batch([agg_c[h] if comp[h] else agg[h, :Nl] for h in (0, 1)] + [x], ups, [d_w_in, d_w_out, m_loop], plan,
                          keep=gkeep, keep_scale=ctx.keep_scale,
                          rows=[plan.n_c[h] if comp[h] else Nl for h in (0, 1)] + [Nl] if any(comp) else None)   # [D, Dout] each
            if ctx.has_bias:
                torch.sum(d_out, 0, out=flat[3 * D * Dout + T * D:])

        # ---- d(agg) = d_res @ W^T on the tensor cores (3xTF32), main stream
        hybrid = coll is not None and coll.p2p is not None and coll.p2p.hybrid
        if grp is None:
            g3 = coll.p2p.g3_planes() if hybrid else plan.scratch('g3', (3, Nb, D))
        else:
            # the grouped d_x pass takes the self-loop plane as addend on its node rows and the zero rows behind it on its
            # group rows (never written after allocation)
            g3_all = plan.scratch('g3grp', (3 * Nb + grp.n_out, D), zeros=True)
            g3 = g3_all[:3 * Nb].view(3, Nb, D)
        if not any(comp):
            gemm_nt_batch(ups, [packed_b[0], packed_b[1], packed_b[2]],
                          [g3[0, :Nl], g3[1, :Nl], g3[2, :Nl]], keep=gkeep, keep_scale=ctx.keep_scale)
        else:
            # a compacted half: d(agg) of its occupied rows, scattered into their rows of g3 (the only rows of that plane the
            # aggregation backward reads: its edges' destinations)
            dense = [h for h in (0, 1) if not comp[h]]
            for h in (0, 1):
                n_c = plan.n_c[h]
                if comp[h] and n_c:
                    g3_c = plan.scratch('g3_c%d' % h, (n_c, D))
                    gemm_nt(d_res[h][:n_c], None, g3_c, packed=packed_b[h])
                    rows_copy(g3_c, None, g3[h], plan.rows[h], n_c)
            gemm_nt_batch([ups[h] for h in dense] + [d_out], [packed_b[h] for h in dense] + [packed_b[2]],
                          [g3[h, :Nl] for h in dense] + [g3[2, :Nl]])
        if n_hub:
            coll.spread_hub_rows(g3, 2, n_loc)                       # the virtual rows see their hub's upstream gradient
        if hybrid:
            coll.p2p.gather_g()                                      # K10: upstream rows of the remote destinations, from their owners
        # ---- K3: d_x (+ self-loop term) and d_ee over src-sorted rows, d_rel over type-sorted rows
        p2p = None if coll is None else coll.p2p
        d_ee = torch.empty_like(ee)
        if grp is not None:
            # d_x / d_ee over the grouped src stream: d_x of the in-half records and the out-half group rows Q behind it; then
            # d_x += rel (.) Q and d_rel from the group rows - no second pass over the edge table
            dxq = torch.empty((plan.num_nodes + grp.n_out, D), dtype=torch.float32, device=dev)
            d_x_full, Q = dxq[:plan.num_nodes], dxq[plan.num_nodes:]
            addend_g = g3_all[2 * Nb:]

            def level0_src(sp, out_final, carry):
                _lib.call('kgc_agg_bwd_src_grouped', p(x_full), p(relp), T, p(ee), p(g3), p(grp.rec_s), p(sp.rowflags),
                          p(grp.xrow_s), p(sp.chunks), sp.n_rec, plan.num_dst_rows, plan.num_edges_in, grp.n_out, p(addend_g),
                          p(d_ee), p(out_final), p(carry), D, st())
            plan.run_reduction(grp.src, level0_src, dxq, D, addend=addend_g, tag='sg')
            grp.dx.run(plan, Q, relp, d_x_full, D, accumulate=True, tag='gx')
            P = agg_all[2 * plan.num_dst_rows:]
            grp.drel_in.run(plan, P, g3[0], d_relp, D, tag='gri')
            grp.drel_out.run(plan, Q, x_full, d_relp, D, accumulate=True, tag='gro')
        else:
            d_x_full = p2p.partial if (p2p is not None and not hybrid) else torch.empty((plan.num_nodes, D), dtype=torch.float32,
                                                                                        device=dev)
            # self-loop term: added by the aggregation itself when its output rows are final (one GPU; hybrid cut: the remote
            # rows of plane 2 are zero), otherwise by the owner-side reduction
            loop_addend = g3[2] if (coll is None or hybrid) else None

            def level0_src(sp, out_final, carry):
                _lib.call('kgc_agg_bwd_src', p(x_full), p(relp), relp.shape[0], p(ee), p(g3), p(plan.rec_src), p(sp.rowflags),
                          p(sp.chunks), sp.n_rec, plan.num_dst_rows, plan.num_edges_in, p(loop_addend), p(d_ee), p(out_final),
                          p(carry), D, st())
            plan.run_reduction(plan.bwd_src, level0_src, d_x_full, D, addend=loop_addend, tag='s')
        scatter = None
        if hybrid:
            # K10 on the exchange stream: partial rows of the remote sources to symmetric memory, barrier (own channel), the
            # owners add the other ranks' partial rows to the few rows that have any - next to the d_rel pass
            ex = p2p.exchange_stream
            ex.wait_stream(main)
            with torch.cuda.stream(ex):
                p2p.reduce_dx(d_x_full, channel=1)
            d_x = d_x_full[:Nl]
        elif p2p is not None:
            # K10 on the exchange stream, next to the d_rel pass and the replicated-gradient all-reduce of the main stream:
            # barrier (own channel), then every owner pulls the partial rows of the ranks that touched its rows (rank order,
            # deterministic) and adds the self-loop term - reduce-scatter + add in one kernel over peer memory
            d_x = torch.empty((Nl, D), dtype=torch.float32, device=dev)
            ex = p2p.exchange_stream
            ex.wait_stream(main)
            with torch.cuda.stream(ex):
                p2p.reduce(g3[2, :Nl], Nl, out=d_x, channel=1)
        compact = coll is not None and coll.halo_rows is not None
        if coll is not None and p2p is None and not compact:   # source-row gradients go back to their owners while the d_rel pass runs
            d_x, scatter = coll.reduce_scatter_rows(d_x_full, async_op=True)

        if grp is None:
            def level0_rel(sp, out_final, carry):
                _lib.call('kgc_agg_bwd_rel', p(x_full), p(ee), p(g3), p(plan.rec_type), p(sp.rowflags), p(sp.chunks), sp.n_rec,
                          plan.num_dst_rows, plan.num_edges_in, p(out_final), p(carry), D, st())
            plan.run_rel_reduction(level0_rel, d_relp, D)

        main.wait_stream(side)                                        # the weight gradients are part of `flat`
        if coll is None:
            d_x = d_x_full
        elif p2p is not None:
            coll.all_reduce(flat, 'flat')
            main.wait_stream(p2p.exchange_stream)
        elif compact:
            coll.all_reduce(flat, 'flat')
            d_x = coll.reduce_compact(d_x_full, Nb)[:Nl] + g3[2, :Nl]
        else:
            coll.all_reduce(flat, 'flat')
            if scatter is not None:
                scatter.wait()
            d_x = d_x[:Nl] + g3[2, :Nl]                               # self-loop term of this rank's (real) rows
        d_bias = flat[3 * D * Dout + T * D:] * 3.0 if ctx.has_bias else None
        # K0 backward: self-loop vectors, relation transform (model.py:107; replicated inputs, identical on every rank)
        small = torch.empty((2 * D * Dout + 2 * D + (T - 1) * D,), dtype=torch.float32, device=dev)
        d_w_loop, d_w_rel = small[:D * Dout].view(D, Dout), small[D * Dout:2 * D * Dout].view(D, Dout)
        o = 2 * D * Dout
        d_loop_rel, d_loop_edge, d_rels = small[o:o + D].view(1, D), small[o + D:o + 2 * D].view(1, D), small[o + 2 * D:].view(T - 1, D)
        g_rel_c = None if g_rel is None else g_rel.contiguous()
        rel_add = None
        if g_rel_c is not None and T - 1 >= 256 and g_rel_c.data_ptr() % 16 == 0 and Dout % 4 == 0 and (D * Dout) % 32 == 0:
            # many relations (Wikidata5M shape: 1,644 rows): the two products over the relation rows on the tensor cores
            rel_add = gemm_nt(g_rel_c, None, torch.empty((T - 1, D), dtype=torch.float32, device=dev), packed=packed_b[3])
            gemm_tn(relp[:T - 1], g_rel_c, d_w_rel, plan)
        _lib.call('kgc_conv_param_grads', p(m_loop), p(w_loop.detach().contiguous()), p(loop_rel.detach()), p(loop_edge.detach()),
                  p(relp), p(w_rel.detach().contiguous()), p(g_rel_c), p(d_relp), T - 1, D, Dout, p(d_w_loop), p(d_loop_rel),
                  p(d_loop_edge), p(d_rels), p(d_w_rel), p(rel_add), st())
        return (d_x, d_rels, d_ee, d_w_in, d_w_out, d_w_loop, d_w_rel, d_loop_rel, d_loop_edge, d_gamma, d_beta, d_bias,
                None, None, None, None, None, None, None, None, None, None, None, None, None)


class MGCNConv(nn.Module):
    """Drop-in for the reference MGCNConv (model.py:47-127): same ctor, parameters, forward."""

    def __init__(self, in_channels, out_channels, num_relations, bias=False, dropout=0.1, **kwargs):
        super(MGCNConv, self).__init__()
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.num_relations = num_relations
        self.aggr = 'add'

        self.ent_bn = nn.BatchNorm1d(out_channels)
        self.drop = nn.Dropout(dropout)
        self.act = torch.tanh

        self.loop_weight = get_param((in_channels, out_channels))
        self.in_weight = get_param((in_channels, out_channels))
        self.out_weight = get_param((in_channels, out_channels))
        self.rels_weight = get_param((in_channels, out_channels))
        self.loop_rel = get_param((1, in_channels))
        self.loop_edge = get_param((1, in_channels))

        if bias is True:
            self.register_parameter('bias', nn.Parameter(torch.zeros(out_channels)))
        else:
            self.register_parameter('bias', None)
        self._forced_masks = None
        # dropout stream of the CUDA path: a device-resident counter (not part of the state dict); every training
        # forward advances it and the tail kernels key a Philox4x32-10 generator with it (K4, no mask tensors)
        self.register_buffer('_drop_seed', torch.zeros(1, dtype=torch.int64), persistent=False)
        self._drop_seeded = False

    def set_dropout_masks(self, mask_in, mask_out):
        """Inject the two keep masks ([N, Dout], 0/1) the next training forward uses instead of drawing
        them - the parity tests replay the reference's own Bernoulli draws this way.  None clears."""
        self._forced_masks = None if mask_in is None else (mask_in, mask_out)

    def compute_norm(self, edge_index, num_ent):
        """model.py:72-80 for one half's edge_index [2, E_h]; evaluated by K1."""
        ei = torch.cat([edge_index, edge_index], 1).contiguous()
        et = torch.zeros(ei.size(1), dtype=torch.int64, device=ei.device)
        return get_plan(ei, et, num_ent, 1).norm[:edge_index.size(1)].clone()

    def _masks(self, n_rows, device):
        """-> (mask_in, mask_out, keep_scale, seed, drop_p).  Training with p > 0: injected masks if set, otherwise a
        fresh seed for the in-kernel counter-based generator (first seed drawn from torch's generator, so
        torch.manual_seed makes runs reproducible)."""
        p = self.drop.p
        if not self.training or p == 0.0:
            return None, None, 1.0, None, 0.0
        if self._forced_masks is not None:
            m_in, m_out = self._forced_masks
            return (m_in.to(device=device, dtype=torch.uint8).contiguous(),
                    m_out.to(device=device, dtype=torch.uint8).contiguous(), 1.0 / (1.0 - p), None, p)
        if not self._drop_seeded:
            self._drop_seed.fill_(int(torch.randint(0, 2 ** 62, (1,)).item()))
            self._drop_seeded = True
        self._drop_seed.add_(0x9E3779B97F4A7C15 & 0x7FFFFFFFFFFFFFFF)     # new stream every step (device op: graph-capturable)
        return None, None, 1.0 / (1.0 - p), self._drop_seed.clone(), p

    def _out_drop_cfg(self, p, seed):
        """(p, seed) of the output dropout of this forward, or None.  It shares the tail's Philox seed (plane 2); when the
        tail itself does not draw (p = 0 or injected masks) the seed counter is advanced here."""
        if not self.training or not p or p <= 0.0:
            return None
        if seed is None:
            if not self._drop_seeded:
                self._drop_seed.fill_(int(torch.randint(0, 2 ** 62, (1,)).item()))
                self._drop_seeded = True
            self._drop_seed.add_(0x9E3779B97F4A7C15 & 0x7FFFFFFFFFFFFFFF)
            seed = self._drop_seed.clone()
        self._last_out_seed = seed
        return float(p), seed

    def dropout_masks(self, seed, n_rows):
        """The two keep masks [n_rows, Dout] the tail kernels derive from ``seed`` (int64 device tensor): for tests."""
        out = []
        for plane in (0, 1):
            m = torch.empty((n_rows, self.out_channels), dtype=torch.uint8, device=seed.device)
            _lib.call('kgc_dropout_mask', _lib.ptr(seed), plane, float(self.drop.p), m.numel(), _lib.ptr(m), _lib.stream())
            out.append(m)
        return out

    def forward(self, x, edge_index, edge_type, edge_norm, edge_embs, rels_embs, size=None, _out_drop=0.0):
        # edge_norm and size are accepted and ignored, exactly as the reference does (model.py:82, SURVEY fact 6).
        # _out_drop (private, used by MGCN.encode): dropout probability applied to all_ent inside the tail kernel
        num_ent = x.size(0)
        plan = get_plan(edge_index, edge_type, num_ent, rels_embs.size(0) + 1)
        m_in, m_out, keep_scale, seed, drop_p = self._masks(num_ent, x.device)
        self._last_seed = seed
        bn = self.ent_bn
        use_batch_stats = self.training or bn.running_mean is None
        # running statistics of nn.BatchNorm1d: updated inside the statistics kernel when the momentum is a number
        track = self.training and bn.track_running_stats and bn.running_mean is not None
        fused = track and bn.momentum is not None
        all_ent, all_rel, stats = _ConvFn.apply(
            x, rels_embs, edge_embs, self.in_weight, self.out_weight, self.loop_weight, self.rels_weight,
            self.loop_rel, self.loop_edge, bn.weight, bn.bias, self.bias, plan, m_in, m_out, keep_scale,
            use_batch_stats, bn.running_mean, bn.running_var, bn.eps, None, seed, drop_p,
            (float(bn.momentum), bn.num_batches_tracked) if fused else None, self._out_drop_cfg(_out_drop, seed))
        if track and not fused:
            self._update_running_stats(stats, num_ent)
        return all_ent, all_rel

    def _update_running_stats(self, stats, n_rows):
        bn = self.ent_bn
        if self.training and bn.track_running_stats and bn.running_mean is not None:
            with torch.no_grad():           # nn.BatchNorm1d bookkeeping: momentum update with the UNBIASED variance
                bn.num_batches_tracked += 1
                mom = bn.momentum if bn.momentum is not None else 1.0 / float(bn.num_batches_tracked)
                unbias = float(n_rows) / float(max(n_rows - 1, 1))
                bn.running_mean.mul_(1.0 - mom).add_(stats[0], alpha=mom)
                bn.running_var.mul_(1.0 - mom).add_(stats[1], alpha=mom * unbias)

    def forward_partitioned(self, x_local, part, edge_embs_local, rels_embs, _out_drop=0.0):
        """The same layer on a dst-partitioned graph (SURVEY.md 8(e)): ``x_local`` = this rank's node rows,
        ``edge_embs_local`` = the rows of the edges it owns (``part.owned_eids`` order), ``part`` = a
        GraphPartition.  Exchanges: all-gather of x (forward), reduce-scatter of d_x (backward), all-reduce of the
        BatchNorm column sums (2 x Dout doubles, both ways) and of the replicated-parameter gradients.
        ``_out_drop`` as in ``forward`` (used by the sharded MGCN's encoder)."""
        m_in, m_out, keep_scale, seed, drop_p = self._masks(x_local.size(0), x_local.device)
        if seed is not None:
            seed = seed + part.rank          # decorrelate the row blocks of different ranks
        self._last_seed = seed
        out_drop = self._out_drop_cfg(_out_drop, seed)
        if out_drop is not None and seed is None:
            out_drop = (out_drop[0], out_drop[1] + part.rank)       # its own stream: decorrelated as above
        bn = self.ent_bn
        use_batch_stats = self.training or bn.running_mean is None
        coll = part.collectives(x_local.shape[1])
        all_ent, all_rel, stats = _ConvFn.apply(
            x_local, rels_embs, edge_embs_local, self.in_weight, self.out_weight, self.loop_weight, self.rels_weight,
            self.loop_rel, self.loop_edge, bn.weight, bn.bias, self.bias, part.plan, m_in, m_out, keep_scale,
            use_batch_stats, bn.running_mean, bn.running_var, bn.eps, coll, seed, drop_p, None, out_drop)
        self._update_running_stats(stats, part.num_nodes)
        return all_ent, all_rel

    def __repr__(self):
        return '{}({}, {}, num_relations={})'.format(self.__class__.__name__, self.in_channels, self.out_channels,
                                                     self.num_relations)
