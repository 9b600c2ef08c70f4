"""ctypes binding of libkgc_b200.so (the C ABI declared in include/kgc_b200.h).

There is no CPU fallback and no alternative backend: if the shared library is missing or a call
fails, a RuntimeError is raised.  PyTorch is used only for device memory, streams and
torch.distributed; every pointer handed to the library is a raw device address.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('KGC_LIB_PATH') or os.path.join(_HERE, 'libkgc_b200.so')     # KGC_LIB_PATH: A/B runs of two builds
_LIB = None

_vp, _i64, _i32, _f32, _sz = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_float, ctypes.c_size_t

# name -> (restype, argtypes); must list every symbol include/kgc_b200.h declares (tests check this)
SIGNATURES = {
    'kgc_last_error': (ctypes.c_char_p, []),
    'kgc_abi_version': (ctypes.c_int, []),
    'kgc_csr_workspace_bytes': (_sz, [_i64, _i64, _i64]),
    'kgc_csr_build': (ctypes.c_int, [_vp, _vp, _vp, _i64, _i64, _i64, _i64, _i64, _i64, _i32, _vp, _vp, _vp, _vp, _vp,
                                     _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _sz, _vp]),
    'kgc_csr_type_rows': (_i64, [_i64, _i64, _i64]),
    'kgc_block_sum': (ctypes.c_int, [_vp, _i64, _i64, _vp, _vp]),
    'kgc_stream_plan_flags': (ctypes.c_int, [_vp, _vp, _vp, _i64, _i64, _i32, _vp, _vp, _vp, _vp]),
    'kgc_agg_fwd': (ctypes.c_int, [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _i32, _vp]),
    'kgc_rows_fill': (ctypes.c_int, [_vp, _i64, _vp, _vp, _i32, _vp]),
    'kgc_rows_reduce': (ctypes.c_int, [_vp, _vp, _i64, _i64, _vp, _vp, _vp, _i32, _vp]),
    'kgc_agg_bwd_src': (ctypes.c_int, [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _i32, _vp]),
    'kgc_agg_bwd_rel': (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _vp, _vp, _i32, _vp]),
    'kgc_tail_num_blocks': (_i64, [_i64]),
    'kgc_dropout_mask': (ctypes.c_int, [_vp, _i32, _f32, _i64, _vp, _vp]),
    'kgc_keep_pitch': (_i32, []),
    'kgc_tail_fwd': (ctypes.c_int, [_vp, _vp, _vp, _vp, _f32, _f32, _vp, _i64, _i32, _vp, _vp, _vp, _vp]),
    'kgc_tail_fwd_rows': (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f32, _f32, _vp, _i64, _i32, _vp, _vp, _vp, _vp]),
    'kgc_rows_copy': (ctypes.c_int, [_vp, _i64, _vp, _vp, _i64, _vp, _i64, _i32, _vp]),
    'kgc_colsum_finalize': (ctypes.c_int, [_vp, _i64, _i32, _vp, _vp]),
    'kgc_colstats_from_sums': (ctypes.c_int, [_vp, _i64, _i32, _f32, _i32, _vp, _vp, _vp, _vp]),
    'kgc_colstats_finalize': (ctypes.c_int, [_vp, _i64, _i64, _i32, _f32, _f32, _vp, _vp, _vp, _vp, _vp, _vp]),
    'kgc_colsum_finalize2': (ctypes.c_int, [_vp, _i64, _i32, _vp, _vp, _vp]),
    'kgc_tail_apply': (ctypes.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp, _f32, _vp, _vp]),
    'kgc_tail_bwd_reduce': (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp, _f32, _vp]),
    'kgc_tail_bwd_apply': (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _i64, _i32, _vp, _vp, _f32, _vp, _vp, _f32, _vp]),
    'kgc_tail_bwd_apply_rows': (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _i64, _i32, _vp, _vp, _f32, _vp, _vp, _vp,
                                               _vp, _vp, _f32, _vp]),
    'kgc_gemm_packed_b_bytes': (_sz, [_i32, _i32]),
    'kgc_gemm_pack_b': (ctypes.c_int, [_vp, _i64, _i64, _i32, _i32, _vp, _vp]),
    'kgc_gemm_nt': (ctypes.c_int, [_vp, _i64, _i32, _i64, _vp, _i32, _vp, _i64, _vp]),
    'kgc_conv_prep': (ctypes.c_int, [_vp, _i32] + [_vp] * 6 + [_i32, _i32] + [_vp] * 5),
    'kgc_conv_param_grads': (ctypes.c_int, [_vp] * 8 + [_i32, _i32, _i32] + [_vp] * 7),
    'kgc_gemm_nt_batch': (ctypes.c_int, [_i32, _vp, _i64, _i32, _i64, _vp, _i32, _vp, _i64, _vp]),
    'kgc_gemm_nt_batch_masked': (ctypes.c_int, [_i32, _vp, _i64, _i32, _i64, _vp, _i32, _vp, _i64, _vp, _i32, _f32, _vp]),
    'kgc_gemm_tn_tc_batch_masked': (ctypes.c_int, [_i32, _vp, _i64, _vp, _i64, _i64, _i32, _i32, _vp, _vp, _sz, _vp, _i32, _f32, _vp]),
    'kgc_gemm_nt_trans': (ctypes.c_int, [_vp, _i64, _i32, _i64, _vp, _i32, _vp, _i64, _vp]),
    'kgc_gemm_nt_splitk': (ctypes.c_int, [_vp, _i64, _vp, _i64, _i64, _i32, _i32, _vp, _vp, _sz, _vp]),
    'kgc_gemm_set_debug': (None, [_vp]),
    'kgc_gemm_tn_workspace_bytes': (_sz, [_i64, _i32, _i32]),
    'kgc_gemm_tn_tc_workspace_bytes': (_sz, [_i64, _i32, _i32]),
    'kgc_gemm_tn_tc': (ctypes.c_int, [_vp, _i64, _vp, _i64, _i64, _i32, _i32, _vp, _vp, _sz, _vp]),
    'kgc_gemm_tn_tc_batch': (ctypes.c_int, [_i32, _vp, _i64, _vp, _i64, _i64, _i32, _i32, _vp, _vp, _sz, _vp]),
    'kgc_gemm_tn_tc_batch_rows': (ctypes.c_int, [_i32, _vp, _i64, _vp, _i64, _vp, _i64, _i32, _i32, _vp, _vp, _sz, _vp]),
    'kgc_gemm_tn': (ctypes.c_int, [_vp, _i64, _vp, _i64, _i64, _i32, _i32, _vp, _vp, _sz, _vp]),
    'kgc_label_build': (ctypes.c_int, [_vp, _i64, _vp, _vp, _vp, _i64, _f32, _f32, _vp, _vp, _vp]),
    'kgc_neg_sample': (ctypes.c_int, [_vp, _i64, _vp, _vp, _i64, _vp, _i32, _i32, _vp, _vp]),
    'kgc_pos_sample': (ctypes.c_int, [_vp, _i64, _vp, _vp, _vp, _i32, _vp, _vp]),
    'kgc_edge_sample': (ctypes.c_int, [_vp, _vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp]),
    'kgc_bn2d_partials_bytes': (_sz, [_i32]),
    'kgc_bn2d_relu_drop_fwd': (ctypes.c_int, [_vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _f32, _f32, _i32, _i32, _vp, _f32, _vp, _vp, _vp, _vp]),
    'kgc_bn2d_relu_drop_bwd': (ctypes.c_int, [_vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp, _i32, _i32, _vp, _f32, _vp, _vp, _vp, _vp]),
    'kgc_conv1ch_supported': (_i32, [_i32, _i32, _i32, _i32]),
    'kgc_conv1ch_bwd_workspace_bytes': (_sz, [_i64, _i32, _i32]),
    'kgc_conv1ch_fwd': (ctypes.c_int, [_vp, _vp, _vp, _i64, _i32, _i32, _i32, _i32, _vp, _vp]),
    'kgc_conv1ch_bwd': (ctypes.c_int, [_vp, _vp, _vp, _i64, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp]),
    'kgc_opt_chunk_elems': (_i32, []),
    'kgc_clip_adam_step': (ctypes.c_int, [_vp, _vp, _i64, _vp, _vp, _vp, _vp]),
    'kgc_p2p_allreduce': (ctypes.c_int, [_vp, _i64, _vp, _i32, _i32, _vp, _vp, _vp, _vp, _i64, _i32, _vp]),
    'kgc_p2p_barrier': (ctypes.c_int, [_vp, _i32, _i32, _vp, _vp, _vp]),
    'kgc_p2p_halo_gather': (ctypes.c_int, [_vp, _i32, _vp, _vp, _i64, _i64, _i32, _vp]),
    'kgc_p2p_halo_reduce': (ctypes.c_int, [_vp, _i32, _vp, _vp, _i64, _vp, _vp, _i32, _vp]),
    'kgc_ingest_open': (ctypes.c_int, [ctypes.c_char_p, _vp]),
    'kgc_ingest_close': (None, [_vp]),
    'kgc_ingest_count': (_i64, [_vp, _i32]),
    'kgc_ingest_copy': (ctypes.c_int, [_vp, _i32, _vp, _i64]),
    'kgc_ingest_name': (ctypes.c_char_p, [_vp, _i32, _i64]),
    'kgc_score_1n_fwd': (ctypes.c_int, [_vp, _i64, _i32, _i64, _vp, _i32, _vp, _vp, _i64, _vp]),
    'kgc_score_1n_logits': (ctypes.c_int, [_vp, _i64, _i32, _i64, _vp, _i32, _vp, _vp, _i64, _vp]),
    'kgc_rank_count_dense': (ctypes.c_int, [_vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp]),
    'kgc_score_1n_bwd_logit': (ctypes.c_int, [_vp, _i64, _vp, _i64, _i64, _i32, _i32, _vp, _vp, _vp]),
    'kgc_label_mask_words': (_i64, [_i64]),
    'kgc_label_mask_build': (ctypes.c_int, [_vp, _i64, _vp, _vp, _vp, _i64, _vp, _vp, _vp]),
    'kgc_bce_1n_bwd_logit': (ctypes.c_int, [_vp, _i64, _vp, _i64, _i32, _i32, _f32, _f32, _vp, _vp, _vp, _vp, _vp]),
    'kgc_score_1n_fwd_t': (ctypes.c_int, [_vp, _i64, _i32, _i64, _vp, _i32, _vp, _vp, _i64, _vp]),
    'kgc_bce_1n_t_blocks': (_i64, [_i64]),
    'kgc_label_mask_t_build': (ctypes.c_int, [_vp, _i64, _vp, _vp, _i64, _vp, _vp]),
    'kgc_bce_1n_bwd_logit_t': (ctypes.c_int, [_vp, _vp, _i64, _i32, _i32, _f32, _f32, _vp, _vp, _vp, _vp]),
    'kgc_score_kpad': (_i32, [_i32]),
    'kgc_score_pack_entities': (ctypes.c_int, [_vp, _vp, _i64, _i32, _vp, _vp]),
    'kgc_score_pack_queries': (ctypes.c_int, [_vp, _i64, _i32, _vp, _vp]),
    'kgc_score_pairs_workspace_bytes': (_sz, [_i64, _i32]),
    'kgc_score_pairs': (ctypes.c_int, [_vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp, _sz, _vp]),
    'kgc_score_rank': (ctypes.c_int, [_vp, _vp, _i64, _i64, _i32, _vp, _vp, _vp, _vp]),
    'kgc_rank_finalize': (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp]),
    'kgc_score_topk_workspace_bytes': (_sz, [_i64, _i64, _i32, _i32]),
    'kgc_score_topk': (ctypes.c_int, [_vp, _vp, _i64, _i64, _i32, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _sz, _vp]),
    'kgc_topk_dense_workspace_bytes': (_sz, [_i64, _i64, _i32]),
    'kgc_topk_dense': (ctypes.c_int, [_vp, _i64, _i64, _i64, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _sz, _vp]),
    'kgc_topk_merge': (ctypes.c_int, [_vp, _vp, _i64, _i64, _i32, _vp, _vp, _vp, _vp]),
    'kgc_sampled_bce_fwd_blocks': (_i64, [_i64]),
    'kgc_sampled_bce_fwd': (ctypes.c_int, [_vp, _i64, _i32, _vp, _i64, _i64, _vp, _vp, _i32, _i32, _f32, _f32, _vp, _vp, _vp, _vp,
                                           _vp, _vp]),
    'kgc_sampled_adv_fwd': (ctypes.c_int, [_vp, _i64, _i32, _vp, _i64, _i64, _vp, _vp, _i32, _i32, _f32, _f32, _f32, _vp, _vp, _vp,
                                           _vp, _vp, _vp]),
    'kgc_sampled_bce_bwd_table_workspace_bytes': (_sz, [_i64, _i64]),
    'kgc_sampled_bce_bwd_table': (ctypes.c_int, [_vp, _i64, _i32, _vp, _i32, _vp, _vp, _i64, _vp, _i64, _vp, _vp, _sz, _vp]),
}


def lib():
    """Load libkgc_b200.so once; fail loudly when it has not been built."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError('{} is missing: build it with `python -c "import __graft_entry__ as g; g.build()"` '
                               '(nvcc, sm_100a). There is no CPU or PyTorch fallback.'.format(LIB_PATH))
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)       # AttributeError if the symbol is not exported
            fn.restype, fn.argtypes = res, args
        if handle.kgc_abi_version() != 1:
            raise RuntimeError('libkgc_b200.so ABI version mismatch')
        _LIB = handle
    return _LIB


LAUNCHES = 0     # kernels launched through the C ABI since import (bench.py reports it as gpu_launches)
_KERNELS_PER_CALL = {'kgc_csr_build': 16, 'kgc_label_mask_build': 2, 'kgc_bce_1n_bwd_logit': 2, 'kgc_bce_1n_bwd_logit_t': 2, 'kgc_label_mask_t_build': 2, 'kgc_score_pairs': 3, 'kgc_rank_finalize': 2, 'kgc_score_topk': 2, 'kgc_topk_dense': 2, 'kgc_sampled_bce_fwd': 4, 'kgc_sampled_adv_fwd': 4, 'kgc_sampled_bce_bwd_table': 7, 'kgc_gemm_tn': 2, 'kgc_gemm_tn_tc': 2, 'kgc_gemm_tn_tc_batch': 2, 'kgc_gemm_tn_tc_batch_rows': 2, 'kgc_gemm_tn_tc_batch_masked': 2}   # (kgc_p2p_allreduce: 1 or 3)


def call(name, *args):
    """Invoke an int-returning entry point; raise RuntimeError with kgc_last_error() on failure."""
    global LAUNCHES
    h = lib()
    LAUNCHES += _KERNELS_PER_CALL.get(name, 1)
    rc = getattr(h, name)(*args)
    if rc != 0:
        raise RuntimeError('{} failed: {}'.format(name, h.kgc_last_error().decode('utf-8', 'replace')))


_WARNED = set()


def library_path(site, reason):
    """A call site is about to leave the hand-written kernels for a torch / cuDNN / cuBLAS library operation (a shape or
    dtype the kernel does not take).  Never silent: raises under KGC_STRICT=1 (the GPU tests run that way), otherwise warns
    once per site."""
    msg = 'kgc_gcn_b200: {} is running on the torch library path ({})'.format(site, reason)
    if os.environ.get('KGC_STRICT', '0') not in ('', '0'):
        raise RuntimeError(msg + ' and KGC_STRICT=1 forbids it')
    if site not in _WARNED:
        _WARNED.add(site)
        import warnings
        warnings.warn(msg, RuntimeWarning, stacklevel=3)


def ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda(t, dtype, name):
    if not (torch.is_tensor(t) and t.is_cuda):
        raise RuntimeError('{} must be a CUDA tensor: the M-GCN hot path runs on the GPU only (no CPU fallback)'.format(name))
    if t.dtype != dtype:
        raise TypeError('{} must be {}, got {}'.format(name, dtype, t.dtype))
    return t if t.is_contiguous() else t.contiguous()
