"""kgc_gcn_b200: B200-native hot path of M-GCN (weilonghu/KGC-GCN) behind the reference's module API.

    from kgc_gcn_b200 import MGCN, MGCNConv, ConvE, DataLoader, KBDataset

Compute runs in libkgc_b200.so (hand-written sm_100a CUDA behind the C ABI of include/kgc_b200.h);
there is no CPU fallback.
"""
from .conv import (MGCNConv, get_param, gemm_nt, gemm_tn, gemm_nt_trans, gemm_nt_splitk,   # noqa: F401
                   linear_tc, linear_tc_supported)
from .model import MGCN, ConvE, ShardedMGCN      # noqa: F401
from .data_loader import DataLoader, KBDataset, GraphData, BatchIterator, epoch_permutation   # noqa: F401
from .plan import GraphPlan, get_plan, build_levels, build_stream_plan   # noqa: F401
from .scoring import (EntityTable, filtered_rank, pack_queries, pair_scores, predict, evaluate,   # noqa: F401
                      score_kpad, topk, merge_topk, score_sampled_bce, score_sampled_ce, score_shared_bce,
                      score_shared_ce, score_1n_bce_shard)
from .partition import GraphPartition, partition_edges   # noqa: F401
from .train import GraphedTrainStep             # noqa: F401
from .optim import ClipAdam                      # noqa: F401
from .utils import save_checkpoint, load_checkpoint   # noqa: F401
from . import _lib                               # noqa: F401

__all__ = ['MGCN', 'MGCNConv', 'ConvE', 'DataLoader', 'KBDataset', 'GraphData', 'BatchIterator', 'GraphPlan',
           'get_plan', 'build_levels', 'build_stream_plan', 'get_param', 'gemm_nt', 'gemm_tn', 'gemm_nt_trans', 'gemm_nt_splitk', 'linear_tc', 'linear_tc_supported', 'epoch_permutation', 'EntityTable', 'filtered_rank', 'pack_queries',
           'pair_scores', 'topk', 'merge_topk', 'predict', 'evaluate', 'score_kpad', 'score_sampled_bce', 'score_sampled_ce', 'score_shared_bce', 'score_shared_ce', 'GraphPartition', 'partition_edges', 'GraphedTrainStep', 'ClipAdam',
           'save_checkpoint', 'load_checkpoint']
