"""Batch-shared negatives, host side: the broadcast candidate matrix that defines the shared losses, the argument checks
of score_shared_bce / score_shared_ce, KBDataset.shared_negatives, MGCN.loss_sampled(shared_negatives=...) and
GraphedTrainStep(shared_negatives=...) (no GPU needed)."""
import numpy as np
import pytest
import torch

import kgc_gcn_b200 as k


def _csr(lists):
    ptr = np.zeros(len(lists) + 1, dtype=np.int64)
    ptr[1:] = np.cumsum([len(l) for l in lists])
    return torch.from_numpy(ptr), torch.from_numpy(np.concatenate([np.asarray(l, np.int32) for l in lists]))


def test_shared_candidates_follow_the_definition():
    """Row b = [pos_cand[b] | shared with each known object of query qid[b] set to -1]; duplicates stay separate slots."""
    rng = np.random.default_rng(0)
    N, K, B = 20, 15, 9
    lists = [sorted(set(rng.integers(0, N, int(rng.integers(0, 7))).tolist())) or [0] for _ in range(12)]
    ptr, idx = _csr(lists)
    shared = torch.from_numpy(rng.integers(0, N, K).astype(np.int32))
    shared[3] = shared[4]
    qid = torch.from_numpy(rng.integers(0, 12, B)).long()
    pos = torch.from_numpy(rng.integers(-1, N, (B, 2)).astype(np.int32))
    cand = k.scoring.shared_candidates(pos, shared, qid, ptr, idx)
    assert cand.dtype == torch.int32 and tuple(cand.shape) == (B, 2 + K)
    for b in range(B):
        known = set(lists[int(qid[b])])
        want = pos[b].tolist() + [-1 if int(s) in known else int(s) for s in shared]
        assert cand[b].tolist() == want


def _args(B=4, D=8, N=10, K=5, n_pos=1):
    return (torch.zeros(B, D), torch.zeros(N, D), torch.zeros(N), torch.zeros((B, n_pos), dtype=torch.int32),
            torch.zeros(K, dtype=torch.int32), torch.zeros(B, dtype=torch.int64), torch.zeros(11, dtype=torch.int64),
            torch.zeros(0, dtype=torch.int32))


@pytest.mark.parametrize('fn', ['score_shared_bce', 'score_shared_ce'])
def test_shared_argument_errors(fn):
    f = getattr(k, fn)
    with pytest.raises(ValueError, match='D % 4'):
        f(*_args(D=6))
    with pytest.raises(ValueError, match='D % 4'):
        f(*_args(D=228))
    with pytest.raises(ValueError, match='k >= 1'):
        f(*_args(K=0))
    with pytest.raises(ValueError, match='n_pos >= 1'):
        f(*_args(n_pos=0))
    a = list(_args())
    a[4] = a[4].long()
    with pytest.raises(ValueError, match='int32'):
        f(*a)
    a = list(_args())
    a[5] = torch.zeros(3, dtype=torch.int64)
    with pytest.raises(ValueError, match='shape mismatch'):
        f(*a)
    with pytest.raises(RuntimeError, match='CUDA tensor'):
        f(*_args())


def test_shared_option_errors():
    with pytest.raises(ValueError, match='adversarial_temperature'):
        k.score_shared_bce(*_args(), adversarial_temperature=-1.0)
    with pytest.raises(ValueError, match='label_smoothing'):
        k.score_shared_ce(*_args(), label_smoothing=1.5)


def test_shared_negatives_sampler_is_gpu_only_and_checks_k():
    ds = k.KBDataset.__new__(k.KBDataset)
    ds.num_entity = 7
    with pytest.raises(ValueError, match='k must be'):
        ds.shared_negatives(0, device='cpu')
    with pytest.raises(RuntimeError, match='GPU only'):
        ds.shared_negatives(4, device='cpu')


def test_loss_sampled_shared_rejects_tries():
    with pytest.raises(ValueError, match='tries'):
        k.MGCN.loss_sampled(object(), [0], None, None, 4, tries=3, shared_negatives=True)


def test_graphed_step_shared_errors():
    with pytest.raises(ValueError, match='needs negatives=k'):
        k.GraphedTrainStep(None, None, None, None, 4, shared_negatives=True)
    with pytest.raises(ValueError, match='tries'):
        k.GraphedTrainStep(None, None, None, None, 4, negatives=8, tries=2, shared_negatives=True)
