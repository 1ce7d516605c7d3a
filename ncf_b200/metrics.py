"""Leave-one-out evaluation — the drop-in for reference src/training/metrics.py:4-25.

`metrics(model, test_loader, top_k) -> (HR list, NDCG list)` keeps the reference signature, but
instead of one forward + torch.topk + two host syncs per user it scores every user's candidates in
one fused launch and ranks them with one warp per user (ncf_eval_users).  The held-out item is
column 0 of each candidate row (reference src/data/datasets.py:31-34); ties go to the lower
candidate index.  NDCG is derived from the device rank on the host as 1/np.log2(rank+2) in float64,
which is the reference's own expression (metrics.py:22), so the returned lists compare equal.

A NaN score is not a candidate, so a user whose held-out score is NaN is a miss (HR 0, NDCG 0).  A
model that has diverged to NaN, or an id outside the tables (the forward gives NaN for it), scores
HR = 0 rather than a perfect one.  This departs from the reference on purpose: its torch.topk ranks
NaN above every number and counts a NaN held-out item as a hit.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch

from . import _lib, ops


@dataclass
class EvalResult:
    hit: torch.Tensor     # uint8 [n]
    rank: torch.Tensor    # int32 [n], -1 = held-out item not in the top k
    ndcg: torch.Tensor    # float32 [n] (device value)
    topk: torch.Tensor    # int32 [n, k] candidate indices, best first
    scores: torch.Tensor  # float32 [n, C]

    def lists(self):
        """(HR, NDCG) as the reference returns them: python ints and float64s."""
        rank = self.rank.cpu().numpy()
        HR = (rank >= 0).astype(np.int64).tolist()
        NDCG = [0.0 if r < 0 else float(1.0 / np.log2(r + 2)) for r in rank.tolist()]
        return HR, NDCG


def evaluate(model, users: torch.Tensor, cands: torch.Tensor, top_k: int) -> EvalResult:
    """users int64[n], cands int64[n, C] on the model's device."""
    if cands.dim() != 2:
        raise _lib.NcfError("evaluate: cands must be a dense [n, C] tensor (ragged test sets are rejected; "
                            "the reference silently misaligns users in that case, SURVEY.md H5)")
    hit, rank, ndcg, topk, scores = ops.eval_users(model.abi_struct(), users.contiguous(),
                                                   cands.contiguous(), int(top_k))
    return EvalResult(hit, rank, ndcg, topk, scores)


def evaluate_top_k(model, users: torch.Tensor, cands: torch.Tensor, max_k: int = 10):
    """HR@K and NDCG@K for every K = 1..max_k from ONE scoring + ranking pass: the rank of the held-out
    item among its candidates decides every K at once (hit iff rank < K).  Replaces the `max_k` full
    evaluation passes of reference scripts/evaluate_models.py:22-32 (`metrics(model, loader, k)` per k).
    Returns (hr_at_k, ndcg_at_k): dicts {k: mean over users}, the reference function's return value."""
    res = evaluate(model, users, cands, max_k)
    rank = res.rank.cpu().numpy().astype(np.int64)          # -1 = not within the top max_k
    gain = np.where(rank >= 0, 1.0 / np.log2(np.maximum(rank, 0) + 2.0), 0.0)
    hr_at_k, ndcg_at_k = {}, {}
    for k in range(1, max_k + 1):
        hit = (rank >= 0) & (rank < k)
        hr_at_k[k] = float(np.mean(hit.astype(np.float64)))
        ndcg_at_k[k] = float(np.mean(np.where(hit, gain, 0.0)))
    return hr_at_k, ndcg_at_k


def evaluate_full_ranking(model, users: torch.Tensor, targets: torch.Tensor, exclude, ks=(1, 5, 10, 20)):
    """Full-ranking leave-one-out protocol: the held-out item targets[r] is ranked against every item user
    users[r] has not seen (exclude = (rowptr, col) of ops.csr_build over the training pairs), ties to the
    lower item id.  One ncf_recommend pass (k = 1: only the target's rank is needed).
    Returns (rank int32 [n] on the device, -1 = target excluded; {K: HR@K}; {K: NDCG@K}), means over users
    with NDCG = 1/log2(rank+2) in float64 as EvalResult.lists() computes it."""
    from .recommend import recommend_ranked
    _, _, rank = recommend_ranked(model, users, 1, exclude, target=targets)
    r = rank.cpu().numpy().astype(np.int64)
    gain = np.where(r >= 0, 1.0 / np.log2(np.maximum(r, 0) + 2.0), 0.0)
    hr_at_k, ndcg_at_k = {}, {}
    for k in ks:
        hit = (r >= 0) & (r < k)
        hr_at_k[k] = float(np.mean(hit.astype(np.float64))) if r.size else 0.0
        ndcg_at_k[k] = float(np.mean(np.where(hit, gain, 0.0))) if r.size else 0.0
    return rank, hr_at_k, ndcg_at_k


def evaluate_top_k_performance(model, test_loader, max_k=10):
    """Drop-in for reference scripts/evaluate_models.py:22-32 (same name, arguments and return value)."""
    device = next(model.parameters()).device
    users, cands = _test_tensors(test_loader, device)
    with torch.no_grad():
        return evaluate_top_k(model, users, cands, max_k)


def _test_tensors(test_loader, device):
    """Pulls (users [n], cands [n, C]) out of a reference-style test DataLoader / NCFData."""
    ds = getattr(test_loader, "dataset", test_loader)
    C = getattr(test_loader, "batch_size", None)
    feats = getattr(ds, "features_ps", None)
    if feats is None or C is None:
        raise _lib.NcfError("metrics: need a DataLoader over NCFData (features_ps) with batch_size = C")
    arr = feats if torch.is_tensor(feats) else torch.as_tensor(np.asarray(feats, dtype=np.int64))
    if arr.shape[0] % C != 0:
        raise _lib.NcfError(f"metrics: {arr.shape[0]} test rows are not a multiple of batch_size {C}")
    arr = arr.to(device).reshape(-1, C, 2)
    return arr[:, 0, 0].contiguous(), arr[:, :, 1].contiguous()


def metrics(model, test_loader, top_k):
    device = next(model.parameters()).device
    users, cands = _test_tensors(test_loader, device)
    with torch.no_grad():
        return evaluate(model, users, cands, top_k).lists()
