"""Full-catalog top-K recommendation: given users, the best K items of the whole catalog, leaving out the
items each user already has.

One ncf_recommend call scores the users against every item with the forward kernels (ncf_forward's tile
paths), sets the excluded items to NaN and selects the K best per user on the GPU, `chunk_users` users at
a time, so memory stays bounded by the chunk rather than by users x items.  Order: larger score first,
equal scores to the lower item id (the rule of the sampled evaluation, metrics.evaluate).

The parameters are read as they are.  A model trained with FusedTrainStep holds lazily updated Adam rows:
call `ts.flush()` first (train_loop.fit does so at the end of every epoch).
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from . import _lib, ops

WORKSPACE_BUDGET = 1 << 30   # default chunk_users keeps the workspace at or below 1 GiB
MAX_CHUNK_PAIRS = 1 << 28    # (user, item) pairs one chunk may score (ncf_recommend)


def default_chunk_users(m: _lib.NcfModel, n: int, k: int, budget: int = WORKSPACE_BUDGET) -> int:
    """The largest chunk (at most n users, at least 1) whose workspace fits `budget` bytes."""
    chunk = max(1, min(n, MAX_CHUNK_PAIRS // m.item_num))
    while chunk > 1:
        need = ops.recommend_workspace_bytes(m, chunk, k)
        if need <= budget:
            break
        chunk = max(1, min(chunk - 1, chunk * budget // need))
    return chunk


def recommend_ranked(model, users: torch.Tensor, k: int = 10, exclude=None, chunk_users: Optional[int] = None,
                     target: Optional[torch.Tensor] = None):
    """recommend() plus, when `target` (int64 [n] item ids) is given, the full rank of each user's target
    among the items not excluded (-1: the target is excluded or out of range)."""
    users = users.reshape(-1).to(torch.int64).contiguous()
    m = model.abi_struct()
    n = users.numel()
    if chunk_users is None:
        chunk_users = default_chunk_users(m, max(n, 1), k)
    rowptr, col = exclude if exclude is not None else (None, None)
    if target is not None:
        target = target.reshape(-1).to(torch.int64).contiguous()
    with torch.no_grad():
        return ops.recommend(m, users, int(k), int(chunk_users), rowptr, col, target)


def recommend(model, users: torch.Tensor, k: int = 10, exclude=None,
              chunk_users: Optional[int] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """users int64 [n] on the model's device -> (items int64 [n, k], scores float32 [n, k]), best first.

    exclude: (rowptr, col) of ops.csr_build over the pairs to leave out (typically the training pairs);
    None ranks every item.  A user with fewer than k items left gets -1 / NaN in the remaining slots.
    chunk_users: users scored per forward; default: as many as keep the workspace within 1 GiB."""
    items, scores, _ = recommend_ranked(model, users, k, exclude, chunk_users)
    return items, scores
