"""Reference for ``kgat_recommend_capped_round`` / ``KGAT.recommend_capped`` written with stock torch ops and a plain Python greedy
(CPU or CUDA tensors).

Definition (include/kgat_b200.h): problem ``p`` is a member of capped group ``j`` when CSR row ``user_num + p`` of the attentive
matrix stores a column ``user_num + e`` for some entity ``e`` of the group (``require``'s membership rule).  For each row ``b``:

1. the eligible candidates are ``items``, then the ``require`` filter, minus ``exclude[users[b]]``;
2. they are walked in ``recommend``'s order: the ``topk_rows`` key of the score descending, then the earlier position in
   ``items``;
3. ``p`` is accepted when every group it is a member of has ``count_j < cap_j``; accepting adds 1 to each such ``count_j``;
4. the walk stops at ``k`` acceptances.

The result is the accepted problems in acceptance order with their scores and their number, padded with -1 / -inf.

The scores are an input (``scores[b, x]`` = score of row ``b`` and item id ``x``), so a test can feed the bit-exact ``PREDICT``
scores and expect identical results.
"""

from __future__ import annotations

import torch

from oracle.recommend_ref import filter_ref, float_key

_I64 = torch.int64


def recommend_capped_ref(scores, users, items, k: int, caps, row_ptr, col_idx, user_num: int, exclude_ptr=None, exclude_items=None,
                         require=None):
    """(items int64 [U, k], scores fp32 [U, k], count int32 [U]).  ``scores``: fp32 [U, N] over item ids 0 .. N-1 (every
    candidate below N); ``users``: ids into ``exclude_ptr``; ``caps``: list of ``(group, cap)`` pairs; ``row_ptr`` / ``col_idx``:
    the attentive matrix's CSR; ``exclude_ptr`` / ``exclude_items``: per user the excluded item ids (any order); ``require``:
    the filter's groups."""
    dev = scores.device
    users = users.to(device=dev, dtype=_I64)
    cand = items.to(device=dev, dtype=_I64)
    if require is not None:
        cand = cand[filter_ref(row_ptr, col_idx, cand, require, user_num).to(dev)]
    U, n = users.numel(), cand.numel()
    out_items = torch.full((U, k), -1, dtype=_I64, device=dev)
    out_scores = torch.full((U, k), float("-inf"), dtype=torch.float32, device=dev)
    count = torch.zeros(U, dtype=torch.int32, device=dev)
    if U == 0 or n == 0:
        return out_items, out_scores, count
    # member[c, j]: candidate c is in capped group j
    member = torch.zeros(n, len(caps), dtype=torch.bool, device=dev)
    for j, (group, _) in enumerate(caps):
        member[filter_ref(row_ptr, col_idx, cand, [list(group)], user_num).to(dev), j] = True
    groups_of = [torch.nonzero(member[c]).flatten().tolist() for c in range(n)]
    cap = [int(c) for _, c in caps]
    s = scores[:, cand]  # [U, n]
    key = float_key(s)
    for b in range(U):
        eligible = torch.ones(n, dtype=torch.bool, device=dev)
        if exclude_ptr is not None:
            u = int(users[b])
            eligible &= ~torch.isin(cand, exclude_items.to(device=dev, dtype=_I64)[int(exclude_ptr[u]) : int(exclude_ptr[u + 1])])
        idx = torch.nonzero(eligible).flatten()
        # stable sort on -key keeps the ascending position order among equal keys
        order = idx[torch.sort(-key[b, idx], stable=True).indices].tolist()
        used = [0] * len(caps)
        m = 0
        for c in order:
            if m == k:
                break
            if any(used[j] >= cap[j] for j in groups_of[c]):
                continue
            for j in groups_of[c]:
                used[j] += 1
            out_items[b, m] = cand[c]
            out_scores[b, m] = s[b, c]
            m += 1
        count[b] = m
    return out_items, out_scores, count
