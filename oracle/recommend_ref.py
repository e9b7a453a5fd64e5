"""Reference for ``kgat_recommend_filter`` / ``kgat_recommend_topk`` / ``KGAT.recommend`` written with stock torch ops (CPU or
CUDA tensors).

Definition (include/kgat_b200.h): candidate ``p`` of ``items`` passes the filter when, for every group, CSR row
``user_num + p`` of the attentive matrix stores a column ``user_num + e`` for some entity ``e`` of the group.  User ``u``'s
eligible candidates are the passing ones not in ``u``'s exclusion list; they are ranked by the fp32 score
``table[u] . table[p]`` descending (the ``topk_rows`` key: NaN largest, -0 below +0), then by position in ``items``; the top
``k`` are returned as item ids, scores and their number, padded with -1 / -inf.

The scores here come from ``table[u] @ table[c].T``, whose summation order is not the kernel's sequential fmaf chain, so they
can differ in the last bits; near-ties can then swap places.
"""

from __future__ import annotations

import torch

_I64 = torch.int64


def filter_ref(row_ptr, col_idx, items, groups, user_num: int) -> torch.Tensor:
    """Positions into ``items`` (int64, ascending) of the items that pass every group."""
    items = items.to(_I64)
    keep = torch.ones(items.numel(), dtype=torch.bool, device=items.device)
    if items.numel() == 0:
        return torch.zeros(0, dtype=_I64, device=items.device)
    rp = row_ptr.to(_I64).to(items.device)
    col = col_idx.to(_I64).to(items.device)
    n = rp.numel() - 1
    rows = torch.repeat_interleave(torch.arange(n, device=items.device), rp[1:] - rp[:-1])
    keys = rows * n + col  # ascending: rows ascend, columns ascend within a row
    node = items + user_num
    for g in groups:
        ent = torch.tensor(list(g), dtype=_I64, device=items.device) + user_num
        q = (node[:, None] * n + ent[None, :]).flatten()
        pos = torch.searchsorted(keys, q).clamp(max=max(keys.numel() - 1, 0))
        hit = (keys[pos] == q) if keys.numel() else torch.zeros_like(q, dtype=torch.bool)
        keep &= hit.view(items.numel(), ent.numel()).any(1)
    return torch.nonzero(keep).flatten()


def float_key(s: torch.Tensor) -> torch.Tensor:
    """topk_rows' order-preserving uint32 key of fp32 values, as int64."""
    u = s.contiguous().view(torch.int32).to(_I64) & 0xFFFFFFFF
    return torch.where(u >= 0x80000000, 0xFFFFFFFF - u, u | 0x80000000)


def recommend_ref(table, users, items, k: int, exclude_ptr=None, exclude_items=None, groups=None, row_ptr=None, col_idx=None,
                  user_num: int = 0):
    """(items int64 [U, k], scores fp32 [U, k], count int32 [U]).  ``table``: concatenated propagated rows [N, W];
    ``exclude_ptr`` / ``exclude_items``: per user the excluded item ids (any order); ``groups``: the filter (needs ``row_ptr``,
    ``col_idx`` of the attentive matrix and ``user_num``)."""
    dev = table.device
    users = users.to(device=dev, dtype=_I64)
    cand = items.to(device=dev, dtype=_I64)
    if groups is not None:
        cand = cand[filter_ref(row_ptr, col_idx, cand, groups, user_num).to(dev)]
    U, n = users.numel(), cand.numel()
    out_items = torch.full((U, k), -1, dtype=_I64, device=dev)
    out_scores = torch.full((U, k), float("-inf"), dtype=torch.float32, device=dev)
    count = torch.zeros(U, dtype=torch.int32, device=dev)
    if U == 0 or n == 0:
        return out_items, out_scores, count
    scores = table[users] @ table[cand].T  # [U, n]
    eligible = torch.ones(U, n, dtype=torch.bool, device=dev)
    if exclude_ptr is not None:
        ptr = exclude_ptr.to(device=dev, dtype=_I64)
        ex = exclude_items.to(device=dev, dtype=_I64)
        for b in range(U):
            u = int(users[b])
            eligible[b] &= ~torch.isin(cand, ex[ptr[u] : ptr[u + 1]])
    key = float_key(scores)
    pos = torch.arange(n, device=dev, dtype=_I64)
    for b in range(U):
        idx = torch.nonzero(eligible[b]).flatten()
        # stable sort on -key keeps the ascending position order among equal keys
        order = idx[torch.sort(-key[b, idx], stable=True).indices][:k]
        m = order.numel()
        out_items[b, :m] = cand[pos[order]]
        out_scores[b, :m] = scores[b, order]
        count[b] = m
    return out_items, out_scores, count
