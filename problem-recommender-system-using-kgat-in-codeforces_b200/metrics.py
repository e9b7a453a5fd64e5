"""Evaluation on the device: the reference's ``evaluate`` loop (src/model/KGAT/main.py:70-130) and
``metrics_at_k`` (src/utils/metrics_calculator.py:84-131) without the per-batch device->host copy of a
256 x n_items score matrix and the full CPU ``torch.sort``.

Per 256-user batch: scores from the cached propagated tables (gather + SGEMM), training positives masked
to -inf, exact top-K on the device (K = max(k_list); ties lowest item first, the CPU ``torch.sort`` order),
then precision / recall / nDCG from the K hit flags:

    precision@k = hits[:k].sum / k
    recall@k    = hits[:k].sum / |test items of the user|        (NaN when the user has none, as in the reference)
    ndcg@k      = sum_i hit_i / log2(i + 2)  /  sum_{i < min(k, |test|)} 1 / log2(i + 2)

The reference builds its denominators from the *full* ranking (``hits.sum()`` and the sorted full-row
hits); every item appears exactly once in a full ranking, so they equal the number of test items of the
user -- which is what is used here.
"""

from __future__ import annotations

import numpy as np
import torch

from . import ops


class InteractionCSR:
    """{user: [items]} as device CSR (int32), for masking and hit tests."""

    def __init__(self, inter, user_num: int, item_num: int, device):
        if isinstance(inter, dict):
            counts = np.array([len(inter.get(u, ())) for u in range(user_num)], dtype=np.int64)
            flat = np.concatenate([np.asarray(inter.get(u, ()), dtype=np.int64) for u in range(user_num)] + [np.zeros(0, np.int64)])
        else:  # (M, 2) array of (user, item)
            pairs = np.asarray(inter, dtype=np.int64).reshape(-1, 2)
            order = np.lexsort((pairs[:, 1], pairs[:, 0]))
            pairs = pairs[order]
            counts = np.bincount(pairs[:, 0], minlength=user_num)
            flat = pairs[:, 1]
        # the reference derives hits and denominators from a binary item mask (metrics_calculator.py:112-122): an item listed twice for a
        # user counts once
        users_all = np.repeat(np.arange(user_num, dtype=np.int64), counts)
        keys = np.unique(users_all * item_num + flat.astype(np.int64))
        counts = np.bincount(keys // item_num, minlength=user_num).astype(np.int64)
        flat = keys % item_num
        self.user_num, self.item_num = user_num, item_num
        self.ptr_host = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
        self.items = torch.from_numpy(flat.astype(np.int32)).to(device)
        self.counts = torch.from_numpy(counts.astype(np.int64)).to(device)
        users = np.repeat(np.arange(user_num, dtype=np.int64), counts)
        self.keys = torch.from_numpy(np.sort(users * item_num + flat)).to(device)  # sorted (user, item) keys
        self._ptr_dev = None

    @property
    def ptr_dev(self) -> torch.Tensor:
        """Row pointer over all users as int32 on the device of ``items`` (built on first use; ``KGAT.recommend`` reads it)."""
        if self._ptr_dev is None:
            if self.ptr_host[-1] > np.iinfo(np.int32).max:
                raise ValueError("more than 2^31 - 1 interactions do not fit the int32 row pointer")
            self._ptr_dev = torch.from_numpy(self.ptr_host.astype(np.int32)).to(self.items.device)
        return self._ptr_dev

    def batch(self, start: int, stop: int):
        """(ptr int32 [b+1] relative to the batch, items int32) for users [start, stop)."""
        ptr = torch.from_numpy((self.ptr_host[start : stop + 1] - self.ptr_host[start]).astype(np.int32)).to(self.items.device)
        return ptr, self.items[self.ptr_host[start] : self.ptr_host[stop]]

    def contains(self, users: torch.Tensor, items: torch.Tensor) -> torch.Tensor:
        keys = users.to(torch.int64) * self.item_num + items.to(torch.int64)
        pos = torch.searchsorted(self.keys, keys).clamp_(max=max(self.keys.numel() - 1, 0))
        return (self.keys[pos] == keys) if self.keys.numel() else torch.zeros_like(keys, dtype=torch.bool)


@torch.no_grad()
def evaluate(model, train: InteractionCSR, test: InteractionCSR, k_list=(20, 40, 60, 80, 100), batch_size: int = 256, users=None):
    """Ranking metrics for ``users`` (default: every user with at least one test item -- the reference iterates
    ``eval_interaction_dict.keys()``), averaged like main.py:123-128.  Returns ({k: {metric: float}}, top-K indices)."""
    model.eval()
    dev = model._device()
    kmax = max(k_list)
    if users is None:
        users = torch.nonzero(test.counts > 0).flatten().cpu().numpy()
    users = np.asarray(users, dtype=np.int64)
    items = torch.arange(train.item_num, device=dev)
    disc = 1.0 / torch.log2(torch.arange(2, kmax + 2, device=dev, dtype=torch.float32))
    cum_ideal = torch.cumsum(disc, 0)
    sums = {k: {"precision": 0.0, "recall": 0.0, "ndcg": 0.0} for k in k_list}
    tops = []
    n_done = 0
    for s in range(0, users.shape[0], batch_size):
        ub = users[s : s + batch_size]
        contiguous = ub.shape[0] > 0 and bool((np.diff(ub) == 1).all())
        if contiguous:
            ptr, flat = train.batch(int(ub[0]), int(ub[-1]) + 1)
        else:
            cnt = train.ptr_host[ub + 1] - train.ptr_host[ub]
            ptr = torch.from_numpy(np.concatenate([[0], np.cumsum(cnt)]).astype(np.int32)).to(dev)
            idx = np.concatenate([np.arange(train.ptr_host[u], train.ptr_host[u + 1]) for u in ub] + [np.zeros(0, np.int64)]).astype(np.int64)
            flat = train.items[torch.from_numpy(idx).to(dev)]
        ub_dev = torch.from_numpy(ub).to(dev)
        top = model.recommend_topk(ub_dev, items, kmax, ptr, flat).to(torch.int64)  # [b, kmax]
        tops.append(top)
        hits = test.contains(ub_dev[:, None].expand_as(top), top).to(torch.float32)
        n_test = test.counts[ub_dev].to(torch.float32)
        for k in k_list:
            hk = hits[:, :k]
            tp = hk.sum(1)
            dcg = (hk * disc[:k]).sum(1)
            n_ideal = torch.clamp(n_test, max=k).to(torch.int64)
            idcg = torch.where(n_ideal > 0, cum_ideal[(n_ideal - 1).clamp(min=0)], torch.full_like(dcg, float("inf")))
            sums[k]["precision"] += float((tp / k).sum())
            sums[k]["recall"] += float((tp / n_test).sum())  # NaN for users without test items, as in the reference
            sums[k]["ndcg"] += float((dcg / idcg).sum())
        n_done += ub.shape[0]
    out = {k: {m: v / max(n_done, 1) for m, v in d.items()} for k, d in sums.items()}
    return out, (torch.cat(tops) if tops else torch.zeros(0, kmax, dtype=torch.int64, device=dev))
