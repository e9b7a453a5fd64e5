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


def metrics_from_ranks(ranks, n_test: np.ndarray, k_list) -> torch.Tensor:
    """Mean ranking metrics of the rows of ``ranks`` (a ``model.TargetRanks``, or anything with its fields) as one fp64 tensor:
    for each k of ``k_list`` precision, recall, ndcg and hit, then mrr, auc and mean_rank (see ``rank_metrics``).  ``n_test``
    (host array): the denominator ``T_u`` of each row.  Per-row terms in fp64 (integer counts exact), each row summed in target order and the
    rows summed in a fixed order, so the result is deterministic; works on CPU or CUDA tensors alike."""
    dev = ranks.rank.device
    U = ranks.ptr.numel() - 1
    rk = ranks.rank
    seg = torch.repeat_interleave(torch.arange(U, device=dev), ranks.ptr.diff(), output_size=rk.numel())
    valid = rk >= 0
    max_t = int(min(max(k_list), max(int(n_test.max()) if U else 0, 1)))  # the ideal DCG needs min(k, T_u) <= max_t terms
    n_test = torch.from_numpy(np.asarray(n_test, dtype=np.float64)).to(dev)

    def per_row(x):  # integer sum per row
        return torch.zeros(U, dtype=torch.int64, device=dev).index_add_(0, seg, x.to(torch.int64)).to(torch.float64)

    def mean(x, mask=None):
        if mask is None:
            return x.sum() / max(U, 1)
        return torch.where(mask, x, 0.0).sum() / mask.sum().clamp(min=1)

    cum_ideal = torch.from_numpy(np.cumsum(1.0 / np.log2(np.arange(2, max_t + 2, dtype=np.float64)))).to(dev)
    gain = torch.where(valid, 1.0 / torch.log2(rk.clamp(min=0).to(torch.float64) + 2.0), 0.0)
    out = []
    for k in k_list:
        in_k = valid & (rk < k)
        h = per_row(in_k)
        dcg = torch.segment_reduce(torch.where(in_k, gain, 0.0), "sum", offsets=ranks.ptr, unsafe=True)
        n_ideal = n_test.clamp(max=k).to(torch.int64)
        idcg = torch.where(n_ideal > 0, cum_ideal[(n_ideal - 1).clamp(min=0, max=max_t - 1)], float("inf"))
        out += [mean(h / k), mean(h / n_test), mean(dcg / idcg), mean((h > 0).to(torch.float64))]
    P = per_row(valid)
    S = per_row(torch.where(valid, rk, 0))
    big = torch.iinfo(torch.int64).max
    best = torch.full((U,), big, dtype=torch.int64, device=dev).scatter_reduce_(0, seg, torch.where(valid, rk, big), "amin")
    mrr = torch.where(P > 0, 1.0 / (1.0 + best.clamp(max=2**53).to(torch.float64)), 0.0)
    N = ranks.eligible.to(torch.float64) - P
    auc = 1.0 - (S - P * (P - 1) / 2) / (P * N)
    out += [mean(mrr), mean(auc, (P > 0) & (N > 0)), mean(S / P, P > 0)]
    return torch.stack(out)


@torch.no_grad()
def rank_metrics(model, train: InteractionCSR, test: InteractionCSR, k_list=(20, 40, 60, 80, 100), users=None) -> dict:
    """Full-ranking metrics of ``users`` (default: every user with at least one test item, as ``evaluate``), from the exact rank
    of each test item among all problems not in the user's training positives (``model.rank(users, train.item_num, test,
    exclude=train)``); no score matrix.  With ``T_u`` = the user's number of test items (``evaluate``'s denominator) and
    ``h_k`` = the test items of rank < k, per user:

        precision@k = h_k / k                  recall@k = h_k / T_u (NaN when T_u = 0, as the reference)
        ndcg@k      = sum_{rank < k} 1 / log2(rank + 2)  /  sum_{i < min(k, T_u)} 1 / log2(i + 2)
        hit@k       = [h_k > 0]                mrr = 1 / (1 + lowest rank), 0 when no test item is eligible
        mean_rank   = the mean rank of the user's eligible test items
        auc         = 1 - sum_i (r_(i) - i) / (P' N'), r_(0) < r_(1) < ... the eligible test items' ranks, P' their number,
                      N' = eligible problems - P': the fraction of (test item, other eligible problem) pairs ordered correctly

    A test item that is also a training positive is not eligible: it counts in ``T_u`` but has no rank.  Users without an
    eligible test item, or without any other eligible problem, have no AUC and no mean rank, and are left out of those two
    means; every other metric is the mean over all ``users``.  ``k`` may be any positive int.  Exactly the top-k that
    ``evaluate`` sees for k <= 128 when the user has at least k eligible problems (``evaluate`` then has no masked entry in its
    top-k).  Per-user terms are computed on the device in fp64 and reduced in a fixed order; the result is read back once.

    Returns ``{k: {"precision", "recall", "ndcg", "hit"} for k in k_list, "mrr": float, "auc": float, "mean_rank": float}``."""
    k_list = [int(k) for k in k_list]
    if not k_list or min(k_list) < 1:
        raise ValueError(f"k_list must hold positive ints, got {k_list}")
    model.eval()
    if users is None:
        users = np.nonzero(np.diff(test.ptr_host) > 0)[0]
    users = torch.as_tensor(np.asarray(users, dtype=np.int64))
    ranks = model.rank(users, train.item_num, test, exclude=train)
    vals = metrics_from_ranks(ranks, np.diff(test.ptr_host)[users.numpy()], k_list).tolist()
    out: dict = {k: dict(zip(("precision", "recall", "ndcg", "hit"), vals[4 * j : 4 * j + 4])) for j, k in enumerate(k_list)}
    out.update(zip(("mrr", "auc", "mean_rank"), vals[4 * len(k_list) :]))
    return out


class TripleSet:
    """A set of CKG triples ``(h, r, t)`` as sorted unique int64 keys ``(h * relation_num + r) * node_num + t`` on the device:
    the known triples of the filtered link-prediction protocol (``KGAT.complete`` / ``KGAT.kg_rank`` ``exclude``)."""

    def __init__(self, heads, relations, tails, node_num: int, relation_num: int, device):
        node_num, relation_num = int(node_num), int(relation_num)
        if node_num < 1 or relation_num < 1:
            raise ValueError("node_num and relation_num must be positive")
        if node_num * node_num * relation_num > np.iinfo(np.int64).max:
            raise ValueError(f"keys of {node_num} nodes and {relation_num} relations do not fit int64")
        cols = [torch.as_tensor(x).to(device=device, dtype=torch.int64).flatten() for x in (heads, relations, tails)]
        if not cols[0].numel() == cols[1].numel() == cols[2].numel():
            raise ValueError("heads, relations and tails differ in length")
        h, r, t = cols
        if h.numel():
            lo = torch.stack([h.min(), r.min(), t.min()]).min()
            hi_h, hi_r, hi_t = torch.stack([h.max(), r.max(), t.max()]).tolist()
            if int(lo) < 0 or hi_h >= node_num or hi_t >= node_num or hi_r >= relation_num:
                raise ValueError(f"triples must hold node ids in [0, {node_num}) and relation ids in [0, {relation_num})")
        self.node_num, self.relation_num = node_num, relation_num
        self.keys = torch.unique((h * relation_num + r) * node_num + t)  # sorted

    @classmethod
    def from_ckg(cls, g, device="cuda") -> "TripleSet":
        """Every triple of the CKG edge list (``g.heads / relations / tails``): what TransR trains on."""
        return cls(torch.from_numpy(np.asarray(g.heads)), torch.from_numpy(np.asarray(g.relations)), torch.from_numpy(np.asarray(g.tails)),
                   g.node_num, g.relation_num, device)

    def __len__(self) -> int:
        return int(self.keys.numel())

    def triples(self):
        """(heads, relations, tails) int64 on the device, in key order."""
        t = self.keys % self.node_num
        hr = self.keys // self.node_num
        return hr // self.relation_num, hr % self.relation_num, t


def link_terms(rank: torch.Tensor, hits) -> torch.Tensor:
    """Per-query fp64 terms [Q, 3 + len(hits)] of the filtered link-prediction metrics from 0-based ranks (-1 = not ranked):
    ranked flag, 1 / (rank + 1), rank + 1, then [rank < k] for every k of ``hits``; zeros for unranked queries."""
    ok = rank >= 0
    r1 = (rank + 1).to(torch.float64)
    cols = [ok.to(torch.float64), torch.where(ok, 1.0 / r1, 0.0), torch.where(ok, r1, 0.0)]
    cols += [(ok & (rank < k)).to(torch.float64) for k in hits]
    return torch.stack(cols, 1)


@torch.no_grad()
def link_metrics(model, triples, known, hits=(1, 3, 10), candidates="relation") -> dict:
    """Filtered link prediction of the trained TransR half: the rank of each held-out triple's tail (``KGAT.kg_rank``) among the
    candidates, with every other triple of ``known`` (a ``TripleSet``) filtered out (Bordes et al. 2013).

    ``triples``: a ``TripleSet`` or ``(heads, relations, tails)`` of the triples to rank.  ``candidates``: ``"relation"`` -- the
    tail nodes of the query's relation in ``known`` (type-constrained), ``"all"`` -- every CKG node, or a 1-D tensor of node
    ids.  Head prediction needs no second call: every CKG relation has its inverse in the edge list.  Queries are grouped by
    relation, one ``kg_rank`` call per relation; per-query terms are fp64 on the device, summed in a fixed order and read back
    once.  A triple whose tail is not a candidate is skipped (``n_skipped``).

    Returns ``{"mrr", "mean_rank" (1-based), "hits": {k: ...}, "per_relation": {r: {"mrr", "mean_rank", "hits", "n_ranked"}},
    "n_ranked", "n_skipped"}``; means over the ranked queries (NaN when there is none)."""
    hits = [int(k) for k in hits]
    if not hits or min(hits) < 1:
        raise ValueError(f"hits must hold positive ints, got {hits}")
    dev = model._device()
    N, R = model.node_num, model._relation_num
    if known.node_num != N or known.relation_num != R:
        raise ValueError(f"known is a TripleSet over {known.node_num} nodes and {known.relation_num} relations, the model has {N} and {R}")
    if isinstance(triples, TripleSet):
        h, r, t = triples.triples()
    else:
        h, r, t = (torch.as_tensor(x).to(device=dev, dtype=torch.int64).flatten() for x in triples)
    if isinstance(candidates, str) and candidates not in ("relation", "all"):
        raise ValueError(f'candidates must be "relation", "all" or a tensor of node ids, got {candidates!r}')
    rels = torch.unique(r).tolist()
    if rels and (rels[0] < 0 or rels[-1] >= R):
        raise ValueError(f"relation ids must lie in [0, {R})")
    if isinstance(candidates, str) and candidates == "relation":
        _, kr, kt = known.triples()
    sums, per = [], []
    for rel in rels:
        sel = torch.nonzero(r == rel).flatten()
        if isinstance(candidates, str):
            cand = N if candidates == "all" else torch.unique(kt[kr == rel])
        else:
            cand = candidates
        ranks = model.kg_rank(h[sel], r[sel], t[sel], cand, exclude=known)
        per.append(link_terms(ranks.rank, hits).sum(0))
    terms = torch.stack(per) if per else torch.zeros(0, 3 + len(hits), dtype=torch.float64, device=dev)
    vals = torch.cat([terms, terms.sum(0, keepdim=True)]).tolist()  # rows: relations in ascending id, then the total

    def summary(v):
        n = v[0]
        div = (lambda x: x / n) if n > 0 else (lambda x: float("nan"))
        return {"mrr": div(v[1]), "mean_rank": div(v[2]), "hits": {k: div(v[3 + j]) for j, k in enumerate(hits)}, "n_ranked": int(n)}

    total = summary(vals[-1])
    return {"mrr": total["mrr"], "mean_rank": total["mean_rank"], "hits": total["hits"],
            "per_relation": {rel: summary(v) for rel, v in zip(rels, vals[:-1])}, "n_ranked": total["n_ranked"],
            "n_skipped": int(h.numel()) - total["n_ranked"]}
