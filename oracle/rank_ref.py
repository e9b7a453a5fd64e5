"""Reference for ``kgat_rank_targets`` / ``KGAT.rank`` written with stock torch ops (CPU or CUDA tensors).

Definition (include/kgat_b200.h): the candidates are ``items`` in their given order; candidate ``c`` is eligible for user ``u``
unless it is in ``u``'s exclusion list.  The key of ``c`` is ``(float_key(s(u, c)), -position(c))`` compared
lexicographically -- the ``topk_rows`` key (NaN largest, -0 below +0), then the earlier position -- which is
``recommend``'s order.  For each target ``p`` of ``u`` that is an eligible candidate:

    rank(u, p) = #{ c eligible for u : key(c) > key(p) }

and -1 for any other target.  ``eligible`` counts the eligible candidates.

The scores are an input (``scores[b, x]`` = score of user row ``b`` and item id ``x``), so a test can feed the bit-exact
``PREDICT`` scores and expect identical ranks.
"""

from __future__ import annotations

import torch

from oracle.recommend_ref import float_key

_I64 = torch.int64


def rank_ref(scores, users, items, target_ptr, target_items, exclude_ptr=None, exclude_items=None):
    """(ptr int64 [U+1], items int64 [M], scores fp32 [M], rank int64 [M], eligible int64 [U]).  ``scores``: fp32 [U, N] over
    item ids 0 .. N-1 (every candidate and target below N); ``users``: ids into ``target_ptr`` / ``exclude_ptr``, repeats
    allowed; ``target_ptr`` / ``target_items``: per user the targets, ascending; ``exclude_ptr`` / ``exclude_items``: per user
    the excluded item ids (any order)."""
    dev = scores.device
    users = users.to(device=dev, dtype=_I64)
    cand = items.to(device=dev, dtype=_I64)
    tptr = target_ptr.to(device=dev, dtype=_I64)
    titems = target_items.to(device=dev, dtype=_I64)
    U, n = users.numel(), cand.numel()
    pos = torch.arange(n, device=dev)
    key = float_key(scores)
    out_ptr = [0]
    out_items, out_scores, out_rank, eligible = [], [], [], []
    for b in range(U):
        u = int(users[b])
        tg = titems[tptr[u] : tptr[u + 1]]
        elig = torch.ones(n, dtype=torch.bool, device=dev)
        if exclude_ptr is not None:
            elig &= ~torch.isin(cand, exclude_items[exclude_ptr[u] : exclude_ptr[u + 1]].to(device=dev, dtype=_I64))
        eligible.append(int(elig.sum()))
        ck, cp = key[b, cand][elig], pos[elig]
        match = tg[:, None] == cand[None, :]  # [T, n]
        found = match.any(1)
        tpos = torch.where(found, match.to(torch.int8).argmax(1), 0)
        t_elig = found & elig[tpos]
        tk = key[b, tg]
        beats = (ck[None, :] > tk[:, None]) | ((ck[None, :] == tk[:, None]) & (cp[None, :] < tpos[:, None]))
        out_rank.append(torch.where(t_elig, beats.sum(1), -1))
        out_items.append(tg)
        out_scores.append(scores[b, tg])
        out_ptr.append(out_ptr[-1] + tg.numel())
    cat = lambda xs, dt: torch.cat(xs) if xs else torch.zeros(0, dtype=dt, device=dev)  # noqa: E731
    return (torch.tensor(out_ptr, dtype=_I64, device=dev), cat(out_items, _I64), cat(out_scores, torch.float32), cat(out_rank, _I64),
            torch.tensor(eligible, dtype=_I64, device=dev))


def auc_pairs(scores_row, items, targets, excluded=()):
    """AUC of one user by brute-force pair counting: the fraction of (eligible target, eligible non-target) candidate pairs in
    which the target's key is the larger.  NaN when either side is empty."""
    cand = items.to(_I64).tolist()
    ex = set(int(x) for x in excluded)
    tg = set(int(x) for x in targets)
    key = float_key(scores_row).tolist()
    k = {c: (key[c], -j) for j, c in enumerate(cand) if c not in ex}
    pos = [k[c] for c in k if c in tg]
    neg = [k[c] for c in k if c not in tg]
    if not pos or not neg:
        return float("nan")
    return sum(p > q for p in pos for q in neg) / (len(pos) * len(neg))
