"""Reference for ``kgat_complete_topk`` / ``kgat_complete_rank`` / ``KGAT.complete`` / ``KGAT.kg_rank`` written with stock torch
ops (CPU or CUDA tensors).

Definition (include/kgat_b200.h): a query is ``(h, r)``; its candidates are ``candidates`` in their given order.  Candidate
``c`` is eligible unless ``(h, r, c)`` is a known triple; for a rank with target ``t`` the target itself stays eligible.  The
key of ``c`` is ``(key32(E(h, r, c)), -position(c))`` compared lexicographically, where ``key32(E) = float_key(-E)`` (lower
energy ranks first, -0 below +0) and a NaN energy takes the largest key.  Then

    complete: the first k eligible candidates in key order (node ids, energies, their number; padded with -1 / +inf)
    rank(q)  = #{ c eligible, c != t : key(c) > key(t) },  -1 when t is not a candidate

The energies are an input (``energy[q, x]`` = energy of query ``q`` and node ``x``), so a test can feed the kernel's bit-exact
energies and expect identical results.  ``energy_f64`` gives the energy in fp64 for tolerance checks.
"""

from __future__ import annotations

import numpy as np
import torch

from oracle.recommend_ref import float_key

_I64 = torch.int64


def key32(energy: torch.Tensor) -> torch.Tensor:
    """int64 key of the energies: float_key of the sign-flipped value, NaN largest."""
    flipped = (energy.contiguous().view(torch.int32) ^ torch.tensor(-(2**31), dtype=torch.int32)).view(torch.float32)
    k = float_key(flipped)
    return torch.where(torch.isnan(energy), torch.full_like(k, 0xFFFFFFFF), k)


def _known(keys, h, r, cand, node_num, relation_num):
    """bool [n]: (h, r, cand[i]) is in the sorted key tensor."""
    if keys is None or keys.numel() == 0:
        return torch.zeros(cand.numel(), dtype=torch.bool, device=cand.device)
    q = (h * relation_num + r) * node_num + cand
    pos = torch.searchsorted(keys, q).clamp(max=keys.numel() - 1)
    return keys[pos] == q


def complete_ref(energy, heads, relations, candidates, k, known_keys=None, node_num=None, relation_num=None):
    """(tails int64 [Q, k], energy fp32 [Q, k], count int32 [Q]); ``known_keys``: sorted int64 keys (h R + r) N + t."""
    dev = energy.device
    cand = candidates.to(device=dev, dtype=_I64)
    Q, n = heads.numel(), cand.numel()
    out_t = torch.full((Q, k), -1, dtype=_I64, device=dev)
    out_e = torch.full((Q, k), float("inf"), dtype=torch.float32, device=dev)
    count = torch.zeros(Q, dtype=torch.int32, device=dev)
    pos = torch.arange(n, device=dev)
    for q in range(Q):
        ok = ~_known(known_keys, int(heads[q]), int(relations[q]), cand, node_num, relation_num)
        kq = key32(energy[q, cand])[ok]
        # key descending, then position ascending: sort by position first, then a stable sort on the key
        idx = torch.sort(kq, descending=True, stable=True).indices[:k]
        sel = pos[ok][idx]
        m = sel.numel()
        out_t[q, :m] = cand[sel]
        out_e[q, :m] = energy[q, cand[sel]]
        count[q] = m
    return out_t, out_e, count


def kg_rank_ref(energy, heads, relations, tails, candidates, known_keys=None, node_num=None, relation_num=None):
    """(energy fp32 [Q], rank int64 [Q], eligible int64 [Q])."""
    dev = energy.device
    cand = candidates.to(device=dev, dtype=_I64)
    Q, n = heads.numel(), cand.numel()
    pos = torch.arange(n, device=dev)
    ranks, elig = [], []
    for q in range(Q):
        t = int(tails[q])
        ok = ~_known(known_keys, int(heads[q]), int(relations[q]), cand, node_num, relation_num) | (cand == t)
        elig.append(int(ok.sum()))
        hit = torch.nonzero(cand == t).flatten()
        if hit.numel() == 0:
            ranks.append(-1)
            continue
        tp = int(hit[0])
        kc = key32(energy[q, cand])
        kt = kc[tp]
        beats = (kc > kt) | ((kc == kt) & (pos < tp))
        ranks.append(int((beats & ok & (cand != t)).sum()))
    return (energy[torch.arange(Q, device=dev), tails.to(device=dev, dtype=_I64)], torch.tensor(ranks, dtype=_I64, device=dev),
            torch.tensor(elig, dtype=_I64, device=dev))


def link_metrics_ref(ranks, hits=(1, 3, 10)) -> dict:
    """MRR, 1-based mean rank and Hits@k of 0-based ranks (-1 = skipped), in numpy fp64."""
    r = np.asarray(ranks, dtype=np.int64)
    r = r[r >= 0].astype(np.float64) + 1.0
    if r.size == 0:
        return {"mrr": float("nan"), "mean_rank": float("nan"), "hits": {k: float("nan") for k in hits}, "n_ranked": 0}
    return {"mrr": float(np.mean(1.0 / r)), "mean_rank": float(np.mean(r)), "hits": {k: float(np.mean(r <= k)) for k in hits},
            "n_ranked": int(r.size)}


def energy_f64(emb, rel_emb, W, heads, relations, tails) -> torch.Tensor:
    """||e_h W_r + e_r - e_t W_r||^2 in fp64 for each (heads[i], relations[i], tails[i])."""
    e, er, w = emb.double(), rel_emb.double(), W.double()
    h, r, t = (x.to(device=e.device, dtype=_I64) for x in (heads, relations, tails))
    xh = torch.bmm(e[h][:, None, :], w[r])[:, 0]
    xt = torch.bmm(e[t][:, None, :], w[r])[:, 0]
    return ((xh + er[r] - xt) ** 2).sum(1)
