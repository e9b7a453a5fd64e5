"""Reference for ``kgat_explain_paths`` / ``KGAT.explain`` written with stock torch ops (CPU or CUDA tensors).

Definition (include/kgat_b200.h): for every pair (s, t) the simple paths s = v0 -> ... -> vh = t, 1 <= h <= H <= 3,
whose hops are stored entries of the attentive matrix A (CSR: row_ptr, col_idx, vals; columns sorted, unique per row).
Weight = fp32 product of the hop values, left to right.  Ranked by weight descending, then h ascending, then (v1, v2)
ascending; the top k are returned with -1 / 0 padding, plus the number of paths (``count``) and their summed weight in
fp64 (``mass``) per length.

Every stored entry (v, w) is found by a binary search of the key v * n + w among the CSR's keys, which ascend in
slot order.  3-hop paths s -> a -> b -> t are enumerated per (pair, a) from the shorter of row a and In(t) (the
column t of A), so the work is the same probe count the kernel has; pairs are processed in chunks of bounded size.
"""

from __future__ import annotations

import torch

_I64 = torch.int64


def _expand(starts: torch.Tensor, lens: torch.Tensor):
    """For segments [starts[i], starts[i] + lens[i]): (owner segment of every element, its position)."""
    owner = torch.repeat_interleave(torch.arange(lens.numel(), device=lens.device), lens)
    first = torch.cumsum(lens, 0) - lens
    pos = torch.arange(owner.numel(), device=lens.device) - first[owner] + starts[owner]
    return owner, pos


def _lookup(keys: torch.Tensor, q: torch.Tensor):
    """(found, slot) of every key in q among the ascending ``keys``."""
    pos = torch.searchsorted(keys, q)
    pos_c = pos.clamp(max=max(keys.numel() - 1, 0))
    found = (pos < keys.numel()) & (keys[pos_c] == q) if keys.numel() else torch.zeros_like(q, dtype=torch.bool)
    return found, pos_c


def explain_paths_ref(row_ptr, col_idx, vals, src, dst, k: int, max_hops: int, max_probes: int = 1 << 24):
    """Returns (nodes [P,k,H+1] int64, slots [P,k,H] int64, hops [P,k] int32, weight [P,k] fp32, count [P,H] int64,
    mass [P,H] fp64) on the device of ``col_idx``."""
    if not 1 <= k <= 64 or max_hops not in (1, 2, 3):
        raise ValueError("k must be in [1, 64] and max_hops in {1, 2, 3}")
    dev = col_idx.device
    H = int(max_hops)
    rp = row_ptr.to(dev, _I64)
    col = col_idx.to(dev, _I64)
    vals = vals.to(dev, torch.float32)
    n = rp.numel() - 1
    deg = rp[1:] - rp[:-1]
    row_of = torch.repeat_interleave(torch.arange(n, device=dev), deg)
    keys = row_of * n + col
    # In(t): the slots of column t, ordered by row
    t_perm = torch.argsort(col * n + row_of, stable=True)
    t_deg = torch.bincount(col, minlength=n)
    t_ptr = torch.cat([torch.zeros(1, dtype=_I64, device=dev), torch.cumsum(t_deg, 0)])
    src = torch.as_tensor(src).to(dev, _I64).flatten()
    dst = torch.as_tensor(dst).to(dev, _I64).flatten()
    P = src.numel()
    nodes = torch.full((P, k, H + 1), -1, dtype=_I64, device=dev)
    slots = torch.full((P, k, H), -1, dtype=_I64, device=dev)
    hops = torch.zeros(P, k, dtype=torch.int32, device=dev)
    weight = torch.zeros(P, k, dtype=torch.float32, device=dev)
    count = torch.zeros(P, H, dtype=_I64, device=dev)
    mass = torch.zeros(P, H, dtype=torch.float64, device=dev)
    if P == 0:
        return nodes, slots, hops, weight, count, mass
    valid = (src >= 0) & (src < n) & (dst >= 0) & (dst < n) & (src != dst)
    s_all, t_all = src.clamp(0, max(n - 1, 0)), dst.clamp(0, max(n - 1, 0))
    # per-pair probe count (chunking only)
    work = torch.ones(P, dtype=_I64, device=dev) + deg[s_all]
    if H >= 3:
        o, p = _expand(rp[s_all], deg[s_all])
        a = col[p]
        work.index_add_(0, o, torch.minimum(deg[a], t_deg[t_all[o]]))
    bounds, start, acc = [], 0, 0
    for j, w in enumerate(work.tolist()):
        if acc and acc + w > max_probes:
            bounds.append((start, j))
            start, acc = j, 0
        acc += w
    bounds.append((start, P))
    for lo, hi in bounds:
        _chunk(lo, hi, s_all, t_all, valid, rp, col, vals, deg, keys, n, t_perm, t_ptr, t_deg, k, H, nodes, slots, hops, weight, count,
               mass)
    return nodes, slots, hops, weight, count, mass


def _chunk(lo, hi, s_all, t_all, valid, rp, col, vals, deg, keys, n, t_perm, t_ptr, t_deg, k, H, nodes, slots, hops, weight, count, mass):
    dev = col.device
    pid = torch.arange(lo, hi, device=dev)
    pid = pid[valid[lo:hi]]
    s, t = s_all[pid], t_all[pid]
    parts = []  # (pair, h, v1, v2, w, slot0, slot1, slot2)
    none = lambda m: torch.full((m,), -1, dtype=_I64, device=dev)  # noqa: E731
    # 1 hop
    f, sl = _lookup(keys, s * n + t)
    parts.append((pid[f], 1, t[f], none(int(f.sum())), vals[sl[f]], sl[f], none(int(f.sum())), none(int(f.sum()))))
    if H >= 2:
        o, slot0 = _expand(rp[s], deg[s])
        a = col[slot0]
        f, slot1 = _lookup(keys, a * n + t[o])
        f &= (a != s[o]) & (a != t[o])
        w = vals[slot0[f]] * vals[slot1[f]]
        parts.append((pid[o[f]], 2, a[f], t[o[f]], w, slot0[f], slot1[f], none(int(f.sum()))))
        if H >= 3:
            keep = (a != s[o]) & (a != t[o])
            o, slot0, a = o[keep], slot0[keep], a[keep]
            tt = t[o]
            from_row = deg[a] <= t_deg[tt]
            for branch in (True, False):
                m = from_row == branch
                oo, s0, aa, t3 = o[m], slot0[m], a[m], tt[m]
                if branch:  # b from row a, look up (b, t)
                    q, slot1 = _expand(rp[aa], deg[aa])
                    b = col[slot1]
                    f, slot2 = _lookup(keys, b * n + t3[q])
                else:  # b from In(t), look up (a, b)
                    q, tpos = _expand(t_ptr[t3], t_deg[t3])
                    slot2 = t_perm[tpos]
                    b = _row_of_slot(rp, slot2)
                    f, slot1 = _lookup(keys, aa[q] * n + b)
                f &= (b != s[oo[q]]) & (b != aa[q]) & (b != t3[q])
                q = q[f]
                w = (vals[s0[q]] * vals[slot1[f]]) * vals[slot2[f]]
                parts.append((pid[oo[q]], 3, aa[q], b[f], w, s0[q], slot1[f], slot2[f]))
    pair = torch.cat([p[0] for p in parts])
    h = torch.cat([torch.full((p[0].numel(),), p[1], dtype=_I64, device=dev) for p in parts])
    v1, v2, w = (torch.cat([p[i] for p in parts]) for i in (2, 3, 4))
    sl = torch.stack([torch.cat([p[i] for p in parts]) for i in (5, 6, 7)], dim=1)
    count.view(-1).index_add_(0, pair * H + h - 1, torch.ones_like(pair))
    mass.view(-1).index_add_(0, pair * H + h - 1, w.to(torch.float64))
    # rank: pair asc, weight desc, h asc, v1 asc, v2 asc (stable sorts from the last key to the first)
    order = torch.argsort(v2, stable=True)
    for key, desc in ((v1, False), (h, False), (w, True), (pair, False)):
        order = order[torch.sort(key[order], stable=True, descending=desc).indices]
    pair, h, v1, v2, w, sl = pair[order], h[order], v1[order], v2[order], w[order], sl[order]
    first = torch.searchsorted(pair, pair)  # pair is ascending now: index of the first entry of each pair
    rank = torch.arange(pair.numel(), device=dev) - first
    m = rank < k
    pair, rank, h, v1, v2, w, sl = pair[m], rank[m], h[m], v1[m], v2[m], w[m], sl[m]
    hops[pair, rank] = h.to(torch.int32)
    weight[pair, rank] = w
    s, t = s_all[pair], t_all[pair]
    nodes[pair, rank, 0] = s
    nodes[pair, rank, h] = t
    nodes[pair, rank, 1] = torch.where(h >= 2, v1, nodes[pair, rank, 1])
    if H >= 3:
        nodes[pair, rank, 2] = torch.where(h == 3, v2, nodes[pair, rank, 2])
    for j in range(H):
        slots[pair, rank, j] = torch.where(h > j, sl[:, j], slots[pair, rank, j])


def _row_of_slot(rp: torch.Tensor, slot: torch.Tensor) -> torch.Tensor:
    return torch.searchsorted(rp, slot, right=True) - 1
