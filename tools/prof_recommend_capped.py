#!/usr/bin/env python
"""Capped top-k recommendations (``KGAT.recommend_capped``) at codeforces-full (200,000 users x 10,000 problems), k = 20, training
positives excluded, for three cap sets:
  (a) at most 2 problems per tag;  (b) at most 3 per tag and 4 per rating;  (tight) at most 1 per tag.
For each: the time of one call, its rounds and the active rows per round; next to it, in the same run:
  * ``recommend`` at k = 20 and at k = m (the capped call's candidates per row and round);
  * an exact torch baseline per 256-user batch: cuBLAS fp32 scores, -inf on the exclusions, a full stable sort, and the greedy
    vectorised over the batch, stopping once every row of the batch is finished (its scores sum in another order, so it is
    reported as an agreement fraction);
  * the over-fetch workaround: ``recommend(k=128)`` and the greedy over those 128 only, with the share of users it gets wrong
    (a different list) or leaves short (fewer than k while the exact list has k);
  * the mean number of distinct tags and ratings per list, for plain ``recommend(k=20)`` and for the capped lists.

Every GPU time is the median of --reps warmed calls (CUDA events around the call, read-backs included); the torch baseline is
slow and is timed over --torch-reps calls.  The card's name and power limit are read in the same run.

    python tools/prof_recommend_capped.py [--out profiles/recommend_capped_b200.json]
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

from kgat_b200 import ops, synthetic  # noqa: E402
from kgat_b200.metrics import InteractionCSR  # noqa: E402
from kgat_b200.trainer import build_model  # noqa: E402
from oracle.recommend_ref import filter_ref  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=10)
ap.add_argument("--torch-reps", type=int, default=1)
ap.add_argument("--k", type=int, default=20)
ap.add_argument("--batch", type=int, default=256)
ap.add_argument("--out", default=None)
args = ap.parse_args()


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"], capture_output=True,
                       text=True)
    line = q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 and q.stdout.strip() else ""
    parts = [p.strip() for p in line.split(",")] if line else []
    out = {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": line}
    if len(parts) == 3:
        out["power_limit_w"] = float(parts[1])
        out["max_sm_clock_mhz"] = float(parts[2])
    return out


def timed(fn, reps: int, warm: int = 2):
    for _ in range(warm):
        out = fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return out, {"ms_median": float(np.median(ts)), "ms_min": float(min(ts)), "ms_max": float(max(ts)), "reps": len(ts)}


def greedy(order_items, member, cap, k):
    """The capped greedy over the columns of order_items (int64 [B, L], -1 = no candidate), vectorised over the rows;
    member: bool [n_items, G].  Stops once every row is finished.  Returns (items [B, k], count [B])."""
    B, L = order_items.shape
    dev = order_items.device
    cnt = torch.zeros(B, member.shape[1], dtype=torch.int32, device=dev)
    n = torch.zeros(B, dtype=torch.int64, device=dev)
    out = torch.full((B, k + 1), -1, dtype=torch.int64, device=dev)  # column k takes the writes of finished rows
    rows = torch.arange(B, device=dev)
    for j0 in range(0, L, 64):  # one read-back per 64 steps to stop early
        for j in range(j0, min(j0 + 64, L)):
            it = order_items[:, j]
            mem = member[it.clamp(min=0)] & (it >= 0)[:, None]
            ok = (it >= 0) & (n < k) & ~(mem & (cnt >= cap)).any(1)
            cnt += (mem & ok[:, None]).int()
            out[rows, torch.where(ok, n, k)] = torch.where(ok, it, -1)
            n += ok.long()
        if bool((n == k).all()):
            break
    return out[:, :k], n


hw = card()
dev = torch.device("cuda")
k = args.k
t0 = time.time()
g = synthetic.make_ckg("codeforces-full", with_dicts=False)
m = build_model(g, "cuda").eval()
train = InteractionCSR(g.train_interactions, g.user_num, g.item_num, "cuda")
U, n = g.user_num, g.item_num
t_ent = n + 1_913 + 5  # first tag entity (synthetic._codeforces_triples: problems, contests, divisions, tags, ratings)
r_ent = t_ent + 37     # first rating entity
tags, ratings = list(range(t_ent, t_ent + 37)), list(range(r_ent, r_ent + 28))
graph = m._graph()
items = torch.arange(n, device=dev)


def membership(groups):
    mem = torch.zeros(n, len(groups), dtype=torch.bool, device=dev)
    for j, grp in enumerate(groups):
        mem[filter_ref(graph.row_ptr, graph.col_idx, items, [grp], g.user_num), j] = True
    return mem


tag_mem, rating_mem = membership([[t] for t in tags]), membership([[r] for r in ratings])


def diversity(lst):
    valid = (lst >= 0)[:, :, None]
    x = lst.clamp(min=0)
    return {"distinct_tags": float(((tag_mem[x] & valid).any(1)).sum(1).float().mean()),
            "distinct_ratings": float(((rating_mem[x] & valid).any(1)).sum(1).float().mean())}


table = torch.cat(m._tables(), 1)
item_rows = table[:n].contiguous()
batches = []
for s in range(0, U, args.batch):
    e = min(s + args.batch, U)
    ptr, flat = train.batch(s, e)
    rows = torch.repeat_interleave(torch.arange(e - s, device=dev), (ptr[1:] - ptr[:-1]).long())
    batches.append((s, e, rows, flat.long()))
setup_s = time.time() - t0
users = torch.arange(U)

plain, t_plain = timed(lambda: m.recommend(users, n, k=k, exclude=train), args.reps)
results = {"card": hw, "shape": "codeforces-full", "users": U, "items": n, "k": k, "m": max(k, 64), "setup_s": setup_s,
           "recommend_k": {"time": t_plain, **diversity(plain.items)}, "runs": []}
_, t_m = timed(lambda: m.recommend(users, n, k=max(k, 64), exclude=train), args.reps)
results["recommend_k_m"] = {"time": t_m}
over, t_over = timed(lambda: m.recommend(users, n, k=128, exclude=train), args.reps)
results["recommend_k128"] = {"time": t_over}
print(json.dumps(results), flush=True)

cap_sets = {"a: 2 per tag": [([t], 2) for t in tags],
            "b: 3 per tag, 4 per rating": [([t], 3) for t in tags] + [([r], 4) for r in ratings],
            "tight: 1 per tag": [([t], 1) for t in tags]}
for name, caps in cap_sets.items():
    groups, values = ops.cap_groups(caps, g.entity_num)
    member = membership(groups)
    cap = torch.tensor(values, dtype=torch.int32, device=dev)
    got, t_cap = timed(lambda: m.recommend_capped(users, n, k, caps, exclude=train), args.reps)
    active = []
    tables = m._tables()
    ops.launch_recommend_capped(tables, graph, users.to(dev, torch.int32), items.int(), k, groups, values, g.user_num, train.ptr_dev,
                                train.items, active_rows=active)

    def torch_exact():
        out = torch.empty(U, k, dtype=torch.int64, device=dev)
        for s, e, rows, cols in batches:
            sc = table[s:e] @ item_rows.T
            sc[rows, cols] = -float("inf")
            order = torch.sort(sc, dim=1, descending=True, stable=True).indices
            order = torch.where(torch.gather(sc, 1, order) == -float("inf"), -1, order)  # excluded: no candidate
            out[s:e] = greedy(order, member, cap, k)[0]
        return out

    th, t_torch = timed(torch_exact, args.torch_reps, warm=1)

    def overfetch():
        r = m.recommend(users, n, k=128, exclude=train)
        return greedy(r.items, member, cap, k)

    (of_items, of_n), t_of = timed(overfetch, args.reps)
    exact_full = got.count == k
    r = {"caps": name, "groups": len(caps), "recommend_capped": t_cap, "rounds": len(active), "active_rows_per_round": active,
         "torch_exact_256_batches": t_torch, "speedup_vs_torch_exact": t_torch["ms_median"] / t_cap["ms_median"],
         "index_agreement_with_torch_exact": float((th == got.items).float().mean()),
         "overfetch_recommend128_plus_filter": t_of,
         "overfetch_users_wrong": float((of_items != got.items).any(1).float().mean()),
         "overfetch_users_short": float(((of_n < k) & exact_full).float().mean()),
         "users_with_k": int(exact_full.sum()), **diversity(got.items)}
    print(json.dumps(r), flush=True)
    results["runs"].append(r)
    assert len(active) <= len(caps) + 1, r

if args.out:
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(results, indent=1) + "\n")
