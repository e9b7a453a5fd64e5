#!/usr/bin/env python
"""Top-k recommendations for every user in one call (``KGAT.recommend``) against the batched paths it replaces.

C4 (Yelp2018 shape, 45,919 users x 45,538 items), k = 20, training positives excluded:
  * ``model.recommend`` -- one call;
  * the existing ``recommend_topk`` loop over 256-user batches (gather + SGEMM + mask + radix top-k per batch, the scheme of
    ``metrics.evaluate`` and test_yelp2018_shape_full_graph_top20), masks prepared before timing;
  * torch: cuBLAS fp32 matmul + index_put of -inf + ``torch.topk`` per 256-user batch, masks prepared before timing.
  The one call must equal the loop bit for bit; torch sums in another order and is reported as an agreement fraction.
Codeforces-full (200,000 users x 10,000 problems), k = 20, training positives excluded: ``model.recommend`` unfiltered and with
``require = [four adjacent rating entities, one tag]``.

Every time is the median of --reps warmed calls (CUDA events around the call; a call that reads back its range checks
synchronises anyway).  FLOPs = 2 * users * candidates * concatenated width; the FP32 FFMA peak is 148 SMs x 128 lanes x 2 x
the max SM clock read from nvidia-smi in the same run.

    python tools/prof_recommend.py [--out profiles/recommend_b200.json]
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

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=10)
ap.add_argument("--k", type=int, default=20)
ap.add_argument("--batch", type=int, default=256)
ap.add_argument("--out", default=None)
args = ap.parse_args()


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"], capture_output=True,
                       text=True)
    line = q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 and q.stdout.strip() else ""
    parts = [p.strip() for p in line.split(",")] if line else []
    out = {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": line, "sm_count": torch.cuda.get_device_properties(0).multi_processor_count}
    if len(parts) == 3:
        out["power_limit_w"] = float(parts[1])
        out["max_sm_clock_mhz"] = float(parts[2])
    return out


def timed(fn, reps: int):
    for _ in range(2):
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
    return out, ts


def stats(ts, users, n_cand, width, peak):
    med = float(np.median(ts))
    flops = 2.0 * users * n_cand * width
    return {"ms_median": med, "ms_min": float(min(ts)), "ms_max": float(max(ts)), "reps": len(ts), "users_per_s": users / (med * 1e-3),
            "flops": flops, "tflops": flops / (med * 1e-3) / 1e12, "fraction_of_fp32_ffma_peak": flops / (med * 1e-3) / peak if peak else None}


hw = card()
peak = hw["sm_count"] * 128 * 2 * hw["max_sm_clock_mhz"] * 1e6 if "max_sm_clock_mhz" in hw else None
results = {"card": hw, "fp32_ffma_peak_tflops": peak / 1e12 if peak else None, "k": args.k, "runs": []}
dev = torch.device("cuda")
k = args.k

# ---------------------------------------------------------------------------------------------------- C4
t0 = time.time()
g = synthetic.make_ckg("yelp2018", with_dicts=False)
m = build_model(g, "cuda").eval()
train = InteractionCSR(g.train_interactions, g.user_num, g.item_num, "cuda")
tables = m._tables()
width = sum(t.shape[1] for t in tables)
U, n = g.user_num, g.item_num
items = torch.arange(n, device=dev)
batches = []
for s in range(0, U, args.batch):
    e = min(s + args.batch, U)
    ptr, flat = train.batch(s, e)
    rows = torch.repeat_interleave(torch.arange(e - s, device=dev), (ptr[1:] - ptr[:-1]).long())
    batches.append((s, e, torch.arange(s, e, device=dev), ptr, flat, rows, flat.long()))
setup_s = time.time() - t0

one, t_one = timed(lambda: m.recommend(torch.arange(U), n, k=k, exclude=train), args.reps)


def loop():
    out = torch.empty(U, k, dtype=torch.int32, device=dev)
    val = torch.empty(U, k, dtype=torch.float32, device=dev)
    for s, e, ub, ptr, flat, _, _ in batches:
        out[s:e], val[s:e] = m.recommend_topk(ub, items, k, ptr, flat, want_values=True)
    return out, val


table = torch.cat(tables, 1)
item_rows = table[:n].contiguous()


def torch_loop():
    out = torch.empty(U, k, dtype=torch.int64, device=dev)
    for s, e, ub, _, _, rows, cols in batches:
        sc = table[ub] @ item_rows.T
        sc[rows, cols] = -float("inf")
        out[s:e] = torch.topk(sc, k, dim=1).indices
    return out


(lp_items, lp_vals), t_loop = timed(loop, args.reps)
th_items, t_torch = timed(torch_loop, args.reps)
exact = bool(torch.equal(one.items, lp_items.long()) and torch.equal(one.scores.view(torch.int32), lp_vals.view(torch.int32)))
users_all = torch.arange(U, device=dev)[:, None].expand(-1, k)
no_train = not bool(train.contains(users_all, one.items).any())
r = {"shape": "yelp2018 (C4)", "users": U, "candidates": n, "width": width, "setup_s": setup_s,
     "recommend_one_call": stats(t_one, U, n, width, peak),
     "recommend_topk_256_loop": stats(t_loop, U, n, width, peak),
     "torch_cublas_mask_topk_256_loop": stats(t_torch, U, n, width, peak),
     "speedup_vs_recommend_topk_loop": float(np.median(t_loop) / np.median(t_one)),
     "speedup_vs_torch_loop": float(np.median(t_torch) / np.median(t_one)),
     "bit_identical_to_recommend_topk_loop": exact,
     "index_agreement_with_torch": float((th_items == one.items).float().mean()),
     "recommends_no_training_positive": no_train,
     "not_slower_than_recommend_topk_loop": bool(np.median(t_one) <= np.median(t_loop))}
print(json.dumps(r), flush=True)
results["runs"].append(r)
assert exact and no_train, r
del m, tables, table, item_rows, batches, one, lp_items, lp_vals, th_items, train
torch.cuda.empty_cache()

# ---------------------------------------------------------------------------------------------------- Codeforces-full
t0 = time.time()
g = synthetic.make_ckg("codeforces-full", with_dicts=False)
m = build_model(g, "cuda").eval()
train = InteractionCSR(g.train_interactions, g.user_num, g.item_num, "cuda")
width = sum(t.shape[1] for t in m._tables())
U, n = g.user_num, g.item_num
t_ent = n + 1_913 + 5  # first tag entity (synthetic._codeforces_triples: problems, contests, divisions, tags, ratings)
r_ent = t_ent + 37     # first rating entity
require = [[r_ent + 8, r_ent + 9, r_ent + 10, r_ent + 11], [t_ent + 1]]
setup_s = time.time() - t0
for name, req in (("unfiltered", None), ("require 4 ratings AND 1 tag", require)):
    rec, ts = timed(lambda: m.recommend(torch.arange(U), n, k=k, exclude=train, require=req), args.reps)
    n_cand = n if req is None else int(ops.recommend_filter(m._graph(), torch.arange(n), req, g.user_num)[2])
    again = m.recommend(torch.arange(U), n, k=k, exclude=train, require=req)
    users_all = torch.arange(U, device=dev)[:, None].expand(-1, k)
    valid = rec.items >= 0
    r = {"shape": "codeforces-full (C2)", "mode": name, "require": req, "users": U, "items": n, "candidates": n_cand, "width": width,
         "setup_s": setup_s, "recommend_one_call": stats(ts, U, n_cand, width, peak),
         "users_with_k": int((rec.count == k).sum()), "repeatable": bool(torch.equal(rec.items, again.items)),
         "recommends_no_training_positive": not bool(train.contains(users_all[valid], rec.items[valid]).any())}
    print(json.dumps(r), flush=True)
    results["runs"].append(r)
    assert r["repeatable"] and r["recommends_no_training_positive"], r

if args.out:
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(results, indent=1) + "\n")
