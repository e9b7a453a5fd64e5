#!/usr/bin/env python
"""Full-ranking evaluation in one call (``KGAT.rank`` / ``metrics.rank_metrics``) against the batched paths it replaces.

At C4 (Yelp2018 shape, 45,919 users x 45,538 items) and C2 (full Codeforces, 200,000 users x 10,000 problems), for every
user with a test item, k_list = 20, 40, 60, 80, 100, training positives excluded:
  * ``model.rank`` -- one call (the exact rank of every test item);
  * ``metrics.rank_metrics`` -- one call (rank + the per-user terms + the means, one read-back);
  * ``metrics.evaluate`` -- the 256-user ``recommend_topk`` loop (gather + SGEMM + mask + top-100 per batch, host reductions);
  * torch: per 256-user batch a cuBLAS fp32 score matrix, -inf on the training positives, and for every test item the number of
    candidates whose (score, position) beats it -- the same ranks from a materialised matrix.
Hit counts and P / R / nDCG of ``rank_metrics`` must equal ``evaluate``'s; torch sums the scores in another order and is reported
as the fraction of ranks it gets exactly.

Every time is the median of --reps warmed calls (CUDA events around the call; every path reads its result back).  FLOPs =
2 * users * candidates * concatenated width; the FP32 FFMA peak is 148 SMs x 128 lanes x 2 x the max SM clock read from
nvidia-smi in the same run.

    python tools/prof_rank.py [--out profiles/rank_b200.json]
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

from kgat_b200 import synthetic  # noqa: E402
from kgat_b200.metrics import InteractionCSR, evaluate, rank_metrics  # noqa: E402
from kgat_b200.trainer import build_model  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=10)
ap.add_argument("--batch", type=int, default=256)
ap.add_argument("--shapes", default="yelp2018,codeforces-full")
ap.add_argument("--out", default=None)
args = ap.parse_args()
K_LIST = (20, 40, 60, 80, 100)


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
results = {"card": hw, "fp32_ffma_peak_tflops": peak / 1e12 if peak else None, "k_list": list(K_LIST), "runs": []}
dev = torch.device("cuda")

for shape in args.shapes.split(","):
    t0 = time.time()
    g = synthetic.make_ckg(shape)
    m = build_model(g, "cuda").eval()
    train = InteractionCSR(g.train_interactions, g.user_num, g.item_num, "cuda")
    test = InteractionCSR(g.test_dict, g.user_num, g.item_num, "cuda")
    users = np.nonzero(np.diff(test.ptr_host) > 0)[0]
    users_t = torch.from_numpy(users)
    tables = m._tables()
    width = sum(t.shape[1] for t in tables)
    U, n = users.size, g.item_num
    table = torch.cat(tables, 1)
    item_rows = table[:n].contiguous()
    pos = torch.arange(n, device=dev)
    batches = []
    for s in range(0, U, args.batch):
        ub = users[s : s + args.batch]
        cnt = train.ptr_host[ub + 1] - train.ptr_host[ub]
        idx = np.concatenate([np.arange(train.ptr_host[u], train.ptr_host[u + 1]) for u in ub])
        rows = torch.from_numpy(np.repeat(np.arange(ub.size), cnt)).to(dev)
        cols = train.items[torch.from_numpy(idx).to(dev)].long()
        tcnt = test.ptr_host[ub + 1] - test.ptr_host[ub]
        tidx = np.concatenate([np.arange(test.ptr_host[u], test.ptr_host[u + 1]) for u in ub])
        trows = torch.from_numpy(np.repeat(np.arange(ub.size), tcnt)).to(dev)
        tcols = test.items[torch.from_numpy(tidx).to(dev)].long()
        batches.append((torch.from_numpy(ub).to(dev), rows, cols, trows, tcols))
    setup_s = time.time() - t0

    one, t_rank = timed(lambda: m.rank(users_t, n, test, exclude=train), args.reps)
    met, t_met = timed(lambda: rank_metrics(m, train, test, k_list=K_LIST), args.reps)
    (ev, top), t_ev = timed(lambda: evaluate(m, train, test, k_list=K_LIST), args.reps)

    def torch_ranks():
        out = []
        for ub, rows, cols, trows, tcols in batches:
            sc = table[ub] @ item_rows.T
            sc[rows, cols] = -float("inf")
            ts, excluded = sc[trows, tcols], torch.isinf(sc[trows, tcols])
            r = torch.empty(trows.numel(), dtype=torch.int64, device=dev)
            for c in range(0, trows.numel(), 2048):  # bounded [targets x items] comparison blocks
                s_ = sc[trows[c : c + 2048]]
                t_ = ts[c : c + 2048, None]
                beat = (s_ > t_) | ((s_ == t_) & (pos[None, :] < tcols[c : c + 2048, None]))
                r[c : c + 2048] = (beat & ~torch.isinf(s_)).sum(1)
            out.append(torch.where(excluded, -1, r))
        return torch.cat(out)

    th_rank, t_torch = timed(torch_ranks, args.reps)
    # exactness: hit counts and metrics against evaluate
    hits = test.contains(torch.from_numpy(users).to(dev)[:, None].expand_as(top), top)
    b = torch.repeat_interleave(torch.arange(U, device=dev), one.ptr.diff())
    hit_equal = all(bool(torch.equal(torch.zeros(U, dtype=torch.int64, device=dev).index_add_(0, b, ((one.rank >= 0) & (one.rank < k)).long()),
                                     hits[:, :k].sum(1))) for k in K_LIST)
    max_rel = max(abs(met[k][x] - ev[k][x]) / max(abs(ev[k][x]), 1e-30) for k in K_LIST for x in ("precision", "recall", "ndcg"))
    r = {"shape": shape, "users": int(U), "candidates": n, "targets": int(one.items.numel()), "width": width, "setup_s": setup_s,
         "rank_one_call": stats(t_rank, U, n, width, peak),
         "rank_metrics_one_call": stats(t_met, U, n, width, peak),
         "evaluate_256_loop": stats(t_ev, U, n, width, peak),
         "torch_cublas_mask_count_256_loop": stats(t_torch, U, n, width, peak),
         "speedup_rank_metrics_vs_evaluate": float(np.median(t_ev) / np.median(t_met)),
         "speedup_rank_metrics_vs_torch": float(np.median(t_torch) / np.median(t_met)),
         "hit_counts_equal_evaluate": hit_equal, "max_rel_diff_vs_evaluate": max_rel,
         "rank_agreement_with_torch": float((th_rank == one.rank).float().mean()),
         "metrics": {str(k): v for k, v in met.items()}}
    print(json.dumps(r), flush=True)
    results["runs"].append(r)
    assert hit_equal and max_rel <= 1e-6, r
    del m, tables, table, item_rows, batches, one, met, top, th_rank, train, test
    torch.cuda.empty_cache()

if args.out:
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(results, indent=1) + "\n")
