#!/usr/bin/env python
"""Knowledge-graph completion (``KGAT.complete`` / ``KGAT.kg_rank`` / ``metrics.link_metrics``) against a torch baseline, and the
first quality number of the trained TransR half.

Workloads (d = k = 64):
  (a) codeforces-full (211,983 nodes, 10 relations): rating prediction for every problem without a rating edge (top-5 of the
      28 ratings) and tag completion for every problem (top-5 of the 37 tags), CKG triples filtered;
  (b) amazon-book (159,251 nodes, 80 relations): filtered ranks of 10,000 sampled CKG triples against all nodes
      (``link_metrics(candidates="all")``, one ``kg_rank`` call per relation);
  (c) codeforces-sm: 10 % of the rating edges held out (``build_ckg`` on the remaining triples), a few epochs with the training
      engine, then filtered MRR / Hits@1/3/10 of the held-out ratings among the 28 ratings, next to a random ranking's.
(a) and (b) time random-initialised parameters: the kernels' work does not depend on the values.  The torch baseline per
relation: cuBLAS candidate projections E @ W_r, then per query chunk the energies |q|^2 + |P|^2 - 2 q P^T (cuBLAS), +inf on
known triples, and topk (complete) or a count of better keys (rank); it sums in another order, so it is reported as the
fraction of results it gets exactly.

Every time is the median of --reps warmed calls (CUDA events around the call, result read back).  FLOPs counted from shapes:
projection 2 n_cand d k per relation, scoring 3 k per (query, candidate) pair (subtract, fma, tree add).  The card's name and
power limit are read in the same run.

    python tools/prof_complete.py [--out profiles/complete_b200.json]
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

from kgat_b200 import synthetic  # noqa: E402
from kgat_b200.ckg import build_ckg, interaction_dict  # noqa: E402
from kgat_b200.engine import TrainEngine  # noqa: E402
from kgat_b200.metrics import TripleSet, link_metrics  # noqa: E402
from kgat_b200.trainer import EpochData, build_model  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--epochs", type=int, default=4)
ap.add_argument("--workloads", default="a,b,c")
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


def timed(fn, reps: int):
    for _ in range(2):
        out = fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return float(np.median(ms)), out


def relation_between(g, head_lo, head_hi, tails):
    """The CKG relation id whose edges go from nodes [head_lo, head_hi) to exactly the node set ``tails``."""
    for r in np.unique(g.relations):
        sel = g.relations == r
        if g.heads[sel].min() >= head_lo and g.heads[sel].max() < head_hi and np.array_equal(np.unique(g.tails[sel]), np.sort(tails)):
            return int(r)
    raise RuntimeError("relation not found")


def torch_complete(emb, rel, w, heads, rels, cand, k, known, chunk=256):
    """Baseline: per relation cuBLAS projections, chunked energies, +inf on known triples, topk."""
    N, R = emb.shape[0], rel.shape[0]
    out_t = torch.empty(heads.numel(), k, dtype=torch.int64, device=emb.device)
    out_e = torch.empty(heads.numel(), k, device=emb.device)
    for r in torch.unique(rels).tolist():
        idx = torch.nonzero(rels == r).flatten()
        P = emb[cand] @ w[r]
        p2 = (P * P).sum(1)
        for s in range(0, idx.numel(), chunk):
            qi = idx[s : s + chunk]
            q = emb[heads[qi]] @ w[r] + rel[r]
            E = (q * q).sum(1, keepdim=True) + p2[None, :] - 2.0 * (q @ P.T)
            key = (heads[qi, None] * R + r) * N + cand[None, :]
            pos = torch.searchsorted(known, key).clamp(max=known.numel() - 1)
            E.masked_fill_(known[pos] == key, float("inf"))
            v, j = torch.topk(E, k, dim=1, largest=False)
            out_t[qi], out_e[qi] = cand[j], v
    return out_t, out_e


def torch_rank(emb, rel, w, heads, rels, tails, known, chunk=128):
    """Baseline: ranks against all nodes -- per relation projections, chunked energies, known triples other than the target
    masked, count of better (energy, position) keys."""
    N, R = emb.shape[0], rel.shape[0]
    rank = torch.empty(heads.numel(), dtype=torch.int64, device=emb.device)
    ar = torch.arange(N, device=emb.device)
    for r in torch.unique(rels).tolist():
        idx = torch.nonzero(rels == r).flatten()
        P = emb @ w[r]
        p2 = (P * P).sum(1)
        for s in range(0, idx.numel(), chunk):
            qi = idx[s : s + chunk]
            q = emb[heads[qi]] @ w[r] + rel[r]
            E = (q * q).sum(1, keepdim=True) + p2[None, :] - 2.0 * (q @ P.T)
            key = (heads[qi, None] * R + r) * N + ar[None, :]
            pos = torch.searchsorted(known, key).clamp(max=known.numel() - 1)
            E.masked_fill_((known[pos] == key) & (ar[None, :] != tails[qi, None]), float("inf"))
            et = E.gather(1, tails[qi, None])
            rank[qi] = ((E < et) | ((E == et) & (ar[None, :] < tails[qi, None]))).sum(1)
    return rank


def flops(n_rel_used, n_cand, n_pairs, d, k):
    return 2.0 * n_rel_used * n_cand * d * k + 3.0 * n_pairs * k


def workload_a():
    shape = synthetic.SHAPES["codeforces-full"]
    rng = np.random.default_rng(synthetic.SEED)
    triples = synthetic._codeforces_triples(rng, shape)
    users = np.arange(shape.user_num)
    g = build_ckg(shape.user_num, shape.entity_num, shape.item_num, shape.kg_relation_num, np.stack([users, users % shape.item_num], 1), triples)
    m = build_model(g, "cuda").eval()
    U, P = g.user_num, shape.item_num
    g0 = shape.entity_num - 28
    t0 = g0 - 37
    r_rating = relation_between(g, U, U + P, U + g0 + np.arange(28))
    r_tag = relation_between(g, U, U + P, np.unique(g.tails[(g.tails >= U + t0) & (g.tails < U + g0)]))
    known = TripleSet.from_ckg(g)
    rated = np.unique(g.heads[g.relations == r_rating])
    unrated = torch.from_numpy(np.setdiff1d(np.arange(U, U + P), rated))
    problems = torch.arange(U, U + P)
    ratings = torch.arange(U + g0, U + g0 + 28)
    tags = torch.arange(U + t0, U + g0)
    emb, rel, w = m._transr_params()
    res = {"nodes": g.node_num, "relations": g.relation_num, "unrated_problems": int(unrated.numel()), "problems": P}
    for name, heads, r, cand in (("rating_unrated", unrated, r_rating, ratings), ("tags_all", problems, r_tag, tags)):
        rels = torch.full_like(heads, r)

        def kern():
            out = m.complete(heads, rels, cand, k=5, exclude=known)
            return out.tails.cpu(), out.energy.cpu()

        hc, rc, cc = heads.cuda(), rels.cuda(), cand.cuda()

        def base():
            t, e = torch_complete(emb, rel, w, hc, rc, cc, 5, known.keys)
            return t.cpu(), e.cpu()

        t_k, (tk, ek) = timed(kern, args.reps)
        t_b, (tb, _) = timed(base, args.reps)
        res[name] = {"queries": int(heads.numel()), "candidates": int(cand.numel()), "k": 5, "complete_ms": t_k, "torch_ms": t_b,
                     "torch_rows_equal": float((tk == tb).all(1).float().mean()),
                     "gflop": flops(1, cand.numel(), heads.numel() * cand.numel(), 64, 64) / 1e9}
        print(json.dumps({name: res[name]}), flush=True)
    return res


def workload_b():
    g = synthetic.make_ckg("amazon-book", with_dicts=False)
    m = build_model(g, "cuda").eval()
    known = TripleSet.from_ckg(g)
    rng = np.random.default_rng(0)
    sel = rng.choice(g.nnz, 10_000, replace=False)
    h, r, t = (torch.from_numpy(np.asarray(x[sel]).astype(np.int64)).cuda() for x in (g.heads, g.relations, g.tails))
    n_rel_used = int(torch.unique(r).numel())

    def kern():
        return link_metrics(m, (h, r, t), known, candidates="all")

    emb, rel, w = m._transr_params()

    def base():
        return torch_rank(emb, rel, w, h, r, t, known.keys).cpu()

    t_k, met = timed(kern, args.reps)
    t_b, rb = timed(base, max(1, args.reps // 2))
    rk = torch.cat([m.kg_rank(h[r == x], r[r == x], t[r == x], g.node_num, exclude=known).rank.cpu() for x in torch.unique(r).tolist()])
    order = torch.cat([torch.nonzero(r == x).flatten().cpu() for x in torch.unique(r).tolist()])
    rb_sorted = rb[order]
    f = flops(n_rel_used, g.node_num, 10_000 * g.node_num, 64, 64)
    res = {"nodes": g.node_num, "relations": g.relation_num, "relations_queried": n_rel_used, "triples": 10_000, "link_metrics_ms": t_k,
           "torch_ms": t_b, "torch_ranks_equal": float((rk == rb_sorted).float().mean()), "gflop": f / 1e9,
           "link_metrics_gflops": f / (t_k * 1e6), "mrr_untrained": met["mrr"]}
    print(json.dumps({"amazon_book": res}), flush=True)
    return res


def workload_c():
    shape = synthetic.SHAPES["codeforces-sm"]
    rng = np.random.default_rng(synthetic.SEED)
    pairs = synthetic._interactions(rng, shape, 1.3, 50.0)
    triples = synthetic._codeforces_triples(rng, shape)
    train, _, _ = synthetic.split_interactions(rng, pairs, shape.user_num)
    hold_rng = np.random.default_rng(1)
    rated = np.nonzero(triples[:, 1] == 1)[0]
    held = hold_rng.choice(rated, rated.size // 10, replace=False)
    keep = np.ones(triples.shape[0], bool)
    keep[held] = False
    g = build_ckg(shape.user_num, shape.entity_num, shape.item_num, shape.kg_relation_num, train, triples[keep])
    g.train_interactions, g.train_dict = train, interaction_dict(train, shape.user_num)  # what the epoch sampler draws from
    U, P = g.user_num, shape.item_num
    g0 = shape.entity_num - 28
    r_rating = relation_between(g, U, U + P, U + g0 + np.arange(28))
    h = torch.from_numpy(U + triples[held, 0])
    t = torch.from_numpy(U + triples[held, 2])
    r = torch.full_like(h, r_rating)
    known = TripleSet.from_ckg(g)
    ratings = torch.arange(U + g0, U + g0 + 28)
    m = build_model(g, "cuda")
    eng = TrainEngine(m)
    out = {"held_out": int(held.size), "epochs": args.epochs, "by_epoch": []}
    n = 28
    out["random"] = {"mrr": float(np.mean(1.0 / np.arange(1, n + 1))), "hits": {k: k / n for k in (1, 3, 10)}}
    for e in range(args.epochs + 1):
        if e > 0:
            eng.run_epoch(EpochData.sample(g, seed=e))
        met = link_metrics(m, (h, r, t), known, candidates=ratings)
        out["by_epoch"].append({"epoch": e, "mrr": met["mrr"], "mean_rank": met["mean_rank"], "hits": met["hits"], "n_ranked": met["n_ranked"]})
        print(json.dumps(out["by_epoch"][-1]), flush=True)
    return out


results = {"card": card(), "note": "B200; times are medians of warmed calls with the result read back"}
WORKLOADS = {"a": ("codeforces_full", workload_a), "b": ("amazon_book", workload_b), "c": ("codeforces_sm_quality", workload_c)}
for wl in args.workloads.split(","):
    name, fn = WORKLOADS[wl]
    results[name] = fn()
print(json.dumps(results["card"]))
if args.out:
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(results, indent=1) + "\n")
