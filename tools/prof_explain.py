#!/usr/bin/env python
"""Path explanations at an evaluation batch: 256 users with test items x their top-20 recommendations (train positives
masked) = 5,120 (user, problem) pairs, H = 3 hops, k = 10 paths, after one eval-mode attention refresh, so that A holds
real attention values.  Times ``ops.explain_paths`` (the two kernels plus the id conversion and the range-check read-back,
CUDA events, warmed, median of --reps) and the torch reference ``oracle/explain_ref.py`` on the same GPU, asserts that the
two agree, and writes one JSON object per shape.

    python tools/prof_explain.py [--shapes amazon-book codeforces-full] [--out profiles/explain_b200.json]
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
from kgat_b200.model import KGATMode  # noqa: E402
from kgat_b200.trainer import build_model  # noqa: E402
from oracle.explain_ref import explain_paths_ref  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--shapes", nargs="+", default=["amazon-book", "codeforces-full"])
ap.add_argument("--users", type=int, default=256)
ap.add_argument("--topn", type=int, default=20)
ap.add_argument("--k", type=int, default=10)
ap.add_argument("--hops", type=int, default=3)
ap.add_argument("--reps", type=int, default=20)
ap.add_argument("--ref-reps", type=int, default=3)
ap.add_argument("--out", default=None)
args = ap.parse_args()


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 and q.stdout.strip() else ""
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": line}


def timed(fn, reps: int):
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return out, ts


def probes(graph, src: np.ndarray, dst: np.ndarray, H: int) -> int:
    """Binary-search probes of the kernel's enumeration: min(deg s, |In t|) + sum over a in row s of min(deg a, |In t|)."""
    rp = graph.row_ptr.cpu().numpy().astype(np.int64)
    tp = graph.t_ptr.cpu().numpy().astype(np.int64)
    col = graph.col_idx.cpu().numpy()
    deg, tdeg = np.diff(rp), np.diff(tp)
    total = len(src)
    for s, t in zip(src, dst):
        if s == t:
            continue
        if H >= 2:
            total += min(deg[s], tdeg[t])
        if H >= 3:
            a = col[rp[s] : rp[s + 1]]
            a = a[(a != s) & (a != t)]
            total += int(np.minimum(deg[a], tdeg[t]).sum())
    return int(total)


results = []
for shape in args.shapes:
    t0 = time.time()
    g = synthetic.make_ckg(shape, with_dicts=True)
    model = build_model(g, "cuda").eval()
    dev = torch.device("cuda")
    edges = (torch.from_numpy(np.asarray(g.heads)).to(dev), torch.from_numpy(np.asarray(g.relations)).to(dev),
             torch.from_numpy(np.asarray(g.tails)).to(dev), torch.from_numpy(np.asarray(g.adjacency_relations, np.int64)).to(dev))
    model(*edges, mode=KGATMode.UPDATE_ATTENTION)
    users = np.array(sorted(u for u, items in g.test_dict.items() if len(items) > 0))
    users = np.random.default_rng(0).choice(users, args.users, replace=False)
    users.sort()
    train = [np.asarray(sorted(g.train_dict.get(int(u), [])), np.int32) for u in users]
    mask_ptr = torch.from_numpy(np.concatenate([[0], np.cumsum([len(x) for x in train])]).astype(np.int32)).to(dev)
    mask_items = torch.from_numpy(np.concatenate(train).astype(np.int32)).to(dev)
    top = model.recommend_topk(torch.from_numpy(users).to(dev), torch.arange(g.item_num, device=dev), args.topn, mask_ptr, mask_items)
    src = torch.from_numpy(users).to(dev).repeat_interleave(args.topn)
    dst = top.flatten().to(torch.int64) + g.user_num
    graph = model._graph()
    setup_s = time.time() - t0

    run = lambda: ops.explain_paths(graph, src, dst, args.k, args.hops)  # noqa: E731
    for _ in range(3):
        run()
    got, ts = timed(run, args.reps)
    again = run()
    repeatable = all(torch.equal(a, b) for a, b in zip(got, again))

    ref, ref_ts = timed(lambda: explain_paths_ref(graph.row_ptr, graph.col_idx, graph.vals, src, dst, args.k, args.hops), 1)
    if ref_ts[0] < 60e3:
        _, more = timed(lambda: explain_paths_ref(graph.row_ptr, graph.col_idx, graph.vals, src, dst, args.k, args.hops), args.ref_reps - 1)
        ref_ts += more
    exact = {n: bool(torch.equal(a, b)) for n, a, b in zip(("nodes", "slots", "hops", "weight", "count"), got[:5], ref[:5])}
    mass_rel = float(((got[5].double() - ref[5]).abs() / ref[5].abs().clamp_min(1e-30)).max())
    n_probes = probes(graph, src.cpu().numpy(), dst.cpu().numpy(), args.hops)
    med, ref_med = float(np.median(ts)), float(np.median(ref_ts))
    r = {
        "shape": shape,
        "card": card(),
        "nodes": graph.n,
        "nnz": graph.nnz,
        "pairs": int(src.numel()),
        "k": args.k,
        "max_hops": args.hops,
        "probes": n_probes,
        "paths_per_length": ref[4].sum(0).tolist(),
        "kernel_ms_median": med,
        "kernel_ms_min": float(min(ts)),
        "kernel_ms_max": float(max(ts)),
        "kernel_reps": len(ts),
        "pairs_per_s": src.numel() / (med * 1e-3),
        "probes_per_s": n_probes / (med * 1e-3),
        "torch_reference_ms": ref_ts,
        "torch_reference_ms_median": ref_med,
        "speedup_vs_torch_reference": ref_med / med,
        "exact": exact,
        "mass_max_rel_err": mass_rel,
        "repeatable": repeatable,
        "setup_s": setup_s,
    }
    print(json.dumps(r), flush=True)
    assert all(exact.values()) and mass_rel <= 1e-5 and repeatable, r
    results.append(r)
    del model, graph, got, ref
    torch.cuda.empty_cache()

if args.out:
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(results, indent=1) + "\n")
