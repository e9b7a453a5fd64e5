#!/usr/bin/env python
"""Benchmark of the KGAT hot path on the Amazon-book-shaped synthetic CKG (BASELINE.json configs[2]).

    python bench.py --gpus N --steps K --warmup W             # our arm (CUDA kernels)
    python bench.py --impl reference --steps K --warmup W     # reference arm: CPU oracle port
    python bench.py --steps K --warmup W --dump-outputs DIR   # + what the last timed epoch computed, as DIR/<name>.npy

Metric (BASELINE.json): **KGAT epoch seconds** -- one "step" is one reference epoch body
(main.py:290-361: n_cf CF steps + n_kg KG steps + one attention refresh) over pre-sampled synthetic
batches; ``value`` is measured with the batches resident in HBM, ``e2e`` through the same public
model API with the batches in pinned host memory, a host->device copy of every step's ids and a
device->host read of every step's loss inside the timed region.  Extra keys report propagation
edges/s, the per-kernel time split, the roofline of the dominant kernel (live CUDA-event timing) and
the CPU baseline (the oracle port of the reference's PyTorch-CPU path, timed on this box's cores on a
bounded sample and extrapolated to one epoch).
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "kgat_epoch_seconds"
UNIT = "s"
WORKLOAD = "amazon-book"


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


# ----------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int = 0):
        self.rows: list[list[str]] = []
        self.proc = None
        self.index = index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
            )
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) >= 6:
                self.rows.append(parts)

    def __exit__(self, *exc):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self) -> dict:
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


# ----------------------------------------------------------------------------------------------
# reference arm / baselines: the UNMODIFIED reference KGAT (oracle/_ref, staged by oracle/build_ref.py) through its own
# public API, on the host cores or -- the same-box incumbent -- on the B200 with stock ATen kernels.  The oracle port
# (oracle/kgat_oracle.py) is the fallback when the staged reference is missing.
# ----------------------------------------------------------------------------------------------
def _att_coo(g):
    n = g.node_num
    return torch.sparse_coo_tensor(torch.from_numpy(np.vstack([g.att_rows, g.att_cols])).long(), torch.from_numpy(g.att_vals), size=(n, n))


def reference_model(g, params, device):
    """The staged, unmodified reference ``KGAT`` with our initial parameters; None when oracle/_ref is absent."""
    from oracle import build_ref

    mods = build_ref.load()
    if mods is None:
        print("bench.py: oracle/_ref is not staged (build() with KGAT_REFERENCE set stages it): the baselines run the oracle port",
              file=sys.stderr)
        return None
    ref, _ = mods
    m = ref.KGAT(ref.KGATArgs(user_num=g.user_num, entity_num=g.entity_num, relation_num=g.relation_num, attentive_matrix=_att_coo(g)))
    m.load_state_dict(params, strict=False)
    m = m.to(device)
    m.build_optimizer(cf_lr=1e-3, kg_lr=1e-4)  # two torch.optim.Adam over all parameters (model.py:393-405)
    m.train()
    return m, ref.KGATMode


class ReferenceRunner:
    """Bounded samples of the reference epoch body (main.py:290-361) through the reference model's own API."""

    def __init__(self, g, params, data, device="cpu", refresh_relations: int = 2):
        self.g, self.data, self.device = g, data, torch.device(device)
        if self.device.type == "cpu":
            torch.set_num_threads(os.cpu_count() or 1)
        built = reference_model(g, params, self.device)
        self.kind = "reference" if built is not None else "port"
        self.cf_i = self.kg_i = 0
        self.warm = False
        rels = np.asarray(g.adjacency_relations[:refresh_relations])
        sel = np.isin(g.relations, rels)
        self.share = float(sel.sum()) / max(g.nnz, 1)
        if built is not None:
            self.model, self.Mode = built
            # main.py:351-353 hands over the whole edge list; relation_indices selects the relations to score
            self.edges = (torch.from_numpy(g.heads.astype(np.int64)).to(self.device), torch.from_numpy(g.relations.astype(np.int64)).to(self.device),
                          torch.from_numpy(g.tails.astype(np.int64)).to(self.device), torch.from_numpy(rels.astype(np.int64)).to(self.device))
        else:
            from oracle import kgat_oracle as O

            self.O = O
            self.att = _att_coo(g).to(self.device)
            self.p = {k: v.detach().clone().to(self.device).requires_grad_(True) for k, v in params.items()}
            self.opt = {"cf": torch.optim.Adam(list(self.p.values()), lr=1e-3), "kg": torch.optim.Adam(list(self.p.values()), lr=1e-4)}
            self.sel, self.rels = sel, rels

    def _sync(self):
        if self.device.type == "cuda":
            torch.cuda.synchronize(self.device)

    def _step(self, kind):
        d = self.data
        if kind == "cf":
            b = [torch.from_numpy(a[self.cf_i % d.n_cf]).to(self.device) for a in d.cf]
            self.cf_i += 1
        else:
            b = [torch.from_numpy(a[self.kg_i % d.n_kg]).to(self.device) for a in d.kg]
            self.kg_i += 1
        self._sync()
        t0 = time.perf_counter()
        if self.kind == "reference":
            m = self.model
            loss = m(*b, mode=self.Mode.TRAIN_CF if kind == "cf" else self.Mode.TRAIN_KG)
            loss.backward()
            (m.update_cf_weights if kind == "cf" else m.update_kg_weights)()
            loss.item()  # main.py:314 / 343 read the loss every step
        else:
            loss = self.O.cf_loss(self.p, self.att, *b) if kind == "cf" else self.O.kg_loss(self.p, *b)
            loss.backward()
            self.opt[kind].step()
            self.opt[kind].zero_grad()
            float(loss)
        self._sync()
        return time.perf_counter() - t0

    def _refresh(self):
        self._sync()
        t0 = time.perf_counter()
        if self.kind == "reference":
            m = self.model
            keep = m.attentive_matrix.data
            m(*self.edges, mode=self.Mode.UPDATE_ATTENTION)  # train() mode, no no_grad: as main.py:350-361
            m.attentive_matrix.data = keep  # the sample scored a subset of the relations: keep the full matrix for the CF steps
        else:
            g, O = self.g, self.O
            with torch.no_grad():
                q = {k: v.detach() for k, v in self.p.items()}
                heads = torch.from_numpy(g.heads[self.sel].astype(np.int64)).to(self.device)
                tails = torch.from_numpy(g.tails[self.sel].astype(np.int64)).to(self.device)
                rel_of = torch.from_numpy(g.relations[self.sel].astype(np.int64)).to(self.device)
                rows, cols, vals = [], [], []
                for r in self.rels.tolist():
                    idx = torch.where(rel_of == r)[0]
                    rows.append(heads[idx])
                    cols.append(tails[idx])
                    vals.append(O.attention_by_relation(q, heads[idx], tails[idx], r, g.node_num))
                mtx = torch.sparse_coo_tensor(torch.stack([torch.cat(rows), torch.cat(cols)]), torch.cat(vals), size=(g.node_num, g.node_num))
                torch.sparse.softmax(mtx.cpu(), dim=1).to(self.device)
        self._sync()
        return (time.perf_counter() - t0) / max(self.share, 1e-9)

    def sample(self, n_cf: int = 3, n_kg: int = 3):
        """One bounded sample: (one warm-up CF + KG step the first time,) n_cf CF steps, n_kg KG steps, the refresh of a
        relation subset -- extrapolated to one epoch with the reference's own batch counts."""
        if not self.warm:
            self._step("cf")
            self._step("kg")
            self.warm = True
        t_cf = float(np.mean([self._step("cf") for _ in range(n_cf)]))
        t_kg = float(np.mean([self._step("kg") for _ in range(n_kg)]))
        t_ref = self._refresh()
        d = self.data
        return {"epoch_s_extrapolated": d.n_cf * t_cf + d.n_kg * t_kg + t_ref, "cf_step_s": t_cf, "kg_step_s": t_kg, "refresh_s_extrapolated": t_ref,
                "cores": (os.cpu_count() or 1) if self.device.type == "cpu" else 0, "kind": self.kind,
                "sample": f"{n_cf} CF + {n_kg} KG steps (after one warm-up step each) + attention refresh of {self.share:.1%} of the edges, "
                          f"extrapolated x({d.n_cf}, {d.n_kg}, 1/share)"}


def make_workload(workload: str, seed: int = 2024):
    from kgat_b200 import synthetic
    from kgat_b200.trainer import EpochData

    g = synthetic.make_ckg(workload, seed=seed, with_dicts=False)
    data = EpochData.sample(g, seed=seed)
    return g, data


def init_params(g, seed: int = 2024):
    """Reference-initialised parameters (KGAT module constructed on the CPU under the seed)."""
    from kgat_b200.model import KGAT, KGATArgs

    torch.manual_seed(seed)
    m = KGAT(KGATArgs(user_num=g.user_num, entity_num=g.entity_num, relation_num=g.relation_num))
    return {k: v.detach().clone() for k, v in m.state_dict().items() if not v.is_sparse}


def config_dict(g, data, n_gpus):
    return {
        "workload": f"synthetic {WORKLOAD}-shaped CKG (configs[2]): users={g.user_num} items={g.item_num} entities={g.entity_num} "
                    f"relations={g.relation_num} nodes={g.node_num} nnz={g.nnz}; 3 layers 64->64->32->16, d=64, fp32",
        "epoch": f"{data.n_cf} CF steps (B=256) + {data.n_kg} KG steps (B=512) + 1 attention refresh",
        "batches": "one epoch of batches is sampled up front (seed 2024) and replayed by every bench step (step s uses batch s mod n), so "
                   "the losses keep falling across bench steps; timing does not depend on it",
        "l2_policy": "inputs larger than L2: the epoch streams >1 TB through 126 MB of L2; every step rewrites the 41 MB table, its Adam moments and ~0.3 GB of activations",
        "cf_pruning": "each CF step computes layer l only for the rows the batch can reach (exact; frontier.py): same loss and gradients as "
                      "the reference's full-graph propagation per batch",
        "parallelism": f"row-sharded x{n_gpus}" if n_gpus > 1 else "single GPU",
    }


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    g, data = make_workload(WORKLOAD)
    runner = ReferenceRunner(g, init_params(g), data, "cpu")
    vals, last = [], None
    for i in range(args.warmup + args.steps):
        last = runner.sample()
        if i >= args.warmup:
            vals.append(last["epoch_s_extrapolated"])
    v = float(np.mean(vals)) if vals else last["epoch_s_extrapolated"]
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": v * 1e3, "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(g, data, 1),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": last["cores"], "kind": last["kind"], "sample": last["sample"]},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "detail": {k: last[k] for k in ("cf_step_s", "kg_step_s", "refresh_s_extrapolated")},
        "note": "the unmodified reference KGAT (oracle/_ref: src/model/KGAT/{model,aggregator,multi_head_attention}.py) driven through its own "
                "API with torch.optim.Adam on the host cores" if last["kind"] == "reference" else "oracle port (oracle/_ref not staged)",
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------
def frontier_stats(engine, graph):
    """Rows and edges per frontier level of the engine's last CF step (host side, from the device row lists)."""
    f = getattr(engine, "frontier", None)
    if f is None:
        return None
    deg = (graph.row_ptr[1:] - graph.row_ptr[:-1]).to(torch.int64)
    deg_t = (graph.t_ptr[1:] - graph.t_ptr[:-1]).to(torch.int64)
    out = {}
    counts = f.counts.cpu().tolist()
    for level in range(1, f.n_layers + 1):
        rows = f.rows(level)[: counts[level - 1]].long()
        out[f"L{level}"] = {"rows": counts[level - 1], "edges": int(deg[rows].sum()), "edges_t": int(deg_t[rows].sum())}
    return out


def algorithmic_bytes(name: str, g, graph, fr) -> float | None:
    """Compulsory-traffic model B_min of SURVEY.md section 8d per launch of the named kernel (every distinct byte once),
    restricted to the rows / edges the pruned step touches (``fr``: frontier_stats)."""
    n, nnz = g.node_num, graph.nnz
    m = __import__("re").match(r"(spmmT?)_d(\d+)(?:_(rows|edges|scatter|pruned))?(?:_L(\d+))?$", name)
    if m:
        kind, d, var, lvl = m.group(1), int(m.group(2)), m.group(3), int(m.group(4)) if m.group(4) else None
        t = kind == "spmmT"
        if var is None or fr is None or lvl is None:
            plan = graph.t_plan if t else graph.plan
            return 8.0 * nnz + 16.0 * plan.n_tasks + 4.0 * n * d * (3 if t else 2)
        cur = fr[f"L{lvl}"]
        if not t:  # forward rows of level l: their edges, the distinct source rows (level l-1, or all of E0), the outputs
            src_rows = fr[f"L{lvl - 1}"]["rows"] if lvl > 1 else n
            return 8.0 * cur["edges"] + 16.0 * cur["rows"] + 4.0 * d * (min(src_rows, cur["edges"]) + cur["rows"])
        if var == "scatter":  # edges of the source rows (level l), their g rows, zero + reduce into level l-1 rows
            dst = fr[f"L{lvl - 1}"]["rows"]
            return 8.0 * cur["edges"] + 16.0 * cur["rows"] + 4.0 * d * (2 * cur["rows"] + 2 * dst)
        dst_rows, dst_edges = (fr[f"L{lvl - 1}"]["rows"], fr[f"L{lvl - 1}"]["edges_t"]) if lvl > 1 else (n, nnz)
        return 8.0 * dst_edges + 16.0 * dst_rows + 4.0 * d * (2 * cur["rows"] + dst_rows)  # gather: all edges of the dst rows are streamed
    m = __import__("re").match(r"biagg_(fwd|bwd)_(\d+)x(\d+)(?:_rows)?(?:_L(\d+))?$", name)
    if m:
        di, do = int(m.group(2)), int(m.group(3))
        rows = fr[f"L{int(m.group(4))}"]["rows"] if (fr is not None and m.group(4)) else n
        if m.group(1) == "fwd":
            return rows * (4.0 * (2 * di + do) + 4 + do)
        return rows * (4.0 * (2 * do + 2 * di + 2 * di) + 4 + do)
    return None


def gathered_bytes(name: str, g, graph, fr) -> float | None:
    """Bytes the gather moves from L2 to the SMs: one d-wide row per live edge (the L2-resident regime's real traffic)."""
    m = __import__("re").match(r"(spmmT?)_d(\d+)(?:_(rows|edges|scatter|pruned))?(?:_L(\d+))?$", name)
    if not m:
        return None
    d, var, lvl = int(m.group(2)), m.group(3), int(m.group(4)) if m.group(4) else None
    if var is None or fr is None or lvl is None:
        return 4.0 * d * graph.nnz
    key = "edges" if (m.group(1) == "spmm" or var == "scatter") else "edges_t"
    # transposed gather over the level below: live edges = edges out of this level's rows (A is structurally symmetric)
    return 4.0 * d * fr[f"L{lvl}"]["edges" if key == "edges" else "edges"]


def l2_gather_peak():
    """Measured L2 -> SM random row-gather peak of this GPU (tools/microbench/l2_gather, ~2 s); None if the binary is absent."""
    exe = ROOT / "tools" / "microbench" / "l2_gather"
    if not exe.exists():
        return None
    try:
        out = subprocess.run([str(exe), "--json"], capture_output=True, text=True, timeout=120, check=True).stdout.strip().splitlines()[-1]
        return json.loads(out)
    except Exception as e:  # noqa: BLE001
        return {"unavailable": f"{type(e).__name__}: {e}"[:200]}


def time_cuda(fn, reps: int, warm: int = 2) -> float:
    for _ in range(warm):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3 / reps


def extra_shape_block(shape: str, dev, n_cf: int = 20, n_kg: int = 100, topk_users: bool = False):
    """A secondary BASELINE.json configuration on this GPU: measured CF / KG step and refresh through the CUDA-graph engine,
    extrapolated to that shape's epoch with the reference's batch counts; optionally the full-graph top-20 for all users."""
    from kgat_b200 import synthetic
    from kgat_b200.engine import TrainEngine
    from kgat_b200.trainer import EpochData, build_model

    t0 = time.perf_counter()
    g = synthetic.make_ckg(shape, with_dicts=topk_users)
    data = EpochData.sample(g, n_cf=n_cf, n_kg=n_kg)
    model = build_model(g, dev)
    eng = TrainEngine(model)
    eng.bind_resident(data.tensors())
    eng.run_epoch(n_cf=2, n_kg=2)  # captures the graphs, first refresh
    eng.run_epoch(n_cf=n_cf, n_kg=n_kg)
    ph = dict(eng.last_phase_ms)
    from kgat_b200.sampler import BatchSampler

    s = BatchSampler(g)
    e_cf, e_kg = s.cf_batches_per_epoch(256), s.kg_batches_per_epoch(512)
    cf_us, kg_us = 1e3 * ph["cf"] / n_cf, 1e3 * ph["kg"] / n_kg
    out = {"shape": shape, "nodes": g.node_num, "nnz": g.nnz, "cf_step_us": cf_us, "kg_step_us": kg_us, "refresh_ms": ph["refresh"],
           "epoch_steps": [e_cf, e_kg], "epoch_s_extrapolated": (e_cf * cf_us + e_kg * kg_us) / 1e6 + ph["refresh"] / 1e3,
           "frontier": frontier_stats(eng, model._graph()), "setup_s": None,
           "measured": f"{n_cf} CF + {n_kg} KG graph-replayed steps and one refresh; epoch = steps x the reference's batch counts (main.py:297, 324)"}
    if topk_users:
        from kgat_b200.metrics import InteractionCSR, evaluate

        model.eval()
        train = InteractionCSR(g.train_dict, g.user_num, g.item_num, dev)
        test = InteractionCSR(g.test_dict, g.user_num, g.item_num, dev)
        users = np.arange(g.user_num)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        res, _ = evaluate(model, train, test, k_list=(20,), batch_size=256, users=users)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t1
        out["full_graph_top20"] = {"users": int(g.user_num), "items": int(g.item_num), "seconds": dt, "users_per_s": g.user_num / dt,
                                   "recall@20": float(res[20]["recall"]), "ndcg@20": float(res[20]["ndcg"]), "precision@20": float(res[20]["precision"]),
                                   "what": "one propagation (cached across batches) + per 256 users: score GEMM, train-positive mask, exact top-20, metrics"}
    out["setup_s"] = time.perf_counter() - t0
    del eng, model
    torch.cuda.empty_cache()
    return out


def c5_scaled_block(dev, peak):
    """configs[4] scaled 5x down (2.2 M nodes, 40 M edges, d = 128, layers 128-64-32-16): one full propagation step, forward +
    backward, where the 1.1 GB table no longer fits the L2 and HBM is the bound."""
    from kgat_b200 import synthetic
    from kgat_b200.functions import DropoutSpec, propagate_backward, propagate_forward
    from kgat_b200.graph import AttentiveGraph

    n5, d5 = 2_200_000, 128
    h5, _, t5 = synthetic.make_edges_only(n5, 40_000_000, 64)
    deg5 = np.bincount(h5, minlength=n5).astype(np.float32)
    g5 = AttentiveGraph.from_coo(torch.from_numpy(h5.astype(np.int64)).to(dev), torch.from_numpy(t5.astype(np.int64)).to(dev),
                                 torch.from_numpy((1.0 / deg5[h5]).astype(np.float32)).to(dev), n5)
    dims = [d5, 128, 64, 32, 16]
    torch.manual_seed(0)
    layers = [(torch.randn(dims[i + 1], dims[i], device=dev) * 0.1, torch.zeros(dims[i + 1], device=dev),
               torch.randn(dims[i + 1], dims[i], device=dev) * 0.1, torch.zeros(dims[i + 1], device=dev)) for i in range(4)]
    e0 = torch.randn(n5, d5, device=dev) * 0.1
    drop = DropoutSpec(ps=[0.1] * 4, seed=1)

    def step():
        st = propagate_forward(g5, e0, layers, drop, save=True)
        g_last = torch.ones_like(st.tables[-1])
        propagate_backward(g5, st, layers, g_last, lambda l, buf: None)

    x5 = e0
    y5 = torch.empty_like(x5)
    t_spmm = time_cuda(lambda: g5.matmul(x5, out=y5), 5)
    tfile = ROOT / "profiles" / "ncu_traffic.json"
    c5_traffic = json.loads(tfile.read_text()).get("spmm_d128_c5_scaled") if tfile.exists() else None
    t_step = time_cuda(step, 3, warm=1)
    b_gather = 8.0 * g5.nnz + 16.0 * g5.plan.n_tasks + 4.0 * g5.nnz * d5 + 4.0 * n5 * d5
    out = {"nodes": n5, "nnz": g5.nnz, "dims": dims, "table_bytes": 4.0 * n5 * d5,
           "propagation_step_ms": t_step * 1e3, "propagated_edges_per_s": g5.nnz * 4 * 2 / t_step,
           "spmm_d128": {"ms": t_spmm * 1e3, "algorithmic_bytes": b_gather, "achieved": b_gather / t_spmm / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": b_gather / t_spmm / 1e9 / peak, "edges_per_s": g5.nnz / t_spmm,
                         # what the launch really moves through HBM (ncu dram__bytes_read + write, profiles/r2_c5_spmm_d128_ncu.csv:
                         # 14.81 + 1.12 GB, L2 hit rate 21 %) over the time measured here
                         "traffic": c5_traffic, "achieved_by_traffic": (c5_traffic / t_spmm / 1e9) if c5_traffic else None,
                         "frac_by_traffic": (c5_traffic / t_spmm / 1e9 / peak) if c5_traffic else None,
                         "model": "B_gather (SURVEY.md 8d): the table is 9x the L2, one 512 B neighbour row per edge is compulsory HBM traffic; "
                                  "Zipf hubs still hit the L2, so the figure can exceed the copy peak; frac_by_traffic uses the DRAM bytes ncu counts"},
           "what": "full (unpruned) 4-layer propagation forward + backward with message dropout, one GPU; the sharded run is in the N > 1 lines"}
    del g5, e0, layers, x5, y5
    torch.cuda.empty_cache()
    try:  # the same full training step the N > 1 lines report (sharding.ShardedEngine), here with one rank: the N-GPU c5_scaled.step_ms compare to it
        from kgat_b200.sharded_pruned import c5_sharded_block

        out["sharded_step_world1"] = c5_sharded_block(dev, 1, 0)
    except Exception as e:  # noqa: BLE001
        out["sharded_step_world1"] = {"unavailable": f"{type(e).__name__}: {e}"[:300]}
    return out


DUMP_LIMIT_BYTES = 64 << 20
DUMP_ATT_ENTRIES = 1 << 20


def dump_outputs(out_dir: Path, model, losses) -> None:
    """What ``TrainEngine.run_epoch`` leaves its caller after the last timed epoch: the epoch's mean CF and KG losses and the
    trained model -- every dense parameter in full, and the refreshed attention weights at a fixed, seeded sample of their
    entries (all of them would not fit the dump's 64 MB next to the entity table).  The inputs and the gradients' summation
    order are fixed, so two runs of one build with the same arguments write bit-identical arrays."""
    arrays = {"cf_loss": np.array(losses[0], np.float64), "kg_loss": np.array(losses[1], np.float64)}
    for k, v in model.state_dict().items():
        if not v.is_sparse:
            arrays[k] = v.detach().float().cpu().numpy()
    vals = model.attentive_matrix.data._values()
    pick = np.sort(np.random.default_rng(0).choice(vals.numel(), size=min(DUMP_ATT_ENTRIES, vals.numel()), replace=False))
    arrays["attentive_matrix.values_sample"] = vals[torch.from_numpy(pick).to(vals.device)].float().cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES} byte limit")
    out_dir.mkdir(parents=True, exist_ok=True)
    for k, a in arrays.items():
        np.save(out_dir / f"{k}.npy", a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-hbm-regime", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary shapes (Yelp2018 top-20, scaled C5, full Codeforces)")
    ap.add_argument("--budget-s", type=float, default=330.0, help="wall-clock budget: optional blocks are skipped once it is spent")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path,
                    help="write what the last timed epoch left the caller (losses, trained parameters, refreshed attention) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and (args.impl != "ours" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs covers the single-GPU run of our implementation")
    if args.impl == "reference":
        run_reference_arm(args)
        return
    t_start = time.perf_counter()

    import kgat_b200  # noqa: F401
    from kgat_b200 import _lib, ops
    from kgat_b200.engine import TrainEngine
    from kgat_b200.trainer import build_model, run_epoch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist

        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl")
        if args.gpus != world:
            raise SystemExit(f"--gpus {args.gpus} != WORLD_SIZE {world}")
        from kgat_b200 import sharded_pruned

        sharded_pruned.bench_main(args, METRIC, UNIT, WORKLOAD, make_workload, config_dict, ClockSampler)
        return
    if args.gpus != 1:
        raise SystemExit("launch N>1 with torch.distributed.run (one rank per GPU)")

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    _lib.load()
    g, data = make_workload(WORKLOAD)
    model = build_model(g, dev)
    init_state = {k: v.detach().clone().cpu() for k, v in model.state_dict().items() if not v.is_sparse}
    dev_data = data.tensors(device=dev)
    host_data = data.tensors(pin=True)

    def barrier():
        torch.cuda.synchronize()

    engine = TrainEngine(model)
    engine.bind_resident(data.tensors())

    # ---- set-up (never timed): two 2-step mini-epochs capture the step graphs and take the one-off structure swap of
    #      the first attention refresh, so that even --warmup 0 times steady-state epochs only
    for _ in range(2):
        engine.run_epoch(n_cf=2, n_kg=2)
    # ---- warm-up: W full epochs (>= 3 by contract) through the CUDA-graph engine ----
    for _ in range(max(args.warmup, 0)):
        engine.run_epoch()
    barrier()

    # ---- timed: K epochs, inputs resident in HBM ----
    _lib.LaunchCounter.count = 0
    with ClockSampler(local_rank) as clocks:
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        t0.record()
        losses = None
        for _ in range(args.steps):
            losses = engine.run_epoch()
        t1.record()
        barrier()
    launches = _lib.LaunchCounter.count
    if args.dump_outputs is not None:  # before the e2e leg below trains the same model further
        dump_outputs(args.dump_outputs, model, losses)
    phases = dict(engine.last_phase_ms)
    epoch_s = t0.elapsed_time(t1) / 1e3 / max(args.steps, 1)
    clk = clocks.summary()
    graph = model._graph()
    fr = frontier_stats(engine, graph)

    # ---- e2e: one epoch through the reference-facing model API (model(...), loss.backward(),
    #      update_*_weights(), loss.item()) from pinned host buffers; and the same through the engine ----
    e2e = None
    if not args.no_e2e:
        steps_in_epoch = data.n_cf + data.n_kg
        run_epoch(model, host_data, read_loss_every_step=True, n_cf=8, n_kg=8, refresh=False)  # capture the API graphs (untimed)
        barrier()
        w0 = time.perf_counter()
        _, _, h2d, d2h = run_epoch(model, host_data, read_loss_every_step=True)
        barrier()
        e2e_s = time.perf_counter() - w0
        engine = TrainEngine(model)  # re-read the Adam step counts the API epoch advanced
        engine.bind_resident(data.tensors())
        engine.run_epoch(host_data, read_loss_every_step=True, n_cf=8, n_kg=8, refresh=False)  # capture host-mode graphs
        barrier()
        w0 = time.perf_counter()
        engine.run_epoch(host_data, read_loss_every_step=True)
        barrier()
        e2e_engine_s = time.perf_counter() - w0
        e2e = {"value": e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "api": "model(..., mode=TRAIN_CF/TRAIN_KG/UPDATE_ATTENTION) + loss.backward() + update_*_weights() + loss.item()",
               "engine_value": e2e_engine_s,
               "note": f"bytes are per epoch (= one bench step: {steps_in_epoch} model steps; every model step copies its ids from pinned host "
                       "memory and reads its loss back on the host); engine_value = same host buffers through the CUDA-graph TrainEngine"}

    # ---- per-kernel split + roofline of the dominant kernel (live CUDA events, same process) ----
    n_probe_cf, n_probe_kg = 30, 60
    # eager (un-captured) launches so that every kernel can be bracketed by its own pair of CUDA events
    probe = TrainEngine(model, use_graphs=False)
    probe.bind_resident(data.tensors())
    with ops.KernelTimer() as kt:
        probe.run_epoch(n_cf=n_probe_cf, n_kg=n_probe_kg, refresh=False)
    ksum = kt.summary()
    per_epoch_ms = {}
    for name, (cnt, ms) in ksum.items():
        cf_kernel = not (name.startswith("transr") or name.startswith("adam_rolling"))
        if name == "adam_apply":
            continue
        scale = (data.n_cf / n_probe_cf) if cf_kernel else (data.n_kg / n_probe_kg)
        per_epoch_ms[name] = {"launches_per_epoch": int(cnt * scale), "avg_us": 1e3 * ms / cnt, "epoch_ms": ms * scale}
    if "adam_apply" in kt.events:
        ev = kt.events["adam_apply"]
        cf_ms = sum(a.elapsed_time(b) for a, b in ev[:n_probe_cf])
        kg_ms = sum(a.elapsed_time(b) for a, b in ev[n_probe_cf:])
        per_epoch_ms["adam_apply_cf"] = {"launches_per_epoch": data.n_cf, "avg_us": 1e3 * cf_ms / n_probe_cf, "epoch_ms": cf_ms * data.n_cf / n_probe_cf}
        if len(ev) > n_probe_cf:  # (only when the KG phase runs the dense sweep: kg_adam="dense"; the rolling kernels are timed under their own names)
            per_epoch_ms["adam_apply_kg"] = {"launches_per_epoch": data.n_kg, "avg_us": 1e3 * kg_ms / max(n_probe_kg, 1), "epoch_ms": kg_ms * data.n_kg / max(n_probe_kg, 1)}
    # dominant kernel = the propagation kernel (north_star) with the largest share of the epoch
    prop = [k for k in per_epoch_ms if k.startswith("spmm") or k.startswith("biagg_fwd") or k.startswith("biagg_bwd")]
    top = max(prop, key=lambda k: per_epoch_ms[k]["epoch_ms"])
    top_spmm = max((k for k in prop if k.startswith("spmm")), key=lambda k: per_epoch_ms[k]["epoch_ms"])
    peak, peak_kind = peaks()
    traffic_all = {}
    tfile = ROOT / "profiles" / "ncu_traffic.json"
    if tfile.exists():
        traffic_all = json.loads(tfile.read_text())

    def roof(name):
        abytes = algorithmic_bytes(name, g, graph, fr)
        us = per_epoch_ms[name]["avg_us"]
        ach = abytes / (us * 1e-6) / 1e9 if abytes else None
        return {"kernel": name, "bound": "hbm", "avg_us": us, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": (ach / peak) if ach else None,
                "traffic": traffic_all.get(name), "peak_source": f"{peak_kind} (MEASURED_PEAKS.json hbm_gbs, burst copy)",
                "algorithmic_bytes_per_launch": abytes,
                "model": "B_min (every distinct byte once, SURVEY.md 8d) over the rows / edges the pruned step touches"}

    # `roofline` follows the attentive SpMM (the HBM / L2 gather kernel north_star's 60 % target is about, and the kernel round 1's
    # verdict named); the bi-interaction kernels are tensor-pipe / latency bound and are listed in roofline_propagation_kernels
    roofline = roof(top_spmm)
    roofline["largest_propagation_kernel"] = top
    roofline_all = {k: {kk: vv for kk, vv in roof(k).items() if kk in ("avg_us", "achieved", "frac", "algorithmic_bytes_per_launch")} for k in prop}
    # the same kernel against what actually bounds it while the 41 MB table sits in the L2: the L2 -> SM gather fabric
    l2 = l2_gather_peak()
    roofline_l2 = None
    if l2 and "gather_peak_gbs" in l2:
        gb = gathered_bytes(top_spmm, g, graph, fr)
        ab = algorithmic_bytes(top_spmm, g, graph, fr)
        us = per_epoch_ms[top_spmm]["avg_us"]
        ach = (gb + ab) / (us * 1e-6) / 1e9
        roofline_l2 = {"kernel": top_spmm, "bound": "l2_gather", "avg_us": us, "achieved": ach, "peak": l2["gather_peak_gbs"], "unit": "GB/s",
                       "frac": ach / l2["gather_peak_gbs"], "gathered_bytes_per_launch": gb, "streamed_bytes_per_launch": ab,
                       "peak_source": "tools/microbench/l2_gather run in this process's job: random 256 B rows out of a 41 MB table, all SMs, no compute",
                       "microbench": l2}
    elif l2:
        roofline_l2 = l2
    # the dense Adam sweep (the CF phase's optimiser step; the KG phase used it too until the rolling window replaced it there),
    # timed back to back over the KG parameter set so launch gaps do not count
    ad = engine.kg_adam
    snap = ad.snapshot()
    adam_s = time_cuda(lambda: ad.apply(engine.kg_grads), 20, warm=1)
    ad.restore(snap)
    adam_bytes = 7.0 * 4 * sum(p.numel() for p in ad.params)
    roofline_adam = {"kernel": "adam_kernel (dense sweep over the entity table + moments)", "bound": "hbm", "avg_us": adam_s * 1e6, "algorithmic_bytes_per_launch": adam_bytes,
                     "achieved": adam_bytes / adam_s / 1e9, "peak": peak, "unit": "GB/s", "frac": adam_bytes / adam_s / 1e9 / peak}

    def left():
        return args.budget_s - (time.perf_counter() - t_start)

    # ---- baselines: the unmodified reference on the host cores (bounded sample) and on this GPU (the same-box incumbent) ----
    cpu = incumbent = None
    if not args.no_cpu_baseline:
        try:
            r = ReferenceRunner(g, init_state, data, "cpu")
            c = r.sample(n_cf=3, n_kg=3)
            cpu = {"value": c["epoch_s_extrapolated"], "unit": UNIT, "cores": c["cores"], "kind": c["kind"], "sample": c["sample"],
                   "cf_step_s": c["cf_step_s"], "kg_step_s": c["kg_step_s"], "refresh_s": c["refresh_s_extrapolated"]}
            del r
        except Exception as e:  # noqa: BLE001 - a baseline must never take the bench line down
            cpu = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
        try:
            r = ReferenceRunner(g, init_state, data, dev)
            c = r.sample(n_cf=3, n_kg=10)
            incumbent = {"value": c["epoch_s_extrapolated"], "unit": UNIT, "kind": c["kind"],
                         "what": "the unmodified reference KGAT moved to this B200 (.to('cuda'): stock ATen / cuSPARSE kernels, torch.optim.Adam, the "
                                 "device -> host -> device round trip of model.py:364-366, loss read every step)",
                         "cf_step_s": c["cf_step_s"], "kg_step_s": c["kg_step_s"], "refresh_s": c["refresh_s_extrapolated"], "sample": c["sample"]}
            del r
            torch.cuda.empty_cache()
        except Exception as e:  # noqa: BLE001
            incumbent = {"unavailable": f"{type(e).__name__}: {e}"[:200]}

    # ---- secondary configurations (BASELINE.json configs[3], [4] scaled, [1]) while the wall-clock budget lasts ----
    extras = {}
    if not args.no_extra:
        for key, cost, fn in (("c4_yelp2018", 40, lambda: extra_shape_block("yelp2018", dev, topk_users=True)),
                              ("c5_scaled", 60, lambda: c5_scaled_block(dev, peak)),
                              ("c2_codeforces_full", 150, lambda: extra_shape_block("codeforces-full", dev, n_cf=10, n_kg=50))):
            if key == "c5_scaled" and args.no_hbm_regime:
                continue
            if left() < cost:
                extras[key] = {"skipped": f"wall-clock budget ({args.budget_s:.0f} s) spent; run with a larger --budget-s"}
                continue
            try:
                extras[key] = fn()
            except Exception as e:  # noqa: BLE001
                extras[key] = {"unavailable": f"{type(e).__name__}: {e}"[:300]}

    n_layers = 3
    ref_edges_per_epoch = graph.nnz * n_layers * 2 * data.n_cf
    touched = sum(v["edges"] for v in fr.values()) * 2 * data.n_cf if fr else ref_edges_per_epoch
    line = {
        "metric": METRIC, "value": epoch_s, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": epoch_s * 1e3, "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(g, data, 1),
        "propagation_edges_per_s": ref_edges_per_epoch / epoch_s,
        "propagation_edges_per_s_note": "reference-equivalent: nnz x 3 layers x (fwd + bwd) x CF steps of the reference's full-graph propagation per "
                                        "batch, divided by the measured epoch; edges_touched_per_s counts only the frontier's edges actually processed",
        "edges_touched_per_s": touched / epoch_s, "frontier": fr,
        "cf_loss": losses[0], "kg_loss": losses[1],
        "phases": {"cf_phase_s": phases["cf"] / 1e3, "kg_phase_s": phases["kg"] / 1e3, "refresh_s": phases["refresh"] / 1e3,
                   "cf_step_us": 1e3 * phases["cf"] / max(phases["n_cf"], 1), "kg_step_us": 1e3 * phases["kg"] / max(phases["n_kg"], 1)},
        "kg_adam": {"engine": {"mode": engine.kg_adam_mode, "window": engine.kg_window},
                    "api": {"deferred": bool(model.kg_deferred_adam), "window": model.kg_window},
                    "optimiser_state_bytes_per_step": 6.0 * 4 * model._emb_raw().numel() / max(engine.kg_window, 1),
                    "dense_sweep_bytes_per_step": 6.0 * 4 * model._emb_raw().numel(),
                    "what": "KG-phase Adam over the entity table: batch rows + a rotating 1/window slice per step, zero-gradient updates "
                            "replayed in registers; bit-identical to the per-step sweep of torch.optim.Adam (tests: rolling / deferred / "
                            "arithmetic_core)"},
        "e2e": e2e, "gpu_launches": launches, "clocks": clk,
        "roofline": roofline, "roofline_l2": roofline_l2, "roofline_adam": roofline_adam, "roofline_propagation_kernels": roofline_all,
        "cpu_baseline": cpu, "gpu_incumbent": incumbent,
        **extras,
        "kernels": {k: {kk: round(vv, 3) if isinstance(vv, float) else vv for kk, vv in v.items()} for k, v in sorted(per_epoch_ms.items(), key=lambda kv: -kv[1]["epoch_ms"])},
        "bench_wall_s": time.perf_counter() - t_start,
    }
    print(json.dumps(line))


if __name__ == "__main__":
    main()
