#!/usr/bin/env python
"""Per-kernel device time of the KG training step (TransR forward + backward, its deterministic reduce, the loss reduction and the
rolling-window Adam kernels) at the Amazon-book shape, from a torch.profiler trace of eager (un-captured) steps of the epoch engine.

    python tools/prof_kg_kernels.py [--steps 200] [--out profiles/kg_kernels.json] [--label NAME]

Prints and writes {kernel: {launches_per_step, avg_us, us_per_step}} with the card's name and power limit read in the same run.
"""
import argparse
import json
import re
import subprocess
import sys
from pathlib import Path

import torch
from torch.profiler import ProfilerActivity, profile

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

from kgat_b200 import synthetic  # noqa: E402
from kgat_b200.engine import TrainEngine  # noqa: E402
from kgat_b200.trainer import KG_BATCH, EpochData, build_model  # noqa: E402


def short_name(name: str) -> str:
    """'void kgat::(anonymous namespace)::transr_reduce_kernel<2, 2>(...)' -> 'transr_reduce_kernel<2, 2>'"""
    name = re.sub(r"\(.*\)$", "", name.strip().replace("(anonymous namespace)::", ""))
    name = re.sub(r"^void ", "", name)
    return name.split("::")[-1] if "<" not in name else name[name.rfind("::", 0, name.index("<")) + 2:]


def gpu_info() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = (s.strip() for s in out.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:  # noqa: BLE001
        return {"name": torch.cuda.get_device_name(), "power_limit": f"unavailable ({type(e).__name__})"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shape", default="amazon-book")
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--out", type=Path, default=None)
    ap.add_argument("--label", default="")
    args = ap.parse_args()

    g = synthetic.make_ckg(args.shape)
    model = build_model(g, "cuda").train()
    data = EpochData.sample(g, n_cf=1, n_kg=args.steps)
    eng = TrainEngine(model, use_graphs=False)
    eng.bind_resident(data.tensors())
    eng.run_epoch(n_cf=0, n_kg=args.steps, refresh=False)  # warm-up: module loads, first touches
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.run_epoch(n_cf=0, n_kg=args.steps, refresh=False)
        torch.cuda.synchronize()
    per = {}
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA or ev.device_time_total <= 0:
            continue
        k = short_name(ev.name)
        c, t = per.get(k, (0, 0.0))
        per[k] = (c + 1, t + ev.device_time_total)
    kernels = {k: {"launches_per_step": c / args.steps, "avg_us": t / c, "us_per_step": t / args.steps}
               for k, (c, t) in sorted(per.items(), key=lambda kv: -kv[1][1])}
    res = {"label": args.label, "shape": args.shape, "kg_batch": KG_BATCH,
           "steps": args.steps, "gpu": gpu_info(), "sum_us_per_step": sum(v["us_per_step"] for v in kernels.values()),
           "what": "torch.profiler CUDA activity of eager KG steps (TrainEngine(use_graphs=False)); kernel device time only, no launch gaps",
           "kernels": kernels}
    print(json.dumps(res, indent=1))
    if args.out is not None:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
