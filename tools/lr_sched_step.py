"""Step time with a device-evaluated learning-rate schedule (optim.LRSchedule) against the same trainer without one.

    python tools/lr_sched_step.py [--steps 200] [--rounds 5]

Legs, each timed as A (no schedule) / B (LRSchedule.cosine with warm-up) alternately in `rounds` rounds on the same GPU:
  hhi_graph   HHI TranslatorTrainer at the benchmark shape (256 clips x 90 tokens, H 128), whole-step CUDA graph: the
              advance kernel replaces the step-count increment on the graph's side branch
  hhi_eager   the same trainer with use_graphs=False: one extra one-thread launch before the fused Adam
  hhi_g       HHI EgoT2-g PromptTranslatorTrainer (bench.py's hhi_g_train batches): graph replay + eager Adam, one extra
              launch before it
Inputs come from bench.py's pools (distinct batches, together >= 2 x L2).  Prints one JSON line per leg with the median
us/step of A and B over the rounds, every round's numbers, and the GPU name and power limit they were measured at."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
from egot2_b200 import synth  # noqa: E402
from egot2_b200.optim import LRSchedule  # noqa: E402
from egot2_b200.trainer import PromptTranslatorTrainer, TranslatorTrainer  # noqa: E402


def power_limit() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:      # noqa: BLE001 - reported, not fatal
        return f"unknown ({e!r})"


def make_trainer(leg, schedule):
    if leg == "hhi_g":
        wl = bench.WORKLOADS["hhi_g_train"]
        spec = wl["spec"]()
        kw = {} if schedule is None else dict(lr_schedule=schedule)
        tr = PromptTranslatorTrainer(256, 4, 3, 0.1, "cuda:0", "bf16", **kw)
    else:
        wl = bench.WORKLOADS["hhi_ttm3_train_b256"]
        spec = wl["spec"]()
        tr = TranslatorTrainer(spec, "cuda:0", "bf16", use_graphs=(leg == "hhi_graph"), lr_schedule=schedule)
    tr.load_state_dict(synth.make_state_dict(spec, 0))
    return tr, wl, spec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--legs", default="hhi_graph,hhi_eager,hhi_g")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    gpu = dict(name=torch.cuda.get_device_name(0), power_limit=power_limit())
    total = args.steps * (args.rounds + 1)
    for leg in args.legs.split(","):
        sched = LRSchedule.cosine(5e-4, total, end_lr=1e-6, warmup_steps=total // 10)
        arms = {}
        for name, s in (("none", None), ("cosine", sched)):
            tr, wl, spec = make_trainer(leg, s)
            pool, _ = bench.build_pool(wl, spec, wl["batch"], dev, "bf16", 0)
            arms[name] = (tr, pool)

        def run(name, n):
            tr, pool = arms[name]
            for i in range(n):
                fe, la = pool[i % len(pool)]
                tr.train_step(fe, la, graph_key=i % len(pool) if tr.use_graphs else None)
        for name in arms:                                 # capture every pool graph, warm both arms
            run(name, max(len(arms[name][1]), 10))
        us = {"none": [], "cosine": []}
        for r in range(args.rounds):
            for name in (("none", "cosine") if r % 2 == 0 else ("cosine", "none")):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize(dev)
                e0.record()
                run(name, args.steps)
                e1.record()
                torch.cuda.synchronize(dev)
                us[name].append(1000.0 * e0.elapsed_time(e1) / args.steps)
        print(json.dumps(dict(leg=leg, steps=args.steps, rounds=args.rounds, gpu=gpu,
                              us_per_step_none=round(statistics.median(us["none"]), 2),
                              us_per_step_cosine=round(statistics.median(us["cosine"]), 2),
                              rounds_none=[round(x, 2) for x in us["none"]],
                              rounds_cosine=[round(x, 2) for x in us["cosine"]])), flush=True)
        del arms
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
