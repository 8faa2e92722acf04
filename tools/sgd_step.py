"""Step time with SGD (egot2_sgd_step_fused: momentum with Nesterov) against the same trainer with the default Adam / AdamW.

    python tools/sgd_step.py [--steps 200] [--rounds 6] [--legs hhi_graph,hoi_lta,hhi_g]

Legs, each timed as A (default Adam) / B (SGD(momentum=0.9, nesterov=True), same weight decay) alternately in `rounds` rounds
on the same GPU:
  hhi_graph   HHI TranslatorTrainer at the benchmark shape (256 clips x 90 tokens, H 128), whole-step CUDA graph
  hoi_lta     HOI LTA TranslatorTrainer at b512, whole-step graph: the largest arena (~28 M parameters), where the optimizer's
              share of the step is largest.  Per parameter SGD moves 26 B (reads parameter, gradient, buffer; writes
              parameter, buffer, bf16 shadow, cleared gradient), Adam 34 B
  hhi_g       HHI EgoT2-g PromptTranslatorTrainer (bench.py's hhi_g_train batches): graph replay, then the optimizer as an
              eager launch (Adam: the fused launch on the host step count; SGD: the SGD launch on the host step count)
Inputs come from bench.py's pools (distinct batches, together >= 2 x L2).  Prints one JSON line per leg with the median, min
and max us/step of A and B over the rounds, every round's numbers, and the GPU name and power limit they were measured at."""
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
from egot2_b200.optim import SGD  # noqa: E402
from egot2_b200.trainer import PromptTranslatorTrainer, TranslatorTrainer  # noqa: E402

NESTEROV = SGD(momentum=0.9, nesterov=True)


def power_limit() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:      # noqa: BLE001 - reported, not fatal
        return f"unknown ({e!r})"


def make_trainer(leg, sgd, device="cuda:0"):
    kw = dict(optimizer=sgd, weight_decay=1e-4)
    if leg == "hhi_g":
        wl = bench.WORKLOADS["hhi_g_train"]
        spec = wl["spec"]()
        kw.pop("weight_decay")                     # the EgoT2-g HHI recipe is Adam without weight decay
        tr = PromptTranslatorTrainer(256, 4, 3, 0.1, device, "bf16", **kw)
    else:
        wl = bench.WORKLOADS["hoi_lta_train_b512" if leg == "hoi_lta" else "hhi_ttm3_train_b256"]
        spec = wl["spec"]()
        tr = TranslatorTrainer(spec, device, "bf16", use_graphs=True, **kw)
    tr.load_state_dict(synth.make_state_dict(spec, 0))
    return tr, wl, spec


def time_leg(leg, steps, rounds, device="cuda:0"):
    dev = torch.device(device)
    arms = {}
    for name, g in (("adam", None), ("sgd", NESTEROV)):
        tr, wl, spec = make_trainer(leg, g, device)
        pool, _ = bench.build_pool(wl, spec, wl["batch"], dev, "bf16", 0)
        arms[name] = (tr, pool)

    def run(name, n):
        tr, pool = arms[name]
        for i in range(n):
            fe, la = pool[i % len(pool)]
            tr.train_step(fe, la, graph_key=i % len(pool))
    for name in arms:                                 # capture every pool graph, warm both arms
        run(name, max(len(arms[name][1]), 10))
    us = {"adam": [], "sgd": []}
    for r in range(rounds):
        for name in (("adam", "sgd") if r % 2 == 0 else ("sgd", "adam")):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(dev)
            e0.record()
            run(name, steps)
            e1.record()
            torch.cuda.synchronize(dev)
            us[name].append(1000.0 * e0.elapsed_time(e1) / steps)
    numel = arms["adam"][0].engine.arena.numel
    del arms
    torch.cuda.empty_cache()
    return us, numel


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--legs", default="hhi_graph,hoi_lta,hhi_g")
    args = ap.parse_args()
    gpu = dict(name=torch.cuda.get_device_name(0), power_limit=power_limit(), count=torch.cuda.device_count())
    for leg in args.legs.split(","):
        us, numel = time_leg(leg, args.steps, args.rounds)
        out = dict(leg=leg, steps=args.steps, rounds=args.rounds, gpu=gpu, arena_numel=numel)
        for arm in ("adam", "sgd"):
            out[f"us_per_step_{arm}"] = round(statistics.median(us[arm]), 2)
            out[f"spread_{arm}"] = [round(min(us[arm]), 2), round(max(us[arm]), 2)]
            out[f"rounds_{arm}"] = [round(x, 2) for x in us[arm]]
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
