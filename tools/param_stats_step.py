"""Step time with per-parameter statistics (param_stats: one egot2_param_stats launch before every optimizer launch) against
the same trainer without them.

    python tools/param_stats_step.py [--steps 200] [--rounds 5] [--legs hhi_graph,hoi_lta,hhi_g]

Arms, timed alternately in `rounds` rounds on the same GPU (the order rotates every round):
  off         no statistics
  every100    ParamStats(100): a due step every 100 steps, the others exit at once (the amortised case)
  every1_nh   ParamStats(1, histograms=False): every step due, moments and norms only
  every1      ParamStats(1): every step due, with histograms (the worst case)
Legs:
  hhi_graph   HHI TranslatorTrainer at the benchmark shape (256 clips x 90 tokens, H 128), whole-step CUDA graph
  hoi_lta     HOI LTA TranslatorTrainer at b512, whole-step graph: the largest arena (~28 M parameters)
  hhi_g       HHI EgoT2-g PromptTranslatorTrainer (bench.py's hhi_g_train batches): graph replay, then the eager optimizer
Inputs come from bench.py's pools.  Prints one JSON line per leg with the median and the range of us/step of every arm over
the rounds, and the GPU name and power limit they were measured at."""
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
from egot2_b200.stats import ParamStats  # noqa: E402
from egot2_b200.trainer import PromptTranslatorTrainer, TranslatorTrainer  # noqa: E402

ARMS = {"off": None, "every100": ParamStats(100), "every1_nh": ParamStats(1, histograms=False), "every1": ParamStats(1)}


def power_limit() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:      # noqa: BLE001 - reported, not fatal
        return f"unknown ({e!r})"


def make_trainer(leg, ps, device="cuda:0"):
    kw = {} if ps is None else dict(param_stats=ps)
    if leg == "hhi_g":
        wl = bench.WORKLOADS["hhi_g_train"]
        spec = wl["spec"]()
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
    for name, ps in ARMS.items():
        tr, wl, spec = make_trainer(leg, ps, device)
        pool, _ = bench.build_pool(wl, spec, wl["batch"], dev, "bf16", 0)
        arms[name] = (tr, pool)

    def run(name, n):
        tr, pool = arms[name]
        for i in range(n):
            fe, la = pool[i % len(pool)]
            tr.train_step(fe, la, graph_key=i % len(pool))
    for name in arms:                                 # capture every pool graph, warm every arm
        run(name, max(len(arms[name][1]), 10))
    us = {name: [] for name in arms}
    order = list(arms)
    for r in range(rounds):
        for name in order[r % len(order):] + order[:r % len(order)]:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(dev)
            e0.record()
            run(name, steps)
            e1.record()
            torch.cuda.synchronize(dev)
            us[name].append(1000.0 * e0.elapsed_time(e1) / steps)
    del arms
    torch.cuda.empty_cache()
    return us


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--legs", default="hhi_graph,hoi_lta,hhi_g")
    args = ap.parse_args()
    gpu = dict(name=torch.cuda.get_device_name(0), power_limit=power_limit())
    for leg in args.legs.split(","):
        us = time_leg(leg, args.steps, args.rounds)
        print(json.dumps(dict(leg=leg, steps=args.steps, rounds=args.rounds, gpu=gpu,
                              median_us={k: round(statistics.median(v), 2) for k, v in us.items()},
                              range_us={k: [round(min(v), 2), round(max(v), 2)] for k, v in us.items()},
                              rounds_us={k: [round(x, 2) for x in v] for k, v in us.items()})), flush=True)


if __name__ == "__main__":
    main()
