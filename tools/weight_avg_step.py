"""Step time with a weight average (weight_average: one egot2_weight_avg_update launch after every optimizer launch) against
the same trainer without it.

    python tools/weight_avg_step.py [--steps 200] [--rounds 5] [--legs hhi_graph,hoi_lta,hhi_g,kernel]

Arms, timed alternately in `rounds` rounds on the same GPU (the order rotates every round):
  off         no average
  ema1        WeightAverage.ema(0.999): every step due (reads the parameters and the average, writes the average)
  ema10       WeightAverage.ema(0.999, every=10): a due step every 10 steps, the others exit at once
  swa1        WeightAverage.swa(): every step due, the running mean
Legs:
  hhi_graph   HHI TranslatorTrainer at the benchmark shape (256 clips x 90 tokens, H 128), whole-step CUDA graph
  hoi_lta     HOI LTA TranslatorTrainer at b512, whole-step graph: the largest arena (~28 M parameters)
  hhi_g       HHI EgoT2-g PromptTranslatorTrainer (bench.py's hhi_g_train batches): graph replay, then the eager optimizer
  kernel      egot2_weight_avg_update alone on the LTA b512 arena, due (EMA) and not due, back to back (its 336 MB working
              set exceeds the 126 MB L2): us per launch and the achieved bytes/s of a due launch
Inputs come from bench.py's pools.  Prints one JSON line per leg with the median and the range of us/step of every arm over
the rounds, the bytes a due step moves, and the GPU name and power limit they were measured at."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
from egot2_b200 import synth  # noqa: E402
from egot2_b200.optim import WeightAverage  # noqa: E402
from egot2_b200.trainer import PromptTranslatorTrainer, TranslatorTrainer  # noqa: E402
from param_stats_step import power_limit  # noqa: E402

ARMS = {"off": None, "ema1": WeightAverage.ema(0.999), "ema10": WeightAverage.ema(0.999, every=10),
        "swa1": WeightAverage.swa()}


def make_trainer(leg, wa, device="cuda:0"):
    kw = {} if wa is None else dict(weight_average=wa)
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
    for name, wa in ARMS.items():
        tr, wl, spec = make_trainer(leg, wa, device)
        pool, _ = bench.build_pool(wl, spec, wl["batch"], dev, "bf16", 0)
        arms[name] = (tr, pool)
    numel = arms["off"][0].engine.arena.numel

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
    return us, numel


def time_kernel(rounds, launches=200, device="cuda:0"):
    from egot2_b200 import _lib as L
    from egot2_b200.engine import ParamArena
    numel = ParamArena(bench.WORKLOADS["hoi_lta_train_b512"]["spec"](), "meta").numel
    param = torch.randn(numel, device=device)
    avg = torch.randn(numel, device=device)
    wa = WeightAverage.ema(0.999)
    steps = {"due": torch.full((1,), 2, dtype=torch.int32, device=device),
             "not_due": torch.full((1,), 0, dtype=torch.int32, device=device)}
    st = torch.cuda.current_stream().cuda_stream

    def run(name, n):
        for _ in range(n):
            L.call("egot2_weight_avg_update", param.data_ptr(), avg.data_ptr(), numel, wa.kind, wa.ema_weight, wa.every,
                   wa.start, steps[name].data_ptr(), None, st)
    us = {name: [] for name in steps}
    for name in steps:
        run(name, 10)
    for r in range(rounds):
        for name in (list(steps) if r % 2 == 0 else list(steps)[::-1]):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            run(name, launches)
            e1.record()
            torch.cuda.synchronize()
            us[name].append(1000.0 * e0.elapsed_time(e1) / launches)
    return us, numel


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--legs", default="hhi_graph,hoi_lta,hhi_g,kernel")
    args = ap.parse_args()
    gpu = dict(name=torch.cuda.get_device_name(0), power_limit=power_limit())
    for leg in args.legs.split(","):
        us, numel = time_kernel(args.rounds) if leg == "kernel" else time_leg(leg, args.steps, args.rounds)
        extra = {}
        if leg == "kernel":
            extra["due_tb_per_s"] = round(12 * numel / statistics.median(us["due"]) / 1e6, 3)
        print(json.dumps(dict(leg=leg, steps=args.steps, rounds=args.rounds, gpu=gpu, arena_numel=numel,
                              due_step_bytes=12 * numel, **extra,
                              median_us={k: round(statistics.median(v), 2) for k, v in us.items()},
                              range_us={k: [round(min(v), 2), round(max(v), 2)] for k, v in us.items()},
                              rounds_us={k: [round(x, 2) for x in v] for k, v in us.items()})), flush=True)


if __name__ == "__main__":
    main()
