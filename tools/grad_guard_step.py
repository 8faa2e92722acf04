"""Step time with the gradient guard (max_grad_norm: egot2_grad_norm + the guarded optimizer) against the same trainer
without it.

    python tools/grad_guard_step.py [--steps 200] [--rounds 5] [--legs hhi_graph,hoi_lta,hhi_g,peer]

Legs, each timed as A (no guard) / B (max_grad_norm=1.0) alternately in `rounds` rounds on the same GPU:
  hhi_graph   HHI TranslatorTrainer at the benchmark shape (256 clips x 90 tokens, H 128), whole-step CUDA graph: the norm
              launch is captured between the backward and the optimizer
  hoi_lta     HOI LTA TranslatorTrainer at b512, whole-step graph: the largest arena (~28 M fp32 gradients, ~112 MB), where
              the extra read of the gradient arena costs most
  hhi_g       HHI EgoT2-g PromptTranslatorTrainer (bench.py's hhi_g_train batches): graph replay, then the norm and the
              guarded Adam as eager launches
  peer        the hhi_graph leg on 2 ranks over the peer-memory exchange (EGOT2_DP_FUSED=1), which the guard splits into two
              launches with one more flag round trip; only with more than one GPU
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
from egot2_b200.trainer import PromptTranslatorTrainer, TranslatorTrainer  # noqa: E402

MAX_NORM = 1.0


def power_limit() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:      # noqa: BLE001 - reported, not fatal
        return f"unknown ({e!r})"


def make_trainer(leg, guard, device="cuda:0"):
    kw = {} if guard is None else dict(max_grad_norm=guard)
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
    for name, g in (("none", None), ("guard", MAX_NORM)):
        tr, wl, spec = make_trainer("hhi_graph" if leg == "peer" else leg, g, device)
        pool, _ = bench.build_pool(wl, spec, wl["batch"], dev, "bf16", 0)
        arms[name] = (tr, pool)

    def run(name, n):
        tr, pool = arms[name]
        for i in range(n):
            fe, la = pool[i % len(pool)]
            tr.train_step(fe, la, graph_key=i % len(pool))
    for name in arms:                                 # capture every pool graph, warm both arms
        run(name, max(len(arms[name][1]), 10))
    us = {"none": [], "guard": []}
    for r in range(rounds):
        for name in (("none", "guard") if r % 2 == 0 else ("guard", "none")):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(dev)
            e0.record()
            run(name, steps)
            e1.record()
            torch.cuda.synchronize(dev)
            us[name].append(1000.0 * e0.elapsed_time(e1) / steps)
    skipped = int(arms["guard"][0].skipped_steps)
    del arms
    torch.cuda.empty_cache()
    return us, skipped


def _peer_worker(rank, world, port, steps, rounds, q):
    import torch.distributed as dist
    os.environ.update(EGOT2_DP_FUSED="1", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank),
                      WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        out = time_leg("peer", steps, rounds, f"cuda:{rank}")
        if rank == 0:
            q.put(out)
        dist.barrier()
    finally:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--legs", default="hhi_graph,hoi_lta,hhi_g,peer")
    args = ap.parse_args()
    gpu = dict(name=torch.cuda.get_device_name(0), power_limit=power_limit(), count=torch.cuda.device_count())
    for leg in args.legs.split(","):
        if leg == "peer":
            if torch.cuda.device_count() < 2:
                print(json.dumps(dict(leg=leg, gpu=gpu, skipped="needs 2 GPUs")), flush=True)
                continue
            import socket

            import torch.multiprocessing as mp
            with socket.socket() as s:
                s.bind(("127.0.0.1", 0))
                port = s.getsockname()[1]
            ctx = mp.get_context("spawn")
            q = ctx.Queue()
            procs = [ctx.Process(target=_peer_worker, args=(r, 2, port, args.steps, args.rounds, q)) for r in range(2)]
            for p in procs:
                p.start()
            us, skipped = q.get(timeout=600)
            for p in procs:
                p.join(timeout=60)
        else:
            us, skipped = time_leg(leg, args.steps, args.rounds)
        print(json.dumps(dict(leg=leg, steps=args.steps, rounds=args.rounds, gpu=gpu, max_grad_norm=MAX_NORM,
                              skipped_steps=skipped,
                              us_per_step_none=round(statistics.median(us["none"]), 2),
                              us_per_step_guard=round(statistics.median(us["guard"]), 2),
                              rounds_none=[round(x, 2) for x in us["none"]],
                              rounds_guard=[round(x, 2) for x in us["guard"]])), flush=True)


if __name__ == "__main__":
    main()
