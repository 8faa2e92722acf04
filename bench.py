#!/usr/bin/env python
"""Benchmark of the EgoT2 task-translation hot path on B200 (contract: see the task statement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dtype bf16|fp32]
                    [--dump-outputs DIR]

Metric (BASELINE.json): translator forward+backward clips/sec.  Default workload = BASELINE config 2:
HHI TaskFusionMFTransformer3Task (LAM+TTM+ASD -> TTM) training, 1 layer, hidden 128, 4 heads, FFN 2048,
256 clips per GPU x 3 tasks x 30 frames (T = 90 tokens), synthetic per-frame features (256-wide), seeded weights.
One step = forward + fused weighted-CE loss + backward of every translator parameter + (N>1: one NCCL
all-reduce of the flat gradient arena) + one fused Adam launch.

Lines printed by rank 0 (ONE JSON line):
  value     whole-job clips/s over exactly K timed steps, features already resident in HBM (rotating pool larger than L2),
            CUDA-event timed, max over ranks; at the default K = 2000 that window lasts about 0.66 s (0.33 ms steps on one
            B200 at 1000 W), while K = 20 gives a window of a few milliseconds.  Only this figure follows --steps exactly:
            e2e, fwd_only, fp32, module_path and the other workloads each time their own count, derived from K but clamped;
  e2e       same step driven from pinned HOST buffers through TranslatorTrainer.train_stream_host: every step's H2D copy of
            features+labels and D2H read of its loss are inside the timed region (double-buffered on a copy stream);
  roofline  the dominant kernel of the step (largest share of the summed kernel time), timed by CUDA events that the
            library records around each launch on the launch stream during a pass of eager steps after the timed region;
  cpu_baseline  the CPU oracle (torch restatement of the reference translator) on this box's host cores.
`--impl reference` times that CPU implementation as the reference arm.

--dump-outputs DIR: after the K timed steps, rank 0 writes what the last of them computed - the loss it returned
(loss.npy) and, where the step runs from a CUDA graph of the single-model trainer, the translator output it computed
(logits.npy) - in float32, so that two builds run with the same arguments (same seeded weights and inputs) can be compared
output for output.  The updated parameters are deliberately not written: the kernels' reductions add partial sums in no
fixed order, and Adam turns those last-bit differences into whole learning-rate steps wherever a gradient is rounding
noise (the attention key bias has an exactly zero gradient), so the parameters differ between two runs of one build by
far more than rounding, while what the step computes from them does not.
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

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from egot2_b200 import specs, synth  # noqa: E402

WORKLOADS = {
    # BASELINE.json configs[1]
    "hhi_ttm3_train_b256": dict(spec=lambda: specs.hhi_ttm_spec(128, 4, 1, 0.5, True), batch=256, seg_tokens=(30, 30, 30)),
    # BASELINE.json configs[3] (per-frame features; bf16)
    "hoi_pnr_train_b256": dict(spec=lambda: specs.hoi_pnr_spec(128, 6, 16, 0.5, 0.1), batch=256, seg_tokens=(16, 16, 8, 8)),
    # BASELINE.json configs[4]
    "hoi_lta_train_b512": dict(spec=lambda: specs.hoi_lta_spec(512, 4, 8, 0.5), batch=512, seg_tokens=(2, 2, 2, 2)),
    # BASELINE.json configs[2]: HHI EgoT2-g, one step = the three forwards of video_tasktranslation.py:39-66 on
    # lam (64 clips x 7 tokens), ttm (8 clips x 3x30 tokens), asd (20 clips x 3x30 tokens -> 600 frame rows); H256 L3+3
    "hhi_g_train": dict(spec=lambda: specs.hhi_g_spec(256, 4, 3, 0.1, "ttm"), batch=92, seg_tokens=(30, 30, 30), prompt=True,
                        g_batches=dict(lam=(64, 7), ttm=(8, 30), asd=(20, 30))),
    # SURVEY 8f-2: HOI EgoT2-g at the reference defaults (hidden 512, 8 heads, 3+3 layers, HOI/configs/multitask/config.py:49-53),
    # one step = the three forwards of Unified3TaskTranslation.training_step (pnr, oscc and action batches of 32 clips x 48 tokens)
    "hoi_g_train": dict(spec=lambda: specs.hoi_g_spec(512, 8, 3, 0.1, 600), batch=96, seg_tokens=(16, 16, 8, 8), prompt=True,
                        g_kind="hoi", g_batches=dict(pnr=32, oscc=32, action=32)),
}
L2_BYTES = 126 * 2 ** 20
DUMP_BYTES = 60 * 2 ** 20         # array payload of --dump-outputs: with the .npy headers the files stay under 64 MB


def dump_outputs(out_dir, arrays):
    """Write {name: tensor} as out_dir/<name>.npy in float32.  When all of them together exceed DUMP_BYTES, every tensor is
    replaced by the same fraction of its elements (at least one), picked by a fixed seed (flattened, in index order), so
    that two runs sample identical positions."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    keep = min(1.0, (DUMP_BYTES // 4 - len(arrays)) / sum(t.numel() for t in arrays.values()))
    g = torch.Generator().manual_seed(0)
    for name, t in arrays.items():
        a = t.detach().float().cpu()
        if keep < 1.0:
            flat = a.reshape(-1)
            a = flat[torch.randperm(flat.numel(), generator=g)[:max(1, int(flat.numel() * keep))].sort().values]
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy())


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"], bf16_tflops_sustained=d["bf16_tflops_sustained"],
                    source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


def load_ncu_traffic(tag: str):
    """dram bytes (read+write) per launch of the dominant kernel, from the committed `ncu --set full` summary
    (profiles/ncu_traffic.json: {launcher-tag prefix: bytes}); None when that kernel has no capture yet."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(p):
        return None
    try:
        table = json.load(open(p))
    except Exception:
        return None
    for k, v in table.items():
        if not k.startswith("_") and tag.startswith(k):
            return v
    return None


def make_g_batch(wl, seed, fdt):
    """EgoT2-g step inputs: 7 feature tensors [lam | lam,ttm,asd | lam,ttm,asd] + concatenated (rows,3) targets."""
    feats, labels = [], []
    if wl.get("g_kind") == "hoi":          # 12 feature tensors = 3 x [pnr, oscc, slow, fast] + concatenated (clips,3) targets
        sp = wl["spec"]()
        for i, task in enumerate(("pnr", "oscc", "action")):
            b = wl["g_batches"][task]
            f = synth.make_features(sp, b, seed=seed * 7 + i, dtype=fdt)
            feats += [f[s_.name] for s_ in sp.segments]
            labels.append(synth.make_labels(sp, b, seed=seed * 7 + i))
        return feats, torch.cat(labels, dim=0)
    for mode in ("lam", "ttm", "asd"):
        b, d = wl["g_batches"][mode]
        sp = specs.hhi_g_spec(256, 4, 3, 0.1, mode)
        seg = (d,) if mode == "lam" else (d, d, d)
        f = synth.make_features(sp, b, seg, seed=seed * 7 + len(mode), dtype=fdt)
        feats += [f[s_.name] for s_ in sp.segments]
        labels.append(synth.make_labels(sp, b, seg, seed=seed * 7 + len(mode)))
    return feats, torch.cat(labels, dim=0)


def g_flops_per_step(wl, backward=True):
    tot = 0.0
    if wl.get("g_kind") == "hoi":
        return sum(wl["g_batches"].values()) * wl["spec"]().flops_per_clip(wl["seg_tokens"], backward=backward)
    for mode in ("lam", "ttm", "asd"):
        b, d = wl["g_batches"][mode]
        sp = specs.hhi_g_spec(256, 4, 3, 0.1, mode)
        seg = (d,) if mode == "lam" else (d, d, d)
        tot += b * sp.flops_per_clip(seg, backward=backward)      # encoder + projections; the 2-token decoder is < 2 %
    return tot


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------- reference legs
# SURVEY.md section 8(d): which roofline bounds each configuration (the table, not a self-made byte count)
TABLE_BOUND = {"hhi_ttm3_train_b256": "tensor", "hoi_pnr_train_b256": "hbm+tensor", "hoi_lta_train_b512": "tensor",
               "hhi_g_train": "tensor", "hoi_g_train": "tensor"}


def time_reference_cpu(name, wl, steps, warmup, batch=0, budget_s=25.0):
    """The UNMODIFIED reference translator class (oracle/ref_shims: source tree here, oracle/_ref on the GPU box; the oracle
    port only if neither exists) on the host cores, all threads, fp32: forward (train mode) + loss + backward + Adam.
    Bounded: stops early when `budget_s` is exceeded.  Returns (clips/s, s/step, steps done, kind, info)."""
    torch.set_num_threads(os.cpu_count() or 1)
    B = batch or wl["batch"]
    from oracle import ref_bench
    step = None
    if ref_bench.available():
        try:
            step, info = ref_bench.make_step(name, wl, "cpu", autocast_bf16=False, adam=True, batch=B)
            kind = "reference"
        except Exception as e:        # e.g. oracle/_ref incomplete on this box: fall back to the restatement, and say so
            print(f"bench: reference classes unavailable ({e!r}); timing the oracle port instead", file=sys.stderr)
    if step is None:
        spec = wl["spec"]()
        fn = cpu_oracle_g_step_fn(wl) if wl.get("prompt") else cpu_oracle_step_fn(spec, B, wl["seg_tokens"])
        step, info, kind = (lambda i: fn()), {"class": "oracle port", "source": "oracle/translator_oracle.py"}, "port"
    for i in range(warmup):
        step(i)
    t0 = time.perf_counter()
    done = 0
    for i in range(steps):
        step(warmup + i)
        done += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return B * done / dt, dt / done, done, kind, info


def cpu_oracle_step_fn(spec, batch, seg_tokens, seed=0):
    """Fallback when the reference classes are unavailable: the CPU oracle port (fwd train mode + loss + backward)."""
    from oracle import translator_oracle as O
    sd = synth.make_state_dict(spec, seed)
    P = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    feats = synth.make_features(spec, batch, seg_tokens, seed)
    labels = synth.make_labels(spec, batch, seg_tokens, seed)
    cw = torch.tensor([0.266, 0.734])

    def step():
        for p in P.values():
            p.grad = None
        if spec.family == "hhi_ttm":
            out = O.hhi_ttm_forward(P, feats, spec.heads, spec.p_layer, True)
            loss = O.ce_loss(out, labels, cw)
        elif spec.family == "hoi_pnr":
            out = O.hoi_pnr_forward(P, feats["pnr"], feats["oscc"], feats["slow"], feats["fast"], spec.heads,
                                    spec.p_feat, spec.p_layer, True)
            loss = O.bce_sigmoid_loss(out, torch.nn.functional.one_hot(labels, 16).float())
        else:
            out = O.hoi_lta_forward(P, feats["pnr"], feats["oscc"], feats["action"], feats["lta"], spec.heads,
                                    spec.p_layer, spec.p_head, True)
            loss = O.lta_loss(out, labels, spec.head_groups)
        loss.backward()
        return float(loss)
    return step


def cpu_oracle_g_step_fn(wl, seed=0):
    """EgoT2-g fallback: the three forwards + summed CE + backward of the CPU oracle port."""
    from oracle import translator_oracle as O
    spec = wl["spec"]()
    sd = synth.make_state_dict(spec, seed)
    P = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    feats, labels = make_g_batch(wl, seed, torch.float32)
    if wl.get("g_kind") == "hoi":

        def hoi_step():
            for p in P.values():
                p.grad = None
            off, loss = 0, 0.0
            for i in range(3):
                pnr, oscc, slow, fast = feats[4 * i:4 * i + 4]
                tgt = labels[off:off + pnr.shape[0]]
                off += pnr.shape[0]
                out = O.hoi_g_forward(P, pnr, oscc, slow, fast, tgt[:, :-1], spec.heads, spec.p_layer, True)
                loss = loss + torch.nn.functional.cross_entropy(out, tgt[:, 1:])
            loss.backward()
            return float(loss)
        return hoi_step
    groups = {"lam": dict(lam=feats[0]), "ttm": dict(lam=feats[1], ttm=feats[2], asd=feats[3]),
              "asd": dict(lam=feats[4], ttm=feats[5], asd=feats[6])}

    def step():
        for p in P.values():
            p.grad = None
        off, loss = 0, 0.0
        for mode in ("lam", "ttm", "asd"):
            b, d = wl["g_batches"][mode]
            rows = b * d if mode == "asd" else b
            tgt = labels[off:off + rows]
            off += rows
            out = O.hhi_g_forward(P, groups[mode], tgt[:, :-1], mode, spec.heads, spec.p_layer, True)
            loss = loss + torch.nn.functional.cross_entropy(out, tgt[:, 1:])
        loss.backward()
        return float(loss)
    return step


def run_reference(args, wl, spec):
    """--impl reference: the reference's own implementation of the path on the host cores (rank 0 only), same steps/warmup as
    our arm; every step is the workload's full batch unless the run would exceed the time budget (then it stops early and
    says so in `sample`)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warm = max(1, args.steps), max(1, args.warmup)
    cps, sec, done, kind, info = time_reference_cpu(args.workload, wl, steps, min(warm, 3), budget_s=150.0)
    cores = torch.get_num_threads()
    sample = (f"{done} of {steps} requested steps x {wl['batch']} clips; {info.get('class')} from {info.get('source')}; "
              f"{info.get('step', 'fwd + loss + bwd')}; fp32; {cores} host threads; bounded at 150 s of CPU work")
    line = {"impl": "reference", "metric": "translator fwd+bwd clips/sec", "value": cps, "unit": "clips/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "steps_timed": done, "ms_per_step": sec * 1e3,
            "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_of(args.workload, wl, spec, wl["batch"]),
            "cpu_baseline": {"value": cps, "unit": "clips/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": cps, "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def config_of(name, wl, spec, B):
    """The workload description both arms print (identical keys and values: the driver compares them)."""
    return {"workload": name, "translator": spec.family, "hidden": spec.hidden, "layers": spec.layers, "heads": spec.heads,
            "ffn": spec.ffn, "clips_per_gpu": B, "tokens_per_clip": sum(wl["seg_tokens"]),
            "step": "fwd (train mode, dropout on) + loss + bwd (all translator grads) + Adam"}


# ---------------------------------------------------------------------------------------------- our arm
def build_trainer(name, wl, spec, dev, dtype, use_graphs=True):
    from egot2_b200.trainer import HoiPromptTranslatorTrainer, PromptTranslatorTrainer, TranslatorTrainer
    if wl.get("prompt") and wl.get("g_kind") == "hoi":
        tr = HoiPromptTranslatorTrainer(spec.hidden, spec.heads, spec.layers, spec.p_layer, spec.vocab, dev, dtype)
    elif wl.get("prompt"):
        tr = PromptTranslatorTrainer(256, 4, 3, 0.1, dev, dtype)
    else:
        tr = TranslatorTrainer(spec, dev, dtype, use_graphs=use_graphs)
    tr.load_state_dict(synth.make_state_dict(spec, 0))          # identical weights on every rank
    return tr


def build_pool(wl, spec, B, dev, dtype, rank, max_pool=64):
    """Distinct input batches resident in HBM, together >= 2 x L2, so that no step finds its inputs in L2."""
    fdt = torch.bfloat16 if dtype == "bf16" else torch.float32
    seg = wl["seg_tokens"]
    if wl.get("prompt"):
        feat_bytes = sum(t.numel() * t.element_size() for t in make_g_batch(wl, 0, fdt)[0])
    else:
        feat_bytes = spec.feature_elems_per_clip(seg) * B * (2 if dtype == "bf16" else 4)
    n_pool = min(max_pool, max(3, -(-2 * L2_BYTES // feat_bytes)))
    pool = []
    for i in range(n_pool):
        if wl.get("prompt"):
            fe, la = make_g_batch(wl, 1000 * rank + i, fdt)
            pool.append(([t.to(dev) for t in fe], la.to(dev)))
            continue
        f = synth.make_features(spec, B, seg, seed=1000 * rank + i, dtype=fdt)
        pool.append(([f[s.name].to(dev) for s in spec.segments], synth.make_labels(spec, B, seg, seed=1000 * rank + i).to(dev)))
    return pool, feat_bytes


def timed(fn, n, dev, world):
    """CUDA-event time of fn(0..n-1) in ms, barrier + synchronize on both sides, max over ranks."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize(dev)
    e0.record()
    for i in range(n):
        fn(i)
    e1.record()
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize(dev)
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
    return float(ms.item())


def measure_train(name, wl, spec, B, dev, dtype, rank, world, steps, warmup, use_graphs=True):
    """Device-resident training throughput of one workload at `world` GPUs: (trainer, pool, ms_total)."""
    tr = build_trainer(name, wl, spec, dev, dtype, use_graphs)
    pool, feat_bytes = build_pool(wl, spec, B, dev, dtype, rank)
    n_pool = len(pool)

    def step(i):
        fe, la = pool[i % n_pool]
        tr.train_step(fe, la, graph_key=i % n_pool)
    for i in range(max(warmup, n_pool if tr.use_graphs else warmup)):      # capture every pool graph first
        step(i)
    ms = timed(lambda i: step(i + 1), steps, dev, world)
    return tr, pool, feat_bytes, ms


def other_workload_line(name, dev, rank, world, steps, warmup, batch=0):
    """A further BASELINE.json configuration, device-resident at `world` GPUs (weak scaling), compact record."""
    wl = dict(WORKLOADS[name])
    if batch:
        wl["batch"] = batch
    spec = wl["spec"]()
    B = wl["batch"]
    tr, pool, feat_bytes, ms = measure_train(name, wl, spec, B, dev, "bf16", rank, world, steps, warmup)
    peaks = load_peaks()
    is_g = bool(wl.get("prompt"))
    flops = g_flops_per_step(wl) if is_g else spec.flops_per_clip(wl["seg_tokens"], backward=True) * B
    sec = ms * 1e-3 / steps
    rec = {"workload": name, "clips_per_gpu": B, "n_gpus": world, "value": world * B / sec, "unit": "clips/s",
           "ms_per_step": sec * 1e3, "steps": steps, "model_tflops_per_s_per_gpu": flops / sec / 1e12,
           "frac_tensor_sustained": flops / sec / 1e12 / peaks["bf16_tflops_sustained"], "bound_8d": TABLE_BOUND.get(name)}
    if not is_g:
        # SURVEY 8(d): Bytes_fwd+bwd = 2 x feature bytes (+ 3 x parameter bytes, which matter at small batch)
        pbytes = 3 * sum(v.numel() for v in synth.make_state_dict(spec, 0).values()) * 2
        rec["frac_hbm"] = (2 * feat_bytes + pbytes) / sec / 1e9 / peaks["hbm_gbs"]
    del tr, pool
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="hhi_ttm3_train_b256", choices=sorted(WORKLOADS))
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--batch", type=int, default=0, help="clips per GPU (default: the workload's)")
    ap.add_argument("--no-graphs", action="store_true")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-extras", action="store_true", help="headline line only (A/B runs): no fwd_only / fp32 / "
                    "module_path / gpu_baseline / other workloads")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's loss and translator output "
                    "as DIR/<name>.npy (float32, under 64 MB in all)")
    args = ap.parse_args()
    wl = dict(WORKLOADS[args.workload])
    if args.batch:
        wl["batch"] = args.batch
    spec = wl["spec"]()
    if args.impl == "reference":
        return run_reference(args, wl, spec)
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    from egot2_b200.parallel import bind_to_gpu_numa
    numa = bind_to_gpu_numa(local_rank)            # pinned staging buffers land on the GPU's own NUMA node
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=dev)
    from egot2_b200 import _lib as L

    B, seg = wl["batch"], wl["seg_tokens"]
    fdt = torch.bfloat16 if args.dtype == "bf16" else torch.float32
    is_g = bool(wl.get("prompt"))
    lib = L.load()

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident throughput over the K timed steps
    clocks = ClockSampler(local_rank)
    tr = build_trainer(args.workload, wl, spec, dev, args.dtype, not args.no_graphs)
    pool, feat_bytes = build_pool(wl, spec, B, dev, args.dtype, rank)
    n_pool = len(pool)
    last = []            # (loss, graph key) of the latest step

    def run_steps(n, start=0):
        for i in range(n):
            fe, la = pool[(start + i) % n_pool]
            last[:] = [tr.train_step(fe, la, graph_key=(start + i) % n_pool), (start + i) % n_pool]

    run_steps(max(args.warmup, n_pool if tr.use_graphs else args.warmup))     # capture every pool graph first
    barrier()
    l0 = lib.egot2_launch_count()
    tr.use_graphs, keep = False, tr.use_graphs
    run_steps(1)                                                                # one eager step to count our launches
    launches_per_step = lib.egot2_launch_count() - l0
    tr.use_graphs = keep
    barrier()
    if rank == 0:
        clocks.start()
    try:
        ms_total = timed(lambda i: run_steps(1, start=1 + i), args.steps, dev, world)
    finally:
        clock_info = clocks.stop() if rank == 0 else None
    value = world * B * args.steps / (ms_total * 1e-3)
    if args.dump_outputs and rank == 0:
        # the step's buffers are overwritten by the legs below: copied out before any of them runs
        from egot2_b200.engine import Activations
        from egot2_b200.trainer import TranslatorTrainer
        outputs = {"loss": last[0].reshape(1)}
        if isinstance(tr, TranslatorTrainer) and tr.use_graphs:
            act = tr._graphs[last[1]][-1]          # the graph cache entry ends with the activations its replays write
            assert isinstance(act, Activations), f"unexpected graph cache entry {type(act)}: no logits to dump"
            outputs["logits"] = act.t["out"]
        dump_outputs(args.dump_outputs, outputs)

    # ---- end-to-end from pinned host buffers (H2D + step + D2H of the loss inside the timed region)
    host = []
    for i in range(2):
        if is_g:
            fe, la = make_g_batch(wl, 5000 + 10 * rank + i, fdt)
            host.append(([t.pin_memory() for t in fe], la.pin_memory()))
            continue
        f = synth.make_features(spec, B, seg, seed=5000 + 10 * rank + i, dtype=fdt)
        host.append(([f[s.name].pin_memory() for s in spec.segments],
                     synth.make_labels(spec, B, seg, seed=5000 + 10 * rank + i).pin_memory()))
    e2e_steps = max(5, min(args.steps, 200))
    tr.train_stream_host(host, 4)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    losses = tr.train_stream_host(host, e2e_steps)        # returns after the last loss has been read back
    e1.record()
    barrier()
    assert len(losses) == e2e_steps and all(l == l for l in losses), f"e2e: loss read-back failed: {losses}"
    ms2 = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        torch.distributed.all_reduce(ms2, op=torch.distributed.ReduceOp.MAX)
    e2e_value = world * B * e2e_steps / (float(ms2.item()) * 1e-3)
    h2d = sum(t.numel() * t.element_size() for t in host[0][0]) + host[0][1].numel() * 8
    # what the box's host -> device path allows: the same pinned buffers copied back to back, nothing else running
    # (the e2e step cannot be faster than this copy; on a shared VM it varies from box to box)
    devb = [torch.empty_like(t, device=dev) for t in host[0][0]]
    for _ in range(3):
        for d_, t in zip(devb, host[0][0]):
            d_.copy_(t, non_blocking=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(20):
        for d_, t in zip(devb, host[0][0]):
            d_.copy_(t, non_blocking=True)
    e1.record()
    torch.cuda.synchronize(dev)
    h2d_ms = e0.elapsed_time(e1) / 20
    h2d_gbs = sum(t.numel() * t.element_size() for t in host[0][0]) / (h2d_ms * 1e-3) / 1e9
    del devb

    # ---- the other BASELINE.json configurations at this GPU count (every rank takes part: they all-reduce too)
    others = []
    if not args.skip_extras and args.workload == "hhi_ttm3_train_b256" and args.dtype == "bf16":
        del host
        o_steps, o_warm = max(10, min(args.steps, 30)), 3
        for name in ("hoi_pnr_train_b256", "hoi_lta_train_b512", "hhi_g_train"):
            try:
                others.append(other_workload_line(name, dev, rank, world, o_steps, o_warm))
            except Exception as e:      # a secondary line must not take the headline down
                others.append({"workload": name, "error": repr(e)[:200]})
        # BASELINE configs[4]: batch sweep 64..4096 clips GLOBAL over the GPUs of this run (weight-HBM <-> tensor crossover)
        sweep = []
        for gb in (64, 256, 1024, 4096):
            if gb % world or gb // world < 8:
                continue
            try:
                r = other_workload_line("hoi_lta_train_b512", dev, rank, world, o_steps, o_warm, batch=gb // world)
                sweep.append({"global_batch": gb, "clips_per_gpu": gb // world, "value": r["value"], "ms_per_step": r["ms_per_step"],
                              "frac_tensor_sustained": r["frac_tensor_sustained"], "frac_hbm": r.get("frac_hbm")})
            except Exception as e:
                sweep.append({"global_batch": gb, "error": repr(e)[:200]})
        others.append({"workload": "hoi_lta batch sweep", "n_gpus": world, "sweep": sweep})

    if rank != 0:
        if world > 1:
            torch.distributed.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (timed alone, CUDA events on its launch stream)
    peaks = load_peaks()
    es = 2 if args.dtype == "bf16" else 4
    prof_steps = max(3, min(args.steps, 10))
    rows = profile_step_launchers(tr, [(fe, la) for fe, la in pool], n_pool, prof_steps, es)
    roof = dominant_kernel_roofline(rows, prof_steps, peaks, es, ms_total / args.steps * 1e3, TABLE_BOUND.get(args.workload))
    traffic = load_ncu_traffic(roof["kernel"])
    if traffic is not None:
        roof["traffic"] = traffic

    flops_step = g_flops_per_step(wl) if is_g else spec.flops_per_clip(seg, backward=True) * B
    tfs = flops_step * world * args.steps / (ms_total * 1e-3) / 1e12
    line = {
        "metric": "translator fwd+bwd clips/sec", "value": value, "unit": "clips/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if args.dtype == "bf16" else "f32", "data": "synthetic",
        "config": config_of(args.workload, wl, spec, B),       # identical in the reference arm's line
        "run": {"l2_policy": f"inputs rotate over a pool of {n_pool} batches = {n_pool * feat_bytes / 2**20:.0f} MiB "
                             f"> 126 MiB L2; saved activations add more per step",
                "cuda_graphs": bool(tr.use_graphs), "numa_bind": numa,
                "parallelism": f"dp{world} (clips sharded; one gradient exchange per step)",
                "exchange": ("none" if world == 1 else ("peer-memory kernel: reduce-scatter + Adam + all-gather (csrc/peer.cu)"
                                                        if getattr(tr, "peer", None) is not None else
                                                        "NCCL all-reduce overlapped with the embedding backward + fused Adam"))},
        "model_tflops_per_s": tfs,
        "step_roofline": {"bound": "tensor", "achieved": tfs / world, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                          "frac": tfs / world / peaks["bf16_tflops_sustained"],
                          "note": "whole step, per GPU: SURVEY 8(d) FLOPs_fwd+bwd per clip x clips / step time"},
        "clocks": clock_info,
        "e2e": {"value": e2e_value, "unit": "clips/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 4,
                "steps": e2e_steps, "h2d_copy_alone_ms": h2d_ms, "h2d_copy_alone_gbs": h2d_gbs,
                "h2d_bound_clips_per_s": world * B / (h2d_ms * 1e-3)},
        "gpu_launches": int(launches_per_step * args.steps),
        "gpu_launches_per_step": int(launches_per_step),
        "roofline": roof,
    }
    if others:
        line["other_workloads"] = others

    if world == 1 and not args.skip_extras and not is_g:
        extras = extra_legs(args, wl, spec, tr, pool, dev)
        line.update(extras)
    # ---- CPU baseline (rank 0, N=1 only): the reference class on the host cores, bounded sample
    if world == 1 and not args.skip_cpu_baseline:
        cps, sec, done, kind, info = time_reference_cpu(args.workload, wl, steps=5, warmup=1, budget_s=20.0)
        line["cpu_baseline"] = {"value": cps, "unit": "clips/s", "cores": torch.get_num_threads(), "kind": kind,
                                "sample": f"{done} steps x {B} clips; {info.get('class')} from {info.get('source')}; "
                                          f"{info.get('step', 'fwd + loss + bwd')}; fp32"}
    print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


def extra_legs(args, wl, spec, tr, pool, dev):
    """N = 1 only, rank 0: forward-only, fp32 mode, the drop-in nn.Module path, and the reference classes in stock torch
    eager on this same GPU (the comparator SURVEY 8(d) names)."""
    out = {}
    B, seg, n_pool = wl["batch"], wl["seg_tokens"], len(pool)
    n = max(20, min(args.steps, 200))

    def rec(ms, steps, **kw):
        return dict({"value": B * steps / (ms * 1e-3), "unit": "clips/s", "ms_per_step": ms / steps, "steps": steps}, **kw)
    # forward only (eval mode, no dropout), device-resident, eager launches
    try:
        for i in range(3):
            tr.infer(pool[i % n_pool][0])
        ms = timed(lambda i: tr.infer(pool[i % n_pool][0]), n, dev, 1)
        fl = spec.flops_per_clip(seg, backward=False) * B
        out["fwd_only"] = rec(ms, n, dtype=args.dtype, model_tflops_per_s=fl * n / (ms * 1e-3) / 1e12, mode="eval forward, eager launches")
    except Exception as e:
        out["fwd_only"] = {"error": repr(e)[:200]}
    # fp32 parity mode (CUDA-core fp32 kernels: the mode whose argmax is bit-exact against the reference)
    try:
        tr32 = build_trainer(args.workload, wl, spec, dev, "fp32", True)
        pool32, _ = build_pool(wl, spec, B, dev, "fp32", 0, max_pool=6)
        for i in range(max(3, len(pool32))):
            tr32.train_step(*pool32[i % len(pool32)], graph_key=i % len(pool32))
        n32 = max(5, min(n, 20))
        ms = timed(lambda i: tr32.train_step(*pool32[i % len(pool32)], graph_key=i % len(pool32)), n32, dev, 1)
        out["fp32"] = rec(ms, n32, dtype="f32", mode="fp32 parity mode, full training step")
        del tr32, pool32
    except Exception as e:
        out["fp32"] = {"error": repr(e)[:200]}
    # the drop-in nn.Module (what run_ttm.py gets): module forward + torch loss + loss.backward() + torch.optim.Adam
    try:
        out["module_path"] = module_path_leg(wl, spec, pool, dev, n)
    except Exception as e:
        out["module_path"] = {"error": repr(e)[:300]}
    # the reference classes in torch eager on this GPU
    try:
        from oracle import ref_bench
        gb = {"kind": "reference classes (oracle/ref_shims) in stock torch eager on the same GPU" if ref_bench.available() else "unavailable"}
        if ref_bench.available():
            for key, ac in (("fp32", False), ("bf16_autocast", True)):
                step, info = ref_bench.make_step(args.workload, wl, str(dev), autocast_bf16=ac, adam=True, n_batches=4)
                for i in range(5):
                    step(i)
                nb = max(10, min(n, 50))
                ms = timed(step, nb, dev, 1)
                gb[key] = rec(ms, nb)
                gb["class"], gb["source"], gb["step"] = info["class"], info["source"], info["step"]
                fstep, _ = ref_bench.make_step(args.workload, wl, str(dev), autocast_bf16=ac, training=False, n_batches=4)
                for i in range(3):
                    fstep(i)
                ms = timed(fstep, nb, dev, 1)
                gb[key + "_fwd_only"] = rec(ms, nb)
                del step, fstep
        out["gpu_baseline"] = gb
    except Exception as e:
        out["gpu_baseline"] = {"error": repr(e)[:300]}
    torch.cuda.empty_cache()
    return out


def module_path_leg(wl, spec, pool, dev, n):
    from types import SimpleNamespace
    from egot2_b200 import hhi
    from egot2_b200.modules import PrecomputedFeatures
    if spec.family != "hhi_ttm" or len(spec.segments) != 3:
        return {"skipped": "module-path leg is wired for the HHI 3-task translator"}

    class _Talk(torch.nn.Module):
        def forward_audio_frontend(self, a): return a
        def forward_visual_frontend(self, v): return v
        def forward_cross_attention(self, a, v): return a, v
        def forward_audio_visual_backend(self, a, v): return v["asd"].reshape(-1, v["asd"].shape[-1])

    class _Feats(dict):
        @property
        def shape(self):
            b, d, _ = self["asd"].shape
            return (b, d, 1, 1)
    margs = SimpleNamespace(lam_checkpoint="x", ttm_checkpoint="x", asd_checkpoint="x", nofreeze=False, hidden_dim=spec.hidden,
                            num_heads=spec.heads, dropout=spec.p_layer, num_layers=spec.layers)
    m = hhi.ttm.TaskFusionMFTransformer3Task(margs, backbones={"lam_model": PrecomputedFeatures("lam"), "ttm_model": PrecomputedFeatures("ttm"),
                                                               "asd_model": _Talk()})
    m.load_state_dict(synth.make_state_dict(spec, 0), strict=False)
    m.to(dev).set_compute_dtype("bf16").train()
    opt = torch.optim.Adam([p for p in m.parameters() if p.requires_grad], lr=5e-4)
    cw = torch.tensor([0.266, 0.734], device=dev)
    names = [s.name for s in spec.segments]

    def step(i):
        fe, la = pool[i % len(pool)]
        v = _Feats({k: t for k, t in zip(names, fe)})
        opt.zero_grad(set_to_none=True)
        out = m(v, v, None, None)
        loss = torch.nn.functional.cross_entropy(out.float(), la, weight=cw)
        loss.backward()
        opt.step()
    for i in range(5):
        step(i)
    ms = timed(step, n, dev, 1)
    return {"value": wl["batch"] * n / (ms * 1e-3), "unit": "clips/s", "ms_per_step": ms / n, "steps": n,
            "mode": "egot2_b200.hhi.ttm.TaskFusionMFTransformer3Task (bf16 compute) + torch cross_entropy + loss.backward() + torch.optim.Adam"}


def launcher_cost(tag: str, es: int):
    """Algorithmic (flops, bytes) of ONE launch of the launcher `tag` (the tags carry the problem shape).
    bytes = operands read once + results written once; es = bytes per activation element.  None = not modelled."""
    import re
    def ints(pat):
        m = re.search(pat, tag)
        return [int(x) for x in m.groups()] if m else None
    if tag.startswith("ffn_fwd_sm100"):
        M, FF = ints(r"M(\d+) H128 FF(\d+)")
        H = 128          # x1 in, W1+W2, hid saved for backward, y2 + x_out out
        return 4.0 * M * H * FF, (M * H + 2 * H * FF + M * FF + 2 * M * H) * es
    if tag.startswith("ffn_bwd_dx_sm100"):
        M, FF = ints(r"M(\d+) H128 FF(\d+)")
        H = 128          # dhid = gate(d2 . W2), d3 = dhid . W1 + d1; reads d2, d1, gate bits, W1+W2; writes dhid and d3
        return 4.0 * M * H * FF, (3 * M * H + 2 * H * FF + M * FF) * es + M * FF // 8
    if tag.startswith("ffn_bwd_sm100"):
        M, FF = ints(r"M(\d+) H128 FF(\d+)")
        H = 128          # dX GEMMs (2) + dW GEMMs (2); reads d2, x1, hid, W1, W2; writes d3 + fp32 dW1/dW2
        return 8.0 * M * H * FF, (3 * M * H + M * FF + 2 * H * FF) * es + 2 * H * FF * 4
    if tag.startswith("gemm_"):
        M, N, K = ints(r"M(\d+) N(\d+) K(\d+)")
        out_es = 4 if ",f32>" in tag or "<f32>" in tag else es
        extra = M * N * es if ("+mask" in tag or "+res" in tag) else 0
        return 2.0 * M * N * K, (M * K + N * K) * es + M * N * out_es + extra
    if tag.startswith("attn_"):
        B, T, H = ints(r"B(\d+) T(\d+) H(\d+)")
        if "_fwd" in tag:      # QK^T + PV ; reads qkv, writes out
            return 4.0 * B * T * T * H, B * T * 4 * H * es
        return 10.0 * B * T * T * H, B * T * 8 * H * es      # S, dP, dV, dQ, dK ; reads qkv,out,dout, writes dqkv
    m = ints(r"^ln_(?:fwd|bwd) rows(\d+) H(\d+)")
    if m:
        rows, H = m
        return 8.0 * rows * H, rows * H * es * (2 if tag.startswith("ln_fwd") else 3)
    m = ints(r"^colsum M(\d+) N(\d+)")
    if m:
        return float(m[0] * m[1]), m[0] * m[1] * es
    m = ints(r"^dropout_inplace n(\d+)")
    if m:
        return float(m[0]), 2 * m[0] * es
    return None


def profile_step_launchers(tr, pool, n_pool, steps, es):
    """Per-launcher CUDA-event timing of `steps` eager (un-graphed) training steps, through the library's own
    egot2_prof_* hooks: every launcher brackets its kernel(s) with events on the launch stream."""
    from egot2_b200 import _lib as L
    keep, keep_world, keep_peer = tr.use_graphs, tr.world, getattr(tr, "peer", None)
    tr.use_graphs, tr.world, tr.peer = False, 1, None      # rank 0 profiles alone: no collective / peer exchange in this pass
    for i in range(2):
        tr.train_step(*pool[i % n_pool])
    torch.cuda.synchronize()
    L.prof_enable(True)
    for i in range(steps):
        tr.train_step(*pool[(2 + i) % n_pool])
    torch.cuda.synchronize()
    rows = L.prof_report()
    L.prof_enable(False)
    tr.use_graphs, tr.world, tr.peer = keep, keep_world, keep_peer
    return rows


def dominant_kernel_roofline(rows, steps, peaks, es, step_us_graph, table_bound=None):
    """rows: [(tag, launches, total_us)] from the profiled pass.  The dominant launcher = the largest share of the
    summed kernel time; its achieved rate = algorithmic flops|bytes of one launch / its mean event-timed duration."""
    tot = sum(r[2] for r in rows) or 1.0
    ridge = peaks["bf16_tflops_sustained"] * 1e12 / (peaks["hbm_gbs"] * 1e9)
    breakdown = []
    for tag, n, us in rows[:8]:
        c = launcher_cost(tag, es)
        ent = {"launcher": tag, "launches_per_step": n / steps, "us_per_step": us / steps, "share": us / tot}
        if c:
            f, b = c
            ent["tflops"] = f * n / (us * 1e-6) / 1e12
            ent["gbs"] = b * n / (us * 1e-6) / 1e9
        breakdown.append(ent)
    tag, n, us = next(r for r in rows if launcher_cost(r[0], es))
    flops, nbytes = launcher_cost(tag, es)
    sec = us * 1e-6 / n
    ai = flops / nbytes
    # inside a long step the sustained tensor figure is the fair ceiling (MEASURED_PEAKS.json: burst vs sustained)
    # Which roofline bounds the kernel: SURVEY 8(d)'s table for the configuration (a contraction kernel of a tensor-bound
    # configuration is measured against the tensor pipe even when its own byte count - which includes activations that
    # are saved by design choice, not by necessity - would put it a hair under the ridge); otherwise by arithmetic intensity.
    contraction = tag.startswith(("ffn_", "gemm_", "attn_"))
    if es == 2 and ((table_bound == "tensor" and contraction) or ai >= ridge):
        bound, achieved, peak, unit = "tensor", flops / sec / 1e12, peaks["bf16_tflops_sustained"], "TFLOP/s"
    else:
        bound, achieved, peak, unit = "hbm", nbytes / sec / 1e9, peaks["hbm_gbs"], "GB/s"
    return {"kernel": tag, "bound": bound, "achieved": achieved, "peak": peak, "unit": unit, "frac": achieved / peak,
            "traffic": None, "us_per_launch": sec * 1e6, "launches_per_step": n / steps, "share_of_step": us / tot,
            "algorithmic_flops_per_launch": flops, "algorithmic_bytes_per_launch": nbytes,
            "arith_intensity_flop_per_byte": ai, "peak_source": peaks["source"] + " (sustained, timed inside the step)",
            "timing": "CUDA events recorded by the library around the launch, on the launch stream, %d eager steps" % steps,
            "sum_kernel_us_per_step": tot / steps, "graph_step_us": step_us_graph, "breakdown": breakdown}


if __name__ == "__main__":
    main()
