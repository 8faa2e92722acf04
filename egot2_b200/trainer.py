"""Fused training / inference steps over a TranslatorEngine: the public API the benchmark and
the end-to-end path use.

One training step = forward (fused loss) -> backward into the flat gradient arena ->
[data-parallel: ONE NCCL all-reduce of that arena over NVLink] -> one fused Adam launch.
Clips shard across ranks (each rank steps its own clips; no data-path collective), the only
exchange is the translator-gradient all-reduce (SURVEY.md §8e).  The forward+backward launch
sequence is captured once per input batch into a CUDA graph (the step is launch-bound at the
reference's batch sizes), replayed afterwards.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import ctypes as C
import os

import torch

from . import _lib as L
from .engine import Activations, TranslatorEngine
from .optim import LRSchedule
from .parallel import allreduce_gradients
from .specs import TranslatorSpec


def _cur_stream(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _dev_guard(device):
    """Make `device` current for library calls that own per-device state (side streams, the dropout-epoch slot)."""
    import contextlib
    return torch.cuda.device(device) if torch.device(device).type == "cuda" else contextlib.nullcontext()


def _make_peer_exchange(engine, process_group, world):
    """parallel.PeerExchange for this engine, or None (one rank, EGOT2_DP_FUSED=0, CPU group, or the IPC set-up failed on
    some rank - decided collectively, so that every rank takes the same path)."""
    import os
    # EGOT2_DP_FUSED: "1" always, "0" never, default "auto" = from 3 ranks on.  Measured on B200 (HHI b256, us per step,
    # peer-memory kernel vs NCCL all-reduce overlapped with the embedding backward + fused Adam): N=2 365.8 vs 358.3,
    # N=8 373.9 vs 393.0 - NCCL's small-message latency grows with the rank count, the one-kernel exchange's barely does.
    mode = os.environ.get("EGOT2_DP_FUSED", "auto")
    if world <= 1 or mode == "0" or (mode == "auto" and world < 3) or engine.device.type != "cuda" or world > 8:
        return None
    import torch.distributed as dist
    from .parallel import PeerExchange
    peer, ok = None, 1
    try:
        peer = PeerExchange(engine, process_group)
    except Exception as e:      # noqa: BLE001 - any failure means "use NCCL", never a silent wrong answer
        import warnings
        warnings.warn(f"egot2_b200: peer-memory exchange unavailable ({e!r}); using the NCCL all-reduce path")
        ok = 0
    flag = torch.tensor([ok], device=engine.device, dtype=torch.int32)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=process_group)
    return peer if int(flag.item()) == 1 else None


def _check_max_grad_norm(x) -> float:
    x = float(x)
    if not x > 0.0:                        # also rejects NaN
        raise ValueError(f"max_grad_norm must be positive (math.inf: skip non-finite steps, never clip), got {x}")
    return x


class _OptimizerState:
    """Learning-rate schedule, gradient guard and resumable optimizer state of the fused trainers.

    With `lr_schedule` (optim.LRSchedule) the trainer owns three device buffers: the egot2_lr_sched descriptor, the lr of
    the last step and the optimizer step count.  Every step, on every path, is egot2_opt_advance (step count + 1, lr of
    that step) followed by an optimizer launch that reads both from the device, so a replayed CUDA graph follows the
    schedule and `set_lr_schedule` takes effect without a new capture.

    With `max_grad_norm` the trainer also owns an egot2_grad_guard: right before the optimizer launch, after any gradient
    all-reduce, egot2_grad_norm computes the global L2 norm of the gradient the optimizer would apply; the update is then
    clipped to max_grad_norm (torch.nn.utils.clip_grad_norm_), or skipped when the norm is not finite - parameters, shadow
    and moments unchanged, gradient cleared, the device step count taken back, so the bias corrections and the schedule
    count applied steps only (GradScaler + LambdaLR, by contrast, advances the schedule on a skipped step).  The device
    step count is then authoritative: only construction and load_optimizer_state_dict set it from the host.

    Without either, nothing here adds a launch."""

    def _init_optimizer_state(self, lr_schedule: Optional[LRSchedule], lr: float, default_lr: float,
                              max_grad_norm: Optional[float] = None):
        if lr_schedule is not None and lr != default_lr:
            raise ValueError("pass either lr or lr_schedule, not both")
        self.max_grad_norm = None
        if max_grad_norm is not None:
            max_grad_norm = _check_max_grad_norm(max_grad_norm)
            if os.environ.get("EGOT2_DP_SPLIT", "0") == "1":
                raise ValueError("max_grad_norm is incompatible with EGOT2_DP_SPLIT=1: the split peer exchange updates most "
                                 "parameters before the embedding gradients, and so the global norm, exist")
        self.lr_schedule = None
        self._epoch = 0                    # dropout epoch of the next step: the trainer advances it once per step from 0
        if not hasattr(self, "_step_dev"):
            self._step_dev = torch.zeros(1, device=self.device, dtype=torch.int32)
            self._step_dev_val = 0
        if lr_schedule is not None:
            self._sched_dev = torch.zeros(C.sizeof(L.LrSched), device=self.device, dtype=torch.uint8)
            self._lr_dev = torch.zeros(1, device=self.device, dtype=torch.float32)
            self.lr_schedule = lr_schedule
            self.set_lr_schedule(lr_schedule)
        if max_grad_norm is not None:
            self._guard_dev = torch.zeros(C.sizeof(L.GradGuard), device=self.device, dtype=torch.uint8)
            self.engine.grad_norm_workspace()
            self.max_grad_norm = max_grad_norm
            self.set_max_grad_norm(max_grad_norm)

    def set_lr_schedule(self, schedule: LRSchedule):
        """Rewrite the device descriptor (in stream order): the next step follows `schedule` at its current step count, in
        graph mode without a new capture.  To drive the lr from host code, call set_lr_schedule(LRSchedule.constant(x))
        before each step."""
        if self.lr_schedule is None:
            raise ValueError("this trainer was built without lr_schedule; its optimizer launches take hp['lr']")
        host = torch.frombuffer(bytearray(bytes(schedule.pack())), dtype=torch.uint8)
        # pageable source: the copy is staged before copy_ returns, so `host` may go away at once
        self._sched_dev.copy_(host, non_blocking=True)
        self.lr_schedule = schedule

    def _guard_field(self, name: str, value=None, dtype=torch.float32) -> torch.Tensor:
        """The device bytes of one egot2_grad_guard field as a 0-dim tensor view; with `value`, write it first (stream
        order, only that field: the others belong to the kernels)."""
        f = getattr(L.GradGuard, name)
        view = self._guard_dev[f.offset:f.offset + f.size]
        if value is not None:
            host = torch.frombuffer(bytearray(bytes((C.c_float if dtype == torch.float32 else C.c_int32)(value))),
                                    dtype=torch.uint8)
            view.copy_(host, non_blocking=True)        # pageable source: staged before copy_ returns
        return view.view(dtype)[0]

    def set_max_grad_norm(self, max_grad_norm: float):
        """Rewrite the guard's max_norm on the device (in stream order): the next step clips to it, in graph mode without a
        new capture.  math.inf: skip non-finite steps, never clip."""
        if self.max_grad_norm is None:
            raise ValueError("this trainer was built without max_grad_norm; its optimizer launches have no gradient guard")
        x = _check_max_grad_norm(max_grad_norm)
        self._guard_field("max_norm", x)
        self.max_grad_norm = x

    @property
    def last_grad_norm(self) -> torch.Tensor:
        """The unclipped global gradient norm of the last step (what clip_grad_norm_ returns; NaN / inf on a skipped step), as
        a 0-dim device tensor: no sync."""
        if self.max_grad_norm is None:
            raise ValueError("this trainer was built without max_grad_norm; no gradient norm is computed")
        return self._guard_field("total_norm")

    @property
    def skipped_steps(self) -> torch.Tensor:
        """The number of steps skipped for a non-finite gradient, as a 0-dim device int32 tensor: no sync."""
        if self.max_grad_norm is None:
            raise ValueError("this trainer was built without max_grad_norm; no step is ever skipped")
        return self._guard_field("skipped", dtype=torch.int32)

    @property
    def last_lr(self) -> torch.Tensor:
        """The lr the last step used, as a 0-dim device tensor (with a schedule a view of the device lr: no sync)."""
        if self.lr_schedule is None:
            return torch.tensor(float(self.hp["lr"]), device=self.device)
        return self._lr_dev[0]

    def _opt_advance(self, stream: int):
        with _dev_guard(self.device):
            L.call("egot2_opt_advance", self._step_dev.data_ptr(), self._sched_dev.data_ptr(), self._lr_dev.data_ptr(),
                   stream)

    def _advance_eager(self) -> dict:
        """Before an eager optimizer launch: with a schedule or a guard, advance the device step count (and lr) on the
        current stream and return the launch's step_dev / lr_dev / guard arguments; without either, nothing ({})."""
        if self.lr_schedule is None and self.max_grad_norm is None:
            return {}
        if self.max_grad_norm is None and self._step_dev_val != self.step_count - 1:
            self._step_dev.fill_(self.step_count - 1)      # with a guard the device count is authoritative (skips)
        if self.lr_schedule is not None:
            self._opt_advance(_cur_stream(self.device))
        else:
            self._step_dev.add_(1)
        self._step_dev_val = self.step_count
        return self._opt_args(self._step_dev)

    def _opt_args(self, step_dev: torch.Tensor) -> dict:
        """step_dev / lr_dev (/ guard) of an optimizer launch that reads the device step count."""
        opt = dict(step_dev=step_dev, lr_dev=None if self.lr_schedule is None else self._lr_dev)
        if self.max_grad_norm is not None:
            opt["guard"] = self._guard_dev
        return opt

    def optimizer_state_dict(self) -> dict:
        """What a run needs beyond the parameters (state_dict) to resume as if uninterrupted: the Adam moments keyed by
        parameter name, the step count (train_step calls), the schedule, the dropout epoch and, with a guard, max_grad_norm and
        the number of skipped steps (read from the device: this syncs).  Under the peer-memory exchange every rank holds the
        moments of its own arena slice only: save and load per rank."""
        arena = self.engine.arena
        zeros = None if "m" in self.opt_state else torch.zeros_like(arena.param)
        return {"step": self.step_count,
                "exp_avg": arena.state_dict(self.opt_state.get("m", zeros)),
                "exp_avg_sq": arena.state_dict(self.opt_state.get("v", zeros)),
                "lr_schedule": None if self.lr_schedule is None else self.lr_schedule.to_dict(),
                "dropout_epoch": self._epoch,
                "max_grad_norm": self.max_grad_norm,
                "skipped_steps": 0 if self.max_grad_norm is None else int(self.skipped_steps)}

    def load_optimizer_state_dict(self, sd: dict):
        if (sd["lr_schedule"] is None) != (self.lr_schedule is None):
            raise ValueError("optimizer state saved " + ("without" if sd["lr_schedule"] is None else "with") +
                             " an lr_schedule: build the trainer the same way")
        if (sd.get("max_grad_norm") is None) != (self.max_grad_norm is None):
            raise ValueError("optimizer state saved " + ("without" if sd.get("max_grad_norm") is None else "with") +
                             " max_grad_norm: build the trainer the same way")
        arena = self.engine.arena
        for k, key in (("m", "exp_avg"), ("v", "exp_avg_sq")):
            if k in self.opt_state:        # in place: captured graphs hold these buffers
                self.opt_state[k].zero_()
            else:
                self.opt_state[k] = torch.zeros_like(arena.param)
            arena.load_state_dict(sd[key], base=self.opt_state[k])
        self.step_count = int(sd["step"])
        skipped = int(sd.get("skipped_steps", 0))
        self._step_dev.fill_(self.step_count - skipped)     # the device count counts applied steps
        self._step_dev_val = self.step_count
        if self.lr_schedule is not None:
            self.set_lr_schedule(LRSchedule.from_dict(sd["lr_schedule"]))
        if self.max_grad_norm is not None:
            self.set_max_grad_norm(sd["max_grad_norm"])
            self._guard_field("skipped", skipped, dtype=torch.int32)
        self._epoch = int(sd["dropout_epoch"])
        if self.dropout_epoch:
            with _dev_guard(self.device):
                L.call("egot2_dropout_epoch_set", self._epoch, _cur_stream(self.device))


class _PromptStepGraphs(_OptimizerState):
    """Optional CUDA-graph replay of an EgoT2-g step's forward/backward launch sequence (several hundred small eager
    launches per step otherwise).  On by default since it ran green on hardware (round 2); EGOT2_G_GRAPH=0 keeps eager
    launches.  One graph per `graph_key` (= one fixed set of input
    buffers); the captured kernels keep their dropout seeds, the library's device-resident dropout epoch (advanced once per
    step) gives every replay fresh masks; gradient all-reduce (N > 1) and the fused Adam / AdamW stay eager launches behind
    the replay, which also leaves the gradient arena cleared and the bf16 shadow current for the next replay."""

    def _init_step_graphs(self):
        import os
        g = os.environ.get("EGOT2_G_GRAPH", "auto")          # "1" on, "0" off, default: on for CUDA devices
        self.use_graphs = g == "1" or (g == "auto" and torch.device(self.device).type == "cuda")
        self._graphs: Dict[int, tuple] = {}
        self._grad_clean = False
        self.dropout_epoch = self.use_graphs and os.environ.get("EGOT2_DROPOUT_EPOCH", "1") != "0"
        if self.dropout_epoch:
            with _dev_guard(self.device):      # the slot and the per-translation-unit pointers are per device
                L.call("egot2_dropout_epoch_enable", 1)
                L.call("egot2_dropout_epoch_set", 0, _cur_stream(self.device))

    def _capture_graph(self, body):
        """body(): forward/backward launches accumulating into a CLEAN gradient arena, returns the loss tensor."""
        cur = torch.cuda.current_stream(self.device)
        s = torch.cuda.Stream(device=self.device)
        s.wait_stream(cur)
        with torch.cuda.stream(s):                       # warm-up: buffer allocation, workspace sizing
            body()
        cur.wait_stream(s)
        arena = self.engine.arena
        arena.grad.zero_()
        if self.engine.dtype == "bf16":
            arena.refresh_shadow()
            arena.shadow_fresh = True
        torch.cuda.synchronize(self.device)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            total = body()
        return g.replay, total

    def _graph_step(self, body, graph_key: int, decoupled: bool):
        arena = self.engine.arena
        entry = self._graphs.get(graph_key)
        if entry is None:
            entry = self._graphs[graph_key] = self._capture_graph(body)
        replay, total = entry
        if not self._grad_clean:
            arena.grad.zero_()
        if self.engine.dtype == "bf16" and not arena.shadow_fresh:
            arena.refresh_shadow()
        replay()
        if getattr(self, "peer", None) is not None:
            self.peer.step(self.opt_state, self.step_count, self.hp, _cur_stream(self.device), decoupled=decoupled,
                           **self._advance_eager())
        else:
            scale = 1.0
            if self.world > 1:
                scale = allreduce_gradients(arena.grad, self.pg)
            self.engine.adam_step(self.opt_state, self.step_count, self.hp["lr"], self.hp["betas"], self.hp["eps"],
                                  self.hp["weight_decay"], grad_scale=scale, fused=True, decoupled=decoupled,
                                  **self._advance_eager())
        self._grad_clean = True
        if self.dropout_epoch:
            with _dev_guard(self.device):
                L.call("egot2_dropout_epoch_advance", _cur_stream(self.device))
            self._epoch += 1
        return total


class PromptTranslatorTrainer(_PromptStepGraphs):
    """EgoT2-g training step (HHI/tasks/multitask/video_tasktranslation.py:39-66): THREE forwards of one shared model
    per step - 'lam' (LAM tokens only), 'ttm' (lam+ttm+asd tokens) and 'asd' (same encoder, 3-token memory per frame) -
    an unweighted CE over the 7-word vocabulary at the two answer positions of each, loss = sum_i ratio_i * loss_i,
    one backward into ONE gradient arena, [DP: one all-reduce], one fused Adam launch.

    Step inputs: feats = [lam | lam, ttm, asd (ttm batch) | lam, ttm, asd (asd batch)] (7 tensors),
                 labels = the three (rows_i, 3) target-token tensors concatenated along rows."""

    def __init__(self, hidden=256, heads=4, layers=3, dropout=0.1, device="cuda:0", dtype: str = "bf16", lr: float = 5e-4,
                 ratios=(1.0, 1.0, 1.0), process_group=None, lr_schedule: Optional[LRSchedule] = None,
                 max_grad_norm: Optional[float] = None):
        from .hhi import PositionalEncoding
        from .specs import hhi_g_spec
        self.device = torch.device(device)
        self.specs = {m: hhi_g_spec(hidden, heads, layers, dropout, m) for m in ("lam", "ttm", "asd")}
        self.spec = self.specs["ttm"]
        self.engine = TranslatorEngine(self.specs["ttm"], self.device, dtype)
        self.engines = {"ttm": self.engine}
        for m in ("lam", "asd"):
            self.engines[m] = TranslatorEngine(self.specs[m], self.device, dtype, arena=self.engine.arena)
        pe = PositionalEncoding(hidden).pe
        for e in self.engines.values():
            e.set_sinusoid(pe)
        self.ratios = ratios
        self.hp = dict(lr=lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0)
        self.opt_state: Dict[str, torch.Tensor] = {}
        self.step_count = 0
        self.pg = process_group
        self.world = 1
        if process_group is not None or (torch.distributed.is_available() and torch.distributed.is_initialized()):
            self.world = torch.distributed.get_world_size(process_group)
        self.peer = _make_peer_exchange(self.engine, process_group, self.world)
        self._init_step_graphs()           # one CUDA graph per step unless EGOT2_G_GRAPH=0
        self._branch_streams = self._branch_grads = None
        if os.environ.get("EGOT2_G_STREAMS", "1") != "0" and self.device.type == "cuda":
            self._branch_streams = {m: torch.cuda.Stream(device=self.device) for m in ("lam", "asd")}
            self._branch_grads = {m: torch.zeros_like(self.engine.arena.grad) for m in ("lam", "asd")}
        self._h2d: Dict[int, List[torch.Tensor]] = {}
        self.copy_stream = torch.cuda.Stream(device=self.device)
        self.loss_kind, self.class_weight = L.LOSS_CE, None
        self._init_optimizer_state(lr_schedule, lr, 5e-4, max_grad_norm)

    def load_state_dict(self, sd):
        self.engine.arena.load_state_dict(sd)

    def _fwd_bwd_all(self, feats, labels, seed0: int):
        """The three forward/backward passes into a clean gradient arena (the graph-captured body).

        The three passes are independent until their gradients meet, and each is a chain of several hundred tiny kernels
        (7 / 90 / 90 tokens x at most 64 clips) that leave most of the GPU idle: they run SIDE BY SIDE on three streams
        (three parallel branches of the CUDA graph).  The shared arena's accumulation is not atomic everywhere, so 'lam' and
        'asd' write their gradients to buffers of their own, and one launch (egot2_sum_into_f32) adds both into the arena
        and clears them.  EGOT2_G_STREAMS=0: one after the other on the caller's stream."""
        groups = {"lam": list(feats[0:1]), "ttm": list(feats[1:4]), "asd": list(feats[4:7])}
        import contextlib
        par = self._branch_streams is not None
        cur = torch.cuda.current_stream(self.device) if par else None
        off, total, losses = 0, None, []
        for mi, (ratio, mode) in enumerate(zip(self.ratios, ("lam", "ttm", "asd"))):
            rows = groups[mode][0].shape[0] * (groups[mode][0].shape[1] if mode == "asd" else 1)
            tgt = labels[off:off + rows]
            off += rows
            eng = self.engines[mode]
            side = par and mode != "ttm"
            if side:
                self._branch_streams[mode].wait_stream(cur)
            with (torch.cuda.stream(self._branch_streams[mode]) if side else contextlib.nullcontext()):
                act = eng.forward(groups[mode], training=True, seed=seed0 + mi, labels=tgt[:, 1:], loss=L.LOSS_CE,
                                  persistent=True, prompt=tgt[:, :-1])
                eng.backward(act, dloss_scale=float(ratio), zero_grad=False, grad=self._branch_grads[mode] if side else None)
            losses.append((act.t["loss"], ratio))
        if par:
            for mode in ("lam", "asd"):
                cur.wait_stream(self._branch_streams[mode])
            g = self.engine.arena.grad
            with _dev_guard(self.device):
                L.call("egot2_sum_into_f32", g.data_ptr(), self._branch_grads["lam"].data_ptr(),
                       self._branch_grads["asd"].data_ptr(), g.numel(), _cur_stream(self.device))
        for lt, ratio in losses:
            l = lt[0] * ratio
            total = l if total is None else total + l
        return total

    def train_step(self, feats: Sequence[torch.Tensor], labels: torch.Tensor, graph_key: Optional[int] = None):
        self.step_count += 1
        if self.use_graphs and graph_key is not None:
            return self._graph_step(lambda: self._fwd_bwd_all(feats, labels, 4 * (abs(graph_key) + 1)), graph_key, False)
        if not self._grad_clean:
            self.engine.arena.grad.zero_()
        total = self._fwd_bwd_all(feats, labels, self.step_count * 4)         # one arena, accumulated over the three
        if self.peer is not None:
            self.peer.step(self.opt_state, self.step_count, self.hp, _cur_stream(self.device), **self._advance_eager())
            self._grad_clean = True
            return total
        scale = 1.0
        if self.world > 1:
            scale = allreduce_gradients(self.engine.arena.grad, self.pg)
        sched = self._advance_eager()      # a schedule needs the fused launch (the one that reads the device lr)
        self.engine.adam_step(self.opt_state, self.step_count, self.hp["lr"], self.hp["betas"], self.hp["eps"],
                              self.hp["weight_decay"], grad_scale=scale, fused=bool(sched), **sched)
        self._grad_clean = bool(sched)     # the plain Adam launch leaves the gradients in place
        return total

    train_stream_host = None     # bound below to TranslatorTrainer's implementation (same double-buffered host path)


class HoiPromptTranslatorTrainer(_PromptStepGraphs):
    """HOI EgoT2-g training step (Unified3TaskTranslation, HOI/tasks/multitask/video_task.py:182-204): THREE forwards of
    one model per step - a PNR batch, an OSCC batch and an action batch, each the (pnr16, oscc16, slow8, fast8) features
    of its clips plus (B_i, 3) target tokens [task word, answer, answer] - an unweighted CE over the vocabulary at the two
    answer positions, loss = sum_i ratio_i * loss_i, one backward into ONE gradient arena, [DP: one all-reduce], AdamW
    (lr 1e-4, weight decay 1e-4, :265-268; defaults hidden 512 / 8 heads / 3 layers, HOI/configs/multitask/config.py:49-53).

    Step inputs: feats = 3 x [pnr, oscc, slow, fast] (12 tensors), labels = the three target tensors concatenated."""

    def __init__(self, hidden=512, heads=8, layers=3, dropout=0.1, vocab=600, device="cuda:0", dtype: str = "bf16",
                 lr: float = 1e-4, weight_decay: float = 1e-4, ratios=(1.0, 1.0, 1.0), n_tasks: int = 3, process_group=None,
                 lr_schedule: Optional[LRSchedule] = None, max_grad_norm: Optional[float] = None):
        from .hhi import PositionalEncoding
        from .specs import hoi_g_spec
        self.device = torch.device(device)
        self.spec = hoi_g_spec(hidden, heads, layers, dropout, vocab, "clip", n_tasks)
        self.engine = TranslatorEngine(self.spec, self.device, dtype)
        self.engine.set_sinusoid(PositionalEncoding(hidden, max_len=200).pe)
        self.ratios = ratios
        self.hp = dict(lr=lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=weight_decay)
        self.opt_state: Dict[str, torch.Tensor] = {}
        self.step_count = 0
        self.pg = process_group
        self.world = 1
        if process_group is not None or (torch.distributed.is_available() and torch.distributed.is_initialized()):
            self.world = torch.distributed.get_world_size(process_group)
        self.peer = _make_peer_exchange(self.engine, process_group, self.world)
        self._init_step_graphs()           # one CUDA graph per step unless EGOT2_G_GRAPH=0; _grad_clean: True after a fused AdamW
        # the three forward/backward passes of a step side by side (see PromptTranslatorTrainer._fwd_bwd_all): passes 2 and 3 get
        # engines (workspaces, saved activations), streams and gradient arenas of their own; one arena of parameters
        self.engines = [self.engine]
        self._branch_streams = self._branch_grads = None
        if os.environ.get("EGOT2_G_STREAMS", "1") != "0" and self.device.type == "cuda":
            pe = PositionalEncoding(hidden, max_len=200).pe
            for _ in range(2):
                e = TranslatorEngine(self.spec, self.device, dtype, arena=self.engine.arena)
                e.set_sinusoid(pe)
                self.engines.append(e)
            self._branch_streams = [torch.cuda.Stream(device=self.device) for _ in range(2)]
            self._branch_grads = [torch.zeros_like(self.engine.arena.grad) for _ in range(2)]
        self._h2d: Dict[int, List[torch.Tensor]] = {}
        self.copy_stream = None if self.device.type != "cuda" else torch.cuda.Stream(device=self.device)
        self.loss_kind, self.class_weight = L.LOSS_CE, None
        self._init_optimizer_state(lr_schedule, lr, 1e-4, max_grad_norm)

    def load_state_dict(self, sd):
        self.engine.arena.load_state_dict(sd)

    def _fwd_bwd_all(self, feats, labels, seed0: int):
        """The three forward/backward passes into a clean gradient arena (the graph-captured body)."""
        import contextlib
        par = self._branch_streams is not None
        cur = torch.cuda.current_stream(self.device) if par else None
        off, total, losses = 0, None, []
        for i, ratio in enumerate(self.ratios):
            group = list(feats[4 * i:4 * i + 4])
            tgt = labels[off:off + group[0].shape[0]]
            off += group[0].shape[0]
            side = par and i > 0
            eng = self.engines[i] if par else self.engine
            if side:
                self._branch_streams[i - 1].wait_stream(cur)
            with (torch.cuda.stream(self._branch_streams[i - 1]) if side else contextlib.nullcontext()):
                act = eng.forward(group, training=True, seed=seed0 + i, labels=tgt[:, 1:], loss=L.LOSS_CE,
                                  persistent=True, prompt=tgt[:, :-1])
                eng.backward(act, dloss_scale=float(ratio), zero_grad=False, grad=self._branch_grads[i - 1] if side else None)
            losses.append((act.t["loss"], ratio))
        if par:
            for st in self._branch_streams:
                cur.wait_stream(st)
            g = self.engine.arena.grad
            with _dev_guard(self.device):
                L.call("egot2_sum_into_f32", g.data_ptr(), self._branch_grads[0].data_ptr(), self._branch_grads[1].data_ptr(),
                       g.numel(), _cur_stream(self.device))
        for lt, ratio in losses:
            l = lt[0] * ratio
            total = l if total is None else total + l
        return total

    def train_step(self, feats: Sequence[torch.Tensor], labels: torch.Tensor, graph_key: Optional[int] = None):
        assert len(feats) == 12, "three batches x (pnr, oscc, slow, fast)"
        self.step_count += 1
        if self.use_graphs and graph_key is not None:
            return self._graph_step(lambda: self._fwd_bwd_all(feats, labels, 4 * (abs(graph_key) + 1)), graph_key, True)
        eng = self.engine
        off, total = 0, None
        for i, ratio in enumerate(self.ratios):
            group = list(feats[4 * i:4 * i + 4])
            rows = group[0].shape[0]
            tgt = labels[off:off + rows]
            off += rows
            act = eng.forward(group, training=True, seed=self.step_count * 4 + i, labels=tgt[:, 1:], loss=L.LOSS_CE,
                              persistent=True, prompt=tgt[:, :-1])
            # one arena, accumulated over the three; cleared here only if the previous step's optimizer did not
            eng.backward(act, dloss_scale=float(ratio), zero_grad=(i == 0 and not self._grad_clean))
            l = act.t["loss"][0] * ratio
            total = l if total is None else total + l
        if self.peer is not None:
            self.peer.step(self.opt_state, self.step_count, self.hp, _cur_stream(self.device), decoupled=True,
                           **self._advance_eager())
            self._grad_clean = True
            return total
        scale = 1.0
        if self.world > 1:
            scale = allreduce_gradients(eng.arena.grad, self.pg)
        # AdamW (decoupled decay) + bf16 shadow + gradient clear in one launch
        eng.adam_step(self.opt_state, self.step_count, self.hp["lr"], self.hp["betas"], self.hp["eps"],
                      self.hp["weight_decay"], grad_scale=scale, fused=True, decoupled=True, **self._advance_eager())
        self._grad_clean = True
        return total


def default_loss(spec: TranslatorSpec):
    """(loss kind, class weights) the reference task uses for this translator (SURVEY.md F10)."""
    if spec.family == "hhi_ttm":
        return L.LOSS_CE, torch.tensor([0.266, 0.734])
    if spec.family == "hoi_pnr":
        return (L.LOSS_BCE_SIGMOID if spec.n_out == 16 else L.LOSS_CE), None
    if spec.family in ("hoi_lta", "hoi_ar"):
        return L.LOSS_CE_GROUPS, None
    raise ValueError(f"{spec.family}: the loss lives outside the translator (use the nn.Module API)")


class TranslatorTrainer(_OptimizerState):
    def __init__(self, spec: TranslatorSpec, device, dtype: str = "bf16", lr: float = 5e-4, betas=(0.9, 0.999),
                 eps: float = 1e-8, weight_decay: float = 0.0, process_group=None, use_graphs: bool = True,
                 sinusoid: Optional[torch.Tensor] = None, lr_schedule: Optional[LRSchedule] = None,
                 max_grad_norm: Optional[float] = None):
        self.spec = spec
        self.device = torch.device(device)
        self.engine = TranslatorEngine(spec, self.device, dtype)
        if spec.embed == "task_sinusoid":
            if sinusoid is None:
                from .hhi import PositionalEncoding
                sinusoid = PositionalEncoding(spec.hidden).pe
            self.engine.set_sinusoid(sinusoid)
        self.loss_kind, cw = default_loss(spec)
        self.class_weight = None if cw is None else cw.to(self.device)
        self.hp = dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay)
        self.opt_state: Dict[str, torch.Tensor] = {}
        self.step_count = 0
        self.pg = process_group
        self.world = 1
        if process_group is not None or (torch.distributed.is_available() and torch.distributed.is_initialized()):
            self.world = torch.distributed.get_world_size(process_group)
        self.use_graphs = use_graphs
        self._grad_clean = False           # True right after the fused Adam: the gradient arena is all zeros
        # Whole-step graphs (single GPU): the fused Adam is captured behind forward+backward, with the optimizer's step
        # count kept ON THE DEVICE (a counter kernel on a side branch of the graph advances it, the Adam kernel reads
        # it), so one graph launch is one optimisation step.  EGOT2_GRAPH_UPDATE=0 keeps Adam as an eager launch after
        # the replay.
        import os
        gu = os.environ.get("EGOT2_GRAPH_UPDATE", "1")
        # N > 1: capturing torch.distributed's NCCL all-reduce hung on the 2xB200 box (round 1), so the data-parallel step
        # keeps [graph: forward+backward] -> eager all-reduce -> eager fused Adam unless forced with EGOT2_GRAPH_UPDATE=force
        self.graph_update = gu == "force" or (gu != "0" and self.world == 1)
        # N > 1 with graphs: the step is TWO graphs - [forward + backward down to the encoder input] and [embedding
        # backward] - so that the all-reduce of everything but the embedding-stage gradients (arena[embed_numel:],
        # most of the bytes) runs on NCCL's stream WHILE the second graph executes; only the small embedding bucket is
        # reduced after it.  EGOT2_DP_OVERLAP=0: one graph, one all-reduce behind it.
        ov = os.environ.get("EGOT2_DP_OVERLAP", "1")       # "force": also with one rank (tests; needs an initialised group)
        self.dp_overlap = ((self.world > 1 and ov != "0") or ov == "force") and spec.head != "decoder"
        # N > 1, preferred: the exchange as ONE kernel over NVLink peer memory (parallel.PeerExchange / csrc/peer.cu: gradient
        # reduce-scatter + Adam on this rank's slice + parameter all-gather).  No NCCL call and no host launch inside the step,
        # so the whole step is again ONE CUDA graph, exactly like on one GPU.  EGOT2_DP_FUSED=0 keeps the NCCL path above.
        self.peer = _make_peer_exchange(self.engine, process_group, self.world)
        if self.peer is not None:
            self.dp_overlap = False
            self.graph_update = gu != "0"
        if self.dp_overlap:
            self.graph_update = False
        # Graph replays re-run kernels whose dropout keys were frozen at capture: the library's device-resident dropout
        # epoch (advanced once per step, XORed into every key at execution time) gives every replay fresh masks.
        self.dropout_epoch = bool(use_graphs) and os.environ.get("EGOT2_DROPOUT_EPOCH", "1") != "0"
        if self.dropout_epoch:
            with _dev_guard(self.device):
                L.call("egot2_dropout_epoch_enable", 1)
                L.call("egot2_dropout_epoch_set", 0, torch.cuda.current_stream(self.device).cuda_stream)
        self._step_dev = torch.zeros(1, device=self.device, dtype=torch.int32)
        self._step_dev_val = 0
        self._init_optimizer_state(lr_schedule, lr, 5e-4, max_grad_norm)
        self._bump_stream = torch.cuda.Stream(device=self.device)
        self._peer_stream = torch.cuda.Stream(device=self.device)
        self._graphs: Dict[int, tuple] = {}
        self._h2d: Dict[int, List[torch.Tensor]] = {}
        self.copy_stream = torch.cuda.Stream(device=self.device)

    # ------------------------------------------------------------------ parameters
    def load_state_dict(self, sd):
        self.engine.arena.load_state_dict(sd)

    def state_dict(self):
        return self.engine.arena.state_dict()

    # ------------------------------------------------------------------ device-resident step
    def _fwd_bwd(self, feats: Sequence[torch.Tensor], labels: torch.Tensor, seed: int, stage: str = "all") -> Activations:
        act = self.engine.forward(feats, training=True, seed=seed, labels=labels, loss=self.loss_kind,
                                  class_weight=self.class_weight, persistent=True)
        # the fused Adam of the previous step left the gradient arena cleared (and the bf16 shadow current)
        self.engine.backward(act, zero_grad=not self._grad_clean, stage=stage)
        self._grad_clean = False
        return act

    def train_step(self, feats: Sequence[torch.Tensor], labels: torch.Tensor, graph_key: Optional[int] = None):
        """One optimisation step on device-resident features.  Returns the (device) loss tensor.
        graph_key: a stable id for this exact set of input buffers; its launch sequence is captured into a CUDA
        graph on first use.  The captured kernels keep the dropout seed they were captured with; the device-resident
        dropout epoch (advanced once per step, folded into every key at execution time) makes each replay draw fresh
        masks all the same."""
        self.step_count += 1
        if self.dropout_epoch:
            self._epoch += 1               # every path below advances the device epoch once
        if graph_key is not None and self.use_graphs:
            entry = self._graphs.get(graph_key)
            if entry is None:
                entry = self._capture(feats, labels, graph_key)
            if len(entry) == 3:                           # data-parallel, two graphs with the all-reduce in between
                return self._dp_overlap_step(entry)
            graph, act = entry
            if not self._grad_clean:                      # e.g. the first graphed step after eager ones
                self.engine.arena.grad.zero_()
            if self.engine.dtype == "bf16" and not self.engine.arena.shadow_fresh:
                self.engine.arena.refresh_shadow()
            if self.graph_update and self.max_grad_norm is None and self._step_dev_val != self.step_count - 1:
                self._step_dev.fill_(self.step_count - 1)
            graph.replay()
            if self.graph_update:                         # the graph ended with fused Adam (+ the epoch advance)
                self._step_dev_val = self.step_count
                self._grad_clean = True
                self.engine.arena.shadow_fresh = self.engine.dtype == "bf16"
                return act.t["loss"][0]
            self._grad_clean = False
        else:
            act = self._fwd_bwd(feats, labels, seed=self.step_count)
        self._reduce_and_update()
        self._advance_epoch()
        return act.t["loss"][0]

    def _dp_overlap_step(self, entry):
        import torch.distributed as dist
        g1, g2, act = entry
        eng = self.engine
        if not self._grad_clean:
            eng.arena.grad.zero_()
        if eng.dtype == "bf16" and not eng.arena.shadow_fresh:
            eng.arena.refresh_shadow()
        nb = eng.arena.embed_numel
        g1.replay()                                       # forward + backward of head and encoder layers
        work = dist.all_reduce(eng.arena.grad[nb:], group=self.pg, async_op=True)      # overlaps the embedding backward
        g2.replay()
        dist.all_reduce(eng.arena.grad[:nb], group=self.pg)
        work.wait()
        eng.adam_step(self.opt_state, self.step_count, self.hp["lr"], self.hp["betas"], self.hp["eps"],
                      self.hp["weight_decay"], grad_scale=1.0 / self.world, fused=True, **self._advance_eager())
        self._grad_clean = True
        self._advance_epoch()
        return act.t["loss"][0]

    def _capture(self, feats, labels, key):
        # labels are NOT converted here: engine.forward() does it inside the captured region, so a caller's int32 / strided
        # label buffer is re-read (and re-converted) on every replay instead of being frozen at capture-time values
        if self.engine.spec.p_layer > 0 or self.engine.spec.p_embed > 0 or self.engine.spec.p_feat > 0 or self.engine.spec.p_head > 0:
            if not self.dropout_epoch:
                raise L.Egot2Error("graph replay with training dropout needs the device-resident dropout epoch "
                                   "(EGOT2_DROPOUT_EPOCH=0 would replay ONE frozen mask): use use_graphs=False")
        # warm-up on a side stream (allocations, workspace sizing), then capture
        s = torch.cuda.Stream(device=self.device)
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            self._fwd_bwd(feats, labels, seed=self._graph_seed(key))
        torch.cuda.current_stream().wait_stream(s)
        # the captured sequence is the steady state: shadow current and gradient arena cleared by the previous step's
        # fused Adam, so neither the cast nor the fill is part of the graph
        self.engine.arena.grad.zero_()
        if self.engine.dtype == "bf16":
            self.engine.arena.refresh_shadow()
            self.engine.arena.shadow_fresh = True
        self._grad_clean = True
        if self.graph_update:
            if "m" not in self.opt_state:                 # optimizer state must exist before capture
                self.opt_state["m"] = torch.zeros_like(self.engine.arena.param)
                self.opt_state["v"] = torch.zeros_like(self.engine.arena.param)
            if self.world > 1 and self.peer is None:      # communicator warm-up outside the capture (grad arena is zero)
                allreduce_gradients(self.engine.arena.grad, self.pg)
            if self.max_grad_norm is None:             # with a guard the device count is authoritative (skips)
                self._step_dev.fill_(self.step_count - 1)
            self._step_dev_val = self.step_count - 1
        if self.dp_overlap and not self.graph_update:
            torch.cuda.synchronize(self.device)
            g1, g2 = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
            with torch.cuda.graph(g1):
                act = self._fwd_bwd(feats, labels, seed=self._graph_seed(key), stage="pre_embed")
            with torch.cuda.graph(g2, pool=g1.pool()):
                self.engine.backward(act, zero_grad=False, stage="embed")
            self._graphs[key] = (g1, g2, act)
            return self._graphs[key]
        torch.cuda.synchronize(self.device)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            cur = torch.cuda.current_stream(self.device)
            if self.graph_update:                         # side branch: advance the device-resident step count
                self._bump_stream.wait_stream(cur)
                with torch.cuda.stream(self._bump_stream):
                    if self.lr_schedule is not None:      # ... and the lr of that step
                        self._opt_advance(self._bump_stream.cuda_stream)
                    else:
                        self._step_dev.add_(1)
            split = self.graph_update and self.peer is not None and self.engine.spec.head != "decoder" \
                and os.environ.get("EGOT2_DP_SPLIT", "0") == "1"
            if split:
                # peer-memory exchange in two pieces: everything but the embedding-stage parameters (most of the bytes) is
                # reduced + updated + gathered on a side stream WHILE the embedding backward runs (it reads only prefix
                # parameters), the small embedding prefix right after it
                act = self._fwd_bwd(feats, labels, seed=self._graph_seed(key), stage="pre_embed")
                cur.wait_stream(self._bump_stream)            # the step count both exchange launches read
                nb, n = self.engine.arena.embed_numel, self.engine.arena.numel
                self._peer_stream.wait_stream(cur)
                with torch.cuda.stream(self._peer_stream):
                    self.peer.step(self.opt_state, self.step_count, self.hp, self._peer_stream.cuda_stream,
                                   step_dev=self._step_dev, lo=nb, hi=n, channel=0, lr_dev=self._graph_lr_dev())
                self.engine.backward(act, zero_grad=False, stage="embed")
                self._bump_stream.wait_stream(cur)
                with torch.cuda.stream(self._bump_stream):
                    self._advance_epoch()
                self.peer.step(self.opt_state, self.step_count, self.hp, cur.cuda_stream, step_dev=self._step_dev,
                               lo=0, hi=nb, channel=1, lr_dev=self._graph_lr_dev())
                cur.wait_stream(self._peer_stream)
                cur.wait_stream(self._bump_stream)
                self._grad_clean = True
                self._graphs[key] = (g, act)
                return g, act
            act = self._fwd_bwd(feats, labels, seed=self._graph_seed(key))
            if self.graph_update:
                cur.wait_stream(self._bump_stream)
                # every dropout consumer of this step has been enqueued before this point: the epoch advances for the
                # NEXT replay on the side branch, beside the Adam launch (which reads no dropout key)
                self._bump_stream.wait_stream(cur)
                with torch.cuda.stream(self._bump_stream):
                    self._advance_epoch()
                self._reduce_and_update(step_dev=self._step_dev)
                cur.wait_stream(self._bump_stream)
        self._graphs[key] = (g, act)
        return g, act

    @staticmethod
    def _graph_seed(key: int) -> int:
        """Dropout seed a graph is captured with: positive, distinct for every key (device pool keys are >= 0, the host
        path's double-buffer slots are -(slot + 1))."""
        return 2 * abs(int(key)) + (1 if key >= 0 else 2) + 1000

    def _advance_epoch(self):
        if self.dropout_epoch:
            with _dev_guard(self.device):
                L.call("egot2_dropout_epoch_advance", torch.cuda.current_stream(self.device).cuda_stream)      # current = the stream in effect

    def _graph_lr_dev(self) -> Optional[torch.Tensor]:
        """lr_dev of an optimizer launch inside the whole-step graph (advanced on its side branch), None without a schedule."""
        return None if self.lr_schedule is None else self._lr_dev

    def _reduce_and_update(self, step_dev: Optional[torch.Tensor] = None):
        """step_dev: the launch sits in the whole-step graph, whose side branch advances the step count (and lr).  With a
        guard, the norm launch follows the all-reduce (engine.adam_step) or is part of the peer exchange."""
        eng = self.engine
        opt = self._advance_eager() if step_dev is None else self._opt_args(step_dev)
        if self.peer is not None:                         # one kernel: reduce-scatter + Adam + all-gather over peer memory
            self.peer.step(self.opt_state, self.step_count, self.hp, torch.cuda.current_stream(self.device).cuda_stream,
                           **opt)
            self._grad_clean = True
            return
        scale = 1.0
        if self.world > 1:
            scale = allreduce_gradients(eng.arena.grad, self.pg)            # ONE flat NCCL all-reduce (NVLink)
        eng.adam_step(self.opt_state, self.step_count, self.hp["lr"], self.hp["betas"], self.hp["eps"],
                      self.hp["weight_decay"], grad_scale=scale, fused=True, **opt)
        self._grad_clean = True

    # ------------------------------------------------------------------ host-buffer (end-to-end) step
    def train_step_host(self, host_feats: Sequence[torch.Tensor], host_labels: torch.Tensor, slot: int = 0) -> float:
        """End-to-end step from pinned HOST buffers: H2D copy of the features + labels, the step, and a D2H read
        of the loss.  Device staging buffers are double-buffered per `slot`."""
        bufs = self._h2d.get(slot)
        if bufs is None:
            bufs = [torch.empty(f.shape, device=self.device, dtype=f.dtype) for f in host_feats]
            bufs.append(torch.empty(host_labels.shape, device=self.device, dtype=torch.int64))
            self._h2d[slot] = bufs
        for b, f in zip(bufs[:-1], host_feats):
            b.copy_(f, non_blocking=True)
        bufs[-1].copy_(host_labels, non_blocking=True)
        loss = self.train_step(bufs[:-1], bufs[-1], graph_key=-(slot + 1) if self.use_graphs else None)
        return float(loss.item())

    def train_stream_host(self, host_batches, n_steps: int) -> List[float]:
        """End-to-end training over a stream of pinned HOST batches [(feats..., labels)], double-buffered: the H2D
        copy of step i+1 runs on a copy stream while step i computes, and every step's loss comes back with an
        asynchronous D2H copy that is only read at the end.  Every step still pays its own H2D + D2H."""
        cur = torch.cuda.current_stream(self.device)
        ev_h2d = [torch.cuda.Event() for _ in range(2)]
        ev_done = [torch.cuda.Event() for _ in range(2)]
        if not hasattr(self, "_loss_host") or self._loss_host.numel() < n_steps:
            self._loss_host = torch.empty(max(n_steps, 1), dtype=torch.float32).pin_memory()
        for i in range(n_steps):
            slot = i % 2
            host_feats, host_labels = host_batches[i % len(host_batches)]
            bufs = self._h2d.get(slot)
            if bufs is None:
                # allocate ON the copy stream: a block the caching allocator recycles from the compute stream may still
                # be in use by kernels in flight there, and the copy stream would overwrite it without waiting
                with torch.cuda.stream(self.copy_stream):
                    bufs = [torch.empty(f.shape, device=self.device, dtype=f.dtype) for f in host_feats]
                    bufs.append(torch.empty(host_labels.shape, device=self.device, dtype=torch.int64))
                self._h2d[slot] = bufs
            with torch.cuda.stream(self.copy_stream):
                if i >= 2:
                    self.copy_stream.wait_event(ev_done[slot])      # the step that last used this slot has finished
                for b, f in zip(bufs[:-1], host_feats):
                    b.copy_(f, non_blocking=True)
                bufs[-1].copy_(host_labels, non_blocking=True)
                ev_h2d[slot].record(self.copy_stream)
            cur.wait_event(ev_h2d[slot])
            loss = self.train_step(bufs[:-1], bufs[-1], graph_key=-(slot + 1) if self.use_graphs else None)
            self._loss_host[i:i + 1].copy_(loss.reshape(1), non_blocking=True)
            ev_done[slot].record(cur)
        cur.synchronize()
        return self._loss_host[:n_steps].tolist()

    # ------------------------------------------------------------------ inference
    @torch.no_grad()
    def infer(self, feats: Sequence[torch.Tensor]) -> torch.Tensor:
        act = self.engine.forward(feats, training=False, persistent=True)
        return act.t["out"]


PromptTranslatorTrainer.train_stream_host = TranslatorTrainer.train_stream_host
HoiPromptTranslatorTrainer.train_stream_host = TranslatorTrainer.train_stream_host
