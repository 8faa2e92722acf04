"""Learning-rate schedules of the fused trainers (trainer.py), evaluated ON THE DEVICE.

A trainer's step is one CUDA-graph replay with no host work in between, and its optimizer step count already lives on the
device.  So the lr lives there too: `egot2_opt_advance` advances the step count and writes the lr of that step from a
device-resident `egot2_lr_sched` descriptor (include/egot2.h, where lr_at is defined), and the Adam / AdamW / peer-exchange
kernels read it when they execute.  `LRSchedule` is the host description of that descriptor; it validates and packs, and
deliberately does not evaluate the schedule (the only host restatement of lr_at is in the tests).

The policies are the SlowFast-style ones the HOI configs select (SURVEY.md §2.2, §3.5: Adam + warm-up cosine,
HOI/optimizers/lta/lr_scheduler.py:21-26,67-91): 'constant', 'cosine' (with end_lr), 'steps' (steps with relative lrs), each
with an optional linear warm-up.  Steps are optimizer steps; callers that think in epochs convert.

`ParamGroup` is the fused trainers' form of torch.optim's param groups (per-group weight decay and lr multiplier, frozen
parameters).  They are applied per element by the optimizer kernels, from a device-resident `egot2_param_groups` descriptor
and a map of one group per 64-element block of the parameter arena (include/egot2.h); `resolve_param_groups` builds both.

`SGD` selects torch.optim.SGD (momentum, dampening, Nesterov) instead of Adam / AdamW for a fused trainer
(egot2_sgd_step_fused, egot2_dp_desc.sgd): SlowFast's construct_optimizer builds it beside Adam and AdamW (HOI/optimizers/).

`WeightAverage` selects an averaged copy of the weights (torch.optim.swa_utils.AveragedModel: EMA or SWA), kept by one
egot2_weight_avg_update launch after every optimizer launch.
"""
from __future__ import annotations

import dataclasses
import fnmatch
import math
from dataclasses import dataclass
from typing import Dict, Mapping, Optional, Sequence, Tuple

import numpy as np

from . import _lib as L


@dataclass(frozen=True)
class LRSchedule:
    """lr of optimizer step t (1-based) = lr_at(t - 1), see include/egot2.h.  Build with the constructors below."""
    kind: int
    base_lr: float
    total_steps: int = 0
    end_lr: float = 0.0
    warmup_steps: int = 0
    warmup_start_lr: float = 0.0
    milestones: Tuple[int, ...] = ()
    factors: Tuple[float, ...] = ()

    @classmethod
    def constant(cls, lr: float) -> "LRSchedule":
        return cls(L.LR_CONSTANT, float(lr))

    @classmethod
    def cosine(cls, base_lr: float, total_steps: int, end_lr: float = 0.0, warmup_steps: int = 0,
               warmup_start_lr: float = 0.0) -> "LRSchedule":
        """end_lr + (base_lr - end_lr) * (1 + cos(pi * s / total_steps)) / 2, held at end_lr from s = total_steps on."""
        return cls(L.LR_COSINE, float(base_lr), int(total_steps), float(end_lr), int(warmup_steps), float(warmup_start_lr))

    @classmethod
    def steps(cls, base_lr: float, milestones: Sequence[int], factors: Sequence[float], warmup_steps: int = 0,
              warmup_start_lr: float = 0.0) -> "LRSchedule":
        """base_lr * factors[i], i = the number of milestones <= s (MultiStepLR: factors[i] = gamma ** i)."""
        return cls(L.LR_STEPS, float(base_lr), 0, 0.0, int(warmup_steps), float(warmup_start_lr),
                   tuple(int(m) for m in milestones), tuple(float(f) for f in factors))

    def __post_init__(self):
        if self.kind not in (L.LR_CONSTANT, L.LR_COSINE, L.LR_STEPS):
            raise ValueError(f"LRSchedule: unknown kind {self.kind}")
        if self.warmup_steps < 0:
            raise ValueError("LRSchedule: warmup_steps must be >= 0")
        if self.kind == L.LR_COSINE and self.total_steps <= 0:
            raise ValueError("LRSchedule.cosine: total_steps must be positive")
        if self.kind == L.LR_STEPS:
            ms = self.milestones
            if len(ms) > L.LR_MAX_MILESTONES:
                raise ValueError(f"LRSchedule.steps: at most {L.LR_MAX_MILESTONES} milestones")
            if any(b <= a for a, b in zip(ms, ms[1:])) or any(m < 0 for m in ms):
                raise ValueError("LRSchedule.steps: milestones must be non-negative and strictly increasing")
            if len(self.factors) != len(ms) + 1:
                raise ValueError("LRSchedule.steps: factors must have exactly one entry more than milestones")
        elif self.milestones or self.factors:
            raise ValueError("LRSchedule: milestones / factors belong to the 'steps' schedule only")

    def pack(self) -> L.LrSched:
        """The egot2_lr_sched this schedule is on the device."""
        d = L.LrSched()
        d.kind, d.n_milestones = self.kind, len(self.milestones)
        d.warmup_steps, d.total_steps = self.warmup_steps, self.total_steps
        d.base_lr, d.warmup_start_lr, d.end_lr = self.base_lr, self.warmup_start_lr, self.end_lr
        for i, m in enumerate(self.milestones):
            d.milestones[i] = m
        for i, f in enumerate(self.factors):
            d.factors[i] = f
        return d

    def to_dict(self) -> dict:
        """Plain fields (ints, floats, tuples) for a checkpoint that torch.load(weights_only=True) reads back."""
        return dataclasses.asdict(self)

    @classmethod
    def from_dict(cls, d: dict) -> "LRSchedule":
        return cls(**{**d, "milestones": tuple(d["milestones"]), "factors": tuple(d["factors"])})


def check_group_hp(name: str, x: float) -> float:
    x = float(x)
    if not (math.isfinite(x) and x >= 0.0):
        raise ValueError(f"ParamGroup: {name} must be finite and >= 0, got {x}")
    return x


@dataclass(frozen=True)
class ParamGroup:
    """One optimizer parameter group of a fused trainer (trainer.py): the parameters whose reference state_dict names
    (spec.param_shapes() keys) match one of `patterns` (fnmatch).  Their lr is the trainer's lr (fixed or scheduled) times
    lr_mult; weight_decay None inherits the trainer's; frozen is requires_grad=False (parameters and moments stay as they
    are, and the gradient stays out of the max_grad_norm norm).  A parameter joins the first group that matches it;
    unmatched parameters form group 0 with lr_mult 1 and the trainer's weight_decay."""
    patterns: Tuple[str, ...]
    lr_mult: float = 1.0
    weight_decay: Optional[float] = None
    frozen: bool = False

    def __post_init__(self):
        pats = (self.patterns,) if isinstance(self.patterns, str) else tuple(self.patterns)
        if not pats or not all(isinstance(p, str) for p in pats):
            raise ValueError(f"ParamGroup: patterns must be one or more strings, got {self.patterns!r}")
        object.__setattr__(self, "patterns", pats)
        object.__setattr__(self, "lr_mult", check_group_hp("lr_mult", self.lr_mult))
        if self.weight_decay is not None:
            object.__setattr__(self, "weight_decay", check_group_hp("weight_decay", self.weight_decay))
        object.__setattr__(self, "frozen", bool(self.frozen))


def resolve_param_groups(groups: Sequence[ParamGroup], shapes: Mapping[str, Tuple[int, ...]], offsets: Mapping[str, int],
                         numel: int, block: int = 64) -> np.ndarray:
    """The uint8 map of one group per `block`-element block of an arena of `numel` elements with these offsets: a parameter's
    group is the first ParamGroup with a pattern that matches its name.  Group 0 is the default group, groups[i] is group
    i + 1.  Raises ValueError for a pattern that matches nothing, more than MAX_PARAM_GROUPS groups, or two parameters of
    different groups in one block."""
    if len(groups) + 1 > L.MAX_PARAM_GROUPS:
        raise ValueError(f"at most {L.MAX_PARAM_GROUPS} parameter groups, the default group included: got {len(groups) + 1}")
    names = list(shapes)
    for g in groups:
        for pat in g.patterns:
            if not fnmatch.filter(names, pat):
                raise ValueError(f"ParamGroup pattern {pat!r} matches no parameter")
    index = []
    for n in names:
        index.append(next((i + 1 for i, g in enumerate(groups) if any(fnmatch.fnmatchcase(n, p) for p in g.patterns)), 0))
    group_of = dict(zip(names, index))
    bmap = np.zeros((numel + block - 1) // block, dtype=np.uint8)
    edge: Dict[int, str] = {}                 # first / last block of a parameter -> the parameter that claimed it
    for n, k in zip(names, index):
        size = int(np.prod(shapes[n], dtype=np.int64))
        if size == 0:
            continue
        b0, b1 = offsets[n] // block, (offsets[n] + size - 1) // block
        for b in {b0, b1}:                     # only a first or last block can be shared (parameters do not overlap)
            other = edge.setdefault(b, n)
            if group_of[other] != k:
                raise ValueError(f"parameters {other!r} (group {group_of[other]}) and {n!r} (group {k}) share a "
                                 f"{block}-element block of the arena and must be in the same parameter group")
        bmap[b0:b1 + 1] = k
    return bmap


def pack_param_groups(hp: Sequence[Tuple[float, float, bool]]) -> L.ParamGroups:
    """The egot2_param_groups of (lr_mult, weight_decay, frozen) per group."""
    d = L.ParamGroups()
    d.n_groups = len(hp)
    for i, (lr_mult, wd, frozen) in enumerate(hp):
        d.lr_mult[i], d.weight_decay[i], d.frozen[i] = lr_mult, wd, int(frozen)
    return d


@dataclass(frozen=True)
class SGD:
    """torch.optim.SGD(momentum, dampening, nesterov) for a fused trainer's `optimizer=`; lr and weight decay stay the trainer's
    (lr / lr_schedule, weight_decay, param_groups).  The checks are torch's: momentum >= 0, dampening finite, Nesterov needs
    momentum > 0 and dampening 0.  SlowFast's SGD default is SGD(momentum=0.9, nesterov=True) with weight_decay 1e-4."""
    momentum: float = 0.0
    dampening: float = 0.0
    nesterov: bool = False

    def __post_init__(self):
        momentum, dampening = float(self.momentum), float(self.dampening)
        if not (math.isfinite(momentum) and momentum >= 0.0):
            raise ValueError(f"SGD: momentum must be finite and >= 0, got {momentum}")
        if not math.isfinite(dampening):
            raise ValueError(f"SGD: dampening must be finite, got {dampening}")
        if self.nesterov and (momentum <= 0.0 or dampening != 0.0):
            raise ValueError("SGD: Nesterov momentum requires a momentum and zero dampening")
        object.__setattr__(self, "momentum", momentum)
        object.__setattr__(self, "dampening", dampening)
        object.__setattr__(self, "nesterov", bool(self.nesterov))

    def to_dict(self) -> dict:
        return dataclasses.asdict(self)


_INT32_MAX = 2 ** 31 - 1


@dataclass(frozen=True)
class WeightAverage:
    """An averaged copy of a fused trainer's parameters (`weight_average=`), updated on the device by egot2_weight_avg_update
    after every due step: torch.optim.swa_utils.AveragedModel fed with the trainer's parameters.  Step t (the optimizer's
    applied-step count, 1-based) is due when t >= start and (t - start) % every == 0; the first due step copies the
    parameters, every later one lerps towards them.  Build with the constructors below."""
    kind: int
    decay: float = 0.0
    every: int = 1
    start: int = 1

    @classmethod
    def ema(cls, decay: float = 0.999, every: int = 1, start: int = 1) -> "WeightAverage":
        """AveragedModel(multi_avg_fn=get_ema_multi_avg_fn(decay)): avg = lerp(avg, param, 1 - decay)."""
        return cls(L.AVG_EMA, decay, every, start)

    @classmethod
    def swa(cls, every: int = 1, start: int = 1) -> "WeightAverage":
        """AveragedModel() with its default average: the equal-weight running mean of the parameters on the due steps."""
        return cls(L.AVG_SWA, 0.0, every, start)

    def __post_init__(self):
        if self.kind not in (L.AVG_EMA, L.AVG_SWA):
            raise ValueError(f"WeightAverage: unknown kind {self.kind!r}")
        try:
            decay = float(self.decay)
        except (TypeError, ValueError):
            decay = math.nan
        if not (math.isfinite(decay) and 0.0 <= decay <= 1.0):
            raise ValueError(f"WeightAverage: decay must be finite and in [0, 1], got {self.decay!r}")
        for name in ("every", "start"):
            v = getattr(self, name)
            if isinstance(v, bool) or not isinstance(v, (int, np.integer)) or not 0 < int(v) <= _INT32_MAX:
                raise ValueError(f"WeightAverage: {name} must be a positive int that fits in int32, got {v!r}")
            object.__setattr__(self, name, int(v))
        object.__setattr__(self, "decay", decay)

    @property
    def ema_weight(self) -> float:
        """The lerp weight of an EMA update, float(1 - decay) with the subtraction in double as torch does it (0 for SWA,
        whose weight the kernel computes from the update count)."""
        return 1.0 - self.decay if self.kind == L.AVG_EMA else 0.0

    def to_dict(self) -> dict:
        return dataclasses.asdict(self)

    @classmethod
    def from_dict(cls, d: dict) -> "WeightAverage":
        return cls(**{k: d[k] for k in ("kind", "decay", "every", "start")})
