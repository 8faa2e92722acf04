"""Learning-rate schedules of the fused trainers (trainer.py), evaluated ON THE DEVICE.

A trainer's step is one CUDA-graph replay with no host work in between, and its optimizer step count already lives on the
device.  So the lr lives there too: `egot2_opt_advance` advances the step count and writes the lr of that step from a
device-resident `egot2_lr_sched` descriptor (include/egot2.h, where lr_at is defined), and the Adam / AdamW / peer-exchange
kernels read it when they execute.  `LRSchedule` is the host description of that descriptor; it validates and packs, and
deliberately does not evaluate the schedule (the only host restatement of lr_at is in the tests).

The policies are the SlowFast-style ones the HOI configs select (SURVEY.md §2.2, §3.5: Adam + warm-up cosine,
HOI/optimizers/lta/lr_scheduler.py:21-26,67-91): 'constant', 'cosine' (with end_lr), 'steps' (steps with relative lrs), each
with an optional linear warm-up.  Steps are optimizer steps; callers that think in epochs convert.
"""
from __future__ import annotations

import dataclasses
from dataclasses import dataclass
from typing import Sequence, Tuple

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
