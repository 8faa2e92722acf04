"""Per-parameter gradient and weight statistics of the fused trainers (trainer.py, `param_stats=`), computed on the device.

The reference logs histograms of every weight and of every gradient each LOG_GRADIENT_PERIOD steps (an `on_after_backward`
hook calling SummaryWriter.add_histogram, HOI/tasks/lta/video_task.py:112-125), and Lightning users log per-parameter
gradient norms (lightning.pytorch.utilities.grad_norm).  The fused trainers apply and clear the gradient arena inside their
optimizer launch, so nothing is left to inspect after a step.  Instead, on a due step one launch (egot2_param_stats,
include/egot2.h) right before the optimizer reduces the gradient the optimizer applies and the parameters before the update
to what TensorBoard needs: num, min, max, sum, sum of squares, the non-finite count, the L2 norm and the bucket counts over
TensorBoard's default edges.

This module owns that histogram format: `ParamStats` (the trainers' option), the default edges, the work units of the
launch, and the host-side trimming that turns bucket counts into `SummaryWriter.add_histogram_raw` arguments equal to what
`add_histogram(tag, tensor)` writes.
"""
from __future__ import annotations

import ctypes as C
import numbers
from dataclasses import dataclass
from typing import Mapping, Optional, Sequence, Tuple

import numpy as np

from . import _lib as L

# elements per work unit: big enough that the per-unit histogram flush is small next to the unit's reads, small enough that
# the 28 M-element HOI LTA arena spreads over every SM
UNIT_ELEMS = 32768


@dataclass(frozen=True)
class ParamStats:
    """Statistics of every parameter and of every trainable gradient on the optimizer steps t (1-based) with
    (t - 1) % every == 0 (Lightning's global_step % every == 0 before optimizer.step()); histograms=False keeps the norms and
    moments only."""
    every: int
    histograms: bool = True

    def __post_init__(self):
        if isinstance(self.every, bool) or not isinstance(self.every, numbers.Integral) or self.every <= 0:
            raise ValueError(f"ParamStats: every must be a positive int, got {self.every!r}")
        object.__setattr__(self, "every", int(self.every))
        object.__setattr__(self, "histograms", bool(self.histograms))


def default_edges() -> np.ndarray:
    """TensorBoard's default histogram bucket edges (SummaryWriter.default_bins), with the same loop, so the doubles are the
    same: 1549 edges, 1548 buckets."""
    v = 1e-12
    pos = []
    while v < 1e20:
        pos.append(v)
        v *= 1.1
    edges = np.array([-x for x in reversed(pos)] + [0.0] + pos, dtype=np.float64)
    assert edges.size == L.STATS_BUCKETS + 1
    return edges


def plan_units(shapes: Mapping[str, Tuple[int, ...]], offsets: Mapping[str, int], has_grad: Sequence[bool],
               unit: int = UNIT_ELEMS):
    """The egot2_stats_param table (one entry per parameter, in `shapes` order) and the egot2_stats_unit list: array 0 (the
    gradient) of the parameters with a gradient, then array 1 (the weights) of every parameter, each parameter cut into
    chunks of at most `unit` elements.  A unit never spans two parameters, also where the stacked LTA / AR head biases sit
    back to back inside one 64-element block."""
    names = list(shapes)
    params = (L.StatsParam * len(names))()
    units = []
    for a in (0, 1):
        for p, n in enumerate(names):
            numel = int(np.prod(shapes[n], dtype=np.int64))
            pr = params[p]
            pr.offset, pr.numel, pr.has_grad = offsets[n], numel, int(bool(has_grad[p]))
            pr.first_unit[a] = len(units)
            if a == 1 or has_grad[p]:
                for b in range(0, numel, unit):
                    units.append((p, a, offsets[n] + b, offsets[n] + min(b + unit, numel)))
            pr.n_units[a] = len(units) - pr.first_unit[a]
    table = (L.StatsUnit * len(units))(*[L.StatsUnit(*u) for u in units])
    return params, table


def histogram_raw(stat: L.ParamStat, counts: np.ndarray, edges: np.ndarray) -> Optional[dict]:
    """The add_histogram_raw keyword arguments of one (array, parameter): the bucket counts trimmed exactly as
    torch.utils.tensorboard.summary.make_histogram trims np.histogram's (the support, plus the empty bucket left of it), so
    the buckets and limits equal those add_histogram(tag, tensor) writes.  min, max, sum and sum_squares cover the finite
    values (make_histogram's min and max would be NaN with a NaN present).  None when no value falls into a bucket."""
    counts = np.asarray(counts, dtype=np.int64)
    cum = np.cumsum(np.greater(counts, 0))
    if cum[-1] == 0:
        return None
    start, end = np.searchsorted(cum, [0, cum[-1] - 1], side="right")
    start, end = int(start), int(end) + 1
    c = counts[start - 1:end] if start > 0 else np.concatenate([[0], counts[:end]])
    return dict(min=float(stat.min), max=float(stat.max), num=int(stat.num), sum=float(stat.sum),
                sum_squares=float(stat.sum_squares), bucket_limits=edges[start:end + 1].tolist(),
                bucket_counts=c.tolist())


def pack_desc(ps: ParamStats, n_params: int) -> bytes:
    return bytes(L.ParamStatsDesc(every=ps.every, histograms=int(ps.histograms), n_params=n_params, step=0, grad_norm=0.0))


def read_stats(host: bytes, n_params: int):
    """(descriptor, [2 * n_params] egot2_param_stat records) from the bytes of a trainer's stats buffer."""
    d = L.ParamStatsDesc.from_buffer_copy(host[:C.sizeof(L.ParamStatsDesc)])
    off = stats_offset()
    recs = (L.ParamStat * (2 * n_params)).from_buffer_copy(host[off:off + 2 * n_params * C.sizeof(L.ParamStat)])
    return d, recs


def stats_offset() -> int:
    """Byte offset of the records in a trainer's stats buffer [descriptor | records [2][P] | counts [2][P][1548] int32]."""
    return (C.sizeof(L.ParamStatsDesc) + 63) // 64 * 64


def buffer_bytes(n_params: int, histograms: bool) -> int:
    return stats_offset() + 2 * n_params * C.sizeof(L.ParamStat) + (2 * n_params * L.STATS_BUCKETS * 4 if histograms else 0)
