"""Data-parallel plumbing of the translator path (SURVEY.md §8e): clips are independent units, so they
shard across ranks with NO data-path collective; the only exchange of a training step is the all-reduce of
the flat translator-gradient arena (what the reference gets from Lightning DDP's bucketed all-reduce:
HOI/scripts/lta/run_lta.py:249, HOI/configs/recognition/defaults.py:494; DP averaging of per-GPU losses:
HOI/tasks/pnr/video_task.py:39-42).

Everything here is host logic over torch.distributed (NCCL on the GPUs, gloo in the CPU tests).
"""
from __future__ import annotations

from typing import Optional, Sequence, Tuple

import torch
import torch.distributed as dist


def bind_to_gpu_numa(device_index: int):
    """Pin this process to the CPUs of the NUMA node its GPU hangs off, BEFORE it allocates pinned host buffers (first touch
    then places them on that node).  With 8 ranks each streaming features to its own GPU every step, buffers on the wrong
    socket halve the host->device rate.  Best effort: returns (numa node, #cpus) or None when sysfs / the PCI ids are missing."""
    import os
    try:
        p = torch.cuda.get_device_properties(device_index)
        bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        base = f"/sys/bus/pci/devices/{bdf}"
        node = int(open(f"{base}/numa_node").read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node, len(cpus)
    except Exception:      # noqa: BLE001 - purely an optimisation
        return None


def shard_range(n_clips: int, world: int, rank: int) -> Tuple[int, int]:
    """Contiguous, balanced clip range [lo, hi) of `rank`: the first n % world ranks get one extra clip
    (reference: DistributedSampler's per-GPU batch = BATCH_SIZE / NUM_GPUS, HOI/dataset/lta/loader.py:73-74)."""
    if not (0 <= rank < world):
        raise ValueError(f"rank {rank} outside world of {world}")
    base, extra = divmod(n_clips, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def shard_clips(tensors: Sequence[torch.Tensor], world: int, rank: int):
    """Slice every per-clip tensor (leading dimension = clips) to this rank's shard."""
    lo, hi = shard_range(int(tensors[0].shape[0]), world, rank)
    return [t[lo:hi] for t in tensors]


def allreduce_gradients(flat_grad: torch.Tensor, group=None, local_weight: Optional[float] = None) -> float:
    """Combine the ranks' flat gradient arenas in place with ONE all-reduce and return the scale the optimizer must
    apply to the summed buffer.

    local_weight None  -> DDP semantics (what the reference does): mean over ranks, scale = 1 / world.
    local_weight w_r   -> exact full-batch gradient for mean-type losses with unequal shards: every rank scales its
                          arena by w_r first (w_r = its clips, or its summed class weights for the weighted CE), the
                          buffers are summed and the returned scale is 1 / sum_r w_r.
    """
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if world == 1:
        return 1.0
    if local_weight is None:
        dist.all_reduce(flat_grad, group=group)
        return 1.0 / world
    w = torch.tensor([float(local_weight)], dtype=torch.float64, device=flat_grad.device)
    flat_grad.mul_(float(local_weight))
    dist.all_reduce(flat_grad, group=group)
    dist.all_reduce(w, group=group)
    return 1.0 / float(w.item())


def gather_outputs(local_out: torch.Tensor, n_clips: int, group=None) -> torch.Tensor:
    """Inference: concatenate the ranks' per-clip outputs in clip order (shards may differ by one clip)."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if world == 1:
        return local_out
    base, extra = divmod(n_clips, world)
    pad_rows = base + (1 if extra else 0)
    padded = local_out.new_zeros((pad_rows,) + tuple(local_out.shape[1:]))
    padded[: local_out.shape[0]] = local_out
    parts = [torch.empty_like(padded) for _ in range(world)]
    dist.all_gather(parts, padded, group=group)
    out = []
    for r, p in enumerate(parts):
        lo, hi = shard_range(n_clips, world, r)
        out.append(p[: hi - lo])
    return torch.cat(out, dim=0)


# ---------------------------------------------------------------------------------------------------------------------
# The exchange step as one kernel over NVLink peer memory (csrc/peer.cu)
# ---------------------------------------------------------------------------------------------------------------------
def slab_layout(numel: int, with_shadow: bool, flag_bytes: int):
    """Byte offsets of (param fp32, grad fp32, shadow bf16 | -1, flags) inside a rank's slab and the slab size; identical
    on every rank by construction (a pure function of the arena size)."""
    a = lambda x: (x + 255) // 256 * 256
    off_param = 0
    off_grad = a(off_param + 4 * numel)
    off_shadow = a(off_grad + 4 * numel) if with_shadow else -1
    off_flags = a((off_shadow + 2 * numel) if with_shadow else (off_grad + 4 * numel))
    return off_param, off_grad, off_shadow, off_flags, off_flags + flag_bytes


class _DeviceMemory:
    """Zero-copy view of raw device memory for torch (CUDA array interface v2)."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (int(ptr), False), "version": 2}


class PeerExchange:
    """Puts an engine's parameter / gradient / bf16-shadow arenas into an IPC-shared slab, maps every peer's slab, and runs
    `egot2_dp_reduce_adam` - gradient reduce-scatter + Adam on this rank's slice + parameter all-gather in ONE kernel - in
    place of [NCCL all-reduce + fused Adam].  One node, at most 8 ranks, every GPU peer-accessible (NVSwitch).

    `available()` is False (and the trainer keeps the NCCL path) for CPU process groups, more than 8 ranks, or when the
    handle exchange fails."""

    def __init__(self, engine, group=None):
        import ctypes as C
        from . import _lib as L
        self.engine, self.group = engine, group
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        if not (1 < self.world <= 8) or engine.device.type != "cuda":
            raise L.Egot2Error("PeerExchange: needs 2..8 CUDA ranks on one node")
        arena = engine.arena
        with_shadow = engine.dtype == "bf16"
        lib = L.load()
        self.offs = slab_layout(arena.numel, with_shadow, int(lib.egot2_dp_flag_bytes()))
        off_param, off_grad, off_shadow, off_flags, nbytes = self.offs
        with torch.cuda.device(engine.device):
            ptr = C.c_void_p()
            L.call("egot2_peer_alloc", nbytes, C.byref(ptr))
            self.local = int(ptr.value)
            hb = int(lib.egot2_peer_handle_bytes())
            handle = C.create_string_buffer(hb)
            L.call("egot2_peer_export", self.local, handle)
            handles = [None] * self.world
            dist.all_gather_object(handles, bytes(handle.raw), group=group)
            self.slabs = []
            for r, h in enumerate(handles):
                if r == self.rank:
                    self.slabs.append(self.local)
                    continue
                p = C.c_void_p()
                L.call("egot2_peer_import", C.create_string_buffer(h, hb), C.byref(p))
                self.slabs.append(int(p.value))
            raw = torch.as_tensor(_DeviceMemory(self.local, nbytes), device=engine.device)
            self._raw = raw                                            # keeps the view alive; the slab itself is freed in close()
            param = raw[off_param:off_param + 4 * arena.numel].view(torch.float32)
            grad = raw[off_grad:off_grad + 4 * arena.numel].view(torch.float32)
            shadow = raw[off_shadow:off_shadow + 2 * arena.numel].view(torch.bfloat16) if with_shadow else None
            arena.rebase(param, grad, shadow)
            torch.cuda.synchronize(engine.device)
        dist.barrier(group=group)                                      # every slab is mapped everywhere before the first step
        self.desc = L.DpDesc()
        self.desc.world, self.desc.rank, self.desc.numel = self.world, self.rank, arena.numel
        for r, p in enumerate(self.slabs):
            self.desc.slab[r] = p
        self.desc.off_param, self.desc.off_grad, self.desc.off_shadow, self.desc.off_flags = off_param, off_grad, off_shadow, off_flags

    def step(self, state, step: int, hp, stream: int, step_dev: Optional[torch.Tensor] = None, decoupled: bool = False,
             lo: int = 0, hi: Optional[int] = None, channel: int = 0, lr_dev: Optional[torch.Tensor] = None,
             guard: Optional[torch.Tensor] = None, groups: Optional[Tuple[torch.Tensor, torch.Tensor]] = None, sgd=None):
        """The exchange + optimizer step of this rank for arena elements [lo, hi) (default: everything) on flag `channel`;
        afterwards that part of the gradient arena is cleared (stream order).  lr_dev: the learning rate is read from this
        device float when the kernel executes (optim.py), instead of hp["lr"].  guard: a device egot2_grad_guard - the
        update is clipped by the global norm of the rank-averaged gradient, or skipped on every rank when it is not finite
        (two launches); it must cover the whole arena.  groups: (device egot2_param_groups, block map of the whole arena), as
        in engine.adam_step; hp["weight_decay"] is then unused.  sgd: an optim.SGD - torch.optim.SGD on this rank's slice
        instead of Adam (engine.sgd_step's semantics; state["buf"] is the local momentum buffer, hp["betas"] / hp["eps"] and
        `decoupled` are unused)."""
        import ctypes as C
        from . import _lib as L
        arena = self.engine.arena
        d = self.desc
        if sgd is None:
            if "m" not in state:
                state["m"] = torch.zeros_like(arena.param)
                state["v"] = torch.zeros_like(arena.param)
            d.exp_avg, d.exp_avg_sq = state["m"].data_ptr(), state["v"].data_ptr()
            d.sgd, d.momentum, d.dampening, d.nesterov = 0, 0.0, 0.0, 0
        else:
            if sgd.momentum != 0.0 and "buf" not in state:
                state["buf"] = torch.zeros_like(arena.param)
            d.exp_avg, d.exp_avg_sq = (state["buf"].data_ptr() if sgd.momentum != 0.0 else None), None
            d.sgd, d.momentum, d.dampening, d.nesterov = 1, sgd.momentum, sgd.dampening, int(sgd.nesterov)
        d.lr, (d.beta1, d.beta2), d.eps, d.weight_decay = hp["lr"], hp["betas"], hp["eps"], hp["weight_decay"]
        d.step = int(step)
        d.step_dev = step_dev.data_ptr() if step_dev is not None else None
        d.lr_dev = lr_dev.data_ptr() if lr_dev is not None else None
        d.decoupled = 1 if decoupled else 0
        hi = arena.numel if hi is None else hi
        if guard is not None and (lo, hi) != (0, arena.numel):
            raise L.Egot2Error("PeerExchange.step: a gradient guard needs the norm of the whole arena (lo=0, hi=numel)")
        d.guard = guard.data_ptr() if guard is not None else None
        d.groups, d.block_group = (None, None) if groups is None else (groups[0].data_ptr(), groups[1].data_ptr())
        # small exchanges: the slice owners clear the gradients in the same kernel; large ones: one local clear afterwards
        # (clearing over NVLink would double the remote traffic)
        remote_zero = (hi - lo) * 4 <= (16 << 20)
        d.zero_grads_remote = 1 if remote_zero else 0
        with torch.cuda.device(self.engine.device):
            L.call("egot2_dp_reduce_adam_range", C.byref(d), int(lo), int(hi), int(channel), stream)
        if not remote_zero:
            arena.grad[lo:hi].zero_() # safe: the kernel returned only after every peer finished reading these gradients
        arena.shadow_fresh = self.engine.dtype == "bf16"

    def close(self):
        from . import _lib as L
        with torch.cuda.device(self.engine.device):
            torch.cuda.synchronize(self.engine.device)
            for r, p in enumerate(self.slabs):
                if r != self.rank and p:
                    L.call("egot2_peer_unimport", p)
            self.slabs = []
