"""Learning-rate schedules evaluated on the device (optim.LRSchedule, egot2_opt_advance, egot2_adam_step_fused_sched,
egot2_dp_desc.lr_dev) and resumable optimizer state of the fused trainers.

CPU: the host restatement of lr_at against torch.optim.lr_scheduler, the ABI mirrors, the launch plan of a scheduled step,
LRSchedule's input checks.  GPU (-m gpu): the kernels against the restatement and torch.optim, the trainers' scheduled
graph steps against host-set lrs, resume, and the two-rank exchange."""
import contextlib
import ctypes as C
import math
import os

import numpy as np
import pytest
import torch

from egot2_b200 import _lib as L
from egot2_b200.optim import LRSchedule

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def lr_at(s: LRSchedule, t: int) -> float:
    """Host restatement of the device's lr_at (include/egot2.h) for optimizer step index t = 0, 1, ... (the lr of step t + 1).

    The policies are SlowFast's, as selected by the HOI configs (SURVEY.md §2.2 and §3.5: Adam + warm-up cosine,
    HOI/optimizers/lta/lr_scheduler.py:21-26,67-91): cosine from base_lr to end_lr over total_steps, steps with relative lrs,
    and a linear warm-up from warmup_start_lr to the policy's value at warmup_steps.  The reference tree is not part of this
    checkout, so these formulas were written from the survey's description and were NOT re-read against lr_scheduler.py."""
    def policy(k):
        if s.kind == L.LR_COSINE:
            if k >= s.total_steps:
                return s.end_lr
            return s.end_lr + (s.base_lr - s.end_lr) * (1.0 + math.cos(math.pi * k / s.total_steps)) / 2.0
        if s.kind == L.LR_STEPS:
            return s.base_lr * s.factors[sum(1 for m in s.milestones if m <= k)]
        return s.base_lr
    if t < s.warmup_steps:
        return s.warmup_start_lr + (policy(s.warmup_steps) - s.warmup_start_lr) * t / s.warmup_steps
    return policy(t)


SCHEDULES = {
    "constant": LRSchedule.constant(3e-4),
    "cosine": LRSchedule.cosine(1e-3, 20, end_lr=1e-5),
    "cosine_warmup": LRSchedule.cosine(1e-3, 20, end_lr=1e-5, warmup_steps=5, warmup_start_lr=1e-6),
    "steps": LRSchedule.steps(1e-3, [4, 9, 15], [1.0, 0.3, 0.1, 0.01]),
    "steps_warmup": LRSchedule.steps(1e-3, [4, 9, 15], [1.0, 0.3, 0.1, 0.01], warmup_steps=3),
}


# ------------------------------------------------------------------------------------------------ CPU: the restatement
def _torch_lrs(sched_fn, base_lr, n):
    p = torch.nn.Parameter(torch.zeros(1))
    opt = torch.optim.SGD([p], lr=base_lr)
    sch = sched_fn(opt)
    out = []
    for _ in range(n):
        out.append(opt.param_groups[0]["lr"])
        opt.step()
        sch.step()
    return out


def test_cosine_matches_cosine_annealing_lr():
    s = LRSchedule.cosine(1e-3, 20, end_lr=1e-5)
    want = _torch_lrs(lambda o: torch.optim.lr_scheduler.CosineAnnealingLR(o, T_max=20, eta_min=1e-5), 1e-3, 21)
    got = [lr_at(s, t) for t in range(21)]
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-15)
    assert lr_at(s, 25) == s.end_lr                     # held at end_lr after total_steps


def test_steps_matches_multistep_lr():
    gamma, ms = 0.2, [3, 7, 12]
    s = LRSchedule.steps(1e-3, ms, [gamma ** i for i in range(len(ms) + 1)])
    want = _torch_lrs(lambda o: torch.optim.lr_scheduler.MultiStepLR(o, milestones=ms, gamma=gamma), 1e-3, 16)
    np.testing.assert_allclose([lr_at(s, t) for t in range(16)], want, rtol=1e-12)


@pytest.mark.parametrize("name", ["cosine_warmup", "steps_warmup"])
def test_warmup_matches_lambda_lr_and_is_continuous(name):
    s = SCHEDULES[name]
    w = s.warmup_steps

    def lam(t):                     # the warm-up formula restated independently of lr_at
        target = lr_at(dataclass_replace(s, warmup_steps=0), w)
        return (s.warmup_start_lr + (target - s.warmup_start_lr) * t / w if t < w else lr_at(s, t)) / s.base_lr
    want = _torch_lrs(lambda o: torch.optim.lr_scheduler.LambdaLR(o, lam), s.base_lr, 20)
    np.testing.assert_allclose([lr_at(s, t) for t in range(20)], want, rtol=1e-12)
    assert lr_at(s, 0) == s.warmup_start_lr
    # the warm-up's end point is the policy's value: no jump at t = warmup_steps
    step_in = lr_at(s, w - 1) - lr_at(s, w - 2)
    assert abs(lr_at(s, w) - lr_at(s, w - 1) - step_in) <= 1e-12


def dataclass_replace(s, **kw):
    import dataclasses
    return dataclasses.replace(s, **kw)


# ------------------------------------------------------------------------------------------------ CPU: host checks
@pytest.mark.parametrize("make", [
    lambda: LRSchedule.cosine(1e-3, 0),
    lambda: LRSchedule.cosine(1e-3, -5),
    lambda: LRSchedule.steps(1e-3, [5, 3], [1.0, 0.1, 0.01]),
    lambda: LRSchedule.steps(1e-3, [3, 3], [1.0, 0.1, 0.01]),
    lambda: LRSchedule.steps(1e-3, [3, 5], [1.0, 0.1]),
    lambda: LRSchedule.steps(1e-3, list(range(1, 10)), [1.0] * 10),
    lambda: LRSchedule.steps(1e-3, [-1], [1.0, 0.1]),
    lambda: LRSchedule.cosine(1e-3, 10, warmup_steps=-1),
    lambda: LRSchedule(7, 1e-3),
    lambda: LRSchedule(L.LR_CONSTANT, 1e-3, milestones=(3,), factors=(1.0, 0.1)),
])
def test_schedule_rejects_malformed_input(make):
    with pytest.raises(ValueError):
        make()


def test_schedule_packs_and_round_trips():
    s = SCHEDULES["steps_warmup"]
    d = s.pack()
    assert (d.kind, d.n_milestones, d.warmup_steps) == (L.LR_STEPS, 3, 3)
    assert list(d.milestones[:3]) == [4, 9, 15] and list(d.factors[:4]) == [1.0, 0.3, 0.1, 0.01]
    assert LRSchedule.from_dict(s.to_dict()) == s
    c = LRSchedule.cosine(2e-3, 100, end_lr=1e-6, warmup_steps=10, warmup_start_lr=1e-7).pack()
    assert (c.kind, c.total_steps, c.base_lr, c.end_lr, c.warmup_start_lr) == (L.LR_COSINE, 100, 2e-3, 1e-6, 1e-7)


@pytest.fixture(scope="module")
def built():
    from egot2_b200 import build
    return build.build()


def test_struct_layouts_match_header(built):
    """sizeof and every field offset of egot2_lr_sched and of the extended egot2_dp_desc equal the ctypes mirrors."""
    import subprocess
    import tempfile
    names = {"egot2_lr_sched": L.LrSched, "egot2_dp_desc": L.DpDesc}
    fields = [(n, f[0]) for n, cls in names.items() for f in cls._fields_]
    prog = '#include <stdio.h>\n#include <stddef.h>\n#include "egot2.h"\nint main(){' + "".join(
        f'printf("{n} %zu\\n", sizeof({n}));' for n in names) + "".join(
        f'printf("{n}.{f} %zu\\n", offsetof({n}, {f}));' for n, f in fields) + \
        'printf("kinds %d %d %d\\n", EGOT2_LR_CONSTANT, EGOT2_LR_COSINE, EGOT2_LR_STEPS);return 0;}'
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "probe.c")
        open(src, "w").write(prog)
        exe = os.path.join(td, "probe")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
        out = subprocess.check_output([exe], text=True)
    for line in out.strip().splitlines():
        n, *v = line.split()
        if n == "kinds":
            assert [int(x) for x in v] == [L.LR_CONSTANT, L.LR_COSINE, L.LR_STEPS]
        elif "." in n:
            st, f = n.split(".")
            assert getattr(names[st], f).offset == int(v[0]), f"{n}: ctypes offset {getattr(names[st], f).offset} != C {v[0]}"
        else:
            assert C.sizeof(names[n]) == int(v[0]), f"{n}: ctypes {C.sizeof(names[n])} != C {v[0]}"


# ------------------------------------------------------------------------------------------------ CPU: launch plan
class _FakeStream:
    cuda_stream = 0

    def wait_stream(self, other):
        pass


class _FakeGraph:
    def __init__(self):
        self.replays = 0

    def replay(self):
        self.replays += 1


@pytest.fixture
def recorder(monkeypatch):
    """The C ABI replaced by a recorder and the CUDA-graph machinery by stand-ins, so the trainer's launch sequence runs on
    the CPU.  ('capture', i) / ('end', i) markers delimit what a captured graph contains."""
    from egot2_b200 import engine as E, trainer as T
    calls = []

    def fake_call(name, *args):
        calls.append((name, args))
        return 0

    @contextlib.contextmanager
    def fake_graph(g, *a, **k):
        calls.append(("<capture>", ()))
        yield
        calls.append(("</capture>", ()))
    monkeypatch.setattr(L, "call", fake_call)
    monkeypatch.setattr(E, "_stream", lambda: 0)
    monkeypatch.setattr(T, "_cur_stream", lambda device: 0)
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    monkeypatch.setattr(torch.cuda, "Stream", lambda device=None: _FakeStream())
    monkeypatch.setattr(torch.cuda, "current_stream", lambda device=None: _FakeStream())
    monkeypatch.setattr(torch.cuda, "stream", lambda s: contextlib.nullcontext())
    monkeypatch.setattr(torch.cuda, "synchronize", lambda device=None: None)
    monkeypatch.setattr(torch.cuda, "CUDAGraph", _FakeGraph)
    monkeypatch.setattr(torch.cuda, "graph", fake_graph)
    return calls


def _hhi_trainer(schedule=None, **kw):
    from egot2_b200 import specs, synth
    from egot2_b200.trainer import TranslatorTrainer
    spec = specs.hhi_ttm_spec(128, 4, 1, 0.5, True)
    tr = TranslatorTrainer(spec, "cpu", "bf16", lr_schedule=schedule, **kw)
    tr.load_state_dict(synth.make_state_dict(spec, 0))
    f = synth.make_features(spec, 4, (6, 6, 6), seed=1, dtype=torch.bfloat16)
    return tr, [f[s.name] for s in spec.segments], synth.make_labels(spec, 4, (6, 6, 6), seed=1)


def _captured(calls):
    names = [c[0] for c in calls]
    i, j = names.index("<capture>"), names.index("</capture>")
    return names[i + 1:j]


# The launch sequence of this HHI trainer without a schedule, as the commit before device-side schedules recorded it with
# the same stand-ins: construction, the first graph step (warm-up, capture), a replay (nothing), an eager step.
_FWD_BWD = ["egot2_hhi_tok_table_fwd", "egot2_embed_fwd", "egot2_encoder_layer_fwd", "egot2_head_loss_fwd",
            "egot2_head_loss_bwd", "egot2_encoder_layer_bwd", "egot2_embed_bwd"]
_PARENT_GRAPH = _FWD_BWD + ["egot2_dropout_epoch_advance", "egot2_adam_step_fused_dev"]
_PARENT_PLAN = (["egot2_dropout_epoch_enable", "egot2_dropout_epoch_set", "egot2_cast_f32_to_bf16"] + _FWD_BWD
                + ["egot2_cast_f32_to_bf16", "<capture>"] + _PARENT_GRAPH + ["</capture>"]
                + _FWD_BWD + ["egot2_adam_step_fused", "egot2_dropout_epoch_advance"])


def test_unscheduled_step_plan_is_unchanged(recorder):
    tr, feats, labels = _hhi_trainer()
    tr.train_step(feats, labels, graph_key=0)
    tr.train_step(feats, labels, graph_key=0)
    tr.use_graphs = False
    tr.train_step(feats, labels)
    assert [c[0] for c in recorder] == _PARENT_PLAN


def test_scheduled_graph_step_plan(recorder):
    tr, feats, labels = _hhi_trainer(LRSchedule.cosine(1e-3, 10, warmup_steps=2))
    tr.train_step(feats, labels, graph_key=0)
    body = _captured(recorder)
    assert body.count("egot2_opt_advance") == 1 and body.count("egot2_adam_step_fused_sched") == 1
    assert "egot2_adam_step_fused_dev" not in body
    # the advance replaces the side branch's counter increment: the forward/backward chain is the parent's
    assert [n for n in body if n not in ("egot2_opt_advance", "egot2_adam_step_fused_sched")] == _PARENT_GRAPH[:-1]
    (adv,) = [a for n, a in recorder if n == "egot2_opt_advance"]
    (adam,) = [a for n, a in recorder if n == "egot2_adam_step_fused_sched"]
    assert adv[0] == tr._step_dev.data_ptr() and adv[1] == tr._sched_dev.data_ptr() and adv[2] == tr._lr_dev.data_ptr()
    assert adam[5] == tr._lr_dev.data_ptr() and adam[10] == tr._step_dev.data_ptr() and adam[14] == 0     # Adam, not AdamW
    # set_lr_schedule between replays: the descriptor changes in place, no capture
    tr.set_lr_schedule(LRSchedule.constant(5e-5))
    del recorder[:]
    tr.train_step(feats, labels, graph_key=0)
    assert recorder == [] and len(tr._graphs) == 1
    assert bytes(tr._sched_dev.numpy()) == bytes(LRSchedule.constant(5e-5).pack())


@pytest.mark.parametrize("use_graphs", [False, True])
def test_scheduled_eager_update_plan(use_graphs, recorder, monkeypatch):
    """Eager optimizer launches (no graphs, or EGOT2_GRAPH_UPDATE=0): one advance right before the optimizer."""
    monkeypatch.setenv("EGOT2_GRAPH_UPDATE", "0")
    tr, feats, labels = _hhi_trainer(LRSchedule.constant(1e-4), use_graphs=use_graphs)
    for step in (1, 2):
        del recorder[:]
        tr.train_step(feats, labels, graph_key=0)
        names = [c[0] for c in recorder if not c[0].startswith("<")]
        i = names.index("egot2_adam_step_fused_sched")
        assert names[i - 1] == "egot2_opt_advance" and names.count("egot2_opt_advance") == 1
        assert "egot2_adam_step_fused" not in names and "egot2_adam_step_fused_dev" not in names
        assert tr._step_dev_val == step                # what the advance kernel (not run here) leaves in _step_dev


def test_scheduled_peer_split_hands_lr_to_both_exchanges(recorder, monkeypatch):
    """EGOT2_DP_SPLIT=1: the peer exchange runs as two launches inside the graph; both read the device lr."""
    monkeypatch.setenv("EGOT2_DP_SPLIT", "1")
    got = []

    class FakePeer:
        def step(self, state, step, hp, stream, **kw):
            got.append(kw)
    tr, feats, labels = _hhi_trainer(LRSchedule.cosine(1e-3, 10))
    tr.peer, tr.graph_update = FakePeer(), True
    tr.train_step(feats, labels, graph_key=0)
    assert len(got) == 2 and {k["channel"] for k in got} == {0, 1}
    assert all(k["lr_dev"] is tr._lr_dev and k["step_dev"] is tr._step_dev for k in got)
    assert _captured(recorder).count("egot2_opt_advance") == 1


def test_adamw_with_device_step_takes_the_sched_entry(recorder):
    """engine.adam_step(step_dev=..., decoupled=True) runs AdamW through egot2_adam_step_fused_sched (the _dev entry has
    no decoupled decay), with the fixed lr handed over on the device."""
    tr, _, _ = _hhi_trainer()
    del recorder[:]
    tr.engine.adam_step({}, 1, 2e-4, weight_decay=1e-2, fused=True, step_dev=tr._step_dev, decoupled=True)
    ((name, args),) = [c for c in recorder if "adam" in c[0]]
    assert name == "egot2_adam_step_fused_sched" and args[14] == 1 and args[10] == tr._step_dev.data_ptr()
    del recorder[:]
    tr.engine.adam_step({}, 1, 2e-4, fused=True, step_dev=tr._step_dev, lr_dev=tr._step_dev.float())
    assert [n for n, _ in recorder] == ["egot2_adam_step_fused_sched"] and recorder[0][1][14] == 0
    with pytest.raises(L.Egot2Error):                        # a device lr without a device step count
        tr.engine.adam_step({}, 1, fused=True, lr_dev=tr._step_dev.float())


def test_lr_and_schedule_together_is_an_error(recorder):
    with pytest.raises(ValueError):
        _hhi_trainer(LRSchedule.constant(1e-4), lr=1e-3)
    tr, _, _ = _hhi_trainer()
    with pytest.raises(ValueError):
        tr.set_lr_schedule(LRSchedule.constant(1e-4))


def test_optimizer_state_dict_round_trip(recorder):
    """Moments keyed by parameter name (the arena's name-to-slice mapping), step count, schedule and dropout epoch."""
    s = LRSchedule.cosine(1e-3, 10, warmup_steps=2)
    tr, feats, labels = _hhi_trainer(s)
    for _ in range(3):
        tr.train_step(feats, labels, graph_key=0)
    arena = tr.engine.arena
    torch.manual_seed(0)
    tr.opt_state["m"].copy_(torch.randn(arena.numel))
    tr.opt_state["v"].copy_(torch.rand(arena.numel))
    sd = tr.optimizer_state_dict()
    assert sd["step"] == 3 and sd["dropout_epoch"] == 3 and LRSchedule.from_dict(sd["lr_schedule"]) == s
    assert set(sd["exp_avg"]) == set(arena.shapes)
    tr2, _, _ = _hhi_trainer(LRSchedule.constant(1.0))
    del recorder[:]
    tr2.load_optimizer_state_dict(sd)
    assert tr2.step_count == 3 and int(tr2._step_dev[0]) == 3 and tr2._epoch == 3 and tr2.lr_schedule == s
    assert [(n, a[0]) for n, a in recorder] == [("egot2_dropout_epoch_set", 3)]
    for k in ("m", "v"):
        for name in arena.shapes:
            assert torch.equal(arena.view(name, tr2.opt_state[k]), arena.view(name, tr.opt_state[k]))
    with pytest.raises(ValueError):                           # saved with a schedule, loaded into a trainer without one
        _hhi_trainer()[0].load_optimizer_state_dict(sd)


# ------------------------------------------------------------------------------------------------ GPU
def _dev_sched(s: LRSchedule, dev="cuda:0"):
    return torch.frombuffer(bytearray(bytes(s.pack())), dtype=torch.uint8).to(dev)


def _f32(x: float) -> float:
    return float(np.float32(x))


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SCHEDULES))
def test_opt_advance_matches_oracle(name):
    s = SCHEDULES[name]
    st = torch.cuda.current_stream().cuda_stream
    sched = _dev_sched(s)
    step = torch.zeros(1, device="cuda", dtype=torch.int32)
    lr = torch.zeros(1, device="cuda", dtype=torch.float32)
    n = 30
    got = torch.empty(n, device="cuda", dtype=torch.float32)
    for t in range(n):
        L.call("egot2_opt_advance", step.data_ptr(), sched.data_ptr(), lr.data_ptr(), st)
        got[t:t + 1].copy_(lr)
    got = got.cpu().numpy()
    assert int(step.item()) == n
    for t in range(1, n + 1):
        want = np.float32(lr_at(s, t - 1))
        assert abs(float(got[t - 1]) - float(want)) <= float(np.spacing(want)), (t, got[t - 1], want)


@pytest.mark.gpu
@pytest.mark.parametrize("decoupled", [False, True])
def test_adam_sched_matches_torch(decoupled):
    """egot2_adam_step_fused_sched (Adam / AdamW) == torch.optim.Adam / AdamW + LambdaLR over 10 scheduled steps."""
    s = LRSchedule.cosine(1e-3, 8, end_lr=1e-5, warmup_steps=3, warmup_start_lr=1e-5)
    torch.manual_seed(2)
    n = 10007
    p = torch.randn(n, device="cuda")
    ref = p.clone().requires_grad_(True)
    wd = 0.1 if decoupled else 0.01
    opt = (torch.optim.AdamW if decoupled else torch.optim.Adam)([ref], lr=s.base_lr, weight_decay=wd)
    lam = torch.optim.lr_scheduler.LambdaLR(opt, lambda t: lr_at(s, t) / s.base_lr)
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    shadow = torch.empty(n, device="cuda", dtype=torch.bfloat16)
    step = torch.zeros(1, device="cuda", dtype=torch.int32)
    lr = torch.zeros(1, device="cuda", dtype=torch.float32)
    sched = _dev_sched(s)
    st = torch.cuda.current_stream().cuda_stream
    for _ in range(10):
        g = torch.randn(n, device="cuda")
        ref.grad = g.clone()
        opt.step()
        lam.step()
        L.call("egot2_opt_advance", step.data_ptr(), sched.data_ptr(), lr.data_ptr(), st)
        L.call("egot2_adam_step_fused_sched", p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), n, lr.data_ptr(),
               0.9, 0.999, 1e-8, wd, step.data_ptr(), 1.0, shadow.data_ptr(), 1, int(decoupled), st)
        assert float((p - ref.detach()).abs().max()) < 1e-6
        assert float(g.abs().max()) == 0.0 and torch.equal(shadow, p.to(torch.bfloat16))


def _hhi_setup(dropout: bool, batch=16, seed=1):
    import dataclasses
    from egot2_b200 import specs, synth
    spec = specs.hhi_ttm_spec(128, 4, 1, 0.5 if dropout else 0.0, True)
    if not dropout:
        spec = dataclasses.replace(spec, p_embed=0.0)
    seg = (30, 30, 30)
    f = synth.make_features(spec, batch, seg, seed=seed, dtype=torch.bfloat16)
    feats = [f[s.name].cuda() for s in spec.segments]
    return spec, feats, synth.make_labels(spec, batch, seg, seed=seed).cuda()


def _hhi_trainer_gpu(spec, **kw):
    from egot2_b200 import synth
    from egot2_b200.trainer import TranslatorTrainer
    tr = TranslatorTrainer(spec, torch.device("cuda:0"), "bf16", **kw)
    tr.load_state_dict(synth.make_state_dict(spec, 0))
    return tr


@pytest.mark.gpu
def test_scheduled_whole_step_graph_matches_host_set_lr():
    """HHI TranslatorTrainer, whole-step graph, warm-up from lr 0 + cosine over 12 replays == an eager trainer whose host
    lr is set to the same value before each step; last_lr reports it; set_lr_schedule needs no new capture.  Peak lr 5e-4
    (the HHI recipe's): Adam turns the fp32-atomic rounding of near-zero gradients into steps of about lr, so the parameter
    tolerance of the fixed-lr graph test holds at that lr."""
    s = LRSchedule.cosine(5e-4, 12, end_lr=1e-5, warmup_steps=3, warmup_start_lr=0.0)
    spec, feats, labels = _hhi_setup(dropout=False)
    tg = _hhi_trainer_gpu(spec, use_graphs=True, lr_schedule=s)
    te = _hhi_trainer_gpu(spec, use_graphs=False)
    assert tg.graph_update
    p0 = tg.engine.arena.param.clone()
    lrs, lg, le = [], [], []
    for t in range(1, 13):
        lg.append(tg.train_step(feats, labels, graph_key=0).clone())
        lrs.append(tg.last_lr.clone())
        te.hp["lr"] = lr_at(s, t - 1)
        le.append(te.train_step(feats, labels).clone())
        if t == 1:
            assert torch.equal(tg.engine.arena.param, p0)            # lr 0: the first step moves nothing
        if t == 2:
            assert not torch.equal(tg.engine.arena.param, p0)
    torch.cuda.synchronize()
    assert [float(x) for x in lrs] == [_f32(lr_at(s, t)) for t in range(12)]
    pg, pe = tg.engine.arena.param, te.engine.arena.param
    assert float((pg - pe).abs().max()) <= 5e-4 * float(pe.abs().max())
    assert all(abs(float(a) - float(b)) <= 2e-2 * abs(float(b)) + 1e-4 for a, b in zip(lg, le))
    assert float(lg[-1]) != float(lg[0])
    # a new schedule between replays: lr 0 freezes the parameters, then a constant lr moves them; still one graph
    n_graphs = len(tg._graphs)
    tg.set_lr_schedule(LRSchedule.constant(0.0))
    before = tg.engine.arena.param.clone()
    tg.train_step(feats, labels, graph_key=0)
    torch.cuda.synchronize()
    assert float(tg.last_lr) == 0.0 and torch.equal(tg.engine.arena.param, before)
    tg.set_lr_schedule(LRSchedule.constant(1e-3))
    tg.train_step(feats, labels, graph_key=0)
    torch.cuda.synchronize()
    assert float(tg.last_lr) == _f32(1e-3) and not torch.equal(tg.engine.arena.param, before)
    assert len(tg._graphs) == n_graphs and tg.step_count == 14 and int(tg._step_dev.item()) == 14


@pytest.mark.gpu
@pytest.mark.parametrize("scheduled", [True, False])
def test_resume_continues_like_an_uninterrupted_run(scheduled):
    """6 graph steps with dropout, save, a fresh trainer loads and runs 6 more == 12 uninterrupted steps: per-step losses and
    final parameters to rounding.  Negative control: the same resume with the dropout epoch left at 0 draws other masks.
    The parameters are compared by the L2 norm of the difference relative to how far training moved them: two identical
    uninterrupted runs already differ by ~2e-3 at single elements (Adam turns the fp32-atomic rounding of near-zero
    gradients into steps of about lr), but by ~0.5 % in that norm, against ~5-12 % for the control."""
    from egot2_b200.engine import _stream
    kw = dict(use_graphs=True)
    if scheduled:
        kw["lr_schedule"] = LRSchedule.cosine(5e-4, 12, warmup_steps=2, warmup_start_lr=1e-5)
    spec, feats, labels = _hhi_setup(dropout=True)

    def run(tr, n):
        out = [tr.train_step(feats, labels, graph_key=0).clone() for _ in range(n)]
        torch.cuda.synchronize()
        return [float(x) for x in out]
    full = _hhi_trainer_gpu(spec, **kw)
    p0 = full.engine.arena.param.clone()
    l_full = run(full, 12)
    p_full = full.engine.arena.param.clone()
    del full
    first = _hhi_trainer_gpu(spec, **kw)
    run(first, 6)
    sd, osd = first.state_dict(), first.optimizer_state_dict()
    assert osd["step"] == 6 and osd["dropout_epoch"] == 6
    del first
    results = {}
    for restore_epoch in (True, False):
        tr = _hhi_trainer_gpu(spec, **kw)
        tr.load_state_dict(sd)
        tr.load_optimizer_state_dict(osd)
        if not restore_epoch:
            L.call("egot2_dropout_epoch_set", 0, _stream())
        results[restore_epoch] = (run(tr, 6), tr.engine.arena.param.clone())
        del tr
    (l_res, p_res), (l_ctl, p_ctl) = results[True], results[False]
    moved = float((p_full - p0).norm())
    assert float((p_res - p_full).norm()) <= 2e-2 * moved
    assert float((p_ctl - p_full).norm()) > 2e-2 * moved
    err = max(abs(a - b) for a, b in zip(l_res, l_full[6:]))
    ctl = max(abs(a - b) for a, b in zip(l_ctl, l_full[6:]))
    assert err <= 2e-2 * abs(l_full[6]) + 1e-4
    assert ctl > 10 * err, (err, ctl)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["hhi", "hoi"])
def test_prompt_trainer_scheduled_graph_matches_host_set_lr(kind, monkeypatch):
    """EgoT2-g trainers (HHI: Adam, HOI: AdamW), graph mode: a scheduled run == the same trainer without a schedule whose
    host lr is set to the schedule's value before each step.  In these trainers the optimizer after the graph replay is an
    eager launch that takes hp["lr"], so the reference is graph mode too: an eager-mode run would draw other dropout masks
    (the prompt-embedding dropout cannot be switched off), and the two runs go one after the other because trainers share
    the device's dropout epoch."""
    from egot2_b200 import specs, synth, trainer as T
    monkeypatch.setenv("EGOT2_G_GRAPH", "1")
    s = LRSchedule.steps(5e-4, [2, 4], [1.0, 0.5, 0.25], warmup_steps=1, warmup_start_lr=1e-5)
    feats, labels = [], []
    if kind == "hoi":
        sp = specs.hoi_g_spec(128, 4, 1, 0.1, 40)
        for i, B in enumerate((8, 8, 8)):
            f = synth.make_features(sp, B, seed=60 + i, dtype=torch.bfloat16)
            feats += [f[s_.name].cuda() for s_ in sp.segments]
            labels.append(synth.make_labels(sp, B, seed=60 + i))
    else:
        for mode, (B, D) in (("lam", (16, 7)), ("ttm", (4, 10)), ("asd", (4, 10))):
            sp = specs.hhi_g_spec(128, 4, 1, 0.1, mode)
            seg = (D,) if mode == "lam" else (D, D, D)
            f = synth.make_features(sp, B, seg, seed=70, dtype=torch.bfloat16)
            feats += [f[s_.name].cuda() for s_ in sp.segments]
            labels.append(synth.make_labels(sp, B, seg, seed=70))
    labels = torch.cat(labels).cuda()

    def run(schedule):
        cls = T.HoiPromptTranslatorTrainer if kind == "hoi" else T.PromptTranslatorTrainer
        extra = dict(vocab=40) if kind == "hoi" else {}
        tr = cls(hidden=128, heads=4, layers=1, device="cuda:0", dtype="bf16", lr_schedule=schedule, **extra)
        tr.load_state_dict(synth.make_state_dict(tr.spec, 3))
        assert tr.use_graphs
        losses, lrs = [], []
        for t in range(1, 7):
            if schedule is None:
                tr.hp["lr"] = lr_at(s, t - 1)
            losses.append(tr.train_step(feats, labels, graph_key=0).clone())
            lrs.append(tr.last_lr.clone())
        torch.cuda.synchronize()
        return [float(x) for x in losses], [float(x) for x in lrs], tr.engine.arena.param.clone()
    lg, lrs, pg = run(s)
    le, _, pe = run(None)
    assert lrs == [_f32(lr_at(s, t)) for t in range(6)]
    assert float((pg - pe).abs().max()) <= 5e-4 * float(pe.abs().max())
    assert all(abs(a - b) <= 2e-2 * abs(b) + 1e-4 for a, b in zip(lg, le))
    assert lg[-1] != lg[0]


def _sched_rank_worker(rank, world, port, q, fused, split, steps):
    os.environ["EGOT2_DP_FUSED"] = fused
    os.environ["EGOT2_DP_SPLIT"] = split
    import dataclasses

    import torch
    import torch.distributed as dist

    from egot2_b200 import specs, synth
    from egot2_b200.optim import LRSchedule
    from egot2_b200.trainer import TranslatorTrainer
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        sp = dataclasses.replace(specs.hhi_ttm_spec(128, 4, 1, 0.0, True), p_embed=0.0)
        B, seg = 16, (10, 10, 10)
        f = synth.make_features(sp, B, seg, seed=77, dtype=torch.bfloat16)
        lab = synth.make_labels(sp, B, seg, seed=77)
        lo, hi = rank * B // world, (rank + 1) * B // world
        tr = TranslatorTrainer(sp, f"cuda:{rank}", "bf16", use_graphs=True,
                               lr_schedule=LRSchedule.cosine(2e-3, 6, end_lr=1e-4, warmup_steps=2))
        assert (tr.peer is not None) == (fused == "1"), "the exchange path is not the one asked for"
        tr.load_state_dict(synth.make_state_dict(sp, 9))
        feats = [f[s.name][lo:hi].cuda() for s in sp.segments]
        labels = lab[lo:hi].cuda()
        for _ in range(steps):
            tr.train_step(feats, labels, graph_key=0)
        torch.cuda.synchronize()
        q.put((rank, {k: v.cpu() for k, v in tr.state_dict().items()}))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def _run_two_ranks(fused, split="0", steps=6):
    import socket

    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_sched_rank_worker, args=(r, 2, port, q, fused, split, steps)) for r in range(2)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=170) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return got[0], got[1]


@pytest.mark.gpu
def test_two_rank_scheduled_exchange():
    """Scheduled, 6 whole-step graph replays on 2 ranks: the peer-memory exchange (also split in two launches) leaves
    bit-identical ranks, and it agrees with the NCCL all-reduce path to bf16-training accuracy."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    a0, a1 = _run_two_ranks("1")
    for k in a0:
        assert torch.equal(a0[k], a1[k]), f"{k}: ranks diverged"
    s0, s1 = _run_two_ranks("1", split="1")
    n0, _ = _run_two_ranks("0")
    for k in a0:
        assert torch.equal(s0[k], s1[k]), f"{k}: ranks diverged (split exchange)"
        for other in (n0, s0):
            assert float((a0[k] - other[k]).abs().max()) <= 2e-4 + 1e-3 * float(other[k].abs().max()), k
