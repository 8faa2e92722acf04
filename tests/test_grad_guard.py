"""Gradient-norm clipping and skipping of non-finite steps on the device (egot2_grad_guard, egot2_grad_norm,
egot2_adam_step_fused_guard, egot2_dp_desc.guard) and the trainers' max_grad_norm.

CPU: the launch plans of guarded and unguarded steps, input checks, the optimizer-state round trip, the ABI mirrors.
GPU (-m gpu): the norm kernel against torch in float64, the guarded Adam / AdamW against clip_grad_norm_ + torch.optim, skipped
steps in the trainers, graph against eager, resume after a skip, and the two-rank exchange."""
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


@pytest.fixture(scope="module")
def built():
    from egot2_b200 import build
    return build.build()


def test_struct_layouts_match_header(built):
    """sizeof and every field offset of egot2_grad_guard and of the extended egot2_dp_desc equal the ctypes mirrors."""
    import subprocess
    import tempfile
    names = {"egot2_grad_guard": L.GradGuard, "egot2_dp_desc": L.DpDesc}
    fields = [(n, f[0]) for n, cls in names.items() for f in cls._fields_]
    prog = '#include <stdio.h>\n#include <stddef.h>\n#include "egot2.h"\nint main(){' + "".join(
        f'printf("{n} %zu\\n", sizeof({n}));' for n in names) + "".join(
        f'printf("{n}.{f} %zu\\n", offsetof({n}, {f}));' for n, f in fields) + "return 0;}"
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "probe.c")
        open(src, "w").write(prog)
        exe = os.path.join(td, "probe")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
        out = subprocess.check_output([exe], text=True)
    for line in out.strip().splitlines():
        n, v = line.split()
        if "." in n:
            st, f = n.split(".")
            assert getattr(names[st], f).offset == int(v), f"{n}: ctypes {getattr(names[st], f).offset} != C {v}"
        else:
            assert C.sizeof(names[n]) == int(v), f"{n}: ctypes {C.sizeof(names[n])} != C {v}"


# ------------------------------------------------------------------------------------------------ CPU: launch plans
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
def recorder(monkeypatch, built):
    """The C ABI replaced by a recorder and the CUDA-graph machinery by stand-ins, so the trainer's launch sequence runs on
    the CPU.  ('<capture>', ()) / ('</capture>', ()) delimit what a captured graph contains."""
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


def _hhi_trainer(**kw):
    from egot2_b200 import specs, synth
    from egot2_b200.trainer import TranslatorTrainer
    spec = specs.hhi_ttm_spec(128, 4, 1, 0.5, True)
    tr = TranslatorTrainer(spec, "cpu", "bf16", **kw)
    tr.load_state_dict(synth.make_state_dict(spec, 0))
    f = synth.make_features(spec, 4, (6, 6, 6), seed=1, dtype=torch.bfloat16)
    return tr, [f[s.name] for s in spec.segments], synth.make_labels(spec, 4, (6, 6, 6), seed=1)


def _captured(calls):
    names = [c[0] for c in calls]
    i, j = names.index("<capture>"), names.index("</capture>")
    return names[i + 1:j]


# The launch sequence of this HHI trainer without a guard or schedule as the parent commit records it with the same
# stand-ins: construction, the first graph step (warm-up, capture), a replay (nothing), an eager step.
_FWD_BWD = ["egot2_hhi_tok_table_fwd", "egot2_embed_fwd", "egot2_encoder_layer_fwd", "egot2_head_loss_fwd",
            "egot2_head_loss_bwd", "egot2_encoder_layer_bwd", "egot2_embed_bwd"]
_PARENT_GRAPH = _FWD_BWD + ["egot2_dropout_epoch_advance", "egot2_adam_step_fused_dev"]
_PARENT_PLAN = (["egot2_dropout_epoch_enable", "egot2_dropout_epoch_set", "egot2_cast_f32_to_bf16"] + _FWD_BWD
                + ["egot2_cast_f32_to_bf16", "<capture>"] + _PARENT_GRAPH + ["</capture>"]
                + _FWD_BWD + ["egot2_adam_step_fused", "egot2_dropout_epoch_advance"])
_GUARD_PAIR = ["egot2_grad_norm", "egot2_adam_step_fused_guard"]


def test_unguarded_step_plan_is_unchanged(recorder):
    tr, feats, labels = _hhi_trainer()
    assert tr.max_grad_norm is None
    tr.train_step(feats, labels, graph_key=0)
    tr.train_step(feats, labels, graph_key=0)
    tr.use_graphs = False
    tr.train_step(feats, labels)
    assert [c[0] for c in recorder] == _PARENT_PLAN


@pytest.mark.parametrize("scheduled", [False, True])
def test_guarded_graph_step_plan(scheduled, recorder):
    sched = LRSchedule.cosine(1e-3, 10, warmup_steps=2) if scheduled else None
    tr, feats, labels = _hhi_trainer(max_grad_norm=1.0, lr_schedule=sched)
    tr._step_dev.fill_(7)                     # stands for skips: the host must never rewrite the device count from step_count
    tr.train_step(feats, labels, graph_key=0)
    body = _captured(recorder)
    assert body.count("egot2_grad_norm") == 1 and body.count("egot2_adam_step_fused_guard") == 1
    assert "egot2_adam_step_fused_dev" not in body and "egot2_adam_step_fused_sched" not in body
    i = body.index("egot2_grad_norm")
    assert body[i + 1] == "egot2_adam_step_fused_guard"
    assert i > body.index("egot2_embed_bwd")                          # after the last backward launch
    assert [n for n in body if n not in _GUARD_PAIR + ["egot2_opt_advance"]] == _PARENT_GRAPH[:-1]
    (norm,) = [a for n, a in recorder if n == "egot2_grad_norm"]
    (adam,) = [a for n, a in recorder if n == "egot2_adam_step_fused_guard"]
    g = tr._guard_dev.data_ptr()
    assert norm[0] == tr.engine.arena.grad.data_ptr() and norm[2] == 1.0 and norm[3] == g
    assert norm[4] == tr._step_dev.data_ptr()
    assert adam[11] == tr._step_dev.data_ptr() and adam[16] == g and adam[15] == 0           # Adam, not AdamW
    assert adam[6] == (tr._lr_dev.data_ptr() if scheduled else None)
    # nothing filled the device count from step_count; without a schedule the side branch's increment ran (on the CPU
    # here), with one egot2_opt_advance advances it (recorded, not run)
    assert int(tr._step_dev[0]) == (7 if scheduled else 8)
    # set_max_grad_norm between replays: the descriptor's max_norm changes in place, no launch, no capture
    tr.set_max_grad_norm(0.25)
    del recorder[:]
    tr.train_step(feats, labels, graph_key=0)
    tr.train_step(feats, labels, graph_key=0)
    assert recorder == [] and len(tr._graphs) == 1
    assert bytes(tr._guard_dev[:4].numpy()) == bytes(C.c_float(0.25)) and float(tr.max_grad_norm) == 0.25
    assert float(tr._guard_field("max_norm")) == 0.25


@pytest.mark.parametrize("use_graphs", [False, True])
def test_guarded_eager_update_plan(use_graphs, recorder, monkeypatch):
    """Eager optimizer launches (no graphs, or EGOT2_GRAPH_UPDATE=0): the norm and the guarded Adam right after the advance,
    on the device step count, which the host never rewrites."""
    monkeypatch.setenv("EGOT2_GRAPH_UPDATE", "0")
    tr, feats, labels = _hhi_trainer(max_grad_norm=math.inf, use_graphs=use_graphs)
    tr._step_dev.fill_(3)
    for step in (1, 2):
        del recorder[:]
        tr.train_step(feats, labels, graph_key=0)
        names = [c[0] for c in recorder if not c[0].startswith("<")]
        i = names.index("egot2_grad_norm")
        assert names[i:i + 2] == _GUARD_PAIR and "egot2_embed_bwd" not in names[i:]
        assert names.count("egot2_grad_norm") == 1 and [n for n in names if "adam" in n] == _GUARD_PAIR[1:]
        assert int(tr._step_dev[0]) == 3 + step
    sched = LRSchedule.constant(1e-4)
    tr, feats, labels = _hhi_trainer(max_grad_norm=2.0, use_graphs=use_graphs, lr_schedule=sched)
    del recorder[:]
    tr.train_step(feats, labels, graph_key=0)
    names = [c[0] for c in recorder if not c[0].startswith("<")]
    i = names.index("egot2_opt_advance")
    assert names[i + 1:i + 3] == _GUARD_PAIR


def test_guarded_peer_exchange_receives_the_guard(recorder):
    got = []

    class FakePeer:
        def step(self, state, step, hp, stream, **kw):
            got.append(kw)
    tr, feats, labels = _hhi_trainer(max_grad_norm=1.0)
    tr.peer, tr.graph_update = FakePeer(), True
    tr.train_step(feats, labels, graph_key=0)
    tr.use_graphs = False
    tr.train_step(feats, labels)
    assert len(got) == 2 and all(k["guard"] is tr._guard_dev and k["step_dev"] is tr._step_dev for k in got)
    assert "egot2_grad_norm" not in [n for n, _ in recorder]          # the exchange computes the norm itself


def test_prompt_trainer_eager_guard_takes_the_fused_entry(recorder):
    """PromptTranslatorTrainer's eager step without a schedule uses the plain egot2_adam_step; with a guard it must run the
    norm and the fused guarded entry on the device step count."""
    from egot2_b200 import specs, synth
    from egot2_b200.trainer import PromptTranslatorTrainer
    tr = PromptTranslatorTrainer(hidden=128, heads=4, layers=1, device="cpu", max_grad_norm=1.0)
    assert not tr.use_graphs
    feats, labels = [], []
    for mode, (B, D) in (("lam", (4, 7)), ("ttm", (2, 4)), ("asd", (2, 4))):
        sp = specs.hhi_g_spec(128, 4, 1, 0.1, mode)
        seg = (D,) if mode == "lam" else (D, D, D)
        f = synth.make_features(sp, B, seg, seed=5, dtype=torch.bfloat16)
        feats += [f[s.name] for s in sp.segments]
        labels.append(synth.make_labels(sp, B, seg, seed=5))
    del recorder[:]
    tr.train_step(feats, torch.cat(labels))
    names = [n for n, _ in recorder]
    assert names[-2:] == _GUARD_PAIR and "egot2_adam_step" not in names
    assert int(tr._step_dev[0]) == 1 and tr._grad_clean


@pytest.mark.parametrize("bad", [0.0, -1.0, float("nan"), -math.inf])
def test_bad_max_grad_norm_is_rejected(bad, recorder):
    with pytest.raises(ValueError):
        _hhi_trainer(max_grad_norm=bad)
    tr, _, _ = _hhi_trainer(max_grad_norm=1.0)
    with pytest.raises(ValueError):
        tr.set_max_grad_norm(bad)
    assert tr.max_grad_norm == 1.0


def test_guard_misuse_is_rejected(recorder, monkeypatch):
    tr, _, _ = _hhi_trainer()
    for f in (lambda: tr.set_max_grad_norm(1.0), lambda: tr.last_grad_norm, lambda: tr.skipped_steps):
        with pytest.raises(ValueError):
            f()
    with pytest.raises(L.Egot2Error):          # the guard takes the step back on a skip: it needs the device step count
        tr.engine.adam_step({}, 1, fused=True, guard=torch.zeros(C.sizeof(L.GradGuard), dtype=torch.uint8))
    monkeypatch.setenv("EGOT2_DP_SPLIT", "1")
    with pytest.raises(ValueError, match="EGOT2_DP_SPLIT"):
        _hhi_trainer(max_grad_norm=1.0)


def test_optimizer_state_dict_round_trip(recorder):
    """max_grad_norm and skipped_steps travel with the optimizer state; the restored device count is step - skipped."""
    tr, feats, labels = _hhi_trainer(max_grad_norm=0.5, lr_schedule=LRSchedule.cosine(1e-3, 10))
    for _ in range(3):
        tr.train_step(feats, labels, graph_key=0)
    tr._guard_field("skipped", 2, dtype=torch.int32)         # what two skipped steps leave on the device
    sd = tr.optimizer_state_dict()
    assert sd["step"] == 3 and sd["max_grad_norm"] == 0.5 and sd["skipped_steps"] == 2
    tr2, _, _ = _hhi_trainer(max_grad_norm=4.0, lr_schedule=LRSchedule.constant(1.0))
    del recorder[:]
    tr2.load_optimizer_state_dict(sd)
    assert tr2.step_count == 3 and int(tr2._step_dev[0]) == 1 and int(tr2.skipped_steps) == 2
    assert tr2.max_grad_norm == 0.5 and float(tr2._guard_field("max_norm")) == 0.5
    assert [n for n, _ in recorder] == ["egot2_dropout_epoch_set"]
    with pytest.raises(ValueError):                           # saved with a guard, loaded into a trainer without one
        _hhi_trainer(lr_schedule=LRSchedule.constant(1.0))[0].load_optimizer_state_dict(sd)
    plain = _hhi_trainer()[0].optimizer_state_dict()
    assert plain["max_grad_norm"] is None and plain["skipped_steps"] == 0
    with pytest.raises(ValueError):                           # ... and the reverse
        _hhi_trainer(max_grad_norm=1.0)[0].load_optimizer_state_dict(plain)


# ------------------------------------------------------------------------------------------------ GPU: kernels
def _guard(max_norm=1.0, skipped=0, dev="cuda"):
    g = L.GradGuard(max_norm=max_norm, total_norm=0.0, coef=0.0, skip=0, skipped=skipped)
    return torch.frombuffer(bytearray(bytes(g)), dtype=torch.uint8).to(dev)


def _read_guard(t):
    return L.GradGuard.from_buffer_copy(t.cpu().numpy().tobytes())


def _norm_ws():
    return torch.zeros(int(L.load().egot2_grad_norm_workspace_bytes()), device="cuda", dtype=torch.uint8)


def _grad_norm(g, n, scale, guard, step, ws):
    L.call("egot2_grad_norm", g.data_ptr(), n, scale, guard.data_ptr(), None if step is None else step.data_ptr(),
           ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream)


def _lta_arena_numel():
    from egot2_b200 import specs
    from egot2_b200.engine import ParamArena
    return ParamArena(specs.hoi_lta_spec(512, 4, 8, 0.5), "meta").numel


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 3, 255, 256, 257, 4099, 1_000_003, "hoi_lta"])
@pytest.mark.parametrize("aligned", [True, False])
def test_grad_norm_matches_torch_float64(n, aligned):
    if n == "hoi_lta":
        n = _lta_arena_numel()
        assert n > 20_000_000
    torch.manual_seed(n % 1000)
    buf = torch.randn(n + 1, device="cuda")
    g = buf[:n] if aligned else buf[1:]           # a 4-byte offset takes the scalar path
    ws, scale = _norm_ws(), 0.5
    want = float(torch.linalg.vector_norm(g.double() * scale))
    results = []
    for _ in range(2):
        guard = _guard(max_norm=0.25 * want)
        _grad_norm(g, n, scale, guard, None, ws)
        results.append(_read_guard(guard))
    a, b = results
    assert abs(a.total_norm - want) <= 1e-6 * want
    assert bytes(a) == bytes(b)                   # bit-identical across launches
    assert a.skip == 0 and a.skipped == 0
    assert a.coef == np.float32(np.float32(0.25 * want) / (np.float32(a.total_norm) + np.float32(1e-6)))
    assert int(ws.sum()) != 0 and int(ws[-16:].sum()) == 0   # partial sums written; the grid counter reset itself


@pytest.mark.gpu
@pytest.mark.parametrize("value", [float("nan"), math.inf, -math.inf])
@pytest.mark.parametrize("where", ["first", "middle", "last"])
def test_grad_norm_detects_non_finite(value, where):
    n = 100_003
    g = torch.randn(n, device="cuda")
    g[{"first": 0, "middle": n // 2, "last": n - 1}[where]] = value
    guard, ws = _guard(max_norm=1.0, skipped=4), _norm_ws()
    step = torch.tensor([9], device="cuda", dtype=torch.int32)
    _grad_norm(g, n, 1.0, guard, step, ws)
    r = _read_guard(guard)
    assert r.skip == 1 and r.skipped == 5 and not math.isfinite(r.total_norm) and int(step) == 8
    g.normal_()                                  # the next, finite step clears the flag and leaves count and step alone
    _grad_norm(g, n, 1.0, guard, step, ws)
    r = _read_guard(guard)
    assert r.skip == 0 and r.skipped == 5 and math.isfinite(r.total_norm) and int(step) == 8


@pytest.mark.gpu
def test_grad_norm_huge_finite_elements_are_not_flagged():
    n = 1_000_000
    g = torch.randn(n, device="cuda")
    g[::9973] = 1e30
    guard, ws = _guard(max_norm=1.0), _norm_ws()
    _grad_norm(g, n, 1.0, guard, None, ws)
    r = _read_guard(guard)
    want = float(torch.linalg.vector_norm(g.double()))
    assert r.skip == 0 and abs(r.total_norm - want) <= 1e-6 * want and r.coef > 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("decoupled", [False, True])
@pytest.mark.parametrize("scheduled", [False, True])
@pytest.mark.parametrize("clip", ["active", "inactive"])
def test_guarded_adam_matches_clip_grad_norm_and_torch(decoupled, scheduled, clip):
    """egot2_grad_norm + egot2_adam_step_fused_guard == clip_grad_norm_ + torch.optim.Adam / AdamW (+ LambdaLR) over 8 steps."""
    s = LRSchedule.cosine(1e-3, 6, end_lr=1e-5, warmup_steps=2, warmup_start_lr=1e-5)
    torch.manual_seed(3)
    n = 10007
    max_norm = 40.0 if clip == "active" else 1e4      # the norm of randn(n) * [0.8, 1.2] is ~80 - 120
    p = torch.randn(n, device="cuda")
    ref = p.clone().requires_grad_(True)
    wd = 0.1 if decoupled else 0.01
    opt = (torch.optim.AdamW if decoupled else torch.optim.Adam)([ref], lr=s.base_lr if scheduled else 2e-3, weight_decay=wd)
    if scheduled:
        from test_lr_schedule import lr_at
        lam = torch.optim.lr_scheduler.LambdaLR(opt, lambda t: lr_at(s, t) / s.base_lr)
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    shadow = torch.empty(n, device="cuda", dtype=torch.bfloat16)
    step = torch.zeros(1, device="cuda", dtype=torch.int32)
    lr = torch.zeros(1, device="cuda", dtype=torch.float32)
    sched = torch.frombuffer(bytearray(bytes(s.pack())), dtype=torch.uint8).cuda()
    guard, ws = _guard(max_norm), _norm_ws()
    st = torch.cuda.current_stream().cuda_stream
    for i in range(8):
        g = torch.randn(n, device="cuda") * (0.8 + 0.05 * i)
        ref.grad = g.clone()
        want_norm = float(torch.nn.utils.clip_grad_norm_([ref], max_norm))
        opt.step()
        if scheduled:
            lam.step()
            L.call("egot2_opt_advance", step.data_ptr(), sched.data_ptr(), lr.data_ptr(), st)
        else:
            step.add_(1)
        _grad_norm(g, n, 1.0, guard, step, ws)
        L.call("egot2_adam_step_fused_guard", p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), n, 2e-3,
               lr.data_ptr() if scheduled else None, 0.9, 0.999, 1e-8, wd, step.data_ptr(), 1.0, shadow.data_ptr(), 1,
               int(decoupled), guard.data_ptr(), st)
        r = _read_guard(guard)
        assert abs(r.total_norm - want_norm) <= 1e-6 * want_norm
        assert (r.coef < 1.0) == (clip == "active") and r.skip == 0
        assert float((p - ref.detach()).abs().max()) < 1e-6
        assert float(g.abs().max()) == 0.0 and torch.equal(shadow, p.to(torch.bfloat16))
    assert int(step) == 8


# ------------------------------------------------------------------------------------------------ GPU: trainers
def _hhi_setup(batch=16, seed=1):
    import dataclasses
    from egot2_b200 import specs, synth
    spec = dataclasses.replace(specs.hhi_ttm_spec(128, 4, 1, 0.0, True), p_embed=0.0)
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


def _snapshot(tr):
    a = tr.engine.arena
    return [a.param.clone(), a.shadow.clone(), tr.opt_state["m"].clone(), tr.opt_state["v"].clone()]


@contextlib.contextmanager
def _nan_feature(feats):
    """A NaN in one element of the first feature tensor, in place (graph replays read these buffers), restored after."""
    old = feats[0][0, 0, 0].clone()
    feats[0][0, 0, 0] = float("nan")
    try:
        yield
    finally:
        feats[0][0, 0, 0] = old


@pytest.mark.gpu
def test_gradient_arena_padding_stays_zero():
    """The arena's alignment padding never receives a gradient, so it adds nothing to the norm."""
    spec, feats, labels = _hhi_setup()
    tr = _hhi_trainer_gpu(spec, use_graphs=False)
    tr._fwd_bwd(feats, labels, seed=1)
    a = tr.engine.arena
    used = torch.zeros(a.numel, dtype=torch.bool, device="cuda")
    for name, o in a.offsets.items():
        used[o:o + a.view(name).numel()] = True
    assert int((~used).sum()) > 0 and float(a.grad[~used].abs().max()) == 0.0
    assert float(a.grad[used].abs().max()) > 0.0


@pytest.mark.gpu
def test_skipped_step_whole_step_graph():
    """A NaN feature: the whole-step graph leaves parameters, shadow and moments bit for bit, clears the gradient, counts the
    skip and keeps the device step count; the next step uses the lr of the applied count and trains on."""
    from test_lr_schedule import lr_at
    s = LRSchedule.cosine(5e-4, 10, end_lr=1e-5, warmup_steps=2, warmup_start_lr=1e-5)
    spec, feats, labels = _hhi_setup()
    tr = _hhi_trainer_gpu(spec, use_graphs=True, lr_schedule=s, max_grad_norm=1.0)
    assert tr.graph_update
    for _ in range(2):
        tr.train_step(feats, labels, graph_key=0)
    before = _snapshot(tr)
    with _nan_feature(feats):
        loss = tr.train_step(feats, labels, graph_key=0)
    torch.cuda.synchronize()
    assert not math.isfinite(float(loss)) and not math.isfinite(float(tr.last_grad_norm))
    for x, y in zip(before, _snapshot(tr)):
        assert torch.equal(x, y)
    assert float(tr.engine.arena.grad.abs().max()) == 0.0
    assert int(tr.skipped_steps) == 1 and int(tr._step_dev) == 2 and tr.step_count == 3
    loss = tr.train_step(feats, labels, graph_key=0)
    torch.cuda.synchronize()
    assert math.isfinite(float(loss)) and math.isfinite(float(tr.last_grad_norm))
    assert float(tr.last_lr) == float(np.float32(lr_at(s, 2))) and int(tr._step_dev) == 3
    assert not torch.equal(tr.engine.arena.param, before[0]) and len(tr._graphs) == 1


@pytest.mark.gpu
def test_guarded_graph_matches_guarded_eager_with_clipping():
    """Clipping active on every step: the guarded whole-step graph == the guarded eager trainer.

    In both, every step's first-moment update reveals the gradient Adam applied, whose norm must be max_grad_norm.  The
    parameters are compared by the L2 norm of the difference relative to how far training moved them, not element by element:
    an element whose gradient is fp32-atomic rounding noise moves by about +-lr per step in a random direction under Adam,
    whatever the scale, so after 8 steps at lr 5e-4 single elements of two runs of the SAME path differ by 1e-3 and more."""
    spec, feats, labels = _hhi_setup()
    max_norm = 0.05
    tg = _hhi_trainer_gpu(spec, use_graphs=True, max_grad_norm=max_norm)
    te = _hhi_trainer_gpu(spec, use_graphs=False, max_grad_norm=max_norm)
    p0 = te.engine.arena.param.clone()
    b1 = tg.hp["betas"][0]
    lg, le, ng, ne = [], [], [], []
    for _ in range(8):
        for tr, losses, norms in ((tg, lg, ng), (te, le, ne)):
            m0 = tr.opt_state["m"].clone() if "m" in tr.opt_state else torch.zeros_like(p0)
            losses.append(float(tr.train_step(feats, labels, graph_key=0 if tr is tg else None)))
            norms.append(float(tr.last_grad_norm))
            applied = (tr.opt_state["m"].double() - b1 * m0.double()) / (1.0 - b1)
            assert abs(float(applied.norm()) - max_norm) <= 1e-3 * max_norm
    assert all(x > max_norm for x in ng + ne)                         # clipping was active
    assert all(abs(a - b) <= 2e-2 * b for a, b in zip(ng, ne))
    pg, pe = tg.engine.arena.param, te.engine.arena.param
    assert float((pg - pe).norm()) <= 2e-2 * float((pe - p0).norm())
    assert all(abs(a - b) <= 2e-2 * abs(b) + 1e-4 for a, b in zip(lg, le))
    assert int(tg._step_dev) == 8 and int(te._step_dev) == 8 and int(tg.skipped_steps) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("graphs", ["1", "0"])
@pytest.mark.parametrize("kind", ["hhi", "hoi"])
def test_prompt_trainers_clip_and_skip(kind, graphs, monkeypatch):
    """EgoT2-g trainers (HHI: Adam, HOI: AdamW), graph replay and eager: the first moment's update reveals the gradient the
    optimizer applied, whose norm must be min(last_grad_norm, max_grad_norm); a NaN batch is skipped bit for bit."""
    from egot2_b200 import specs, synth, trainer as T
    monkeypatch.setenv("EGOT2_G_GRAPH", graphs)
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
    cls = T.HoiPromptTranslatorTrainer if kind == "hoi" else T.PromptTranslatorTrainer
    extra = dict(vocab=40) if kind == "hoi" else {}
    max_norm = 0.05
    tr = cls(hidden=128, heads=4, layers=1, device="cuda:0", dtype="bf16", max_grad_norm=max_norm, **extra)
    tr.load_state_dict(synth.make_state_dict(tr.spec, 3))
    assert tr.use_graphs == (graphs == "1")
    b1 = tr.hp["betas"][0]
    for _ in range(3):
        m0 = tr.opt_state["m"].clone() if "m" in tr.opt_state else torch.zeros_like(tr.engine.arena.param)
        tr.train_step(feats, labels, graph_key=0)
        torch.cuda.synchronize()
        applied = (tr.opt_state["m"].double() - b1 * m0.double()) / (1.0 - b1)
        norm = float(tr.last_grad_norm)
        assert norm > max_norm
        assert abs(float(applied.norm()) - max_norm) <= 1e-3 * max_norm
    before = _snapshot(tr)
    with _nan_feature(feats):
        tr.train_step(feats, labels, graph_key=0)
    torch.cuda.synchronize()
    for x, y in zip(before, _snapshot(tr)):
        assert torch.equal(x, y)
    assert float(tr.engine.arena.grad.abs().max()) == 0.0
    assert int(tr.skipped_steps) == 1 and int(tr._step_dev) == 3 and tr.step_count == 4
    loss = tr.train_step(feats, labels, graph_key=0)
    torch.cuda.synchronize()
    assert math.isfinite(float(loss)) and int(tr._step_dev) == 4


@pytest.mark.gpu
def test_resume_after_a_skipped_step():
    """Steps 1-2, a NaN step 3, save, a fresh trainer loads and runs steps 4-6 == six uninterrupted steps (parameters by the L2
    norm of the difference relative to how far training moved them, as the schedule's resume test)."""
    s = LRSchedule.cosine(5e-4, 8, warmup_steps=2, warmup_start_lr=1e-5)
    spec, feats, labels = _hhi_setup()
    kw = dict(use_graphs=True, lr_schedule=s, max_grad_norm=0.5)

    def run(tr, steps):
        for t in steps:
            with (_nan_feature(feats) if t == 3 else contextlib.nullcontext()):
                tr.train_step(feats, labels, graph_key=0)
        torch.cuda.synchronize()
    full = _hhi_trainer_gpu(spec, **kw)
    p0 = full.engine.arena.param.clone()
    run(full, range(1, 7))
    p_full = full.engine.arena.param.clone()
    assert int(full.skipped_steps) == 1 and int(full._step_dev) == 5
    del full
    first = _hhi_trainer_gpu(spec, **kw)
    run(first, range(1, 4))
    sd, osd = first.state_dict(), first.optimizer_state_dict()
    assert osd["step"] == 3 and osd["skipped_steps"] == 1 and osd["max_grad_norm"] == 0.5
    del first
    tr = _hhi_trainer_gpu(spec, **kw)
    tr.load_state_dict(sd)
    tr.load_optimizer_state_dict(osd)
    assert int(tr._step_dev) == 2 and int(tr.skipped_steps) == 1
    run(tr, range(4, 7))
    assert int(tr._step_dev) == 5 and int(tr.skipped_steps) == 1
    moved = float((p_full - p0).norm())
    assert float((tr.engine.arena.param - p_full).norm()) <= 2e-2 * moved


# ------------------------------------------------------------------------------------------------ GPU: two ranks
def _guard_rank_worker(rank, world, port, q, fused, nan_rank, steps):
    os.environ["EGOT2_DP_FUSED"] = fused
    import dataclasses

    import torch
    import torch.distributed as dist

    from egot2_b200 import specs, synth
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
        tr = TranslatorTrainer(sp, f"cuda:{rank}", "bf16", use_graphs=True, max_grad_norm=0.05)
        assert (tr.peer is not None) == (fused == "1"), "the exchange path is not the one asked for"
        tr.load_state_dict(synth.make_state_dict(sp, 9))
        feats = [f[s.name][lo:hi].cuda() for s in sp.segments]
        labels = lab[lo:hi].cuda()
        norms = []
        for t in range(steps):
            nan = rank == nan_rank and t == steps - 1
            with (_nan_feature(feats) if nan else contextlib.nullcontext()):
                tr.train_step(feats, labels, graph_key=0)
            norms.append(tr.last_grad_norm.clone())
        torch.cuda.synchronize()
        q.put((rank, dict(norms=[float(x) for x in norms], skipped=int(tr.skipped_steps), step=int(tr._step_dev),
                          params={k: v.cpu() for k, v in tr.state_dict().items()})))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def _run_two_ranks(fused, nan_rank=-1, steps=4):
    import socket

    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_guard_rank_worker, args=(r, 2, port, q, fused, nan_rank, steps)) for r in range(2)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=170) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return got[0], got[1]


@pytest.mark.gpu
@pytest.mark.parametrize("fused", ["1", "0"])
def test_two_rank_guarded_exchange(fused):
    """Peer-memory exchange and NCCL: both ranks see the identical norm and keep bit-identical parameters; the first norm
    matches one rank on the whole batch (to the class-weighted CE's per-shard normalisation); a NaN on one rank only makes
    both ranks skip."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import dataclasses
    from egot2_b200 import specs, synth
    r0, r1 = _run_two_ranks(fused)
    assert r0["norms"] == r1["norms"] and r0["skipped"] == r1["skipped"] == 0
    for k in r0["params"]:
        assert torch.equal(r0["params"][k], r1["params"][k]), f"{k}: ranks diverged"
    sp = dataclasses.replace(specs.hhi_ttm_spec(128, 4, 1, 0.0, True), p_embed=0.0)
    f = synth.make_features(sp, 16, (10, 10, 10), seed=77, dtype=torch.bfloat16)
    one = _hhi_trainer_gpu(sp, use_graphs=True, max_grad_norm=0.05)
    one.load_state_dict(synth.make_state_dict(sp, 9))
    one.train_step([f[s.name].cuda() for s in sp.segments], synth.make_labels(sp, 16, (10, 10, 10), seed=77).cuda(),
                   graph_key=0)
    want = float(one.last_grad_norm)
    assert abs(r0["norms"][0] - want) <= 5e-2 * want
    n0, n1 = _run_two_ranks(fused, nan_rank=1)
    for r in (n0, n1):
        assert r["skipped"] == 1 and r["step"] == 3 and not math.isfinite(r["norms"][-1])
    for k in n0["params"]:
        assert torch.equal(n0["params"][k], n1["params"][k]), f"{k}: ranks diverged after a skip"
