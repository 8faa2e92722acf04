"""Parameter groups of the fused trainers (optim.ParamGroup, egot2_param_groups, egot2_adam_step_fused_groups,
egot2_grad_norm_groups, egot2_dp_desc.groups): per-group weight decay and lr multipliers, and frozen parameters.

CPU: group resolution and its input checks, the launch plans with and without groups, the ABI mirrors, the optimizer-state
round trip.  GPU (-m gpu): the grouped Adam / AdamW against torch.optim with the equivalent param groups (with LambdaLR and
with clip_grad_norm_ over the trainable parameters), NaNs in frozen and in trainable gradients, the no-op check against the
ungrouped launch inside a replayed graph, frozen parameters in every trainer, graph against eager, set_param_group between
replays, resume, and the two-rank exchange."""
import contextlib
import ctypes as C
import math
import os

import numpy as np
import pytest
import torch

from egot2_b200 import _lib as L
from egot2_b200.optim import LRSchedule, ParamGroup

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# frozen first, so that the biases of the frozen layer stay frozen (the first matching group wins)
GROUPS = [ParamGroup("*layers.0.*", frozen=True), ParamGroup("proj*", lr_mult=0.1),
          ParamGroup(["*bias", "*norm*", "ln.*"], weight_decay=0.0)]


@pytest.fixture(scope="module")
def built():
    from egot2_b200 import build
    return build.build()


def test_struct_layouts_match_header(built):
    """sizeof and every field offset of egot2_param_groups and of the extended egot2_dp_desc equal the ctypes mirrors."""
    import subprocess
    import tempfile
    names = {"egot2_param_groups": L.ParamGroups, "egot2_dp_desc": L.DpDesc}
    fields = [(n, f[0]) for n, cls in names.items() for f in cls._fields_]
    prog = '#include <stdio.h>\n#include <stddef.h>\n#include "egot2.h"\nint main(){' + "".join(
        f'printf("{n} %zu\\n", sizeof({n}));' for n in names) + "".join(
        f'printf("{n}.{f} %zu\\n", offsetof({n}, {f}));' for n, f in fields) + \
        'printf("max %d\\n", EGOT2_MAX_PARAM_GROUPS);return 0;}'
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "probe.c")
        open(src, "w").write(prog)
        exe = os.path.join(td, "probe")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
        out = subprocess.check_output([exe], text=True)
    for line in out.strip().splitlines():
        n, v = line.split()
        if n == "max":
            assert L.MAX_PARAM_GROUPS == int(v)
        elif "." in n:
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

    def pool(self):
        return None


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


def _names(calls):
    return [c[0] for c in calls]


def _captured(calls):
    names = _names(calls)
    i, j = names.index("<capture>"), names.index("</capture>")
    return names[i + 1:j]


# The launch sequence of this HHI trainer without groups, guard or schedule as the parent commit records it with the same
# stand-ins: construction, the first graph step (warm-up, capture), a replay (nothing), an eager step.
_FWD_BWD = ["egot2_hhi_tok_table_fwd", "egot2_embed_fwd", "egot2_encoder_layer_fwd", "egot2_head_loss_fwd",
            "egot2_head_loss_bwd", "egot2_encoder_layer_bwd", "egot2_embed_bwd"]
_PARENT_GRAPH = _FWD_BWD + ["egot2_dropout_epoch_advance", "egot2_adam_step_fused_dev"]
_PARENT_PLAN = (["egot2_dropout_epoch_enable", "egot2_dropout_epoch_set", "egot2_cast_f32_to_bf16"] + _FWD_BWD
                + ["egot2_cast_f32_to_bf16", "<capture>"] + _PARENT_GRAPH + ["</capture>"]
                + _FWD_BWD + ["egot2_adam_step_fused", "egot2_dropout_epoch_advance"])
_GROUPED = "egot2_adam_step_fused_groups"


def _plan(tr, feats, labels):
    tr.train_step(feats, labels, graph_key=0)
    tr.train_step(feats, labels, graph_key=0)
    tr.use_graphs = False
    tr.train_step(feats, labels)


def test_ungrouped_plan_is_unchanged(recorder):
    tr, feats, labels = _hhi_trainer()
    assert tr.param_groups is None and tr._groups is None
    _plan(tr, feats, labels)
    assert _names(recorder) == _PARENT_PLAN


@pytest.mark.parametrize("guard", [False, True])
def test_grouped_plan_has_the_same_launches(guard, recorder):
    """Whole-step graph and eager step: the same launches as without groups, with the grouped entry (and, with a guard, the
    grouped norm) in place of the ungrouped one; it reads the descriptor, the block map and the device step count."""
    kw = dict(max_grad_norm=1.0) if guard else {}
    tr, feats, labels = _hhi_trainer(**kw)
    _plan(tr, feats, labels)
    ref = list(recorder)
    del recorder[:]
    tr, feats, labels = _hhi_trainer(param_groups=GROUPS, weight_decay=0.01, **kw)
    _plan(tr, feats, labels)
    got = _names(recorder)
    assert len(got) == len(ref)
    swap = {"egot2_adam_step_fused_dev": _GROUPED, "egot2_adam_step_fused": _GROUPED,
            "egot2_adam_step_fused_guard": _GROUPED, "egot2_grad_norm": "egot2_grad_norm_groups"}
    assert got == [swap.get(n, n) for n in _names(ref)]
    assert _captured(recorder)[-1] == _GROUPED
    desc, bmap = tr._groups
    adams = [a for n, a in recorder if n == _GROUPED]
    assert len(adams) == 2
    for a in adams:
        assert a[10] == tr._step_dev.data_ptr() and a[16] == desc.data_ptr() and a[17] == bmap.data_ptr()
        assert a[14] == 0 and a[15] == (tr._guard_dev.data_ptr() if guard else None)
    if guard:
        for a in [a for n, a in recorder if n == "egot2_grad_norm_groups"]:
            assert a[5] == desc.data_ptr() and a[6] == bmap.data_ptr()


def _prompt_batch(kind):
    from egot2_b200 import specs, synth
    feats, labels = [], []
    if kind == "hoi":
        sp = specs.hoi_g_spec(128, 4, 1, 0.1, 40)
        for i in range(3):
            f = synth.make_features(sp, 4, seed=60 + i, dtype=torch.bfloat16)
            feats += [f[s.name] for s in sp.segments]
            labels.append(synth.make_labels(sp, 4, seed=60 + i))
    else:
        for mode, (B, D) in (("lam", (4, 7)), ("ttm", (2, 4)), ("asd", (2, 4))):
            sp = specs.hhi_g_spec(128, 4, 1, 0.1, mode)
            seg = (D,) if mode == "lam" else (D, D, D)
            f = synth.make_features(sp, B, seg, seed=5, dtype=torch.bfloat16)
            feats += [f[s.name] for s in sp.segments]
            labels.append(synth.make_labels(sp, B, seg, seed=5))
    return feats, torch.cat(labels)


@pytest.mark.parametrize("graphs", ["1", "0"])
@pytest.mark.parametrize("kind", ["hhi", "hoi"])
def test_prompt_trainer_plans(kind, graphs, recorder, monkeypatch):
    """EgoT2-g trainers, graph replay and eager: two steps issue as many launches with groups as without, and the optimizer
    launch is the grouped entry on the device step count (HOI: AdamW).  The HHI eager step without groups runs the unfused
    egot2_adam_step, so every forward re-casts the bf16 shadow; the grouped launch writes the shadow itself, which saves
    those casts."""
    from egot2_b200 import trainer as T
    monkeypatch.setenv("EGOT2_G_GRAPH", graphs)
    cls = T.HoiPromptTranslatorTrainer if kind == "hoi" else T.PromptTranslatorTrainer
    extra = dict(vocab=40) if kind == "hoi" else {}
    feats, labels = _prompt_batch(kind)
    plans = []
    for groups in (None, [ParamGroup("proj*", frozen=True), ParamGroup("*bias", weight_decay=0.0)]):
        del recorder[:]
        tr = cls(hidden=128, heads=4, layers=1, device="cpu", param_groups=groups, **extra)
        assert tr.use_graphs == (graphs == "1")
        for _ in range(2):
            tr.train_step(feats, labels, graph_key=0)
        plans.append(_names(recorder))
    plain, grouped = plans
    if kind == "hhi" and graphs == "0":
        cast = "egot2_cast_f32_to_bf16"
        assert grouped.count(cast) < plain.count(cast)
        plain, grouped = [n for n in plain if n != cast], [n for n in grouped if n != cast]
    assert len(plain) == len(grouped)
    assert [n for n in plain if "adam" not in n] == [n for n in grouped if "adam" not in n]
    assert [n for n in grouped if "adam" in n] == [_GROUPED] * 2
    assert int(tr._step_dev[0]) == 2 and tr._grad_clean
    (a, _) = [a for n, a in recorder if n == _GROUPED]
    assert a[14] == (1 if kind == "hoi" else 0) and a[16] == tr._groups[0].data_ptr()


def test_peer_exchange_receives_the_groups(recorder):
    got = []

    class FakePeer:
        def step(self, state, step, hp, stream, **kw):
            got.append(kw)
    counts = []
    for groups in (None, GROUPS):
        tr, feats, labels = _hhi_trainer(param_groups=groups)
        tr.peer, tr.graph_update = FakePeer(), True
        del recorder[:]
        tr.train_step(feats, labels, graph_key=0)
        tr.use_graphs = False
        tr.train_step(feats, labels)
        counts.append(len(recorder))
    assert counts[0] == counts[1]
    assert all("groups" not in k for k in got[:2])
    assert len(got) == 4 and all(k["groups"] is tr._groups and k["step_dev"] is tr._step_dev for k in got[2:])


def test_peer_desc_carries_the_groups(built, monkeypatch):
    """PeerExchange.step writes the descriptor and block-map pointers into egot2_dp_desc (NULL without groups)."""
    from egot2_b200.parallel import PeerExchange
    descs = []

    class Eng:
        device = torch.device("cpu")
        dtype = "bf16"

        class arena:
            numel = 128
            param = torch.zeros(128)
            grad = torch.zeros(128)
            shadow_fresh = False
    ex = PeerExchange.__new__(PeerExchange)
    ex.engine, ex.desc = Eng, L.DpDesc()
    hp = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0)
    groups = (torch.zeros(C.sizeof(L.ParamGroups), dtype=torch.uint8), torch.zeros(2, dtype=torch.uint8))
    monkeypatch.setattr(L, "call", lambda name, d, *a: descs.append((d._obj.groups, d._obj.block_group)))
    monkeypatch.setattr(torch.cuda, "device", lambda d: contextlib.nullcontext())
    ex.step({}, 1, hp, 0, step_dev=torch.zeros(1, dtype=torch.int32))
    ex.step({}, 1, hp, 0, step_dev=torch.zeros(1, dtype=torch.int32), groups=groups)
    assert descs[0] == (None, None)
    assert descs[1] == (groups[0].data_ptr(), groups[1].data_ptr())


# ------------------------------------------------------------------------------------------------ CPU: resolution, checks
def test_group_resolution(recorder):
    """First match wins, unmatched parameters form group 0 with the trainer's weight decay, weight_decay=None inherits it."""
    tr, _, _ = _hhi_trainer(weight_decay=0.05, param_groups=[
        ParamGroup("proj_lam.*", frozen=True), ParamGroup(["proj_*", "task_embed"], lr_mult=0.5),
        ParamGroup("*bias", weight_decay=0.0)])
    a = tr.engine.arena
    bmap = tr._groups[1].numpy()
    assert bmap.size == (a.numel + 63) // 64

    def group(name):
        ks = set(bmap[a.offsets[name] // 64:(a.offsets[name] + a.view(name).numel() - 1) // 64 + 1].tolist())
        assert len(ks) == 1
        return ks.pop()
    assert group("proj_lam.weight") == group("proj_lam.bias") == 1            # not 3: the first match wins
    assert group("proj_ttm.bias") == group("task_embed") == 2
    assert group("transformer_encoder.layers.0.linear1.bias") == group("ln.bias") == 3
    assert group("transformer_encoder.layers.0.linear1.weight") == group("linear_head.1.weight") == 0
    assert tr._group_hp == [(1.0, 0.05, False), (1.0, 0.05, True), (0.5, 0.05, False), (1.0, 0.0, False)]
    d = L.ParamGroups.from_buffer_copy(tr._groups[0].numpy().tobytes())
    assert d.n_groups == 4 and list(d.frozen)[:4] == [0, 1, 0, 0]
    assert np.allclose(list(d.lr_mult)[:4], [1.0, 1.0, 0.5, 1.0]) and np.allclose(list(d.weight_decay)[:4], [0.05] * 3 + [0])


def test_stacked_head_biases_split_across_groups_are_rejected(recorder):
    """The LTA head's biases sit back to back inside 64-element blocks: splitting them across groups names both."""
    from egot2_b200 import specs
    from egot2_b200.trainer import TranslatorTrainer
    spec = specs.hoi_lta_spec(128, 1, 4, 0.5)
    with pytest.raises(ValueError, match=r"head\.projections\.0\.bias.*head\.projections\.1\.bias"):
        TranslatorTrainer(spec, "cpu", "bf16", param_groups=[ParamGroup("head.projections.0.bias", weight_decay=0.0)])
    tr = TranslatorTrainer(spec, "cpu", "bf16", param_groups=[ParamGroup("head.projections.*.bias", weight_decay=0.0)])
    assert tr._group_hp[1] == (1.0, 0.0, False)


@pytest.mark.parametrize("bad", [-1.0, float("nan"), math.inf])
def test_bad_hyperparameters_are_rejected(bad, recorder):
    for kw in (dict(lr_mult=bad), dict(weight_decay=bad)):
        with pytest.raises(ValueError):
            ParamGroup("*", **kw)
    tr, _, _ = _hhi_trainer(param_groups=[ParamGroup("*bias", lr_mult=0.0)])
    for kw in (dict(lr_mult=bad), dict(weight_decay=bad)):
        with pytest.raises(ValueError):
            tr.set_param_group(1, **kw)
    assert tr._group_hp[1] == (0.0, 0.0, False)


def test_bad_groups_are_rejected(recorder):
    with pytest.raises(ValueError, match="matches no parameter"):
        _hhi_trainer(param_groups=[ParamGroup(["*bias", "no_such_param*"])])
    with pytest.raises(ValueError, match="at most 8"):
        _hhi_trainer(param_groups=[ParamGroup(f"*{i}*") for i in range(8)])
    _hhi_trainer(param_groups=[ParamGroup("*bias")] * 7)                       # 8 with the default group
    with pytest.raises(ValueError):
        ParamGroup([])
    tr, _, _ = _hhi_trainer()
    with pytest.raises(ValueError):
        tr.set_param_group(0, lr_mult=1.0)
    tr, _, _ = _hhi_trainer(param_groups=GROUPS)
    with pytest.raises(ValueError):
        tr.set_param_group(4, lr_mult=1.0)
    with pytest.raises(L.Egot2Error):
        tr.engine.adam_step({}, 1, fused=True, groups=tr._groups)              # needs the device step count


def test_set_param_group_rewrites_the_descriptor_without_a_launch(recorder):
    tr, feats, labels = _hhi_trainer(param_groups=GROUPS, weight_decay=0.01)
    tr.train_step(feats, labels, graph_key=0)
    del recorder[:]
    tr.set_param_group(2, lr_mult=0.25)
    tr.set_param_group(0, weight_decay=0.5)
    tr.train_step(feats, labels, graph_key=0)
    assert recorder == [] and len(tr._graphs) == 1
    d = L.ParamGroups.from_buffer_copy(tr._groups[0].numpy().tobytes())
    assert d.lr_mult[2] == 0.25 and d.weight_decay[2] == np.float32(0.01) and d.weight_decay[0] == 0.5
    assert d.frozen[1] == 1


def test_optimizer_state_dict_round_trip(recorder):
    tr, feats, labels = _hhi_trainer(param_groups=GROUPS, weight_decay=0.01)
    tr.train_step(feats, labels, graph_key=0)
    tr.set_param_group(2, lr_mult=0.3)
    sd = tr.optimizer_state_dict()
    assert [g["patterns"] for g in sd["param_groups"]] == [None] + [list(g.patterns) for g in GROUPS]
    assert sd["param_groups"][2]["lr_mult"] == 0.3 and sd["param_groups"][1]["frozen"]
    tr2, _, _ = _hhi_trainer(param_groups=GROUPS, weight_decay=0.01)
    del recorder[:]
    tr2.load_optimizer_state_dict(sd)
    assert tr2._group_hp == tr._group_hp and torch.equal(tr2._groups[0], tr._groups[0])
    assert _names(recorder) == ["egot2_dropout_epoch_set"]
    for other in (None, GROUPS[:2], [ParamGroup("*layers.0.*"), *GROUPS[1:]]):      # none, fewer, not frozen
        with pytest.raises(ValueError, match="param"):
            _hhi_trainer(param_groups=other)[0].load_optimizer_state_dict(sd)
    plain = _hhi_trainer()[0].optimizer_state_dict()
    assert plain["param_groups"] is None
    with pytest.raises(ValueError):
        _hhi_trainer(param_groups=GROUPS)[0].load_optimizer_state_dict(plain)


# ------------------------------------------------------------------------------------------------ GPU: kernels
def _guard(max_norm=1.0):
    g = L.GradGuard(max_norm=max_norm, total_norm=0.0, coef=0.0, skip=0, skipped=0)
    return torch.frombuffer(bytearray(bytes(g)), dtype=torch.uint8).to("cuda")


def _read_guard(t):
    return L.GradGuard.from_buffer_copy(t.cpu().numpy().tobytes())


def _arena(kind):
    from egot2_b200 import specs
    from egot2_b200.engine import ParamArena
    spec = {"hhi": specs.hhi_ttm_spec(), "pnr": specs.hoi_pnr_spec(), "lta": specs.hoi_lta_spec(512, 4, 8, 0.5)}[kind]
    return ParamArena(spec, "meta")


def _device_groups(arena, groups, wd):
    from egot2_b200.optim import pack_param_groups, resolve_param_groups
    bmap = resolve_param_groups(groups, arena.shapes, arena.offsets, arena.numel)
    hp = [(1.0, wd, False)] + [(g.lr_mult, wd if g.weight_decay is None else g.weight_decay, g.frozen) for g in groups]
    desc = torch.frombuffer(bytearray(bytes(pack_param_groups(hp))), dtype=torch.uint8).cuda()
    return desc, torch.from_numpy(bmap).cuda(), hp


def _group_of(arena, bmap):
    bm = bmap.cpu().numpy()
    return {n: int(bm[arena.offsets[n] // 64]) for n in arena.shapes}


@pytest.mark.gpu
@pytest.mark.parametrize("clip", [False, True])
@pytest.mark.parametrize("scheduled", [False, True])
@pytest.mark.parametrize("decoupled", [False, True])
@pytest.mark.parametrize("kind", ["hhi", "pnr", "lta"])
def test_grouped_adam_matches_torch(kind, decoupled, scheduled, clip):
    """egot2_adam_step_fused_groups (+ egot2_grad_norm_groups) over a translator arena == torch.optim.Adam / AdamW with one
    param group per ParamGroup at lr = base_lr * lr_mult (+ LambdaLR, + clip_grad_norm_ over the trainable parameters) over 6
    steps; the frozen group's parameters, shadow and moments stay bit for bit, every gradient is cleared."""
    arena = _arena(kind)
    wd = 0.1 if decoupled else 0.01
    desc, bmap, hp = _device_groups(arena, GROUPS, wd)
    gid = _group_of(arena, bmap)
    assert sorted(set(gid.values())) == [0, 1, 2, 3]
    s = LRSchedule.cosine(1e-3, 5, end_lr=1e-5, warmup_steps=2, warmup_start_lr=1e-5)
    base = s.base_lr if scheduled else 2e-3
    n = arena.numel
    torch.manual_seed(11)
    p = torch.zeros(n, device="cuda")
    for name in arena.shapes:                 # init-sized weights: fp32 rounding of the two sides stays far below 1e-6
        arena.view(name, p).normal_(0.0, 0.1)
    p0 = p.clone()
    refs = {name: arena.view(name, p).clone() for name in arena.shapes}
    for name in refs:
        refs[name].requires_grad_(hp[gid[name]][2] is False)
    pgroups = [dict(params=[refs[nm] for nm in refs if gid[nm] == k], lr=base * hp[k][0], weight_decay=hp[k][1])
               for k in range(len(hp)) if not hp[k][2]]
    opt = (torch.optim.AdamW if decoupled else torch.optim.Adam)(pgroups, lr=base)
    if scheduled:
        from test_lr_schedule import lr_at
        lam = torch.optim.lr_scheduler.LambdaLR(opt, lambda t: lr_at(s, t) / s.base_lr)
    trainable = [refs[nm] for nm in refs if refs[nm].requires_grad]
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    shadow = p.to(torch.bfloat16)
    shadow0 = shadow.clone()
    step = torch.zeros(1, device="cuda", dtype=torch.int32)
    lr = torch.zeros(1, device="cuda", dtype=torch.float32)
    sched = torch.frombuffer(bytearray(bytes(s.pack())), dtype=torch.uint8).cuda()
    ws = torch.zeros(int(L.load().egot2_grad_norm_workspace_bytes()), device="cuda", dtype=torch.uint8)
    frozen = torch.zeros(n, dtype=torch.bool, device="cuda")
    for name in arena.shapes:
        if hp[gid[name]][2]:
            arena.view(name, frozen).fill_(True)
    st = torch.cuda.current_stream().cuda_stream
    guard = None
    for i in range(6):
        g = torch.zeros(n, device="cuda")
        for name in arena.shapes:
            arena.view(name, g).normal_().mul_(0.8 + 0.05 * i)
        for name, r in refs.items():
            r.grad = arena.view(name, g).clone() if r.requires_grad else None
        if clip:
            want = float(torch.linalg.vector_norm(g[~frozen].double()))
            max_norm = 0.5 * want
            assert abs(float(torch.nn.utils.clip_grad_norm_(trainable, max_norm)) - want) <= 1e-5 * want
            guard = _guard(max_norm)
        opt.step()
        if scheduled:
            lam.step()
            L.call("egot2_opt_advance", step.data_ptr(), sched.data_ptr(), lr.data_ptr(), st)
        else:
            step.add_(1)
        if clip:
            L.call("egot2_grad_norm_groups", g.data_ptr(), n, 1.0, guard.data_ptr(), step.data_ptr(), desc.data_ptr(),
                   bmap.data_ptr(), ws.data_ptr(), ws.numel(), st)
        L.call("egot2_adam_step_fused_groups", p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), n, base,
               lr.data_ptr() if scheduled else None, 0.9, 0.999, 1e-8, step.data_ptr(), 1.0, shadow.data_ptr(), 1,
               int(decoupled), None if guard is None else guard.data_ptr(), desc.data_ptr(), bmap.data_ptr(), st)
        if clip:
            r = _read_guard(guard)
            assert r.skip == 0 and r.coef < 1.0 and abs(r.total_norm - want) <= 1e-6 * want
        assert float(g.abs().max()) == 0.0
    err = max(float((arena.view(name, p) - r.detach()).abs().max()) for name, r in refs.items())
    assert err < 1e-6, err
    assert torch.equal(p[frozen], p0[frozen]) and torch.equal(shadow[frozen], shadow0[frozen])
    assert float(m[frozen].abs().max()) == 0.0 and float(v[frozen].abs().max()) == 0.0
    assert torch.equal(shadow[~frozen], p[~frozen].to(torch.bfloat16)) and not torch.equal(p, p0)


def _nan_case(nan_in_frozen):
    """One grouped AdamW step with clipping over the HHI arena after a NaN in one gradient element of a frozen or of a
    trainable parameter; returns (arena, state before, state after, guard, the gradient without the NaN, max_norm)."""
    arena = _arena("hhi")
    desc, bmap, hp = _device_groups(arena, GROUPS, 0.1)
    gid = _group_of(arena, bmap)
    n = arena.numel
    torch.manual_seed(5)
    p, g = torch.randn(n, device="cuda"), torch.randn(n, device="cuda")
    m, v = torch.rand(n, device="cuda") * 1e-2, torch.rand(n, device="cuda") * 1e-4
    shadow = p.to(torch.bfloat16)
    clean = g.clone()
    name = next(nm for nm in arena.shapes if hp[gid[nm]][2] == nan_in_frozen)
    arena.view(name, g).view(-1)[3] = float("nan")
    frozen = torch.zeros(n, dtype=torch.bool, device="cuda")
    for nm in arena.shapes:
        if hp[gid[nm]][2]:
            arena.view(nm, frozen).fill_(True)
    clean[frozen] = 0.0
    max_norm = 0.5 * float(torch.linalg.vector_norm(clean.double()))
    guard = _guard(max_norm)
    step = torch.tensor([3], device="cuda", dtype=torch.int32)
    ws = torch.zeros(int(L.load().egot2_grad_norm_workspace_bytes()), device="cuda", dtype=torch.uint8)
    before = [t.clone() for t in (p, shadow, m, v)]
    st = torch.cuda.current_stream().cuda_stream
    L.call("egot2_grad_norm_groups", g.data_ptr(), n, 1.0, guard.data_ptr(), step.data_ptr(), desc.data_ptr(),
           bmap.data_ptr(), ws.data_ptr(), ws.numel(), st)
    L.call("egot2_adam_step_fused_groups", p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), n, 1e-3, None, 0.9,
           0.999, 1e-8, step.data_ptr(), 1.0, shadow.data_ptr(), 1, 1, guard.data_ptr(), desc.data_ptr(), bmap.data_ptr(), st)
    assert float(g.abs().max()) == 0.0
    return frozen, before, [p, shadow, m, v], _read_guard(guard), clean, max_norm, int(step)


@pytest.mark.gpu
def test_nan_in_a_frozen_gradient_neither_skips_nor_clips():
    """The norm leaves frozen gradients out: the step is clipped by the trainable norm, exactly as the same step without the
    NaN (which only clip_grad_norm_ over the trainable parameters would also ignore)."""
    frozen, before, after, r, clean, max_norm, step = _nan_case(True)
    want = float(torch.linalg.vector_norm(clean.double()))
    assert r.skip == 0 and r.skipped == 0 and step == 3 and abs(r.total_norm - want) <= 1e-6 * want
    assert r.coef == np.float32(np.float32(max_norm) / (np.float32(r.total_norm) + np.float32(1e-6)))
    for x, y in zip(before, after):
        assert torch.equal(x[frozen], y[frozen]) and not torch.equal(x[~frozen], y[~frozen])
    assert bool(torch.isfinite(after[0]).all())


@pytest.mark.gpu
def test_nan_in_a_trainable_gradient_skips_bit_for_bit():
    _, before, after, r, _, _, step = _nan_case(False)
    assert r.skip == 1 and r.skipped == 1 and step == 2 and not math.isfinite(r.total_norm)
    for x, y in zip(before, after):
        assert torch.equal(x, y)


# ------------------------------------------------------------------------------------------------ GPU: trainers
def _hhi_setup(batch=16, seed=1):
    import dataclasses
    from egot2_b200 import specs, synth
    spec = dataclasses.replace(specs.hhi_ttm_spec(128, 4, 2, 0.0, True), p_embed=0.0)
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


def _frozen_mask(tr):
    a = tr.engine.arena
    mask = torch.zeros(a.numel, dtype=torch.bool, device=a.param.device)
    for k, (_, _, frozen) in enumerate(tr._group_hp):
        if frozen:
            mask |= (tr._groups[1].repeat_interleave(64)[:a.numel] == k)
    return mask


@pytest.mark.gpu
@pytest.mark.parametrize("guard", [False, True])
def test_catch_all_group_is_bit_identical_to_no_groups(guard):
    """A single catch-all group with default values == no groups, bit for bit, over 8 graph-replayed steps.

    The backward's fp32 atomics make two trainers' gradients differ in the last bits, so the ungrouped update runs in the
    SAME graph, on the same gradient: the trainer's captured optimizer call is wrapped so that the graph first runs the
    launch the ungrouped graph ends with (egot2_adam_step_fused_dev; egot2_grad_norm + egot2_adam_step_fused_guard with a
    guard) on a twin of the parameters, shadow and moments, then the grouped one."""
    spec, feats, labels = _hhi_setup()
    kw = dict(max_grad_norm=0.05) if guard else {}
    tr = _hhi_trainer_gpu(spec, use_graphs=True, weight_decay=0.01, param_groups=[ParamGroup("*")], **kw)
    eng, a = tr.engine, tr.engine.arena
    a.refresh_shadow()
    p0 = a.param.clone()
    twin = dict(p=a.param.clone(), s=a.shadow.clone(), m=torch.zeros_like(a.param), v=torch.zeros_like(a.param))
    twin_guard = _guard(0.05) if guard else None
    ws = torch.zeros(int(L.load().egot2_grad_norm_workspace_bytes()), device="cuda", dtype=torch.uint8)
    real = eng.adam_step

    def both(state, step, lr, betas, eps, weight_decay, grad_scale=1.0, fused=False, step_dev=None, groups=None,
             guard=None, **k):
        st = torch.cuda.current_stream().cuda_stream
        if guard is None:
            L.call("egot2_adam_step_fused_dev", twin["p"].data_ptr(), a.grad.data_ptr(), twin["m"].data_ptr(),
                   twin["v"].data_ptr(), a.numel, lr, betas[0], betas[1], eps, weight_decay, step_dev.data_ptr(),
                   float(grad_scale), twin["s"].data_ptr(), 0, st)
        else:                                             # the twin norm leaves the step count to the trainer's
            L.call("egot2_grad_norm", a.grad.data_ptr(), a.numel, float(grad_scale), twin_guard.data_ptr(), None,
                   ws.data_ptr(), ws.numel(), st)
            L.call("egot2_adam_step_fused_guard", twin["p"].data_ptr(), a.grad.data_ptr(), twin["m"].data_ptr(),
                   twin["v"].data_ptr(), a.numel, lr, None, betas[0], betas[1], eps, weight_decay, step_dev.data_ptr(),
                   float(grad_scale), twin["s"].data_ptr(), 0, 0, twin_guard.data_ptr(), st)
        return real(state, step, lr, betas, eps, weight_decay, grad_scale=grad_scale, fused=fused, step_dev=step_dev,
                    groups=groups, guard=guard, **k)
    eng.adam_step = both
    for _ in range(8):
        tr.train_step(feats, labels, graph_key=0)
    torch.cuda.synchronize()
    assert len(tr._graphs) == 1 and int(tr._step_dev) == 8
    assert not torch.equal(a.param, p0)
    for x, y in zip((a.param, a.shadow, tr.opt_state["m"], tr.opt_state["v"]), (twin["p"], twin["s"], twin["m"], twin["v"])):
        assert torch.equal(x, y)
    if guard:
        assert bytes(_read_guard(twin_guard)) == bytes(L.GradGuard.from_buffer_copy(tr._guard_dev.cpu().numpy().tobytes()))


@pytest.mark.gpu
def test_frozen_parameters_stay_in_the_whole_step_graph():
    spec, feats, labels = _hhi_setup()
    tr = _hhi_trainer_gpu(spec, use_graphs=True, weight_decay=0.01, max_grad_norm=1.0, param_groups=GROUPS)
    p0 = tr.engine.arena.param.clone()
    for _ in range(6):
        tr.train_step(feats, labels, graph_key=0)
    torch.cuda.synchronize()
    fz = _frozen_mask(tr)
    assert int(fz.sum()) > 0
    p, s, m, v = _snapshot(tr)
    assert torch.equal(p[fz], p0[fz]) and torch.equal(s[fz], p0[fz].to(torch.bfloat16))
    assert float(m[fz].abs().max()) == 0.0 and float(v[fz].abs().max()) == 0.0
    assert float((p[~fz] - p0[~fz]).abs().max()) > 0.0 and float(tr.engine.arena.grad.abs().max()) == 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("graphs", ["1", "0"])
@pytest.mark.parametrize("kind", ["hhi", "hoi"])
def test_frozen_parameters_stay_in_the_prompt_trainers(kind, graphs, monkeypatch):
    from egot2_b200 import synth, trainer as T
    monkeypatch.setenv("EGOT2_G_GRAPH", graphs)
    feats, labels = _prompt_batch(kind)
    feats, labels = [f.cuda() for f in feats], labels.cuda()
    cls = T.HoiPromptTranslatorTrainer if kind == "hoi" else T.PromptTranslatorTrainer
    extra = dict(vocab=40) if kind == "hoi" else {}
    tr = cls(hidden=128, heads=4, layers=1, device="cuda:0", dtype="bf16", param_groups=GROUPS, **extra)
    tr.load_state_dict(synth.make_state_dict(tr.spec, 3))
    p0 = tr.engine.arena.param.clone()
    for _ in range(4):
        tr.train_step(feats, labels, graph_key=0)
    torch.cuda.synchronize()
    fz = _frozen_mask(tr)
    assert int(fz.sum()) > 0
    p, s, m, v = _snapshot(tr)
    assert torch.equal(p[fz], p0[fz]) and torch.equal(s[fz], p0[fz].to(torch.bfloat16))
    assert float(m[fz].abs().max()) == 0.0 and float(v[fz].abs().max()) == 0.0
    assert float((p[~fz] - p0[~fz]).abs().max()) > 0.0 and int(tr._step_dev) == 4


@pytest.mark.gpu
def test_grouped_graph_matches_grouped_eager():
    """Grouped whole-step graph == grouped eager trainer (the parameters by the L2 norm of the difference relative to how far
    training moved them: the backward's fp32 atomics make single elements of two runs differ, see test_grad_guard)."""
    spec, feats, labels = _hhi_setup()
    kw = dict(weight_decay=0.01, lr_schedule=LRSchedule.cosine(5e-4, 8, warmup_steps=2), param_groups=GROUPS)
    tg = _hhi_trainer_gpu(spec, use_graphs=True, **kw)
    te = _hhi_trainer_gpu(spec, use_graphs=False, **kw)
    p0 = te.engine.arena.param.clone()
    for _ in range(6):
        lg = float(tg.train_step(feats, labels, graph_key=0))
        le = float(te.train_step(feats, labels))
        assert abs(lg - le) <= 2e-2 * abs(le) + 1e-4
    pg, pe = tg.engine.arena.param, te.engine.arena.param
    assert float((pg - pe).norm()) <= 2e-2 * float((pe - p0).norm())
    fz = _frozen_mask(tg)
    assert torch.equal(pg[fz], pe[fz]) and torch.equal(pg[fz], p0[fz])


@pytest.mark.gpu
def test_set_param_group_takes_effect_at_the_next_replay():
    spec, feats, labels = _hhi_setup()
    tr = _hhi_trainer_gpu(spec, use_graphs=True, weight_decay=0.01, param_groups=GROUPS)
    tr.train_step(feats, labels, graph_key=0)
    for k in range(4):
        tr.set_param_group(k, lr_mult=0.0)
    before = tr.engine.arena.param.clone()
    tr.train_step(feats, labels, graph_key=0)
    torch.cuda.synchronize()
    assert torch.equal(tr.engine.arena.param, before)                  # lr 0 for every group: nothing moves
    tr.set_param_group(0, lr_mult=1.0)
    tr.train_step(feats, labels, graph_key=0)
    torch.cuda.synchronize()
    moved = tr.engine.arena.param != before
    g0 = (tr._groups[1].repeat_interleave(64)[:tr.engine.arena.numel] == 0)
    assert bool(moved[g0].any()) and not bool(moved[~g0].any())
    assert len(tr._graphs) == 1


@pytest.mark.gpu
def test_resume_mid_run():
    """Steps 1-3, save (with a rewritten group), a fresh trainer loads and runs 4-6 == six uninterrupted steps."""
    spec, feats, labels = _hhi_setup()
    kw = dict(use_graphs=True, weight_decay=0.01, max_grad_norm=0.5, param_groups=GROUPS)

    def run(tr, steps):
        for t in steps:
            if t == 2:
                tr.set_param_group(2, lr_mult=0.5)
            tr.train_step(feats, labels, graph_key=0)
        torch.cuda.synchronize()
    full = _hhi_trainer_gpu(spec, **kw)
    p0 = full.engine.arena.param.clone()
    run(full, range(1, 7))
    p_full = full.engine.arena.param.clone()
    del full
    first = _hhi_trainer_gpu(spec, **kw)
    run(first, range(1, 4))
    sd, osd = first.state_dict(), first.optimizer_state_dict()
    del first
    tr = _hhi_trainer_gpu(spec, **kw)
    tr.load_state_dict(sd)
    tr.load_optimizer_state_dict(osd)
    assert tr._group_hp[2][0] == 0.5
    run(tr, range(4, 7))
    assert float((tr.engine.arena.param - p_full).norm()) <= 2e-2 * float((p_full - p0).norm())
    fz = _frozen_mask(tr)
    assert torch.equal(tr.engine.arena.param[fz], p0[fz])


# ------------------------------------------------------------------------------------------------ GPU: two ranks
def _rank_worker(rank, world, port, q):
    os.environ["EGOT2_DP_FUSED"] = "1"
    import dataclasses

    import torch
    import torch.distributed as dist

    from egot2_b200 import specs, synth
    from egot2_b200.trainer import TranslatorTrainer
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        sp = dataclasses.replace(specs.hhi_ttm_spec(128, 4, 2, 0.0, True), p_embed=0.0)
        B, seg = 16, (10, 10, 10)
        f = synth.make_features(sp, B, seg, seed=77, dtype=torch.bfloat16)
        lab = synth.make_labels(sp, B, seg, seed=77)
        lo, hi = rank * B // world, (rank + 1) * B // world
        tr = TranslatorTrainer(sp, f"cuda:{rank}", "bf16", use_graphs=True, weight_decay=0.01, max_grad_norm=0.05,
                               param_groups=GROUPS)
        assert tr.peer is not None
        tr.load_state_dict(synth.make_state_dict(sp, 9))
        p0 = tr.engine.arena.param.clone()
        feats = [f[s.name][lo:hi].cuda() for s in sp.segments]
        labels = lab[lo:hi].cuda()
        for _ in range(4):
            tr.train_step(feats, labels, graph_key=0)
        torch.cuda.synchronize()
        fz = _frozen_mask(tr)
        q.put((rank, dict(frozen_kept=bool(torch.equal(tr.engine.arena.param[fz], p0[fz])),
                          params={k: v.cpu() for k, v in tr.state_dict().items()})))
        dist.barrier()
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_two_rank_grouped_peer_exchange():
    """The peer-memory exchange (EGOT2_DP_FUSED=1) with groups and a guard: ranks stay bit-identical, frozen parameters stay."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import socket

    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_rank_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=170) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert got[0]["frozen_kept"] and got[1]["frozen_kept"]
    for k in got[0]["params"]:
        assert torch.equal(got[0]["params"][k], got[1]["params"][k]), f"{k}: ranks diverged"
