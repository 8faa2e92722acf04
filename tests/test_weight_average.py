"""Weight averaging of the fused trainers (optim.WeightAverage, egot2_weight_avg_update): torch.optim.swa_utils.AveragedModel's
EMA and SWA over the parameter arena, updated on the device after the optimizer launch.

CPU: the input checks of WeightAverage and of the C entry, the launch plans (one update right after every optimizer launch
or peer exchange, on the trainer's device step count and guard), the optimizer-state round trip and its rejections, and the
checks of averaged_state_dict() / averaged_weights().  GPU (-m gpu): the kernel against AveragedModel bit for bit over the
HHI, PNR and LTA-b512 arenas, the trainers against AveragedModel fed with their own parameters, the guard, resume,
averaged_weights(), training unperturbed, and two ranks."""
import io
import math
import os

import pytest
import torch

from egot2_b200 import _lib as L
from egot2_b200.optim import SGD, LRSchedule, ParamGroup, WeightAverage
from egot2_b200.stats import ParamStats
from test_param_groups import (GROUPS, _arena, _hhi_setup, _hhi_trainer, _hhi_trainer_gpu, _names,  # noqa: F401
                               _prompt_batch, built, recorder)

_AVG = "egot2_weight_avg_update"
_OPT = {"egot2_adam_step", "egot2_adam_step_fused", "egot2_adamw_step_fused", "egot2_adam_step_fused_dev",
        "egot2_adam_step_fused_sched", "egot2_adam_step_fused_guard", "egot2_adam_step_fused_groups", "egot2_sgd_step_fused"}
_PEER = "<peer>"


# ------------------------------------------------------------------------------------------------ CPU: input checks
@pytest.mark.parametrize("bad", [dict(decay=-0.1), dict(decay=1.0 + 1e-9), dict(decay=math.nan), dict(decay=math.inf),
                                 dict(decay="x"), dict(decay=None), dict(every=0), dict(every=-2), dict(every=1.5),
                                 dict(every=True), dict(every="2"), dict(every=2 ** 31), dict(start=0), dict(start=-1),
                                 dict(start=2.0), dict(start=None), dict(start=2 ** 31)])
def test_weight_average_input_checks(bad):
    with pytest.raises(ValueError):
        WeightAverage.ema(**bad)
    if "decay" not in bad:
        with pytest.raises(ValueError):
            WeightAverage.swa(**bad)


def test_weight_average_fields_and_round_trip():
    import numpy as np
    e = WeightAverage.ema(0.999, every=np.int64(3), start=2 ** 31 - 1)
    assert (e.kind, e.decay, e.every, e.start) == (L.AVG_EMA, 0.999, 3, 2 ** 31 - 1) and type(e.every) is int
    assert e.ema_weight == 1.0 - 0.999                      # the subtraction in double, as torch does with the scalar
    s = WeightAverage.swa()
    assert (s.kind, s.every, s.start, s.ema_weight) == (L.AVG_SWA, 1, 1, 0.0)
    assert WeightAverage.ema(0).decay == 0.0 and WeightAverage.ema(1).decay == 1.0
    for wa in (e, s):
        d = wa.to_dict()
        assert WeightAverage.from_dict(d) == wa and all(isinstance(v, (int, float)) for v in d.values())
    with pytest.raises(ValueError):
        WeightAverage(7)


def test_c_entry_checks(built):
    lib = L.load()
    ok = dict(param=256, avg=512, n=64, kind=L.AVG_EMA, w=0.001, every=1, start=1, step=768, guard=None)
    bad_cases = [dict(param=None), dict(avg=None), dict(step=None), dict(kind=2), dict(kind=-1), dict(every=0),
                 dict(every=-1), dict(start=0), dict(start=-5), dict(w=-0.01), dict(w=1.01), dict(w=math.nan),
                 dict(n=66), dict(param=260), dict(avg=520)]
    for bad in bad_cases:
        a = {**ok, **bad}
        rc = lib.egot2_weight_avg_update(a["param"], a["avg"], a["n"], a["kind"], a["w"], a["every"], a["start"], a["step"],
                                         a["guard"], None)
        assert rc != 0, bad
        assert b"weight_avg_update" in lib.egot2_last_error()


def test_trainer_rejects_other_types(recorder):
    with pytest.raises(ValueError, match="weight_average"):
        _hhi_trainer(weight_average=0.999)
    tr, _, _ = _hhi_trainer()
    assert tr.weight_average is None and tr._avg is None
    with pytest.raises(ValueError, match="weight_average"):
        tr.averaged_state_dict()
    with pytest.raises(ValueError, match="weight_average"):
        with tr.averaged_weights():
            pass


# ------------------------------------------------------------------------------------------------ CPU: launch plans
def _check_avg_after_every_update(calls, tr, wa):
    """Exactly one egot2_weight_avg_update right after every optimizer launch and every peer exchange, none elsewhere, each
    with the trainer's arena, average, step_dev and guard and the WeightAverage's fields; returns the number of updates."""
    names = _names(calls)
    n = 0
    for i, nm in enumerate(names):
        if nm in _OPT or nm == _PEER:
            n += 1
            assert i + 1 < len(names) and names[i + 1] == _AVG, names[i - 1:i + 3]
        if nm == _AVG:
            assert names[i - 1] in _OPT or names[i - 1] == _PEER, names[i - 2:i + 1]
            a = calls[i][1]
            arena = tr.engine.arena
            assert a[:3] == (arena.param.data_ptr(), tr._avg.data_ptr(), arena.numel)
            assert a[3:7] == (wa.kind, wa.ema_weight, wa.every, wa.start)
            assert a[7] == tr._step_dev.data_ptr()
            assert a[8] == (None if tr.max_grad_norm is None else tr._guard_dev.data_ptr())
    assert names.count(_AVG) == n > 0
    return n


def _plan(tr, feats, labels):
    tr.train_step(feats, labels, graph_key=0)
    tr.train_step(feats, labels, graph_key=0)
    tr.use_graphs = False
    tr.train_step(feats, labels)


_CONFIGS = {"plain": {}, "guard": dict(max_grad_norm=1.0), "groups": dict(param_groups=GROUPS),
            "sgd": dict(optimizer=SGD(momentum=0.9), max_grad_norm=1.0),
            "sched": dict(lr_schedule=LRSchedule.cosine(1e-3, 10)), "stats": dict(param_stats=ParamStats(2))}


@pytest.mark.parametrize("config", list(_CONFIGS))
def test_plan_has_one_update_after_every_optimizer_launch(config, recorder):
    """Whole-step graph (the update is captured, right after the optimizer) and eager step: the launches without an average,
    plus one update after every optimizer launch.  Without a guard, groups, schedule or statistics the eager optimizer reads
    the device step count."""
    kw = _CONFIGS[config]
    tr, feats, labels = _hhi_trainer(**kw)
    _plan(tr, feats, labels)
    ref = _names(recorder)
    assert _AVG not in ref
    del recorder[:]
    wa = WeightAverage.ema(0.99, every=3, start=2)
    tr, feats, labels = _hhi_trainer(weight_average=wa, **kw)
    _plan(tr, feats, labels)
    got = _names(recorder)
    assert _check_avg_after_every_update(recorder, tr, wa) == 2
    cap = got[got.index("<capture>") + 1:got.index("</capture>")]
    assert cap[-1] == _AVG and cap[-2] in _OPT
    dev_step = {"egot2_adam_step_fused": "egot2_adam_step_fused_dev"}
    assert [n for n in got if n != _AVG] == [dev_step.get(n, n) for n in ref]


def test_dp_overlap_plan(recorder, monkeypatch):
    import torch.distributed as dist
    monkeypatch.setenv("EGOT2_DP_OVERLAP", "force")

    class Work:
        def wait(self):
            pass
    monkeypatch.setattr(dist, "all_reduce", lambda *a, **k: Work())
    wa = WeightAverage.swa(every=2)
    tr, feats, labels = _hhi_trainer(weight_average=wa, max_grad_norm=1.0)
    assert tr.dp_overlap
    tr.world = 2
    for _ in range(2):
        tr.train_step(feats, labels, graph_key=0)
    assert _check_avg_after_every_update(recorder, tr, wa) == 2


def test_nccl_path_plan(recorder, monkeypatch):
    from egot2_b200 import trainer as T
    monkeypatch.setattr(T, "allreduce_gradients", lambda grad, pg: 0.5)
    wa = WeightAverage.ema(0.9)
    for kw in ({}, dict(max_grad_norm=1.0, param_groups=GROUPS)):
        tr, feats, labels = _hhi_trainer(weight_average=wa, **kw)
        tr.world, tr.use_graphs = 2, False
        del recorder[:]
        tr.train_step(feats, labels)
        assert _check_avg_after_every_update(recorder, tr, wa) == 1


def _fake_peer(monkeypatch, recorder):
    """_make_peer_exchange stubbed by a peer whose step() is recorded as ('<peer>', kwargs)."""
    from egot2_b200 import trainer as T

    class FakePeer:
        def step(self, state, step, hp, stream, **kw):
            recorder.append((_PEER, kw))
    monkeypatch.setattr(T, "_make_peer_exchange", lambda engine, pg, world: FakePeer())


@pytest.mark.parametrize("config", ["plain", "guard+groups", "sgd"])
def test_peer_path_plan(config, recorder, monkeypatch):
    """The peer exchange, captured in the whole-step graph and eager: one update right after every exchange."""
    _fake_peer(monkeypatch, recorder)
    kw = {"plain": {}, "guard+groups": dict(max_grad_norm=1.0, param_groups=GROUPS),
          "sgd": dict(optimizer=SGD(momentum=0.9))}[config]
    wa = WeightAverage.ema(0.999, start=3)
    tr, feats, labels = _hhi_trainer(weight_average=wa, **kw)
    assert tr.peer is not None and tr.graph_update
    _plan(tr, feats, labels)
    assert _check_avg_after_every_update(recorder, tr, wa) == 2
    names = _names(recorder)
    cap = names[names.index("<capture>") + 1:names.index("</capture>")]
    assert cap[-2:] == [_PEER, _AVG]
    assert all(k["step_dev"] is tr._step_dev for n, k in recorder if n == _PEER)


def test_split_peer_exchange_updates_once(recorder, monkeypatch):
    """EGOT2_DP_SPLIT=1: the exchange runs in two pieces; the average is updated once, after both are joined."""
    _fake_peer(monkeypatch, recorder)
    monkeypatch.setenv("EGOT2_DP_SPLIT", "1")
    wa = WeightAverage.swa()
    tr, feats, labels = _hhi_trainer(weight_average=wa)
    for _ in range(2):
        tr.train_step(feats, labels, graph_key=0)
    names = _names(recorder)
    cap = names[names.index("<capture>") + 1:names.index("</capture>")]
    assert cap.count(_PEER) == 2 and cap.count(_AVG) == 1 and cap[-1] == _AVG
    assert names.count(_AVG) == 1
    (a,) = [a for n, a in recorder if n == _AVG]
    assert a[1] == tr._avg.data_ptr() and a[7] == tr._step_dev.data_ptr() and a[8] is None


@pytest.mark.parametrize("graphs", ["1", "0"])
@pytest.mark.parametrize("kind", ["hhi", "hoi"])
def test_prompt_trainer_plans(kind, graphs, recorder, monkeypatch):
    """EgoT2-g trainers, graph replay and eager, plain and with a guard and groups: one update after every optimizer launch,
    which is a fused launch on the device step count (the HHI eager step too)."""
    from egot2_b200 import trainer as T
    monkeypatch.setenv("EGOT2_G_GRAPH", graphs)
    cls = T.HoiPromptTranslatorTrainer if kind == "hoi" else T.PromptTranslatorTrainer
    extra = dict(vocab=40) if kind == "hoi" else {}
    feats, labels = _prompt_batch(kind)
    wa = WeightAverage.ema(0.5, every=2)
    for kw in ({}, dict(max_grad_norm=1.0, param_groups=[ParamGroup("proj*", frozen=True)]),
               dict(optimizer=SGD(momentum=0.9)), dict(lr_schedule=LRSchedule.cosine(1e-3, 10))):
        del recorder[:]
        tr = cls(hidden=128, heads=4, layers=1, device="cpu", weight_average=wa, **extra, **kw)
        for _ in range(2):
            tr.train_step(feats, labels, graph_key=0)
        assert _check_avg_after_every_update(recorder, tr, wa) == 2
        assert "egot2_adam_step" not in _names(recorder) and tr._grad_clean
        if "lr_schedule" not in kw:                        # with a schedule egot2_opt_advance counts (not run here)
            assert int(tr._step_dev[0]) == 2


@pytest.mark.parametrize("kind", ["hhi", "hoi"])
def test_prompt_trainer_peer_plans(kind, recorder, monkeypatch):
    from egot2_b200 import trainer as T
    _fake_peer(monkeypatch, recorder)
    cls = T.HoiPromptTranslatorTrainer if kind == "hoi" else T.PromptTranslatorTrainer
    extra = dict(vocab=40) if kind == "hoi" else {}
    feats, labels = _prompt_batch(kind)
    wa = WeightAverage.swa()
    for graphs in ("1", "0"):
        monkeypatch.setenv("EGOT2_G_GRAPH", graphs)
        del recorder[:]
        tr = cls(hidden=128, heads=4, layers=1, device="cpu", weight_average=wa, **extra)
        for _ in range(2):
            tr.train_step(feats, labels, graph_key=0)
        assert _check_avg_after_every_update(recorder, tr, wa) == 2


# ------------------------------------------------------------------------------------------------ CPU: state
def _filled_trainer(wa, **kw):
    tr, feats, labels = _hhi_trainer(weight_average=wa, **kw)
    g = torch.Generator().manual_seed(5)
    arena = tr.engine.arena                                # the parameters only: the padding stays 0, as the kernel keeps it
    arena.load_state_dict({n: torch.randn(shp, generator=g) for n, shp in arena.shapes.items()}, base=tr._avg)
    return tr, feats, labels


def test_optimizer_state_dict_round_trip(recorder):
    wa = WeightAverage.ema(0.9, every=2, start=3)
    tr, feats, labels = _filled_trainer(wa, max_grad_norm=1.0)
    tr.train_step(feats, labels, graph_key=0)
    sd = tr.optimizer_state_dict()
    w = sd["weight_average"]
    assert {k: w[k] for k in ("kind", "decay", "every", "start")} == wa.to_dict()
    assert w["average"].keys() == tr.engine.arena.shapes.keys()
    buf = io.BytesIO()
    torch.save(sd, buf)
    buf.seek(0)
    sd = torch.load(buf, weights_only=True)
    tr2, _, _ = _hhi_trainer(weight_average=wa, max_grad_norm=1.0)
    ptr = tr2._avg.data_ptr()
    tr2.load_optimizer_state_dict(sd)
    assert tr2._avg.data_ptr() == ptr and torch.equal(tr2._avg, tr._avg)
    tr2.load_state_dict(tr.state_dict())                 # the parameters only: the average stays
    assert torch.equal(tr2._avg, tr._avg)
    assert _hhi_trainer()[0].optimizer_state_dict()["weight_average"] is None


@pytest.mark.parametrize("other", [None, WeightAverage.swa(every=2, start=3), WeightAverage.ema(0.8, every=2, start=3),
                                   WeightAverage.ema(0.9, every=1, start=3), WeightAverage.ema(0.9, every=2, start=1)])
def test_optimizer_state_load_rejections(other, recorder):
    wa = WeightAverage.ema(0.9, every=2, start=3)
    tr, _, _ = _filled_trainer(wa)
    sd = tr.optimizer_state_dict()
    dst, _, _ = _hhi_trainer(weight_average=other)
    before = None if dst._avg is None else dst._avg.clone()
    with pytest.raises(ValueError, match="weight_average|fixed at construction"):
        dst.load_optimizer_state_dict(sd)
    if before is not None:
        assert torch.equal(dst._avg, before)
    # and the reverse: a state saved without an average
    plain = _hhi_trainer()[0].optimizer_state_dict()
    with pytest.raises(ValueError, match="weight_average"):
        _hhi_trainer(weight_average=wa)[0].load_optimizer_state_dict(plain)


def test_no_average_before_the_first_update(recorder):
    wa = WeightAverage.swa(every=4, start=3)
    tr, feats, labels = _filled_trainer(wa)
    for t in (0, 2):
        tr._step_dev.fill_(t)
        with pytest.raises(ValueError, match="first update"):
            tr.averaged_state_dict()
        with pytest.raises(ValueError, match="first update"):
            with tr.averaged_weights():
                pass
    tr._step_dev.fill_(3)
    sd = tr.averaged_state_dict()
    arena = tr.engine.arena
    assert all(torch.equal(sd[n], arena.view(n, tr._avg)) for n in arena.shapes)
    sd[next(iter(sd))].fill_(7.0)                          # a copy
    assert not torch.equal(arena.view(next(iter(sd)), tr._avg), sd[next(iter(sd))])
    assert tr._averaged_updates() == 1
    tr._step_dev.fill_(11)
    assert tr._averaged_updates() == 3


def test_averaged_weights_swaps_in_and_back(recorder):
    """CPU: inside the block the arena holds the average and train_step raises; afterwards the parameters, shadow and its
    freshness are back and training goes on."""
    wa = WeightAverage.ema(0.9)
    tr, feats, labels = _filled_trainer(wa)
    tr.train_step(feats, labels, graph_key=0)
    arena = tr.engine.arena
    tr._step_dev.fill_(1)
    arena.shadow.copy_(arena.param)                        # the cast is recorded, not run, here
    p0 = arena.param.clone()
    s0 = arena.shadow.clone()
    fresh = arena.shadow_fresh
    del recorder[:]
    with tr.averaged_weights():
        assert torch.equal(arena.param, tr._avg) and arena.shadow_fresh
        assert _names(recorder) == ["egot2_cast_f32_to_bf16"]
        with pytest.raises(ValueError, match="averaged_weights"):
            tr.train_step(feats, labels, graph_key=0)
        with pytest.raises(ValueError, match="already"):
            with tr.averaged_weights():
                pass
        assert tr.state_dict()[next(iter(arena.shapes))].equal(arena.view(next(iter(arena.shapes)), tr._avg))
    assert torch.equal(arena.param, p0) and torch.equal(arena.shadow, s0) and arena.shadow_fresh == fresh
    assert tr.step_count == 1
    tr.train_step(feats, labels, graph_key=0)
    assert tr.step_count == 2


# ------------------------------------------------------------------------------------------------ GPU: the kernel
def _ref_model(numel):
    """A module holding one flat fp32 parameter of `numel` elements (the arena), for AveragedModel."""
    m = torch.nn.Module()
    m.p = torch.nn.Parameter(torch.zeros(numel, device="cuda"))
    return m


def _averaged_model(model, wa):
    from torch.optim.swa_utils import AveragedModel, get_ema_multi_avg_fn
    if wa.kind == L.AVG_EMA:
        return AveragedModel(model, multi_avg_fn=get_ema_multi_avg_fn(wa.decay))
    return AveragedModel(model)


def _due(wa, t):
    return t >= wa.start and (t - wa.start) % wa.every == 0


def _launch(param, avg, wa, step_dev, guard=None):
    L.call(_AVG, param.data_ptr(), avg.data_ptr(), param.numel(), wa.kind, wa.ema_weight, wa.every, wa.start,
           step_dev.data_ptr(), None if guard is None else guard.data_ptr(), torch.cuda.current_stream().cuda_stream)


_KERNEL_CASES = [WeightAverage.ema(0.999), WeightAverage.ema(0.9, every=3, start=2), WeightAverage.ema(0.3),
                 WeightAverage.ema(0.5, every=2), WeightAverage.ema(0.0), WeightAverage.ema(1.0, start=2),
                 WeightAverage.swa(), WeightAverage.swa(every=2, start=3)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(_KERNEL_CASES)))
@pytest.mark.parametrize("kind", ["hhi", "pnr", "lta"])
def test_kernel_matches_averaged_model(kind, case):
    """The kernel and AveragedModel driven through the same parameter arrays: bit-identical after every step; a step that is
    not due, and a due step whose guard says skip, leave the average bit-identical."""
    wa = _KERNEL_CASES[case]
    n = _arena(kind).numel
    model = _ref_model(n)
    ref = _averaged_model(model, wa)
    avg = torch.full((n,), 123.0, device="cuda")
    step = torch.zeros(1, dtype=torch.int32, device="cuda")
    guard = torch.frombuffer(bytearray(bytes(L.GradGuard(max_norm=1.0))), dtype=torch.uint8).cuda()
    skip = guard[L.GradGuard.skip.offset:L.GradGuard.skip.offset + 4].view(torch.int32)
    g = torch.Generator(device="cuda").manual_seed(case)
    x = torch.randn(n, device="cuda", generator=g)
    steps = 3 * wa.every + wa.start + 1
    for t in range(1, steps + 1):
        x = x + 0.3 * torch.randn(n, device="cuda", generator=g) * (1 + (t % 3))
        with torch.no_grad():
            model.p.copy_(x)
        step.fill_(t)
        before = avg.clone()
        if _due(wa, t) and t > wa.start:                 # a skipped step first: nothing may change
            skip.fill_(1)
            _launch(model.p, avg, wa, step, guard)
            assert torch.equal(avg, before)
            skip.fill_(0)
        _launch(model.p, avg, wa, step, guard if t % 2 else None)
        if _due(wa, t):
            ref.update_parameters(model)
            assert torch.equal(avg, ref.module.p), (t, float((avg - ref.module.p).abs().max()))
        else:
            assert torch.equal(avg, before)
    assert int(ref.n_averaged) == sum(_due(wa, t) for t in range(1, steps + 1)) >= 4


# ------------------------------------------------------------------------------------------------ GPU: trainers
def _drive(tr, steps, wa, step_fn, ref=None, applied=None, t0=0):
    """Run step_fn(i) for `steps` steps and feed AveragedModel `ref` (a fresh one by default) with the trainer's own
    parameters after every applied step that is due; returns it.  applied(i) -> False marks a step the guard skips; t0 is
    the device step count before the first."""
    arena = tr.engine.arena
    model = _ref_model(arena.numel)
    if ref is None:
        ref = _averaged_model(model, wa)
    t = t0
    for i in range(steps):
        step_fn(i)
        if applied is not None and not applied(i):
            continue
        t += 1
        if _due(wa, t):
            with torch.no_grad():
                model.p.copy_(arena.param)
            ref.update_parameters(model)
    torch.cuda.synchronize()
    assert int(tr._step_dev) == t
    return ref


def _assert_avg_equals(tr, ref):
    arena = tr.engine.arena
    sd = tr.averaged_state_dict()
    want = arena.state_dict(ref.module.p.detach())
    for nm in arena.shapes:
        assert torch.equal(sd[nm], want[nm]), nm


_TRAINER_CASES = {"eager_ema": (dict(use_graphs=False), WeightAverage.ema(0.9)),
                  "graph_swa": (dict(use_graphs=True), WeightAverage.swa(every=2, start=2)),
                  "graph_sgd_ema": (dict(use_graphs=True, optimizer=SGD(momentum=0.9)), WeightAverage.ema(0.7, every=3)),
                  "graph_frozen_swa": (dict(use_graphs=True, param_groups=GROUPS, weight_decay=0.01), WeightAverage.swa()),
                  "eager_frozen_ema": (dict(use_graphs=False, param_groups=GROUPS, max_grad_norm=1.0),
                                       WeightAverage.ema(0.99, start=3))}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(_TRAINER_CASES))
def test_trainer_matches_averaged_model(case):
    kw, wa = _TRAINER_CASES[case]
    spec, feats, labels = _hhi_setup()
    tr = _hhi_trainer_gpu(spec, weight_average=wa, **kw)
    p0 = tr.engine.arena.param.clone()
    ref = _drive(tr, 8, wa, step_fn=lambda i: tr.train_step(feats, labels, graph_key=0))
    _assert_avg_equals(tr, ref)
    if "param_groups" in kw:
        from test_param_groups import _frozen_mask
        fz = _frozen_mask(tr)
        assert int(fz.sum()) > 0 and torch.equal(tr._avg[fz], p0[fz])


@pytest.mark.gpu
@pytest.mark.parametrize("graphs", ["1", "0"])
@pytest.mark.parametrize("kind", ["hhi", "hoi"])
def test_prompt_trainers_match_averaged_model(kind, graphs, monkeypatch):
    from egot2_b200 import synth, trainer as T
    monkeypatch.setenv("EGOT2_G_GRAPH", graphs)
    feats, labels = _prompt_batch(kind)
    feats, labels = [f.cuda() for f in feats], labels.cuda()
    cls = T.HoiPromptTranslatorTrainer if kind == "hoi" else T.PromptTranslatorTrainer
    extra = dict(vocab=40) if kind == "hoi" else {}
    wa = WeightAverage.ema(0.8, every=2) if kind == "hoi" else WeightAverage.swa()
    tr = cls(hidden=128, heads=4, layers=1, device="cuda:0", dtype="bf16", weight_average=wa, **extra)
    tr.load_state_dict(synth.make_state_dict(tr.spec, 3))
    ref = _drive(tr, 5, wa, step_fn=lambda i: tr.train_step(feats, labels, graph_key=0))
    _assert_avg_equals(tr, ref)


@pytest.mark.gpu
def test_guard_skip_leaves_the_average():
    """A NaN step leaves the average bit for bit; the next applied step updates it exactly once."""
    from test_grad_guard import _nan_feature
    spec, feats, labels = _hhi_setup()
    wa = WeightAverage.ema(0.9)
    tr = _hhi_trainer_gpu(spec, use_graphs=True, max_grad_norm=1.0, weight_average=wa)
    seen = {}

    def step(i):
        if i == 2:
            seen["before"] = tr._avg.clone()
            with _nan_feature(feats):
                tr.train_step(feats, labels, graph_key=0)
            torch.cuda.synchronize()
            assert int(tr.skipped_steps) == 1 and torch.equal(tr._avg, seen["before"])
        else:
            tr.train_step(feats, labels, graph_key=0)
    ref = _drive(tr, 5, wa, step_fn=step, applied=lambda i: i != 2)
    assert int(ref.n_averaged) == 4
    _assert_avg_equals(tr, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("wa", [WeightAverage.swa(start=2), WeightAverage.ema(0.8, every=2)], ids=["swa", "ema"])
def test_resume_mid_run(wa):
    """Steps 1-3, save, a fresh trainer loads and runs 4-6.  The loaded average equals the saved one bit for bit; the later
    average equals AveragedModel started from the loaded average (n_averaged restored) and fed with the resumed trainer's
    parameters; against an uninterrupted run it agrees to the tolerance of test_param_groups.py::test_resume_mid_run."""
    spec, feats, labels = _hhi_setup()
    kw = dict(use_graphs=True, weight_decay=0.01, max_grad_norm=0.5, weight_average=wa)

    def run(tr, n):
        for _ in range(n):
            tr.train_step(feats, labels, graph_key=0)
        torch.cuda.synchronize()
    full = _hhi_trainer_gpu(spec, **kw)
    p0 = full.engine.arena.param.clone()
    run(full, 6)
    avg_full = full._avg.clone()
    del full
    first = _hhi_trainer_gpu(spec, **kw)
    run(first, 3)
    sd, osd = first.state_dict(), first.optimizer_state_dict()
    saved, n_saved = first._avg.clone(), first._averaged_updates()
    del first
    buf = io.BytesIO()
    torch.save(osd, buf)
    buf.seek(0)
    osd = torch.load(buf, weights_only=True)
    tr = _hhi_trainer_gpu(spec, **kw)
    tr.load_state_dict(sd)
    tr.load_optimizer_state_dict(osd)
    assert torch.equal(tr._avg, saved)
    model = _ref_model(tr.engine.arena.numel)
    ref = _averaged_model(model, wa)
    with torch.no_grad():
        ref.module.p.copy_(saved)
    ref.n_averaged.fill_(n_saved)
    ref = _drive(tr, 3, wa, ref=ref, step_fn=lambda i: tr.train_step(feats, labels, graph_key=0), t0=3)
    _assert_avg_equals(tr, ref)
    assert float((tr._avg - avg_full).norm()) <= 2e-2 * float((avg_full - p0).norm())


@pytest.mark.gpu
def test_averaged_weights_block():
    """Inside: the arena is the average, the shadow its bf16 cast, infer() agrees with a fresh trainer that loaded
    averaged_state_dict().  After: parameters, shadow, moments and gradient arena equal the snapshot; no new capture."""
    spec, feats, labels = _hhi_setup()
    wa = WeightAverage.ema(0.5)
    tr = _hhi_trainer_gpu(spec, use_graphs=True, weight_average=wa)
    for _ in range(4):
        tr.train_step(feats, labels, graph_key=0)
    torch.cuda.synchronize()
    arena = tr.engine.arena
    snap = [arena.param.clone(), arena.shadow.clone(), tr.opt_state["m"].clone(), tr.opt_state["v"].clone(),
            arena.grad.clone()]
    avg_sd = tr.averaged_state_dict()
    fresh = _hhi_trainer_gpu(spec, use_graphs=True)
    fresh.load_state_dict(avg_sd)
    want = fresh.infer(feats).float().clone()
    with tr.averaged_weights():
        assert torch.equal(arena.param, tr._avg) and torch.equal(arena.shadow, tr._avg.to(torch.bfloat16))
        assert all(torch.equal(v, avg_sd[k]) for k, v in tr.state_dict().items())
        got = tr.infer(feats).float().clone()
    torch.cuda.synchronize()
    assert float((got - want).abs().max()) <= 2e-2 * float(want.abs().max())
    after = [arena.param, arena.shadow, tr.opt_state["m"], tr.opt_state["v"], arena.grad]
    for x, y in zip(snap, after):
        assert torch.equal(x, y)
    assert len(tr._graphs) == 1
    tr.train_step(feats, labels, graph_key=0)
    torch.cuda.synchronize()
    assert len(tr._graphs) == 1 and int(tr._step_dev) == 5


@pytest.mark.gpu
def test_training_is_not_perturbed():
    """One update on a due step leaves the parameters, shadow and gradient bit for bit; a trainer with an average trains as
    one without, within the graph-vs-eager tolerance."""
    spec, feats, labels = _hhi_setup()
    tr = _hhi_trainer_gpu(spec, use_graphs=True, weight_average=WeightAverage.swa())
    tr.train_step(feats, labels, graph_key=0)
    torch.cuda.synchronize()
    arena = tr.engine.arena
    arena.grad.normal_()
    snap = [arena.param.clone(), arena.shadow.clone(), arena.grad.clone()]
    _launch(arena.param, tr._avg, WeightAverage.ema(0.5), torch.full((1,), 2, dtype=torch.int32, device="cuda"))
    torch.cuda.synchronize()
    assert all(torch.equal(x, y) for x, y in zip(snap, (arena.param, arena.shadow, arena.grad)))
    runs = []
    for wa in (None, WeightAverage.ema(0.9)):
        tr = _hhi_trainer_gpu(spec, use_graphs=True, weight_average=wa)
        p0 = tr.engine.arena.param.clone()
        losses = [float(tr.train_step(feats, labels, graph_key=0)) for _ in range(8)]
        torch.cuda.synchronize()
        runs.append((losses, tr.engine.arena.param.clone()))
    for a, b in zip(runs[0][0], runs[1][0]):
        assert abs(a - b) <= 2e-2 * abs(a) + 1e-4
    assert float((runs[0][1] - runs[1][1]).norm()) <= 2e-2 * float((runs[0][1] - p0).norm())


# ------------------------------------------------------------------------------------------------ GPU: two ranks
def _rank_worker(rank, world, port, q, fused):
    os.environ["EGOT2_DP_FUSED"] = fused
    import dataclasses

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
        tr = TranslatorTrainer(sp, f"cuda:{rank}", "bf16", use_graphs=True, max_grad_norm=1.0,
                               weight_average=WeightAverage.ema(0.8))
        assert (tr.peer is not None) == (fused == "1")
        tr.load_state_dict(synth.make_state_dict(sp, 9))
        feats = [f[s.name][lo:hi].cuda() for s in sp.segments]
        labels = lab[lo:hi].cuda()
        for _ in range(4):
            tr.train_step(feats, labels, graph_key=0)
        torch.cuda.synchronize()
        q.put((rank, dict(avg=tr._avg.cpu(), param=tr.engine.arena.param.cpu())))
        dist.barrier()
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.parametrize("fused", ["0", "1"], ids=["nccl", "peer"])
def test_two_rank_averages_are_identical(fused):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import socket

    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_rank_worker, args=(r, 2, port, q, fused)) for r in range(2)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=170) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert torch.equal(got[0]["param"], got[1]["param"])
    assert torch.equal(got[0]["avg"], got[1]["avg"]) and not torch.equal(got[0]["avg"], torch.zeros_like(got[0]["avg"]))
