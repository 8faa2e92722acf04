"""SGD for the fused trainers (optim.SGD, egot2_sgd_step_fused, egot2_dp_desc.sgd): torch.optim.SGD with momentum, dampening
and Nesterov inside the one optimizer launch and the peer exchange.

CPU: SGD's input checks against torch's, the C entry's checks, the extended egot2_dp_desc against a compiled probe, the launch
plans (unchanged without SGD; with it the same launches with egot2_sgd_step_fused in place of every Adam entry) and the
optimizer-state round trip.  GPU (-m gpu): the entry against torch.optim.SGD(foreach=False) over three arenas (with LambdaLR,
clip_grad_norm_ and parameter groups), skipped NaN steps, graph against eager, both EgoT2-g trainers against torch.optim.SGD
on the engine's own gradient, resume, and the two-rank exchange."""
import contextlib
import ctypes as C
import math
import os

import pytest
import torch

from egot2_b200 import _lib as L
from egot2_b200.optim import SGD, LRSchedule, ParamGroup
from test_param_groups import (GROUPS, _PARENT_PLAN, _arena, _captured, _device_groups, _group_of, _guard, _hhi_setup,  # noqa: F401
                               _hhi_trainer, _hhi_trainer_gpu, _names, _plan, _prompt_batch, _read_guard, built, recorder)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_SGD = "egot2_sgd_step_fused"
NESTEROV = SGD(momentum=0.9, nesterov=True)

# egot2_sgd_step_fused's arguments by position
A_BUF, A_LR_DEV, A_MOM, A_DAMP, A_NEST, A_WD, A_STEP, A_STEP_DEV, A_GUARD, A_GROUPS, A_BMAP = 2, 5, 6, 7, 8, 9, 10, 11, 15, 16, 17


# ------------------------------------------------------------------------------------------------ CPU: checks, ABI
@pytest.mark.parametrize("kw", [dict(momentum=-0.1), dict(momentum=0.0, nesterov=True), dict(momentum=0.9, dampening=0.1,
                                nesterov=True), dict(momentum=math.nan), dict(momentum=math.inf), dict(dampening=math.nan),
                                dict(dampening=-math.inf)])
def test_sgd_rejects_what_torch_rejects(kw):
    """Every torch.optim.SGD rejection (negative momentum; Nesterov without momentum or with dampening) and non-finite values."""
    if math.isfinite(kw.get("momentum", 0.0)) and math.isfinite(kw.get("dampening", 0.0)):
        with pytest.raises(ValueError):
            torch.optim.SGD([torch.zeros(1, requires_grad=True)], lr=0.1, **kw)
    with pytest.raises(ValueError):
        SGD(**kw)


def test_sgd_accepts_what_torch_accepts():
    for kw in (dict(), dict(momentum=0.9), dict(momentum=0.9, dampening=0.1), dict(momentum=0.9, nesterov=True),
               dict(momentum=0.5, dampening=-0.5)):
        torch.optim.SGD([torch.zeros(1, requires_grad=True)], lr=0.1, **kw)
        s = SGD(**kw)
        assert SGD(**s.to_dict()) == s and isinstance(s.momentum, float)


@pytest.mark.parametrize("bad", [dict(momentum=-1.0), dict(nesterov=1), dict(momentum=0.9, buf=True, dampening=0.1, nesterov=1),
                                 dict(dampening=math.nan), dict(momentum=0.9), dict(buf=True), dict(step=0),
                                 dict(guard=True)])
def test_c_entry_checks(bad, built):
    """The entry's own checks, which run before any device work (n = 0 would otherwise return at once)."""
    kw = {**dict(momentum=0.0, dampening=0.0, nesterov=0, buf=False, step=1, guard=False), **bad}
    with pytest.raises(L.Egot2Error):
        L.call(_SGD, None, None, 8 if kw["buf"] else None, 0, 1e-3, None, kw["momentum"], kw["dampening"], kw["nesterov"],
               0.0, kw["step"], None, 1.0, None, 1, 8 if kw["guard"] else None, None, None, None)
    L.call(_SGD, None, None, None, 0, 1e-3, None, 0.0, 0.0, 0, 0.0, 1, None, 1.0, None, 1, None, None, None, None)


def test_dp_desc_layout_matches_header(built):
    import subprocess
    import tempfile
    fields = [f[0] for f in L.DpDesc._fields_]
    assert fields[-4:] == ["sgd", "momentum", "dampening", "nesterov"]
    prog = '#include <stdio.h>\n#include <stddef.h>\n#include "egot2.h"\nint main(){' + \
        'printf("size %zu\\n", sizeof(egot2_dp_desc));' + "".join(
            f'printf("{f} %zu\\n", offsetof(egot2_dp_desc, {f}));' for f in fields) + "return 0;}"
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "probe.c")
        open(src, "w").write(prog)
        exe = os.path.join(td, "probe")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
        out = subprocess.check_output([exe], text=True)
    for line in out.strip().splitlines():
        n, v = line.split()
        want = C.sizeof(L.DpDesc) if n == "size" else getattr(L.DpDesc, n).offset
        assert want == int(v), f"{n}: ctypes {want} != C {v}"


# ------------------------------------------------------------------------------------------------ CPU: launch plans
def test_adam_plan_is_unchanged(recorder):
    tr, feats, labels = _hhi_trainer()
    assert tr.sgd is None
    _plan(tr, feats, labels)
    assert _names(recorder) == _PARENT_PLAN


def _swap(names):
    return [_SGD if "adam" in n else n for n in names]


@pytest.mark.parametrize("momentum", [0.0, 0.9])
@pytest.mark.parametrize("groups", [False, True])
@pytest.mark.parametrize("guard", [False, True])
def test_sgd_plan_has_the_same_launches(guard, groups, momentum, recorder):
    """Whole-step graph and eager step: the launches of the Adam trainer with egot2_sgd_step_fused in place of every Adam entry,
    on the trainer's step_dev / lr_dev / guard / descriptor / block map, with a NULL buffer when momentum is 0."""
    kw = dict(max_grad_norm=1.0) if guard else {}
    if groups:
        kw["param_groups"] = GROUPS
    tr, feats, labels = _hhi_trainer(weight_decay=1e-4, **kw)
    _plan(tr, feats, labels)
    ref = _names(recorder)
    del recorder[:]
    sgd = SGD(momentum=momentum)
    tr, feats, labels = _hhi_trainer(weight_decay=1e-4, optimizer=sgd, **kw)
    _plan(tr, feats, labels)
    assert _names(recorder) == _swap(ref)
    assert _captured(recorder)[-1] == _SGD
    assert ("m" not in tr.opt_state) and (("buf" in tr.opt_state) == (momentum != 0.0))
    launches = [a for n, a in recorder if n == _SGD]
    assert len(launches) == 2
    graph, eager = launches
    for a in launches:
        assert a[A_BUF] == (tr.opt_state["buf"].data_ptr() if momentum else None)
        assert (a[A_MOM], a[A_DAMP], a[A_NEST]) == (momentum, 0.0, 0)
        assert a[A_GUARD] == (tr._guard_dev.data_ptr() if guard else None)
        assert (a[A_GROUPS], a[A_BMAP]) == ((tr._groups[0].data_ptr(), tr._groups[1].data_ptr()) if groups else (None, None))
        assert a[A_WD] == pytest.approx(1e-4)
    assert graph[A_STEP_DEV] == tr._step_dev.data_ptr()
    if guard or groups:
        assert eager[A_STEP_DEV] == tr._step_dev.data_ptr()
    else:
        assert eager[A_STEP_DEV] is None and eager[A_STEP] == 3


def test_scheduled_sgd_reads_the_device_lr(recorder):
    tr, feats, labels = _hhi_trainer(optimizer=NESTEROV, lr_schedule=LRSchedule.cosine(1e-2, 10))
    _plan(tr, feats, labels)
    launches = [a for n, a in recorder if n == _SGD]
    assert len(launches) == 2
    for a in launches:
        assert a[A_LR_DEV] == tr._lr_dev.data_ptr() and a[A_STEP_DEV] == tr._step_dev.data_ptr() and a[A_NEST] == 1


@pytest.mark.parametrize("extra", [{}, dict(max_grad_norm=1.0, param_groups=[ParamGroup("proj*", frozen=True),
                                                                           ParamGroup("*bias", weight_decay=0.0)])])
@pytest.mark.parametrize("graphs", ["1", "0"])
@pytest.mark.parametrize("kind", ["hhi", "hoi"])
def test_prompt_trainer_plans(kind, graphs, extra, recorder, monkeypatch):
    """EgoT2-g trainers, graph replay and eager: two steps issue the Adam trainer's launches with egot2_sgd_step_fused in place
    of the Adam entry.  The HHI eager step with plain Adam runs the unfused egot2_adam_step, so every forward re-casts the
    bf16 shadow; the SGD launch writes the shadow itself and leaves the gradient arena clean, which saves those casts."""
    from egot2_b200 import trainer as T
    monkeypatch.setenv("EGOT2_G_GRAPH", graphs)
    cls = T.HoiPromptTranslatorTrainer if kind == "hoi" else T.PromptTranslatorTrainer
    kw = dict(vocab=40) if kind == "hoi" else {}
    feats, labels = _prompt_batch(kind)
    plans = []
    for opt in (None, NESTEROV):
        del recorder[:]
        tr = cls(hidden=128, heads=4, layers=1, device="cpu", optimizer=opt, **kw, **extra)
        for _ in range(2):
            tr.train_step(feats, labels, graph_key=0)
        plans.append(_names(recorder))
    adam, sgd = plans
    if kind == "hhi" and graphs == "0" and not extra:
        cast = "egot2_cast_f32_to_bf16"
        assert sgd.count(cast) < adam.count(cast)
        adam, sgd = [n for n in adam if n != cast], [n for n in sgd if n != cast]
    assert sgd == _swap(adam)
    assert tr._grad_clean and "m" not in tr.opt_state
    launches = [a for n, a in recorder if n == _SGD]
    assert len(launches) == 2
    wd = 1e-4 if kind == "hoi" else 0.0           # HOI: AdamW's weight decay becomes SGD's coupled decay
    for a in launches:
        assert a[A_BUF] == tr.opt_state["buf"].data_ptr() and a[A_NEST] == 1 and a[A_WD] == pytest.approx(wd)
        assert a[A_STEP_DEV] == (tr._step_dev.data_ptr() if extra else None)
        assert a[A_GUARD] == (tr._guard_dev.data_ptr() if extra else None)


def test_nccl_path_takes_the_sgd_launch(recorder, monkeypatch):
    """Two ranks without the peer exchange: the all-reduce's scale reaches the SGD launch."""
    from egot2_b200 import trainer as T
    monkeypatch.setattr(T, "allreduce_gradients", lambda grad, pg: 0.5)
    tr, feats, labels = _hhi_trainer(optimizer=NESTEROV)
    tr.world, tr.use_graphs = 2, False
    del recorder[:]
    tr.train_step(feats, labels)
    (a,) = [a for n, a in recorder if n == _SGD]
    assert a[12] == 0.5 and "adam" not in " ".join(_names(recorder))


@pytest.mark.parametrize("split", ["0", "1"])
def test_peer_exchange_receives_the_sgd(split, recorder, monkeypatch):
    """Whole-step graph (one exchange, or two with EGOT2_DP_SPLIT=1) and eager step: every exchange gets the trainer's SGD and
    never `decoupled`; an Adam trainer's exchanges get sgd=None."""
    monkeypatch.setenv("EGOT2_DP_SPLIT", split)
    got = []

    class FakePeer:
        def step(self, state, step, hp, stream, **kw):
            got.append(kw)
    for opt in (None, NESTEROV):
        del got[:]
        tr, feats, labels = _hhi_trainer(optimizer=opt)
        tr.peer, tr.graph_update = FakePeer(), True
        tr.train_step(feats, labels, graph_key=0)
        tr.use_graphs = False
        tr.train_step(feats, labels)
        assert len(got) == (3 if split == "1" else 2)
        assert all(k["sgd"] is opt and not k.get("decoupled", False) for k in got)


def test_hoi_prompt_peer_exchange_drops_decoupled(recorder, monkeypatch):
    from egot2_b200 import trainer as T
    monkeypatch.setenv("EGOT2_G_GRAPH", "0")
    got = []

    class FakePeer:
        def step(self, state, step, hp, stream, **kw):
            got.append(kw)
    feats, labels = _prompt_batch("hoi")
    for opt in (None, NESTEROV):
        del got[:]
        tr = T.HoiPromptTranslatorTrainer(hidden=128, heads=4, layers=1, vocab=40, device="cpu", optimizer=opt)
        tr.peer = FakePeer()
        tr.train_step(feats, labels)
        assert got[0]["decoupled"] == (opt is None) and got[0]["sgd"] is opt


def test_peer_desc_carries_the_sgd(built, monkeypatch):
    """PeerExchange.step writes the SGD fields and the momentum buffer (NULL without momentum) into egot2_dp_desc."""
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
    hp = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-4)

    def rec(name, d, *a):
        o = d._obj
        descs.append((o.sgd, o.momentum, o.dampening, o.nesterov, o.exp_avg, o.exp_avg_sq, o.decoupled))
    monkeypatch.setattr(L, "call", rec)
    monkeypatch.setattr(torch.cuda, "device", lambda d: contextlib.nullcontext())
    states = [{}, {}, {}]
    ex.step(states[0], 1, hp, 0, decoupled=True)
    ex.step(states[1], 1, hp, 0, sgd=SGD(momentum=0.9, dampening=0.25))
    ex.step(states[2], 1, hp, 0, sgd=SGD())
    assert descs[0][:4] == (0, 0.0, 0.0, 0) and descs[0][4] == states[0]["m"].data_ptr() and descs[0][6] == 1
    assert set(states[1]) == {"buf"} and descs[1] == (1, pytest.approx(0.9), 0.25, 0, states[1]["buf"].data_ptr(), None, 0)
    assert states[2] == {} and descs[2] == (1, 0.0, 0.0, 0, None, None, 0)


def test_trainer_input_checks(recorder):
    from egot2_b200 import specs
    from egot2_b200.trainer import TranslatorTrainer
    spec = specs.hhi_ttm_spec(128, 4, 1, 0.5, True)
    for kw in (dict(betas=(0.8, 0.999)), dict(eps=1e-6)):
        with pytest.raises(ValueError, match="betas and eps"):
            TranslatorTrainer(spec, "cpu", "bf16", optimizer=NESTEROV, **kw)
    with pytest.raises(ValueError, match="optim.SGD"):
        TranslatorTrainer(spec, "cpu", "bf16", optimizer=torch.optim.SGD)
    TranslatorTrainer(spec, "cpu", "bf16", betas=(0.8, 0.999))
    with pytest.raises(L.Egot2Error):
        _hhi_trainer()[0].engine.sgd_step({}, 1, 1e-3, NESTEROV, guard=torch.zeros(4))     # needs the device step count


def test_optimizer_state_dict_round_trip(recorder):
    sgd = SGD(momentum=0.9, dampening=0.1)
    tr, feats, labels = _hhi_trainer(optimizer=sgd, weight_decay=1e-4, max_grad_norm=1.0)
    tr.train_step(feats, labels, graph_key=0)
    for name in tr.engine.arena.shapes:                          # the buffer outside the parameters' slots stays zero
        tr.engine.arena.view(name, tr.opt_state["buf"]).normal_()
    sd = tr.optimizer_state_dict()
    assert "exp_avg" not in sd and "exp_avg_sq" not in sd and sd["sgd"] == dict(momentum=0.9, dampening=0.1, nesterov=False)
    assert set(sd["momentum_buffer"]) == set(tr.engine.arena.shapes)
    tr2, _, _ = _hhi_trainer(optimizer=sgd, weight_decay=1e-4, max_grad_norm=1.0)
    tr2.load_optimizer_state_dict(sd)
    assert torch.equal(tr2.opt_state["buf"], tr.opt_state["buf"]) and tr2.step_count == 1 and int(tr2._step_dev) == 1
    assert "m" not in tr2.opt_state
    buf = tr2.opt_state["buf"]
    tr2.load_optimizer_state_dict(sd)
    assert tr2.opt_state["buf"] is buf                           # in place: captured graphs hold it
    # momentum 0: no buffer at all
    plain_sgd = _hhi_trainer(optimizer=SGD())[0]
    sd0 = plain_sgd.optimizer_state_dict()
    assert sd0["momentum_buffer"] is None and sd0["sgd"] == dict(momentum=0.0, dampening=0.0, nesterov=False)
    tr3 = _hhi_trainer(optimizer=SGD())[0]
    tr3.load_optimizer_state_dict(sd0)
    assert tr3.opt_state == {}
    # the Adam dict keeps its keys
    adam_sd = _hhi_trainer(max_grad_norm=1.0)[0].optimizer_state_dict()
    assert "exp_avg" in adam_sd and "sgd" not in adam_sd and "momentum_buffer" not in adam_sd
    # rejections: Adam <-> SGD, and other SGD fields
    with pytest.raises(ValueError, match="Adam"):
        _hhi_trainer(optimizer=sgd, max_grad_norm=1.0)[0].load_optimizer_state_dict(adam_sd)
    with pytest.raises(ValueError, match="SGD"):
        _hhi_trainer(max_grad_norm=1.0)[0].load_optimizer_state_dict(sd)
    for other in (SGD(momentum=0.9), SGD(momentum=0.8, dampening=0.1), SGD(momentum=0.9, nesterov=True), SGD()):
        with pytest.raises(ValueError, match="fixed at construction"):
            _hhi_trainer(optimizer=other, max_grad_norm=1.0)[0].load_optimizer_state_dict(sd)


# ------------------------------------------------------------------------------------------------ GPU: the entry
CONFIGS = [SGD(), SGD(momentum=0.9), SGD(momentum=0.9, dampening=0.1), SGD(momentum=0.9, nesterov=True)]


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["plain", "sched", "clip", "groups"])
@pytest.mark.parametrize("wd", [0.0, 1e-4])
@pytest.mark.parametrize("sgd", CONFIGS, ids=["m0", "m09", "m09_d01", "nesterov"])
@pytest.mark.parametrize("kind", ["hhi", "pnr", "lta"])
def test_sgd_matches_torch(kind, sgd, wd, variant):
    """egot2_sgd_step_fused over a translator arena == torch.optim.SGD(foreach=False) over 5 steps on fresh gradients (the first
    step initialises the buffer), with LambdaLR (sched), clip_grad_norm_ (clip) or one param group per ParamGroup (groups);
    after every step the shadow is bf16(param) bit for bit and the gradient arena is zero."""
    arena = _arena(kind)
    n = arena.numel
    groups = variant == "groups"
    if groups:
        desc, bmap, hp = _device_groups(arena, GROUPS, wd)
        gid = _group_of(arena, bmap)
    else:
        desc = bmap = None
        hp, gid = [(1.0, wd, False)], {name: 0 for name in arena.shapes}
    s = LRSchedule.cosine(2e-2, 5, end_lr=1e-4, warmup_steps=2, warmup_start_lr=1e-3)
    base = s.base_lr if variant == "sched" else 1e-2
    torch.manual_seed(7)
    p = torch.zeros(n, device="cuda")
    for name in arena.shapes:
        arena.view(name, p).normal_(0.0, 0.1)
    p0 = p.clone()
    refs = {name: arena.view(name, p).clone() for name in arena.shapes}
    for name in refs:
        refs[name].requires_grad_(not hp[gid[name]][2])
    pgroups = [dict(params=[refs[nm] for nm in refs if gid[nm] == k], lr=base * hp[k][0], weight_decay=hp[k][1])
               for k in range(len(hp)) if not hp[k][2]]
    opt = torch.optim.SGD(pgroups, lr=base, momentum=sgd.momentum, dampening=sgd.dampening, nesterov=sgd.nesterov,
                          foreach=False)
    if variant == "sched":
        from test_lr_schedule import lr_at
        lam = torch.optim.lr_scheduler.LambdaLR(opt, lambda t: lr_at(s, t) / s.base_lr)
    trainable = [r for r in refs.values() if r.requires_grad]
    frozen = torch.zeros(n, dtype=torch.bool, device="cuda")
    for name in arena.shapes:
        if hp[gid[name]][2]:
            arena.view(name, frozen).fill_(True)
    buf = torch.zeros(n, device="cuda") if sgd.momentum else None
    shadow = p.to(torch.bfloat16)
    step = torch.zeros(1, device="cuda", dtype=torch.int32)
    lr = torch.zeros(1, device="cuda", dtype=torch.float32)
    sched = torch.frombuffer(bytearray(bytes(s.pack())), dtype=torch.uint8).cuda()
    ws = torch.zeros(int(L.load().egot2_grad_norm_workspace_bytes()), device="cuda", dtype=torch.uint8)
    st = torch.cuda.current_stream().cuda_stream
    on_dev = variant != "plain"
    for i in range(5):
        g = torch.zeros(n, device="cuda")
        for name in arena.shapes:
            arena.view(name, g).normal_().mul_(0.8 + 0.05 * i)
        for name, r in refs.items():
            r.grad = arena.view(name, g).clone() if r.requires_grad else None
        guard = None
        if variant == "clip":
            want = float(torch.linalg.vector_norm(g.double()))
            torch.nn.utils.clip_grad_norm_(trainable, 0.5 * want)
            guard = _guard(0.5 * want)
        opt.step()
        if variant == "sched":
            lam.step()
            L.call("egot2_opt_advance", step.data_ptr(), sched.data_ptr(), lr.data_ptr(), st)
        else:
            step.add_(1)
        if guard is not None:
            L.call("egot2_grad_norm", g.data_ptr(), n, 1.0, guard.data_ptr(), step.data_ptr(), ws.data_ptr(), ws.numel(), st)
        L.call(_SGD, p.data_ptr(), g.data_ptr(), None if buf is None else buf.data_ptr(), n, base,
               lr.data_ptr() if variant == "sched" else None, sgd.momentum, sgd.dampening, int(sgd.nesterov), wd, i + 1,
               step.data_ptr() if on_dev else None, 1.0, shadow.data_ptr(), 1, None if guard is None else guard.data_ptr(),
               None if desc is None else desc.data_ptr(), None if bmap is None else bmap.data_ptr(), st)
        if guard is not None:
            r = _read_guard(guard)
            assert r.skip == 0 and r.coef < 1.0
        assert float(g.abs().max()) == 0.0
        assert torch.equal(shadow, p.to(torch.bfloat16))
    err = max(float((arena.view(name, p) - r.detach()).abs().max()) for name, r in refs.items())
    assert err < 1e-6, err
    if buf is not None:
        berr = max(float((arena.view(name, buf) - opt.state[r]["momentum_buffer"]).abs().max() / (
            1.0 + opt.state[r]["momentum_buffer"].abs().max())) for name, r in refs.items() if r.requires_grad)
        assert berr < 1e-6, berr
        if groups:
            assert float(buf[frozen].abs().max()) == 0.0
    if groups:
        assert torch.equal(p[frozen], p0[frozen]) and bool(frozen.any())
    assert not torch.equal(p[~frozen], p0[~frozen])


def _nan_setup():
    arena = _arena("hhi")
    n = arena.numel
    torch.manual_seed(3)
    p = torch.randn(n, device="cuda") * 0.1
    buf = torch.zeros(n, device="cuda")
    shadow = p.to(torch.bfloat16)
    step = torch.zeros(1, device="cuda", dtype=torch.int32)
    ws = torch.zeros(int(L.load().egot2_grad_norm_workspace_bytes()), device="cuda", dtype=torch.uint8)
    guard = _guard(math.inf)
    st = torch.cuda.current_stream().cuda_stream

    def step_with(g):
        step.add_(1)
        L.call("egot2_grad_norm", g.data_ptr(), n, 1.0, guard.data_ptr(), step.data_ptr(), ws.data_ptr(), ws.numel(), st)
        L.call(_SGD, p.data_ptr(), g.data_ptr(), buf.data_ptr(), n, 1e-2, None, 0.9, 0.0, 1, 0.0, 1, step.data_ptr(), 1.0,
               shadow.data_ptr(), 1, guard.data_ptr(), None, None, st)
        assert float(g.abs().max()) == 0.0
    return n, p, buf, shadow, step, guard, step_with


@pytest.mark.gpu
def test_nan_step_is_skipped_bit_for_bit():
    n, p, buf, shadow, step, guard, step_with = _nan_setup()
    for _ in range(3):
        step_with(torch.randn(n, device="cuda"))
    before = [t.clone() for t in (p, buf, shadow)]
    g = torch.randn(n, device="cuda")
    g[n // 2] = float("nan")
    step_with(g)
    r = _read_guard(guard)
    assert r.skip == 1 and r.skipped == 1 and int(step) == 3
    for x, y in zip(before, (p, buf, shadow)):
        assert torch.equal(x, y)


@pytest.mark.gpu
def test_nan_first_step_leaves_the_initialisation_to_the_next():
    """A skipped first step takes the count back to 0, so the next applied step starts the buffer from its own gradient
    (GradScaler skips optimizer.step(), and torch's buffer stays None until then)."""
    n, p, buf, shadow, step, guard, step_with = _nan_setup()
    g = torch.randn(n, device="cuda")
    g[0] = float("nan")
    step_with(g)
    assert int(step) == 0 and float(buf.abs().max()) == 0.0
    g = torch.randn(n, device="cuda")
    want = g.clone()
    step_with(g)
    assert int(step) == 1 and _read_guard(guard).skip == 0
    assert torch.equal(buf, want)


# ------------------------------------------------------------------------------------------------ GPU: trainers
@pytest.mark.gpu
def test_graph_matches_eager_with_sgd_and_clipping():
    """Whole-step graph == eager TranslatorTrainer with SGD and clipping active (dropout off).  Parameters by the L2 norm of the
    difference relative to how far training moved them: the backward's fp32 atomics make single elements of two runs
    differ (test_grad_guard)."""
    spec, feats, labels = _hhi_setup()
    kw = dict(optimizer=NESTEROV, weight_decay=1e-4, lr=2e-2, max_grad_norm=0.05)
    tg = _hhi_trainer_gpu(spec, use_graphs=True, **kw)
    te = _hhi_trainer_gpu(spec, use_graphs=False, **kw)
    p0 = te.engine.arena.param.clone()
    for _ in range(6):
        lg = float(tg.train_step(feats, labels, graph_key=0))
        le = float(te.train_step(feats, labels))
        assert abs(lg - le) <= 2e-2 * abs(le) + 1e-4
    torch.cuda.synchronize()
    assert float(tg.last_grad_norm) > 0.05 and float(te.last_grad_norm) > 0.05           # clipping was active
    pg, pe = tg.engine.arena.param, te.engine.arena.param
    assert float((pg - pe).norm()) <= 2e-2 * float((pe - p0).norm())
    bg, be = tg.opt_state["buf"], te.opt_state["buf"]
    assert float((bg - be).norm()) <= 2e-2 * float(be.norm())
    assert float(tg.engine.arena.grad.abs().max()) == 0.0 and torch.equal(tg.engine.arena.shadow, pg.to(torch.bfloat16))


@pytest.mark.gpu
@pytest.mark.parametrize("graphs", ["1", "0"])
@pytest.mark.parametrize("kind", ["hhi", "hoi"])
def test_prompt_trainers_match_torch_sgd(kind, graphs, monkeypatch):
    """Two EgoT2-g steps (dropout 0) == torch.optim.SGD applied to the gradient the engine produced for the same batches.

    The reference takes that gradient from the arena right before each optimizer launch (the launch is always eager in these
    trainers), so the order of the backward's fp32 atomic accumulations does not enter: a second forward/backward would
    give a gradient that differs in the last bits.  What remains is the fp32 rounding of the update itself, hence 1e-6."""
    from egot2_b200 import synth, trainer as T
    monkeypatch.setenv("EGOT2_G_GRAPH", graphs)
    feats, labels = _prompt_batch(kind)
    feats, labels = [f.cuda() for f in feats], labels.cuda()
    cls = T.HoiPromptTranslatorTrainer if kind == "hoi" else T.PromptTranslatorTrainer
    extra = dict(vocab=40) if kind == "hoi" else {}
    tr = cls(hidden=128, heads=4, layers=1, dropout=0.0, device="cuda:0", dtype="bf16", lr=5e-2, optimizer=NESTEROV, **extra)
    tr.load_state_dict(synth.make_state_dict(tr.spec, 3))
    a = tr.engine.arena
    ref = {name: a.view(name).clone().requires_grad_(True) for name in a.shapes}
    start = {name: r.detach().clone() for name, r in ref.items()}
    opt = torch.optim.SGD(list(ref.values()), lr=tr.hp["lr"], momentum=0.9, nesterov=True,
                          weight_decay=tr.hp["weight_decay"], foreach=False)
    real = tr.engine.sgd_step

    def spy(state, step, lr, sgd, weight_decay=0.0, grad_scale=1.0, **k):
        for name, r in ref.items():
            r.grad = a.view(name, a.grad) * grad_scale
        opt.step()
        return real(state, step, lr, sgd, weight_decay, grad_scale=grad_scale, **k)
    tr.engine.sgd_step = spy
    for _ in range(2):
        tr.train_step(feats, labels, graph_key=0)
    torch.cuda.synchronize()
    err = max(float((a.view(name) - r.detach()).abs().max()) for name, r in ref.items())
    scale = max(1.0, max(float(r.detach().abs().max()) for r in ref.values()))
    assert err <= 1e-6 * scale, err
    berr = max(float((a.view(name, tr.opt_state["buf"]) - opt.state[r]["momentum_buffer"]).abs().max())
               for name, r in ref.items())
    assert berr <= 1e-6 * max(1.0, max(float(opt.state[r]["momentum_buffer"].abs().max()) for r in ref.values())), berr
    assert tr._grad_clean and float(a.grad.abs().max()) == 0.0
    assert max(float((a.view(name) - p).abs().max()) for name, p in start.items()) > 1e-3          # training moved them


@pytest.mark.gpu
def test_resume_mid_run():
    """Steps 1-3 on the whole-step graph, save, a fresh trainer loads: its parameters, buffer and device step count equal the
    saved run's bit for bit, and three more optimizer steps on the same fixed gradients (through the trainers' eager
    optimizer path, with a schedule and a guard) keep both bit-identical.  Without the restored step count the resumed
    trainer would start the buffer afresh."""
    spec, feats, labels = _hhi_setup()
    kw = dict(use_graphs=True, optimizer=NESTEROV, weight_decay=1e-4, lr_schedule=LRSchedule.cosine(2e-2, 8),
              max_grad_norm=1e3)
    full = _hhi_trainer_gpu(spec, **kw)
    for _ in range(3):
        full.train_step(feats, labels, graph_key=0)
    torch.cuda.synchronize()
    sd, osd = full.state_dict(), full.optimizer_state_dict()
    tr = _hhi_trainer_gpu(spec, **kw)
    tr.load_state_dict(sd)
    tr.load_optimizer_state_dict(osd)
    assert torch.equal(tr.engine.arena.param, full.engine.arena.param)
    assert torch.equal(tr.opt_state["buf"], full.opt_state["buf"]) and int(tr._step_dev) == int(full._step_dev) == 3
    torch.manual_seed(4)
    grads = [torch.randn(full.engine.arena.numel, device="cuda") * 1e-3 for _ in range(3)]
    for t in (full, tr):
        for g in grads:
            t.step_count += 1
            t.engine.arena.grad.copy_(g)
            t._reduce_and_update()
    torch.cuda.synchronize()
    assert torch.equal(tr.engine.arena.param, full.engine.arena.param)
    assert torch.equal(tr.opt_state["buf"], full.opt_state["buf"]) and int(tr._step_dev) == 6
    # ... and the resumed trainer keeps training on its graph
    p = tr.engine.arena.param.clone()
    tr.train_step(feats, labels, graph_key=0)
    torch.cuda.synchronize()
    assert not torch.equal(tr.engine.arena.param, p) and int(tr._step_dev) == 7


# ------------------------------------------------------------------------------------------------ GPU: two ranks
def _rank_worker(rank, world, port, case, q):
    os.environ["EGOT2_DP_FUSED"] = "1"
    if case == "split":
        os.environ["EGOT2_DP_SPLIT"] = "1"
    import dataclasses

    import torch
    import torch.distributed as dist

    from egot2_b200 import specs, synth
    from egot2_b200.trainer import TranslatorTrainer
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        solo = [dist.new_group([r]) for r in range(world)]
        sp = dataclasses.replace(specs.hhi_ttm_spec(128, 4, 2, 0.0, True), p_embed=0.0)
        B, seg = 16, (10, 10, 10)
        f = synth.make_features(sp, B, seg, seed=77, dtype=torch.bfloat16)
        lab = synth.make_labels(sp, B, seg, seed=77)
        kw = dict(use_graphs=True, lr=2e-2, weight_decay=1e-4, optimizer=SGD(momentum=0.9, nesterov=True))
        if case == "guard":
            kw["max_grad_norm"] = 0.05
        if case == "groups":
            kw["param_groups"] = GROUPS

        def run(tr, lo, hi):
            tr.load_state_dict(synth.make_state_dict(sp, 9))
            start = tr.engine.arena.param.cpu()
            feats = [f[s.name][lo:hi].cuda() for s in sp.segments]
            labels = lab[lo:hi].cuda()
            for _ in range(4):
                tr.train_step(feats, labels, graph_key=0)
            torch.cuda.synchronize()
            return start, tr.engine.arena.param.cpu(), tr.opt_state["buf"].cpu()
        tr = TranslatorTrainer(sp, f"cuda:{rank}", "bf16", **kw)
        assert tr.peer is not None
        _, p, buf = run(tr, rank * B // world, (rank + 1) * B // world)
        out = dict(p=p, buf=buf)
        if rank == 0:                                  # the one-rank run on the concatenated batch
            one = TranslatorTrainer(sp, "cuda:0", "bf16", process_group=solo[0], **kw)
            assert one.peer is None and one.world == 1
            out["one"] = run(one, 0, B)
        q.put((rank, out))
        dist.barrier()
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["plain", "guard", "groups", "split"])
def test_two_rank_sgd_peer_exchange(case):
    """The peer-memory exchange with SGD (EGOT2_DP_FUSED=1; split: EGOT2_DP_SPLIT=1, two [lo, hi) exchanges): ranks are
    bit-identical, and match one rank on the concatenated batch (by the L2 norm of the difference relative to how far training
    moved the parameters: the rank-order sum and the backward's fp32 atomics reorder the additions).  Each rank holds the
    momentum buffer of its own slices only (the rest stays zero), so the two ranks' buffers add up to the one-rank buffer."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import socket

    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_rank_worker, args=(r, 2, port, case, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=240) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert torch.equal(got[0]["p"], got[1]["p"]), "ranks diverged"
    start, p_one, buf_one = got[0]["one"]
    assert float((got[0]["p"] - p_one).norm()) <= 2e-2 * float((p_one - start).norm())
    assert bool(((got[0]["buf"] != 0) & (got[1]["buf"] != 0)).sum() == 0)
    assert float((got[0]["buf"] + got[1]["buf"] - buf_one).norm()) <= 2e-2 * float(buf_one.norm())
