"""Per-parameter gradient and weight statistics of the fused trainers (stats.ParamStats, egot2_param_stats).

CPU: the bucket edges against SummaryWriter's, the host trimming against make_histogram, the launch plans (one stats launch
right before every optimizer launch, on the trainer's device step count), input checks, the ABI mirrors and the C entry's
checks.  GPU (-m gpu): the kernel against numpy over the HHI, PNR and LTA-b512 arenas, the statistics inside the trainers
against the arrays their optimizer received, the guard, frozen groups, the EgoT2-g trainers, TensorBoard end to end, training
unperturbed, and two ranks on the NCCL path."""
import contextlib
import ctypes as C
import os

import numpy as np
import pytest
import torch

from egot2_b200 import _lib as L
from egot2_b200.optim import ParamGroup
from egot2_b200.stats import ParamStats, default_edges, histogram_raw, plan_units
from test_param_groups import (GROUPS, _arena, _hhi_setup, _hhi_trainer, _hhi_trainer_gpu, _names,  # noqa: F401
                               _prompt_batch, built, recorder)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_STATS = "egot2_param_stats"
_OPT = {"egot2_adam_step", "egot2_adam_step_fused", "egot2_adamw_step_fused", "egot2_adam_step_fused_dev",
        "egot2_adam_step_fused_sched", "egot2_adam_step_fused_guard", "egot2_adam_step_fused_groups", "egot2_sgd_step_fused"}
_NORM = {"egot2_grad_norm", "egot2_grad_norm_groups"}


# ------------------------------------------------------------------------------------------------ CPU: format
def test_edges_equal_summary_writer_default_bins(tmp_path):
    from torch.utils.tensorboard import SummaryWriter
    w = SummaryWriter(log_dir=str(tmp_path))
    want = w.default_bins
    w.close()
    got = default_edges()
    assert len(want) == got.size == L.STATS_BUCKETS + 1
    assert all(float(a) == b for a, b in zip(got, want))


def _f32_inside(x):
    """The fp32 value nearest to x on the side of 0 (fp32 values are what the kernel bins)."""
    f = np.float32(x)
    return float(np.nextafter(f, np.float32(0)) if abs(float(f)) > abs(x) else f)


def _values_cases():
    rng = np.random.default_rng(3)
    e = default_edges()
    mag = 10.0 ** rng.uniform(-14, 22, 5000)
    yield "random", mag * rng.choice([-1.0, 1.0], mag.size)
    yield "one bucket", np.full(100, 0.37)
    yield "first bucket", np.array([_f32_inside(e[0]), _f32_inside(e[0] * 0.99)])
    yield "last bucket", np.array([_f32_inside(e[-1]), _f32_inside(e[-1] * 0.99)])
    yield "zeros", np.array([0.0, -0.0, 0.0])
    yield "outside", np.array([1e30, -1e30, 3.0, -2.5, e[-1] * 1.0001])
    yield "edges", e[::7].copy()


@pytest.mark.parametrize("case", [c for c, _ in _values_cases()])
def test_trimming_equals_make_histogram(case):
    from torch.utils.tensorboard.summary import make_histogram
    values = dict(_values_cases())[case].astype(np.float32).astype(np.float64)
    edges = default_edges()
    counts, _ = np.histogram(values, bins=edges)
    stat = L.ParamStat(sum=values.sum(), sum_squares=values.dot(values), min=values.min(), max=values.max(), norm=0.0,
                       nonfinite=0, num=values.size)
    h = histogram_raw(stat, counts, edges)
    ref = make_histogram(values, edges.tolist())
    assert h["bucket_limits"] == list(ref.bucket_limit) and h["bucket_counts"] == list(ref.bucket)
    assert h["num"] == ref.num and h["min"] == ref.min and h["max"] == ref.max


def test_trimming_of_an_empty_histogram():
    assert histogram_raw(L.ParamStat(), np.zeros(L.STATS_BUCKETS, np.int32), default_edges()) is None


@pytest.mark.parametrize("bad", [0, -3, 1.5, True, "2", None])
def test_param_stats_input_checks(bad):
    with pytest.raises(ValueError):
        ParamStats(bad)
    assert ParamStats(np.int64(4)).every == 4 and ParamStats(1, histograms=False).histograms is False


def test_units_never_span_two_parameters():
    """LTA: the stacked head biases sit back to back; every unit lies inside one parameter and the units of a parameter are
    consecutive and cover it exactly, gradient units first."""
    arena = _arena("lta")
    names = list(arena.shapes)
    has_grad = [i % 3 != 0 for i in range(len(names))]
    params, units = plan_units(arena.shapes, arena.offsets, has_grad, unit=1000)
    assert [u.array for u in units] == sorted(u.array for u in units)
    for p, n in enumerate(names):
        pr = params[p]
        numel = arena.view(n).numel()
        assert pr.offset == arena.offsets[n] and pr.numel == numel and pr.has_grad == int(has_grad[p])
        for a in (0, 1):
            us = units[pr.first_unit[a]:pr.first_unit[a] + pr.n_units[a]]
            if a == 0 and not has_grad[p]:
                assert pr.n_units[0] == 0
                continue
            assert all(u.param == p and u.array == a for u in us)
            assert us[0].begin == arena.offsets[n] and us[-1].end == arena.offsets[n] + numel
            assert all(x.end == y.begin for x, y in zip(us, us[1:]))
    assert any(arena.offsets[b] % 64 for b in arena.head_b_names)


def test_struct_layouts_match_header(built):
    import subprocess
    import tempfile
    names = {"egot2_param_stats_desc": L.ParamStatsDesc, "egot2_stats_param": L.StatsParam,
             "egot2_stats_unit": L.StatsUnit, "egot2_param_stat": L.ParamStat}
    fields = [(n, f[0]) for n, cls in names.items() for f in cls._fields_]
    prog = '#include <stdio.h>\n#include <stddef.h>\n#include "egot2.h"\nint main(){' + "".join(
        f'printf("{n} %zu\\n", sizeof({n}));' for n in names) + "".join(
        f'printf("{n}.{f} %zu\\n", offsetof({n}, {f}));' for n, f in fields) + \
        'printf("buckets %d\\n", EGOT2_STATS_BUCKETS);return 0;}'
    with tempfile.TemporaryDirectory() as td:
        src = os.path.join(td, "probe.c")
        open(src, "w").write(prog)
        exe = os.path.join(td, "probe")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
        out = subprocess.check_output([exe], text=True)
    for line in out.strip().splitlines():
        n, v = line.split()
        if n == "buckets":
            assert L.STATS_BUCKETS == int(v)
        elif "." in n:
            st, f = n.split(".")
            assert getattr(names[st], f).offset == int(v), f"{n}: ctypes {getattr(names[st], f).offset} != C {v}"
        else:
            assert C.sizeof(names[n]) == int(v), f"{n}: ctypes {C.sizeof(names[n])} != C {v}"


def test_c_entry_checks(built):
    lib = L.load()
    assert lib.egot2_param_stats_workspace_bytes(0, 4) == 0 and lib.egot2_param_stats_workspace_bytes(3, 0) == 0
    need = lib.egot2_param_stats_workspace_bytes(3, 5)
    assert need >= 5 * 16 + 2 * 3 * L.STATS_BUCKETS * 4
    ok = dict(grad=256, param=512, scale=1.0, step=768, desc=1024, params=1280, P=3, units=1536, U=5, edges=1792,
              stats=2048, counts=2304, ws=4096, ws_bytes=need)
    bad_cases = [dict(grad=None), dict(step=None), dict(desc=None), dict(stats=None), dict(ws=None), dict(P=0), dict(U=-1),
                 dict(edges=None), dict(counts=None), dict(scale=float("nan")), dict(ws_bytes=need - 1), dict(ws=4100)]
    for bad in bad_cases:
        a = {**ok, **bad}
        rc = lib.egot2_param_stats(a["grad"], a["param"], a["scale"], a["step"], a["desc"], a["params"], a["P"], a["units"],
                                   a["U"], a["edges"], a["stats"], a["counts"], a["ws"], a["ws_bytes"], None)
        assert rc != 0, bad
        assert b"param_stats" in lib.egot2_last_error()


# ------------------------------------------------------------------------------------------------ CPU: launch plans
def _check_stats_before_every_optimizer(calls, step_dev, scale=None):
    """Exactly one egot2_param_stats right before every optimizer launch (before the guard's norm, when there is one), none
    elsewhere, each on the trainer's step_dev; returns the number of optimizer launches."""
    names = _names(calls)
    n_opt = 0
    for i, n in enumerate(names):
        if n in _OPT:
            n_opt += 1
            j = i - 1 if names[i - 1] not in _NORM else i - 2
            assert names[j] == _STATS, names[max(0, j - 2):i + 1]
        if n == _STATS:
            assert names[i + 1] in _OPT or (names[i + 1] in _NORM and names[i + 2] in _OPT)
            a = calls[i][1]
            assert a[3] == step_dev.data_ptr()
            if scale is not None:
                assert a[2] == scale
    assert names.count(_STATS) == n_opt > 0
    return n_opt


def _plan(tr, feats, labels):
    tr.train_step(feats, labels, graph_key=0)
    tr.train_step(feats, labels, graph_key=0)
    tr.use_graphs = False
    tr.train_step(feats, labels)


@pytest.mark.parametrize("config", ["plain", "guard", "groups", "guard+groups", "sgd", "sched"])
def test_plan_has_one_stats_launch_before_every_optimizer_launch(config, recorder):
    """Whole-step graph (the stats launch is captured) and eager step: the launches without stats, plus one stats launch in
    front of every optimizer launch.  Without a guard, groups or schedule the eager optimizer reads the device step count."""
    from egot2_b200.optim import SGD, LRSchedule
    kw = {"plain": {}, "guard": dict(max_grad_norm=1.0), "groups": dict(param_groups=GROUPS),
          "guard+groups": dict(max_grad_norm=1.0, param_groups=GROUPS), "sgd": dict(optimizer=SGD(momentum=0.9)),
          "sched": dict(lr_schedule=LRSchedule.cosine(1e-3, 10))}[config]
    tr, feats, labels = _hhi_trainer(**kw)
    _plan(tr, feats, labels)
    ref = _names(recorder)
    del recorder[:]
    tr, feats, labels = _hhi_trainer(param_stats=ParamStats(3), **kw)
    _plan(tr, feats, labels)
    got = _names(recorder)
    assert _check_stats_before_every_optimizer(recorder, tr._step_dev, 1.0) == 2
    cap = got[got.index("<capture>"):got.index("</capture>")]
    assert _STATS in cap
    dev_step = {"egot2_adam_step_fused": "egot2_adam_step_fused_dev"}
    assert [n for n in got if n != _STATS] == [dev_step.get(n, n) for n in ref]


def test_dp_overlap_plan(recorder, monkeypatch):
    """The data-parallel overlap path (two graphs with the all-reduce between them): the stats launch follows the all-reduce
    and precedes the optimizer, on the all-reduce's scale."""
    import torch.distributed as dist
    monkeypatch.setenv("EGOT2_DP_OVERLAP", "force")

    class Work:
        def wait(self):
            pass
    monkeypatch.setattr(dist, "all_reduce", lambda *a, **k: Work())
    tr, feats, labels = _hhi_trainer(param_stats=ParamStats(1))
    assert tr.dp_overlap
    tr.world = 2
    for _ in range(2):
        tr.train_step(feats, labels, graph_key=0)
    assert _check_stats_before_every_optimizer(recorder, tr._step_dev, 0.5) == 2


def test_nccl_path_plan(recorder, monkeypatch):
    from egot2_b200 import trainer as T
    monkeypatch.setattr(T, "allreduce_gradients", lambda grad, pg: 0.5)
    tr, feats, labels = _hhi_trainer(param_stats=ParamStats(2), max_grad_norm=1.0)
    tr.world, tr.use_graphs = 2, False
    del recorder[:]
    tr.train_step(feats, labels)
    assert _check_stats_before_every_optimizer(recorder, tr._step_dev, 0.5) == 1


@pytest.mark.parametrize("graphs", ["1", "0"])
@pytest.mark.parametrize("kind", ["hhi", "hoi"])
def test_prompt_trainer_plans(kind, graphs, recorder, monkeypatch):
    from egot2_b200 import trainer as T
    monkeypatch.setenv("EGOT2_G_GRAPH", graphs)
    cls = T.HoiPromptTranslatorTrainer if kind == "hoi" else T.PromptTranslatorTrainer
    extra = dict(vocab=40) if kind == "hoi" else {}
    feats, labels = _prompt_batch(kind)
    for kw in ({}, dict(max_grad_norm=1.0, param_groups=[ParamGroup("proj*", frozen=True)])):
        del recorder[:]
        tr = cls(hidden=128, heads=4, layers=1, device="cpu", param_stats=ParamStats(1), **extra, **kw)
        for _ in range(2):
            tr.train_step(feats, labels, graph_key=0)
        assert _check_stats_before_every_optimizer(recorder, tr._step_dev, 1.0) == 2
        assert int(tr._step_dev[0]) == 2


def test_trainer_input_checks(recorder, monkeypatch):
    from egot2_b200 import trainer as T
    with pytest.raises(ValueError):
        _hhi_trainer(param_stats=5)
    tr, _, _ = _hhi_trainer()
    for f in (lambda: tr.grad_norms(), lambda: tr.histograms(), lambda: tr.param_stats_step):
        with pytest.raises(ValueError, match="param_stats"):
            f()
    tr, _, _ = _hhi_trainer(param_stats=ParamStats(1, histograms=False))
    with pytest.raises(ValueError, match="histograms"):
        tr.histograms()
    assert set(tr.grad_norms()) == set(tr.engine.arena.shapes) | {"total"}
    assert int(tr.param_stats_step) == 0
    tr, _, _ = _hhi_trainer(param_stats=ParamStats(1), param_groups=GROUPS)
    frozen = {n for n in tr.engine.arena.shapes if n.startswith("transformer_encoder.layers.0.")}
    assert frozen and not frozen & set(tr.grad_norms())
    assert tr.histograms() == (0, [])
    monkeypatch.setattr(T, "_make_peer_exchange", lambda engine, pg, world: object())
    with pytest.raises(ValueError, match="EGOT2_DP_FUSED=0"):
        _hhi_trainer(param_stats=ParamStats(1))
    _hhi_trainer()


def test_optimizer_state_is_unchanged(recorder):
    tr, feats, labels = _hhi_trainer(param_stats=ParamStats(1))
    tr.train_step(feats, labels, graph_key=0)
    ref, _, _ = _hhi_trainer()
    ref.train_step(feats, labels, graph_key=0)
    a, b = tr.optimizer_state_dict(), ref.optimizer_state_dict()
    assert a.keys() == b.keys() and a["step"] == b["step"]


# ------------------------------------------------------------------------------------------------ GPU: the kernel
class _Kernel:
    """egot2_param_stats over an arena, with every buffer it needs."""

    def __init__(self, arena, every=1, histograms=True, has_grad=None):
        from egot2_b200 import stats as S
        self.arena, self.names = arena, list(arena.shapes)
        self.P = len(self.names)
        self.has_grad = [True] * self.P if has_grad is None else has_grad
        params, units = plan_units(arena.shapes, arena.offsets, self.has_grad)
        self.params = torch.frombuffer(bytearray(bytes(params)), dtype=torch.uint8).cuda()
        self.units = torch.frombuffer(bytearray(bytes(units)), dtype=torch.uint8).cuda()
        self.U = len(units)
        self.out = torch.zeros(S.buffer_bytes(self.P, histograms), dtype=torch.uint8, device="cuda")
        self.out[:C.sizeof(L.ParamStatsDesc)].copy_(torch.frombuffer(bytearray(S.pack_desc(ParamStats(every, histograms),
                                                                                               self.P)), dtype=torch.uint8))
        self.edges = torch.from_numpy(default_edges()).cuda() if histograms else None
        self.ws = torch.zeros(int(L.load().egot2_param_stats_workspace_bytes(self.P, self.U)), dtype=torch.uint8,
                              device="cuda")
        self.hist = histograms

    def __call__(self, grad, param, scale, step):
        from egot2_b200 import stats as S
        base = self.out.data_ptr()
        rec = base + S.stats_offset()
        L.call("egot2_param_stats", grad.data_ptr(), param.data_ptr(), float(scale), step.data_ptr(), base,
               self.params.data_ptr(), self.P, self.units.data_ptr(), self.U,
               self.edges.data_ptr() if self.hist else None, rec,
               rec + 2 * self.P * C.sizeof(L.ParamStat) if self.hist else None, self.ws.data_ptr(), self.ws.numel(),
               torch.cuda.current_stream().cuda_stream)

    def read(self):
        from egot2_b200 import stats as S
        host = self.out.cpu().numpy().tobytes()
        d, recs = S.read_stats(host, self.P)
        counts = None
        if self.hist:
            c0 = S.stats_offset() + 2 * self.P * C.sizeof(L.ParamStat)
            counts = np.frombuffer(host[c0:], dtype=np.int32).reshape(2, self.P, L.STATS_BUCKETS)
        return d, recs, counts


def _adversarial(n, seed):
    """Magnitudes log-uniform in [1e-14, 1e22] with random signs, exact +-0 and the fp32 neighbours of bucket edges."""
    g = torch.Generator().manual_seed(seed)
    x = torch.pow(10.0, torch.rand(n, generator=g, dtype=torch.float64) * 36 - 14)
    x = (x * (torch.randint(0, 2, (n,), generator=g) * 2 - 1)).float()
    e = torch.from_numpy(default_edges()).float()
    near = torch.cat([e, torch.nextafter(e, torch.tensor(np.inf)), torch.nextafter(e, torch.tensor(-np.inf)),
                      torch.tensor([0.0, -0.0])])
    idx = torch.randint(0, n, (min(n // 8, near.numel()),), generator=g)
    x[idx] = near[torch.randint(0, near.numel(), (idx.numel(),), generator=g)]
    return x


def _check_pair(rec, counts, vals, edges):
    """One (array, parameter) record + counts against numpy on the fp32 values `vals` (CPU tensor)."""
    v = vals.double().numpy()
    fin = v[np.isfinite(v)]
    assert rec.num == v.size and rec.nonfinite == v.size - fin.size
    if fin.size:
        assert rec.min == fin.min() and rec.max == fin.max()
        assert abs(rec.sum - fin.sum()) <= 1e-12 * np.abs(fin).sum()
        assert abs(rec.sum_squares - fin.dot(fin)) <= 1e-12 * fin.dot(fin)
    want_counts, _ = np.histogram(fin, bins=edges)
    assert np.array_equal(counts, want_counts)
    ref = float(torch.linalg.vector_norm(vals.double()))
    if np.isnan(ref):
        assert np.isnan(rec.norm)
    else:
        assert rec.norm == np.float32(ref) or abs(rec.norm - ref) <= 2 ** -23 * ref


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [1.0, 0.5, 1.0 / 3.0])
@pytest.mark.parametrize("kind", ["hhi", "pnr", "lta"])
def test_kernel_matches_numpy(kind, scale):
    """Every (array, parameter): counts over the default edges equal np.histogram's, trimmed limits and counts equal
    make_histogram's, min / max / num exact, sums to 1e-12, norms to fp32 rounding; two runs are bit-identical; a step that is
    not due leaves every output untouched."""
    from torch.utils.tensorboard.summary import make_histogram
    arena = _arena(kind)
    k = _Kernel(arena, every=2)
    n = arena.numel
    grad, param = _adversarial(n, 1).cuda(), _adversarial(n, 2).cuda()
    step = torch.tensor([3], dtype=torch.int32, device="cuda")
    k(grad, param, scale, step)
    d, recs, counts = k.read()
    assert d.step == 3 and d.every == 2
    first = k.out.clone()
    g32 = (grad * np.float32(scale)).cpu()
    p32 = param.cpu()
    edges = default_edges()
    tot = 0.0
    for p, name in enumerate(k.names):
        o, m = arena.offsets[name], arena.view(name).numel()
        for a, src in ((0, g32), (1, p32)):
            vals = src[o:o + m]
            _check_pair(recs[a * k.P + p], counts[a, p], vals, edges)
            if kind == "hhi" or p % 10 == 0:
                h = histogram_raw(recs[a * k.P + p], counts[a, p], edges)
                ref = make_histogram(vals.double().numpy(), edges.tolist())
                assert h["bucket_limits"] == list(ref.bucket_limit) and h["bucket_counts"] == list(ref.bucket)
                assert h["min"] == ref.min and h["max"] == ref.max and h["num"] == ref.num
        tot += recs[p].sum_squares
    assert abs(d.grad_norm - np.sqrt(tot)) <= 2 ** -23 * np.sqrt(tot)
    k(grad, param, scale, step)                       # bit-identical repeat (the workspace reset itself)
    assert torch.equal(k.out, first)
    step.fill_(4)                                     # (4 - 1) % 2 != 0: not due
    grad.fill_(1.0)
    k(grad, param, scale, step)
    assert torch.equal(k.out, first)


@pytest.mark.gpu
@pytest.mark.parametrize("value", [float("nan"), float("inf"), -float("inf")])
def test_non_finite_elements(value):
    """NaN / +-inf at the first, a middle and the last element of a parameter and across the boundary of two stacked LTA
    head biases: exact non-finite counts, finite statistics as without them, norms NaN / inf as torch's."""
    arena = _arena("lta")
    k = _Kernel(arena)
    n = arena.numel
    grad = torch.randn(n, device="cuda")
    param = torch.randn(n, device="cuda")
    step = torch.ones(1, dtype=torch.int32, device="cuda")
    name = "head.projections.0.weight" if "head.projections.0.weight" in arena.shapes else k.names[-3]
    o, m = arena.offsets[name], arena.view(name).numel()
    b0, b1 = arena.head_b_names[0], arena.head_b_names[1]
    hit = [o, o + m // 2, o + m - 1, arena.offsets[b0] + arena.view(b0).numel() - 1, arena.offsets[b1]]
    assert (hit[3] + 1) // 64 == hit[4] // 64 or hit[3] + 1 == hit[4]
    for arr in (grad, param):
        arr[hit] = value
    k(grad, param, 1.0, step)
    d, recs, counts = k.read()
    edges = default_edges()
    for p, nm in enumerate(k.names):
        oo, mm = arena.offsets[nm], arena.view(nm).numel()
        for a, src in ((0, grad.cpu()), (1, param.cpu())):
            _check_pair(recs[a * k.P + p], counts[a, p], src[oo:oo + mm], edges)
    want = {name: 3, b0: 1, b1: 1}
    for p, nm in enumerate(k.names):
        assert recs[p].nonfinite == recs[k.P + p].nonfinite == want.get(nm, 0)
    assert np.isnan(d.grad_norm) if value != value else np.isinf(d.grad_norm)


@pytest.mark.gpu
def test_frozen_parameters_have_no_gradient_statistics():
    arena = _arena("hhi")
    has_grad = [i % 2 == 0 for i in range(len(arena.shapes))]
    k = _Kernel(arena, has_grad=has_grad)
    grad, param = torch.randn(arena.numel, device="cuda"), torch.randn(arena.numel, device="cuda")
    k(grad, param, 1.0, torch.ones(1, dtype=torch.int32, device="cuda"))
    d, recs, counts = k.read()
    tot = 0.0
    for p, nm in enumerate(k.names):
        o, m = arena.offsets[nm], arena.view(nm).numel()
        assert recs[k.P + p].num == m
        if has_grad[p]:
            tot += float(grad[o:o + m].double().pow(2).sum())
            assert recs[p].num == m
        else:
            assert recs[p].num == 0 and counts[0, p].sum() == 0
    assert abs(d.grad_norm - np.sqrt(tot)) <= 1e-6 * np.sqrt(tot)


# ------------------------------------------------------------------------------------------------ GPU: trainers
def _capture_optimizer_inputs(eng, store, method="adam_step"):
    """Wrap engine.adam_step / sgd_step: clone fp32(grad * grad_scale) and the parameters before the original runs."""
    real = getattr(eng, method)

    def wrapped(*a, grad_scale=1.0, **k):
        store.append(((eng.arena.grad * np.float32(grad_scale)).cpu(), eng.arena.param.cpu()))
        return real(*a, grad_scale=grad_scale, **k)
    setattr(eng, method, wrapped)


def _check_trainer_stats(tr, grad, param):
    """histograms() / grad_norms() of a trainer against the arrays its optimizer received."""
    from torch.utils.tensorboard.summary import make_histogram
    arena = tr.engine.arena
    step, hists = tr.histograms()
    hists = dict(hists)
    edges = default_edges().tolist()
    norms = tr.grad_norms()
    tot = 0.0
    for nm in arena.shapes:
        o, m = arena.offsets[nm], arena.view(nm).numel()
        for tag, src in ((nm, param), (nm + ".grad", grad)):
            if tag not in hists:
                assert tag.endswith(".grad") and nm not in norms
                continue
            ref = make_histogram(src[o:o + m].double().numpy(), edges)
            h = hists[tag]
            assert h["bucket_limits"] == list(ref.bucket_limit) and h["bucket_counts"] == list(ref.bucket), tag
            assert h["min"] == ref.min and h["max"] == ref.max and h["num"] == ref.num
            assert abs(h["sum_squares"] - ref.sum_squares) <= 1e-12 * ref.sum_squares
        if nm in norms:
            ref = float(torch.linalg.vector_norm(grad[o:o + m].double()))
            assert abs(float(norms[nm]) - ref) <= 2 ** -23 * ref
            tot += ref * ref
    assert abs(float(norms["total"]) - np.sqrt(tot)) <= 1e-6 * np.sqrt(tot)
    return step


@pytest.mark.gpu
@pytest.mark.parametrize("sgd", [False, True])
def test_trainer_stats_are_those_of_the_optimizer_inputs(sgd, monkeypatch):
    """every=3 over 7 steps.  Whole-step graph: stamps 1, 1, 1, 4, 4, 4, 7.  With EGOT2_GRAPH_UPDATE=0 (eager optimizer after
    the replay) the statistics equal those of the arrays the optimizer received on the due steps."""
    from egot2_b200.optim import SGD
    spec, feats, labels = _hhi_setup()
    kw = dict(optimizer=SGD(momentum=0.9)) if sgd else {}
    tr = _hhi_trainer_gpu(spec, use_graphs=True, param_stats=ParamStats(3), **kw)
    assert tr.graph_update
    stamps = []
    for _ in range(7):
        tr.train_step(feats, labels, graph_key=0)
        stamps.append(int(tr.param_stats_step))
    assert stamps == [1, 1, 1, 4, 4, 4, 7]
    monkeypatch.setenv("EGOT2_GRAPH_UPDATE", "0")
    tr = _hhi_trainer_gpu(spec, use_graphs=True, param_stats=ParamStats(3), **kw)
    assert not tr.graph_update
    seen = []
    _capture_optimizer_inputs(tr.engine, seen, "sgd_step" if sgd else "adam_step")
    for t in range(1, 8):
        tr.train_step(feats, labels, graph_key=0)
        if (t - 1) % 3 == 0:
            assert _check_trainer_stats(tr, *seen[-1]) == t


@pytest.mark.gpu
def test_guard_skip_records_and_the_retry_overwrites():
    from test_grad_guard import _nan_feature
    spec, feats, labels = _hhi_setup()
    tr = _hhi_trainer_gpu(spec, use_graphs=True, max_grad_norm=1.0, param_stats=ParamStats(1))
    tr.train_step(feats, labels, graph_key=0)
    n = tr.grad_norms()
    assert abs(float(n["total"]) - float(tr.last_grad_norm)) <= 1e-6 * float(tr.last_grad_norm)
    with _nan_feature(feats):
        tr.train_step(feats, labels, graph_key=0)
    torch.cuda.synchronize()
    assert int(tr.skipped_steps) == 1 and int(tr.param_stats_step) == 2 and int(tr._step_dev) == 1
    step, recs = _records(tr)
    P = len(tr._stats["names"])
    assert sum(recs[p].nonfinite for p in range(P)) > 0 and all(recs[P + p].nonfinite == 0 for p in range(P))
    tr.train_step(feats, labels, graph_key=0)
    step, recs = _records(tr)
    assert step == 2 and int(tr._step_dev) == 2 and all(recs[p].nonfinite == 0 for p in range(2 * P))
    assert abs(float(tr.grad_norms()["total"]) - float(tr.last_grad_norm)) <= 1e-6 * float(tr.last_grad_norm)


def _records(tr):
    from egot2_b200 import stats as S
    d, recs = S.read_stats(tr._stats["out"].cpu().numpy().tobytes(), len(tr._stats["names"]))
    return d.step, recs


@pytest.mark.gpu
def test_frozen_groups_in_the_trainer(monkeypatch):
    monkeypatch.setenv("EGOT2_GRAPH_UPDATE", "0")
    spec, feats, labels = _hhi_setup()
    tr = _hhi_trainer_gpu(spec, use_graphs=True, param_groups=GROUPS, param_stats=ParamStats(2))
    seen = []
    _capture_optimizer_inputs(tr.engine, seen)
    for _ in range(3):
        tr.train_step(feats, labels, graph_key=0)
    frozen = [n for n in tr.engine.arena.shapes if n.startswith("transformer_encoder.layers.0.")]
    tags = dict(tr.histograms()[1])
    assert frozen and all(n in tags and n + ".grad" not in tags for n in frozen)
    assert _check_trainer_stats(tr, *seen[-1]) == 3


@pytest.mark.gpu
@pytest.mark.parametrize("graphs", ["1", "0"])
@pytest.mark.parametrize("kind", ["hhi", "hoi"])
def test_prompt_trainers(kind, graphs, monkeypatch):
    from egot2_b200 import synth, trainer as T
    monkeypatch.setenv("EGOT2_G_GRAPH", graphs)
    feats, labels = _prompt_batch(kind)
    feats, labels = [f.cuda() for f in feats], labels.cuda()
    cls = T.HoiPromptTranslatorTrainer if kind == "hoi" else T.PromptTranslatorTrainer
    extra = dict(vocab=40) if kind == "hoi" else {}
    tr = cls(hidden=128, heads=4, layers=1, device="cuda:0", dtype="bf16", param_stats=ParamStats(2), **extra)
    tr.load_state_dict(synth.make_state_dict(tr.spec, 3))
    seen = []
    _capture_optimizer_inputs(tr.engine, seen)
    for _ in range(3):
        tr.train_step(feats, labels, graph_key=0)
    assert len(seen) == 3 and _check_trainer_stats(tr, *seen[-1]) == 3


@pytest.mark.gpu
def test_tensorboard_end_to_end(tmp_path, monkeypatch):
    """add_histogram_raw(**h) and add_histogram(tag, tensor) of the same step read back as equal HistogramProtos."""
    from tensorboard.backend.event_processing.event_file_loader import EventFileLoader
    from torch.utils.tensorboard import SummaryWriter
    monkeypatch.setenv("EGOT2_GRAPH_UPDATE", "0")
    spec, feats, labels = _hhi_setup()
    tr = _hhi_trainer_gpu(spec, use_graphs=True, param_stats=ParamStats(1))
    seen = []
    _capture_optimizer_inputs(tr.engine, seen)
    tr.train_step(feats, labels, graph_key=0)
    step, hists = tr.histograms()
    grad, param = seen[-1]
    arena = tr.engine.arena
    dirs = [str(tmp_path / "raw"), str(tmp_path / "ref")]
    w_raw, w_ref = SummaryWriter(dirs[0]), SummaryWriter(dirs[1])
    for tag, h in hists:
        nm = tag[:-5] if tag.endswith(".grad") else tag
        src = grad if tag.endswith(".grad") else param
        w_raw.add_histogram_raw(tag, global_step=step - 1, **h)
        w_ref.add_histogram(tag, arena.view(nm, src), global_step=step - 1)
    w_raw.close()
    w_ref.close()

    def load(d):
        out = {}
        for f in os.listdir(d):
            for ev in EventFileLoader(os.path.join(d, f)).Load():
                for v in ev.summary.value:
                    out[(v.tag, ev.step)] = v.histo
        return out
    a, b = load(dirs[0]), load(dirs[1])
    assert a.keys() == b.keys() and len(a) == len(hists) > 0
    for key in a:
        x, y = a[key], b[key]
        assert list(x.bucket_limit) == list(y.bucket_limit) and list(x.bucket) == list(y.bucket), key
        assert x.min == y.min and x.max == y.max and x.num == y.num


@pytest.mark.gpu
def test_training_is_not_perturbed():
    spec, feats, labels = _hhi_setup()
    runs = []
    for ps in (None, ParamStats(1)):
        tr = _hhi_trainer_gpu(spec, use_graphs=True, param_stats=ps)
        p0 = tr.engine.arena.param.clone()
        for _ in range(8):
            tr.train_step(feats, labels, graph_key=0)
        torch.cuda.synchronize()
        runs.append(tr.engine.arena.param.clone())
    assert float((runs[0] - runs[1]).norm()) <= 2e-2 * float((runs[0] - p0).norm())


# ------------------------------------------------------------------------------------------------ GPU: two ranks
def _rank_worker(rank, world, port, q):
    os.environ["EGOT2_DP_FUSED"] = "0"
    os.environ["EGOT2_GRAPH_UPDATE"] = "0"
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
        tr = TranslatorTrainer(sp, f"cuda:{rank}", "bf16", use_graphs=True, param_stats=ParamStats(1))
        assert tr.peer is None
        tr.load_state_dict(synth.make_state_dict(sp, 9))
        seen = []
        _capture_optimizer_inputs(tr.engine, seen)
        feats = [f[s.name][lo:hi].cuda() for s in sp.segments]
        labels = lab[lo:hi].cuda()
        for _ in range(2):
            tr.train_step(feats, labels, graph_key=0)
        step = _check_trainer_stats(tr, *seen[-1])
        q.put((rank, dict(step=step, out=tr._stats["out"].cpu())))
        dist.barrier()
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_two_rank_nccl_stats_are_identical():
    """Two ranks on the NCCL all-reduce path: every rank records the statistics of the rank-mean gradient, bit-identically."""
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
    assert got[0]["step"] == got[1]["step"] == 2
    assert torch.equal(got[0]["out"], got[1]["out"])
