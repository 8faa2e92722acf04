"""On-device PNR / OSCC metrics (egot2_b200/metrics.py -> egot2_pnr_metrics) against the CPU restatement, and the
restatement against the reference's own functions (HOI/evaluation/pnr/metrics.py) where oracle/ref_shims finds them."""
import importlib

import pytest
import torch

from oracle import metrics_oracle as MO


def _inputs(B, seed, ties=False):
    g = torch.Generator().manual_seed(seed)
    preds = torch.randn(B, 16, generator=g)
    if ties:
        preds = torch.round(preds)                       # repeated maxima: first-index tie-break must match torch.argmax
    key = torch.randint(0, 16, (B,), generator=g)
    labels = torch.nn.functional.one_hot(key, 16).float()
    sc = torch.randint(0, 2, (B,), generator=g)
    fps = torch.tensor([30.0, 29.97, 24.0, 59.94])[torch.randint(0, 4, (B,), generator=g)].double()
    start = torch.randint(0, 5000, (B,), generator=g)
    end = start + torch.randint(16, 400, (B,), generator=g)
    pnr = start + torch.randint(0, 400, (B,), generator=g)
    info = {"clip_start_frame": start, "clip_end_frame": end, "pnr_frame": pnr}
    oscc_pred = torch.randn(B, 2, generator=g)
    oscc_lab = torch.randint(0, 2, (B,), generator=g)
    return preds, labels, sc, fps, info, oscc_pred, oscc_lab


@pytest.mark.requires_reference
@pytest.mark.parametrize("B,seed,ties", [(1, 0, False), (37, 1, False), (256, 2, True)])
def test_oracle_matches_reference_metrics(B, seed, ties):
    import sys
    import types
    for name in ("torchmetrics", "editdistance"):               # imported further down the reference file, unused here
        if name not in sys.modules:
            try:
                importlib.import_module(name)
            except Exception:
                stub = types.ModuleType(name)
                stub.Metric = object
                sys.modules[name] = stub
    from oracle import ref_shims
    ref = ref_shims._load_file("ref_pnr_metrics", "HOI/evaluation/pnr/metrics.py")
    preds, labels, sc, fps, info, op, ol = _inputs(B, seed, ties)
    assert MO.state_change_accuracy(op, ol) == ref.state_change_accuracy(op, ol)
    assert MO.keyframe_accuracy(preds, labels, sc) == ref.keyframe_accuracy(preds, labels, sc)
    for kw in (dict(), dict(sum=True)):
        a, b = MO.keyframe_distance(preds, labels, sc, fps, info, **kw), ref.keyframe_distance(preds, labels, sc, fps, info, **kw)
        assert abs(a - float(b)) <= 1e-12 * max(1.0, abs(a))
    none_sc = torch.zeros(B, dtype=torch.int64)
    assert MO.keyframe_distance(preds, labels, none_sc, fps, info, evaluate_trained=True) is None
    assert ref.keyframe_distance(preds, labels, none_sc, fps, info, evaluate_trained=True) is None


@pytest.mark.gpu
@pytest.mark.parametrize("B,seed,ties", [(1, 0, False), (37, 1, False), (256, 2, True), (3000, 3, True)])
def test_device_metrics_match_oracle(B, seed, ties):
    from egot2_b200 import metrics as M
    preds, labels, sc, fps, info, op, ol = _inputs(B, seed, ties)
    dev = torch.device("cuda:0")
    cu = lambda t: t.to(dev)
    cinfo = {k: cu(v) for k, v in info.items()}
    assert M.state_change_accuracy(cu(op), cu(ol)) == MO.state_change_accuracy(op, ol)
    assert M.keyframe_accuracy(cu(preds), cu(labels), cu(sc)) == MO.keyframe_accuracy(preds, labels, sc)
    for kw in (dict(), dict(sum=True)):
        a = M.keyframe_distance(cu(preds), cu(labels), cu(sc), cu(fps), cinfo, **kw)
        b = MO.keyframe_distance(preds, labels, sc, fps, info, **kw)
        assert abs(a - b) <= 1e-9 * max(1.0, abs(b))
    none_sc = torch.zeros(B, dtype=torch.int64)
    assert M.keyframe_distance(cu(preds), cu(labels), cu(none_sc), cu(fps), cinfo, evaluate_trained=True) is None
    assert M.keyframe_distance(cu(preds), cu(labels), cu(none_sc), cu(fps), cinfo) == 0.0
    # list-of-tensors inputs like the reference call sites (preds / labels / sc_labels zipped per clip)
    assert M.keyframe_accuracy(list(cu(preds)), list(cu(labels)), list(cu(sc))) == MO.keyframe_accuracy(preds, labels, sc)


def test_metrics_refuse_cpu_tensors():
    from egot2_b200 import _lib as L, metrics as M
    with pytest.raises(L.Egot2Error):
        M.state_change_accuracy(torch.zeros(2, 2), torch.zeros(2, dtype=torch.int64))
