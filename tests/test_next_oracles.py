"""Oracles of SURVEY.md §8(f) rows that have no CUDA path yet (oracle/next_rows.py): the HOI EgoT2-g restatement against its
committed golden (made from the real reference class), and live against the reference classes where oracle/ref_shims finds them."""
import numpy as np
import pytest
import torch

from oracle import next_rows as NR
from oracle import translator_oracle as O
from oracle.cases import grad_digest


def test_hoi_g_oracle_matches_golden():
    gold = np.load(NR.GOLDEN)
    sd, feats, target = NR.inputs()
    P = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    out, loss = NR.oracle_outputs(P, feats, target)
    ref = torch.from_numpy(gold["output"])
    assert out.shape == ref.shape == (NR.B, NR.VOCAB, 2)
    assert float((out.detach() - ref).abs().max()) <= 2e-5 + 1e-4 * float(ref.abs().max())
    assert abs(float(loss) - float(gold["loss"])) <= 1e-4 * abs(float(gold["loss"]))
    names = [k[len("grad/"):] for k in gold.files if k.startswith("grad/")]
    grads = torch.autograd.grad(loss, [P[k] for k in names], allow_unused=True)
    for k, g in zip(names, grads):
        d = grad_digest(g if g is not None else torch.zeros_like(P[k]))
        r = torch.from_numpy(gold["grad/" + k])
        assert float((d - r).abs().max()) <= 2e-4 * (float(r.abs().max()) + 1e-6) + 1e-6, k
    toks = O.hoi_g_predict_ac(sd, feats["pnr"], feats["oscc"], feats["slow"], feats["fast"], 4, NR.HEADS)
    assert torch.equal(toks, torch.from_numpy(gold["predict_ac"]))


def test_hoi_g_action_task_shares_one_position_run():
    """The action task's 16 tokens (slow8 | fast8) carry positions 0..15, not 0..7 twice (encode_prepare is applied to the
    concatenated action features): permuting which half is 'slow' must change the memory."""
    sd, feats, _ = NR.inputs()
    mem = O.hoi_g_encode(sd, feats["pnr"], feats["oscc"], feats["slow"], feats["fast"], NR.HEADS)
    assert mem.shape == (NR.B, 48, NR.H)
    H = NR.H
    pe = O.sinusoid_table(16, H)
    x = O.layer_norm(torch.cat([O.linear(feats["slow"], sd["proj_action_slow.weight"], sd["proj_action_slow.bias"]),
                                O.linear(feats["fast"], sd["proj_action_fast.weight"], sd["proj_action_fast.bias"])], dim=1),
                     sd["ln.weight"], sd["ln.bias"]) + sd["task_embed"][:, 2, :] + pe
    assert x.shape == (NR.B, 16, H) and not torch.allclose(pe[:8], pe[8:])


@pytest.mark.requires_reference
def test_hoi_g_oracle_matches_reference_live():
    rec = NR.main(write=False)                         # asserts oracle == reference class on the spot
    gold = np.load(NR.GOLDEN)
    assert np.allclose(rec["output"], gold["output"], atol=2e-5, rtol=1e-4)
    assert np.array_equal(rec["predict_ac"], gold["predict_ac"])


@pytest.mark.parametrize("three_task", [False, True])
def test_simple_vit_oracle_matches_golden(three_task):
    """simple_vit siblings (pre-norm, GELU, bias-free qkv/out with dim_head 128 x 8 heads on a 256-wide model): the
    restatement against the golden made from the reference classes (oracle/next_rows.py main_vit)."""
    gold = np.load(NR.GOLDEN_VIT)
    tag = "3task" if three_task else "2task"
    sd, feats, labels = NR.vit_inputs(three_task)
    P = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    out, loss = NR.vit_oracle(P, feats, labels, three_task)
    ref = torch.from_numpy(gold[tag + "/output"])
    assert float((out.detach() - ref).abs().max()) <= 2e-5 + 1e-4 * float(ref.abs().max())
    assert abs(float(loss) - float(gold[tag + "/loss"])) <= 1e-4 * abs(float(gold[tag + "/loss"]))
    names = [k[len(tag + "/grad/"):] for k in gold.files if k.startswith(tag + "/grad/")]
    grads = torch.autograd.grad(loss, [P[k] for k in names])
    for k, g in zip(names, grads):
        d, r = grad_digest(g), torch.from_numpy(gold[tag + "/grad/" + k])
        assert float((d - r).abs().max()) <= 2e-4 * (float(r.abs().max()) + 1e-6) + 1e-6, k
    assert torch.equal(out.argmax(-1), ref.argmax(-1))          # keyframe index


@pytest.mark.requires_reference
def test_simple_vit_oracle_matches_reference_live():
    rec = NR.main_vit(write=False)
    gold = np.load(NR.GOLDEN_VIT)
    for tag in ("2task", "3task"):
        assert np.allclose(rec[tag + "/output"], gold[tag + "/output"], atol=2e-5, rtol=1e-4)
