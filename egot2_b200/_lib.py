"""ctypes binding of libegot2.so (the C ABI declared in include/egot2.h).

There is deliberately NO fallback: if the CUDA library is missing or fails to load, importing
the ops raises — the product path never routes through PyTorch eager or the CPU oracle.
"""
from __future__ import annotations

import ctypes as C
import os

MAX_SEG = 8
MAX_GROUPS = 4
F32, BF16 = 0, 1
LOSS_NONE, LOSS_CE, LOSS_BCE_SIGMOID, LOSS_CE_GROUPS = 0, 1, 2, 3
LR_CONSTANT, LR_COSINE, LR_STEPS = 0, 1, 2
LR_MAX_MILESTONES = 8
AVG_EMA, AVG_SWA = 0, 1

# EGOT2_LIB: an alternative build of the same library (instrumented / experimental variants for tools/); never a fallback
_LIB_PATH = os.environ.get("EGOT2_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libegot2.so")

i32, u64, f32, vp, sz = C.c_int32, C.c_uint64, C.c_float, C.c_void_p, C.c_size_t


class EmbedDesc(C.Structure):
    _fields_ = [("dtype", i32), ("feat_dtype", i32), ("B", i32), ("T", i32), ("H", i32), ("n_seg", i32),
                ("seg_tokens", i32 * MAX_SEG), ("seg_in_dim", i32 * MAX_SEG), ("seg_offset", i32 * MAX_SEG),
                ("seg_has_proj", i32 * MAX_SEG), ("training", i32), ("p_feat", f32), ("p_embed", f32),
                ("ln_eps", f32), ("seed", u64), ("no_ln", i32), ("feat_drop_tokens", i32)]


class EmbedIn(C.Structure):
    _fields_ = [("feat", vp * MAX_SEG), ("proj_w", vp * MAX_SEG), ("proj_b", vp * MAX_SEG), ("ln_g", vp),
                ("ln_b", vp), ("tok_table", vp)]


class EmbedOut(C.Structure):
    _fields_ = [("z", vp), ("stat", vp), ("x", vp)]


class EmbedGrads(C.Structure):
    _fields_ = [("proj_w", vp * MAX_SEG), ("proj_b", vp * MAX_SEG), ("ln_g", vp), ("ln_b", vp), ("tok_table", vp),
                ("dfeat", vp * MAX_SEG), ("seg_embed", vp * MAX_SEG)]


class LayerDesc(C.Structure):
    _fields_ = [("dtype", i32), ("B", i32), ("T", i32), ("H", i32), ("FF", i32), ("heads", i32), ("training", i32),
                ("layer_index", i32), ("p_drop", f32), ("ln_eps", f32), ("seed", u64)]


_LAYER_FIELDS = ["in_proj_w", "out_proj_w", "lin1_w", "lin2_w", "in_proj_b", "out_proj_b", "lin1_b", "lin2_b",
                 "norm1_g", "norm1_b", "norm2_g", "norm2_b"]


class LayerParams(C.Structure):
    _fields_ = [(n, vp) for n in _LAYER_FIELDS]


class LayerGrads(C.Structure):
    _fields_ = [(n, vp) for n in _LAYER_FIELDS]


class LayerSaved(C.Structure):
    _fields_ = [(n, vp) for n in ["qkv", "attn", "lse", "y1", "stat1", "x1", "hid", "y2", "stat2", "hid_mask", "ffn_scratch"]]


class DecoderDesc(C.Structure):
    _fields_ = [("dtype", i32), ("rows", i32), ("S", i32), ("mem_rows", i32), ("M", i32), ("kv_inner", i32),
                ("kv_outer", i32), ("kv_jstride", i32), ("kv_istride", i32), ("H", i32), ("FF", i32), ("heads", i32),
                ("training", i32), ("layer_index", i32), ("p_drop", f32), ("ln_eps", f32), ("seed", u64)]


_DEC_FIELDS = ["sa_in_w", "sa_out_w", "ca_in_w", "ca_out_w", "lin1_w", "lin2_w", "sa_in_b", "sa_out_b", "ca_in_b",
               "ca_out_b", "lin1_b", "lin2_b", "norm1_g", "norm1_b", "norm2_g", "norm2_b", "norm3_g", "norm3_b"]


class DecoderParams(C.Structure):
    _fields_ = [(n, vp) for n in _DEC_FIELDS]


class DecoderGrads(C.Structure):
    _fields_ = [(n, vp) for n in _DEC_FIELDS]


class DecoderSaved(C.Structure):
    _fields_ = [(n, vp) for n in ["qkv", "a1", "y1", "stat1", "x1", "qc", "kvc", "a2", "y2", "stat2", "x2", "hid", "y3",
                                  "stat3"]]


class HeadDesc(C.Structure):
    _fields_ = [("dtype", i32), ("B", i32), ("T", i32), ("H", i32), ("pool", i32), ("row_tokens", i32),
                ("use_ln", i32), ("n_out", i32), ("loss", i32), ("n_groups", i32), ("group_size", i32 * MAX_GROUPS),
                ("sub_rows", i32), ("training", i32), ("p_head", f32), ("ln_eps", f32), ("seed", u64)]


class HeadIn(C.Structure):
    _fields_ = [(n, vp) for n in ["x", "ln_g", "ln_b", "w", "b", "labels", "class_weight"]]


class HeadOut(C.Structure):
    _fields_ = [(n, vp) for n in ["pooled", "stat", "g", "logits", "loss", "argmax", "row_loss"]]


class DpDesc(C.Structure):
    _fields_ = [("world", i32), ("rank", i32), ("numel", C.c_int64), ("slab", vp * 8), ("off_param", C.c_int64),
                ("off_grad", C.c_int64), ("off_shadow", C.c_int64), ("off_flags", C.c_int64), ("exp_avg", vp), ("exp_avg_sq", vp),
                ("lr", f32), ("beta1", f32), ("beta2", f32), ("eps", f32), ("weight_decay", f32), ("step", i32), ("step_dev", vp),
                ("decoupled", i32), ("zero_grads_remote", i32), ("lr_dev", vp), ("guard", vp), ("groups", vp),
                ("block_group", vp), ("sgd", i32), ("momentum", f32), ("dampening", f32), ("nesterov", i32)]


class GradGuard(C.Structure):
    _fields_ = [("max_norm", f32), ("total_norm", f32), ("coef", f32), ("skip", i32), ("skipped", i32)]


MAX_PARAM_GROUPS = 8


class ParamGroups(C.Structure):
    _fields_ = [("n_groups", i32), ("lr_mult", f32 * MAX_PARAM_GROUPS), ("weight_decay", f32 * MAX_PARAM_GROUPS),
                ("frozen", i32 * MAX_PARAM_GROUPS)]


STATS_BUCKETS = 1548


class ParamStatsDesc(C.Structure):
    _fields_ = [("every", i32), ("histograms", i32), ("n_params", i32), ("step", i32), ("grad_norm", f32)]


class StatsParam(C.Structure):
    _fields_ = [("offset", C.c_int64), ("numel", C.c_int64), ("has_grad", i32), ("first_unit", i32 * 2), ("n_units", i32 * 2)]


class StatsUnit(C.Structure):
    _fields_ = [("param", i32), ("array", i32), ("begin", C.c_int64), ("end", C.c_int64)]


class ParamStat(C.Structure):
    _fields_ = [("sum", C.c_double), ("sum_squares", C.c_double), ("min", f32), ("max", f32), ("norm", f32),
                ("nonfinite", i32), ("num", C.c_int64)]


class LrSched(C.Structure):
    _fields_ = [("kind", i32), ("n_milestones", i32), ("warmup_steps", C.c_int64), ("total_steps", C.c_int64),
                ("base_lr", C.c_double), ("warmup_start_lr", C.c_double), ("end_lr", C.c_double),
                ("milestones", C.c_int64 * LR_MAX_MILESTONES), ("factors", C.c_double * (LR_MAX_MILESTONES + 1))]


class HeadGrads(C.Structure):
    _fields_ = [(n, vp) for n in ["ln_g", "ln_b", "w", "b"]]


class VitDesc(C.Structure):
    _fields_ = [("dtype", i32), ("B", i32), ("T", i32), ("D", i32), ("heads", i32), ("dim_head", i32), ("mlp", i32),
                ("layer_index", i32), ("ln_eps", f32)]


_VIT_PARAM_FIELDS = ["qkv_w", "out_w", "ff1_w", "ff2_w", "norm_a_g", "norm_a_b", "norm_f_g", "norm_f_b", "ff1_b", "ff2_b"]


class VitParams(C.Structure):
    _fields_ = [(n, vp) for n in _VIT_PARAM_FIELDS]


class VitGrads(C.Structure):
    _fields_ = [(n, vp) for n in _VIT_PARAM_FIELDS]


class VitSaved(C.Structure):
    _fields_ = [(n, vp) for n in ["h", "stat_a", "qkv", "attn", "lse", "x1", "h2", "stat_f", "u", "act"]]


P = C.POINTER

# name -> (restype, argtypes); every symbol declared in include/egot2.h must be listed here
SIGNATURES = {
    "egot2_version": (C.c_char_p, []),
    "egot2_last_error": (C.c_char_p, []),
    "egot2_sm_count": (C.c_int, []),
    "egot2_launch_count": (C.c_uint64, []),
    "egot2_dropout_epoch_enable": (C.c_int, [C.c_int]),
    "egot2_dropout_epoch_set": (C.c_int, [u64, vp]),
    "egot2_dropout_epoch_advance": (C.c_int, [vp]),
    "egot2_dropout_epoch_host": (C.c_int, [u64]),
    "egot2_pnr_metrics": (C.c_int, [i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "egot2_row_softmax": (C.c_int, [C.c_int64, i32, vp, vp, vp]),
    "egot2_segment_softmax_mean": (C.c_int, [i32, i32, vp, vp, vp, vp]),
    "egot2_topk_correct": (C.c_int, [i32, i32, vp, vp, i32, vp, vp, vp]),
    "egot2_edit_distance_prefix": (C.c_int, [i32, i32, i32, vp, vp, vp, vp, vp]),
    "egot2_prof_enable": (C.c_int, [C.c_int]),
    "egot2_peer_alloc": (C.c_int, [C.c_size_t, C.POINTER(vp)]),
    "egot2_peer_free": (C.c_int, [vp]),
    "egot2_peer_handle_bytes": (C.c_int, []),
    "egot2_peer_export": (C.c_int, [vp, vp]),
    "egot2_peer_import": (C.c_int, [vp, C.POINTER(vp)]),
    "egot2_peer_unimport": (C.c_int, [vp]),
    "egot2_dp_flag_bytes": (C.c_size_t, []),
    "egot2_dp_reduce_adam": (C.c_int, [vp, vp]),
    "egot2_dp_reduce_adam_range": (C.c_int, [vp, C.c_int64, C.c_int64, i32, vp]),
    "egot2_side_defer": (C.c_int, [C.c_int]),
    "egot2_side_join_all": (C.c_int, [vp]),
    "egot2_timeline_set": (C.c_int, [vp]),
    "egot2_prof_report": (C.c_int, [C.c_char_p, sz]),
    "egot2_embed_workspace_bytes": (sz, [P(EmbedDesc), C.c_int]),
    "egot2_embed_fwd": (C.c_int, [P(EmbedDesc), P(EmbedIn), P(EmbedOut), vp, sz, vp]),
    "egot2_embed_bwd": (C.c_int, [P(EmbedDesc), P(EmbedIn), P(EmbedOut), vp, P(EmbedGrads), vp, sz, vp]),
    "egot2_hhi_tok_table_fwd": (C.c_int, [vp, vp, i32, i32, P(i32), P(i32), i32, vp, vp]),
    "egot2_hhi_tok_table_bwd": (C.c_int, [vp, i32, P(i32), P(i32), i32, vp, vp]),
    "egot2_ffn_scratch_bytes": (sz, [i32]),
    "egot2_encoder_layer_workspace_bytes": (sz, [P(LayerDesc), C.c_int]),
    "egot2_encoder_layer_fwd": (C.c_int, [P(LayerDesc), P(LayerParams), vp, vp, P(LayerSaved), vp, sz, vp]),
    "egot2_encoder_layer_bwd": (C.c_int, [P(LayerDesc), P(LayerParams), vp, P(LayerSaved), vp, vp, P(LayerGrads),
                                          vp, sz, vp]),
    "egot2_decoder_layer_workspace_bytes": (sz, [P(DecoderDesc)]),
    "egot2_decoder_layer_fwd": (C.c_int, [P(DecoderDesc), P(DecoderParams), vp, vp, vp, P(DecoderSaved), vp]),
    "egot2_decoder_layer_bwd": (C.c_int, [P(DecoderDesc), P(DecoderParams), vp, vp, P(DecoderSaved), vp, vp, vp,
                                          P(DecoderGrads), vp, sz, vp]),
    "egot2_vit_layer_workspace_bytes": (sz, [P(VitDesc)]),
    "egot2_vit_layer_fwd": (C.c_int, [P(VitDesc), P(VitParams), vp, vp, P(VitSaved), vp]),
    "egot2_vit_layer_bwd": (C.c_int, [P(VitDesc), P(VitParams), vp, P(VitSaved), vp, vp, P(VitGrads), vp, sz, vp]),
    "egot2_prompt_embed_fwd": (C.c_int, [i32, i32, i32, i32, vp, vp, vp, f32, i32, u64, vp, vp]),
    "egot2_prompt_embed_bwd": (C.c_int, [i32, i32, i32, i32, vp, vp, f32, i32, u64, vp, vp]),
    "egot2_head_rows": (C.c_int, [P(HeadDesc)]),
    "egot2_head_workspace_bytes": (sz, [P(HeadDesc)]),
    "egot2_head_loss_fwd": (C.c_int, [P(HeadDesc), P(HeadIn), P(HeadOut), vp]),
    "egot2_head_loss_bwd": (C.c_int, [P(HeadDesc), P(HeadIn), P(HeadOut), vp, f32, vp, P(HeadGrads), vp, sz, vp]),
    "egot2_slowfast_pool_fwd": (C.c_int, [vp, i32, i32, i32, i32, i32, i32, vp, i32, vp]),
    "egot2_cast_f32_to_bf16": (C.c_int, [vp, vp, sz, vp]),
    "egot2_sum_into_f32": (C.c_int, [vp, vp, vp, sz, vp]),
    "egot2_cast_bf16_to_f32": (C.c_int, [vp, vp, sz, vp]),
    "egot2_adam_step": (C.c_int, [vp, vp, vp, vp, sz, f32, f32, f32, f32, f32, i32, f32, vp]),
    "egot2_adam_step_fused": (C.c_int, [vp, vp, vp, vp, sz, f32, f32, f32, f32, f32, i32, f32, vp, i32, vp]),
    "egot2_adamw_step_fused": (C.c_int, [vp, vp, vp, vp, sz, f32, f32, f32, f32, f32, i32, f32, vp, i32, vp]),
    "egot2_adam_step_fused_dev": (C.c_int, [vp, vp, vp, vp, sz, f32, f32, f32, f32, f32, vp, f32, vp, i32, vp]),
    "egot2_adam_step_fused_sched": (C.c_int, [vp, vp, vp, vp, sz, vp, f32, f32, f32, f32, vp, f32, vp, i32, i32, vp]),
    "egot2_opt_advance": (C.c_int, [vp, vp, vp, vp]),
    "egot2_grad_norm_workspace_bytes": (sz, []),
    "egot2_grad_norm": (C.c_int, [vp, sz, f32, vp, vp, vp, sz, vp]),
    "egot2_adam_step_fused_guard": (C.c_int, [vp, vp, vp, vp, sz, f32, vp, f32, f32, f32, f32, vp, f32, vp, i32, i32, vp, vp]),
    "egot2_adam_step_fused_groups": (C.c_int, [vp, vp, vp, vp, sz, f32, vp, f32, f32, f32, vp, f32, vp, i32, i32, vp, vp, vp,
                                               vp]),
    "egot2_grad_norm_groups": (C.c_int, [vp, sz, f32, vp, vp, vp, vp, vp, sz, vp]),
    "egot2_sgd_step_fused": (C.c_int, [vp, vp, vp, sz, f32, vp, f32, f32, i32, f32, i32, vp, f32, vp, i32, vp, vp, vp, vp]),
    "egot2_param_stats_workspace_bytes": (sz, [i32, i32]),
    "egot2_param_stats": (C.c_int, [vp, vp, f32, vp, vp, vp, i32, vp, i32, vp, vp, vp, vp, sz, vp]),
    "egot2_weight_avg_update": (C.c_int, [vp, vp, sz, i32, f32, i32, i32, vp, vp, vp]),
    "egot2_gemm": (C.c_int, [i32, i32, i32, i32, vp, i32, vp, i32, vp, i32, vp, i32, i32, vp]),
    "egot2_gemm_last_impl": (C.c_char_p, []),
    "egot2_layernorm_fwd": (C.c_int, [i32, i32, i32, vp, vp, vp, f32, vp, vp, vp]),
    "egot2_attention_fwd": (C.c_int, [i32, i32, i32, i32, i32, vp, vp, vp, f32, i32, u64, vp]),
    "egot2_attention_bwd": (C.c_int, [i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, f32, i32, u64, vp, sz, vp]),
    "egot2_attention_bwd_workspace_bytes": (sz, [i32, i32, i32, i32, i32]),
    "egot2_pool_fwd": (C.c_int, [i32, i32, i32, i32, i32, i32, vp, vp, vp]),
    "egot2_pool_bwd": (C.c_int, [i32, i32, i32, i32, i32, i32, vp, vp, vp]),
}

_lib = None


class Egot2Error(RuntimeError):
    pass


def lib_path() -> str:
    return _LIB_PATH


def load():
    """Load libegot2.so (once).  Raises if it has not been built — there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise Egot2Error(f"{_LIB_PATH} not found: build it with `python -m egot2_b200.build` "
                         "(the CUDA library is mandatory; there is no PyTorch/CPU fallback)")
    lib = C.CDLL(_LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError if a declared symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().egot2_last_error().decode(errors="replace")
        raise Egot2Error(f"{what or 'egot2 call'} failed (rc={rc}): {msg}")


def call(name: str, *args):
    """Call an int-returning entry point and raise Egot2Error on failure."""
    check(getattr(load(), name)(*args), name)


def prof_enable(on: bool = True):
    check(load().egot2_prof_enable(1 if on else 0), "egot2_prof_enable")


def prof_report():
    """[(launcher tag, launches, total_us)] recorded since prof_enable(True), sorted by total time."""
    buf = C.create_string_buffer(1 << 20)
    check(load().egot2_prof_report(buf, len(buf)), "egot2_prof_report")
    rows = []
    for line in buf.value.decode().splitlines():
        tag, n, us = line.split("\t")
        rows.append((tag, int(n), float(us)))
    return sorted(rows, key=lambda r: -r[2])
