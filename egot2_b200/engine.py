"""Host-side driver of the translator hot path: parameter arena, activation buffers, and the
sequence of C-ABI stage calls (embed -> L x encoder layer -> head[+loss]) forward and backward.

PyTorch is used here for device memory (caching allocator), streams and views only; every
FLOP on the path is executed by libegot2.so.
"""
from __future__ import annotations

import ctypes as C
import os
import re
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _lib as L
from .specs import TranslatorSpec

_ALIGN = 64  # elements: keeps every tensor 256 B (fp32) / 128 B (bf16) aligned for vector + TMA access


def _dt(dtype: str) -> int:
    return {"fp32": L.F32, "bf16": L.BF16}[dtype]


def _torch_dt(dtype: str) -> torch.dtype:
    return {"fp32": torch.float32, "bf16": torch.bfloat16}[dtype]


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _stream() -> int:
    """Current stream of the CURRENT device: every public engine entry point runs under torch.cuda.device(engine.device)
    (`_on_device`), so this is the engine's device whatever the caller's current device is."""
    return torch.cuda.current_stream().cuda_stream


def _on_device(fn):
    """Run an engine method with the engine's device current: the library's launches, its per-device side streams and
    dropout-epoch slot and torch's current stream then all refer to `self.device`, also for an engine on cuda:1 in a
    process whose current device is cuda:0."""
    import functools

    @functools.wraps(fn)
    def wrapped(self, *a, **k):
        if self.device.type != "cuda":            # CPU only under tests/abi_emulator.py (host-wiring checks)
            return fn(self, *a, **k)
        with torch.cuda.device(self.device):
            return fn(self, *a, **k)
    return wrapped


class ParamArena:
    """All translator parameters in ONE flat fp32 buffer (+ same-layout gradient buffer and bf16
    shadow).  One buffer = one NCCL all-reduce, one Adam launch, one fp32->bf16 cast launch.
    The LTA head's Z independent Linear layers are laid out back to back so that they form one
    (Z*593, H) matrix for a single GEMM."""

    def __init__(self, spec: TranslatorSpec, device: torch.device):
        self.spec = spec
        self.device = torch.device(device)
        shapes = spec.param_shapes()
        self.shapes = shapes
        self.offsets: Dict[str, int] = {}
        off = 0

        def place(name, numel, align=True):
            nonlocal off
            if align:
                off = (off + _ALIGN - 1) // _ALIGN * _ALIGN
            self.offsets[name] = off
            off += numel

        # stacked heads (LTA: head.projections.z ; AR: linear_head1.1 / linear_head2.1): contiguous, no padding between
        head_w = [n for n in shapes if re.fullmatch(r"head\.projections\.\d+\.weight|linear_head\d\.1\.weight", n)]
        head_b = [n for n in shapes if re.fullmatch(r"head\.projections\.\d+\.bias|linear_head\d\.1\.bias", n)]
        # The embedding-stage parameters (per-task projections, task/positional embeddings, the shared LayerNorm) come
        # FIRST and contiguous: their gradients are the last ones backward produces, so under data parallelism the rest
        # of the arena [embed_numel:] can be all-reduced while the embedding backward still runs (trainer.py).
        proj_names = {s.proj for s in spec.segments if s.proj is not None}
        def _is_embed(n):
            return n.rsplit(".", 1)[0] in proj_names or n in ("task_embed", "pe", "ln.weight", "ln.bias")
        for name, shp in shapes.items():
            if _is_embed(name):
                place(name, _numel(shp))
        self.embed_numel = (off + _ALIGN - 1) // _ALIGN * _ALIGN
        off = self.embed_numel
        for name, shp in shapes.items():
            if name in head_w or name in head_b or _is_embed(name):
                continue
            place(name, _numel(shp))
        for i, name in enumerate(head_w):      # contiguous block, no padding between heads
            place(name, _numel(shapes[name]), align=(i == 0))
        for i, name in enumerate(head_b):
            place(name, _numel(shapes[name]), align=(i == 0))
        self.numel = (off + _ALIGN - 1) // _ALIGN * _ALIGN
        self.param = torch.zeros(self.numel, device=self.device, dtype=torch.float32)
        self.grad = torch.zeros(self.numel, device=self.device, dtype=torch.float32)
        self.shadow: Optional[torch.Tensor] = None
        # True while `shadow` is known to equal bf16(param): set by the fused Adam (which writes both), cleared by
        # anything else that may change the parameters.  The drop-in nn.Module path never sets it (a torch optimizer
        # updates the arena views behind our back), so there every forward re-casts.
        self.shadow_fresh = False
        self.head_w_names, self.head_b_names = head_w, head_b

    def rebase(self, param: torch.Tensor, grad: torch.Tensor, shadow: Optional[torch.Tensor]):
        """Move the arena into caller-provided storage (same layout; e.g. an IPC-shared slab, parallel.PeerExchange): the
        current contents are copied over and every later call reads the new buffers.  Only for trainer-owned arenas, before
        any CUDA graph is captured - the drop-in nn.Modules alias their nn.Parameters to the original storage."""
        assert param.numel() == self.numel and grad.numel() == self.numel and param.dtype == grad.dtype == torch.float32
        param.copy_(self.param)
        grad.copy_(self.grad)
        if shadow is not None:
            assert shadow.numel() == self.numel and shadow.dtype == torch.bfloat16
            if self.shadow is not None:
                shadow.copy_(self.shadow)
            else:
                self.shadow_fresh = False
        self.param, self.grad = param, grad
        if shadow is not None:
            self.shadow = shadow

    def view(self, name: str, base: Optional[torch.Tensor] = None) -> torch.Tensor:
        base = self.param if base is None else base
        shp = self.shapes[name]
        o = self.offsets[name]
        return base[o:o + _numel(shp)].view(shp)

    def stacked_head(self, base: Optional[torch.Tensor] = None):
        """(sum of head rows, H) weight and (sum of head rows,) bias views of the stacked heads (LTA / AR)."""
        base = self.param if base is None else base
        w0, b0 = self.head_w_names[0], self.head_b_names[0]
        H = self.shapes[w0][1]
        rows = sum(self.shapes[n][0] for n in self.head_w_names)
        ow, ob = self.offsets[w0], self.offsets[b0]
        return base[ow:ow + rows * H].view(rows, H), base[ob:ob + rows]

    def load_state_dict(self, sd: Dict[str, torch.Tensor], base: Optional[torch.Tensor] = None):
        """base: another buffer of the arena's layout (e.g. Adam moments) to fill instead of the parameters."""
        with torch.no_grad():
            for name in self.shapes:
                self.view(name, base).copy_(sd[name].to(device=self.device, dtype=torch.float32))
        if base is None:
            self.shadow_fresh = False

    def state_dict(self, base: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        return {name: self.view(name, base).clone() for name in self.shapes}

    @_on_device
    def refresh_shadow(self):
        """fp32 -> bf16 shadow of the whole arena (one launch)."""
        if self.shadow is None:
            self.shadow = torch.empty(self.numel, device=self.device, dtype=torch.bfloat16)
            self.shadow_fresh = False
        if self.shadow_fresh:
            return
        L.call("egot2_cast_f32_to_bf16", self.param.data_ptr(), self.shadow.data_ptr(), self.numel, _stream())


def _numel(shp) -> int:
    n = 1
    for d in shp:
        n *= d
    return n


@dataclass
class Activations:
    """Everything one forward leaves behind for its backward (device buffers + the descriptors)."""
    B: int
    seg_tokens: Tuple[int, ...]
    T: int
    training: bool
    seed: int
    feats: List[torch.Tensor] = field(default_factory=list)
    t: Dict[str, torch.Tensor] = field(default_factory=dict)     # named buffers
    embed_desc: Optional[L.EmbedDesc] = None
    embed_in: Optional[L.EmbedIn] = None
    embed_out: Optional[L.EmbedOut] = None
    layer_desc: List[L.LayerDesc] = field(default_factory=list)
    layer_params: List[L.LayerParams] = field(default_factory=list)
    layer_saved: List[L.LayerSaved] = field(default_factory=list)
    head_desc: Optional[L.HeadDesc] = None
    head_in: Optional[L.HeadIn] = None
    head_out: Optional[L.HeadOut] = None
    rows: int = 0
    dec_desc: List[L.DecoderDesc] = field(default_factory=list)
    dec_params: List[L.DecoderParams] = field(default_factory=list)
    dec_saved: List[L.DecoderSaved] = field(default_factory=list)
    prompt: Optional[torch.Tensor] = None


class TranslatorEngine:
    """Runs one translator variant (`spec`) on one GPU in `dtype` ("fp32" parity mode or "bf16")."""

    def __init__(self, spec: TranslatorSpec, device, dtype: str = "fp32", arena: Optional[ParamArena] = None):
        L.load()
        if not torch.cuda.is_available():
            raise L.Egot2Error("egot2_b200 needs a CUDA device (no CPU fallback)")
        self.spec = spec
        self.device = torch.device(device)
        self.dtype = dtype
        self.dt = _dt(dtype)
        self.tdt = _torch_dt(dtype)
        self.arena = arena if arena is not None else ParamArena(spec, self.device)
        self.pe_buffer: Optional[torch.Tensor] = None     # HHI: (max_len, H) sinusoid table (pos_embed.pe)
        self.lossav: Optional[Dict[str, torch.Tensor]] = None
        self._ws: Optional[torch.Tensor] = None
        self._ws_alt: Dict[int, torch.Tensor] = {}
        # measured on B200 (HHI b256, PNR b256, LTA b512): 347.1 vs 345.2, 1064 vs 1050, 1644 vs 1655 us per step with / without
        # deferral - the parameter-gradient backlog is real SM time, not an idle gap, so the default stays "join per layer"
        self.defer_joins = os.environ.get("EGOT2_DEFER_JOIN", "0") == "1"
        self._ws_retired: List[torch.Tensor] = []     # outgrown workspaces: CUDA graphs captured earlier still point into them
        self._persistent: Dict[Tuple, Activations] = {}

    # ------------------------------------------------------------------ helpers
    def _mat(self, name: str) -> torch.Tensor:
        """Matrix parameter in the compute dtype."""
        if self.dtype == "bf16":
            return self.arena.view(name, self.arena.shadow)
        return self.arena.view(name)

    def _vec(self, name: str) -> torch.Tensor:
        return self.arena.view(name)

    def _workspace(self, nbytes: int, slot: int = 0) -> torch.Tensor:
        """slot 0: the shared scratch of every stage; slots 1, 2: the alternate encoder-layer workspace and the embedding
        stage's own one, used by backward() while the side-stream joins are deferred (egot2_side_defer)."""
        if slot:
            cur = self._ws_alt.get(slot)
            if cur is None or cur.numel() < nbytes:
                if cur is not None:
                    self._ws_retired.append(cur)
                cur = torch.empty(int(nbytes), device=self.device, dtype=torch.uint8)
                self._ws_alt[slot] = cur
            return cur
        if self._ws is None or self._ws.numel() < nbytes:
            if self._ws is not None:
                # never hand an outgrown workspace back to the allocator: a graph captured for a smaller batch has its raw
                # pointer baked in and would scribble over whatever reuses the block
                self._ws_retired.append(self._ws)
            self._ws = torch.empty(int(nbytes), device=self.device, dtype=torch.uint8)
        return self._ws

    def set_sinusoid(self, pe: torch.Tensor):
        """pe: the module's registered buffer pos_embed.pe, (max_len, 1, H) or (max_len, H)."""
        self.pe_buffer = pe.reshape(pe.shape[0], -1).to(device=self.device, dtype=torch.float32).contiguous()

    # ------------------------------------------------------------------ forward
    @_on_device
    def forward(self, feats: Sequence[torch.Tensor], training: bool = False, seed: int = 0,
                labels: Optional[torch.Tensor] = None, loss: int = L.LOSS_NONE,
                class_weight: Optional[torch.Tensor] = None, persistent: bool = False,
                prompt: Optional[torch.Tensor] = None) -> Activations:
        sp = self.spec
        assert len(feats) == len(sp.segments), f"expected {len(sp.segments)} feature streams"
        B = int(feats[0].shape[0])
        seg_tokens = tuple(int(f.shape[1]) for f in feats)
        for f, s in zip(feats, sp.segments):
            assert f.shape[0] == B and f.shape[2] == s.in_dim, f"{s.name}: bad feature shape {tuple(f.shape)}"
            assert s.tokens is None or f.shape[1] == s.tokens, f"{s.name}: expected {s.tokens} tokens"
        feat_dt = feats[0].dtype
        if self.dtype == "fp32":
            feats = [f.float().contiguous() for f in feats]
            feat_dt = torch.float32
        else:
            if any(f.dtype != feat_dt for f in feats) or feat_dt not in (torch.float32, torch.bfloat16):
                feats = [f.to(torch.bfloat16) for f in feats]
                feat_dt = torch.bfloat16
            feats = [f.contiguous() for f in feats]
        T = sum(seg_tokens)
        H, FF = sp.hidden, sp.ffn
        M = B * T
        dev, tdt = self.device, self.tdt
        st = _stream()
        if self.dtype == "bf16":
            self.arena.refresh_shadow()

        key = (B, seg_tokens, bool(training), feat_dt, loss, None if prompt is None else tuple(prompt.shape))
        act = self._persistent.get(key) if persistent else None
        fresh = act is None
        if fresh:
            act = Activations(B, seg_tokens, T, bool(training), int(seed))
            if persistent:
                self._persistent[key] = act
        act.seed = int(seed)
        act.feats = list(feats)
        t = act.t

        def buf(name, shape, dtype):
            if name not in t:
                t[name] = torch.empty(shape, device=dev, dtype=dtype)
            return t[name]

        # ---- token table (what is added after the shared LN)
        if sp.embed == "task_sinusoid":
            if self.pe_buffer is None:
                raise L.Egot2Error("HHI translator: call set_sinusoid(pos_embed.pe) first")
            table = buf("tok_table", (T, H), torch.float32)
            runs = sp.table_runs(seg_tokens)          # one position run per segment (HOI EgoT2-g: slow|fast share one)
            segs = (C.c_int32 * len(runs))(*[r[0] for r in runs])
            ids = (C.c_int32 * len(runs))(*[r[1] for r in runs])
            L.call("egot2_hhi_tok_table_fwd", self._vec("task_embed").data_ptr(), self.pe_buffer.data_ptr(),
                   int(self.pe_buffer.shape[0]), len(runs), segs, ids, H, table.data_ptr(), st)
        else:
            table = self._vec("pe").view(T, H)

        # ---- embed
        if fresh or act.embed_desc is None:
            d = L.EmbedDesc()
            d.dtype = self.dt
            d.B, d.T, d.H, d.n_seg = B, T, H, len(seg_tokens)
            off = 0
            for k, (s, dk) in enumerate(zip(sp.segments, seg_tokens)):
                d.seg_tokens[k], d.seg_in_dim[k], d.seg_offset[k] = dk, s.in_dim, off
                d.seg_has_proj[k] = 1 if s.proj is not None else 0
                off += dk
            d.ln_eps = 1e-5
            act.embed_desc = d
            act.embed_in, act.embed_out = L.EmbedIn(), L.EmbedOut()
        d = act.embed_desc
        d.feat_dtype = L.F32 if feat_dt == torch.float32 else L.BF16
        d.training, d.p_feat, d.p_embed, d.seed = int(training), sp.p_feat, sp.p_embed, int(seed)
        ein, eout = act.embed_in, act.embed_out
        for k, s in enumerate(sp.segments):
            ein.feat[k] = feats[k].data_ptr()
            if s.proj is not None:
                ein.proj_w[k] = self._mat(s.proj + ".weight").data_ptr()
                ein.proj_b[k] = self._vec(s.proj + ".bias").data_ptr()
        d.no_ln = 0 if sp.embed_ln else 1
        d.feat_drop_tokens = sp.feat_drop_tokens
        if sp.embed_ln:
            ein.ln_g, ein.ln_b = self._vec("ln.weight").data_ptr(), self._vec("ln.bias").data_ptr()
        ein.tok_table = table.data_ptr()
        eout.z = buf("z", (B, T, H), tdt).data_ptr()
        eout.stat = buf("stat0", (M, 2), torch.float32).data_ptr()
        x = buf("x0", (B, T, H), tdt)
        eout.x = x.data_ptr()
        ws_bytes = L.load().egot2_embed_workspace_bytes(C.byref(d), 0)
        ws = self._workspace(ws_bytes)
        L.call("egot2_embed_fwd", C.byref(d), C.byref(ein), C.byref(eout), ws.data_ptr(), ws.numel(), st)

        # ---- encoder layers
        if sp.encoder == "simple_vit":
            x = self._vit_forward(act, x, buf)
            n_torch_layers = 0
        else:
            n_torch_layers = sp.layers
        if n_torch_layers and (fresh or not act.layer_desc):
            act.layer_desc, act.layer_params, act.layer_saved = [], [], []
            for i in range(sp.layers):
                ld = L.LayerDesc()
                ld.dtype, ld.B, ld.T, ld.H, ld.FF, ld.heads = self.dt, B, T, H, FF, sp.heads
                ld.layer_index, ld.ln_eps = i, 1e-5
                act.layer_desc.append(ld)
                act.layer_params.append(L.LayerParams())
                act.layer_saved.append(L.LayerSaved())
        for i in range(n_torch_layers):
            ld, lp, ls = act.layer_desc[i], act.layer_params[i], act.layer_saved[i]
            ld.training, ld.p_drop, ld.seed = int(training), sp.p_layer, int(seed)
            self._fill_layer_params(lp, i)
            ls.qkv = buf(f"qkv{i}", (M, 3 * H), tdt).data_ptr()
            ls.attn = buf(f"attn{i}", (M, H), tdt).data_ptr()
            ls.lse = buf(f"lse{i}", (B, sp.heads, T), torch.float32).data_ptr()
            ls.y1 = buf(f"y1_{i}", (M, H), tdt).data_ptr()
            ls.stat1 = buf(f"stat1_{i}", (M, 2), torch.float32).data_ptr()
            ls.x1 = buf(f"x1_{i}", (M, H), tdt).data_ptr()
            ls.hid = buf(f"hid{i}", (M, FF), tdt).data_ptr()
            ls.y2 = buf(f"y2_{i}", (M, H), tdt).data_ptr()
            ls.stat2 = buf(f"stat2_{i}", (M, 2), torch.float32).data_ptr()
            if self.dtype == "bf16" and H == 128 and FF % 128 == 0:     # gate bits of the fused tcgen05 FFN
                ls.hid_mask = buf(f"hmask{i}", (FF // 64, M, 2), torch.int32).data_ptr()
                nscr = int(L.load().egot2_ffn_scratch_bytes(M)) // 4
                if nscr > 0:            # zeroed once; the fused FFN kernels leave it zeroed (see include/egot2.h)
                    if "ffn_scratch" not in t:
                        t["ffn_scratch"] = torch.zeros(nscr, device=dev, dtype=torch.float32)
                    ls.ffn_scratch = t["ffn_scratch"].data_ptr()
            x_out = buf(f"x{i + 1}", (B, T, H), tdt)
            L.call("egot2_encoder_layer_fwd", C.byref(ld), C.byref(lp), x.data_ptr(), x_out.data_ptr(), C.byref(ls),
                   None, 0, st)
            x = x_out
        t["x_last"] = x

        # ---- EgoT2-g: task-prompt decoder over the encoder memory, then the vocabulary head
        if sp.head == "decoder":
            return self._decoder_forward(act, x, prompt, training, seed, labels, loss, buf)

        # ---- head
        if sp.head == "tokens":
            D0 = seg_tokens[0]
            act.rows = B * D0
            out = buf("pooled", (act.rows, H), torch.float32)
            L.call("egot2_pool_fwd", self.dt, B, T, H, 0, D0, x.data_ptr(), out.data_ptr(), st)
            t["out"] = out
            return act
        if fresh or act.head_desc is None:
            hd = L.HeadDesc()
            hd.dtype, hd.B, hd.T, hd.H, hd.pool, hd.row_tokens = self.dt, B, T, H, 1, 0
            hd.use_ln = 1 if sp.head in ("pool_ln_linear", "pool_ln_multilinear") else 0
            hd.n_out, hd.ln_eps = sp.n_out, 1e-5
            if sp.head in ("pool_multilinear", "pool_ln_multilinear"):
                hd.n_groups, hd.sub_rows = len(sp.head_groups), sp.n_heads_out
                for gi, gs in enumerate(sp.head_groups):
                    hd.group_size[gi] = gs
            act.head_desc, act.head_in, act.head_out = hd, L.HeadIn(), L.HeadOut()
        hd, hin, hout = act.head_desc, act.head_in, act.head_out
        hd.loss, hd.training, hd.p_head, hd.seed = int(loss), int(training), sp.p_head, int(seed)
        rows = B
        act.rows = rows
        hin.x = x.data_ptr()
        if sp.head == "pool_ln_linear":
            ln_name = "ln" if sp.head_ln_shared else "linear_head.0"
            hin.ln_g, hin.ln_b = self._vec(ln_name + ".weight").data_ptr(), self._vec(ln_name + ".bias").data_ptr()
            hin.w, hin.b = self._mat("linear_head.1.weight").data_ptr(), self._vec("linear_head.1.bias").data_ptr()
        elif sp.head == "pool_linear":
            hin.w, hin.b = self._mat("linear_head.weight").data_ptr(), self._vec("linear_head.bias").data_ptr()
        else:
            base = self.arena.shadow if self.dtype == "bf16" else self.arena.param
            w, _ = self.arena.stacked_head(base)
            _, bvec = self.arena.stacked_head(self.arena.param)
            hin.w, hin.b = w.data_ptr(), bvec.data_ptr()
            if sp.head == "pool_ln_multilinear":      # AR: the shared ln in front of both heads
                hin.ln_g, hin.ln_b = self._vec("ln.weight").data_ptr(), self._vec("ln.bias").data_ptr()
        if loss != L.LOSS_NONE:
            assert labels is not None
            lab = labels.to(device=dev, dtype=torch.int64).contiguous()
            t["labels"] = lab
            hin.labels = lab.data_ptr()
            if class_weight is not None:
                cw = class_weight.to(device=dev, dtype=torch.float32).contiguous()
                t["class_weight"] = cw
                hin.class_weight = cw.data_ptr()
            else:
                hin.class_weight = None
            segs = rows * (sp.n_heads_out * len(sp.head_groups)
                           if sp.head in ("pool_multilinear", "pool_ln_multilinear") else 1)
            hout.row_loss = buf("row_loss", (segs, 2), torch.float32).data_ptr()
            hout.loss = buf("loss", (2,), torch.float32).data_ptr()
            hout.argmax = buf("argmax", (segs,), torch.int32).data_ptr()
        hout.pooled = buf("pooled", (rows, H), torch.float32).data_ptr()
        hout.stat = buf("stat_head", (rows, 2), torch.float32).data_ptr()
        hout.g = buf("g_head", (rows, H), tdt).data_ptr()
        logits = buf("logits", (rows, sp.n_out), torch.float32)
        hout.logits = logits.data_ptr()
        L.call("egot2_head_loss_fwd", C.byref(hd), C.byref(hin), C.byref(hout), st)
        t["out"] = logits
        return act

    # ------------------------------------------------------------------ simple_vit encoder (HOI PNR "simple_vit" sibling)
    _VIT_NAMES = {"qkv_w": "0.to_qkv.weight", "out_w": "0.to_out.weight", "ff1_w": "1.net.1.weight", "ff2_w": "1.net.3.weight",
                  "norm_a_g": "0.norm.weight", "norm_a_b": "0.norm.bias", "norm_f_g": "1.net.0.weight",
                  "norm_f_b": "1.net.0.bias", "ff1_b": "1.net.1.bias", "ff2_b": "1.net.3.bias"}

    def _fill_vit_params(self, vp, i: int, grads_base: Optional[torch.Tensor] = None):
        pre = f"{self.spec.encoder_prefix}layers.{i}."
        for f, n in self._VIT_NAMES.items():
            if grads_base is not None:
                setattr(vp, f, self.arena.view(pre + n, grads_base).data_ptr())
            elif f.endswith("_w"):
                setattr(vp, f, self._mat(pre + n).data_ptr())
            else:
                setattr(vp, f, self._vec(pre + n).data_ptr())

    def _vit_forward(self, act: Activations, x: torch.Tensor, buf) -> torch.Tensor:
        """depth x egot2_vit_layer_fwd (HOI/models/pnr/simple_vit.py:93-107); x: (B, T, D) tokens after ln + pe."""
        sp = self.spec
        B, T, D, tdt, st = act.B, act.T, sp.hidden, self.tdt, _stream()
        M, inner = B * T, sp.heads * sp.dim_head
        if not act.layer_desc:
            for i in range(sp.layers):
                vd = L.VitDesc()
                vd.dtype, vd.B, vd.T, vd.D, vd.heads, vd.dim_head, vd.mlp = self.dt, B, T, D, sp.heads, sp.dim_head, sp.ffn
                vd.layer_index, vd.ln_eps = i, 1e-5
                act.layer_desc.append(vd)
                act.layer_params.append(L.VitParams())
                act.layer_saved.append(L.VitSaved())
        for i in range(sp.layers):
            vd, vp, vs = act.layer_desc[i], act.layer_params[i], act.layer_saved[i]
            self._fill_vit_params(vp, i)
            for name, shape, dty in (("h", (M, D), tdt), ("stat_a", (M, 2), torch.float32), ("qkv", (M, 3 * inner), tdt),
                                     ("attn", (M, inner), tdt), ("lse", (B, sp.heads, T), torch.float32), ("x1", (M, D), tdt),
                                     ("h2", (M, D), tdt), ("stat_f", (M, 2), torch.float32), ("u", (M, sp.ffn), tdt),
                                     ("act", (M, sp.ffn), tdt)):
                setattr(vs, name, buf(f"vit{i}_{name}", shape, dty).data_ptr())
            x_out = buf(f"x{i + 1}", (B, T, D), tdt)
            L.call("egot2_vit_layer_fwd", C.byref(vd), C.byref(vp), x.data_ptr(), x_out.data_ptr(), C.byref(vs), st)
            x = x_out
        return x

    def _vit_backward(self, act: Activations, dx: torch.Tensor, grad: torch.Tensor):
        sp, t, st = self.spec, act.t, _stream()
        for i in reversed(range(sp.layers)):
            vd = act.layer_desc[i]
            vg = L.VitGrads()
            self._fill_vit_params(vg, i, grads_base=grad)
            x_in = t["x0"] if i == 0 else t[f"x{i}"]
            ws = self._workspace(L.load().egot2_vit_layer_workspace_bytes(C.byref(vd)))
            L.call("egot2_vit_layer_bwd", C.byref(vd), C.byref(act.layer_params[i]), x_in.data_ptr(),
                   C.byref(act.layer_saved[i]), dx.data_ptr(), dx.data_ptr(), C.byref(vg), ws.data_ptr(), ws.numel(), st)

    # ------------------------------------------------------------------ EgoT2-g decoder
    _DEC_NAMES = {"sa_in_w": "self_attn.in_proj_weight", "sa_out_w": "self_attn.out_proj.weight",
                  "ca_in_w": "multihead_attn.in_proj_weight", "ca_out_w": "multihead_attn.out_proj.weight",
                  "lin1_w": "linear1.weight", "lin2_w": "linear2.weight", "sa_in_b": "self_attn.in_proj_bias",
                  "sa_out_b": "self_attn.out_proj.bias", "ca_in_b": "multihead_attn.in_proj_bias",
                  "ca_out_b": "multihead_attn.out_proj.bias", "lin1_b": "linear1.bias", "lin2_b": "linear2.bias",
                  "norm1_g": "norm1.weight", "norm1_b": "norm1.bias", "norm2_g": "norm2.weight", "norm2_b": "norm2.bias",
                  "norm3_g": "norm3.weight", "norm3_b": "norm3.bias"}

    def _fill_decoder_params(self, dp, i: int, grads_base: Optional[torch.Tensor] = None):
        pre = f"transformer_decoder.layers.{i}."
        for f, n in self._DEC_NAMES.items():
            if grads_base is not None:
                setattr(dp, f, self.arena.view(pre + n, grads_base).data_ptr())
            elif f.endswith("_w"):
                setattr(dp, f, self._mat(pre + n).data_ptr())
            else:
                setattr(dp, f, self._vec(pre + n).data_ptr())

    def _decoder_forward(self, act: Activations, mem: torch.Tensor, prompt, training, seed, labels, loss, buf):
        """decode() of TaskTranslationPromptTransformer (task_prompt_model.py:260-269) + CE over the vocabulary
        (HHI/tasks/multitask/video_tasktranslation.py:48-61).  prompt: (rows, S) int64 decoder input tokens."""
        sp = self.spec
        if prompt is None:
            raise L.Egot2Error("EgoT2-g translator: forward() needs the decoder prompt tokens")
        if self.pe_buffer is None:
            raise L.Egot2Error("EgoT2-g translator: call set_sinusoid(pos_embed.pe) first")
        B, T, H, FF = act.B, act.T, sp.hidden, sp.ffn
        dev, tdt, st = self.device, self.tdt, _stream()
        t = act.t
        if sp.g_mode == "asd":
            if len(set(act.seg_tokens)) != 1:
                raise L.Egot2Error("EgoT2-g 'asd' regroups the memory per frame: the three tasks need equal lengths")
            Tt = act.seg_tokens[0]
            rows, M, inner, outer, jstr, istr = B * Tt, 3, Tt, T, Tt, 1
        else:
            rows, M, inner, outer, jstr, istr = B, T, 1, T, 1, 0
        prompt = prompt.to(device=dev, dtype=torch.int64).contiguous()
        assert prompt.dim() == 2 and prompt.shape[0] == rows, f"prompt must be ({rows}, S), got {tuple(prompt.shape)}"
        S = int(prompt.shape[1])
        R = rows * S
        act.prompt, act.rows = prompt, R
        t["prompt"] = prompt
        y = buf("dec_y0", (rows, S, H), tdt)
        L.call("egot2_prompt_embed_fwd", self.dt, rows, S, H, prompt.data_ptr(), self._vec("embedding.weight").data_ptr(),
               self.pe_buffer.data_ptr(), 0.1, int(training), int(seed), y.data_ptr(), st)
        if not act.dec_desc:
            for i in range(sp.decoder_layers):
                dd = L.DecoderDesc()
                dd.dtype, dd.rows, dd.S, dd.mem_rows, dd.M = self.dt, rows, S, B * T, M
                dd.kv_inner, dd.kv_outer, dd.kv_jstride, dd.kv_istride = inner, outer, jstr, istr
                dd.H, dd.FF, dd.heads, dd.layer_index, dd.ln_eps = H, FF, sp.heads, i, 1e-5
                act.dec_desc.append(dd)
                act.dec_params.append(L.DecoderParams())
                act.dec_saved.append(L.DecoderSaved())
        for i in range(sp.decoder_layers):
            dd, dp, ds = act.dec_desc[i], act.dec_params[i], act.dec_saved[i]
            dd.training, dd.p_drop, dd.seed = int(training), sp.p_layer, int(seed)
            self._fill_decoder_params(dp, i)
            for name, shape, dty in (("qkv", (R, 3 * H), tdt), ("a1", (R, H), tdt), ("y1", (R, H), tdt),
                                     ("stat1", (R, 2), torch.float32), ("x1", (R, H), tdt), ("qc", (R, H), tdt),
                                     ("kvc", (B * T, 2 * H), tdt), ("a2", (R, H), tdt), ("y2", (R, H), tdt),
                                     ("stat2", (R, 2), torch.float32), ("x2", (R, H), tdt), ("hid", (R, FF), tdt),
                                     ("y3", (R, H), tdt), ("stat3", (R, 2), torch.float32)):
                setattr(ds, name, buf(f"dec{i}_{name}", shape, dty).data_ptr())
            y_out = buf(f"dec_y{i + 1}", (rows, S, H), tdt)
            L.call("egot2_decoder_layer_fwd", C.byref(dd), C.byref(dp), y.data_ptr(), mem.data_ptr(), y_out.data_ptr(),
                   C.byref(ds), st)
            y = y_out
        t["dec_last"] = y
        # vocabulary head on every prompt position: rows*S rows, no pooling, no LayerNorm
        if act.head_desc is None:
            hd = L.HeadDesc()
            hd.dtype, hd.B, hd.T, hd.H, hd.pool, hd.row_tokens, hd.use_ln = self.dt, rows, S, H, 0, S, 0
            hd.n_out, hd.ln_eps = sp.vocab, 1e-5
            act.head_desc, act.head_in, act.head_out = hd, L.HeadIn(), L.HeadOut()
        hd, hin, hout = act.head_desc, act.head_in, act.head_out
        hd.loss, hd.training, hd.p_head, hd.seed = int(loss), int(training), 0.0, int(seed)
        hin.x = y.data_ptr()
        hin.w, hin.b = self._mat("fc.weight").data_ptr(), self._vec("fc.bias").data_ptr()
        if loss != L.LOSS_NONE:
            assert labels is not None
            lab = labels.to(device=dev, dtype=torch.int64).reshape(-1).contiguous()
            assert lab.numel() == R, f"expected {R} target tokens, got {lab.numel()}"
            t["labels"] = lab
            hin.labels = lab.data_ptr()
            hin.class_weight = None
            hout.row_loss = buf("row_loss", (R, 2), torch.float32).data_ptr()
            hout.loss = buf("loss", (2,), torch.float32).data_ptr()
            hout.argmax = buf("argmax", (R,), torch.int32).data_ptr()
        hout.pooled = buf("pooled", (R, H), torch.float32).data_ptr()
        hout.stat = buf("stat_head", (R, 2), torch.float32).data_ptr()
        hout.g = buf("g_head", (R, H), tdt).data_ptr()
        logits = buf("logits", (R, sp.vocab), torch.float32)
        hout.logits = logits.data_ptr()
        L.call("egot2_head_loss_fwd", C.byref(hd), C.byref(hin), C.byref(hout), st)
        t["out"] = logits
        return act

    @_on_device
    def decode_again(self, act: Activations, prompt: torch.Tensor) -> Activations:
        """Greedy decoding step of EgoT2-g (predict_ac, HOI/models/multitask/video_model_builder.py:264-275): only the
        decoder and the vocabulary head run, for a new (longer) prompt, over the encoder memory `act` already holds.
        Inference only; the returned activations own their decoder buffers and share the memory."""
        if self.spec.head != "decoder" or "x_last" not in act.t:
            raise L.Egot2Error("decode_again: needs the activations of an EgoT2-g forward")
        act2 = Activations(act.B, act.seg_tokens, act.T, False, 0)
        t, dev = act2.t, self.device
        t["x_last"] = act.t["x_last"]

        def buf(name, shape, dtype):
            if name not in t:
                t[name] = torch.empty(shape, device=dev, dtype=dtype)
            return t[name]
        return self._decoder_forward(act2, t["x_last"], prompt, False, 0, None, L.LOSS_NONE, buf)

    def _decoder_backward(self, act: Activations, dout, dloss_scale, grad, gv) -> torch.Tensor:
        """Backward of the vocabulary head, the decoder layers and the prompt embedding; returns d(loss)/d(memory) in the
        activation dtype, i.e. the gradient entering the encoder."""
        sp = self.spec
        B, T, H = act.B, act.T, sp.hidden
        dev, tdt, st = self.device, self.tdt, _stream()
        t = act.t
        rows, S = act.dec_desc[0].rows, act.dec_desc[0].S
        R = rows * S
        hd = act.head_desc
        if hd.loss == L.LOSS_NONE:
            assert dout is not None
            dlogits = dout.to(device=dev, dtype=torch.float32).reshape(R, sp.vocab).contiguous().clone()
        else:
            dlogits = torch.empty((R, sp.vocab), device=dev, dtype=torch.float32)
        hg = L.HeadGrads()
        hg.w, hg.b = gv("fc.weight").data_ptr(), gv("fc.bias").data_ptr()
        dy = torch.empty((rows, S, H), device=dev, dtype=tdt)
        ws = self._workspace(L.load().egot2_head_workspace_bytes(C.byref(hd)))
        L.call("egot2_head_loss_bwd", C.byref(hd), C.byref(act.head_in), C.byref(act.head_out), dlogits.data_ptr(),
               float(dloss_scale), dy.data_ptr(), C.byref(hg), ws.data_ptr(), ws.numel(), st)
        dmem = torch.zeros((B * T, H), device=dev, dtype=torch.float32)
        mem = t["x_last"]
        for i in reversed(range(sp.decoder_layers)):
            dd = act.dec_desc[i]
            dg = L.DecoderGrads()
            self._fill_decoder_params(dg, i, grads_base=grad)
            y_in = t[f"dec_y{i}"]
            ws = self._workspace(L.load().egot2_decoder_layer_workspace_bytes(C.byref(dd)))
            L.call("egot2_decoder_layer_bwd", C.byref(dd), C.byref(act.dec_params[i]), y_in.data_ptr(), mem.data_ptr(),
                   C.byref(act.dec_saved[i]), dy.data_ptr(), dy.data_ptr(), dmem.data_ptr(), C.byref(dg), ws.data_ptr(),
                   ws.numel(), st)
        L.call("egot2_prompt_embed_bwd", self.dt, rows, S, H, act.prompt.data_ptr(), dy.data_ptr(), 0.1,
               int(act.training), int(act.seed), gv("embedding.weight").data_ptr(), st)
        return dmem.view(B, T, H).to(tdt)

    def _fill_layer_params(self, lp: L.LayerParams, i: int, grads_base: Optional[torch.Tensor] = None):
        p = f"{self.spec.encoder_prefix}layers.{i}."
        names = {"in_proj_w": "self_attn.in_proj_weight", "out_proj_w": "self_attn.out_proj.weight",
                 "lin1_w": "linear1.weight", "lin2_w": "linear2.weight", "in_proj_b": "self_attn.in_proj_bias",
                 "out_proj_b": "self_attn.out_proj.bias", "lin1_b": "linear1.bias", "lin2_b": "linear2.bias",
                 "norm1_g": "norm1.weight", "norm1_b": "norm1.bias", "norm2_g": "norm2.weight", "norm2_b": "norm2.bias"}
        for f, n in names.items():
            if grads_base is not None:
                setattr(lp, f, self.arena.view(p + n, grads_base).data_ptr())
            elif f.endswith("_w"):
                setattr(lp, f, self._mat(p + n).data_ptr())
            else:
                setattr(lp, f, self._vec(p + n).data_ptr())

    # ------------------------------------------------------------------ backward
    @_on_device
    def backward(self, act: Activations, dout: Optional[torch.Tensor] = None, dloss_scale: float = 1.0,
                 grad: Optional[torch.Tensor] = None, zero_grad: bool = True,
                 want_dfeat: Sequence[bool] = (), stage: str = "all") -> Tuple[torch.Tensor, List[Optional[torch.Tensor]]]:
        """Gradients of every translator parameter, accumulated into `grad` (a flat fp32 buffer with the
        arena layout; default: arena.grad).  `dout`: gradient w.r.t. the forward output when the loss was
        computed outside (drop-in autograd path); with a fused loss pass dloss_scale instead."""
        sp = self.spec
        B, T, H = act.B, act.T, sp.hidden
        grad = self.arena.grad if grad is None else grad
        assert stage in ("all", "pre_embed", "embed")
        if zero_grad and stage != "embed":
            grad.zero_()
        st = _stream()
        tdt, dev = self.tdt, self.device
        t = act.t
        gv = lambda name: self.arena.view(name, grad)
        # stage = "pre_embed" | "embed": the two halves of backward as separate calls (separate CUDA graphs in the
        # data-parallel trainer, so that most of the gradient all-reduce overlaps the embedding backward); the gradient
        # w.r.t. the encoder input then lives in a persistent buffer between the two
        if stage == "all":
            dx = torch.empty((B, T, H), device=dev, dtype=tdt)
        else:
            assert sp.head != "decoder", "staged backward is not wired for the EgoT2-g decoder head"
            if "dx_chain" not in t:
                t["dx_chain"] = torch.empty((B, T, H), device=dev, dtype=tdt)
            dx = t["dx_chain"]
        if stage == "embed":
            return self._embed_backward(act, dx, grad, gv, want_dfeat)

        # ---- head
        if sp.head == "decoder":
            dx = self._decoder_backward(act, dout, dloss_scale, grad, gv).contiguous()
        elif sp.head == "tokens":
            assert dout is not None
            dp = dout.to(device=dev, dtype=torch.float32).contiguous()
            L.call("egot2_pool_bwd", self.dt, B, T, H, 0, act.seg_tokens[0], dp.data_ptr(), dx.data_ptr(), st)
        else:
            hd = act.head_desc
            if hd.loss == L.LOSS_NONE:
                assert dout is not None
                dlogits = dout.to(device=dev, dtype=torch.float32).contiguous().clone()
            else:
                dlogits = torch.empty((act.rows, sp.n_out), device=dev, dtype=torch.float32)
            hg = L.HeadGrads()
            if sp.head == "pool_ln_linear":
                ln_name = "ln" if sp.head_ln_shared else "linear_head.0"
                hg.ln_g, hg.ln_b = gv(ln_name + ".weight").data_ptr(), gv(ln_name + ".bias").data_ptr()
                hg.w, hg.b = gv("linear_head.1.weight").data_ptr(), gv("linear_head.1.bias").data_ptr()
            elif sp.head == "pool_linear":
                hg.w, hg.b = gv("linear_head.weight").data_ptr(), gv("linear_head.bias").data_ptr()
            else:
                w, bvec = self.arena.stacked_head(grad)
                hg.w, hg.b = w.data_ptr(), bvec.data_ptr()
                if sp.head == "pool_ln_multilinear":
                    hg.ln_g, hg.ln_b = gv("ln.weight").data_ptr(), gv("ln.bias").data_ptr()
            ws = self._workspace(L.load().egot2_head_workspace_bytes(C.byref(hd)))
            L.call("egot2_head_loss_bwd", C.byref(hd), C.byref(act.head_in), C.byref(act.head_out), dlogits.data_ptr(),
                   float(dloss_scale), dx.data_ptr(), C.byref(hg), ws.data_ptr(), ws.numel(), st)

        # ---- encoder layers (reverse)
        if sp.encoder == "simple_vit":
            self._vit_backward(act, dx, grad)
        # The parameter-gradient branches of a layer (side streams) are not joined at the layer boundary: they overlap the
        # next layer's chain (two alternating workspaces) and the embedding backward (its own workspace), and everything is
        # joined once before this call returns.
        n_enc = sp.layers if sp.encoder == "torch" else 0
        defer = self.defer_joins and n_enc > 0
        if defer:
            L.call("egot2_side_defer", 1)
        try:
            for i in reversed(range(n_enc)):
                ld = act.layer_desc[i]
                lg = L.LayerGrads()
                self._fill_layer_params(lg, i, grads_base=grad)
                x_in = t["x0"] if i == 0 else t[f"x{i}"]
                ws = self._workspace(L.load().egot2_encoder_layer_workspace_bytes(C.byref(ld), 1),
                                     slot=(i & 1) if defer else 0)
                L.call("egot2_encoder_layer_bwd", C.byref(ld), C.byref(act.layer_params[i]), x_in.data_ptr(),
                       C.byref(act.layer_saved[i]), dx.data_ptr(), dx.data_ptr(), C.byref(lg), ws.data_ptr(), ws.numel(), st)
            if stage == "pre_embed":
                return grad, [None] * len(sp.segments)
            return self._embed_backward(act, dx, grad, gv, want_dfeat, ws_slot=2 if defer else 0)
        finally:
            if defer:
                L.call("egot2_side_defer", 0)
                L.call("egot2_side_join_all", st)

    def _embed_backward(self, act: Activations, dx: torch.Tensor, grad: torch.Tensor, gv, want_dfeat, ws_slot: int = 0):
        sp = self.spec
        B, T, H = act.B, act.T, sp.hidden
        dev, st = self.device, _stream()
        # ---- embed
        eg = L.EmbedGrads()
        dfeats: List[Optional[torch.Tensor]] = [None] * len(sp.segments)
        for k, s in enumerate(sp.segments):
            if s.proj is not None:
                eg.proj_w[k] = gv(s.proj + ".weight").data_ptr()
                eg.proj_b[k] = gv(s.proj + ".bias").data_ptr()
            if k < len(want_dfeat) and want_dfeat[k]:
                dfeats[k] = torch.empty((B, act.seg_tokens[k], s.in_dim), device=dev, dtype=torch.float32)
                eg.dfeat[k] = dfeats[k].data_ptr()
        if sp.embed_ln:
            eg.ln_g, eg.ln_b = gv("ln.weight").data_ptr(), gv("ln.bias").data_ptr()
        if sp.embed == "task_sinusoid":
            # table row = task_embed[task_k] + fixed sinusoid: the column sums of each segment go straight into
            # d(task_embed[task_k]) (no (T,H) table gradient, no second reduction pass)
            te = gv("task_embed").view(-1, H)
            for k, s in enumerate(sp.segments):
                eg.seg_embed[k] = te[s.task_id].data_ptr()
        else:
            eg.tok_table = gv("pe").view(T, H).data_ptr()
        d = act.embed_desc
        ws = self._workspace(L.load().egot2_embed_workspace_bytes(C.byref(d), 1), slot=ws_slot)
        L.call("egot2_embed_bwd", C.byref(d), C.byref(act.embed_in), C.byref(act.embed_out), dx.data_ptr(), C.byref(eg),
               ws.data_ptr(), ws.numel(), st)
        return grad, dfeats

    # ------------------------------------------------------------------ fused optimizer
    @_on_device
    def adam_step(self, state: Dict[str, torch.Tensor], step: int, lr: float = 5e-4, betas=(0.9, 0.999),
                  eps: float = 1e-8, weight_decay: float = 0.0, grad_scale: float = 1.0, fused: bool = False,
                  step_dev: Optional[torch.Tensor] = None, decoupled: bool = False, lr_dev: Optional[torch.Tensor] = None,
                  guard: Optional[torch.Tensor] = None):
        """torch.optim.Adam over the whole arena in one launch (HHI/tasks/ttm/video_task.py:64-66: lr 5e-4).
        fused: the same launch also writes the bf16 shadow of the updated parameters (bf16 engines) and clears the
        gradient arena, so the next step needs neither the cast launch nor a fill (callers then pass
        zero_grad=False to backward()).
        step_dev / lr_dev: the step count (int32) and the learning rate (float32) are read from device memory when the
        kernel executes (graph replays, device-evaluated schedules: optim.py); lr_dev needs step_dev.
        guard: a device egot2_grad_guard (_lib.GradGuard bytes; fused, needs step_dev): egot2_grad_norm of grad_scale * the
        gradient arena first, then the update clipped by that norm, or skipped (gradient cleared, step count taken back)
        when it is not finite."""
        if "m" not in state:
            state["m"] = torch.zeros_like(self.arena.param)
            state["v"] = torch.zeros_like(self.arena.param)
        if lr_dev is not None and step_dev is None:
            raise L.Egot2Error("adam_step: lr_dev needs step_dev (egot2_opt_advance keeps both on the device)")
        if guard is not None and (step_dev is None or not fused):
            raise L.Egot2Error("adam_step: a gradient guard needs the fused launch and step_dev (a skip takes the step back)")
        if fused:
            shadow = None
            if self.dtype == "bf16":
                if self.arena.shadow is None:
                    self.arena.refresh_shadow()
                shadow = self.arena.shadow.data_ptr()
            if guard is not None:
                ws = self.grad_norm_workspace()
                L.call("egot2_grad_norm", self.arena.grad.data_ptr(), self.arena.numel, float(grad_scale), guard.data_ptr(),
                       step_dev.data_ptr(), ws.data_ptr(), ws.numel(), _stream())
                L.call("egot2_adam_step_fused_guard", self.arena.param.data_ptr(), self.arena.grad.data_ptr(),
                       state["m"].data_ptr(), state["v"].data_ptr(), self.arena.numel, float(lr),
                       None if lr_dev is None else lr_dev.data_ptr(), betas[0], betas[1], eps, weight_decay,
                       step_dev.data_ptr(), float(grad_scale), shadow, 1, 1 if decoupled else 0, guard.data_ptr(), _stream())
            elif step_dev is not None and (lr_dev is not None or decoupled):
                if lr_dev is None:          # AdamW with a device step count: the fixed lr goes to the device as well
                    lr_dev = torch.full((1,), float(lr), device=self.device, dtype=torch.float32)
                L.call("egot2_adam_step_fused_sched", self.arena.param.data_ptr(), self.arena.grad.data_ptr(),
                       state["m"].data_ptr(), state["v"].data_ptr(), self.arena.numel, lr_dev.data_ptr(), betas[0],
                       betas[1], eps, weight_decay, step_dev.data_ptr(), float(grad_scale), shadow, 1,
                       1 if decoupled else 0, _stream())
            elif step_dev is not None:      # step count read on the device (graph-resident update)
                L.call("egot2_adam_step_fused_dev", self.arena.param.data_ptr(), self.arena.grad.data_ptr(),
                       state["m"].data_ptr(), state["v"].data_ptr(), self.arena.numel, lr, betas[0], betas[1], eps,
                       weight_decay, step_dev.data_ptr(), float(grad_scale), shadow, 1, _stream())
            elif decoupled:                 # torch.optim.AdamW (HOI EgoT2-g)
                L.call("egot2_adamw_step_fused", self.arena.param.data_ptr(), self.arena.grad.data_ptr(),
                       state["m"].data_ptr(), state["v"].data_ptr(), self.arena.numel, lr, betas[0], betas[1], eps,
                       weight_decay, int(step), float(grad_scale), shadow, 1, _stream())
            else:
                L.call("egot2_adam_step_fused", self.arena.param.data_ptr(), self.arena.grad.data_ptr(),
                       state["m"].data_ptr(), state["v"].data_ptr(), self.arena.numel, lr, betas[0], betas[1], eps,
                       weight_decay, int(step), float(grad_scale), shadow, 1, _stream())
            self.arena.shadow_fresh = shadow is not None
            return
        if decoupled:
            raise L.Egot2Error("adam_step: decoupled weight decay (AdamW) is only built into the fused launch")
        L.call("egot2_adam_step", self.arena.param.data_ptr(), self.arena.grad.data_ptr(), state["m"].data_ptr(),
               state["v"].data_ptr(), self.arena.numel, lr, betas[0], betas[1], eps, weight_decay, int(step),
               float(grad_scale), _stream())
        self.arena.shadow_fresh = False

    def grad_norm_workspace(self) -> torch.Tensor:
        """The egot2_grad_norm workspace of this engine: zero-filled once, and every launch leaves it so.  Trainers allocate it
        at construction, outside any CUDA-graph capture."""
        ws = getattr(self, "_norm_ws", None)
        if ws is None:
            ws = self._norm_ws = torch.zeros(int(L.load().egot2_grad_norm_workspace_bytes()), device=self.device,
                                             dtype=torch.uint8)
        return ws
