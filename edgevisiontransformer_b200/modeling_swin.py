"""Drop-in B200 Swin Transformer classifier (SURVEY.md section 8f rank 4).

The reference builds ``swin_{tiny,small,base}_patch4_window7_224`` from an external checkout of microsoft/Swin-Transformer
(utils.py:14-47 ``get_swin``) and exports / benchmarks it (tools.py:265-292 ``export_onnx_swin``); the same network with HF
key names is ``transformers.SwinForImageClassification`` (SITE/models/swin/modeling_swin.py), which is what
:meth:`B200SwinForImageClassification.from_hf` takes.  ``from_microsoft`` renames a state dict of the original repository.
The 384-pixel checkpoints ``swin_{base,large}_patch4_window12_384`` (12 x 12 windows of 144 tokens) run as well.

Data layout: inside a stage the f32 residual stream ``[B*T, C]`` is kept in the WINDOW ORDER of the current block (image,
window, token in window).  A block whose cyclic shift differs from the previous one starts with a row gather fused into its
``layernorm_before`` (``evt_gather_layernorm``: LN output for the QKV GEMM + the permuted residual copy); patch merging is
the same kernel with a 4-row gather.  Everything between -- QKV / out-proj / FC1+GELU / FC2 -- is the tcgen05 GEMM of the
ViT path with its TMA reduce-add epilogue, attention is ``evt_window_attention_fwd``.  bf16 operands, f32 accumulate /
residual / LayerNorm / softmax; logits within 2e-2 of the f32 reference.  No CPU fallback.
"""
from __future__ import annotations

import math
from typing import Dict, List, Sequence

import torch
import torch.nn as nn

import ctypes as ct

from . import _lib, ops
from .modeling_vit import ImageClassifierOutput

LOG2E = 1.4426950408889634


def window_order(H: int, W: int, ws: int, shift: int) -> torch.Tensor:
    """raster index (y*W + x) of every position of the window order: r = ((wh*nWw + ww)*ws + i)*ws + j holds the token
    at y = (wh*ws + i + shift) % H, x = (ww*ws + j + shift) % W   (roll by -shift, then window_partition, :606-613)."""
    wh, ww, i, j = torch.meshgrid(torch.arange(H // ws), torch.arange(W // ws), torch.arange(ws), torch.arange(ws), indexing="ij")
    y = (wh * ws + i + shift) % H
    x = (ww * ws + j + shift) % W
    return (y * W + x).reshape(-1)


def _inverse(perm: torch.Tensor) -> torch.Tensor:
    inv = torch.empty_like(perm)
    inv[perm] = torch.arange(perm.numel())
    return inv


def relative_position_index(ws: int) -> torch.Tensor:
    coords = torch.stack(torch.meshgrid([torch.arange(ws), torch.arange(ws)], indexing="ij")).flatten(1)
    rel = (coords[:, :, None] - coords[:, None, :]).permute(1, 2, 0).contiguous()
    rel[:, :, 0] += ws - 1
    rel[:, :, 1] += ws - 1
    rel[:, :, 0] *= 2 * ws - 1
    return rel.sum(-1)


def shift_mask(H: int, W: int, ws: int, shift: int) -> torch.Tensor:
    """[nW, ws*ws, ws*ws] additive 0 / -100 mask of SW-MSA (SwinLayer.get_attn_mask, :556-582)."""
    img = torch.zeros(H, W)
    cnt = 0
    for hs in (slice(0, -ws), slice(-ws, -shift), slice(-shift, None)):
        for wsl in (slice(0, -ws), slice(-ws, -shift), slice(-shift, None)):
            img[hs, wsl] = cnt
            cnt += 1
    mw = img.view(H // ws, ws, W // ws, ws).permute(0, 2, 1, 3).reshape(-1, ws * ws)
    m = mw.unsqueeze(1) - mw.unsqueeze(2)
    return torch.where(m != 0, torch.full_like(m, -100.0), torch.zeros_like(m))


def attention_table(bias_table: torch.Tensor, heads: int, ws: int, mask: torch.Tensor = None) -> torch.Tensor:
    """(relative position bias [+ shift mask]) * log2(e) in the kernel's layout: padded to [n_tab, heads, 64, 56] for 7 x 7
    windows, [n_tab, heads, 144, 144] for 12 x 12."""
    N = ws * ws
    bias = bias_table[relative_position_index(ws).view(-1)].view(N, N, heads).permute(2, 0, 1).float()      # [heads, N, N]
    full = bias.unsqueeze(0) if mask is None else bias.unsqueeze(0) + mask.unsqueeze(1)
    rows, cols = ops.window_table_shape(N)
    out = torch.zeros(full.shape[0], heads, rows, cols)
    out[:, :, :, N:] = -float("inf")
    out[:, :, :N, :N] = full * LOG2E
    return out.contiguous()


class B200SwinConfig:
    """The attributes the reference's callers (and eval_loop.PipelinedClassifier) read off ``model.config``."""

    def __init__(self, depths, num_heads, embed_dim, window_size, patch_size, image_size, layer_norm_eps, num_labels):
        self.depths, self.num_heads, self.embed_dim = list(depths), list(num_heads), embed_dim
        self.window_size, self.patch_size, self.image_size = window_size, patch_size, image_size
        self.layer_norm_eps, self.num_labels = layer_norm_eps, num_labels
        self.hidden_size = embed_dim * 2 ** (len(self.depths) - 1)


class B200SwinForImageClassification(nn.Module):
    """Inference-only.  ``state_dict`` uses HF key names (``swin.embeddings...``, ``swin.encoder.layers.{s}.blocks.{b}...``).
    ``window`` 7 (224 pixels) or 12 (384 pixels)."""

    def __init__(self, state_dict: Dict[str, torch.Tensor], depths: Sequence[int], num_heads: Sequence[int], embed_dim: int,
                 window: int = 7, patch: int = 4, image_size: int = 224, eps: float = 1e-5, device="cuda", max_batch: int = 1024):
        super().__init__()
        dev = torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError("B200SwinForImageClassification runs only on a CUDA (sm_100a) device; no CPU fallback")
        if window not in (7, 12) or any(embed_dim * 2 ** s != 32 * h for s, h in enumerate(num_heads)):
            raise ValueError("only 7x7 and 12x12 windows with head size 32 are implemented "
                             "(swin_{tiny,small,base,large}_patch4_window7_224, swin_{base,large}_patch4_window12_384)")
        grid = image_size // patch
        if image_size % patch or grid % (window * 2 ** (len(depths) - 1)):
            raise ValueError("image_size / patch must be a multiple of window * 2^(stages-1)")
        self.depths, self.num_heads, self.embed_dim = list(depths), list(num_heads), embed_dim
        self.window, self.patch, self.image_size, self.eps = window, patch, image_size, eps
        self.max_batch, self._device = int(max_batch), dev
        self._graphs: dict = {}
        sd = {k: v.detach() for k, v in state_dict.items()}

        def f32(k):
            return sd[k].to(device=dev, dtype=torch.float32).contiguous()

        def bf16(k):
            return sd[k].to(device=dev, dtype=torch.float32).reshape(sd[k].shape[0], -1).to(torch.bfloat16).contiguous()

        e = "swin.embeddings."
        self.w_patch, self.b_patch = bf16(e + "patch_embeddings.projection.weight"), f32(e + "patch_embeddings.projection.bias")
        self.g_embed, self.be_embed = f32(e + "norm.weight"), f32(e + "norm.bias")
        self.stages: List[dict] = []
        H = grid
        order = torch.arange(H * H)                               # raster after the patch embedding
        first = window_order(H, H, window, 0)
        self.idx_embed = _inverse(order)[first].to(torch.int32).to(dev)
        order = first
        for s, depth in enumerate(depths):
            C, heads = embed_dim * 2 ** s, num_heads[s]
            blocks = []
            for b in range(depth):
                p = f"swin.encoder.layers.{s}.blocks.{b}."
                shift = window // 2 if (b % 2 == 1 and H > window) else 0
                want = window_order(H, H, window, shift)
                blk = dict(shift=shift, idx=None)
                if not torch.equal(want, order):
                    blk["idx"] = _inverse(order)[want].to(torch.int32).to(dev)
                    order = want
                blk["ln1"] = (f32(p + "layernorm_before.weight"), f32(p + "layernorm_before.bias"))
                blk["wqkv"] = torch.cat([bf16(p + f"attention.self.{n}.weight") for n in ("query", "key", "value")], 0).contiguous()
                blk["bqkv"] = torch.cat([f32(p + f"attention.self.{n}.bias") for n in ("query", "key", "value")], 0).contiguous()
                mask = shift_mask(H, H, window, shift) if shift > 0 else None
                blk["table"] = attention_table(sd[p + "attention.self.relative_position_bias_table"].float().cpu(), heads, window,
                                               mask).to(dev)
                blk["wo"], blk["bo"] = bf16(p + "attention.output.dense.weight"), f32(p + "attention.output.dense.bias")
                blk["ln2"] = (f32(p + "layernorm_after.weight"), f32(p + "layernorm_after.bias"))
                blk["w1"], blk["b1"] = bf16(p + "intermediate.dense.weight"), f32(p + "intermediate.dense.bias")
                blk["w2"], blk["b2"] = bf16(p + "output.dense.weight"), f32(p + "output.dense.bias")
                blocks.append(blk)
            st = dict(C=C, heads=heads, H=H, blocks=blocks, merge=None)
            if s + 1 < len(depths):
                p = f"swin.encoder.layers.{s}.downsample."
                H2 = H // 2
                nxt = window_order(H2, H2, window, 0)             # the next stage starts in (unshifted) window order
                y2, x2 = nxt // H2, nxt % H2
                src = torch.stack([(2 * y2) * H + 2 * x2, (2 * y2 + 1) * H + 2 * x2, (2 * y2) * H + 2 * x2 + 1,
                                   (2 * y2 + 1) * H + 2 * x2 + 1], dim=1)                        # :334-343 concat order
                st["merge"] = dict(idx=_inverse(order)[src].to(torch.int32).contiguous().to(dev),
                                   ln=(f32(p + "norm.weight"), f32(p + "norm.bias")), w=bf16(p + "reduction.weight"))
                order, H = nxt, H2
            self.stages.append(st)
        self.g_final, self.b_final = f32("swin.layernorm.weight"), f32("swin.layernorm.bias")
        self.w_cls, self.b_cls = bf16("classifier.weight"), f32("classifier.bias")
        self.num_labels = self.w_cls.shape[0]
        self.config = B200SwinConfig(depths, num_heads, embed_dim, window, patch, image_size, eps, self.num_labels)
        self._param = nn.Parameter(self.b_cls, requires_grad=False)       # next(model.parameters()).device works
        # The C++ runtime (evt_swin_*, csrc/swin_model.cu): same weights under their HF names, the window orders / gathers /
        # bias + mask tables recomputed on the host inside the library; one call issues the whole launch sequence.  The
        # op-level composition above (_run_ops) stays as the cross-check of the tests.
        self._lib = _lib.load()
        self._handle = ct.c_void_p()
        self._ws, self._ws_batch = None, 0
        spec = _lib.SwinSpec()
        spec.image, spec.patch, spec.window, spec.embed_dim = image_size, patch, window, embed_dim
        spec.stages, spec.num_labels, spec.eps = len(self.depths), self.num_labels, float(eps)
        for i, (d, h) in enumerate(zip(self.depths, self.num_heads)):
            spec.depths[i], spec.heads[i] = int(d), int(h)
        with torch.cuda.device(dev):
            _lib.check(self._lib.evt_swin_create(ct.byref(spec), ct.byref(self._handle)), "swin_create")
            dev_sd = {k: v.to(device=dev, dtype=torch.float32).contiguous() for k, v in sd.items()
                      if torch.is_tensor(v) and v.is_floating_point()}
            views = (_lib.TensorView * len(dev_sd))()
            keep = []
            for i, (k, v) in enumerate(dev_sd.items()):
                name = k.encode()
                keep.append(name)
                views[i].name, views[i].data, views[i].ndim = name, v.data_ptr(), 1
                views[i].shape[0] = v.numel()
            _lib.check(self._lib.evt_swin_load_weights(self._handle, views, len(dev_sd), torch.cuda.current_stream().cuda_stream),
                       "swin_load_weights")
        self.use_ops = False        # True: the Python-composed op sequence instead of the C++ runtime (tests)

    # ------------------------------------------------------------------ constructors
    @classmethod
    def from_hf(cls, model: nn.Module, **kw):
        c = model.config
        return cls(model.state_dict(), depths=c.depths, num_heads=c.num_heads, embed_dim=c.embed_dim, window=c.window_size,
                   patch=c.patch_size, image_size=c.image_size, eps=c.layer_norm_eps, **kw)

    @classmethod
    def from_microsoft(cls, state_dict: Dict[str, torch.Tensor], depths, num_heads, embed_dim, **kw):
        """State dict of microsoft/Swin-Transformer's ``SwinTransformer`` (what ``get_swin`` + ``load_state_dict(sd['model'])``
        holds, tools.py:284-288): fused ``attn.qkv``, ``patch_embed`` / ``layers.{s}.blocks.{b}`` / ``norm`` / ``head`` names.
        Unless given, the window is read off the (2w-1)^2 rows of the first relative position bias table and the image size
        is that of the published checkpoints with that window (7: 224, 12: 384)."""
        sd = microsoft_to_hf(state_dict)
        if "window" not in kw:
            n = sd["swin.encoder.layers.0.blocks.0.attention.self.relative_position_bias_table"].shape[0]
            side = math.isqrt(n)
            if side * side != n or side % 2 == 0:
                raise ValueError(f"relative_position_bias_table has {n} rows, not (2 * window - 1)^2")
            kw["window"] = (side + 1) // 2
        kw.setdefault("image_size", {7: 224, 12: 384}.get(kw["window"], 224))
        return cls(sd, depths=depths, num_heads=num_heads, embed_dim=embed_dim, **kw)

    def num_parameters(self) -> int:
        n = sum(t.numel() for t in (self.w_patch, self.b_patch, self.g_embed, self.be_embed, self.g_final, self.b_final,
                                    self.w_cls, self.b_cls))
        for st in self.stages:
            for blk in st["blocks"]:
                n += sum(blk[k].numel() for k in ("wqkv", "bqkv", "wo", "bo", "w1", "b1", "w2", "b2"))
                n += sum(t.numel() for t in blk["ln1"] + blk["ln2"]) + (2 * self.window - 1) ** 2 * st["heads"]
            if st["merge"] is not None:
                n += st["merge"]["w"].numel() + sum(t.numel() for t in st["merge"]["ln"])
        return n

    def train(self, mode: bool = True):
        if mode:
            raise RuntimeError("B200SwinForImageClassification is inference-only")
        return super().train(False)

    def __del__(self):
        try:
            if getattr(self, "_handle", None) is not None and self._handle.value:
                self._lib.evt_swin_destroy(self._handle)
                self._handle = ct.c_void_p()
        except Exception:
            pass

    def launches_per_forward(self) -> int:
        return int(self._lib.evt_swin_launches_per_forward(self._handle))

    # ------------------------------------------------------------------ forward
    def _workspace(self, batch: int) -> torch.Tensor:
        if self._ws is None or batch > self._ws_batch:
            n = ct.c_size_t()
            _lib.check(self._lib.evt_swin_workspace_bytes(self._handle, batch, ct.byref(n)), "swin_workspace_bytes")
            self._ws = torch.empty(n.value, dtype=torch.uint8, device=self._device)
            self._ws_batch = batch
            self._graphs.clear()       # captured graphs hold the old workspace pointer
        return self._ws

    def _run(self, x: torch.Tensor) -> torch.Tensor:
        if self.use_ops:
            return self._run_ops(x)
        B = x.shape[0]
        ws = self._workspace(B)
        logits = torch.empty((B, self.num_labels), dtype=torch.float32, device=x.device)
        _lib.check(self._lib.evt_swin_forward(self._handle, x.data_ptr(), B, logits.data_ptr(), ws.data_ptr(), ws.numel(),
                                              torch.cuda.current_stream().cuda_stream), "swin_forward")
        return logits

    def _run_ops(self, x: torch.Tensor) -> torch.Tensor:
        with ops.static_weights():          # every linear() below multiplies by a weight matrix this module owns
            return self._run_impl(x)

    def _run_impl(self, x: torch.Tensor) -> torch.Tensor:
        B = x.shape[0]
        eps, ws2 = self.eps, self.window * self.window
        cols = ops.im2col_patch(x, self.patch)
        y = ops.linear(cols, self.w_patch, self.b_patch, out_dtype=torch.float32)
        T = (self.image_size // self.patch) ** 2
        resid, _ = ops.gather_layernorm(y, self.idx_embed, self.g_embed, self.be_embed, eps, B, T, T, out_dtype=torch.float32)
        for st in self.stages:
            C, heads, T = st["C"], st["heads"], st["H"] * st["H"]
            for blk in st["blocks"]:
                if blk["idx"] is not None:
                    xn, resid = ops.gather_layernorm(resid, blk["idx"], *blk["ln1"], eps, B, T, T, copy=True)
                else:
                    xn = ops.layernorm(resid, *blk["ln1"], eps)
                qkv = ops.linear(xn, blk["wqkv"], blk["bqkv"])
                ctx = ops.window_attention(qkv, blk["table"], B * T // ws2, heads, ws2, 32)
                ops.linear(ctx, blk["wo"], blk["bo"], residual=resid, out=resid, out_dtype=torch.float32)
                xn = ops.layernorm(resid, *blk["ln2"], eps)
                h = ops.linear(xn, blk["w1"], blk["b1"], act="gelu_erf")
                ops.linear(h, blk["w2"], blk["b2"], residual=resid, out=resid, out_dtype=torch.float32)
            if st["merge"] is not None:
                mg = st["merge"]
                xm, _ = ops.gather_layernorm(resid, mg["idx"], *mg["ln"], eps, B, T, T // 4, G=4)
                resid = ops.linear(xm, mg["w"], None, out_dtype=torch.float32)
        last = self.stages[-1]
        pooled = ops.layernorm_mean_tokens(resid, self.g_final, self.b_final, eps, B, last["H"] * last["H"])
        return ops.linear(pooled, self.w_cls, self.b_cls, out_dtype=torch.float32)

    @torch.no_grad()
    def forward(self, pixel_values: torch.Tensor = None, head_mask=None, labels=None, output_attentions=None,
                output_hidden_states=None, interpolate_pos_encoding=None, return_dict=None) -> ImageClassifierOutput:
        if pixel_values is None:
            raise ValueError("You have to specify pixel_values")
        for name, v in (("head_mask", head_mask), ("labels", labels), ("output_attentions", output_attentions),
                        ("output_hidden_states", output_hidden_states), ("interpolate_pos_encoding", interpolate_pos_encoding)):
            if v is not None and v is not False:
                raise NotImplementedError(f"B200SwinForImageClassification.forward does not support {name}")
        x = pixel_values
        if not x.is_cuda:
            raise RuntimeError("pixel_values must be a CUDA tensor (no CPU fallback); move the batch with .to(device)")
        if x.dim() != 4 or x.shape[1] != 3 or x.shape[2] != self.image_size or x.shape[3] != self.image_size:
            raise ValueError(f"Input image size ({tuple(x.shape[2:])}) doesn't match model ({self.image_size}*{self.image_size}).")
        x = x.float().contiguous()
        outs = []
        with torch.cuda.device(self._device):
            for s in range(0, x.shape[0], self.max_batch):
                outs.append(self._run(x[s:s + self.max_batch]))
        return ImageClassifierOutput(logits=outs[0] if len(outs) == 1 else torch.cat(outs, 0))


def _swin_forward_graphed(self, pixel_values: torch.Tensor) -> ImageClassifierOutput:
    """Same result as forward(); the ~110 launches of one forward are replayed from a CUDA graph (latency path)."""
    if not pixel_values.is_cuda:
        raise RuntimeError("pixel_values must be a CUDA tensor (no CPU fallback)")
    if pixel_values.shape[0] > self.max_batch:
        return self.forward(pixel_values)
    from .graph_util import graphed_call
    with torch.no_grad():
        return ImageClassifierOutput(logits=graphed_call(self._graphs, pixel_values, self._run, self._device))


B200SwinForImageClassification.forward_graphed = _swin_forward_graphed


def microsoft_to_hf(sd: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    """microsoft/Swin-Transformer ``SwinTransformer.state_dict()`` (or its ``{'model': ...}`` checkpoint) -> HF key names."""
    if "model" in sd and isinstance(sd["model"], dict):
        sd = sd["model"]
    out: Dict[str, torch.Tensor] = {}
    top = {"patch_embed.proj.": "swin.embeddings.patch_embeddings.projection.", "patch_embed.norm.": "swin.embeddings.norm.",
           "norm.": "swin.layernorm.", "head.": "classifier."}
    blk = {"norm1.": "layernorm_before.", "norm2.": "layernorm_after.", "attn.proj.": "attention.output.dense.",
           "mlp.fc1.": "intermediate.dense.", "mlp.fc2.": "output.dense.",
           "attn.relative_position_bias_table": "attention.self.relative_position_bias_table"}
    for k, v in sd.items():
        if k.endswith("attn_mask") or k.endswith("relative_position_index"):
            continue                                      # buffers, recomputed here
        for a, b in top.items():
            if k.startswith(a):
                out[b + k[len(a):]] = v
                break
        else:
            if not k.startswith("layers."):
                raise ValueError(f"unexpected key {k!r} in a Swin state dict")
            _, s, kind, rest = k.split(".", 3)
            if kind == "downsample":
                out[f"swin.encoder.layers.{s}.downsample.{rest}"] = v
                continue
            b, rest = rest.split(".", 1)
            p = f"swin.encoder.layers.{s}.blocks.{b}."
            if rest.startswith("attn.qkv."):
                C = v.shape[0] // 3
                for i, n in enumerate(("query", "key", "value")):
                    out[p + f"attention.self.{n}." + rest[len("attn.qkv."):]] = v[i * C:(i + 1) * C].contiguous()
                continue
            for a, bname in blk.items():
                if rest.startswith(a):
                    out[p + bname + rest[len(a):]] = v
                    break
            else:
                raise ValueError(f"unexpected key {k!r} in a Swin state dict")
    return out
