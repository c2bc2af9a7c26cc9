"""Drop-in B200 Swin V2 classifier: the 256-pixel ImageNet-1k checkpoints of microsoft/Swin-Transformer
(``swinv2_{tiny,small,base}_patch4_window{8,16}_256``, ``swinv2_{base,large}_patch4_window12to16_192to256_22kto1k_ft``), the
network of ``transformers.Swinv2ForImageClassification`` (SITE/models/swinv2/modeling_swinv2.py).

The forward is one call into the Swin runtime of libevt (``evt_swin_*`` with ``spec.version = 2``, csrc/swin_model.cu): the
window orders, gathers, continuous-position-bias tables and logit scales are computed there at load, from the weights under
their HF names.  Blocks are post-norm (``x + LN(attn(x))``, ``x + LN(mlp(x))``), attention is cosine attention in 8 x 8 or
16 x 16 windows (``evt_cosine_window_attention_fwd``), patch merging is reduction then LayerNorm.  bf16 GEMM and attention
operands, f32 accumulate / residual / LayerNorm / softmax; there is no tf32 mode for V2.  No CPU fallback.

The shift mask: the installed HF forward adds SW-MSA's -100 mask twice (Swinv2SelfAttention.forward :463-468), the original
code once.  ``from_hf`` reproduces the HF module it is given (mask_adds = 2); ``from_microsoft`` and the factories run the
original arithmetic (1), the one the published checkpoints were trained with, whichever key layout their weights come in.
"""
from __future__ import annotations

import ctypes as ct
import math
import os
from typing import Dict, Sequence

import torch
import torch.nn as nn

from . import _lib
from .modeling_swin import B200SwinConfig, B200SwinForImageClassification

# name -> (embed_dim, depths, heads, window, pretrained_window_sizes); every one at 256 pixels, patch 4, head size 32
SWINV2 = {
    "swinv2_tiny_patch4_window8_256": (96, [2, 2, 6, 2], [3, 6, 12, 24], 8, [0, 0, 0, 0]),
    "swinv2_small_patch4_window8_256": (96, [2, 2, 18, 2], [3, 6, 12, 24], 8, [0, 0, 0, 0]),
    "swinv2_base_patch4_window8_256": (128, [2, 2, 18, 2], [4, 8, 16, 32], 8, [0, 0, 0, 0]),
    "swinv2_tiny_patch4_window16_256": (96, [2, 2, 6, 2], [3, 6, 12, 24], 16, [0, 0, 0, 0]),
    "swinv2_small_patch4_window16_256": (96, [2, 2, 18, 2], [3, 6, 12, 24], 16, [0, 0, 0, 0]),
    "swinv2_base_patch4_window16_256": (128, [2, 2, 18, 2], [4, 8, 16, 32], 16, [0, 0, 0, 0]),
    "swinv2_base_patch4_window12to16_192to256_22kto1k_ft": (128, [2, 2, 18, 2], [4, 8, 16, 32], 16, [12, 12, 12, 6]),
    "swinv2_large_patch4_window12to16_192to256_22kto1k_ft": (192, [2, 2, 18, 2], [6, 12, 24, 48], 16, [12, 12, 12, 6]),
}
SUPPORTED = ("8 x 8 and 16 x 16 windows at head size 32: swinv2_{tiny,small,base}_patch4_window{8,16}_256, "
             "swinv2_{base,large}_patch4_window12to16_192to256_22kto1k_ft")
_BUFFERS = ("relative_coords_table", "relative_position_index", "attn_mask")


def stage_windows(image_size: int, patch: int, window: int, stages: int):
    """[(tokens per side, window)] per stage: the window is min(resolution, window) (Swinv2Layer._compute_window_shift)."""
    H, out = image_size // patch, []
    for _ in range(stages):
        out.append((H, min(H, window)))
        H //= 2
    return out


def check_geometry(image_size: int, patch: int, window: int, embed_dim: int, num_heads: Sequence[int], precision: str = "bf16"):
    """Raise ValueError for what the V2 runtime does not run, before anything is allocated."""
    if precision != "bf16":
        raise ValueError(f"Swin V2 runs in bf16 only; precision {precision!r} (tf32) is not implemented for it")
    if patch != 4 or image_size % patch:
        raise ValueError(f"only patch size 4 is implemented; supported: {SUPPORTED}")
    if any(embed_dim * 2 ** s != 32 * h for s, h in enumerate(num_heads)):
        raise ValueError(f"only head size 32 is implemented; supported: {SUPPORTED}")
    for H, ws in stage_windows(image_size, patch, window, len(num_heads)):
        if ws not in (8, 16) or H % ws:
            raise ValueError(f"a {ws} x {ws} window over {H} x {H} tokens is not implemented; supported: {SUPPORTED}")


class B200Swinv2ForImageClassification(B200SwinForImageClassification):
    """Inference-only.  ``state_dict`` uses HF key names (``swinv2.embeddings...``, ``swinv2.encoder.layers.{s}.blocks.{b}...``,
    ``swinv2.layernorm``, ``classifier``).  ``mask_adds``: how often the -100 shift mask is added to a masked score (2: the
    installed HF forward, 1: microsoft/Swin-Transformer).  forward / forward_graphed / launches_per_forward are those of the
    V1 class, over the same runtime handle."""

    def __init__(self, state_dict: Dict[str, torch.Tensor], depths: Sequence[int], num_heads: Sequence[int], embed_dim: int,
                 window: int = 8, pretrained_window_sizes: Sequence[int] = (0, 0, 0, 0), patch: int = 4, image_size: int = 256,
                 eps: float = 1e-5, mask_adds: int = 1, device="cuda", max_batch: int = 1024, precision: str = "bf16"):
        nn.Module.__init__(self)
        check_geometry(image_size, patch, window, embed_dim, num_heads, precision)
        if len(depths) != len(num_heads) or len(pretrained_window_sizes) != len(depths) or len(depths) > _lib.SWIN_MAX_STAGES:
            raise ValueError("depths, num_heads and pretrained_window_sizes need one entry per stage")
        if mask_adds not in (1, 2):
            raise ValueError("mask_adds must be 1 (microsoft/Swin-Transformer) or 2 (the installed HF forward)")
        dev = torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError("B200Swinv2ForImageClassification runs only on a CUDA (sm_100a) device; no CPU fallback")
        self.depths, self.num_heads, self.embed_dim = list(depths), list(num_heads), embed_dim
        self.window, self.patch, self.image_size, self.eps = window, patch, image_size, eps
        self.pretrained_window_sizes, self.mask_adds = list(pretrained_window_sizes), int(mask_adds)
        self.max_batch, self._device, self.precision = int(max_batch), dev, precision
        self._graphs: dict = {}
        self.use_ops = False            # there is no op-level composition of the V2 forward: the runtime is the only path
        sd = {k: v.detach() for k, v in state_dict.items() if not k.endswith(_BUFFERS)}
        self.num_labels = int(sd["classifier.weight"].shape[0])
        self._n_params = sum(v.numel() for v in sd.values())
        self.config = B200SwinConfig(depths, num_heads, embed_dim, window, patch, image_size, eps, self.num_labels)
        self.config.pretrained_window_sizes = list(pretrained_window_sizes)
        self._param = nn.Parameter(sd["classifier.bias"].to(device=dev, dtype=torch.float32), requires_grad=False)
        self._lib = _lib.load()
        self._handle = ct.c_void_p()
        self._ws, self._ws_batch = None, 0
        spec = _lib.SwinSpec()
        spec.image, spec.patch, spec.window, spec.embed_dim = image_size, patch, window, embed_dim
        spec.stages, spec.num_labels, spec.eps = len(self.depths), self.num_labels, float(eps)
        spec.precision, spec.version, spec.mask_adds = _lib.PREC_BF16, 2, self.mask_adds
        for i, (d, h, pw) in enumerate(zip(self.depths, self.num_heads, self.pretrained_window_sizes)):
            spec.depths[i], spec.heads[i], spec.pretrained_window[i] = int(d), int(h), int(pw)
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

    # ------------------------------------------------------------------ constructors
    @classmethod
    def from_hf(cls, model: nn.Module, **kw):
        """A ``transformers.Swinv2ForImageClassification``; reproduces its forward, including the shift mask added twice."""
        c = model.config
        kw.setdefault("mask_adds", 2)
        return cls(model.state_dict(), depths=c.depths, num_heads=c.num_heads, embed_dim=c.embed_dim, window=c.window_size,
                   pretrained_window_sizes=list(c.pretrained_window_sizes), patch=c.patch_size, image_size=c.image_size,
                   eps=c.layer_norm_eps, **kw)

    @classmethod
    def from_microsoft(cls, state_dict: Dict[str, torch.Tensor], depths, num_heads, embed_dim, window: int,
                       pretrained_window_sizes: Sequence[int] = (0, 0, 0, 0), image_size: int = 256, **kw):
        """State dict of microsoft/Swin-Transformer's ``SwinTransformerV2`` (bare, or its ``{'model': ...}`` checkpoint).  The
        relative_position_index / relative_coords_table buffers it carries are checked against the geometry given here (a
        wrong window or pretrained window size is refused); attn_mask buffers are ignored (recomputed in the runtime)."""
        sd = _unwrap(state_dict)
        verify_microsoft_buffers(sd, image_size, window, pretrained_window_sizes, len(depths))
        return cls(microsoft_to_canonical(sd), depths=depths, num_heads=num_heads, embed_dim=embed_dim, window=window,
                   pretrained_window_sizes=pretrained_window_sizes, image_size=image_size, **kw)

    def num_parameters(self) -> int:
        return self._n_params


def _unwrap(sd):
    if "model" in sd and isinstance(sd["model"], dict):
        sd = sd["model"]
    return sd


def hf_to_canonical(sd: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    """HF ``Swinv2ForImageClassification`` state dict -> the names the runtime loads (the same, without buffers)."""
    return {k: v for k, v in sd.items() if not k.endswith(_BUFFERS)}


def microsoft_to_canonical(sd: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    """microsoft/Swin-Transformer ``SwinTransformerV2.state_dict()`` -> HF ``Swinv2ForImageClassification`` names.  The fused
    ``attn.qkv.weight`` is split; ``attn.q_bias`` / ``attn.v_bias`` become the query / value biases (the key has none)."""
    sd = _unwrap(sd)
    out: Dict[str, torch.Tensor] = {}
    top = {"patch_embed.proj.": "swinv2.embeddings.patch_embeddings.projection.", "patch_embed.norm.": "swinv2.embeddings.norm.",
           "norm.": "swinv2.layernorm.", "head.": "classifier."}
    blk = {"norm1.": "layernorm_before.", "norm2.": "layernorm_after.", "attn.proj.": "attention.output.dense.",
           "mlp.fc1.": "intermediate.dense.", "mlp.fc2.": "output.dense.", "attn.logit_scale": "attention.self.logit_scale",
           "attn.cpb_mlp.": "attention.self.continuous_position_bias_mlp.", "attn.q_bias": "attention.self.query.bias",
           "attn.v_bias": "attention.self.value.bias"}
    for k, v in sd.items():
        if k.endswith(_BUFFERS):
            continue
        for a, b in top.items():
            if k.startswith(a):
                out[b + k[len(a):]] = v
                break
        else:
            if not k.startswith("layers."):
                raise ValueError(f"unexpected key {k!r} in a Swin V2 state dict")
            _, s, kind, rest = k.split(".", 3)
            if kind == "downsample":
                out[f"swinv2.encoder.layers.{s}.downsample.{rest}"] = v
                continue
            b, rest = rest.split(".", 1)
            p = f"swinv2.encoder.layers.{s}.blocks.{b}."
            if rest == "attn.qkv.weight":
                C = v.shape[0] // 3
                for i, n in enumerate(("query", "key", "value")):
                    out[p + f"attention.self.{n}.weight"] = v[i * C:(i + 1) * C].contiguous()
                continue
            for a, bname in blk.items():
                if rest.startswith(a):
                    out[p + bname + rest[len(a):]] = v
                    break
            else:
                raise ValueError(f"unexpected key {k!r} in a Swin V2 state dict")
    return out


def relative_coords_table(ws: int, pws: int) -> torch.Tensor:
    """[1, 2ws-1, 2ws-1, 2] log-spaced CPB input coordinates (Swinv2SelfAttention.create_coords_table_and_index :490-506)."""
    r = torch.arange(-(ws - 1), ws, dtype=torch.float32)
    t = torch.stack(torch.meshgrid([r, r], indexing="ij")).permute(1, 2, 0).contiguous().unsqueeze(0)
    t /= (pws - 1) if pws > 0 else max(ws - 1, 1)
    t *= 8
    return torch.sign(t) * torch.log2(t.abs() + 1.0) / math.log2(8)


def verify_microsoft_buffers(sd, image_size, window, pretrained_window_sizes, stages):
    from .modeling_swin import relative_position_index
    for k, v in sd.items():
        if not (k.endswith("relative_position_index") or k.endswith("relative_coords_table")):
            continue
        s = int(k.split(".")[1])
        if s >= stages:
            raise ValueError(f"{k}: stage {s} does not exist in a {stages}-stage model")
        _, ws = stage_windows(image_size, 4, window, stages)[s]
        if k.endswith("relative_position_index"):
            ok = tuple(v.shape) == (ws * ws, ws * ws) and torch.equal(v.long().cpu(), relative_position_index(ws))
        else:
            want = relative_coords_table(ws, pretrained_window_sizes[s])
            ok = tuple(v.shape) == tuple(want.shape) and torch.allclose(v.float().cpu(), want, atol=1e-5)
        if not ok:
            raise ValueError(f"{k} does not match window {ws} / pretrained window {pretrained_window_sizes[s]} at stage {s}: "
                             f"the checkpoint is not the model named")


def _swinv2_factory(name: str, weights, **kw) -> B200Swinv2ForImageClassification:
    """A Swin V2 checkpoint (file or state dict; microsoft/Swin-Transformer or HF Swinv2ForImageClassification key names) as the
    named model: its shapes must match the name."""
    embed_dim, depths, heads, window, pws = SWINV2[name]
    sd = weights
    if isinstance(sd, (str, os.PathLike)):
        sd = torch.load(sd, map_location="cpu", weights_only=True)
    sd = _unwrap(sd)
    hf = any(k.startswith("swinv2.") for k in sd)
    if not hf:
        verify_microsoft_buffers(sd, 256, window, pws, len(depths))
    can = hf_to_canonical(sd) if hf else microsoft_to_canonical(sd)
    e = can.get("swinv2.embeddings.patch_embeddings.projection.weight")
    got_depths = [len({k.split(".")[5] for k in can if k.startswith(f"swinv2.encoder.layers.{s}.blocks.")}) for s in range(4)]
    got_heads = [can.get(f"swinv2.encoder.layers.{s}.blocks.0.attention.self.logit_scale", torch.empty(0)).numel() for s in range(4)]
    got = (None if e is None else tuple(e.shape), got_depths, got_heads)
    want = ((embed_dim, 3, 4, 4), depths, heads)
    if got != want or any(k.startswith("swinv2.encoder.layers.4.") for k in can):
        raise ValueError(f"the weights are not {name}: patch embedding / blocks per stage / heads per stage {got}, expected {want}")
    kw.setdefault("mask_adds", 1)                     # trained with the mask added once, whatever the key layout
    return B200Swinv2ForImageClassification(can, depths=depths, num_heads=heads, embed_dim=embed_dim, window=window,
                                            pretrained_window_sizes=pws, image_size=256, **kw)


def swinv2_tiny_patch4_window8_256(weights, **kw):
    return _swinv2_factory("swinv2_tiny_patch4_window8_256", weights, **kw)


def swinv2_small_patch4_window8_256(weights, **kw):
    return _swinv2_factory("swinv2_small_patch4_window8_256", weights, **kw)


def swinv2_base_patch4_window8_256(weights, **kw):
    return _swinv2_factory("swinv2_base_patch4_window8_256", weights, **kw)


def swinv2_tiny_patch4_window16_256(weights, **kw):
    return _swinv2_factory("swinv2_tiny_patch4_window16_256", weights, **kw)


def swinv2_small_patch4_window16_256(weights, **kw):
    return _swinv2_factory("swinv2_small_patch4_window16_256", weights, **kw)


def swinv2_base_patch4_window16_256(weights, **kw):
    return _swinv2_factory("swinv2_base_patch4_window16_256", weights, **kw)


def swinv2_base_patch4_window12to16_192to256_22kto1k_ft(weights, **kw):
    return _swinv2_factory("swinv2_base_patch4_window12to16_192to256_22kto1k_ft", weights, **kw)


def swinv2_large_patch4_window12to16_192to256_22kto1k_ft(weights, **kw):
    return _swinv2_factory("swinv2_large_patch4_window12to16_192to256_22kto1k_ft", weights, **kw)
