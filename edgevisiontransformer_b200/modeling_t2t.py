"""B200 T2T-ViT (tokens-to-token + transformer), the reference's ``modeling/models/t2t_vit.py`` (TensorFlow).

Input is NHWC ``[B,224,224,3]`` as in the reference (t2t_vit.py:65).  Weight names follow the flat scheme documented in
INTEGRATION.md (one entry per Keras variable; Dense kernels ``[in, out]``).  The tokens-to-token module runs as

    unfold(7,4,2)+LN -> kqv GEMM -> performer -> attn_output GEMM (+v) -> LN -> MLP GEMMs (+skip)   [T=3136, 147->64]
    unfold(3,2,1)+LN -> ... same ...                                                                 [T= 784, 576->64]
    unfold(3,2,1)    -> the [B*196, 576] matrix that is the A operand of the ``project`` GEMM

and the rest (project + cls + sinusoid position table + 14 TF-dialect encoder blocks + LN + classifier) is the
model-level C entry point ``evt_model_forward_embedded``.

``B200T2TViTTorch`` and ``t2t_vit_{7,10,12,14,19,24}`` run the published PyTorch checkpoints (yitu-opensource/T2T-ViT,
``tokens_type='performer'``; the files the reference's tools.py:347-365 loads): NCHW f32 / bf16 / uint8 pixels, the same
front-end kernels with the stage-1 soft split reading planar pixels (``spec.t2t = 2``), erf-GELU performers and a pre-LN
(HF-dialect) encoder.  Weights go through ``dialects.t2t_torch_to_canonical``.  The same class and ``t2t_vit_t_{14,19,24}`` run
the ``tokens_type='transformer'`` checkpoints (``spec.t2t = 3``): each token stage is a one-head ``Token_transformer`` whose exact
softmax attention runs over all 3136 (stage 1) or 784 (stage 2) tokens of an image.
"""
from __future__ import annotations

import argparse
import os
from typing import Dict, List, Optional

import torch
import torch.nn as nn

from . import ops
from .dialects import T2T_TORCH_HEAD_SIZE, _encoder_to_canonical, t2t_torch_to_canonical, unwrap_checkpoint
from .modeling_vit import B200ViTForImageClassification, ImageClassifierOutput, config_from_state_dict

TF_EPS = 1e-5


def _pad_cols(w: torch.Tensor, mult: int = 8) -> torch.Tensor:
    n, k = w.shape
    ld = (k + mult - 1) // mult * mult
    if ld == k:
        return w.contiguous()
    out = torch.zeros((n, ld), dtype=w.dtype, device=w.device)
    out[:, :k] = w
    return out


class _Performer:
    """Device-side weights of one TokenPerformer (transformer_encoder.py:39-65)."""

    def __init__(self, sd: Dict[str, torch.Tensor], p: str, dev):
        f32 = lambda t: t.detach().to(dev, torch.float32).contiguous()      # noqa: E731
        bf = lambda t: _pad_cols(t.detach().to(dev, torch.float32).t().contiguous()).to(torch.bfloat16)   # noqa: E731
        self.in_dim = sd[p + ".kqv.kernel"].shape[0]
        self.g1, self.b1 = f32(sd[p + ".norm1.gamma"]), f32(sd[p + ".norm1.beta"])
        self.wkqv, self.bkqv = bf(sd[p + ".kqv.kernel"]), f32(sd[p + ".kqv.bias"])
        self.w = f32(sd[p + ".w"])
        self.wo, self.bo = bf(sd[p + ".attn_output.kernel"]), f32(sd[p + ".attn_output.bias"])
        self.g2, self.b2 = f32(sd[p + ".norm2.gamma"]), f32(sd[p + ".norm2.beta"])
        self.w1, self.bb1 = bf(sd[p + ".mlp.fc1.kernel"]), f32(sd[p + ".mlp.fc1.bias"])
        self.w2, self.bb2 = bf(sd[p + ".mlp.fc2.kernel"]), f32(sd[p + ".mlp.fc2.bias"])

    def __call__(self, x_nhwc: torch.Tensor, k: int, s: int, p: int) -> torch.Tensor:
        B, H, W, _ = x_nhwc.shape
        oh, ow = (H + 2 * p - k) // s + 1, (W + 2 * p - k) // s + 1
        T = oh * ow
        X = ops.unfold_ln_nhwc(x_nhwc, k, s, p, self.g1, self.b1, TF_EPS, ld=self.wkqv.shape[1])
        kqv = ops.linear(X, self.wkqv, self.bkqv, k=self.in_dim)                    # bf16 [B*T, 192]
        yattn, y = ops.performer(kqv, self.w, B, T)                                  # y = v (f32)
        # y = v + attn_output(.) ; y += mlp(LN(y))   (transformer_encoder.py:93-99), one kernel
        ops.performer_mlp(yattn, y, self.wo, self.bo, self.g2, self.b2, self.w1, self.bb1, self.w2, self.bb2, TF_EPS)
        return y.view(B, oh, ow, 64)


class B200T2TViT(nn.Module):
    """get_t2t_vit_{7,10,12,14} (t2t_vit.py:138-148) on libevt.  ``sd`` uses the oracle / INTEGRATION.md naming."""

    def __init__(self, sd: Dict[str, torch.Tensor], depth: int, num_heads: int, device="cuda", max_batch: int = 1024,
                 precision: str = "bf16"):
        super().__init__()
        dev = torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError("B200T2TViT runs only on a CUDA (sm_100a) device; no CPU fallback")
        if precision != "bf16":
            raise NotImplementedError("the T2T front-end is implemented for the bf16 mode")
        D = sd["cls_tokens"].shape[-1]
        self.hidden, self.depth, self.num_heads = D, depth, num_heads
        self.max_batch = int(max_batch)
        self._dev = dev
        self.p1 = _Performer(sd, "t2t.performer1", dev)
        self.p2 = _Performer(sd, "t2t.performer2", dev)
        heads: List[int] = [num_heads] * depth
        c: Dict[str, torch.Tensor] = {}
        c["vit.embeddings.patch_embeddings.projection.weight"] = sd["t2t.project.kernel"].t().contiguous()   # [D, 576]
        c["vit.embeddings.patch_embeddings.projection.bias"] = sd["t2t.project.bias"]
        c["vit.embeddings.cls_token"] = sd["cls_tokens"].reshape(1, 1, D)
        c["vit.embeddings.position_embeddings"] = sd["pos_embedding"].reshape(1, -1, D)
        _encoder_to_canonical(sd, c, heads, D // num_heads)
        c["vit.layernorm.weight"], c["vit.layernorm.bias"] = sd["norm.gamma"], sd["norm.beta"]
        c["classifier.weight"] = sd["classifier_head.kernel"].t().contiguous()
        c["classifier.bias"] = sd["classifier_head.bias"]
        # The tokens-to-token module runs inside the library too (evt_model_forward with spec.t2t = 1: soft splits, the two
        # TokenPerformers and the project GEMM are part of the C++ launch sequence); its Keras variables go in under their own
        # names.  `tokens()` below keeps an op-level composition of the same module for tests that look at the tokens.
        for k, v in sd.items():
            if k.startswith("t2t.performer"):
                c[k] = v
        self.core = B200ViTForImageClassification.from_state_dict(
            c, device=dev, max_batch=max_batch, dialect="tf", hidden_act="gelu_tanh", layer_norm_eps=TF_EPS, final_ln=True,
            head_size=D // num_heads, embed_k=sd["t2t.project.kernel"].shape[0], precision=precision, t2t=True)
        self.config = self.core.config
        self._graphs: dict = {}
        # The graphs captured by forward_graphed bake in the core's activation workspace pointer: drop them whenever the core
        # reallocates it (a larger batch arrived), or a replay would write into memory already returned to the allocator.
        self.core.on_workspace_realloc(self._graphs.clear)
        self.eval()

    @torch.no_grad()
    def tokens(self, x: torch.Tensor) -> torch.Tensor:
        """tokens-to-token module up to (not including) ``project``: bf16 [B*196, 576]."""
        with ops.static_weights():       # the performers' linear() calls multiply by weights this module owns
            y = self.p1(x, 7, 4, 2)          # [B,56,56,64] f32
            y = self.p2(y, 3, 2, 1)          # [B,28,28,64] f32
        return ops.unfold_ln_nhwc(y, 3, 2, 1)

    @torch.no_grad()
    def forward(self, x: torch.Tensor) -> ImageClassifierOutput:
        if not x.is_cuda:
            raise RuntimeError("input must be a CUDA tensor (no CPU fallback)")
        if x.dim() != 4 or x.shape[-1] != 3:
            raise ValueError("T2T-ViT takes channel-last images [B, H, W, 3] (t2t_vit.py:65)")
        x = x.float().contiguous()
        return ImageClassifierOutput(logits=self._forward_core(x))

    def _forward_core(self, x: torch.Tensor) -> torch.Tensor:
        """One C call per chunk: front-end + encoder + head (evt_model_forward on NHWC f32 pixels)."""
        c = self.config
        if x.shape[1] != c.image_size or x.shape[2] != c.image_size:
            raise ValueError(f"Input image size ({tuple(x.shape[1:3])}) doesn't match model ({c.image_size}*{c.image_size}).")
        logits = torch.empty((x.shape[0], c.num_labels), dtype=torch.float32, device=x.device)
        with torch.cuda.device(self._dev):
            for s in range(0, x.shape[0], self.max_batch):
                self.core._run(x[s:s + self.max_batch], logits[s:s + self.max_batch])
        return logits

    @torch.no_grad()
    def forward_graphed(self, x: torch.Tensor) -> ImageClassifierOutput:
        """Same result as forward(); front-end and encoder launches replayed from one CUDA graph (latency path)."""
        if not x.is_cuda:
            raise RuntimeError("input must be a CUDA tensor (no CPU fallback)")
        if x.shape[0] > self.max_batch:
            return self.forward(x)
        from .graph_util import graphed_call
        return ImageClassifierOutput(logits=graphed_call(self._graphs, x.float(), self._forward_core, self._dev))

    def launches_per_forward(self) -> int:
        return self.core.launches_per_forward()


def get_t2t_vit_14(sd, **kw):
    return B200T2TViT(sd, depth=14, num_heads=6, **kw)


def get_t2t_vit_12(sd, **kw):
    return B200T2TViT(sd, depth=12, num_heads=4, **kw)


def get_t2t_vit_10(sd, **kw):
    return B200T2TViT(sd, depth=10, num_heads=4, **kw)


def get_t2t_vit_7(sd, **kw):
    return B200T2TViT(sd, depth=7, num_heads=4, **kw)


# ---------------------------------------------------------------------------------------------- PyTorch T2T-ViT checkpoints
# upstream factories (models/t2t_vit.py): embed_dim, depth, num_heads, mlp_ratio; t2t_vit_t_* are tokens_type='transformer'
T2T_TORCH = {"t2t_vit_7": (256, 7, 4, 2.0), "t2t_vit_10": (256, 10, 4, 2.0), "t2t_vit_12": (256, 12, 4, 2.0),
             "t2t_vit_14": (384, 14, 6, 3.0), "t2t_vit_19": (448, 19, 7, 3.0), "t2t_vit_24": (512, 24, 8, 3.0),
             "t2t_vit_t_14": (384, 14, 6, 3.0), "t2t_vit_t_19": (448, 19, 7, 3.0), "t2t_vit_t_24": (512, 24, 8, 3.0)}


def tokens_type_of(sd: Dict[str, torch.Tensor]) -> str:
    """'transformer' for a state dict with Token_transformer stages (tokens_to_token.attention1.attn.qkv), else 'performer'."""
    return "transformer" if "tokens_to_token.attention1.attn.qkv.weight" in sd else "performer"


def load_t2t_checkpoint(path) -> dict:
    """``torch.load`` of a T2T-ViT ``.pth`` / ``.pth.tar`` with ``weights_only=True``.  timm's checkpoint saver, which wrote the
    published files, stores the training ``argparse.Namespace`` under ``args``: that one class is allow-listed."""
    with torch.serialization.safe_globals([argparse.Namespace]):
        return torch.load(os.fspath(path), map_location="cpu", weights_only=True)


class B200T2TViTTorch(B200ViTForImageClassification):
    """PyTorch ``T2T_ViT`` (``tokens_type='performer'`` or ``'transformer'``, detected from the keys; ``tokens_type`` says which)
    on libevt: the whole forward, front-end included, is one C call per chunk.  Input is NCHW ``[B, 3, 224, 224]`` in f32, bf16 or uint8 (uint8 is normalised with ``pixel_mean`` / ``pixel_std``
    inside the first soft split; the zero padding applies to the normalised image, as upstream pads the normalised tensor).

    ``checkpoint_or_sd``: a file path, a checkpoint dict (``state_dict_ema`` -- used unless ``use_ema=False`` --,
    ``state_dict`` or ``model``) or a flat state dict.  Depth and embed_dim come from the weights; ``num_heads`` defaults to
    embed_dim / 64 (the head size of every published config).  ``qk_scale`` defaults to head_dim ** -0.5 as upstream's class
    does; the ``t2t_vit_*`` factories default it to embed_dim ** -0.5, as upstream's do for ``pretrained=True``."""

    def __init__(self, checkpoint_or_sd, num_heads: Optional[int] = None, qk_scale: Optional[float] = None, device="cuda",
                 max_batch: int = 1024, precision: str = "bf16", image_size: int = 224, use_ema: bool = True, keep_params: bool = True):
        if precision != "bf16":
            raise NotImplementedError("the T2T front-end is implemented for the bf16 mode")
        if image_size != 224:
            raise ValueError(f"image_size {image_size}: only the 224-pixel T2T-ViT is supported")
        sd = load_t2t_checkpoint(checkpoint_or_sd) if isinstance(checkpoint_or_sd, (str, os.PathLike)) else checkpoint_or_sd
        csd, kw = t2t_torch_to_canonical(sd, qk_scale=qk_scale, use_ema=use_ema)
        D = csd["vit.embeddings.cls_token"].shape[-1]
        nh = D // T2T_TORCH_HEAD_SIZE if num_heads is None else int(num_heads)
        if nh <= 0 or D % nh or D // nh != T2T_TORCH_HEAD_SIZE:
            raise ValueError(f"embed_dim {D} with num_heads {nh} gives head size {D / max(nh, 1):g}; only head size "
                             f"{T2T_TORCH_HEAD_SIZE} is implemented")
        super().__init__(config_from_state_dict(csd, **kw), csd, device=device, max_batch=max_batch, keep_params=keep_params)
        self.num_heads, self.depth, self.hidden = nh, self.config.num_hidden_layers, D
        self.tokens_type = "transformer" if kw["t2t"] == 3 else "performer"

    @classmethod
    def from_checkpoint(cls, path, **kw) -> "B200T2TViTTorch":
        """A published checkpoint file: the factory of its embed_dim (and depth) supplies the defaults."""
        sd = unwrap_checkpoint(load_t2t_checkpoint(path), kw.get("use_ema", True))
        name = _factory_of(sd)
        if name is None and kw.get("qk_scale") is None:
            raise ValueError("checkpoint shape matches no published t2t_vit_* config; pass qk_scale= explicitly")
        return globals()[name](sd, **kw) if name is not None else cls(sd, **kw)


def _factory_of(sd: Dict[str, torch.Tensor]) -> Optional[str]:
    if "cls_token" not in sd:
        return None
    D, depth = sd["cls_token"].shape[-1], 0
    while f"blocks.{depth}.attn.qkv.weight" in sd:
        depth += 1
    tt = tokens_type_of(sd) == "transformer"
    by_dim = [name for name, (d, _, _, _) in T2T_TORCH.items()              # same heads, mlp ratio and qk_scale for one D
              if d == D and ("_t_" in name) == tt]
    exact = [name for name in by_dim if T2T_TORCH[name][1] == depth]
    return (exact or by_dim or [None])[0]


def _t2t_factory(name: str, checkpoint_or_sd, **kw) -> B200T2TViTTorch:
    D, _, heads, ratio = T2T_TORCH[name]     # depth comes from the weights
    sd = load_t2t_checkpoint(checkpoint_or_sd) if isinstance(checkpoint_or_sd, (str, os.PathLike)) else checkpoint_or_sd
    sd = unwrap_checkpoint(sd, kw.get("use_ema", True))
    want_tt = "transformer" if "_t_" in name else "performer"
    if tokens_type_of(sd) != want_tt:
        raise ValueError(f"{name} is a tokens_type='{want_tt}' T2T-ViT; the weights are tokens_type='{tokens_type_of(sd)}' "
                         f"({'t2t_vit_t_*' if want_tt == 'performer' else 't2t_vit_*'} runs them)")
    if "cls_token" in sd and "blocks.0.mlp.fc1.weight" in sd:
        got = (sd["cls_token"].shape[-1], sd["blocks.0.mlp.fc1.weight"].shape[0])
        if got != (D, int(D * ratio)):
            raise ValueError(f"{name} is embed_dim {D} with an MLP of {int(D * ratio)}; the weights have {got[0]} and {got[1]}")
    kw.setdefault("num_heads", heads)
    kw.setdefault("qk_scale", D ** -0.5)           # upstream's t2t_vit_* with pretrained=True
    return B200T2TViTTorch(sd, **kw)


def t2t_vit_7(checkpoint_or_sd, **kw):
    return _t2t_factory("t2t_vit_7", checkpoint_or_sd, **kw)


def t2t_vit_10(checkpoint_or_sd, **kw):
    return _t2t_factory("t2t_vit_10", checkpoint_or_sd, **kw)


def t2t_vit_12(checkpoint_or_sd, **kw):
    return _t2t_factory("t2t_vit_12", checkpoint_or_sd, **kw)


def t2t_vit_14(checkpoint_or_sd, **kw):
    return _t2t_factory("t2t_vit_14", checkpoint_or_sd, **kw)


def t2t_vit_19(checkpoint_or_sd, **kw):
    return _t2t_factory("t2t_vit_19", checkpoint_or_sd, **kw)


def t2t_vit_24(checkpoint_or_sd, **kw):
    return _t2t_factory("t2t_vit_24", checkpoint_or_sd, **kw)


def t2t_vit_t_14(checkpoint_or_sd, **kw):
    return _t2t_factory("t2t_vit_t_14", checkpoint_or_sd, **kw)


def t2t_vit_t_19(checkpoint_or_sd, **kw):
    return _t2t_factory("t2t_vit_t_19", checkpoint_or_sd, **kw)


def t2t_vit_t_24(checkpoint_or_sd, **kw):
    return _t2t_factory("t2t_vit_t_24", checkpoint_or_sd, **kw)
