"""Oracle: the tokens-to-token module of the PyTorch T2T-ViT with ``tokens_type='transformer'`` (yitu-opensource/T2T-ViT,
``models/t2t_vit.py`` ``T2T_module``, ``models/token_transformer.py`` ``Token_transformer`` / ``Attention``), restated
channel-last on the canonical weights the runtime loads (test infrastructure).

PARITY UNPINNED: no copy of the upstream repository and no checkpoint is available; this follows the published code as known.
Readings it rests on (the runtime makes the same ones):

* the token attention's scale is ``dim ** -0.5`` with dim = 147 (stage 1) / 576 (stage 2) -- ``Attention`` takes
  ``head_dim = dim // num_heads`` from the INPUT width, not from in_dim = 64 -- and the factories' ``qk_scale`` does not reach it
  (``T2T_module`` builds its ``Token_transformer`` s without one);
* ``qkv_bias=False``: ``attn.qkv`` has no bias;
* the skip connection of the attention starts from v, not from x (x is 147 / 576 wide, the output 64): ``v + proj(ctx)``;
* ``Mlp(64, 64, 64)`` names ``fc1`` / ``fc2`` and uses ``nn.GELU`` (erf);
* LayerNorm eps 1e-5 (``nn.LayerNorm``'s default) for norm1 and norm2.

Weight names (INTEGRATION.md §3): ``t2t.transformer{1,2}.norm1.{gamma,beta}`` and ``.qkv.kernel`` ([in, 192], rows in
``(kh, kw, c)`` order), ``.attn_output.{kernel,bias}``, ``.norm2.{gamma,beta}``, ``.mlp.fc{1,2}.{kernel,bias}``;
``t2t.project.{kernel,bias}`` as in ``oracle.t2t``.
"""
from __future__ import annotations

import math
from typing import Dict

import torch
import torch.nn.functional as F

from .t2t import unfold_nhwc
from .tf_vit import TF_EPS, dense


def token_transformer(sd: Dict[str, torch.Tensor], p: str, x: torch.Tensor) -> torch.Tensor:
    """Token_transformer.forward on [B, T, in_dim] rows -> [B, T, 64]."""
    in_dim = x.shape[-1]
    x = F.layer_norm(x, (in_dim,), sd[p + ".norm1.gamma"], sd[p + ".norm1.beta"], TF_EPS)
    q, k, v = torch.split(dense(x, sd, p + ".qkv", bias=False), 64, dim=-1)
    attn = torch.softmax((q * in_dim ** -0.5) @ k.transpose(-2, -1), dim=-1)
    y = v + dense(attn @ v, sd, p + ".attn_output")
    z = F.layer_norm(y, (64,), sd[p + ".norm2.gamma"], sd[p + ".norm2.beta"], TF_EPS)
    return y + dense(F.gelu(dense(z, sd, p + ".mlp.fc1")), sd, p + ".mlp.fc2")


def t2t_module(sd: Dict[str, torch.Tensor], x: torch.Tensor) -> torch.Tensor:
    """T2T_module(tokens_type='transformer').forward on NHWC pixels [B, 224, 224, 3] -> [B, 196, D]."""
    B = x.shape[0]
    x = token_transformer(sd, "t2t.transformer1", unfold_nhwc(x, 7, 4, 2))
    hw = int(math.isqrt(x.shape[1]))
    x = token_transformer(sd, "t2t.transformer2", unfold_nhwc(x.reshape(B, hw, hw, -1), 3, 2, 1))
    hw = int(math.isqrt(x.shape[1]))
    return dense(unfold_nhwc(x.reshape(B, hw, hw, -1), 3, 2, 1), sd, "t2t.project")
