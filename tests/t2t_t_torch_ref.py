"""The PyTorch T2T-ViT with ``tokens_type='transformer'`` (yitu-opensource/T2T-ViT ``t2t_vit_t_{14,19,24}``) restated as
``nn.Module`` s with upstream's ``state_dict()`` keys: the reference ``modeling_t2t.t2t_vit_t_*`` is tested against.  Test
infrastructure; the product never imports it.  The encoder, head and stress init are ``t2t_torch_ref`` 's.

PARITY UNPINNED, as for the performer models: there is no copy of the upstream repository and no checkpoint here.  This follows
``models/token_transformer.py`` (``Attention``, ``Token_transformer``) and ``models/t2t_vit.py`` (``T2T_module`` with
``tokens_type='transformer'``, the ``t2t_vit_t_*`` factories) as published.  Readings that cannot be checked offline:

* the token attention's scale is ``dim ** -0.5`` with dim = 147 / 576 (head_dim = dim // num_heads of the INPUT width), not
  64 ** -0.5, and the factories' ``qk_scale`` does not reach it;
* ``qkv_bias=False`` in the token transformers;
* the attention's skip connection is ``v + proj(ctx)`` (v squeezed from the one head), not ``x + ...``;
* ``Mlp`` names ``fc1`` / ``fc2`` and uses ``nn.GELU`` (erf); mlp_ratio 1.0;
* LayerNorm eps 1e-5 (``nn.LayerNorm`` 's default).
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn

import t2t_torch_ref as ref

# name -> (embed_dim, depth, num_heads, mlp_ratio), models/t2t_vit.py
CONFIGS = {"t2t_vit_t_14": (384, 14, 6, 3.0), "t2t_vit_t_19": (448, 19, 7, 3.0), "t2t_vit_t_24": (512, 24, 8, 3.0)}


class TokenAttention(nn.Module):
    """models/token_transformer.py ``Attention`` (num_heads = 1 as T2T_module builds it)."""

    def __init__(self, dim, in_dim, num_heads=1, qkv_bias=False, qk_scale=None):
        super().__init__()
        self.num_heads = num_heads
        self.in_dim = in_dim
        head_dim = dim // num_heads
        self.scale = qk_scale or head_dim ** -0.5
        self.qkv = nn.Linear(dim, in_dim * 3, bias=qkv_bias)
        self.proj = nn.Linear(in_dim, in_dim)

    def forward(self, x):
        B, N, C = x.shape
        qkv = self.qkv(x).reshape(B, N, 3, self.num_heads, self.in_dim).permute(2, 0, 3, 1, 4)
        q, k, v = qkv[0], qkv[1], qkv[2]
        attn = ((q * self.scale) @ k.transpose(-2, -1)).softmax(dim=-1)
        x = self.proj((attn @ v).transpose(1, 2).reshape(B, N, self.in_dim))
        return v.squeeze(1) + x


class Token_transformer(nn.Module):
    def __init__(self, dim, in_dim, num_heads=1, mlp_ratio=1.0, qkv_bias=False, qk_scale=None):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim)
        self.attn = TokenAttention(dim, in_dim=in_dim, num_heads=num_heads, qkv_bias=qkv_bias, qk_scale=qk_scale)
        self.norm2 = nn.LayerNorm(in_dim)
        self.mlp = ref.Mlp(in_dim, int(in_dim * mlp_ratio))

    def forward(self, x):
        x = self.attn(self.norm1(x))
        return x + self.mlp(self.norm2(x))


class T2T_module(nn.Module):
    """T2T_module(tokens_type='transformer')."""

    def __init__(self, img_size=224, in_chans=3, embed_dim=768, token_dim=64):
        super().__init__()
        self.soft_split0 = nn.Unfold(kernel_size=(7, 7), stride=(4, 4), padding=(2, 2))
        self.soft_split1 = nn.Unfold(kernel_size=(3, 3), stride=(2, 2), padding=(1, 1))
        self.soft_split2 = nn.Unfold(kernel_size=(3, 3), stride=(2, 2), padding=(1, 1))
        self.attention1 = Token_transformer(dim=in_chans * 7 * 7, in_dim=token_dim, num_heads=1, mlp_ratio=1.0)
        self.attention2 = Token_transformer(dim=token_dim * 3 * 3, in_dim=token_dim, num_heads=1, mlp_ratio=1.0)
        self.project = nn.Linear(token_dim * 3 * 3, embed_dim)
        self.num_patches = (img_size // (4 * 2 * 2)) * (img_size // (4 * 2 * 2))

    def forward(self, x):
        x = self.attention1(self.soft_split0(x).transpose(1, 2))
        B, new_HW, C = x.shape
        x = x.transpose(1, 2).reshape(B, C, int(math.isqrt(new_HW)), int(math.isqrt(new_HW)))
        x = self.attention2(self.soft_split1(x).transpose(1, 2))
        B, new_HW, C = x.shape
        x = x.transpose(1, 2).reshape(B, C, int(math.isqrt(new_HW)), int(math.isqrt(new_HW)))
        return self.project(self.soft_split2(x).transpose(1, 2))


class T2T_ViT(ref.T2T_ViT):
    """T2T_ViT(tokens_type='transformer'): the performer model's encoder and head around the transformer token module."""

    def __init__(self, img_size=224, in_chans=3, embed_dim=768, token_dim=64, **kw):
        super().__init__(img_size=img_size, in_chans=in_chans, embed_dim=embed_dim, token_dim=token_dim, **kw)
        self.tokens_to_token = T2T_module(img_size=img_size, in_chans=in_chans, embed_dim=embed_dim, token_dim=token_dim)


def t2t_vit_t(name: str, depth=None, qk_scale="factory", **kw) -> T2T_ViT:
    """Upstream factory ``name`` (optionally at reduced ``depth``).  qk_scale="factory": embed_dim ** -0.5 in the encoder
    blocks, as the factories set it for the published weights; the token transformers keep in_dim ** -0.5 either way."""
    D, L, heads, ratio = CONFIGS[name]
    scale = D ** -0.5 if qk_scale == "factory" else qk_scale
    return T2T_ViT(embed_dim=D, depth=L if depth is None else depth, num_heads=heads, mlp_ratio=ratio, qk_scale=scale, **kw).eval()


def stress_model(name: str, depth=None, seed: int = 0, **kw) -> T2T_ViT:
    torch.manual_seed(seed)
    return ref.stress_init_(t2t_vit_t(name, depth=depth, **kw), seed=seed)
