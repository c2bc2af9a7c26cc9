"""The PyTorch T2T-ViT (yitu-opensource/T2T-ViT, ``tokens_type='performer'``) restated as ``nn.Module`` s: the reference that
``modeling_t2t.B200T2TViTTorch`` is tested and benchmarked against.  Test infrastructure; the product never imports it.

PARITY UNPINNED: there is no copy of the upstream repository here and no checkpoint to compare with.  This follows the
published code as known -- ``models/t2t_vit.py`` (``T2T_module``, ``T2T_ViT``, ``get_sinusoid_encoding``, the ``t2t_vit_*``
factories), ``models/token_performer.py`` (``Token_performer``) and ``models/transformer_block.py`` (``Mlp``, ``Attention``,
``Block``).  ``state_dict()`` keys and shapes are upstream's.  Points that cannot be checked offline:

* softmax scale: the class defaults ``qk_scale`` to head_dim ** -0.5; the published factories built with ``pretrained=True``
  set embed_dim ** -0.5.  ``t2t_vit(name, ...)`` below follows the factories; both take ``qk_scale=``.
* LayerNorm eps 1e-5 everywhere (``nn.LayerNorm`` defaults, performers and blocks).
* ``nn.GELU`` (erf) in the performer MLP and the blocks; the performer divides by ``D + 1e-8``, uses m = 32 random features,
  and stores ``w`` already multiplied by sqrt(m).

Upstream's ``prm_exp`` / ``single_attn`` cast to float32 (``x.float()``); here the module's own dtype is kept so that a float64
copy is an exact reference (in float32 the two are the same).  ``gelu="tanh"`` swaps the performers' GELU for the tanh form:
only so that ``T2T_module`` can be compared with the TensorFlow restatement ``oracle.t2t.t2t_module``.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn

from oracle.t2t import sinusoid_table

# name -> (embed_dim, depth, num_heads, mlp_ratio), models/t2t_vit.py
CONFIGS = {"t2t_vit_7": (256, 7, 4, 2.0), "t2t_vit_10": (256, 10, 4, 2.0), "t2t_vit_12": (256, 12, 4, 2.0),
           "t2t_vit_14": (384, 14, 6, 3.0), "t2t_vit_19": (448, 19, 7, 3.0), "t2t_vit_24": (512, 24, 8, 3.0)}


class Token_performer(nn.Module):
    def __init__(self, dim, in_dim, head_cnt=1, kernel_ratio=0.5, gelu="erf"):
        super().__init__()
        self.emb = in_dim * head_cnt
        self.kqv = nn.Linear(dim, 3 * self.emb)
        self.proj = nn.Linear(self.emb, self.emb)
        self.head_cnt = head_cnt
        self.norm1 = nn.LayerNorm(dim)
        self.norm2 = nn.LayerNorm(self.emb)
        self.epsilon = 1e-8
        self.mlp = nn.Sequential(nn.Linear(self.emb, self.emb), nn.GELU(approximate="tanh" if gelu == "tanh" else "none"),
                                 nn.Linear(self.emb, self.emb), nn.Dropout(0.0))
        self.m = int(self.emb * kernel_ratio)
        self.w = nn.Parameter(nn.init.orthogonal_(torch.randn(self.m, self.emb)) * math.sqrt(self.m), requires_grad=False)

    def prm_exp(self, x):
        xd = ((x * x).sum(dim=-1, keepdim=True)).repeat(1, 1, self.m) / 2
        wtx = torch.einsum("bti,mi->btm", x, self.w)
        return torch.exp(wtx - xd) / math.sqrt(self.m)

    def single_attn(self, x):
        k, q, v = torch.split(self.kqv(x), self.emb, dim=-1)
        kp, qp = self.prm_exp(k), self.prm_exp(q)
        D = torch.einsum("bti,bi->bt", qp, kp.sum(dim=1)).unsqueeze(dim=2)
        kptv = torch.einsum("bin,bim->bnm", v, kp)
        y = torch.einsum("bti,bni->btn", qp, kptv) / (D.repeat(1, 1, self.emb) + self.epsilon)
        return v + self.proj(y)

    def forward(self, x):
        x = self.single_attn(self.norm1(x))
        return x + self.mlp(self.norm2(x))


class T2T_module(nn.Module):
    def __init__(self, img_size=224, in_chans=3, embed_dim=768, token_dim=64, gelu="erf"):
        super().__init__()
        self.soft_split0 = nn.Unfold(kernel_size=(7, 7), stride=(4, 4), padding=(2, 2))
        self.soft_split1 = nn.Unfold(kernel_size=(3, 3), stride=(2, 2), padding=(1, 1))
        self.soft_split2 = nn.Unfold(kernel_size=(3, 3), stride=(2, 2), padding=(1, 1))
        self.attention1 = Token_performer(dim=in_chans * 7 * 7, in_dim=token_dim, kernel_ratio=0.5, gelu=gelu)
        self.attention2 = Token_performer(dim=token_dim * 3 * 3, in_dim=token_dim, kernel_ratio=0.5, gelu=gelu)
        self.project = nn.Linear(token_dim * 3 * 3, embed_dim)
        self.num_patches = (img_size // (4 * 2 * 2)) * (img_size // (4 * 2 * 2))

    def forward(self, x):
        x = self.soft_split0(x).transpose(1, 2)
        x = self.attention1(x)
        B, new_HW, C = x.shape
        x = x.transpose(1, 2).reshape(B, C, int(math.isqrt(new_HW)), int(math.isqrt(new_HW)))
        x = self.soft_split1(x).transpose(1, 2)
        x = self.attention2(x)
        B, new_HW, C = x.shape
        x = x.transpose(1, 2).reshape(B, C, int(math.isqrt(new_HW)), int(math.isqrt(new_HW)))
        x = self.soft_split2(x).transpose(1, 2)
        return self.project(x)


class Mlp(nn.Module):
    def __init__(self, in_features, hidden_features):
        super().__init__()
        self.fc1 = nn.Linear(in_features, hidden_features)
        self.act = nn.GELU()
        self.fc2 = nn.Linear(hidden_features, in_features)

    def forward(self, x):
        return self.fc2(self.act(self.fc1(x)))


class Attention(nn.Module):
    def __init__(self, dim, num_heads=8, qkv_bias=False, qk_scale=None):
        super().__init__()
        self.num_heads = num_heads
        head_dim = dim // num_heads
        self.scale = qk_scale or head_dim ** -0.5
        self.qkv = nn.Linear(dim, dim * 3, bias=qkv_bias)
        self.proj = nn.Linear(dim, dim)

    def forward(self, x):
        B, N, C = x.shape
        qkv = self.qkv(x).reshape(B, N, 3, self.num_heads, C // self.num_heads).permute(2, 0, 3, 1, 4)
        q, k, v = qkv[0], qkv[1], qkv[2]
        attn = ((q @ k.transpose(-2, -1)) * self.scale).softmax(dim=-1)
        return self.proj((attn @ v).transpose(1, 2).reshape(B, N, C))


class Block(nn.Module):
    def __init__(self, dim, num_heads, mlp_ratio=4.0, qkv_bias=False, qk_scale=None):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim)
        self.attn = Attention(dim, num_heads=num_heads, qkv_bias=qkv_bias, qk_scale=qk_scale)
        self.norm2 = nn.LayerNorm(dim)
        self.mlp = Mlp(dim, int(dim * mlp_ratio))

    def forward(self, x):
        x = x + self.attn(self.norm1(x))
        return x + self.mlp(self.norm2(x))


class T2T_ViT(nn.Module):
    def __init__(self, img_size=224, in_chans=3, num_classes=1000, embed_dim=768, depth=12, num_heads=12, mlp_ratio=4.0,
                 qkv_bias=False, qk_scale=None, token_dim=64, gelu="erf"):
        super().__init__()
        self.tokens_to_token = T2T_module(img_size=img_size, in_chans=in_chans, embed_dim=embed_dim, token_dim=token_dim, gelu=gelu)
        num_patches = self.tokens_to_token.num_patches
        self.cls_token = nn.Parameter(torch.zeros(1, 1, embed_dim))
        self.pos_embed = nn.Parameter(sinusoid_table(num_patches + 1, embed_dim).unsqueeze(0), requires_grad=False)
        self.blocks = nn.ModuleList([Block(embed_dim, num_heads, mlp_ratio, qkv_bias, qk_scale) for _ in range(depth)])
        self.norm = nn.LayerNorm(embed_dim)
        self.head = nn.Linear(embed_dim, num_classes)

    def forward(self, x):
        x = self.tokens_to_token(x)
        x = torch.cat((self.cls_token.expand(x.shape[0], -1, -1), x), dim=1) + self.pos_embed
        for blk in self.blocks:
            x = blk(x)
        return self.head(self.norm(x)[:, 0])


def t2t_vit(name: str, depth=None, qk_scale="factory", **kw) -> T2T_ViT:
    """Upstream factory ``name`` (optionally at reduced ``depth``).  qk_scale="factory": embed_dim ** -0.5, as the
    factories set it for the published weights; None: the class default head_dim ** -0.5."""
    D, L, heads, ratio = CONFIGS[name]
    scale = D ** -0.5 if qk_scale == "factory" else qk_scale
    return T2T_ViT(embed_dim=D, depth=L if depth is None else depth, num_heads=heads, mlp_ratio=ratio, qk_scale=scale, **kw).eval()


@torch.no_grad()
def stress_init_(model: nn.Module, seed: int = 0) -> nn.Module:
    """Seeded weights a wrong layout cannot pass: Glorot-normal Linear weights, non-zero biases, LayerNorm affine away from
    (1, 0) -- the performers' norm1, whose rows the converter permutes, strongly so and asymmetrically --, orthogonal w times
    sqrt(m), a random cls token.  pos_embed keeps the sinusoid table (upstream stores it in the checkpoint)."""
    g = torch.Generator().manual_seed(seed)
    rn = lambda *s: torch.randn(*s, generator=g)       # noqa: E731
    for name, mod in model.named_modules():
        if isinstance(mod, nn.Linear):
            fan_out, fan_in = mod.weight.shape
            mod.weight.copy_(rn(fan_out, fan_in) * math.sqrt(2.0 / (fan_in + fan_out)))
            if mod.bias is not None:
                mod.bias.copy_(rn(fan_out) * 0.1)
        elif isinstance(mod, nn.LayerNorm):
            n = mod.weight.numel()
            if name.endswith("norm1") and "tokens_to_token" in name:
                mod.weight.copy_(torch.linspace(0.3, 1.7, n) + 0.2 * rn(n))
                mod.bias.copy_(torch.linspace(-0.5, 0.5, n) + 0.1 * rn(n))
            else:
                mod.weight.copy_(1.0 + 0.1 * rn(n))
                mod.bias.copy_(0.1 * rn(n))
        elif isinstance(mod, Token_performer):
            q, _ = torch.linalg.qr(rn(mod.emb, mod.m))
            mod.w.copy_(q.t() * math.sqrt(mod.m))
    if hasattr(model, "cls_token"):
        model.cls_token.copy_(rn(*model.cls_token.shape) * 0.05)
    return model
