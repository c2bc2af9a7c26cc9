"""DeiT III (facebookresearch/deit ``models_v2.py``: ``vit_models`` with ``Layer_scale_init_Block``) restated as nn.Modules with
upstream's state-dict keys (``patch_embed.proj``, ``cls_token``, ``pos_embed``, ``blocks.{l}.{norm1,attn.qkv,attn.proj,norm2,
mlp.fc1,mlp.fc2,gamma_1,gamma_2}``, ``norm``, ``head``), test infrastructure for tests/test_deit3_cpu.py and
tests/test_gpu_deit3.py.

No upstream code was available when this was written, so these are readings of ``models_v2`` and of timm's ``deit3_*``, not
checks against it:
  * LayerNorm eps 1e-6 (``partial(nn.LayerNorm, eps=1e-6)`` in every ``deit_*_LS`` factory);
  * erf-GELU (``nn.GELU()``) in the MLP;
  * ``qkv_bias=True``;
  * softmax scale ``head_dim ** -0.5``;
  * the position embedding is ``[1, patches, D]`` and is added to the patch tokens only, before the cls token is
    prepended (the cls token gets no position row);
  * ``x + gamma_1 * attn(norm1(x))``, ``x + gamma_2 * mlp(norm2(x))``;
  * the classifier reads row 0 after the final norm.
timm's ``deit3_*`` names LayerScale ``blocks.{l}.ls{1,2}.gamma``; ``to_timm_keys`` renames.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

# name -> (embed dim, depth, heads, patch)
CONFIGS = {
    "small": (384, 12, 6, 16), "medium": (512, 12, 8, 16), "base": (768, 12, 12, 16), "large": (1024, 24, 16, 16),
    "huge": (1280, 32, 16, 14),
}


class Attention(nn.Module):
    def __init__(self, dim, num_heads):
        super().__init__()
        self.num_heads = num_heads
        self.scale = (dim // num_heads) ** -0.5
        self.qkv = nn.Linear(dim, dim * 3, bias=True)
        self.proj = nn.Linear(dim, dim)

    def forward(self, x):
        B, N, C = x.shape
        qkv = self.qkv(x).reshape(B, N, 3, self.num_heads, C // self.num_heads).permute(2, 0, 3, 1, 4)
        q, k, v = qkv[0], qkv[1], qkv[2]
        attn = ((q * self.scale) @ k.transpose(-2, -1)).softmax(dim=-1)
        return self.proj((attn @ v).transpose(1, 2).reshape(B, N, C))


class Mlp(nn.Module):
    def __init__(self, dim, hidden):
        super().__init__()
        self.fc1 = nn.Linear(dim, hidden)
        self.fc2 = nn.Linear(hidden, dim)

    def forward(self, x):
        return self.fc2(F.gelu(self.fc1(x)))


class Layer_scale_init_Block(nn.Module):
    def __init__(self, dim, num_heads, mlp_ratio=4.0, init_values=1e-4):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim, eps=1e-6)
        self.attn = Attention(dim, num_heads)
        self.norm2 = nn.LayerNorm(dim, eps=1e-6)
        self.mlp = Mlp(dim, int(dim * mlp_ratio))
        self.gamma_1 = nn.Parameter(init_values * torch.ones(dim))
        self.gamma_2 = nn.Parameter(init_values * torch.ones(dim))

    def forward(self, x):
        x = x + self.gamma_1 * self.attn(self.norm1(x))
        return x + self.gamma_2 * self.mlp(self.norm2(x))


class PatchEmbed(nn.Module):
    def __init__(self, patch, dim):
        super().__init__()
        self.proj = nn.Conv2d(3, dim, kernel_size=patch, stride=patch)

    def forward(self, x):
        return self.proj(x).flatten(2).transpose(1, 2)


class vit_models(nn.Module):
    def __init__(self, img_size=224, patch_size=16, num_classes=1000, embed_dim=768, depth=12, num_heads=12, mlp_ratio=4.0):
        super().__init__()
        self.patch_embed = PatchEmbed(patch_size, embed_dim)
        self.cls_token = nn.Parameter(torch.zeros(1, 1, embed_dim))
        self.pos_embed = nn.Parameter(torch.zeros(1, (img_size // patch_size) ** 2, embed_dim))
        self.blocks = nn.ModuleList([Layer_scale_init_Block(embed_dim, num_heads, mlp_ratio) for _ in range(depth)])
        self.norm = nn.LayerNorm(embed_dim, eps=1e-6)
        self.head = nn.Linear(embed_dim, num_classes)

    def forward(self, x):
        x = self.patch_embed(x)
        x = x + self.pos_embed
        x = torch.cat((self.cls_token.expand(x.shape[0], -1, -1), x), dim=1)
        for blk in self.blocks:
            x = blk(x)
        return self.head(self.norm(x)[:, 0])


def build(name: str, image: int = 224, depth: Optional[int] = None, seed: int = 0, num_classes: int = 1000,
          dims: Optional[tuple] = None) -> vit_models:
    """Seeded, stress-initialised DeiT III: LayerScale gamma drawn from [0.1, 1] (not the 1e-4 init, under which the residual
    branches would hardly reach the logits), biases and LayerNorm affine from N(0, 0.1), cls / position rows from N(0, 0.02).
    ``dims`` = (embed dim, heads, patch) overrides the named shape (small test models)."""
    D, L, H, P = CONFIGS[name] if dims is None else (dims[0], 2, dims[1], dims[2])
    torch.manual_seed(seed)
    m = vit_models(img_size=image, patch_size=P, num_classes=num_classes, embed_dim=D, depth=L if depth is None else depth,
                   num_heads=H).eval()
    g = torch.Generator().manual_seed(seed + 1000)
    with torch.no_grad():
        for n, p in m.named_parameters():
            if "gamma_" in n:
                p.copy_(0.1 + 0.9 * torch.rand(p.shape, generator=g))
            elif n.endswith("bias"):
                p.copy_(torch.randn(p.shape, generator=g) * 0.1)
            elif "norm" in n:
                p.copy_(1.0 + torch.randn(p.shape, generator=g) * 0.1)
            elif n in ("cls_token", "pos_embed"):
                p.copy_(torch.randn(p.shape, generator=g) * 0.02)
            else:   # Linear / Conv weights: N(0, 0.02), the trunc_normal_ init of models_v2, untruncated
                p.copy_(torch.randn(p.shape, generator=g) * 0.02)
    return m


def to_timm_keys(sd: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    """models_v2 keys -> timm deit3_* keys (``gamma_i`` -> ``ls{i}.gamma``)."""
    out = {}
    for k, v in sd.items():
        for i in (1, 2):
            if k.endswith(f".gamma_{i}"):
                k = k[:-len(f"gamma_{i}")] + f"ls{i}.gamma"
        out[k] = v
    return out
