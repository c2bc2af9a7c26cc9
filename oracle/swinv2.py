"""Oracle: seeded HF ``Swinv2ForImageClassification`` models (test infrastructure).

The installed ``transformers`` carries Swin V2 (SITE/models/swinv2/modeling_swinv2.py), so the parity tests run that module
itself in float32 as the reference rather than a restatement.  ``build_hf_swinv2`` makes one of a given width (the variants
of the microsoft/Swin-Transformer configs), depth, window and pretrained window sizes.

``stress=True`` randomises what HF initialises to constants, so that every term of the arithmetic matters:
biases, LayerNorm affine and the ``continuous_position_bias_mlp`` weights ~ N(0, 0.1) (LayerNorm weights 1 + N(0, 0.1)), and
``logit_scale`` per head uniform in [0, ln 100 + 0.5], so some heads sit at the clamp exp(ln 100) = 100.

``halve_shift_masks`` divides the shift masks of an HF module by two: its forward adds the mask twice (:463-468), which with
halved masks is the -100 of the original code once (what ``B200Swinv2ForImageClassification.from_microsoft`` reproduces).
"""
from __future__ import annotations

import math

import torch

SWINV2_WIDTHS = {"tiny": (96, [3, 6, 12, 24]), "small": (96, [3, 6, 12, 24]), "base": (128, [4, 8, 16, 32]),
                 "large": (192, [6, 12, 24, 48])}
SWINV2_DEPTHS = {"tiny": [2, 2, 6, 2], "small": [2, 2, 18, 2], "base": [2, 2, 18, 2], "large": [2, 2, 18, 2]}


def build_hf_swinv2(kind: str, seed: int, depths=None, window: int = 8, pretrained_window_sizes=(0, 0, 0, 0), stress: bool = False,
                    image_size: int = 256, num_labels: int = 1000):
    from transformers import Swinv2Config, Swinv2ForImageClassification
    embed_dim, heads = SWINV2_WIDTHS[kind]
    cfg = Swinv2Config(image_size=image_size, patch_size=4, window_size=window, embed_dim=embed_dim,
                       depths=list(depths or SWINV2_DEPTHS[kind]), num_heads=heads, num_labels=num_labels,
                       pretrained_window_sizes=list(pretrained_window_sizes))
    torch.manual_seed(seed)
    model = Swinv2ForImageClassification(cfg).eval()
    if stress:
        g = torch.Generator().manual_seed(seed + 1000)
        with torch.no_grad():
            for name, p in model.named_parameters():
                if name.endswith("logit_scale"):
                    p.copy_(torch.rand(p.shape, generator=g) * (math.log(100.0) + 0.5))
                elif "continuous_position_bias_mlp" in name:
                    p.copy_(torch.randn(p.shape, generator=g) * 0.1)
                elif ("norm" in name) and name.endswith("weight"):
                    p.copy_(1.0 + torch.randn(p.shape, generator=g) * 0.1)
                elif name.endswith("bias"):
                    p.copy_(torch.randn(p.shape, generator=g) * 0.1)
    return model


def halve_shift_masks(model) -> None:
    """Make every shifted block of an HF Swinv2 module build a -50 mask, so that its double add gives the original -100."""
    for layer in model.modules():
        if type(layer).__name__ == "Swinv2Layer" and not hasattr(layer, "_orig_get_attn_mask"):
            layer._orig_get_attn_mask = layer.get_attn_mask

            def halved(height, width, dtype, _f=layer._orig_get_attn_mask):
                m = _f(height, width, dtype)
                return None if m is None else m / 2
            layer.get_attn_mask = halved


def to_microsoft(model) -> dict:
    """The HF module's weights under microsoft/Swin-Transformer ``SwinTransformerV2`` names (fused qkv, q_bias / v_bias,
    cpb_mlp, norm1 / norm2, head), with the buffers that repository's state dicts carry."""
    sd = model.state_dict()
    out = {}
    for k, v in sd.items():
        k2 = k
        if k.startswith("swinv2.embeddings.patch_embeddings.projection."):
            k2 = "patch_embed.proj." + k.rsplit(".", 1)[1]
        elif k.startswith("swinv2.embeddings.norm."):
            k2 = "patch_embed.norm." + k.rsplit(".", 1)[1]
        elif k.startswith("swinv2.layernorm."):
            k2 = "norm." + k.rsplit(".", 1)[1]
        elif k.startswith("classifier."):
            k2 = "head." + k.rsplit(".", 1)[1]
        elif k.startswith("swinv2.encoder.layers."):
            k2 = k[len("swinv2.encoder."):]
            for a, b in (("layernorm_before.", "norm1."), ("layernorm_after.", "norm2."), ("attention.output.dense.", "attn.proj."),
                         ("intermediate.dense.", "mlp.fc1."), ("output.dense.", "mlp.fc2."),
                         ("attention.self.continuous_position_bias_mlp.", "attn.cpb_mlp."),
                         ("attention.self.logit_scale", "attn.logit_scale")):
                k2 = k2.replace(a, b)
            if "attention.self." in k2:
                continue                               # q / k / v handled below
        out[k2] = v.clone()
    for name, attn in model.named_modules():
        if type(attn).__name__ == "Swinv2SelfAttention":
            p = name[len("swinv2.encoder."):].replace(".attention.self", ".attn.")
            out[p + "qkv.weight"] = torch.cat([attn.query.weight, attn.key.weight, attn.value.weight], 0).detach().clone()
            out[p + "q_bias"] = attn.query.bias.detach().clone()
            out[p + "v_bias"] = attn.value.bias.detach().clone()
            out[p + "relative_coords_table"] = attn.relative_coords_table.clone()
            out[p + "relative_position_index"] = attn.relative_position_index.clone()
    return out
