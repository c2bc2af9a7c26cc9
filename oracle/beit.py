"""Oracle: seeded HF ``BeitForImageClassification`` / ``Data2VecVisionForImageClassification`` models (test infrastructure).

The installed ``transformers`` carries both (SITE/models/beit/modeling_beit.py, SITE/models/data2vec/modeling_data2vec_vision.py),
so the parity tests run those modules themselves in float32 as the reference.

``stress=True`` randomises what HF initialises to constants, so that every path the library adds moves the logits: the
relative position bias tables (zeros in HF) ~ N(0, 1), LayerScale ``lambda_{1,2}`` (0.1 in HF) uniform in [0.1, 1], biases
and LayerNorm shifts ~ N(0, 0.1) and LayerNorm weights 1 + N(0, 0.1).
"""
from __future__ import annotations

import torch

BEIT_SIZES = {"base": (768, 12, 12), "large": (1024, 24, 16)}   # hidden, layers, heads


def build_hf_beit(kind: str = "base", seed: int = 0, layers=None, image_size: int = 224, num_labels: int = 1000, stress: bool = True,
                  data2vec: bool = False, use_mean_pooling: bool = True, use_relative_position_bias: bool = True,
                  use_shared_relative_position_bias: bool = False, use_absolute_position_embeddings: bool = False,
                  attn_implementation: str = "eager"):
    from transformers import BeitConfig, BeitForImageClassification, Data2VecVisionConfig, Data2VecVisionForImageClassification
    D, L, heads = BEIT_SIZES[kind]
    Config, Model = (Data2VecVisionConfig, Data2VecVisionForImageClassification) if data2vec else (BeitConfig, BeitForImageClassification)
    cfg = Config(hidden_size=D, num_hidden_layers=int(layers or L), num_attention_heads=heads, intermediate_size=4 * D,
                 image_size=image_size, patch_size=16, num_labels=num_labels, use_mean_pooling=use_mean_pooling,
                 use_relative_position_bias=use_relative_position_bias,
                 use_shared_relative_position_bias=use_shared_relative_position_bias,
                 use_absolute_position_embeddings=use_absolute_position_embeddings, layer_scale_init_value=0.1,
                 attn_implementation=attn_implementation)
    torch.manual_seed(seed)
    model = Model(cfg).eval()
    if stress:
        g = torch.Generator().manual_seed(seed + 1000)
        with torch.no_grad():
            for name, p in model.named_parameters():
                if name.endswith("relative_position_bias_table"):
                    p.copy_(torch.randn(p.shape, generator=g))
                elif name.endswith(("lambda_1", "lambda_2")):
                    p.copy_(0.1 + 0.9 * torch.rand(p.shape, generator=g))
                elif ("norm" in name) and name.endswith("weight"):
                    p.copy_(1.0 + torch.randn(p.shape, generator=g) * 0.1)
                elif name.endswith("bias") or name.endswith("position_embeddings") or name.endswith("cls_token"):
                    p.copy_(torch.randn(p.shape, generator=g) * 0.1)
    return model


def images(n: int, image_size: int = 224, seed: int = 0) -> torch.Tensor:
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, 3, image_size, image_size, generator=g)


@torch.no_grad()
def hf_logits(model, x: torch.Tensor) -> torch.Tensor:
    """fp32 CPU forward of the HF module (TF32 matmuls off)."""
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        return model.float().cpu()(pixel_values=x.float().cpu()).logits
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
