"""BEiT and data2vec-vision image classifiers on the ViT runtime.

HF ``BeitForImageClassification`` and ``Data2VecVisionForImageClassification`` (SITE/models/beit/modeling_beit.py; data2vec-vision
is the same network under the ``data2vec_vision.`` prefix) are pre-LN ViT encoders with head size 64, erf-GELU and eps 1e-12.
What differs from ViT, and how the library runs it:

  * relative position bias: ``table[rel(q, k), h]`` added to the scaled scores of every layer (``BeitRelativePositionBias``,
    :511-591), per layer (``use_relative_position_bias``) or one table shared by all layers
    (``use_shared_relative_position_bias``, expanded here to every layer).  The attention kernels read the compact table
    (``evt_attention_rel_bias_fwd``); no dense [heads, S, S] bias exists anywhere.
  * mean-pooled head (``use_mean_pooling``): ``classifier(LayerNorm(mean of rows 1..S-1))``; ``pooler.layernorm`` becomes the
    runtime's final norm with ``final_ln = 2``.  Without mean pooling, ``beit.layernorm`` then row 0, as in ViT.
  * LayerScale ``lambda_1`` / ``lambda_2``: folded into ``attention.output.dense`` / ``output.dense`` at load
    (``dialects.fold_layerscale``).
  * no key bias (a zero one is supplied), and no absolute position embeddings unless ``use_absolute_position_embeddings``
    (zero position rows otherwise).

bf16 only; every refusal below is raised before anything is allocated on the device.
"""
from __future__ import annotations

import json
import os
from typing import Dict, Tuple

import torch

from .dialects import fold_layerscale
from .modeling_vit import B200ViTConfig, B200ViTForImageClassification, config_from_state_dict

BEIT_MODEL_TYPES = ("beit", "data2vec-vision")
_PREFIXES = ("beit.", "data2vec_vision.")
_CLASSIFIERS = ("BeitForImageClassification", "Data2VecVisionForImageClassification")
_TABLE = "attention.attention.relative_position_bias.relative_position_bias_table"
_SHARED = "vit.encoder.relative_position_bias."
HEAD_SIZE = 64
MAX_TOKENS = 1026  # EVT_ATTN_MAX_TOKENS
# BeitConfig / Data2VecVisionConfig defaults, for config.json files that leave a key out
_DEFAULTS = dict(image_size=224, patch_size=16, num_channels=3, use_mean_pooling=True, use_relative_position_bias=False,
                 use_shared_relative_position_bias=False, use_absolute_position_embeddings=False, layer_norm_eps=1e-12,
                 hidden_act="gelu", pruned_heads={})


def _get(config, name):
    v = config.get(name, _DEFAULTS.get(name)) if isinstance(config, dict) else getattr(config, name, _DEFAULTS.get(name))
    return v[0] if isinstance(v, (tuple, list)) and name in ("image_size", "patch_size") else v


def relative_position_index(grid: int) -> torch.Tensor:
    """generate_relative_position_index (:521-544) for a grid x grid patch image: [grid^2 + 1, grid^2 + 1] int64.  Used to check
    the ``relative_position_index`` buffers that checkpoints saved by older transformers carry."""
    coords = torch.stack(torch.meshgrid(torch.arange(grid), torch.arange(grid), indexing="ij")).flatten(1)
    rel = coords[:, :, None] - coords[:, None, :]
    n = (2 * grid - 1) ** 2 + 3
    idx = torch.empty((grid * grid + 1,) * 2, dtype=torch.int64)
    idx[1:, 1:] = (rel[0] + grid - 1) * (2 * grid - 1) + rel[1] + grid - 1
    idx[0, :] = n - 3
    idx[:, 0] = n - 2
    idx[0, 0] = n - 1
    return idx


def _check_index(sd: Dict[str, torch.Tensor], key: str, grid: int) -> None:
    t = sd.pop(key, None)
    if t is not None and not torch.equal(t.long(), relative_position_index(grid)):
        raise ValueError(f"{key} does not match a {grid} x {grid} patch grid: the checkpoint was made for another image or patch "
                         "size (running it at another resolution is not implemented)")


def beit_to_canonical(sd: Dict[str, torch.Tensor], config) -> Tuple[Dict[str, torch.Tensor], B200ViTConfig]:
    """HF BEiT / data2vec-vision classifier state dict + its config (a ``BeitConfig``-like object or the config.json dict) ->
    (canonical ``vit.``-named state dict, B200ViTConfig).  Raises ValueError for what the library does not run."""
    D, L = int(_get(config, "hidden_size")), int(_get(config, "num_hidden_layers"))
    heads = int(_get(config, "num_attention_heads"))
    image, patch = int(_get(config, "image_size")), int(_get(config, "patch_size"))
    if D != heads * HEAD_SIZE:
        raise ValueError(f"BEiT: hidden size {D} with {heads} heads is head size {D / heads:g}; only head size {HEAD_SIZE} is "
                         "implemented")
    if _get(config, "pruned_heads"):
        raise ValueError("head-pruned BEiT models are not implemented")
    if int(_get(config, "num_channels")) != 3:
        raise ValueError("BEiT: only 3-channel images are implemented")
    if image % patch:
        raise ValueError(f"BEiT: image size {image} is not a multiple of the patch size {patch}")
    W = image // patch
    S = W * W + 1
    if S > MAX_TOKENS:
        raise ValueError(f"BEiT: {image} px with {patch}-pixel patches is {S} tokens; at most {MAX_TOKENS} are implemented")
    out: Dict[str, torch.Tensor] = {}
    found = [p for p in _PREFIXES if any(k.startswith(p) for k in sd)]
    if len(found) != 1:
        raise ValueError(f"BEiT state dict must have exactly one of the prefixes {_PREFIXES}; found {found}")
    for k, v in sd.items():
        if k.startswith(found[0]):
            out["vit." + k[len(found[0]):]] = v
        elif k.startswith("classifier."):
            out[k] = v
        else:
            raise ValueError(f"BEiT: unexpected key {k!r} (only image classifiers are implemented: no masked-image-modeling or "
                             "segmentation heads)")
    if "classifier.weight" not in out:
        raise ValueError("BEiT state dict has no classifier.weight: only image classifiers (BeitForImageClassification, "
                         "Data2VecVisionForImageClassification) are implemented")
    if "classifier.bias" not in out:
        out["classifier.bias"] = torch.zeros(out["classifier.weight"].shape[0])
    out.pop("vit.embeddings.mask_token", None)
    n = (2 * W - 1) ** 2 + 3
    shared = out.pop(_SHARED + "relative_position_bias_table", None)
    _check_index(out, _SHARED + "relative_position_index", W)
    if (shared is not None) != bool(_get(config, "use_shared_relative_position_bias")):
        raise ValueError("BEiT: use_shared_relative_position_bias and the shared relative_position_bias_table disagree")
    per_layer = bool(_get(config, "use_relative_position_bias"))
    for l in range(L):
        p = f"vit.encoder.layer.{l}."
        a = out[p + "attention.attention.query.weight"].shape[0]
        table = out.get(p + _TABLE)
        _check_index(out, p + "attention.attention.relative_position_bias.relative_position_index", W)
        if (table is not None) != per_layer:
            raise ValueError(f"BEiT layer {l}: use_relative_position_bias and the layer's relative_position_bias_table disagree")
        if table is not None and shared is not None:   # HF adds both biases
            if table.shape != shared.shape:
                raise ValueError(f"BEiT layer {l}: the per-layer and the shared bias tables differ in shape")
            table = table.float() + shared.float()
        elif shared is not None:
            table = shared
        if table is not None:
            if table.dim() != 2 or table.shape[0] != n:
                raise ValueError(f"BEiT layer {l}: relative_position_bias_table is {tuple(table.shape)}, expected [{n}, heads] for a "
                                 f"{W} x {W} patch grid")
            if a != HEAD_SIZE * table.shape[1]:
                raise ValueError(f"BEiT layer {l}: {a} query rows for {table.shape[1]} bias heads; head-pruned or uneven heads are "
                                 "not implemented")
            out[p + _TABLE] = table
        if a != D:
            raise ValueError(f"BEiT layer {l}: {a} query rows, expected {D}; head-pruned models are not implemented")
        if p + "attention.attention.key.bias" not in out:
            out[p + "attention.attention.key.bias"] = torch.zeros(a)
        g1, g2 = out.pop(p + "lambda_1", None), out.pop(p + "lambda_2", None)
        if (g1 is None) != (g2 is None):
            raise ValueError(f"BEiT layer {l} has LayerScale on one residual branch only")
        if g1 is not None:
            fold_layerscale(out, p + "attention.output.dense", g1, D, f"BEiT layer {l}")
            fold_layerscale(out, p + "output.dense", g2, D, f"BEiT layer {l}")
    if f"vit.encoder.layer.{L}.attention.attention.query.weight" in out:
        raise ValueError(f"BEiT state dict has more than num_hidden_layers = {L} layers")
    pos = out.get("vit.embeddings.position_embeddings")
    if bool(_get(config, "use_absolute_position_embeddings")):
        if pos is None or pos.shape[-2:] != (S, D):
            raise ValueError(f"BEiT: use_absolute_position_embeddings needs position_embeddings [1, {S}, {D}]")
    else:
        if pos is not None:
            raise ValueError("BEiT: position_embeddings present although use_absolute_position_embeddings is off")
        out["vit.embeddings.position_embeddings"] = torch.zeros(1, S, D)
    mean_pool = bool(_get(config, "use_mean_pooling"))
    if mean_pool:
        if "vit.layernorm.weight" in out:
            raise ValueError("BEiT: a final layernorm with use_mean_pooling (where it is an Identity)")
        out["vit.layernorm.weight"] = out.pop("vit.pooler.layernorm.weight")
        out["vit.layernorm.bias"] = out.pop("vit.pooler.layernorm.bias")
    elif any(k.startswith("vit.pooler.") for k in out):
        raise ValueError("BEiT: a pooler layernorm without use_mean_pooling")
    cfg = config_from_state_dict(out, layer_norm_eps=float(_get(config, "layer_norm_eps")), hidden_act=_get(config, "hidden_act"),
                                 head_size=HEAD_SIZE, image_size=image, patch_size=patch, final_ln=True)
    if cfg.num_hidden_layers != L:
        raise ValueError(f"BEiT state dict has {cfg.num_hidden_layers} layers, config says {L}")
    if mean_pool:
        cfg.final_ln = 2   # evt_model_spec.final_ln = 2: LayerNorm of the mean of the patch rows
    return out, cfg


class B200BeitForImageClassification(B200ViTForImageClassification):
    """HF ``BeitForImageClassification`` / ``Data2VecVisionForImageClassification`` forward inside libevt (bf16).  forward,
    forward_graphed, the pixel dtypes, head_mask and context capture are those of B200ViTForImageClassification."""

    @classmethod
    def from_state_dict(cls, sd: Dict[str, torch.Tensor], config=None, **kw):
        """``sd``: HF-named state dict (``beit.*`` or ``data2vec_vision.*`` + ``classifier.*``); ``config``: its BeitConfig /
        Data2VecVisionConfig or the config.json dict."""
        if config is None:
            raise ValueError("B200BeitForImageClassification.from_state_dict needs the model's config (image and patch size, "
                             "pooling and bias options are not in the weights)")
        precision = kw.pop("precision", "bf16")
        if precision != "bf16":
            raise ValueError(f"BEiT runs in the bf16 mode only (precision={precision!r}): the tf32 attention has no relative "
                             "position bias")
        csd, cfg = beit_to_canonical(sd, config)
        return cls(cfg, csd, **kw)

    @classmethod
    def from_hf(cls, model, **kw):
        """Build from a live HF BeitForImageClassification or Data2VecVisionForImageClassification."""
        if type(model).__name__ not in _CLASSIFIERS:
            raise ValueError(f"{type(model).__name__} is not implemented; B200BeitForImageClassification runs {_CLASSIFIERS}")
        return cls.from_state_dict(dict(model.state_dict()), model.config, **kw)

    @classmethod
    def from_pretrained(cls, model_dir: str, **kw):
        """A checkpoint directory: config.json with model_type "beit" or "data2vec-vision" and model.safetensors or
        pytorch_model.bin (read_beit_checkpoint)."""
        sd, config = read_beit_checkpoint(model_dir)
        return cls.from_state_dict(sd, config, **kw)


def read_beit_checkpoint(model_dir: str) -> Tuple[Dict[str, torch.Tensor], dict]:
    """(state dict, config.json dict) of a BEiT / data2vec-vision classifier directory; no nn_pruning zero-row pass."""
    from .checkpoint import read_state_dict
    with open(os.path.join(model_dir, "config.json")) as f:
        config = json.load(f)
    if config.get("model_type") not in BEIT_MODEL_TYPES:
        raise ValueError(f"config.json model_type {config.get('model_type')!r} is not one of {BEIT_MODEL_TYPES}")
    arch = config.get("architectures") or []
    if arch and not any(a in _CLASSIFIERS for a in arch):
        raise ValueError(f"architectures {arch} is not implemented; B200BeitForImageClassification runs {_CLASSIFIERS}")
    return read_state_dict(model_dir), config
