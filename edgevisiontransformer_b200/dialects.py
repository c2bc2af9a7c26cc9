"""Weight-layout adapters: the reference's TensorFlow-dialect models -> the canonical (HF-named,
``[out, in]`` Linear) layout libevt loads.

TF dialect facts handled here (modeling/models/vit.py:9-55, modeling/layers/attention.py:17-20):
  * Keras ``Dense`` kernels are ``[in, out]``                    -> transposed
  * fused no-bias ``to_qkv`` with columns ordered (qkv, head, d)   -> split into query / key / value
  * patch pixels flattened ``(p1 p2 c)``                           -> rows permuted to ``(c p1 p2)`` (our im2col order)
  * no final LayerNorm, head = Dense(mlp_dim, gelu) -> Dense(classes) -> pre_classifier + classifier
The different skip-connection semantics (skip carries LN(x)) is a runtime flag (dialect="tf").

timm / facebookresearch-deit dialect (``torch.hub.load('facebookresearch/deit:main', 'deit_*_patch16_224')``,
utils.py:52-62, tools.py:244-263): same function as HF ViT with a fused ``attn.qkv`` Linear (rows q | k | v, head-major
inside each), LayerNorm eps 1e-6 and flat key names -> pure renaming + split, see ``timm_vit_to_canonical``.

DeiT III (facebookresearch-deit ``models_v2``: ``deit_{small,medium,base,large}_patch16_LS``, ``deit_huge_patch14_LS``; timm
``deit3_*``): the same blocks with LayerScale, ``x + gamma_1 * attn(norm1(x))`` and ``x + gamma_2 * mlp(norm2(x))`` (keys
``blocks.{l}.gamma_{1,2}`` or timm's ``blocks.{l}.ls{1,2}.gamma``), and a position embedding of the patches only (no cls row).
LayerScale is folded into the two residual projections, ``W' = diag(gamma) W``, ``b' = gamma * b``; the cls token gets a zero
position row.  See ``timm_vit_to_canonical``.

PyTorch T2T-ViT (yitu-opensource/T2T-ViT, ``tokens_type='performer'``; the reference's tools.py:347-365 loads these files):
timm-layout encoder blocks without qkv bias, plus the tokens-to-token module, whose ``nn.Unfold`` soft splits order their
columns ``(c, kh, kw)`` -> permuted to the ``(kh, kw, c)`` order of the library's soft splits, see ``t2t_torch_to_canonical``.
"""
from __future__ import annotations

import math
import re
from typing import Dict, List, Optional, Tuple

import torch


def _encoder_to_canonical(sd: Dict[str, torch.Tensor], out: Dict[str, torch.Tensor], heads: List[int], head_size: int,
                          prefix: str = "layers") -> None:
    for l, nh in enumerate(heads):
        p, q = f"{prefix}.{l}", f"vit.encoder.layer.{l}"
        a = nh * head_size
        wqkv = sd[p + ".attn.to_qkv.kernel"].t().contiguous()          # [3a, D], rows (qkv, head, d)
        for i, n in enumerate(("query", "key", "value")):
            out[f"{q}.attention.attention.{n}.weight"] = wqkv[i * a:(i + 1) * a].contiguous()
        out[f"{q}.attention.output.dense.weight"] = sd[p + ".attn.to_out.kernel"].t().contiguous()
        out[f"{q}.attention.output.dense.bias"] = sd[p + ".attn.to_out.bias"]
        out[f"{q}.layernorm_before.weight"] = sd[p + ".attn.norm.gamma"]
        out[f"{q}.layernorm_before.bias"] = sd[p + ".attn.norm.beta"]
        out[f"{q}.layernorm_after.weight"] = sd[p + ".ffn.norm.gamma"]
        out[f"{q}.layernorm_after.bias"] = sd[p + ".ffn.norm.beta"]
        out[f"{q}.intermediate.dense.weight"] = sd[p + ".ffn.fc1.kernel"].t().contiguous()
        out[f"{q}.intermediate.dense.bias"] = sd[p + ".ffn.fc1.bias"]
        out[f"{q}.output.dense.weight"] = sd[p + ".ffn.fc2.kernel"].t().contiguous()
        out[f"{q}.output.dense.bias"] = sd[p + ".ffn.fc2.bias"]


def tf_vit_to_canonical(sd: Dict[str, torch.Tensor], heads: List[int], head_size: int = 64, patch: int = 16
                        ) -> Tuple[Dict[str, torch.Tensor], dict]:
    """modeling/models/vit.py ViT / ViT_Pruned weights -> (canonical state dict, from_state_dict kwargs)."""
    out: Dict[str, torch.Tensor] = {}
    D = sd["cls_token"].shape[-1]
    k = sd["patch_to_embedding.kernel"]                                  # [(p1 p2 c), D]
    w = k.t().reshape(D, patch, patch, 3).permute(0, 3, 1, 2).contiguous()   # [D, c, p1, p2]
    out["vit.embeddings.patch_embeddings.projection.weight"] = w
    out["vit.embeddings.patch_embeddings.projection.bias"] = sd["patch_to_embedding.bias"]
    out["vit.embeddings.cls_token"] = sd["cls_token"].reshape(1, 1, D)
    out["vit.embeddings.position_embeddings"] = sd["pos_embedding"].reshape(1, -1, D)
    _encoder_to_canonical(sd, out, heads, head_size)
    out["pre_classifier.weight"] = sd["mlp_head.0.kernel"].t().contiguous()
    out["pre_classifier.bias"] = sd["mlp_head.0.bias"]
    out["classifier.weight"] = sd["mlp_head.1.kernel"].t().contiguous()
    out["classifier.bias"] = sd["mlp_head.1.bias"]
    kw = dict(dialect="tf", hidden_act="gelu_tanh", layer_norm_eps=1e-5, final_ln=False, head_size=head_size, patch_size=patch)
    return out, kw


def timm_vit_to_canonical(sd: Dict[str, torch.Tensor], patch: int = 16) -> Tuple[Dict[str, torch.Tensor], dict]:
    """timm ``VisionTransformer`` / facebookresearch DeiT state dict -> (canonical state dict, from_state_dict kwargs).

    Accepts the hub checkpoints' ``{'model': state_dict}`` wrapper.  The reference asks the hub for
    ``deit_{type}_patch16_{224,384}`` (utils.py:52-62); the hub's distilled variants (``DistilledVisionTransformer``:
    ``dist_token``, ``head_dist``, eval output ``(head(x[:, 0]) + head_dist(x[:, 1])) / 2``) map onto the two-head layout that
    ``modeling_vit.normalise_keys`` folds into one classifier.  Half of that layout is refused."""
    if "model" in sd and isinstance(sd["model"], dict):
        sd = sd["model"]
    _refuse_deit3_variants(sd)
    distilled = "dist_token" in sd
    if distilled != ("head_dist.weight" in sd):
        raise ValueError("distilled DeiT checkpoint needs both dist_token and head_dist")
    D = sd["cls_token"].shape[-1]
    pos = sd["pos_embed"].reshape(1, -1, D)
    n_prefix = 2 if distilled else 1
    if math.isqrt(pos.shape[1]) ** 2 == pos.shape[1]:   # patches only (DeiT III): the prefix tokens get no position row
        pos = torch.cat((pos.new_zeros(1, n_prefix, D), pos), dim=1)
    out: Dict[str, torch.Tensor] = {
        "vit.embeddings.cls_token": sd["cls_token"].reshape(1, 1, D),
        "vit.embeddings.position_embeddings": pos,
        "vit.embeddings.patch_embeddings.projection.weight": sd["patch_embed.proj.weight"],
        "vit.embeddings.patch_embeddings.projection.bias": sd["patch_embed.proj.bias"],
        "vit.layernorm.weight": sd["norm.weight"], "vit.layernorm.bias": sd["norm.bias"],
    }
    if distilled:
        out["vit.embeddings.distillation_token"] = sd["dist_token"].reshape(1, 1, D)
        out["cls_classifier.weight"], out["cls_classifier.bias"] = sd["head.weight"], sd["head.bias"]
        out["distillation_classifier.weight"], out["distillation_classifier.bias"] = sd["head_dist.weight"], sd["head_dist.bias"]
    else:
        out["classifier.weight"], out["classifier.bias"] = sd["head.weight"], sd["head.bias"]
    depth = _timm_blocks_to_canonical(sd, out, D)
    if depth == 0:
        raise ValueError("not a timm VisionTransformer state dict (no blocks.0.attn.qkv.weight)")
    stray = [k for k in sd if _LAYERSCALE.search(k) and int(k.split(".")[1]) >= depth]
    if stray:
        raise ValueError(f"LayerScale parameters of blocks the state dict does not have: {stray[:4]}")
    return out, dict(layer_norm_eps=1e-6, hidden_act="gelu", patch_size=patch)


_LAYERSCALE = re.compile(r"^blocks\.\d+\.(gamma_[12]|ls[12]\.gamma)$")
DEIT3_HUGE_DIM, DEIT3_GIANT_DIM = 1280, 1408


def _refuse_deit3_variants(sd: Dict[str, torch.Tensor]) -> None:
    """The DeiT III variants this library does not run, refused by name rather than loaded wrong."""
    if any(re.match(r"^blocks\.\d+\.(attn1|mlp1|norm11|norm21|gamma_1_1|gamma_2_1)\.?", k) for k in sd):
        raise ValueError("parallel-block DeiT III (deit_huge_patch14_26x2_LS: two attention and two MLP branches per block) "
                         "is not implemented")
    if "cls_token" in sd and sd["cls_token"].shape[-1] == DEIT3_GIANT_DIM and any(_LAYERSCALE.search(k) for k in sd):
        raise ValueError("DeiT III Giant (deit_giant_patch14_LS, embed dim 1408, head size 88) is not implemented")


def deit3_head_size(sd: Dict[str, torch.Tensor]) -> int:
    """Head size of a DeiT III state dict (80 for Huge, embed dim 1280; 64 for every smaller model), else 64."""
    if "model" in sd and isinstance(sd["model"], dict):
        sd = sd["model"]
    layerscale = any(_LAYERSCALE.search(k) for k in sd)
    return 80 if layerscale and "cls_token" in sd and sd["cls_token"].shape[-1] == DEIT3_HUGE_DIM else 64


def _layerscale(sd: Dict[str, torch.Tensor], l: int, i: int) -> Optional[torch.Tensor]:
    """gamma_i of block l in either key layout (None without LayerScale); both layouts at once are refused."""
    a, b = sd.get(f"blocks.{l}.gamma_{i}"), sd.get(f"blocks.{l}.ls{i}.gamma")
    if a is not None and b is not None:
        raise ValueError(f"block {l} has both blocks.{l}.gamma_{i} and blocks.{l}.ls{i}.gamma")
    return a if a is not None else b


def _timm_blocks_to_canonical(sd: Dict[str, torch.Tensor], out: Dict[str, torch.Tensor], D: int, q_scale: float = 1.0) -> int:
    """timm ``Block`` s ``blocks.{l}.*`` (fused ``attn.qkv``, rows q | k | v) -> ``vit.encoder.layer.{l}.*``; returns the depth.
    ``q_scale`` multiplies the query rows (weight and bias): how a softmax scale other than head_size ** -0.5 is folded in.
    LayerScale (DeiT III) is folded in f32 into the rows of ``attn.proj`` (gamma_1) and ``mlp.fc2`` (gamma_2)."""
    l = 0
    while f"blocks.{l}.attn.qkv.weight" in sd:
        p, q = f"blocks.{l}.", f"vit.encoder.layer.{l}."
        w = sd[p + "attn.qkv.weight"]
        if w.shape[0] != 3 * D:
            raise ValueError(f"blocks.{l}.attn.qkv.weight has {w.shape[0]} rows, expected 3 x {D}")
        b = sd.get(p + "attn.qkv.bias")
        for i, n in enumerate(("query", "key", "value")):
            for t, suffix in ((w, "weight"), (b, "bias")):
                if t is not None:
                    rows = t[i * D:(i + 1) * D]
                    out[q + f"attention.attention.{n}.{suffix}"] = (rows * q_scale if i == 0 and q_scale != 1.0 else rows).contiguous()
        for src, dst in (("attn.proj", "attention.output.dense"), ("mlp.fc1", "intermediate.dense"), ("mlp.fc2", "output.dense"),
                         ("norm1", "layernorm_before"), ("norm2", "layernorm_after")):
            out[q + dst + ".weight"] = sd[p + src + ".weight"]
            out[q + dst + ".bias"] = sd[p + src + ".bias"]
        g1, g2 = _layerscale(sd, l, 1), _layerscale(sd, l, 2)
        if (g1 is None) != (g2 is None):
            raise ValueError(f"block {l} has LayerScale on one residual branch only")
        for g, dst in ((g1, "attention.output.dense"), (g2, "output.dense")):
            if g is not None:
                fold_layerscale(out, q + dst, g, D, f"block {l}")
        l += 1
    return l


def fold_layerscale(sd: Dict[str, torch.Tensor], linear: str, gamma: torch.Tensor, D: int, where: str) -> None:
    """In place: LayerScale ``gamma * linear(x)`` folded into the Linear ``linear`` of ``sd`` (``.weight`` [D, in], ``.bias`` [D]):
    ``W' = diag(gamma) W``, ``b' = gamma * b``, computed in f32 at least (f64 weights stay f64).  ``where`` names the block in
    the error for a gamma of the wrong length."""
    w, b = sd[linear + ".weight"], sd[linear + ".bias"]
    dt = torch.promote_types(w.dtype, torch.float32)
    g = gamma.to(dt).reshape(-1)
    if g.numel() != D:
        raise ValueError(f"{where}: LayerScale has {g.numel()} entries, expected {D}")
    sd[linear + ".weight"] = w.to(dt) * g[:, None]
    sd[linear + ".bias"] = b.to(dt) * g


def unwrap_checkpoint(ck: dict, use_ema: bool = True) -> Dict[str, torch.Tensor]:
    """The state dict inside a training checkpoint: ``state_dict_ema`` (when ``use_ema``), ``state_dict`` or ``model``, else
    ``ck`` itself; ``module.`` (DataParallel / DDP) prefixes stripped.  timm's checkpoint saver writes the first two."""
    for k in (("state_dict_ema",) if use_ema else ()) + ("state_dict", "model"):
        if isinstance(ck.get(k), dict):
            ck = ck[k]
            break
    return {(k[len("module."):] if k.startswith("module.") else k): v for k, v in ck.items() if torch.is_tensor(v)}


def _ckk_to_kkc(t: torch.Tensor, C: int, k: int) -> torch.Tensor:
    """Last dimension ordered (c, kh, kw) -- nn.Unfold's columns -- reordered to (kh, kw, c)."""
    lead = t.shape[:-1]
    return t.reshape(*lead, C, k, k).movedim(-3, -1).reshape(*lead, C * k * k).contiguous()


T2T_TORCH_HEAD_SIZE = 64


def t2t_torch_to_canonical(sd: Dict[str, torch.Tensor], qk_scale: Optional[float] = None, use_ema: bool = True
                           ) -> Tuple[Dict[str, torch.Tensor], dict]:
    """PyTorch T2T-ViT (``T2T_ViT`` with ``tokens_type='performer'`` or ``'transformer'``) state dict or training checkpoint ->
    (canonical state dict, from_state_dict kwargs).  The token type is read from the keys.

    * performer: ``tokens_to_token.attention{1,2}.*`` -> ``t2t.performer{1,2}.*`` in the Keras naming the runtime loads
      (INTEGRATION.md §3): kernels ``[in, out]``; the rows of ``kqv.kernel`` and of ``norm1.{gamma,beta}`` permuted from
      ``(c, kh, kw)`` to ``(kh, kw, c)`` (stage 1: C = 3, k = 7; stage 2: C = 64, k = 3); ``w`` as stored (already times
      sqrt(m)).  ``t2t = 2``.
    * transformer (``Token_transformer``, one head): -> ``t2t.transformer{1,2}.*``: ``norm1`` and the input rows of
      ``qkv.kernel`` (from ``attn.qkv.weight``, which has no bias) permuted the same way, ``attn.proj`` -> ``attn_output``,
      ``mlp.fc{1,2}`` -> ``mlp.fc{1,2}``.  The token attention's scale (in_dim ** -0.5) is the runtime's.  ``t2t = 3``.
    * ``tokens_to_token.project`` -> the token-embedding projection, its 576 input columns permuted the same way (C = 64, k = 3).
    * ``cls_token``, ``pos_embed`` (the sinusoid table stored in the checkpoint) -> the embeddings.
    * ``blocks.*``, ``norm.*``, ``head.*`` as in ``timm_vit_to_canonical``.  ``qk_scale`` (default head_size ** -0.5, the
      scale the runtime applies) is folded into the query rows.
    Refuses a dict holding both token types, a ``Token_transformer`` with a qkv bias and any image size other than 224."""
    sd = unwrap_checkpoint(sd, use_ema)
    performer = "tokens_to_token.attention1.kqv.weight" in sd
    transformer = "tokens_to_token.attention1.attn.qkv.weight" in sd
    if performer and transformer:
        raise ValueError("state dict mixes tokens_type='performer' (attention1.kqv) and tokens_type='transformer' (attention1.attn.qkv) "
                         "token modules: not one T2T-ViT")
    if not (performer or transformer) or "blocks.0.attn.qkv.weight" not in sd:
        raise ValueError("not a PyTorch T2T-ViT state dict (no tokens_to_token.attention1.kqv.weight / .attn.qkv.weight or "
                         "blocks.0.attn.qkv.weight)")
    if transformer and any(f"tokens_to_token.attention{i}.attn.qkv.bias" in sd for i in (1, 2)):
        raise ValueError("tokens_type='transformer' with a qkv bias: upstream's Token_transformer has none and it is not implemented")
    D = sd["cls_token"].shape[-1]
    if sd["pos_embed"].shape[-2] != 197:
        raise ValueError(f"pos_embed has {sd['pos_embed'].shape[-2]} rows: only the 224-pixel T2T-ViT (197 tokens) is supported")
    out: Dict[str, torch.Tensor] = {}
    for i, (C, k) in ((1, (3, 7)), (2, (64, 3))):
        if transformer:
            _token_transformer_to_canonical(sd, out, i, C, k)
            continue
        s, d = f"tokens_to_token.attention{i}.", f"t2t.performer{i}."
        out[d + "norm1.gamma"] = _ckk_to_kkc(sd[s + "norm1.weight"], C, k)
        out[d + "norm1.beta"] = _ckk_to_kkc(sd[s + "norm1.bias"], C, k)
        out[d + "kqv.kernel"] = _ckk_to_kkc(sd[s + "kqv.weight"], C, k).t().contiguous()
        out[d + "kqv.bias"] = sd[s + "kqv.bias"]
        out[d + "w"] = sd[s + "w"]
        for src, dst in (("proj", "attn_output"), ("mlp.0", "mlp.fc1"), ("mlp.2", "mlp.fc2")):
            out[d + dst + ".kernel"] = sd[s + src + ".weight"].t().contiguous()
            out[d + dst + ".bias"] = sd[s + src + ".bias"]
        out[d + "norm2.gamma"], out[d + "norm2.beta"] = sd[s + "norm2.weight"], sd[s + "norm2.bias"]
    out["vit.embeddings.patch_embeddings.projection.weight"] = _ckk_to_kkc(sd["tokens_to_token.project.weight"], 64, 3)
    out["vit.embeddings.patch_embeddings.projection.bias"] = sd["tokens_to_token.project.bias"]
    out["vit.embeddings.cls_token"] = sd["cls_token"].reshape(1, 1, D)
    out["vit.embeddings.position_embeddings"] = sd["pos_embed"].reshape(1, -1, D)
    scale = T2T_TORCH_HEAD_SIZE ** -0.5 if qk_scale is None else float(qk_scale)
    _timm_blocks_to_canonical(sd, out, D, q_scale=scale * math.sqrt(T2T_TORCH_HEAD_SIZE))
    out["vit.layernorm.weight"], out["vit.layernorm.bias"] = sd["norm.weight"], sd["norm.bias"]
    out["classifier.weight"], out["classifier.bias"] = sd["head.weight"], sd["head.bias"]
    kw = dict(dialect="hf", hidden_act="gelu", layer_norm_eps=1e-5, final_ln=True, head_size=T2T_TORCH_HEAD_SIZE, patch_size=16,
              image_size=224, embed_k=576, t2t=3 if transformer else 2)
    return out, kw


T2T_TOKEN_DIM = 64


def _token_transformer_to_canonical(sd: Dict[str, torch.Tensor], out: Dict[str, torch.Tensor], i: int, C: int, k: int) -> None:
    """``tokens_to_token.attention{i}`` (a one-head ``Token_transformer``, token_dim 64) -> ``t2t.transformer{i}.*``."""
    s, d = f"tokens_to_token.attention{i}.", f"t2t.transformer{i}."
    w = sd[s + "attn.qkv.weight"]
    if tuple(w.shape) != (3 * T2T_TOKEN_DIM, C * k * k):
        raise ValueError(f"{s}attn.qkv.weight is {tuple(w.shape)}, expected ({3 * T2T_TOKEN_DIM}, {C * k * k}): only token_dim "
                         f"{T2T_TOKEN_DIM} is implemented")
    out[d + "norm1.gamma"] = _ckk_to_kkc(sd[s + "norm1.weight"], C, k)
    out[d + "norm1.beta"] = _ckk_to_kkc(sd[s + "norm1.bias"], C, k)
    out[d + "qkv.kernel"] = _ckk_to_kkc(w, C, k).t().contiguous()
    for src, dst in (("attn.proj", "attn_output"), ("mlp.fc1", "mlp.fc1"), ("mlp.fc2", "mlp.fc2")):
        out[d + dst + ".kernel"] = sd[s + src + ".weight"].t().contiguous()
        out[d + dst + ".bias"] = sd[s + src + ".bias"]
    out[d + "norm2.gamma"], out[d + "norm2.beta"] = sd[s + "norm2.weight"], sd[s + "norm2.bias"]
