"""Transformer-token T2T-ViT checkpoints (t2t_vit_t_*) without a GPU: the converter against nn.Unfold in float64, key conversion,
factory selection, checkpoint files and the refusals."""
import argparse
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import t2t_t_torch_ref as tref  # noqa: E402
import t2t_torch_ref as ref  # noqa: E402
from edgevisiontransformer_b200 import modeling_t2t  # noqa: E402
from edgevisiontransformer_b200.dialects import t2t_torch_to_canonical  # noqa: E402
from edgevisiontransformer_b200.modeling_t2t import B200T2TViTTorch, _factory_of  # noqa: E402
from oracle import t2t_transformer as ot2t  # noqa: E402


def _sd(name="t2t_vit_t_14", depth=1, seed=0):
    return {k: v.clone() for k, v in tref.stress_model(name, depth, seed).state_dict().items()}


def test_state_dict_keys_are_upstreams():
    sd = _sd()
    for k, shape in (("tokens_to_token.attention1.norm1.weight", (147,)), ("tokens_to_token.attention1.attn.qkv.weight", (192, 147)),
                     ("tokens_to_token.attention1.attn.proj.weight", (64, 64)), ("tokens_to_token.attention1.norm2.weight", (64,)),
                     ("tokens_to_token.attention1.mlp.fc1.weight", (64, 64)), ("tokens_to_token.attention1.mlp.fc2.bias", (64,)),
                     ("tokens_to_token.attention2.attn.qkv.weight", (192, 576)), ("tokens_to_token.project.weight", (384, 576)),
                     ("cls_token", (1, 1, 384)), ("pos_embed", (1, 197, 384)), ("blocks.0.attn.qkv.weight", (1152, 384))):
        assert tuple(sd[k].shape) == shape, k
    for i in (1, 2):
        assert f"tokens_to_token.attention{i}.attn.qkv.bias" not in sd
        assert f"tokens_to_token.attention{i}.kqv.weight" not in sd


def test_t2t_module_matches_the_oracle_float64():
    """nn.Unfold on NCHW pixels (columns (c, kh, kw)) == the channel-last oracle (columns (kh, kw, c)) on the converted weights:
    pins the norm1 and qkv column permutations and the project columns to nn.Unfold itself."""
    m = tref.stress_model("t2t_vit_t_14", depth=1, seed=3).double()
    csd, kw = t2t_torch_to_canonical(m.state_dict())
    assert kw["t2t"] == 3
    osd = {k: v.double() for k, v in csd.items() if k.startswith("t2t.transformer")}
    osd["t2t.project.kernel"] = csd["vit.embeddings.patch_embeddings.projection.weight"].double().t()
    osd["t2t.project.bias"] = csd["vit.embeddings.patch_embeddings.projection.bias"].double()
    x = torch.randn(2, 3, 224, 224, generator=torch.Generator().manual_seed(4), dtype=torch.float64)
    with torch.no_grad():
        want = m.tokens_to_token(x)
        got = ot2t.t2t_module(osd, x.permute(0, 2, 3, 1).contiguous())
    assert got.shape == want.shape == (2, 196, 384)
    assert (got - want).abs().max().item() <= 1e-9
    # a 64 ** -0.5 token-attention scale (the reading the oracle does not take) is visible at this precision
    assert m.tokens_to_token.attention1.attn.scale == 147 ** -0.5
    assert m.tokens_to_token.attention2.attn.scale == 576 ** -0.5


def test_key_conversion():
    sd = _sd()
    csd, kw = t2t_torch_to_canonical(sd)
    assert kw["t2t"] == 3 and kw["hidden_act"] == "gelu" and kw["layer_norm_eps"] == 1e-5
    assert not any(k.startswith("t2t.performer") for k in csd)
    for i, (C, k, n) in ((1, (3, 7, 147)), (2, (64, 3, 576))):
        s, d = f"tokens_to_token.attention{i}.", f"t2t.transformer{i}."
        g = sd[s + "norm1.weight"]
        perm = g.reshape(C, k, k).permute(1, 2, 0).reshape(-1)
        assert not torch.equal(csd[d + "norm1.gamma"], g)
        assert torch.equal(csd[d + "norm1.gamma"], perm)
        w = sd[s + "attn.qkv.weight"]
        assert tuple(csd[d + "qkv.kernel"].shape) == (n, 192)
        assert torch.equal(csd[d + "qkv.kernel"], w.reshape(192, C, k, k).permute(0, 2, 3, 1).reshape(192, n).t())
        assert torch.equal(csd[d + "attn_output.kernel"], sd[s + "attn.proj.weight"].t())
        assert torch.equal(csd[d + "mlp.fc1.kernel"], sd[s + "mlp.fc1.weight"].t())
        assert torch.equal(csd[d + "mlp.fc2.bias"], sd[s + "mlp.fc2.bias"])
        assert torch.equal(csd[d + "norm2.beta"], sd[s + "norm2.bias"])
        assert d + "qkv.bias" not in csd


def test_factory_selection(tmp_path):
    assert _factory_of(_sd("t2t_vit_t_14")) == "t2t_vit_t_14"
    assert _factory_of(_sd("t2t_vit_t_19")) == "t2t_vit_t_19"
    assert _factory_of(_sd("t2t_vit_t_24", depth=24)) == "t2t_vit_t_24"
    assert _factory_of(_sd("t2t_vit_t_14", depth=14)) == "t2t_vit_t_14"
    perf = {k: v.clone() for k, v in ref.stress_init_(ref.t2t_vit("t2t_vit_14", depth=1)).state_dict().items()}
    assert _factory_of(perf) == "t2t_vit_14"
    assert modeling_t2t.tokens_type_of(perf) == "performer" and modeling_t2t.tokens_type_of(_sd()) == "transformer"
    for name, D, L, heads, ratio in (("t2t_vit_t_14", 384, 14, 6, 3.0), ("t2t_vit_t_19", 448, 19, 7, 3.0),
                                     ("t2t_vit_t_24", 512, 24, 8, 3.0)):
        assert modeling_t2t.T2T_TORCH[name] == (D, L, heads, ratio) == tref.CONFIGS[name]
    with pytest.raises(ValueError, match="t2t_vit_t_14 is a tokens_type='transformer'"):
        modeling_t2t.t2t_vit_t_14(perf)
    with pytest.raises(ValueError, match="t2t_vit_14 is a tokens_type='performer'"):
        modeling_t2t.t2t_vit_14(_sd())
    with pytest.raises(ValueError, match="t2t_vit_t_19 is embed_dim 448"):
        modeling_t2t.t2t_vit_t_19(_sd())


def test_pth_tar_in_upstream_layout_loads_weights_only(tmp_path):
    """timm's checkpoint saver layout (state_dict_ema / args): read with weights_only=True and converted as transformer tokens."""
    sd = _sd()
    path = tmp_path / "82.6_T2T_ViTt_24.pth.tar"
    torch.save({"epoch": 309, "arch": "t2t_vit_t_14", "state_dict": sd, "state_dict_ema": sd, "version": 2, "metric": 81.7,
                "args": argparse.Namespace(model="t2t_vit_t_14", lr=5e-4, img_size=224)}, path)
    ck = modeling_t2t.load_t2t_checkpoint(path)
    csd, kw = t2t_torch_to_canonical(ck)
    assert kw["t2t"] == 3 and csd["vit.embeddings.cls_token"].shape == (1, 1, 384)


def test_rejections():
    sd = _sd()
    perf = {k: v.clone() for k, v in ref.stress_init_(ref.t2t_vit("t2t_vit_7", depth=1)).state_dict().items()}
    mixed = dict(sd, **{k: v for k, v in perf.items() if k.startswith("tokens_to_token.attention1.kqv")})
    for bad in (mixed, dict(perf, **{"tokens_to_token.attention1.attn.qkv.weight": sd["tokens_to_token.attention1.attn.qkv.weight"]})):
        with pytest.raises(ValueError, match="tokens_type='transformer'"):
            t2t_torch_to_canonical(bad)
        with pytest.raises(ValueError, match="tokens_type='transformer'"):
            B200T2TViTTorch(bad)
    biased = dict(sd, **{"tokens_to_token.attention2.attn.qkv.bias": torch.zeros(192)})
    with pytest.raises(ValueError, match="qkv bias"):
        t2t_torch_to_canonical(biased)
    with pytest.raises(ValueError, match="224"):
        t2t_torch_to_canonical(dict(sd, pos_embed=torch.zeros(1, 577, 384)))
    with pytest.raises(ValueError, match="224"):
        B200T2TViTTorch(sd, image_size=384)
    with pytest.raises(ValueError, match="224"):
        modeling_t2t.t2t_vit_t_14(sd, image_size=384)
    with pytest.raises(NotImplementedError):
        B200T2TViTTorch(sd, precision="tf32")
    with pytest.raises(NotImplementedError):
        modeling_t2t.t2t_vit_t_14(sd, precision="tf32")
    wide = dict(sd, **{"tokens_to_token.attention1.attn.qkv.weight": torch.zeros(3 * 128, 147)})
    with pytest.raises(ValueError, match="token_dim 64"):
        t2t_torch_to_canonical(wide)
