"""PyTorch T2T-ViT checkpoints without a GPU: the weight converter against nn.Unfold, checkpoint wrappers and files, rejections."""
import argparse
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import t2t_torch_ref as ref  # noqa: E402
from edgevisiontransformer_b200.dialects import t2t_torch_to_canonical  # noqa: E402
from edgevisiontransformer_b200.modeling_t2t import B200T2TViTTorch, load_t2t_checkpoint, t2t_vit_14  # noqa: E402
from oracle import t2t as ot2t  # noqa: E402


def _model(name="t2t_vit_7", depth=1, seed=0, **kw):
    torch.manual_seed(seed)
    return ref.stress_init_(ref.t2t_vit(name, depth=depth, **kw), seed=seed)


def _sd(name="t2t_vit_7", depth=1, seed=0):
    return {k: v.clone() for k, v in _model(name, depth, seed).state_dict().items()}


def test_state_dict_keys_are_upstreams():
    sd = _sd()
    for k, shape in (("tokens_to_token.attention1.kqv.weight", (192, 147)), ("tokens_to_token.attention1.w", (32, 64)),
                     ("tokens_to_token.attention1.mlp.0.weight", (64, 64)), ("tokens_to_token.attention1.mlp.2.weight", (64, 64)),
                     ("tokens_to_token.attention2.norm1.weight", (576,)), ("tokens_to_token.project.weight", (256, 576)),
                     ("cls_token", (1, 1, 256)), ("pos_embed", (1, 197, 256)), ("blocks.0.attn.qkv.weight", (768, 256)),
                     ("blocks.0.mlp.fc1.weight", (512, 256)), ("norm.weight", (256,)), ("head.weight", (1000, 256))):
        assert tuple(sd[k].shape) == shape, k
    assert "blocks.0.attn.qkv.bias" not in sd


def test_t2t_module_matches_the_tf_restatement_float64():
    """nn.Unfold on NCHW pixels (columns (c, kh, kw)) == the channel-last restatement (columns (kh, kw, c)) on the converted
    weights: pins every column permutation of the converter to nn.Unfold itself."""
    m = _model(gelu="tanh", seed=3).double()
    csd, _ = t2t_torch_to_canonical(m.state_dict())
    osd = {k: v.double() for k, v in csd.items() if k.startswith("t2t.performer")}
    osd["t2t.project.kernel"] = csd["vit.embeddings.patch_embeddings.projection.weight"].double().t()
    osd["t2t.project.bias"] = csd["vit.embeddings.patch_embeddings.projection.bias"].double()
    x = torch.randn(2, 3, 224, 224, generator=torch.Generator().manual_seed(4), dtype=torch.float64)
    with torch.no_grad():
        want = m.tokens_to_token(x)
        got = ot2t.t2t_module(osd, x.permute(0, 2, 3, 1).contiguous())
    assert got.shape == want.shape == (2, 196, 256)
    assert (got - want).abs().max().item() <= 1e-9


def test_norm1_permutation_is_not_symmetric():
    """the stress init gives norm1 a profile that a missing or wrong permutation changes"""
    sd = _sd()
    csd, _ = t2t_torch_to_canonical(sd)
    g = sd["tokens_to_token.attention1.norm1.weight"]
    assert not torch.equal(csd["t2t.performer1.norm1.gamma"], g)
    assert torch.equal(csd["t2t.performer1.norm1.gamma"], g.reshape(3, 7, 7).permute(1, 2, 0).reshape(-1))


def test_qk_scale_folds_into_the_query_rows():
    sd = _sd()
    a, _ = t2t_torch_to_canonical(sd)
    b, _ = t2t_torch_to_canonical(sd, qk_scale=0.05)
    w = sd["blocks.0.attn.qkv.weight"]
    assert torch.equal(a["vit.encoder.layer.0.attention.attention.query.weight"], w[:256])
    torch.testing.assert_close(b["vit.encoder.layer.0.attention.attention.query.weight"], w[:256] * 0.05 * 8, rtol=0, atol=0)
    assert torch.equal(b["vit.encoder.layer.0.attention.attention.key.weight"], w[256:512])
    assert torch.equal(b["vit.encoder.layer.0.attention.attention.value.weight"], w[512:])


def test_checkpoint_wrappers_and_module_prefix():
    sd, other = _sd(seed=0), _sd(seed=1)
    ref_csd, _ = t2t_torch_to_canonical(sd)
    alt_csd, _ = t2t_torch_to_canonical(other)
    pre = {"module." + k: v for k, v in sd.items()}
    key = "t2t.performer1.kqv.kernel"
    for ck, want in ((sd, ref_csd), ({"state_dict_ema": sd, "state_dict": other}, ref_csd), ({"state_dict": pre}, ref_csd),
                     ({"model": pre, "epoch": 3}, ref_csd), ({"state_dict_ema": pre, "state_dict": other}, ref_csd)):
        got, _ = t2t_torch_to_canonical(ck)
        assert got.keys() == want.keys()
        assert torch.equal(got[key], want[key])
    got, _ = t2t_torch_to_canonical({"state_dict_ema": sd, "state_dict": other}, use_ema=False)
    assert torch.equal(got[key], alt_csd[key])


def test_pth_tar_with_args_namespace_loads_weights_only(tmp_path):
    """timm's checkpoint saver layout: an argparse.Namespace under 'args' loads with weights_only=True (allow-listed)."""
    sd = _sd()
    path = tmp_path / "81.5_T2T_ViT_14.pth.tar"
    torch.save({"epoch": 309, "arch": "t2t_vit_7", "state_dict": sd, "state_dict_ema": sd, "version": 2, "metric": 71.7,
                "args": argparse.Namespace(model="t2t_vit_7", lr=5e-4, img_size=224)}, path)
    with pytest.raises(Exception):
        torch.load(path, map_location="cpu", weights_only=True)       # without the allow-list: refused
    ck = load_t2t_checkpoint(path)
    assert ck["args"].model == "t2t_vit_7"
    csd, kw = t2t_torch_to_canonical(ck)
    assert kw["t2t"] == 2 and csd["vit.embeddings.cls_token"].shape == (1, 1, 256)


def test_rejections():
    sd = _sd()
    tt = dict(sd, **{"tokens_to_token.attention1.attn.qkv.weight": torch.zeros(147 * 3, 147)})
    with pytest.raises(ValueError, match="tokens_type='transformer'"):
        t2t_torch_to_canonical(tt)
    with pytest.raises(ValueError, match="tokens_type='transformer'"):
        B200T2TViTTorch(tt)
    big = dict(sd, pos_embed=torch.zeros(1, 577, 256))
    with pytest.raises(ValueError, match="224"):
        t2t_torch_to_canonical(big)
    with pytest.raises(ValueError, match="224"):
        B200T2TViTTorch(sd, image_size=384)
    with pytest.raises(NotImplementedError):
        B200T2TViTTorch(sd, precision="tf32")
    with pytest.raises(ValueError, match="head size"):
        B200T2TViTTorch(sd, num_heads=8)
    with pytest.raises(ValueError, match="not a PyTorch T2T-ViT"):
        t2t_torch_to_canonical({"cls_token": torch.zeros(1, 1, 256)})
    with pytest.raises(ValueError, match="t2t_vit_14 is embed_dim 384"):
        t2t_vit_14(sd)
