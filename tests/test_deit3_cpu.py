"""DeiT III loading on the CPU: LayerScale folded into the residual projections, cls-free position rows, both key layouts,
and the variants that are refused.  The folded canonical weights through oracle.vit match the models_v2 restatement
(tests/deit3_ref.py) in float64."""
import os
import sys

import pytest
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import deit3_ref as ref  # noqa: E402
from edgevisiontransformer_b200 import modeling_vit  # noqa: E402
from edgevisiontransformer_b200.dialects import deit3_head_size, timm_vit_to_canonical  # noqa: E402
from oracle import vit as ovit  # noqa: E402
from oracle.spec import ViTSpec  # noqa: E402


def _oracle64(csd, spec, x):
    """oracle.vit's embeddings / encoder layers / head composed in float64 (vit_forward casts its input to f32)."""
    h = ovit.patch_embed(csd, x, spec.patch)
    h = torch.cat((csd["vit.embeddings.cls_token"].expand(x.shape[0], -1, -1), h), dim=1) + csd["vit.embeddings.position_embeddings"]
    for l in range(spec.layers):
        h = ovit.encoder_layer(csd, l, h, spec)
    h = F.layer_norm(h, (spec.hidden,), csd["vit.layernorm.weight"], csd["vit.layernorm.bias"], spec.eps)
    return F.linear(h[:, 0], csd["classifier.weight"], csd["classifier.bias"])


def test_restatement_uses_models_v2_keys():
    sd = ref.build("small", depth=1).state_dict()
    assert {"cls_token", "pos_embed", "patch_embed.proj.weight", "norm.weight", "head.weight"} <= set(sd)
    assert {f"blocks.0.{n}" for n in ("gamma_1", "gamma_2", "attn.qkv.bias", "attn.proj.weight", "mlp.fc2.bias")} <= set(sd)
    assert sd["pos_embed"].shape == (1, 196, 384)
    assert "blocks.0.ls1.gamma" in ref.to_timm_keys(sd)


@pytest.mark.parametrize("dims,image", [((128, 2, 16), 64), ((160, 2, 14), 56), ((128, 2, 16), 48)])
def test_folded_weights_match_restatement_f64(dims, image):
    m = ref.build("small", image=image, seed=3, num_classes=10, dims=dims).double()
    x = torch.randn(2, 3, image, image, generator=torch.Generator().manual_seed(4), dtype=torch.float64)
    with torch.no_grad():
        want = m(x)
    csd, kw = timm_vit_to_canonical(m.state_dict(), patch=dims[2])
    assert csd["vit.embeddings.position_embeddings"].shape[1] == (image // dims[2]) ** 2 + 1
    assert torch.all(csd["vit.embeddings.position_embeddings"][0, 0] == 0)
    spec = ViTSpec(hidden=dims[0], layers=2, heads=[dims[1]] * 2, inter=[4 * dims[0]] * 2, head_size=dims[0] // dims[1],
                   tokens=(image // dims[2]) ** 2 + 1, eps=kw["layer_norm_eps"], num_labels=10, image=image, patch=dims[2])
    got = _oracle64(csd, spec, x)
    assert (got - want).abs().max().item() <= 1e-9


def test_layerscale_moves_logits():
    """The fold is not a no-op on stress-initialised gammas: dropping it changes the logits."""
    m = ref.build("small", image=48, seed=5, num_classes=10, dims=(128, 2, 16)).double()
    x = torch.randn(1, 3, 48, 48, dtype=torch.float64)
    sd = {k: v for k, v in m.state_dict().items() if "gamma" not in k}
    plain, _ = timm_vit_to_canonical(sd, patch=16)
    folded, _ = timm_vit_to_canonical(m.state_dict(), patch=16)
    spec = ViTSpec(hidden=128, layers=2, heads=[2] * 2, inter=[512] * 2, tokens=10, eps=1e-6, num_labels=10, image=48)
    assert (_oracle64(plain, spec, x) - _oracle64(folded, spec, x)).abs().max().item() > 1e-2


def test_both_key_layouts_give_the_same_canonical_dict():
    sd = ref.build("small", depth=2, seed=7).state_dict()
    a, ka = timm_vit_to_canonical(sd)
    b, kb = timm_vit_to_canonical(ref.to_timm_keys(sd))
    c, _ = timm_vit_to_canonical({"model": sd})
    assert ka == kb and set(a) == set(b) == set(c)
    for k in a:
        assert torch.equal(a[k], b[k]) and torch.equal(a[k], c[k]), k


def test_fold_is_f32_and_exact():
    sd = ref.build("small", depth=1, seed=9).state_dict()
    csd, _ = timm_vit_to_canonical(sd)
    w = csd["vit.encoder.layer.0.output.dense.weight"]
    assert w.dtype == torch.float32
    assert torch.equal(w, sd["blocks.0.mlp.fc2.weight"] * sd["blocks.0.gamma_2"][:, None])
    assert torch.equal(csd["vit.encoder.layer.0.attention.output.dense.bias"], sd["blocks.0.attn.proj.bias"] * sd["blocks.0.gamma_1"])
    half, _ = timm_vit_to_canonical({k: v.bfloat16() for k, v in sd.items()})
    assert half["vit.encoder.layer.0.output.dense.weight"].dtype == torch.float32


def test_head_size_of_deit3():
    huge = {"cls_token": torch.zeros(1, 1, 1280), "blocks.0.gamma_1": torch.zeros(1280)}
    assert deit3_head_size(huge) == 80
    assert deit3_head_size({"model": huge}) == 80
    assert deit3_head_size({"cls_token": torch.zeros(1, 1, 1280)}) == 64      # a plain ViT-H keeps the default
    assert deit3_head_size(ref.build("base", depth=1).state_dict()) == 64


def test_refusals():
    sd = ref.build("small", depth=2, seed=11).state_dict()
    par = dict(sd, **{"blocks.0.attn1.qkv.weight": torch.zeros(3 * 384, 384), "blocks.0.gamma_1_1": torch.zeros(384)})
    with pytest.raises(ValueError, match="deit_huge_patch14_26x2_LS"):
        timm_vit_to_canonical(par)
    giant = {k: (torch.zeros(1, 1, 1408) if k == "cls_token" else v) for k, v in sd.items()}
    with pytest.raises(ValueError, match="Giant.*head size 88"):
        timm_vit_to_canonical(giant)
    one = {k: v for k, v in sd.items() if k != "blocks.1.gamma_2"}
    with pytest.raises(ValueError, match="one residual branch"):
        timm_vit_to_canonical(one)
    stray = dict(sd, **{"blocks.5.gamma_1": torch.ones(384)})
    with pytest.raises(ValueError, match="LayerScale parameters of blocks"):
        timm_vit_to_canonical(stray)
    both = dict(sd, **{"blocks.0.ls1.gamma": sd["blocks.0.gamma_1"]})
    with pytest.raises(ValueError, match="both"):
        timm_vit_to_canonical(both)
    bad = dict(sd, **{"blocks.0.gamma_2": torch.ones(100)})
    with pytest.raises(ValueError, match="LayerScale has 100 entries"):
        timm_vit_to_canonical(bad)


def test_factories_check_shapes_before_building():
    small = ref.build("small", depth=1).state_dict()
    with pytest.raises(ValueError, match="deit3_base_patch16_224 is embed dim 768"):
        modeling_vit.deit3_base_patch16_224(small)
    with pytest.raises(ValueError, match="deit3_huge_patch14_224 is embed dim 1280"):
        modeling_vit.deit3_huge_patch14_224(small)
    with pytest.raises(ValueError, match="576 patches; the weights have 196"):
        modeling_vit.deit3_small_patch16_384(small)
    with pytest.raises(ValueError, match="no blocks.*gamma_1"):
        modeling_vit.deit3_small_patch16_224({k: v for k, v in small.items() if "gamma" not in k})
    par = dict(small, **{"blocks.0.mlp1.fc1.weight": torch.zeros(1536, 384)})
    with pytest.raises(ValueError, match="parallel-block"):
        modeling_vit.deit3_small_patch16_224(par)


def test_factory_reads_a_checkpoint_file(tmp_path):
    sd = ref.build("small", depth=1).state_dict()
    p = tmp_path / "deit_3_small_224_1k.pth"
    torch.save({"model": ref.to_timm_keys(sd)}, p)
    with pytest.raises(ValueError, match="deit3_medium_patch16_224 is embed dim 512"):
        modeling_vit.deit3_medium_patch16_224(str(p))
