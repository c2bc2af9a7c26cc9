"""BEiT / data2vec-vision without a GPU: the kernels' bias index arithmetic against the installed HF module, the LayerScale
fold, the key renaming and table expansion, config.json reading and every refusal."""
import copy

import pytest
import torch

from oracle import beit as ob


def _tiny(**kw):
    kw.setdefault("layers", 2)
    kw.setdefault("image_size", 64)
    kw.setdefault("num_labels", 10)
    return ob.build_hf_beit("base", seed=kw.pop("seed", 0), **kw)


@pytest.mark.parametrize("grid", [2, 7, 14, 24, 32])
def test_score_bias_matches_hf_index(grid):
    from transformers import BeitConfig
    from transformers.models.beit.modeling_beit import BeitRelativePositionBias
    from edgevisiontransformer_b200 import ops
    heads = 3
    rpb = BeitRelativePositionBias(BeitConfig(num_attention_heads=heads), window_size=(grid, grid))
    table = torch.randn(rpb.num_relative_distance, heads)   # asymmetric: rel(q, k) != rel(k, q) gives other values
    idx = rpb.generate_relative_position_index((grid, grid))
    want = table[idx.view(-1)].view(grid * grid + 1, grid * grid + 1, heads).permute(2, 0, 1)
    got = ops.beit_score_bias(table, grid)
    assert torch.equal(got, want)
    assert not torch.equal(got, got.transpose(1, 2))


@pytest.mark.parametrize("grid", [2, 7, 14, 32])
def test_relative_position_index_restatement(grid):
    from transformers import BeitConfig
    from transformers.models.beit.modeling_beit import BeitRelativePositionBias
    from edgevisiontransformer_b200.modeling_beit import relative_position_index
    rpb = BeitRelativePositionBias(BeitConfig(), window_size=(grid, grid))
    assert torch.equal(relative_position_index(grid), rpb.generate_relative_position_index((grid, grid)).long())


def test_layerscale_fold_float64():
    """The HF module in float64 with its lambdas against a copy holding the folded weights and lambdas = 1."""
    from edgevisiontransformer_b200.modeling_beit import beit_to_canonical
    m = _tiny().double()
    x = ob.images(2, 64, seed=3).double()
    with torch.no_grad():
        want = m(pixel_values=x).logits
        csd, _ = beit_to_canonical(dict(m.state_dict()), m.config)
        folded = copy.deepcopy(m)
        for l, layer in enumerate(folded.beit.encoder.layer):
            p = f"vit.encoder.layer.{l}."
            layer.attention.output.dense.weight.copy_(csd[p + "attention.output.dense.weight"])
            layer.attention.output.dense.bias.copy_(csd[p + "attention.output.dense.bias"])
            layer.output.dense.weight.copy_(csd[p + "output.dense.weight"])
            layer.output.dense.bias.copy_(csd[p + "output.dense.bias"])
            layer.lambda_1.fill_(1.0)
            layer.lambda_2.fill_(1.0)
        got = folded(pixel_values=x).logits
    assert (got - want).abs().max().item() <= 1e-9
    assert (m.beit.encoder.layer[0].lambda_1 != 1).any()


def test_beit_and_data2vec_prefixes_give_the_same_dict():
    from edgevisiontransformer_b200.modeling_beit import beit_to_canonical
    a = _tiny(seed=1)
    b = _tiny(seed=1, data2vec=True)
    b.load_state_dict({k.replace("beit.", "data2vec_vision.", 1): v for k, v in a.state_dict().items()})
    ca, cfa = beit_to_canonical(dict(a.state_dict()), a.config)
    cb, cfb = beit_to_canonical(dict(b.state_dict()), b.config)
    assert cfa == cfb and cfa.final_ln == 2 and cfa.tokens == 17
    assert set(ca) == set(cb) and all(torch.equal(ca[k], cb[k]) for k in ca)
    L = cfa.num_hidden_layers
    assert all(f"vit.encoder.layer.{l}.attention.attention.key.bias" in ca for l in range(L))
    assert torch.equal(ca["vit.embeddings.position_embeddings"], torch.zeros(1, 17, 768))
    assert not any("lambda" in k or "pooler" in k for k in ca)


def test_shared_table_expands_to_every_layer():
    from edgevisiontransformer_b200.modeling_beit import beit_to_canonical
    m = _tiny(layers=3, use_relative_position_bias=False, use_shared_relative_position_bias=True)
    sd = dict(m.state_dict())
    shared = sd["beit.encoder.relative_position_bias.relative_position_bias_table"]
    csd, _ = beit_to_canonical(sd, m.config)
    for l in range(3):
        assert torch.equal(csd[f"vit.encoder.layer.{l}.attention.attention.relative_position_bias.relative_position_bias_table"], shared)
    assert not any(k.startswith("vit.encoder.relative_position_bias") for k in csd)


def test_cls_pooling_keeps_the_final_layernorm():
    from edgevisiontransformer_b200.modeling_beit import beit_to_canonical
    m = _tiny(use_mean_pooling=False, use_absolute_position_embeddings=True)
    csd, cfg = beit_to_canonical(dict(m.state_dict()), m.config)
    assert cfg.final_ln is True and torch.equal(csd["vit.layernorm.weight"], m.beit.layernorm.weight)
    assert torch.equal(csd["vit.embeddings.position_embeddings"], m.beit.embeddings.position_embeddings)


def test_relative_position_index_buffers_are_checked():
    from edgevisiontransformer_b200.modeling_beit import beit_to_canonical, relative_position_index
    m = _tiny()
    sd = dict(m.state_dict())
    key = "beit.encoder.layer.1.attention.attention.relative_position_bias.relative_position_index"
    csd, _ = beit_to_canonical({**sd, key: relative_position_index(4)}, m.config)
    assert not any(k.endswith("relative_position_index") for k in csd)
    with pytest.raises(ValueError, match="does not match a 4 x 4 patch grid"):
        beit_to_canonical({**sd, key: relative_position_index(4).t().contiguous()}, m.config)


@pytest.mark.parametrize("data2vec", [False, True])
def test_config_json_round_trip(tmp_path, data2vec):
    from edgevisiontransformer_b200.modeling_beit import beit_to_canonical, read_beit_checkpoint
    m = _tiny(seed=2, data2vec=data2vec, use_shared_relative_position_bias=True, use_relative_position_bias=False)
    m.save_pretrained(tmp_path)
    sd, config = read_beit_checkpoint(str(tmp_path))
    assert config["model_type"] == ("data2vec-vision" if data2vec else "beit")
    got, gcfg = beit_to_canonical(sd, config)
    want, wcfg = beit_to_canonical(dict(m.state_dict()), m.config)
    assert gcfg == wcfg and set(got) == set(want) and all(torch.equal(got[k], want[k]) for k in want)


def test_config_json_of_another_model_is_refused(tmp_path):
    from edgevisiontransformer_b200.modeling_beit import read_beit_checkpoint
    (tmp_path / "config.json").write_text('{"model_type": "vit"}')
    with pytest.raises(ValueError, match="model_type"):
        read_beit_checkpoint(str(tmp_path))
    (tmp_path / "config.json").write_text('{"model_type": "beit", "architectures": ["BeitForMaskedImageModeling"]}')
    with pytest.raises(ValueError, match="architectures"):
        read_beit_checkpoint(str(tmp_path))


def _refuses(match, fn):
    """ValueError, raised before the constructor touches the device (on a machine without a GPU it would fail otherwise)."""
    with pytest.raises(ValueError, match=match):
        fn()


def test_refusals_before_allocation():
    from transformers import BeitConfig, BeitForMaskedImageModeling, BeitForSemanticSegmentation
    from edgevisiontransformer_b200.modeling_beit import B200BeitForImageClassification as B
    m = _tiny()
    sd = dict(m.state_dict())
    _refuses("bf16 mode only", lambda: B.from_hf(m, precision="tf32"))
    _refuses("is not implemented", lambda: B.from_hf(BeitForMaskedImageModeling(BeitConfig(num_hidden_layers=1, image_size=32))))
    _refuses("is not implemented", lambda: B.from_hf(BeitForSemanticSegmentation(BeitConfig(num_hidden_layers=4, image_size=32, out_indices=[0, 1, 2, 3]))))
    _refuses("no classifier.weight", lambda: B.from_state_dict({k: v for k, v in sd.items() if not k.startswith("classifier.")}, m.config))
    _refuses("unexpected key", lambda: B.from_state_dict({**sd, "lm_head.weight": torch.zeros(1)}, m.config))
    big = copy.deepcopy(m.config)
    big.image_size = 528    # 33 x 33 patches + cls = 1090 tokens
    _refuses("at most 1026", lambda: B.from_state_dict(sd, big))
    pruned = copy.deepcopy(m.config)
    pruned.pruned_heads = {0: [1]}
    _refuses("head-pruned", lambda: B.from_state_dict(sd, pruned))
    uneven = dict(sd)
    t = "beit.encoder.layer.1.attention.attention.relative_position_bias.relative_position_bias_table"
    uneven[t] = sd[t][:, :11]
    _refuses("uneven heads", lambda: B.from_state_dict(uneven, m.config))
    h80 = copy.deepcopy(m.config)
    h80.num_attention_heads = 8
    _refuses("only head size 64", lambda: B.from_state_dict(sd, h80))
    _refuses("needs the model's config", lambda: B.from_state_dict(sd))
    nolayer = {k: v for k, v in sd.items() if "lambda_2" not in k or ".0." not in k}
    _refuses("one residual branch", lambda: B.from_state_dict(nolayer, m.config))


def test_mean_pooling_without_any_bias_is_plain_vit_with_a_pooled_head():
    """Accepted on purpose: no tables (the runtime's bias-free attention) and the mean-pooled head."""
    from edgevisiontransformer_b200.modeling_beit import beit_to_canonical
    m = _tiny(use_relative_position_bias=False)
    csd, cfg = beit_to_canonical(dict(m.state_dict()), m.config)
    assert cfg.final_ln == 2 and not any("relative_position" in k for k in csd)
