"""Swin V2 without a GPU: the host-side CPB tables and the kernel's index / mask arithmetic against the installed HF
Swinv2 module, the microsoft -> HF renaming, the factory shape checks and every refusal."""
import pytest
import torch

from oracle import swinv2 as osv2


@pytest.mark.parametrize("window,pretrained", [(8, 0), (16, 0), (8, 12), (16, 12), (8, 6)])
def test_cpb_table_matches_hf(window, pretrained):
    from transformers import Swinv2Config
    from transformers.models.swinv2.modeling_swinv2 import Swinv2SelfAttention
    from edgevisiontransformer_b200 import ops
    torch.manual_seed(window + pretrained)
    heads = 6
    attn = Swinv2SelfAttention(Swinv2Config(), 192, heads, window, [pretrained, pretrained]).eval()
    with torch.no_grad():
        for p in attn.continuous_position_bias_mlp.parameters():
            p.copy_(torch.randn(p.shape) * 0.1)
    mlp = attn.continuous_position_bias_mlp
    with torch.no_grad():
        want = 16 * torch.sigmoid(mlp.double()(attn.relative_coords_table.double()).view(-1, heads)).t().float()
    got = ops.swinv2_cpb_table(mlp[0].weight, mlp[0].bias, mlp[2].weight, window, pretrained)
    assert got.shape == want.shape == (heads, (2 * window - 1) ** 2)
    assert (got - want).abs().max().item() <= 1e-6


@pytest.mark.parametrize("window,grid,shift", [(8, 64, 4), (8, 16, 4), (16, 64, 8), (16, 32, 8), (8, 8, 0), (16, 16, 0)])
def test_score_bias_index_and_mask_match_hf(window, grid, shift):
    """Dense restatement of the kernel's bias index and shift-mask region against relative_position_index + get_attn_mask."""
    from transformers import Swinv2Config
    from transformers.models.swinv2.modeling_swinv2 import Swinv2Layer, Swinv2SelfAttention
    from edgevisiontransformer_b200 import ops
    heads, N = 2, window * window
    table = torch.randn(heads, (2 * window - 1) ** 2)
    got = ops.swinv2_score_bias(table, window, grid, shift, mask=-200.0)
    rpi = Swinv2SelfAttention(Swinv2Config(), 64, heads, window).relative_position_index
    bias = table.t()[rpi.view(-1)].view(N, N, heads).permute(2, 0, 1)
    layer = Swinv2Layer(Swinv2Config(window_size=window), 64, (grid, grid), heads, shift_size=shift)
    assert layer.shift_size == shift and layer.window_size == window
    mask = layer.get_attn_mask(grid, grid, torch.float32)
    want = bias.unsqueeze(0).expand((grid // window) ** 2, -1, -1, -1).clone()
    if mask is not None:
        want += 2 * mask.unsqueeze(1)                   # -100 added twice = the -200 given above
        assert (mask != 0).any()
    assert torch.equal(got, want)


def test_microsoft_names_equal_hf_names():
    from edgevisiontransformer_b200.modeling_swinv2 import hf_to_canonical, microsoft_to_canonical
    hf = osv2.build_hf_swinv2("tiny", seed=3, depths=[2, 2, 2, 2], stress=True, num_labels=10)
    a = hf_to_canonical(hf.state_dict())
    b = microsoft_to_canonical({"model": osv2.to_microsoft(hf)})
    assert sorted(a) == sorted(b)
    for k in a:
        assert torch.equal(a[k], b[k]), k


def test_microsoft_buffers_are_verified():
    from edgevisiontransformer_b200.modeling_swinv2 import verify_microsoft_buffers
    ms = osv2.to_microsoft(osv2.build_hf_swinv2("tiny", seed=1, depths=[2, 2, 2, 2], window=16, num_labels=10))
    verify_microsoft_buffers(ms, 256, 16, [0, 0, 0, 0], 4)
    with pytest.raises(ValueError, match="pretrained window"):
        verify_microsoft_buffers(ms, 256, 16, [12, 12, 12, 6], 4)
    with pytest.raises(ValueError, match="window 8"):
        verify_microsoft_buffers(ms, 256, 8, [0, 0, 0, 0], 4)


def test_factory_checks_shapes():
    from edgevisiontransformer_b200 import modeling_swinv2 as m
    sd = osv2.build_hf_swinv2("tiny", seed=0, depths=[2, 2, 2, 2], num_labels=10).state_dict()
    with pytest.raises(ValueError, match="not swinv2_tiny_patch4_window8_256"):
        m.swinv2_tiny_patch4_window8_256(sd)          # depths 2, 2, 2, 2 are not tiny's 2, 2, 6, 2
    with pytest.raises(ValueError, match="not swinv2_base_patch4_window16_256"):
        m.swinv2_base_patch4_window16_256(sd)
    ms = osv2.to_microsoft(osv2.build_hf_swinv2("tiny", seed=0, depths=[2, 2, 2, 2], window=8, num_labels=10))
    with pytest.raises(ValueError, match="does not match window 16"):
        m.swinv2_tiny_patch4_window16_256({"model": ms})   # the buffers say window 8


@pytest.mark.parametrize("kw,match", [
    (dict(precision="tf32"), "bf16 only"),
    (dict(image_size=192, window=12), "12 x 12 window"),                 # the 192-pixel 22k models
    (dict(image_size=384, window=24), "24 x 24 window"),                 # window12to24_384: 576-token windows
    (dict(image_size=224, window=7), "7 x 7 window"),
    (dict(embed_dim=64), "head size 32"),
])
def test_refusals_before_allocation(kw, match):
    """Raised before any device or library call: the same refusals on a machine without a GPU."""
    from edgevisiontransformer_b200.modeling_swinv2 import B200Swinv2ForImageClassification
    args = dict(state_dict={}, depths=[2, 2, 6, 2], num_heads=[3, 6, 12, 24], embed_dim=96, window=8, image_size=256)
    args.update(kw)
    with pytest.raises(ValueError, match=match):
        B200Swinv2ForImageClassification(**args)


def test_timm_names_are_refused():
    from edgevisiontransformer_b200.modeling_swinv2 import microsoft_to_canonical
    with pytest.raises(ValueError, match="unexpected key"):
        microsoft_to_canonical({"stages.0.blocks.0.attn.qkv.weight": torch.zeros(3, 1)})


def test_header_declares_v2_spec_fields():
    import ctypes as C
    from edgevisiontransformer_b200 import _lib
    # image, patch, window, embed_dim, stages, depths[8], heads[8], num_labels, eps, precision, version, pretrained_window[8], mask_adds
    assert C.sizeof(_lib.SwinSpec) == 4 * (5 + 8 + 8 + 3 + 1 + 8 + 1)
    assert _lib.SwinSpec.version.offset == 4 * (5 + 16 + 3)
