"""GPU parity of the 12 x 12-window Swin path (swin_{base,large}_patch4_window12_384): the 144-token window attention
against float32 torch, and whole models against the installed HF SwinForImageClassification run in float32 on the CPU.
Swin-L widths are covered at both window sizes.  bf16 mode: logits max-abs <= 2e-2."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import swin as osw  # noqa: E402
from oracle import vit as ovit  # noqa: E402

LOG2E = 1.4426950408889634
WIDTHS = {"base": (128, [4, 8, 16, 32]), "large": (192, [6, 12, 24, 48])}


def build_hf_swin(kind: str, depths, seed: int, image_size: int = 384, window: int = 12, stress: bool = True):
    """Random-init HF SwinForImageClassification of the given widths and geometry; ``stress`` randomises what HF initialises
    to 0 / 1 (biases, LayerNorm affine, the relative position bias tables), as oracle.swin.build_hf_swin does."""
    from transformers import SwinConfig, SwinForImageClassification
    embed_dim, heads = WIDTHS[kind]
    cfg = SwinConfig(image_size=image_size, patch_size=4, window_size=window, embed_dim=embed_dim, depths=list(depths),
                     num_heads=heads, num_labels=1000)
    torch.manual_seed(seed)
    model = SwinForImageClassification(cfg).eval()
    if stress:
        g = torch.Generator().manual_seed(seed + 1000)
        with torch.no_grad():
            for name, prm in model.named_parameters():
                if name.endswith("relative_position_bias_table"):
                    prm.copy_(torch.randn(prm.shape, generator=g) * 0.5)
                elif "norm" in name and name.endswith("weight"):
                    prm.copy_(1.0 + torch.randn(prm.shape, generator=g) * 0.1)
                elif name.endswith("bias"):
                    prm.copy_(torch.randn(prm.shape, generator=g) * 0.1)
    return model


def hf_logits(hf, x):
    with torch.no_grad():
        return hf(pixel_values=x).logits


def assert_close(got, want):
    r = ovit.compare_logits(got, want)
    assert r["max_abs"] <= 2e-2 and r["top1_agree"] == 1.0, r


@pytest.mark.parametrize("heads,n_win,n_tab", [(4, 9, 4), (4, 5, 1), (48, 3, 1), (48, 7, 4)])
def test_window_attention_144_matches_torch(heads, n_win, n_tab):
    from edgevisiontransformer_b200 import ops
    from edgevisiontransformer_b200.modeling_swin import attention_table, shift_mask
    g = torch.Generator().manual_seed(100 + heads + n_win)
    C, N = heads * 32, 144
    q, k, v = (torch.randn(n_win * N, C, generator=g) * s for s in (2.0, 2.0, 1.5))   # scores up to ~20: the row max matters
    qkv = torch.cat([q, k, v], 1).bfloat16()
    tab = torch.randn(23 * 23, heads, generator=g)
    mask = shift_mask(24, 24, 12, 6) if n_tab == 4 else None                         # the four windows of a 24 x 24 stage
    table = attention_table(tab, heads, 12, mask)
    assert tuple(table.shape) == (n_tab, heads, N, N)
    if mask is not None:
        assert (mask == -100).any() and (mask == 0).any()
    got = ops.window_attention(qkv.cuda(), table.cuda(), n_win, heads, window_tokens=N).float().cpu()
    q, k, v = [t.float().view(n_win, N, heads, 32).transpose(1, 2) for t in qkv.split(C, dim=1)]
    s = q @ k.transpose(-1, -2) / 32 ** 0.5 + table[torch.arange(n_win) % n_tab] / LOG2E
    want = (s.softmax(-1) @ v).transpose(1, 2).reshape(n_win * N, C)
    assert (got - want).abs().max() < 0.03          # bf16 probabilities and bf16 output
    assert (got - want).abs().mean() < 2e-3


def test_window_attention_rejects_other_windows():
    from edgevisiontransformer_b200 import ops
    qkv = torch.zeros(100, 3 * 32, dtype=torch.bfloat16, device="cuda")
    with pytest.raises(RuntimeError, match="49.*144"):
        ops.window_attention(qkv, torch.zeros(1, 1, 100, 100, device="cuda"), 1, 1, window_tokens=100)
    with pytest.raises(ValueError):                 # a 144-token call with the 49-token table layout
        ops.window_attention(torch.zeros(144, 96, dtype=torch.bfloat16, device="cuda"), torch.zeros(1, 1, 64, 56, device="cuda"),
                             1, 1, window_tokens=144)


def _check_model(hf, n_images, seed):
    """from_hf on n_images (max_batch 2: the chunk loop runs) against HF, then forward_graphed, the C runtime against the
    op-level composition with split-K off, and the launch count."""
    from edgevisiontransformer_b200 import ops
    from edgevisiontransformer_b200.modeling_swin import B200SwinForImageClassification
    c = hf.config
    x = ovit.synthetic_images(n_images, seed=seed, size=c.image_size)
    want = hf_logits(hf, x)
    m = B200SwinForImageClassification.from_hf(hf, max_batch=2)
    assert m.window == c.window_size and m.image_size == c.image_size
    got = m(pixel_values=x.cuda()).logits
    assert_close(got, want)
    assert_close(m.forward_graphed(x[:1].cuda()).logits, want[:1])
    try:
        ops.set_gemm_split_k(False)
        a = m(pixel_values=x[:2].cuda()).logits
        m.use_ops = True
        b = m(pixel_values=x[:2].cuda()).logits
        assert torch.equal(a, b)
    finally:
        m.use_ops = False
        ops.set_gemm_split_k(True)
    assert m.launches_per_forward() == 3 + 7 * sum(c.depths) + 2 * (len(c.depths) - 1) + 2
    assert m.num_parameters() == sum(p.numel() for p in hf.parameters())
    return m, x, want


def test_swin_base_384_reduced_depth_matches_hf():
    hf = build_hf_swin("base", [1, 1, 3, 1], seed=12)
    m, x, want = _check_model(hf, 3, seed=4)
    # the CPU oracle's restatement agrees at window 12 as well
    assert_close(m(pixel_values=x.cuda()).logits, osw.swin_forward(ovit.state_dict_of(hf), x, hf.config.depths, hf.config.num_heads,
                                                                  window=12))
    # microsoft/Swin-Transformer key names: window and image size read off the bias tables
    from edgevisiontransformer_b200.modeling_swin import B200SwinForImageClassification
    m2 = B200SwinForImageClassification.from_microsoft(osw.hf_to_microsoft(ovit.state_dict_of(hf)), depths=hf.config.depths,
                                                       num_heads=hf.config.num_heads, embed_dim=128)
    assert m2.window == 12 and m2.image_size == 384
    assert_close(m2(x[:2].cuda()).logits, want[:2])


def test_swin_base_384_full_depth_matches_hf():
    hf = build_hf_swin("base", [2, 2, 18, 2], seed=13)
    _check_model(hf, 3, seed=5)


@pytest.mark.parametrize("image_size,window", [(384, 12), (224, 7)])
def test_swin_large_matches_hf(image_size, window):
    """Swin-L widths: the widest patch-merging gather (4 x 768 = 3072) and the widest final pool (1536)."""
    hf = build_hf_swin("large", [1, 1, 3, 1], seed=14, image_size=image_size, window=window)
    _check_model(hf, 3, seed=6)


def test_swin_rejects_unsupported_windows():
    from edgevisiontransformer_b200.modeling_swin import B200SwinForImageClassification
    hf = build_hf_swin("base", [1, 1, 1, 1], seed=15, stress=False)
    sd = hf.state_dict()
    kw = dict(depths=[1, 1, 1, 1], num_heads=WIDTHS["base"][1], embed_dim=128)
    with pytest.raises(ValueError, match="7x7 and 12x12"):
        B200SwinForImageClassification(sd, window=10, image_size=320, **kw)
    with pytest.raises(ValueError):                 # 96 / (7 * 8) is not whole: the 384-pixel geometry needs window 12
        B200SwinForImageClassification(sd, window=7, image_size=384, **kw)
