"""GPU tests of the classification-row tail: the last encoder layer runs its attention for the cls query only and its
out-projection, LayerNorm, FC1 and FC2 on one row per image (csrc/model.cu).  Asking for the last layer's context
(`capture_context`) makes that layer run on every row, so each case compares the default forward with the full one on the
same model.  K splitting is off wherever bits are compared: split-K reduce-adds land in any order."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import ViTSpec  # noqa: E402
from oracle import pruning as opr  # noqa: E402
from oracle import tf_vit as otf  # noqa: E402
from oracle import vit as ovit  # noqa: E402


@pytest.fixture
def no_split_k():
    from edgevisiontransformer_b200 import ops
    ops.set_gemm_split_k(False)
    yield
    ops.set_gemm_split_k(True)


def _model(sd, **kw):
    from edgevisiontransformer_b200 import B200ViTForImageClassification
    return B200ViTForImageClassification.from_state_dict(sd, **kw)


def _tail_and_full(m, x, **kw):
    """-> (logits of the default forward, logits with every layer on all rows)."""
    m.capture_context(False)
    tail = m(x, **kw).logits.clone()
    m.capture_context(True)
    full = m(x, **kw).logits.clone()
    m.capture_context(False)
    return tail, full


def _last_layer_mask(layers, heads):
    mask = torch.ones(layers, heads)
    mask[layers - 1, 0] = 0.0
    mask[layers - 1, heads - 1] = 0.5
    mask[2, heads // 2] = 0.0
    return mask


@pytest.mark.parametrize("S", [197, 198, 50])
@pytest.mark.parametrize("Sq", [1, 2])
@pytest.mark.parametrize("B", [3, 160])
def test_attention_query_rows_are_the_full_rows(S, Sq, B):
    """Rows < Sq of the query-row mode are bit-identical to the same rows of the full kernel (B = 3 splits the query tiles
    of a pair across CTAs in the full run, B = 160 does not)."""
    from edgevisiontransformer_b200 import ops
    heads = 3
    g = torch.Generator().manual_seed(S * 10 + Sq)
    qkv = (torch.randn(B * S, 3 * heads * 64, generator=g) * 2).bfloat16().cuda()
    mask = torch.tensor([1.0, 0.0, 0.5], device="cuda")
    for hm in (None, mask):
        full = ops.attention(qkv, B, S, heads, head_mask=hm).view(B, S, -1)
        rows = ops.attention(qkv, B, S, heads, head_mask=hm, q_rows=Sq)
        assert rows.shape == (B * Sq, heads * 64)
        assert torch.equal(rows.view(B, Sq, -1), full[:, :Sq])


@pytest.mark.parametrize("kind", ["tiny", "small"])
@pytest.mark.parametrize("bs", [1, 5, 64])
def test_deit_tail_is_bit_identical(kind, bs, no_split_k):
    spec = ViTSpec.deit(kind)
    sd = ovit.state_dict_of(ovit.build_hf_model(spec, seed=3, stress=True))
    m = _model(sd)
    x = ovit.synthetic_images(bs, seed=4).cuda()
    tail, full = _tail_and_full(m, x)
    assert torch.equal(tail, full)
    mask = _last_layer_mask(spec.layers, spec.heads[0])
    tail_m, full_m = _tail_and_full(m, x, head_mask=mask)
    assert torch.equal(tail_m, full_m)
    assert (tail_m - tail).abs().max().item() > 1e-3     # the mask reaches the tail's attention


def test_base_sized_tail_on_cta_pair_shapes(no_split_k):
    """D = 768 at a batch where the full-size GEMMs run on CTA pairs; the launch structure is that of the full layer."""
    spec = ViTSpec.deit("base")
    sd = ovit.state_dict_of(ovit.build_hf_model(spec, seed=1, stress=True))
    m = _model(sd)
    x = ovit.synthetic_images(256, seed=2).cuda()
    tail, full = _tail_and_full(m, x)
    assert torch.equal(tail, full)
    assert m.launches_per_forward() == 3 + 7 * 12 + 2
    m.profile_begin()
    m(x[:4])
    st = m.profile_end()
    L = spec.layers
    assert {k: n for k, (_, n) in st.items()} == {"embed": 3, "layernorm": 2 * L, "qkv": L, "attention": L, "out_proj": L,
                                                  "fc1": L, "fc2": L, "head": 2}


def test_tf_dialect_tail_is_bit_identical(no_split_k):
    """TF dialect: the LayerNorms copy their output into the residual stream; LN2 of the tail writes the cls rows only."""
    from edgevisiontransformer_b200.dialects import tf_vit_to_canonical
    sd, heads, _ = otf.init_tf_vit(dim=192, depth=12, seed=1, stress=True)
    csd, kw = tf_vit_to_canonical(sd, heads)
    m = _model(csd, **kw)
    x = ovit.synthetic_images(5, seed=2).cuda()
    tail, full = _tail_and_full(m, x)
    assert torch.equal(tail, full)


def test_t2t_tail_is_bit_identical(no_split_k):
    from edgevisiontransformer_b200.modeling_t2t import B200T2TViT
    from oracle import t2t as ot2t
    sd = ot2t.init_t2t_vit(hidden=384, depth=3, num_heads=6, mlp_ratio=3.0, seed=0, stress=True)
    m = B200T2TViT(sd, depth=3, num_heads=6)
    x = ovit.synthetic_images(3, seed=4, channels_last=True).cuda()
    tail = m(x).logits
    c = m.core.config
    ctx = [torch.empty((3 * c.tokens, h * c.head_size), dtype=torch.bfloat16, device="cuda") for h in c.heads]
    full = torch.empty_like(tail)
    m.core._run(x, full, ctx=ctx)
    assert torch.equal(tail, full)


@pytest.mark.parametrize("case", ["h1_d230", "head18_uneven"])
def test_pruned_tiny_tail_is_bit_identical(case, golden_dir, no_split_k):
    import os
    spec = ViTSpec.deit("tiny")
    sd = ovit.state_dict_of(ovit.build_hf_model(spec, seed=4, stress=True))
    f = np.load(os.path.join(golden_dir, f"pruned_tiny_{case}.npz"))
    heads_kept = [[0]] * 12 if case == "h1_d230" else opr.kept_heads_from_pruned_str(opr.DEIT_TINY_HEAD18, 12, 3)
    _, pruned, _ = opr.synthesize_pruned(sd, heads_kept, [int(v) for v in f["inter_kept"]], seed=7)
    m = _model(pruned)
    x = ovit.synthetic_images(5, seed=1).cuda()
    tail, full = _tail_and_full(m, x)
    assert torch.equal(tail, full)


def test_distilled_two_heads_keep_the_full_layer(no_split_k):
    """head_rows = 2 reads rows 0 and 1 of every image; the last layer stays whole for it (same launches, same bits)."""
    from transformers import DeiTConfig, DeiTForImageClassificationWithTeacher
    from edgevisiontransformer_b200 import B200ViTForImageClassification
    cfg = DeiTConfig(hidden_size=192, num_hidden_layers=12, num_attention_heads=3, intermediate_size=768, num_labels=1000,
                     attn_implementation="eager")
    torch.manual_seed(21)
    hf = DeiTForImageClassificationWithTeacher(cfg).eval()
    m = B200ViTForImageClassification.from_hf(hf)
    assert m.config.head_rows == 2
    x = ovit.synthetic_images(5, seed=9)
    tail, full = _tail_and_full(m, x.cuda())
    assert torch.equal(tail, full)
    with torch.no_grad():
        want = hf(pixel_values=x).logits
    r = ovit.compare_logits(tail, want)
    assert r["max_abs"] <= 2e-2 and r["top1_agree"] == 1.0, r


def test_row_ln_models_at_large_batch(no_split_k):
    """D = 192 / 384 at large batch: the full layer-11 out-projection carries LN2 in its epilogue (gemm_rowln), the tail
    runs the plain GEMM and the LayerNorm kernel.  The two give the same logits bit for bit (measured on a B200), and the
    test holds them to that."""
    for kind in ("tiny", "small"):
        spec = ViTSpec.deit(kind)
        sd = ovit.state_dict_of(ovit.build_hf_model(spec, seed=0, stress=True))
        m = _model(sd)
        x = ovit.synthetic_images(128, seed=3).cuda()
        tail, full = _tail_and_full(m, x)
        assert torch.equal(tail, full), (kind, (tail - full).abs().max().item())
