"""GPU tests of sequences longer than 256 tokens: the 384-pixel DeiT / ViT models (577 tokens, 578 with a distillation token)
and the key-blocked attention kernel behind them (csrc/attention.cu, attention_long_kernel), from the op up to the model
classes.  Checkers: the fp32 attention oracle, the CPU model oracle and the live HF modules on the same weights."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import ViTSpec  # noqa: E402
from oracle import vit as ovit  # noqa: E402

BF16_TOL = 2e-2
MAX_TOKENS = 1026       # EVT_ATTN_MAX_TOKENS (include/evt.h)


@pytest.fixture
def no_split_k():
    from edgevisiontransformer_b200 import ops
    ops.set_gemm_split_k(False)
    yield
    ops.set_gemm_split_k(True)


def _ops():
    from edgevisiontransformer_b200 import ops
    return ops


def _qkv(B, S, heads, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(B * S, 3 * heads * 64, generator=g) * scale).bfloat16().cuda()


def _attn_ref(qkv, B, S, heads, hs=64):
    a = heads * hs
    q, k, v = qkv[:, :a].float(), qkv[:, a:2 * a].float(), qkv[:, 2 * a:3 * a].float()
    return ovit.attention(q.view(B, S, a), k.view(B, S, a), v.view(B, S, a), hs).reshape(B * S, a)


def _check(got, want, tol=BF16_TOL):
    r = ovit.compare_logits(got, want)
    assert r["max_abs"] <= tol, r
    assert r["top1_agree"] == 1.0, r
    return r


def _model(sd, **kw):
    from edgevisiontransformer_b200 import B200ViTForImageClassification
    return B200ViTForImageClassification.from_state_dict(sd, **kw)


def _spec384(kind):
    return ViTSpec.deit(kind, image=384, tokens=577)


# ------------------------------------------------------------------------------------------------ op level

# B = 1 leaves most SMs idle; B = 40 at 12 heads and S = 577 (2400 items) fills every SM several times over.  S = 257 / 300
# have one / 44 valid keys in their last 128-key block, 1025 / 1026 one / two.
@pytest.mark.parametrize("B,S,heads", [(1, 257, 1), (2, 300, 3), (3, 577, 12), (1, 577, 3), (40, 577, 12), (2, 578, 3),
                                       (1, 1025, 12), (2, 1025, 3), (1, MAX_TOKENS, 1)])
def test_long_attention_matches_fp32(B, S, heads):
    ops = _ops()
    qkv = _qkv(B, S, heads, seed=S + B)
    ctx = ops.attention(qkv, B, S, heads)
    assert ctx.shape == (B * S, heads * 64)
    err = (ctx.float() - _attn_ref(qkv, B, S, heads)).abs().max().item()
    assert err < 2e-2, f"attention B={B} S={S} heads={heads}: err {err}"


def test_long_attention_head_mask_and_peaky_scores():
    """Large logits make the row maximum jump between key blocks, which exercises the lazy rescale of O and the sum."""
    ops = _ops()
    B, S, heads = 2, 577, 3
    qkv = _qkv(B, S, heads, seed=7, scale=3.0)
    mask = torch.tensor([1.0, 0.0, 1.0], device="cuda")
    ctx = ops.attention(qkv, B, S, heads, head_mask=mask)
    ref = _attn_ref(qkv, B, S, heads).view(B * S, heads, 64) * mask.view(1, heads, 1)
    assert (ctx.float() - ref.reshape(B * S, -1)).abs().max().item() < 6e-2
    assert ctx.view(B * S, heads, 64)[:, 1].abs().max().item() == 0.0


def test_long_attention_late_maximum():
    """Scores that grow along the key axis: every block raises the row maximum far past the rescale margin."""
    ops = _ops()
    B, S, heads = 2, 577, 2
    a = heads * 64
    qkv = _qkv(B, S, heads, seed=8, scale=0.5).float()
    qkv[:, :a] = 1.0 / 8                                               # q . k = sum(k) / 8
    ramp = torch.linspace(0, 6, S, device="cuda").repeat(B)[:, None]
    qkv[:, a:2 * a] += ramp
    qkv = qkv.bfloat16()
    err = (ops.attention(qkv, B, S, heads).float() - _attn_ref(qkv, B, S, heads)).abs().max().item()
    assert err < 2e-2, err


@pytest.mark.parametrize("S", [577, 1025])
@pytest.mark.parametrize("B", [3, 40])
def test_long_attention_query_rows_are_the_full_rows(S, B):
    ops = _ops()
    heads = 3
    qkv = _qkv(B, S, heads, seed=S * 10 + B, scale=2.0)
    mask = torch.tensor([1.0, 0.0, 0.5], device="cuda")
    for hm in (None, mask):
        full = ops.attention(qkv, B, S, heads, head_mask=hm).view(B, S, -1)
        for Sq in (1, 2, 130):
            rows = ops.attention(qkv, B, S, heads, head_mask=hm, q_rows=Sq)
            assert rows.shape == (B * Sq, heads * 64)
            assert torch.equal(rows.view(B, Sq, -1), full[:, :Sq]), (S, B, Sq)


GUARD = 4096
SENT = -12345.0


# B * heads * query tiles: 15 / 9 / 27 items (an odd count leaves the last unit of a CTA with one item); S = 577 ends in a
# 65-row query tile, S = 1025 in a 1-row one.
@pytest.mark.parametrize("B,S", [(1, 577), (3, 577), (1, 1025), (3, 1025)])
@pytest.mark.parametrize("Sq", ["S", 1])
def test_long_attention_stays_in_bounds(B, S, Sq):
    from edgevisiontransformer_b200 import _lib
    lib = _lib.load()
    heads = 3
    Sq = S if Sq == "S" else Sq
    qkv = _qkv(B, S, heads, seed=5)
    n = B * Sq * heads * 64
    buf = torch.full((n + 2 * GUARD,), SENT, dtype=torch.bfloat16, device="cuda")
    out = buf[GUARD:GUARD + n]
    _lib.check(lib.evt_attention_query_rows_fwd(qkv.data_ptr(), qkv.stride(0), out.data_ptr(), heads * 64, None, B, S, Sq, heads, 64,
                                                0.125, torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert bool((buf[:GUARD] == SENT).all()) and bool((buf[GUARD + n:] == SENT).all())
    assert bool((out != SENT).all()), "output not fully written"


def test_long_attention_limits():
    ops = _ops()
    with pytest.raises(RuntimeError, match="1026"):
        ops.attention(_qkv(1, MAX_TOKENS + 1, 1, seed=1), 1, MAX_TOKENS + 1, 1)
    with pytest.raises(RuntimeError, match="256"):
        ops.attention(_qkv(1, 300, 1, seed=1).float(), 1, 300, 1)     # the tf32 kernel keeps its S <= 256


def test_torch_layers_attention_long_sequence():
    from edgevisiontransformer_b200 import torch_layers as tl
    torch.manual_seed(3)
    m = tl.Attention(192, 3).cuda().eval()
    x = torch.randn(2, 577, 192, device="cuda")
    got = m(x)
    with torch.no_grad():
        q, k, v = (lin(x).view(2, 577, 3, 64).transpose(1, 2) for lin in (m.to_query, m.to_key, m.to_value))
        p = torch.softmax(q @ k.transpose(-1, -2) * 0.125, -1)
        want = m.to_out((p @ v).transpose(1, 2).reshape(2, 577, 192))
    assert (got - want).abs().max().item() < 3e-2


# ------------------------------------------------------------------------------------------------ model level

@pytest.mark.parametrize("kind,big", [("tiny", 256), ("small", 256), ("base", 256)])
def test_deit_384_matches_oracle(kind, big):
    """DeiT-{Tiny,Small,Base} patch16-384: batch 1 and 5 and a large-M batch against the CPU oracle; the same images through
    the small-batch kernels agree with their large-batch logits; a second pass reproduces the first bit for bit."""
    spec = _spec384(kind)
    sd = ovit.state_dict_of(ovit.build_hf_model(spec, seed=2, stress=True))
    m = _model(sd, image_size=384, max_batch=big)
    assert m.config.tokens == 577 and m.config.image_size == 384
    x1 = ovit.synthetic_images(5, seed=3, size=384)
    want = ovit.vit_forward(sd, spec, x1)
    _check(m(x1[:1].cuda()).logits, want[:1])
    _check(m(x1.cuda()).logits, want)
    g = torch.Generator(device="cuda").manual_seed(4)
    x = torch.randn(big, 3, 384, 384, device="cuda", generator=g)
    logits = m(x).logits
    assert logits.shape == (big, 1000) and torch.isfinite(logits).all()
    pick = torch.tensor([0, 1, big // 2, big - 1], device="cuda")
    ops = _ops()
    try:
        ops.set_gemm_split_k(False)
        small = m(x[pick].contiguous()).logits
    finally:
        ops.set_gemm_split_k(True)
    r = ovit.compare_logits(logits[pick], small)
    assert r["max_abs"] <= 5e-3 and r["top1_agree"] == 1.0, r
    _check(logits[pick[:2]], ovit.vit_forward(sd, spec, x[pick[:2]].cpu()))
    assert torch.equal(m(x).logits, logits)


def test_hf_deit_384_and_distilled():
    """HF DeiTForImageClassification (578 tokens, classifier on the cls row) and the two-head distilled DeiT at 384 against
    the live HF modules."""
    from transformers import DeiTConfig, DeiTForImageClassification, DeiTForImageClassificationWithTeacher
    from edgevisiontransformer_b200 import B200ViTForImageClassification
    cfg = DeiTConfig(hidden_size=192, num_hidden_layers=12, num_attention_heads=3, intermediate_size=768, num_labels=1000,
                     image_size=384, attn_implementation="eager")
    x = ovit.synthetic_images(3, seed=5, size=384)
    for cls_ in (DeiTForImageClassification, DeiTForImageClassificationWithTeacher):
        torch.manual_seed(17)
        hf = cls_(cfg).eval()
        with torch.no_grad():
            for n, p in hf.named_parameters():
                if n.endswith("bias") or "layernorm" in n:
                    p.add_(torch.randn_like(p) * 0.1)
            for t in (hf.deit.embeddings.cls_token, hf.deit.embeddings.distillation_token, hf.deit.embeddings.position_embeddings):
                t.normal_(0, 0.02)
            want = hf(pixel_values=x).logits
        m = B200ViTForImageClassification.from_hf(hf)
        assert m.config.tokens == 578 and m.config.image_size == 384
        assert m.config.head_rows == (2 if cls_ is DeiTForImageClassificationWithTeacher else 1)
        _check(m(x.cuda()).logits, want)


def test_timm_384_state_dict():
    """A deit_*_patch16_384 checkpoint in the timm layout: the image size comes from the 577 position rows."""
    from edgevisiontransformer_b200 import B200ViTForImageClassification
    from oracle import timm_vit as otimm
    spec = ViTSpec.deit("tiny", image=384, tokens=577, eps=1e-6)
    tsd = otimm.hf_to_timm(ovit.state_dict_of(ovit.build_hf_model(spec, seed=6, stress=True)))
    x = ovit.synthetic_images(2, seed=7, size=384)
    want = otimm.timm_vit_forward(tsd, x, num_heads=3)
    m = B200ViTForImageClassification.from_timm(tsd)
    assert m.config.image_size == 384 and m.config.tokens == 577
    _check(m(x.cuda()).logits, want)


def test_head_mask_and_context_capture_at_577_tokens():
    spec = ViTSpec.deit("tiny", image=384, tokens=577, layers=4, heads=[3] * 4, inter=[768] * 4)
    sd = ovit.state_dict_of(ovit.build_hf_model(spec, seed=8, stress=True))
    m = _model(sd, image_size=384)
    x = ovit.synthetic_images(2, seed=9, size=384)
    mask = torch.ones(4, 3)
    mask[1, 2] = 0.0
    mask[3, 0] = 0.5
    ctx_want = []
    want = ovit.vit_forward(sd, spec, x, head_mask=mask, ctx_out=ctx_want)
    m.capture_context(True)
    got = m(x.cuda(), head_mask=mask).logits
    _check(got, want)
    assert len(m.context_layers) == 4
    for got_c, want_c in zip(m.context_layers, ctx_want):
        assert got_c.shape == (2, 3, 577, 64) == want_c.shape
        assert (got_c.float().cpu() - want_c).abs().max().item() < 5e-2
    assert m.context_layers[1][:, 2].abs().max().item() == 0.0
    m.capture_context(False)


@pytest.mark.parametrize("bs", [1, 5, 64])
def test_cls_tail_at_577_tokens_is_bit_identical(bs, no_split_k):
    """The last layer runs its attention for the cls query only (q_rows = 1 of the long kernel) and the rest on one row per
    image; capturing the context forces the full layer.  Same bits with and without a head mask."""
    spec = _spec384("tiny")
    sd = ovit.state_dict_of(ovit.build_hf_model(spec, seed=3, stress=True))
    m = _model(sd, image_size=384)
    x = ovit.synthetic_images(bs, seed=4, size=384).cuda()
    mask = torch.ones(12, 3)
    mask[11, 0] = 0.0
    mask[11, 2] = 0.5
    for kw in ({}, {"head_mask": mask}):
        m.capture_context(False)
        tail = m(x, **kw).logits.clone()
        m.capture_context(True)
        full = m(x, **kw).logits.clone()
        m.capture_context(False)
        assert torch.equal(tail, full), kw


def test_launch_count_at_577_tokens():
    from edgevisiontransformer_b200 import _lib
    spec = _spec384("small")
    m = _model(ovit.state_dict_of(ovit.build_hf_model(spec, seed=1)), image_size=384)
    x = ovit.synthetic_images(4, seed=2, size=384).cuda()
    m(x)
    torch.cuda.synchronize()
    lib = _lib.load()
    lib.evt_launch_count_reset()
    m(x)
    torch.cuda.synchronize()
    assert lib.evt_launch_count() == m.launches_per_forward()


def test_rejections():
    spec = _spec384("tiny")
    sd = ovit.state_dict_of(ovit.build_hf_model(spec, seed=1))
    with pytest.raises(RuntimeError, match="tf32"):
        _model(sd, image_size=384, precision="tf32")
    # 528 px, a 33 x 33 grid: 1090 tokens, past EVT_ATTN_MAX_TOKENS
    big = ViTSpec.deit("tiny", image=528, tokens=33 * 33 + 1, layers=1, heads=[3], inter=[768])
    with pytest.raises(RuntimeError, match="1026"):
        _model(ovit.state_dict_of(ovit.build_hf_model(big, seed=1)), image_size=528)
