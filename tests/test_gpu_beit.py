"""GPU parity of the BEiT / data2vec-vision path: attention with the relative position bias (197, 577 and 1025 tokens, the cls-row
query path) against float64 torch, the mean-pooled head against torch, and whole models against the installed HF modules run in
float32 (TF32 off) on the same stress-initialised weights.  bf16 mode: logits max-abs <= 2e-2, top-1 agreement (tie-aware)."""

import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import beit as ob  # noqa: E402
from oracle import vit as ovit  # noqa: E402



def _inputs(g, B, S, heads, kind):
    C = heads * 64
    q, k, v = (torch.randn(B * S, C, generator=g) for _ in range(3))
    if kind == "late_max":          # every query's best key is the image's last token: the online softmax must rescale
        kv, qv = k.view(B, S, heads, 64), q.view(B, S, heads, 64)
        kv[:, -1] = qv.mean(1) * 6
    elif kind == "peaky":           # each query equals one key, scaled: near one-hot probabilities
        k = q.view(B, S, C).flip(1).reshape(B * S, C).clone() * 3
    return torch.cat([q, k, v], 1).bfloat16()


def _reference(qkv, bias, B, S, heads, head_mask=None, Sq=None, transpose=False):
    q, k, v = [t.double().view(B, S, heads, 64).transpose(1, 2) for t in qkv.cpu().split(heads * 64, dim=1)]
    b = bias.double().transpose(-1, -2) if transpose else bias.double()
    p = ((q @ k.transpose(-1, -2)) * 0.125 + b).softmax(-1)
    if head_mask is not None:
        p = p * head_mask.double().cpu().view(1, heads, 1, 1)
    out = (p @ v).transpose(1, 2)
    Sq = S if Sq is None else Sq
    return out[:, :Sq].reshape(B * Sq, heads * 64)


CASES = [  # grid (S = grid^2 + 1), B, heads, kind
    (2, 3, 1, "random"), (7, 2, 12, "peaky"), (14, 3, 12, "random"), (14, 2, 16, "late_max"), (24, 2, 12, "random"),
    (24, 1, 16, "peaky"), (32, 2, 16, "late_max"), (32, 1, 1, "random"),
]


@pytest.mark.parametrize("cls_rows", [False, True])
@pytest.mark.parametrize("grid,B,heads,kind", CASES)
def test_attention_rel_bias_matches_float64(grid, B, heads, kind, cls_rows):
    from edgevisiontransformer_b200 import ops
    S = grid * grid + 1
    g = torch.Generator().manual_seed(grid * 100 + B * 10 + heads)
    qkv = _inputs(g, B, S, heads, kind)
    table = torch.randn((2 * grid - 1) ** 2 + 3, heads, generator=g) * 2
    hm = None
    if heads > 1:
        hm = torch.rand(heads, generator=g) + 0.5
        hm[1] = 0.0
    Sq = 1 if cls_rows else None
    got = ops.attention_rel_bias(qkv.cuda(), table, grid, B, heads, head_mask=None if hm is None else hm.cuda(), q_rows=Sq)
    got = got.float().cpu().double()
    bias = ops.beit_score_bias(table, grid)
    want = _reference(qkv, bias, B, S, heads, hm, Sq)
    err = (got - want).abs()
    assert err.max() < 0.04, err.max()
    assert err.mean() < 3e-3, err.mean()
    if not cls_rows and kind != "peaky":
        # the index and its transpose must be told apart: the same table with query and key roles swapped is far off (the cls
        # row alone cannot tell them apart, its bias is one value for every patch key either way; near one-hot rows barely move)
        swapped = (got - _reference(qkv, bias, B, S, heads, hm, Sq, transpose=True)).abs()
        assert swapped.max() > 0.2, swapped.max()
    if not cls_rows:   # the cls-row path gives the same bits as the full call
        one = ops.attention_rel_bias(qkv.cuda(), table, grid, B, heads, head_mask=None if hm is None else hm.cuda(), q_rows=1)
        assert torch.equal(one.float().cpu().double(), got.view(B, S, -1)[:, 0])


@pytest.mark.parametrize("grid,Sq", [(14, 197), (24, 1), (32, 1025)])
def test_attention_rel_bias_guard_band(grid, Sq):
    """Canaries in a row above and below the context and in the columns beside the heads' columns stay untouched."""
    from edgevisiontransformer_b200 import _lib, ops
    B, heads, S = 2, 12, grid * grid + 1
    g = torch.Generator().manual_seed(grid)
    qkv = _inputs(g, B, S, heads, "random").cuda()
    table = torch.randn((2 * grid - 1) ** 2 + 3, heads, generator=g)
    ld = heads * 64 + 64
    buf = torch.full((B * Sq + 2, ld), 7.0, dtype=torch.bfloat16, device="cuda")
    tab = ops._beit_table(table, grid).cuda()
    ctx = buf[1:1 + B * Sq]
    _lib.check(_lib.load().evt_attention_rel_bias_fwd(qkv.data_ptr(), qkv.stride(0), ctx.data_ptr(), ld, None, tab.data_ptr(), grid, B, S,
                                                      Sq, heads, 64, 0.125, torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert (buf[0] == 7).all() and (buf[-1] == 7).all() and (ctx[:, heads * 64:] == 7).all()
    want = ops.attention_rel_bias(qkv, table, grid, B, heads, q_rows=Sq)
    assert torch.equal(ctx[:, :heads * 64], want)


def test_attention_rel_bias_refusals():
    from edgevisiontransformer_b200 import _lib
    lib = _lib.load()
    qkv = torch.zeros(2 * 197, 3 * 64, dtype=torch.bfloat16, device="cuda")
    ctx = torch.zeros(2 * 197, 80, dtype=torch.bfloat16, device="cuda")
    tab = torch.zeros(732, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    assert lib.evt_attention_rel_bias_fwd(qkv.data_ptr(), 192, ctx.data_ptr(), 64, None, tab.data_ptr(), 14, 2, 197, 197, 1, 64, 0.125, st) == 0
    for args, msg in (((14, 2, 198, 198, 1, 64), b"grid^2 + 1"), ((14, 2, 197, 197, 1, 80), b"head size 64")):
        rc = lib.evt_attention_rel_bias_fwd(qkv.data_ptr(), 240, ctx.data_ptr(), 80, None, tab.data_ptr(), *args, 0.125, st)
        assert rc == _lib.EVT_ERR_UNSUPPORTED and msg in lib.evt_last_error()


@pytest.mark.parametrize("T,D", [(197, 768), (577, 1024), (1025, 1024), (5, 64)])
def test_layernorm_patch_mean_matches_torch(T, D):
    from edgevisiontransformer_b200 import ops
    g = torch.Generator().manual_seed(T + D)
    images = 3
    x = torch.randn(images * T, D, generator=g) * 2 + 0.5
    gamma, beta = 1 + torch.randn(D, generator=g) * 0.1, torch.randn(D, generator=g) * 0.1
    got = ops.layernorm_patch_mean(x.cuda(), gamma.cuda(), beta.cuda(), 1e-12, images, T).float().cpu()
    xd = x.double().view(images, T, D)[:, 1:].mean(1)
    want = torch.nn.functional.layer_norm(xd, (D,), gamma.double(), beta.double(), 1e-12)
    assert (got.double() - want).abs().max() <= 0.01 * want.abs().max()


def _hf_logits(hf, x):
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = False, False
    with torch.no_grad():
        out = hf.cuda()(pixel_values=x.float().cuda()).logits.float().cpu()
    hf.cpu()
    return out


def _check(m, hf, n_images, image_size, seed, bound=2e-2):
    x = ob.images(n_images, image_size, seed=seed)
    want = _hf_logits(hf, x)
    got = m(x.cuda()).logits.cpu()
    r = ovit.compare_logits(got, want)
    assert r["max_abs"] <= bound and r["top1_agree"] == 1.0, r
    return x, want


MODELS = [  # kind, layers, image size, options
    ("base", None, 224, {}),
    ("large", 4, 224, {}),
    ("base", 2, 384, {}),
    ("large", 2, 512, {}),
    ("base", 3, 224, dict(use_relative_position_bias=False, use_shared_relative_position_bias=True)),
    ("base", 3, 224, dict(use_relative_position_bias=False)),                     # plain ViT encoder, mean-pooled head
    ("base", 3, 224, dict(data2vec=True)),
    ("base", 2, 224, dict(num_labels=21841, use_absolute_position_embeddings=True)),
]


@pytest.mark.parametrize("kind,layers,image,opts", MODELS)
def test_from_hf_matches_hf_fp32(kind, layers, image, opts):
    from edgevisiontransformer_b200.modeling_beit import B200BeitForImageClassification
    hf = ob.build_hf_beit(kind, seed=len(opts) + (layers or 0), layers=layers, image_size=image, **opts)
    m = B200BeitForImageClassification.from_hf(hf, max_batch=8)
    assert m.config.final_ln == 2
    _check(m, hf, 4, image, seed=image + (layers or 0))


def test_cls_pooling_tail_is_bit_identical_to_the_full_layer():
    """use_mean_pooling=False: beit.layernorm then row 0, so the last layer runs on the cls rows only (biased Sq = 1
    attention); its logits equal those of a forward that keeps the whole last layer (context capture turns the tail off)."""
    from edgevisiontransformer_b200.modeling_beit import B200BeitForImageClassification
    hf = ob.build_hf_beit("base", seed=5, layers=3, use_mean_pooling=False)
    m = B200BeitForImageClassification.from_hf(hf, max_batch=8)
    assert m.config.final_ln is True
    x, want = _check(m, hf, 4, 224, seed=11)
    tail = m(x.cuda()).logits
    m.capture_context(True)
    full = m(x.cuda()).logits
    m.capture_context(False)
    assert torch.equal(tail, full)


def test_uint8_graphed_pipelined_pretrained_and_launch_count(tmp_path):
    from edgevisiontransformer_b200 import _lib
    from edgevisiontransformer_b200.eval_loop import PipelinedClassifier
    from edgevisiontransformer_b200.modeling_beit import B200BeitForImageClassification
    hf = ob.build_hf_beit("base", seed=7, layers=2)
    m = B200BeitForImageClassification.from_hf(hf, max_batch=4)
    x, want = _check(m, hf, 6, 224, seed=13)           # 6 images at max_batch 4: two chunks
    r = ovit.compare_logits(m.forward_graphed(x[:1].cuda()).logits.cpu(), want[:1])
    assert r["max_abs"] <= 2e-2 and r["top1_agree"] == 1.0, r
    got = PipelinedClassifier(m, chunk=4).logits(x.pin_memory())
    r = ovit.compare_logits(got.cpu(), want)
    assert r["max_abs"] <= 2e-2 and r["top1_agree"] == 1.0, r
    # uint8 pixels are normalised inside the patch gather
    u8 = torch.randint(0, 256, (3, 3, 224, 224), dtype=torch.uint8, generator=torch.Generator().manual_seed(1))
    mean, std = torch.tensor(m.pixel_mean).view(1, 3, 1, 1), torch.tensor(m.pixel_std).view(1, 3, 1, 1)
    r = ovit.compare_logits(m(u8.cuda()).logits.cpu(), _hf_logits(hf, (u8.float() / 255 - mean) / std))
    assert r["max_abs"] <= 2e-2 and r["top1_agree"] == 1.0, r
    hf.save_pretrained(tmp_path)
    m2 = B200BeitForImageClassification.from_pretrained(str(tmp_path), max_batch=4)
    assert torch.equal(m2(x[:4].cuda()).logits, m(x[:4].cuda()).logits)
    lib = _lib.load()
    torch.cuda.synchronize()
    lib.evt_launch_count_reset()
    m(x[:4].cuda())
    torch.cuda.synchronize()
    assert lib.evt_launch_count() == m.launches_per_forward() == 3 + 7 * 2 + 2


def test_head_mask_zeroes_a_head():
    """A zero in head_mask removes that head's context: the HF module with the head's value rows zeroed is the reference
    (HF BEiT's forward takes no head_mask)."""
    import copy
    from edgevisiontransformer_b200.modeling_beit import B200BeitForImageClassification
    hf = ob.build_hf_beit("base", seed=8, layers=2)
    m = B200BeitForImageClassification.from_hf(hf, max_batch=4)
    hm = torch.ones(2, 12)
    hm[0, 3] = hm[1, 7] = 0.0
    ref = copy.deepcopy(hf)
    with torch.no_grad():
        for l, h in ((0, 3), (1, 7)):
            v = ref.beit.encoder.layer[l].attention.attention.value
            v.weight[h * 64:(h + 1) * 64] = 0
            v.bias[h * 64:(h + 1) * 64] = 0
    x = ob.images(2, 224, seed=17)
    r = ovit.compare_logits(m(x.cuda(), head_mask=hm).logits.cpu(), _hf_logits(ref, x))
    assert r["max_abs"] <= 2e-2 and r["top1_agree"] == 1.0, r
    assert ovit.compare_logits(m(x.cuda()).logits.cpu(), _hf_logits(ref, x))["max_abs"] > 2e-2


def test_runtime_refusals():
    """The C runtime itself refuses the bias in the tf32 mode, with a distillation token, and final_ln = 2 in tf32."""
    from edgevisiontransformer_b200 import _lib
    from edgevisiontransformer_b200.modeling_beit import beit_to_canonical
    from edgevisiontransformer_b200.modeling_vit import B200ViTForImageClassification
    hf = ob.build_hf_beit("base", seed=9, layers=1)
    sd, cfg = beit_to_canonical(dict(hf.state_dict()), hf.config)
    cfg.precision = "tf32"
    with pytest.raises(_lib.EvtError, match="bf16 mode only"):
        B200ViTForImageClassification(cfg, sd)
    cfg.precision, cfg.final_ln = "tf32", True
    with pytest.raises(_lib.EvtError, match="relative position bias .BEiT. is implemented in the bf16 mode only"):
        B200ViTForImageClassification(cfg, sd)
