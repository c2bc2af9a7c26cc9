"""GPU parity of the Swin V2 path: the cosine window attention (64 and 256 tokens) against a float64 torch reference, the
post-norm residual kernel against torch, and whole models against the installed HF Swinv2ForImageClassification run in
float32 (TF32 off) on the same weights.  bf16 mode: logits max-abs <= 2e-2, top-1 agreement (tie-aware)."""
import ctypes as ct
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import swinv2 as osv2  # noqa: E402
from oracle import vit as ovit  # noqa: E402

LOG2E = 1.4426950408889634


def _reference(qkv, table, logit_scale, n_win, heads, window, grid, shift, mask):
    from edgevisiontransformer_b200 import ops
    N, C = window * window, heads * 32
    q, k, v = [t.double().view(n_win, N, heads, 32).transpose(1, 2) for t in qkv.cpu().split(C, dim=1)]
    cos = torch.nn.functional.normalize(q, dim=-1) @ torch.nn.functional.normalize(k, dim=-1).transpose(-1, -2)
    scale = logit_scale.double().clamp(max=math.log(100.0)).exp().view(1, heads, 1, 1)
    bias = ops.swinv2_score_bias(table, window, grid, shift, mask).double()          # [nW, heads, N, N]
    s = cos * scale + bias[torch.arange(n_win) % bias.shape[0]]
    return (s.softmax(-1) @ v).transpose(1, 2).reshape(n_win * N, C)


def _inputs(g, n_win, heads, window, kind):
    N, C = window * window, heads * 32
    q, k, v = (torch.randn(n_win * N, C, generator=g) for _ in range(3))
    if kind == "late_max":                 # every query's best key is the window's last token: the online softmax must rescale
        qv = q.view(n_win, N, heads, 32)
        kv = k.view(n_win, N, heads, 32)
        kv[:, -1] = qv.mean(1) * 8
    elif kind == "peaky":                  # each query equals one key: cosine 1 against the rest's ~0, times scale 100
        k = q.view(n_win, N, C).flip(1).reshape(n_win * N, C).clone()
    return torch.cat([q, k, v * 1.5], 1).bfloat16()


@pytest.mark.parametrize("window,heads,grid,shift,kind", [
    (8, 3, 64, 0, "random"), (8, 3, 16, 4, "random"), (8, 32, 8, 0, "peaky"), (8, 1, 16, 4, "late_max"), (8, 12, 32, 4, "peaky"),
    (8, 1, 8, 0, "random"), (8, 3, 8, 0, "peaky"),
    (16, 1, 32, 8, "late_max"), (16, 4, 32, 0, "random"), (16, 8, 32, 8, "peaky"), (16, 32, 16, 0, "random"), (16, 6, 64, 8, "random"),
])
def test_cosine_window_attention_matches_float64(window, heads, grid, shift, kind):
    from edgevisiontransformer_b200 import ops
    g = torch.Generator().manual_seed(window * 100 + heads + grid + shift)
    per_img = (grid // window) ** 2
    n_win = per_img * (2 if per_img < 8 else 1) + (1 if per_img == 1 else 0)      # grid == window: 3 windows, odd item counts
    qkv = _inputs(g, n_win, heads, window, kind)
    table = 16 * torch.sigmoid(torch.randn(heads, (2 * window - 1) ** 2, generator=g))
    logit_scale = torch.rand(heads, generator=g) * (math.log(100.0) + 0.5)
    logit_scale[0] = math.log(100.0) + 0.5                                          # clamped
    mask = -200.0 if shift else -100.0
    got = ops.cosine_window_attention(qkv.cuda(), (table * LOG2E).cuda(),
                                      (logit_scale.clamp(max=math.log(100.0)).exp() * LOG2E).cuda(), n_win, heads, window, grid,
                                      shift, mask).float().cpu()
    want = _reference(qkv, table, logit_scale, n_win, heads, window, grid, shift, mask)
    err = (got.double() - want).abs()
    # bf16 probabilities and output (|v| up to ~6), f16 q / k hats times scales up to 100
    assert err.max() < 0.06, err.max()
    assert err.mean() < 3e-3, err.mean()


@pytest.mark.parametrize("window,grid", [(8, 16), (16, 32)])
def test_cosine_window_attention_honours_the_mask_value(window, grid):
    """Masks small enough to leave masked pairs a visible weight: the kernel adds the value it is given, and a different value
    gives a different context (at -100 or -200 the masked probabilities vanish either way)."""
    from edgevisiontransformer_b200 import ops
    g = torch.Generator().manual_seed(77 + window)
    heads, n_win = 2, (grid // window) ** 2
    qkv = _inputs(g, n_win, heads, window, "random")
    table = 16 * torch.sigmoid(torch.randn(heads, (2 * window - 1) ** 2, generator=g))
    logit_scale = torch.full((heads,), math.log(10.0))
    sc = (logit_scale.exp() * LOG2E).cuda()
    got = {}
    for mask in (-1.0, -3.0):
        got[mask] = ops.cosine_window_attention(qkv.cuda(), (table * LOG2E).cuda(), sc, n_win, heads, window, grid, window // 2,
                                                mask).float().cpu()
        want = _reference(qkv, table, logit_scale, n_win, heads, window, grid, window // 2, mask)
        assert (got[mask].double() - want).abs().max() < 0.03
    assert (got[-1.0] - got[-3.0]).abs().max() > 0.05


def test_cosine_window_attention_guard_band():
    """Canary rows before and after the context, and the columns of other heads beside it, stay untouched."""
    from edgevisiontransformer_b200 import _lib
    heads, window, grid, n_win = 2, 16, 32, 4
    N, C = window * window, heads * 32
    g = torch.Generator().manual_seed(5)
    qkv = _inputs(g, n_win, heads, window, "random").cuda()
    ldc, pad = C + 32, 64
    buf = torch.full(((n_win * N + 2 * pad) * ldc,), -7.0, dtype=torch.bfloat16, device="cuda")
    ctx = buf[pad * ldc:]
    tab = torch.zeros(heads, (2 * window - 1) ** 2, device="cuda")
    sc = torch.full((heads,), 10 * LOG2E, device="cuda")
    lib = _lib.load()
    _lib.check(lib.evt_cosine_window_attention_fwd(qkv.data_ptr(), qkv.stride(0), ctx.data_ptr(), ldc, tab.data_ptr(), sc.data_ptr(),
                                                   n_win, window, heads, 32, grid, 8, -100.0, torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    m = buf.view(-1, ldc)
    assert (m[:pad] == -7).all() and (m[pad + n_win * N:] == -7).all()
    assert (m[pad:pad + n_win * N, C:] == -7).all()
    assert torch.isfinite(m[pad:pad + n_win * N, :C].float()).all()


def test_cosine_window_attention_refuses_other_windows():
    from edgevisiontransformer_b200 import ops
    z = torch.zeros(144, 96, dtype=torch.bfloat16, device="cuda")
    with pytest.raises(RuntimeError, match="8x8.*16x16"):
        ops.cosine_window_attention(z, torch.zeros(1, 23 * 23, device="cuda"), torch.ones(1, device="cuda"), 1, 1, 12, 12)


@pytest.mark.parametrize("C,G,gather,add", [(96, 1, False, True), (192, 1, True, True), (768, 1, True, True), (96, 4, True, True),
                                            (384, 4, True, True), (1536, 1, False, False), (192, 1, True, False)])
def test_postnorm_residual_matches_torch(C, G, gather, add):
    from edgevisiontransformer_b200 import ops
    g = torch.Generator().manual_seed(C + G)
    images, T = 3, 64
    T_out = T // G
    y, resid = torch.randn(images * T, C, generator=g) * 3, torch.randn(images * T, C, generator=g)
    gamma, beta = 1 + 0.1 * torch.randn(C, generator=g), 0.1 * torch.randn(C, generator=g)
    idx = torch.randperm(T, generator=g)[:T_out * G].to(torch.int32) if gather else None
    o32, o16 = ops.postnorm_residual(y.cuda(), resid.cuda() if add else None, idx.cuda() if gather else None, gamma.cuda(),
                                     beta.cuda(), 1e-5, images, T_out, G)
    v = torch.nn.functional.layer_norm(y.double(), (C,), gamma.double(), beta.double(), 1e-5) + (resid.double() if add else 0)
    src = (torch.arange(images).view(-1, 1) * T + (idx.long().view(1, -1) if gather else torch.arange(T).view(1, -1))).view(-1)
    want = v[src].view(images * T_out, G * C)
    assert (o32.cpu().double() - want).abs().max() < 1e-4
    assert (o16.cpu().double() - want).abs().max() < 0.02 * (want.abs().max() + 1) / 4


def _hf_logits(hf, x):
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = False, False
    with torch.no_grad():
        return hf.cuda()(pixel_values=x.cuda()).logits.float().cpu()


def _check(m, hf, n_images, seed, bound=2e-2):
    x = torch.randn(n_images, 3, 256, 256, generator=torch.Generator().manual_seed(seed))
    want = _hf_logits(hf, x)
    got = m(x.cuda()).logits.cpu()
    r = ovit.compare_logits(got, want)
    assert r["max_abs"] <= bound and r["top1_agree"] == 1.0, r
    return m, x, want


MODELS = [  # kind, depths, window, pretrained window sizes
    ("tiny", [2, 2, 2, 2], 8, [0, 0, 0, 0]),
    ("tiny", None, 8, [0, 0, 0, 0]),
    ("tiny", None, 16, [0, 0, 0, 0]),
    ("base", [2, 2, 2, 2], 16, [0, 0, 0, 0]),
    ("base", [2, 2, 2, 2], 16, [12, 12, 12, 6]),
]


@pytest.mark.parametrize("stress", [False, True])
@pytest.mark.parametrize("kind,depths,window,pws", MODELS)
def test_from_hf_matches_hf_fp32(kind, depths, window, pws, stress):
    from edgevisiontransformer_b200.modeling_swinv2 import B200Swinv2ForImageClassification
    hf = osv2.build_hf_swinv2(kind, seed=11 + window, depths=depths, window=window, pretrained_window_sizes=pws, stress=stress)
    m = B200Swinv2ForImageClassification.from_hf(hf, max_batch=8)
    _check(m, hf, 4, seed=window)
    del m
    torch.cuda.empty_cache()


@pytest.mark.parametrize("kind,pws,bound", [("base", [0, 0, 0, 0], 2.5e-2), ("large", [12, 12, 12, 6], 3.3e-2)])
def test_full_depth_bf16_error_is_the_weight_rounding(kind, pws, bound):
    """Full-depth base / large window-16 models (HF init) exceed 2e-2 against fp32: 2.12e-2 and 2.80e-2 measured on these 8
    images (tools/swinv2_error_sites.py).  The cause is the bf16 rounding of the weights, which post-norm blocks carry into the
    stream at full scale: the fp32 HF forward with only its GEMM weights rounded to bf16 is already 1.93e-2 / 2.51e-2 away.
    So: the measured bound against fp32, and the 2e-2 contract against the fp32 forward of the bf16-rounded weights."""
    from edgevisiontransformer_b200.modeling_swinv2 import B200Swinv2ForImageClassification
    hf = osv2.build_hf_swinv2(kind, seed=0, window=16, pretrained_window_sizes=pws)
    m = B200Swinv2ForImageClassification.from_hf(hf, max_batch=8)
    _, x, _ = _check(m, hf, 8, seed=0, bound=bound)
    for name, mod in hf.named_modules():
        if isinstance(mod, (torch.nn.Linear, torch.nn.Conv2d)) and "continuous_position_bias_mlp" not in name:
            mod.weight.data = mod.weight.data.bfloat16().float()
    r = ovit.compare_logits(m(x.cuda()).logits.cpu(), _hf_logits(hf, x))
    assert r["max_abs"] <= 2e-2 and r["top1_agree"] == 1.0, r
    del m
    torch.cuda.empty_cache()


@pytest.mark.parametrize("window", [8, 16])
def test_from_microsoft_matches_hf_with_halved_mask(window):
    from edgevisiontransformer_b200.modeling_swinv2 import B200Swinv2ForImageClassification
    hf = osv2.build_hf_swinv2("tiny", seed=21, depths=[2, 2, 2, 2], window=window, stress=True)
    ms = {"model": osv2.to_microsoft(hf)}
    osv2.halve_shift_masks(hf)
    m = B200Swinv2ForImageClassification.from_microsoft(ms, depths=[2, 2, 2, 2], num_heads=[3, 6, 12, 24], embed_dim=96, window=window)
    _check(m, hf, 4, seed=3)


def test_factory_graphed_pipelined_and_launch_count():
    from edgevisiontransformer_b200 import _lib, modeling_swinv2
    from edgevisiontransformer_b200.eval_loop import PipelinedClassifier
    hf = osv2.build_hf_swinv2("tiny", seed=4, window=8, stress=True)
    m = modeling_swinv2.swinv2_tiny_patch4_window8_256(hf.state_dict(), max_batch=4)
    assert m.mask_adds == 1                                   # the factories run the original arithmetic, mask once
    osv2.halve_shift_masks(hf)
    m, x, want = _check(m, hf, 6, seed=9)                      # 6 images at max_batch 4: two chunks
    r = ovit.compare_logits(m.forward_graphed(x[:1].cuda()).logits.cpu(), want[:1])
    assert r["max_abs"] <= 2e-2 and r["top1_agree"] == 1.0, r
    r = ovit.compare_logits(m.forward_graphed(x[1:3].cuda()).logits.cpu(), want[1:3])
    assert r["max_abs"] <= 2e-2 and r["top1_agree"] == 1.0, r
    got = PipelinedClassifier(m, chunk=4).logits(x.pin_memory())
    r = ovit.compare_logits(got.cpu(), want)
    assert r["max_abs"] <= 2e-2 and r["top1_agree"] == 1.0, r
    lib = _lib.load()
    torch.cuda.synchronize()
    lib.evt_launch_count_reset()
    m(x[:2].cuda())
    torch.cuda.synchronize()
    assert lib.evt_launch_count() == m.launches_per_forward() == 3 + 7 * 12 + 2 * 3 + 2


def test_runtime_refuses_v2_tf32_and_other_windows():
    from edgevisiontransformer_b200 import _lib
    lib = _lib.load()
    s = _lib.SwinSpec()
    s.image, s.patch, s.window, s.embed_dim, s.stages, s.num_labels, s.eps, s.version = 192, 4, 12, 96, 4, 10, 1e-5, 2
    for i, (d, h) in enumerate(zip([2, 2, 2, 2], [3, 6, 12, 24])):
        s.depths[i], s.heads[i] = d, h
    h = ct.c_void_p()
    assert lib.evt_swin_create(ct.byref(s), ct.byref(h)) == _lib.EVT_ERR_UNSUPPORTED
    assert b"16 x 16" in lib.evt_last_error()
    s.image, s.window, s.precision = 256, 8, _lib.PREC_TF32
    assert lib.evt_swin_create(ct.byref(s), ct.byref(h)) == _lib.EVT_ERR_UNSUPPORTED
    assert b"tf32" in lib.evt_last_error()
