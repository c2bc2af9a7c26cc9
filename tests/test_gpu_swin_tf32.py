"""The Swin tf32 accuracy mode (precision="tf32"): the tf32 window attention for 49- and 144-token windows against a float64
emulation of its arithmetic, whole models against the installed HF SwinForImageClassification run in float32 on the CPU
(logits max-abs <= 1e-3, the project's tf32 contract; 1.5e-3 for the stress-initialised 384-pixel models, DESIGN.md section 4),
the C runtime against the op-level composition, and the Python / C
surface of the new precision field."""
import ctypes as ct

import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import swin as osw  # noqa: E402
from oracle import vit as ovit  # noqa: E402

LOG2E = 1.4426950408889634
WIDTHS = {"base": (128, [4, 8, 16, 32]), "large": (192, [6, 12, 24, 48])}
SENT = -12345.0


def build_hf_swin_384(kind, depths, seed, stress=True):
    """Random-init HF SwinForImageClassification at 384 pixels / window 12; ``stress`` randomises the bias tables, biases and
    LayerNorm affine (as tests/test_gpu_swin_window12.py does)."""
    from transformers import SwinConfig, SwinForImageClassification
    embed_dim, heads = WIDTHS[kind]
    cfg = SwinConfig(image_size=384, patch_size=4, window_size=12, embed_dim=embed_dim, depths=list(depths), num_heads=heads,
                     num_labels=1000)
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


def assert_tf32_close(got, want, bound=1e-3):
    r = ovit.compare_logits(got, want)
    assert r["max_abs"] <= bound and r["top1_agree"] == 1.0, r
    return r


# ------------------------------------------------------------------------------------------------------------ op level
def emulate(qkv, table, n_win, n_tab, heads, N):
    """float64 restatement of the kernel's arithmetic: scores from the (tf32) operands, s * scale * log2e + table, row max,
    2^(z - max) rounded to tf32, sum of the rounded values, context / sum rounded to tf32.  Also the unrounded attention."""
    from edgevisiontransformer_b200 import ops
    C = heads * 32
    q, k, v = [t.double().view(n_win, N, heads, 32).transpose(1, 2) for t in qkv.split(C, dim=1)]
    rows, cols = ops.window_table_shape(N)
    tab = table[torch.arange(n_win) % n_tab][:, :, :N, :N].double()
    z = (q @ k.transpose(-1, -2)) * (32 ** -0.5 * LOG2E) + tab
    p = torch.exp2(z - z.amax(-1, keepdim=True))
    exact = ((p / p.sum(-1, keepdim=True)) @ v).transpose(1, 2).reshape(n_win * N, C)
    p = ops.round_tf32(p.float()).double()
    o = (p @ v) / p.sum(-1, keepdim=True)
    want = ops.round_tf32(o.float()).double().transpose(1, 2).reshape(n_win * N, C)
    vmax = v.abs().amax(dim=(-2, -1), keepdim=True).expand(-1, -1, N, 32).transpose(1, 2).reshape(n_win * N, C)
    return want, exact, vmax


def run_window_tf32(heads, n_win, n_tab, N, seed, scales):
    """qkv tf32-representable (rounded as the QKV GEMM's epilogue rounds it); the context lands in a guarded buffer with
    ldc = heads*32 + 8 and 5 spare rows: the padding columns and spare rows must keep their sentinel."""
    from edgevisiontransformer_b200 import _lib, ops
    from edgevisiontransformer_b200.modeling_swin import attention_table, shift_mask
    g = torch.Generator().manual_seed(seed)
    C = heads * 32
    q, k, v = (torch.randn(n_win * N, C, generator=g) * s for s in scales)
    qkv = ops.round_tf32(torch.cat([q, k, v], 1))
    ws = 7 if N == 49 else 12
    mask = shift_mask(2 * ws, 2 * ws, ws, ws // 2) if n_tab == 4 else None        # the four windows of a two-window-wide stage
    table = attention_table(torch.randn((2 * ws - 1) ** 2, heads, generator=g), heads, ws, mask)
    ldc, spare = C + 8, 5
    buf = torch.full((n_win * N + spare, ldc), SENT, device="cuda")
    lib = _lib.load()
    qd, td = qkv.cuda(), table.cuda()
    _lib.check(lib.evt_window_attention_fwd_tf32(qd.data_ptr(), qd.stride(0), buf.data_ptr(), ldc, td.data_ptr(), n_tab, n_win, N, heads,
                                                 32, 32 ** -0.5, torch.cuda.current_stream().cuda_stream), "window_attention_tf32")
    out = buf.cpu()
    assert (out[:n_win * N, C:] == SENT).all() and (out[n_win * N:] == SENT).all(), "context written outside [rows, heads*32]"
    got = out[:n_win * N, :C].double()
    assert torch.equal(ops.round_tf32(got.float()).double(), got)                  # stored values are tf32
    # the op wrapper dispatches on the f32 dtype to the same kernel
    assert torch.equal(ops.window_attention(qd, td, n_win, heads, N).cpu().double(), got)
    want, exact, vmax = emulate(qkv, table, n_win, n_tab, heads, N)
    err = (got - want).abs()
    bound = 2.0 ** -10 * (want.abs() + vmax)
    assert (err <= bound).all(), f"max excess {(err - bound).max().item():.3e}, max err {err.max().item():.3e}"
    print(f"tf32 window attention N={N} heads={heads} n_win={n_win} n_tab={n_tab}: max |got - emulation| {err.max().item():.3e}, "
          f"max |got - float64 attention| {(got - exact).abs().max().item():.3e}")


@pytest.mark.parametrize("heads,n_win,n_tab", [(3, 8, 4), (6, 5, 1), (24, 3, 1)])
def test_window_attention_tf32_49(heads, n_win, n_tab):
    run_window_tf32(heads, n_win, n_tab, 49, seed=heads, scales=(1.5, 1.5, 1.5))


@pytest.mark.parametrize("heads,n_win,n_tab", [(4, 9, 4), (4, 5, 1), (48, 3, 1), (48, 7, 4)])
def test_window_attention_tf32_144(heads, n_win, n_tab):
    run_window_tf32(heads, n_win, n_tab, 144, seed=100 + heads + n_win, scales=(2.0, 2.0, 1.5))


def test_tf32_ops_round_their_outputs():
    """gather_layernorm, layernorm_mean_tokens and im2col_patch with out_dtype=TF32 write the f32 result rounded to tf32."""
    from edgevisiontransformer_b200 import ops
    g = torch.Generator().manual_seed(5)
    x = (torch.randn(2 * 196, 96, generator=g) * 2).cuda()
    idx = torch.randperm(196, generator=g).to(torch.int32).cuda()
    gamma, beta = torch.randn(96, generator=g).cuda(), torch.randn(96, generator=g).cuda()
    y32, _ = ops.gather_layernorm(x, idx, gamma, beta, 1e-5, 2, 196, 196, out_dtype=torch.float32)
    yt, _ = ops.gather_layernorm(x, idx, gamma, beta, 1e-5, 2, 196, 196, out_dtype=ops.TF32)
    assert torch.equal(yt, ops.round_tf32(y32))
    xm = (torch.randn(3 * 49, 768, generator=g) * 3).cuda()
    gm, bm = torch.randn(768, generator=g).cuda(), torch.randn(768, generator=g).cuda()
    pt = ops.layernorm_mean_tokens(xm, gm, bm, 1e-5, 3, 49, out_dtype=ops.TF32)
    want = torch.nn.functional.layer_norm(xm.cpu().double(), (768,), gm.cpu().double(), bm.cpu().double(), 1e-5).view(3, 49, 768).mean(1)
    assert pt.dtype == torch.float32 and torch.equal(pt, ops.round_tf32(pt)) and (pt.cpu().double() - want).abs().max() < 2e-3
    px = torch.randn(2, 3, 56, 56, generator=g).cuda()
    ct_ = ops.im2col_patch(px, 4, out_dtype=ops.TF32)
    want = px.cpu().view(2, 3, 14, 4, 14, 4).permute(0, 2, 4, 1, 3, 5).reshape(2 * 196, 48)
    assert torch.equal(ct_.cpu(), ops.round_tf32(want))
    assert torch.equal(ops.im2col_patch(px, 4).float().cpu(), want.bfloat16().float())


# ------------------------------------------------------------------------------------------------------------ model level
def check_model(hf, n_images, seed, bound=1e-3):
    """tf32 model on n_images (max_batch 2: the chunk loop runs) against fp32 HF on the CPU, the C runtime against the op-level
    composition (bit-identical) and the launch count."""
    from edgevisiontransformer_b200 import ops
    from edgevisiontransformer_b200.modeling_swin import B200SwinForImageClassification
    c = hf.config
    x = ovit.synthetic_images(n_images, seed=seed, size=c.image_size)
    want = hf_logits(hf, x)
    m = B200SwinForImageClassification.from_hf(hf, max_batch=2, precision="tf32")
    assert m.precision == "tf32"
    got = m(pixel_values=x.cuda()).logits
    r = assert_tf32_close(got, want, bound)
    print(f"Swin embed_dim={c.embed_dim} window={c.window_size} depths={c.depths} tf32: {r}")
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
    return m, x, want, got


def test_swin_tiny_hf_init_tf32():
    hf = osw.build_hf_swin("tiny", seed=0, stress=False)
    check_model(hf, 2, seed=1)


def test_swin_tiny_stress_tf32():
    hf = osw.build_hf_swin("tiny", seed=7, stress=True)
    m, x, want, got = check_model(hf, 3, seed=2)
    # the microsoft/Swin-Transformer key layout loads to the same function
    from edgevisiontransformer_b200.modeling_swin import B200SwinForImageClassification
    m2 = B200SwinForImageClassification.from_microsoft(osw.hf_to_microsoft(ovit.state_dict_of(hf)), depths=hf.config.depths,
                                                       num_heads=hf.config.num_heads, embed_dim=96, max_batch=2, precision="tf32")
    assert torch.equal(m2(pixel_values=x.cuda()).logits, got)


# The two stress-initialised 384-pixel models measure 1.0e-3 and 1.14e-3: stock PyTorch with TF32 matmuls lands at the same
# place on them (1.01e-3, 1.18e-3), and so does this runtime with float64 window attention, so the excess comes from tf32 GEMM
# operands, not from the attention's rounding points.  DESIGN.md section 4 records the measurement; the bound is 1.5e-3 there.
def test_swin_base_384_stress_tf32():
    hf = build_hf_swin_384("base", [2, 2, 2, 2], seed=21)
    check_model(hf, 3, seed=3, bound=1.5e-3)


def test_swin_large_384_tf32():
    hf = build_hf_swin_384("large", [1, 1, 1, 1], seed=22)
    check_model(hf, 2, seed=4, bound=1.5e-3)


# ------------------------------------------------------------------------------------------------------------ surface
def test_tf32_graphed_and_eval_loop():
    from edgevisiontransformer_b200.eval_loop import PipelinedClassifier, evaluate
    from edgevisiontransformer_b200.modeling_swin import B200SwinForImageClassification
    hf = osw.build_hf_swin("tiny", seed=8, stress=True, depths=[1, 1, 3, 1])
    m = B200SwinForImageClassification.from_hf(hf, max_batch=4, precision="tf32")
    x = ovit.synthetic_images(6, seed=3)
    want = hf_logits(hf, x)
    for _ in range(2):                                # capture, then replay
        assert torch.equal(m.forward_graphed(x[:1].cuda()).logits, m(pixel_values=x[:1].cuda()).logits)
    got = PipelinedClassifier(m, chunk=4).logits(x.pin_memory())
    assert_tf32_close(got, want)
    labels = want.argmax(-1)
    res = evaluate([(x[:4], labels[:4]), (x[4:], labels[4:])], m, eval_batch_size=4)
    assert res["eval_accuracy"] == 1.0


def test_precision_argument_and_spec_field():
    from edgevisiontransformer_b200 import _lib
    from edgevisiontransformer_b200.modeling_swin import B200SwinForImageClassification
    hf = osw.build_hf_swin("tiny", seed=9, stress=False, depths=[1, 1, 1, 1])
    with pytest.raises(ValueError, match="precision"):
        B200SwinForImageClassification.from_hf(hf, precision="fp8")
    lib = _lib.load()

    def spec(precision=None):
        s = _lib.SwinSpec()
        s.image, s.patch, s.window, s.embed_dim, s.stages, s.num_labels, s.eps = 224, 4, 7, 96, 4, 1000, 1e-5
        for i, h in enumerate([3, 6, 12, 24]):
            s.depths[i], s.heads[i] = 1, h
        if precision is not None:
            s.precision = precision
        return s

    def ws_bytes(s):
        h = ct.c_void_p()
        _lib.check(lib.evt_swin_create(ct.byref(s), ct.byref(h)), "swin_create")
        try:
            n = ct.c_size_t()
            _lib.check(lib.evt_swin_workspace_bytes(h, 8, ct.byref(n)), "swin_workspace_bytes")
            return n.value
        finally:
            lib.evt_swin_destroy(h)

    zero, bf16, tf32 = ws_bytes(spec()), ws_bytes(spec(_lib.PREC_BF16)), ws_bytes(spec(_lib.PREC_TF32))
    assert zero == bf16 < tf32                        # a zero-initialised spec is the bf16 model; tf32 operands take 4 bytes
    for bad in (2, -1):
        h = ct.c_void_p()
        assert lib.evt_swin_create(ct.byref(spec(bad)), ct.byref(h)) == _lib.EVT_ERR_INVALID
