"""Transformer-token T2T-ViT (t2t_vit_t_*, spec.t2t = 3) on the B200: the token-transformer block at the op level against torch
f32, and the models against the nn.Module restatement in fp32 on the CPU at the bf16 contract (max-abs logit error <= 2e-2,
top-1 agreement)."""
import os
import sys

import pytest
import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import t2t_t_torch_ref as tref  # noqa: E402
from oracle import vit as ovit  # noqa: E402

pytestmark = pytest.mark.gpu
BF16_TOL = 2e-2
MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
GUARD = 4096
SENT = -12345.0


def _b200(name, m, **kw):
    from edgevisiontransformer_b200 import modeling_t2t
    return getattr(modeling_t2t, name)(m.state_dict(), **kw)


def _images(B, seed):
    return torch.randn(B, 3, 224, 224, generator=torch.Generator().manual_seed(seed))


def _check(got, want, tol=BF16_TOL):
    r = ovit.compare_logits(got, want)
    assert r["max_abs"] <= tol and r["top1_agree"] == 1.0, r
    return r


# ------------------------------------------------------------------------------------------------ op level

def _block_inputs(B, T, seed):
    g = torch.Generator().manual_seed(seed)
    # q and k at 3 x unit scale: scores q.k * in_dim ** -0.5 have a spread of a few units, so the softmax is neither flat nor
    # one-hot; v at unit scale, so |y| ~ 1-4
    qkv = torch.randn(B * T, 192, generator=g)
    qkv[:, :128] *= 3
    qkv = qkv.bfloat16().cuda()
    w = [(torch.randn(64, 64, generator=g) / 8).bfloat16().cuda() for _ in range(3)]
    v = [(torch.randn(64, generator=g) * 0.1).cuda() for _ in range(5)]
    v[1] += 1.0                                                  # gamma around 1
    return qkv, w, v


def _block_ref(qkv, B, T, scale, w, v, eps=1e-5):
    """torch f32 on the same bf16 qkv and bf16 weights"""
    wo, w1, w2 = (t.float() for t in w)
    bo, gamma, beta, b1, b2 = v
    q, k, vv = (qkv.float().view(B, T, 192)[..., i * 64:(i + 1) * 64] for i in range(3))
    ctx = F.scaled_dot_product_attention(q, k, vv, scale=scale)
    y = vv + ctx @ wo.t() + bo
    z = F.layer_norm(y, (64,), gamma, beta, eps)
    return (y + F.gelu(z @ w1.t() + b1) @ w2.t() + b2).reshape(B * T, 64)


# T = 3136 / 784: the two T2T stages (25 / 7 query tiles and key blocks, 64 / 16 valid keys in the last block); 1000 and 257 other
# key-blocked lengths (one valid key in the last block at 257); 50 takes the short kernel (every key on chip).
@pytest.mark.parametrize("B,T", [(1, 3136), (2, 3136), (3, 784), (2, 1000), (3, 257), (4, 50)])
def test_token_transformer_block_matches_fp32(B, T):
    """Tolerance 3e-2 on |y| ~ 1-4: P is rounded to bf16 as the P V operand, ctx and the LayerNorm / GELU outputs are bf16
    operands of the 64 x 64 products, and a row averages up to 3136 keys; the one-layer long-sequence attention test
    (test_gpu_long_seq.py) holds its context to 3e-2 for the same reasons."""
    from edgevisiontransformer_b200 import _lib
    lib = _lib.load()
    scale = {3136: 147 ** -0.5, 784: 576 ** -0.5}.get(T, 0.125)
    qkv, w, v = _block_inputs(B, T, seed=T + B)
    n = B * T * 64
    buf = torch.full((n + 2 * GUARD,), SENT, dtype=torch.float32, device="cuda")
    y = buf[GUARD:GUARD + n]
    import ctypes as C
    nb = C.c_size_t()
    _lib.check(lib.evt_token_transformer_workspace_bytes(B, T, C.byref(nb)))
    assert nb.value == B * T * 64 * 2
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
    wo, w1, w2 = w
    bo, gamma, beta, b1, b2 = v
    _lib.check(lib.evt_token_transformer_block_fwd(qkv.data_ptr(), 192, y.data_ptr(), ws.data_ptr(), B, T, scale, wo.data_ptr(),
                                                   bo.data_ptr(), gamma.data_ptr(), beta.data_ptr(), w1.data_ptr(), b1.data_ptr(),
                                                   w2.data_ptr(), b2.data_ptr(), 1e-5, torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert bool((buf[:GUARD] == SENT).all()) and bool((buf[GUARD + n:] == SENT).all()), "write outside y"
    want = _block_ref(qkv, B, T, scale, w, v)
    err = (y.view(B * T, 64) - want).abs().max().item()
    assert err < 3e-2, f"token transformer B={B} T={T}: err {err}"
    # the Python wrapper is the same call
    from edgevisiontransformer_b200 import ops
    y2 = ops.token_transformer_block(qkv, B, T, scale, wo, bo, gamma, beta, w1, b1, w2, b2, 1e-5)
    assert torch.equal(y2, y.view(B * T, 64))


def test_public_attention_cap_is_unchanged():
    from edgevisiontransformer_b200 import ops
    qkv = torch.zeros(3136, 192, dtype=torch.bfloat16, device="cuda")
    with pytest.raises(RuntimeError, match="1026"):
        ops.attention(qkv, 1, 3136, 1)


# ------------------------------------------------------------------------------------------------ models

@pytest.mark.parametrize("name,depth,B", [("t2t_vit_t_14", 2, 2), ("t2t_vit_t_14", None, 2), ("t2t_vit_t_19", None, 2),
                                          ("t2t_vit_t_24", None, 2)])
def test_matches_restatement(name, depth, B):
    m = tref.stress_model(name, depth, seed=1)
    b = _b200(name, m, max_batch=8)
    D, L, heads, _ = tref.CONFIGS[name]
    assert (b.hidden, b.num_heads, b.config.num_hidden_layers, b.tokens_type) == (D, heads, L if depth is None else depth, "transformer")
    x = _images(B, seed=2)
    with torch.no_grad():
        want = m(x)
    got = b(x.cuda()).logits
    torch.cuda.synchronize()
    r = _check(got, want)
    print(name, "depth", depth, "max_abs", r["max_abs"])


@pytest.fixture(scope="module")
def t14():
    m = tref.stress_model("t2t_vit_t_14", depth=3, seed=5)
    return m, _b200("t2t_vit_t_14", m, max_batch=4)


def test_pixel_dtypes(t14):
    """bf16 and uint8 NCHW pixels against f32 pixels of the same images (uint8: normalised inside the soft split, the padding of
    the 7 x 7 windows is 0 after normalisation)."""
    m, b = t14
    x = _images(3, seed=6)
    with torch.no_grad():
        xb = x.bfloat16()
        _check(b(xb.cuda()).logits, b(xb.float().cuda()).logits)
        u8 = torch.randint(0, 256, (3, 3, 224, 224), dtype=torch.uint8, generator=torch.Generator().manual_seed(7))
        xn = (u8.float() / 255 - torch.tensor(MEAN).view(1, 3, 1, 1)) / torch.tensor(STD).view(1, 3, 1, 1)
        got = b(u8.cuda()).logits
        _check(got, b(xn.cuda()).logits)
        r = _check(got, m(xn))
        print("uint8 max_abs", r["max_abs"])


def test_forward_graphed_and_chunks(t14):
    from edgevisiontransformer_b200 import ops
    m, b = t14
    x = _images(6, seed=10).cuda()
    try:
        ops.set_gemm_split_k(False)           # fixed summation order: the replay and the chunks are bit-identical
        b._graphs.clear()
        want = b(x[:2]).logits
        assert torch.equal(b.forward_graphed(x[:2]).logits, want)
        big = b(x).logits                     # 6 images > max_batch 4: chunks of 4 and 2
        assert torch.equal(big[:4], b(x[:4]).logits)
        assert torch.equal(big[4:], b(x[4:]).logits)
    finally:
        ops.set_gemm_split_k(True)
        b._graphs.clear()


def test_launch_count(t14):
    from edgevisiontransformer_b200 import _lib
    _, b = t14
    x = _images(2, seed=12).cuda()
    b(x)
    torch.cuda.synchronize()
    lib = _lib.load()
    lib.evt_launch_count_reset()
    b(x)
    torch.cuda.synchronize()
    assert lib.evt_launch_count() == b.launches_per_forward()
    # per token stage 4 launches (soft split + LN, qkv GEMM, attention, tail) instead of the performer's 5
    from edgevisiontransformer_b200 import modeling_t2t
    import t2t_torch_ref as ref
    pm = modeling_t2t.t2t_vit_14(ref.stress_init_(ref.t2t_vit("t2t_vit_14", depth=3)).state_dict(), max_batch=4)
    assert pm.launches_per_forward() - b.launches_per_forward() == 2
    b.profile_begin()
    b(x)
    stages = b.profile_end()
    assert stages["embed"][1] >= 2 * 4 + 1 and stages["embed"][0] > 0


def test_t2t_vit_t_14_batch_256():
    """Batch 256 (802 816 stage-1 token rows, 6400 attention work items): finite, and picked rows agree with a small batch of the
    same images (split-K off) and with the restatement."""
    from edgevisiontransformer_b200 import ops
    m = tref.stress_model("t2t_vit_t_14", seed=2)
    b = _b200("t2t_vit_t_14", m, max_batch=256)
    g = torch.Generator(device="cuda").manual_seed(23)
    x = torch.randn(256, 3, 224, 224, device="cuda", generator=g)
    big = b(x).logits
    assert big.shape == (256, 1000) and torch.isfinite(big).all()
    idx = torch.tensor([0, 1, 128, 255], device="cuda")
    try:
        ops.set_gemm_split_k(False)
        small = b(x[idx].contiguous()).logits
    finally:
        ops.set_gemm_split_k(True)
    _check(big[idx], small)
    with torch.no_grad():
        want = m(x[idx[:2]].cpu())
    r = _check(big[idx[:2]], want)
    print("t2t_vit_t_14 bs256 max_abs", r["max_abs"])
