"""GPU parity tests of the op-level C ABI against plain torch fp32 references (same seeded inputs).

Tolerances: bf16 operands + fp32 accumulation -> compare against the fp32 reference computed from the SAME
bf16-rounded operands, so only accumulation order and the bf16 rounding of the output remain."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import vit as ovit  # noqa: E402


def _ops():
    from edgevisiontransformer_b200 import ops
    return ops


def _rand(shape, seed, scale=1.0, device="cuda"):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(shape, generator=g) * scale).to(device)


@pytest.mark.parametrize("rows,D,eps", [(197, 192, 1e-12), (197 * 3 + 5, 384, 1e-12), (1000, 768, 1e-5),
                                        (64, 64, 1e-5), (33, 576, 1e-5), (50, 147, 1e-5), (7, 1000, 1e-12), (101, 96, 1e-5), (3, 64, 1e-5)])
@pytest.mark.parametrize("out_dtype", [torch.bfloat16, torch.float32])
def test_layernorm(rows, D, eps, out_dtype):
    ops = _ops()
    x = _rand((rows, D), 1, 2.0) + 0.5
    g = 1 + _rand((D,), 2, 0.1)
    b = _rand((D,), 3, 0.1)
    y = ops.layernorm(x, g, b, eps, out_dtype=out_dtype)
    ref = torch.nn.functional.layer_norm(x, (D,), g, b, eps)
    tol = 2e-2 if out_dtype == torch.bfloat16 else 2e-5
    assert (y.float() - ref).abs().max().item() < tol


def test_layernorm_constant_row_and_writeback():
    ops = _ops()
    x = torch.full((4, 192), 3.25, device="cuda")
    g = torch.ones(192, device="cuda")
    b = torch.zeros(192, device="cuda")
    y = ops.layernorm(x, g, b, 1e-12, out_dtype=torch.float32)
    assert torch.isfinite(y).all() and y.abs().max().item() == 0.0      # centred variance: exactly 0, no NaN
    x = _rand((10, 384), 4)
    ref = torch.nn.functional.layer_norm(x, (384,), g.new_ones(384), g.new_zeros(384), 1e-5)
    y = ops.layernorm(x, g.new_ones(384), g.new_zeros(384), 1e-5, write_back=True)
    assert (x - ref).abs().max().item() < 2e-5 and (y.float() - ref).abs().max().item() < 2e-2


def test_layernorm2d():
    ops = _ops()
    x = _rand((3, 197, 192), 5)
    add = _rand((3, 197, 192), 6)
    g = 1 + _rand((197, 192), 7, 0.1)
    b = _rand((197, 192), 8, 0.1)
    y = ops.layernorm2d(x, g, b, 1e-5, addend=add)
    ref = torch.nn.functional.layer_norm(x + add, (197, 192), g, b, 1e-5)
    assert (y - ref).abs().max().item() < 5e-5


GEMM_SHAPES = [
    # (M, N, K)  -- DeiT shapes, pruned widths, alignment cliffs from the reference's sweeps (SURVEY 4.3)
    (197, 576, 192), (197 * 4, 192, 192), (197 * 2, 768, 192), (197 * 2, 192, 768),
    (394, 2304, 768), (300, 768, 3072), (256, 3072, 768),
    (197, 192, 64), (197, 64, 192), (197, 230, 192), (197, 192, 230), (197, 231, 192),
    (1, 1000, 192), (5, 1000, 768), (129, 160, 200), (128, 8, 8), (1000, 1, 64), (63, 3072, 768), (16, 32, 4096),
]


@pytest.mark.parametrize("M,N,K", GEMM_SHAPES)
def test_gemm_bias(M, N, K):
    ops = _ops()
    lda, ldw = (K + 7) // 8 * 8, (K + 7) // 8 * 8
    a = torch.zeros((M, lda), dtype=torch.bfloat16, device="cuda")
    w = torch.zeros((N, ldw), dtype=torch.bfloat16, device="cuda")
    a[:, :K] = _rand((M, K), 1).bfloat16()
    w[:, :K] = _rand((N, K), 2, 0.05).bfloat16()
    if lda > K:   # garbage in the pad columns must be ignored (TMA zero fill past K)
        a[:, K:] = 7.0
        w[:, K:] = -3.0
    bias = _rand((N,), 3, 0.1)
    ref = a[:, :K].float() @ w[:, :K].float().t() + bias
    out = ops.linear(a, w, bias, out_dtype=torch.float32, k=K)
    err = (out - ref).abs().max().item()
    assert err < 2e-3 * max(1.0, math.sqrt(K) * 0.05), f"f32-out err {err}"
    outb = ops.linear(a, w, bias, out_dtype=torch.bfloat16, k=K)
    errb = (outb.float() - ref).abs().max().item()
    assert errb < 1e-2 * max(1.0, ref.abs().max().item()), f"bf16-out err {errb}"


PAIR_SHAPES = [
    # (M, N, K): exercise the CTA-pair (cta_group::2) kernel -- 256-row tiles with an M tail inside the leader's half,
    # inside the peer's half, N tiles of 256 / 192 / 128 incl. N tails, K tails, several tiles per pair (pipeline wrap).
    (256 * 3 + 57, 768, 192), (256 * 2 + 128 + 31, 2304, 768), (197 * 40, 3072, 768), (197 * 40, 768, 3072),
    (1000, 576, 192), (1000, 384, 384), (777, 230, 192), (777, 192, 230), (130, 128, 64), (256 * 80, 256, 64),
]


@pytest.mark.parametrize("M,N,K", PAIR_SHAPES)
def test_gemm_pair_kernel_matches_single_cta(M, N, K):
    """The CTA-pair kernel must reproduce the single-CTA kernel bit for bit (same K order, same epilogue) and both
    must match the fp32 reference."""
    ops = _ops()
    ld = (K + 7) // 8 * 8
    a = torch.zeros((M, ld), dtype=torch.bfloat16, device="cuda")
    w = torch.zeros((N, ld), dtype=torch.bfloat16, device="cuda")
    a[:, :K] = _rand((M, K), 11).bfloat16()
    w[:, :K] = _rand((N, K), 12, 0.05).bfloat16()
    bias = _rand((N,), 13, 0.1)
    res0 = _rand((M, N), 14)
    ref = a[:, :K].float() @ w[:, :K].float().t() + bias
    outs = {}
    try:
        for mode in (0, 1):
            ops.set_gemm_pair_mode(mode)
            ldo = (N + 7) // 8 * 8
            ob = torch.zeros((M, ldo), dtype=torch.bfloat16, device="cuda")
            ops.linear(a, w, bias, act="gelu_erf", out=ob, out_dtype=torch.bfloat16, k=K, n=N)
            of = None
            if N % 4 == 0:
                of = res0.clone()
                ops.linear(a, w, bias, residual=of, out=of, out_dtype=torch.float32, k=K)
            outs[mode] = (ob, of)
    finally:
        ops.set_gemm_pair_mode(-1)
    torch.cuda.synchronize()
    assert torch.equal(outs[0][0], outs[1][0])
    assert (outs[1][0][:, :N].float() - ovit.gelu_erf(ref)).abs().max().item() < 1e-2 * max(1.0, ref.abs().max().item())
    if outs[0][1] is not None:
        assert torch.equal(outs[0][1], outs[1][1])
        assert (outs[1][1] - (ref + res0)).abs().max().item() < 2e-3 * max(1.0, math.sqrt(K) * 0.05)


@pytest.mark.parametrize("M,N,K", [(197 * 3, 768, 768), (1000, 384, 384), (777, 192, 768), (256 * 3 + 5, 768, 3072),
                                   (130, 64, 64), (600, 320, 192), (197 * 40, 768, 230), (256 * 80 + 129, 768, 768)])
def test_gemm_residual_layernorm_fused(M, N, K):
    """x += a w^T + b ; xn = LN(x): the fused kernel against fp32 torch, and bit-exact residual against the
    unfused GEMM (same accumulation, same single f32 add)."""
    ops = _ops()
    ld = (K + 7) // 8 * 8
    a = torch.zeros((M, ld), dtype=torch.bfloat16, device="cuda")
    w = torch.zeros((N, ld), dtype=torch.bfloat16, device="cuda")
    a[:, :K] = _rand((M, K), 21).bfloat16()
    w[:, :K] = _rand((N, K), 22, 0.05).bfloat16()
    bias = _rand((N,), 23, 0.1)
    res0 = _rand((M, N), 24) + 0.5 * _rand((M, 1), 25)       # rows with different means
    gamma = 1 + _rand((N,), 26, 0.1)
    beta = _rand((N,), 27, 0.1)
    eps = 1e-12
    want_res = res0 + a[:, :K].float() @ w[:, :K].float().t() + bias
    want_xn = torch.nn.functional.layer_norm(want_res, (N,), gamma, beta, eps)
    res = res0.clone()
    unfused = res0.clone()
    try:
        # Deterministic accumulation order on both sides: by default the entry point issues the residual GEMM and the
        # LayerNorm kernel (a single-kernel version lost its A/B test and was removed), and a small-M residual GEMM
        # splits K over idle SMs, whose reduce-adds land in any order.
        ops.set_gemm_split_k(False)
        xn = ops.linear_residual_layernorm(a, w, bias, res, gamma, beta, eps, k=K)
        torch.cuda.synchronize()
        ops.set_gemm_pair_mode(0)           # forced kernel choice: the 1-CTA kernel
        ops.linear(a, w, bias, residual=unfused, out=unfused, out_dtype=torch.float32, k=K)
    finally:
        ops.set_gemm_pair_mode(-1)
        ops.set_gemm_split_k(True)
    assert torch.equal(res, unfused)
    assert (res - want_res).abs().max().item() < 2e-3 * max(1.0, math.sqrt(K) * 0.05)
    ref_xn = torch.nn.functional.layer_norm(res, (N,), gamma, beta, eps)
    assert (xn.float() - ref_xn).abs().max().item() < 2e-2          # bf16 output of O(1..4) values
    assert (xn.float() - ref_xn.bfloat16().float()).abs().mean().item() < 1e-3
    assert (xn.float() - want_xn).abs().max().item() < 4e-2


@pytest.mark.parametrize("rows", [16, 37, 3136 * 3 + 5])
def test_performer_tail_in_one_kernel(rows):
    """evt_performer_mlp_fwd: y = v + attn_output(ya); y += fc2(gelu_tanh(fc1(LN(y)))) for 64-wide tokens -- against fp32 torch on the
    bf16-rounded operands, and against the four kernels it replaces (same operand roundings: agreement to summation order)."""
    ops = _ops()
    ya = _rand((rows, 64), 51).bfloat16()
    v = _rand((rows, 64), 52) + 0.3 * _rand((rows, 1), 53)
    wo, w1, w2 = (_rand((64, 64), 54 + i, 0.15).bfloat16() for i in range(3))
    bo, b1, b2 = (_rand((64,), 57 + i, 0.1) for i in range(3))
    gamma, beta = 1 + _rand((64,), 60, 0.1), _rand((64,), 61, 0.1)
    eps = 1e-5
    canary = torch.full((8, 64), 7.0, device="cuda")
    buf = torch.cat([v, canary])
    y = ops.performer_mlp(ya, buf[:rows], wo, bo, gamma, beta, w1, b1, w2, b2, eps)
    # the four-kernel path
    y4 = v.clone()
    ops.linear(ya, wo, bo, residual=y4, out=y4, out_dtype=torch.float32)
    z = ops.layernorm(y4, gamma, beta, eps)
    h = ops.linear(z, w1, b1, act="gelu_tanh")
    ops.linear(h, w2, b2, residual=y4, out=y4, out_dtype=torch.float32)
    torch.cuda.synchronize()
    assert torch.equal(buf[rows:], canary)
    # fp32 reference with the same roundings of the two intermediate operands
    y1 = v + ya.float() @ wo.float().t() + bo
    zr = torch.nn.functional.layer_norm(y1, (64,), gamma, beta, eps).bfloat16().float()
    hr = torch.nn.functional.gelu(zr @ w1.float().t() + b1, approximate="tanh").bfloat16().float()
    want = y1 + hr @ w2.float().t() + b2
    assert (y - want).abs().max().item() < 2e-2
    assert (y - want).abs().mean().item() < 1e-3
    assert (y - y4).abs().max().item() < 2e-2 and (y - y4).abs().mean().item() < 1e-3


@pytest.mark.parametrize("B,T", [(2, 784), (3, 100), (1, 3136)])
def test_performer_block_equals_its_two_halves(B, T):
    """evt_performer_block_fwd (the apply kernel carries each tile through attn_output + LayerNorm + MLP) is bit-identical to
    evt_performer_fwd followed by evt_performer_mlp_fwd; T = 100 leaves a partial 16-token tile and a partial 256-token chunk."""
    ops = _ops()
    kqv = _rand((B * T, 192), 71, 0.5).bfloat16()
    w = _rand((32, 64), 72) * math.sqrt(32) / 8
    wo, w1, w2 = (_rand((64, 64), 73 + i, 0.15).bfloat16() for i in range(3))
    bo, b1, b2 = (_rand((64,), 76 + i, 0.1) for i in range(3))
    gamma, beta = 1 + _rand((64,), 79, 0.1), _rand((64,), 80, 0.1)
    ya, v = ops.performer(kqv, w, B, T)
    two = ops.performer_mlp(ya, v, wo, bo, gamma, beta, w1, b1, w2, b2, 1e-5)
    one = ops.performer_block(kqv, w, B, T, wo, bo, gamma, beta, w1, b1, w2, b2, 1e-5)
    torch.cuda.synchronize()
    assert torch.isfinite(one).all() and torch.equal(one, two)


@pytest.mark.parametrize("M,N,K,copy_ln", [(256 * 80 + 129, 192, 64, False), (256 * 90 + 1, 192, 230, False), (256 * 75, 384, 384, False),
                                         (256 * 74 + 255, 384, 1536, False), (256 * 80 + 129, 192, 230, True),
                                         (256 * 77 + 33, 384, 1152, True), (197 * 1024, 192, 64, False)])
def test_gemm_residual_layernorm_rows_in_tmem(M, N, K, copy_ln):
    """csrc/gemm_rowln.cu (N = 192 / 384, every CTA pair gets a 256-row block): the new residual stream is bit-identical to the
    TMA reduce-add GEMM (same accumulation, same single f32 add), the normalised rows match the LayerNorm of that stream, and
    the TF dialect (copy_ln) leaves the unrounded normalised rows in the stream.  Row tails, K tails (230) and K = 64 included."""
    ops = _ops()
    ld = (K + 7) // 8 * 8
    a = torch.zeros((M, ld), dtype=torch.bfloat16, device="cuda")
    w = torch.zeros((N, ld), dtype=torch.bfloat16, device="cuda")
    a[:, :K] = _rand((M, K), 31).bfloat16()
    w[:, :K] = _rand((N, K), 32, 0.05).bfloat16()
    bias = _rand((N,), 33, 0.1)
    res0 = _rand((M, N), 34) + 0.5 * _rand((M, 1), 35)
    res0[:, 7] += 40.0                                         # an outlier channel, as trained ViTs have
    gamma = 1 + _rand((N,), 36, 0.1)
    beta = _rand((N,), 37, 0.1)
    eps = 1e-5 if copy_ln else 1e-12
    res = res0.clone()
    canary = torch.full((64, N), 7.0, device="cuda", dtype=torch.bfloat16)
    xn_buf = torch.cat([torch.empty((M, N), dtype=torch.bfloat16, device="cuda"), canary])
    xn = ops.linear_residual_layernorm(a, w, bias, res, gamma, beta, eps, k=K, xn=xn_buf[:M], copy_ln=copy_ln)
    unfused = res0.clone()
    ops.linear(a, w, bias, residual=unfused, out=unfused, out_dtype=torch.float32, k=K)
    torch.cuda.synchronize()
    assert torch.equal(xn_buf[M:], canary)                     # nothing written past row M
    ref_xn = torch.nn.functional.layer_norm(unfused, (N,), gamma, beta, eps)
    if copy_ln:
        assert (res - ref_xn).abs().max().item() < 2e-4 * max(1.0, ref_xn.abs().max().item())
        assert torch.equal(xn, res.bfloat16())
    else:
        assert torch.equal(res, unfused)
        assert (xn.float() - ref_xn).abs().max().item() < 1e-2 * max(1.0, ref_xn.abs().max().item())
        assert (xn.float() - ref_xn.bfloat16().float()).abs().mean().item() < 1e-3
    want = res0 + a[:, :K].float() @ w[:, :K].float().t() + bias
    assert (unfused - want).abs().max().item() < 2e-3 * max(1.0, math.sqrt(K) * 0.05)


def test_gemm_residual_layernorm_rows_in_tmem_constant_rows():
    """Exactly constant rows with eps = 1e-12: the centred variance is exactly 0, so xn == beta (no NaN / inf)."""
    ops = _ops()
    M, N, K = 256 * 80, 192, 64
    a = torch.zeros((M, K), dtype=torch.bfloat16, device="cuda")
    w = _rand((N, K), 41, 0.05).bfloat16()
    res = torch.full((M, N), 3.25, device="cuda")
    gamma, beta = 1 + _rand((N,), 42, 0.1), _rand((N,), 43, 0.1)
    xn = ops.linear_residual_layernorm(a, w, None, res, gamma, beta, 1e-12)
    assert torch.isfinite(xn.float()).all()
    assert (xn.float() - beta.bfloat16().float()).abs().max().item() == 0.0


@pytest.mark.parametrize("M,N,K,act", [(128 * 3 + 5, 576, 192, None), (1000, 230, 192, "gelu_erf"), (777, 1152, 384, None),
                                       (300, 1536, 384, "gelu_erf"), (130, 192, 64, "gelu_tanh"), (515, 768, 256, "gelu_tanh"),
                                       (128 * 150 + 77, 192, 192, None), (64, 100, 128, None)])
def test_layernorm_fused_into_the_projection(M, N, K, act):
    """evt_layernorm_gemm: act(LN(x) W^T + b) in one kernel against fp32 torch, and against the two-kernel path (LayerNorm
    kernel + GEMM) -- same f32 statistics, same bf16 rounding of the normalised rows, so the outputs agree to bf16
    rounding of the result.  Also the TF-dialect write-back of the normalised rows."""
    ops = _ops()
    x = _rand((M, K), 41) * 2 + 0.3 * _rand((M, 1), 42)
    gamma = 1 + _rand((K,), 43, 0.1)
    beta = _rand((K,), 44, 0.1)
    w = _rand((N, K), 45, 0.05).bfloat16()
    bias = _rand((N,), 46, 0.1)
    eps = 1e-12 if K != 256 else 1e-5
    xn_ref = torch.nn.functional.layer_norm(x, (K,), gamma, beta, eps)
    z = xn_ref.bfloat16().float() @ w.float().t() + bias
    ref = z if act is None else (ovit.gelu_erf(z) if act == "gelu_erf" else ovit.gelu_tanh(z))
    got = ops.layernorm_linear(x, gamma, beta, eps, w, bias, act=act)
    assert got.shape == (M, N) and got.dtype == torch.bfloat16
    tol = 2e-2 * max(1.0, ref.abs().max().item())
    assert (got.float() - ref).abs().max().item() < tol
    xn = ops.layernorm(x, gamma, beta, eps)
    two = ops.linear(xn, w, bias, act=act)
    assert (got.float() - two.float()).abs().max().item() <= 1.6e-2 * max(1.0, ref.abs().max().item())
    assert (got.float() - two.float()).abs().mean().item() < 1e-4
    x2 = x.clone()
    got2 = ops.layernorm_linear(x2, gamma, beta, eps, w, bias, act=act, write_back=True)
    assert torch.equal(got2, got)
    assert (x2 - xn_ref).abs().max().item() < 2e-5 * max(1.0, xn_ref.abs().max().item())


def test_gemm_residual_layernorm_constant_rows():
    """eps = 1e-12 and rows that are exactly constant: the centred variance must be exactly 0 -> xn == beta."""
    ops = _ops()
    M, N, K = 300, 768, 64
    a = _rand((M, K), 1).bfloat16()
    w = torch.zeros((N, K), dtype=torch.bfloat16, device="cuda")
    # constants whose 768-term sums are exact in f32 (multiples of 1/4 up to 64): the mean is then exact for any
    # summation order, which is what "exactly constant" needs with eps = 1e-12
    res = (torch.round(_rand((M, 1), 2) * 100).clamp(-256, 256) / 4).expand(M, N).contiguous()
    gamma = 1 + _rand((N,), 3, 0.1)
    beta = _rand((N,), 4, 0.1)
    xn = ops.linear_residual_layernorm(a, w, None, res, gamma, beta, 1e-12)
    assert torch.isfinite(xn.float()).all()
    assert (xn.float() - beta.bfloat16().float()).abs().max().item() == 0.0


@pytest.mark.parametrize("M,N,K", [(197, 768, 3072), (197, 768, 768), (198, 384, 1536), (394, 192, 768), (1, 768, 3072)])
def test_gemm_split_k_small_m(M, N, K):
    """Batch-1 shapes: the residual GEMMs split K over the idle SMs (partial products meet in the TMA reduce-add)."""
    ops = _ops()
    a = _rand((M, K), 31).bfloat16()
    w = _rand((N, K), 32, 0.05).bfloat16()
    bias = _rand((N,), 33, 0.1)
    res0 = _rand((M, N), 34)
    want = res0 + a.float() @ w.float().t() + bias
    res = res0.clone()
    ops.linear(a, w, bias, residual=res, out=res, out_dtype=torch.float32)
    assert (res - want).abs().max().item() < 2e-3 * max(1.0, math.sqrt(K) * 0.05)
    # plain-store outputs at the same small M use narrow tiles (no split): still exact against the reference
    out = ops.linear(a, w, bias, out_dtype=torch.float32)
    assert (out - (want - res0)).abs().max().item() < 2e-3 * max(1.0, math.sqrt(K) * 0.05)


@pytest.mark.parametrize("act", ["gelu_erf", "gelu_tanh"])
def test_gemm_gelu_and_residual(act):
    ops = _ops()
    M, N, K = 197 * 3, 768, 192
    a = _rand((M, K), 1).bfloat16()
    w = _rand((N, K), 2, 0.08).bfloat16()
    bias = _rand((N,), 3, 0.2)
    z = a.float() @ w.float().t() + bias
    ref = ovit.gelu_erf(z) if act == "gelu_erf" else ovit.gelu_tanh(z)
    out = ops.linear(a, w, bias, act=act, out_dtype=torch.float32)
    assert (out - ref).abs().max().item() < 2e-3
    # residual, in place: out aliases residual
    res = _rand((M, N), 4)
    want = z + res
    got = ops.linear(a, w, bias, residual=res, out=res, out_dtype=torch.float32)
    assert got.data_ptr() == res.data_ptr()
    assert (res - want).abs().max().item() < 2e-3


def test_gemm_tf32():
    ops = _ops()
    M, N, K = 197, 576, 192
    a = _rand((M, K), 1)
    w = _rand((N, K), 2, 0.05)
    bias = _rand((N,), 3, 0.1)
    ref = a @ w.t() + bias
    out = ops.linear(a, w, bias, out_dtype=torch.float32)
    assert (out - ref).abs().max().item() < 5e-3           # tf32: 10-bit mantissa operands


def _attn_ref(qkv, B, S, heads, hs=64):
    a = heads * hs
    q, k, v = qkv[:, :a].float(), qkv[:, a:2 * a].float(), qkv[:, 2 * a:3 * a].float()
    return ovit.attention(q.view(B, S, a), k.view(B, S, a), v.view(B, S, a), hs).reshape(B * S, a)


@pytest.mark.parametrize("B,S,heads", [(2, 197, 3), (1, 198, 1), (3, 128, 2), (2, 40, 6), (1, 256, 2), (5, 197, 12), (2, 16, 1), (1, 1, 1)])
def test_attention(B, S, heads):
    ops = _ops()
    qkv = _rand((B * S, 3 * heads * 64), 1, 1.0).bfloat16()
    ctx = ops.attention(qkv, B, S, heads)
    ref = _attn_ref(qkv, B, S, heads)
    err = (ctx.float() - ref).abs().max().item()
    assert err < 2e-2, f"attention err {err}"


@pytest.mark.parametrize("B,S,heads", [(2, 197, 3), (1, 198, 1), (3, 128, 2), (1, 256, 2), (2, 16, 1)])
def test_attention_tf32(B, S, heads):
    ops = _ops()
    qkv = _rand((B * S, 3 * heads * 64), 1, 1.0)
    ctx = ops.attention(qkv, B, S, heads)
    ref = _attn_ref(qkv, B, S, heads)
    err = (ctx - ref).abs().max().item()
    assert ctx.dtype == torch.float32 and err < 3e-3, f"tf32 attention err {err}"


def test_attention_head_mask_and_peaky_scores():
    ops = _ops()
    B, S, heads = 2, 197, 3
    qkv = _rand((B * S, 3 * heads * 64), 2, 3.0).bfloat16()       # large logits: softmax near one-hot
    mask = torch.tensor([1.0, 0.0, 1.0], device="cuda")
    ctx = ops.attention(qkv, B, S, heads, head_mask=mask)
    ref = _attn_ref(qkv, B, S, heads).view(B * S, heads, 64) * mask.view(1, heads, 1)
    assert (ctx.float() - ref.reshape(B * S, -1)).abs().max().item() < 6e-2
    assert ctx.view(B * S, heads, 64)[:, 1].abs().max().item() == 0.0


def test_im2col_and_cast_and_unfold():
    ops = _ops()
    x = _rand((3, 3, 224, 224), 1)
    cols = ops.im2col_patch(x, 16)
    ref = x.reshape(3, 3, 14, 16, 14, 16).permute(0, 2, 4, 1, 3, 5).reshape(3 * 196, 768).bfloat16()
    assert torch.equal(cols, ref)                                   # pure gather + RN rounding: bit exact
    v = _rand((1003,), 2)
    assert torch.equal(ops.cast_bf16(v), v.bfloat16())
    from oracle import t2t as ot2t
    img = _rand((2, 30, 30, 3), 3)
    u = ops.unfold_nhwc(img, 7, 4, 2)
    refu = ot2t.unfold_nhwc(img.cpu(), 7, 4, 2).reshape(-1, 147)
    assert u.shape[1] == 152
    assert torch.equal(u[:, :147].cpu(), refu.bfloat16()) and u[:, 147:].abs().max().item() == 0


@pytest.mark.parametrize("kind,B,D", [("vit", 3, 192), ("deit", 2, 384), ("vit", 140, 192)])
def test_patch_embed_matches_hf_embeddings(kind, B, D):
    """evt_patch_embed_fwd = `ViTEmbeddings.forward` / `DeiTEmbeddings.forward` of the installed transformers (the module the
    reference calls): Conv2d patch projection + cls (and distillation) token + position embeddings, f32 / bf16 / raw uint8
    pixels.  The live HF module is the checker.  B = 140: 27 580 token rows, the CTA-pair GEMM path."""
    from transformers import DeiTConfig, DeiTModel, ViTConfig, ViTModel
    ops = _ops()
    torch.manual_seed(11)
    kw = dict(hidden_size=D, num_hidden_layers=1, num_attention_heads=D // 64, intermediate_size=2 * D)
    emb = (ViTModel(ViTConfig(**kw), add_pooling_layer=False) if kind == "vit" else DeiTModel(DeiTConfig(**kw), add_pooling_layer=False)).embeddings.eval()
    with torch.no_grad():
        for prm in emb.parameters():
            prm.copy_(torch.randn_like(prm) * (0.05 if prm.dim() == 4 else 0.5))
    conv = emb.patch_embeddings.projection
    prefix = emb.cls_token[0] if kind == "vit" else torch.cat((emb.cls_token[0], emb.distillation_token[0]), 0)
    args = [t.detach().cuda() for t in (conv.weight, conv.bias, prefix, emb.position_embeddings[0])]
    x = torch.randn(B, 3, 224, 224, generator=torch.Generator().manual_seed(12))
    with torch.no_grad():
        ref = emb(x)
    out = ops.patch_embed(x.cuda(), *args)
    assert out.shape == ref.shape == (B, 197 if kind == "vit" else 198, D)
    # bf16 pixels and weights, f32 accumulation over K = 768: |sum| ~ 1.4, rounding ~ 2^-9 per operand
    assert (out.cpu() - ref).abs().max().item() < 2e-2
    assert torch.equal(out[:, : prefix.shape[0]].cpu(), (prefix + emb.position_embeddings[0, : prefix.shape[0]]).detach().expand(B, -1, -1))
    outb = ops.patch_embed(x.bfloat16().cuda(), *args)
    # the f32 path rounds its pixels to bf16 in the gather: same operands; split K at small M leaves the f32 add order open
    assert (outb - out).abs().max().item() < 1e-4
    if B <= 3:
        mean, std = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)    # deit_pruning/src/utils.py:105-107
        u8 = torch.randint(0, 256, (B, 3, 224, 224), dtype=torch.uint8, generator=torch.Generator().manual_seed(13))
        xn = (u8.float() / 255 - torch.tensor(mean).view(1, 3, 1, 1)) / torch.tensor(std).view(1, 3, 1, 1)
        with torch.no_grad():
            refu = emb(xn)
        outu = ops.patch_embed(u8.cuda(), *args, mean=mean, std=std)
        assert (outu.cpu() - refu).abs().max().item() < 4e-2        # normalised pixels reach |x| ~ 2.6


def test_errors_are_loud():
    ops = _ops()
    with pytest.raises(RuntimeError):
        ops.layernorm(torch.zeros(4, 8), torch.ones(8), torch.zeros(8), 1e-5)          # CPU tensor
    a = torch.zeros((4, 12), dtype=torch.bfloat16, device="cuda")
    with pytest.raises(ValueError):
        ops.linear(a[:, :9], a[:, :9], None)           # 24-byte rows: not a legal TMA leading dimension -> EVT_ERR_INVALID


@pytest.mark.parametrize("B,T", [(2, 784), (3, 50), (1, 3136), (2, 257)])
def test_performer_core_matches_restatement(B, T):
    """evt_performer_fwd (TokenPerformer.single_attn core, transformer_encoder.py:67-94) against oracle.t2t.prm_exp; T values
    cover partial 16-token tiles and partial 256-token blocks."""
    import math
    from edgevisiontransformer_b200 import ops
    from oracle import t2t as ot2t
    g = torch.Generator().manual_seed(T)
    kqv = (torch.randn(B * T, 192, generator=g) * 0.7).bfloat16()
    q_, _ = torch.linalg.qr(torch.randn(64, 32, generator=g))
    w = (q_.t() * math.sqrt(32)).contiguous()
    k, q, v = [t.float().view(B, T, 64) for t in kqv.split(64, dim=1)]
    kp, qp = ot2t.prm_exp(k, w), ot2t.prm_exp(q, w)
    D = torch.einsum("bti,bi->bt", qp, kp.sum(dim=1)).unsqueeze(2)
    want = torch.einsum("bti,bni->btn", qp, torch.einsum("bin,bim->bnm", v, kp)) / (D + 1e-8)
    yattn, vout = ops.performer(kqv.cuda(), w.cuda(), B, T)
    assert torch.equal(vout.cpu(), v.reshape(B * T, 64))                      # the skip input is an exact copy
    err = (yattn.float().cpu().view(B, T, 64) - want).abs().max().item()
    assert err < 2e-2 * max(1.0, want.abs().max().item()), err                # bf16 operands / output
    assert (yattn.float().cpu().view(B, T, 64) - want).abs().mean().item() < 2e-3
