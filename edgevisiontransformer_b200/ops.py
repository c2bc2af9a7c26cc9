"""Op-level torch wrappers over the libevt C ABI.  torch supplies device memory and the stream only.

Every function requires CUDA tensors; a CPU tensor raises (there is no CPU path in the product).
"""
from __future__ import annotations

from typing import Optional

import torch

from . import _lib
from ._lib import ACT_GELU_ERF, ACT_GELU_TANH, ACT_NONE, EVT_BF16, EVT_F32, EVT_TF32  # noqa: F401

# out_dtype of layernorm / linear / gather_layernorm / layernorm_mean_tokens / im2col_patch: an f32 tensor whose values are
# rounded to nearest tf32 when written (the operand of a tf32 GEMM or attention, whose tensor cores would truncate).
TF32 = "tf32"

ACTS = {None: ACT_NONE, "none": ACT_NONE, "gelu": ACT_GELU_ERF, "gelu_erf": ACT_GELU_ERF, "erf": ACT_GELU_ERF,
        "gelu_tanh": ACT_GELU_TANH, "gelu_new": ACT_GELU_TANH, "gelu_pytorch_tanh": ACT_GELU_TANH}
# "tanh" is not an alias: HF's ACT2FN["tanh"] is plain nn.Tanh, which the fused epilogue does not implement.


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _need_cuda(*ts: Optional[torch.Tensor]) -> None:
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("edgevisiontransformer_b200 ops need CUDA tensors on a B200 (sm_100a); "
                               "there is no CPU fallback")


def _storage(out_dtype) -> torch.dtype:
    return torch.float32 if out_dtype == TF32 else out_dtype


def _dt(t: torch.Tensor, out_dtype=None) -> int:
    if out_dtype == TF32:
        return EVT_TF32
    if t.dtype == torch.float32:
        return EVT_F32
    if t.dtype == torch.bfloat16:
        return EVT_BF16
    raise ValueError(f"unsupported dtype {t.dtype}")


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def round_tf32(x: torch.Tensor) -> torch.Tensor:
    """f32 -> the nearest tf32 value (ties away from zero), as f32: what ``cvt.rna.tf32.f32`` gives, i.e. what the tf32 mode's
    kernels write.  Finite inputs; any device."""
    b = x.float().contiguous().view(torch.int32)
    return ((b + 0x1000) & ~0x1FFF).view(torch.float32)


def layernorm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float,
              out_dtype: torch.dtype = torch.bfloat16, write_back: bool = False) -> torch.Tensor:
    """LayerNorm over the last dim of an f32 tensor whose rows are contiguous (out_dtype bf16, f32 or TF32).
    write_back: x <- LN(x) too."""
    _need_cuda(x, gamma, beta)
    if x.dtype != torch.float32 or x.stride(-1) != 1:
        raise ValueError("layernorm wants an f32 tensor with unit inner stride")
    D = x.shape[-1]
    x2 = x.reshape(-1, D)
    if x2.data_ptr() != x.data_ptr():
        raise ValueError("layernorm wants a tensor viewable as [rows, D]")
    y = torch.empty(x2.shape, dtype=_storage(out_dtype), device=x.device)
    lib = _lib.load()
    _lib.check(lib.evt_layernorm_fwd(x2.data_ptr(), x2.stride(0), gamma.data_ptr(), beta.data_ptr(), y.data_ptr(), _dt(y, out_dtype),
                                     y.stride(0), x2.data_ptr() if write_back else None, x2.shape[0], D, float(eps),
                                     _stream()), "layernorm")
    return y.view(*x.shape)


def layernorm_rows(x: torch.Tensor, row_stride: int, rows: int, D: int, gamma, beta, eps, out_dtype=torch.bfloat16):
    """LayerNorm of `rows` rows of length D spaced row_stride elements apart (cls rows of [B,S,D])."""
    _need_cuda(x, gamma, beta)
    y = torch.empty((rows, D), dtype=out_dtype, device=x.device)
    lib = _lib.load()
    _lib.check(lib.evt_layernorm_fwd(x.data_ptr(), row_stride, gamma.data_ptr(), beta.data_ptr(), y.data_ptr(), _dt(y), D,
                                     None, rows, D, float(eps), _stream()), "layernorm")
    return y


def layernorm2d(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-5,
                addend: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Joint LayerNorm over the last two dims of f32 x[B,n,h] (+addend), affine [n,h]."""
    _need_cuda(x, gamma, beta, addend)
    x = x.contiguous()
    if addend is not None:
        addend = addend.contiguous()
    B = x.shape[0]
    nh = x[0].numel()
    if gamma.numel() != nh or beta.numel() != nh:
        raise ValueError("layernorm2d: affine parameters must have n*h elements")
    y = torch.empty_like(x)
    lib = _lib.load()
    _lib.check(lib.evt_layernorm2d_fwd(x.data_ptr(), _ptr(addend), gamma.contiguous().data_ptr(),
                                       beta.contiguous().data_ptr(), y.data_ptr(), B, nh, float(eps), _stream()),
               "layernorm2d")
    return y


def linear(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor] = None, act=None,
           residual: Optional[torch.Tensor] = None, out_dtype: torch.dtype = torch.bfloat16,
           out: Optional[torch.Tensor] = None, n: Optional[int] = None, k: Optional[int] = None) -> torch.Tensor:
    """out[M,N] = act(a[M,K] @ w[N,K]^T + bias) (+ residual).  a, w bf16 (tensor cores, f32 accumulate) or
    both f32 (tf32 mode; out_dtype f32 or TF32).  Row strides may exceed the logical K / N (padded leading dimensions)."""
    _need_cuda(a, w, bias, residual, out)
    if a.dim() != 2 or w.dim() != 2 or a.stride(1) != 1 or w.stride(1) != 1:
        raise ValueError("linear wants 2-D operands with unit inner stride")
    if a.dtype != w.dtype:
        raise ValueError("linear: a and w must have the same dtype")
    M = a.shape[0]
    K = k if k is not None else a.shape[1]
    N = n if n is not None else w.shape[0]
    if w.shape[1] < K or a.shape[1] < K:
        raise ValueError("linear: K exceeds operand width")
    rounded = out_dtype == TF32
    if out is None:
        out = torch.empty((M, N), dtype=_storage(out_dtype), device=a.device)
    if residual is not None and (residual.dtype != torch.float32 or residual.stride(1) != 1):
        raise ValueError("linear: residual must be f32 with unit inner stride")
    lib = _lib.load()
    act_id = ACTS[act] if not isinstance(act, int) else act
    if a.dtype == torch.bfloat16:
        if rounded:
            raise ValueError("linear: a TF32 output needs f32 (tf32-mode) operands")
        rc = lib.evt_gemm_bias_act(a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), _ptr(bias), _ptr(residual),
                                   residual.stride(0) if residual is not None else 0, 0, 0, out.data_ptr(), _dt(out),
                                   out.stride(0), 0, 0, 0, M, N, K, act_id, _stream())
    elif a.dtype == torch.float32:
        if out.dtype != torch.float32:
            raise ValueError("linear: tf32 mode writes f32")
        if rounded:
            rc = lib.evt_gemm_bias_act_tf32_ex(a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), _ptr(bias), _ptr(residual),
                                               residual.stride(0) if residual is not None else 0, 0, 0, out.data_ptr(), EVT_TF32,
                                               out.stride(0), 0, 0, 0, M, N, K, act_id, _stream())
        else:
            rc = lib.evt_gemm_bias_act_tf32(a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), _ptr(bias), _ptr(residual),
                                            residual.stride(0) if residual is not None else 0, 0, 0, out.data_ptr(),
                                            out.stride(0), 0, 0, 0, M, N, K, act_id, _stream())
    else:
        raise ValueError(f"linear: unsupported dtype {a.dtype}")
    _lib.check(rc, "gemm")
    return out


def layernorm_linear(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float, w: torch.Tensor,
                     bias: Optional[torch.Tensor] = None, act=None, write_back: bool = False,
                     out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """act(LayerNorm(x) @ w^T + bias) in ONE kernel (the LayerNorm is the producer of the GEMM's A operand): x f32 [M, K]
    with K in {64, 128, 192, 256, 384}, w bf16 [N, >=K] -> bf16 [M, N].  write_back: x <- LayerNorm(x) (TF dialect)."""
    _need_cuda(x, gamma, beta, w, bias, out)
    if x.dtype != torch.float32 or w.dtype != torch.bfloat16 or x.dim() != 2 or w.dim() != 2 or x.stride(1) != 1 or w.stride(1) != 1:
        raise ValueError("layernorm_linear wants a 2-D f32 x and a 2-D bf16 w with unit inner strides")
    M, K = x.shape
    N = w.shape[0]
    if w.shape[1] < K:
        raise ValueError("layernorm_linear: w has fewer columns than x")
    if out is None:
        ld = (N + 7) // 8 * 8
        out = torch.empty((M, ld), dtype=torch.bfloat16, device=x.device)[:, :N]
    lib = _lib.load()
    rc = lib.evt_layernorm_gemm(x.data_ptr(), x.stride(0), gamma.contiguous().data_ptr(), beta.contiguous().data_ptr(), float(eps),
                                x.data_ptr() if write_back else None, w.data_ptr(), w.stride(0), _ptr(bias), out.data_ptr(),
                                out.stride(0), M, N, K, ACTS[act], _stream())
    _lib.check(rc, "layernorm_gemm")
    return out


def linear_residual_layernorm(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], resid: torch.Tensor,
                              gamma: torch.Tensor, beta: torch.Tensor, eps: float, k: Optional[int] = None,
                              xn: Optional[torch.Tensor] = None, copy_ln: bool = False) -> torch.Tensor:
    """resid[M,N] += a[M,K] @ w[N,K]^T + bias (f32, in place); returns xn = LayerNorm(resid) * gamma + beta (bf16).
    N = 192 / 384 at large M: one kernel, the LayerNorm runs in the GEMM epilogue on rows held in tensor memory; otherwise the
    GEMM and the LayerNorm kernel.  copy_ln (TF dialect): resid ends up holding the normalised rows (f32)."""
    _need_cuda(a, w, bias, resid, gamma, beta, xn)
    if a.dtype != torch.bfloat16 or w.dtype != torch.bfloat16 or resid.dtype != torch.float32:
        raise ValueError("linear_residual_layernorm wants bf16 operands and an f32 residual stream")
    if a.dim() != 2 or w.dim() != 2 or resid.dim() != 2 or a.stride(1) != 1 or w.stride(1) != 1 or resid.stride(1) != 1:
        raise ValueError("linear_residual_layernorm wants 2-D operands with unit inner stride")
    M, N = resid.shape
    K = k if k is not None else a.shape[1]
    if a.shape[0] != M or w.shape[0] != N or a.shape[1] < K or w.shape[1] < K:
        raise ValueError("linear_residual_layernorm: shape mismatch")
    if xn is None:
        xn = torch.empty((M, N), dtype=torch.bfloat16, device=a.device)
    lib = _lib.load()
    rc = lib.evt_gemm_residual_layernorm_ex(a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), _ptr(bias), resid.data_ptr(),
                                            resid.stride(0), gamma.contiguous().data_ptr(), beta.contiguous().data_ptr(),
                                            float(eps), int(copy_ln), xn.data_ptr(), xn.stride(0), M, N, K, _stream())
    _lib.check(rc, "gemm_residual_layernorm")
    return xn


def attention(qkv: torch.Tensor, B: int, S: int, heads: int, head_size: int = 64, scale: Optional[float] = None,
              head_mask: Optional[torch.Tensor] = None, q_rows: Optional[int] = None) -> torch.Tensor:
    """qkv bf16 [B*S, 3*heads*head_size] (q | k | v blocks) -> ctx bf16 [B*S, heads*head_size].  S up to 1026
    (EVT_ATTN_MAX_TOKENS) in bf16, up to 256 for f32 qkv (the tf32 mode).
    q_rows (bf16 only): just the first q_rows queries of every image, against all S keys -> ctx [B*q_rows, heads*head_size]."""
    _need_cuda(qkv, head_mask)
    if qkv.dtype not in (torch.bfloat16, torch.float32) or qkv.dim() != 2 or qkv.stride(1) != 1:
        raise ValueError("attention wants a 2-D bf16 (or f32 for the tf32 mode) qkv matrix")
    if qkv.shape[0] != B * S or qkv.shape[1] < 3 * heads * head_size:
        raise ValueError("attention: qkv shape does not match B, S, heads")
    if q_rows is not None and qkv.dtype != torch.bfloat16:
        raise ValueError("attention: q_rows is implemented for bf16 only")
    Sq = S if q_rows is None else int(q_rows)
    ctx = torch.empty((B * Sq, heads * head_size), dtype=qkv.dtype, device=qkv.device)
    scale = float(head_size ** -0.5 if scale is None else scale)
    lib = _lib.load()
    if q_rows is not None:
        rc = lib.evt_attention_query_rows_fwd(qkv.data_ptr(), qkv.stride(0), ctx.data_ptr(), ctx.stride(0), _ptr(head_mask), B, S,
                                              Sq, heads, head_size, scale, _stream())
    else:
        fn = lib.evt_attention_fwd if qkv.dtype == torch.bfloat16 else lib.evt_attention_fwd_tf32
        rc = fn(qkv.data_ptr(), qkv.stride(0), ctx.data_ptr(), ctx.stride(0), _ptr(head_mask), B, S, heads, head_size, scale,
                _stream())
    _lib.check(rc, "attention")
    return ctx


LOG2E = 1.4426950408889634


def _beit_table(table: torch.Tensor, grid: int) -> torch.Tensor:
    """HF relative_position_bias_table [(2 grid - 1)^2 + 3, heads] -> the library's [heads, n] f32 in log2 units."""
    n = (2 * grid - 1) ** 2 + 3
    if table.dim() != 2 or table.shape[0] != n:
        raise ValueError(f"relative_position_bias_table must be [{n}, heads] for grid {grid}")
    return (table.detach().double().t() * LOG2E).float().contiguous()


def attention_rel_bias(qkv: torch.Tensor, table: torch.Tensor, grid: int, B: int, heads: int, scale: Optional[float] = None,
                       head_mask: Optional[torch.Tensor] = None, q_rows: Optional[int] = None) -> torch.Tensor:
    """BEiT attention (include/evt.h evt_attention_rel_bias_fwd): softmax(q k^T * scale + table[rel(q, k), h]) v for images of
    grid x grid patches behind a cls token (S = grid^2 + 1), head size 64.  qkv bf16 [B*S, 3*heads*64]; table: the HF
    relative_position_bias_table [(2 grid - 1)^2 + 3, heads] (natural-log units; repacked here); q_rows: just the first q_rows
    queries of every image -> ctx bf16 [B*q_rows, heads*64]."""
    _need_cuda(qkv, head_mask)
    S = grid * grid + 1
    if qkv.dtype != torch.bfloat16 or qkv.dim() != 2 or qkv.stride(1) != 1 or qkv.shape[0] != B * S or qkv.shape[1] < 3 * heads * 64:
        raise ValueError("attention_rel_bias wants a bf16 [B*(grid^2+1), >= 3*heads*64] qkv matrix")
    tab = _beit_table(table, grid).to(qkv.device)
    Sq = S if q_rows is None else int(q_rows)
    ctx = torch.empty((B * Sq, heads * 64), dtype=torch.bfloat16, device=qkv.device)
    scale = float(64 ** -0.5 if scale is None else scale)
    _lib.check(_lib.load().evt_attention_rel_bias_fwd(qkv.data_ptr(), qkv.stride(0), ctx.data_ptr(), ctx.stride(0), _ptr(head_mask),
                                                      tab.data_ptr(), grid, B, S, Sq, heads, 64, scale, _stream()), "attention_rel_bias")
    return ctx


def beit_score_bias(table: torch.Tensor, grid: int) -> torch.Tensor:
    """Dense [heads, S, S] form (S = grid^2 + 1) of what evt_attention_rel_bias_fwd adds to the scores, in natural-log units,
    from the kernels' index arithmetic (evt_beit_score_bias).  table: HF layout [(2 grid - 1)^2 + 3, heads].  No GPU."""
    n = (2 * grid - 1) ** 2 + 3
    if table.dim() != 2 or table.shape[0] != n:
        raise ValueError(f"beit_score_bias: table must be [{n}, heads]")
    t = table.detach().float().cpu().t().contiguous()
    S = grid * grid + 1
    out = torch.empty((t.shape[0], S, S), dtype=torch.float32)
    _lib.check(_lib.load().evt_beit_score_bias(t.data_ptr(), t.shape[0], grid, out.data_ptr()), "beit_score_bias")
    return out


def layernorm_patch_mean(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float, images: int, T: int) -> torch.Tensor:
    """BEiT's mean-pooled head input: LayerNorm of the mean of rows 1..T-1 of each image, x f32 [images*T, D] -> bf16 [images, D]."""
    _need_cuda(x, gamma, beta)
    if x.dtype != torch.float32 or x.dim() != 2 or not x.is_contiguous() or x.shape[0] != images * T:
        raise ValueError("layernorm_patch_mean wants a contiguous f32 [images*T, D] matrix")
    y = torch.empty((images, x.shape[1]), dtype=torch.bfloat16, device=x.device)
    _lib.check(_lib.load().evt_layernorm_patch_mean(x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), y.data_ptr(), images, T, x.shape[1],
                                                    float(eps), _stream()), "layernorm_patch_mean")
    return y


def gather_layernorm(x: torch.Tensor, idx: torch.Tensor, gamma: Optional[torch.Tensor], beta: Optional[torch.Tensor], eps: float,
                     images: int, T_in: int, T_out: int, G: int = 1, out_dtype: Optional[torch.dtype] = torch.bfloat16,
                     copy: bool = False):
    """Row gather fused with LayerNorm (Swin window partition / shift / patch merging, include/evt.h).
    x f32 [images*T_in, C]; idx int32 [T_out*G] -> (LN output [images*T_out, G*C] (out_dtype bf16, f32 or TF32) or None, raw
    gathered f32 copy or None)."""
    _need_cuda(x, idx, gamma, beta)
    if x.dtype != torch.float32 or x.dim() != 2 or not x.is_contiguous() or x.shape[0] != images * T_in:
        raise ValueError("gather_layernorm wants a contiguous f32 [images*T_in, C] matrix")
    if idx.dtype != torch.int32 or idx.numel() != T_out * G or not idx.is_contiguous():
        raise ValueError("gather_layernorm: idx must be a contiguous int32 [T_out*G] tensor")
    C = x.shape[1]
    y = torch.empty((images * T_out, G * C), dtype=_storage(out_dtype), device=x.device) if out_dtype is not None else None
    cp = torch.empty((images * T_out, G * C), dtype=torch.float32, device=x.device) if copy else None
    lib = _lib.load()
    _lib.check(lib.evt_gather_layernorm(x.data_ptr(), idx.data_ptr(), _ptr(gamma), _ptr(beta), _ptr(y),
                                        _dt(y, out_dtype) if y is not None else EVT_BF16, _ptr(cp), images, T_in, T_out, G, C, float(eps),
                                        _stream()), "gather_layernorm")
    return y, cp


def window_table_shape(window_tokens: int):
    """(rows, key columns) of one head's bias + mask table in evt_window_attention_fwd: 7 x 7 windows pad 49 to 64 x 56
    (columns 49..55 -inf), 12 x 12 windows use 144 x 144 as is."""
    return (64, 56) if window_tokens == 49 else (window_tokens, window_tokens)


def window_attention(qkv: torch.Tensor, table: torch.Tensor, n_windows: int, heads: int, window_tokens: int = 49,
                     head_size: int = 32, scale: Optional[float] = None) -> torch.Tensor:
    """qkv bf16 [n_windows*N, 3*heads*32] in window order (N = window_tokens, 49 or 144), table f32
    [n_tab, heads, *window_table_shape(N)] (log2 domain, include/evt.h) -> ctx bf16 [n_windows*N, heads*32].
    f32 qkv (tf32-representable values, e.g. from a TF32 linear) runs the tf32 kernel -> ctx f32, rounded to tf32."""
    _need_cuda(qkv, table)
    if qkv.dtype not in (torch.bfloat16, torch.float32) or qkv.dim() != 2 or qkv.stride(1) != 1 or qkv.shape[0] != n_windows * window_tokens:
        raise ValueError("window_attention wants a bf16 (or f32 for the tf32 mode) [n_windows*tokens, 3*heads*head_size] matrix")
    want = (heads, *window_table_shape(window_tokens))
    if table.dtype != torch.float32 or table.dim() != 4 or tuple(table.shape[1:]) != want or not table.is_contiguous():
        raise ValueError(f"window_attention: table must be a contiguous f32 [n_tab, {want[0]}, {want[1]}, {want[2]}] tensor")
    ctx = torch.empty((qkv.shape[0], heads * head_size), dtype=qkv.dtype, device=qkv.device)
    scale = float(head_size ** -0.5 if scale is None else scale)
    lib = _lib.load()
    fn = lib.evt_window_attention_fwd if qkv.dtype == torch.bfloat16 else lib.evt_window_attention_fwd_tf32
    _lib.check(fn(qkv.data_ptr(), qkv.stride(0), ctx.data_ptr(), ctx.stride(0), table.data_ptr(),
                                            table.shape[0], n_windows, window_tokens, heads, head_size, scale, _stream()),
               "window_attention")
    return ctx


def layernorm_mean_tokens(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float, images: int, T: int,
                          out_dtype=torch.bfloat16) -> torch.Tensor:
    """mean over tokens of LayerNorm(x): x f32 [images*T, D] -> [images, D] bf16 or TF32 (Swin final norm + pooler)."""
    _need_cuda(x, gamma, beta)
    if x.dtype != torch.float32 or x.dim() != 2 or not x.is_contiguous() or x.shape[0] != images * T:
        raise ValueError("layernorm_mean_tokens wants a contiguous f32 [images*T, D] matrix")
    if out_dtype not in (torch.bfloat16, TF32):
        raise ValueError("layernorm_mean_tokens: out_dtype must be bf16 or TF32")
    y = torch.empty((images, x.shape[1]), dtype=_storage(out_dtype), device=x.device)
    lib = _lib.load()
    _lib.check(lib.evt_layernorm_mean_tokens_ex(x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), y.data_ptr(), _dt(y, out_dtype), images,
                                                T, x.shape[1], float(eps), _stream()), "layernorm_mean_tokens")
    return y


def cosine_window_attention(qkv: torch.Tensor, table: torch.Tensor, head_scale: torch.Tensor, n_windows: int, heads: int,
                            window: int, grid: int, shift: int = 0, mask: float = -100.0) -> torch.Tensor:
    """Swin V2 cosine window attention (include/evt.h evt_cosine_window_attention_fwd): qkv bf16 [n_windows*window^2, 3*heads*32]
    in window order, table f32 [heads, (2*window-1)^2] = 16 sigmoid(cpb) * log2(e), head_scale f32 [heads] =
    exp(min(logit_scale, ln 100)) * log2(e); grid = tokens per image side, shift = the block's cyclic shift (0: no mask), mask =
    what a masked score gets added -> ctx bf16 [n_windows*window^2, heads*32]."""
    _need_cuda(qkv, table, head_scale)
    N = window * window
    if qkv.dtype != torch.bfloat16 or qkv.dim() != 2 or qkv.stride(1) != 1 or qkv.shape[0] != n_windows * N:
        raise ValueError("cosine_window_attention wants a bf16 [n_windows*window^2, 3*heads*32] matrix")
    nt = (2 * window - 1) ** 2
    if table.dtype != torch.float32 or tuple(table.shape) != (heads, nt) or not table.is_contiguous():
        raise ValueError(f"cosine_window_attention: table must be a contiguous f32 [{heads}, {nt}] tensor")
    if head_scale.dtype != torch.float32 or head_scale.numel() != heads or not head_scale.is_contiguous():
        raise ValueError(f"cosine_window_attention: head_scale must be a contiguous f32 [{heads}] tensor")
    ctx = torch.empty((qkv.shape[0], heads * 32), dtype=torch.bfloat16, device=qkv.device)
    lib = _lib.load()
    _lib.check(lib.evt_cosine_window_attention_fwd(qkv.data_ptr(), qkv.stride(0), ctx.data_ptr(), ctx.stride(0), table.data_ptr(),
                                                   head_scale.data_ptr(), n_windows, window, heads, 32, grid, shift, float(mask),
                                                   _stream()), "cosine_window_attention")
    return ctx


def postnorm_residual(y: torch.Tensor, resid: Optional[torch.Tensor], idx: Optional[torch.Tensor], gamma: torch.Tensor,
                      beta: torch.Tensor, eps: float, images: int, T_out: int, G: int = 1, f32: bool = True, bf16: bool = True):
    """Post-norm residual update (include/evt.h evt_postnorm_residual): row r, group g of the output =
    (resid[s] if resid is given else 0) + LayerNorm(y[s]), s = image * T_in + (idx[t * G + g] if idx is given else t).
    y / resid f32 [images*T_in, C] -> (f32 [images*T_out, G*C] or None, bf16 [images*T_out, G*C] or None)."""
    _need_cuda(y, resid, idx, gamma, beta)
    if y.dtype != torch.float32 or y.dim() != 2 or not y.is_contiguous() or y.shape[0] % images:
        raise ValueError("postnorm_residual wants a contiguous f32 [images*T_in, C] matrix")
    if resid is not None and (resid.dtype != torch.float32 or resid.shape != y.shape or not resid.is_contiguous()):
        raise ValueError("postnorm_residual: resid must be a contiguous f32 tensor shaped like y")
    if idx is not None and (idx.dtype != torch.int32 or idx.numel() != T_out * G or not idx.is_contiguous()):
        raise ValueError("postnorm_residual: idx must be a contiguous int32 [T_out*G] tensor")
    T_in, C = y.shape[0] // images, y.shape[1]
    o32 = torch.empty((images * T_out, G * C), dtype=torch.float32, device=y.device) if f32 else None
    o16 = torch.empty((images * T_out, G * C), dtype=torch.bfloat16, device=y.device) if bf16 else None
    lib = _lib.load()
    _lib.check(lib.evt_postnorm_residual(y.data_ptr(), _ptr(resid), _ptr(idx), gamma.data_ptr(), beta.data_ptr(), _ptr(o32), _ptr(o16),
                                         images, T_in, T_out, G, C, float(eps), _stream()), "postnorm_residual")
    return o32, o16


def swinv2_cpb_table(w1: torch.Tensor, b1: torch.Tensor, w2: torch.Tensor, window: int, pretrained_window: int = 0) -> torch.Tensor:
    """16 sigmoid(cpb_mlp(relative_coords_table)) as the Swin V2 load computes it on the host: CPU f32 [heads, (2*window-1)^2]
    from continuous_position_bias_mlp.{0.weight [512, 2], 0.bias [512], 2.weight [heads, 512]}.  Needs no GPU."""
    w1, b1, w2 = (t.detach().float().cpu().contiguous() for t in (w1, b1, w2))
    if tuple(w1.shape) != (512, 2) or tuple(b1.shape) != (512,) or w2.dim() != 2 or w2.shape[1] != 512:
        raise ValueError("swinv2_cpb_table wants w1 [512, 2], b1 [512], w2 [heads, 512]")
    out = torch.empty((w2.shape[0], (2 * window - 1) ** 2), dtype=torch.float32)
    _lib.check(_lib.load().evt_swinv2_cpb_table(w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), w2.shape[0], window, pretrained_window,
                                                out.data_ptr()), "swinv2_cpb_table")
    return out


def swinv2_score_bias(table: torch.Tensor, window: int, grid: int, shift: int, mask: float = -100.0) -> torch.Tensor:
    """Dense [(grid/window)^2, heads, N, N] form of what evt_cosine_window_attention_fwd adds to the scores (bias from the compact
    CPU f32 table [heads, (2*window-1)^2], plus `mask` between shift regions), from the kernel's index arithmetic.  No GPU."""
    table = table.detach().float().cpu().contiguous()
    heads, N = table.shape[0], window * window
    if table.dim() != 2 or table.shape[1] != (2 * window - 1) ** 2:
        raise ValueError("swinv2_score_bias: table must be [heads, (2*window-1)^2]")
    out = torch.empty(((grid // window) ** 2, heads, N, N), dtype=torch.float32)
    _lib.check(_lib.load().evt_swinv2_score_bias(table.data_ptr(), heads, window, grid, shift, float(mask), out.data_ptr()),
               "swinv2_score_bias")
    return out


def im2col_patch(pixels: torch.Tensor, patch: int = 16, out_dtype=torch.bfloat16) -> torch.Tensor:
    """f32 NCHW pixels -> the patch matrix [B*(H/P)*(W/P), 3*P*P] in (c, i, j) order, bf16 or TF32."""
    _need_cuda(pixels)
    if out_dtype not in (torch.bfloat16, TF32):
        raise ValueError("im2col_patch: out_dtype must be bf16 or TF32")
    if pixels.dtype != torch.float32 or pixels.dim() != 4 or pixels.shape[1] != 3:
        raise ValueError("im2col_patch wants f32 NCHW pixels with 3 channels")
    pixels = pixels.contiguous()
    B, _, H, W = pixels.shape
    cols = torch.empty((B * (H // patch) * (W // patch), 3 * patch * patch), dtype=_storage(out_dtype), device=pixels.device)
    lib = _lib.load()
    _lib.check(lib.evt_im2col_patch_ex(pixels.data_ptr(), cols.data_ptr(), _dt(cols, out_dtype), B, H, W, patch, _stream()), "im2col")
    return cols


def patch_embed(pixels: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, prefix: torch.Tensor, pos: torch.Tensor,
                patch: int = 16, mean=None, std=None) -> torch.Tensor:
    """`ViTEmbeddings.forward` (SITE/models/vit/modeling_vit.py:95-126) as one library call: NCHW pixels (f32, bf16, or raw
    uint8 with per-channel `mean` / `std` of the reference's `Normalize`, deit_pruning/src/utils.py:105-107) ->
    f32 [B, tokens, D].  weight: the conv kernel [D, 3, P, P] (or [D, 3*P*P]); prefix: [n_prefix, D] cls (+ distillation)
    token rows; pos: [tokens, D]."""
    import ctypes as C
    _need_cuda(pixels, weight, bias, prefix, pos)
    if pixels.dim() != 4 or pixels.shape[1] != 3:
        raise ValueError("patch_embed wants NCHW pixels with 3 channels")
    pix = {torch.float32: _lib.PIX_F32, torch.bfloat16: _lib.PIX_BF16, torch.uint8: _lib.PIX_U8}.get(pixels.dtype)
    if pix is None:
        raise ValueError("patch_embed: pixels must be f32, bf16 or uint8")
    pixels = pixels.contiguous()
    B, _, H, W = pixels.shape
    D = weight.shape[0]
    K = 3 * patch * patch
    w = weight.reshape(D, -1)
    if w.shape[1] != K:
        raise ValueError(f"patch_embed: weight has {w.shape[1]} inputs per filter, expected {K}")
    w = w.to(torch.bfloat16)
    if patch == 14:   # the library's P = 14 patch rows are 592 wide: 588 columns and 4 zero ones
        w = torch.nn.functional.pad(w, (0, 592 - K))
    w = w.contiguous()
    prefix = prefix.reshape(-1, D).float().contiguous()
    tokens = prefix.shape[0] + (H // patch) * (W // patch)
    pos = pos.reshape(-1, D).float().contiguous()
    if pos.shape[0] != tokens:
        raise ValueError(f"patch_embed: {pos.shape[0]} position rows for {tokens} tokens")
    scale = shift = None
    if pix == _lib.PIX_U8:
        if mean is None or std is None:
            raise ValueError("patch_embed: uint8 pixels need mean and std")
        scale = (C.c_float * 3)(*[1.0 / (255.0 * float(s_)) for s_ in std])
        shift = (C.c_float * 3)(*[-float(m_) / float(s_) for m_, s_ in zip(mean, std)])
    lib = _lib.load()
    n = C.c_size_t()
    _lib.check(lib.evt_patch_embed_workspace_bytes(B, H, W, patch, prefix.shape[0], C.byref(n)), "patch_embed_workspace_bytes")
    ws = torch.empty(n.value + 1024, dtype=torch.uint8, device=pixels.device)
    ws_ptr = (ws.data_ptr() + 1023) // 1024 * 1024
    out = torch.empty((B, tokens, D), dtype=torch.float32, device=pixels.device)
    _lib.check(lib.evt_patch_embed_fwd(pixels.data_ptr(), pix, scale, shift, w.data_ptr(), w.shape[1], bias.float().contiguous().data_ptr(),
                                       prefix.data_ptr(), pos.data_ptr(), out.data_ptr(), ws_ptr, B, H, W, patch, D,
                                       prefix.shape[0], _stream()), "patch_embed")
    return out


def cast_bf16(x: torch.Tensor) -> torch.Tensor:
    _need_cuda(x)
    x = x.contiguous()
    if x.dtype != torch.float32:
        raise ValueError("cast_bf16 wants f32")
    y = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    lib = _lib.load()
    _lib.check(lib.evt_cast_f32_bf16(x.data_ptr(), y.data_ptr(), x.numel(), _stream()), "cast")
    return y


def unfold_nhwc(x: torch.Tensor, k: int, s: int, p: int, ld: Optional[int] = None) -> torch.Tensor:
    """tf_Unfold (channel-last): x [B,H,W,C] f32|bf16 -> bf16 [B*oh*ow, ld] (ld >= k*k*C, zero padded)."""
    _need_cuda(x)
    x = x.contiguous()
    B, H, W, Cc = x.shape
    oh, ow = (H + 2 * p - k) // s + 1, (W + 2 * p - k) // s + 1
    ld = ld or (k * k * Cc + 7) // 8 * 8
    out = torch.empty((B * oh * ow, ld), dtype=torch.bfloat16, device=x.device)
    lib = _lib.load()
    _lib.check(lib.evt_unfold_nhwc(x.data_ptr(), _dt(x), out.data_ptr(), ld, B, H, W, Cc, k, s, p, _stream()), "unfold")
    return out


def unfold_ln_nhwc(x: torch.Tensor, k: int, s: int, p: int, gamma: Optional[torch.Tensor] = None,
                   beta: Optional[torch.Tensor] = None, eps: float = 1e-5, ld: Optional[int] = None) -> torch.Tensor:
    """tf_Unfold fused with the LayerNorm over each unfolded row (gamma/beta None -> plain unfold)."""
    _need_cuda(x, gamma, beta)
    x = x.contiguous()
    B, H, W, Cc = x.shape
    oh, ow = (H + 2 * p - k) // s + 1, (W + 2 * p - k) // s + 1
    ld = ld or (k * k * Cc + 7) // 8 * 8
    out = torch.empty((B * oh * ow, ld), dtype=torch.bfloat16, device=x.device)
    lib = _lib.load()
    _lib.check(lib.evt_unfold_ln_nhwc(x.data_ptr(), _dt(x), out.data_ptr(), ld, _ptr(gamma), _ptr(beta), float(eps), B, H, W,
                                      Cc, k, s, p, _stream()), "unfold_ln")
    return out


def performer(kqv: torch.Tensor, w: torch.Tensor, B: int, T: int, eps: float = 1e-8):
    """TokenPerformer.single_attn core: kqv bf16 [B*T, >=192] (k|q|v) -> (yattn bf16 [B*T,64], v f32 [B*T,64])."""
    _need_cuda(kqv, w)
    if kqv.dtype != torch.bfloat16 or kqv.dim() != 2 or kqv.shape[0] != B * T or kqv.stride(1) != 1:
        raise ValueError("performer wants a bf16 [B*T, 192] kqv matrix")
    if tuple(w.shape) != (32, 64) or w.dtype != torch.float32:
        raise ValueError("performer: w must be f32 [32, 64]")
    import ctypes as C
    lib = _lib.load()
    n = C.c_size_t()
    _lib.check(lib.evt_performer_workspace_bytes(B, T, C.byref(n)), "performer_workspace_bytes")
    ws = torch.empty(n.value, dtype=torch.uint8, device=kqv.device)
    yattn = torch.empty((B * T, 64), dtype=torch.bfloat16, device=kqv.device)
    vout = torch.empty((B * T, 64), dtype=torch.float32, device=kqv.device)
    _lib.check(lib.evt_performer_fwd(kqv.data_ptr(), kqv.stride(0), w.contiguous().data_ptr(), yattn.data_ptr(),
                                     vout.data_ptr(), ws.data_ptr(), B, T, 64, 32, float(eps), _stream()), "performer")
    return yattn, vout


def performer_mlp(yattn: torch.Tensor, y: torch.Tensor, wo, bo, gamma, beta, w1, b1, w2, b2, eps: float) -> torch.Tensor:
    """In place on y (f32 [rows, 64], holding v): y += attn_output(yattn); y += fc2(gelu_tanh(fc1(LayerNorm(y)))).
    yattn bf16 [rows, 64]; wo / w1 / w2 bf16 [64, 64] ([out, in]); one kernel (csrc/performer.cu)."""
    _need_cuda(yattn, y, wo, bo, gamma, beta, w1, b1, w2, b2)
    if yattn.dtype != torch.bfloat16 or y.dtype != torch.float32 or yattn.shape != y.shape or y.dim() != 2 or y.shape[1] != 64:
        raise ValueError("performer_mlp wants yattn bf16 [rows, 64] and y f32 [rows, 64]")
    if not (yattn.is_contiguous() and y.is_contiguous()):
        raise ValueError("performer_mlp wants contiguous rows")
    for w in (wo, w1, w2):
        if w.dtype != torch.bfloat16 or tuple(w.shape) != (64, 64) or not w.is_contiguous():
            raise ValueError("performer_mlp: weights must be contiguous bf16 [64, 64]")
    lib = _lib.load()
    _lib.check(lib.evt_performer_mlp_fwd(yattn.data_ptr(), y.data_ptr(), wo.data_ptr(), _ptr(bo), gamma.contiguous().data_ptr(),
                                         beta.contiguous().data_ptr(), w1.data_ptr(), _ptr(b1), w2.data_ptr(), _ptr(b2),
                                         y.shape[0], float(eps), _stream()), "performer_mlp")
    return y


def performer_block(kqv: torch.Tensor, w: torch.Tensor, B: int, T: int, wo, bo, gamma, beta, w1, b1, w2, b2, ln_eps: float,
                    eps: float = 1e-8) -> torch.Tensor:
    """performer() followed by performer_mlp() in three launches (the apply kernel carries each tile through the tail):
    kqv bf16 [B*T, >=192] -> y f32 [B*T, 64].  Bit-identical to the two calls."""
    _need_cuda(kqv, w, wo, bo, gamma, beta, w1, b1, w2, b2)
    if kqv.dtype != torch.bfloat16 or kqv.dim() != 2 or kqv.shape[0] != B * T or kqv.stride(1) != 1:
        raise ValueError("performer_block wants a bf16 [B*T, 192] kqv matrix")
    if tuple(w.shape) != (32, 64) or w.dtype != torch.float32:
        raise ValueError("performer_block: w must be f32 [32, 64]")
    for m in (wo, w1, w2):
        if m.dtype != torch.bfloat16 or tuple(m.shape) != (64, 64) or not m.is_contiguous():
            raise ValueError("performer_block: weights must be contiguous bf16 [64, 64]")
    import ctypes as C
    lib = _lib.load()
    n = C.c_size_t()
    _lib.check(lib.evt_performer_workspace_bytes(B, T, C.byref(n)), "performer_workspace_bytes")
    ws = torch.empty(n.value, dtype=torch.uint8, device=kqv.device)
    y = torch.empty((B * T, 64), dtype=torch.float32, device=kqv.device)
    _lib.check(lib.evt_performer_block_fwd(kqv.data_ptr(), kqv.stride(0), w.contiguous().data_ptr(), y.data_ptr(), ws.data_ptr(), B, T,
                                           float(eps), wo.data_ptr(), _ptr(bo), gamma.contiguous().data_ptr(), beta.contiguous().data_ptr(),
                                           w1.data_ptr(), _ptr(b1), w2.data_ptr(), _ptr(b2), float(ln_eps), _stream()), "performer_block")
    return y


def token_transformer_block(qkv: torch.Tensor, B: int, T: int, scale: float, wo, bo, gamma, beta, w1, b1, w2, b2,
                            ln_eps: float) -> torch.Tensor:
    """T2T-ViT ``Token_transformer`` after its qkv projection, in two launches: ctx = softmax(q k^T * scale) v over all T tokens
    of an image (one head of 64, any T), y = v + proj(ctx); y += fc2(gelu_erf(fc1(LayerNorm(y)))).
    qkv bf16 [B*T, >=192] (q | k | v) -> y f32 [B*T, 64]."""
    _need_cuda(qkv, wo, bo, gamma, beta, w1, b1, w2, b2)
    if qkv.dtype != torch.bfloat16 or qkv.dim() != 2 or qkv.shape[0] != B * T or qkv.stride(1) != 1:
        raise ValueError("token_transformer_block wants a bf16 [B*T, 192] qkv matrix")
    for m in (wo, w1, w2):
        if m.dtype != torch.bfloat16 or tuple(m.shape) != (64, 64) or not m.is_contiguous():
            raise ValueError("token_transformer_block: weights must be contiguous bf16 [64, 64]")
    import ctypes as C
    lib = _lib.load()
    n = C.c_size_t()
    _lib.check(lib.evt_token_transformer_workspace_bytes(B, T, C.byref(n)), "token_transformer_workspace_bytes")
    ws = torch.empty(n.value, dtype=torch.uint8, device=qkv.device)
    y = torch.empty((B * T, 64), dtype=torch.float32, device=qkv.device)
    _lib.check(lib.evt_token_transformer_block_fwd(qkv.data_ptr(), qkv.stride(0), y.data_ptr(), ws.data_ptr(), B, T, float(scale),
                                                   wo.data_ptr(), _ptr(bo), gamma.contiguous().data_ptr(), beta.contiguous().data_ptr(),
                                                   w1.data_ptr(), _ptr(b1), w2.data_ptr(), _ptr(b2), float(ln_eps), _stream()),
               "token_transformer_block")
    return y


def set_gemm_pair_mode(mode: int) -> None:
    """-1 automatic, 0 single-CTA GEMM kernel only, 1 CTA-pair (cta_group::2) kernel whenever applicable."""
    _lib.load().evt_gemm_set_pair_mode(int(mode))


def set_gemm_split_k(enable: bool) -> None:
    """Split K over idle SMs for small-batch residual GEMMs (default on: lower latency, last-bit run-to-run variation)."""
    _lib.load().evt_gemm_set_split_k(1 if enable else 0)


class static_weights:
    """Context manager: the ``w`` operands of the ``linear`` calls inside are weights (never produced by the preceding
    kernel), so the GEMM may request their first tiles ahead of the programmatic dependency wait (evt_gemm_weights_static)."""

    def __enter__(self):
        _lib.load().evt_gemm_weights_static(1)
        return self

    def __exit__(self, *exc):
        _lib.load().evt_gemm_weights_static(-1)
        return False


def launch_count(reset: bool = False) -> int:
    lib = _lib.load()
    n = int(lib.evt_launch_count())
    if reset:
        lib.evt_launch_count_reset()
    return n
