import torch
import torch.nn as nn

from .. import ops
from ._packed import PackedWeights


class Attention(nn.Module):
    """modeling/torch_layers/attention.py:4-48: q/k/v Linear(+bias) -> softmax(q k^T * head_size^-0.5) v -> to_out.

    B200 path: x -> bf16, ONE GEMM on the concatenated [3*h*d, hidden] weight (bias in the epilogue), the fused
    attention kernel (n up to EVT_ATTN_MAX_TOKENS = 1026), then the to_out GEMM (f32 out; an optional residual is added in its epilogue).
    """

    def __init__(self, hidden_size, num_heads, head_size=None):
        if head_size is None:
            if hidden_size % num_heads != 0:
                raise ValueError(f'hidden_size {head_size} must be a multiple of num_heads {num_heads}.')
            self.head_size = hidden_size // num_heads
        else:
            self.head_size = head_size
        super().__init__()
        self.num_heads = num_heads
        self.scale = self.head_size ** -0.5
        self.hidden_size = hidden_size
        a = self.num_heads * self.head_size
        self.to_query = nn.Linear(in_features=hidden_size, out_features=a)
        self.to_key = nn.Linear(in_features=hidden_size, out_features=a)
        self.to_value = nn.Linear(in_features=hidden_size, out_features=a)
        self.to_out = nn.Linear(in_features=a, out_features=hidden_size)
        self._packed = PackedWeights()

    def _weights(self):
        ps = [self.to_query.weight, self.to_key.weight, self.to_value.weight, self.to_query.bias, self.to_key.bias,
              self.to_value.bias, self.to_out.weight, self.to_out.bias]

        def build():
            wqkv = torch.cat([self.to_query.weight, self.to_key.weight, self.to_value.weight], 0).to(torch.bfloat16).contiguous()
            bqkv = torch.cat([self.to_query.bias, self.to_key.bias, self.to_value.bias], 0).float().contiguous()
            return wqkv, bqkv, self.to_out.weight.to(torch.bfloat16).contiguous(), self.to_out.bias.float().contiguous()
        return self._packed.get(ps, build)

    @torch.no_grad()
    def forward(self, x, residual=None):
        if not x.is_cuda:
            raise RuntimeError("edgevisiontransformer_b200.torch_layers.Attention needs CUDA tensors (no CPU fallback)")
        if self.head_size not in (64, 80):
            raise NotImplementedError("the fused attention kernel implements head_size 64 (every DeiT / T2T configuration) and 80 "
                                      "(DeiT III Huge)")
        B, n, h = x.shape
        wqkv, bqkv, wo, bo = self._weights()
        xb = ops.cast_bf16(x.float().reshape(B * n, h))
        qkv = ops.linear(xb, wqkv, bqkv)
        ctx = ops.attention(qkv, B, n, self.num_heads, self.head_size, self.scale)
        res = None if residual is None else residual.float().reshape(B * n, h).contiguous()
        out = ops.linear(ctx, wo, bo, residual=res, out_dtype=torch.float32)
        return out.view(B, n, h)
