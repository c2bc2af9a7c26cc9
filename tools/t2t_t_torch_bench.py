"""T2T-ViT_t-14 (tokens_type='transformer') on one GPU; prints one JSON line.

    python tools/t2t_t_torch_bench.py [--batch 1024] [--steps 5] [--reps 5] [--preroll-s 3]

* Throughput of T2T-ViT_t-14 (stress-initialised, bf16, device-resident random NCHW f32 and uint8 pixels, `--batch` images in
  one forward), the two pixel types alternated `--reps` times after a power pre-roll; medians.
* The front-end share: EVT_STAGE_EMBED (soft splits, token transformers, project GEMM) over the whole forward, from the model's
  profiling events on one forward of `--batch` images.
* The stage-1 token attention alone (one head of 64 over 3136 tokens, `--batch` images): its kernel time from torch.profiler
  over the op-level token-transformer block (attention_long_kernel), the block's time from CUDA events, the achieved TFLOP/s at
  4 * 3136^2 * 64 = 2.52 GFLOP per image, and F.scaled_dot_product_attention on the same q / k / v (contiguous copies) timed
  the same two ways.
* Stock PyTorch bf16 of the nn.Module restatement (tests/t2t_t_torch_ref.py) with F.scaled_dot_product_attention in both token
  transformers and in the encoder blocks, same images, same chunk: the baseline.  (Eager attention would materialise a 20 GB
  bf16 score tensor per 1024-image chunk at stage 1.)
The GPU name and power limit are read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
import types

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import t2t_t_torch_ref as tref  # noqa: E402
import t2t_torch_ref as ref  # noqa: E402
from edgevisiontransformer_b200 import ops  # noqa: E402
from edgevisiontransformer_b200.modeling_t2t import t2t_vit_t_14  # noqa: E402

T1 = 3136
ATTN_FLOP_PER_IMAGE = 4 * T1 * T1 * 64


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--id=%d" % torch.cuda.current_device(), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    return {"name": torch.cuda.get_device_name(), "nvidia_smi": q}


def event_ms(fn, steps):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def kernel_ms(fn, calls, match):
    """summed device time per call of the CUDA kernels whose name contains one of `match`, from torch.profiler"""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile as tprof
    fn()
    torch.cuda.synchronize()
    with tprof(activities=[ProfilerActivity.CUDA]) as p:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    ms = {}
    for e in p.events():
        if e.device_type == DeviceType.CUDA and any(m in e.name for m in match):
            ms[e.name] = ms.get(e.name, 0.0) + e.time_range.elapsed_us() / 1e3 / calls
    return ms


def _sdpa_token_attention(self, x):
    B, N, _ = x.shape
    q, k, v = self.qkv(x).reshape(B, N, 3, 1, self.in_dim).permute(2, 0, 3, 1, 4)
    ctx = F.scaled_dot_product_attention(q, k, v, scale=self.scale)
    return v.squeeze(1) + self.proj(ctx.transpose(1, 2).reshape(B, N, self.in_dim))


def _sdpa_attention(self, x):
    B, N, C = x.shape
    q, k, v = self.qkv(x).reshape(B, N, 3, self.num_heads, C // self.num_heads).permute(2, 0, 3, 1, 4)
    return self.proj(F.scaled_dot_product_attention(q, k, v, scale=self.scale).transpose(1, 2).reshape(B, N, C))


def stock_sdpa(model):
    for mod in model.modules():
        if isinstance(mod, tref.TokenAttention):
            mod.forward = types.MethodType(_sdpa_token_attention, mod)
        elif isinstance(mod, ref.Attention):
            mod.forward = types.MethodType(_sdpa_attention, mod)
    return model


def token_attention(a):
    B = a.batch
    g = torch.Generator(device="cuda").manual_seed(1)
    qkv = (torch.randn(B * T1, 192, device="cuda", generator=g) * 3).bfloat16()
    w = [(torch.randn(64, 64, device="cuda", generator=g) / 8).bfloat16() for _ in range(3)]
    v = [torch.randn(64, device="cuda", generator=g) * 0.1 for _ in range(5)]
    scale = 147 ** -0.5
    block = lambda: ops.token_transformer_block(qkv, B, T1, scale, w[0], v[0], v[1], v[2], w[1], v[3], w[2], v[4], 1e-5)  # noqa: E731
    q, k, vv = (qkv.view(B, T1, 192)[..., i * 64:(i + 1) * 64].unsqueeze(1).contiguous() for i in range(3))
    sdpa = lambda: F.scaled_dot_product_attention(q, k, vv, scale=scale)  # noqa: E731
    block()
    sdpa()
    block_ms = statistics.median(event_ms(block, a.steps) for _ in range(3))
    sdpa_ms = statistics.median(event_ms(sdpa, a.steps) for _ in range(3))
    ours = kernel_ms(block, a.steps, ("attention_long_kernel",))
    theirs = kernel_ms(sdpa, a.steps, ("",))
    attn_ms, sdpa_kernel_ms = sum(ours.values()), sum(theirs.values())
    flop = ATTN_FLOP_PER_IMAGE * B
    return {"images": B, "gflop_per_image": round(ATTN_FLOP_PER_IMAGE / 1e9, 3),
            "attention_kernel_ms": round(attn_ms, 3), "attention_tflops": round(flop / attn_ms / 1e9, 1),
            "block_ms_events": round(block_ms, 3),
            "sdpa_kernels": {n: round(t, 3) for n, t in theirs.items()}, "sdpa_kernel_ms": round(sdpa_kernel_ms, 3),
            "sdpa_ms_events": round(sdpa_ms, 3), "sdpa_tflops": round(flop / sdpa_kernel_ms / 1e9, 1),
            "sdpa_over_ours_kernel_time": round(sdpa_kernel_ms / attn_ms, 3)}


def throughput(a):
    g = torch.Generator(device="cuda").manual_seed(0)
    m_ref = tref.stress_model("t2t_vit_t_14", seed=0)
    m = t2t_vit_t_14(m_ref.state_dict(), max_batch=a.batch)
    x = torch.randn(a.batch, 3, 224, 224, device="cuda", generator=g)
    u8 = torch.randint(0, 256, (a.batch, 3, 224, 224), device="cuda", dtype=torch.uint8, generator=g)
    runs = {"f32": lambda: m(x), "u8": lambda: m(u8)}
    with torch.no_grad():
        for f in runs.values():
            f()
        t0 = time.perf_counter()
        while time.perf_counter() - t0 < a.preroll_s:
            for f in runs.values():
                f()
            torch.cuda.synchronize()
        rates = {k: [] for k in runs}
        for _ in range(a.reps):                          # alternate the pixel types, one timed window each per repetition
            for k, f in runs.items():
                rates[k].append(a.batch / (event_ms(f, a.steps) / 1e3))
        m.profile_begin()
        m(x)
        stages = m.profile_end()
        total = sum(ms for ms, _ in stages.values())
        out = {"img_per_s": {k: [round(r, 1) for r in v] for k, v in rates.items()},
               "median_img_per_s": {k: round(statistics.median(v), 1) for k, v in rates.items()},
               "embed_ms": round(stages["embed"][0], 3), "forward_ms_profiled": round(total, 3),
               "front_end_share": round(stages["embed"][0] / total, 4)}
        del m
        torch.cuda.empty_cache()
        stock = stock_sdpa(m_ref.cuda().bfloat16())
        xb = x.bfloat16()
        stock(xb)
        stock_rates = [a.batch / (event_ms(lambda: stock(xb), max(1, a.steps // 2)) / 1e3) for _ in range(3)]
    out["pytorch_bf16_sdpa_img_per_s"] = [round(r, 1) for r in stock_rates]
    out["b200_f32_over_pytorch_sdpa"] = round(statistics.median(rates["f32"]) / statistics.median(stock_rates), 2)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--preroll-s", type=float, default=3.0)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("t2t_t_torch_bench needs a B200: the library has no CPU path")
    res = {"gpu": gpu_info(), "batch": a.batch}
    res["token_attention_stage1"] = token_attention(a)
    torch.cuda.empty_cache()
    res.update(throughput(a))
    res["gpu_after"] = gpu_info()
    print(json.dumps(res))


if __name__ == "__main__":
    main()
