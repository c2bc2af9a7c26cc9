"""256-pixel Swin V2 models and the cosine window attention kernel on one GPU; prints one JSON line.

    python tools/swinv2_bench.py [--chunk 256] [--batch 1024] [--steps 5] [--preroll-s 2]

* swinv2_tiny_window8, swinv2_tiny_window16, swinv2_base_window16 (random init, HF Swinv2ForImageClassification via from_hf),
  bf16, device-resident random inputs, `--batch` images per step in forwards of `--chunk`, after a power pre-roll.
* Batch-1 p50 of forward_graphed (CUDA-graph replay).
* Stock PyTorch on the same GPU and the same weights: HF Swinv2ForImageClassification in bf16, same chunks.
* Logit max-abs and top-1 agreement of 8 images against the fp32 HF forward (TF32 off).
* The cosine window attention alone at the stage-1 shapes of one chunk (64- and 256-token windows, plain and shifted).
* Kernel time by name over one chunk of each model from torch.profiler (a separate pass after the timed ones).
The GPU name and power limit are read in the same run.
"""
import argparse
import json
import math
import os
import re
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from edgevisiontransformer_b200 import ops  # noqa: E402
from edgevisiontransformer_b200.modeling_swinv2 import B200Swinv2ForImageClassification  # noqa: E402
from oracle import swinv2 as osv2  # noqa: E402
from oracle import vit as ovit  # noqa: E402

MODELS = (("swinv2_tiny_window8", "tiny", 8), ("swinv2_tiny_window16", "tiny", 16), ("swinv2_base_window16", "base", 16))


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


def preroll(fn, seconds):
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        fn()
        torch.cuda.synchronize()


def chunked(model, x, chunk):
    def step():
        for s in range(0, x.shape[0], chunk):
            model(x[s:s + chunk])
    return step


def batch1_p50(m, x1, n=200):
    for _ in range(20):
        m.forward_graphed(x1)
    torch.cuda.synchronize()
    ts = []
    for _ in range(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        m.forward_graphed(x1)
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2]


def attention_alone(g):
    """Stage-1 shapes of a 256-image chunk of swinv2_base: 64 x 64 tokens, 4 heads, windows of 64 and 256 tokens."""
    res = {}
    heads, grid, C = 4, 64, 128
    for window in (8, 16):
        N = window * window
        n_win = 256 * (grid // window) ** 2
        qkv = torch.randn(n_win * N, 3 * C, device="cuda", generator=g).bfloat16()
        tab = torch.rand(heads, (2 * window - 1) ** 2, device="cuda", generator=g) * 16 * math.log2(math.e)
        sc = torch.full((heads,), 10 * math.log2(math.e), device="cuda")
        for kind, shift in (("plain", 0), ("shifted", window // 2)):
            f = lambda: ops.cosine_window_attention(qkv, tab, sc, n_win, heads, window, grid, shift)  # noqa: E731
            f()
            preroll(f, 0.5)
            ms = event_ms(f, 50)
            flop = 4.0 * N * N * 32 * n_win * heads
            io_bytes = n_win * N * 4 * C * 2
            res[f"window{window}_{kind}"] = {"windows": n_win, "tokens": N, "heads": heads, "ms": round(ms, 4),
                                            "tflops": round(flop / ms / 1e9, 1), "qkv_ctx_GBps": round(io_bytes / ms / 1e6, 1)}
        del qkv
    return res


def profile(m, x):
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile as tprof
    m(x)
    torch.cuda.synchronize()
    with tprof(activities=[ProfilerActivity.CUDA]) as p:
        m(x)
        torch.cuda.synchronize()
    by_name = {}
    for e in p.events():
        if e.device_type == DeviceType.CUDA:
            key = re.sub(r"<.*", "", e.name).split("::")[-1].split("(")[0]      # the kernel's own name
            by_name[key] = by_name.get(key, 0) + e.time_range.elapsed_us()
    total = sum(by_name.values())
    return {"kernel_ms": round(total / 1e3, 2),
            "shares": {k: round(v / total, 4) for k, v in sorted(by_name.items(), key=lambda kv: -kv[1])[:8]}}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--chunk", type=int, default=256)
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--preroll-s", type=float, default=2.0)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        print("swinv2_bench needs a B200 (sm_100a)")
        return 2
    g = torch.Generator(device="cuda").manual_seed(0)
    out = {"gpu": gpu_info(), "image": 256, "batch": a.batch, "chunk": a.chunk, "models": {}}
    x = torch.randn(a.batch, 3, 256, 256, device="cuda", generator=g)
    for label, kind, window in MODELS:
        hf = osv2.build_hf_swinv2(kind, seed=0, window=window)
        m = B200Swinv2ForImageClassification.from_hf(hf, max_batch=a.chunk)
        step = chunked(m, x, a.chunk)
        step()
        preroll(step, a.preroll_s)
        ms = event_ms(step, a.steps)
        r = {"img_per_s": round(a.batch / ms * 1e3, 1), "ms_per_step": round(ms, 2),
             "batch1_graphed_p50_ms": round(batch1_p50(m, x[:1].contiguous()), 4)}
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = False, False
        hf = hf.cuda()
        ref = hf(pixel_values=x[:8]).logits.float()
        c = ovit.compare_logits(m(x[:8]).logits, ref)
        r["vs_fp32_hf"] = {"images": 8, "max_abs": round(c["max_abs"], 5), "top1_agree": c["top1_agree"],
                           "ref_logit_std": round(ref.std().item(), 4)}
        r["profile_chunk"] = profile(m, x[:a.chunk])
        del m
        torch.cuda.empty_cache()
        tm = hf.bfloat16().eval()
        xb = x.bfloat16()
        step = chunked(lambda t: tm(pixel_values=t), xb, a.chunk)
        step()
        preroll(step, a.preroll_s)
        tms = event_ms(step, max(2, a.steps // 2))
        r["torch_bf16"] = {"img_per_s": round(a.batch / tms * 1e3, 1), "ms_per_step": round(tms, 2), "torch": torch.__version__}
        r["speedup_vs_torch"] = round(r["img_per_s"] / r["torch_bf16"]["img_per_s"], 3)
        out["models"][label] = r
        del tm, hf, xb
        torch.cuda.empty_cache()
    out["cosine_window_attention"] = attention_alone(g)
    print(json.dumps(out))
    return 0


if __name__ == "__main__":
    with torch.no_grad():
        sys.exit(main())
