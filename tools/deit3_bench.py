"""DeiT III (deit3_base / deit3_large at 224 px, deit3_huge_patch14 at 224 px) on one GPU in bf16; prints one JSON line.

    python tools/deit3_bench.py [--steps 5] [--preroll-s 2]
    python tools/deit3_bench.py --profile

* img/s of each model (stress-initialised weights from the models_v2 restatement in tests/deit3_ref.py, device-resident random
  inputs): base and large at batch 1024, huge at batch 256, one forward per step, after a power pre-roll as in bench.py.
* Stock PyTorch on the same GPU and weights: the restatement in bf16 with its attention through
  torch.nn.functional.scaled_dot_product_attention, same batch.
* Logit max-abs and top-1 agreement of 8 images against the fp32 restatement on the GPU (TF32 off).
* --profile (a run of its own, tracing slows the host): torch.profiler over one forward of huge at batch 256, kernel time by
  name, and the head-80 attention kernel's time and share of the forward.
The GPU name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import deit3_ref as ref  # noqa: E402
from edgevisiontransformer_b200 import modeling_vit  # noqa: E402
from oracle import vit as ovit  # noqa: E402

MODELS = {"deit3_base_patch16_224": ("base", 1024), "deit3_large_patch16_224": ("large", 1024), "deit3_huge_patch14_224": ("huge", 256)}


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


def sdpa_forward(self, x):
    """ref.Attention.forward with the softmax(q k^T) v of torch's fused SDPA."""
    B, N, C = x.shape
    qkv = self.qkv(x).reshape(B, N, 3, self.num_heads, C // self.num_heads).permute(2, 0, 3, 1, 4)
    o = F.scaled_dot_product_attention(qkv[0], qkv[1], qkv[2], scale=self.scale)
    return self.proj(o.transpose(1, 2).reshape(B, N, C))


def profile(g):
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile as tprof
    m = modeling_vit.deit3_huge_patch14_224(ref.build("huge").state_dict(), max_batch=256)
    x = torch.randn(256, 3, 224, 224, device="cuda", generator=g)
    m(x)
    torch.cuda.synchronize()
    with tprof(activities=[ProfilerActivity.CUDA]) as p:
        m(x)
        torch.cuda.synchronize()
    by_name = {}
    for e in p.events():
        if e.device_type == DeviceType.CUDA:
            by_name[e.name] = by_name.get(e.name, 0) + e.time_range.elapsed_us()
    total = sum(by_name.values())
    att = sum(v for k, v in by_name.items() if "attention_long_kernel" in k)
    top = sorted(by_name.items(), key=lambda kv: -kv[1])[:8]
    # 4 S^2 d per (image, head, layer) over 31 full layers; the last layer's cls-row attention is negligible
    flop = 4.0 * 257 * 257 * 80 * 16 * 256 * 31
    return {"model": "deit3_huge_patch14_224", "batch": 256, "kernel_ms": round(total / 1e3, 2),
            "attention80_ms": round(att / 1e3, 2), "attention80_share": round(att / total, 4),
            "attention80_tflops": round(flop / (att / 1e6) / 1e12, 1),
            "top": [{"kernel": k[:90], "ms": round(v / 1e3, 2), "share": round(v / total, 4)} for k, v in top]}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--preroll-s", type=float, default=2.0)
    ap.add_argument("--profile", action="store_true", help="kernel shares with torch.profiler only (no timing)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        print("deit3_bench needs a B200 (sm_100a)")
        return 2
    g = torch.Generator(device="cuda").manual_seed(0)
    out = {"gpu": gpu_info()}
    if a.profile:
        out["profile"] = profile(g)
        print(json.dumps(out))
        return 0
    out["models"] = {}
    eager = ref.Attention.forward
    for name, (kind, batch) in MODELS.items():
        rm = ref.build(kind)
        m = getattr(modeling_vit, name)(rm.state_dict(), max_batch=batch)
        x = torch.randn(batch, 3, 224, 224, device="cuda", generator=g)
        step = lambda: m(x)  # noqa: E731
        step()
        preroll(step, a.preroll_s)
        ms = event_ms(step, a.steps)
        r = {"batch": batch, "img_per_s": round(batch / ms * 1e3, 1), "ms_per_step": round(ms, 2)}
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = False, False
        rm = rm.cuda()
        xs = x[:8]
        want = rm(xs).float()
        c = ovit.compare_logits(m(xs).logits, want)
        r["vs_fp32"] = {"images": 8, "max_abs": round(c["max_abs"], 5), "top1_agree": c["top1_agree"]}
        del m
        torch.cuda.empty_cache()
        ref.Attention.forward = sdpa_forward
        tm = rm.bfloat16()
        xb = x.bfloat16()
        tstep = lambda: tm(xb)  # noqa: E731
        tstep()
        preroll(tstep, a.preroll_s)
        tms = event_ms(tstep, max(2, a.steps // 2))
        r["torch_bf16_sdpa"] = {"img_per_s": round(batch / tms * 1e3, 1), "ms_per_step": round(tms, 2), "torch": torch.__version__}
        r["speedup_vs_torch"] = round(r["img_per_s"] / r["torch_bf16_sdpa"]["img_per_s"], 3)
        ref.Attention.forward = eager
        out["models"][name] = r
        del tm, rm, xb, x
        torch.cuda.empty_cache()
    print(json.dumps(out))
    return 0


if __name__ == "__main__":
    with torch.no_grad():
        sys.exit(main())
