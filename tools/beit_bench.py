"""BEiT (mean-pooled head, per-layer relative position bias) on one GPU in bf16; prints one JSON line.

    python tools/beit_bench.py [--steps 5] [--preroll-s 2] [--models beit_base_224,beit_large_224,...]

* img/s of each model (stress-initialised weights from oracle/beit.py, device-resident random inputs), one forward per step
  after a power pre-roll as in bench.py: base and large at 224 px at batch 1024, large at 384 px at batch 256 and at 512 px
  at batch 64.
* Stock PyTorch on the same GPU and weights: the HF module in bf16 with SDPA attention, same batch.
* Logit max-abs and top-1 agreement of 8 images against the HF module in fp32 on the GPU (TF32 off).
* What the bias costs: the attention kernel alone with and without a table (evt_attention_rel_bias_fwd against
  evt_attention_fwd, same qkv, calls alternating, CUDA events) at the beit-base-224, large-384 and large-512 shapes.
The GPU name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from edgevisiontransformer_b200 import _lib, ops  # noqa: E402
from edgevisiontransformer_b200.modeling_beit import B200BeitForImageClassification  # noqa: E402
from oracle import beit as ob  # noqa: E402
from oracle import vit as ovit  # noqa: E402

MODELS = {"beit_base_224": ("base", 224, 1024), "beit_large_224": ("large", 224, 1024), "beit_large_384": ("large", 384, 256),
          "beit_large_512": ("large", 512, 64)}
ATTN_SHAPES = {"beit_base_224": (14, 12, 1024), "beit_large_384": (24, 16, 256), "beit_large_512": (32, 16, 64)}  # grid, heads, B


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


def bench_model(name, steps, preroll_s):
    kind, image, batch = MODELS[name]
    hf = ob.build_hf_beit(kind, seed=0, image_size=image, attn_implementation="sdpa")
    ours = B200BeitForImageClassification.from_hf(hf, max_batch=batch, keep_params=False)
    x = torch.randn(batch, 3, image, image, device="cuda")
    # accuracy: 8 images against the fp32 HF forward (TF32 off)
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    hf32 = hf.cuda()
    with torch.no_grad():
        want = hf32(pixel_values=x[:8]).logits.float()
    acc = ovit.compare_logits(ours(x[:8]).logits, want)
    stock = hf32.to(torch.bfloat16)
    xb = x.to(torch.bfloat16)

    def run_ours():
        ours(x)

    def run_stock():
        with torch.no_grad():
            stock(pixel_values=xb)

    out = {"batch": batch, "image": image, "accuracy_vs_fp32_8img": acc}
    for label, fn in (("ours", run_ours), ("stock_pytorch_bf16_sdpa", run_stock)):
        fn()
        preroll(fn, preroll_s)
        ms = event_ms(fn, steps)
        out[label] = {"ms_per_batch": round(ms, 3), "img_per_s": round(batch / ms * 1e3, 1)}
    out["speedup_vs_stock"] = round(out["stock_pytorch_bf16_sdpa"]["ms_per_batch"] / out["ours"]["ms_per_batch"], 2)
    del ours, stock, hf, hf32
    torch.cuda.empty_cache()
    return out


def bench_bias_cost(name, reps):
    """Attention kernel alone, with and without the bias table, same qkv, calls alternating."""
    grid, heads, B = ATTN_SHAPES[name]
    S = grid * grid + 1
    lib, st = _lib.load(), torch.cuda.current_stream().cuda_stream
    qkv = (torch.randn(B * S, 3 * heads * 64, device="cuda") * 0.5).bfloat16()
    ctx = torch.empty(B * S, heads * 64, dtype=torch.bfloat16, device="cuda")
    tab = ops._beit_table(torch.randn((2 * grid - 1) ** 2 + 3, heads), grid).cuda()

    def plain():
        _lib.check(lib.evt_attention_fwd(qkv.data_ptr(), qkv.stride(0), ctx.data_ptr(), ctx.stride(0), None, B, S, heads, 64, 0.125, st))

    def biased():
        _lib.check(lib.evt_attention_rel_bias_fwd(qkv.data_ptr(), qkv.stride(0), ctx.data_ptr(), ctx.stride(0), None, tab.data_ptr(),
                                                  grid, B, S, S, heads, 64, 0.125, st))

    for fn in (plain, biased):
        for _ in range(5):
            fn()
    t = {"plain": [], "bias": []}
    for _ in range(reps):
        t["plain"].append(event_ms(plain, 10))
        t["bias"].append(event_ms(biased, 10))
    med = {k: sorted(v)[len(v) // 2] for k, v in t.items()}
    return {"B": B, "S": S, "heads": heads, "plain_ms": round(med["plain"], 4), "bias_ms": round(med["bias"], 4),
            "bias_cost_pct": round(100 * (med["bias"] / med["plain"] - 1), 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--preroll-s", type=float, default=2.0)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--models", default=",".join(MODELS))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        print("tools/beit_bench.py needs a B200: there is no CPU path")
        return 2
    res = {"gpu": gpu_info(), "bias_cost": {n: bench_bias_cost(n, a.reps) for n in ATTN_SHAPES}, "models": {}}
    for n in a.models.split(","):
        res["models"][n] = bench_model(n, a.steps, a.preroll_s)
    print(json.dumps(res))
    return 0


if __name__ == "__main__":
    sys.exit(main())
