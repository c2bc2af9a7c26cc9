"""384-pixel DeiT models (577 tokens) and the long-sequence attention kernel on one GPU; prints one JSON line.

    python tools/long_seq_bench.py [--chunk 1024] [--batch 2048] [--steps 5] [--preroll-s 2]

* DeiT-Tiny / -Small / -Base patch16-384, bf16, device-resident random inputs, `--batch` images per step in forwards of
  `--chunk`, after a power pre-roll as in bench.py; per-stage times from evt_model_profile_begin/end over one chunk.
* Stock PyTorch on the same GPU and the same DeiT-Base weights: HF ViTForImageClassification at image_size=384 in bf16
  (cuBLAS + SDPA), same chunks.
* The attention op alone at B = 1024, S = 577, 12 heads against torch.nn.functional.scaled_dot_product_attention (default
  backend selection) on the same bf16 q / k / v; TFLOP/s from 4 S^2 64 heads B.
* Logit max-abs and top-1 agreement of a few images of DeiT-Base-384 against the fp32 HF forward.
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

from edgevisiontransformer_b200 import B200ViTForImageClassification, ops  # noqa: E402
from edgevisiontransformer_b200.benchmark.b200 import _random_hf  # noqa: E402
from oracle import vit as ovit  # noqa: E402


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


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--chunk", type=int, default=1024)
    ap.add_argument("--batch", type=int, default=2048)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--preroll-s", type=float, default=2.0)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        print("long_seq_bench needs a B200 (sm_100a)")
        return 2
    out = {"gpu": gpu_info(), "image": 384, "tokens": 577, "batch": a.batch, "chunk": a.chunk, "models": {}}
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(a.batch, 3, 384, 384, device="cuda", generator=g)
    hf_base = None
    for name in ("deit_tiny", "deit_small", "deit_base"):
        hf = _random_hf(name, image_size=384)
        m = B200ViTForImageClassification.from_hf(hf, max_batch=a.chunk, keep_params=False)
        step = chunked(m, x, a.chunk)
        step()
        preroll(step, a.preroll_s)
        ms = event_ms(step, a.steps)
        m.profile_begin()
        m(x[:a.chunk])
        stages = {k: {"ms": round(v[0], 3), "launches": v[1]} for k, v in m.profile_end().items()}
        out["models"][name] = {"img_per_s": round(a.batch / ms * 1e3, 1), "ms_per_step": round(ms, 2), "stages_one_chunk": stages}
        if name == "deit_base":
            hf_base = hf
            ref = hf.cuda()(pixel_values=x[:8]).logits.float()
            r = ovit.compare_logits(m(x[:8]).logits, ref)
            out["deit_base_vs_fp32_hf"] = {"images": 8, "max_abs": round(r["max_abs"], 5), "top1_agree": r["top1_agree"]}
        del m
        torch.cuda.empty_cache()

    # stock PyTorch: the same DeiT-Base weights, bf16, SDPA
    hf_base.config._attn_implementation = "sdpa"       # the modules share this config
    tm = hf_base.cuda().bfloat16().eval()
    xb = x.bfloat16()
    with torch.no_grad():
        step = chunked(lambda t: tm(pixel_values=t), xb, a.chunk)
        step()
        preroll(step, a.preroll_s)
        ms = event_ms(step, a.steps)
    out["torch_bf16_sdpa_deit_base"] = {"img_per_s": round(a.batch / ms * 1e3, 1), "ms_per_step": round(ms, 2),
                                        "torch": torch.__version__}
    out["deit_base_speedup_vs_torch"] = round(out["models"]["deit_base"]["img_per_s"] / out["torch_bf16_sdpa_deit_base"]["img_per_s"], 3)
    del tm, hf_base, xb
    torch.cuda.empty_cache()

    # attention alone
    B, S, H = 1024, 577, 12
    qkv = torch.randn(B * S, 3 * H * 64, device="cuda", generator=g).bfloat16()
    flop = 4.0 * S * S * 64 * H * B
    q, k, v = qkv.view(B, S, 3, H, 64).permute(2, 0, 3, 1, 4)
    f_evt = lambda: ops.attention(qkv, B, S, H)  # noqa: E731
    f_sdpa = lambda: torch.nn.functional.scaled_dot_product_attention(q, k, v)  # noqa: E731
    res = {}
    for nm, f in (("evt", f_evt), ("sdpa", f_sdpa)):
        f()
        preroll(f, 1.0)
        ms = event_ms(f, 20)
        res[nm] = {"ms": round(ms, 4), "tflops": round(flop / ms / 1e9, 1)}
    ctx = f_evt().view(B, S, H, 64).float()
    ref = f_sdpa().transpose(1, 2).float()
    res["max_abs_vs_sdpa"] = (ctx - ref).abs().max().item()
    res["shape"] = {"B": B, "S": S, "heads": H, "head_size": 64}
    out["attention"] = res
    print(json.dumps(out))
    return 0


if __name__ == "__main__":
    with torch.no_grad():
        sys.exit(main())
