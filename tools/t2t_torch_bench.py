"""T2T-ViT-14 from the PyTorch checkpoint layout against the TensorFlow layout on one GPU; prints one JSON line.

    python tools/t2t_torch_bench.py [--batch 1024] [--chunk 1024] [--steps 5] [--reps 5] [--preroll-s 3]
    python tools/t2t_torch_bench.py --profile [--chunk 1024]

* Throughput of T2T-ViT-14 (random init, bf16, device-resident random inputs, `--batch` images per step in forwards of
  `--chunk`): the PyTorch-layout model (`B200T2TViTTorch`, NCHW f32 and uint8 pixels) and the TF-layout model (`B200T2TViT`,
  NHWC f32), alternated `--reps` times after a power pre-roll.
* Stock PyTorch bf16 eager of the nn.Module restatement (tests/t2t_torch_ref.py) on the same GPU, same chunks: the baseline.
* --profile (a run of its own, tracing slows the host): torch.profiler over one chunk of each layout; the time of the stage-1
  soft split kernel (`unfold773_kernel`, NHWC and NCHW instantiations) and of the whole front-end.
The GPU name and power limit are read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import t2t_torch_ref as ref  # noqa: E402
from edgevisiontransformer_b200.modeling_t2t import B200T2TViT, t2t_vit_14  # noqa: E402
from oracle import t2t as ot2t  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--id=%d" % torch.cuda.current_device(), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    return {"name": torch.cuda.get_device_name(), "nvidia_smi": q}


def chunked(model, x, chunk):
    def step():
        for s in range(0, x.shape[0], chunk):
            model(x[s:s + chunk])
    return step


def event_ms(fn, steps):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def build(chunk):
    torch.manual_seed(0)
    pt_ref = ref.stress_init_(ref.t2t_vit("t2t_vit_14"), seed=0)
    pt = t2t_vit_14(pt_ref.state_dict(), max_batch=chunk, keep_params=True)
    tf = B200T2TViT(ot2t.init_t2t_vit(hidden=384, depth=14, num_heads=6, mlp_ratio=3.0, seed=0), depth=14, num_heads=6,
                    max_batch=chunk)
    return pt_ref, pt, tf


def inputs(batch, g):
    x = torch.randn(batch, 3, 224, 224, device="cuda", generator=g)
    u8 = torch.randint(0, 256, (batch, 3, 224, 224), device="cuda", dtype=torch.uint8, generator=g)
    return x, u8, x.permute(0, 2, 3, 1).contiguous()


def throughput(a):
    g = torch.Generator(device="cuda").manual_seed(0)
    pt_ref, pt, tf = build(a.chunk)
    x, u8, x_nhwc = inputs(a.batch, g)
    runs = {"torch_layout_f32": chunked(pt, x, a.chunk), "torch_layout_u8": chunked(pt, u8, a.chunk),
            "tf_layout_f32": chunked(tf, x_nhwc, a.chunk)}
    with torch.no_grad():
        for f in runs.values():
            f()
        t0 = time.perf_counter()
        while time.perf_counter() - t0 < a.preroll_s:
            for f in runs.values():
                f()
            torch.cuda.synchronize()
        rates = {k: [] for k in runs}
        for _ in range(a.reps):                          # alternate the layouts, one timed window each per repetition
            for k, f in runs.items():
                rates[k].append(a.batch / (event_ms(f, a.steps) / 1e3))
        # stock PyTorch bf16 eager of the restatement, same weights and chunks
        eager = pt_ref.cuda().bfloat16()
        xb = x.bfloat16()
        fe = chunked(eager, xb, a.chunk)
        fe()
        eager_rates = [a.batch / (event_ms(fe, max(1, a.steps // 2)) / 1e3) for _ in range(3)]
    med = {k: statistics.median(v) for k, v in rates.items()}
    return {"img_per_s": {k: [round(r, 1) for r in v] for k, v in rates.items()},
            "median_img_per_s": {k: round(v, 1) for k, v in med.items()},
            "torch_f32_over_tf": round(med["torch_layout_f32"] / med["tf_layout_f32"], 4),
            "torch_u8_over_tf": round(med["torch_layout_u8"] / med["tf_layout_f32"], 4),
            "pytorch_bf16_eager_img_per_s": [round(r, 1) for r in eager_rates],
            "b200_torch_f32_over_eager": round(med["torch_layout_f32"] / statistics.median(eager_rates), 2)}


def profile(a):
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile as tprof
    g = torch.Generator(device="cuda").manual_seed(0)
    _, pt, tf = build(a.chunk)
    x, u8, x_nhwc = inputs(a.chunk, g)
    out = {}
    for label, model, inp in (("torch_layout_f32", pt, x), ("torch_layout_u8", pt, u8), ("tf_layout_f32", tf, x_nhwc)):
        with torch.no_grad():
            for _ in range(2):
                model(inp)
            torch.cuda.synchronize()
            with tprof(activities=[ProfilerActivity.CUDA]) as p:
                for _ in range(3):
                    model(inp)
                torch.cuda.synchronize()
        k = {}
        for e in p.events():
            if e.device_type == DeviceType.CUDA:
                k[e.name] = k.get(e.name, 0.0) + e.time_range.elapsed_us() / 1e3 / 3      # ms per forward
        total = sum(k.values())
        split = {n: round(v, 4) for n, v in k.items() if "unfold773" in n}
        front = sum(v for n, v in k.items() if "unfold" in n or "performer" in n)
        out[label] = {"forward_kernel_ms": round(total, 3), "stage1_soft_split_ms": split,
                      "soft_splits_and_performers_ms": round(front, 3)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--chunk", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--preroll-s", type=float, default=3.0)
    ap.add_argument("--profile", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("t2t_torch_bench needs a B200: the library has no CPU path")
    res = {"gpu": gpu_info(), "batch": a.batch, "chunk": a.chunk}
    res.update({"profile": profile(a)} if a.profile else throughput(a))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
