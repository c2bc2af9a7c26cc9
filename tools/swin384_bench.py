"""384-pixel Swin models (12 x 12 windows) and the 144-token window attention kernel on one GPU; prints one JSON line.

    python tools/swin384_bench.py [--chunk 256] [--batch 1024] [--steps 5] [--preroll-s 2]
    python tools/swin384_bench.py --profile [--chunk 256]

* Swin-B / Swin-L patch4_window12_384 (random init), bf16, device-resident random inputs, `--batch` images per step in
  forwards of `--chunk`, after a power pre-roll as in bench.py.  The workspace the runtime asks for is reported for the
  chunk and for the whole batch.
* Stock PyTorch on the same GPU and the same weights: HF SwinForImageClassification in bf16, same chunks.
* Logit max-abs and top-1 agreement of a few images against the fp32 HF forward (TF32 off).
* The window attention op alone at the stage-1 shapes of one chunk, plain (n_tab = 1) and shifted (n_tab = windows per
  image), next to the 49-token kernel on the stage-1 shape of the 224-pixel model: time, tensor TFLOP/s from
  4 N^2 32 per (window, head), and the bytes each call reads (q / k / v, table) and writes.
* --profile (a run of its own, tracing slows the host): torch.profiler over one chunk of each model, kernel time by name
  and the window attention's share.
The GPU name and power limit are read in the same run.
"""
import argparse
import ctypes as ct
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from edgevisiontransformer_b200 import ops  # noqa: E402
from edgevisiontransformer_b200.benchmark.b200 import SWIN  # noqa: E402
from edgevisiontransformer_b200.modeling_swin import B200SwinForImageClassification, attention_table, shift_mask  # noqa: E402
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


def random_hf(name, image_size=384, window=12):
    from transformers import SwinConfig, SwinForImageClassification
    dim, depths, heads = SWIN[name]
    torch.manual_seed(0)
    return SwinForImageClassification(SwinConfig(image_size=image_size, patch_size=4, window_size=window, embed_dim=dim,
                                                 depths=depths, num_heads=heads, num_labels=1000)).eval()


def workspace_bytes(m, batch):
    n = ct.c_size_t()
    assert m._lib.evt_swin_workspace_bytes(m._handle, batch, ct.byref(n)) == 0
    return n.value


def window_attention_alone(g):
    """Stage-1 shapes of a 256-image chunk: Swin-B-384 / Swin-L-384 (64 windows of 144 per image) and Swin-B-224 (64 of 49)."""
    res = {}
    for label, N, ws, H, heads in (("swin_base_384_stage1", 144, 12, 96, 4), ("swin_large_384_stage1", 144, 12, 96, 6),
                                   ("swin_base_224_stage1", 49, 7, 56, 4)):
        per_img = (H // ws) ** 2
        n_win = 256 * per_img
        C = heads * 32
        qkv = torch.randn(n_win * N, 3 * C, device="cuda", generator=g).bfloat16()
        bias = torch.randn((2 * ws - 1) ** 2, heads, generator=torch.Generator().manual_seed(0))
        rows, cols = ops.window_table_shape(N)
        for kind, mask in (("plain", None), ("shifted", shift_mask(H, H, ws, ws // 2))):
            table = attention_table(bias, heads, ws, mask).cuda()
            f = lambda: ops.window_attention(qkv, table, n_win, heads, window_tokens=N)  # noqa: E731
            f()
            preroll(f, 0.5)
            ms = event_ms(f, 50)
            items = n_win * heads
            flop = 4.0 * N * N * 32 * items                    # the useful work, not the padded tiles of N = 49
            io_bytes = n_win * N * (3 * C + C) * 2             # q, k, v read, ctx written
            tab_read = items * rows * cols * 4                 # every (window, head) reads its whole table from L2
            res[f"{label}_{kind}"] = {"windows": n_win, "tokens": N, "heads": heads, "n_tab": table.shape[0], "ms": round(ms, 4),
                                      "tflops": round(flop / ms / 1e9, 1), "qkv_ctx_GBps": round(io_bytes / ms / 1e6, 1),
                                      "table_bytes_distinct": table.numel() * 4, "table_read_GBps": round(tab_read / ms / 1e6, 1),
                                      "us_per_1k_tokens": round(ms * 1e3 / (n_win * N / 1e3), 4)}
        del qkv
    return res


def profile(chunk, g):
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile as tprof
    out = {}
    for name in ("swin_base", "swin_large"):
        m = B200SwinForImageClassification.from_hf(random_hf(name), max_batch=chunk)
        x = torch.randn(chunk, 3, 384, 384, device="cuda", generator=g)
        m(x)
        torch.cuda.synchronize()
        with tprof(activities=[ProfilerActivity.CUDA]) as p:
            m(x)
            torch.cuda.synchronize()
        by_name = {}
        for e in p.events():                           # kernels only: the trace has CUDA activities and nothing else
            if e.device_type == DeviceType.CUDA:
                by_name[e.name] = by_name.get(e.name, 0) + e.time_range.elapsed_us()
        total = sum(by_name.values())
        top = sorted(by_name.items(), key=lambda kv: -kv[1])[:8]
        wa = sum(v for k, v in by_name.items() if "window_attention" in k)
        out[name] = {"chunk": chunk, "kernel_ms": round(total / 1e3, 2), "window_attention_ms": round(wa / 1e3, 2),
                     "window_attention_share": round(wa / total, 4),
                     "top": [{"kernel": k[:90], "ms": round(v / 1e3, 2), "share": round(v / total, 4)} for k, v in top]}
        del m
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--chunk", type=int, default=256)
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--preroll-s", type=float, default=2.0)
    ap.add_argument("--profile", action="store_true", help="kernel shares with torch.profiler only (no timing)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        print("swin384_bench needs a B200 (sm_100a)")
        return 2
    g = torch.Generator(device="cuda").manual_seed(0)
    out = {"gpu": gpu_info(), "image": 384, "window": 12}
    if a.profile:
        out["profile"] = profile(a.chunk, g)
        print(json.dumps(out))
        return 0
    out.update({"batch": a.batch, "chunk": a.chunk, "models": {}})
    x = torch.randn(a.batch, 3, 384, 384, device="cuda", generator=g)
    for name in ("swin_base", "swin_large"):
        hf = random_hf(name)
        m = B200SwinForImageClassification.from_hf(hf, max_batch=a.chunk)
        r = {"workspace_GB_chunk": round(workspace_bytes(m, a.chunk) / 1e9, 2),
             "workspace_GB_batch": round(workspace_bytes(m, a.batch) / 1e9, 2)}
        step = chunked(m, x, a.chunk)
        step()
        preroll(step, a.preroll_s)
        ms = event_ms(step, a.steps)
        r.update({"img_per_s": round(a.batch / ms * 1e3, 1), "ms_per_step": round(ms, 2)})
        # accuracy: fp32 HF forward, TF32 off
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = False, False
        hf = hf.cuda()
        xs = x[:8]
        ref = hf(pixel_values=xs).logits.float()
        c = ovit.compare_logits(m(xs).logits, ref)
        r["vs_fp32_hf"] = {"images": 8, "max_abs": round(c["max_abs"], 5), "top1_agree": c["top1_agree"],
                           "ref_logit_std": round(ref.std().item(), 4)}
        del m
        torch.cuda.empty_cache()
        # stock PyTorch: the same weights in bf16
        tm = hf.bfloat16().eval()
        xb = x.bfloat16()
        step = chunked(lambda t: tm(pixel_values=t), xb, a.chunk)
        step()
        preroll(step, a.preroll_s)
        tms = event_ms(step, max(2, a.steps // 2))
        r["torch_bf16"] = {"img_per_s": round(a.batch / tms * 1e3, 1), "ms_per_step": round(tms, 2), "torch": torch.__version__}
        r["speedup_vs_torch"] = round(r["img_per_s"] / r["torch_bf16"]["img_per_s"], 3)
        out["models"][name] = r
        del tm, hf, xb
        torch.cuda.empty_cache()
    out["window_attention"] = window_attention_alone(g)
    print(json.dumps(out))
    return 0


if __name__ == "__main__":
    with torch.no_grad():
        sys.exit(main())
