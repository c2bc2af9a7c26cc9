"""The Swin tf32 accuracy mode next to the bf16 mode on one GPU; prints one JSON line.

    python tools/swin_tf32_bench.py [--reps 5] [--preroll-s 2]

* Swin-T (224 px) at batch 1024 in forwards of 256 and Swin-B-384 at batch 256, bf16 and tf32 (random init, the same
  weights), device-resident random inputs, after a power pre-roll as in bench.py.  The two modes alternate, `--reps` times;
  medians are reported.
* Batch-1 p50 latency of forward_graphed in both modes (200 replays each).
* Stock PyTorch: HF SwinForImageClassification in fp32 with torch.backends.cuda.matmul.allow_tf32 = True, the same weights
  and batches.
* The window attention op alone at the stage-1 shapes of one 256-image chunk (Swin-T: 49-token windows, 3 heads; Swin-B-384:
  144-token windows, 4 heads), plain and shifted, bf16 kernel next to the tf32 kernel: time and the bytes read and written.
* Logit max-abs and top-1 agreement of 8 images against the fp32 HF forward (TF32 off), both modes.
The GPU name and power limit are read in the same run.
"""
import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from edgevisiontransformer_b200 import ops  # noqa: E402
from edgevisiontransformer_b200.modeling_swin import B200SwinForImageClassification, attention_table, shift_mask  # noqa: E402
from oracle import vit as ovit  # noqa: E402
from swin384_bench import chunked, event_ms, gpu_info, preroll, random_hf  # noqa: E402

MODELS = {"swin_tiny_224": ("swin_tiny", 224, 7, 1024), "swin_base_384": ("swin_base", 384, 12, 256)}
CHUNK = 256


def set_tf32(on):
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = on, on


def p50_graphed(m, x1, n=200):
    for _ in range(10):
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
    return statistics.median(ts)


def model_rows(reps, preroll_s, g):
    out = {}
    for label, (name, size, window, batch) in MODELS.items():
        hf = random_hf(name, image_size=size, window=window)
        x = torch.randn(batch, 3, size, size, device="cuda", generator=g)
        ms = {p: B200SwinForImageClassification.from_hf(hf, max_batch=CHUNK, precision=p) for p in ("bf16", "tf32")}
        steps = {p: chunked(m, x, CHUNK) for p, m in ms.items()}
        for s in steps.values():
            s()
        preroll(lambda: [s() for s in steps.values()], preroll_s)
        times = {p: [] for p in ms}
        for _ in range(reps):                              # alternate the modes
            for p, s in steps.items():
                times[p].append(event_ms(s, 1))
        r = {"batch": batch, "chunk": CHUNK, "image": size, "window": window}
        for p in ms:
            t = statistics.median(times[p])
            r[p] = {"img_per_s": round(batch / t * 1e3, 1), "ms_per_batch": round(t, 2),
                    "ms_all": [round(v, 2) for v in times[p]],
                    "batch1_graphed_p50_ms": round(p50_graphed(ms[p], x[:1]), 4)}
        r["tf32_over_bf16_time"] = round(r["bf16"]["img_per_s"] / r["tf32"]["img_per_s"], 3)
        # accuracy against the fp32 HF forward (TF32 off)
        set_tf32(False)
        hf = hf.cuda()
        ref = hf(pixel_values=x[:8]).logits.float()
        for p, m in ms.items():
            c = ovit.compare_logits(m(x[:8]).logits, ref)
            r[p]["vs_fp32_hf"] = {"images": 8, "max_abs": float(f"{c['max_abs']:.3g}"), "top1_agree": c["top1_agree"]}
        r["ref_logit_std"] = round(ref.std().item(), 4)
        del ms, steps
        torch.cuda.empty_cache()
        # stock PyTorch fp32 with TF32 matmuls, the same weights and batch
        set_tf32(True)
        tstep = chunked(lambda t: hf(pixel_values=t), x, CHUNK)
        tstep()
        preroll(tstep, preroll_s)
        tt = statistics.median([event_ms(tstep, 1) for _ in range(3)])
        r["torch_fp32_allow_tf32"] = {"img_per_s": round(batch / tt * 1e3, 1), "ms_per_batch": round(tt, 2), "torch": torch.__version__}
        r["tf32_speedup_vs_torch"] = round(r["tf32"]["img_per_s"] / r["torch_fp32_allow_tf32"]["img_per_s"], 3)
        set_tf32(False)
        out[label] = r
        del hf, x
        torch.cuda.empty_cache()
    return out


def window_attention_alone(g):
    res = {}
    for label, N, ws, H, heads in (("swin_tiny_224_stage1", 49, 7, 56, 3), ("swin_base_384_stage1", 144, 12, 96, 4)):
        n_win = CHUNK * (H // ws) ** 2
        C = heads * 32
        q32 = ops.round_tf32(torch.randn(n_win * N, 3 * C, device="cuda", generator=g))
        bias = torch.randn((2 * ws - 1) ** 2, heads, generator=torch.Generator().manual_seed(0))
        rows, cols = ops.window_table_shape(N)
        for kind, mask in (("plain", None), ("shifted", shift_mask(H, H, ws, ws // 2))):
            table = attention_table(bias, heads, ws, mask).cuda()
            r = {"windows": n_win, "tokens": N, "heads": heads, "n_tab": table.shape[0], "table_bytes_distinct": table.numel() * 4}
            for p, qkv in (("bf16", q32.bfloat16()), ("tf32", q32)):
                f = lambda: ops.window_attention(qkv, table, n_win, heads, window_tokens=N)  # noqa: E731
                f()
                preroll(f, 0.5)
                ms = event_ms(f, 50)
                eb = qkv.element_size()
                rd = n_win * N * 3 * C * eb                 # q, k, v
                wr = n_win * N * C * eb                     # ctx
                r[p] = {"ms": round(ms, 4), "bytes_read_qkv": rd, "bytes_written_ctx": wr, "table_bytes_read": n_win * heads * rows * cols * 4,
                        "qkv_ctx_GBps": round((rd + wr) / ms / 1e6, 1),
                        "tflops": round(4.0 * N * N * 32 * n_win * heads / ms / 1e9, 1)}
            r["tf32_over_bf16_time"] = round(r["tf32"]["ms"] / r["bf16"]["ms"], 3)
            res[f"{label}_{kind}"] = r
        del q32
        torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--preroll-s", type=float, default=2.0)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        print("swin_tf32_bench needs a B200 (sm_100a)")
        return 2
    g = torch.Generator(device="cuda").manual_seed(0)
    out = {"gpu": gpu_info(), "models": model_rows(a.reps, a.preroll_s, g), "window_attention": window_attention_alone(g)}
    print(json.dumps(out))
    return 0


if __name__ == "__main__":
    with torch.no_grad():
        sys.exit(main())
