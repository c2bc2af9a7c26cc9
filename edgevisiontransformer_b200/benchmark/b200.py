"""``b200_benchmark``: latency / throughput of a model on the B200 backend.

Mirrors the reference's GPU timing convention (utils.py:860-900 ``trt_benchmark`` and tools.py:993-1009
``trt_benchmark_cmd``): device-resident synthetic ``randn`` input, ``warmup_runs`` untimed runs, then ``num_runs`` runs
each bracketed by a stream synchronise and ``timeit.default_timer``; optional ``--topk`` keeps the fastest runs
(benchmark/tensorrt/onnx_trt_test.py:103-105); prints ``Avg latency: X ms, Std: Y ms`` and one JSON line.

    python -m edgevisiontransformer_b200.benchmark --model deit_tiny --batch 1 --precision tf32 --graph
    python -m edgevisiontransformer_b200.benchmark --model deit_base --image-size 384 --batch 256
    python -m edgevisiontransformer_b200.benchmark --model swin_large --image-size 384 --batch 256
    python -m edgevisiontransformer_b200.benchmark --model /path/to/pruned_checkpoint --batch 1024
    python -m edgevisiontransformer_b200.benchmark --model attention --h 768 --a 12 --n 197      (op-level, tools.py:735-758)
"""
from __future__ import annotations

import argparse
import json
import os
import timeit
from typing import Optional, Sequence, Tuple

import numpy as np
import torch

DEIT = {"deit_tiny": (192, 3, 768), "deit_small": (384, 6, 1536), "deit_base": (768, 12, 3072)}
SWIN = {"swin_tiny": (96, [2, 2, 6, 2], [3, 6, 12, 24]), "swin_small": (96, [2, 2, 18, 2], [3, 6, 12, 24]),
        "swin_base": (128, [2, 2, 18, 2], [4, 8, 16, 32]), "swin_large": (192, [2, 2, 18, 2], [6, 12, 24, 48])}
# swin_*_patch4_window7_224 (tools.py:280); --image-size 384 takes the window12_384 geometry (published for base / large;
# tiny / small run the same geometry)
SWIN_WINDOW = {224: 7, 384: 12}
T2T = {"t2t_vit_7": (256, 7, 4, 2.0), "t2t_vit_10": (256, 10, 4, 2.0), "t2t_vit_12": (256, 12, 4, 2.0),
       "t2t_vit_14": (384, 14, 6, 3.0)}


def _random_hf(name: str, seed: int = 0, image_size: int = 224):
    from transformers import ViTConfig, ViTForImageClassification
    d, h, i = DEIT[name]
    torch.manual_seed(seed)
    return ViTForImageClassification(ViTConfig(hidden_size=d, num_hidden_layers=12, num_attention_heads=h, intermediate_size=i,
                                               image_size=image_size, num_labels=1000, attn_implementation="eager")).eval()


def _random_t2t_weights(hidden, depth, heads, mlp_ratio, seed=0):
    """Keras-default random weights in the naming of INTEGRATION.md (no checkpoints offline)."""
    import math
    g = torch.Generator().manual_seed(seed)

    def glorot(i, o):
        lim = math.sqrt(6.0 / (i + o))
        return (torch.rand(i, o, generator=g) * 2 - 1) * lim
    sd = {}
    for name, ind in (("t2t.performer1", 147), ("t2t.performer2", 576)):
        sd[name + ".norm1.gamma"], sd[name + ".norm1.beta"] = torch.ones(ind), torch.zeros(ind)
        sd[name + ".kqv.kernel"], sd[name + ".kqv.bias"] = glorot(ind, 192), torch.zeros(192)
        q, _ = torch.linalg.qr(torch.randn(64, 32, generator=g))
        sd[name + ".w"] = q.t().contiguous() * math.sqrt(32)
        for n in ("attn_output", "mlp.fc1", "mlp.fc2"):
            sd[f"{name}.{n}.kernel"], sd[f"{name}.{n}.bias"] = glorot(64, 64), torch.zeros(64)
        sd[name + ".norm2.gamma"], sd[name + ".norm2.beta"] = torch.ones(64), torch.zeros(64)
    sd["t2t.project.kernel"], sd["t2t.project.bias"] = glorot(576, hidden), torch.zeros(hidden)
    sd["cls_tokens"] = torch.randn(1, 1, hidden, generator=g) * 0.05
    pos = torch.arange(197, dtype=torch.float64)[:, None] / torch.pow(
        torch.tensor(10000.0, dtype=torch.float64), 2 * (torch.arange(hidden) // 2).double() / hidden)[None, :]
    pos[:, 0::2], pos[:, 1::2] = torch.sin(pos[:, 0::2]), torch.cos(pos[:, 1::2])
    sd["pos_embedding"] = pos.float()
    inter = int(mlp_ratio * hidden)
    a = hidden
    for l in range(depth):
        p = f"layers.{l}"
        sd[p + ".attn.norm.gamma"], sd[p + ".attn.norm.beta"] = torch.ones(hidden), torch.zeros(hidden)
        sd[p + ".attn.to_qkv.kernel"] = glorot(hidden, 3 * a)
        sd[p + ".attn.to_out.kernel"], sd[p + ".attn.to_out.bias"] = glorot(a, hidden), torch.zeros(hidden)
        sd[p + ".ffn.norm.gamma"], sd[p + ".ffn.norm.beta"] = torch.ones(hidden), torch.zeros(hidden)
        sd[p + ".ffn.fc1.kernel"], sd[p + ".ffn.fc1.bias"] = glorot(hidden, inter), torch.zeros(inter)
        sd[p + ".ffn.fc2.kernel"], sd[p + ".ffn.fc2.bias"] = glorot(inter, hidden), torch.zeros(hidden)
    sd["norm.gamma"], sd["norm.beta"] = torch.ones(hidden), torch.zeros(hidden)
    sd["classifier_head.kernel"], sd["classifier_head.bias"] = glorot(hidden, 1000), torch.zeros(1000)
    return sd


def build_model(name: str, precision: str = "bf16", max_batch: int = 512, device="cuda", image_size: int = 224, **op_kw):
    """-> (callable taking one CUDA tensor, input shape without batch, description).  image_size: deit_* and swin_* (224 or
    384: deit_*_patch16_{224,384}, swin_*_patch4_window7_224 / swin_*_patch4_window12_384)."""
    from .. import B200ViTForImageClassification
    if name in DEIT:
        m = B200ViTForImageClassification.from_hf(_random_hf(name, image_size=image_size), device=device, max_batch=max_batch,
                                                  precision=precision, keep_params=False)
        return m, (3, image_size, image_size), f"{name} random-init ({precision}, {image_size} px)"
    if name in T2T:
        from ..modeling_t2t import B200T2TViT
        hidden, depth, heads, ratio = T2T[name]
        m = B200T2TViT(_random_t2t_weights(hidden, depth, heads, ratio), depth=depth, num_heads=heads, device=device,
                       max_batch=min(max_batch, 1024), precision=precision)
        return m, (224, 224, 3), f"{name} random-init ({precision}), NHWC input"
    if name in SWIN:
        from transformers import SwinConfig, SwinForImageClassification
        from ..modeling_swin import B200SwinForImageClassification
        dim, depths, heads = SWIN[name]
        window = SWIN_WINDOW[image_size]
        torch.manual_seed(0)
        hf = SwinForImageClassification(SwinConfig(image_size=image_size, patch_size=4, window_size=window, embed_dim=dim,
                                                   depths=depths, num_heads=heads, num_labels=1000)).eval()
        m = B200SwinForImageClassification.from_hf(hf, device=device, max_batch=min(max_batch, 1024))
        return m, (3, image_size, image_size), f"{name} random-init (bf16, {image_size} px, window {window})"
    if name in ("attention", "ffn"):
        from .. import torch_layers as tl
        h, n = op_kw.get("h", 768), op_kw.get("n", 128)
        if name == "attention":
            m = tl.get_attention(h=h, a=op_kw.get("a", 12), h_k=op_kw.get("h_k"), n=n).to(device).eval()
        else:
            m = tl.get_ffn(h=h, i=op_kw.get("i", 3072), n=n).to(device).eval()
        return m, (n, h), f"torch_layers {name} h={h} n={n}"
    if os.path.isdir(name):
        m = B200ViTForImageClassification.from_pretrained(name, device=device, max_batch=max_batch, precision=precision,
                                                          keep_params=False)
        return m, (3, m.config.image_size, m.config.image_size), f"checkpoint {name} heads={m.config.heads} ffn={m.config.intermediate}"
    raise ValueError(f"unknown model {name!r}")


def b200_benchmark(model, input_shape: Sequence[int], num_runs: int = 50, warmup_runs: int = 20, topk: Optional[int] = None,
                   graph: bool = False, device="cuda") -> Tuple[float, float, np.ndarray]:
    """(avg_ms, std_ms, all run times in ms).  ``graph=True`` replays a captured CUDA graph (latency path)."""
    x = torch.randn(*input_shape, device=device)
    run = model
    if graph and hasattr(model, "forward_graphed"):
        run = model.forward_graphed
    stream = torch.cuda.current_stream()
    with torch.no_grad():
        for _ in range(warmup_runs):
            run(x)
        times = []
        for _ in range(num_runs):
            stream.synchronize()
            t0 = timeit.default_timer()
            run(x)
            stream.synchronize()
            times.append((timeit.default_timer() - t0) * 1e3)
    t = np.sort(np.asarray(times))
    if topk:
        t = t[:topk]
    return float(t.mean()), float(t.std()), np.asarray(times)


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(prog="b200_benchmark", description=__doc__.split("\n")[0])
    ap.add_argument("--model", required=True, help="deit_{tiny,small,base} | swin_{tiny,small,base,large} | t2t_vit_{7,10,12,14} | attention | ffn | checkpoint dir")
    ap.add_argument("--batch", type=int, default=1)
    ap.add_argument("--precision", default="bf16", choices=["bf16", "tf32"])
    ap.add_argument("--num_runs", type=int, default=50)
    ap.add_argument("--warmup_runs", type=int, default=20)
    ap.add_argument("--topk", type=int, default=None)
    ap.add_argument("--graph", action="store_true", help="CUDA-graph replay (small-batch latency path)")
    ap.add_argument("--image-size", type=int, default=224,
                    help="deit_* / swin_* input resolution (384: deit_*_patch16_384, 577 tokens; swin_*_patch4_window12_384)")
    for k, d in (("h", 768), ("a", 12), ("i", 3072), ("n", 128)):
        ap.add_argument(f"--{k}", type=int, default=d)
    ap.add_argument("--h_k", type=int, default=None)
    a = ap.parse_args(argv)
    if not torch.cuda.is_available():
        print("b200_benchmark needs a B200 (sm_100a): the backend has no CPU path")
        return 2
    if a.image_size != 224 and a.model not in DEIT and a.model not in SWIN:
        ap.error("--image-size applies to the deit_* and swin_* models only")
    if a.model in SWIN and a.image_size not in SWIN_WINDOW:
        ap.error("swin_* runs at --image-size 224 (window 7) or 384 (window 12)")
    model, shape, desc = build_model(a.model, a.precision, max_batch=max(a.batch, 1), image_size=a.image_size, h=a.h, a=a.a, i=a.i,
                                     n=a.n, h_k=a.h_k)
    avg, std, times = b200_benchmark(model, (a.batch, *shape), a.num_runs, a.warmup_runs, a.topk, graph=a.graph)
    print(f"{desc}: batch {a.batch}")
    print(f"Avg latency: {avg: .3f} ms, Std: {std: .3f} ms")          # tools.py:1009 format
    p50 = float(np.percentile(times, 50))
    print(json.dumps({"model": a.model, "batch": a.batch, "precision": a.precision, "image_size": a.image_size, "graph": bool(a.graph),
                      "avg_ms": avg, "std_ms": std, "p50_ms": p50, "images_per_sec": a.batch / (avg / 1e3),
                      "num_runs": a.num_runs, "warmup_runs": a.warmup_runs}))
    return 0
