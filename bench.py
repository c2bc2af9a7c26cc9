#!/usr/bin/env python
"""Headline benchmark: DeiT-Base patch16-224 bf16 inference forward, images/s, batch-sharded over N B200s.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run)
    python bench.py --impl reference ...                      (the reference's CPU forward on the host cores)
    python bench.py ... --dump-outputs DIR                    (also save the last timed step's logits under DIR)

One "step" = one forward of the hot path over the rank's shard of the global batch (BASELINE.json config 3:
global batch 4096 sharded 4096/2048/1024/512 per GPU; strong scaling, no collective on the data path).
Prints ONE JSON line on rank 0.  See DESIGN.md section "Measurement" for every field.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOADS = {
    # name: (hidden, heads, inter, default global batch)
    "deit_base": (768, 12, 3072, 4096),
    "deit_small": (384, 6, 1536, 256),
    "deit_tiny": (192, 3, 768, 1024),
}
GFLOP_PER_IMG = {"deit_base": 35.128, "deit_small": 9.198, "deit_tiny": 2.507}   # SURVEY.md section 8d


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tf_burst": d["bf16_tflops"], "tf_sustained": d["bf16_tflops_sustained"], "src": "measured"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "src": "fallback"}


def matmul_gflop(hidden, heads, inter, tokens=197, labels=1000, patches=196, patch_k=768):
    """SURVEY.md section 8d: algorithmic matmul FLOPs per image, 2 M N K per GEMM, HF dialect."""
    f = 2.0 * patches * patch_k * hidden
    for h, i in zip(heads, inter):
        a = 64 * h
        f += 3 * 2 * tokens * hidden * a + 2 * 2 * tokens * tokens * a + 2 * tokens * a * hidden + 2 * 2 * tokens * hidden * i
    return (f + 2.0 * hidden * labels) / 1e9


def hbm_mb_per_img(hidden, heads, inter, tokens=197):
    """SURVEY.md section 8d: algorithmic HBM bytes per image (bf16 activations, one pass per op with epilogue fusion,
    LayerNorm separate, weights amortised): per layer 2 S [2D + (D+3a) + (3a+a) + (a+2D) + 2D + (D+i) + (i+2D)]."""
    b = 0.0
    for h, i in zip(heads, inter):
        a, D = 64 * h, hidden
        b += 2.0 * tokens * (2 * D + (D + 3 * a) + (3 * a + a) + (a + 2 * D) + 2 * D + (D + i) + (i + 2 * D))
    return b / 1e6


def traffic_lookup(kernel: str, M: int, N: int, K: int):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of a kernel at a shape, from the committed ncu
    captures indexed in profiles/traffic.json.  No matching capture -> (None, True): the line then says traffic_stale."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        tab = json.load(open(p))
    except Exception:
        return None, True, None
    ent = tab.get(f"{kernel}|M={M},N={N},K={K}")
    if not ent:
        return None, True, None
    return float(ent["dram_read"]) + float(ent["dram_write"]), False, ent.get("source")


def timed_steps(fn, steps, warmup=3):
    """CUDA-event time per call on the current stream after `warmup` untimed calls."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(dirname: str, logits: torch.Tensor, rank: int, world: int) -> str:
    """Save what the timed path returned in its last step (the [per-GPU batch, 1000] f32 logits) as DIR/logits.npy, or
    DIR/logits_rank<r>.npy per rank when sharded.  Above 64 MB in all, every k-th row is kept (a fixed stride, so two runs
    with the same arguments save the same images).  Inputs and weights are seeded: two builds compare output for output."""
    import numpy as np
    a = logits.float().cpu().numpy()
    stride = -(-a.nbytes // (DUMP_LIMIT_BYTES // world))
    os.makedirs(dirname, exist_ok=True)
    path = os.path.join(dirname, "logits.npy" if world == 1 else f"logits_rank{rank}.npy")
    np.save(path, np.ascontiguousarray(a[::stride]))
    return path


def build_hf(workload: str, seed: int = 0):
    """Random-init HF ViTForImageClassification of the named architecture (no checkpoints offline)."""
    from transformers import ViTConfig, ViTForImageClassification
    d, h, i, _ = WORKLOADS[workload]
    cfg = ViTConfig(hidden_size=d, num_hidden_layers=12, num_attention_heads=h, intermediate_size=i, num_labels=1000,
                    image_size=224, patch_size=16, attn_implementation="eager")
    torch.manual_seed(seed)
    return ViTForImageClassification(cfg).eval()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.stop, self.t = index, [], threading.Event(), None

    def _run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.05)

    def __enter__(self):
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.t.join(timeout=6)

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
            except Exception:
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_forward_rate(workload: str, batch: int, budget_s: float, threads: int):
    """images/s of the reference's own forward (HF ViT, fp32, eager attention) on the host cores."""
    torch.set_num_threads(threads)
    model = build_hf(workload)
    x = torch.randn(batch, 3, 224, 224, generator=torch.Generator().manual_seed(1))
    with torch.no_grad():
        model(pixel_values=x)                                   # warm-up
        t0, n = time.perf_counter(), 0
        while True:
            model(pixel_values=x)
            n += 1
            el = time.perf_counter() - t0
            if el > budget_s or n >= 50:
                break
    return batch * n / el, n, el


def run_reference(args):
    """--impl reference: the reference path (HF ViTForImageClassification called as deit_pruning/src/utils.py:194-195
    does) on the host CPU, each step a bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    sample = args.ref_batch
    model = build_hf(args.workload)
    x = torch.randn(sample, 3, 224, 224, generator=torch.Generator().manual_seed(1))
    with torch.no_grad():
        for _ in range(max(1, min(args.warmup, 2))):
            model(pixel_values=x)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            out = model(pixel_values=x).logits
        el = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out, 0, 1)
    ips = sample * args.steps / el
    line = {
        "impl": "reference", "metric": "images_per_sec", "value": ips, "unit": "img/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": el / args.steps * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.workload} patch16-224, HF ViTForImageClassification forward on host CPU",
                   "sample": f"{sample} images per step"},
        "cpu_baseline": {"value": ips, "unit": "img/s", "cores": threads, "kind": "reference",
                         "sample": f"{args.steps} steps x {sample} synthetic images, fp32, eager attention, torch {torch.__version__}"},
        "e2e": {"value": ips, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def pruned_tiny_state_dict(case: str):
    """BASELINE config 4 on random-init DeiT-Tiny weights, built the way the reference's eval does it (eval_main.py:87-103):
    nn_pruning leaves all-zero FC1 rows / FC2 columns and zeroed head blocks in a full-size checkpoint; the product's
    checkpoint surgery (prune_heads_ / drop_zero_ffn_ = HF prune_heads + optimize_model) then yields the small shapes.
      h1_d230        layerwise_thresholds "h_0.50_d_0.3" x 12: 1 head, 230 FFN units per layer (SURVEY.md section 8d)
      head18_uneven  are16heads tiny-18 heads [1,1,1,1,2,1,2,2,2,2,1,2] (draw.py:104-106) with uneven FFN widths"""
    from edgevisiontransformer_b200 import checkpoint as ck
    from edgevisiontransformer_b200.modeling_vit import normalise_keys
    sd = normalise_keys({k: v.detach().clone() for k, v in build_hf("deit_tiny").state_dict().items()})
    if case == "h1_d230":
        heads, inter = [1] * 12, [230] * 12
    else:
        heads, inter = [1, 1, 1, 1, 2, 1, 2, 2, 2, 2, 1, 2], [230, 231, 200, 256, 1, 8, 407, 230, 300, 150, 768, 64]
    g = torch.Generator().manual_seed(7)
    for l in range(12):
        p = f"vit.encoder.layer.{l}."
        drop = torch.randperm(768, generator=g)[: 768 - inter[l]]
        sd[p + "intermediate.dense.weight"][drop] = 0
        sd[p + "intermediate.dense.bias"][drop] = 0
        sd[p + "output.dense.weight"][:, drop] = 0
    ck.prune_heads_(sd, {l: list(range(heads[l], 3)) for l in range(12)}, 64, n_orig=3)
    ck.drop_zero_ffn_(sd)
    return sd, heads, inter


def extra_configs(dev, steps, pk):
    """BASELINE configs 2, 4 and 5 in the same run (device-resident inputs, CUDA events): images/s and the roofline
    fraction SURVEY.md section 8d assigns to each (tensor for Small and T2T, HBM for the pruned Tiny)."""
    from edgevisiontransformer_b200 import B200ViTForImageClassification
    from edgevisiontransformer_b200.benchmark.b200 import _random_t2t_weights
    out = {}

    def run(name, model, x, batch, gflop, hbm_mb=None, note=None):
        ms = timed_steps(lambda: model(x).logits, steps, warmup=3)
        ips = batch / ms * 1e3
        ent = {"batch": batch, "img_per_s": ips, "ms_per_forward": ms, "gflop_per_img": gflop, "model_tflops": ips * gflop / 1e3,
               "frac_tensor_sustained": ips * gflop / 1e3 / pk["tf_sustained"], "steps": steps}
        if hbm_mb is not None:
            ent["hbm_mb_per_img"] = hbm_mb
            ent["hbm_roofline_img_per_s"] = pk["hbm_gbs"] * 1e3 / hbm_mb
            ent["frac_hbm"] = ips / ent["hbm_roofline_img_per_s"]
        if note:
            ent["note"] = note
        out[name] = ent

    m = B200ViTForImageClassification.from_hf(build_hf("deit_small"), device=dev, max_batch=256, keep_params=False)
    x = torch.randn(256, 3, 224, 224, device=dev)
    run("config2_deit_small_bs256", m, x, 256, GFLOP_PER_IMG["deit_small"], hbm_mb_per_img(384, [6] * 12, [1536] * 12))
    del m
    x = torch.randn(1024, 3, 224, 224, device=dev)
    for case in ("h1_d230", "head18_uneven"):
        sd, heads, inter = pruned_tiny_state_dict(case)
        m = B200ViTForImageClassification.from_state_dict(sd, device=dev, max_batch=1024, keep_params=False)
        assert m.config.heads == heads and m.config.intermediate == inter
        run(f"config4_pruned_tiny_{case}_bs1024", m, x, 1024, matmul_gflop(192, heads, inter), hbm_mb_per_img(192, heads, inter),
            note="HBM-bound config: frac_hbm is the roofline fraction")
        del m
    from edgevisiontransformer_b200.modeling_t2t import B200T2TViT
    m = B200T2TViT(_random_t2t_weights(384, 14, 6, 3.0), depth=14, num_heads=6, device=dev, max_batch=1024)
    x = torch.randn(1024, 224, 224, 3, device=dev)
    run("config5_t2t_vit_14_bs1024", m, x, 1024, 9.567, note="NHWC input, one chunk of 1024 (6.4 GB workspace; chunks of 256: -8 %); "
                                                             "9.567 GF/img = front-end 0.598 + encoder 8.969")
    del m, x
    torch.cuda.empty_cache()
    return out


def library_baseline(dev, batch, steps):
    """SURVEY.md section 8d: the reference's own module (HF ViTForImageClassification, DeiT-Base) in bf16 on the SAME GPU
    through stock PyTorch kernels (cuBLAS + SDPA, and eager attention as the reference's pinned transformers runs it)."""
    from transformers import ViTConfig, ViTForImageClassification
    out = {"what": "HF ViTForImageClassification DeiT-Base bf16 on this GPU via stock PyTorch (cuBLAS/cuDNN/ATen)", "batch": batch,
           "torch": torch.__version__}
    x = torch.randn(batch, 3, 224, 224, device=dev, dtype=torch.bfloat16)
    for impl in ("sdpa", "eager"):
        cfg = ViTConfig(hidden_size=768, num_hidden_layers=12, num_attention_heads=12, intermediate_size=3072, num_labels=1000,
                        image_size=224, patch_size=16, attn_implementation=impl)
        torch.manual_seed(0)
        model = ViTForImageClassification(cfg).eval().to(dev).bfloat16()
        with torch.no_grad():
            ms = timed_steps(lambda: model(pixel_values=x).logits, steps, warmup=3)
        out[impl + "_img_per_s"] = batch / ms * 1e3
        del model
        torch.cuda.empty_cache()
    return out


def config1_latency(dev, runs=200):
    """BASELINE config 1 as written: DeiT-Tiny patch16-224, random-init (seed 0), batch 1, the tf32 accuracy mode: p50
    over `runs` CUDA-graph replays, and max-abs error / top-1 agreement against the reference's fp32 forward on the CPU
    (the HF module itself, not the oracle) on the same synthetic image."""
    from edgevisiontransformer_b200 import B200ViTForImageClassification
    hf = build_hf("deit_tiny", seed=0)
    x = torch.randn(1, 3, 224, 224, generator=torch.Generator().manual_seed(1))
    with torch.no_grad():
        want = hf(pixel_values=x).logits
    out = {}
    for prec in ("tf32", "bf16"):
        m = B200ViTForImageClassification.from_hf(hf, device=dev, max_batch=1, precision=prec, keep_params=False)
        xd = x.to(dev)
        for _ in range(30):
            got = m.forward_graphed(xd).logits
        torch.cuda.synchronize()
        ts = []
        for _ in range(runs):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            m.forward_graphed(xd)
            torch.cuda.synchronize()
            ts.append((time.perf_counter() - t0) * 1e3)
        ts.sort()
        out[prec] = {"p50_ms": ts[len(ts) // 2], "p90_ms": ts[int(len(ts) * 0.9)], "runs": runs,
                     "max_abs_vs_reference_fp32": float((got.cpu() - want).abs().max()),
                     "top1_agrees": bool((got.cpu().argmax(-1) == want.argmax(-1)).all())}
        del m
    out["model"] = "deit_tiny patch16-224 random-init seed 0, batch 1, synthetic randn image seed 1"
    out["tolerance"] = {"tf32": 1e-3, "bf16": 2e-2}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="deit_base", choices=sorted(WORKLOADS))
    ap.add_argument("--global-batch", type=int, default=0)
    ap.add_argument("--chunk", type=int, default=1024, help="images per forward call inside a step")
    ap.add_argument("--ref-batch", type=int, default=16)
    ap.add_argument("--preroll-s", type=float, default=2.0, help="seconds of untimed steps before the timed region (sustained clocks)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the other BASELINE configs, the library baseline and config 1")
    ap.add_argument("--dump-outputs", metavar="DIR", help="save the logits of the last timed step as DIR/logits.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        print("bench.py needs a B200: the product has no CPU path (use --impl reference for the CPU baseline)", file=sys.stderr)
        return 2
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = max(world, 1)
    gbatch = args.global_batch or WORKLOADS[args.workload][3]
    per = gbatch // n_gpus
    assert per * n_gpus == gbatch, "global batch must divide by the GPU count"
    chunk = min(args.chunk, per)

    from edgevisiontransformer_b200 import B200ViTForImageClassification, ops
    hf = build_hf(args.workload)
    model = B200ViTForImageClassification.from_hf(hf, device=dev, max_batch=chunk, keep_params=False)
    del hf
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    x = torch.randn(per, 3, 224, 224, device=dev, generator=g)           # resident in HBM, >> L2 (126 MB)

    def step():
        return model(x).logits

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    warm = max(args.warmup, 3)
    for _ in range(warm):
        out = step()
    torch.cuda.synchronize()
    # Power pre-roll: the same step, untimed, for >= preroll_s on every rank, so that the timed steps run at the clocks
    # the GPU SUSTAINS under its power cap.  Without it a short timed region (8 GPUs: 0.4 s) runs at boost clocks and the
    # scaling efficiency reads above 1 (round-1 verdict).
    pre_steps = 0
    t_pre = time.perf_counter()
    while time.perf_counter() - t_pre < args.preroll_s:
        step()
        torch.cuda.synchronize()
        pre_steps += 1

    # ------------------------------------------------------------------ timed region (device-resident inputs)
    barrier()
    ops.launch_count(reset=True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        e0.record()
        for _ in range(args.steps):
            out = step()
        e1.record()
        torch.cuda.synchronize()
    launches = ops.launch_count()
    ms = e0.elapsed_time(e1)
    barrier()
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    value = gbatch / (ms_step / 1e3)
    assert torch.isfinite(out).all()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out, rank, n_gpus)

    # ------------------------------------------------------------------ end to end through the public API, host buffers
    # Headline e2e: f32 pinned pixels (what the reference's loader hands over).  The C ABI also takes bf16 and raw u8
    # pixels (conversion / normalisation fused into the patch gather): 2x / 4x fewer bytes over PCIe, reported beside it.
    from edgevisiontransformer_b200.eval_loop import PipelinedClassifier
    runner = PipelinedClassifier(model, chunk=chunk)

    def e2e_run(host, pipelined=True):
        """K steps through the public host-tensor API.  pipelined: `submit` step i+1 before collecting step i (what an
        evaluation loop does: the next batch's H2D runs under this batch's last forwards); otherwise one synchronous
        `logits()` call per step.  Either way every step's pixels cross PCIe and every step's logits come back inside the
        timed region."""
        for _ in range(2):
            runner.logits(host)
        barrier()
        t0 = time.perf_counter()
        e0.record()
        if pipelined:
            prev = None
            for _ in range(args.steps):
                h = runner.submit(host)          # H2D (pinned, chunked) -> forward -> D2H logits, queued
                if prev is not None:
                    lg = prev.result()
                prev = h
            lg = prev.result()
        else:
            for _ in range(args.steps):
                lg = runner.logits(host)
        e1.record()
        torch.cuda.synchronize()
        el = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)
        tt = torch.tensor([el], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        assert lg.shape == (per, 1000) and not lg.is_cuda
        step_s = float(tt.item()) / args.steps / 1e3
        e2e_run.h2d_gbs = host.numel() * host.element_size() / step_s / 1e9     # per-GPU host -> device rate this implies
        return gbatch / step_s

    # pinned host batches are allocated with the process bound to the GPU's own NUMA node (restored right after: the CPU
    # baseline leg below must see every core)
    from edgevisiontransformer_b200.eval_loop import near_gpu
    with near_gpu(dev) as numa_note:
        host = torch.empty((per, 3, 224, 224), dtype=torch.float32).pin_memory()
    host.copy_(x)
    e2e_pipe = e2e_run(host)
    e2e_h2d_gbs = e2e_run.h2d_gbs
    e2e_sync = e2e_run(host, pipelined=False)
    # Both are the public API; the headline is the better one and says which (one batch queued ahead hides the one copy per step
    # that a synchronous call exposes: N = 8, f32 pixels: 201.6 k against 188.4 k img/s).
    e2e_value, e2e_mode = (e2e_pipe, "pipelined") if e2e_pipe >= e2e_sync else (e2e_sync, "per_call_synchronous")
    if e2e_mode != "pipelined":
        e2e_h2d_gbs = e2e_run.h2d_gbs
    e2e_alt = {}
    with near_gpu(dev):
        hb = torch.empty((per, 3, 224, 224), dtype=torch.bfloat16).pin_memory()
    hb.copy_(x)
    del host
    e2e_alt["bf16_pixels"] = {"value": e2e_run(hb), "unit": "img/s", "h2d_bytes_per_step": per * 3 * 224 * 224 * 2,
                              "h2d_gb_per_s_per_gpu": e2e_run.h2d_gbs}
    del hb
    with near_gpu(dev):
        hu = torch.empty((per, 3, 224, 224), dtype=torch.uint8).pin_memory()
    hu.copy_(torch.randint(0, 256, (per, 3, 224, 224), dtype=torch.uint8))
    e2e_alt["u8_pixels"] = {"value": e2e_run(hu), "unit": "img/s", "h2d_bytes_per_step": per * 3 * 224 * 224,
                            "h2d_gb_per_s_per_gpu": e2e_run.h2d_gbs,
                            "note": "raw uint8 images, ImageNet mean/std normalisation fused into the patch gather"}
    del hu

    # ------------------------------------------------------------------ roofline of the dominant kernel (FC1 GEMM)
    # Second pass over the SAME K steps with the library's event tap on: a CUDA event on the launching stream after
    # every launch (evt_model_profile_begin/end), so each stage's time is measured inside the step, GPU at its
    # sustained (power-capped) clocks.  `value` above comes from the untapped pass.
    pk = peaks()
    roof = None
    stage_line = None
    if rank == 0:
        d, _, inter, _ = WORKLOADS[args.workload]
        M = chunk * 197
        model.profile_begin()
        e0.record()
        for _ in range(args.steps):
            step()
        e1.record()
        stages = model.profile_end()
        tapped_ms = e0.elapsed_time(e1)
        tot = sum(ms for ms, _ in stages.values())
        stage_line = {k: {"ms_per_launch": ms / max(n, 1), "launches": n, "share": ms / tot} for k, (ms, n) in stages.items()}
        stage_line["_tapped_step_ms"] = tapped_ms / args.steps
        fc1_ms, fc1_n = stages["fc1"]
        kms = fc1_ms / max(fc1_n, 1)
        flops = 2.0 * M * inter * d                       # algorithmic FLOPs of one FC1 launch (chunk x 197 rows)
        ach = flops / (kms / 1e3) / 1e12
        # the same kernel timed alone (burst clocks) for comparison with the burst peak
        a = torch.randn(M, d, device=dev).bfloat16()
        w = (torch.randn(inter, d, device=dev) * 0.02).bfloat16()
        b = torch.zeros(inter, device=dev)
        o = torch.empty(M, inter, device=dev, dtype=torch.bfloat16)
        alone_ms = timed_steps(lambda: ops.linear(a, w, b, act="gelu_erf", out=o), 10, warmup=3)
        alone = flops / (alone_ms / 1e3) / 1e12
        kname = "gemm_pair_kernel<256,bf16,gelu_erf>"
        traffic, stale, tsrc = traffic_lookup(kname, M, inter, d)
        roof = {"bound": "tensor", "kernel": "%s (FC1: M=%d N=%d K=%d)" % (kname, M, inter, d),
                "achieved": ach, "peak": pk["tf_sustained"], "unit": "TFLOP/s", "frac": ach / pk["tf_sustained"],
                "peak_source": pk["src"] + " (sustained: kernel timed inside the step, %d launches)" % fc1_n,
                "ms_per_launch": kms, "share_of_step": fc1_ms / tot,
                "alone": {"achieved": alone, "peak": pk["tf_burst"], "frac": alone / pk["tf_burst"], "ms_per_launch": alone_ms,
                          "peak_source": pk["src"] + " (burst: kernel timed alone)"},
                # dram__bytes_read.sum + dram__bytes_write.sum per launch of this kernel at this shape, looked up in the index of
                # committed ncu --set full captures (profiles/traffic.json); null + traffic_stale when no capture matches
                "traffic": traffic, "traffic_stale": stale, "traffic_source": tsrc,
                "algorithmic_bytes": 2.0 * M * d + 2.0 * inter * d + 2.0 * M * inter,
                "model_frac_sustained": value / n_gpus * GFLOP_PER_IMG[args.workload] / 1e3 / pk["tf_sustained"]}
        del a, w, b, o

    # ------------------------------------------------------------------ batch-1 latency (BASELINE metric: bs1 p50)
    lat = None
    if rank == 0:
        x1 = x[:1].contiguous()
        for _ in range(30):
            model.forward_graphed(x1)
        torch.cuda.synchronize()
        ts = []
        for _ in range(200):                      # sync-bracketed wall clock per run, as utils.py:866-872 times a model
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            model.forward_graphed(x1)
            torch.cuda.synchronize()
            ts.append((time.perf_counter() - t0) * 1e3)
        ts.sort()
        lat = {"batch": 1, "model": args.workload + " bf16", "p50_ms": ts[len(ts) // 2], "p90_ms": ts[int(len(ts) * 0.9)], "runs": len(ts),
               "how": "CUDA-graph replay of the forward incl. the device-side input copy, host wall clock around each run"}

    extras, lib_base = None, None
    if rank == 0 and n_gpus == 1 and not args.no_extras:
        del x
        torch.cuda.empty_cache()
        lat["config1"] = config1_latency(dev)
        extras = extra_configs(dev, max(5, min(args.steps, 10)), pk)
        lib_base = library_baseline(dev, chunk, 5)

    cpu = None
    if rank == 0 and n_gpus == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        ips, n, el = cpu_forward_rate(args.workload, 16, 15.0, threads)
        cpu = {"value": ips, "unit": "img/s", "cores": threads, "kind": "reference",
               "sample": f"{n} forwards of 16 synthetic images in {el:.1f}s, HF ViTForImageClassification fp32 eager on host CPU"}

    if rank == 0:
        line = {
            "metric": "images_per_sec", "value": value, "unit": "img/s", "n_gpus": n_gpus, "steps": args.steps,
            "warmup": warm, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"{args.workload} patch16-224 bf16 forward, random-init weights", "global_batch": gbatch,
                       "per_gpu_batch": per, "chunk": chunk, "parallelism": f"batch-sharded x{n_gpus}, no collective",
                       "l2": "inputs larger than L2 (%.0f MB of pixels per step)" % (per * 3 * 224 * 224 * 4 / 1e6),
                       "preroll": "%d untimed steps over %.1f s before the timed region (sustained clocks)" % (pre_steps, args.preroll_s)},
            "e2e": {"value": e2e_value, "unit": "img/s", "h2d_bytes_per_step": per * 3 * 224 * 224 * 4,
                    "d2h_bytes_per_step": per * 1000 * 4, "pixels": "f32 pinned host memory",
                    "host_numa": numa_note or "not bound (NVML affinity unavailable)",
                    "mode": e2e_mode,
                    "how": "every step copies its pixels in and its logits out inside the timed region; value = the better of the two loops below",
                    "pipelined": {"value": e2e_pipe, "unit": "img/s", "how": "PipelinedClassifier.submit/result, step i+1 queued before "
                                  "step i is collected (its H2D runs under step i's last forwards)"},
                    "per_call_synchronous": {"value": e2e_sync, "unit": "img/s", "how": "one PipelinedClassifier.logits(host) per step"},
                    "h2d_gb_per_s_per_gpu": e2e_h2d_gbs, "ratio_to_device_resident": e2e_value / value,
                    "other_pixel_types": e2e_alt},
            "gpu_launches": int(launches),
            "clocks": clk.summary(),
            "roofline": roof,
            "stages": stage_line,
            "latency": lat,
            "configs": extras,
            "gpu_library_baseline": lib_base,
            "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
