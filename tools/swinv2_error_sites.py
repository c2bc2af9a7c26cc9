"""Where the bf16 error of the Swin V2 forward comes from; prints one JSON line.

    python tools/swinv2_error_sites.py [--images 8]

The fp32 HF Swinv2ForImageClassification (TF32 off) is run again with its tensors rounded to bf16 at one of the places where
the library's forward stores or reads bf16, one place at a time and all together, and each run's logits are compared with the
fp32 ones.  The sites are those of csrc/swin_model.cu v2_block: GEMM weights, the pixels (im2col), the bf16 copy of the residual
stream that the QKV and FC1 GEMMs read, the qkv GEMM output, the softmax probabilities (P of P V), the attention context, the
FC1 output, the patch-merging input and the pooled features.  With the library's own logits beside them this separates the
error one rounding site adds from the rest.  Also measured: how far the HF forward (shift mask added twice) and the original
arithmetic (once) lie apart on stress-initialised weights, with logit scales up to the clamp.
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from edgevisiontransformer_b200.modeling_swinv2 import B200Swinv2ForImageClassification  # noqa: E402
from oracle import swinv2 as osv2  # noqa: E402
from oracle import vit as ovit  # noqa: E402

SITES = ("weights", "pixels", "stream_a", "qkv_out", "probs", "ctx", "fc1_out", "merge_a", "pooled")


def _bf(t):
    return t.bfloat16().float()


def round_at(model, sites):
    """Hooks that round the named sites to bf16; returns the handles (weights are rounded in place)."""
    hs = []
    pre = lambda m, a: (_bf(a[0]),) + tuple(a[1:])  # noqa: E731
    post = lambda m, a, o: _bf(o)  # noqa: E731
    for name, mod in model.named_modules():
        leaf = name.rsplit(".", 1)[-1]
        if "weights" in sites and isinstance(mod, (torch.nn.Linear, torch.nn.Conv2d)) and "continuous_position_bias_mlp" not in name:
            mod.weight.data = _bf(mod.weight.data)
        if "pixels" in sites and leaf == "projection":
            hs.append(mod.register_forward_pre_hook(pre))
        if "stream_a" in sites and (leaf in ("query", "key", "value") or name.endswith("intermediate.dense")):
            hs.append(mod.register_forward_pre_hook(pre))
        if "qkv_out" in sites and leaf in ("query", "key", "value"):
            hs.append(mod.register_forward_hook(post))
        if "probs" in sites and name.endswith("attention.self.dropout"):
            hs.append(mod.register_forward_hook(post))
        if "ctx" in sites and name.endswith("attention.output.dense"):
            hs.append(mod.register_forward_pre_hook(pre))
        if "fc1_out" in sites and name.endswith(".output.dense") and "attention" not in name:
            hs.append(mod.register_forward_pre_hook(pre))
        if "merge_a" in sites and leaf == "reduction":
            hs.append(mod.register_forward_pre_hook(pre))
        if "pooled" in sites and name == "classifier":
            hs.append(mod.register_forward_pre_hook(pre))
    return hs


def logits(model, x):
    with torch.no_grad():
        return model(pixel_values=x).logits.float()


def sites_of(kind, window, pws, x, seed=0, stress=False):
    hf = osv2.build_hf_swinv2(kind, seed=seed, window=window, pretrained_window_sizes=pws, stress=stress).cuda()
    ref = logits(hf, x)
    lib = B200Swinv2ForImageClassification.from_hf(hf, max_batch=x.shape[0])
    out = {"library": round(ovit.compare_logits(lib(x).logits, ref)["max_abs"], 5), "ref_logit_std": round(ref.std().item(), 4)}
    del lib
    sd = {k: v.clone() for k, v in hf.state_dict().items()}
    for s in SITES + ("all",):
        hf.load_state_dict(sd, strict=False)
        hs = round_at(hf, SITES if s == "all" else (s,))
        out[s] = round(ovit.compare_logits(logits(hf, x), ref)["max_abs"], 5)
        for h in hs:
            h.remove()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--images", type=int, default=8)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        print("swinv2_error_sites needs a GPU")
        return 2
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = False, False
    x = torch.randn(a.images, 3, 256, 256, generator=torch.Generator().manual_seed(0)).cuda()
    out = {"gpu": torch.cuda.get_device_name(), "images": a.images, "max_abs_vs_fp32": {}}
    for label, kind, window, pws in (("tiny_w8", "tiny", 8, [0] * 4), ("base_w16", "base", 16, [0] * 4),
                                     ("base_w12to16", "base", 16, [12, 12, 12, 6]), ("large_w12to16", "large", 16, [12, 12, 12, 6])):
        out["max_abs_vs_fp32"][label] = sites_of(kind, window, pws, x)
        torch.cuda.empty_cache()
    # mask added twice (HF) vs once (original code), fp32 both, stress weights with logit scales up to the clamp
    mask = {}
    for label, kind, window in (("tiny_w8_stress", "tiny", 8), ("base_w16_stress", "base", 16)):
        hf = osv2.build_hf_swinv2(kind, seed=7, window=window, stress=True).cuda()
        twice = logits(hf, x)
        osv2.halve_shift_masks(hf)
        once = logits(hf, x)
        mask[label] = {"max_abs": float((twice - once).abs().max()), "logit_std": round(twice.std().item(), 4)}
        del hf
        torch.cuda.empty_cache()
    out["mask_twice_vs_once"] = mask
    print(json.dumps(out))
    return 0


if __name__ == "__main__":
    sys.exit(main())
