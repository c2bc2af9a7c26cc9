"""Build libevt.so in-tree with nvcc for sm_100a (no torch headers: the boundary is a plain C ABI).

    python -m edgevisiontransformer_b200.build [--force]

Objects and the shared library land next to the sources (git-ignored, shipped to the GPU box).
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
# EVT_BUILD_OUT / EVT_NVCC_EXTRA: build a second library (another commit's sources, or extra nvcc flags) under its own name for
# same-box A/B runs against the shipped one (loaded through EVT_LIB_PATH), e.g. EVT_BUILD_OUT=libevt_prev.so
OUT = os.path.join(HERE, os.environ.get("EVT_BUILD_OUT", "libevt.so"))
OBJ_DIR = os.path.join(CSRC, "build" + ("_" + os.path.splitext(os.path.basename(OUT))[0] if "EVT_BUILD_OUT" in os.environ else ""))

SOURCES = ["common.cu", "gemm.cu", "gemm2.cu", "gemm_ln.cu", "gemm_rowln.cu", "attention.cu", "layernorm.cu", "embed.cu", "performer.cu", "swin.cu", "swinv2.cu", "swin_model.cu", "model.cu"]
# Kernels that lost their A/B tests are not kept in the tree: DESIGN.md records each result and the commit its source is at.

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
    "-Xptxas", "-v",
] + os.environ.get("EVT_NVCC_EXTRA", "").split()


def nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libevt cannot be built (there is no prebuilt or CPU fallback)")


def _digest(paths) -> str:
    h = hashlib.sha256()
    for p in sorted(paths):
        with open(p, "rb") as f:
            h.update(p.encode())
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ_DIR, exist_ok=True)
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "evt.h"))
    stamp_path = os.path.join(OBJ_DIR, "stamp")
    want = _digest(srcs + headers)
    if not force and os.path.exists(OUT) and os.path.exists(stamp_path) and open(stamp_path).read() == want:
        return OUT
    cc = nvcc()

    def compile_one(src):
        obj = os.path.join(OBJ_DIR, os.path.basename(src) + ".o")
        cmd = [cc] + NVCC_FLAGS + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log = r.stdout + r.stderr
        with open(obj + ".log", "w") as f:
            f.write(log)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{log[-6000:]}")
        if verbose:
            print(log)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        objs = list(ex.map(compile_one, srcs))
    cmd = [cc, "-shared", "-o", OUT] + objs + ["-cudart", "static", "-Xlinker", "--exclude-libs=ALL"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    with open(stamp_path, "w") as f:
        f.write(want)
    return OUT


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(path)
