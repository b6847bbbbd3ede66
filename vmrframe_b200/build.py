"""Builds the in-tree CUDA library ``vmrframe_b200/libseqpan_b200.so`` for sm_100a with nvcc.

The shared object is git-ignored but travels to the GPU box with the ``gpurun`` snapshot; nothing is
JIT-compiled at run time.  ``python -m vmrframe_b200.build`` rebuilds unconditionally; translation units
are compiled in parallel into ``csrc/_obj`` (git-ignored) and only re-compiled when they or a header changed.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
OBJ = os.path.join(CSRC, os.environ.get("SEQPAN_OBJDIR", "_obj"))
LIB = os.environ.get("SEQPAN_LIB") or os.path.join(PKG, "libseqpan_b200.so")
SOURCES = ["kernels_f32.cu", "linear_tc.cu", "chain_tc.cu", "tail_tc.cu", "attn_tc.cu", "cq_tc.cu", "train_ops.cu", "train_tc.cu", "seqpan_api.cu"]
# diagnostics (tcgen05 descriptor probe) live in their own library: the product library exports no test entry points
DIAG_SOURCES = ["umma_probe.cu"]
DIAG_LIB = os.path.join(os.path.dirname(LIB), "libseqpan_diag.so")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
CFLAGS = ARCH + ["-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC"] + \
    (["-DSEQPAN_TIMELINE"] if os.environ.get("SEQPAN_TIMELINE") == "1" else []) + \
    [f"-D{d}" for d in os.environ.get("SEQPAN_DEFINES", "").split()]


def _headers() -> list[str]:
    hs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h", ".def"))]
    return hs + [os.path.join(PKG, "..", "include", "seqpan_b200.h")]


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    if not os.path.exists(DIAG_LIB):
        return True
    t = min(t, os.path.getmtime(DIAG_LIB))
    deps = [os.path.join(CSRC, f) for f in SOURCES + DIAG_SOURCES] + _headers()
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "nvcc")
    os.makedirs(OBJ, exist_ok=True)
    hdr_t = max(os.path.getmtime(h) for h in _headers())

    def compile_one(src: str):
        s, o = os.path.join(CSRC, src), os.path.join(OBJ, src + ".o")
        if not force and os.path.exists(o) and os.path.getmtime(o) > max(os.path.getmtime(s), hdr_t):
            return None
        cmd = [nvcc] + CFLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
        return res.stderr

    with ThreadPoolExecutor(max_workers=len(SOURCES) + len(DIAG_SOURCES)) as ex:
        logs = list(ex.map(compile_one, SOURCES + DIAG_SOURCES))
    if verbose:
        for src, log in zip(SOURCES + DIAG_SOURCES, logs):
            if log:
                print(f"== {src}\n{log}")
    cmd = [nvcc] + ARCH + ["-shared", "-cudart", "static", "-o", LIB] + [os.path.join(OBJ, s + ".o") for s in SOURCES]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    cmd = [nvcc] + ARCH + ["-shared", "-cudart", "static", "-o", DIAG_LIB] + [os.path.join(OBJ, s + ".o") for s in DIAG_SOURCES]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n" + " ".join(cmd) + "\n" + res.stdout + res.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="-f" in sys.argv or "--force" in sys.argv, verbose="-v" in sys.argv))
