"""Builds lz4net_b200/liblz4b200.so in-tree with nvcc for sm_100a (the only target: no multi-arch fallback).

    python -m lz4net_b200.build            # incremental
    python -m lz4net_b200.build --force

nvcc cross-compiles without a GPU, so this also runs in the CPU-only build container.  The .so is git-ignored but
travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "liblz4b200.so")
SOURCES = ["capi.cu", "decode.cu", "encode.cu", "util.cu", "stream.cu", "framing.cpp"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def _stale() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(os.path.dirname(HERE), "include", "lz4b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return OUT
    objs = []
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.rsplit(".", 1)[0] + ".o")
        cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError(f"nvcc failed on {src}")
    # symbols: only the extern "C" ABI is exported (visibility=hidden + explicit default on the ABI via version script)
    vs = os.path.join(objdir, "exports.map")
    with open(vs, "w") as f:
        f.write("{ global: lz4b200_*; local: *; };\n")
    cmd = [_nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", OUT] + objs + ["-Xlinker", f"--version-script={vs}", "-lcudart_static", "-ldl", "-lrt", "-lpthread"]
    subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
