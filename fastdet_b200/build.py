"""Builds fastdet_b200/libfastdet_b200.so in-tree with nvcc for sm_100a (and nothing else).

    python -m fastdet_b200.build [--force] [--dev]

The shared object is git-ignored but travels to the GPU box with the repo snapshot.  cudart is linked
statically and the driver API (tensor-map encoders) is resolved at run time, so the library loads — and its
host-side logic (ONNX parse, fusion, BatchNorm folding, weight packing) runs — on a machine without a GPU.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libfastdet_b200.so")
SOURCES = ["capi.cu", "conv_tc.cu", "conv_halo.cu", "conv_stem.cu", "conv_block.cu", "jpeg.cu", "pre.cu", "pool.cu", "post.cu", "plan.cc", "onnx_reader.cc", "options.cc", "server.cc"]
HEADERS = ["conv_tc.h", "conv_halo.h", "conv_stem.h", "conv_block.h", "kernels.h", "jpeg.h", "plan.h", "onnx_reader.h", "options.h", "ptx.cuh", "act.cuh", os.path.join("..", "..", "include", "fastdet_b200.h")]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def nvcc() -> str:
    exe = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(exe):
        raise RuntimeError("nvcc not found: fastdet_b200 needs the CUDA toolkit to build its sm_100a library")
    return exe


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    deps = srcs + [os.path.join(CSRC, h) for h in HEADERS]
    if not force and not _stale(LIB, deps):
        return LIB
    objdir = os.path.join(HERE, "csrc", "_obj")
    os.makedirs(objdir, exist_ok=True)
    common = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC"] + ARCH
    if verbose:
        common += ["-Xptxas", "-v"]
    procs = []
    objs = []
    for s in srcs:
        o = os.path.join(objdir, os.path.basename(s) + ".o")
        objs.append(o)
        if force or _stale(o, [s] + deps[len(srcs):]):
            cmd = [nvcc()] + common + (["-x", "cu"] if s.endswith(".cc") else []) + ["-c", s, "-o", o]
            procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for cmd, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError("nvcc failed: " + " ".join(cmd) + "\n" + out)
        if verbose and out:
            print(out)
    link = [nvcc()] + ARCH + ["-shared", "-o", LIB] + objs + ["-cudart", "static"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed: " + " ".join(link) + "\n" + r.stdout)
    return LIB


def build_dev_harness() -> str:
    """csrc/dev/test_conv: stand-alone conv kernel checker/timer (developer tool)."""
    out = os.path.join(os.path.dirname(HERE), "build", "test_conv")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    srcs = [os.path.join(CSRC, "conv_tc.cu"), os.path.join(CSRC, "conv_halo.cu"), os.path.join(CSRC, "options.cc"),
            os.path.join(CSRC, "dev", "test_conv.cu")]
    if os.path.exists(out) and not _stale(out, srcs + [os.path.join(CSRC, h) for h in HEADERS]):
        return out
    # -DFASTDET_DEV: the harness build is the only one that carries the kernels' cycle counters / skip switches
    cmd = [nvcc(), "-O3", "-std=c++17", "-lineinfo", "-DFASTDET_DEV"] + ARCH + ["-x", "cu"] + srcs + ["-o", out]
    subprocess.run(cmd, check=True)
    return out


def build_stem_harness() -> str:
    """csrc/dev/test_stem: stand-alone checker/timer of the fused stem kernel against a float64 loop and the two-kernel path."""
    out = os.path.join(os.path.dirname(HERE), "build", "test_stem")
    srcs = [os.path.join(CSRC, f) for f in ("conv_tc.cu", "conv_halo.cu", "conv_stem.cu", "conv_block.cu", "pre.cu", "options.cc", os.path.join("dev", "test_stem.cu"))]
    if os.path.exists(out) and not _stale(out, srcs + [os.path.join(CSRC, h) for h in HEADERS]):
        return out
    cmd = [nvcc(), "-O3", "-std=c++17", "-lineinfo", "-DFASTDET_DEV"] + ARCH + ["-x", "cu"] + srcs + ["-o", out]
    subprocess.run(cmd, check=True)
    return out


if __name__ == "__main__":
    lib = build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(lib)
    if "--dev" in sys.argv:
        print(build_dev_harness())
        print(build_stem_harness())
