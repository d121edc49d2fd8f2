"""Builds libsimdjson_b200.so (CUDA, sm_100a) and the synthetic-workload generator in-tree.

nvcc cross-compiles without a GPU; the built .so files are git-ignored but travel to the GPU box.
"""
from __future__ import annotations

import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libsimdjson_b200.so")
SYNTH_SRC = os.path.join(PKG, "synth", "gen.c")
SYNTH_LIB = os.path.join(PKG, "synth", "libsjb200_synth.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "-shared",
]


def _stale(target: str, sources: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def build_cuda(force: bool = False, verbose: bool = False) -> str:
    sources = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))]
    sources.append(os.path.join(PKG, "..", "include", "simdjson_b200.h"))
    if force or _stale(LIB, sources):
        nvcc = os.environ.get("NVCC", "nvcc")
        cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB, os.path.join(CSRC, "capi.cu")]
        subprocess.check_call(cmd)
    return LIB


def build_synth(force: bool = False) -> str:
    if force or _stale(SYNTH_LIB, [SYNTH_SRC]):
        subprocess.check_call(["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-o", SYNTH_LIB, SYNTH_SRC])
    return SYNTH_LIB


def build_cpp_tests(force: bool = False) -> str:
    """tests/cpp/batch_test: the multi-GPU batch driver driven from C++ alone (links the product library, the workload
    generator and -- as the checker -- the CPU oracle)."""
    root = os.path.dirname(PKG)
    src = os.path.join(root, "tests", "cpp", "batch_test.cpp")
    out = os.path.join(root, "tests", "cpp", "batch_test")
    oracle_dir = os.path.join(root, "oracle")
    if force or _stale(out, [src, LIB, SYNTH_LIB]):
        subprocess.check_call(["make", "-s", "-C", oracle_dir, "liboracle_stage1.so"])
        nvcc = os.environ.get("NVCC", "nvcc")
        subprocess.check_call([nvcc, "-O2", "-std=c++17", "-o", out, src, f"-L{PKG}", "-lsimdjson_b200", f"-L{os.path.dirname(SYNTH_LIB)}",
                               "-lsjb200_synth", f"-L{oracle_dir}", "-loracle_stage1",
                               "-Xlinker", "-rpath=$ORIGIN/../../mojo_simdjson_b200", "-Xlinker", "-rpath=$ORIGIN/../../mojo_simdjson_b200/synth",
                               "-Xlinker", "-rpath=$ORIGIN/../../oracle", "-Wno-deprecated-gpu-targets"])
    return out


def build_all(force: bool = False, verbose: bool = False) -> None:
    build_cuda(force, verbose)
    build_synth(force)
    build_cpp_tests(force)


if __name__ == "__main__":
    build_all(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(LIB)
