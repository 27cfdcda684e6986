"""Builds libminorseq_b200.so (CUDA kernels + C ABI) in-tree with nvcc for sm_100a."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libminorseq_b200.so")
SOURCES = ["abi_core.cu", "pileup.cu", "format.cu", "synth.cu", "call.cu", "phase.cu", "phase_order.cu", "cooc_tc.cu", "fuse.cu", "comm.cu", "pass.cu", "nw.cu", "events.cu", "tiles.cu", "linkage.cu", "group.cu", "align.cu", "abundance.cu", "indel.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-fmad=false",  # K2's fp64 path must not contract a*b+c (fisher_core.h)
    "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall", "-shared", "-ldl",
]


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "minorseq_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force=False, verbose=False):
    if not force and not _stale():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    res = subprocess.run(cmd + ["-ccbin", "/usr/bin/g++"], capture_output=True, text=True, env=env)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed building libminorseq_b200.so")
    if verbose:
        sys.stderr.write(res.stderr)
    return LIB


HOST = os.path.join(HERE, "host")
BIN = os.path.join(HERE, "bin")
HOST_PROGRAMS = {"juliet": "juliet_main.cpp", "fuse": "fuse_main.cpp", "host_selftest": "host_selftest.cpp", "mixdata": "mixdata_main.cpp", "packed2bam": "packed2bam_main.cpp", "cleric": "cleric_main.cpp", "align": "align_main.cpp", "julietflow": "julietflow_main.cpp"}


def build_host(force=False):
    """The C++ host layer above the C ABI: juliet / fuse mains and the CPU-only self test (g++, zlib)."""
    os.makedirs(BIN, exist_ok=True)
    hdrs = [os.path.join(HOST, f) for f in os.listdir(HOST)] + [os.path.join(HERE, "..", "include", "minorseq_b200.h"), LIB]
    for name, src in HOST_PROGRAMS.items():
        out = os.path.join(BIN, name)
        if not force and os.path.exists(out) and all(os.path.getmtime(d) <= os.path.getmtime(out) for d in hdrs if os.path.exists(d)):
            continue
        cmd = ["/usr/bin/g++", "-O3", "-std=c++17", "-Wall", "-I/usr/local/cuda/include", "-o", out, os.path.join(HOST, src), "-lz", "-pthread", "-ldl"]
        if name in ("juliet", "fuse", "cleric", "align"):
            cmd += ["-L" + HERE, "-lminorseq_b200", "-Wl,-rpath,$ORIGIN/..", "-Wl,-rpath," + HERE]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            sys.stderr.write(res.stdout + res.stderr)
            raise RuntimeError(f"g++ failed building {name}")
    return BIN


if __name__ == "__main__":
    print(build_library(force=True, verbose="-v" in sys.argv))
    print(build_host(force=True))
