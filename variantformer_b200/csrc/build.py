"""Build libvf_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m variantformer_b200.csrc.build [--force] [--verbose]
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = ["vf_api.cu", "vf_gemm.cu", "vf_attention_mc.cu", "vf_elementwise.cu", "vf_encode.cu", "vf_forward.cu",
           "vf_attn_probs.cu"]
HEADERS = ["vf_common.cuh", "vf_internal.h", os.path.join("..", "..", "include", "vf_b200.h")]
LIB = os.path.join(HERE, "libvf_b200.so")
INGEST_SRC = os.path.join(HERE, "vf_ingest.cpp")
INGEST_LIB = os.path.join(HERE, "libvf_ingest.so")
CXX = os.environ.get("CXX", "g++")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
         "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-Xptxas", "-v"]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    hdrs = [os.path.join(HERE, h) for h in HEADERS]
    objs = []
    procs = []
    for src in SOURCES:
        s = os.path.join(HERE, src)
        o = os.path.join(HERE, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + hdrs):
            cmd = [NVCC] + FLAGS + ["-c", s, "-o", o]
            procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            print(f"--- {src} ---\n{out}")
        if p.returncode != 0:
            failed = True
    if failed:
        raise RuntimeError("nvcc failed")
    if force or procs or _stale(LIB, objs):
        subprocess.run([NVCC, "-shared", "-o", LIB] + objs + ["-lcudart"], check=True)
    build_ingest(force)
    return LIB


def build_ingest(force=False):
    """libvf_ingest.so: host-side FASTA / VCF ingest (C++17, zlib, threads; no CUDA)."""
    hdr = os.path.join(HERE, "..", "..", "include", "vf_ingest.h")
    if force or _stale(INGEST_LIB, [INGEST_SRC, hdr]):
        subprocess.run([CXX, "-O3", "-std=c++17", "-shared", "-fPIC", "-Wall", INGEST_SRC, "-o", INGEST_LIB, "-lz",
                        "-lpthread"], check=True)
    return INGEST_LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
