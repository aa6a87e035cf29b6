"""Builds cutseq_b200/libcutseq_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""

from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libcutseq_b200.so")
SOURCES = ["kernels.cu", "tail.cu", "emit_stage.cu", "gz_deflate.cu", "gz_inflate.cu", "gz_stream.cu", "plan.cu", "prefilter.cu", "parse.cu", "synth.cu", "fastq_io.cpp", "text_reader.cpp", "inflate.cpp", "pinflate.cpp", "pipeline.cpp", "host_numa.cpp"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-O3,-pthread,-Wall", "-cudart", "static",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    return "nvcc"


def sources():
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


STAMP = os.path.join(HERE, "build", "sources.sha256")


def _deps():
    deps = sources() + [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".h", ".cuh"))]
    deps.append(os.path.join(HERE, "..", "include", "cutseq_b200.h"))
    return deps


def sources_hash() -> str:
    """sha256 over everything the library is built from (contents, not time stamps: a checkout, a stash or the copy
    to a GPU box changes mtimes without changing a byte)."""
    import hashlib

    h = hashlib.sha256()
    for d in _deps():
        h.update(os.path.basename(d).encode() + b"\0")
        with open(d, "rb") as f:
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def needs_build() -> bool:
    if not os.path.exists(LIB):
        return True
    try:
        with open(STAMP) as f:
            return f.read().strip() != sources_hash()
    except OSError:
        return True


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    import fcntl

    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    # one builder at a time (torchrun ranks, pytest workers): the others wait and find the work done
    with open(os.path.join(objdir, ".lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        if not force and not needs_build():
            return LIB
        return _build_locked(objdir, verbose)


def _build_locked(objdir: str, verbose: bool) -> str:
    want = sources_hash()
    objs = []
    procs = []
    for src in sources():
        obj = os.path.join(objdir, os.path.basename(src) + ".o")
        objs.append(obj)
        cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-x", "cu", "-c", src, "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            sys.stderr.write(out)
            raise RuntimeError(f"nvcc failed on {src}")
        if verbose or "warning" in out:
            sys.stderr.write(out)
    tmp = LIB + f".tmp{os.getpid()}"
    cmd = [_nvcc(), "-shared", "-Wno-deprecated-gpu-targets", "-gencode", "arch=compute_100a,code=sm_100a", "-o", tmp] + objs + ["-cudart", "static", "-lz", "-lpthread"]
    subprocess.check_call(cmd)
    os.replace(tmp, LIB)  # a process that maps the old file keeps it
    with open(STAMP + ".tmp", "w") as f:
        f.write(want + "\n")
    os.replace(STAMP + ".tmp", STAMP)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
