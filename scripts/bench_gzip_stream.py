#!/usr/bin/env python
"""Ordinary-gzip decoder benchmark: the device decoder (csq_gz_stream_inflate, csrc/gz_stream.cu) against the host
decoder of the file driver (csq_pinflate_mem, csrc/pinflate.cpp, at the driver's thread count for paired input), on one
mate of seeded config-2 FASTQ (4 M reads by default) as a single gzip member at levels 1 and 6, plus the slow inputs
(level 0 = stored blocks, and Z_FIXED: no block start the search can find); GB/s of text.  Host and device runs
alternate (A B A B) in one process, and both outputs must equal the text.  The GPU name and power limit are read in the
same run.

    python scripts/bench_gzip_stream.py --reads 4000000 --out gzip_stream.json
"""

import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.abspath(os.path.dirname(__file__)))
sys.path.insert(0, ROOT)

from scripts.bench_files import gzip_single_member  # noqa: E402


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def decoder_leg(text: bytes, comp: bytes, threads: int, reps: int):
    from cutseq_b200 import native

    L = native.lib()
    src = np.frombuffer(comp + b"\0" * 16, dtype=np.uint8)
    out = np.empty(len(text) + 1, dtype=np.uint8)
    n = C.c_uint64()
    want = hashlib.sha256(text).hexdigest()
    runs = {"host": [], "device": []}
    for _ in range(reps):
        for route in ("host", "device"):
            out[:16] = 0
            t0 = time.perf_counter()
            if route == "host":
                rc = L.csq_pinflate_mem(src.ctypes.data, len(comp), out.ctypes.data, out.size, threads, 0, C.byref(n))
            else:
                rc = L.csq_gz_stream_inflate(0, src.ctypes.data, len(comp), out.ctypes.data, out.size, 0, 0, C.byref(n))
            dt = time.perf_counter() - t0
            native.check(rc)
            if n.value != len(text) or hashlib.sha256(out[: n.value]).hexdigest() != want:
                raise SystemExit(f"{route} decoder output differs from the text")
            runs[route].append(round(len(text) / dt / 1e9, 3))
    return {"text_bytes": len(text), "comp_bytes": len(comp), "gb_per_s": runs}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=4_000_000, help="reads of the decoder-alone input (one mate)")
    ap.add_argument("--slow-reads", type=int, default=1_000_000, help="reads of the level-0 and Z_FIXED inputs")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--threads", type=int, default=os.cpu_count() or 8)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from cutseq_b200 import native

    res = {"gpu": gpu_info(), "decoder": {}}
    # pinflate's thread count in the file driver for paired input: the host's cores shared by the two mates
    host_threads = min(16, max(2, (os.cpu_count() or 8) // 2))
    res["pinflate_threads"] = host_threads
    batch = native.synth_batch(2, args.reads, first_index=0, buffer=14)
    text = bytes(native.format_fastq(batch, 0))
    native.lib().csq_synth_free()
    for level in (1, 6):
        comp = gzip_single_member(text, args.threads, level=level)
        res["decoder"][f"level{level}"] = decoder_leg(text, comp, host_threads, args.reps)
        print(json.dumps({f"level{level}": res["decoder"][f"level{level}"]}), flush=True)
    slow = text[: len(text) * args.slow_reads // max(args.reads, 1)]
    slow = slow[: slow.rfind(b"\n") + 1]
    for name, level, strategy in (("level0", 0, zlib.Z_DEFAULT_STRATEGY), ("fixed", 6, zlib.Z_FIXED)):
        c = zlib.compressobj(level, zlib.DEFLATED, 31, 8, strategy)
        comp = c.compress(slow) + c.flush()
        res["decoder"][name] = decoder_leg(slow, comp, host_threads, 1)
        print(json.dumps({name: res["decoder"][name]}), flush=True)
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
