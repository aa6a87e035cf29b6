#!/usr/bin/env python
"""FASTA file benchmark: seeded FASTA pairs (BASELINE.json config 2, csq_synth_batch) on disk, trimmed through the
command line twice - the native route (the library parses and writes FASTA, CSQ_PLAN_FASTA) and the pump route (the
converting Python pumps of cutseq_b200.transcode around a FASTQ plan, what the command line did before) - for
unwrapped and 60-column records, plain and .gz.  Reports pairs/s of both routes, the sha256 of every decompressed
output (the routes must agree) and the GPU name and power limit read in the same run.

    python scripts/bench_fasta.py --pairs 10000000 --out fasta.json
"""

import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from scripts.bench_files import gzip_single_member, hash_outputs  # noqa: E402

BLOCK_PAIRS = 1_000_000  # pairs generated and converted at a time; larger fixtures repeat this block


def fasta_block(fastq: bytes, width):
    """FASTQ text as csq_format_fastq writes it -> FASTA records, the sequence wrapped at `width` columns (None: not)."""
    lines = fastq.split(b"\n")
    heads, seqs = lines[0:-1:4], lines[1:-1:4]
    if width is None:
        return b"".join(b">" + h[1:] + b"\n" + s + b"\n" for h, s in zip(heads, seqs))
    return b"".join(b">" + h[1:] + b"\n" + b"".join(s[o:o + width] + b"\n" for o in range(0, len(s), width))
                    for h, s in zip(heads, seqs))


def write_fixtures(d, pairs, threads):
    """{variant: [R1, R2]} for unwrapped / wrapped60 x plain / gz."""
    from cutseq_b200 import native

    block = min(pairs, BLOCK_PAIRS)
    reps, rest = divmod(pairs, block)
    paths = {f"{shape}_{comp}": [os.path.join(d, f"{shape}_R{m + 1}.fa" + (".gz" if comp == "gz" else "")) for m in range(2)]
             for shape in ("unwrapped", "wrapped60") for comp in ("plain", "gz")}
    handles = {k: [open(p, "wb") for p in v] for k, v in paths.items()}
    try:
        for n, times in ((block, reps), (rest, 1 if rest else 0)):
            if not times:
                continue
            batch = native.synth_batch(2, n, first_index=0, buffer=14)
            for m in range(2):
                fastq = bytes(native.format_fastq(batch, m))
                for shape, width in (("unwrapped", None), ("wrapped60", 60)):
                    text = fasta_block(fastq, width)
                    gz = gzip_single_member(text, threads)
                    for _ in range(times):
                        handles[f"{shape}_plain"][m].write(text)
                        handles[f"{shape}_gz"][m].write(gz)
    finally:
        for v in handles.values():
            for f in v:
                f.close()
        native.lib().csq_synth_free()
    return paths


def run_route(route, inputs, out_dir, threads, gz_out):
    from cutseq_b200 import run
    from cutseq_b200.transcode import Transcoders

    ext = ".fa.gz" if gz_out else ".fa"
    outs = [os.path.join(out_dir, f"{route}_{n}{ext}") for n in ("trimmed_R1", "trimmed_R2", "short_R1", "short_R2")]
    argv = ["-A", "TAKARAV3", "--trim-polyA", "-t", str(threads)] + inputs + ["-o", outs[0], outs[1], "-s", outs[2], outs[3]]
    orig = Transcoders.__init__
    if route == "pump":  # the converting pumps around a FASTQ plan
        Transcoders.__init__ = lambda self, i, o, fasta_native=False: orig(self, i, o)
    try:
        t0 = time.perf_counter()
        run.main(argv)
        dt = time.perf_counter() - t0
    finally:
        Transcoders.__init__ = orig
    hashes = hash_outputs(outs, gz_out)
    for p in outs:
        os.remove(p)
    return dt, hashes


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=10_000_000)
    ap.add_argument("--threads", type=int, default=min(16, os.cpu_count() or 8))
    ap.add_argument("--variants", default="unwrapped_plain,wrapped60_plain,unwrapped_gz,wrapped60_gz")
    ap.add_argument("--routes", default="native,pump")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    tmp = tempfile.mkdtemp(prefix="bench_fasta_")
    res = {"pairs": args.pairs, "gpu": gpu_info(), "threads": args.threads, "variants": {}}
    try:
        t0 = time.perf_counter()
        paths = write_fixtures(tmp, args.pairs, args.threads)
        res["fixture_s"] = round(time.perf_counter() - t0, 1)
        for v in args.variants.split(","):
            row = {}
            for route in args.routes.split(","):
                dt, hashes = run_route(route, paths[v], tmp, args.threads, gz_out=v.endswith("_gz"))
                row[route] = {"seconds": round(dt, 2), "pairs_per_s": round(args.pairs / dt), "sha256": hashes}
                print(f"{v:16s} {route:6s} {dt:8.2f} s  {args.pairs / dt / 1e6:7.2f} M pairs/s", flush=True)
            hs = [r["sha256"] for r in row.values()]
            row["outputs_equal"] = all(h == hs[0] for h in hs)
            res["variants"][v] = row
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    print(json.dumps(res, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
