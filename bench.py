#!/usr/bin/env python
"""bench.py - read-pairs/s of the trimming chain on BASELINE.json's workload (config 2).

    python bench.py [--gpus N] [--steps K] [--warmup W]          # this implementation
    python bench.py --impl reference [...]                       # CPU arm (oracle port, all host cores)
    torchrun --nproc-per-node N bench.py --gpus N ...            # one rank per GPU

One "step" = one pass of the whole hot path (FASTQ parse, all ALIGN ops, cuts, quality trim, filters, FASTQ
emission) over the 10 M synthetic 2x150 read pairs of config 2 (`-A TAKARAV3 --trim-polyA`), held as 5 batches
of 2 M pairs per GPU.
  value  kernel throughput with the batches resident in HBM (CUDA events around exactly K steps, max over ranks)
  e2e    the same chain through csq_submit_text / csq_wait with pinned HOST buffers, host->device and device->host
         copies inside the timed region; roofline_e2e relates it to the measured PCIe copy ceiling (csq_pcie_peak)
  files  FASTQ files on disk -> csq_run_files (all GPUs of the job, driven by rank 0) -> trimmed FASTQ files, plain and
         .gz, with the sha256 of every output and its equality to the 1-GPU run of the same files
Prints ONE JSON line (rank 0).
"""

from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "read-pairs/s (2x150, TAKARAV3)"
UNIT = "pairs/s"
BATCH_PAIRS = 2_000_000      # pairs per batch and GPU
N_BATCHES = 5                # resident batches per GPU: 5 x 2M = the 10M pairs of config 2 = one step
ARGV = ["-A", "TAKARAV3", "--trim-polyA"]


def takara_program():
    from cutseq_b200 import program, run
    from cutseq_b200.common import BarcodeConfig

    args = run.build_parser().parse_args(ARGV + ["r1.fq", "r2.fq"])
    scheme = run.resolve_scheme(args)
    return program.compile_paired(BarcodeConfig(scheme), run.settings_from_args(args))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "25", "-i", str(self.device)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        rows = [l for (t, l) in self.lines if t0 - 0.05 <= t <= t1 + 0.15] or [l for (_, l) in self.lines]
        for l in rows:
            parts = [p.strip() for p in l.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def h2d_bytes(batch):
    total = 0
    for m in range(batch.n_mates):
        mi = batch.mate[m]
        total += 2 * mi.seq_bytes + 8 * batch.n_reads + mi.name_bytes + 4 * (batch.n_reads + 1)
    return int(total)


def kernel_sources_hash():
    """sha256 over the CUDA sources: numbers taken from a committed ncu capture are only printed next to live times
    when the kernels are still the ones that were profiled."""
    h = hashlib.sha256()
    csrc = os.path.join(ROOT, "cutseq_b200", "csrc")
    for fn in sorted(os.listdir(csrc)):
        if fn.endswith((".cu", ".cuh", ".h")):
            with open(os.path.join(csrc, fn), "rb") as f:
                h.update(f.read())
    return h.hexdigest()[:16]


DUMP_SEED = 20241020
DUMP_READS = 1 << 15                 # per-read results kept per batch
DUMP_WINDOWS, DUMP_WINDOW = 16, 1024  # windows of FASTQ text kept per output stream (bytes each)


def dump_outputs(out_dir, plan, slots, P, first_index, capacity):
    """Writes what the last timed step computed - each slot's outputs as Plan.results / Plan.fetch_text hand them to a
    caller - to out_dir/<name>.npy (the untimed profiling step behind the timed ones reruns the first slot's batch:
    same outputs).  The full outputs are GBs, so beside the exact size and sha256 of every FASTQ stream only a fixed,
    seeded sample is kept: DUMP_READS reads per batch and DUMP_WINDOWS text windows per stream.
      read_index                  [n]            global index of each sampled read
      read_{start,stop,dest,matched} [n, mate]   csq_read_result of those reads
      text_bytes                  [batch, dest, mate]
      text_sha256                 [batch, dest, mate, 8]   digest of the whole stream as big-endian 32-bit words
      text_windows                [batch, dest, mate, window, byte]   float32 byte values, -1 past the end"""
    import numpy as np

    rng = np.random.default_rng(DUMP_SEED)
    index, fields = [], {k: [] for k in ("start", "stop", "dest", "matched")}
    text_bytes, sha, windows = [], [], []
    for b, slot in enumerate(slots):
        pick = np.sort(rng.choice(P, size=min(DUMP_READS, P), replace=False))
        index.append(first_index + b * P + pick)
        res = [plan.results(slot, m, P)[pick] for m in range(2)]
        for k in fields:
            fields[k].append(np.stack([r[k] for r in res], axis=1))
        texts = plan.fetch_text(slot, capacity)
        text_bytes.append([[len(t) for t in row] for row in texts])
        sha.append([[np.frombuffer(hashlib.sha256(t).digest(), dtype=">u4") for t in row] for row in texts])
        win = np.full((len(texts), 2, DUMP_WINDOWS, DUMP_WINDOW), -1, dtype=np.float32)
        for d, row in enumerate(texts):
            for m, t in enumerate(row):
                starts = (rng.random(DUMP_WINDOWS) * max(len(t) - DUMP_WINDOW, 0)).astype(np.int64)
                for w, s in enumerate(starts):
                    piece = np.frombuffer(t[s : s + DUMP_WINDOW], dtype=np.uint8)
                    win[d, m, w, : len(piece)] = piece
        windows.append(win)
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"read_index": np.concatenate(index), "text_bytes": np.array(text_bytes), "text_sha256": np.array(sha),
              "text_windows": np.stack(windows)}
    arrays.update({f"read_{k}": np.concatenate(v) for k, v in fields.items()})
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a if a.dtype == np.float32 else a.astype(np.float64))


def real_reference_available():
    """A real cutadapt 5.x + a reference tree: then the CPU arm is the reference itself (scripts/bless_against_cutadapt.py)."""
    try:
        from scripts import bless_against_cutadapt as bless

        mod, info = bless.real_cutadapt()
        if mod is None:
            return None
        for cand in (os.environ.get("CUTSEQ_REFERENCE"), "/root/reference", os.path.join(ROOT, "baseline", "_ref")):
            if cand and os.path.exists(os.path.join(cand, "cutseq", "run.py")):
                return {"cutadapt": info, "reference": cand}
    except Exception:
        pass
    return None


def cpu_leg_real(ref, steps, sample_pairs):
    """`cutseq -A TAKARAV3 --trim-polyA -t <cores>` of the REAL reference on files of the same generator."""
    import shutil
    import tempfile

    from oracle import oracle
    from scripts import bench_files

    tmp = tempfile.mkdtemp()
    try:
        batch = oracle.synth_batch(2, sample_pairs)
        ins = [os.path.join(tmp, f"in_R{m}.fq") for m in (1, 2)]
        bench_files.write_fastq_from_soa(batch, ins)
        cores = os.cpu_count() or 1
        env = dict(os.environ, PYTHONPATH=ref["reference"] + os.pathsep + os.environ.get("PYTHONPATH", ""))
        t0 = time.perf_counter()
        for _ in range(steps):
            subprocess.check_call([sys.executable, "-m", "cutseq.run"] + ARGV + ["-t", str(cores), "-O", os.path.join(tmp, "out")] + ins,
                                  env=env, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        dt = time.perf_counter() - t0
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return steps * sample_pairs / dt, cores, dt / steps


def cpu_leg(prog, steps, warmup, sample_pairs, first_index=0):
    """The oracle port on all host cores over bounded samples of the same workload (generator: oracle/libsynth.so,
    the CUDA-free build of cutseq_b200/csrc/synth.cu - nothing of the product library is mapped here)."""
    from oracle import oracle

    threads = oracle.lib().orc_max_threads()
    batch = oracle.synth_batch(2, sample_pairs, first_index=first_index)
    for _ in range(max(0, warmup)):
        oracle.run_batch(prog, batch, n_threads=threads, want_matches=False)
    t0 = time.perf_counter()
    for _ in range(steps):
        oracle.run_batch(prog, batch, n_threads=threads, want_matches=False)
    dt = time.perf_counter() - t0
    return steps * sample_pairs / dt, threads, dt / steps


def files_leg(prog, pairs_plain, pairs_gz, n_devices, threads, pairs_gzip=0):
    """FASTQ files on disk -> csq_run_files -> trimmed FASTQ files, plain and .gz (BGZF members in, gzip members out);
    host stages reported separately; with n_devices > 1 the same files also go through ONE GPU and the outputs must
    have the same sha256 (order-preserving reassembly, reference run.py:751-758 / 793-794 `-t N` runner)."""
    import shutil
    import tempfile

    from cutseq_b200 import native
    from scripts import bench_files

    tmp = tempfile.mkdtemp(dir=os.environ.get("CSQ_BENCH_TMP"))
    out = {"host_threads": threads, "n_devices": n_devices}
    try:
        for variant, pairs in (("plain", pairs_plain), ("gz", pairs_gz), ("gzip", pairs_gzip)):
            if pairs <= 0:
                continue
            ext = ".fq" if variant == "plain" else ".fq.gz"
            ins = [os.path.join(tmp, f"in_R{m}{ext}") for m in (1, 2)]
            t0 = time.time()
            bench_files.write_fixture(ins, pairs, {"plain": False, "gz": "bgzf", "gzip": "gzip"}[variant], threads)
            gen_s = time.time() - t0
            res = {"pairs": pairs, "input_bytes": sum(os.path.getsize(p) for p in ins), "fixture_s": gen_s}
            hashes = {}
            for nd in sorted({1, n_devices}):
                outs = {"trimmed": [os.path.join(tmp, f"out{nd}_trimmed_R{m}{ext}") for m in (1, 2)],
                        "short": [os.path.join(tmp, f"out{nd}_short_R{m}{ext}") for m in (1, 2)]}
                best = None
                for rep in range(2):
                    for q in outs["trimmed"] + outs["short"]:  # a fresh run writes new files
                        if os.path.exists(q):
                            os.remove(q)
                    t0 = time.time()
                    counters, timing = native.run_files(prog, ins, outs, gpus=nd, threads=threads)
                    wall = time.time() - t0
                    if best is None or wall < best[0]:
                        best = (wall, timing, counters)
                wall, timing, counters = best
                hashes[nd] = bench_files.hash_outputs(outs["trimmed"] + outs["short"], variant != "plain")
                res[f"n{nd}"] = {"pairs_per_s": pairs / wall, "wall_s": wall, "read_inflate_s": timing.read_inflate,
                                 "gpu_h2d_kernels_d2h_s": timing.h2d_kernels_d2h, "gpu_kernels_s": timing.kernels,
                                 "deflate_write_s": timing.write_deflate, "written_pairs": int(counters.written),
                                 "output_bytes": sum(os.path.getsize(p) for p in outs["trimmed"] + outs["short"])}
                for p in outs["trimmed"] + outs["short"]:
                    if os.path.exists(p):
                        os.remove(p)
            res["pairs_per_s"] = res[f"n{n_devices}"]["pairs_per_s"]
            res["sha256"] = hashes[n_devices]
            res["same_as_1gpu"] = hashes[n_devices] == hashes[1]
            out[variant] = res
            for p in ins:
                if os.path.exists(p):
                    os.remove(p)
        out["note"] = ("whole runs incl. plan set-up and pinned allocations; stage seconds are busy times of overlapping stages; "
                       "sha256 over the (decompressed) bytes of trimmed_R1, trimmed_R2, short_R1, short_R2; "
                       "gz: input = BGZF members (64 KiB blocks, level 1, inflated on the device); gzip: input = ordinary gzip, one member "
                       "per 4 M pairs at level 6 (one DEFLATE stream, decoded by the host threads in parallel: csrc/pinflate.cpp); "
                       ".gz output = concatenated gzip members made on the device")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return out


def e2e_gz_leg(args, prog, plan_flags, device, batches, P, B, world, barrier, max_over_ranks, bgzf_in=True):
    """csq_submit_bgzf / csq_wait with CSQ_PLAN_GZIP_OUT: the two pinned text batches of the e2e leg, compressed once on the
    host into BGZF members (64 KiB, zlib level 1 - what bgzip or this library's own writer produces), go through the
    device inflate, the chain and the device deflate; compressed bytes only cross PCIe in both directions.
    bgzf_in=False: the pinned FASTQ text goes up as it is (csq_submit_text) and only the outputs are gzip members - plain
    files in, the reference's default .fastq.gz out: the upload has the link to itself."""
    import ctypes as C

    import numpy as np
    import torch

    from cutseq_b200 import _abi as A
    from cutseq_b200 import native
    from scripts import bench_files

    threads = max(2, (os.cpu_count() or 4) // max(1, world))
    inputs = []  # per batch: (csq_batch_bgzf, keep-alive)
    comp_bytes = 0
    for tb in batches if bgzf_in else []:
        b = A.csq_batch_bgzf()
        b.n_reads, b.n_mates, b.first_record = P, 2, tb.c.first_record
        keep = []
        for m in range(2):
            text = memoryview(tb.keep[m].numpy())
            z = bench_files.bgzf_compress(text, threads)
            run = native.BgzfRun(z)
            pinned = torch.empty(len(z) + 64, dtype=torch.uint8, pin_memory=True)
            pinned[: len(z)] = torch.frombuffer(bytearray(z), dtype=torch.uint8)
            b.mate[m] = run.c
            b.mate[m].data = pinned.data_ptr()
            keep += [run, pinned]
            comp_bytes += len(z) if tb is batches[0] else 0
        inputs.append((b, keep))
    plan = native.Plan(prog, device, plan_flags | A.PLAN_GZIP_OUT)
    try:
        text_bytes = int(sum(batches[0].c.mate[m].bytes for m in range(2)))
        cap = text_bytes // 3 + 4096
        n_fly = 3
        outs, keep_out = [], []
        for s in range(n_fly):
            out = A.csq_batch_out()
            for d in range(A.CSQ_N_DEST):
                for m in range(2):
                    size = cap if d == 0 else cap // 4
                    buf = torch.empty(size, dtype=torch.uint8, pin_memory=True)
                    keep_out.append(buf)
                    out.text[d][m].data = buf.data_ptr()
                    out.text[d][m].capacity = size
            outs.append(out)

        def run_batches(k):
            d2h, submitted = 0, 0
            for i in range(k):
                while submitted < k and submitted < i + n_fly:
                    if bgzf_in:
                        native.check(native.lib().csq_submit_bgzf(plan._h, submitted % n_fly, C.byref(inputs[submitted % len(inputs)][0]), C.byref(outs[submitted % n_fly])))
                    else:
                        plan.submit_text(submitted % n_fly, batches[submitted % len(batches)].c, outs[submitted % n_fly])
                    submitted += 1
                plan.wait(i % n_fly)
                o = outs[i % n_fly]
                d2h += sum(o.text[d][m].bytes for d in range(A.CSQ_N_DEST) for m in range(2))
            return d2h

        steps = max(2, min(args.steps, 12))
        run_batches(3)
        barrier()
        w0 = time.perf_counter()
        d2h = run_batches(steps * B)
        torch.cuda.synchronize()
        w1 = time.perf_counter()
        barrier()
        dt = max_over_ranks(w1 - w0)
        return {"value": world * steps * B * P / dt, "unit": UNIT, "h2d_bytes_per_step": (comp_bytes if bgzf_in else text_bytes) * B,
                "d2h_bytes_per_step": int(d2h // steps),
                "ms_per_step": dt / steps * 1e3, "steps": steps, "text_bytes_per_step": text_bytes * B,
                "input": "BGZF members (zlib level 1, 0xFF00-byte pieces), inflated on the device, one warp per member" if bgzf_in
                         else "pinned FASTQ text (csq_submit_text)",
                "output": "gzip members (BGZF framing, dynamic-Huffman literal coding) encoded on the device",
                "timing": f"wall clock between device-synchronised points, {n_fly} batches in flight through "
                          f"{'csq_submit_bgzf' if bgzf_in else 'csq_submit_text'}/csq_wait, max over ranks"}
    finally:
        plan.close()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    prog = takara_program()
    ref = real_reference_available()
    if ref:
        sample = 400_000
        value, threads, step_s = cpu_leg_real(ref, max(1, min(args.steps, 3)), sample)
        kind, what = "reference", f"real cutseq (cutadapt {ref['cutadapt']}) -t {threads} on FASTQ files of the config-2 generator, parse and write included"
    else:
        sample = 200_000
        value, threads, step_s = cpu_leg(prog, args.steps, min(args.warmup, 1), sample)
        kind, what = "port", ("oracle/cutseq_oracle.c (restated cutadapt chain; the reference needs the absent cutadapt package), "
                              "gzip/parse excluded")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": step_s * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int32", "data": "synthetic",
        "config": {"workload": f"config2: synthetic 2x150 read pairs, cutseq {' '.join(ARGV)}; step = {sample} pairs (bounded sample of the 10M-pair workload)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind,
                         "sample": f"{args.steps} x {sample} pairs of the config-2 generator, {what}",
                         "cutadapt_importable": bool(ref)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=60, help="timed steps of the headline (resident) leg; a step is one pass over the 10M-pair workload "
                    "(default: ~1 s timed). The end-to-end legs time the same count clamped to 2..12 steps and report it "
                    "in their own \"steps\"")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch-pairs", type=int, default=BATCH_PAIRS)
    ap.add_argument("--batches", type=int, default=N_BATCHES)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-numa", action="store_true", help="do not bind the rank to the GPU's NUMA node (A/B runs)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-e2e-gz", action="store_true", help="skip the end-to-end leg with compressed host buffers (BGZF in, gzip out)")
    ap.add_argument("--no-files", action="store_true", help="skip the whole-file leg (FASTQ files on disk -> csq_run_files -> files)")
    ap.add_argument("--file-pairs", type=int, default=20_000_000, help="pairs in the plain whole-file leg (config 5: streamed, <= 20M-pair on-disk file)")
    ap.add_argument("--file-pairs-gz", type=int, default=20_000_000, help="pairs in the .gz whole-file leg")
    ap.add_argument("--file-pairs-gzip", type=int, default=4_000_000, help="pairs in the ordinary-gzip whole-file leg (single-member input)")
    ap.add_argument("--no-prefilter", action="store_true", help="exact DP on every read (CSQ_PLAN_NO_PREFILTER)")
    ap.add_argument("--emit", default="stage", choices=["stage", "g16"], help="emit kernel (A/B runs); stage (k_emit_stage, through shared memory) is the product default")
    ap.add_argument("--no-exact-stop", action="store_true", help="exact DP walks on after an error-free full match (CSQ_PLAN_NO_EXACT_STOP, A/B runs)")
    ap.add_argument("--one-stream", action="store_true", help="mate chains on one stream (CSQ_PLAN_ONE_STREAM), for A/B runs")
    ap.add_argument("--input", default="text", choices=["text", "soa"], help="batch form handed to the library")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy "
                    "(rank 0's batches; sizes and sha256 of every output stream, a seeded sample of reads and text)")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)

    # stdout carries exactly ONE JSON line: anything libraries print there (e.g. NCCL's version banner)
    # is sent to stderr by pointing fd 1 at fd 2 until the result is written to the saved descriptor.
    sys.stdout.flush()
    result_fd = os.dup(1)
    os.dup2(2, 1)

    import torch

    from cutseq_b200 import _abi as A
    from cutseq_b200 import build, native

    from cutseq_b200 import dist as csq_dist

    group = csq_dist.Group()  # NCCL process group when launched by torchrun with WORLD_SIZE > 1
    rank, local_rank, world = group.rank, group.local_rank, group.world
    torch.cuda.set_device(local_rank)
    build.build()
    native.lib()  # fails loudly when the CUDA library is missing
    # one process per GPU: this rank's threads and pinned buffers stay on the GPU's NUMA node (-1: nothing to bind to)
    numa_node = -1 if args.no_numa else native.bind_host_to_device(local_rank)

    def barrier():
        torch.cuda.synchronize()
        group.barrier()
        torch.cuda.synchronize()

    max_over_ranks = group.max

    prog = takara_program()
    P, B = args.batch_pairs, args.batches
    plan_flags = ((A.PLAN_NO_PREFILTER if args.no_prefilter else 0) | {"stage": 0, "g16": A.PLAN_EMIT_G16}[args.emit]
                  | (A.PLAN_ONE_STREAM if args.one_stream else 0) | (A.PLAN_NO_EXACT_STOP if args.no_exact_stop else 0))
    plan = native.Plan(prog, local_rank, plan_flags)
    # this rank's contiguous index range of the workload: [rank*B*P, (rank+1)*B*P)
    # Host copies: batches 0 and 1 stay in pinned memory for the end-to-end leg; later batches reuse one
    # staging buffer (csq_upload is synchronous), so a rank pins three batches, not B.
    batches = []
    text_mode = args.input == "text"
    for b in range(B):
        batch = native.synth_batch(2, P, first_index=(rank * B + b) * P, buffer=min(b, 2))
        if text_mode:  # the FASTQ bytes of the batch, as a file would hold them, in pinned host memory
            texts = []
            for m in range(2):
                mi = batch.mate[m]
                buf = torch.empty(int(mi.name_bytes) + 2 * int(mi.seq_bytes) + 6 * P + 64, dtype=torch.uint8, pin_memory=True)
                n_bytes = native.format_fastq(batch, m, out=buf).numel()
                texts.append(buf[:n_bytes])
            tb = native.TextBatch(texts, P, first_record=(rank * B + b) * P)
            plan.upload_text(b, tb.c)
            if b < 2:
                batches.append(tb)
        else:
            plan.upload(b, batch)
            if b < 2:
                batches.append(batch)
    slots = list(range(B))

    def in_bytes(bt):
        return int(sum(bt.c.mate[m].bytes for m in range(2))) if text_mode else h2d_bytes(bt)

    def submit(slot, bt, out):
        if text_mode:
            plan.submit_text(slot, bt.c, out)
        else:
            plan.submit(slot, bt, out)

    # ---- kernel throughput, inputs resident in HBM: a step = the B resident batches, one after the other ----
    if args.warmup > 0:
        plan.run_steps(slots, args.warmup * B)
    c0 = plan.stats()
    l0 = plan.launch_count()
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    t0 = time.time()
    ms = plan.run_steps(slots, args.steps * B)  # untimed sizing pass inside, then K x B batches between two CUDA events
    t1 = time.time()
    barrier()
    launches = plan.launch_count() - l0
    c1 = plan.stats()
    job_counters = group.sum_counters(c1)  # the one reduction of trim statistics (NCCL all-reduce when N > 1)
    ktimes = plan.kernel_times(slots[0])
    ms = max_over_ranks(ms)
    value = world * args.steps * B * P / (ms * 1e-3)
    # csq_run_steps = B sizing batches + K*B timed batches + 1 per-kernel profiling batch; only the timed ones count
    n_passes = args.steps * B + B + 1
    per_batch_launches = launches // n_passes
    timed_launches = per_batch_launches * args.steps * B

    def cells(c):
        return sum(sum(c.dp_cells[m]) for m in range(2))

    cells_per_batch = (cells(c1) - cells(c0)) / n_passes
    step_ms = ms / args.steps
    gcups_nominal = cells_per_batch * B / (step_ms * 1e-3) / 1e9
    clocks = sampler.stop(t0, t1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, plan, slots, P, rank * B * P, int(in_bytes(batches[0]) // 2 + 64 * P + 4096))

    # ---- end to end through the C ABI with host buffers (H2D + kernels + D2H timed); a step = B batches ----
    e2e = None
    roofline_e2e = None
    if not args.no_e2e:
        cap = int(in_bytes(batches[0]) // 2 + 64 * P + 4096)
        outs, keep = [], []
        n_e2e = 3 if B + 2 < A.CSQ_N_SLOTS else 2  # batches in flight: keeps the H2D engine busy while a D2H drains
        for s in range(n_e2e):
            out = A.csq_batch_out()
            for d in range(A.CSQ_N_DEST):
                for m in range(2):
                    size = cap if d == 0 else cap // 4
                    buf = torch.empty(size, dtype=torch.uint8, pin_memory=True)
                    keep.append(buf)
                    out.text[d][m].data = buf.data_ptr()
                    out.text[d][m].capacity = size
            outs.append(out)
        e2e_slots = [B + i for i in range(n_e2e)] if B + n_e2e <= A.CSQ_N_SLOTS else list(range(n_e2e))

        def e2e_batches(k):
            """k batches, up to n_e2e in flight (submit of batch i+n-1 is issued before the wait of batch i)."""
            d2h = 0
            submitted = 0
            for i in range(k):
                while submitted < k and submitted < i + n_e2e:
                    submit(e2e_slots[submitted % n_e2e], batches[submitted % len(batches)], outs[submitted % n_e2e])
                    submitted += 1
                plan.wait(e2e_slots[i % n_e2e])
                o = outs[i % n_e2e]
                d2h += sum(o.text[d][m].bytes for d in range(A.CSQ_N_DEST) for m in range(2))
            return d2h

        e2e_steps = max(2, min(args.steps, 12))  # 12 steps = 120 M pairs, ~2 s: enough for a copy-bound rate
        e2e_batches(max(2, min(args.warmup, 3)))
        barrier()
        w0 = time.perf_counter()
        d2h = e2e_batches(e2e_steps * B)
        torch.cuda.synchronize()
        w1 = time.perf_counter()
        barrier()
        e2e_s = max_over_ranks(w1 - w0)
        e2e = {"value": world * e2e_steps * B * P / e2e_s, "unit": UNIT, "h2d_bytes_per_step": in_bytes(batches[0]) * B,
               "d2h_bytes_per_step": int(d2h // e2e_steps), "ms_per_step": e2e_s / e2e_steps * 1e3, "steps": e2e_steps,
               "timing": f"wall clock between device-synchronised points, {n_e2e} batches in flight through csq_submit_text/csq_wait, max over ranks"}
        # the ceiling of this path: the same byte counts per batch as plain pinned copies, both directions at once,
        # every rank between the same barriers (the ranks of one box share its PCIe root / host memory)
        try:
            hb, db = in_bytes(batches[0]), int(d2h // (e2e_steps * B))
            native.pcie_peak(local_rank, hb, db, reps=1, mode=2)
            barrier()
            up, down = native.pcie_peak(local_rank, hb, db, reps=4, mode=2)
            barrier()
            t_ceiling = max_over_ranks(hb / (up * 1e9))  # seconds per batch of the slowest rank (both directions share the time)
            ceiling_pairs = world * P / t_ceiling
            roofline_e2e = {"bound": "pcie (pinned host <-> device copies, both directions at once)", "achieved": e2e["value"], "peak": ceiling_pairs,
                            "unit": UNIT, "frac": e2e["value"] / ceiling_pairs, "h2d_GBps_ceiling": up, "d2h_GBps_ceiling": down,
                            "h2d_GBps_achieved": e2e["h2d_bytes_per_step"] / (e2e["ms_per_step"] * 1e-3) / 1e9,
                            "d2h_GBps_achieved": e2e["d2h_bytes_per_step"] / (e2e["ms_per_step"] * 1e-3) / 1e9,
                            "how": "csq_pcie_peak(mode 2): cudaMemcpyAsync of one batch's input bytes up and output bytes down, 4 repetitions, "
                                   "all ranks at once; peak = pairs/s if the chain cost nothing but those copies (rank 0's GB/s shown, time = max over ranks)"}
        except native.NativeError as exc:
            roofline_e2e = {"error": str(exc)}

    # ---- the same end to end with COMPRESSED host buffers: BGZF members in (device inflate), gzip members out (device
    # deflate) - what the reference's default .fastq.gz files hold; ~1/3 of the bytes cross PCIe ----
    e2e_gz = e2e_gzout = None
    if not args.no_e2e and not args.no_e2e_gz and text_mode:
        try:
            e2e_gz = e2e_gz_leg(args, prog, plan_flags, local_rank, batches, P, B, world, barrier, max_over_ranks)
        except Exception as exc:
            e2e_gz = {"error": repr(exc)}
        try:  # plain text up, gzip members down
            e2e_gzout = e2e_gz_leg(args, prog, plan_flags, local_rank, batches, P, B, world, barrier, max_over_ranks, bgzf_in=False)
        except Exception as exc:
            e2e_gzout = {"error": repr(exc)}

    native.unbind_host()  # the host legs below (files, CPU baseline) use every core of the box
    if rank != 0:
        plan.close()
        torch.cuda.synchronize()
        # rank 0 drives every GPU of the job in the files leg: wait here so that the job ends together - on the host
        # (a GPU barrier would spin on this rank's GPU while rank 0's file run needs it)
        group.host_wait("csq_files_leg_done")
        group.close()
        return 0

    # ---- roofline of the dominant kernel (per-kernel CUDA events of one untimed batch behind the timed region) ----
    alu_peak, mixed_peak = native.int_peak(local_rank)
    dom_name, dom_ms = max(ktimes, key=lambda kv: kv[1]) if ktimes else ("n/a", 0.0)
    hbm_peak, hbm_src = 6650.0, "fallback (B200_PROFILING.md)"
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            hbm_peak, hbm_src = json.load(f)["hbm_gbs"], "measured (MEASURED_PEAKS.json, copy read+write)"
    except Exception:
        pass
    d2h_per_batch = e2e["d2h_bytes_per_step"] // B if e2e else int(0.78 * in_bytes(batches[0]))
    emit_bytes = in_bytes(batches[0]) + d2h_per_batch  # input records read once + FASTQ text written once (~1.27 KB / pair)
    emit_ms = sum(kms for name, kms in ktimes if name == "k_emit")
    roofline = {"bound": "hbm", "kernel": {"stage": "k_emit_stage", "g16": "k_emit<16>"}[args.emit],
                "achieved": (emit_bytes / (emit_ms * 1e-3) / 1e9) if emit_ms else None, "peak": hbm_peak, "unit": "GB/s",
                "peak_source": hbm_src, "traffic": None, "ms": emit_ms, "share_of_step": emit_ms * B / step_ms if step_ms else None,
                "how": "algorithmic bytes per launch (the batch's FASTQ text read once + the trimmed FASTQ text written once) / CUDA-event "
                       "duration of that launch (one untimed batch, events on the launching stream)"}
    if roofline["achieved"]:
        roofline["frac"] = roofline["achieved"] / hbm_peak
    src_hash = kernel_sources_hash()
    try:  # DRAM bytes of one launch from the committed ncu capture (per pair, scaled to this batch size) - only if the sources still match
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            tr = json.load(f)
        if tr.get("sources_sha256_16") == src_hash:
            roofline["traffic"] = tr[{"stage": "k_emit", "g16": "k_emit_g16"}[args.emit]]["dram_bytes_per_pair"] * P
            roofline["traffic_source"] = tr["source"]
        else:
            roofline["traffic_source"] = "committed ncu capture is older than the kernel sources: not shown"
    except Exception:
        pass
    # integer side: time of every ALIGN op (prefilter + exact DP) and nominal GCUPS; executed lane-ops only from a capture of THESE sources
    align_ops = []
    for name, kms in ktimes:
        if name.startswith("k_prefilter"):
            align_ops.append([name.replace("k_prefilter", "k_prefilter+k_align"), kms, True])
        elif name.startswith("k_align"):
            if align_ops and align_ops[-1][2]:
                align_ops[-1][1] += kms
                align_ops[-1][2] = False
            else:
                align_ops.append([name, kms, False])
    align_cells = []
    for m, ops in enumerate((prog.ops_r1, prog.ops_r2)):
        for t, op in enumerate(ops):
            if op.kind == A.OP_ALIGN:
                align_cells.append((c1.dp_cells[m][t] - c0.dp_cells[m][t]) / n_passes)
    dp_kernels = [{"kernel": name, "ms": kms, "nominal_gcups": cl / (kms * 1e-3) / 1e9 if kms > 0 else None}
                  for (name, kms, _), cl in zip(align_ops, align_cells)]
    roofline_dp_executed = None
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            tr = json.load(f)
        if tr.get("sources_sha256_16") == src_hash and dp_kernels and not args.no_prefilter:
            dom = max(dp_kernels, key=lambda r: r["ms"])
            kind = dom["kernel"][dom["kernel"].index("("):]
            lane_ops = tr["dp_lane_ops_per_read"]["k_prefilter" + kind] + tr["dp_lane_ops_per_read"]["k_align" + kind]
            achieved = lane_ops * P / (dom["ms"] * 1e-3) / 1e9
            peak = max(alu_peak, mixed_peak) / 1e9
            roofline_dp_executed = {"bound": "int_issue", "kernel": dom["kernel"], "achieved": achieved, "peak": peak, "unit": "Gop/s",
                                    "frac": achieved / peak, "sources_sha256_16": src_hash,
                                    "how": "executed integer lane-ops per read (smsp__inst_executed x 32, " + tr["source"] + ") x reads per launch / "
                                           "live CUDA-event duration; peak = csq_int_peak measured live (ALU + FMA pipe mix)"}
    except Exception:
        pass

    # ---- whole files: read / inflate, GPU chain, deflate / write (rank 0 drives all GPUs of the job) ----
    files = None
    if not args.no_files:
        try:
            files = files_leg(prog, args.file_pairs, args.file_pairs_gz, world, os.cpu_count() or 4, pairs_gzip=args.file_pairs_gzip)
        except Exception as exc:  # the headline numbers must not die with a full /tmp
            files = {"error": repr(exc)}
    group.host_signal("csq_files_leg_done")

    cpu = None
    if not args.no_cpu and world == 1:
        v, threads, step_s = cpu_leg(prog, 3, 1, 100_000)
        cpu = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": "3 x 100000 pairs of the same config-2 generator through oracle/cutseq_oracle.c (restated cutadapt chain), "
                         "gzip/parse excluded"}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32",
        "data": "synthetic",
        "config": {"workload": f"config2: synthetic 2x150 read pairs, cutseq {' '.join(ARGV)}; step = {B} resident batches x {P} pairs per GPU "
                               f"(= {B * P} pairs); consecutive batches are different data "
                               f"({in_bytes(batches[0]) / 1e9:.2f} GB in each, far larger than the 126 MB L2, no flush needed); "
                               f"input form: {'raw FASTQ text, record index built on the device' if text_mode else 'host-parsed SoA'}",
                   "parallelism": f"dp{world} (contiguous index ranges per GPU, no collective on the data path)",
                   "prefilter": not args.no_prefilter, "emit": args.emit, "exact_stop": not args.no_exact_stop, "numa_node": numa_node},
        "nominal_gcups": gcups_nominal, "cells_per_pair": cells_per_batch / P,
        "roofline": roofline, "roofline_e2e": roofline_e2e, "roofline_dp_executed": roofline_dp_executed,
        "int_peak_Gops": {"alu_only": alu_peak / 1e9, "alu_fma_mix": mixed_peak / 1e9},
        "kernels": [{"kernel": n, "ms": t} for n, t in ktimes], "kernels_note": "one batch of the step, one stream, CUDA event after every kernel",
        "dp_kernels": dp_kernels, "cpu_baseline": cpu, "e2e": e2e, "e2e_gz": e2e_gz, "e2e_gzout": e2e_gzout, "files": files, "gpu_launches": int(timed_launches), "clocks": clocks,
        "job_counters": {"pairs": int(job_counters.n), "written": int(job_counters.written), "too_short": int(job_counters.too_short)},
        "sources_sha256_16": src_hash,
    }
    sys.stdout.flush()
    os.write(result_fd, (json.dumps(line) + "\n").encode())
    plan.close()
    group.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
