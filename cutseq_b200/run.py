"""Command line and run driver: cutseq's CLI surface on top of the B200 chain.

Mirror of the reference ``cutseq/run.py``:

* ``main``              run.py:866-1109  (flags, scheme lookup, output naming)
* ``run_cutseq``        run.py:815-863
* ``pipeline_single``   run.py:305-490   (same signature)
* ``pipeline_paired``   run.py:493-812   (same signature)
* ``CutadaptConfig``    run.py:198-219

Where the reference builds cutadapt modifier objects and runs them read by read, this
module compiles the same operation order into an op program (``program.py``) and hands
whole files to the native library (``csq_run_files``), which parses FASTQ on the host,
runs the chain on the GPU(s) and writes the outputs in input order.  There is no CPU
fallback: without the CUDA library / a B200 the run fails.
"""

from __future__ import annotations

import argparse
import json
import logging
import re
import sys

from . import __version__, program
from .common import BUILDIN_ADAPTERS, BarcodeConfig, print_builtin_adapters, remove_fq_suffix

logging.basicConfig(level=logging.INFO, format="%(asctime)s -  %(levelname)s - %(message)s")


class CutadaptConfig:
    """Settings bag with the reference's field names and defaults (run.py:206-219)."""

    def __init__(self):
        self.rname_suffix = False
        self.ensure_inline_barcode = False
        self.trim_polyA = False
        self.trim_polyA_wo_direction = False
        self.conditional_cutter = True
        self.min_length = 20
        self.min_quality = 20
        self.auto_rc = False
        self.dry_run = False
        self.threads = 1
        self.json_file = None
        self.force_trim_min_length = 50
        self.force_anywhere = False
        # additions of this implementation
        self.gpus = 1
        self.batch_reads = 0


def _emit_notes(prog):
    for note in prog.notes:
        level, _, text = note.partition(":")
        (logging.warning if level == "WARNING" else logging.info)(text)


def minimal_report_text(counters, prog) -> str:
    """cutadapt ``minimal_report`` table from the device counters.

    With several AdapterCutters per mate cutadapt's ``Statistics._collect_modifier``
    asserts on the second one; the reference swallows that (run.py:58-73), so
    ``w/adapters`` is the count of the FIRST AdapterCutter of each mate only.
    """
    from . import _abi as A

    def first_align(ops):
        for i, op in enumerate(ops):
            if op.kind == A.OP_ALIGN:
                return i
        return None

    def w_adapters(mate, ops):
        i = first_align(ops)
        return int(counters.with_adapters[mate][i]) if i is not None else 0

    header = ["status", "in_reads", "in_bp", "too_short", "too_long", "too_many_n", "out_reads", "w/adapters", "qualtrim_bp", "out_bp"]
    total_bp = int(counters.total_bp[0]) + (int(counters.total_bp[1]) if prog.paired else 0)
    fields = ["OK", int(counters.n), total_bp, int(counters.too_short), 0, 0, int(counters.written),
              w_adapters(0, prog.ops_r1), int(counters.quality_trimmed_bp[0]), int(counters.written_bp[0])]
    if prog.paired:
        header += ["w/adapters2", "qualtrim_bp2", "out2_bp"]
        fields += [w_adapters(1, prog.ops_r2), int(counters.quality_trimmed_bp[1]), int(counters.written_bp[1])]
    return "\t".join(header) + "\n" + "\t".join(str(x) for x in fields)


_ADAPTER_TYPES = None


def _adapter_types():
    """csq adapter kind -> (cutadapt ``descriptive_identifier``, is 5' end).  Recalled from cutadapt 5.x adapters.py
    (unverified here, like everything below the boundary: DESIGN.md section 2)."""
    global _ADAPTER_TYPES
    if _ADAPTER_TYPES is None:
        from . import _abi as A

        _ADAPTER_TYPES = {
            A.AD_FRONT: ("regular_five_prime", True), A.AD_RIGHTMOST_FRONT: ("rightmost_five_prime", True),
            A.AD_NI_FRONT: ("noninternal_five_prime", True), A.AD_PREFIX: ("anchored_five_prime", True),
            A.AD_BACK: ("regular_three_prime", False), A.AD_BACK_ANYWHERE: ("regular_three_prime", False),
            A.AD_NI_BACK: ("noninternal_three_prime", False), A.AD_SUFFIX: ("anchored_three_prime", False),
        }
    return _ADAPTER_TYPES


def _error_lengths(length: int, rate: float):
    """cutadapt ``ErrorRanges(length, error_rate).lengths()``: the last overlap length of every allowed-error count
    but the final one (rate 0.2, 20 nt: 0 errors up to 4, 1 up to 9, 2 up to 14, 3 up to 19 -> [4, 9, 14, 19])."""
    out, prev = [], 0
    for n in range(1, length + 1):
        k = int(n * rate)
        if k != prev:
            out.append(n - 1)
            prev = k
    return out


def _adjacent_bases(counters, mate):
    """cutadapt ``EndStatistics.adjacent_bases`` of a 3' end: the read base in front of every match; a match at the
    read start and a base outside ACGT both count under "" (cutadapt's ``except KeyError: adjacent_bases[""] = 1``
    resets that entry instead of adding to it - a result that depends on how reads fall into worker chunks; the sum
    is reported here)."""
    a = counters.adjacent_bases[mate]
    return {"A": int(a[0]), "C": int(a[1]), "G": int(a[2]), "T": int(a[3]), "": int(a[4]) + int(a[5])}


def _dominant_adjacent_base(adjacent):
    """cutadapt ``EndStatistics`` report rule: the base (or "none/other") in front of more than 80 % of at least 20
    matches, else None."""
    total = sum(adjacent.values())
    if total < 20:
        return None
    for base in ("A", "C", "G", "T", ""):
        if adjacent[base] / total > 0.8:
            return base if base else "none/other"
    return None


def _adapter_entries(counters, mate, ops):
    """``adapters_read1`` / ``adapters_read2`` of cutadapt's ``Statistics.as_json()``.  With several AdapterCutters
    per mate only the FIRST one reaches the statistics (the reference swallows the assertion of the second,
    run.py:58-73); cutadapt numbers unnamed adapters "1", "2", ... in the order run.py creates them, so the first
    cutter of mate 1 holds adapter "1" and that of mate 2 adapter "2" (single-end: "1").  The reference empties
    ``trimmed_lengths`` (run.py:286-301); a 5' end keeps no adjacent-base statistics."""
    from . import _abi as A

    for i, op in enumerate(ops):
        if op.kind != A.OP_ALIGN:
            continue
        kind, five = _adapter_types()[op.adapter_kind]
        anchored = op.adapter_kind in (A.AD_PREFIX, A.AD_SUFFIX)
        end = {
            "type": kind, "sequence": op.adapter, "error_rate": op.max_error_rate, "indels": True,
            "error_lengths": None if anchored else _error_lengths(len(op.adapter), op.max_error_rate),
            "matches": int(counters.with_adapters[mate][i]), "adjacent_bases": None if five else _adjacent_bases(counters, mate),
            "dominant_adjacent_base": None if five else _dominant_adjacent_base(_adjacent_bases(counters, mate)),
            "trimmed_lengths": [],
        }
        return [{"name": str(mate + 1), "total_matches": end["matches"], "on_reverse_complement": None, "linked": False,
                 "five_prime_end": end if five else None, "three_prime_end": None if five else end}]
    return []


def json_report(file, counters, prog, barcode, input1, input2, output1, output2, short1, short2, untrimmed1, untrimmed2):
    """``--json-file`` (reference run.py:222-302): paths, barcode dict and ``stats.as_json()`` - read / base-pair
    counters and the adapter entries in cutadapt's layout (recalled, see ``_adapter_entries``); per-length
    histograms are not collected (the reference throws them away)."""
    from . import _abi as A

    paired = bool(input2)
    total_bp = int(counters.total_bp[0]) + (int(counters.total_bp[1]) if paired else 0)
    qt = [int(counters.quality_trimmed_bp[0]), int(counters.quality_trimmed_bp[1]) if paired else None]
    has_qtrim = [any(op.kind == A.OP_QTRIM for op in ops) for ops in (prog.ops_r1, prog.ops_r2 if paired else [])] + [False]
    qt = [q if (q is not None and has_qtrim[i]) else None for i, q in enumerate(qt)]
    entries = [_adapter_entries(counters, 0, prog.ops_r1), _adapter_entries(counters, 1, prog.ops_r2) if paired else None]
    d = {
        "tag": "Cutadapt report",
        "cutadapt_version": f"cutseq_b200 {__version__}",
        "input": {"path1": input1, "path2": input2, "paired": paired},
        "output": {"output1": output1, "output2": output2, "short1": short1, "short2": short2,
                   "untrimmed1": untrimmed1, "untrimmed2": untrimmed2},
        "barcode": barcode.to_dict(),
        "read_counts": {
            "input": int(counters.n),
            # cutadapt lists its own filters (None = not used); cutseq's IsUntrimmedAny predicate is not one of them,
            # its count is kept under its descriptive identifier
            "filtered": {"too_short": int(counters.too_short), "too_long": None, "too_many_n": None,
                         "too_many_expected_errors": None, "casava_filtered": None, "discard_trimmed": None,
                         "discard_untrimmed": None, "is_untrimmed_any": int(counters.untrimmed)},
            "output": int(counters.written),
            "reverse_complemented": None,
            "read1_with_adapter": entries[0][0]["total_matches"] if entries[0] else None,
            "read2_with_adapter": (entries[1][0]["total_matches"] if entries[1] else None) if paired else None,
        },
        "basepair_counts": {
            "input": total_bp,
            "input_read1": int(counters.total_bp[0]),
            "input_read2": int(counters.total_bp[1]) if paired else None,
            "quality_trimmed": sum(q for q in qt if q is not None) if any(q is not None for q in qt) else None,
            "quality_trimmed_read1": qt[0],
            "quality_trimmed_read2": qt[1],
            "poly_a_trimmed": None,
            "poly_a_trimmed_read1": None,
            "poly_a_trimmed_read2": None,
            "output": int(counters.written_bp[0]) + (int(counters.written_bp[1]) if paired else 0),
            "output_read1": int(counters.written_bp[0]),
            "output_read2": int(counters.written_bp[1]) if paired else None,
        },
        "adapters_read1": entries[0],
        "adapters_read2": entries[1],
        "poly_a_trimmed_read1": None,
        "poly_a_trimmed_read2": None,
    }
    with open(file, "w") as fh:
        fh.write(json.dumps(d, indent=2))


def _run_program(prog, inputs, outputs, settings):
    from . import _abi as A
    from . import native
    from .transcode import Transcoders

    # .bz2 / .xz files (xopen handles them in the reference) go through named pipes and Python's codecs; FASTA files
    # are parsed and written by the library itself (CSQ_PLAN_FASTA)
    with Transcoders(inputs, outputs, fasta_native=True) as tc:
        return native.run_files(prog, tc.inputs, tc.outputs, gpus=getattr(settings, "gpus", 1),
                                threads=settings.threads, batch_reads=getattr(settings, "batch_reads", 0),
                                flags=A.PLAN_FASTA if tc.fasta_native else 0)


def pipeline_single(input1, output1, short1, untrimmed1, barcode, settings):
    """Single-end run (reference run.py:305-490)."""
    prog = program.compile_single(barcode, settings, untrimmed1)
    _emit_notes(prog)
    if settings.dry_run:
        for line in prog.describe():
            print(line)
        return None
    counters, timing = _run_program(prog, [input1], {"trimmed": [output1], "short": [short1], "untrimmed": [untrimmed1]}, settings)
    if settings.json_file is not None:
        json_report(settings.json_file, counters, prog, barcode, input1, None, output1, None, short1, None, untrimmed1, None)
    print(minimal_report_text(counters, prog), file=sys.stderr)
    return counters


def pipeline_paired(input1, input2, output1, output2, short1, short2, untrimmed1, untrimmed2, barcode, settings):
    """Paired-end run (reference run.py:493-812)."""
    prog = program.compile_paired(barcode, settings, untrimmed1, untrimmed2)
    _emit_notes(prog)
    if settings.dry_run:
        for part in ("p5", "p7", "inline5", "inline3", "umi5", "umi3", "mask5", "mask3", "strand"):
            print(f"{part}: {getattr(barcode, part)}")
        for line in prog.describe():
            logging.info(line)
        return None
    counters, timing = _run_program(
        prog, [input1, input2],
        {"trimmed": [output1, output2], "short": [short1, short2], "untrimmed": [untrimmed1, untrimmed2]}, settings)
    if settings.json_file is not None:
        json_report(settings.json_file, counters, prog, barcode, input1, input2, output1, output2, short1, short2, untrimmed1, untrimmed2)
    print(minimal_report_text(counters, prog), file=sys.stderr)
    return counters


def settings_from_args(args) -> CutadaptConfig:
    s = CutadaptConfig()
    s.rname_suffix = args.with_rname_suffix  # accepted, has no effect (as in the reference)
    s.ensure_inline_barcode = args.ensure_inline_barcode
    s.trim_polyA = args.trim_polyA
    s.trim_polyA_wo_direction = args.trim_polyA_wo_direction
    s.conditional_cutter = args.conditional_cutter
    s.threads = args.threads
    s.min_length = args.min_length
    s.min_quality = args.min_quality
    s.dry_run = args.dry_run
    s.auto_rc = args.auto_rc
    s.json_file = args.json_file
    s.force_trim_min_length = args.force_trim_min_length
    s.force_anywhere = args.force_anywhere
    s.gpus = args.gpus
    s.batch_reads = args.batch_reads
    return s


def run_cutseq(args):
    """reference run.py:815-863"""
    barcode = BarcodeConfig(args.adapter_scheme)
    settings = settings_from_args(args)
    if len(args.input_file) == 1:
        return pipeline_single(args.input_file[0], args.output_file[0], args.short_file[0], args.untrimmed_file[0], barcode, settings)
    return pipeline_paired(
        args.input_file[0], args.input_file[1], args.output_file[0], args.output_file[1],
        args.short_file[0], args.short_file[1], args.untrimmed_file[0], args.untrimmed_file[1], barcode, settings)


def build_parser() -> argparse.ArgumentParser:
    """Same flags, defaults and meaning as the reference parser (run.py:874-1020); ``--gpus`` and
    ``--batch-reads`` are the only additions."""
    p = argparse.ArgumentParser(
        prog="cutseq",
        description="Trim sequencing adapters, barcodes, UMIs and masks from NGS reads on NVIDIA B200 GPUs "
        "(cutseq-compatible command line).",
        epilog="Limits (explicit errors, no CPU fallback): reads <= 895 bases, adapters <= 128, headers <= 65535 bytes; "
        "sm_100 GPUs only; .zst files need the zstandard module or the zstd program.",
    )
    p.add_argument("input_file", type=str, nargs="*", help="One (single-end) or two (paired-end) FASTQ files: plain, .gz (incl. bgzip), .bz2 or .xz.")
    p.add_argument("-a", "--adapter-scheme", type=str,
                   help="Library scheme, e.g. P5(INLINE5)NNNNXXX>XXXNNNN(INLINE3)P7: adapters, optional inline barcodes in "
                   "parentheses, N = UMI bases, X = masked bases, and the strand symbol > (forward), < (reverse) or - (unknown).")
    p.add_argument("-A", "--adapter-name", help="Name of a built-in scheme. choices:\n" + ",".join(BUILDIN_ADAPTERS.keys()))
    p.add_argument("-O", "--output-prefix", type=str,
                   help="Prefix for the trimmed/short/untrimmed output files; default: derived from the input file names.")
    p.add_argument("-o", "--output-file", type=str, nargs="+", help="Output file(s) for trimmed reads, one per input file.")
    p.add_argument("-s", "--short-file", type=str, nargs="+", help="Output file(s) for reads that end up shorter than --min-length.")
    p.add_argument("-u", "--untrimmed-file", type=str, nargs="+",
                   help="Output file(s) for reads in which an expected inline barcode was not found.")
    p.add_argument("--json-file", type=str, help="Write trimming statistics as JSON to this file.")
    p.add_argument("-q", "--min-quality", type=int, default=20, help="Quality cutoff for 3' quality trimming. (Default: 20)")
    p.add_argument("-m", "--min-length", type=int, default=20, help="Reads shorter than this after trimming go to the short file. (Default: 20)")
    p.add_argument("--with-rname-suffix", action="store_true",
                   help="Read names carry /1 /2 or .1 .2 suffixes (they are stripped in any case).")
    p.add_argument("--ensure-inline-barcode", action="store_true",
                   help="Send reads without the scheme's inline barcode(s) to the untrimmed files.")
    p.add_argument("--trim-polyA", action="store_true", help="Trim poly-A / poly-T tails.")
    p.add_argument("--trim-polyA-wo-direction", action="store_true",
                   help="Trim poly-A and poly-T on both mates regardless of the scheme's strand.")
    p.add_argument("--conditional-cutter", action=argparse.BooleanOptionalAction, default=True,
                   help="UMI/mask cuts on the far mate only happen if an adapter was found or the read is at least "
                   "--force-trim-min-length long (default); --no-conditional-cutter always cuts.")
    p.add_argument("--force-trim-min-length", type=int, default=50,
                   help="Read length from which conditional UMI/mask cuts are applied without an adapter match. (Default: 50)")
    p.add_argument("--force-anywhere", action="store_true", help="Let the 3' adapter match anywhere in the read.")
    p.add_argument("--auto-rc", action="store_true",
                   help="For '<' libraries: reverse complement single-end reads / swap R1 and R2 outputs of paired reads.")
    p.add_argument("-t", "--threads", type=int, default=1, help="Host threads for FASTQ (de)compression. (Default: 1)")
    p.add_argument("-n", "--dry-run", action="store_true", help="Print the operation list instead of running; writes nothing.")
    p.add_argument("-V", "--version", action="version", version=f"%(prog)s {__version__}")
    p.add_argument("--list-adapters", action="store_true", help="List the built-in schemes and exit.")
    p.add_argument("--gpus", type=int, default=1, help="Number of GPUs to shard batches over. (Default: 1)")
    p.add_argument("--batch-reads", type=int, default=0, help="Reads (pairs) per GPU batch; 0 = library default.")
    return p


def resolve_scheme(args) -> str:
    """-A / -a resolution and normalisation (reference run.py:1041-1056)."""
    if args.adapter_name is not None:
        if args.adapter_scheme is not None:
            logging.info("Adapter scheme is provided, ignoring adapter name.")
        else:
            args.adapter_scheme = BUILDIN_ADAPTERS.get(args.adapter_name.upper())
            if args.adapter_scheme is None:
                logging.error(f"Adapter name '{args.adapter_name} not found in built-in adapters.")
                args.adapter_scheme = args.adapter_name  # the reference falls back to using the name as scheme
    elif args.adapter_scheme is None:
        logging.error("Adapter scheme or name is required. Use -a or -A.")
        sys.exit(1)
    args.adapter_scheme = args.adapter_scheme.replace(" ", "").upper()
    return args.adapter_scheme


def _default_outputs(given, inputs, prefix, label):
    """Output naming rules of the reference (run.py:1058-1086)."""
    tails = [f"_{label}_R1.fastq.gz", f"_{label}_R2.fastq.gz"]
    if given:
        if len(given) != len(inputs):
            logging.error(f"Number of {label} output files ({len(given)}) must match number of input files ({len(inputs)}).")
            sys.exit(1)
        return given
    if prefix is not None:
        return [prefix + tails[i] for i in range(len(inputs))]
    return [remove_fq_suffix(inputs[i]) + tails[i] for i in range(len(inputs))]


def main(argv=None):
    parser = build_parser()
    argv = sys.argv[1:] if argv is None else list(argv)
    if not argv:
        parser.print_help(sys.stdout)
        sys.exit(0)
    args = parser.parse_args(argv)
    if args.list_adapters:
        print_builtin_adapters()
        sys.exit(0)
    if args.input_file is None:
        logging.error("Input file is required.")
        sys.exit(1)
    elif len(args.input_file) > 2:
        logging.error("Input file can not be more than two.")
        sys.exit(1)
    resolve_scheme(args)
    args.output_file = _default_outputs(args.output_file, args.input_file, args.output_prefix, "trimmed")
    args.short_file = _default_outputs(args.short_file, args.input_file, args.output_prefix, "short")
    has_inline = re.match(r".*\([ATGCatgc]+\).*", args.adapter_scheme) is not None
    if args.untrimmed_file or (args.ensure_inline_barcode and has_inline):
        args.untrimmed_file = _default_outputs(args.untrimmed_file, args.input_file, args.output_prefix, "untrimmed")
    else:
        args.untrimmed_file = [None] * len(args.input_file)
    return run_cutseq(args)


if __name__ == "__main__":
    main()
