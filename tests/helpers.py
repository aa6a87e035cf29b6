"""Shared test helpers: golden-fixture access, settings objects, FASTQ record lists."""

import argparse
import gzip
import json
import os

from cutseq_b200 import program
from cutseq_b200.common import BUILDIN_ADAPTERS, BarcodeConfig

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def manifest():
    with open(os.path.join(GOLD, "manifest.json")) as f:
        return json.load(f)


def golden_cases(hash_only=False):
    """Cases with expected files committed (default) or the hash-only cases over the full bundled input."""
    return [c for c in manifest() if bool(c.get("hash_only")) == hash_only]


def read_fastq_gz(path):
    data = gzip.open(path).read()
    lines = data.split(b"\n")
    if lines and lines[-1] == b"":
        lines.pop()
    assert len(lines) % 4 == 0, path
    return [(lines[i][1:].decode("latin-1"), lines[i + 1].decode("latin-1"), lines[i + 3].decode("latin-1")) for i in range(0, len(lines), 4)]


def golden_inputs(case):
    return [read_fastq_gz(os.path.join(GOLD, f"in_{case['input']}_R{m}.fq.gz")) for m in range(1, case["n_mates"] + 1)]


def golden_input_paths(case):
    return [os.path.join(GOLD, f"in_{case['input']}_R{m}.fq.gz") for m in range(1, case["n_mates"] + 1)]


def golden_expected(case, key):
    p = os.path.join(GOLD, f"exp_{case['case']}_{key}.fastq.gz")
    return gzip.open(p).read() if os.path.exists(p) else None


def parse_cli(argv):
    """Parse cutseq flags the way cutseq_b200.run.main does, returning (scheme, settings namespace)."""
    from cutseq_b200 import run

    args = run.build_parser().parse_args(list(argv) + ["dummy.fq"])
    scheme = run.resolve_scheme(args)
    return scheme, run.settings_from_args(args), args


def program_for(argv, n_mates):
    scheme, settings, args = parse_cli(argv)
    bc = BarcodeConfig(scheme)
    want_untrimmed = bool(settings.ensure_inline_barcode and (bc.inline5.len + bc.inline3.len > 0))
    u = "x" if want_untrimmed else None
    if n_mates == 2:
        return program.compile_paired(bc, settings, u, u)
    return program.compile_single(bc, settings, u)


DEST_KEYS = ("trimmed", "short", "untrimmed")


def expected_by_dest(case, prog):
    """-> {(dest, mate): bytes} as the reference wrote them (sink swap undone)."""
    out = {}
    for d, dk in enumerate(DEST_KEYS):
        for m in range(case["n_mates"]):
            fm = m
            if d == 0 and prog.swap_sink:
                fm = 1 - m  # R1 was written to the R2 file and vice versa (run.py:785-792)
            data = golden_expected(case, f"{dk}_R{fm + 1}")
            out[(d, m)] = data if data is not None else b""
    return out
