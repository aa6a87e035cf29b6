#!/usr/bin/env python
"""Generate tests/golden/reference_common.json: what ``cutseq/common.py`` of the original cutseq (stdlib only) returns
for the scheme table, the scheme grammar, the file-name rule, the reverse complement and ``--list-adapters``.
tests/test_scheme.py compares cutseq_b200.common with these values.

    python scripts/make_golden_common.py <cutseq source tree>   # the directory that holds cutseq/common.py
    python scripts/make_golden_common.py --snapshot             # no original at hand: cutseq_b200/common.py's own values

The file's "source" field says which of the two wrote it.  A snapshot only guards cutseq_b200.common against changes
of its own; run the first form where a cutseq source tree is available to turn it into a comparison with the original.
"""

import contextlib
import io
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
OUT = os.path.join(ROOT, "tests", "golden", "reference_common.json")

EXTRA_SCHEMES = ["ACGT>ACGTJUNK", "acgt(tt)NNXX<XN(gg)acgt", "A-C", "ACGT(AC)NNNNXX-XN(GT)TTTT"]
PARTS = ("p5", "p7", "inline5", "inline3", "umi5", "umi3", "mask5", "mask3")
FILE_NAMES = ["x_R1.fastq.gz", "x_R2_001.fq", "x.fq.gz", "dir.fq/x", "x_R1_001.fastq", "_R1.fq", "x.txt"]
SEQUENCES = ["ACGTN", "acgtRYn", ""]


def golden(common, source: str) -> dict:
    schemes = {}
    for s in list(common.BUILDIN_ADAPTERS.values()) + EXTRA_SCHEMES:
        b = common.BarcodeConfig(s)
        schemes[s] = {"to_dict": b.to_dict(), "parts": {p: [getattr(b, p).rc, repr(getattr(b, p))] for p in PARTS}}
    listing = io.StringIO()
    with contextlib.redirect_stdout(listing):
        common.print_builtin_adapters()
    return {
        "source": source,
        "adapters": list(common.BUILDIN_ADAPTERS.items()),
        "schemes": schemes,
        "remove_fq_suffix": {f: common.remove_fq_suffix(f) for f in FILE_NAMES},
        "reverse_complement": {s: common.reverse_complement(s) for s in SEQUENCES},
        "list_adapters": listing.getvalue(),
    }


def main():
    if sys.argv[1:] == ["--snapshot"]:
        sys.path.insert(0, ROOT)
        from cutseq_b200 import common

        source = ("SNAPSHOT of cutseq_b200/common.py, not values of the original cutseq (which was not available "
                  "when this file was written)")
    elif len(sys.argv) == 2 and os.path.isfile(os.path.join(sys.argv[1], "cutseq", "common.py")):
        sys.path.insert(0, os.path.abspath(sys.argv[1]))
        from cutseq import common

        source = "cutseq/common.py of the original cutseq"
    else:
        sys.exit(__doc__)
    with open(OUT, "w") as f:
        json.dump(golden(common, source), f, indent=1)
        f.write("\n")
    print(OUT)


if __name__ == "__main__":
    main()
