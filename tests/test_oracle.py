"""The CPU oracle (oracle/cutseq_oracle.c) against (a) the golden vectors produced by the unmodified
reference run.py on the restated cutadapt, (b) the independent pure-Python restatement of
Aligner.locate, (c) known answers that follow cutadapt's documented behaviour."""

import os
import random
import sys

import pytest

from oracle import oracle
from tests import helpers

SHIM = os.path.join(helpers.ROOT, "oracle", "cutadapt_shim")


def shim_align():
    sys.path.insert(0, SHIM)
    try:
        from cutadapt import align, qualtrim
    finally:
        sys.path.pop(0)
    return align, qualtrim


BACK, FRONT, PREFIX, SUFFIX, NI_FRONT, NI_BACK, ANYWHERE = 14, 11, 8, 2, 9, 6, 15


def test_known_answers():
    ad = "ACGTTGCATA"  # stands in for "ADAPTER" of the cutadapt guide (ACGT alphabet only)
    read = "ccccc".upper() + ad + "GGGGG" + ad + "TTTTT"
    # 3' adapter: leftmost full occurrence wins, everything after it is removed
    assert oracle.locate(ad, read, 0.1, BACK, 3) == (0, 10, 5, 15, 10, 0)
    # partial occurrence at the 3' end, and the min_overlap rule
    p7 = "AGATCGGAAGAGCACACGTC"
    assert oracle.locate(p7, "ACGTACGTACGTAGATC", 0.2, BACK, 3) == (0, 5, 12, 17, 5, 0)
    assert oracle.locate(p7, "ACGTACGTACGTAG", 0.2, BACK, 3) is None
    # poly-A as non-internal 3' adapter
    assert oracle.locate("A" * 100, "ACGTACGTCC" + "A" * 20, 0.15, NI_BACK, 3) == (0, 20, 10, 30, 20, 0)
    # anchored 5'
    assert oracle.locate("ATCACG", "ATCACGTTTTTTTT", 0.2, PREFIX, 6) == (0, 6, 0, 6, 6, 0)
    # a leading extra read base costs one error but no score: row 0 only accumulates cost
    assert oracle.locate("ATCACG", "TATCACGTTTTTTT", 0.2, PREFIX, 6) == (0, 6, 0, 7, 6, 1)
    # no match at all
    assert oracle.locate("CTGATCTGGCCG", "AAAAGGG", 0.1, BACK, 1) is None
    # shape of cutadapt's own tests/test_align.py::test_polya (poly-A found after ACAG)
    s = "A" * 17
    assert oracle.locate(s, "ACAG" + s, 0.0, BACK, 1) == (0, len(s), 4, 4 + len(s), len(s), 0)
    assert oracle.locate(s, "ACAG" + "A" * 15, 0.0, BACK, 1) == (0, 15, 4, 19, 15, 0)


def test_rightmost_front_known_answer():
    from cutseq_b200 import _abi as A
    from cutseq_b200.program import Op

    ad = "ACGTTGCATA"
    read = "CCCCC" + ad + "GGGGG" + ad + "TTTTT"
    op = Op(A.OP_ALIGN, adapter_kind=A.AD_RIGHTMOST_FRONT, adapter=ad, min_overlap=3, max_error_rate=0.1)
    assert oracle.adapter_match(op, read) == (0, 10, 20, 30, 10, 0)  # keeps read[30:] == TTTTT
    op = Op(A.OP_ALIGN, adapter_kind=A.AD_FRONT, adapter=ad, min_overlap=3, max_error_rate=0.1)
    assert oracle.adapter_match(op, read)[3] == 15  # regular 5' adapter: leftmost


def test_error_thresholds():
    # 0.2: one error needs >= 5 aligned adapter characters
    p7 = "AGATCGGAAGAGCACACGTC"
    assert oracle.locate(p7, "TTTTTTTTTTAGAT", 0.2, BACK, 3) == (0, 4, 10, 14, 4, 0)
    assert oracle.locate(p7, "TTTTTTTTTTAGTT", 0.2, BACK, 3) is None
    assert oracle.locate(p7, "TTTTTTTTTAGTTC", 0.2, BACK, 3) == (0, 5, 9, 14, 3, 1)


def plant_copy(rng, ref, q, alpha, max_edits=3, cut=None):
    """Overwrite part of the read q (a list) with a prefix or suffix of ref that carries up to max_edits random
    substitutions / deletions / insertions: at the read start, at its end or anywhere."""
    m, n = len(ref), len(q)
    cut = rng.randint(1, m) if cut is None else cut
    piece = list(ref[:cut] if rng.random() < 0.5 else ref[m - cut:])
    for _ in range(rng.randint(0, max_edits)):
        r = rng.random()
        pos = rng.randrange(len(piece)) if piece else 0
        if r < 0.5 and piece:
            piece[pos] = rng.choice(alpha)
        elif r < 0.75 and piece:
            del piece[pos]
        else:
            piece.insert(pos, rng.choice(alpha))
    pos = rng.choice([0, n - len(piece), rng.randint(0, max(0, n - len(piece)))])
    pos = max(0, pos)
    q[pos : pos + len(piece)] = piece


@pytest.mark.parametrize("flags", [BACK, FRONT, PREFIX, SUFFIX, NI_FRONT, NI_BACK, ANYWHERE])
def test_c_oracle_equals_python_restatement(flags):
    align, _ = shim_align()
    rng = random.Random(flags)
    for it in range(1500):
        m = rng.choice([1, 2, 3, 6, 8, 13, 20, 20, 33])
        alpha = "ACGT" if it % 3 else "AC"
        ref = "".join(rng.choice(alpha) for _ in range(m))
        n = rng.choice([0, 1, 2, 5, 17, 30, 45, 60])
        q = [rng.choice(alpha + "N") for _ in range(n)]
        if n and m <= n and rng.random() < 0.7:  # plant a mutated (partial) copy
            plant_copy(rng, ref, q, alpha)
        q = "".join(q)
        rate = rng.choice([0.0, 0.1, 0.15, 0.2, 0.2, 0.34, 0.5])
        mo = rng.choice([1, 3, 3, 10, m])
        mo = max(1, min(mo, m))
        want = align.Aligner(ref, rate, flags=flags, min_overlap=mo).locate(q)
        got = oracle.locate(ref, q, rate, flags, mo)
        assert got == want, (ref, q, rate, flags, mo)


def shim_adapter(kind, sequence, max_errors, min_overlap):
    """The restated cutadapt adapter class an ALIGN op of this kind stands for."""
    from cutseq_b200 import _abi as A

    sys.path.insert(0, SHIM)
    try:
        from cutadapt import adapters as ad
    finally:
        sys.path.pop(0)
    cls, extra = {
        A.AD_BACK: (ad.BackAdapter, {}),
        A.AD_BACK_ANYWHERE: (ad.BackAdapter, {"force_anywhere": True}),
        A.AD_RIGHTMOST_FRONT: (ad.RightmostFrontAdapter, {}),
        A.AD_PREFIX: (ad.PrefixAdapter, {}),
        A.AD_SUFFIX: (ad.SuffixAdapter, {}),
        A.AD_NI_FRONT: (ad.NonInternalFrontAdapter, {}),
        A.AD_NI_BACK: (ad.NonInternalBackAdapter, {}),
        A.AD_FRONT: (ad.FrontAdapter, {}),
    }[kind]
    return cls(sequence, max_errors=max_errors, min_overlap=min_overlap, **extra)


@pytest.mark.parametrize("kind", range(1, 9))
def test_c_oracle_equals_python_restatement_long_adapters(kind):
    """Adapters of 64, 65, 97 and CSQ_MAX_ADAPTER bases against reads of up to CSQ_MAX_READ_LEN bases, with error
    rates whose double rounding decides (0.29: 100 * 0.29 < 29) and absolute error counts: the whole adapter match of
    the C oracle (count -> rate, min_overlap rules, RightmostFront's reversal) against the restated adapter classes."""
    from cutseq_b200 import _abi as A
    from cutseq_b200.program import Op

    rng = random.Random(500 + kind)
    for it in range(400):
        m = rng.choice([64, 65, 97, A.CSQ_MAX_ADAPTER])
        alpha = "ACGT" if it % 4 else "AC"
        ref = "".join(rng.choice(alpha) for _ in range(m))
        n = rng.choice([0, 1, m - 1, m, 150, 300, 600, A.CSQ_MAX_READ_LEN - 1, A.CSQ_MAX_READ_LEN])
        q = [rng.choice(alpha) if rng.random() > 0.02 else "N" for _ in range(n)]
        for _ in range(rng.choice([0, 1, 1, 2]) if n else 0):
            plant_copy(rng, ref, q, alpha, max_edits=rng.choice([0, 3, 12, 30]), cut=m if rng.random() < 0.3 else None)
        q = "".join(q)[:n]
        if rng.random() < 0.05:
            q = q.lower()
        max_errors = rng.choice([0.0, 0.1, 0.2, 0.29, 0.35, 0.45, 1.0, 7.0, 18.0, 30.0])  # >= 1: a count
        mo = rng.choice([1, 3, 10, m])
        op = Op(A.OP_ALIGN, adapter_kind=kind, adapter=ref, min_overlap=mo, max_error_rate=max_errors)
        want = shim_adapter(kind, ref, max_errors, mo).match_to(q)
        want = None if want is None else want.as_tuple()
        assert oracle.adapter_match(op, q) == want, (kind, ref, q, max_errors, mo)


def test_homopolymer_equals_python_restatement():
    align, _ = shim_align()
    rng = random.Random(5)
    for it in range(300):
        n = rng.randint(0, 140)
        base = "A" if it % 2 else "T"
        flags = NI_BACK if it % 2 else NI_FRONT
        run = base * rng.randint(0, 40)
        body = "".join(rng.choice("ACGT") for _ in range(n))
        q = (body + run) if flags == NI_BACK else (run + body)
        q = "".join(c if rng.random() > 0.03 else rng.choice("ACGTN") for c in q)
        ref = base * 100
        assert oracle.locate(ref, q, 0.15, flags, 3) == align.Aligner(ref, 0.15, flags=flags, min_overlap=3).locate(q)


def test_record_names_match_rule():
    """dnaio's record_names_match as documented upstream: ids end at the first space or tab, "/1" "/2" and ".1" ".2"
    style mate numbers are ignored, anything else must be identical.  C oracle == Python restatement on a table and
    on random headers."""
    from cutadapt._record import record_names_match

    ok = [("r", "r"), ("r 1", "r 2"), ("r/1", "r/2"), ("r.1 x", "r.2 y"), ("r1", "r3"), ("r\t1", "r 2"), ("abc/1 c", "abc/2")]
    bad = [("r", "s"), ("r1", "r4"), ("r", "r1"), ("ab", "abc"), ("abc", "ab"), ("rA", "rB"), ("r\x0b1", "r 2"), ("", "r"), ("r", ""), (" r", "r")]
    for a, b in ok:
        assert oracle.names_match(a, b) and record_names_match(a, b), (a, b)
    for a, b in bad:
        assert not oracle.names_match(a, b) and not record_names_match(a, b), (a, b)
    rng = random.Random(5)
    for _ in range(20000):
        a = "".join(rng.choice("ab12 3\t/.") for _ in range(rng.randint(0, 7)))
        b = a if rng.random() < 0.3 else "".join(rng.choice("ab12 3\t/.") for _ in range(rng.randint(0, 7)))
        if rng.random() < 0.3 and a:
            b = a[:-1] + rng.choice("123 x")
        if b[:1] in (" ", "\t") or b == "":
            continue  # id of length 0: upstream reads header1[-1], undefined
        assert oracle.names_match(a, b) == record_names_match(a, b), (a, b)


def test_quality_trim_index():
    _, qualtrim = shim_align()
    rng = random.Random(3)
    assert oracle.quality_trim_index("IIII", 0, 20) == (0, 4)
    assert oracle.quality_trim_index("II##", 0, 20) == (0, 2)
    assert oracle.quality_trim_index("####", 0, 20) == (0, 0)
    assert oracle.quality_trim_index("", 0, 20) == (0, 0)
    for _ in range(2000):
        q = "".join(rng.choice("I9-#!5?") for _ in range(rng.randint(0, 60)))
        cf, cb = rng.choice([0, 0, 10, 20]), rng.choice([0, 15, 20, 30])
        assert oracle.quality_trim_index(q, cf, cb) == qualtrim.quality_trim_index(q, cf, cb), (q, cf, cb)


@pytest.mark.parametrize("case", helpers.golden_cases(), ids=lambda c: c["case"])
def test_oracle_reproduces_golden(case):
    prog = helpers.program_for(case["argv"], case["n_mates"])
    mates = helpers.golden_inputs(case)
    batch, keep = oracle.make_batch(*mates)
    out = oracle.run_batch(prog, batch, n_threads=3)
    assert out["status"] == 0
    want = helpers.expected_by_dest(case, prog)
    for (d, m), data in want.items():
        assert out["text"][d][m] == data, (case["case"], helpers.DEST_KEYS[d], m)
    # minimal report numbers (w/adapters = first AdapterCutter only, the monkey-patch quirk)
    from cutseq_b200.run import minimal_report_text

    if case["minimal_report"]:
        assert minimal_report_text(out["counters"], prog).splitlines()[1] == case["minimal_report"][-1]


@pytest.mark.parametrize("case", helpers.golden_cases(hash_only=True), ids=lambda c: c["case"])
def test_oracle_full_bundled(case):
    import hashlib

    prog = helpers.program_for(case["argv"], 2)
    batch, keep = oracle.make_batch(*helpers.golden_inputs(case))
    out = oracle.run_batch(prog, batch, n_threads=4)
    for d, dk in enumerate(helpers.DEST_KEYS[:2]):
        for m in range(2):
            assert hashlib.sha256(out["text"][d][m]).hexdigest() == case["outputs"][f"{dk}_R{m + 1}"]["sha256"]


def test_thread_count_does_not_change_output():
    case = helpers.golden_cases()[2]
    prog = helpers.program_for(case["argv"], case["n_mates"])
    batch, keep = oracle.make_batch(*helpers.golden_inputs(case))
    a = oracle.run_batch(prog, batch, n_threads=1)
    b = oracle.run_batch(prog, batch, n_threads=7)
    assert a["text"] == b["text"]


def test_pinning_status_is_honest():
    """tests/golden/PINNING.json says whether the expectations were ever compared with a real cutadapt.  Without one
    it must say "unpinned"; with one importable, scripts/bless_against_cutadapt.py must agree byte for byte."""
    import json
    import subprocess

    with open(os.path.join(helpers.GOLD, "PINNING.json")) as f:
        pin = json.load(f)
    rc = subprocess.call([sys.executable, os.path.join(helpers.ROOT, "scripts", "bless_against_cutadapt.py")],
                         stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    if rc == 3:  # no real cutadapt in this environment
        assert pin["pinned"] is False or pin["checked_against"], "PINNING.json claims a check that cannot have run here"
    else:
        assert rc == 0, "the real cutadapt disagrees with tests/golden (run scripts/bless_against_cutadapt.py)"


def test_long_headers_come_back_whole():
    """Headers up to the product's 65 535 bytes, with and without RENAME; a longer one is CSQ_ERR_LIMIT."""
    from cutseq_b200 import _abi as A
    from cutseq_b200.program import Filters, Op, Program

    rng = random.Random(8)
    for n in (4001, 20000, 65535):
        heads = ["".join(rng.choice("abc:/") for _ in range(n)), "i" * 10 + " " + "c" * (n - 11)]
        recs = [(h, "ACGTACGT", "IIIIIIII") for h in heads]
        batch, keep = oracle.make_batch(recs)
        for ops, names in (([], heads), ([Op(A.OP_RENAME)], [heads[0], "i" * 10])):
            out = oracle.run_batch(Program(False, ops, [], Filters(0)), batch)
            assert out["status"] == 0
            assert [r[0] for r in oracle.parse_fastq_text(out["text"][0][0])] == names
    batch, keep = oracle.make_batch([("x" * 65536, "ACGT", "IIII")])
    assert oracle.run_batch(Program(False, [], [], Filters(0)), batch)["status"] == A.ERR_LIMIT


def test_longest_renamed_name():
    """A 65 535-byte id behind which PairedEndRenamer puts two UMI parts of 895 bases: the longest name a record
    can get, byte for byte."""
    from cutseq_b200 import _abi as A
    from cutseq_b200.program import Filters, Op, Program

    rng = random.Random(9)
    n = A.CSQ_MAX_READ_LEN
    s1, s2 = ("".join(rng.choice("ACGT") for _ in range(n)) for _ in range(2))
    h = "".join(rng.choice("abcdefgh0123456789") for _ in range(65535))
    ops = [Op(A.OP_CUT, length=n), Op(A.OP_RENAME, rename_parts=A.REN_R1_PREFIX | A.REN_R2_PREFIX)]
    batch, keep = oracle.make_batch([(h, s1, "I" * n)], [(h, s2, "I" * n)])
    out = oracle.run_batch(Program(True, ops, ops, Filters(0)), batch)
    assert out["status"] == 0
    for m in range(2):
        assert out["text"][0][m] == f"@{h}_{s1}{s2}\n\n+\n\n".encode()


def shim_modifiers():
    sys.path.insert(0, SHIM)
    try:
        from cutadapt import modifiers
        from cutadapt._record import SequenceRecord
        from cutadapt.info import ModificationInfo
    finally:
        sys.path.pop(0)
    return modifiers, SequenceRecord, ModificationInfo


def shim_run(prog, mates):
    """The generated program as cutadapt modifiers, per read (pair): final names, bases, qualities, destinations."""
    from cutseq_b200 import _abi as A
    from cutseq_b200.program import rename_template

    mods, Record, Info = shim_modifiers()
    n_mates = len(mates)
    opss = [prog.ops_r1, prog.ops_r2][:n_mates]
    steps = []
    for t in range(len(opss[0])):
        row = []
        for ops in opss:
            op = ops[t]
            if op.kind == A.OP_STRIP_SUFFIX:
                row.append(mods.SuffixRemover(op.suffix))
            elif op.kind == A.OP_ALIGN:
                row.append((mods.AdapterCutter([shim_adapter(op.adapter_kind, op.adapter, op.max_error_rate, op.min_overlap)]), op.adapter_id))
            elif op.kind == A.OP_CUT:
                row.append(mods.UnconditionalCutter(op.length))
            elif op.kind == A.OP_QTRIM:
                row.append(mods.QualityTrimmer(op.cutoff_front, op.cutoff_back, op.quality_base))
            elif op.kind == A.OP_RENAME:
                tpl = rename_template(op.rename_parts)
                row.append(mods.PairedEndRenamer(tpl) if n_mates == 2 else mods.Renamer(tpl))
            else:
                raise AssertionError(op)
        steps.append(row)
    out = []
    flt = prog.filters
    for i in range(len(mates[0])):
        reads = [Record(*mates[m][i]) for m in range(n_mates)]
        infos = [Info(r) for r in reads]
        matched = [0] * n_mates
        for row in steps:
            if isinstance(row[0], mods.PairedEndRenamer):
                reads = list(row[0](reads[0], reads[1], infos[0], infos[1]))
                continue
            for m in range(n_mates):
                mod = row[m]
                if isinstance(mod, tuple):
                    mod, aid = mod
                    before = len(infos[m].matches)
                    reads[m] = mod(reads[m], infos[m])
                    if len(infos[m].matches) > before and aid >= 0:
                        matched[m] |= 1 << aid
                else:
                    reads[m] = mod(reads[m], infos[m])
        if any(len(r) < flt.min_length for r in reads):
            dest = A.DEST_SHORT
        elif flt.untrimmed_enabled and any(req & ~matched[m] for m, req in enumerate([flt.required_r1, flt.required_r2][:n_mates])):
            dest = A.DEST_UNTRIMMED
        else:
            dest = A.DEST_TRIMMED
        out.append((dest, [(r.name, r.sequence, r.qualities) for r in reads]))
    return out


def test_generated_programs_equal_cutadapt_modifiers():
    """Programs of tests/program_gen.py without COND_CUT and REVCOMP (cutseq's own classes, checked by known answers
    elsewhere) through the restated cutadapt modifiers, read by read, against oracle.run_batch."""
    from cutseq_b200 import _abi as A
    from tests import program_gen as G

    n_reads = 0
    for seed in range(20):
        rng = random.Random(3300 + seed)
        prog = G.random_program(rng, paired=seed % 2 == 1, cond_cut=False, revcomp=False)
        mates = G.random_mates(rng, prog, 100, lengths=G.EDGE_LENGTHS[:-1] + [40, 64, 100, 150, 300])
        batch, keep = oracle.make_batch(*mates)
        want = oracle.run_batch(prog, batch)
        assert want["status"] == 0
        got = shim_run(prog, mates)
        texts = {}
        for d in range(A.CSQ_N_DEST):
            for m in range(len(mates)):
                texts[d, m] = iter(oracle.parse_fastq_text(want["text"][d][m]))
        for i, (dest, recs) in enumerate(got):
            assert int(want["results"][0]["dest"][i]) == dest, (seed, i)
            for m, rec in enumerate(recs):
                assert next(texts[dest, m]) == rec, (seed, i, m)
        n_reads += len(got)
    assert n_reads == 2000
