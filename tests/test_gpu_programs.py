"""Hand-built op programs against the CPU oracle: the per-read scalar ops (CUT, COND_CUT, RENAME) anywhere in a
program, quality trimming with both cutoffs and either quality base, the Renamer id, header suffixes, UMI parts,
REVCOMP, the filters and both FASTQ emitters, over the whole space that csq_plan_create accepts rather than the
corner the command line reaches.  Bit-exact: every comparison is ==."""

import functools
import os
import random
import re
from types import SimpleNamespace

import numpy as np
import pytest

from cutseq_b200 import _abi as A
from cutseq_b200 import native
from cutseq_b200.program import Filters, Op, Program
from oracle import oracle
from tests import program_gen as G
from tests.test_gpu_gz import gunzip_members
from tests.test_gpu_parity import assert_equals_oracle, check_locate

MAX_N = A.CSQ_MAX_READ_LEN
N_THREADS = min(8, os.cpu_count() or 1)
SIZES = [2000, 1, 31, 33, 255, 257]
FLAGS = [0, A.PLAN_NO_PREFILTER, A.PLAN_EMIT_G16, A.PLAN_ONE_STREAM, A.PLAN_GZIP_OUT, A.PLAN_NO_EXACT_STOP]
N_SEEDS = 24  # even seeds single-end, odd seeds paired


@functools.lru_cache(maxsize=None)
def program_case(seed):
    rng = random.Random(9200 + seed)
    prog = G.random_program(rng, paired=seed % 2 == 1)
    return prog, G.random_mates(rng, prog, sum(SIZES))


def batches(mates):
    """The records of a case cut into batches of SIZES reads."""
    out, at = [], 0
    for n in SIZES:
        out.append([m[at : at + n] for m in mates])
        at += n
    return out


def oracle_run(prog, mates):
    batch, keep = oracle.make_batch(*mates)
    return oracle.run_batch(prog, batch, n_threads=N_THREADS)


def capacity_for(want):
    return 2 * max(len(t) for row in want["text"] for t in row) + 4096


COUNTERS = ("n", "written", "too_short", "untrimmed", "total_bp", "written_bp", "quality_trimmed_bp", "with_adapters",
            "dp_cells", "adjacent_bases")


def counters(c):
    return {f: np.array(np.ctypeslib.as_array(getattr(c, f)) if not isinstance(getattr(c, f), int) else getattr(c, f),
                        dtype=np.int64) for f in COUNTERS}


def run_on_plan(plan, prog, mates, capacity, slot=0, text_eol=None):
    """One batch on an existing plan (SoA, or FASTQ text with the given line end).  The counters are this batch's
    share: the plan sums them over its batches."""
    before = counters(plan.stats())
    n = len(mates[0])
    if text_eol is None:
        batch, keep = oracle.make_batch(*mates)
        text, records = plan.run_batch(batch, capacity, slot)
    else:
        text, records = plan.run_text([G.fastq_text(m, text_eol) for m in mates], n, capacity, slot)
    if plan.flags & A.PLAN_GZIP_OUT:
        text = [[gunzip_members(t) if t else b"" for t in row] for row in text]
    results = [plan.results(slot, m, n) for m in range(len(mates))]
    matches = [{t: plan.matches(slot, m, t, n) for t, op in enumerate(prog.ops_r1 if m == 0 else prog.ops_r2)
                if op.kind == A.OP_ALIGN} for m in range(len(mates))]
    after = counters(plan.stats())
    stats = SimpleNamespace(**{f: (after[f] - before[f]).tolist() for f in COUNTERS})
    return text, records, results, matches, stats


class FlagPlan(native.Plan):
    def __init__(self, prog, flags):
        super().__init__(prog, 0, A.PLAN_KEEP_MATCHES | flags)
        self.flags = flags


def check(prog, mates, want, plan, capacity, slot=0, text_eol=None):
    got = run_on_plan(plan, prog, mates, capacity, slot, text_eol)
    assert_equals_oracle(prog, mates, want, *got)


# ---- a. random valid programs ----

@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(N_SEEDS))
def test_random_program(seed):
    """One generated program: the 2000-read batch under every plan flag, then on the same plan and slot a smaller
    batch (buffers only grow: nothing of the larger batch may leak into it), and as FASTQ text with both emitters."""
    prog, mates = program_case(seed)
    parts = batches(mates)
    wants = [oracle_run(prog, b) for b in parts]
    cap = max(capacity_for(w) for w in wants)
    for j, flags in enumerate(FLAGS):
        small = 1 + (j + seed) % (len(SIZES) - 1)
        with FlagPlan(prog, flags) as plan:
            check(prog, parts[0], wants[0], plan, cap)
            check(prog, parts[small], wants[small], plan, cap)
            if flags in (0, A.PLAN_EMIT_G16):
                check(prog, parts[0], wants[0], plan, cap, slot=1, text_eol="\n")
                if seed % 3 == 0:
                    check(prog, parts[0], wants[0], plan, cap, slot=2, text_eol="\r\n")


def test_random_programs_reach_the_edges():
    """The fixed seeds of test_random_program reach what the generator is there for (no GPU needed)."""
    seen = set()
    for seed in range(N_SEEDS):
        prog, mates = program_case(seed)
        paired = "paired" if prog.paired else "single"
        for ops in (prog.ops_r1, prog.ops_r2) if prog.paired else (prog.ops_r1,):
            kinds = [op.kind for op in ops]
            seen |= {("op", k) for k in kinds}
            seen |= {("align", op.adapter_kind) for op in ops if op.kind == A.OP_ALIGN}
            seen |= {("qtrim_front",) for op in ops if op.kind == A.OP_QTRIM and op.cutoff_front > 0}
            seen |= {("base64",) for op in ops if op.kind == A.OP_QTRIM and op.quality_base == 64}
            if G.max_scalar_run(ops) == G.MAX_PRE:
                seen.add(("run12",))
            if A.OP_ALIGN not in kinds:
                seen.add(("no_align",))
            if A.OP_RENAME in kinds:
                r, aligns = kinds.index(A.OP_RENAME), [t for t, k in enumerate(kinds) if k == A.OP_ALIGN]
                if aligns:
                    seen.add(("rename", "front" if r < aligns[0] else "back" if r > aligns[-1] else "between"))
        want = oracle_run(prog, mates)
        seen |= {("dest", paired, int(d)) for d in want["results"][0]["dest"]}
        for m, recs in enumerate(mates):
            seen |= {("header", len(h)) for h, _, _ in recs if len(h) == 65535}
            seen |= {("blank", c) for h, _, _ in recs for c in G.TEXT_BLANKS if chr(c) in h}
        for row in want["text"]:
            for text in row:
                for umi in re.findall(rb"_([A-Za-z]{17,})$", text, re.M):  # (17 letters in a row: not in a random header)
                    seen |= {("umi>16",)} if len(umi) > 16 else set()
                    seen |= {("umi895",)} if len(umi) >= MAX_N else set()
    need = {("op", k) for k in range(1, 8)} | {("align", k) for k in G.KINDS}
    need |= {("qtrim_front",), ("base64",), ("run12",), ("no_align",), ("umi>16",), ("umi895",), ("header", 65535)}
    need |= {("rename", p) for p in ("front", "between", "back")} | {("blank", c) for c in G.TEXT_BLANKS}
    need |= {("dest", p, d) for p in ("single", "paired") for d in range(A.CSQ_N_DEST)}
    assert need <= seen, sorted(need - seen)


# ---- b. targeted tests ----

def soa_and_text(prog, mates, flags=0, forms=("soa", "text")):
    """The records as an SoA batch and as a FASTQ text batch, in two slots of one plan, against one oracle run."""
    want = oracle_run(prog, mates)
    cap = capacity_for(want)
    with FlagPlan(prog, flags) as plan:
        for slot, form in enumerate(forms):
            check(prog, mates, want, plan, cap, slot, text_eol=None if form == "soa" else "\n")
    return want


QT_CUTOFFS = [0, 1, 10, 20, 40]
NARROW = {"whole": [], "cut5": [Op(A.OP_CUT, length=5)], "cut_7": [Op(A.OP_CUT, length=-7)],
          "align": [Op(A.OP_ALIGN, adapter_kind=A.AD_PREFIX, adapter="ACGTAC", max_error_rate=0.0),
                    Op(A.OP_ALIGN, adapter_kind=A.AD_BACK, adapter="TTGCAGGT", max_error_rate=0.0)]}


def quality_reads(rng, base, cutoffs, n_reads=400):
    """Quality patterns at the edges of the two 16-byte scans: low runs of 15-17 / 31-33 at either end or both, runs
    whose sums return to exactly 0 for the cutoffs, qualities below the base; reads of 0 .. CSQ_MAX_READ_LEN."""
    recs = []
    npr = np.random.default_rng(rng.getrandbits(64))
    for i in range(n_reads):
        n = rng.choice([0, 1, 2, 15, 16, 17, 18, 31, 32, 33, 34, 47, 48, 49, 64, 100, 300, MAX_N, rng.randint(0, MAX_N)])
        q = npr.integers(base + 30, min(126, base + 45) + 1, n).tolist()
        pattern = i % 6
        k = min(n, rng.choice(G.LOW_RUNS))
        if pattern == 1:  # low run at the start / end / both
            q[:k] = [rng.randint(33, base + 2) for _ in range(k)]
        elif pattern == 2:
            q[n - k:] = [rng.randint(33, base + 2) for _ in range(k)]
        elif pattern == 3:
            q[:k] = [rng.randint(33, base + 2) for _ in range(k)]
            q[n - k:] = [rng.randint(33, base + 2) for _ in range(k)]
        elif pattern == 4:  # running sums that reach exactly 0 again (the `s > max` tie)
            for side in (0, 1):
                c = base + cutoffs[side]
                run = []
                while len(run) < k:
                    d = rng.randint(1, 5)
                    run += [c - d, c + d] if rng.random() < 0.7 else [c, c]
                run = [min(126, max(33, x)) for x in run[:k]]
                if side == 0:
                    q[:k] = run
                else:
                    q[n - k:] = run[::-1]
        elif pattern == 5:
            q = npr.integers(33, 127, n).tolist()  # anything, below the base too
        s = list(G.draw(npr, "ACGT", n))
        if n >= 6 and i % 3 == 0:
            s[:6] = "ACGTAC"
        if n >= 14 and i % 4 == 0:
            s[n - 8:] = "TTGCAGGT"
        recs.append((f"q{i}", "".join(s), "".join(map(chr, q))))
    return recs


@pytest.mark.gpu
@pytest.mark.parametrize("narrow", list(NARROW))
@pytest.mark.parametrize("base", [33, 64])
def test_quality_trim_grid(base, narrow):
    """QualityTrimmer over the cutoff grid {0, 1, 10, 20, 40}^2 on whole reads and on intervals narrowed in front of
    it (the 16-byte fetches then start at a > 0).  Each cutoff pair runs behind one of the four narrowings, every
    quality pattern behind all of them."""
    rng = random.Random(base * 10 + len(narrow))
    grid = [(cf, cb) for cf in QT_CUTOFFS for cb in QT_CUTOFFS]
    for i, (cf, cb) in enumerate(grid):
        if i % len(NARROW) == list(NARROW).index(narrow):
            ops = NARROW[narrow] + [Op(A.OP_QTRIM, cutoff_front=cf, cutoff_back=cb, quality_base=base)]
            prog = Program(False, ops, [], Filters(0))
            soa_and_text(prog, [quality_reads(rng, base, (cf, cb), 400)])


ID_POSITIONS = [0, 1, 14, 15, 16, 17, 30, 31, 32, 33, 47, 48, 49]
RENAMER_PROGRAMS = {
    "plain": [],
    "rename": [Op(A.OP_CUT, length=3), Op(A.OP_RENAME, rename_parts=A.REN_OWN_PREFIX | A.REN_OWN_SUFFIX), Op(A.OP_CUT, length=-2)],
    "strip": [Op(A.OP_STRIP_SUFFIX, suffix="/1"), Op(A.OP_STRIP_SUFFIX, suffix="x")],
    "strip_rename": [Op(A.OP_STRIP_SUFFIX, suffix="/1"), Op(A.OP_STRIP_SUFFIX, suffix="x"),
                     Op(A.OP_RENAME, rename_parts=A.REN_OWN_SUFFIX), Op(A.OP_CUT, length=-4)],
}


def renamer_headers(blanks):
    """Every blank at the chunk edges of the id scan, leading blank runs, blank-only headers, blanks at the end only,
    header lengths 0 .. 65 535; some end in the suffixes of RENAMER_PROGRAMS."""
    rng = random.Random(len(blanks))
    npr = np.random.default_rng(len(blanks))
    word = lambda n: G.draw(npr, "abcdefghij0123456789:.-", n)  # noqa: E731
    out = []
    for b in blanks:
        c = chr(b)
        for p in ID_POSITIONS:
            h = word(60)
            out.append(h[:p] + c + h[p + 1:])
            out.append(h[:p] + c + c + h[p + 2:p + 20])  # a blank run inside the header, shorter headers
        for run in (15, 16, 17, 33):
            out.append(c * run + word(20) + c + word(5))
            out.append(c * run + word(20))
        out += [c, c * 16, c * 40, word(20) + c, word(31) + c * 3, word(5) + c + word(3) + "/1", word(5) + c + "x"]
    for n in (0, 1, 15, 16, 17, 4001, 65535):
        h = word(n)
        out += [h, h[:n - 2] + "/1" if n >= 2 else h]
        if n > 20:
            out += [h[:14] + chr(rng.choice(blanks)) + h[15:], h[:n - 1] + chr(rng.choice(blanks))]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["soa", "text"])
@pytest.mark.parametrize("variant", list(RENAMER_PROGRAMS))
def test_renamer_id_blanks(variant, form):
    """Renamer.parse_name (str.split(maxsplit=1)) on the device: every Python blank, single-end SoA also '\\n' and
    '\\r', which a text batch cannot hold."""
    headers = renamer_headers(G.PY_BLANKS if form == "soa" else G.TEXT_BLANKS)
    rng = random.Random(5)
    recs = []
    for i, h in enumerate(headers):
        s = "".join(rng.choice("ACGT") for _ in range(rng.choice([0, 5, 20, 40])))
        recs.append((h, s, "I" * len(s)))
    prog = Program(False, RENAMER_PROGRAMS[variant], [], Filters(0))
    for flags in (0, A.PLAN_EMIT_G16):
        soa_and_text(prog, [recs], flags, forms=(form,))


UMI_LENGTHS = [0, 1, 15, 16, 17, 31, 32, 33, 100, MAX_N]
ID_LENGTHS = [0, 31, 32, 33, 65535]


def umi_records(rng, n_mates, width):
    """Ids of 0 .. 65 535 bytes beside short ones in every warp: records that fit the staged emitter's buffers and
    records that do not."""
    mates = [[] for _ in range(n_mates)]
    npr = np.random.default_rng(rng.getrandbits(64))
    for i in range(96):
        idl = ID_LENGTHS[i % len(ID_LENGTHS)] if i % 2 == 0 else rng.choice([0, 3, 31])
        h = G.draw(npr, "abcdef", idl) + (" c" if i % 3 and idl < 65535 else "")
        ln = rng.choice([width, width, min(MAX_N, width + rng.randint(0, 40)), rng.randint(0, width)])
        for m in range(n_mates):
            mates[m].append((h, G.draw(npr, "ACGTN", ln), G.draw(npr, "".join(G.QCHARS), ln)))
    return mates


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, A.PLAN_EMIT_G16], ids=["emit_stage", "emit_g16"])
@pytest.mark.parametrize("paired", [False, True], ids=["single", "paired"])
def test_umi_parts(paired, flags):
    """UMI parts of 0 .. 895 bases: own prefix and suffix (single-end), R1 and R2 prefixes (paired), in front of ids of
    0 .. 65 535 bytes, as SoA and as text batches."""
    rng = random.Random(17 + paired)
    for a, b in zip(UMI_LENGTHS, UMI_LENGTHS[::-1]):
        if paired:
            ops1 = [Op(A.OP_CUT, length=a), Op(A.OP_RENAME, rename_parts=A.REN_R1_PREFIX | A.REN_R2_PREFIX)]
            ops2 = [Op(A.OP_CUT, length=b), Op(A.OP_RENAME, rename_parts=A.REN_R1_PREFIX | A.REN_R2_PREFIX)]
            prog = Program(True, ops1, ops2, Filters(0))
            width = max(a, b)
        else:
            prog = Program(False, [Op(A.OP_CUT, length=a), Op(A.OP_CUT, length=-b),
                                   Op(A.OP_RENAME, rename_parts=A.REN_OWN_PREFIX | A.REN_OWN_SUFFIX)], [], Filters(0))
            width = min(MAX_N, a + b + 10)
        soa_and_text(prog, umi_records(rng, 2 if paired else 1, width), flags)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [A.AD_NI_BACK, A.AD_NI_FRONT], ids=["ni_back", "ni_front"])
def test_homopolymer_prefilter_reads_shorter_than_min_overlap(kind):
    """k_prefilter_homo: a read shorter than min_overlap can still match with deletions ("GGGG" against G x 128 at
    rate 0.3, min_overlap 5: five adapter characters, one error).  The prefilter used to bound the alignment length by
    the read characters plus the foreign ones and dropped such reads; found by test_random_program[21]."""
    reads = [(f"s{i}", "G" * n + tail, "I" * (n + len(tail))) for i, (n, tail) in
             enumerate((n, t) for n in range(0, 9) for t in ("", "T", "TA"))]
    reads = reads + [(r[0] + "r", r[1][::-1], r[2]) for r in reads]
    for m in (13, 20, 100, 128):
        for rate, mo in ((0.3, 5), (0.3, 4), (0.45, 7), (0.2, 6), (1.0, 3)):
            check_locate(Op(A.OP_ALIGN, adapter_kind=kind, adapter="G" * m, min_overlap=mo, max_error_rate=rate), reads)


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, A.PLAN_EMIT_G16], ids=["emit_stage", "emit_g16"])
def test_revcomp_every_byte(flags):
    """REVCOMP: all IUPAC letters in both cases and other printable bytes, with and without UMI parts, with QTRIM in
    front of it."""
    rng = random.Random(3)
    npr = np.random.default_rng(3)
    alphabet = G.IUPAC + G.IUPAC.lower() + "xz*.#0~-"
    recs = []
    for i in range(600):
        n = rng.choice([0, 1, 15, 16, 17, 33, 100, MAX_N, rng.randint(0, MAX_N)])
        recs.append((f"v{i} c", G.draw(npr, alphabet, n), G.draw(npr, "".join(G.QCHARS), n)))
    for ops in ([Op(A.OP_REVCOMP)],
                [Op(A.OP_QTRIM, cutoff_front=10, cutoff_back=20), Op(A.OP_REVCOMP)],
                [Op(A.OP_CUT, length=4), Op(A.OP_CUT, length=-17),
                 Op(A.OP_RENAME, rename_parts=A.REN_OWN_PREFIX | A.REN_OWN_SUFFIX),
                 Op(A.OP_QTRIM, cutoff_front=5, cutoff_back=15, quality_base=64), Op(A.OP_REVCOMP)]):
        soa_and_text(Program(False, ops, [], Filters(0)), [recs], flags)


HEADER_PROGRAM_OPS = [Op(A.OP_STRIP_SUFFIX, suffix="/1"), Op(A.OP_CUT, length=5),
                      Op(A.OP_RENAME, rename_parts=A.REN_R1_PREFIX | A.REN_R2_PREFIX)]


def header_program(paired):
    if paired:
        return Program(True, HEADER_PROGRAM_OPS, [Op(A.OP_STRIP_SUFFIX, suffix="/2")] + HEADER_PROGRAM_OPS[1:], Filters(0))
    return Program(False, HEADER_PROGRAM_OPS[:2] + [Op(A.OP_RENAME, rename_parts=A.REN_OWN_PREFIX)], [], Filters(0))


def header_records(n_mates, long_len, long_mate=None):
    """Short records around one record whose header is long_len bytes (on every mate, or only on long_mate)."""
    mates = [[] for _ in range(n_mates)]
    for i in range(40):
        for m in range(n_mates):
            h = f"h{i} c/{m + 1}"
            if i == 20:  # the same id on both mates
                h = "x" * 10 + " " + "y" * (long_len - 11 if long_mate in (None, m) else 5)
            mates[m].append((h, "ACGTACGTAC" * (i % 5), "I" * (10 * (i % 5))))
    return mates


@pytest.mark.gpu
@pytest.mark.parametrize("paired", [False, True], ids=["single", "paired"])
def test_header_limit_65535_is_accepted(paired):
    mates = header_records(2 if paired else 1, 65535)
    for flags in (0, A.PLAN_EMIT_G16):
        soa_and_text(header_program(paired), mates, flags)
    # the id itself at the limit: the whole header is the id
    mates = [[("z" * 65535 if i == 3 else f"h{i}", r[1], r[2]) for i, r in enumerate(mate)] for mate in mates]
    soa_and_text(header_program(paired), mates)


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["soa", "text"])
@pytest.mark.parametrize("mate", [0, 1], ids=["r1", "r2"])
def test_header_limit_65536_is_an_error(mate, form):
    """A header of 65 536 bytes is CSQ_ERR_LIMIT in both batch forms, on either mate; the plan stays usable."""
    prog = header_program(True)
    bad = header_records(2, 65536, long_mate=mate)
    good = header_records(2, 65535)
    want = oracle_run(prog, good)
    batch, keep = oracle.make_batch(*bad)
    assert oracle.run_batch(prog, batch)["status"] == A.ERR_LIMIT
    with FlagPlan(prog, 0) as plan:
        with pytest.raises(native.NativeError) as e:
            if form == "soa":
                plan.run_batch(batch, 1 << 20)
            else:
                plan.run_text([G.fastq_text(m) for m in bad], len(bad[0]), 1 << 20)
        assert e.value.code == A.ERR_LIMIT and f"{mate + 1}" in str(e.value) and "65535" in str(e.value), str(e.value)
        check(prog, good, want, plan, capacity_for(want))
        check(prog, good, want, plan, capacity_for(want), slot=1, text_eol="\n")


def c_ops(ops, patch=None):
    arr = (A.csq_op * max(1, len(ops)))()
    for i, op in enumerate(ops):
        arr[i] = op.to_c()
    if patch:
        patch(arr)
    return arr


def plan_create(ops1, ops2=None, patch1=None):
    """csq_plan_create on raw csq_op arrays (some rows hold values Op.to_c refuses to build). -> (code, message)"""
    import ctypes as C

    a1 = c_ops(ops1, patch1)
    a2 = c_ops(ops2 or [])
    flt = Filters(0).to_c()
    h = C.c_void_p()
    rc = native.lib().csq_plan_create(a1, len(ops1), a2, len(ops2 or []), C.byref(flt), 0, 0, C.byref(h))
    msg = native.lib().csq_last_error().decode() if rc else ""
    if h:
        native.lib().csq_plan_destroy(h)
    return rc, msg


def cut(n=1):
    return Op(A.OP_CUT, length=n)


def align(**kw):
    args = dict(adapter_kind=A.AD_BACK, adapter="ACGTACGT", max_error_rate=0.1, min_overlap=3)
    args.update(kw)
    return Op(A.OP_ALIGN, **args)


def strip(s):
    return Op(A.OP_STRIP_SUFFIX, suffix=s)


def rename(parts=0):
    return Op(A.OP_RENAME, rename_parts=parts)


def set_field(i, **kw):
    def patch(arr):
        for k, v in kw.items():
            setattr(arr[i], k, v)
    return patch


QT = Op(A.OP_QTRIM, cutoff_back=20)
RC = Op(A.OP_REVCOMP)
VALIDATION = [
    # (ops r1, ops r2, patch of r1, expected code, message substring)
    ("32 ops", ([cut()] * 11 + [align()]) * 2 + [cut()] * 8, None, None, 0, ""),
    ("33 ops", ([cut()] * 11 + [align()]) * 2 + [cut()] * 9, None, None, A.ERR_INVALID, "program of 33 ops"),
    ("12 scalar ops", [cut()] * 12 + [align()], None, None, 0, ""),
    ("13 scalar ops", [cut()] * 13 + [align()], None, None, A.ERR_INVALID, "more than 12 scalar ops"),
    ("13 scalar ops behind", [align()] + [cut()] * 13, None, None, A.ERR_INVALID, "more than 12 scalar ops"),
    ("strip after rename", [rename(), strip("/1")], None, None, A.ERR_INVALID, "STRIP_SUFFIX must come before RENAME"),
    ("5 suffixes", [strip("a")] * 5, None, None, A.ERR_INVALID, "too many / too long name suffixes"),
    ("9-byte suffix", [strip("abcdefgh")], None, set_field(0, suffix_len=9), A.ERR_INVALID, "too many / too long"),
    ("empty suffix", [strip("a")], None, set_field(0, suffix_len=0), A.ERR_INVALID, "empty name suffix"),
    ("two renames", [rename(), cut(), rename()], None, None, A.ERR_INVALID, "more than one RENAME"),
    ("cut 65535", [cut(65535), cut(-65535)], None, None, 0, ""),
    ("cut 65536", [cut(65536)], None, None, A.ERR_INVALID, "cut length out of range"),
    ("cut -65536", [Op(A.OP_COND_CUT, length=-65536)], None, None, A.ERR_INVALID, "cut length out of range"),
    ("op behind qtrim", [QT, cut()], None, None, A.ERR_INVALID, "only REVCOMP may follow QTRIM"),
    ("revcomp not last", [RC, cut()], None, None, A.ERR_INVALID, "REVCOMP must be the last op"),
    ("revcomp paired", [cut(), RC], [cut(), RC], None, A.ERR_INVALID, "REVCOMP is a single-end op"),
    ("rename on one mate", [rename()], [cut()], None, A.ERR_INVALID, "paired programs must carry the same RENAME"),
    ("rename parts differ", [rename(A.REN_R1_PREFIX)], [rename(A.REN_R2_PREFIX)], None, A.ERR_INVALID, "the same RENAME"),
    ("own parts paired", [rename(A.REN_OWN_PREFIX)], [rename(A.REN_OWN_PREFIX)], None, A.ERR_INVALID, "uses r1/r2 parts"),
    ("r1 part single", [rename(A.REN_R1_PREFIX)], None, None, A.ERR_INVALID, "single-end RENAME uses own parts"),
    ("adapter of 0", [align()], None, set_field(0, adapter_len=0), A.ERR_LIMIT, "adapter length 0 outside 1..128"),
    ("adapter of 129", [align()], None, set_field(0, adapter_len=129), A.ERR_LIMIT, "adapter length 129 outside"),
    ("adapter of 128", [align(adapter="ACGT" * 32)], None, None, 0, ""),
    ("adapter char", [align(adapter="ACGTNCGT")], None, None, A.ERR_INVALID, "'N' is not one of ACGT"),
    ("negative rate", [align(max_error_rate=-0.1)], None, None, A.ERR_INVALID, "bad max_error_rate"),
    ("min_overlap 0", [align(min_overlap=0)], None, None, A.ERR_INVALID, "min_overlap must be >= 1"),
    ("adapter_id 30", [align(adapter_id=30)], None, None, 0, ""),
    ("adapter_id 31", [align(adapter_id=31)], None, None, A.ERR_INVALID, "adapter_id 31 outside -1..30"),
    ("adapter_id -2", [align(adapter_id=-2)], None, None, A.ERR_INVALID, "adapter_id -2 outside -1..30"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("row", VALIDATION, ids=[r[0] for r in VALIDATION])
def test_program_validation(row):
    name, ops1, ops2, patch, code, needle = row
    rc, msg = plan_create(ops1, ops2, patch)
    assert rc == code and needle in msg, (name, rc, msg)


@pytest.mark.gpu
def test_generated_programs_are_valid():
    for seed in range(N_SEEDS):
        prog, _ = program_case(seed)
        rc, msg = plan_create(prog.ops_r1, prog.ops_r2 if prog.paired else None)
        assert rc == 0, (seed, msg)
