"""Random op programs that csq_plan_create accepts, and reads and headers that reach the edges of the per-read
scalar ops, quality trimming, the Renamer id and the emitters.  Shared by tests/test_gpu_programs.py (GPU against
the oracle) and tests/test_oracle.py (oracle against the restated cutadapt modifiers)."""

import numpy as np

from cutseq_b200 import _abi as A
from cutseq_b200.program import Filters, Op, Program
from oracle import oracle

KINDS = [A.AD_BACK, A.AD_BACK_ANYWHERE, A.AD_RIGHTMOST_FRONT, A.AD_PREFIX, A.AD_SUFFIX, A.AD_NI_FRONT, A.AD_NI_BACK, A.AD_FRONT]
MAX_N = A.CSQ_MAX_READ_LEN
# Python's str.split() blanks; a FASTQ text line cannot hold '\n', and a '\r' in front of a line end is dropped
PY_BLANKS = [9, 10, 11, 12, 13, 28, 29, 30, 31, 32]
TEXT_BLANKS = [9, 11, 12, 28, 29, 30, 31, 32]
EDGE_LENGTHS = [0, 1, 15, 16, 17, 31, 32, 33, MAX_N]
LOW_RUNS = [15, 16, 17, 31, 32, 33]  # fetch16 boundaries of the quality scans
IUPAC = "ACGTUMRWSYKVHDBN"
LONG_HEADERS = [4001, 20000, 65535]
MAX_PRE = 12  # CSQ_MAX_PRE: scalar ops in a row (csq_internal.h)
# header endings the STRIP_SUFFIX ops are drawn from (mate 2 carries '2' where mate 1 carries '1')
ENDINGS = ["/1", ".1", "1", "_1", ":N:0", "x", "ACGT", "1:N:0:1", "abcdefgh", " 1"]


def mate2_suffix(s):
    return s[:-1] + "2" if s.endswith("1") else s


def scalar_op(rng, L, cond_cut=True):
    kind = rng.choice([A.OP_CUT, A.OP_CUT, A.OP_COND_CUT]) if cond_cut else A.OP_CUT
    big = rng.random() < 0.07  # most cuts leave something of the read
    length = rng.choice([L, L + 1, MAX_N, 65535] if big else [0, 1, 1, 15, 16, 17]) * rng.choice([1, -1])
    fmin = rng.choice([0, 1, L, L + 1, MAX_N + 1]) if kind == A.OP_COND_CUT else 0
    return Op(kind, length=length, force_trim_min_length=fmin)


def align_op(rng, adapter_id):
    if rng.random() < 0.75:
        m = rng.choice([1, 2, 3, 4, 6, 8, 8, 10, 12, 12, 13, 15, 16, 17, 20, 20, 20, 25, 31, 32, 33])
    else:
        m = rng.choice([40, 57, 63, 64, 65, 96, 97, 100, 127, 128])
    if m >= 13 and rng.random() < 0.15:
        adapter = rng.choice("ACGT") * m  # the homopolymer kernels
    else:
        adapter = "".join(rng.choice("ACGT") for _ in range(m))
    rate = rng.choice([0.0, 0.05, 0.1, 0.15, 0.2, 0.25, 0.3])
    if m >= 8 and rng.random() < 0.2:
        rate = float(rng.choice([1, 2, 3]))  # >= 1: an absolute error count
    return Op(A.OP_ALIGN, adapter_kind=rng.choice(KINDS), adapter=adapter, min_overlap=rng.choice([1, 2, 3, 5, m, m + 3]),
              max_error_rate=rate, adapter_id=adapter_id)


def max_scalar_run(ops):
    run = best = 0
    for op in ops:
        if op.kind in (A.OP_CUT, A.OP_COND_CUT, A.OP_RENAME):
            run += 1
            best = max(best, run)
        elif op.kind == A.OP_ALIGN:
            run = 0
    return best


def random_program(rng, paired, cond_cut=True, revcomp=True):
    """A program of CSQ_MAX_OPS ops at most: 0-4 STRIP_SUFFIX, 0-6 ALIGN with runs of 0-12 scalar ops around them,
    an optional RENAME in front of, between or behind the ALIGN ops, an optional QTRIM (and, single-end, REVCOMP)
    last.  Paired programs pair step t of mate 1 with step t of mate 2 (same RENAME, independent parameters)."""
    L = rng.choice([16, 32, 100, 150, MAX_N])  # read length the cut lengths and COND_CUT bounds are drawn around
    n_align = rng.choice([0, 1, 1, 2, 2, 3, 4, 6])
    n_suffix = rng.choice([0, 0, 1, 2, 4])
    runs = [rng.choice([0, 0, 0, 1, 1, 2, 3, 5, 12]) for _ in range(n_align + 1)]
    rename_at = rng.choice([None, 0, n_align] + list(range(1, n_align)))  # index of the run that holds it
    qtrim = rng.random() < 0.7
    rc = revcomp and not paired and rng.random() < 0.25
    while n_suffix + n_align + sum(runs) + 2 * (rename_at is not None) + qtrim + rc > A.CSQ_MAX_OPS:
        i = max(range(len(runs)), key=lambda j: runs[j])
        runs[i] -= 1
    if rename_at is not None and runs[rename_at] == 12:
        runs[rename_at] = 11
    parts_bits = [A.REN_R1_PREFIX, A.REN_R2_PREFIX] if paired else [A.REN_OWN_PREFIX, A.REN_OWN_SUFFIX]
    parts = sum(b for b in parts_bits if rng.random() < 0.6)
    if rng.random() < 0.1:
        parts = 0
    ids = rng.sample(range(31), 2 * n_align)
    suffixes = [rng.choice(ENDINGS) if rng.random() < 0.7 else "".join(rng.choice("ab1:/.") for _ in range(rng.randint(1, 8)))
                for _ in range(n_suffix)]
    suffixes = [s if not s.endswith(("2", "3")) else s + "x" for s in suffixes][:4]
    suffixes = [s[:A.CSQ_MAX_SUFFIX] for s in suffixes]
    qt = Op(A.OP_QTRIM, cutoff_front=rng.choice([0, 0, 1, 5, 10, 20, rng.randint(0, 40), 40]),
            cutoff_back=rng.choice([0, 1, 10, 15, 20, 30, rng.randint(0, 40), 40]), quality_base=rng.choice([33, 33, 64]))
    rename_slot = rng.randint(0, runs[rename_at]) if rename_at is not None else 0
    umi_cut = rename_at is not None and runs[rename_at] + 2 <= MAX_PRE and rng.random() < 0.3
    mates = []
    for mate in range(2 if paired else 1):
        ops = [Op(A.OP_STRIP_SUFFIX, suffix=s if mate == 0 else mate2_suffix(s)) for s in suffixes]
        for r in range(n_align + 1):
            run = [scalar_op(rng, L, cond_cut) for _ in range(runs[r])]
            if rename_at == r:  # at the same step in both mates
                run.insert(rename_slot, Op(A.OP_RENAME, rename_parts=parts))
                if umi_cut:  # a UMI part of a whole read
                    run.insert(rename_slot, Op(A.OP_CUT, length=rng.choice([MAX_N, 65535]) * rng.choice([1, -1])))
            ops += run
            if r < n_align:
                ops.append(align_op(rng, rng.choice([-1, ids[2 * r + mate]])))
        if qtrim:
            ops.append(Op(A.OP_QTRIM, cutoff_front=qt.cutoff_front, cutoff_back=qt.cutoff_back, quality_base=qt.quality_base)
                       if mate == 0 or rng.random() < 0.5 else
                       Op(A.OP_QTRIM, cutoff_front=rng.randint(0, 40), cutoff_back=rng.randint(0, 40), quality_base=qt.quality_base))
        if rc:
            ops.append(Op(A.OP_REVCOMP))
        mates.append(ops)
    if paired:  # mate 2 sometimes cuts where mate 1 aligns (compile_paired's inline barcodes)
        for t, op in enumerate(mates[1]):
            if op.kind == A.OP_ALIGN and rng.random() < 0.25:
                trial = mates[1][:t] + [scalar_op(rng, L, cond_cut)] + mates[1][t + 1:]
                if max_scalar_run(trial) <= MAX_PRE:
                    mates[1] = trial
    used = [sorted({op.adapter_id for op in ops if op.kind == A.OP_ALIGN and op.adapter_id >= 0}) for ops in mates]
    flt = Filters(min_length=rng.choice([0, 0, 1, 1, 20, 20, 20, MAX_N, MAX_N + 1]))
    if rng.random() < 0.4:
        flt.untrimmed_enabled = True
        req = []
        for m in range(len(mates)):
            bits = sum(1 << b for b in used[m] if rng.random() < 0.6)
            if rng.random() < 0.15:
                bits |= 1 << rng.choice([b for b in range(31) if b not in used[m]])  # an id no op carries
            req.append(bits)
        flt.required_r1 = req[0]
        flt.required_r2 = req[1] if paired else 0
    return Program(paired, mates[0], mates[1] if paired else [], flt)


# ---- reads ----

def plant(rng, q, adapter, alphabet="ACGT"):
    """A partial, mutated copy of the adapter at the read start, at its end or anywhere (as random_reads does)."""
    n, m = len(q), len(adapter)
    cut = rng.randint(1, m)
    piece = list(adapter[:cut] if rng.random() < 0.5 else adapter[m - cut:])
    for _ in range(rng.choice([0, 0, 1, 1, 2, 3, 5])):
        if not piece:
            break
        pos = rng.randrange(len(piece))
        t = rng.random()
        if t < 0.5:
            piece[pos] = rng.choice(alphabet)
        elif t < 0.75:
            del piece[pos]
        else:
            piece.insert(pos, rng.choice(alphabet))
    where = rng.random()
    pos = 0 if where < 0.3 else (max(0, n - len(piece)) if where < 0.65 else rng.randint(0, max(0, n - 1)))
    q[pos : pos + len(piece)] = piece
    del q[n:]


def draw(npr, alphabet, n):
    """n characters of the alphabet (numpy: drawing reads byte by byte with random.choices is slow)."""
    a = np.frombuffer(alphabet.encode("latin-1"), dtype=np.uint8)
    return a[npr.integers(0, a.size, n)].tobytes().decode("latin-1")


def qual_chars(rng, npr, n, qtrims):
    """Qualities '!'..'~', with runs of low quality of 15-17 / 31-33 at either end, and runs whose running sums
    return to exactly 0 under one of the program's QTRIM cutoffs (the `s > max` tie of quality_trim_index)."""
    base = qtrims[0].quality_base if qtrims else 33
    if rng.random() < 0.7:  # mostly good reads, whose trimming stops near the ends
        q = list(draw(npr, "".join(QCHARS[base - 33 + 28:base - 33 + 45]), n).encode("latin-1"))
    else:
        q = list(draw(npr, "".join(QCHARS), n).encode("latin-1"))
    t = rng.random()
    if n and t < 0.3:
        k = min(n, rng.choice(LOW_RUNS))
        lo = [rng.randint(33, 45) for _ in range(k)]
        if rng.random() < 0.5:
            q[:k] = lo
        else:
            q[n - k:] = lo
    elif n and t < 0.55 and qtrims:
        op = rng.choice(qtrims)
        c = rng.choice([op.cutoff_front, op.cutoff_back]) + op.quality_base
        k = min(n, rng.choice(LOW_RUNS + [2, 4, 8]))
        run = []
        while len(run) < k:
            d = rng.randint(0, 6)
            run += [c - d, c + d] if rng.random() < 0.5 else [c + d, c - d]
        run = [min(126, max(33, x)) for x in run[:k]]
        if rng.random() < 0.5:
            q[:k] = run
        else:
            q[n - k:] = run
    return "".join(map(chr, q))


PRINTABLE = [chr(c) for c in range(33, 127)]
QCHARS = PRINTABLE


def header_text(rng, n, blanks):
    if n > 256:  # long headers: a random block repeated (drawing 65 535 bytes one by one is slow)
        block = header_text(rng, 256, blanks)
        return (block * (n // 256 + 1))[:n]
    return "".join(chr(rng.choice(blanks)) if rng.random() < 0.15 else c for c in rng.choices(PRINTABLE, k=n))


def random_header(rng, i, blanks, endings):
    t = rng.random()
    if t < 0.004 * 3:
        body = f"L{i}" + header_text(rng, rng.choice(LONG_HEADERS), blanks)
    elif t < 0.5:
        body = f"r{i}"
    elif t < 0.8:
        body = f"r{i}" + chr(rng.choice(blanks)) + header_text(rng, rng.randint(0, 40), blanks)
    else:
        body = header_text(rng, rng.randint(0, 60), blanks)
    end = rng.choice(endings) if endings and rng.random() < 0.5 else ""
    return (body + end)[:65535]


def strip(name, ops):
    for op in ops:
        if op.kind == A.OP_STRIP_SUFFIX and name.endswith(op.suffix):
            name = name[: len(name) - len(op.suffix)]
    return name


def paired_ok(h1, h2, prog):
    """dnaio's paired reader on the headers as they stand, and PairedEndRenamer on the stripped ones."""
    if not oracle.names_match(h1, h2):
        return False
    has_rename = any(op.kind == A.OP_RENAME for op in prog.ops_r1)
    return not has_rename or oracle.names_match(strip(h1, prog.ops_r1), strip(h2, prog.ops_r2))


def random_mates(rng, prog, n, lengths=None, blanks=TEXT_BLANKS):
    """n records per mate for the program: read lengths from `lengths` (default: the 16-byte edges and anything up to
    CSQ_MAX_READ_LEN), planted copies of the mate's adapters, N, lower case and (REVCOMP) IUPAC letters and other
    printable bytes; headers that end in the program's suffixes and that pass dnaio's pairing rules."""
    n_mates = 2 if prog.paired else 1
    opss = [prog.ops_r1, prog.ops_r2][:n_mates]
    revcomp = prog.ops_r1 and prog.ops_r1[-1].kind == A.OP_REVCOMP
    out = [[] for _ in range(n_mates)]
    npr = np.random.default_rng(rng.getrandbits(64))
    for i in range(n):
        names = None
        for attempt in range(20):
            endings = [op.suffix for op in opss[0] if op.kind == A.OP_STRIP_SUFFIX] + ["/1", " 1:N:0"]
            h1 = random_header(rng, i, blanks, endings if attempt < 10 else [])
            if n_mates == 1:
                names = [h1]
                break
            h2 = h1[:-1] + "2" if h1.endswith("1") else h1
            if rng.random() < 0.2 and (" " in h1 or "\t" in h1):  # another comment behind the dnaio id
                cut = min(h1.find(c) for c in " \t" if c in h1)
                h2 = h2[:cut] + h2[cut] + header_text(rng, rng.randint(0, 20), [32])
            if paired_ok(h1, h2, prog):
                names = [h1, h2]
                break
        if names is None:
            names = [f"p{i}x", f"p{i}x"]
            assert paired_ok(*names, prog)
        for m, ops in enumerate(opss):
            ln = rng.choice(lengths) if lengths else (rng.choice(EDGE_LENGTHS) if rng.random() < 0.4 else rng.randint(0, MAX_N))
            alphabet = IUPAC + IUPAC.lower() if revcomp and rng.random() < 0.3 else "ACGT"
            q = list(draw(npr, alphabet, ln))
            for _ in range(ln // 50):
                q[rng.randrange(ln)] = "N"
            adapters = [op.adapter for op in ops if op.kind == A.OP_ALIGN]
            if ln and adapters:
                for _ in range(rng.choice([0, 1, 1, 2, 3])):
                    plant(rng, q, rng.choice(adapters))
            if revcomp and ln and rng.random() < 0.2:
                q[rng.randrange(ln)] = rng.choice("xz*.#0~")
            s = "".join(q)
            if rng.random() < 0.05:
                s = s.lower()
            qtrims = [op for op in ops if op.kind == A.OP_QTRIM]
            out[m].append((names[m], s, qual_chars(rng, npr, len(s), qtrims)))
    return out


def fastq_text(records, eol="\n"):
    return "".join(f"@{h}{eol}{s}{eol}+{eol}{q}{eol}" for h, s, q in records).encode("latin-1")
