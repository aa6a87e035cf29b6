"""The adapter aligner across its whole range: every adapter length class up to CSQ_MAX_ADAPTER, reads up to
CSQ_MAX_READ_LEN, every kernel variant of the dispatch (k_align<M> with the column in registers, k_align<0> with the
column in local memory, k_align_split for homopolymer 100-mers; k_prefilter with 1-4 bit-vector words,
k_prefilter_fs, k_prefilter_homo) against the CPU oracle.  Bit-exact: every comparison is ==."""

import math
import random
from fractions import Fraction

import pytest

from cutseq_b200 import _abi as A
from cutseq_b200 import native
from cutseq_b200.program import Filters, Op, Program
from oracle import oracle
from tests.test_gpu_parity import KINDS, check_locate, compare_with_oracle, random_reads

pytestmark = pytest.mark.gpu

MAX_M, MAX_N = A.CSQ_MAX_ADAPTER, A.CSQ_MAX_READ_LEN
# register-resident lengths 1..34 (1, 21 / 22 and 32 are where the prefilter changes form), the local-memory DP from
# 35 on, and the word boundaries of the bit vectors and of peq: the row-m bit (m - 1) & 31 is bit 31 or bit 0 of the
# last word at m = 32, 33, 64, 65, 96, 97, 128
SWEEP_M = [1, 2, 4, 7, 16, 21, 22, 31, 32, 33, 34, 35, 48, 63, 64, 65, 66, 80, 95, 96, 97, 99, 100, 101, MAX_M - 1, MAX_M]
SWEEP_RATES = [0.0, 0.1, 0.2, 0.35]
KIND_IDS = {A.AD_BACK: "back", A.AD_BACK_ANYWHERE: "back_anywhere", A.AD_RIGHTMOST_FRONT: "rightmost_front",
            A.AD_PREFIX: "prefix", A.AD_SUFFIX: "suffix", A.AD_NI_FRONT: "ni_front", A.AD_NI_BACK: "ni_back",
            A.AD_FRONT: "front"}


def random_adapter(rng, m):
    """m random bases, not all the same (homopolymers take other kernels) unless m == 1."""
    while True:
        adapter = "".join(rng.choice("ACGT") for _ in range(m))
        if m == 1 or len(set(adapter)) > 1:
            return adapter


def random_bases(rng, n, alphabet="ACGT"):
    return "".join(rng.choices(alphabet, k=n))


def read(name, seq):
    return (name, seq, "I" * len(seq))


def sweep_case(m, kind):
    """(op, reads) of the length sweep for one adapter length and kind: error rate and minimum overlap rotate over
    the (m, kind) pairs, so that every kind meets every rate and every minimum overlap over consecutive lengths; reads
    of 0 .. CSQ_MAX_READ_LEN bases, a read of the maximum length first and last."""
    mi, ki = SWEEP_M.index(m), KINDS.index(kind)
    i = mi * len(KINDS) + ki
    rng = random.Random(7000 + i)
    adapter = random_adapter(rng, m)
    rate = SWEEP_RATES[(mi + ki) % len(SWEEP_RATES)]  # not i: len(KINDS) is a multiple of len(SWEEP_RATES)
    op = Op(A.OP_ALIGN, adapter_kind=kind, adapter=adapter, min_overlap=[1, 3, m][(mi + ki) % 3], max_error_rate=rate)
    lengths = sorted({0, 1, 2, 5, 17, 31, 32, 33, max(m - 1, 0), m, m + 1, 100, 150, 300, 511, 512, 640, MAX_N - 1, MAX_N})
    reads = random_reads(rng, adapter, 120, lengths=lengths, back_to_back=0.5)
    ends = random_reads(rng, adapter, 2, lengths=[MAX_N], back_to_back=0.5)
    return op, [ends[0]] + reads + [ends[1]]


def test_sweep_rotation_reaches_every_rate_and_overlap():
    for kind in KINDS:
        ops = [sweep_case(m, kind)[0] for m in SWEEP_M]
        assert {op.max_error_rate for op in ops} == set(SWEEP_RATES), kind
        assert {1, 3} <= {op.min_overlap for op in ops} and any(op.min_overlap == len(op.adapter) > 3 for op in ops), kind


@pytest.mark.parametrize("m", SWEEP_M, ids=[f"m{m}" for m in SWEEP_M])
def test_length_sweep(m):
    for kind in KINDS:
        op, reads = sweep_case(m, kind)
        check_locate(op, reads)


def mutate(rng, piece, subs, indel=None):
    """piece with `subs` substitutions at distinct positions (each by a different base) and, if indel is 'ins' /
    'del', one inserted / deleted base."""
    p = list(piece)
    for pos in rng.sample(range(len(p)), min(subs, len(p))):
        p[pos] = rng.choice([c for c in "ACGT" if c != p[pos]])
    if indel == "ins":
        p.insert(rng.randint(1, len(p) - 1), rng.choice("ACGT"))
    elif indel == "del":
        del p[rng.randrange(len(p))]
    return "".join(p)


@pytest.mark.parametrize("kind", KINDS, ids=[KIND_IDS[k] for k in KINDS])
def test_packed_cell_limits(kind):
    """The 10-bit fields of the packed DP cell at their limits: reads of CSQ_MAX_READ_LEN bases (origin + 128 reaches
    1023 for the kinds with a free read start) and adapters of CSQ_MAX_ADAPTER bases (with a free adapter start the
    cells of row m start with origin -128, field value 0), at error rate 0 and 0.45."""
    rng = random.Random(300 + kind)
    for m in (1, MAX_M):
        adapter = random_adapter(rng, m)
        for rate in (0.0, 0.45):
            k = int(rate * m)
            reads = []
            for t in range(3):
                full = adapter if t == 0 else mutate(rng, adapter, min(k, m - 1) if t == 1 else k // 2)
                reads.append(read("start", full + random_bases(rng, MAX_N - len(full))))
                reads.append(read("end", random_bases(rng, MAX_N - len(full)) + full))
                reads.append(read("both", full + random_bases(rng, MAX_N - 2 * len(full)) + full))
                reads.append(read("absent", random_bases(rng, MAX_N) if m > 1 else "N" * MAX_N))
            # partial copies: adapter suffixes at the read start (origin -(m - L)), prefixes at its end
            for length in sorted({x for x in (1, 2, m // 2, m - 1, m) if 1 <= x <= m}):
                reads.append(read("sfx", adapter[m - length:] + random_bases(rng, MAX_N - length)))
                reads.append(read("pfx", random_bases(rng, MAX_N - length) + adapter[:length]))
            reads.insert(1, read("empty", ""))
            reads.append(read("lower", (adapter + random_bases(rng, MAX_N - m)).lower()))  # full length, last
            for mo in (1, m):
                check_locate(Op(A.OP_ALIGN, adapter_kind=kind, adapter=adapter, min_overlap=mo, max_error_rate=rate), reads)


def test_read_length_limit_soa_and_text():
    """A read of CSQ_MAX_READ_LEN + 1 bases is refused (ERR_LIMIT) as an SoA batch and as a text batch; one of
    CSQ_MAX_READ_LEN bases goes through, with a CSQ_MAX_ADAPTER-mer."""
    rng = random.Random(11)
    adapter = random_adapter(rng, MAX_M)
    prog = Program(False, [Op(A.OP_ALIGN, adapter_kind=A.AD_BACK_ANYWHERE, adapter=adapter, min_overlap=3, max_error_rate=0.2)], [],
                   Filters(0, False, 0, 0))
    ok = [read("a", random_bases(rng, MAX_N - MAX_M) + adapter), read("b", random_bases(rng, MAX_N))]
    compare_with_oracle(prog, [ok])
    bad = ok + [read("c", random_bases(rng, MAX_N + 1))]
    batch, keep = oracle.make_batch(bad)
    text = "".join(f"@{n}\n{s}\n+\n{q}\n" for n, s, q in bad).encode()
    with native.Plan(prog) as plan:
        with pytest.raises(native.NativeError) as e:
            plan.run_batch(batch)
        assert e.value.code == A.ERR_LIMIT
        with pytest.raises(native.NativeError) as e:
            plan.run_text([text], len(bad))
        assert e.value.code == A.ERR_LIMIT
        # the plan stays usable
        good = "".join(f"@{n}\n{s}\n+\n{q}\n" for n, s, q in ok).encode()
        ok_batch, keep = oracle.make_batch(ok)
        assert plan.run_text([good], len(ok)) == plan.run_batch(ok_batch)


def rounding_edges(max_errors, m):
    """Aligned lengths L <= m at which cutadapt's floor(L * rate) in doubles is one less than the exact value, for an
    error rate (the decimal fraction written) or an absolute count (rate = count / m, as SingleAdapter.__init__ makes
    it).  Only the L whose double value stays within k = int(rate * m) can decide a match.  -> [(L, floor in doubles)]"""
    rate = max_errors / m if max_errors >= 1 else max_errors
    exact = Fraction(int(max_errors), m) if max_errors >= 1 else Fraction(str(max_errors))
    k = int(rate * m)
    out = []
    for length in range(1, m + 1):
        dbl = math.floor(length * rate)
        if dbl != math.floor(length * exact) and dbl <= k:
            out.append((length, dbl))
    return out


def edge_cases():
    """(max_errors, m, L, thr[L]) where double rounding decides: the three named in the threshold table of the tests
    (rate 0.29 at m = 128, L = 100; 18 errors on a 66-mer at L = 55; 30 errors on a 44-mer at L = 22) plus, over
    more rates, counts and lengths, the shortest and longest such L of every (max_errors, m)."""
    found = {}
    for max_errors in (0.1, 0.15, 0.2, 0.29, 0.3, 0.35, 0.45, 7.0, 13.0, 18.0, 30.0):
        for m in (13, 33, 44, 57, 66, 97, 100, 101, 120, MAX_M):
            if max_errors >= 1 and max_errors >= m:
                continue
            edges = rounding_edges(max_errors, m)
            if edges:
                found[(max_errors, m)] = edges
    named = [(0.29, MAX_M, 100), (18.0, 66, 55), (30.0, 44, 22)]
    cases = []
    for max_errors, m, length in named:
        dbl = dict(found[(max_errors, m)])[length]  # KeyError: the search no longer finds a documented case
        cases.append((max_errors, m, length, dbl))
    for (max_errors, m), edges in sorted(found.items()):
        for length, dbl in {edges[0], edges[-1]}:
            if (max_errors, m, length) not in [c[:3] for c in cases]:
                cases.append((max_errors, m, length, dbl))
    return cases


def test_rounding_edges_are_found():
    cases = edge_cases()
    assert (0.29, MAX_M, 100, 28) in cases and (18.0, 66, 55, 14) in cases and (30.0, 44, 22, 14) in cases
    assert len(cases) >= 8


# partial copies that cover exactly L adapter bases: a prefix at the read's 3' end (last-column rule) for the 3'
# kinds, a suffix at its 5' end (row-m rule, origin -(m - L)) for the 5' kinds; the anchored kinds only at L = m
END_KINDS = (A.AD_BACK, A.AD_BACK_ANYWHERE, A.AD_NI_BACK)
START_KINDS = (A.AD_FRONT, A.AD_RIGHTMOST_FRONT, A.AD_NI_FRONT, A.AD_BACK_ANYWHERE)


@pytest.mark.parametrize("case", edge_cases(), ids=lambda c: f"err{c[0]:g}-m{c[1]}-L{c[2]}")
def test_error_threshold_edges(case):
    """thr[L] - 1, thr[L] and thr[L] + 1 errors on an alignment of exactly L adapter bases: substitutions only, and
    with one inserted or deleted base among them."""
    max_errors, m, length, thr = case
    rng = random.Random(f"{max_errors}/{m}/{length}")
    adapter = random_adapter(rng, m)
    kinds = {A.AD_PREFIX: "start", A.AD_SUFFIX: "end"} if length == m else {}
    kinds.update({k: "end" for k in END_KINDS})
    kinds.update({k: "start" for k in START_KINDS if k not in kinds})
    for kind, where in kinds.items():
        piece = adapter[:length] if where == "end" else adapter[m - length:]
        reads = []
        for errors in (thr - 1, thr, thr + 1):
            if errors < 0 or errors > length:
                continue
            for indel in (None, "ins", "del"):
                subs = errors - (indel is not None)
                if subs < 0 or (indel and length < 2):
                    continue
                for rep in range(4):
                    copy = mutate(rng, piece, subs, indel)
                    filler = random_bases(rng, rng.choice([0, 40, 150]))
                    reads.append(read(f"{errors}{indel}{rep}", copy + filler if where == "start" else filler + copy))
        check_locate(Op(A.OP_ALIGN, adapter_kind=kind, adapter=adapter, min_overlap=1, max_error_rate=max_errors), reads)


def homopolymer_reads(rng, letter, count):
    """Reads of 0 .. CSQ_MAX_READ_LEN bases with a run of `letter` at the start, at the end or both, scattered
    foreign bases (N too), and some runs or whole reads in lower case."""
    reads = []
    for i in range(count):
        n = rng.choice([0, 1, 5, 30, 99, 100, 101, 150, 300, 640, MAX_N - 1, MAX_N])
        body = list(random_bases(rng, n))
        for side in rng.choice([(0,), (1,), (0, 1)]):
            run = min(n, rng.choice([0, 3, 10, 20, 50, 99, 100, 101, 130, 400]))
            if side == 0:
                body[:run] = letter * run
            else:
                body[n - run:] = letter * run
        for _ in range(rng.choice([0, 0, 1, 2, 5, 12]) if n else 0):
            body[rng.randrange(n)] = rng.choice("ACGTN")
        s = "".join(body)
        t = rng.random()
        if t < 0.05:
            s = s.lower()
        elif t < 0.1:
            s = s.replace(letter, letter.lower())
        reads.append(read(f"h{i}", s))
    return reads


@pytest.mark.parametrize("kind", KINDS, ids=[KIND_IDS[k] for k in KINDS])
def test_homopolymer_100mers(kind):
    """k_align_split<100, 2 | 4> (and the prefilters in front of it) for every kind and letter: batches of 1, 63, 64
    and 65 reads leave idle lane pairs that still take part in the shuffles; a batch of a few thousand spreads the
    survivor lists over several CTAs."""
    ki = KINDS.index(kind)
    rng = random.Random(900 + kind)
    for li, letter in enumerate("ACGT"):
        rate = (0.0, 0.15, 0.3)[(ki + li) % 3]
        op = Op(A.OP_ALIGN, adapter_kind=kind, adapter=letter * 100, min_overlap=3, max_error_rate=rate)
        for size in (1, 63, 64, 65) + ((2500,) if li == ki % 4 else ()):
            check_locate(op, homopolymer_reads(rng, letter, size))


@pytest.mark.parametrize("kind", [A.AD_NI_FRONT, A.AD_NI_BACK], ids=["ni_front", "ni_back"])
def test_homopolymer_prefilter_lengths(kind):
    """k_prefilter_homo at adapter lengths other than 100, in front of k_align<M> and the local-memory DP."""
    rng = random.Random(950 + kind)
    for i, m in enumerate((1, 2, 31, 64, MAX_M - 1, MAX_M)):
        letter = "ACGT"[i % 4]
        rate = (0.0, 0.15, 0.3)[i % 3]
        op = Op(A.OP_ALIGN, adapter_kind=kind, adapter=letter * m, min_overlap=(1, 3)[i % 2], max_error_rate=rate)
        check_locate(op, homopolymer_reads(rng, letter, 300))


def chain_reads(rng, p5, mid, p7, count):
    """Reads for the long-adapter chain: a (mutated) copy of the anchored 5' adapter, the rightmost-front adapter
    somewhere inside, a (partial, mutated) 3' adapter and a poly-G tail, each present or not."""
    reads = []
    for i in range(count):
        parts = []
        if rng.random() < 0.6:
            parts.append(mutate(rng, p5, rng.choice([0, 0, 2, 6, 9])))
        parts.append(random_bases(rng, rng.choice([0, 20, 100, 250])))
        if rng.random() < 0.6:
            parts.append(mutate(rng, mid, rng.choice([0, 5, 20, 28, 29])))
            parts.append(random_bases(rng, rng.choice([0, 10, 80])))
        if rng.random() < 0.7:
            cut = rng.choice([len(p7), len(p7), 100, 60, 10, 3])
            parts.append(mutate(rng, p7[:cut], rng.choice([0, 1, 5, cut // 5])))
        if rng.random() < 0.5:
            parts.append("G" * rng.choice([5, 30, 100, 200]) + random_bases(rng, rng.choice([0, 0, 3])))
        s = "".join(parts)[:rng.choice([MAX_N, MAX_N, 400, 151])]
        reads.append(read(f"c{i}", s))
    return reads


@pytest.mark.parametrize("flags", [0, A.PLAN_EMIT_G16], ids=["emit_stage", "emit_g16"])
@pytest.mark.parametrize("paired", [False, True], ids=["single", "paired"])
def test_long_adapter_chain(paired, flags):
    """A 128-mer 3' adapter, an anchored 65-mer, a rightmost 97-mer and a poly-G 100-mer, one after another on the
    same read, through the whole chain (text, per-read results, counters) against the oracle."""
    rng = random.Random(4000 + 2 * paired + (flags != 0))
    p7, p5, mid = random_adapter(rng, MAX_M), random_adapter(rng, 65), random_adapter(rng, 97)

    def ops(p7, p5, mid):
        return [
            Op(A.OP_ALIGN, adapter_kind=A.AD_BACK, adapter=p7, min_overlap=3, max_error_rate=0.2),
            Op(A.OP_ALIGN, adapter_kind=A.AD_PREFIX, adapter=p5, min_overlap=3, max_error_rate=0.1),
            Op(A.OP_ALIGN, adapter_kind=A.AD_RIGHTMOST_FRONT, adapter=mid, min_overlap=5, max_error_rate=0.29),
            Op(A.OP_ALIGN, adapter_kind=A.AD_NI_BACK, adapter="G" * 100, min_overlap=3, max_error_rate=0.15),
        ]

    if paired:
        q7, q5, qmid = random_adapter(rng, MAX_M - 1), random_adapter(rng, 64), random_adapter(rng, 96)
        prog = Program(True, ops(p7, p5, mid), ops(q7, q5, qmid), Filters(0, False, 0, 0))
        r1 = chain_reads(rng, p5, mid, p7, 400)
        r2 = [(n, s, q) for (n, _, _), (_, s, q) in zip(r1, chain_reads(rng, q5, qmid, q7, 400))]
        compare_with_oracle(prog, [r1, r2], flags)
    else:
        prog = Program(False, ops(p7, p5, mid), [], Filters(0, False, 0, 0))
        compare_with_oracle(prog, [chain_reads(rng, p5, mid, p7, 600)], flags)
