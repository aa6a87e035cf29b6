"""Parity tests proper: the CUDA chain (through the C ABI, ctypes) against the CPU oracle and the
committed golden vectors. Bit-exact: every comparison is ==."""

import random

import numpy as np
import pytest

from cutseq_b200 import _abi as A
from cutseq_b200 import native
from cutseq_b200.program import Filters, Op, Program
from oracle import oracle
from tests import helpers

pytestmark = pytest.mark.gpu

KINDS = [A.AD_BACK, A.AD_BACK_ANYWHERE, A.AD_RIGHTMOST_FRONT, A.AD_PREFIX, A.AD_SUFFIX, A.AD_NI_FRONT, A.AD_NI_BACK, A.AD_FRONT]


def random_reads(rng, adapter, n_reads, max_len=160, alphabet="ACGT", lengths=None, back_to_back=0.0):
    """Reads with lengths drawn from `lengths` (default: a fixed list up to max_len) and, in 3 of 4, one or two
    partial, mutated adapter copies at the read start, at its end or anywhere; with probability back_to_back the
    second copy follows the first without a gap (adapter dimers)."""
    if lengths is None:
        lengths = [0, 1, 2, 3, 7, 20, 36, 50, 75, 100, 150, max_len]
    else:
        max_len = max(lengths)
    reads = []
    m = len(adapter)
    for i in range(n_reads):
        n = rng.choice(lengths)
        q = [rng.choice(alphabet + "N") if rng.random() < 0.02 else rng.choice(alphabet) for _ in range(n)]
        r = rng.random()
        if n and r < 0.75:  # plant a (partial, mutated) adapter copy, sometimes two
            end = None  # where the previous copy ends
            for _ in range(1 + (rng.random() < 0.15)):
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
                pos = 0 if where < 0.25 else (max(0, n - len(piece)) if where < 0.6 else rng.randint(0, max(0, n - 1)))
                if end is not None and back_to_back and rng.random() < back_to_back:
                    pos = min(end, n)
                q[pos : pos + len(piece)] = piece
                end = pos + len(piece)
            q = q[:max_len]
        s = "".join(q)
        if rng.random() < 0.05:
            s = s.lower()
        reads.append((f"r{i}", s, "I" * len(s)))
    return reads


def check_locate(op, reads):
    """Both execution modes: exact DP on every read, and bit-parallel prefilter + exact DP on the survivors."""
    batch, keep = oracle.make_batch(reads)
    wants = [oracle.adapter_match(op, s) for (_, s, _) in reads]
    for flags in (A.PLAN_NO_PREFILTER, 0, A.PLAN_NO_EXACT_STOP) + ((A.PLAN_NO_EXACT_STOP | A.PLAN_NO_PREFILTER,) if len(set(op.adapter)) == 1 else ()):
        got = native.locate_batch(op, batch.mate[0], len(reads), flags=flags)
        for i, (_, s, _) in enumerate(reads):
            g = got[i]
            have = None if not g["found"] else tuple(int(g[k]) for k in ("ref_start", "ref_stop", "query_start", "query_stop", "score", "errors"))
            assert have == wants[i], (flags, op.adapter, op.adapter_kind, op.max_error_rate, op.min_overlap, s, have, wants[i])


@pytest.mark.parametrize("kind", KINDS)
def test_locate_matches_oracle(kind):
    rng = random.Random(1000 + kind)
    for m, rate, mo in [(20, 0.2, 3), (20, 0.2, 10), (19, 0.2, 3), (6, 0.2, 3), (1, 0.2, 1), (3, 0.34, 1), (13, 0.1, 5),
                        (32, 0.2, 3), (33, 0.15, 3), (34, 0.3, 4), (40, 0.2, 3), (57, 0.12, 3), (20, 0.0, 3), (8, 0.5, 2)]:
        adapter = "".join(rng.choice("ACGT") for _ in range(m))
        op = Op(A.OP_ALIGN, adapter_kind=kind, adapter=adapter, min_overlap=mo, max_error_rate=rate)
        check_locate(op, random_reads(rng, adapter, 700))


@pytest.mark.parametrize("kind", [A.AD_NI_FRONT, A.AD_NI_BACK, A.AD_BACK, A.AD_RIGHTMOST_FRONT])
def test_locate_homopolymer_and_low_complexity(kind):
    rng = random.Random(77 + kind)
    for adapter, rate in [("A" * 100, 0.15), ("T" * 100, 0.15), ("AC" * 50, 0.15), ("A" * 30, 0.2), ("G" * 100, 0.1)]:
        op = Op(A.OP_ALIGN, adapter_kind=kind, adapter=adapter, min_overlap=3, max_error_rate=rate)
        reads = []
        for i in range(500):
            n = rng.randint(0, 150)
            body = "".join(rng.choice("ACGT") for _ in range(n))
            run = adapter[0] * rng.randint(0, 60)
            s = (body + run) if rng.random() < 0.5 else (run + body)
            s = "".join(c if rng.random() > 0.04 else rng.choice("ACGTN") for c in s)[:160]
            reads.append((f"h{i}", s, "I" * len(s)))
        check_locate(op, reads)


@pytest.mark.parametrize("kind", [A.AD_BACK, A.AD_RIGHTMOST_FRONT])
def test_locate_column_window_long_reads(kind):
    """The exact pass starts at a column chosen by the prefilter (BACK flags): long reads with several, partly
    damaged adapter copies far apart, near the ends and back to back (adapter dimers) must give cutadapt's match."""
    rng = random.Random(4242 + kind)
    for m, rate, mo in [(20, 0.2, 3), (20, 0.2, 10), (12, 0.25, 3), (31, 0.2, 5), (33, 0.2, 3), (57, 0.12, 3)]:
        adapter = "".join(rng.choice("ACGT") for _ in range(m))
        reads = []
        for i in range(500):
            n = rng.choice([120, 151, 250, 300, 450, 600, 800])
            q = [rng.choice("ACGT") for _ in range(n)]
            copies = rng.choice([0, 1, 1, 2, 2, 3])
            anchor = rng.randint(0, n - 1)
            for c in range(copies):
                piece = list(adapter)
                if rng.random() < 0.3:
                    cut = rng.randint(1, m)
                    piece = piece[:cut] if rng.random() < 0.5 else piece[m - cut:]
                for _ in range(rng.choice([0, 0, 1, 2, 3, 4, 6])):
                    if not piece:
                        break
                    pos = rng.randrange(len(piece))
                    t = rng.random()
                    if t < 0.5:
                        piece[pos] = rng.choice("ACGT")
                    elif t < 0.75:
                        del piece[pos]
                    else:
                        piece.insert(pos, rng.choice("ACGT"))
                where = rng.random()
                if where < 0.2:
                    pos = 0
                elif where < 0.45:
                    pos = max(0, n - len(piece) + rng.choice([0, 0, 1, 3]))
                elif where < 0.7:
                    pos = min(n - 1, anchor + c * (m + rng.choice([0, 0, 1, 2, 5])))  # dimers / near-by copies
                else:
                    pos = rng.randint(0, n - 1)
                q[pos : pos + len(piece)] = piece
            s = "".join(q)[:n]
            reads.append((f"w{i}", s, "I" * len(s)))
        op = Op(A.OP_ALIGN, adapter_kind=kind, adapter=adapter, min_overlap=mo, max_error_rate=rate)
        check_locate(op, reads)


def test_locate_two_letter_alphabet_ties():
    # low-complexity sequence space maximises cost ties, i.e. exercises the tie-breaking rules
    rng = random.Random(5)
    for kind in KINDS:
        for m in (5, 12, 20):
            adapter = "".join(rng.choice("AC") for _ in range(m))
            op = Op(A.OP_ALIGN, adapter_kind=kind, adapter=adapter, min_overlap=2, max_error_rate=0.25)
            check_locate(op, random_reads(rng, adapter, 400, max_len=60, alphabet="AC"))


def run_gpu(prog, mates, flags=0):
    batch, keep = oracle.make_batch(*mates)
    with native.Plan(prog, 0, A.PLAN_KEEP_MATCHES | flags) as plan:
        text, records = plan.run_batch(batch)
        n = batch.n_reads
        results = [plan.results(0, m, n) for m in range(batch.n_mates)]
        matches = []
        for m in range(batch.n_mates):
            ops = prog.ops_r1 if m == 0 else prog.ops_r2
            matches.append({t: plan.matches(0, m, t, n) for t, op in enumerate(ops) if op.kind == A.OP_ALIGN})
        stats = plan.stats()
    return text, records, results, matches, stats, batch, keep


COUNTER_FIELDS = ("n", "written", "too_short", "untrimmed")


def compare_with_oracle(prog, mates, flags=0):
    text, records, results, matches, stats, batch, keep = run_gpu(prog, mates, flags)
    want = oracle.run_batch(prog, batch, n_threads=4)
    n_mates = batch.n_mates
    for m in range(n_mates):
        for t, got in matches[m].items():
            w = want["matches"][m][t]
            for f in ("found", "ref_start", "ref_stop", "query_start", "query_stop", "score", "errors"):
                bad = np.nonzero(got[f] != w[f])[0]
                assert bad.size == 0, (m, t, f, int(bad[0]), got[bad[0]], w[bad[0]], mates[m][int(bad[0])])
        for f in ("start", "stop", "dest", "matched"):
            if prog.ops_r1[-1].kind == A.OP_REVCOMP and f in ("start", "stop"):
                continue
            bad = np.nonzero(results[m][f] != want["results"][m][f])[0]
            assert bad.size == 0, (m, f, int(bad[0]), results[m][bad[0]], want["results"][m][bad[0]])
    for d in range(A.CSQ_N_DEST):
        for m in range(n_mates):
            assert text[d][m] == want["text"][d][m], (d, m)
            assert records[d][m] == want["records"][d][m]
    for f in COUNTER_FIELDS:
        assert getattr(stats, f) == getattr(want["counters"], f), f
    for m in range(n_mates):
        assert stats.total_bp[m] == want["counters"].total_bp[m]
        assert stats.written_bp[m] == want["counters"].written_bp[m]
        assert stats.quality_trimmed_bp[m] == want["counters"].quality_trimmed_bp[m]
        assert list(stats.with_adapters[m]) == list(want["counters"].with_adapters[m])
        assert list(stats.dp_cells[m]) == list(want["counters"].dp_cells[m])
        assert list(stats.adjacent_bases[m]) == list(want["counters"].adjacent_bases[m])
    return text


@pytest.mark.parametrize("flags", [0, A.PLAN_NO_PREFILTER, A.PLAN_EMIT_G16, A.PLAN_NO_EXACT_STOP, A.PLAN_ONE_STREAM], ids=["prefilter", "exact_only", "emit_g16", "no_exact_stop", "one_stream"])
@pytest.mark.parametrize("case", helpers.golden_cases(), ids=lambda c: c["case"])
def test_golden_vectors(case, flags):
    prog = helpers.program_for(case["argv"], case["n_mates"])
    mates = helpers.golden_inputs(case)
    text = compare_with_oracle(prog, mates, flags)
    for (d, m), data in helpers.expected_by_dest(case, prog).items():
        assert text[d][m] == data, (case["case"], helpers.DEST_KEYS[d], m)


def test_empty_and_tiny_batches():
    prog = helpers.program_for(["-A", "TAKARAV3", "--trim-polyA"], 2)
    compare_with_oracle(prog, [[], []])
    compare_with_oracle(prog, [[("a 1", "", "")], [("a 2", "", "")]])
    compare_with_oracle(prog, [[("a", "ACGT", "IIII")], [("a", "TTTTTTTTTTTTTTTTTTTTTTTTTTTTT", "I" * 29)]])


def test_pairing_error_is_reported():
    prog = helpers.program_for(["-A", "TAKARAV3"], 2)
    batch, keep = oracle.make_batch([("x 1", "ACGT" * 10, "I" * 40)], [("y 2", "ACGT" * 10, "I" * 40)])
    with native.Plan(prog) as plan:
        with pytest.raises(native.NativeError) as e:
            plan.run_batch(batch)
        assert e.value.code == A.ERR_PAIRING
    assert oracle.run_batch(prog, batch)["status"] == A.ERR_PAIRING


# dnaio record_names_match / is_mate: header 2's id ends at its first space or tab, header 1 must end or hold a
# space / tab there, one trailing 1-3 on BOTH ids is ignored.  The reference applies it twice: dnaio's paired reader on
# the headers as they stand in the files, PairedEndRenamer (run.py:643-645) on what the SuffixRemovers left.
NAME_PAIRS = [
    ("r", "r"), ("r 1:N:0", "r 2:N:0"), ("r\t1", "r\t2"), ("r/1", "r/2"), ("r.1", "r.2"), ("r_1", "r_2"), ("r1", "r2"),
    ("r3", "r1"), ("SRR1.1.1 1 length=76", "SRR1.1.2 1 length=76"), ("r/1 comment", "r/2 comment"), ("r/1 c", "r/2"),
    ("ab1", "ab3 x"), ("a.1", "a.2"), ("q\x0bz 1", "q\x0bz 2"), ("x" * 70 + "1 c", "x" * 70 + "2 d"),
    ("x" * 15 + " c", "x" * 15 + " d"), ("x" * 16 + " c", "x" * 16 + " d"), ("x" * 17, "x" * 17), ("r/1", "r/2 c"),
    ("x 1", "y 2"), ("rA", "rB"), ("r1", "r4"), ("r", "r1"), ("r1", "r"), ("ab", "abc"), ("abc", "ab"), ("r/1", "r.2x"),
    ("r\x0b1", "r 2"), ("a.1", "a.3"), ("r1.1", "r2.2"), ("x" * 70 + "a", "x" * 70 + "b"), ("x" * 31 + "a c", "x" * 31 + "b c"),
    ("x" * 16 + "y" + "x" * 20, "x" * 37), ("", "r"), ("r", ""), (" r", "r"), ("a.1/1", "a.2/2"), ("a/1.1", "a/2.2"),
]


def reference_accepts(h1, h2):
    """What the reference does with a pair of headers under -A TAKARAV3 (SuffixRemover '.1' '/1' | '.2' '/2')."""
    from oracle import oracle as orc

    def strip(h, sufs):
        for x in sufs:
            if h.endswith(x):
                h = h[: len(h) - len(x)]
        return h

    return orc.names_match(h1, h2) and orc.names_match(strip(h1, (".1", "/1")), strip(h2, (".2", "/2")))


def test_record_names_match_rule():
    prog = helpers.program_for(["-A", "TAKARAV3"], 2)
    seq, q = "ACGTTGCA" * 10, "I" * 80
    good = [(a, b) for a, b in NAME_PAIRS if reference_accepts(a, b)]
    bad = [(a, b) for a, b in NAME_PAIRS if not reference_accepts(a, b)]
    assert ("r/1 comment", "r/2 comment") in good and ("SRR1.1.1 1 length=76", "SRR1.1.2 1 length=76") in good and ("r1", "r2") in good
    assert ("rA", "rB") in bad and ("a.1", "a.3") in bad and ("r1.1", "r2.2") in bad and ("r/1 c", "r/2") in bad and len(bad) >= 15
    r1 = [(a, seq, q) for a, _ in good]
    r2 = [(b, seq, q) for _, b in good]
    text = compare_with_oracle(prog, [r1, r2])
    assert text[0][0].count(b"\n") == 4 * len(good)  # every pair written, each mate under its own id
    for a, b in bad:
        m1, m2 = r1[:3] + [(a, seq, q)] + r1[3:5], r2[:3] + [(b, seq, q)] + r2[3:5]
        batch, keep = oracle.make_batch(m1, m2)
        assert oracle.run_batch(prog, batch)["status"] == A.ERR_PAIRING, (a, b)
        for flags in (0, A.PLAN_EMIT_G16):
            with native.Plan(prog, 0, flags) as plan:
                with pytest.raises(native.NativeError) as e:
                    plan.run_batch(batch)
                assert e.value.code == A.ERR_PAIRING, (a, b)
                texts = [("".join(f"@{n}\n{s}\n+\n{qq}\n" for n, s, qq in m)).encode("latin-1") for m in (m1, m2)]
                with pytest.raises(native.NativeError) as e:
                    plan.run_text(texts, 6)
                assert e.value.code == A.ERR_PAIRING, (a, b)


def test_pairing_error_in_a_pair_that_bypasses_the_staging_buffers():
    """Headers of 30 KB: the pair does not fit the emitter's shared-memory buffers and is written bytewise; the name
    check has to work there too (ids differ in their last character only)."""
    prog = helpers.program_for(["-A", "TAKARAV3"], 2)
    seq, q = "ACGTTGCA" * 10, "I" * 80
    long_id = "x" * 300
    good = [(f"{long_id}a " + "c" * 30000, seq, q), ("r2 1", seq, q)]
    mate = [(f"{long_id}a " + "d" * 30000, seq, q), ("r2 2", seq, q)]
    compare_with_oracle(prog, [good, mate])
    bad = [(f"{long_id}b " + "d" * 30000, seq, q), ("r2 2", seq, q)]
    batch, keep = oracle.make_batch(good, bad)
    with native.Plan(prog) as plan:
        with pytest.raises(native.NativeError) as e:
            plan.run_batch(batch)
        assert e.value.code == A.ERR_PAIRING


def test_read_length_limit_is_an_error():
    prog = helpers.program_for(["-A", "TAKARAV3"], 1)
    batch, keep = oracle.make_batch([("x", "A" * 1000, "I" * 1000)])
    with native.Plan(prog) as plan:
        with pytest.raises(native.NativeError) as e:
            plan.run_batch(batch)
        assert e.value.code == A.ERR_LIMIT


def test_odd_headers_and_names():
    prog = helpers.program_for(["-A", "TAKARAV3"], 1)
    seq, q = "ACGTTGCA" * 10, "I" * 80
    names = ["plain", "with comment here", " leading space", "trailing ", "tab\tsep", "x/1", "x.1", "x/1.1", "x.1/1", "a  b  c", "", " ", "id /1"]
    compare_with_oracle(prog, [[(nm, seq, q) for nm in names]])


@pytest.mark.parametrize("flags", [0, A.PLAN_EMIT_G16], ids=["emit_stage", "emit_g16"])
def test_long_and_mixed_length_pairs(flags):
    """Reads of 250-850 bases beside short ones: the staged emitter has to halve its passes (8 pairs no longer fit its
    shared-memory buffers), down to single pairs, and the DP walks windows far into long reads."""
    prog = helpers.program_for(["-A", "TAKARAV3", "--trim-polyA"], 2)
    rng = random.Random(99)
    comp = {"A": "T", "C": "G", "G": "C", "T": "A", "N": "N"}
    p7, p5rc = "AGATCGGAAGAGCACACGTC", "AGATCGGAAGAGCGTCGTGT"

    def noisy(seq):
        out = []
        for c in seq:
            t = rng.random()
            if t < 0.01:
                out.append(rng.choice("ACGTN"))
            elif t < 0.012:
                continue
            else:
                out.append(c)
        return "".join(out)

    r1, r2 = [], []
    for k in range(360):
        read_len = rng.choice([250, 40, 600, 150, 850, 300])
        insert = rng.randint(10, read_len + 200)
        frag = "".join(rng.choice("ACGT") for _ in range(insert))
        if rng.random() < 0.2:
            frag = "T" * rng.randint(10, 40) + frag  # poly-T at the start of R1 (strand '-')
        rc = "".join(comp[c] for c in reversed(frag))
        s1 = noisy(frag + p7 + "TGAACTCCAGTCAC" + "G" * read_len)[:read_len]
        s2 = noisy(rc + p5rc + "AGATCTCGGTGGTCGCCGTATCATT" + "G" * read_len)[:read_len]
        q1 = "".join(rng.choice("II9-#") for _ in s1)
        q2 = "".join(rng.choice("II9-#") for _ in s2)
        r1.append((f"P{k}:{read_len} 1:N:0:ACGT", s1, q1))
        r2.append((f"P{k}:{read_len} 2:N:0:ACGT", s2, q2))
    want = compare_with_oracle(prog, [r1, r2], flags)
    # the same records as a text batch (one source span per mate and pass in the staged emitter)
    texts = ["".join(f"@{n}\n{s_}\n+\n{q}\n" for (n, s_, q) in recs).encode() for recs in (r1, r2)]
    with native.Plan(prog, 0, flags) as plan:
        got, _ = plan.run_text(texts, len(r1))
    assert got == want


def test_random_programs_against_oracle():
    rng = random.Random(2024)
    for it in range(12):
        def part(n):
            return "".join(rng.choice("ACGT") for _ in range(n))

        scheme = part(rng.choice([12, 19, 20, 25]))
        if rng.random() < 0.5:
            scheme += "(" + part(rng.choice([4, 6, 8])) + ")"
        scheme += "N" * rng.choice([0, 0, 5, 8]) + "X" * rng.choice([0, 1, 3])
        scheme += rng.choice("<>-")
        scheme += "X" * rng.choice([0, 2, 6]) + "N" * rng.choice([0, 0, 6, 10])
        if rng.random() < 0.5:
            scheme += "(" + part(rng.choice([4, 6, 8])) + ")"
        scheme += part(rng.choice([12, 19, 20, 25]))
        argv = ["-a", scheme]
        for flag, p in (("--trim-polyA", 0.5), ("--trim-polyA-wo-direction", 0.3), ("--no-conditional-cutter", 0.3),
                        ("--force-anywhere", 0.3), ("--ensure-inline-barcode", 0.5), ("--auto-rc", 0.3)):
            if rng.random() < p:
                argv.append(flag)
        argv += ["-q", str(rng.choice([0, 10, 20, 30])), "-m", str(rng.choice([0, 15, 20, 40]))]
        n_mates = rng.choice([1, 2])
        prog = helpers.program_for(argv, n_mates)
        from cutseq_b200.common import BarcodeConfig

        bc = BarcodeConfig(scheme.upper())
        import scripts.make_golden as mg

        r1, r2 = mg.synth_pairs(rng.randint(0, 1 << 30), 300, read_len=rng.choice([50, 100, 150]), p5=bc.p5.fw, p7=bc.p7.fw,
                                inline5=bc.inline5.fw, inline3=bc.inline3.fw, umi5=bc.umi5.len, umi3=bc.umi3.len,
                                mask5=bc.mask5.len, mask3=bc.mask3.len, strand=bc.strand or "+", readthrough=0.5,
                                polya=0.2, bc_error=0.03, wrong_bc=0.1, suffix_style=rng.choice([None, "slash", "dot", "bare"]))
        compare_with_oracle(prog, [r1, r2] if n_mates == 2 else [r1])


def test_synthetic_configs_against_oracle():
    """BASELINE.json configs 2-4 (synthetic generator), 30 000 units each, whole chain vs the oracle."""
    cases = [
        (2, ["-A", "TAKARAV3", "--trim-polyA"], 2),
        (3, ["-a", "ACACGACGCTCTTCCGATCT(ATCACG)NNNNNNNNXXX<XXX(CGTGAT)AGATCGGAAGAGCACACGTC", "--ensure-inline-barcode"], 2),
        (3, ["-a", "ACACGACGCTCTTCCGATCT(ATCACG)NNNNNNNNXXX<XXX(CGTGAT)AGATCGGAAGAGCACACGTC"], 2),
        (4, ["-A", "SMALLRNA"], 1),
    ]
    for config, argv, n_mates in cases:
        prog = helpers.program_for(argv, n_mates)
        batch = native.synth_batch(config, 30000, first_index=12345, buffer=3)
        want = oracle.run_batch(prog, batch, n_threads=8)
        for flags in (0, A.PLAN_NO_PREFILTER, A.PLAN_EMIT_G16, A.PLAN_NO_EXACT_STOP, A.PLAN_NO_EXACT_STOP | A.PLAN_NO_PREFILTER):
            with native.Plan(prog, 0, A.PLAN_KEEP_MATCHES | flags) as plan:
                text, records = plan.run_batch(batch)
                stats = plan.stats()
                for m in range(n_mates):
                    ops = prog.ops_r1 if m == 0 else prog.ops_r2
                    for t, op in enumerate(ops):
                        if op.kind == A.OP_ALIGN:
                            got = plan.matches(0, m, t, batch.n_reads)
                            w = want["matches"][m][t]
                            for f in ("found", "ref_start", "ref_stop", "query_start", "query_stop", "score", "errors"):
                                assert (got[f] == w[f]).all(), (config, argv, flags, m, t, f)
            for d in range(A.CSQ_N_DEST):
                for m in range(n_mates):
                    assert text[d][m] == want["text"][d][m], (config, argv, flags, d, m)
            assert list(stats.dp_cells[0]) == list(want["counters"].dp_cells[0])
            assert stats.written == want["counters"].written and stats.untrimmed == want["counters"].untrimmed


# ---- text batches: raw FASTQ bytes in, the device builds the record index (parse.cu) ----
PARSE_FLAGS = [0]
PARSE_IDS = ["parse"]


@pytest.mark.parametrize("pflags", PARSE_FLAGS, ids=PARSE_IDS)
def test_text_batches_equal_soa_batches(pflags):
    cases = [
        (2, ["-A", "TAKARAV3", "--trim-polyA"], 2),
        (3, ["-a", "ACACGACGCTCTTCCGATCT(ATCACG)NNNNNNNNXXX<XXX(CGTGAT)AGATCGGAAGAGCACACGTC", "--ensure-inline-barcode"], 2),
        (4, ["-A", "SMALLRNA"], 1),
    ]
    for config, argv, n_mates in cases:
        prog = helpers.program_for(argv, n_mates)
        for n in (1, 255, 20011):
            batch = native.synth_batch(config, n, first_index=99, buffer=5)
            texts = [native.format_fastq(batch, m).tobytes() for m in range(n_mates)]
            with native.Plan(prog, 0, pflags) as plan:
                want, want_records = plan.run_batch(batch)
                got, got_records = plan.run_text(texts, n, slot=1)
                assert got == want and got_records == want_records, (config, n)
                crlf = [t.replace(b"\n", b"\r\n") for t in texts]
                got, got_records = plan.run_text(crlf, n, slot=2)
                assert got == want and got_records == want_records, (config, n, "crlf")


@pytest.mark.parametrize("pflags", PARSE_FLAGS, ids=PARSE_IDS)
def test_text_batch_odd_records(pflags):
    """'+' line repeating the name, empty reads, a read at the length limit, lower-case bases, header with tabs."""
    prog = helpers.program_for(["-A", "SMALLRNA"], 1)
    recs = [
        ("r1 x", "ACGTACGTACGTACGTACGTACGTAGATCGGAAGAGCACACGTC", True),
        ("r2\ty", "", False),
        ("r3", "A" * A.CSQ_MAX_READ_LEN, False),
        ("r4/1", "acgtacgtnnacgtacgtacgtacgtagatcggaagagcacacgtc", True),
        ("r5.1 z", "ACGTTTGACCATGACCATGACGATTTACGACGATATTACGAGT", False),
    ]
    text = b""
    for name, seq, plus_name in recs:
        text += f"@{name}\n{seq}\n+{name if plus_name else ''}\n{'I' * len(seq)}\n".encode()
    want = oracle_text(prog, [text])
    with native.Plan(prog, 0, pflags) as plan:
        got, _ = plan.run_text([text], len(recs))
    assert got[0][0] == want[0][0] and got[1][0] == want[1][0]


@pytest.mark.parametrize("pflags", PARSE_FLAGS, ids=PARSE_IDS)
def test_text_batch_mixed_line_endings(pflags):
    """CRLF and LF records in one batch, a '\\r' in the middle of a header, a '+' line that repeats the name with
    CRLF: only the '\\r' in front of a line end is dropped (dnaio), wherever the batch-wide CR flag is set."""
    prog = helpers.program_for(["-A", "SMALLRNA"], 1)
    rng = random.Random(21)
    text, clean = b"", b""
    for i in range(3000):
        seq = "".join(rng.choice("ACGT") for _ in range(rng.randint(0, 60))) + "AGATCGGAAGAGCACACGTC"[: rng.randint(0, 20)]
        name = f"r{i} co\rmment" if i % 17 == 3 else f"r{i} comment"
        plus = name if i % 5 == 0 else ""
        eol = "\r\n" if i % 3 else "\n"
        text += f"@{name}{eol}{seq}{eol}+{plus}{eol}{'I' * len(seq)}{eol}".encode()
        clean += f"@{name}\n{seq}\n+{plus}\n{'I' * len(seq)}\n".encode()
    want = oracle_text(prog, [clean])
    with native.Plan(prog, 0, pflags) as plan:
        got, _ = plan.run_text([text], 3000)
    assert got[0][0] == want[0][0] and got[1][0] == want[1][0]


@pytest.mark.parametrize("pflags", PARSE_FLAGS, ids=PARSE_IDS)
def test_text_batch_lines_longer_than_a_parse_tile(pflags):
    """Header comments / '+' lines of 20-50 KB: whole 16 KiB parse tiles without a line end, so the start of the
    open line has to be carried across several tiles by the look-back."""
    prog = helpers.program_for(["-A", "SMALLRNA"], 1)
    rng = random.Random(7)
    text = b""
    n = 0
    for i in range(400):
        seq = "".join(rng.choice("ACGT") for _ in range(rng.randint(0, 120))) + "AGATCGGAAGAGCACACGTC"[: rng.randint(0, 20)]
        comment = "c" * (rng.choice([20000, 33000, 50000]) if i % 57 == 5 else rng.randint(0, 30))
        plus = f"r{i} {comment}" if i % 3 == 0 else ""  # the '+' line may repeat the header
        text += f"@r{i} {comment}\n{seq}\n+{plus}\n{'I' * len(seq)}\n".encode()
        n += 1
    want = oracle_text(prog, [text])
    with native.Plan(prog, 0, pflags) as plan:
        got, _ = plan.run_text([text], n)
    assert got[0][0] == want[0][0] and got[1][0] == want[1][0]


@pytest.mark.parametrize("pflags", PARSE_FLAGS, ids=PARSE_IDS)
def test_text_batch_many_tiny_records(pflags):
    """Empty reads: 6-byte lines, ~2 700 line ends per parse tile; plus a wrong record count in both directions."""
    prog = helpers.program_for(["-A", "SMALLRNA"], 1)
    n = 50000
    text = b"".join(b"@%d\n\n+\n\n" % i for i in range(n))
    with native.Plan(prog, 0, pflags) as plan:
        got, records = plan.run_text([text], n)
        assert records[1][0] == n and got[1][0] == text  # all too short, unchanged
        for wrong in (n - 1, n + 1):
            with pytest.raises(native.NativeError) as e:
                plan.run_text([text], wrong)
            assert e.value.code == A.ERR_FORMAT and "whole FASTQ records" in str(e.value)


def oracle_text(prog, texts):
    """Oracle over FASTQ text: host parser (csq_parse_fastq_mem semantics, Python) -> SoA -> oracle.run_batch."""
    mates = []
    for t in texts:
        lines = t.split(b"\n")
        mates.append([(lines[i][1:].rstrip(b"\r").decode(), lines[i + 1].rstrip(b"\r").decode(), lines[i + 3].rstrip(b"\r").decode())
                      for i in range(0, len(lines) - 1, 4)])
    batch, keep = oracle.make_batch(*mates)
    return oracle.run_batch(prog, batch, n_threads=2)["text"]


@pytest.mark.parametrize("bad,code,needle", [
    (b"@r1\nACGT\n+\nIIII\nr2\nACGT\n+\nIIII\n", A.ERR_FORMAT, "line 5 is expected to start with '@'"),
    (b"@r1\nACGT\n+\nIIII\n@r2\nACGT\n-\nIIII\n", A.ERR_FORMAT, "line 7 is expected to start with '+'"),
    (b"@r1\nACGT\n+\nIII\n@r2\nACGT\n+\nIIII\n", A.ERR_FORMAT, "length of sequence and qualities differ (record at line 1)"),
    (b"@r1\nACGT\n+\nIIII\n@r2\n" + b"A" * 900 + b"\n+\n" + b"I" * 900 + b"\n", A.ERR_LIMIT, "line 5"),
    (b"@r1\nACGT\n+\nIIII\n@r2\nACGT\n+\n", A.ERR_FORMAT, "whole FASTQ records"),
    # dnaio: a description repeated behind the '+' must equal the header
    (b"@r1 x\nACGT\n+r1 x\nIIII\n@r2\nACGT\n+r3\nIIII\n", A.ERR_FORMAT, "descriptions don't match at line 7"),
    (b"@r1 x\nACGT\n+r1\nIIII\n@r2\nACGT\n+\nIIII\n", A.ERR_FORMAT, "descriptions don't match at line 3"),
    (b"@r1\nACGT\n+\nIIII\n@" + b"h" * 70000 + b"\nACGT\n+\nIIII\n", A.ERR_LIMIT, "header at line 5"),
])
@pytest.mark.parametrize("pflags", PARSE_FLAGS, ids=PARSE_IDS)
def test_text_batch_format_errors(bad, code, needle, pflags):
    prog = helpers.program_for(["-A", "SMALLRNA"], 1)
    with native.Plan(prog, 0, pflags) as plan:
        with pytest.raises(native.NativeError) as e:
            plan.run_text([bad], 2, capacity=8192 + len(bad))
        assert e.value.code == code and needle in str(e.value), str(e.value)
        # the plan stays usable
        good = b"@r1\nACGTACGTACGTACGTACGTACGTACGT\n+\nIIIIIIIIIIIIIIIIIIIIIIIIIIII\n"
        got, records = plan.run_text([good], 1, capacity=8192)
        assert got[0][0] == good and records[0][0] == 1
        # a repeated description that matches is fine (and is not written again, like dnaio's fastq_bytes)
        twice = b"@r1 c\r\nACGTACGTACGTACGTACGTACGTACGT\r\n+r1 c\r\nIIIIIIIIIIIIIIIIIIIIIIIIIIII\r\n"
        got, records = plan.run_text([twice], 1, capacity=8192)
        assert got[0][0] == good and records[0][0] == 1  # (the Renamer of this scheme keeps the id only)
