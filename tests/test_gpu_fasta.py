"""FASTA on the device (CSQ_PLAN_FASTA): FASTA text batches parsed, trimmed and written as FASTA by the library, against
the route the command line took before - FASTA -> transcode.fasta_to_fastq -> the chain (here the CPU oracle) ->
transcode.fastq_to_fasta.  Every comparison is ==."""

import bz2
import gzip
import io
import json
import lzma
import random
from types import SimpleNamespace

import pytest

from cutseq_b200 import _abi as A
from cutseq_b200 import native, run, transcode
from cutseq_b200.transcode import Transcoders
from tests import helpers
from tests import program_gen as G
from tests.test_gpu_gz import gunzip_members
from tests.test_gpu_parity import assert_equals_oracle
from tests.test_gpu_programs import COUNTERS, FLAGS, N_SEEDS, N_THREADS, SIZES, counters, program_case
from oracle import oracle

pytestmark = pytest.mark.gpu


def fasta_text(records, width=None, eol="\n", rng=None):
    """FASTA records (header, sequence); width: wrap the sequence (None: one line; "mixed": a random width per record)."""
    out = []
    for h, s, *_ in records:
        w = width if width != "mixed" else rng.choice([None, 1, 7, 60, 80])
        lines = [s] if not w or not s else [s[o:o + w] for o in range(0, len(s), w)]
        out.append(">" + h + eol + "".join(x + eol for x in lines))
    return "".join(out).encode("latin-1")


def pump(text: bytes):
    """The converting pump: FASTA -> FASTQ records (header, sequence, 'I' qualities)."""
    fq = io.BytesIO()
    transcode.fasta_to_fastq(io.BytesIO(text), fq)
    lines = fq.getvalue().split(b"\n")
    return [tuple(x.decode("latin-1") for x in (lines[i][1:], lines[i + 1], lines[i + 3])) for i in range(0, len(lines) - 1, 4)]


def to_fasta(fastq: bytes) -> bytes:
    out = io.BytesIO()
    transcode.fastq_to_fasta(io.BytesIO(fastq), out)
    return out.getvalue()


def expected(prog, texts):
    mates = [pump(t) for t in texts]
    batch, keep = oracle.make_batch(*mates)
    want = oracle.run_batch(prog, batch, n_threads=N_THREADS)
    want["text"] = [[to_fasta(t) for t in row] for row in want["text"]]
    return mates, want


class FastaPlan(native.Plan):
    def __init__(self, prog, flags):
        super().__init__(prog, 0, A.PLAN_KEEP_MATCHES | A.PLAN_FASTA | flags)
        self.flags = flags


def run_fasta(plan, prog, texts, n, capacity, slot=0):
    before = counters(plan.stats())
    text, records = plan.run_text(texts, n, capacity, slot)
    if plan.flags & A.PLAN_GZIP_OUT:
        text = [[gunzip_members(t) if t else b"" for t in row] for row in text]
    results = [plan.results(slot, m, n) for m in range(len(texts))]
    matches = [{t: plan.matches(slot, m, t, n) for t, op in enumerate(prog.ops_r1 if m == 0 else prog.ops_r2)
                if op.kind == A.OP_ALIGN} for m in range(len(texts))]
    after = counters(plan.stats())
    stats = SimpleNamespace(**{f: (after[f] - before[f]).tolist() for f in COUNTERS})
    return text, records, results, matches, stats


def check(plan, prog, texts, slot=0):
    mates, want = expected(prog, texts)
    cap = 2 * max(len(t) for t in texts) + 64 * len(mates[0]) + 4096
    got = run_fasta(plan, prog, texts, len(mates[0]), cap, slot)
    assert_equals_oracle(prog, mates, want, *got)


SHAPES = [None, 60, 1, 80, "mixed"]


@pytest.mark.parametrize("seed", range(N_SEEDS))
def test_random_program_fasta(seed):
    """The generated programs of test_gpu_programs as FASTA (wrapped in a shape that rotates with the seed) under every
    plan flag: a 2000-record batch, then a smaller one on the same slot."""
    prog, mates = program_case(seed)
    rng = random.Random(seed)
    shape = SHAPES[seed % len(SHAPES)]
    big = [fasta_text(m[:SIZES[0]], shape, rng=random.Random(seed)) for m in mates]
    for j, flags in enumerate(FLAGS):
        small_n = SIZES[1 + (j + seed) % (len(SIZES) - 1)]
        small = [fasta_text(m[SIZES[0]:SIZES[0] + small_n], shape, rng=random.Random(seed + 1)) for m in mates]
        with FastaPlan(prog, flags) as plan:
            check(plan, prog, big)
            check(plan, prog, small)
            if flags == 0:
                check(plan, prog, [fasta_text(m[:500], rng.choice(SHAPES), "\r\n", rng=rng) for m in mates], slot=1)


def odd_shapes(rng, n):
    """Blank lines (also in front of the first header), blanks around sequence lines, CRLF, empty sequences, '>' inside
    sequence lines and 895-base reads wrapped."""
    parts = ["\n \n"]
    for i in range(n):
        eol = "\r\n" if i % 5 == 0 else "\n"
        parts.append(f">r{i} x{i % 7}{' ' if i % 3 == 0 else ''}{eol}")
        length = rng.choice([0, 0, 1, 15, 16, 17, 150, 894, 895])
        seq = "".join(rng.choice("ACGTN") for _ in range(length))
        w = rng.choice([1, 3, 60, 80, 1000])
        for o in range(0, len(seq), w):
            piece = seq[o:o + w]
            lead = rng.choice(["", "", " ", "\t"])
            trail = rng.choice(["", "", " ", "\t\x0b\x0c", "\r"])
            if rng.random() < 0.1 and len(piece) >= 2:
                piece = piece[0] + ">" + piece[2:]  # '>' inside a line
            parts.append(lead + piece + trail + eol)
            if rng.random() < 0.1:
                parts.append(eol)
    return "".join(parts).encode("latin-1")


@pytest.mark.parametrize("flags", [0, A.PLAN_EMIT_G16, A.PLAN_GZIP_OUT])
@pytest.mark.parametrize("paired", [False, True])
def test_text_shapes(flags, paired):
    prog, _ = program_case(1 if paired else 0)
    rng = random.Random(11)
    n = 700
    texts = [odd_shapes(rng, n) for _ in range(2 if paired else 1)]
    if paired:  # same headers in both mates
        texts[1] = texts[0]
    with FastaPlan(prog, flags) as plan:
        check(plan, prog, texts)
        check(plan, prog, [t[: t.index(b">r5 ")] for t in texts], slot=0)  # a small batch after a large one


def simple_plan(paired=False, flags=0):
    prog, _ = program_case(1 if paired else 0)
    return prog, FastaPlan(prog, flags)


def run_error(texts, n, paired=False):
    prog, plan = simple_plan(paired)
    with plan:
        with pytest.raises(native.NativeError) as e:
            plan.run_text(texts, n, 1 << 20)
    return e.value


def test_text_before_the_first_header_is_an_error():
    e = run_error([b"\n\nACGT\n>r1\nAC\n"], 1)
    assert e.code == A.ERR_FORMAT and "line 3" in str(e)


def test_read_length_limit():
    seq = "A" * 896
    text = (">ok\n" + "C" * 895 + "\n>long\n" + "\n".join(seq[o:o + 60] for o in range(0, 896, 60)) + "\n").encode()
    e = run_error([text], 2)
    assert e.code == A.ERR_LIMIT and "line 3" in str(e)
    prog, plan = simple_plan()
    with plan:
        check(plan, prog, [text[: text.index(b">long")]])


def test_header_limit():
    prog, plan = simple_plan()
    ok = (">" + "h" * 65535 + "\nACGT\n").encode()
    with plan:
        check(plan, prog, [ok])
    e = run_error([(">" + "h" * 65536 + "\nACGT\n").encode()], 1)
    assert e.code == A.ERR_LIMIT


def test_mismatched_mate_names():
    e = run_error([b">a/1\nAC\n>b/1\nAC\n", b">a/2\nAC\n>c/2\nAC\n"], 2, paired=True)
    assert e.code == A.ERR_PAIRING


def test_fastq_text_and_wrong_counts_are_format_errors():
    assert run_error([b"@r1\nACGT\n+\nIIII\n"], 1).code == A.ERR_FORMAT
    assert run_error([b">r1\nACGT\n>r2\nA\n"], 1).code == A.ERR_FORMAT
    assert run_error([b">r1\nACGT\n"], 2).code == A.ERR_FORMAT


def test_soa_and_bgzf_entry_points_refuse_the_flag():
    prog, plan = simple_plan()
    recs = [("r1", "ACGT", "IIII")]
    with plan:
        batch, keep = oracle.make_batch(recs)
        with pytest.raises(native.NativeError) as e:
            plan.run_batch(batch, 4096, 0)
        assert e.value.code == A.ERR_INVALID
        with pytest.raises(native.NativeError) as e:
            plan.upload(0, batch)
        assert e.value.code == A.ERR_INVALID
    lib = native.lib()
    # csq_submit_bgzf / csq_bgzf_count_lines check the flag before they look at the batch
    with FastaPlan(prog, 0) as plan:
        out = A.csq_batch_out()
        bg = A.csq_batch_bgzf()
        bg.n_mates = 1
        assert lib.csq_submit_bgzf(plan._h, 0, native.C.byref(bg), native.C.byref(out)) == A.ERR_INVALID
        bi = A.csq_bgzf_in()
        assert lib.csq_bgzf_count_lines(plan._h, 0, native.C.byref(bi), None) == A.ERR_INVALID


# ---- the command line: native route against the pump route ----

def cli_inputs(tmp_path, kind, width, name="takarav3_synth_polya"):
    case = [c for c in helpers.golden_cases() if c["case"] == name][0]
    paths = []
    for m, p in enumerate(helpers.golden_input_paths(case)):
        lines = gzip.open(p).read().split(b"\n")
        recs = [(lines[i][1:].decode(), lines[i + 1].decode()) for i in range(0, len(lines) - 1, 4)]
        text = fasta_text(recs, width)
        path = str(tmp_path / (f"in_R{m + 1}.fa" + {"plain": "", "gz": ".gz", "bgzf": ".gz", "bz2": ".bz2"}[kind]))
        if kind == "plain":
            open(path, "wb").write(text)
        elif kind == "gz":
            open(path, "wb").write(gzip.compress(text))
        elif kind == "bgzf":
            from tests.test_fasta_host import bgzf
            open(path, "wb").write(bgzf(text, 0xFF00))
        else:
            open(path, "wb").write(bz2.compress(text))
        paths.append(path)
    return case, paths


def read_any(path):
    for ext, op in ((".gz", gzip.open), (".bz2", bz2.open), (".xz", lzma.open)):
        if path.endswith(ext):
            return op(path, "rb").read()
    return open(path, "rb").read()


def both_routes(tmp_path, monkeypatch, capsys, argv, inputs, outs):
    """argv with -o/-s outputs named `outs` through the native route and through the pump route; -> [(native, pump)]."""
    got = {}
    for route in ("native", "pump"):
        names = [str(tmp_path / f"{route}_{o}") for o in outs]
        extra = []
        if len(names) >= 1:
            extra += ["-o"] + names[: len(inputs)]
        if len(names) > len(inputs):
            extra += ["-s"] + names[len(inputs):]
        js = str(tmp_path / f"{route}.json")
        with monkeypatch.context() as mp:
            if route == "pump":
                orig = Transcoders.__init__
                mp.setattr(Transcoders, "__init__", lambda self, i, o, fasta_native=False: orig(self, i, o))
            capsys.readouterr()
            run.main(argv + extra + ["--json-file", js] + inputs)
            report = capsys.readouterr().out
        got[route] = ([read_any(n) for n in names], report, json.load(open(js)))
    return got


@pytest.mark.parametrize("kind,outs,br", [
    ("plain", ("o1.fa", "o2.fa", "s1.fa", "s2.fa"), "100000"),
    ("gz", ("o1.fa.gz", "o2.fa.gz", "s1.fa.gz", "s2.fa.gz"), "64"),
    ("bgzf", ("o1.fa.bz2", "o2.fa.xz", "s1.fa", "s2.fa.gz"), "1"),
    ("bz2", ("o1.fa", "o2.fa.gz", "s1.fa.xz", "s2.fa"), "64"),
])
def test_cli_native_route_equals_pump_route(tmp_path, monkeypatch, capsys, kind, outs, br):
    case, inputs = cli_inputs(tmp_path, kind, 60 if kind != "plain" else None)
    got = both_routes(tmp_path, monkeypatch, capsys, case["argv"] + ["--batch-reads", br], inputs, outs)
    n_files, n_report, n_json = got["native"]
    p_files, p_report, p_json = got["pump"]
    assert n_files == p_files
    assert n_report == p_report
    for j in (n_json, p_json):
        j.pop("input", None), j.pop("output", None)
    assert n_json["read_counts"] == p_json["read_counts"] and n_json["basepair_counts"] == p_json["basepair_counts"]
    assert n_json["adapters_read1"] == p_json["adapters_read1"] and n_json["adapters_read2"] == p_json["adapters_read2"]
    assert n_files[0].count(b"\n") > 1000


@pytest.mark.parametrize("name", ["se_takarav3_autorc", "se_inline_ensure", "takarav3_autorc"])
def test_cli_auto_rc_and_polya(tmp_path, monkeypatch, capsys, name):
    """Single-end --auto-rc (REVCOMP on the device) and --trim-polyA; paired --auto-rc (swapped sink)."""
    case, inputs = cli_inputs(tmp_path, "plain", 60, name)
    outs = ("o1.fa", "s1.fa") if len(inputs) == 1 else ("o1.fa", "o2.fa", "s1.fa", "s2.fa")
    got = both_routes(tmp_path, monkeypatch, capsys, case["argv"] + ["--batch-reads", "100"], inputs, outs)
    assert got["native"][0] == got["pump"][0] and got["native"][1] == got["pump"][1]
    assert got["native"][0][0].count(b">") > 100


def test_cli_multi_gpu_order(tmp_path, monkeypatch, capsys):
    if native.device_count() < 2:
        pytest.skip("needs two GPUs")
    case, inputs = cli_inputs(tmp_path, "plain", 60)
    got = both_routes(tmp_path, monkeypatch, capsys, case["argv"] + ["--batch-reads", "64", "--gpus", "2"], inputs,
                      ("o1.fa", "o2.fa"))
    assert got["native"][0] == got["pump"][0]
