"""FASTA on the host side of the library (CSQ_PLAN_FASTA): the record-start helper csq_after_kth_fasta_record, the
text reader that cuts FASTA files into batches of whole records, and the pumps Transcoders starts for FASTA files when
the library reads them itself.  No GPU."""
import gzip
import os
import random
import struct
import threading
import zlib

import numpy as np
import pytest

from cutseq_b200 import _abi as A
from cutseq_b200 import native
from cutseq_b200.transcode import Transcoders


def record_starts(text: bytes):
    """Python reference: offsets of the bytes '>' that start a line."""
    return [i for i in range(len(text)) if text[i:i + 1] == b">" and (i == 0 or text[i - 1:i] == b"\n")]


def after_kth(text: bytes, k: int):
    buf = np.frombuffer(text + b"\0" * 64, dtype=np.uint8)
    return native.lib().csq_after_kth_fasta_record(buf.ctypes.data, len(text), k)


def random_fasta(rng, n_records, crlf=False, junk=True):
    eol = b"\r\n" if crlf else b"\n"
    out = []
    for i in range(n_records):
        out.append(b">r%d %s" % (i, bytes(rng.choice(b"ab >") for _ in range(rng.randrange(0, 9)))) + eol)
        for _ in range(rng.randrange(0, 5)):
            line = bytes(rng.choice(b"ACGTN") for _ in range(rng.randrange(0, 90)))
            if junk and rng.random() < 0.3:
                line = rng.choice([b" ", b"\t", b"  >", b"x>"]) + line + rng.choice([b"", b" ", b">"])
            out.append(line + eol)
        if junk and rng.random() < 0.2:
            out.append(eol)
    return b"".join(out)


@pytest.mark.parametrize("seed", range(12))
def test_after_kth_fasta_record_matches_python(seed):
    rng = random.Random(seed)
    text = random_fasta(rng, rng.randrange(0, 200), crlf=seed % 3 == 0)
    if seed % 4 == 1:
        text = b"\n\n  \n" + text  # blank lines in front of the first header
    starts = record_starts(text)
    for k in list(range(min(len(starts) + 3, 40))) + [len(starts) - 1, len(starts), len(starts) + 1, 10 ** 9]:
        if k < 0:
            continue
        want = starts[k] if k < len(starts) else 2 ** 64 - 1
        assert after_kth(text, k) == want, (seed, k)


@pytest.mark.parametrize("at", [0, 1, 15, 16, 63, 64, 65, 127, 128, 4095, 4096, 4097, 8191, 8192])
def test_after_kth_fasta_record_at_chunk_edges(at):
    """Record starts and the line ends in front of them on every side of the 64-byte SIMD steps and 4 KiB blocks."""
    for before in (b"\n", b"\r\n", b" ", b"x"):
        text = b">a\n" + b"C" * max(0, at - 3 - len(before)) + before
        text = text[:at] + b">b\nAC\n>c\n" if len(text) >= at else text + b">b\nAC\n>c\n"
        starts = record_starts(text)
        for k in range(len(starts) + 1):
            want = starts[k] if k < len(starts) else 2 ** 64 - 1
            assert after_kth(text, k) == want, (at, before, k)


def test_after_kth_fasta_record_edge_cases():
    assert after_kth(b"", 0) == 2 ** 64 - 1
    assert after_kth(b">a\nAC\n", 0) == 0
    assert after_kth(b">a\nAC\n", 1) == 2 ** 64 - 1
    assert after_kth(b" >a\n>b\n", 0) == 4  # whitespace in front of '>' makes a sequence line
    assert after_kth(b"A>a\nC>b\n>c\n", 0) == 8  # '>' in the middle of a line
    assert after_kth(b"\r\n>a\r\n>b", 1) == 6


def read_all(path1, path2=None, batch=7):
    got, counts = [[], []], []
    with native.TextReader(path1, path2, flags=A.PLAN_FASTA) as r:
        while True:
            n, texts, first = r.next(batch)
            if n == 0:
                break
            counts.append(n)
            for m, t in enumerate(texts):
                got[m].append(t)
    return counts, got


def check_batches(text, counts, parts, batch):
    body = text if text.endswith(b"\n") or not text else text + b"\n"
    assert b"".join(parts) == body
    assert sum(counts) == len(record_starts(text))
    assert all(c == batch for c in counts[:-1]) and 0 < counts[-1] <= batch
    for i, (c, p) in enumerate(zip(counts, parts)):
        starts = record_starts(p)
        assert len(starts) == c
        if i:
            assert p.startswith(b">")  # every batch but the first starts at a header


def bgzf(text, piece=1000):
    """BGZF members (bgzip framing) of `piece` text bytes each."""
    out = b""
    for o in range(0, len(text), piece):
        raw = zlib.compressobj(6, zlib.DEFLATED, -15)
        data = raw.compress(text[o:o + piece]) + raw.flush()
        extra = b"BC" + struct.pack("<HH", 2, len(data) + 25)
        out += (b"\x1f\x8b\x08\x04" + b"\0" * 4 + b"\0\xff" + struct.pack("<H", len(extra)) + extra + data +
                struct.pack("<II", zlib.crc32(text[o:o + piece]), len(text[o:o + piece])))
    return out


@pytest.mark.parametrize("form", ["plain", "gzip", "bgzf", "fifo"])
@pytest.mark.parametrize("final_eol", [True, False])
def test_text_reader_cuts_fasta_at_record_starts(tmp_path, form, final_eol):
    rng = random.Random(7)
    text = b"\n \n" + random_fasta(rng, 3000, crlf=False)
    if not final_eol:
        text = text.rstrip(b"\n")
    path = str(tmp_path / "in.fa")
    feeder = None
    if form == "plain":
        open(path, "wb").write(text)
    elif form == "gzip":
        open(path, "wb").write(gzip.compress(text))
    elif form == "bgzf":
        open(path, "wb").write(bgzf(text))
    else:
        os.mkfifo(path)

        def feed():
            with open(path, "wb") as f:
                f.write(text)

        feeder = threading.Thread(target=feed)
        feeder.start()
    for batch in (7, 1000):
        if feeder is None or batch == 7:
            counts, got = read_all(path, batch=batch)
            check_batches(text, counts, got[0], batch)
    if feeder:
        feeder.join()


def test_text_reader_pairs_and_preamble_errors(tmp_path):
    rng = random.Random(3)
    a, b = random_fasta(rng, 500), random_fasta(rng, 500)
    pa, pb = str(tmp_path / "a.fa"), str(tmp_path / "b.fa.gz")
    open(pa, "wb").write(a)
    open(pb, "wb").write(gzip.compress(b))
    counts, got = read_all(pa, pb, batch=64)
    check_batches(a, counts, got[0], 64)
    check_batches(b, counts, got[1], 64)
    bad = str(tmp_path / "bad.fa")
    open(bad, "wb").write(b"\n\nno header\n")
    with pytest.raises(native.NativeError) as e:
        read_all(bad)
    assert e.value.code == A.ERR_FORMAT and "line 3" in str(e.value)


def test_transcoders_native_fasta_starts_only_compression_pumps(tmp_path):
    import bz2

    fa = b">r1\nACGT\n>r2\nGG\n"
    plain, gz, bz = str(tmp_path / "a.fa"), str(tmp_path / "b.fa.gz"), str(tmp_path / "c.fa.bz2")
    open(plain, "wb").write(fa)
    open(gz, "wb").write(gzip.compress(fa))
    with bz2.open(bz, "wb") as f:
        f.write(fa)
    outs = {"trimmed": [str(tmp_path / "o1.fa"), str(tmp_path / "o2.fa.xz")], "short": [str(tmp_path / "s1.fa.gz"), None],
            "untrimmed": None}
    with Transcoders([plain, gz], outs, fasta_native=True) as tc:
        assert tc.fasta and tc.fasta_native
        assert tc.inputs == [plain, gz]  # the library reads plain and gzip FASTA itself
        assert tc.outputs["trimmed"][0] == outs["trimmed"][0] and tc.outputs["short"][0] == outs["short"][0]
        assert tc.outputs["trimmed"][1] != outs["trimmed"][1]  # .xz: a compression pump
        with open(tc.outputs["trimmed"][1], "wb") as w:
            w.write(fa)
    import lzma

    assert lzma.open(outs["trimmed"][1]).read() == fa  # the pump only compressed: FASTA stayed FASTA
    with Transcoders([bz], {"trimmed": [str(tmp_path / "o.fa")]}, fasta_native=True) as tc:
        assert tc.fasta_native and tc.inputs[0] != bz
        with open(tc.inputs[0], "rb") as r:
            assert r.read() == fa  # decompressed, not converted to FASTQ
    with Transcoders([plain], {"trimmed": [str(tmp_path / "p.fa")]}) as tc:
        assert tc.fasta and not tc.fasta_native and tc.inputs[0] != plain  # default: the converting pumps
        with open(tc.inputs[0], "rb") as r:
            assert r.read() == b"@r1\nACGT\n+\nIIII\n@r2\nGG\n+\nII\n"
        open(tc.outputs["trimmed"][0], "wb").close()
