"""The device decoder of ordinary gzip files (csrc/gz_stream.cu) run by its host twin against zlib - no GPU needed.

The twin runs the same span search, span decode, window and resolve code as k_gzs_search / k_gzs_decode / k_gzs_window /
k_gzs_resolve, with one lane, under the same round orchestration.  Small spans and rounds make many of both out of
small inputs, so member ends, continuations and round cuts land everywhere."""

import os
import random
import zlib

import pytest

from cutseq_b200 import _abi as A
from cutseq_b200 import native
from tests.test_inflate import fastq, gz


def inflate(comp, cap, span=0, rnd=0):
    return native.gz_stream_inflate_host(comp, cap, span, rnd)


STRATEGIES = [zlib.Z_DEFAULT_STRATEGY, zlib.Z_FIXED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FILTERED]


def deflate(data, level, strategy=zlib.Z_DEFAULT_STRATEGY, mem=8, wbits=31):
    c = zlib.compressobj(level, zlib.DEFLATED, wbits, mem, strategy)
    return c.compress(data) + c.flush()


@pytest.mark.parametrize("level", [0, 1, 6, 9])
def test_levels_strategies_and_memory_levels(level):
    text = fastq(6000, seed=41)
    for strategy in STRATEGIES:
        for mem in (1, 8, 9):
            comp = deflate(text, level, strategy, mem)
            for span, rnd in ((1000, 7000), (20000, 60000), (0, 0)):
                assert inflate(comp, len(text), span, rnd) == text, (level, strategy, mem, span, rnd)


def test_window_bits():
    text = fastq(12000, seed=42)
    for wbits in (25, 28, 31):  # 512-byte, 4 KiB and 32 KiB windows
        comp = deflate(text, 9, wbits=wbits)
        for span, rnd in ((1500, 9000), (30000, 0)):
            assert inflate(comp, len(text), span, rnd) == text, (wbits, span, rnd)


def test_many_spans_and_rounds_match_zlib_with_the_chain_in_order():
    text = fastq(30000, seed=11)
    for level in (1, 6, 9):
        comp = gz(text, level)
        for span, rnd in ((1000, 5000), (20000, 100000), (150000, 0)):
            got, chain = native.gz_stream_inflate_host(comp, len(text), span, rnd, chain=True)
            assert got == text
            # the chain covers the stream without gaps, and its symbols are the text
            assert all(a[1] == b[0] for a, b in zip(chain, chain[1:]))
            assert sum(c[2] for c in chain) == len(text)
            assert len(chain) > 1


def test_members_padding_and_bgzf():
    text = fastq(8000, seed=12)
    # members that are empty, one byte long, or end inside spans; zero padding between and behind them
    parts = [text[:100], b"", text[100:300_000], text[300_000:300_001], text[300_001:]]
    comp = b"".join(gz(p) for p in parts) + bytes(64)
    for span, rnd in ((1000, 4000), (5000, 50_000), (50_000, 0), (1 << 20, 0)):
        assert inflate(comp, len(text), span, rnd) == text, (span, rnd)
    padded = gz(text[:5000]) + bytes(7) + gz(text[5000:])
    assert inflate(padded, len(text), 1000, 3000) == text
    # BGZF framing: thousands of small members, each with an extra field (more than a span holds)
    from scripts import bench_files

    bg = bench_files.bgzf_compress(text, 2)
    for span, rnd in ((1000, 20_000), (100_000, 0)):
        assert inflate(bg, len(text), span, rnd) == text


def test_member_boundary_exactly_at_a_round_cut():
    text = fastq(4000, seed=43)
    a = gz(text[:200_000])
    comp = a + gz(text[200_000:])
    for rnd in (len(a) - 1, len(a), len(a) + 1, len(a) + 8, len(a) + 10):
        assert inflate(comp, len(text), 1000, rnd) == text, rnd


def test_stored_fixed_tiny_and_binary_inputs():
    text = fastq(3000, seed=44)
    for data in (text, b"", b"A", b"ACGT\n" * 3):
        for level, strategy in ((0, zlib.Z_DEFAULT_STRATEGY), (1, zlib.Z_FIXED), (9, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_HUFFMAN_ONLY)):
            assert inflate(gz(data, level, strategy), len(data), 1000, 10_000) == data
    # content that is not text: no block start passes the search, continuations walk the stream
    rng = random.Random(5)
    blob = os.urandom(100_000) + bytes(rng.choice(b"\x00\x01\xfe\xffAB") for _ in range(400_000))
    for span, rnd in ((30_000, 0), (2000, 40_000)):
        assert inflate(gz(blob), len(blob), span, rnd) == blob
    zeros = bytes(3_000_000)  # 1000:1 - a block decodes to more than a span holds
    assert inflate(gz(zeros, 9), len(zeros), 1000, 0) == zeros


def test_random_streams():
    """Random contents, members, levels, strategies, memory levels (tiny blocks), span and round sizes against zlib."""
    rng = random.Random(99)

    def reads(n):
        out = []
        for i in range(n):
            ln = rng.randint(1, 300)
            out.append(f"@M{rng.randint(0, 9)}:{i} {'x' * rng.randint(0, 30)}\n{''.join(rng.choice('ACGTN') for _ in range(ln))}\n+\n"
                       f"{''.join(rng.choice('FFFFFF:,#') for _ in range(ln))}\n")
        return "".join(out).encode()

    for it in range(40):
        kind = rng.choice(["fastq", "fastq", "mixed", "binary", "lines"])
        if kind == "fastq":
            data = reads(rng.randint(1, 4000))
        elif kind == "mixed":
            data = reads(rng.randint(100, 1500)) + os.urandom(rng.randint(0, 50000)) + reads(rng.randint(100, 1500))
        elif kind == "binary":
            data = os.urandom(rng.randint(0, 150000))
        else:
            data = b"".join(bytes(rng.choice(b"ab\n") for _ in range(rng.randint(0, 80))) + b"\n" for _ in range(rng.randint(0, 15000)))
        cuts = sorted(rng.randint(0, len(data)) for _ in range(rng.randint(0, 3)))
        parts = [data[a:b] for a, b in zip([0] + cuts, cuts + [len(data)])]
        comp = b""
        for p in parts:
            comp += deflate(p, rng.choice([1, 1, 4, 6, 6, 9]), rng.choice([zlib.Z_DEFAULT_STRATEGY] * 4 + [zlib.Z_FIXED, zlib.Z_RLE, zlib.Z_HUFFMAN_ONLY, zlib.Z_FILTERED]),
                            rng.choice([1, 8, 9]))
        if rng.random() < 0.2:
            comp += bytes(rng.randint(1, 40))  # zero padding behind the last member
        span, rnd = rng.choice([1000, 3000, 10000, 40000, 200000, 0]), rng.choice([0, 0, 5000, 30000, 100000])
        assert inflate(comp, len(data) + 1, span, rnd) == data, (it, kind, len(data), span, rnd)


def test_bench_fixture():
    from scripts import bench_files

    text = fastq(5000, seed=31)
    comp = bench_files.gzip_single_member(text, 4, level=6, piece=100_000)
    for span, rnd in ((2000, 50_000), (0, 0)):
        assert inflate(comp, len(text), span, rnd) == text


def test_damage_is_an_error():
    text = fastq(20000, seed=13)
    comp = gz(text)
    for pos in (30, len(comp) // 3, len(comp) // 2, len(comp) - 6):  # bit flips in the stream and the trailer
        bad = bytearray(comp)
        bad[pos] ^= 0x55
        with pytest.raises(native.NativeError) as e:
            inflate(bytes(bad), len(text) + 100_000, 2000, 30_000)
        assert e.value.code == A.ERR_IO
    rng = random.Random(17)
    for _ in range(20):
        bad = bytearray(comp)
        bad[rng.randrange(10, len(bad))] ^= 1 << rng.randrange(8)
        with pytest.raises(native.NativeError):
            inflate(bytes(bad), len(text) + 100_000, 5000, 0)
    for cut in (5, 12, len(comp) // 2, len(comp) - 9, len(comp) - 1):  # truncation
        with pytest.raises(native.NativeError):
            inflate(comp[:cut], len(text), 2000, 30_000)
    crc = bytearray(comp)
    crc[-8] ^= 1  # CRC-32
    with pytest.raises(native.NativeError, match="CRC"):
        inflate(bytes(crc), len(text), 2000, 30_000)
    isize = bytearray(comp)
    isize[-4] ^= 1  # ISIZE
    with pytest.raises(native.NativeError, match="ISIZE"):
        inflate(bytes(isize), len(text) + 10, 2000, 30_000)
    with pytest.raises(native.NativeError, match="garbage"):
        inflate(comp + b"garbage!" * 20, len(text), 2000, 30_000)
    with pytest.raises(native.NativeError):
        inflate(b"not gzip at all, not at all", 100)
    with pytest.raises(native.NativeError) as e:
        inflate(comp, len(text) - 1, 2000, 30_000)
    assert e.value.code == A.ERR_CAPACITY
