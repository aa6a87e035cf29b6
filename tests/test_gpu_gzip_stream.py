"""The device decoder of ordinary gzip files (csrc/gz_stream.cu) on the GPU: against zlib and the host twin (outputs
and decode chains), and damage."""

import os
import random
import zlib

import pytest

from cutseq_b200 import _abi as A
from cutseq_b200 import native
from tests.test_gz_stream_host import STRATEGIES, deflate
from tests.test_inflate import fastq, gz

pytestmark = pytest.mark.gpu


def both(comp, cap, span, rnd):
    dev = native.gz_stream_inflate(comp, cap, 0, span, rnd, chain=True)
    host = native.gz_stream_inflate_host(comp, cap, span, rnd, chain=True)
    assert dev[1] == host[1]  # the same spans, starts, ends and symbol counts
    return dev[0]


@pytest.mark.parametrize("level", [0, 1, 6, 9])
def test_device_equals_zlib_and_the_host_twin(level):
    text = fastq(6000, seed=41)
    for strategy in STRATEGIES:
        for mem in (1, 8, 9):
            comp = deflate(text, level, strategy, mem)
            for span, rnd in ((1000, 7000), (20000, 60000), (0, 0)):
                assert both(comp, len(text), span, rnd) == text, (level, strategy, mem, span, rnd)


def test_windows_members_bgzf_binary_and_large():
    text = fastq(12000, seed=42)
    for wbits in (25, 28, 31):
        assert both(deflate(text, 9, wbits=wbits), len(text), 1500, 9000) == text
    parts = [text[:100], b"", text[100:300_000], text[300_000:300_001], text[300_001:]]
    comp = b"".join(gz(p) for p in parts) + bytes(64)
    for span, rnd in ((1000, 4000), (50_000, 0)):
        assert both(comp, len(text), span, rnd) == text
    a = gz(text[:200_000])
    for rnd in (len(a) - 1, len(a), len(a) + 8):
        assert both(a + gz(text[200_000:]), len(text), 1000, rnd) == text
    from scripts import bench_files

    assert both(bench_files.bgzf_compress(text, 2), len(text), 1000, 20_000) == text
    assert both(bench_files.gzip_single_member(text, 4, level=6, piece=100_000), len(text), 2000, 50_000) == text
    blob = os.urandom(100_000) + bytes(random.Random(5).choice(b"\x00\x01\xfe\xffAB") for _ in range(400_000))
    assert both(gz(blob), len(blob), 30_000, 0) == blob
    big = fastq(150_000, seed=45)  # ~30 MB of text: hundreds of spans with the default sizes, several rounds
    comp = gz(big, 6)
    assert native.gz_stream_inflate(comp, len(big)) == big
    assert native.gz_stream_inflate(comp, len(big), 0, 0, len(comp) // 5) == big


def test_random_streams():
    rng = random.Random(77)
    for it in range(40):
        data = fastq(rng.randint(1, 3000), seed=it) if it % 3 else os.urandom(rng.randint(0, 100_000))
        cuts = sorted(rng.randint(0, len(data)) for _ in range(rng.randint(0, 3)))
        comp = b"".join(deflate(data[a:b], rng.choice([1, 4, 6, 9]), rng.choice(STRATEGIES), rng.choice([1, 8, 9]))
                        for a, b in zip([0] + cuts, cuts + [len(data)]))
        span, rnd = rng.choice([1000, 3000, 10000, 40000, 0]), rng.choice([0, 5000, 30000])
        assert both(comp, len(data) + 1, span, rnd) == data, (it, span, rnd)


def test_damage_is_an_error_on_the_device():
    text = fastq(20000, seed=13)
    comp = gz(text)
    rng = random.Random(17)
    for k in range(24):
        bad = bytearray(comp)
        bad[rng.randrange(10, len(bad))] ^= 1 << rng.randrange(8)
        with pytest.raises(native.NativeError):
            native.gz_stream_inflate(bytes(bad), len(text) + 100_000, 0, 5000 if k % 2 else 0, 30_000 if k % 3 else 0)
    for cut in (12, len(comp) // 2, len(comp) - 1):
        with pytest.raises(native.NativeError):
            native.gz_stream_inflate(comp[:cut], len(text), 0, 2000, 30_000)
    for pos, what in ((-8, "CRC"), (-4, "ISIZE")):
        bad = bytearray(comp)
        bad[pos] ^= 1
        with pytest.raises(native.NativeError, match=what):
            native.gz_stream_inflate(bytes(bad), len(text) + 10, 0, 2000, 30_000)
    with pytest.raises(native.NativeError, match="garbage"):
        native.gz_stream_inflate(comp + b"garbage!" * 20, len(text), 0, 2000, 30_000)
    with pytest.raises(native.NativeError) as e:
        native.gz_stream_inflate(comp, len(text) - 1, 0, 2000, 30_000)
    assert e.value.code == A.ERR_CAPACITY
    assert native.gz_stream_inflate(comp, len(text), 0, 2000, 30_000) == text  # the device is still fine
