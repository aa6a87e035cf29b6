"""Compression formats - and the one record format - that the native reader / writer does not speak itself.

The reference opens every file through xopen (behind cutadapt's ``InputPaths`` / ``OutputFiles``, run.py:434-436,
751-753), which handles ``.gz``, ``.bz2``, ``.xz`` and ``.zst`` by file name.  The native library reads plain and gzip
(incl. BGZF) files and writes plain and gzip.  For ``.bz2`` and ``.xz`` this module puts a named pipe between the
file and the library and a Python thread on the other end of it (``bz2`` / ``lzma`` release the GIL while they
work): the library sees a plain FASTQ stream, nothing below the C ABI changes.  ``.zst`` goes the same way through the
``zstandard`` module or the ``zstd`` program when the system has one of them (xopen's fallbacks); this image has neither,
and such files are refused with a clear message instead of being misread as plain text.

FASTA input (records without qualities; the reference hands ``qualities=has_qualities()`` on to its output files,
run.py:439, 756) is read and written by the library itself (``CSQ_PLAN_FASTA``; ``Transcoders(..., fasta_native=True)``
leaves such files alone but for their compression).  The converting pumps below stay as the reference the library is
tested against: the pump turns every record into a FASTQ record with a constant quality far above any cutoff - quality
trimming has nothing to remove, as for a read without qualities - and the output pumps write ``>name`` / sequence
records again (dnaio's FASTA writer does not wrap lines), compressed as the file name says.
(Whether the reference itself survives FASTA input is doubtful - run.py:416 / 720 always add cutadapt's QualityTrimmer,
which takes the length of ``read.qualities`` - see DESIGN.md section 7; here such input simply works.)
"""

from __future__ import annotations

import bz2
import errno
import gzip
import lzma
import os
import shutil
import tempfile
import threading

_OPENERS = {".bz2": bz2.open, ".xz": lzma.open, ".lzma": lzma.open}
_ZSTD = (".zst", ".zstd")


class _PipedProgram:
    """File object over an external (de)compressor, the way xopen falls back to programs: ``zstd -dc file`` for reading,
    ``zstd -c > file`` for writing."""

    def __init__(self, argv, path, mode):
        import subprocess

        self._writing = "w" in mode
        if self._writing:
            self._sink = open(path, "wb")
            self._p = subprocess.Popen(argv, stdin=subprocess.PIPE, stdout=self._sink)
            self._f = self._p.stdin
        else:
            self._sink = None
            self._p = subprocess.Popen(argv + [path], stdout=subprocess.PIPE)
            self._f = self._p.stdout

    def read(self, n=-1):
        return self._f.read(n)

    def readline(self):
        return self._f.readline()

    def __iter__(self):
        return iter(self._f)

    def write(self, data):
        return self._f.write(data)

    def close(self):
        self._f.close()
        rc = self._p.wait()
        if self._sink:
            self._sink.close()
        if rc != 0:
            raise OSError(f"{self._p.args[0]} exited with status {rc}")

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
        return False


def _zstd_opener(path):
    """zstd through the ``zstandard`` module or the ``zstd`` program, whichever the system has (xopen's order); neither
    ships with this image, where such files are refused with a clear message instead of being misread as plain text."""
    try:
        import zstandard  # noqa: F401

        return lambda p, mode: zstandard.open(p, mode)
    except ImportError:
        pass
    prog = shutil.which("zstd")
    if prog:
        return lambda p, mode: _PipedProgram([prog, "-q", "-c"] if "w" in mode else [prog, "-q", "-dc"], p, mode)
    raise ValueError(f"{path}: zstd-compressed files need the zstandard module or the zstd program, and this system has neither "
                     "(use .gz, .bz2, .xz or plain FASTQ)")


def _opener(path):
    if path is None:
        return None
    low = str(path).lower()
    for ext in _ZSTD:
        if low.endswith(ext):
            return _zstd_opener(path)
    for ext, fn in _OPENERS.items():
        if low.endswith(ext):
            return fn
    return None


def _reader(path):
    """Opener for reading a file of any supported compression (used for FASTA inputs and for sniffing)."""
    return _opener(path) or (gzip.open if str(path).lower().endswith(".gz") else open)


def _writer(path):
    """Opener for writing FASTA outputs: compression as the file name says (gzip at level 1 like the native writer)."""
    fn = _opener(path)
    if fn:
        return fn
    if str(path).lower().endswith(".gz"):
        return lambda p, mode: gzip.open(p, mode, compresslevel=1)
    return open


def is_fasta(path) -> bool:
    """dnaio tells the formats apart by the first character of the content: '>' is FASTA, '@' FASTQ."""
    try:
        if not os.path.isfile(path):
            return False
        with _reader(path)(path, "rb") as f:
            while True:
                c = f.read(1)
                if not c:
                    return False
                if c not in b" \t\r\n":
                    return c == b">"
    except (OSError, EOFError, lzma.LZMAError):
        return False


FASTA_QUALITY = b"I"  # Q40 at base 33: above any cutoff, so that quality trimming leaves such reads alone


def fasta_to_fastq(src, dst):
    """FASTA records (sequences may span lines) -> FASTQ records with a constant quality."""
    name, parts = None, []

    def flush():
        if name is not None:
            seq = b"".join(parts)
            dst.write(b"@" + name + b"\n" + seq + b"\n+\n" + FASTA_QUALITY * len(seq) + b"\n")

    for line in src:
        if line.startswith(b">"):
            flush()
            name, parts = line[1:].rstrip(b"\r\n"), []
        elif name is None:
            if line.strip():
                raise ValueError("FASTA input does not start with a '>' header")
        else:
            parts.append(line.strip())
    flush()


def fastq_to_fasta(src, dst):
    """FASTQ records as the library writes them (four lines each) -> '>name' / sequence records."""
    while True:
        header = src.readline()
        if not header:
            return
        seq = src.readline()
        src.readline()
        src.readline()
        dst.write(b">" + header[1:] + seq)


class Transcoders:
    """Context manager: ``tc.inputs`` / ``tc.outputs`` are what the library should open instead of the given paths.

    ``tc.fasta`` tells whether the inputs are FASTA, ``tc.fasta_native`` whether the library is to read them as such.  By default FASTA goes through the converting pumps (the library
    sees FASTQ); with ``fasta_native=True`` only compressions the library cannot read or write get a pump, and the
    caller runs the library with ``CSQ_PLAN_FASTA``."""

    def __init__(self, inputs, outputs, fasta_native=False):
        self.inputs = list(inputs)
        self.outputs = {k: list(v) if v else v for k, v in outputs.items()}
        self._threads = []  # (thread, fifo, "in" | "out")
        self._errors = []
        self._tmp = None
        in_jobs = [(i, p, _opener(p)) for i, p in enumerate(self.inputs)]
        out_jobs = [(k, m, p, _opener(p)) for k, v in self.outputs.items() if v for m, p in enumerate(v)]
        fasta = [is_fasta(p) for p in self.inputs if p]
        self.fasta = bool(fasta) and all(fasta)
        if any(fasta) and not self.fasta:
            raise ValueError("the input files differ in format (FASTA and FASTQ)")
        self.fasta_native = self.fasta and fasta_native  # the library reads and writes these FASTA files itself
        self._convert = self.fasta and not fasta_native
        if self._convert:  # every input and every output goes through a converting pump
            self._in_jobs = [(i, p, _reader(p)) for i, p, _ in in_jobs if p]
            self._out_jobs = [(k, m, p, _writer(p)) for k, m, p, _ in out_jobs if p]
        else:
            self._in_jobs = [j for j in in_jobs if j[2]]
            self._out_jobs = [j for j in out_jobs if j[3]]

    def __enter__(self):
        if not self._in_jobs and not self._out_jobs:
            return self
        self._tmp = tempfile.mkdtemp(prefix="cutseq_b200_")
        for i, path, opener in self._in_jobs:
            fifo = os.path.join(self._tmp, f"in_{i}.fq")
            os.mkfifo(fifo)
            self.inputs[i] = fifo
            self._start(self._feed_fasta if self._convert else self._feed, (path, opener, fifo), fifo, "in")
        for k, m, path, opener in self._out_jobs:
            fifo = os.path.join(self._tmp, f"out_{k}_{m}.fq")  # no compression suffix: the library writes plain text
            os.mkfifo(fifo)
            self.outputs[k][m] = fifo
            self._start(self._drain_fasta if self._convert else self._drain, (path, opener, fifo), fifo, "out")
        return self

    def _start(self, fn, args, fifo, side):
        t = threading.Thread(target=self._guard, args=(fn, args), daemon=True)
        t.start()
        self._threads.append((t, fifo, side))

    def _guard(self, fn, args):
        try:
            fn(*args)
        except BrokenPipeError:
            pass  # the library stopped reading (it reports its own error)
        except Exception as exc:  # surfaced by __exit__
            self._errors.append(exc)

    @staticmethod
    def _feed(path, opener, fifo):
        with opener(path, "rb") as src, open(fifo, "wb") as dst:
            shutil.copyfileobj(src, dst, 1 << 20)

    @staticmethod
    def _drain(path, opener, fifo):
        with open(fifo, "rb") as src, opener(path, "wb") as dst:
            shutil.copyfileobj(src, dst, 1 << 20)

    @staticmethod
    def _feed_fasta(path, opener, fifo):
        with opener(path, "rb") as src, open(fifo, "wb", buffering=1 << 20) as dst:
            fasta_to_fastq(src, dst)

    @staticmethod
    def _drain_fasta(path, opener, fifo):
        with open(fifo, "rb", buffering=1 << 20) as src, opener(path, "wb") as dst:
            fastq_to_fasta(src, dst)

    def __exit__(self, exc_type, exc, tb):
        # The library has returned: a pump that is still running is either busy (it ends at the end of its pipe) or
        # waiting in open() for a pipe the library never opened - the other end is opened for a moment to release it.
        for t, fifo, side in self._threads:
            t.join(timeout=0.05 if exc_type else 0.5)
            while t.is_alive():
                try:
                    fd = os.open(fifo, (os.O_RDONLY if side == "in" else os.O_WRONLY) | os.O_NONBLOCK)
                    os.close(fd)
                except OSError as e:
                    if e.errno not in (errno.ENXIO, errno.ENOENT):
                        raise
                t.join(timeout=0.2)
        if self._tmp:
            shutil.rmtree(self._tmp, ignore_errors=True)
        if exc_type is None and self._errors:
            raise self._errors[0]
        return False
