"""ctypes binding of libcutseq_b200.so (the C ABI of include/cutseq_b200.h).

This is the only execution path of the package: if the CUDA library is missing or no
B200 is visible, calls fail loudly (``NativeError``); there is no CPU fallback.
"""

from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _abi as A

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libcutseq_b200.so")
_lib = None


class NativeError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"cutseq_b200 native error {code}: {message}")
        self.code = code


def lib():
    """Load the CUDA library (built by ``cutseq_b200.build.build()``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError(A.ERR_NO_DEVICE, f"{LIB_PATH} is missing - build it with `python -m cutseq_b200.build` "
                          "(there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    L.csq_last_error.restype = C.c_char_p
    vp, i32, u32, u64p = C.c_void_p, C.c_int, C.c_uint32, C.POINTER(C.c_uint64)
    L.csq_plan_create.argtypes = [C.POINTER(A.csq_op), i32, C.POINTER(A.csq_op), i32, C.POINTER(A.csq_filters), i32, u32, C.POINTER(vp)]
    L.csq_plan_destroy.argtypes = [vp]
    L.csq_plan_destroy.restype = None
    L.csq_submit.argtypes = [vp, i32, C.POINTER(A.csq_batch_in), C.POINTER(A.csq_batch_out)]
    L.csq_submit_text.argtypes = [vp, i32, C.POINTER(A.csq_batch_text), C.POINTER(A.csq_batch_out)]
    L.csq_upload_text.argtypes = [vp, i32, C.POINTER(A.csq_batch_text)]
    L.csq_submit_bgzf.argtypes = [vp, i32, C.POINTER(A.csq_batch_bgzf), C.POINTER(A.csq_batch_out)]
    L.csq_bgzf_count_lines.argtypes = [vp, i32, C.POINTER(A.csq_bgzf_in), vp]
    L.csq_wait.argtypes = [vp, i32]
    L.csq_slot_times.argtypes = [vp, i32, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    L.csq_upload.argtypes = [vp, i32, C.POINTER(A.csq_batch_in)]
    L.csq_run_resident.argtypes = [vp, i32, i32, C.POINTER(C.c_float)]
    L.csq_run_steps.argtypes = [vp, C.POINTER(i32), i32, i32, C.POINTER(C.c_float)]
    L.csq_kernel_times.argtypes = [vp, i32, C.POINTER(C.c_char_p), C.POINTER(C.c_float), i32]
    L.csq_launch_count.argtypes = [vp, u64p]
    L.csq_fetch_results.argtypes = [vp, i32, i32, vp, u32]
    L.csq_fetch_matches.argtypes = [vp, i32, i32, i32, vp, u32]
    L.csq_fetch_text.argtypes = [vp, i32, C.POINTER(A.csq_batch_out)]
    L.csq_stats.argtypes = [vp, C.POINTER(A.csq_counters)]
    L.csq_locate_batch.argtypes = [i32, C.POINTER(A.csq_op), C.POINTER(A.csq_mate_in), u32, u32, vp]
    L.csq_int_peak.argtypes = [i32, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.csq_pcie_peak.argtypes = [i32, C.c_uint64, C.c_uint64, i32, i32, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.csq_bind_host_to_device.argtypes = [i32, C.POINTER(C.c_int)]
    L.csq_unbind_host.argtypes = []
    L.csq_device_count.argtypes = [C.POINTER(i32)]
    if hasattr(L, "csq_run_files"):
        L.csq_run_files.argtypes = [C.POINTER(A.csq_op), i32, C.POINTER(A.csq_op), i32, C.POINTER(A.csq_filters), u32,
                                    C.POINTER(A.csq_files), C.POINTER(A.csq_counters), C.POINTER(A.csq_timing)]
        L.csq_reader_open.argtypes = [C.c_char_p, C.c_char_p, C.POINTER(vp)]
        L.csq_reader_next.argtypes = [vp, i32, u32, C.POINTER(A.csq_batch_in)]
        L.csq_reader_close.argtypes = [vp]
        L.csq_reader_close.restype = None
        L.csq_parse_fastq_mem.argtypes = [vp, C.c_uint64, u32, vp, vp, C.c_uint64, vp, vp, vp, C.c_uint64, vp,
                                          C.POINTER(u32), u64p, u64p]
        L.csq_text_reader_open.argtypes = [C.c_char_p, C.c_char_p, C.POINTER(vp)]
        L.csq_text_reader_open_flags.argtypes = [C.c_char_p, C.c_char_p, u32, C.POINTER(vp)]
        L.csq_text_reader_next.argtypes = [vp, i32, u32, C.POINTER(A.csq_batch_text)]
        L.csq_text_reader_close.argtypes = [vp]
        L.csq_text_reader_close.restype = None
        L.csq_count_newlines.argtypes = [vp, C.c_uint64]
        L.csq_count_newlines.restype = C.c_uint64
        L.csq_after_kth_newline.argtypes = [vp, C.c_uint64, C.c_uint64]
        L.csq_after_kth_newline.restype = C.c_uint64
        L.csq_after_kth_fasta_record.argtypes = [vp, C.c_uint64, C.c_uint64]
        L.csq_after_kth_fasta_record.restype = C.c_uint64
        L.csq_gunzip_mem.argtypes = [vp, C.c_uint64, vp, C.c_uint64, C.c_uint64, u64p]
        L.csq_format_fastq.argtypes = [C.POINTER(A.csq_mate_in), u32, vp, C.c_uint64, u64p]
        L.csq_gz_deflate_host.argtypes = [vp, C.c_uint64, vp, C.c_uint64, u64p]
        L.csq_gz_inflate_host.argtypes = [vp, C.c_uint64, vp, C.c_uint64, u64p, u64p]
        L.csq_pinflate_mem.argtypes = [vp, C.c_uint64, vp, C.c_uint64, C.c_int, C.c_uint64, u64p]
        L.csq_gz_stream_inflate.argtypes = [i32, vp, C.c_uint64, vp, C.c_uint64, C.c_uint64, C.c_uint64, u64p]
        L.csq_gz_stream_inflate_host.argtypes = [vp, C.c_uint64, vp, C.c_uint64, C.c_uint64, C.c_uint64, u64p]
        L.csq_gz_stream_chain.argtypes = [u64p, C.c_uint64]
        L.csq_gz_stream_chain.restype = C.c_uint64
    if hasattr(L, "csq_synth_batch"):
        L.csq_synth_batch.argtypes = [C.POINTER(A.csq_synth), C.c_uint64, u32, i32, C.POINTER(A.csq_batch_in)]
        L.csq_synth_free.restype = None
    if L.csq_abi_version() != A.ABI_VERSION:
        raise NativeError(A.ERR_INVALID, "ABI version mismatch between libcutseq_b200.so and cutseq_b200/_abi.py")
    _lib = L
    return L


def check(rc: int):
    if rc != 0:
        raise NativeError(rc, lib().csq_last_error().decode("utf-8", "replace"))


def device_count() -> int:
    n = C.c_int(0)
    check(lib().csq_device_count(C.byref(n)))
    return n.value


MATCH_DTYPE = np.dtype([(k, "i2") for k in ("found", "ref_start", "ref_stop", "query_start", "query_stop", "score", "errors", "reserved")])
RESULT_DTYPE = np.dtype([("start", "u4"), ("stop", "u4"), ("dest", "u4"), ("matched", "u4")])


class Plan:
    """A compiled op program bound to one GPU (``csq_plan``)."""

    def __init__(self, program, device: int = 0, flags: int = 0):
        self.program = program
        self._ops1, self._n1 = program.c_ops(0)
        self._ops2, self._n2 = program.c_ops(1)
        self._flt = program.filters.to_c()
        self._h = C.c_void_p()
        self.device = device
        check(lib().csq_plan_create(self._ops1, self._n1, self._ops2, self._n2 if program.paired else 0,
                                    C.byref(self._flt), device, flags, C.byref(self._h)))

    def close(self):
        if self._h:
            lib().csq_plan_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ---- batch execution with host buffers (the end-to-end path) ----
    def submit(self, slot: int, batch: A.csq_batch_in, out: A.csq_batch_out):
        check(lib().csq_submit(self._h, slot, C.byref(batch), C.byref(out)))

    def submit_text(self, slot: int, batch: A.csq_batch_text, out: A.csq_batch_out):
        check(lib().csq_submit_text(self._h, slot, C.byref(batch), C.byref(out)))

    def upload_text(self, slot: int, batch: A.csq_batch_text):
        check(lib().csq_upload_text(self._h, slot, C.byref(batch)))

    def run_text(self, texts, n_reads: int, capacity: int | None = None, slot: int = 0, first_record: int = 0):
        """FASTQ text per mate (bytes) through csq_submit_text + csq_wait. -> text[d][m] bytes, records[d][m]"""
        tb = TextBatch(texts, n_reads, first_record)
        if capacity is None:
            capacity = max(len(t) for t in texts) + 64 * n_reads + 4096
        out = A.csq_batch_out()
        bufs = [[np.empty(capacity, dtype=np.uint8) for _ in range(2)] for _ in range(A.CSQ_N_DEST)]
        for d in range(A.CSQ_N_DEST):
            for m in range(2):
                out.text[d][m].data = bufs[d][m].ctypes.data
                out.text[d][m].capacity = capacity
        self.submit_text(slot, tb.c, out)
        self.wait(slot)
        text = [[bufs[d][m][: out.text[d][m].bytes].tobytes() for m in range(2)] for d in range(A.CSQ_N_DEST)]
        records = [[int(out.text[d][m].records) for m in range(2)] for d in range(A.CSQ_N_DEST)]
        return text, records

    def wait(self, slot: int):
        check(lib().csq_wait(self._h, slot))

    def bgzf_count_lines(self, members: "BgzfRun", slot: int = 3):
        """Line ends per member of a run of BGZF members (``csq_bgzf_count_lines``). -> numpy uint32 array"""
        out = np.zeros(max(members.c.n_members, 1), dtype=np.uint32)
        check(lib().csq_bgzf_count_lines(self._h, slot, C.byref(members.c), out.ctypes.data))
        return out[: members.c.n_members] & np.uint32(0x7FFFFFFF)

    def run_bgzf(self, runs, n_reads: int, capacity: int, slot: int = 0, first_record: int = 0):
        """BGZF member runs per mate (BgzfRun) through csq_submit_bgzf + csq_wait. -> out[d][m] bytes, records[d][m]"""
        b = A.csq_batch_bgzf()
        b.n_reads, b.n_mates, b.first_record = n_reads, len(runs), first_record
        for m, r in enumerate(runs):
            b.mate[m] = r.c
        out = A.csq_batch_out()
        bufs = [[np.empty(capacity, dtype=np.uint8) for _ in range(2)] for _ in range(A.CSQ_N_DEST)]
        for d in range(A.CSQ_N_DEST):
            for m in range(2):
                out.text[d][m].data = bufs[d][m].ctypes.data
                out.text[d][m].capacity = capacity
        check(lib().csq_submit_bgzf(self._h, slot, C.byref(b), C.byref(out)))
        self.wait(slot)
        text = [[bufs[d][m][: out.text[d][m].bytes].tobytes() for m in range(2)] for d in range(A.CSQ_N_DEST)]
        records = [[int(out.text[d][m].records) for m in range(2)] for d in range(A.CSQ_N_DEST)]
        return text, records

    def slot_times(self, slot: int):
        t, k = C.c_float(), C.c_float()
        check(lib().csq_slot_times(self._h, slot, C.byref(t), C.byref(k)))
        return t.value, k.value

    def run_batch(self, batch: A.csq_batch_in, capacity: int | None = None, slot: int = 0):
        """submit + wait with freshly allocated numpy output buffers. -> text[d][m] bytes, records[d][m]"""
        if capacity is None:
            capacity = 64
            for m in range(batch.n_mates):
                capacity = max(capacity, int(batch.mate[m].name_bytes) + 2 * int(batch.mate[m].seq_bytes) + 80 * int(batch.n_reads) + 64)
        out = A.csq_batch_out()
        bufs = [[np.empty(capacity, dtype=np.uint8) for _ in range(2)] for _ in range(A.CSQ_N_DEST)]
        for d in range(A.CSQ_N_DEST):
            for m in range(2):
                out.text[d][m].data = bufs[d][m].ctypes.data
                out.text[d][m].capacity = capacity
        self.submit(slot, batch, out)
        self.wait(slot)
        text = [[bufs[d][m][: out.text[d][m].bytes].tobytes() for m in range(2)] for d in range(A.CSQ_N_DEST)]
        records = [[int(out.text[d][m].records) for m in range(2)] for d in range(A.CSQ_N_DEST)]
        return text, records

    # ---- resident mode (measurement) ----
    def upload(self, slot: int, batch: A.csq_batch_in):
        check(lib().csq_upload(self._h, slot, C.byref(batch)))

    def run_resident(self, slot: int, iters: int) -> float:
        ms = C.c_float()
        check(lib().csq_run_resident(self._h, slot, iters, C.byref(ms)))
        return ms.value

    def run_steps(self, slots, steps: int) -> float:
        """`steps` resident steps round-robin over `slots`, back to back on one stream. -> total ms (CUDA events)"""
        arr = (C.c_int * len(slots))(*slots)
        ms = C.c_float()
        check(lib().csq_run_steps(self._h, arr, len(slots), steps, C.byref(ms)))
        return ms.value

    def kernel_times(self, slot: int):
        names = (C.c_char_p * 64)()
        ms = (C.c_float * 64)()
        n = lib().csq_kernel_times(self._h, slot, names, ms, 64)
        return [(names[i].decode(), ms[i]) for i in range(n)]

    def launch_count(self) -> int:
        v = C.c_uint64()
        check(lib().csq_launch_count(self._h, C.byref(v)))
        return v.value

    def results(self, slot: int, mate: int, n: int):
        out = np.zeros(max(n, 1), dtype=RESULT_DTYPE)
        check(lib().csq_fetch_results(self._h, slot, mate, out.ctypes.data, n))
        return out[:n]

    def matches(self, slot: int, mate: int, op_index: int, n: int):
        out = np.zeros(max(n, 1), dtype=MATCH_DTYPE)
        check(lib().csq_fetch_matches(self._h, slot, mate, op_index, out.ctypes.data, n))
        return out[:n]

    def fetch_text(self, slot: int, capacity: int):
        out = A.csq_batch_out()
        bufs = [[np.empty(capacity, dtype=np.uint8) for _ in range(2)] for _ in range(A.CSQ_N_DEST)]
        for d in range(A.CSQ_N_DEST):
            for m in range(2):
                out.text[d][m].data = bufs[d][m].ctypes.data
                out.text[d][m].capacity = capacity
        check(lib().csq_fetch_text(self._h, slot, C.byref(out)))
        return [[bufs[d][m][: out.text[d][m].bytes].tobytes() for m in range(2)] for d in range(A.CSQ_N_DEST)]

    def stats(self) -> A.csq_counters:
        c = A.csq_counters()
        check(lib().csq_stats(self._h, C.byref(c)))
        return c


class TextBatch:
    """csq_batch_text over Python-owned buffers (bytes / numpy uint8 arrays / torch pinned tensors via .data_ptr())."""

    def __init__(self, texts, n_reads: int, first_record: int = 0):
        self.keep = []
        self.c = A.csq_batch_text()
        self.c.n_reads = n_reads
        self.c.n_mates = len(texts)
        self.c.first_record = first_record
        for m, t in enumerate(texts):
            if hasattr(t, "data_ptr"):
                ptr, size = t.data_ptr(), t.numel()
            else:
                arr = np.frombuffer(t, dtype=np.uint8) if not isinstance(t, np.ndarray) else t
                ptr, size = arr.ctypes.data, arr.size
                t = arr
            self.keep.append(t)
            self.c.mate[m].text = ptr
            self.c.mate[m].bytes = size


class BgzfRun:
    """csq_bgzf_in over a bytes object holding whole BGZF members: walks the member headers ('BC' field, ISIZE)."""

    def __init__(self, data: bytes, skip_lines: int = 0, append_newline: bool = False):
        moff, ooff = [0], [0]
        pos = 0
        while pos < len(data):
            if data[pos : pos + 4] != b"\x1f\x8b\x08\x04" or data[pos + 12 : pos + 14] != b"BC":
                raise ValueError("not a BGZF member")
            size = int.from_bytes(data[pos + 16 : pos + 18], "little") + 1
            isize = int.from_bytes(data[pos + size - 4 : pos + size], "little")
            pos += size
            moff.append(pos)
            ooff.append(ooff[-1] + isize)
        self.data = np.frombuffer(data + b"\0" * 16, dtype=np.uint8)
        self.moff = np.array(moff, dtype=np.uint32)
        self.ooff = np.array(ooff, dtype=np.uint32)
        self.c = A.csq_bgzf_in()
        self.c.data = self.data.ctypes.data
        self.c.bytes = len(data)
        self.c.member_off = self.moff.ctypes.data
        self.c.text_off = self.ooff.ctypes.data
        self.c.n_members = len(moff) - 1
        self.c.skip_lines = skip_lines
        self.c.append_newline = int(append_newline)
        self.text_bytes = ooff[-1]


class TextReader:
    """csq_text_reader: batches of raw FASTQ text cut at record boundaries (host side of the file driver).
    flags = PLAN_FASTA: FASTA files, batches of whole FASTA records."""

    def __init__(self, path1, path2=None, flags: int = 0):
        self._h = C.c_void_p()
        check(lib().csq_text_reader_open_flags(os.fsencode(path1), os.fsencode(path2) if path2 else None, flags,
                                               C.byref(self._h)))

    def next(self, max_reads: int, buffer: int = 0):
        """-> (n_reads, [bytes per mate], first_record); n_reads == 0 at the end of the input."""
        b = A.csq_batch_text()
        check(lib().csq_text_reader_next(self._h, buffer, max_reads, C.byref(b)))
        texts = [C.string_at(b.mate[m].text, b.mate[m].bytes) if b.mate[m].bytes else b"" for m in range(b.n_mates)]
        return b.n_reads, texts, b.first_record

    def close(self):
        if self._h:
            lib().csq_text_reader_close(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def format_fastq(batch: A.csq_batch_in, mate: int, out=None):
    """FASTQ text of one mate of a SoA batch (``csq_format_fastq``). -> numpy uint8 array (or fills `out`)."""
    need = C.c_uint64()
    mi = batch.mate[mate]
    if out is None:
        # size: names + 2 * bases + 6 per record
        noff = np.ctypeslib.as_array(C.cast(mi.name_off, C.POINTER(C.c_uint32)), (batch.n_reads + 1,))
        slen = np.ctypeslib.as_array(C.cast(mi.seq_len, C.POINTER(C.c_uint32)), (max(batch.n_reads, 1),))[: batch.n_reads]
        size = int(noff[batch.n_reads] - noff[0]) + 2 * int(slen.sum(dtype=np.uint64)) + 6 * batch.n_reads
        out = np.empty(max(size, 1), dtype=np.uint8)
    ptr, cap = (out.data_ptr(), out.numel()) if hasattr(out, "data_ptr") else (out.ctypes.data, out.size)
    check(lib().csq_format_fastq(C.byref(mi), batch.n_reads, ptr, cap, C.byref(need)))
    return out[: need.value]


def locate_batch(op, mate_in: A.csq_mate_in, n_reads: int, device: int = 0, flags: int = 0):
    """Aligner.locate for a batch of reads on the GPU (``csq_locate_batch``)."""
    cop = op.to_c() if hasattr(op, "to_c") else op
    out = np.zeros(max(n_reads, 1), dtype=MATCH_DTYPE)
    check(lib().csq_locate_batch(device, C.byref(cop), C.byref(mate_in), n_reads, flags, out.ctypes.data))
    return out[:n_reads]


def synth_batch(config: int, n_reads: int, first_index: int = 0, buffer: int = 0, seed: int | None = None,
                read_len: int | None = None, paired: bool | None = None) -> A.csq_batch_in:
    """BASELINE.json configs 2-5 as packed SoA batches in pinned host memory (``csq_synth_batch``)."""
    defaults = {2: (20240419, 150, True), 3: (20240420, 150, True), 4: (20240421, 75, False), 5: (20240419, 150, True)}
    dseed, dlen, dpaired = defaults[config]
    cfg = A.csq_synth(dseed if seed is None else seed, dlen if read_len is None else read_len,
                      int(dpaired if paired is None else paired), 2 if config == 5 else config)
    b = A.csq_batch_in()
    check_plain(lib().csq_synth_batch(C.byref(cfg), first_index, n_reads, buffer, C.byref(b)))
    return b


def check_plain(rc: int):
    if rc != 0:
        raise NativeError(rc, "synthetic generator failed")


def bind_host_to_device(device: int = 0) -> int:
    """Keep this thread, the threads it starts and the memory it pins on the GPU's NUMA node. -> node or -1."""
    node = C.c_int(-1)
    check(lib().csq_bind_host_to_device(device, C.byref(node)))
    return node.value


def unbind_host() -> None:
    check(lib().csq_unbind_host())


def int_peak(device: int = 0):
    a, b = C.c_double(), C.c_double()
    check(lib().csq_int_peak(device, C.byref(a), C.byref(b)))
    return a.value, b.value


def gz_deflate_host(text: bytes) -> bytes:
    """The device gzip writer's algorithm on the host (``csq_gz_deflate_host``): text -> concatenated BGZF members."""
    src = np.frombuffer(text, dtype=np.uint8) if len(text) else np.zeros(1, dtype=np.uint8)
    out = np.empty(len(text) + (len(text) // 32000 + 2) * 64 + 64, dtype=np.uint8)
    n = C.c_uint64()
    check(lib().csq_gz_deflate_host(src.ctypes.data, len(text), out.ctypes.data, out.size, C.byref(n)))
    return out[: n.value].tobytes()


def pinflate(data: bytes, capacity: int, threads: int = 4, span_bytes: int = 0) -> bytes:
    """An ordinary gzip file in memory through the parallel decoder (``csq_pinflate_mem``)."""
    src = np.frombuffer(bytes(data) + b"\0" * 16, dtype=np.uint8)
    out = np.empty(max(capacity, 1), dtype=np.uint8)
    n = C.c_uint64(0)
    check(lib().csq_pinflate_mem(src.ctypes.data, len(data), out.ctypes.data, capacity, threads, span_bytes, C.byref(n)))
    return out[: n.value].tobytes()


def _gz_stream(call, data: bytes, capacity: int, span_bytes: int, round_bytes: int, chain: bool):
    src = np.frombuffer(bytes(data) + b"\0" * 16, dtype=np.uint8)
    out = np.empty(max(capacity, 1), dtype=np.uint8)
    n = C.c_uint64(0)
    check(call(src.ctypes.data, len(data), out.ctypes.data, capacity, span_bytes, round_bytes, C.byref(n)))
    text = out[: n.value].tobytes()
    if not chain:
        return text
    k = lib().csq_gz_stream_chain(None, 0)
    arr = np.zeros(3 * max(k, 1), dtype=np.uint64)
    lib().csq_gz_stream_chain(arr.ctypes.data_as(C.POINTER(C.c_uint64)), k)
    return text, [tuple(int(v) for v in arr[3 * i: 3 * i + 3]) for i in range(k)]


def gz_stream_inflate(data: bytes, capacity: int, device: int = 0, span_bytes: int = 0, round_bytes: int = 0,
                      chain: bool = False):
    """An ordinary gzip file in memory through the device decoder (``csq_gz_stream_inflate``).  chain=True also returns
    the decode chain: (start bit, end bit, symbols) of every span in file order."""
    def call(*a):
        return lib().csq_gz_stream_inflate(device, *a)
    return _gz_stream(call, data, capacity, span_bytes, round_bytes, chain)


def gz_stream_inflate_host(data: bytes, capacity: int, span_bytes: int = 0, round_bytes: int = 0, chain: bool = False):
    """The device decoder's host twin (``csq_gz_stream_inflate_host``), as gz_stream_inflate."""
    return _gz_stream(lib().csq_gz_stream_inflate_host, data, capacity, span_bytes, round_bytes, chain)


def gz_inflate_host(data: bytes, capacity: int):
    """The device gzip reader's decoder on the host (``csq_gz_inflate_host``): BGZF members -> (text, line ends)."""
    src = np.frombuffer(data, dtype=np.uint8) if len(data) else np.zeros(1, dtype=np.uint8)
    out = np.empty(max(capacity, 1), dtype=np.uint8)
    n, lines = C.c_uint64(), C.c_uint64()
    check(lib().csq_gz_inflate_host(src.ctypes.data, len(data), out.ctypes.data, capacity, C.byref(n), C.byref(lines)))
    return out[: n.value].tobytes(), lines.value


def pcie_peak(device: int, bytes_h2d: int, bytes_d2h: int, reps: int = 4, mode: int = 2):
    """Measured pinned-memory copy rates (GB/s): mode 0 host->device, 1 device->host, 2 both at once."""
    a, b = C.c_double(), C.c_double()
    check(lib().csq_pcie_peak(device, bytes_h2d, bytes_d2h, reps, mode, C.byref(a), C.byref(b)))
    return a.value, b.value


def run_files(program, inputs, outputs, gpus: int = 1, threads: int = 1, batch_reads: int = 0, flags: int = 0,
              gzip_level: int = 0):
    """Whole-file run (``csq_run_files``). outputs = {"trimmed": [p1, p2], "short": [...], "untrimmed": [...]}."""
    L = lib()
    if not hasattr(L, "csq_run_files"):
        raise NativeError(A.ERR_INVALID, "library was built without the file pipeline")
    ops1, n1 = program.c_ops(0)
    ops2, n2 = program.c_ops(1)
    flt = program.filters.to_c()
    f = A.csq_files()
    for i, p in enumerate(inputs):
        f.in_[i] = os.fsencode(p)
    for d, key in enumerate(("trimmed", "short", "untrimmed")):
        paths = outputs.get(key) or []
        for m, p in enumerate(paths):
            if p is not None:
                f.out[d][m] = os.fsencode(p)
    f.batch_reads = batch_reads
    f.gzip_level = gzip_level
    f.n_threads = threads
    f.n_devices = gpus
    f.swap_sink = int(program.swap_sink)
    counters, timing = A.csq_counters(), A.csq_timing()
    check(L.csq_run_files(ops1, n1, ops2, n2 if program.paired else 0, C.byref(flt), flags, C.byref(f), C.byref(counters), C.byref(timing)))
    return counters, timing
