"""ctypes mirror of ``include/cutseq_b200.h`` (struct layouts and constants only)."""

from __future__ import annotations

import ctypes as C

ABI_VERSION = 4

CSQ_MAX_ADAPTER = 128
CSQ_MAX_READ_LEN = 895
CSQ_MAX_OPS = 32
CSQ_MAX_SUFFIX = 8
CSQ_N_DEST = 3
CSQ_N_SLOTS = 8

# csq_status
OK, ERR_INVALID, ERR_NO_DEVICE, ERR_CUDA, ERR_NOMEM = 0, -1, -2, -3, -4
ERR_CAPACITY, ERR_FORMAT, ERR_IO, ERR_PAIRING, ERR_LIMIT = -5, -6, -7, -8, -9

# csq_op_kind
OP_STRIP_SUFFIX, OP_ALIGN, OP_CUT, OP_COND_CUT, OP_RENAME, OP_QTRIM, OP_REVCOMP = 1, 2, 3, 4, 5, 6, 7
OP_NAMES = {1: "STRIP_SUFFIX", 2: "ALIGN", 3: "CUT", 4: "COND_CUT", 5: "RENAME", 6: "QTRIM", 7: "REVCOMP"}

# csq_adapter_kind
AD_BACK, AD_BACK_ANYWHERE, AD_RIGHTMOST_FRONT, AD_PREFIX, AD_SUFFIX, AD_NI_FRONT, AD_NI_BACK, AD_FRONT = range(1, 9)
AD_NAMES = {
    AD_BACK: "BackAdapter",
    AD_BACK_ANYWHERE: "BackAdapter(force_anywhere)",
    AD_RIGHTMOST_FRONT: "RightmostFrontAdapter",
    AD_PREFIX: "PrefixAdapter",
    AD_SUFFIX: "SuffixAdapter",
    AD_NI_FRONT: "NonInternalFrontAdapter",
    AD_NI_BACK: "NonInternalBackAdapter",
    AD_FRONT: "FrontAdapter",
}

REN_OWN_PREFIX, REN_OWN_SUFFIX, REN_R1_PREFIX, REN_R2_PREFIX = 1, 2, 4, 8

DEST_TRIMMED, DEST_SHORT, DEST_UNTRIMMED = 0, 1, 2

PLAN_KEEP_MATCHES = 1
PLAN_NO_PREFILTER = 2
PLAN_ONE_STREAM = 64
PLAN_EMIT_G16 = 256
PLAN_NO_EXACT_STOP = 1024
PLAN_GZIP_OUT = 4096
PLAN_FASTA = 8192


class csq_op(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("adapter_kind", C.c_int32),
        ("adapter_len", C.c_int32),
        ("min_overlap", C.c_int32),
        ("adapter_id", C.c_int32),
        ("max_error_rate", C.c_double),
        ("adapter", C.c_char * CSQ_MAX_ADAPTER),
        ("length", C.c_int32),
        ("force_trim_min_length", C.c_int32),
        ("suffix_len", C.c_int32),
        ("suffix", C.c_char * CSQ_MAX_SUFFIX),
        ("rename_parts", C.c_uint32),
        ("cutoff_front", C.c_int32),
        ("cutoff_back", C.c_int32),
        ("quality_base", C.c_int32),
    ]


class csq_filters(C.Structure):
    _fields_ = [
        ("min_length", C.c_int32),
        ("untrimmed_enabled", C.c_int32),
        ("required_r1", C.c_uint32),
        ("required_r2", C.c_uint32),
    ]


class csq_mate_in(C.Structure):
    _fields_ = [
        ("seq", C.c_void_p),
        ("qual", C.c_void_p),
        ("seq_off", C.c_void_p),
        ("seq_len", C.c_void_p),
        ("seq_bytes", C.c_uint64),
        ("name", C.c_void_p),
        ("name_off", C.c_void_p),
        ("name_bytes", C.c_uint64),
    ]


class csq_batch_in(C.Structure):
    _fields_ = [("n_reads", C.c_uint32), ("n_mates", C.c_uint32), ("mate", csq_mate_in * 2)]


class csq_text_in(C.Structure):
    _fields_ = [("text", C.c_void_p), ("bytes", C.c_uint64)]


class csq_batch_text(C.Structure):
    _fields_ = [("n_reads", C.c_uint32), ("n_mates", C.c_uint32), ("first_record", C.c_uint64), ("mate", csq_text_in * 2)]


class csq_bgzf_in(C.Structure):
    _fields_ = [("data", C.c_void_p), ("bytes", C.c_uint64), ("member_off", C.c_void_p), ("text_off", C.c_void_p),
                ("n_members", C.c_uint32), ("skip_lines", C.c_uint32), ("append_newline", C.c_uint32), ("reserved", C.c_uint32)]


class csq_batch_bgzf(C.Structure):
    _fields_ = [("n_reads", C.c_uint32), ("n_mates", C.c_uint32), ("first_record", C.c_uint64), ("mate", csq_bgzf_in * 2)]


class csq_text_out(C.Structure):
    _fields_ = [("data", C.c_void_p), ("capacity", C.c_uint64), ("bytes", C.c_uint64), ("records", C.c_uint64)]


class csq_batch_out(C.Structure):
    _fields_ = [("text", (csq_text_out * 2) * CSQ_N_DEST)]


class csq_match(C.Structure):
    _fields_ = [
        ("found", C.c_int16),
        ("ref_start", C.c_int16),
        ("ref_stop", C.c_int16),
        ("query_start", C.c_int16),
        ("query_stop", C.c_int16),
        ("score", C.c_int16),
        ("errors", C.c_int16),
        ("reserved", C.c_int16),
    ]


class csq_read_result(C.Structure):
    _fields_ = [("start", C.c_uint32), ("stop", C.c_uint32), ("dest", C.c_uint32), ("matched", C.c_uint32)]


class csq_counters(C.Structure):
    _fields_ = [
        ("n", C.c_uint64),
        ("total_bp", C.c_uint64 * 2),
        ("written", C.c_uint64),
        ("written_bp", C.c_uint64 * 2),
        ("too_short", C.c_uint64),
        ("untrimmed", C.c_uint64),
        ("quality_trimmed_bp", C.c_uint64 * 2),
        ("with_adapters", (C.c_uint64 * CSQ_MAX_OPS) * 2),
        ("dp_cells", (C.c_uint64 * CSQ_MAX_OPS) * 2),
        ("adjacent_bases", (C.c_uint64 * 6) * 2),
    ]


class csq_files(C.Structure):
    _fields_ = [
        ("in_", C.c_char_p * 2),
        ("out", (C.c_char_p * 2) * CSQ_N_DEST),
        ("batch_reads", C.c_uint32),
        ("gzip_level", C.c_int32),
        ("n_threads", C.c_int32),
        ("n_devices", C.c_int32),
        ("devices", C.POINTER(C.c_int32)),
        ("swap_sink", C.c_int32),
    ]


class csq_timing(C.Structure):
    _fields_ = [
        ("read_inflate", C.c_double),
        ("parse", C.c_double),
        ("h2d_kernels_d2h", C.c_double),
        ("kernels", C.c_double),
        ("write_deflate", C.c_double),
        ("total", C.c_double),
    ]


class csq_synth(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("read_len", C.c_uint32), ("paired", C.c_uint32), ("config", C.c_uint32)]
