// Internal definitions shared by the CUDA kernels (kernels.cu) and the host side of the
// C ABI (plan.cu). Nothing here is part of the public boundary (include/cutseq_b200.h).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/cutseq_b200.h"

// ---- limits of the packed DP word (see kernels.cu, "DP cell encoding") -------------------
// origin is stored biased by 128 in 10 bits  -> read length <= 895
// cost is stored in 10 bits                  -> m + n <= 1023
#define CSQ_FAST_MAX_READ 895
#define CSQ_MAX_PRE 12 /* scalar ops executed in front of one ALIGN op */
#define CSQ_PF_BINS 5   /* prefilter survivor lists: classes of DP columns left for the exact pass (0..2 long to medium, 4 short)
                           and 3 = reads that hold an error-free copy of the adapter (the exact pass stops there) */

// Scalar (O(1)) ops that sit between alignments: CUT, COND_CUT, RENAME(capture).
struct DevOp {
    int32_t kind;    // csq_op_kind
    int32_t length;  // CUT / COND_CUT
    int32_t fmin;    // COND_CUT
    uint32_t rename_parts;
};

// Per-mate, per-read state carried between kernels: the read is original[a:b].
// Slices of the original read are packed as (offset << 16 | length); length 0 == None/"".
struct __align__(16) ReadState {
    uint16_t a, b;
    uint32_t matched;  // bit31: any AdapterCutter matched (bool(info.matches)); bits 0..30: adapter_id set
    uint32_t cp, cs;   // info.cut_prefix / info.cut_suffix as last assigned
    uint32_t ren_cp, ren_cs;  // ... as they were when the RENAME op ran
    uint16_t id_start, id_end;  // Renamer.parse_name() id within the (suffix-stripped) header
    uint32_t qtrim;    // bases removed by QTRIM (statistics)
};
static_assert(sizeof(ReadState) == 32, "ReadState must stay 32 bytes");

struct MateDev {  // device pointers of one mate of one slot
    // record i: bases seq[seq_off[i] .. +seq_len[i]), qualities qual[qual_off[i] .. +seq_len[i]),
    // header name[name_off[i] .. name_end[i]).
    // SoA batches: qual_off == seq_off and name_end == name_off + 1 (the same arrays);
    // text batches: seq == qual == name == the FASTQ text, all five arrays written by k_records (parse.cu).
    const uint8_t* seq;
    const uint8_t* qual;
    const uint32_t* seq_off;
    const uint32_t* qual_off;
    const uint32_t* seq_len;
    const uint8_t* name;
    const uint32_t* name_off;
    const uint32_t* name_end;
    ReadState* state;
};

struct ParseParams {  // FASTQ text of one mate -> record index (parse.cu)
    const uint8_t* text;
    uint64_t bytes;
    uint32_t n;             // records the host counted (4 n line ends)
    uint32_t* nl;           // four-kernel form: [4 n] byte offsets of the line ends, 16-byte aligned; one-pass form: [n] scratch
    uint32_t* nl_total;     // [1] line ends found
    uint32_t *seq_off, *qual_off, *seq_len, *name_off, *name_end;
    unsigned long long* perr;  // smallest (record << 3 | kind) of a malformed record, ~0 when clean
    uint32_t* any_cr;          // [1] set by k_nl_count when the text holds a '\r' anywhere (CRLF files)
    // BGZF batches: the text is what a run of whole members inflates to, the batch's records sit somewhere inside -
    // `skip` line ends lie in front of the first record (its start is left in *first_off by k_nl_index), lines behind
    // the 4 n of the batch are ignored
    uint32_t skip;
    uint32_t* first_off;       // [1] byte offset of the first record (0 when skip == 0)
};

struct FastaParams {  // FASTA text of one mate -> record index (parse.cu, CSQ_PLAN_FASTA)
    ParseParams p;           // p.nl: [n] offsets of the record starts; p.nl_total: record starts found
    uint8_t* pool;           // wrapped sequences, joined: text + pool0 (one buffer, so that seq_off reaches both)
    uint32_t pool0;
    uint32_t* pad_len;       // [n], 16-byte aligned: padded lengths of the wrapped records, scanned into pool offsets
    uint32_t* pool_total;    // [1]
    uint32_t qual0;          // qual_off of every record: into the constant buffer of 'I' bytes
};
#define CSQ_FASTA_QUAL_BYTES 1024  /* the 'I' buffer: qual_off = 64, then CSQ_MAX_READ_LEN bytes and padding */

struct AlignParams {
    MateDev md;
    csq_match* matches;    // nullable: per-read record of this ALIGN op
    // nullable: prefilter survivors. CSQ_PF_BINS lists of read indices, list b at list[b * n ..), followed by the
    // uint16 first-DP-column of every entry in the same layout (0xFFFF: the aligner's own min_n)
    const uint32_t* list;
    const uint32_t* list_count;  // with list: entries per list (device side)
    uint32_t n;            // reads in the batch
    int32_t first;         // 1: state is initialised here (first segment of the program)
    int32_t count_cells;   // 1: add the nominal DP cells of this launch to the statistics
    int32_t n_pre;
    DevOp pre[CSQ_MAX_PRE];
    // the adapter
    int32_t m, flags, reversed, trim_front, min_overlap, k, adapter_bit, homopolymer;
    uint32_t one;          // == 1: multiplier of the adds that are to run as IMAD on the FMA pipe (opaque to ptxas)
    int32_t exact_stop;    // 1: leave the column loop at an error-free full match, as Aligner.locate does ("exact match, stop early")
    uint8_t thr[CSQ_MAX_ADAPTER + 1];  // thr[L] = floor(L * max_error_rate) with host doubles
    uint32_t peq[4][4];                // [A,C,G,T][word]: bit i-1 set <=> adapter[i-1] == letter
    uint8_t letter;                    // homopolymer base
    unsigned long long* counters;      // csq_counters on the device
    int32_t counter_index;             // word index of with_adapters[mate][op] inside csq_counters
    int32_t adjacent_index;            // word index of adjacent_bases[mate] (first ALIGN op of a mate, 3' kinds), else -1
};

struct FinishParams {
    MateDev md;
    uint32_t n;
    int32_t first;  // program without any ALIGN op: initialise state here
    int32_t n_post;
    DevOp post[CSQ_MAX_PRE];
    int32_t has_qtrim, cutoff_front, cutoff_back, qbase;
    int32_t n_suffix;
    int32_t suffix_len[4];
    char suffix[4][CSQ_MAX_SUFFIX];
    int32_t mate;
    int32_t has_rename;  // 0: the header is written unchanged (after suffix stripping)
    unsigned long long* counters;
    // text batches: the '@' / '+' line starts are checked here, where the header and the end of the bases are
    // fetched anyway (k_records then needs no look at the text); same (record << 3 | kind) key as ParseParams.perr
    unsigned long long* perr;
};

#define CSQ_PAIR_BLOCK 256  // pairs per CTA in the pair/emit kernels (scan granule)

struct PairParams {
    MateDev md[2];
    uint32_t n;
    int32_t n_mates;
    int32_t min_length, untrimmed_enabled;
    uint32_t required[2];
    uint32_t rename_parts;  // of the RENAME op (same on both mates)
    int32_t check_ids;      // paired RENAME present: PairedEndRenamer's record_names_match on the suffix-stripped headers
                            // (dnaio's paired reader check on the raw headers applies to every paired batch)
    int32_t revcomp;        // single-end REVCOMP op present
    uint8_t* dest;          // [n]
    uint32_t* block_tot;    // [nblk][8]: bytes per (dest,mate) stream (6 used)
    uint32_t* block_cnt;    // [nblk][4]: records per dest
    unsigned long long* counters;
    int32_t* error_flag;
};

struct EmitParams {
    PairParams pp;
    const unsigned long long* block_off;  // [nblk][8] exclusive byte offsets per stream
    uint8_t* out[CSQ_N_DEST][2];
};

// ---- device gzip writer (gz_deflate.cu) ----
#define GZ_THREADS 256
#define GZ_RUN 127                       /* literals per thread; odd, so that the runs of a warp spread over the banks */
#define GZ_PIECE (GZ_THREADS * GZ_RUN)   /* 32512 input bytes per member (a multiple of 16)                            */
#define GZ_SLOT 32576                    /* bytes reserved per member before packing (stored piece + framing, 16 | it) */
#define GZ_CODE_STRIDE 260               /* words per stream in GzParams.codes                                         */
#define GZ_HDR_STRIDE 100                /* words per stream in GzParams.hdr: header bits, then their number           */

struct GzParams {  // the six output streams (destination x mate) of one batch
    const uint8_t* text[CSQ_N_DEST * 2];  // emitted FASTQ text
    uint64_t bytes[CSQ_N_DEST * 2];
    uint32_t first_member[CSQ_N_DEST * 2 + 1];  // members in front of every stream (ceil(bytes / GZ_PIECE) each)
    uint32_t* hist;        // [6][256]
    uint32_t* codes;       // [6][GZ_CODE_STRIDE]  code | length << 16 of literal / end-of-block
    uint32_t* hdr;         // [6][GZ_HDR_STRIDE]
    const uint32_t* crc_tab;  // [256]
    const uint32_t* crc_pow;  // [GZ_THREADS]  x^(8 * GZ_RUN * k) mod P
    uint8_t* slots;        // [members][GZ_SLOT]
    uint32_t* msize;       // [members]
    unsigned long long* moff;    // [members] offset inside the packed stream
    unsigned long long* totals;  // [6] packed bytes per stream
    uint8_t* packed[CSQ_N_DEST * 2];
};
cudaError_t csq_launch_gz(const GzParams& p, uint32_t n_members, cudaStream_t stream);
void csq_gz_host_tables(uint32_t* crc_tab, uint32_t* crc_pow);

// ---- device gzip reader (gz_inflate.cu) ----
struct InflateParams {
    const uint8_t* comp;     // the compressed members, back to back as in the file (readable 16 bytes past the end)
    const uint32_t* moff;    // [n + 1] byte offset of every member in comp
    const uint32_t* ooff;    // [n + 1] byte offset of every member's text in out (prefix sums of ISIZE)
    uint32_t n_members;
    uint8_t* out;
    uint32_t* lines;         // nullable: '\n' per member
    int32_t* status;         // atomicMin of (error kind + 16 * member index); INT_MAX when clean
    const uint32_t* crc_tables;  // tables of csq_gz_crc_check_tables: the CRC-32 of every member is verified (error kind 7)
};
cudaError_t csq_launch_inflate(const InflateParams& p, cudaStream_t stream);
void csq_gz_crc_check_tables(uint32_t* t /*[768]*/);

// word indices inside csq_counters viewed as uint64[]
enum {
    CNT_N = 0, CNT_TOTAL_BP = 1, CNT_WRITTEN = 3, CNT_WRITTEN_BP = 4, CNT_TOO_SHORT = 6, CNT_UNTRIMMED = 7,
    CNT_QTRIM_BP = 8, CNT_WITH_ADAPTERS = 10, CNT_DP_CELLS = 10 + 2 * CSQ_MAX_OPS, CNT_ADJACENT = 10 + 4 * CSQ_MAX_OPS
};

// launchers implemented in kernels.cu (all asynchronous on `stream`)
cudaError_t csq_launch_align(const AlignParams& p, uint32_t n_items, cudaStream_t stream);
cudaError_t csq_launch_tail(const FinishParams& f1, const FinishParams& f2, const PairParams& p, bool fasta, cudaStream_t stream);  // tail.cu
cudaError_t csq_launch_scan(uint32_t nblk, const uint32_t* block_tot, const uint32_t* block_cnt,
                            unsigned long long* block_off, unsigned long long* totals, cudaStream_t stream);
// fasta: ">name\nseq\n" records (CSQ_PLAN_FASTA)
cudaError_t csq_launch_emit(const EmitParams& p, bool fasta, cudaStream_t stream);  // kernels.cu: direct, 16 lanes per record
cudaError_t csq_launch_emit_stage(const EmitParams& p, bool fasta, cudaStream_t stream); // emit_stage.cu: staged through shared memory (default)
cudaError_t csq_launch_parse(const ParseParams& p, void* tile_buf, uint16_t* masks, cudaStream_t stream);
uint32_t csq_parse_tiles(uint64_t bytes);
cudaError_t csq_launch_parse_fasta(const FastaParams& f, void* tile_buf, uint16_t* masks, cudaStream_t stream);
uint32_t csq_parse_fasta_launches(uint64_t bytes, uint32_t n);
cudaError_t csq_launch_prefilter(const AlignParams& p, uint32_t* list, uint32_t* list_count, cudaStream_t stream);
bool csq_align_has_exact_kernel(int m);
cudaError_t csq_launch_int_peak(int variant, int iters, unsigned int* sink, int blocks, int threads, cudaStream_t stream);
