/*
 * cutseq_b200.h - C ABI of libcutseq_b200.so: the drop-in boundary for cutseq's
 * per-read trimming path (SURVEY.md section 8(b)).
 *
 * What it replaces in the reference (y9c/cutseq 0.0.68, files under cutseq/):
 *   - the cutadapt modifier/step chain that run.py:326-471 (single-end) and
 *     run.py:533-792 (paired-end) assemble and hand to
 *     runner.run(pipeline, Progress(), outfiles) at run.py:472-473 / 793-794;
 *   - cutseq's own modifiers/predicates run.py:78-110 (IsUntrimmedAny),
 *     run.py:113-161 (ConditionalCutter), run.py:164-187 (ReverseComplementConverter).
 * The arithmetic itself lives in the un-vendored dependency cutadapt~=5.0
 * (reference pyproject.toml:17): Aligner.locate, quality_trim_index, the
 * *Adapter classes, UnconditionalCutter/SuffixRemover/Renamer, TooShort and the
 * paired filters. A call here is batch-granular: one call processes a batch of
 * reads through the whole chain ("op program") on one B200.
 *
 * Conventions
 *   - every function returns 0 on success or a negative csq_status; the text of the
 *     last error of the calling thread is available from csq_last_error();
 *   - nothing throws across this boundary; no torch / C++ types in any signature;
 *   - the library owns all device memory and streams; the caller owns host buffers
 *     and must keep them alive until csq_wait() returns for the slot they were
 *     submitted on;
 *   - a plan is bound to one CUDA device and is used from one host thread at a time;
 *   - there is NO CPU fallback: without a usable CUDA device every compute entry
 *     point fails with CSQ_ERR_NO_DEVICE.
 */
#ifndef CUTSEQ_B200_H
#define CUTSEQ_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CSQ_ABI_VERSION 4

typedef enum csq_status {
    CSQ_OK = 0,
    CSQ_ERR_INVALID = -1,     /* bad argument / malformed program                 */
    CSQ_ERR_NO_DEVICE = -2,   /* no CUDA device, or not an sm_100 part            */
    CSQ_ERR_CUDA = -3,        /* a CUDA runtime call failed (see csq_last_error)  */
    CSQ_ERR_NOMEM = -4,       /* host or device allocation failed                 */
    CSQ_ERR_CAPACITY = -5,    /* an output buffer of the caller is too small      */
    CSQ_ERR_FORMAT = -6,      /* malformed FASTQ input                            */
    CSQ_ERR_IO = -7,          /* open/read/write/inflate/deflate failure          */
    CSQ_ERR_PAIRING = -8,     /* mate ids differ (PairedEndRenamer's ValueError)  */
    CSQ_ERR_LIMIT = -9        /* read or adapter longer than the supported limit  */
} csq_status;

/* Limits of this build. */
#define CSQ_MAX_ADAPTER 128      /* adapter length m                             */
#define CSQ_MAX_READ_LEN 895     /* bases per read (10-bit origin field of the DP word) */
#define CSQ_MAX_OPS 32           /* ops per mate program                         */
#define CSQ_MAX_SUFFIX 8         /* bytes of a STRIP_SUFFIX text                 */

/* ---------------------------------------------------------------------------
 * Op program: one entry per modifier that run.py puts in `modifiers`, in order.
 * ------------------------------------------------------------------------- */
typedef enum csq_op_kind {
    CSQ_OP_STRIP_SUFFIX = 1, /* cutadapt SuffixRemover(text)            run.py:330, 537-542 */
    CSQ_OP_ALIGN = 2,        /* cutadapt AdapterCutter([adapter], times=1, action="trim")
                                run.py:332-368, 544-613, 388-404, 673-707                  */
    CSQ_OP_CUT = 3,          /* cutadapt UnconditionalCutter(length)    run.py:374-386, 599-669 */
    CSQ_OP_COND_CUT = 4,     /* cutseq ConditionalCutter(length, fmin)  run.py:113-161     */
    CSQ_OP_RENAME = 5,       /* cutadapt Renamer / PairedEndRenamer     run.py:377-380, 642-645 */
    CSQ_OP_QTRIM = 6,        /* cutadapt QualityTrimmer(front, back)    run.py:415-417, 718-723 */
    CSQ_OP_REVCOMP = 7       /* cutseq ReverseComplementConverter       run.py:164-187, 420-426 */
} csq_op_kind;

/* cutadapt.align.EndSkip bits of the Aligner ("flags" of Aligner.__cinit__). */
#define CSQ_REFERENCE_START 1u /* a prefix of the adapter may be skipped at no cost */
#define CSQ_QUERY_START 2u     /* a prefix of the read may be skipped at no cost    */
#define CSQ_REFERENCE_END 4u   /* a suffix of the adapter may be skipped            */
#define CSQ_QUERY_STOP 8u      /* a suffix of the read may be skipped               */

/* Which cutadapt adapter class an ALIGN op stands for (decides aligner flags,
 * the reversed-alignment trick and which side of the match is removed). */
typedef enum csq_adapter_kind {
    CSQ_AD_BACK = 1,            /* BackAdapter: flags 14, keep read[:query_start]           */
    CSQ_AD_BACK_ANYWHERE = 2,   /* BackAdapter(force_anywhere=True): flags 15, same trim    */
    CSQ_AD_RIGHTMOST_FRONT = 3, /* RightmostFrontAdapter: reversed adapter vs reversed read,
                                   flags 14, coordinates mapped back, keep read[query_stop:] */
    CSQ_AD_PREFIX = 4,          /* PrefixAdapter: flags 8, min_overlap=m, keep read[query_stop:] */
    CSQ_AD_SUFFIX = 5,          /* SuffixAdapter: flags 2, min_overlap=m, keep read[:query_start] */
    CSQ_AD_NI_FRONT = 6,        /* NonInternalFrontAdapter: flags 9, keep read[query_stop:]  */
    CSQ_AD_NI_BACK = 7,         /* NonInternalBackAdapter: flags 6, keep read[:query_start]  */
    CSQ_AD_FRONT = 8            /* FrontAdapter: flags 11 (not used by run.py; for tests)    */
} csq_adapter_kind;

/* RENAME template parts appended after "{id}_" (0 => template is just "{id}"). */
#define CSQ_REN_OWN_PREFIX 1u /* {cut_prefix}      (single-end template run.py:378)  */
#define CSQ_REN_OWN_SUFFIX 2u /* {cut_suffix}                                        */
#define CSQ_REN_R1_PREFIX 4u  /* {r1.cut_prefix}   (paired template run.py:643)      */
#define CSQ_REN_R2_PREFIX 8u  /* {r2.cut_prefix}                                     */

typedef struct csq_op {
    int32_t kind;                       /* csq_op_kind                                         */
    /* ALIGN */
    int32_t adapter_kind;               /* csq_adapter_kind                                    */
    int32_t adapter_len;                /* m, 1..CSQ_MAX_ADAPTER                               */
    int32_t min_overlap;                /* as passed to the adapter class (clamped to m inside;
                                           PREFIX/SUFFIX force m like cutadapt)                */
    int32_t adapter_id;                 /* 0..30: bit recorded in the mate's "matched adapters"
                                           set when this op finds a match; -1 = not tracked    */
    double max_error_rate;              /* e.g. 0.2 / 0.15 (values < 1: a rate)                */
    char adapter[CSQ_MAX_ADAPTER];      /* ACGT upper-case, not NUL terminated                 */
    /* CUT / COND_CUT: >0 removes from the 5' end, <0 from the 3' end */
    int32_t length;
    int32_t force_trim_min_length;      /* COND_CUT only                                       */
    /* STRIP_SUFFIX */
    int32_t suffix_len;
    char suffix[CSQ_MAX_SUFFIX];
    /* RENAME */
    uint32_t rename_parts;              /* CSQ_REN_* bits                                      */
    /* QTRIM */
    int32_t cutoff_front, cutoff_back, quality_base;
} csq_op;

/* Filters and sink that run.py puts in `steps` (run.py:446-471, 763-792). */
typedef struct csq_filters {
    int32_t min_length;          /* TooShort(min_length); pair is "short" if either mate is   */
    int32_t untrimmed_enabled;   /* second filter present (IsUntrimmedAny)                     */
    uint32_t required_r1;        /* adapter_id bits that must be present on mate 1             */
    uint32_t required_r2;        /* ... on mate 2 (0 for single-end)                           */
} csq_filters;

typedef enum csq_dest { CSQ_DEST_TRIMMED = 0, CSQ_DEST_SHORT = 1, CSQ_DEST_UNTRIMMED = 2, CSQ_N_DEST = 3 } csq_dest;

/* ---------------------------------------------------------------------------
 * Batch in: packed struct-of-arrays, one per mate. Record i has seq_len[i] bases at
 * seq + seq_off[i] and its qualities at qual + seq_off[i]; seq_off[i] is a multiple
 * of 16 and the pools are padded so that [seq_off[i], seq_off[i] + round_up(len,16))
 * is readable. name holds header lines without '@' and without line ends;
 * record i is name[name_off[i] : name_off[i+1]].
 * ------------------------------------------------------------------------- */
typedef struct csq_mate_in {
    const uint8_t* seq;
    const uint8_t* qual;
    const uint32_t* seq_off;   /* n_reads entries */
    const uint32_t* seq_len;   /* n_reads entries */
    uint64_t seq_bytes;        /* size of seq / qual pools (multiple of 16) */
    const uint8_t* name;
    const uint32_t* name_off;  /* n_reads + 1 entries */
    uint64_t name_bytes;
} csq_mate_in;

typedef struct csq_batch_in {
    uint32_t n_reads;          /* reads (single-end) or pairs (paired-end) */
    uint32_t n_mates;          /* 1 or 2 */
    csq_mate_in mate[2];
} csq_batch_in;

/* Batch in, text form: the FASTQ bytes of the batch as they stand in the file (after
 * decompression), whole records only - n_reads records of 4 lines per mate, the last line
 * ended by '\n'. The device builds the record index itself (dnaio's checks: '@' and '+'
 * line starts, equal sequence and quality lengths, "\r\n" line ends accepted); a malformed
 * batch makes csq_wait fail with CSQ_ERR_FORMAT. This is what the whole-file driver uses:
 * the host only cuts the byte stream at record boundaries (csq_count_newlines). */
typedef struct csq_text_in {
    const uint8_t* text;
    uint64_t bytes;
} csq_text_in;

/* Under CSQ_PLAN_FASTA a text batch holds FASTA records instead: a record starts at a line whose first byte is '>'; the
 * header is the rest of that line without its trailing '\r' / '\n' bytes; the sequence is the concatenation of the
 * following lines up to the next header, each stripped of leading and trailing ASCII whitespace (blank lines and empty
 * sequences are allowed).  Blank lines may stand in front of the first header; any other text there is CSQ_ERR_FORMAT.
 * n_reads is the number of headers; a batch holding a different number is CSQ_ERR_FORMAT.  The last line must be
 * ended by '\n' as for FASTQ.  A FASTA read is trimmed as if every quality were 'I' (Q40 at base 33). */
typedef struct csq_batch_text {
    uint32_t n_reads;          /* records per mate in this batch                       */
    uint32_t n_mates;          /* 1 or 2                                               */
    uint64_t first_record;     /* index of the batch's first record in the file (error texts) */
    csq_text_in mate[2];
} csq_batch_text;

/* Batch in, BGZF form: per mate a run of WHOLE BGZF members (bgzip files, this library's own .gz output) as they stand
 * in the file.  The device inflates them (one warp per member) and finds the records itself; the batch's n_reads
 * records start behind `skip_lines` line ends of the inflated text, whatever follows them is ignored - so the host
 * cuts batches at member boundaries and only has to know how many line ends every member holds
 * (csq_bgzf_count_lines).  member_off / text_off are prefix sums over the members: compressed sizes (the 'BC' field)
 * and ISIZE (the last four bytes of a member). */
typedef struct csq_bgzf_in {
    const uint8_t* data;          /* the members, back to back; readable 16 bytes past the end            */
    uint64_t bytes;
    const uint32_t* member_off;   /* n_members + 1 offsets into data                                      */
    const uint32_t* text_off;     /* n_members + 1 offsets into the inflated text                         */
    uint32_t n_members;
    uint32_t skip_lines;          /* line ends of the inflated text in front of the batch's first record  */
    uint32_t append_newline;      /* end of file without a final line end: add one behind the text        */
    uint32_t reserved;
} csq_bgzf_in;

typedef struct csq_batch_bgzf {
    uint32_t n_reads;
    uint32_t n_mates;
    uint64_t first_record;
    csq_bgzf_in mate[2];
} csq_batch_bgzf;

/* Batch out: FASTQ text ("@name\nseq\n+\nqual\n" per record, input order) per
 * destination and mate, written into caller-owned buffers. */
typedef struct csq_text_out {
    uint8_t* data;
    uint64_t capacity;
    uint64_t bytes;     /* out */
    uint64_t records;   /* out */
} csq_text_out;

typedef struct csq_batch_out {
    csq_text_out text[CSQ_N_DEST][2];
} csq_batch_out;

/* Result of one ALIGN op on one read == the tuple Aligner.locate returns, after the
 * coordinate mapping of RightmostFrontAdapter. found==0 means locate returned None. */
typedef struct csq_match {
    int16_t found;
    int16_t ref_start, ref_stop;
    int16_t query_start, query_stop;
    int16_t score, errors;
    int16_t reserved;
} csq_match;

/* Per-mate interval left by the chain: read == original[start:stop]. */
typedef struct csq_read_result {
    uint32_t start, stop;
    uint32_t dest;       /* csq_dest of the read / pair */
    uint32_t matched;    /* adapter_id bits found (bit 31: any AdapterCutter matched) */
} csq_read_result;

/* Counters (sum over processed batches): the fields of cutadapt's minimal report. */
typedef struct csq_counters {
    uint64_t n;                  /* reads / pairs processed                */
    uint64_t total_bp[2];        /* input bases per mate                   */
    uint64_t written;            /* reads / pairs sent to the sink         */
    uint64_t written_bp[2];      /* bases written to the sink per mate     */
    uint64_t too_short;          /* reads / pairs filtered by TooShort     */
    uint64_t untrimmed;          /* reads / pairs filtered by IsUntrimmedAny */
    uint64_t quality_trimmed_bp[2];
    uint64_t with_adapters[2][CSQ_MAX_OPS]; /* matches per ALIGN op, indexed by op position */
    uint64_t dp_cells[2][CSQ_MAX_OPS];      /* nominal DP cells m*(max_n-min_n) per ALIGN op
                                               (SURVEY.md 8(d): the GCUPS numerator)         */
    /* cutadapt's EndStatistics.adjacent_bases of the FIRST ALIGN op of every mate (the one whose statistics the
     * reference's report keeps, run.py:58-73) when that adapter trims behind the match (3' kinds): the read base in
     * front of the match - A, C, G, T, none (the match starts the read), any other character */
    uint64_t adjacent_bases[2][6];
} csq_counters;

typedef struct csq_plan csq_plan;

#define CSQ_PLAN_KEEP_MATCHES 1u  /* keep per-ALIGN csq_match records (tests, statistics) */
#define CSQ_PLAN_NO_PREFILTER 2u  /* run the exact DP on every read (no bit-parallel prefilter) */
#define CSQ_PLAN_ONE_STREAM 64u   /* run the chains of mate 1 and mate 2 on one stream (default: side by side) */
#define CSQ_PLAN_EMIT_G16 256u    /* emit FASTQ text with the direct (global -> global) k_emit, 16 lanes per record, instead of
                                     the default k_emit_stage (staged through shared memory); A/B runs, initcheck runs   */
#define CSQ_PLAN_GZIP_OUT 4096u   /* csq_wait delivers every output stream as concatenated gzip members (BGZF framing, <= 64 KiB
                                     each, dynamic-Huffman DEFLATE encoded on the device) instead of FASTQ text:
                                     csq_text_out.bytes = compressed bytes; what xopen does behind the reference's
                                     default .fastq.gz outputs (run.py:1058-1093), without the text crossing PCIe    */
#define CSQ_PLAN_NO_EXACT_STOP 1024u /* exact DP walks every column even after an error-free full match (results are the same; A/B) */
#define CSQ_PLAN_FASTA 8192u     /* text batches (csq_submit_text, csq_upload_text) hold FASTA records and the emitters write FASTA
                                     (">name\nsequence\n", not wrapped); see csq_batch_text.  csq_submit, csq_upload,
                                     csq_submit_bgzf and csq_bgzf_count_lines return CSQ_ERR_INVALID under this flag          */
/* (flag values 8, 16, 32, 128, 512, 2048 selected slower kernel variants in round 1 - per-pair / 8- / 32-lane emitters,
 * one-pass parse, one-lane / one-column homopolymer DP; those kernels were removed after measurement and the bits are ignored) */

/* Library / device */
int csq_abi_version(void);
const char* csq_last_error(void);
int csq_device_count(int* count);                 /* number of usable sm_100 devices */

/* Plan: the compiled op program for one run (the `modifiers` + `steps` lists). */
int csq_plan_create(const csq_op* ops_r1, int n1, const csq_op* ops_r2, int n2,
                    const csq_filters* filters, int device, uint32_t flags, csq_plan** out);
void csq_plan_destroy(csq_plan* plan);

/* Asynchronous batch execution on slot 0..CSQ_N_SLOTS-1 (each slot = one stream +
 * device buffers): submit copies the batch to the device, runs the chain, emits FASTQ
 * text and copies it back into `out`; wait blocks until that is complete. */
#define CSQ_N_SLOTS 8
int csq_submit(csq_plan* plan, int slot, const csq_batch_in* in, csq_batch_out* out);
int csq_submit_text(csq_plan* plan, int slot, const csq_batch_text* in, csq_batch_out* out);
int csq_submit_bgzf(csq_plan* plan, int slot, const csq_batch_bgzf* in, csq_batch_out* out);
/* Inflates the members on the device and returns the number of line ends in each (host array of n_members; bit 31 of
 * an entry is set when that member's text does not end in a line end); blocks.
 * The file driver's first pass over a BGZF input: from these counts it cuts record-aligned batches. */
int csq_bgzf_count_lines(csq_plan* plan, int slot, const csq_bgzf_in* in, uint32_t* lines);
int csq_wait(csq_plan* plan, int slot);
/* Device time of the last completed submit on this slot, in ms, by CUDA events on the
 * slot's stream: total (H2D + kernels + D2H) and kernels only. */
int csq_slot_times(csq_plan* plan, int slot, float* total_ms, float* kernel_ms);

/* Resident mode (measurement): upload once, run the kernels `iters` times on data that
 * stays in HBM; ms_per_iter is measured with CUDA events on the slot's stream. */
int csq_upload(csq_plan* plan, int slot, const csq_batch_in* in);
int csq_upload_text(csq_plan* plan, int slot, const csq_batch_text* in);
int csq_run_resident(csq_plan* plan, int slot, int iters, float* ms_per_iter);
/* The same over several uploaded slots: after an untimed sizing pass per slot, `steps` steps run
 * back to back on one stream pair, step i on slots[i % n_slots]; total_ms is the CUDA-event time of
 * the whole loop (consecutive steps touch different data, each far larger than L2).  One further,
 * untimed step on a single stream follows for the per-kernel times (csq_kernel_times). */
int csq_run_steps(csq_plan* plan, const int* slots, int n_slots, int steps, float* total_ms);
/* Per-kernel device times (ms, last step of the last csq_run_resident / csq_run_steps call; for
 * csq_run_steps query the first slot of the list). names
 * points at static strings. Returns the number of kernels recorded (<= cap). */
int csq_kernel_times(csq_plan* plan, int slot, const char** names, float* ms, int cap);
int csq_launch_count(csq_plan* plan, uint64_t* launches);   /* kernels launched so far */
/* After csq_wait / csq_run_resident: copy results of the slot back for inspection. */
int csq_fetch_results(csq_plan* plan, int slot, int mate, csq_read_result* out, uint32_t n);
int csq_fetch_matches(csq_plan* plan, int slot, int mate, int op_index, csq_match* out, uint32_t n);
int csq_fetch_text(csq_plan* plan, int slot, csq_batch_out* out);
int csq_stats(csq_plan* plan, csq_counters* out);            /* accumulated counters */

/* Stand-alone aligner call == Aligner(adapter, rate, flags, min_overlap=..).locate(read)
 * for a batch of reads (adapter_kind picks flags / reversal). For parity tests. */
int csq_locate_batch(int device, const csq_op* align_op, const csq_mate_in* reads, uint32_t n_reads,
                     uint32_t plan_flags, csq_match* out);

/* Integer-issue microbenchmark used as the DP roofline denominator: returns measured
 * 32-bit integer lane-ops per second for (0) ALU-pipe only, (1) ALU+FMA-pipe mix. */
int csq_int_peak(int device, double* alu_ops_per_s, double* mixed_ops_per_s);

/* Host <-> device copy ceiling used as the denominator of the end-to-end numbers: pinned buffers of the given
 * sizes, `reps` copies, mode 0 = host->device alone, 1 = device->host alone, 2 = both directions at once (what the
 * pipelined csq_submit_text / csq_wait loop does).  GB/s per direction; in mode 2 over the time both needed. */
int csq_pcie_peak(int device, uint64_t bytes_h2d, uint64_t bytes_d2h, int reps, int mode, double* h2d_gbs, double* d2h_gbs);

/* One process (or thread) per GPU: restrict the calling thread - and the threads and pinned buffers it creates
 * afterwards - to the CPUs / memory of the NUMA node the device's PCIe root port belongs to.  *numa_node = the
 * node, or -1 when nothing was changed (single node, no sysfs entry, cpuset without CPUs of that node).
 * csq_unbind_host() restores the affinity mask and memory policy saved by the first bind.  The reference has no
 * counterpart (cutadapt's worker processes are not placed); used by bench.py / dist runs. */
int csq_bind_host_to_device(int device, int* numa_node);
int csq_unbind_host(void);

/* ---------------------------------------------------------------------------
 * Host FASTQ side (the step either side of the path: dnaio / xopen in the reference).
 * ------------------------------------------------------------------------- */
typedef struct csq_reader csq_reader;
/* Opens 1 or 2 FASTQ files (plain or .gz by magic bytes). */
int csq_reader_open(const char* path1, const char* path2, csq_reader** out);
/* Parses up to max_reads records (pairs) into library-owned pinned SoA buffers that
 * stay valid until the next call with the same buffer index (0..CSQ_N_SLOTS-1).
 * in->n_reads == 0 at end of input. */
int csq_reader_next(csq_reader* r, int buffer, uint32_t max_reads, csq_batch_in* in);
void csq_reader_close(csq_reader* r);
/* Parse FASTQ text that is already in memory into caller-provided SoA arrays (tests). */
int csq_parse_fastq_mem(const uint8_t* text, uint64_t n_bytes, uint32_t max_reads,
                        uint8_t* seq, uint8_t* qual, uint64_t seq_cap, uint32_t* seq_off,
                        uint32_t* seq_len, uint8_t* name, uint64_t name_cap, uint32_t* name_off,
                        uint32_t* n_reads, uint64_t* seq_bytes, uint64_t* consumed);

/* Reader for text batches: opens 1 or 2 FASTQ files (plain, or gzip incl. concatenated members,
 * by magic bytes) and returns max_reads whole records per mate as raw text in library-owned
 * pinned buffers (valid until the next call with the same buffer index). No parsing happens
 * on the host: the stream is cut after 4 * max_reads line ends. in->n_reads == 0 at the end. */
typedef struct csq_text_reader csq_text_reader;
int csq_text_reader_open(const char* path1, const char* path2, csq_text_reader** out);
/* The same with plan flags: under CSQ_PLAN_FASTA the files are FASTA and the stream is cut in front of the
 * (max_reads + 1)-th record start instead (batches hold max_reads records; see csq_batch_text).  BGZF-framed files are
 * read like any gzip file. */
int csq_text_reader_open_flags(const char* path1, const char* path2, uint32_t plan_flags, csq_text_reader** out);
int csq_text_reader_next(csq_text_reader* r, int buffer, uint32_t max_reads, csq_batch_text* in);
void csq_text_reader_close(csq_text_reader* r);
/* Text-batch helpers (host, SIMD): number of '\n' in [text, text + n_bytes); and the offset
 * one past the k-th '\n' (k >= 1), or UINT64_MAX when there are fewer. */
uint64_t csq_count_newlines(const uint8_t* text, uint64_t n_bytes);
uint64_t csq_after_kth_newline(const uint8_t* text, uint64_t n_bytes, uint64_t k);
/* FASTA twin (host, SIMD): the offset of the (k+1)-th record start ('>' as the first byte of a line; the text starts at
 * a line start) in [text, text + n_bytes), or UINT64_MAX when there are fewer.  k = 0: the first record start. */
uint64_t csq_after_kth_fasta_record(const uint8_t* text, uint64_t n_bytes, uint64_t k);
/* gzip data in memory -> dst, decoded in pieces of `piece` bytes with the library's own inflate (tests). */
int csq_gunzip_mem(const uint8_t* src, uint64_t n, uint8_t* dst, uint64_t cap, uint64_t piece, uint64_t* out_n);
/* The device gzip writer's algorithm run on the host, piece by piece (CPU tests of the code construction, the block
 * header, the bit packing and the CRC folding): text -> concatenated BGZF members. */
int csq_gz_deflate_host(const uint8_t* text, uint64_t n, uint8_t* out, uint64_t cap, uint64_t* out_n);
/* The device gzip reader's decoder run on the host, member by member (CPU tests): BGZF members -> text; *lines = '\n' found. */
int csq_gz_inflate_host(const uint8_t* src, uint64_t n, uint8_t* dst, uint64_t cap, uint64_t* out_n, uint64_t* lines);
/* The parallel decoder of ordinary (single-stream) gzip files (csrc/pinflate.cpp; the file driver uses it for .gz inputs
 * without BGZF framing): a whole gzip file in memory -> text.  span_bytes: compressed bytes per thread and round
 * (0: default); tests use small values. */
int csq_pinflate_mem(const uint8_t* src, uint64_t n, uint8_t* dst, uint64_t cap, int threads, uint64_t span_bytes, uint64_t* out_n);
/* The device decoder of ordinary gzip files (csrc/gz_stream.cu; the device counterpart of csq_pinflate_mem, which the
 * file driver keeps using - DESIGN.md section 4.6): a whole gzip file in memory -> text, decoded on `device`.  The stream is decoded in rounds of
 * `round_bytes` compressed bytes, each cut into spans of `span_bytes` (0: the defaults, 64 MiB and 128 KiB); tests use
 * small values.  CSQ_ERR_IO with a message for damaged, truncated or trailing-garbage input and CRC-32 / ISIZE
 * mismatches, CSQ_ERR_CAPACITY when the text does not fit in `cap`. */
int csq_gz_stream_inflate(int device, const uint8_t* src, uint64_t n, uint8_t* dst, uint64_t cap, uint64_t span_bytes,
                          uint64_t round_bytes, uint64_t* out_n);
/* The same decoder's host twin (the same search, decode, window and resolve code with one lane; CPU tests). */
int csq_gz_stream_inflate_host(const uint8_t* src, uint64_t n, uint8_t* dst, uint64_t cap, uint64_t span_bytes,
                               uint64_t round_bytes, uint64_t* out_n);
/* The decode chain of the calling thread's last csq_gz_stream_inflate(_host) call: (start bit, end bit, symbols) of every
 * span in file order, up to max_entries triples into out.  Returns the number of spans (tests). */
uint64_t csq_gz_stream_chain(uint64_t* out, uint64_t max_entries);
/* SoA batch -> FASTQ text of one mate ("@name\nseq\n+\nqual\n"), for tests and benchmarks. */
int csq_format_fastq(const csq_mate_in* mate, uint32_t n_reads, uint8_t* out, uint64_t capacity,
                     uint64_t* bytes);

/* Whole-file driver: read -> (double-buffered) GPU chain -> ordered write. Output paths
 * may be NULL (destination discarded); a ".gz" suffix selects gzip output.  With CSQ_PLAN_FASTA in plan_flags the
 * inputs are FASTA files (plain or gzip) and the outputs FASTA. */
typedef struct csq_files {
    const char* in[2];
    const char* out[CSQ_N_DEST][2];
    uint32_t batch_reads;     /* reads (pairs) per batch; 0 = default                */
    int32_t gzip_level;       /* 1..9; 0 = default (1, as cutadapt/xopen)            */
    int32_t n_threads;        /* host threads for deflate; 0 = default               */
    int32_t n_devices;        /* GPUs to shard over; 0 = 1                           */
    const int32_t* devices;   /* device ordinals (n_devices entries) or NULL = 0..n-1 */
    int32_t swap_sink;        /* paired --auto-rc on '-' strand: R1->out[..][1], R2->out[..][0]
                                 for CSQ_DEST_TRIMMED only (run.py:785-792)            */
} csq_files;

typedef struct csq_timing {   /* seconds, wall clock, summed over batches            */
    double read_inflate, parse, h2d_kernels_d2h, kernels, write_deflate, total;
} csq_timing;

int csq_run_files(const csq_op* ops_r1, int n1, const csq_op* ops_r2, int n2,
                  const csq_filters* filters, uint32_t plan_flags, const csq_files* files,
                  csq_counters* counters, csq_timing* timing);

/* Synthetic workload generator (BASELINE.json configs 2-5; SURVEY.md 8(d)); record i
 * depends only on (seed, first_index + i). Fills library-owned pinned SoA buffers. */
typedef struct csq_synth {
    uint64_t seed;
    uint32_t read_len;          /* 150 (configs 2,3,5) or 75 (config 4)               */
    uint32_t paired;            /* 1 / 0                                              */
    uint32_t config;            /* 2, 3 or 4                                          */
} csq_synth;
int csq_synth_batch(const csq_synth* cfg, uint64_t first_index, uint32_t n_reads, int buffer,
                    csq_batch_in* in);
void csq_synth_free(void);

#ifdef __cplusplus
}
#endif
#endif /* CUTSEQ_B200_H */
