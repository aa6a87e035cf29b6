/*
 * cutseq_oracle.c - TEST INFRASTRUCTURE ONLY.  CPU restatement (plain C) of the reference
 * algorithm for cutseq's per-read trimming path.  Only tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline / --impl reference legs may load this; nothing under
 * cutseq_b200/ does.
 *
 * PARITY UNPINNED.  The arithmetic of this path lives in the reference's un-vendored
 * dependency cutadapt (pyproject.toml:17 "cutadapt~=5.0", no lock file; dnaio/xopen behind
 * it), which is absent from /root/reference and cannot be installed offline.  The
 * reference ships no golden vectors or known-answer tests (its test/ holds two input files
 * only).  This file therefore restates cutadapt's published algorithm (upstream
 * src/cutadapt/_align.pyx Aligner.locate, adapters.py, modifiers.py, qualtrim.pyx,
 * predicates.py, steps.py, pipeline.py) and is anchored on the reference's own call sites:
 *   run.py:326-426 / 533-731   which modifiers, with which parameters, in which order
 *   run.py:113-161             ConditionalCutter
 *   run.py:78-110              IsUntrimmedAny
 *   run.py:164-187             ReverseComplementConverter
 *   run.py:446-471 / 763-792   filters and sink
 * It is cross-checked in tests/ against a second, independent pure-Python restatement
 * (oracle/cutadapt_shim) under which the UNMODIFIED reference run.py is executed to
 * produce tests/golden/.
 *
 * The program it executes is the same csq_op list the product takes
 * (include/cutseq_b200.h), so tests feed both sides identical inputs.
 */
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <pthread.h>
#include <unistd.h>

#include "../include/cutseq_b200.h"

typedef struct orc_entry {
    int cost, score, origin;
} orc_entry;

typedef struct orc_match {
    int found, ref_start, ref_stop, query_start, query_stop, score, errors;
} orc_match;

static int imin(int a, int b) { return a < b ? a : b; }
static int imax(int a, int b) { return a > b ? a : b; }
static char up(char c) { return (c >= 'a' && c <= 'z') ? (char)(c - 32) : c; }

/*
 * Aligner.locate (upstream _align.pyx).  reference s1[0..m), query s2[0..n), flags =
 * EndSkip bits.  One column, Ukkonen band, (cost, score, origin) per cell; best match by the
 * row-m rule while scanning columns, then the last-column search.  The query is compared
 * upper-cased (SingleAdapter.match_to passes sequence.upper()); the adapter is ACGT only so
 * this is plain byte equality (adapter_wildcards is switched off by cutadapt for such
 * adapters, read_wildcards defaults to False: a read 'N' is a mismatch).
 */
int orc_locate(const char* s1, int m, double max_error_rate, int flags, int min_overlap,
               const char* s2, int n, orc_match* out) {
    const int start_in_reference = flags & 1, start_in_query = flags & 2;
    const int stop_in_reference = flags & 4, stop_in_query = flags & 8;
    orc_entry* column = (orc_entry*)malloc(sizeof(orc_entry) * (size_t)(m + 1));
    int i, j;
    int k = (int)(max_error_rate * m);
    int max_n = n, min_n = 0;
    if (!start_in_query) max_n = imin(n, m + k);
    if (!stop_in_query) min_n = imax(0, n - m - k);

    for (i = 0; i <= m; i++) {
        column[i].score = 0;
        if (!start_in_reference && !start_in_query) {
            column[i].cost = imax(i, min_n);
            column[i].origin = 0;
        } else if (start_in_reference && !start_in_query) {
            column[i].cost = min_n;
            column[i].origin = imin(0, min_n - i);
        } else if (!start_in_reference && start_in_query) {
            column[i].cost = i;
            column[i].origin = imax(0, min_n - i);
        } else {
            column[i].cost = imin(i, min_n);
            column[i].origin = min_n - i;
        }
    }

    const int none = m + n + 1;
    int best_cost = none, best_origin = 0, best_score = 0, best_ref_stop = m, best_query_stop = n;
    int last = imin(m, k + 1);
    if (start_in_reference) last = m;

    for (j = min_n + 1; j <= max_n; j++) {
        orc_entry diag = column[0];
        if (start_in_query)
            column[0].origin = j;
        else
            column[0].cost = j;
        const char c2 = up(s2[j - 1]);
        for (i = 1; i <= last; i++) {
            int cost, origin, score;
            if (s1[i - 1] == c2) {
                cost = diag.cost;
                origin = diag.origin;
                score = diag.score + 1;
            } else {
                int cost_diag = diag.cost + 1;
                int cost_deletion = column[i].cost + 1;
                int cost_insertion = column[i - 1].cost + 1;
                if (cost_diag <= cost_deletion && cost_diag <= cost_insertion) {
                    cost = cost_diag;
                    origin = diag.origin;
                    score = diag.score - 1;
                } else if (cost_insertion <= cost_deletion) {
                    cost = cost_insertion;
                    origin = column[i - 1].origin;
                    score = column[i - 1].score - 2;
                } else {
                    cost = cost_deletion;
                    origin = column[i].origin;
                    score = column[i].score - 2;
                }
            }
            diag = column[i];
            column[i].cost = cost;
            column[i].origin = origin;
            column[i].score = score;
        }
        while (last >= 0 && column[last].cost > k) last--;
        if (last < m) {
            last++;
        } else if (stop_in_query) {
            int cost = column[m].cost, score = column[m].score, origin = column[m].origin;
            int length = m + imin(origin, 0);
            int acceptable = length >= min_overlap && (double)cost <= length * max_error_rate;
            int best_length = m + imin(best_origin, 0);
            if (acceptable && (best_cost == none || (origin <= best_origin + m / 2 && score > best_score) ||
                               (length > best_length && score > best_score))) {
                best_score = score;
                best_cost = cost;
                best_origin = origin;
                best_ref_stop = m;
                best_query_stop = j;
                if (cost == 0 && origin >= 0) break;
            }
        }
    }

    if (max_n == n) {
        int first_i = stop_in_reference ? 0 : m;
        for (i = m; i >= first_i; i--) {
            int length = i + imin(column[i].origin, 0);
            int cost = column[i].cost, score = column[i].score;
            int acceptable = length >= min_overlap && (double)cost <= length * max_error_rate;
            if (acceptable && (score > best_score || (score == best_score && cost < best_cost))) {
                best_score = score;
                best_cost = cost;
                best_origin = column[i].origin;
                best_ref_stop = i;
                best_query_stop = n;
            }
        }
    }
    free(column);
    memset(out, 0, sizeof(*out));
    if (best_cost == none) return 0;
    out->found = 1;
    out->ref_start = best_origin >= 0 ? 0 : -best_origin;
    out->query_start = best_origin >= 0 ? best_origin : 0;
    out->ref_stop = best_ref_stop;
    out->query_stop = best_query_stop;
    out->score = best_score;
    out->errors = best_cost;
    return 1;
}

/* Where.* values per adapter class and which side of the match is removed (adapters.py). */
static int kind_flags(int kind) {
    switch (kind) {
        case CSQ_AD_BACK: return 14;
        case CSQ_AD_BACK_ANYWHERE: return 15;
        case CSQ_AD_RIGHTMOST_FRONT: return 14; /* BACK, on reversed adapter and read */
        case CSQ_AD_PREFIX: return 8;
        case CSQ_AD_SUFFIX: return 2;
        case CSQ_AD_NI_FRONT: return 9;
        case CSQ_AD_NI_BACK: return 6;
        case CSQ_AD_FRONT: return 11;
    }
    return -1;
}
static int kind_is_front(int kind) {
    return kind == CSQ_AD_RIGHTMOST_FRONT || kind == CSQ_AD_PREFIX || kind == CSQ_AD_NI_FRONT ||
           kind == CSQ_AD_FRONT;
}

/* <Adapter>.match_to(sequence): SingleAdapter.__init__ clamps min_overlap to m, Prefix/Suffix
 * force it to m; RightmostFrontAdapter reverses adapter and read and maps coordinates back. */
int orc_adapter_match(const csq_op* op, const char* seq, int n, orc_match* out) {
    int m = op->adapter_len;
    int min_overlap = imin(op->min_overlap, m);
    /* SingleAdapter.__init__: max_errors >= 1 is an absolute count */
    const double rate = op->max_error_rate >= 1.0 ? op->max_error_rate / m : op->max_error_rate;
    if (op->adapter_kind == CSQ_AD_PREFIX || op->adapter_kind == CSQ_AD_SUFFIX) min_overlap = m;
    if (op->adapter_kind == CSQ_AD_RIGHTMOST_FRONT) {
        char ref[CSQ_MAX_ADAPTER];
        char* q = (char*)malloc((size_t)n + 1);
        for (int i = 0; i < m; i++) ref[i] = op->adapter[m - 1 - i];
        for (int j = 0; j < n; j++) q[j] = seq[n - 1 - j];
        orc_match r;
        int found = orc_locate(ref, m, rate, 14, min_overlap, q, n, &r);
        free(q);
        memset(out, 0, sizeof(*out));
        if (!found) return 0;
        out->found = 1;
        out->ref_start = m - r.ref_stop;
        out->ref_stop = m - r.ref_start;
        out->query_start = n - r.query_stop;
        out->query_stop = n - r.query_start;
        out->score = r.score;
        out->errors = r.errors;
        return 1;
    }
    return orc_locate(op->adapter, m, rate, kind_flags(op->adapter_kind), min_overlap, seq, n, out);
}

/* quality_trim_index (upstream qualtrim.pyx) */
void orc_quality_trim_index(const char* q, int n, int cutoff_front, int cutoff_back, int base, int* start_out,
                            int* stop_out) {
    int stop = n, start = 0, s = 0, max_qual = 0, i;
    for (i = 0; i < n; i++) {
        s += cutoff_front - ((unsigned char)q[i] - base);
        if (s < 0) break;
        if (s > max_qual) {
            max_qual = s;
            start = i + 1;
        }
    }
    max_qual = 0;
    s = 0;
    for (i = n - 1; i >= 0; i--) {
        s += cutoff_back - ((unsigned char)q[i] - base);
        if (s < 0) break;
        if (s > max_qual) {
            max_qual = s;
            stop = i;
        }
    }
    if (start >= stop) start = stop = 0;
    *start_out = start;
    *stop_out = stop;
}

/* Nominal DP cells of one alignment, m * (max_n - min_n): the GCUPS numerator of SURVEY.md 8(d). */
static uint64_t nominal_cells(const csq_op* op, int n) {
    int m = op->adapter_len, flags = kind_flags(op->adapter_kind);
    double rate = op->max_error_rate >= 1.0 ? op->max_error_rate / m : op->max_error_rate;
    int k = (int)(rate * m), max_n = n, min_n = 0;
    if (!(flags & 2)) max_n = imin(n, m + k);
    if (!(flags & 8)) min_n = imax(0, n - m - k);
    return (uint64_t)m * (uint64_t)(max_n - min_n);
}

/* EndStatistics.adjacent_bases slot of a 3' match: A, C, G, T, none (rstart == 0), other */
static int adjacent_slot(const char* seq, int query_start) {
    if (query_start <= 0) return 4;
    char c = seq[query_start - 1];
    return c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : 5;
}

/* ---- per-read working record (the SequenceRecord + ModificationInfo of one mate) ---- */
/* Longest name a record can carry: the product's 65535-byte header limit, then a renamed id of at most that length
 * plus '_' and two UMI parts of at most CSQ_MAX_READ_LEN bases each. */
#define ORC_NAME_CAP (65535 + 1 + 2 * CSQ_MAX_READ_LEN)

typedef struct orc_read {
    char* seq;   /* working copies, sliced by moving seq/qual and len */
    char* qual;
    int len;
    int orig_off; /* offset of seq[0] inside the original read (undefined after REVCOMP) */
    char* name; /* ORC_NAME_CAP bytes, owned by the chunk worker */
    int name_len;
    /* ModificationInfo */
    int n_matches;
    uint32_t matched_ids;
    const char* cut_prefix;
    int cut_prefix_len; /* -1 == None */
    const char* cut_suffix;
    int cut_suffix_len;
    char* buf_seq; /* owned storage */
    char* buf_qual;
} orc_read;

static int is_py_space(unsigned char c) { return c == ' ' || (c >= 9 && c <= 13) || (c >= 28 && c <= 31); }

/* Renamer.parse_name: fields = name.split(maxsplit=1); id = fields[0] if there are two
 * fields, else the whole name. Returns [id_start, id_end). */
static void parse_name_id(const char* name, int len, int* id_start, int* id_end) {
    int p = 0;
    while (p < len && is_py_space((unsigned char)name[p])) p++;
    int s = p;
    while (p < len && !is_py_space((unsigned char)name[p])) p++;
    int e = p;
    while (p < len && is_py_space((unsigned char)name[p])) p++;
    if (e > s && p < len) { /* a second field exists */
        *id_start = s;
        *id_end = e;
    } else {
        *id_start = 0;
        *id_end = len;
    }
}

/* dnaio record_names_match == SequenceRecord.is_mate (upstream src/dnaio/_core.pyx, record_ids_match): the id of
 * header 2 ends at its first ' ' or '\t' (strcspn; NOT str.split's whitespace set); header 1 must end, or carry a
 * ' ' / '\t', at that very position; when both ids end in '1', '2' or '3' that last character is not compared
 * ("/1" "/2" of old Illumina names, ".1" ".2" of fastq-dump -I); the rest must be byte-identical.  Used twice on the
 * reference's path: by dnaio's paired reader on the headers as they stand in the files, and by cutadapt's
 * PairedEndRenamer (run.py:643-645) on the headers as the SuffixRemovers of run.py:537-542 left them. */
static int names_match(const char* h1, int n1, const char* h2, int n2) {
    int id2 = 0;
    while (id2 < n2 && h2[id2] != ' ' && h2[id2] != '\t') id2++;
    if (n1 < id2) return 0;
    if (id2 < n1 && h1[id2] != ' ' && h1[id2] != '\t') return 0;
    if (id2 > 0 && h1[id2 - 1] >= '1' && h1[id2 - 1] <= '3' && h2[id2 - 1] >= '1' && h2[id2 - 1] <= '3') id2--;
    return memcmp(h1, h2, (size_t)id2) == 0;
}

int orc_names_match(const char* h1, int n1, const char* h2, int n2) { return names_match(h1, n1, h2, n2); }

static void slice(orc_read* r, int start, int stop) { /* python read[start:stop], 0<=start<=stop<=len */
    r->seq += start;
    r->qual += start;
    r->orig_off += start;
    r->len = stop - start;
}

static char complement(char c) {
    static const char* a = "ACGTUMRWSYKVHDBNacgtumrwsykvhdbn";
    static const char* b = "TGCAAKYWSRMBDHVNtgcaakywsrmbdhvn";
    const char* p = strchr(a, c);
    return (p && c) ? b[p - a] : c;
}

static void apply_single(const csq_op* op, orc_read* r, orc_match* match_out, uint64_t* qtrim_bp) {
    switch (op->kind) {
        case CSQ_OP_STRIP_SUFFIX: { /* SuffixRemover */
            int sl = op->suffix_len;
            if (r->name_len >= sl && memcmp(r->name + r->name_len - sl, op->suffix, (size_t)sl) == 0) r->name_len -= sl;
            break;
        }
        case CSQ_OP_ALIGN: { /* AdapterCutter(times=1, action=trim) */
            orc_match mt;
            int found = orc_adapter_match(op, r->seq, r->len, &mt);
            if (match_out) *match_out = mt;
            if (found) {
                r->n_matches++;
                if (op->adapter_id >= 0) r->matched_ids |= 1u << op->adapter_id;
                if (kind_is_front(op->adapter_kind))
                    slice(r, mt.query_stop, r->len); /* RemoveBeforeMatch: read[rstop:] */
                else
                    slice(r, 0, mt.query_start); /* RemoveAfterMatch: read[:rstart] */
            }
            break;
        }
        case CSQ_OP_COND_CUT: /* ConditionalCutter, run.py:154-161 */
            if (r->n_matches == 0 && r->len < op->force_trim_min_length) break;
            /* fall through */
        case CSQ_OP_CUT: { /* UnconditionalCutter */
            int L = op->length;
            if (L > 0) {
                int c = imin(L, r->len);
                r->cut_prefix = r->seq;
                r->cut_prefix_len = c;
                slice(r, c, r->len);
            } else if (L < 0) {
                int c = imin(-L, r->len);
                r->cut_suffix = r->seq + (r->len - c);
                r->cut_suffix_len = c;
                slice(r, 0, r->len - c);
            }
            break;
        }
        case CSQ_OP_QTRIM: {
            int start, stop;
            orc_quality_trim_index(r->qual, r->len, op->cutoff_front, op->cutoff_back, op->quality_base, &start, &stop);
            if (qtrim_bp) *qtrim_bp += (uint64_t)(r->len - (stop - start));
            slice(r, start, stop);
            break;
        }
        case CSQ_OP_REVCOMP: {
            for (int i = 0, j = r->len - 1; i <= j; i++, j--) {
                char a = complement(r->seq[i]), b = complement(r->seq[j]);
                r->seq[i] = b;
                r->seq[j] = a;
                char qa = r->qual[i];
                r->qual[i] = r->qual[j];
                r->qual[j] = qa;
            }
            break;
        }
        default: break;
    }
}

/* Renamer / PairedEndRenamer with the templates run.py builds; out: ORC_NAME_CAP bytes of scratch. */
static int apply_rename(const csq_op* op, orc_read* r, const orc_read* r1, const orc_read* r2, char* out) {
    int s, e;
    parse_name_id(r->name, r->name_len, &s, &e);
    int n = 0;
    memcpy(out, r->name + s, (size_t)(e - s));
    n = e - s;
    if (op->rename_parts) {
        out[n++] = '_';
        if ((op->rename_parts & CSQ_REN_OWN_PREFIX) && r->cut_prefix_len > 0) {
            memcpy(out + n, r->cut_prefix, (size_t)r->cut_prefix_len);
            n += r->cut_prefix_len;
        }
        if ((op->rename_parts & CSQ_REN_OWN_SUFFIX) && r->cut_suffix_len > 0) {
            memcpy(out + n, r->cut_suffix, (size_t)r->cut_suffix_len);
            n += r->cut_suffix_len;
        }
        if ((op->rename_parts & CSQ_REN_R1_PREFIX) && r1 && r1->cut_prefix_len > 0) {
            memcpy(out + n, r1->cut_prefix, (size_t)r1->cut_prefix_len);
            n += r1->cut_prefix_len;
        }
        if ((op->rename_parts & CSQ_REN_R2_PREFIX) && r2 && r2->cut_prefix_len > 0) {
            memcpy(out + n, r2->cut_prefix, (size_t)r2->cut_prefix_len);
            n += r2->cut_prefix_len;
        }
    }
    memcpy(r->name, out, (size_t)n);
    r->name_len = n;
    return 0;
}

typedef struct orc_buf {
    uint8_t* data;
    uint64_t len, cap, records;
} orc_buf;

static void buf_put(orc_buf* b, const void* p, size_t n) {
    if (b->len + n > b->cap) {
        b->cap = (b->cap ? b->cap * 2 : (1u << 16)) + n;
        b->data = (uint8_t*)realloc(b->data, b->cap);
    }
    memcpy(b->data + b->len, p, n);
    b->len += n;
}

static void write_fastq(orc_buf* b, const orc_read* r) { /* dnaio: @name\nseq\n+\nqual\n */
    buf_put(b, "@", 1);
    buf_put(b, r->name, (size_t)r->name_len);
    buf_put(b, "\n", 1);
    buf_put(b, r->seq, (size_t)r->len);
    buf_put(b, "\n+\n", 3);
    buf_put(b, r->qual, (size_t)r->len);
    buf_put(b, "\n", 1);
    b->records++;
}

static void load_read(orc_read* r, const csq_mate_in* in, uint32_t i, char* name_buf) {
    int len = (int)in->seq_len[i];
    r->buf_seq = (char*)malloc((size_t)len + 1);
    r->buf_qual = (char*)malloc((size_t)len + 1);
    memcpy(r->buf_seq, in->seq + in->seq_off[i], (size_t)len);
    if (in->qual)
        memcpy(r->buf_qual, in->qual + in->seq_off[i], (size_t)len);
    else
        memset(r->buf_qual, 'I', (size_t)len);
    r->seq = r->buf_seq;
    r->qual = r->buf_qual;
    r->len = len;
    r->orig_off = 0;
    r->name = name_buf;
    r->name_len = (int)(in->name_off[i + 1] - in->name_off[i]);
    if (r->name_len > 65535) r->name_len = 65535; /* orc_run_batch reports CSQ_ERR_LIMIT, as the product does */
    memcpy(r->name, in->name + in->name_off[i], (size_t)r->name_len);
    r->n_matches = 0;
    r->matched_ids = 0;
    r->cut_prefix = r->cut_suffix = NULL;
    r->cut_prefix_len = r->cut_suffix_len = -1;
}

/*
 * The pipeline of run.py:472-473 / 793-794 over a batch: for each read (pair) run the
 * modifiers in order (both mates in lock-step, as PairedEndModifierWrapper does), then the
 * steps: TooShort filter ("any" mate), optional IsUntrimmedAny filter ("any"), sink.
 * Outputs: FASTQ text per destination and mate (malloc'ed into out->text[][].data, caller
 * frees with orc_free), optional per-mate results and per-op matches.
 * Returns 0, CSQ_ERR_PAIRING when mate ids differ at a paired RENAME, or CSQ_ERR_LIMIT for a header longer than
 * 65535 bytes.
 */
typedef struct orc_job {
    const csq_op *ops1, *ops2;
    int n1, paired;
    const csq_filters* flt;
    const csq_batch_in* in;
    csq_read_result *res1, *res2;
    csq_match *matches1, *matches2;
    uint32_t n, lo, hi;
    orc_buf* b;       /* CSQ_N_DEST*2 buffers of this chunk */
    csq_counters* k;
    int status;
} orc_job;

static void store_match(csq_match* o, const orc_match* mt) {
    o->found = (int16_t)mt->found; o->ref_start = (int16_t)mt->ref_start; o->ref_stop = (int16_t)mt->ref_stop;
    o->query_start = (int16_t)mt->query_start; o->query_stop = (int16_t)mt->query_stop;
    o->score = (int16_t)mt->score; o->errors = (int16_t)mt->errors; o->reserved = 0;
}

static void* chunk_worker(void* arg) {
    orc_job* J = (orc_job*)arg;
    const csq_op *ops1 = J->ops1, *ops2 = J->ops2;
    const int n1 = J->n1, paired = J->paired;
    const csq_filters* flt = J->flt;
    const csq_batch_in* in = J->in;
    const uint32_t n = J->n;
    orc_buf* b = J->b;
    csq_counters* k = J->k;
    int first_align[2] = {-1, -1}; /* the AdapterCutter whose statistics the reference's report keeps (run.py:58-73) */
    for (int t = n1 - 1; t >= 0; t--) {
        if (ops1[t].kind == CSQ_OP_ALIGN) first_align[0] = t;
        if (paired && ops2[t].kind == CSQ_OP_ALIGN) first_align[1] = t;
    }
    char* names = (char*)malloc((size_t)3 * ORC_NAME_CAP); /* mate 1, mate 2, rename scratch */
    for (uint32_t i = J->lo; i < J->hi; i++) {
        orc_read r[2];
        load_read(&r[0], &in->mate[0], i, names);
        if (paired) load_read(&r[1], &in->mate[1], i, names + ORC_NAME_CAP);
        /* dnaio's paired reader: "Records are improperly paired" unless r1.is_mate(r2) */
        if (paired && !names_match(r[0].name, r[0].name_len, r[1].name, r[1].name_len)) J->status = CSQ_ERR_PAIRING;
        for (int mt_i = 0; mt_i < (paired ? 2 : 1); mt_i++)
            if (in->mate[mt_i].name_off[i + 1] - in->mate[mt_i].name_off[i] > 65535u) J->status = CSQ_ERR_LIMIT;
        k->n++;
        k->total_bp[0] += (uint64_t)r[0].len;
        if (paired) k->total_bp[1] += (uint64_t)r[1].len;
        for (int t = 0; t < n1; t++) {
            if (ops1[t].kind == CSQ_OP_RENAME) {
                if (paired) {
                    /* PairedEndRenamer.__call__: ValueError("Input read IDs not identical") unless
                     * record_names_match(read1.name, read2.name); each mate then keeps its OWN id */
                    if (!names_match(r[0].name, r[0].name_len, r[1].name, r[1].name_len)) J->status = CSQ_ERR_PAIRING;
                    orc_read a = r[0], bb = r[1]; /* both names are built from the pre-rename infos */
                    apply_rename(&ops1[t], &r[0], &a, &bb, names + 2 * ORC_NAME_CAP);
                    apply_rename(&ops2[t], &r[1], &a, &bb, names + 2 * ORC_NAME_CAP);
                } else {
                    apply_rename(&ops1[t], &r[0], NULL, NULL, names + 2 * ORC_NAME_CAP);
                }
                continue;
            }
            orc_match mt;
            memset(&mt, 0, sizeof(mt));
            if (ops1[t].kind == CSQ_OP_ALIGN) k->dp_cells[0][t] += nominal_cells(&ops1[t], r[0].len);
            /* adjacent base of a 3' match of the mate's first ALIGN op (BackAdapterStatistics.add_match): looked up before the cut */
            const char* seq_before[2] = {r[0].seq, r[1].seq};
            if (paired && ops2[t].kind == CSQ_OP_ALIGN) k->dp_cells[1][t] += nominal_cells(&ops2[t], r[1].len);
            apply_single(&ops1[t], &r[0], &mt, &k->quality_trimmed_bp[0]);
            if (ops1[t].kind == CSQ_OP_ALIGN) {
                if (mt.found) k->with_adapters[0][t]++;
                if (mt.found && t == first_align[0] && !kind_is_front(ops1[t].adapter_kind)) k->adjacent_bases[0][adjacent_slot(seq_before[0], mt.query_start)]++;
                if (J->matches1) store_match(&J->matches1[(size_t)t * n + i], &mt);
            }
            if (paired) {
                memset(&mt, 0, sizeof(mt));
                apply_single(&ops2[t], &r[1], &mt, &k->quality_trimmed_bp[1]);
                if (ops2[t].kind == CSQ_OP_ALIGN) {
                    if (mt.found) k->with_adapters[1][t]++;
                    if (mt.found && t == first_align[1] && !kind_is_front(ops2[t].adapter_kind)) k->adjacent_bases[1][adjacent_slot(seq_before[1], mt.query_start)]++;
                    if (J->matches2) store_match(&J->matches2[(size_t)t * n + i], &mt);
                }
            }
        }
        /* steps: TooShort filter ("any"), IsUntrimmedAny filter ("any"), sink */
        int dest;
        int too_short = r[0].len < flt->min_length || (paired && r[1].len < flt->min_length);
        if (too_short) {
            dest = CSQ_DEST_SHORT;
            k->too_short++;
        } else if (flt->untrimmed_enabled && (((flt->required_r1 & ~r[0].matched_ids) != 0) ||
                                              (paired && (flt->required_r2 & ~r[1].matched_ids) != 0))) {
            dest = CSQ_DEST_UNTRIMMED;
            k->untrimmed++;
        } else {
            dest = CSQ_DEST_TRIMMED;
            k->written++;
            k->written_bp[0] += (uint64_t)r[0].len;
            if (paired) k->written_bp[1] += (uint64_t)r[1].len;
        }
        write_fastq(&b[dest * 2 + 0], &r[0]);
        if (paired) write_fastq(&b[dest * 2 + 1], &r[1]);
        for (int mt_i = 0; mt_i < (paired ? 2 : 1); mt_i++) {
            csq_read_result* res = mt_i ? J->res2 : J->res1;
            if (res) {
                res[i].start = (uint32_t)r[mt_i].orig_off;
                res[i].stop = (uint32_t)(r[mt_i].orig_off + r[mt_i].len);
                res[i].dest = (uint32_t)dest;
                res[i].matched = r[mt_i].matched_ids | (r[mt_i].n_matches ? 0x80000000u : 0u);
            }
            free(r[mt_i].buf_seq);
            free(r[mt_i].buf_qual);
        }
    }
    free(names);
    return NULL;
}

int orc_run_batch(const csq_op* ops1, int n1, const csq_op* ops2, int n2, const csq_filters* flt,
                  const csq_batch_in* in, csq_batch_out* out, csq_read_result* res1, csq_read_result* res2,
                  csq_match* matches1, csq_match* matches2, csq_counters* counters, int n_threads) {
    const int paired = in->n_mates == 2;
    const uint32_t n = in->n_reads;
    if (paired && n1 != n2) return CSQ_ERR_INVALID;
    if (n_threads < 1) n_threads = 1;
    int n_chunks = n_threads;
    if ((uint32_t)n_chunks > n) n_chunks = n ? (int)n : 1;
    orc_buf* bufs = (orc_buf*)calloc((size_t)n_chunks * CSQ_N_DEST * 2, sizeof(orc_buf));
    csq_counters* cnt = (csq_counters*)calloc((size_t)n_chunks, sizeof(csq_counters));
    orc_job* jobs = (orc_job*)calloc((size_t)n_chunks, sizeof(orc_job));
    pthread_t* tids = (pthread_t*)calloc((size_t)n_chunks, sizeof(pthread_t));
    int status = 0;
    for (int c = 0; c < n_chunks; c++) {
        orc_job* J = &jobs[c];
        J->ops1 = ops1; J->ops2 = ops2; J->n1 = n1; J->paired = paired; J->flt = flt; J->in = in;
        J->res1 = res1; J->res2 = res2; J->matches1 = matches1; J->matches2 = matches2; J->n = n;
        J->lo = (uint32_t)((uint64_t)n * (uint64_t)c / (uint64_t)n_chunks);
        J->hi = (uint32_t)((uint64_t)n * (uint64_t)(c + 1) / (uint64_t)n_chunks);
        J->b = bufs + (size_t)c * CSQ_N_DEST * 2;
        J->k = cnt + c;
        if (n_chunks == 1)
            chunk_worker(J);
        else
            pthread_create(&tids[c], NULL, chunk_worker, J);
    }
    for (int c = 0; c < n_chunks; c++) {
        if (n_chunks > 1) pthread_join(tids[c], NULL);
        if (jobs[c].status) status = jobs[c].status;
    }
    free(jobs);
    free(tids);

    /* concatenate chunk outputs in input order */
    for (int d = 0; d < CSQ_N_DEST; d++)
        for (int mt_i = 0; mt_i < 2; mt_i++) {
            uint64_t total = 0, recs = 0;
            for (int c = 0; c < n_chunks; c++) {
                total += bufs[((size_t)c * CSQ_N_DEST + d) * 2 + mt_i].len;
                recs += bufs[((size_t)c * CSQ_N_DEST + d) * 2 + mt_i].records;
            }
            csq_text_out* t = &out->text[d][mt_i];
            t->data = (uint8_t*)malloc(total ? total : 1);
            t->capacity = total;
            t->bytes = total;
            t->records = recs;
            uint64_t pos = 0;
            for (int c = 0; c < n_chunks; c++) {
                orc_buf* bb = &bufs[((size_t)c * CSQ_N_DEST + d) * 2 + mt_i];
                if (bb->len) memcpy(t->data + pos, bb->data, bb->len);
                pos += bb->len;
                free(bb->data);
            }
        }
    if (counters) {
        for (int c = 0; c < n_chunks; c++) {
            uint64_t* dst = (uint64_t*)counters;
            const uint64_t* src = (const uint64_t*)&cnt[c];
            for (size_t w = 0; w < sizeof(csq_counters) / sizeof(uint64_t); w++) dst[w] += src[w];
        }
    }
    free(bufs);
    free(cnt);
    return status;
}

void orc_free(csq_batch_out* out) {
    for (int d = 0; d < CSQ_N_DEST; d++)
        for (int m = 0; m < 2; m++) {
            free(out->text[d][m].data);
            out->text[d][m].data = NULL;
        }
}

int orc_max_threads(void) {
    long n = sysconf(_SC_NPROCESSORS_ONLN);
    return n > 0 ? (int)n : 1;
}
