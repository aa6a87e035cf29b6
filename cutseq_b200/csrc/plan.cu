// Host side of the C ABI: plans (compiled op programs), slots (stream + device buffers),
// batch submit/wait, resident-mode measurement, result accessors.
// Boundary: include/cutseq_b200.h.  Replaces runner.run(pipeline, ...) of reference
// run.py:472-473 / 793-794 for one batch of reads.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include "csq_internal.h"

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CUDA_TRY(expr)                                                                         \
    do {                                                                                       \
        cudaError_t e_ = (expr);                                                               \
        if (e_ != cudaSuccess)                                                                 \
            return fail(e_ == cudaErrorMemoryAllocation ? CSQ_ERR_NOMEM : CSQ_ERR_CUDA, "%s: %s (%s:%d)", #expr, \
                        cudaGetErrorString(e_), __FILE__, __LINE__);                           \
    } while (0)

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return 0;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        // cudaFree / cudaMalloc synchronise the device and stall every stream of the plan: grow rarely (x1.25 and
        // never below 256 KiB, so that the small per-destination buffers do not creep up batch by batch)
        size_t want = bytes + bytes / 4 + (256u << 10);
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) return fail(CSQ_ERR_NOMEM, "cudaMalloc(%zu): %s", want, cudaGetErrorString(e));
        cap = want;
        return 0;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

struct Segment {  // one ALIGN op with the scalar ops in front of it
    AlignParams ap;
    int op_index;
    const char* name;
    const char* pf_name;
};

struct MateProgram {
    std::vector<Segment> segs;
    FinishParams fin;
    uint32_t rename_parts = 0;
    bool has_rename = false, revcomp = false;
    int n_ops = 0;
    std::vector<int> align_slot;  // op index -> index among ALIGN ops, or -1
    int n_align = 0;
};

struct Slot {
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[6] = {};
    DevBuf seq[2], qual[2], seq_off[2], seq_len[2], name[2], name_off[2], state[2], matches[2];
    DevBuf dest, block_tot, block_cnt, block_off, totals, out[CSQ_N_DEST][2];
    DevBuf list[2], list_count[2];  // per mate: prefilter survivors (indices) and their number
    cudaStream_t stream2 = nullptr;  // chain of mate 2
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    // text batches (csq_submit_text): the FASTQ bytes as they came, and the record index k_records builds
    DevBuf text[2], qual_off[2], name_end[2], nl[2], tiles[2], masks[2], parse_misc;  // parse_misc: nl_total[2] (u32) | perr[2] (u64) at +16 | tile ticket[2] (u32) at +32 | any_cr[2] (u32) at +40
    // device gzip writer (CSQ_PLAN_GZIP_OUT): per-member slots, member sizes / offsets, the packed streams
    DevBuf gz_misc, gz_slots, gz_msize, gz_moff, gz_packed;  // gz_misc: hist | codes | hdr | totals
    unsigned long long* gz_totals_host = nullptr;            // pinned: packed bytes per stream
    const uint8_t* gz_packed_ptr[CSQ_N_DEST * 2] = {};
    bool gz_ready = false;                                   // packed streams of the pending batch are on the device
    DevBuf comp[2], gz_idx[2], gz_lines;   // BGZF batches: compressed members, member / text offsets, line ends per member
    int32_t* inflate_status = nullptr;     // device: smallest (error kind + 16 * member), INT_MAX when clean
    uint32_t skip_lines[2] = {0, 0};
    bool bgzf_mode = false;
    uint64_t text_bytes[2] = {0, 0};
    uint64_t first_record = 0;
    bool text_mode = false;
    unsigned long long* totals_host = nullptr;  // pinned: 12 totals + 2 error flags + 2 parse-error keys
    uint32_t n = 0;
    int n_mates = 0;
    csq_batch_out* pending = nullptr;
    bool front_done = false;
    float total_ms = 0, kernel_ms = 0;
    std::vector<std::pair<const char*, float>> ktimes;
};

}  // namespace

struct csq_plan {
    int device = 0;
    uint32_t flags = 0;
    int n_mates = 1;
    MateProgram prog[2];
    csq_filters flt;
    Slot slots[CSQ_N_SLOTS];
    unsigned long long* counters = nullptr;  // device csq_counters
    int* error_flag = nullptr;
    uint32_t* gz_tables = nullptr;           // device: CRC-32 byte table [256] | fold operators [GZ_THREADS]
    uint32_t* crc_check_tables = nullptr;    // device: tables of the member CRC check behind the device inflate [768]
    uint64_t launches = 0;
};

namespace {

// per-kernel timer labels (csq_plan_kernel_times) of the exact aligner and the prefilter of each adapter kind
struct KindLabels {
    int kind;
    const char *align, *prefilter;
};
constexpr KindLabels KIND_LABELS[] = {
    {CSQ_AD_BACK, "k_align(back)", "k_prefilter(back)"},
    {CSQ_AD_BACK_ANYWHERE, "k_align(back,anywhere)", "k_prefilter(back,anywhere)"},
    {CSQ_AD_RIGHTMOST_FRONT, "k_align(rightmost_front)", "k_prefilter(rightmost_front)"},
    {CSQ_AD_PREFIX, "k_align(prefix)", "k_prefilter(prefix)"},
    {CSQ_AD_SUFFIX, "k_align(suffix)", "k_prefilter(suffix)"},
    {CSQ_AD_NI_FRONT, "k_align(noninternal_front)", "k_prefilter(noninternal_front)"},
    {CSQ_AD_NI_BACK, "k_align(noninternal_back)", "k_prefilter(noninternal_back)"},
    {CSQ_AD_FRONT, "k_align(front)", "k_prefilter(front)"},
};

KindLabels kind_labels(int kind) {
    for (const KindLabels& l : KIND_LABELS)
        if (l.kind == kind) return l;
    return {kind, "k_align", "k_prefilter"};
}

// csq_op(ALIGN) -> aligner parameters (SingleAdapter.__init__ / _make_aligner of adapters.py)
int build_align(const csq_op& op, AlignParams& ap) {
    memset(&ap, 0, sizeof(ap));
    const int m = op.adapter_len;
    if (m < 1 || m > CSQ_MAX_ADAPTER) return fail(CSQ_ERR_LIMIT, "adapter length %d outside 1..%d", m, CSQ_MAX_ADAPTER);
    int flags, reversed = 0, front = 0;
    switch (op.adapter_kind) {
        case CSQ_AD_BACK: flags = 14; break;
        case CSQ_AD_BACK_ANYWHERE: flags = 15; break;
        case CSQ_AD_RIGHTMOST_FRONT: flags = 14; reversed = 1; front = 1; break;
        case CSQ_AD_PREFIX: flags = 8; front = 1; break;
        case CSQ_AD_SUFFIX: flags = 2; break;
        case CSQ_AD_NI_FRONT: flags = 9; front = 1; break;
        case CSQ_AD_NI_BACK: flags = 6; break;
        case CSQ_AD_FRONT: flags = 11; front = 1; break;
        default: return fail(CSQ_ERR_INVALID, "unknown adapter kind %d", op.adapter_kind);
    }
    double rate = op.max_error_rate;
    if (rate >= 1.0) rate /= m;  // an absolute error count (SingleAdapter.__init__)
    if (!(rate >= 0.0)) return fail(CSQ_ERR_INVALID, "bad max_error_rate");
    int mo = op.min_overlap < m ? op.min_overlap : m;
    if (op.adapter_kind == CSQ_AD_PREFIX || op.adapter_kind == CSQ_AD_SUFFIX) mo = m;
    if (mo < 1) return fail(CSQ_ERR_INVALID, "min_overlap must be >= 1");
    ap.m = m;
    ap.flags = flags;
    ap.reversed = reversed;
    ap.trim_front = front;
    ap.min_overlap = mo;
    ap.k = (int)(rate * m);
    // bit 31 of the matched set means "any adapter matched"
    if (op.adapter_id < -1 || op.adapter_id > 30) return fail(CSQ_ERR_INVALID, "adapter_id %d outside -1..30", op.adapter_id);
    ap.adapter_bit = op.adapter_id;
    for (int L = 0; L <= m; L++) {
        // largest integer cost with cost <= L * rate in IEEE double, as Aligner.locate compares
        double lim = L * rate;
        int t = (int)floor(lim);
        if (t > 255) t = 255;
        ap.thr[L] = (uint8_t)t;
    }
    bool homo = true;
    for (int i = 0; i < m; i++) {
        char c = op.adapter[reversed ? (m - 1 - i) : i];
        if (c >= 'a' && c <= 'z') c = (char)(c - 32);
        if (c == 'U') c = 'T';
        int li = c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : -1;
        if (li < 0) return fail(CSQ_ERR_INVALID, "adapter character '%c' is not one of ACGT", c);
        ap.peq[li][i >> 5] |= 1u << (i & 31);
        if (i == 0) ap.letter = (uint8_t)c;
        if ((uint8_t)c != ap.letter) homo = false;
    }
    ap.homopolymer = homo ? 1 : 0;
    return 0;
}

int build_mate_program(const csq_op* ops, int n, int mate, MateProgram& mp) {
    if (n < 0 || n > CSQ_MAX_OPS) return fail(CSQ_ERR_INVALID, "program of %d ops (max %d)", n, CSQ_MAX_OPS);
    mp = MateProgram();
    mp.n_ops = n;
    mp.align_slot.assign(n, -1);
    memset(&mp.fin, 0, sizeof(mp.fin));
    mp.fin.mate = mate;
    std::vector<DevOp> pending;
    bool seen_qtrim = false;
    for (int t = 0; t < n; t++) {
        const csq_op& op = ops[t];
        if (seen_qtrim && op.kind != CSQ_OP_REVCOMP)
            return fail(CSQ_ERR_INVALID, "op %d: only REVCOMP may follow QTRIM", t);
        switch (op.kind) {
            case CSQ_OP_STRIP_SUFFIX:
                if (mp.has_rename) return fail(CSQ_ERR_INVALID, "op %d: STRIP_SUFFIX must come before RENAME", t);
                if (mp.fin.n_suffix >= 4 || op.suffix_len < 0 || op.suffix_len > CSQ_MAX_SUFFIX)
                    return fail(CSQ_ERR_INVALID, "op %d: too many / too long name suffixes", t);
                // SuffixRemover("") would empty every name (name[:-0]); nothing implements that, so it is refused
                if (op.suffix_len == 0) return fail(CSQ_ERR_INVALID, "op %d: empty name suffix", t);
                mp.fin.suffix_len[mp.fin.n_suffix] = op.suffix_len;
                memcpy(mp.fin.suffix[mp.fin.n_suffix], op.suffix, (size_t)op.suffix_len);
                mp.fin.n_suffix++;
                break;
            case CSQ_OP_CUT:
            case CSQ_OP_COND_CUT:
            case CSQ_OP_RENAME: {
                DevOp d = {op.kind, op.length, op.force_trim_min_length, op.rename_parts};
                if (op.kind == CSQ_OP_RENAME) {
                    if (mp.has_rename) return fail(CSQ_ERR_INVALID, "op %d: more than one RENAME", t);
                    mp.has_rename = true;
                    mp.rename_parts = op.rename_parts;
                }
                if (op.kind != CSQ_OP_RENAME && (op.length > 65535 || op.length < -65535))
                    return fail(CSQ_ERR_INVALID, "op %d: cut length out of range", t);
                pending.push_back(d);
                if (pending.size() > CSQ_MAX_PRE) return fail(CSQ_ERR_INVALID, "more than %d scalar ops in a row", CSQ_MAX_PRE);
                break;
            }
            case CSQ_OP_ALIGN: {
                Segment s;
                int rc = build_align(op, s.ap);
                if (rc) return rc;
                s.op_index = t;
                const KindLabels labels = kind_labels(op.adapter_kind);
                s.name = labels.align;
                s.pf_name = labels.prefilter;
                s.ap.n_pre = (int)pending.size();
                for (size_t q = 0; q < pending.size(); q++) s.ap.pre[q] = pending[q];
                pending.clear();
                s.ap.first = mp.segs.empty() ? 1 : 0;
                s.ap.counter_index = CNT_WITH_ADAPTERS + mate * CSQ_MAX_OPS + t;
                s.ap.adjacent_index = (mp.segs.empty() && !s.ap.trim_front) ? CNT_ADJACENT + mate * 6 : -1;
                mp.align_slot[t] = mp.n_align++;
                mp.segs.push_back(s);
                break;
            }
            case CSQ_OP_QTRIM:
                seen_qtrim = true;
                mp.fin.has_qtrim = 1;
                mp.fin.cutoff_front = op.cutoff_front;
                mp.fin.cutoff_back = op.cutoff_back;
                mp.fin.qbase = op.quality_base;
                break;
            case CSQ_OP_REVCOMP:
                if (t != n - 1) return fail(CSQ_ERR_INVALID, "REVCOMP must be the last op");
                mp.revcomp = true;
                break;
            default: return fail(CSQ_ERR_INVALID, "op %d: unknown kind %d", t, op.kind);
        }
    }
    mp.fin.n_post = (int)pending.size();
    for (size_t q = 0; q < pending.size(); q++) mp.fin.post[q] = pending[q];
    mp.fin.first = mp.segs.empty() ? 1 : 0;
    mp.fin.has_rename = mp.has_rename ? 1 : 0;
    return 0;
}

int check_device(int device) {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(CSQ_ERR_NO_DEVICE, "no CUDA device available (%s); this library has no CPU fallback",
                    e == cudaSuccess ? "count is 0" : cudaGetErrorString(e));
    if (device < 0 || device >= count) return fail(CSQ_ERR_NO_DEVICE, "device %d out of range (0..%d)", device, count - 1);
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail(CSQ_ERR_NO_DEVICE, "device %d is sm_%d%d; this build targets sm_100a (B200) only", device, prop.major, prop.minor);
    return 0;
}

// readable bytes in front of and behind every device pool: the 16-byte fetches of k_emit_rec / k_prefilter may
// start up to 15 bytes below a piece and end up to 19 bytes behind it
constexpr size_t TEXT_FRONT_PAD = 64, POOL_PAD = 64;

MateDev mate_dev(Slot& s, int m) {
    MateDev d;
    d.seq_off = (const uint32_t*)s.seq_off[m].p;
    d.seq_len = (const uint32_t*)s.seq_len[m].p;
    d.name_off = (const uint32_t*)s.name_off[m].p;
    d.state = (ReadState*)s.state[m].p;
    if (s.text_mode) {
        d.seq = d.qual = d.name = (const uint8_t*)s.text[m].p + TEXT_FRONT_PAD;
        d.qual_off = (const uint32_t*)s.qual_off[m].p;
        d.name_end = (const uint32_t*)s.name_end[m].p;
    } else {
        d.seq = (const uint8_t*)s.seq[m].p + POOL_PAD;
        d.qual = (const uint8_t*)s.qual[m].p + POOL_PAD;
        d.name = (const uint8_t*)s.name[m].p + POOL_PAD;
        d.qual_off = d.seq_off;
        d.name_end = d.name_off + 1;
    }
    return d;
}

int validate_batch(const csq_plan* plan, const csq_batch_in* in) {
    if (!in) return fail(CSQ_ERR_INVALID, "null batch");
    if ((int)in->n_mates != plan->n_mates) return fail(CSQ_ERR_INVALID, "batch has %u mates, plan has %d", in->n_mates, plan->n_mates);
    for (int m = 0; m < plan->n_mates; m++) {
        const csq_mate_in& mi = in->mate[m];
        if (in->n_reads && (!mi.seq || !mi.qual || !mi.seq_off || !mi.seq_len || !mi.name || !mi.name_off))
            return fail(CSQ_ERR_INVALID, "mate %d: null array (FASTA input without qualities is not supported)", m + 1);
        if (mi.seq_bytes >= (1ull << 32) || mi.name_bytes >= (1ull << 32)) return fail(CSQ_ERR_LIMIT, "batch pools must stay below 4 GiB");
        uint32_t mx = 0;
        for (uint32_t i = 0; i < in->n_reads; i++) mx = mi.seq_len[i] > mx ? mi.seq_len[i] : mx;
        if (mx > CSQ_MAX_READ_LEN) return fail(CSQ_ERR_LIMIT, "mate %d: read of %u bases exceeds the supported %d", m + 1, mx, CSQ_MAX_READ_LEN);
        // the id fields of the per-read state are 16 bits wide (the text path checks the same in k_tail)
        for (uint32_t i = 0; i < in->n_reads; i++)
            if (mi.name_off[i + 1] - mi.name_off[i] > 65535u)
                return fail(CSQ_ERR_LIMIT, "mate %d: header of record %u (%u bytes) exceeds the supported 65535 bytes", m + 1, i,
                            mi.name_off[i + 1] - mi.name_off[i]);
    }
    return 0;
}

int ensure_common(csq_plan* plan, Slot& s, uint32_t n) {
    const uint32_t nblk = (n + CSQ_PAIR_BLOCK - 1) / CSQ_PAIR_BLOCK;
    int rc;
    if ((rc = s.dest.ensure((size_t)n + 16))) return rc;
    if ((rc = s.block_tot.ensure((size_t)nblk * 32 + 32))) return rc;
    if ((rc = s.block_cnt.ensure((size_t)nblk * 16 + 16))) return rc;
    if ((rc = s.block_off.ensure((size_t)nblk * 64 + 64))) return rc;
    if ((rc = s.totals.ensure(16 * 8))) return rc;
    if (!(plan->flags & CSQ_PLAN_NO_PREFILTER)) {
        for (int m = 0; m < plan->n_mates; m++) {
            if ((rc = s.list[m].ensure((size_t)n * CSQ_PF_BINS * 6 + 64))) return rc;
            if ((rc = s.list_count[m].ensure(4 * CSQ_PF_BINS + 16))) return rc;
        }
    }
    return 0;
}

// Per-mate arrays of a text batch of n records and `bytes` bytes of text: the record index the parse kernels build,
// the read states and the kept match records.
int ensure_text_index(csq_plan* plan, Slot& s, int m, uint32_t n, uint64_t bytes) {
    int rc;
    if ((rc = s.seq_off[m].ensure((size_t)n * 4 + 16))) return rc;
    if ((rc = s.qual_off[m].ensure((size_t)n * 4 + 16))) return rc;
    if ((rc = s.seq_len[m].ensure((size_t)n * 4 + 16))) return rc;
    if ((rc = s.name_off[m].ensure((size_t)n * 4 + 16))) return rc;
    if ((rc = s.name_end[m].ensure((size_t)n * 4 + 16))) return rc;
    if ((rc = s.nl[m].ensure(((size_t)n * 4 + 8) * 4))) return rc;
    if ((rc = s.masks[m].ensure(((size_t)csq_parse_tiles(bytes) + 1) * 2048))) return rc;  // 16 bits per 16-byte chunk
    if ((rc = s.tiles[m].ensure(((size_t)csq_parse_tiles(bytes) + 4) * 8))) return rc;
    if ((rc = s.state[m].ensure((size_t)n * sizeof(ReadState) + 32))) return rc;
    if ((plan->flags & CSQ_PLAN_KEEP_MATCHES) && plan->prog[m].n_align)
        if ((rc = s.matches[m].ensure((size_t)n * plan->prog[m].n_align * sizeof(csq_match) + 16))) return rc;
    return 0;
}

// FASTQ text of a batch -> device, as it is; the record index is built by the parse kernels in enqueue_front
int upload_text(csq_plan* plan, Slot& s, const csq_batch_text* in) {
    const uint32_t n = in->n_reads;
    s.n = n;
    s.n_mates = plan->n_mates;
    s.front_done = false;
    s.text_mode = true;
    s.bgzf_mode = false;
    s.first_record = in->first_record;
    int rc;
    for (int m = 0; m < plan->n_mates; m++) {
        const uint64_t bytes = in->mate[m].bytes;
        s.text_bytes[m] = bytes;
        const size_t padded = (size_t)((bytes + 63) & ~(uint64_t)63);
        if ((rc = s.text[m].ensure(TEXT_FRONT_PAD + padded + 128))) return rc;
        if ((rc = ensure_text_index(plan, s, m, n, bytes))) return rc;
        uint8_t* base = (uint8_t*)s.text[m].p;
        CUDA_TRY(cudaMemsetAsync(base, 0, TEXT_FRONT_PAD, s.stream));
        // zero padding behind the text: never a line end, and readable by the 128-bit walks
        CUDA_TRY(cudaMemsetAsync(base + TEXT_FRONT_PAD + (bytes & ~(uint64_t)63), 0, padded - (bytes & ~(uint64_t)63) + 128, s.stream));
        if (bytes) CUDA_TRY(cudaMemcpyAsync(base + TEXT_FRONT_PAD, in->mate[m].text, bytes, cudaMemcpyHostToDevice, s.stream));
    }
    if ((rc = s.parse_misc.ensure(64))) return rc;
    return ensure_common(plan, s, n);
}

// One mate's BGZF members -> device, inflated into the slot's text buffer (k_gz_inflate, one warp per member; k_gz_check: CRC-32 and line ends).
// lines_dev != nullptr: also the line ends per member.  The text buffer is laid out as for csq_submit_text.
int inflate_mate(csq_plan* plan, Slot& s, int m, const csq_bgzf_in& bi, uint32_t* lines_dev, cudaStream_t st) {
    if (bi.n_members && (!bi.data || !bi.member_off || !bi.text_off)) return fail(CSQ_ERR_INVALID, "mate %d: null BGZF arrays", m + 1);
    const uint32_t nm = bi.n_members;
    const uint64_t text_bytes = nm ? bi.text_off[nm] : 0, comp_bytes = nm ? bi.member_off[nm] : 0;
    if (comp_bytes > bi.bytes) return fail(CSQ_ERR_INVALID, "mate %d: member offsets run past the data", m + 1);
    if (text_bytes + 1 >= (1ull << 32) - 4096 || comp_bytes >= (1ull << 32)) return fail(CSQ_ERR_LIMIT, "batch text must stay below 4 GiB");
    const uint64_t bytes = text_bytes + (bi.append_newline ? 1 : 0);
    s.text_bytes[m] = bytes;
    const size_t padded = (size_t)((bytes + 63) & ~(uint64_t)63);
    int rc;
    if ((rc = s.text[m].ensure(TEXT_FRONT_PAD + padded + 128))) return rc;
    if ((rc = s.comp[m].ensure((size_t)comp_bytes + 64))) return rc;
    if ((rc = s.gz_idx[m].ensure(((size_t)nm + 1) * 8 + 16))) return rc;
    uint8_t* base = (uint8_t*)s.text[m].p;
    uint32_t* moff = (uint32_t*)s.gz_idx[m].p;
    uint32_t* ooff = moff + nm + 1;
    CUDA_TRY(cudaMemsetAsync(base, 0, TEXT_FRONT_PAD, st));
    CUDA_TRY(cudaMemsetAsync(base + TEXT_FRONT_PAD + (bytes & ~(uint64_t)63), 0, padded - (bytes & ~(uint64_t)63) + 128, st));
    if (nm) {
        CUDA_TRY(cudaMemcpyAsync(s.comp[m].p, bi.data, comp_bytes, cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemsetAsync((uint8_t*)s.comp[m].p + comp_bytes, 0, 64, st));
        CUDA_TRY(cudaMemcpyAsync(moff, bi.member_off, ((size_t)nm + 1) * 4, cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(ooff, bi.text_off, ((size_t)nm + 1) * 4, cudaMemcpyHostToDevice, st));
        InflateParams ip;
        ip.comp = (const uint8_t*)s.comp[m].p;
        ip.moff = moff;
        ip.ooff = ooff;
        ip.n_members = nm;
        ip.out = base + TEXT_FRONT_PAD;
        ip.lines = lines_dev;
        ip.status = s.inflate_status;
        ip.crc_tables = plan->crc_check_tables;
        CUDA_TRY(csq_launch_inflate(ip, st));
        plan->launches += 1;
    }
    if (bi.append_newline) CUDA_TRY(cudaMemsetAsync(base + TEXT_FRONT_PAD + text_bytes, '\n', 1, st));
    return 0;
}

int upload_bgzf(csq_plan* plan, Slot& s, const csq_batch_bgzf* in) {
    const uint32_t n = in->n_reads;
    s.n = n;
    s.n_mates = plan->n_mates;
    s.front_done = false;
    s.text_mode = true;
    s.bgzf_mode = true;
    s.first_record = in->first_record;
    int rc;
    CUDA_TRY(cudaMemsetAsync(s.inflate_status, 0x7F, sizeof(int32_t), s.stream));
    for (int m = 0; m < plan->n_mates; m++) {
        s.skip_lines[m] = in->mate[m].skip_lines;
        if ((rc = inflate_mate(plan, s, m, in->mate[m], nullptr, s.stream))) return rc;
        if ((rc = ensure_text_index(plan, s, m, n, s.text_bytes[m]))) return rc;
    }
    CUDA_TRY(cudaMemcpyAsync(s.totals_host + 16, s.inflate_status, sizeof(int32_t), cudaMemcpyDeviceToHost, s.stream));
    if ((rc = s.parse_misc.ensure(64))) return rc;
    return ensure_common(plan, s, n);
}

int upload(csq_plan* plan, Slot& s, const csq_batch_in* in) {
    const uint32_t n = in->n_reads;
    s.n = n;
    s.n_mates = plan->n_mates;
    s.front_done = false;
    s.text_mode = false;
    s.bgzf_mode = false;
    for (int m = 0; m < plan->n_mates; m++) {
        const csq_mate_in& mi = in->mate[m];
        int rc;
        if ((rc = s.seq[m].ensure(mi.seq_bytes + 2 * POOL_PAD))) return rc;
        if ((rc = s.qual[m].ensure(mi.seq_bytes + 2 * POOL_PAD))) return rc;
        if ((rc = s.seq_off[m].ensure((size_t)n * 4 + 4))) return rc;
        if ((rc = s.seq_len[m].ensure((size_t)n * 4 + 4))) return rc;
        if ((rc = s.name[m].ensure(mi.name_bytes + 2 * POOL_PAD))) return rc;
        if ((rc = s.name_off[m].ensure(((size_t)n + 1) * 4))) return rc;
        if ((rc = s.state[m].ensure((size_t)n * sizeof(ReadState) + 32))) return rc;
        if ((plan->flags & CSQ_PLAN_KEEP_MATCHES) && plan->prog[m].n_align)
            if ((rc = s.matches[m].ensure((size_t)n * plan->prog[m].n_align * sizeof(csq_match) + 16))) return rc;
        if (n) {
            // the padding is read (and masked off) by the 16-byte fetches: keep it defined
            for (DevBuf* b : {&s.seq[m], &s.qual[m]}) {
                CUDA_TRY(cudaMemsetAsync(b->p, 0, POOL_PAD, s.stream));
                CUDA_TRY(cudaMemsetAsync((uint8_t*)b->p + POOL_PAD + mi.seq_bytes, 0, POOL_PAD, s.stream));
            }
            CUDA_TRY(cudaMemsetAsync(s.name[m].p, 0, POOL_PAD, s.stream));
            CUDA_TRY(cudaMemsetAsync((uint8_t*)s.name[m].p + POOL_PAD + mi.name_bytes, 0, POOL_PAD, s.stream));
            CUDA_TRY(cudaMemcpyAsync((uint8_t*)s.seq[m].p + POOL_PAD, mi.seq, mi.seq_bytes, cudaMemcpyHostToDevice, s.stream));
            CUDA_TRY(cudaMemcpyAsync((uint8_t*)s.qual[m].p + POOL_PAD, mi.qual, mi.seq_bytes, cudaMemcpyHostToDevice, s.stream));
            CUDA_TRY(cudaMemcpyAsync(s.seq_off[m].p, mi.seq_off, (size_t)n * 4, cudaMemcpyHostToDevice, s.stream));
            CUDA_TRY(cudaMemcpyAsync(s.seq_len[m].p, mi.seq_len, (size_t)n * 4, cudaMemcpyHostToDevice, s.stream));
            CUDA_TRY(cudaMemcpyAsync((uint8_t*)s.name[m].p + POOL_PAD, mi.name, mi.name_bytes, cudaMemcpyHostToDevice, s.stream));
            CUDA_TRY(cudaMemcpyAsync(s.name_off[m].p, mi.name_off, ((size_t)n + 1) * 4, cudaMemcpyHostToDevice, s.stream));
        }
    }
    return ensure_common(plan, s, n);
}

struct KernelTimer {  // optional per-kernel CUDA-event timing (resident mode, last iteration)
    bool on = false;
    cudaStream_t stream;
    std::vector<cudaEvent_t> evs;
    std::vector<const char*> names;
    void mark(const char* name) {
        if (!on) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, stream);
        evs.push_back(e);
        names.push_back(name);
    }
};

PairParams pair_params(csq_plan* plan, Slot& s) {
    PairParams pp;
    memset(&pp, 0, sizeof(pp));
    for (int m = 0; m < plan->n_mates; m++) pp.md[m] = mate_dev(s, m);
    pp.n = s.n;
    pp.n_mates = plan->n_mates;
    pp.min_length = plan->flt.min_length;
    pp.untrimmed_enabled = plan->flt.untrimmed_enabled;
    pp.required[0] = plan->flt.required_r1;
    pp.required[1] = plan->flt.required_r2;
    pp.rename_parts = plan->prog[0].rename_parts;
    pp.check_ids = (plan->n_mates == 2 && plan->prog[0].has_rename) ? 1 : 0;
    pp.revcomp = plan->prog[0].revcomp ? 1 : 0;
    pp.dest = (uint8_t*)s.dest.p;
    pp.block_tot = (uint32_t*)s.block_tot.p;
    pp.block_cnt = (uint32_t*)s.block_cnt.p;
    pp.counters = plan->counters;
    pp.error_flag = plan->error_flag;
    return pp;
}

// One mate of a batch: parse (text batches), then prefilter / align per ALIGN op - all on `st` (k_tail follows for both mates).
int enqueue_mate(csq_plan* plan, Slot& s, int m, KernelTimer* kt, cudaStream_t st) {
    const uint32_t n = s.n;
    if (s.text_mode) {
        // FASTQ text -> record index (parse.cu); nl_total[m] at parse_misc + 4 m, perr[m] at parse_misc + 16 + 8 m
        ParseParams pp;
        pp.text = (const uint8_t*)s.text[m].p + TEXT_FRONT_PAD;
        pp.bytes = s.text_bytes[m];
        pp.n = n;
        pp.nl = (uint32_t*)s.nl[m].p;
        pp.nl_total = (uint32_t*)s.parse_misc.p + m;
        pp.seq_off = (uint32_t*)s.seq_off[m].p;
        pp.qual_off = (uint32_t*)s.qual_off[m].p;
        pp.seq_len = (uint32_t*)s.seq_len[m].p;
        pp.name_off = (uint32_t*)s.name_off[m].p;
        pp.name_end = (uint32_t*)s.name_end[m].p;
        pp.perr = (unsigned long long*)((uint8_t*)s.parse_misc.p + 16) + m;
        pp.any_cr = (uint32_t*)((uint8_t*)s.parse_misc.p + 40) + m;
        pp.skip = s.bgzf_mode ? s.skip_lines[m] : 0u;
        pp.first_off = s.bgzf_mode ? (uint32_t*)((uint8_t*)s.parse_misc.p + 48) + m : nullptr;
        CUDA_TRY(csq_launch_parse(pp, s.tiles[m].p, (uint16_t*)s.masks[m].p, st));
        plan->launches += csq_parse_tiles(pp.bytes) ? 4 : 1;
        if (kt) kt->mark(m == 0 ? "k_parse.r1" : "k_parse.r2");
    }
    MateProgram& mp = plan->prog[m];
    for (Segment& sg : mp.segs) {
        AlignParams ap = sg.ap;
        ap.exact_stop = (plan->flags & CSQ_PLAN_NO_EXACT_STOP) ? 0 : 1;
        ap.one = 1u;
        ap.md = mate_dev(s, m);
        ap.n = n;
        ap.list = nullptr;
        ap.list_count = nullptr;
        ap.count_cells = 1;
        ap.counters = plan->counters;
        ap.matches = (plan->flags & CSQ_PLAN_KEEP_MATCHES)
                         ? (csq_match*)s.matches[m].p + (size_t)mp.align_slot[sg.op_index] * n
                         : nullptr;
        if (!(plan->flags & CSQ_PLAN_NO_PREFILTER) && n) {
            // reject-only bit-parallel filter; the exact DP then runs on the compacted survivors
            CUDA_TRY(cudaMemsetAsync(s.list_count[m].p, 0, 4 * CSQ_PF_BINS, st));
            CUDA_TRY(csq_launch_prefilter(ap, (uint32_t*)s.list[m].p, (uint32_t*)s.list_count[m].p, st));
            plan->launches += 1;
            if (kt) kt->mark(sg.pf_name);
            ap.list = (const uint32_t*)s.list[m].p;
            ap.list_count = (const uint32_t*)s.list_count[m].p;
            ap.first = 0;   // the prefilter initialised the state and ran the scalar ops
            ap.n_pre = 0;
            ap.count_cells = 0;
        }
        CUDA_TRY(csq_launch_align(ap, n, st));
        plan->launches += n ? 1 : 0;
        if (kt) kt->mark(sg.name);
    }
    return 0;
}

// parse ... scan, then the 12 totals + error flags to pinned host memory.
// The two mates of a pair do not meet before k_pair: with a second stream (`st2`, nullptr = off) the chain of
// mate 2 runs beside the chain of mate 1, so that the single-CTA scans and the register-bound k_align<100>
// (2 CTAs per SM) of one mate share the machine with the other mate's kernels.  Per-kernel event timing
// (`kt`) keeps everything on one stream.
int enqueue_front(csq_plan* plan, Slot& s, KernelTimer* kt, cudaStream_t st, cudaStream_t st2 = nullptr) {
    const uint32_t n = s.n;
    const uint32_t nblk = (n + CSQ_PAIR_BLOCK - 1) / CSQ_PAIR_BLOCK;
    const bool dual = st2 != nullptr && !kt && plan->n_mates == 2 && n > 0 && !(plan->flags & CSQ_PLAN_ONE_STREAM);
    int rc;
    if (kt) kt->mark("begin");
    if (s.text_mode) CUDA_TRY(cudaMemsetAsync((uint8_t*)s.parse_misc.p + 16, 0xFF, 16, st));
    if (dual) {
        CUDA_TRY(cudaEventRecord(s.ev_fork, st));
        CUDA_TRY(cudaStreamWaitEvent(st2, s.ev_fork, 0));
    }
    for (int m = 0; m < plan->n_mates; m++)
        if ((rc = enqueue_mate(plan, s, m, kt, (dual && m == 1) ? st2 : st))) return rc;
    if (dual) {
        CUDA_TRY(cudaEventRecord(s.ev_join, st2));
        CUDA_TRY(cudaStreamWaitEvent(st, s.ev_join, 0));
    }
    PairParams pp = pair_params(plan, s);
    FinishParams fp[2];
    for (int m = 0; m < 2; m++) {
        fp[m] = plan->prog[m < plan->n_mates ? m : 0].fin;
        fp[m].md = mate_dev(s, m < plan->n_mates ? m : 0);
        fp[m].n = n;
        fp[m].counters = plan->counters;
        fp[m].perr = s.text_mode ? (unsigned long long*)((uint8_t*)s.parse_misc.p + 16) + m : nullptr;
    }
    CUDA_TRY(csq_launch_tail(fp[0], fp[1], pp, st));
    plan->launches += n ? 1 : 0;
    if (kt) kt->mark("k_tail");
    if (s.text_mode)  // parse errors: k_records' and k_tail's ('@' / '+' line starts)
        CUDA_TRY(cudaMemcpyAsync(s.totals_host + 14, (uint8_t*)s.parse_misc.p + 16, 16, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(csq_launch_scan(nblk, (const uint32_t*)s.block_tot.p, (const uint32_t*)s.block_cnt.p,
                             (unsigned long long*)s.block_off.p, (unsigned long long*)s.totals.p, st));
    plan->launches += 1;
    if (kt) kt->mark("k_scan");
    CUDA_TRY(cudaMemcpyAsync(s.totals_host, s.totals.p, 12 * 8, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(s.totals_host + 12, plan->error_flag, sizeof(int), cudaMemcpyDeviceToHost, st));
    s.front_done = true;
    return 0;
}

int size_outputs(Slot& s) {
    for (int d = 0; d < CSQ_N_DEST; d++)
        for (int m = 0; m < 2; m++) {
            int rc = s.out[d][m].ensure((size_t)s.totals_host[d * 2 + m] + 64);
            if (rc) return rc;
        }
    return 0;
}

int enqueue_emit(csq_plan* plan, Slot& s, KernelTimer* kt, cudaStream_t st) {
    EmitParams ep;
    memset(&ep, 0, sizeof(ep));
    ep.pp = pair_params(plan, s);
    ep.block_off = (const unsigned long long*)s.block_off.p;
    for (int d = 0; d < CSQ_N_DEST; d++)
        for (int m = 0; m < 2; m++) ep.out[d][m] = (uint8_t*)s.out[d][m].p;
    // default: staged through shared memory; the direct kernels stay for A/B runs and for the reverse-complementing sink
    if ((plan->flags & CSQ_PLAN_EMIT_G16) || ep.pp.revcomp)
        CUDA_TRY(csq_launch_emit(ep, st));
    else
        CUDA_TRY(csq_launch_emit_stage(ep, st));
    plan->launches += s.n ? 1 : 0;
    if (kt) kt->mark("k_emit");
    return 0;
}

// Device gzip writer behind the emitter (CSQ_PLAN_GZIP_OUT): the six text streams of the slot -> packed BGZF members;
// the packed sizes go to pinned host memory.  Layout of gz_misc: hist [6][256] | codes [6][260] | hdr [6][100] | totals [8] (u64).
int enqueue_gz(csq_plan* plan, Slot& s, KernelTimer* kt, cudaStream_t st) {
    GzParams gp;
    memset(&gp, 0, sizeof(gp));
    uint32_t members = 0;
    size_t packed_cap = 0;
    size_t packed_off[CSQ_N_DEST * 2];
    for (int d = 0; d < CSQ_N_DEST; d++)
        for (int m = 0; m < 2; m++) {
            const int i = d * 2 + m;
            const uint64_t bytes = m < s.n_mates ? s.totals_host[i] : 0;
            gp.text[i] = (const uint8_t*)s.out[d][m].p;
            gp.bytes[i] = bytes;
            gp.first_member[i] = members;
            const uint32_t k = (uint32_t)((bytes + GZ_PIECE - 1) / GZ_PIECE);
            members += k;
            packed_off[i] = packed_cap;
            packed_cap += (size_t)((bytes + 32ull * k + 63) & ~(uint64_t)63);  // a stored piece grows by 31 bytes
        }
    gp.first_member[CSQ_N_DEST * 2] = members;
    int rc;
    const size_t misc_words = 6 * 256 + 6 * GZ_CODE_STRIDE + 6 * GZ_HDR_STRIDE;
    if ((rc = s.gz_misc.ensure(misc_words * 4 + 8 * 8))) return rc;
    if ((rc = s.gz_slots.ensure((size_t)members * GZ_SLOT + 64))) return rc;
    if ((rc = s.gz_msize.ensure((size_t)members * 4 + 16))) return rc;
    if ((rc = s.gz_moff.ensure((size_t)members * 8 + 16))) return rc;
    if ((rc = s.gz_packed.ensure(packed_cap + 64))) return rc;
    uint32_t* misc = (uint32_t*)s.gz_misc.p;
    gp.hist = misc;
    gp.codes = misc + 6 * 256;
    gp.hdr = gp.codes + 6 * GZ_CODE_STRIDE;
    gp.totals = (unsigned long long*)(misc + misc_words);
    gp.crc_tab = plan->gz_tables;
    gp.crc_pow = plan->gz_tables + 256;
    gp.slots = (uint8_t*)s.gz_slots.p;
    gp.msize = (uint32_t*)s.gz_msize.p;
    gp.moff = (unsigned long long*)s.gz_moff.p;
    for (int i = 0; i < CSQ_N_DEST * 2; i++) gp.packed[i] = (uint8_t*)s.gz_packed.p + packed_off[i];
    CUDA_TRY(cudaMemsetAsync(gp.totals, 0, 8 * 8, st));
    CUDA_TRY(csq_launch_gz(gp, members, st));
    plan->launches += members ? 5 : 0;
    if (kt) kt->mark("k_gz");
    CUDA_TRY(cudaMemcpyAsync(s.gz_totals_host, gp.totals, 8 * 8, cudaMemcpyDeviceToHost, st));
    for (int i = 0; i < CSQ_N_DEST * 2; i++) s.gz_packed_ptr[i] = gp.packed[i];
    return 0;
}

// FASTQ format errors found by k_records, worded like dnaio's FastqFormatError
int check_parse_error(Slot& s) {
    if (!s.text_mode) return 0;
    if (s.bgzf_mode) {
        const int32_t st = *(const int32_t*)(s.totals_host + 16);
        if (st != 0x7F7F7F7F)
            return fail(CSQ_ERR_IO, "corrupt BGZF member %d of the batch (%s)", st / 16, st % 16 == 7 ? "CRC-32 mismatch" : "invalid DEFLATE data");
    }
    for (int m = 0; m < s.n_mates; m++) {
        const unsigned long long key = s.totals_host[14 + m];
        if (key == ~0ULL) continue;
        const unsigned long long rec = key >> 3, line = 4 * (s.first_record + rec);
        switch ((int)(key & 7)) {
            case 1: return fail(CSQ_ERR_FORMAT, "input file %d: line %llu is expected to start with '@'", m + 1, line + 1);
            case 2: return fail(CSQ_ERR_FORMAT, "input file %d: line %llu is expected to start with '+'", m + 1, line + 3);
            case 3: return fail(CSQ_ERR_FORMAT, "input file %d: length of sequence and qualities differ (record at line %llu)", m + 1, line + 1);
            case 4: return fail(CSQ_ERR_LIMIT, "input file %d: read at line %llu exceeds the supported %d bases", m + 1, line + 1, CSQ_MAX_READ_LEN);
            case 6:
                return fail(CSQ_ERR_FORMAT, "input file %d: sequence descriptions don't match at line %llu (the second description must be empty or equal to the first)",
                            m + 1, line + 3);
            case 7: return fail(CSQ_ERR_LIMIT, "input file %d: header at line %llu exceeds the supported 65535 bytes", m + 1, line + 1);
            default: return fail(CSQ_ERR_FORMAT, "input file %d: the batch does not hold %u whole FASTQ records (4 lines each)", m + 1, s.n);
        }
    }
    return 0;
}

int check_device_error(Slot& s, int word = 12) {
    if (word == 12) {
        int rc = check_parse_error(s);
        if (rc) return rc;
    }
    int flag = *(int*)(s.totals_host + word);
    if (flag == CSQ_ERR_PAIRING) return fail(CSQ_ERR_PAIRING, "Input read IDs not identical in a pair");
    if (flag) return fail(flag, "device reported error %d", flag);
    return 0;
}

}  // namespace

void csq_set_error(const char* msg) { snprintf(g_err, sizeof(g_err), "%s", msg ? msg : ""); }

extern "C" {

int csq_abi_version(void) { return CSQ_ABI_VERSION; }

const char* csq_last_error(void) { return g_err; }

int csq_device_count(int* count) {
    if (!count) return fail(CSQ_ERR_INVALID, "null argument");
    int c = 0;
    cudaError_t e = cudaGetDeviceCount(&c);
    if (e != cudaSuccess) {
        *count = 0;
        return fail(CSQ_ERR_NO_DEVICE, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    }
    int ok = 0;
    for (int d = 0; d < c; d++) {
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, d) == cudaSuccess && prop.major == 10) ok++;
    }
    *count = ok;
    return 0;
}

int csq_plan_create(const csq_op* ops_r1, int n1, const csq_op* ops_r2, int n2, const csq_filters* filters, int device,
                    uint32_t flags, csq_plan** out) {
    if (!out || !filters || (n1 > 0 && !ops_r1) || (n2 > 0 && !ops_r2)) return fail(CSQ_ERR_INVALID, "null argument");
    *out = nullptr;
    int rc = check_device(device);
    if (rc) return rc;
    csq_plan* plan = new csq_plan();
    plan->device = device;
    // CSQ_PLAN_FLAGS=<int>: extra plan flags for A/B and tool runs without touching the caller (e.g. 256 = direct emitter)
    if (const char* extra = getenv("CSQ_PLAN_FLAGS")) flags |= (uint32_t)strtoul(extra, nullptr, 0);
    plan->flags = flags;
    plan->flt = *filters;
    plan->n_mates = n2 > 0 ? 2 : 1;
    if ((rc = build_mate_program(ops_r1, n1, 0, plan->prog[0])) || (n2 > 0 && (rc = build_mate_program(ops_r2, n2, 1, plan->prog[1])))) {
        delete plan;
        return rc;
    }
    if (plan->n_mates == 2) {
        if (plan->prog[0].has_rename != plan->prog[1].has_rename || plan->prog[0].rename_parts != plan->prog[1].rename_parts) {
            delete plan;
            return fail(CSQ_ERR_INVALID, "paired programs must carry the same RENAME");
        }
        if (plan->prog[0].revcomp || plan->prog[1].revcomp) {
            delete plan;
            return fail(CSQ_ERR_INVALID, "REVCOMP is a single-end op (paired --auto-rc swaps the sink instead)");
        }
        if (plan->prog[0].rename_parts & (CSQ_REN_OWN_PREFIX | CSQ_REN_OWN_SUFFIX)) {
            delete plan;
            return fail(CSQ_ERR_INVALID, "paired RENAME uses r1/r2 parts");
        }
    } else if (plan->prog[0].rename_parts & (CSQ_REN_R1_PREFIX | CSQ_REN_R2_PREFIX)) {
        delete plan;
        return fail(CSQ_ERR_INVALID, "single-end RENAME uses own parts");
    }
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaMalloc((void**)&plan->counters, sizeof(csq_counters));
    if (e == cudaSuccess) e = cudaMemset(plan->counters, 0, sizeof(csq_counters));
    if (e == cudaSuccess) e = cudaMalloc((void**)&plan->error_flag, sizeof(int));
    if (e == cudaSuccess) e = cudaMemset(plan->error_flag, 0, sizeof(int));
    if (e == cudaSuccess) {
        std::vector<uint32_t> tab(768);
        csq_gz_crc_check_tables(tab.data());
        e = cudaMalloc((void**)&plan->crc_check_tables, tab.size() * 4);
        if (e == cudaSuccess) e = cudaMemcpy(plan->crc_check_tables, tab.data(), tab.size() * 4, cudaMemcpyHostToDevice);
    }
    if (e == cudaSuccess && (flags & CSQ_PLAN_GZIP_OUT)) {
        std::vector<uint32_t> tab(256 + GZ_THREADS);
        csq_gz_host_tables(tab.data(), tab.data() + 256);
        e = cudaMalloc((void**)&plan->gz_tables, tab.size() * 4);
        if (e == cudaSuccess) e = cudaMemcpy(plan->gz_tables, tab.data(), tab.size() * 4, cudaMemcpyHostToDevice);
    }
    for (int i = 0; i < CSQ_N_SLOTS && e == cudaSuccess; i++) {
        Slot& s = plan->slots[i];
        e = cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s.stream2, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s.ev_fork, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s.ev_join, cudaEventDisableTiming);
        for (int k = 0; k < 6 && e == cudaSuccess; k++) e = cudaEventCreate(&s.ev[k]);
        if (e == cudaSuccess) e = cudaHostAlloc((void**)&s.totals_host, 24 * 8, cudaHostAllocDefault);
        if (e == cudaSuccess) memset(s.totals_host, 0, 24 * 8);
        if (e == cudaSuccess) e = cudaMalloc((void**)&s.inflate_status, sizeof(int32_t));
        if (e == cudaSuccess && (flags & CSQ_PLAN_GZIP_OUT)) e = cudaHostAlloc((void**)&s.gz_totals_host, 8 * 8, cudaHostAllocDefault);
    }
    if (e != cudaSuccess) {
        rc = fail(CSQ_ERR_CUDA, "plan setup: %s", cudaGetErrorString(e));
        csq_plan_destroy(plan);
        return rc;
    }
    *out = plan;
    return 0;
}

void csq_plan_destroy(csq_plan* plan) {
    if (!plan) return;
    cudaSetDevice(plan->device);
    for (Slot& s : plan->slots) {
        if (s.stream) cudaStreamSynchronize(s.stream);
        for (int m = 0; m < 2; m++) {
            s.seq[m].release(); s.qual[m].release(); s.seq_off[m].release(); s.seq_len[m].release();
            s.name[m].release(); s.name_off[m].release(); s.state[m].release(); s.matches[m].release();
            for (int d = 0; d < CSQ_N_DEST; d++) s.out[d][m].release();
        }
        s.parse_misc.release();
        for (int m = 0; m < 2; m++) { s.list[m].release(); s.list_count[m].release(); }
        if (s.ev_fork) cudaEventDestroy(s.ev_fork);
        if (s.ev_join) cudaEventDestroy(s.ev_join);
        if (s.stream2) cudaStreamDestroy(s.stream2);
        for (int m = 0; m < 2; m++) {
            s.text[m].release(); s.qual_off[m].release(); s.name_end[m].release(); s.nl[m].release(); s.tiles[m].release(); s.masks[m].release();
        }
        s.dest.release(); s.block_tot.release(); s.block_cnt.release(); s.block_off.release(); s.totals.release();
        for (cudaEvent_t& e : s.ev) if (e) cudaEventDestroy(e);
        if (s.totals_host) cudaFreeHost(s.totals_host);
        if (s.inflate_status) cudaFree(s.inflate_status);
        for (int m = 0; m < 2; m++) { s.comp[m].release(); s.gz_idx[m].release(); }
        s.gz_lines.release();
        if (s.gz_totals_host) cudaFreeHost(s.gz_totals_host);
        s.gz_misc.release(); s.gz_slots.release(); s.gz_msize.release(); s.gz_moff.release(); s.gz_packed.release();
        if (s.stream) cudaStreamDestroy(s.stream);
    }
    if (plan->counters) cudaFree(plan->counters);
    if (plan->error_flag) cudaFree(plan->error_flag);
    if (plan->gz_tables) cudaFree(plan->gz_tables);
    if (plan->crc_check_tables) cudaFree(plan->crc_check_tables);
    delete plan;
}

int csq_submit(csq_plan* plan, int slot, const csq_batch_in* in, csq_batch_out* out) {
    if (!plan || slot < 0 || slot >= CSQ_N_SLOTS || !out) return fail(CSQ_ERR_INVALID, "bad plan/slot/out");
    int rc = validate_batch(plan, in);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(plan->device));
    Slot& s = plan->slots[slot];
    if (s.pending) return fail(CSQ_ERR_INVALID, "slot %d still has a batch in flight (call csq_wait)", slot);
    CUDA_TRY(cudaEventRecord(s.ev[0], s.stream));
    if ((rc = upload(plan, s, in))) return rc;
    CUDA_TRY(cudaEventRecord(s.ev[1], s.stream));
    if ((rc = enqueue_front(plan, s, nullptr, s.stream, s.stream2))) return rc;
    CUDA_TRY(cudaEventRecord(s.ev[2], s.stream));
    s.pending = out;
    return 0;
}

static int validate_text(const csq_plan* plan, const csq_batch_text* in) {
    if (!in) return fail(CSQ_ERR_INVALID, "null batch");
    if ((int)in->n_mates != plan->n_mates) return fail(CSQ_ERR_INVALID, "batch has %u mates, plan has %d", in->n_mates, plan->n_mates);
    for (int m = 0; m < plan->n_mates; m++) {
        if (in->mate[m].bytes && !in->mate[m].text) return fail(CSQ_ERR_INVALID, "mate %d: null text", m + 1);
        if (in->mate[m].bytes >= (1ull << 32) - 4096) return fail(CSQ_ERR_LIMIT, "batch text must stay below 4 GiB");
    }
    // the look-back words of the parse kernel count line ends in 30 bits
    if ((uint64_t)in->n_reads * 4 >= (1ull << 30)) return fail(CSQ_ERR_LIMIT, "too many records in one batch (limit 2^28 - 1)");
    return 0;
}

int csq_submit_text(csq_plan* plan, int slot, const csq_batch_text* in, csq_batch_out* out) {
    if (!plan || slot < 0 || slot >= CSQ_N_SLOTS || !out) return fail(CSQ_ERR_INVALID, "bad plan/slot/out");
    int rc = validate_text(plan, in);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(plan->device));
    Slot& s = plan->slots[slot];
    if (s.pending) return fail(CSQ_ERR_INVALID, "slot %d still has a batch in flight (call csq_wait)", slot);
    CUDA_TRY(cudaEventRecord(s.ev[0], s.stream));
    if ((rc = upload_text(plan, s, in))) return rc;
    CUDA_TRY(cudaEventRecord(s.ev[1], s.stream));
    if ((rc = enqueue_front(plan, s, nullptr, s.stream, s.stream2))) return rc;
    CUDA_TRY(cudaEventRecord(s.ev[2], s.stream));
    s.pending = out;
    return 0;
}

int csq_submit_bgzf(csq_plan* plan, int slot, const csq_batch_bgzf* in, csq_batch_out* out) {
    if (!plan || slot < 0 || slot >= CSQ_N_SLOTS || !out || !in) return fail(CSQ_ERR_INVALID, "bad plan/slot/in/out");
    if ((int)in->n_mates != plan->n_mates) return fail(CSQ_ERR_INVALID, "batch has %u mates, plan has %d", in->n_mates, plan->n_mates);
    if ((uint64_t)in->n_reads * 4 >= (1ull << 30)) return fail(CSQ_ERR_LIMIT, "too many records in one batch (limit 2^28 - 1)");
    CUDA_TRY(cudaSetDevice(plan->device));
    Slot& s = plan->slots[slot];
    if (s.pending) return fail(CSQ_ERR_INVALID, "slot %d still has a batch in flight (call csq_wait)", slot);
    int rc;
    CUDA_TRY(cudaEventRecord(s.ev[0], s.stream));
    if ((rc = upload_bgzf(plan, s, in))) return rc;
    CUDA_TRY(cudaEventRecord(s.ev[1], s.stream));
    if ((rc = enqueue_front(plan, s, nullptr, s.stream, s.stream2))) return rc;
    CUDA_TRY(cudaEventRecord(s.ev[2], s.stream));
    s.pending = out;
    return 0;
}

int csq_bgzf_count_lines(csq_plan* plan, int slot, const csq_bgzf_in* in, uint32_t* lines) {
    if (!plan || slot < 0 || slot >= CSQ_N_SLOTS || !in || (in->n_members && !lines)) return fail(CSQ_ERR_INVALID, "bad argument");
    CUDA_TRY(cudaSetDevice(plan->device));
    Slot& s = plan->slots[slot];
    if (s.pending) return fail(CSQ_ERR_INVALID, "slot %d still has a batch in flight (call csq_wait)", slot);
    int rc;
    if ((rc = s.gz_lines.ensure((size_t)in->n_members * 4 + 16))) return rc;
    CUDA_TRY(cudaMemsetAsync(s.inflate_status, 0x7F, sizeof(int32_t), s.stream));
    if ((rc = inflate_mate(plan, s, 0, *in, (uint32_t*)s.gz_lines.p, s.stream))) return rc;
    if (in->n_members) CUDA_TRY(cudaMemcpyAsync(lines, s.gz_lines.p, (size_t)in->n_members * 4, cudaMemcpyDeviceToHost, s.stream));
    CUDA_TRY(cudaMemcpyAsync(s.totals_host + 16, s.inflate_status, sizeof(int32_t), cudaMemcpyDeviceToHost, s.stream));
    CUDA_TRY(cudaStreamSynchronize(s.stream));
    const int32_t st = *(const int32_t*)(s.totals_host + 16);
    if (st != 0x7F7F7F7F)
        return fail(CSQ_ERR_IO, "corrupt BGZF member %d of the range (%s)", st / 16, st % 16 == 7 ? "CRC-32 mismatch" : "invalid DEFLATE data");
    return 0;
}

int csq_upload_text(csq_plan* plan, int slot, const csq_batch_text* in) {
    if (!plan || slot < 0 || slot >= CSQ_N_SLOTS) return fail(CSQ_ERR_INVALID, "bad plan/slot");
    int rc = validate_text(plan, in);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(plan->device));
    Slot& s = plan->slots[slot];
    if ((rc = upload_text(plan, s, in))) return rc;
    CUDA_TRY(cudaStreamSynchronize(s.stream));
    return 0;
}

int csq_wait(csq_plan* plan, int slot) {
    if (!plan || slot < 0 || slot >= CSQ_N_SLOTS) return fail(CSQ_ERR_INVALID, "bad plan/slot");
    CUDA_TRY(cudaSetDevice(plan->device));
    Slot& s = plan->slots[slot];
    if (!s.pending) return fail(CSQ_ERR_INVALID, "nothing submitted on slot %d", slot);
    csq_batch_out* out = s.pending;
    s.pending = nullptr;
    const bool gz = (plan->flags & CSQ_PLAN_GZIP_OUT) != 0;
    int rc;
    // every .bytes field holds the needed size when a buffer is too small: the caller may enlarge its buffers and call
    // csq_wait() again for this slot
    auto capacity_ok = [&]() -> int {
        for (int d = 0; d < CSQ_N_DEST; d++)
            for (int m = 0; m < 2; m++) {
                csq_text_out& t = out->text[d][m];
                if (t.bytes > t.capacity || (t.bytes && !t.data)) {
                    s.pending = out;
                    return fail(CSQ_ERR_CAPACITY, "output buffer [%d][%d] holds %llu bytes, %llu needed", d, m,
                                (unsigned long long)t.capacity, (unsigned long long)t.bytes);
                }
            }
        return 0;
    };
    if (!s.gz_ready) {
        CUDA_TRY(cudaStreamSynchronize(s.stream));
        if ((rc = check_device_error(s))) return rc;
        for (int d = 0; d < CSQ_N_DEST; d++)
            for (int m = 0; m < 2; m++) {
                csq_text_out& t = out->text[d][m];
                t.bytes = s.totals_host[d * 2 + m];
                t.records = (m < s.n_mates) ? s.totals_host[8 + d] : 0;
            }
        if (!gz && (rc = capacity_ok())) return rc;
        if ((rc = size_outputs(s))) return rc;
        CUDA_TRY(cudaEventRecord(s.ev[3], s.stream));
        if ((rc = enqueue_emit(plan, s, nullptr, s.stream))) return rc;
        if (gz) {
            // the text never leaves the device: members are encoded there, their packed sizes come back first
            if ((rc = enqueue_gz(plan, s, nullptr, s.stream))) return rc;
            CUDA_TRY(cudaEventRecord(s.ev[4], s.stream));
            CUDA_TRY(cudaStreamSynchronize(s.stream));
            s.gz_ready = true;
        } else {
            CUDA_TRY(cudaEventRecord(s.ev[4], s.stream));
        }
    }
    if (gz) {
        for (int d = 0; d < CSQ_N_DEST; d++)
            for (int m = 0; m < 2; m++) out->text[d][m].bytes = m < s.n_mates ? s.gz_totals_host[d * 2 + m] : 0;
        if ((rc = capacity_ok())) return rc;
        s.gz_ready = false;
    }
    for (int d = 0; d < CSQ_N_DEST; d++)
        for (int m = 0; m < s.n_mates; m++) {
            csq_text_out& t = out->text[d][m];
            const void* src = gz ? (const void*)s.gz_packed_ptr[d * 2 + m] : s.out[d][m].p;
            if (t.bytes) CUDA_TRY(cudaMemcpyAsync(t.data, src, t.bytes, cudaMemcpyDeviceToHost, s.stream));
        }
    CUDA_TRY(cudaEventRecord(s.ev[5], s.stream));
    CUDA_TRY(cudaStreamSynchronize(s.stream));
    float h2d = 0, front = 0, emit = 0, d2h = 0;
    cudaEventElapsedTime(&h2d, s.ev[0], s.ev[1]);
    cudaEventElapsedTime(&front, s.ev[1], s.ev[2]);
    cudaEventElapsedTime(&emit, s.ev[3], s.ev[4]);
    cudaEventElapsedTime(&d2h, s.ev[4], s.ev[5]);
    s.kernel_ms = front + emit;
    s.total_ms = h2d + front + emit + d2h;
    return 0;
}

int csq_slot_times(csq_plan* plan, int slot, float* total_ms, float* kernel_ms) {
    if (!plan || slot < 0 || slot >= CSQ_N_SLOTS) return fail(CSQ_ERR_INVALID, "bad plan/slot");
    if (total_ms) *total_ms = plan->slots[slot].total_ms;
    if (kernel_ms) *kernel_ms = plan->slots[slot].kernel_ms;
    return 0;
}

int csq_upload(csq_plan* plan, int slot, const csq_batch_in* in) {
    if (!plan || slot < 0 || slot >= CSQ_N_SLOTS) return fail(CSQ_ERR_INVALID, "bad plan/slot");
    int rc = validate_batch(plan, in);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(plan->device));
    Slot& s = plan->slots[slot];
    if ((rc = upload(plan, s, in))) return rc;
    CUDA_TRY(cudaStreamSynchronize(s.stream));
    return 0;
}

int csq_run_resident(csq_plan* plan, int slot, int iters, float* ms_per_iter) {
    if (!plan || slot < 0 || slot >= CSQ_N_SLOTS || iters < 1) return fail(CSQ_ERR_INVALID, "bad plan/slot/iters");
    CUDA_TRY(cudaSetDevice(plan->device));
    Slot& s = plan->slots[slot];
    int rc;
    // sizing pass (not timed): totals are needed on the host before the emit buffers exist
    if ((rc = enqueue_front(plan, s, nullptr, s.stream, s.stream2))) return rc;
    CUDA_TRY(cudaStreamSynchronize(s.stream));
    if ((rc = check_device_error(s))) return rc;
    if ((rc = size_outputs(s))) return rc;
    if ((rc = enqueue_emit(plan, s, nullptr, s.stream))) return rc;
    CUDA_TRY(cudaMemcpyAsync(s.totals_host + 13, plan->error_flag, sizeof(int), cudaMemcpyDeviceToHost, s.stream));
    CUDA_TRY(cudaStreamSynchronize(s.stream));
    if ((rc = check_device_error(s, 13))) return rc;
    if (iters == 1) {  // the sizing pass already did the work once
        if (ms_per_iter) *ms_per_iter = 0.f;
        return 0;
    }
    KernelTimer kt;
    kt.stream = s.stream;
    CUDA_TRY(cudaEventRecord(s.ev[0], s.stream));
    for (int it = 1; it < iters; it++) {
        kt.on = (it == iters - 1);
        if ((rc = enqueue_front(plan, s, kt.on ? &kt : nullptr, s.stream, s.stream2))) return rc;
        if ((rc = enqueue_emit(plan, s, &kt, s.stream))) return rc;
    }
    CUDA_TRY(cudaEventRecord(s.ev[1], s.stream));
    CUDA_TRY(cudaStreamSynchronize(s.stream));
    float ms = 0;
    CUDA_TRY(cudaEventElapsedTime(&ms, s.ev[0], s.ev[1]));
    if (ms_per_iter) *ms_per_iter = ms / (float)(iters - 1);
    s.ktimes.clear();
    for (size_t i = 1; i < kt.evs.size(); i++) {
        float t = 0;
        cudaEventElapsedTime(&t, kt.evs[i - 1], kt.evs[i]);
        s.ktimes.push_back({kt.names[i], t});
    }
    for (cudaEvent_t e : kt.evs) cudaEventDestroy(e);
    return 0;
}

int csq_run_steps(csq_plan* plan, const int* slots, int n_slots, int steps, float* total_ms) {
    if (!plan || !slots || n_slots < 1 || steps < 1) return fail(CSQ_ERR_INVALID, "bad argument");
    for (int i = 0; i < n_slots; i++)
        if (slots[i] < 0 || slots[i] >= CSQ_N_SLOTS) return fail(CSQ_ERR_INVALID, "bad slot");
    CUDA_TRY(cudaSetDevice(plan->device));
    Slot& s0 = plan->slots[slots[0]];
    cudaStream_t st = s0.stream;
    int rc;
    for (int i = 0; i < n_slots; i++) {  // untimed sizing pass: emit buffers must exist
        Slot& s = plan->slots[slots[i]];
        CUDA_TRY(cudaStreamSynchronize(s.stream));
        if ((rc = enqueue_front(plan, s, nullptr, st, s0.stream2))) return rc;
        CUDA_TRY(cudaStreamSynchronize(st));
        if ((rc = check_device_error(s))) return rc;
        if ((rc = size_outputs(s))) return rc;
        if ((rc = enqueue_emit(plan, s, nullptr, st))) return rc;
        CUDA_TRY(cudaMemcpyAsync(s.totals_host + 13, plan->error_flag, sizeof(int), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        if ((rc = check_device_error(s, 13))) return rc;
    }
    CUDA_TRY(cudaStreamSynchronize(st));
    // Timed region: step i on slots[i % n_slots], back to back on the first slot's stream pair (the chains of the two
    // mates side by side).  Running every batch on the streams of its own slot, so that steps overlap, was measured
    // and did not help (4.66 ms against 4.51 ms per step, profiles/r01_overlap_steps.md): the large kernels fill the
    // machine on their own and five batches in flight only add L2 pressure.
    CUDA_TRY(cudaEventRecord(s0.ev[0], st));
    for (int it = 0; it < steps; it++) {
        Slot& s = plan->slots[slots[it % n_slots]];
        if ((rc = enqueue_front(plan, s, nullptr, st, s0.stream2))) return rc;
        if ((rc = enqueue_emit(plan, s, nullptr, st))) return rc;
    }
    CUDA_TRY(cudaEventRecord(s0.ev[1], st));
    CUDA_TRY(cudaStreamSynchronize(st));
    float ms = 0;
    CUDA_TRY(cudaEventElapsedTime(&ms, s0.ev[0], s0.ev[1]));
    if (total_ms) *total_ms = ms;
    // one more step, NOT timed above: everything on one stream with an event after every kernel
    KernelTimer kt;
    kt.stream = st;
    kt.on = true;
    {
        Slot& s = plan->slots[slots[steps % n_slots]];
        if ((rc = enqueue_front(plan, s, &kt, st, nullptr))) return rc;
        if ((rc = enqueue_emit(plan, s, &kt, st))) return rc;
        CUDA_TRY(cudaStreamSynchronize(st));
    }
    s0.ktimes.clear();
    for (size_t i = 1; i < kt.evs.size(); i++) {
        float t = 0;
        cudaEventElapsedTime(&t, kt.evs[i - 1], kt.evs[i]);
        s0.ktimes.push_back({kt.names[i], t});
    }
    for (cudaEvent_t e : kt.evs) cudaEventDestroy(e);
    return 0;
}

int csq_kernel_times(csq_plan* plan, int slot, const char** names, float* ms, int cap) {
    if (!plan || slot < 0 || slot >= CSQ_N_SLOTS) return fail(CSQ_ERR_INVALID, "bad plan/slot");
    Slot& s = plan->slots[slot];
    int n = (int)s.ktimes.size() < cap ? (int)s.ktimes.size() : cap;
    for (int i = 0; i < n; i++) {
        if (names) names[i] = s.ktimes[i].first;
        if (ms) ms[i] = s.ktimes[i].second;
    }
    return n;
}

int csq_launch_count(csq_plan* plan, uint64_t* launches) {
    if (!plan || !launches) return fail(CSQ_ERR_INVALID, "null argument");
    *launches = plan->launches;
    return 0;
}

int csq_fetch_results(csq_plan* plan, int slot, int mate, csq_read_result* out, uint32_t n) {
    if (!plan || slot < 0 || slot >= CSQ_N_SLOTS || mate < 0 || mate >= plan->n_mates || !out) return fail(CSQ_ERR_INVALID, "bad argument");
    CUDA_TRY(cudaSetDevice(plan->device));
    Slot& s = plan->slots[slot];
    if (n > s.n) n = s.n;
    std::vector<ReadState> st(n);
    std::vector<uint8_t> dest(n);
    CUDA_TRY(cudaStreamSynchronize(s.stream));
    if (n) {
        CUDA_TRY(cudaMemcpy(st.data(), s.state[mate].p, (size_t)n * sizeof(ReadState), cudaMemcpyDeviceToHost));
        CUDA_TRY(cudaMemcpy(dest.data(), s.dest.p, n, cudaMemcpyDeviceToHost));
    }
    for (uint32_t i = 0; i < n; i++) {
        out[i].start = st[i].a;
        out[i].stop = st[i].b;
        out[i].dest = dest[i];
        out[i].matched = st[i].matched;
    }
    return 0;
}

int csq_fetch_matches(csq_plan* plan, int slot, int mate, int op_index, csq_match* out, uint32_t n) {
    if (!plan || slot < 0 || slot >= CSQ_N_SLOTS || mate < 0 || mate >= plan->n_mates || !out) return fail(CSQ_ERR_INVALID, "bad argument");
    if (!(plan->flags & CSQ_PLAN_KEEP_MATCHES)) return fail(CSQ_ERR_INVALID, "plan was created without CSQ_PLAN_KEEP_MATCHES");
    MateProgram& mp = plan->prog[mate];
    if (op_index < 0 || op_index >= mp.n_ops || mp.align_slot[op_index] < 0) return fail(CSQ_ERR_INVALID, "op %d is not an ALIGN op", op_index);
    CUDA_TRY(cudaSetDevice(plan->device));
    Slot& s = plan->slots[slot];
    if (n > s.n) n = s.n;
    CUDA_TRY(cudaStreamSynchronize(s.stream));
    if (n)
        CUDA_TRY(cudaMemcpy(out, (csq_match*)s.matches[mate].p + (size_t)mp.align_slot[op_index] * s.n, (size_t)n * sizeof(csq_match),
                            cudaMemcpyDeviceToHost));
    return 0;
}

int csq_fetch_text(csq_plan* plan, int slot, csq_batch_out* out) {
    if (!plan || slot < 0 || slot >= CSQ_N_SLOTS || !out) return fail(CSQ_ERR_INVALID, "bad argument");
    CUDA_TRY(cudaSetDevice(plan->device));
    Slot& s = plan->slots[slot];
    CUDA_TRY(cudaStreamSynchronize(s.stream));
    for (int d = 0; d < CSQ_N_DEST; d++)
        for (int m = 0; m < 2; m++) {
            csq_text_out& t = out->text[d][m];
            t.bytes = m < s.n_mates ? s.totals_host[d * 2 + m] : 0;
            t.records = m < s.n_mates ? s.totals_host[8 + d] : 0;
            if (t.bytes > t.capacity) return fail(CSQ_ERR_CAPACITY, "output buffer [%d][%d] too small (%llu needed)", d, m, (unsigned long long)t.bytes);
            if (t.bytes) CUDA_TRY(cudaMemcpy(t.data, s.out[d][m].p, t.bytes, cudaMemcpyDeviceToHost));
        }
    return 0;
}

int csq_stats(csq_plan* plan, csq_counters* out) {
    if (!plan || !out) return fail(CSQ_ERR_INVALID, "null argument");
    CUDA_TRY(cudaSetDevice(plan->device));
    for (Slot& s : plan->slots) CUDA_TRY(cudaStreamSynchronize(s.stream));
    CUDA_TRY(cudaMemcpy(out, plan->counters, sizeof(csq_counters), cudaMemcpyDeviceToHost));
    return 0;
}

int csq_locate_batch(int device, const csq_op* align_op, const csq_mate_in* reads, uint32_t n_reads, uint32_t plan_flags,
                     csq_match* out) {
    if (!align_op || !reads || !out || align_op->kind != CSQ_OP_ALIGN) return fail(CSQ_ERR_INVALID, "bad argument");
    csq_filters flt = {0, 0, 0, 0};
    csq_plan* plan = nullptr;
    int rc = csq_plan_create(align_op, 1, nullptr, 0, &flt, device, plan_flags | CSQ_PLAN_KEEP_MATCHES, &plan);
    if (rc) return rc;
    csq_batch_in in;
    memset(&in, 0, sizeof(in));
    in.n_reads = n_reads;
    in.n_mates = 1;
    in.mate[0] = *reads;
    rc = csq_upload(plan, 0, &in);
    if (!rc) rc = csq_run_resident(plan, 0, 1, nullptr);
    if (!rc) rc = csq_fetch_matches(plan, 0, 0, 0, out, n_reads);
    csq_plan_destroy(plan);
    return rc;
}

int csq_int_peak(int device, double* alu_ops_per_s, double* mixed_ops_per_s) {
    int rc = check_device(device);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    unsigned int* sink = nullptr;
    CUDA_TRY(cudaMalloc((void**)&sink, 16));
    CUDA_TRY(cudaMemset(sink, 0, 16));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 2000;
    double res[2] = {0, 0};
    for (int v = 0; v < 2; v++) {
        double best = 0;
        for (int rep = 0; rep < 4; rep++) {
            CUDA_TRY(cudaEventRecord(e0, 0));
            CUDA_TRY(csq_launch_int_peak(v, iters, sink, blocks, threads, 0));
            CUDA_TRY(cudaEventRecord(e1, 0));
            CUDA_TRY(cudaEventSynchronize(e1));
            float ms = 0;
            CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
            // 3 integer ops per statement, 64 statements per iteration per thread
            double ops = 3.0 * 64.0 * iters * (double)blocks * threads;
            double r = ops / (ms * 1e-3);
            if (rep > 0 && r > best) best = r;
        }
        res[v] = best;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(sink);
    if (alu_ops_per_s) *alu_ops_per_s = res[0];
    if (mixed_ops_per_s) *mixed_ops_per_s = res[1];
    return 0;
}

// Measured ceiling of the host <-> device path for the end-to-end numbers: pinned host buffers, one stream per
// direction, `reps` copies of bytes_h2d / bytes_d2h each.  mode 0: host -> device alone, 1: device -> host alone,
// 2: both at once (what a pipelined csq_submit_text / csq_wait loop does).  Returns GB/s per direction (for mode 2
// both are bytes moved in that direction over the time until BOTH streams have drained).
int csq_pcie_peak(int device, uint64_t bytes_h2d, uint64_t bytes_d2h, int reps, int mode, double* h2d_gbs, double* d2h_gbs) {
    int rc = check_device(device);
    if (rc) return rc;
    if (reps < 1 || mode < 0 || mode > 2) return fail(CSQ_ERR_INVALID, "bad argument");
    CUDA_TRY(cudaSetDevice(device));
    const bool up = mode != 1 && bytes_h2d > 0, down = mode != 0 && bytes_d2h > 0;
    void *h_in = nullptr, *h_out = nullptr, *d_in = nullptr, *d_out = nullptr;
    cudaStream_t s_up = nullptr, s_down = nullptr;
    cudaEvent_t e0 = nullptr, e_up = nullptr, e_down = nullptr;
    cudaError_t e = cudaSuccess;
    auto step = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
    if (up) {
        step(cudaHostAlloc(&h_in, bytes_h2d, cudaHostAllocDefault));
        step(cudaMalloc(&d_in, bytes_h2d));
        if (e == cudaSuccess) memset(h_in, 0x41, bytes_h2d);
    }
    if (down) {
        step(cudaHostAlloc(&h_out, bytes_d2h, cudaHostAllocDefault));
        step(cudaMalloc(&d_out, bytes_d2h));
        if (e == cudaSuccess) step(cudaMemset(d_out, 0x42, bytes_d2h));
        if (e == cudaSuccess) memset(h_out, 0, bytes_d2h);  // touch the pages before the timed copies
    }
    step(cudaStreamCreateWithFlags(&s_up, cudaStreamNonBlocking));
    step(cudaStreamCreateWithFlags(&s_down, cudaStreamNonBlocking));
    step(cudaEventCreate(&e0));
    step(cudaEventCreate(&e_up));
    step(cudaEventCreate(&e_down));
    float ms_up = 0, ms_down = 0;
    for (int pass = 0; pass < 2 && e == cudaSuccess; pass++) {  // pass 0 warms up (first-touch, page tables)
        const int n = pass == 0 ? 1 : reps;
        step(cudaDeviceSynchronize());
        step(cudaEventRecord(e0, s_up));
        if (down) step(cudaStreamWaitEvent(s_down, e0, 0));
        for (int r = 0; r < n && e == cudaSuccess; r++) {
            if (up) step(cudaMemcpyAsync(d_in, h_in, bytes_h2d, cudaMemcpyHostToDevice, s_up));
            if (down) step(cudaMemcpyAsync(h_out, d_out, bytes_d2h, cudaMemcpyDeviceToHost, s_down));
        }
        step(cudaEventRecord(e_up, s_up));
        step(cudaEventRecord(e_down, s_down));
        step(cudaStreamSynchronize(s_up));
        step(cudaStreamSynchronize(s_down));
        if (e == cudaSuccess) {
            cudaEventElapsedTime(&ms_up, e0, e_up);
            cudaEventElapsedTime(&ms_down, e0, e_down);
        }
    }
    if (e == cudaSuccess) {
        const float both = ms_up > ms_down ? ms_up : ms_down;
        const float t_up = mode == 2 ? both : ms_up, t_down = mode == 2 ? both : ms_down;
        if (h2d_gbs) *h2d_gbs = up && t_up > 0 ? (double)bytes_h2d * reps / (t_up * 1e-3) / 1e9 : 0.0;
        if (d2h_gbs) *d2h_gbs = down && t_down > 0 ? (double)bytes_d2h * reps / (t_down * 1e-3) / 1e9 : 0.0;
    }
    if (e0) cudaEventDestroy(e0);
    if (e_up) cudaEventDestroy(e_up);
    if (e_down) cudaEventDestroy(e_down);
    if (s_up) cudaStreamDestroy(s_up);
    if (s_down) cudaStreamDestroy(s_down);
    if (h_in) cudaFreeHost(h_in);
    if (h_out) cudaFreeHost(h_out);
    if (d_in) cudaFree(d_in);
    if (d_out) cudaFree(d_out);
    if (e != cudaSuccess) return fail(e == cudaErrorMemoryAllocation ? CSQ_ERR_NOMEM : CSQ_ERR_CUDA, "csq_pcie_peak: %s", cudaGetErrorString(e));
    return 0;
}

}  // extern "C"
