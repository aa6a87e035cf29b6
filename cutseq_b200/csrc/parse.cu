// FASTQ text -> record index, on the device.
//
// In text mode (csq_submit_text / csq_upload_text) the host ships the raw FASTQ bytes of a batch - whole
// records, cut at a record boundary by counting line ends - and these kernels do what dnaio's FASTQ
// parser (_core.pyx, behind cutadapt's InputPaths in reference run.py:434, 751) does on the CPU:
//
//   k_nl_count     reads the text once: a line-end bit mask per 16-byte chunk, line ends per 16 KiB tile, and one
//                  flag "there is a '\r' somewhere in this batch"
//   k_tile_scan    exclusive scan of the tile counts (one CTA, 8 tiles per thread and sweep)
//   k_nl_index     from the masks: byte position of every line end, in order, nl[r] = offset of the r-th '\n'
//   k_records      record i = lines 4i .. 4i+3 from the line ends alone: equal sequence / quality lengths, the
//                  read-length limit; writes name / sequence / quality offsets and lengths.  '\r' stripping only
//                  when the flag is set; the '@' / '+' line starts are checked by k_finish (kernels.cu), which
//                  fetches those sectors anyway
//
// The trimming kernels then work on the text where it lies (seq == qual == name pool == the text buffer);
// nothing is copied into a packed layout.  Bound: HBM - the text is read once (plus 1/8 of it written and read
// back as masks and 16 bytes of line-end offsets per record written and read).  A malformed record is reported
// as the smallest (record, kind) key through `perr`, in the order dnaio would meet the problems.
//
// FASTA text (CSQ_PLAN_FASTA) takes its own kernels, as transcode.fasta_to_fastq reads it:
//   k_fa_count     reads the text once: a record-start bit mask per 16-byte chunk ('>' as the first byte of a line)
//                  and record starts per tile; k_tile_scan and k_nl_index then turn the masks into hdr[r] = offset of
//                  the r-th record start, exactly as they do for line ends
//   k_fa_records   thread per record: header = the rest of the '>' line without trailing '\r'; every following line up
//                  to the next record start is stripped of ASCII whitespace and the pieces are joined.  A sequence on
//                  one line (the common unwrapped case, also with CRLF, blank lines or blanks around it) stays
//                  where it is in the text; a wrapped one is marked for the pool.  Text in front of the first header
//                  that is not blank, a different number of headers than the host counted and the read-length limit
//                  are reported through `perr`
//   k_tile_scan    (again) exclusive scan of the 16-byte-padded lengths of the wrapped records = their pool offsets
//   k_fa_compact   thread per wrapped record: its stripped lines, joined, into the pool behind the text
// Qualities are a constant buffer of 'I' bytes (qual_off the same for every record).
#include <cuda_runtime.h>
#include <stdint.h>

#include "csq_internal.h"

namespace {

constexpr int TILE_THREADS = 256;
constexpr int TILE_BYTES = 16384;               // 1024 chunks of 16 bytes; thread t owns the 64 bytes at 64 t
constexpr int TILE_CHUNKS = TILE_BYTES / 16;

// Byte tests on 32-bit words, one LOP3 per step: the constants live in registers (handed in through an opaque asm
// so that ptxas does not turn every step into two immediate-form instructions - the count kernel is ALU bound).
struct ByteConsts {
    uint32_t k7f, k80, k0a, k0d, k01;
};
__device__ __forceinline__ ByteConsts byte_consts() {
    ByteConsts k;
    asm volatile("mov.b32 %0, 0x7F7F7F7F;" : "=r"(k.k7f));
    asm volatile("mov.b32 %0, 0x80808080;" : "=r"(k.k80));
    asm volatile("mov.b32 %0, 0x0A0A0A0A;" : "=r"(k.k0a));
    asm volatile("mov.b32 %0, 0x0D0D0D0D;" : "=r"(k.k0d));
    asm volatile("mov.b32 %0, 0x01010101;" : "=r"(k.k01));
    return k;
}
__device__ __forceinline__ uint32_t lop3(uint32_t a, uint32_t b, uint32_t c, int lut) {
    uint32_t d;
    switch (lut) {  // the look-up table has to be an immediate
        case 0x6A: asm("lop3.b32 %0, %1, %2, %3, 0x6A;" : "=r"(d) : "r"(a), "r"(b), "r"(c)); break;  // (a & b) ^ c
        case 0x02: asm("lop3.b32 %0, %1, %2, %3, 0x02;" : "=r"(d) : "r"(a), "r"(b), "r"(c)); break;  // ~(a | b) & c
        default: asm("lop3.b32 %0, %1, %2, %3, 0xF2;" : "=r"(d) : "r"(a), "r"(b), "r"(c)); break;    // a | (~b & c)
    }
    return d;
}
// bits 7, 15, 23, 31 of the result: byte of w equals the byte replicated in `kc` (which must be < 0x80).
// x = (w & 0x7f..) ^ kc is zero in the low seven bits exactly there; + 0x7f.. then leaves bit 7 clear only for those,
// bytes do not borrow from each other, and w's own bit 7 rules out 0x80 | c.
__device__ __forceinline__ uint32_t eq_marks(uint32_t w, uint32_t kc, const ByteConsts& k) {
    const uint32_t y = lop3(w, k.k7f, kc, 0x6A) + k.k7f;
    return lop3(y, w, k.k80, 0x02);
}
// bit i set <=> byte i of the 16-byte chunk is '\n': the four marks of a word times 0x00204081 land in bits 28..31
// (every partial product has its own bit position, nothing carries)
__device__ __forceinline__ uint32_t nl_mask16(uint4 v, const ByteConsts& k) {
    const uint32_t M = 0x00204081u;
    const uint32_t n0 = (eq_marks(v.x, k.k0a, k) * M) >> 28, n1 = (eq_marks(v.y, k.k0a, k) * M) >> 24;
    const uint32_t n2 = (eq_marks(v.z, k.k0a, k) * M) >> 20, n3 = (eq_marks(v.w, k.k0a, k) * M) >> 16;
    return n0 | (n1 & 0xF0u) | (n2 & 0xF00u) | (n3 & 0xF000u);
}

// Pass 1: the text is read ONCE, fully coalesced (chunk c of the tile by thread c % 256); what survives is a
// 16-bit line-end mask per chunk (1/8 of the text) and the number of line ends per tile.
// The text buffer is 16-byte aligned and zero padded, so whole chunks never leave the allocation and padding
// never counts as a line end.
__global__ void __launch_bounds__(TILE_THREADS) k_nl_count(const uint8_t* __restrict__ text, uint64_t bytes,
                                                           uint16_t* __restrict__ masks, uint32_t* __restrict__ tile_cnt,
                                                           uint32_t* __restrict__ any_cr) {
    __shared__ uint32_t wsum[TILE_THREADS / 32];
    const uint64_t tile_off = (uint64_t)blockIdx.x * TILE_BYTES;
    uint32_t c = 0, cr = 0;
    const ByteConsts k = byte_consts();
#pragma unroll
    for (int i = 0; i < TILE_CHUNKS / TILE_THREADS; i++) {
        const uint32_t chunk = i * TILE_THREADS + threadIdx.x;
        const uint64_t off = tile_off + 16ull * chunk;
        uint32_t m = 0;
        if (off < bytes) {
            const uint4 v = *reinterpret_cast<const uint4*>(text + off);
            m = nl_mask16(v, k);
            // is there a '\r' anywhere?  x = w ^ "\r\r\r\r"; (x - 0x01..) & ~x has bit 7 of some byte set iff x has a
            // zero byte (a borrow can only start at one), accumulated with cr | (~x & (x - 0x01..))
            const uint32_t x0 = v.x ^ k.k0d, x1 = v.y ^ k.k0d, x2 = v.z ^ k.k0d, x3 = v.w ^ k.k0d;
            cr = lop3(cr, x0, x0 - k.k01, 0xF2);
            cr = lop3(cr, x1, x1 - k.k01, 0xF2);
            cr = lop3(cr, x2, x2 - k.k01, 0xF2);
            cr = lop3(cr, x3, x3 - k.k01, 0xF2);
        }
        masks[(size_t)blockIdx.x * TILE_CHUNKS + chunk] = (uint16_t)m;
        c += __popc(m);
    }
    if (__any_sync(0xffffffffu, (cr & 0x80808080u) != 0) && (threadIdx.x & 31) == 0) atomicOr(any_cr, 1u);
    c = __reduce_add_sync(0xffffffffu, c);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
#pragma unroll
        for (int w = 0; w < TILE_THREADS / 32; w++) t += wsum[w];
        tile_cnt[blockIdx.x] = t;
    }
}

// One CTA: exclusive scan of n_tiles counts in place; total[0] = number of line ends.  Thread t takes 8
// consecutive tiles per sweep (two 16-byte loads), so a 715 MB mate (43 600 tiles) needs 6 sweeps.
__global__ void __launch_bounds__(1024) k_tile_scan(uint32_t n_tiles, uint32_t* __restrict__ tile_cnt, uint32_t* __restrict__ total) {
    __shared__ uint32_t warp_sums[32];
    __shared__ uint32_t carry;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n_tiles; base += 8192) {
        const uint32_t i0 = base + threadIdx.x * 8u;
        uint32_t v[8];
        if (i0 + 8 <= n_tiles) {  // the buffer is 16-byte aligned and i0 a multiple of 8
            const uint4 lo = *reinterpret_cast<const uint4*>(tile_cnt + i0), hi = *reinterpret_cast<const uint4*>(tile_cnt + i0 + 4);
            v[0] = lo.x; v[1] = lo.y; v[2] = lo.z; v[3] = lo.w;
            v[4] = hi.x; v[5] = hi.y; v[6] = hi.z; v[7] = hi.w;
        } else {
#pragma unroll
            for (int u = 0; u < 8; u++) v[u] = i0 + u < n_tiles ? tile_cnt[i0 + u] : 0u;
        }
        uint32_t mine = 0;
#pragma unroll
        for (int u = 0; u < 8; u++) mine += v[u];
        uint32_t x = mine;
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) warp_sums[wid] = x;
        __syncthreads();
        if (wid == 0) {
            uint32_t ws = warp_sums[lane];
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, ws, o);
                if (lane >= o) ws += y;
            }
            warp_sums[lane] = ws;
        }
        __syncthreads();
        uint32_t run = carry + (wid ? warp_sums[wid - 1] : 0u) + (x - mine);  // line ends in front of tile i0
        const uint32_t sweep_total = warp_sums[31];
#pragma unroll
        for (int u = 0; u < 8; u++) {
            const uint32_t c = v[u];
            v[u] = run;
            run += c;
        }
        if (i0 + 8 <= n_tiles) {
            *reinterpret_cast<uint4*>(tile_cnt + i0) = make_uint4(v[0], v[1], v[2], v[3]);
            *reinterpret_cast<uint4*>(tile_cnt + i0 + 4) = make_uint4(v[4], v[5], v[6], v[7]);
        } else {
#pragma unroll
            for (int u = 0; u < 8; u++)
                if (i0 + u < n_tiles) tile_cnt[i0 + u] = v[u];
        }
        __syncthreads();
        if (threadIdx.x == 0) carry += sweep_total;
        __syncthreads();
    }
    if (threadIdx.x == 0) total[0] = carry;
}

// Pass 2 reads only the masks: thread t of a tile owns the 64 bytes at 64 t (four masks = one 64-bit word),
// ranks its line ends by a CTA-wide scan and writes their byte offsets, nl[r] = offset of the r-th '\n'.
__global__ void __launch_bounds__(TILE_THREADS) k_nl_index(const uint16_t* __restrict__ masks, const uint32_t* __restrict__ tile_base,
                                                           uint32_t* __restrict__ nl, uint32_t nl_cap, uint32_t skip,
                                                           uint32_t* __restrict__ first_off) {
    __shared__ uint32_t wsum[TILE_THREADS / 32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    unsigned long long m = reinterpret_cast<const unsigned long long*>(masks + (size_t)blockIdx.x * TILE_CHUNKS)[threadIdx.x];
    const uint32_t c = __popcll(m);
    uint32_t x = c;
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) wsum[wid] = x;
    __syncthreads();
    uint32_t r = tile_base[blockIdx.x] + (x - c);
    for (int w = 0; w < wid; w++) r += wsum[w];
    const uint32_t off = blockIdx.x * (uint32_t)TILE_BYTES + threadIdx.x * 64u;
    while (m) {
        const int bit = __ffsll((long long)m) - 1;
        m &= m - 1;
        // line end r of the text is line end r - skip of the batch; the one in front of it marks the first record
        if (r >= skip && r - skip < nl_cap) nl[r - skip] = off + (uint32_t)bit;
        if (r + 1 == skip) first_off[0] = off + (uint32_t)bit + 1u;
        r++;
    }
}

// kinds of a malformed record, in the order dnaio would meet them
enum { PERR_AT = 1, PERR_PLUS = 2, PERR_LEN = 3, PERR_LIMIT = 4, PERR_COUNT = 5 };

__device__ __forceinline__ void report(unsigned long long* perr, uint32_t rec, int kind) {
    atomicMin(perr, ((unsigned long long)rec << 3) | (unsigned long long)kind);
}

__global__ void __launch_bounds__(256) k_records(const ParseParams P) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    // plain text batches hold exactly their records; BGZF batches may hold more lines on either side
    const bool count_ok = P.first_off ? P.nl_total[0] >= P.skip + 4u * P.n : P.nl_total[0] == 4u * P.n;
    if (i == 0 && !count_ok) report(P.perr, 0, PERR_COUNT);
    if (i >= P.n) return;
    if (!count_ok) {  // nl[] is not fully defined: every record becomes an empty one, the host rejects the batch
        P.name_off[i] = P.name_end[i] = P.seq_off[i] = P.seq_len[i] = P.qual_off[i] = 0;
        return;
    }
    // The record index comes from the line ends alone.  The text is only looked at for '\r' stripping, and only when
    // k_nl_count saw a '\r' somewhere (CRLF files); the '@' and '+' line starts are checked by k_finish, which
    // fetches the header and the end of the bases anyway (this kernel used to pull ~5 DRAM sectors per record, 93 %
    // of the text, for six bytes).
    const uint4 e = reinterpret_cast<const uint4*>(P.nl)[i];  // the four line ends of record i
    uint32_t s0 = i ? P.nl[4u * i - 1] + 1u : (P.first_off ? P.first_off[0] : 0u);
    uint32_t e0 = e.x, e1 = e.y, e3 = e.w;
    const uint32_t s1 = e.x + 1, s3 = e.z + 1;
    if (P.any_cr[0]) {
        const uint8_t* __restrict__ t = P.text;
        if (e0 > s0 && t[e0 - 1] == '\r') e0--;
        if (e1 > s1 && t[e1 - 1] == '\r') e1--;
        if (e3 > s3 && t[e3 - 1] == '\r') e3--;
    }
    const uint32_t slen = e1 - s1, qlen = e3 - s3;
    bool ok = true;
    if (slen != qlen || slen > CSQ_MAX_READ_LEN) {
        // rare: this record is reported from here, in the order dnaio would meet its problems (k_finish skips it)
        const uint8_t* __restrict__ t = P.text;
        const uint32_t s2 = e.y + 1;
        uint32_t e2 = e.z;
        if (e2 > s2 && t[e2 - 1] == '\r') e2--;
        const int kind = (e0 == s0 || t[s0] != '@') ? PERR_AT : (e2 == s2 || t[s2] != '+') ? PERR_PLUS : slen != qlen ? PERR_LEN : PERR_LIMIT;
        report(P.perr, i, kind);
        ok = false;
    }
    // a bad record becomes an empty one: the rest of the chain stays in bounds, the batch is rejected by the host
    P.name_off[i] = ok ? min(s0 + 1, e0) : s0;  // behind the '@' (k_finish checks that it is one)
    P.name_end[i] = ok ? e0 : s0;
    P.seq_off[i] = s1;
    P.seq_len[i] = ok ? slen : 0u;
    P.qual_off[i] = s3;
}


// ---- FASTA ----
constexpr uint32_t FA_MULTI = 0x80000000u;  // seq_len bit between k_fa_records and k_fa_compact: sequence spans lines

// bit i set <=> byte i of the 16 equals the byte replicated in kc (< 0x80)
__device__ __forceinline__ uint32_t eq_mask16(uint4 v, uint32_t kc, const ByteConsts& k) {
    const uint32_t M = 0x00204081u;
    const uint32_t n0 = (eq_marks(v.x, kc, k) * M) >> 28, n1 = (eq_marks(v.y, kc, k) * M) >> 24;
    const uint32_t n2 = (eq_marks(v.z, kc, k) * M) >> 20, n3 = (eq_marks(v.w, kc, k) * M) >> 16;
    return n0 | (n1 & 0xF0u) | (n2 & 0xF00u) | (n3 & 0xF000u);
}
__device__ __forceinline__ uint32_t collapse4(uint32_t m) {  // bit 0 of every byte -> bits 0..3
    return (((m & 0x01010101u) * 0x00204081u) >> 21) & 0xFu;
}
// bit i set <=> byte i is ASCII whitespace as bytes.strip() sees it: ' ', '\t', '\n', '\v', '\f', '\r'
__device__ __forceinline__ uint32_t ws_mask16(uint4 v) {
    auto nib = [](uint32_t w) { return collapse4(__vcmpeq4(w, 0x20202020u) | (__vcmpgeu4(w, 0x09090909u) & __vcmpleu4(w, 0x0D0D0D0Du))); };
    return nib(v.x) | (nib(v.y) << 4) | (nib(v.z) << 8) | (nib(v.w) << 12);
}
__device__ __forceinline__ uint32_t nl_bits16(uint4 v) {
    auto nib = [](uint32_t w) { return collapse4(__vcmpeq4(w, 0x0A0A0A0Au)); };
    return nib(v.x) | (nib(v.y) << 4) | (nib(v.z) << 8) | (nib(v.w) << 12);
}
// bits of the 16-byte chunk at c that lie inside [b, e)
__device__ __forceinline__ uint32_t range_bits16(uint32_t c, uint32_t b, uint32_t e) {
    uint32_t valid = 0xFFFFu;
    if (c < b) valid &= 0xFFFFu << (b - c);
    if (e - c < 16u) valid &= (1u << (e - c)) - 1u;
    return valid;
}

// Calls f(s, t) for the stripped content [s, t) of every line in [b, e) that is not blank (the last line may lack its
// line end).  The text is 16-byte aligned and zero padded.
template <class F>
__device__ __forceinline__ void for_each_content(const uint8_t* __restrict__ text, uint32_t b, uint32_t e, F f) {
    int64_t first = -1;  // first and last non-blank byte of the current line
    uint32_t last = 0;
    for (uint32_t c = b & ~15u; c < e; c += 16) {
        const uint4 v = *reinterpret_cast<const uint4*>(text + c);
        const uint32_t valid = range_bits16(c, b, e);
        uint32_t nl = nl_bits16(v) & valid, cont = ~ws_mask16(v) & valid;
        for (;;) {
            const uint32_t bit = nl & (0u - nl);            // the next line end (0: none in this chunk)
            const uint32_t seg = bit ? bit - 1u : 0xFFFFu;  // the bytes in front of it
            const uint32_t cs = cont & seg;
            if (cs) {
                if (first < 0) first = c + (uint32_t)(__ffs(cs) - 1);
                last = c + 31u - (uint32_t)__clz(cs);
            }
            if (!bit) break;
            if (first >= 0) f((uint32_t)first, last + 1u);
            first = -1;
            cont &= ~(seg | bit);
            nl &= ~bit;
        }
    }
    if (first >= 0) f((uint32_t)first, last + 1u);
}

// Pass 1: record starts per 16-byte chunk ('>' behind a '\n', or at offset 0) and per tile.
__global__ void __launch_bounds__(TILE_THREADS) k_fa_count(const uint8_t* __restrict__ text, uint64_t bytes,
                                                           uint16_t* __restrict__ masks, uint32_t* __restrict__ tile_cnt) {
    __shared__ uint32_t wsum[TILE_THREADS / 32];
    const uint64_t tile_off = (uint64_t)blockIdx.x * TILE_BYTES;
    uint32_t c = 0;
    const ByteConsts k = byte_consts();
    uint32_t kgt;
    asm volatile("mov.b32 %0, 0x3E3E3E3E;" : "=r"(kgt));
#pragma unroll 4
    for (int i = 0; i < TILE_CHUNKS / TILE_THREADS; i++) {
        const uint32_t chunk = i * TILE_THREADS + threadIdx.x;
        const uint64_t off = tile_off + 16ull * chunk;
        uint32_t m = 0;
        if (off < bytes) {
            const uint4 v = *reinterpret_cast<const uint4*>(text + off);
            const bool line_start = off == 0 || text[off - 1] == '\n';
            m = eq_mask16(v, kgt, k) & (((eq_mask16(v, k.k0a, k) << 1) | (line_start ? 1u : 0u)) & 0xFFFFu);
        }
        masks[(size_t)blockIdx.x * TILE_CHUNKS + chunk] = (uint16_t)m;
        c += __popc(m);
    }
    c = __reduce_add_sync(0xffffffffu, c);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
#pragma unroll
        for (int w = 0; w < TILE_THREADS / 32; w++) t += wsum[w];
        tile_cnt[blockIdx.x] = t;
    }
}

// kinds of a malformed FASTA batch (same key as the FASTQ kinds; 4 = PERR_LIMIT, 5 = PERR_COUNT, 7 = header limit)
enum { PERR_FA_PREAMBLE = 1 };

__global__ void __launch_bounds__(256) k_fa_records(const FastaParams F) {
    const ParseParams& P = F.p;
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool count_ok = P.nl_total[0] == P.n;
    if (i == 0 && !count_ok) report(P.perr, 0, PERR_COUNT);
    if (i >= P.n) return;
    if (!count_ok) {  // hdr[] is not fully defined: every record becomes an empty one, the host rejects the batch
        P.name_off[i] = P.name_end[i] = P.seq_off[i] = P.seq_len[i] = 0;
        P.qual_off[i] = F.qual0;
        F.pad_len[i] = 0;
        return;
    }
    const uint8_t* __restrict__ t = P.text;
    const uint32_t h = P.nl[i], e = i + 1 < P.n ? P.nl[i + 1] : (uint32_t)P.bytes;
    if (i == 0 && h > 0) {  // only blank lines may stand in front of the first header
        bool blank = true;
        for (uint32_t c = 0; c < h && blank; c += 16) {
            const uint4 v = *reinterpret_cast<const uint4*>(t + c);
            blank = (~ws_mask16(v) & range_bits16(c, 0, h)) == 0;
        }
        if (!blank) report(P.perr, 0, PERR_FA_PREAMBLE);
    }
    // the header line ends at the first '\n' behind the '>'
    uint32_t he = e;
    for (uint32_t c = (h + 1) & ~15u; c < e; c += 16) {
        const uint32_t m = nl_bits16(*reinterpret_cast<const uint4*>(t + c)) & range_bits16(c, h + 1, e);
        if (m) {
            he = c + (uint32_t)(__ffs(m) - 1);
            break;
        }
    }
    uint32_t ne = he;
    while (ne > h + 1 && t[ne - 1] == '\r') ne--;
    const uint32_t body = min(he + 1, e);
    uint32_t lines = 0, len = 0, s0 = body;
    for_each_content(t, body, e, [&](uint32_t s, uint32_t x) {
        if (lines == 0) s0 = s;
        len += x - s;
        lines++;
    });
    const bool ok = len <= CSQ_MAX_READ_LEN;
    if (!ok) report(P.perr, i, PERR_LIMIT);
    P.name_off[i] = h + 1;
    P.name_end[i] = ne;
    P.qual_off[i] = F.qual0;
    const bool multi = ok && lines > 1;
    P.seq_off[i] = multi ? body : s0;  // wrapped: where k_fa_compact starts looking
    P.seq_len[i] = ok ? (multi ? (len | FA_MULTI) : len) : 0u;
    F.pad_len[i] = multi ? (len + 15u) & ~15u : 0u;
}

__global__ void __launch_bounds__(256) k_fa_compact(const FastaParams F) {
    const ParseParams& P = F.p;
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) {  // readable, defined bytes behind the last pool record for the 16-byte fetches
        uint4* z = reinterpret_cast<uint4*>(F.pool + F.pool_total[0]);
        for (int q = 0; q < 4; q++) z[q] = make_uint4(0, 0, 0, 0);
    }
    if (i >= P.n) return;
    const uint32_t sl = P.seq_len[i];
    if (!(sl & FA_MULTI)) return;
    const uint32_t len = sl & ~FA_MULTI, off = F.pad_len[i];
    const uint32_t e = i + 1 < P.n ? P.nl[i + 1] : (uint32_t)P.bytes;
    uint8_t* __restrict__ dst = F.pool + off;
    const uint8_t* __restrict__ t = P.text;
    uint32_t w = 0;
    for_each_content(t, P.seq_off[i], e, [&](uint32_t s, uint32_t x) {
        for (uint32_t y = s; y < x; y++) dst[w++] = t[y];
    });
    for (; w & 15u; w++) dst[w] = 0;
    P.seq_off[i] = F.pool0 + off;
    P.seq_len[i] = len;
}

}  // namespace

uint32_t csq_parse_tiles(uint64_t bytes) { return (uint32_t)((bytes + TILE_BYTES - 1) / TILE_BYTES); }

// `tiles` holds u32 tile counts, `masks` the line-end masks, p.nl the line-end offsets.  (A one-pass form - decoupled
// look-back over per-tile status words, the record index written by the thread that owns a line end - moved 357 MB
// instead of ~560 MB per 1 M pairs but took 240 us against 187 us: one latency chain per 16 KiB tile.  Measured in
// round 1, profiles/r01_ncu_onepass_stage_v1.csv, and removed.)
cudaError_t csq_launch_parse(const ParseParams& p, void* tile_buf, uint16_t* masks, cudaStream_t stream) {
    const uint32_t tiles = csq_parse_tiles(p.bytes);
    uint32_t* tile_cnt = (uint32_t*)tile_buf;
    if (tiles) {
        cudaError_t e = cudaMemsetAsync(p.any_cr, 0, 4, stream);
        if (e != cudaSuccess) return e;
        k_nl_count<<<tiles, TILE_THREADS, 0, stream>>>(p.text, p.bytes, masks, tile_cnt, p.any_cr);
        k_tile_scan<<<1, 1024, 0, stream>>>(tiles, tile_cnt, p.nl_total);
        if (p.first_off) {
            e = cudaMemsetAsync(p.first_off, 0, 4, stream);
            if (e != cudaSuccess) return e;
        }
        k_nl_index<<<tiles, TILE_THREADS, 0, stream>>>(masks, tile_cnt, p.nl, 4u * p.n, p.skip, p.first_off);
    } else {
        cudaError_t e = cudaMemsetAsync(p.nl_total, 0, 4, stream);
        if (e != cudaSuccess) return e;
    }
    k_records<<<(p.n + 255) / 256 + (p.n == 0 ? 1 : 0), 256, 0, stream>>>(p);
    return cudaGetLastError();
}

// FASTA: k_fa_count, k_tile_scan, k_nl_index (not for an empty text), k_fa_records, k_tile_scan, k_fa_compact (not
// for an empty batch).
cudaError_t csq_launch_parse_fasta(const FastaParams& f, void* tile_buf, uint16_t* masks, cudaStream_t stream) {
    const ParseParams& p = f.p;
    const uint32_t tiles = csq_parse_tiles(p.bytes);
    uint32_t* tile_cnt = (uint32_t*)tile_buf;
    if (tiles) {
        k_fa_count<<<tiles, TILE_THREADS, 0, stream>>>(p.text, p.bytes, masks, tile_cnt);
        k_tile_scan<<<1, 1024, 0, stream>>>(tiles, tile_cnt, p.nl_total);
        k_nl_index<<<tiles, TILE_THREADS, 0, stream>>>(masks, tile_cnt, p.nl, p.n, 0u, nullptr);
    } else {
        cudaError_t e = cudaMemsetAsync(p.nl_total, 0, 4, stream);
        if (e != cudaSuccess) return e;
    }
    k_fa_records<<<(p.n + 255) / 256 + (p.n == 0 ? 1 : 0), 256, 0, stream>>>(f);
    if (p.n) {
        k_tile_scan<<<1, 1024, 0, stream>>>(p.n, f.pad_len, f.pool_total);
        k_fa_compact<<<(p.n + 255) / 256, 256, 0, stream>>>(f);
    }
    return cudaGetLastError();
}

uint32_t csq_parse_fasta_launches(uint64_t bytes, uint32_t n) { return (csq_parse_tiles(bytes) ? 3u : 0u) + 1u + (n ? 2u : 0u); }
