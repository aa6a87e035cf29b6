// Device decoder of ORDINARY gzip files: one long DEFLATE stream per member, as gzip, pigz and the sequencers' software
// write them.  The algorithm is the one of pinflate.cpp (pugz / rapidgzip: Kerbiriou & Chikhi 2019), with a warp where
// pinflate has a thread, and the block decoder of gz_inflate_core.h (the one k_gz_inflate runs for BGZF members):
//
//   The stream is decoded in ROUNDS of compressed bytes, each cut into SPANS.  Span 0 of a round starts at the exact bit
//   the previous round ended at, with the 32 KiB window known; every other span is speculative.
//   k_gzs_search  (one warp per span 1..): the first span start at or behind the span's nominal cut - a dynamic-Huffman
//                 block header that passes pinflate's plausible_block tests, or a gzip member header.  The lanes test 32
//                 bit positions at once with the cheap tests; the warp checks the survivors in order.
//   k_gzs_decode  (one warp per span): 16-bit symbols behind 32 768 window places (0x8000 | j where the window is
//                 unknown) up to the first block boundary at or behind the next span's start.  Member ends inside a
//                 span are recorded with their CRC-32 and ISIZE.
//   (host)        the chain: a span counts only when the previous span of the chain ended exactly at its start.
//                 Where it did not (a false positive, a span without a start, a span cut short by its capacity), a
//                 continuation decodes from the chain's end.
//   k_gzs_window  (one CTA): the 32 KiB window in front of every span of the chain, in order (the only serial step).
//   k_gzs_resolve (spans x pieces): markers -> bytes, into one text buffer at exclusive-scan offsets, and the CRC-32 of
//                 every segment between member ends (atomicXor of per-piece CRCs shifted by crc_mulmod, as k_gz_check).
//
// The host twin runs the same search / decode / window / resolve code with a group of one lane, driven by the same
// orchestrator (GzStreamInflater::Impl), so that the CPU tests cover the whole algorithm.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <zlib.h>  // crc32_combine()

#include <algorithm>
#include <string>
#include <vector>

#include "csq_internal.h"
#include "gz_core.h"
#include "gz_inflate_core.h"
#include "host_io.h"

void csq_set_error(const char* msg);  // plan.cu

namespace gzs {

using gzi::BitIn;
using gzi::Group;
using gzi::Tables;

constexpr uint32_t WIN = 32768;
constexpr uint32_t MEMBER_CAP = 64;    // member ends one span records; a span stops behind the 64th
constexpr uint32_t PAD = 4096;         // zero bytes behind the uploaded data (a block header and a token batch fit)
constexpr uint32_t PIECE = 65536;      // symbols per CTA of k_gzs_resolve, 256 per thread
constexpr uint64_t NONE = ~0ull;
constexpr int ERR_GARBAGE = 9;         // bytes behind a member that are neither zero padding nor a gzip header

enum Flags : uint32_t { F_KNOWN = 1, F_EOF = 2, F_SHORT = 4, F_FULL = 8 };

struct SpanRec {
    uint64_t start_bit;  // file bit of the first block (NONE: the search found no start)
    uint64_t stop_bit;   // continuations: decode up to the first block boundary at or behind this bit
    uint64_t end_bit;    // where the decode stopped (a block boundary), or the end of the file
    uint16_t* sym;       // WIN window places, then cap symbols
    uint32_t cap;
    uint32_t n_sym;      // symbols produced (behind the window)
    uint32_t n_members;  // member ends recorded
    int32_t status;      // gzi::Status of a failed decode
    uint32_t flags;      // F_KNOWN (in: the window is wins[0]); F_EOF, F_SHORT (the input ran out), F_FULL (out)
    uint32_t pad_;
};
struct MemberEnd {
    uint32_t out_off;  // symbols of the span in front of the member's end
    uint32_t crc, isize;
};
struct ChainRec {
    uint32_t span;
    uint32_t seg0;      // index of its first segment CRC
    uint64_t text_off;  // exclusive scan of n_sym over the chain
};

struct Params {
    const uint8_t* comp;     // file bytes [base_bit / 8, + comp_len), 4-byte aligned, PAD zero bytes behind
    uint64_t comp_len;
    uint64_t base_bit;
    uint64_t round_end_bit;  // the last span stops at the first block boundary at or behind it
    uint64_t span_bits;      // span k >= 1 searches [base_bit + k span_bits, + span_bits) (clamped to the round)
    uint32_t at_file_end;    // comp reaches the end of the file
    uint32_t n_regular;      // spans of the round (continuations follow them in `spans`)
    SpanRec* spans;
    MemberEnd* members;      // [span][MEMBER_CAP]
    const ChainRec* chain;
    uint32_t n_chain;
    uint8_t* wins;           // [n_chain + 1][WIN]: wins[0] is the window in front of the round
    uint8_t* text;
    uint32_t* seg_crc;       // XOR-accumulated: zero before k_gzs_resolve
    const uint32_t* crc_tab; // [0, 256) CRC-32 byte table; [256 + 256 k + b] x^(8 b 256^k) mod P
};

GZI_HD uint64_t bit_pos(const BitIn& b, const uint8_t* comp) { return (uint64_t)(b.p - comp) * 8 - (uint64_t)b.cnt; }
GZI_HD void seek(BitIn& b, const uint8_t* comp, uint64_t bit) {
    gzi::start(b, comp + (bit >> 3));
    gzi::take(b, (int)(bit & 7));
}

// ---- search ----------------------------------------------------------------------------------------------------------
// Cheap tests of a dynamic block header at `bit`: BFINAL = 0, BTYPE = 2, HLIT / HDIST in range, and the code-length
// code not over-subscribed (complete, when all its lengths are within the 64 bits looked at).
GZI_HD bool cheap_dynamic(const uint8_t* comp, uint64_t bit) {
    const uint8_t* q = comp + (bit >> 3);
    uint64_t lo = 0;
    for (int k = 0; k < 8; k++) lo |= (uint64_t)q[k] << (8 * k);
    const int sh = (int)(bit & 7);
    const uint64_t w = sh ? (lo >> sh) | ((uint64_t)q[8] << (64 - sh)) : lo;
    if ((w & 7u) != 4u) return false;
    const uint64_t v = w >> 3;  // 61 bits
    if ((v & 31u) > 29u || ((v >> 5) & 31u) > 29u) return false;
    const int ncode = (int)((v >> 10) & 15u) + 4;
    const int avail = ncode < 15 ? ncode : 15;
    uint32_t kraft = 0;
    for (int i = 0; i < avail; i++) {
        const int l = (int)((v >> (14 + 3 * i)) & 7u);
        if (l) kraft += 128u >> l;
    }
    return !(kraft > 128u || (avail == ncode && kraft != 128u));
}
GZI_HD bool cheap_member(const uint8_t* comp, uint64_t byte) {
    return comp[byte] == 0x1f && comp[byte + 1] == 0x8b && comp[byte + 2] == 8 && !(comp[byte + 3] & 0xE0u);
}
GZI_HD bool texty(uint32_t c) { return (c >= 32 && c < 127) || c == '\n' || c == '\r' || c == '\t'; }

// pinflate's plausible_block: a complete dynamic header whose first symbols (up to 4096) decode to text literals, or
// to a whole block of at least 64 text symbols
template <int LANES>
GZI_HD bool plausible_block(const Params& P, uint64_t bit, Tables& T, const Group<LANES>& G) {
    BitIn b;
    b.end = P.comp + P.comp_len;
    seek(b, P.comp, bit);
    gzi::refill(b);
    gzi::take(b, 3);
    if (gzi::read_dynamic<LANES>(b, T, G) != gzi::OK) return false;
    uint32_t produced = 0;
    for (int k = 0; k < 4096; k++) {
        if (b.p > b.end + 8) return false;
        gzi::refill(b);
        uint32_t e = gzi::decode_entry<gzi::LBITS, 1>(b, T.llut, T.lcount, T.lsym);
        if (e >= 0x01000000u) {
            if (e == 0xFFFFFFFFu) return false;
            if (e & gzi::E_EOB) return produced >= 64;
            if (!texty((e >> 8) & 0xFFu)) return false;
            produced++;
            continue;
        }
        const uint32_t x = e >> 4 & 15u;
        produced += (e >> 8) + gzi::take(b, (int)x);
        gzi::refill_rare(b);
        e = gzi::decode_entry<gzi::DBITS, 2>(b, T.dlut, T.dcount, T.dsym);
        if (e == 0xFFFFFFFFu) return false;
        gzi::take(b, (int)(e >> 4 & 15u));
    }
    return true;
}

// Span k (>= 1): the first start at or behind its nominal cut, NONE when there is none in front of the next cut.
template <int LANES>
GZI_HD uint64_t search_span(const Params& P, uint32_t k, Tables& T, const Group<LANES>& G) {
    const uint64_t from = (uint64_t)k * P.span_bits, round_bits = P.round_end_bit - P.base_bit;
    const uint64_t to = from + P.span_bits < round_bits ? from + P.span_bits : round_bits;
    for (uint64_t base = from; base < to; base += LANES) {
        const uint64_t bit = base + (uint64_t)G.lane;
        const bool cand = bit < to && (((bit & 7) == 0 && cheap_member(P.comp, bit >> 3)) || cheap_dynamic(P.comp, bit));
        uint32_t m = G.ballot(cand);
        while (m) {
            const uint64_t pb = base + (uint64_t)(GZI_FFS(m) - 1);
            m &= m - 1;
            if ((pb & 7) == 0 && cheap_member(P.comp, pb >> 3)) {
                const uint64_t byte = pb >> 3, left = P.comp_len - byte;
                const uint32_t h = gzi::gzip_header_size(P.comp + byte, (uint32_t)(left < 0xFFFFFFFFu ? left : 0xFFFFFFFFu));
                if (h) return P.base_bit + (byte + h) * 8;  // the member's first block, behind its header
            }
            if (cheap_dynamic(P.comp, pb) && plausible_block<LANES>(P, pb, T, G)) return P.base_bit + pb;
        }
    }
    return NONE;
}

// ---- decode ----------------------------------------------------------------------------------------------------------
GZI_HD uint32_t le32(const uint8_t* p) { return p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }

// Span s from R.start_bit up to the first block boundary at or behind `stop`, or to the end of the file.  Stops early
// (at its last block boundary) when the output does not fit (F_FULL), when the 64th member ends (F_FULL) or when the
// uploaded bytes end before the file does (F_SHORT).
template <int LANES>
GZI_HD void decode_span(const Params& P, uint32_t s, uint64_t stop, Tables& T, const Group<LANES>& G) {
    SpanRec& R = P.spans[s];
    MemberEnd* M = P.members + (size_t)s * MEMBER_CAP;
    uint16_t* sym = R.sym;
    const bool known = (R.flags & F_KNOWN) != 0;
    for (uint32_t j = (uint32_t)G.lane; j < WIN; j += LANES) sym[j] = known ? (uint16_t)P.wins[j] : (uint16_t)(0x8000u | j);
    G.sync();
    const uint32_t cap = WIN + R.cap;
    const uint64_t len_bits = P.comp_len * 8;
    BitIn b;
    b.end = P.comp + P.comp_len;
    seek(b, P.comp, R.start_bit - P.base_bit);
    uint32_t out = WIN, n_mem = 0, flags = 0;
    int status = gzi::OK;
    uint64_t end = R.start_bit - P.base_bit;
    bool first = true;
    for (;;) {
        const uint64_t at = bit_pos(b, P.comp);
        if (!first && at + P.base_bit >= stop) {
            end = at;
            break;
        }
        first = false;
        const uint32_t at_out = out;
        int last = 0, rc = at >= len_bits ? (int)gzi::ERR_INPUT : gzi::inflate_block<LANES, uint16_t>(b, sym, out, cap, T, G, &last);
        uint64_t next = 0;  // byte of the next member's first block
        MemberEnd me = {0, 0, 0};
        if (rc == gzi::OK && last) {  // trailer, zero padding, the next member's header or the end of the file
            uint64_t byte = (bit_pos(b, P.comp) + 7) >> 3;
            if (byte + 8 > P.comp_len) {
                rc = gzi::ERR_INPUT;
            } else {
                me = MemberEnd{out - WIN, le32(P.comp + byte), le32(P.comp + byte + 4)};
                byte += 8;
                while (byte < P.comp_len && P.comp[byte] == 0) byte++;
                if (byte < P.comp_len) {
                    const uint64_t left = P.comp_len - byte;
                    const uint32_t h = gzi::gzip_header_size(P.comp + byte, (uint32_t)(left < 0xFFFFFFFFu ? left : 0xFFFFFFFFu));
                    if (h) next = byte + h;
                    else rc = !P.at_file_end && left < 70000 ? (int)gzi::ERR_INPUT : ERR_GARBAGE;  // (a header may end behind the upload)
                } else if (!P.at_file_end) {
                    rc = gzi::ERR_INPUT;
                }
            }
        }
        if (rc == gzi::ERR_OVERRUN) {
            end = at;
            out = at_out;
            flags |= F_FULL;
            break;
        }
        if (rc != gzi::OK) {
            // what is missing may only not have been uploaded yet: stop at the boundary, the next round goes on from it
            if (!P.at_file_end && (rc == gzi::ERR_INPUT || gzi::byte_pos(b) + 16 > b.end)) {
                end = at;
                out = at_out;
                flags |= F_SHORT;
            } else {
                status = rc == gzi::ERR_INPUT && last ? (int)gzi::ERR_TRAILER : rc;
                end = at;
            }
            break;
        }
        if (last) {
            if (G.lane == 0) M[n_mem] = me;
            n_mem++;
            if (!next) {
                end = len_bits;
                flags |= F_EOF;
                break;
            }
            seek(b, P.comp, next * 8);
            if (n_mem == MEMBER_CAP) {
                end = next * 8;
                flags |= F_FULL;
                break;
            }
        }
    }
    G.sync();
    if (G.lane == 0) {
        R.end_bit = P.base_bit + end;
        R.n_sym = out - WIN;
        R.n_members = n_mem;
        R.status = status;
        R.flags |= flags;
    }
}

// regular span s: up to the next span's start (of the first one that has a start), or to the round's end
GZI_HD uint64_t stop_of(const Params& P, uint32_t s) {
    for (uint32_t q = s + 1; q < P.n_regular; q++)
        if (P.spans[q].start_bit != NONE) return P.spans[q].start_bit;
    return P.round_end_bit;
}

// ---- window and resolve ------------------------------------------------------------------------------------------------
// place j of the window behind chain entry c: the last WIN bytes of (window in front of it ++ its output)
GZI_HD void window_place(const Params& P, uint32_t c, uint32_t j) {
    const SpanRec& R = P.spans[P.chain[c].span];
    const uint8_t* w = P.wins + (size_t)c * WIN;
    const int64_t p = (int64_t)R.n_sym - (int64_t)WIN + (int64_t)j;
    uint8_t v;
    if (p < 0) {
        v = w[j + R.n_sym];
    } else {
        const uint16_t s = R.sym[WIN + (size_t)p];
        v = (s & 0x8000u) ? w[s & 0x7FFFu] : (uint8_t)s;
    }
    P.wins[(size_t)(c + 1) * WIN + j] = v;
}

GZI_HD uint32_t crc_shift(const uint32_t* tab, uint32_t crc, uint32_t n) {  // crc32_combine's "n more bytes follow"
    for (int k = 0; k < 4; k++, n >>= 8)
        if (n & 255u) crc = gz::crc_mulmod(tab[256 + 256 * k + (n & 255u)], crc);
    return crc;
}

// symbols [lo, hi) of chain entry c -> text; their CRC-32 per segment, shifted to the segment's end, XOR-ed in
GZI_HD void resolve_range(const Params& P, uint32_t c, uint32_t lo, uint32_t hi, const uint32_t* byte_tab) {
    const ChainRec& C = P.chain[c];
    const SpanRec& R = P.spans[C.span];
    const MemberEnd* M = P.members + (size_t)C.span * MEMBER_CAP;
    const uint8_t* w = P.wins + (size_t)c * WIN;
    const uint16_t* s = R.sym + WIN;
    uint8_t* t = P.text + C.text_off;
    uint32_t seg_lo = 0;
    for (uint32_t g = 0; g <= R.n_members && seg_lo < hi; g++) {
        const uint32_t seg_hi = g < R.n_members ? M[g].out_off : R.n_sym;
        const uint32_t a = lo > seg_lo ? lo : seg_lo, e = hi < seg_hi ? hi : seg_hi;
        if (a < e) {
            uint32_t crc = 0xFFFFFFFFu;
            for (uint32_t i = a; i < e; i++) {
                const uint16_t v = s[i];
                const uint8_t byte = (v & 0x8000u) ? w[v & 0x7FFFu] : (uint8_t)v;
                t[i] = byte;
                crc = byte_tab[(crc ^ byte) & 0xFFu] ^ (crc >> 8);
            }
            const uint32_t v = crc_shift(P.crc_tab, ~crc, seg_hi - e);
#if defined(__CUDA_ARCH__)
            atomicXor(P.seg_crc + C.seg0 + g, v);
#else
            P.seg_crc[C.seg0 + g] ^= v;
#endif
        }
        seg_lo = seg_hi;
    }
}

// ---- kernels -----------------------------------------------------------------------------------------------------------
constexpr int WARPS = 4;  // spans per CTA of k_gzs_search / k_gzs_decode

__device__ __forceinline__ Group<32> warp_group() {
    Group<32> G;
    G.lane = threadIdx.x & 31;
    G.base = 0;
    G.mask = 0xFFFFFFFFu;
    return G;
}

__global__ void __launch_bounds__(WARPS * 32) k_gzs_search(const __grid_constant__ Params P, uint32_t first, uint32_t count) {
    __shared__ Tables tabs[WARPS];
    const uint32_t i = blockIdx.x * WARPS + threadIdx.x / 32;
    if (i >= count) return;
    const uint64_t start = search_span<32>(P, first + i, tabs[threadIdx.x / 32], warp_group());
    if ((threadIdx.x & 31) == 0) P.spans[first + i].start_bit = start;
}

__global__ void __launch_bounds__(WARPS * 32) k_gzs_decode(const __grid_constant__ Params P, uint32_t first, uint32_t count, int find_stop) {
    __shared__ Tables tabs[WARPS];
    const uint32_t i = blockIdx.x * WARPS + threadIdx.x / 32;
    if (i >= count) return;
    const uint32_t s = first + i;
    if (P.spans[s].start_bit == NONE) return;
    decode_span<32>(P, s, find_stop ? stop_of(P, s) : P.spans[s].stop_bit, tabs[threadIdx.x / 32], warp_group());
}

__global__ void __launch_bounds__(1024) k_gzs_window(const __grid_constant__ Params P) {
    for (uint32_t c = 0; c < P.n_chain; c++) {
        for (uint32_t j = threadIdx.x; j < WIN; j += blockDim.x) window_place(P, c, j);
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256) k_gzs_resolve(const __grid_constant__ Params P) {
    __shared__ uint32_t tab[256];
    tab[threadIdx.x] = P.crc_tab[threadIdx.x];
    __syncthreads();
    const uint32_t c = blockIdx.y, n = P.spans[P.chain[c].span].n_sym;
    const uint32_t lo = blockIdx.x * PIECE + threadIdx.x * (PIECE / 256);
    if (lo >= n) return;
    const uint32_t hi = min(lo + PIECE / 256, n);
    resolve_range(P, c, lo, hi, tab);
}

// ---- where the work runs: the device, or the host twin -----------------------------------------------------------------
struct Backend {
    virtual ~Backend() {}
    virtual void* alloc(size_t n) = 0;   // working memory (zero-filled)
    virtual void release(void* p) = 0;
    virtual void* host_alloc(size_t n) = 0;  // staging memory on the host (pinned for the device)
    virtual void host_release(void* p) = 0;
    virtual bool put(void* dst, const void* src, size_t n) = 0;  // host -> working memory, in order
    virtual bool get(void* dst, const void* src, size_t n) = 0;  // working memory -> host, waits for everything in front
    virtual bool copy(void* dst, const void* src, size_t n) = 0;
    virtual bool zero(void* p, size_t n) = 0;
    virtual bool search(const Params& P, uint32_t first, uint32_t count) = 0;
    virtual bool decode(const Params& P, uint32_t first, uint32_t count, bool find_stop) = 0;
    virtual bool window(const Params& P) = 0;
    virtual bool resolve(const Params& P, uint32_t pieces) = 0;
    virtual bool get_behind(void* dst, const void* src, size_t n) = 0;  // -> host behind what is queued, without waiting
    virtual bool wait_behind() = 0;
    std::string err;
};

struct HostBackend : Backend {
    Tables tab;
    uint32_t byte_tab[256];
    HostBackend() { gz::crc_make_table(byte_tab); }
    void* alloc(size_t n) override { return calloc(1, n + 16); }
    void release(void* p) override { free(p); }
    void* host_alloc(size_t n) override { return malloc(n + 16); }
    void host_release(void* p) override { free(p); }
    bool put(void* d, const void* s, size_t n) override { memcpy(d, s, n); return true; }
    bool get(void* d, const void* s, size_t n) override { memcpy(d, s, n); return true; }
    bool copy(void* d, const void* s, size_t n) override { memmove(d, s, n); return true; }
    bool zero(void* p, size_t n) override { memset(p, 0, n); return true; }
    bool search(const Params& P, uint32_t first, uint32_t count) override {
        const Group<1> one = {0, 1u, 0};
        for (uint32_t s = first; s < first + count; s++) P.spans[s].start_bit = search_span<1>(P, s, tab, one);
        return true;
    }
    bool decode(const Params& P, uint32_t first, uint32_t count, bool find_stop) override {
        const Group<1> one = {0, 1u, 0};
        for (uint32_t s = first; s < first + count; s++)
            if (P.spans[s].start_bit != NONE) decode_span<1>(P, s, find_stop ? stop_of(P, s) : P.spans[s].stop_bit, tab, one);
        return true;
    }
    bool window(const Params& P) override {
        for (uint32_t c = 0; c < P.n_chain; c++)
            for (uint32_t j = 0; j < WIN; j++) window_place(P, c, j);
        return true;
    }
    bool resolve(const Params& P, uint32_t) override {
        for (uint32_t c = 0; c < P.n_chain; c++) {
            const uint32_t n = P.spans[P.chain[c].span].n_sym;
            for (uint32_t lo = 0; lo < n; lo += PIECE / 256)
                resolve_range(P, c, lo, std::min(lo + PIECE / 256, n), byte_tab);
        }
        return true;
    }
    bool get_behind(void* d, const void* s, size_t n) override { memcpy(d, s, n); return true; }
    bool wait_behind() override { return true; }
};

struct DeviceBackend : Backend {
    int dev;
    cudaStream_t st = nullptr, cp = nullptr;  // kernels and copies in; text out (behind the next round's decode)
    cudaEvent_t resolved = nullptr, copied = nullptr;
    explicit DeviceBackend(int device) : dev(device) {
        if (!ok(cudaSetDevice(dev)) || !ok(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking)) ||
            !ok(cudaStreamCreateWithFlags(&cp, cudaStreamNonBlocking)) || !ok(cudaEventCreateWithFlags(&resolved, cudaEventDisableTiming)) ||
            !ok(cudaEventCreateWithFlags(&copied, cudaEventDisableTiming)))
            return;
    }
    ~DeviceBackend() override {
        cudaSetDevice(dev);
        if (st) cudaStreamSynchronize(st);
        if (cp) cudaStreamSynchronize(cp);
        if (resolved) cudaEventDestroy(resolved);
        if (copied) cudaEventDestroy(copied);
        if (st) cudaStreamDestroy(st);
        if (cp) cudaStreamDestroy(cp);
    }
    bool ok(cudaError_t e) {
        if (e == cudaSuccess) return true;
        if (err.empty()) err = std::string("CUDA error in the gzip stream decoder: ") + cudaGetErrorString(e);
        return false;
    }
    void* alloc(size_t n) override {
        void* p = nullptr;
        if (!ok(cudaSetDevice(dev)) || !ok(cudaMalloc(&p, n + 16))) return nullptr;
        if (!ok(cudaMemsetAsync(p, 0, n + 16, st)) || !ok(cudaStreamSynchronize(st))) return nullptr;
        return p;
    }
    void release(void* p) override {
        if (p) cudaFree(p);
    }
    void* host_alloc(size_t n) override {
        void* p = nullptr;
        return ok(cudaHostAlloc(&p, n + 16, cudaHostAllocDefault)) ? p : nullptr;
    }
    void host_release(void* p) override {
        if (p) cudaFreeHost(p);
    }
    bool put(void* d, const void* s, size_t n) override { return ok(cudaMemcpyAsync(d, s, n, cudaMemcpyHostToDevice, st)); }
    bool get(void* d, const void* s, size_t n) override {
        return ok(cudaMemcpyAsync(d, s, n, cudaMemcpyDeviceToHost, st)) && ok(cudaStreamSynchronize(st));
    }
    bool copy(void* d, const void* s, size_t n) override { return ok(cudaMemcpyAsync(d, s, n, cudaMemcpyDeviceToDevice, st)); }
    bool zero(void* p, size_t n) override { return ok(cudaMemsetAsync(p, 0, n, st)); }
    bool search(const Params& P, uint32_t first, uint32_t count) override {
        if (!count) return true;
        k_gzs_search<<<(count + WARPS - 1) / WARPS, WARPS * 32, 0, st>>>(P, first, count);
        return ok(cudaGetLastError());
    }
    bool decode(const Params& P, uint32_t first, uint32_t count, bool find_stop) override {
        if (!count) return true;
        k_gzs_decode<<<(count + WARPS - 1) / WARPS, WARPS * 32, 0, st>>>(P, first, count, find_stop ? 1 : 0);
        return ok(cudaGetLastError());
    }
    bool window(const Params& P) override {
        k_gzs_window<<<1, 1024, 0, st>>>(P);
        return ok(cudaGetLastError());
    }
    bool resolve(const Params& P, uint32_t pieces) override {
        k_gzs_resolve<<<dim3(pieces, P.n_chain), 256, 0, st>>>(P);
        return ok(cudaGetLastError());
    }
    bool get_behind(void* d, const void* s, size_t n) override {
        return ok(cudaEventRecord(resolved, st)) && ok(cudaStreamWaitEvent(cp, resolved, 0)) &&
               ok(cudaMemcpyAsync(d, s, n, cudaMemcpyDeviceToHost, cp)) && ok(cudaEventRecord(copied, cp));
    }
    bool wait_behind() override { return ok(cudaEventSynchronize(copied)); }
};

const char* status_text(int s) {
    switch (s) {
        case gzi::ERR_BLOCK: return "invalid DEFLATE block type or stored-block length";
        case gzi::ERR_CODE: return "invalid Huffman code";
        case gzi::ERR_DIST: return "invalid match distance";
        case gzi::ERR_TRAILER: return "gzip trailer missing";
        case gzi::ERR_INPUT: return "the DEFLATE stream ends in the middle of a member";
        case ERR_GARBAGE: return "trailing garbage behind a gzip member";
        default: return "corrupt DEFLATE stream";
    }
}

}  // namespace gzs

// ---- the orchestrator ----------------------------------------------------------------------------------------------------
namespace csqio {

using namespace gzs;

struct GzStreamInflater::Impl {
    Backend* be = nullptr;
    const uint8_t* data = nullptr;
    size_t n = 0;
    uint64_t span_bytes = 0, round_bytes = 0, overhang = 0;
    uint32_t max_spans = 0, span_cap = 0;
    static constexpr uint32_t MAX_CONT = 32;  // continuations per round; a round may end at any chain end
    // working memory (device, or host for the twin)
    uint8_t* w_comp = nullptr;
    SpanRec* w_spans = nullptr;
    MemberEnd* w_members = nullptr;
    uint16_t* w_sym = nullptr;
    std::vector<uint16_t*> w_cont;
    std::vector<uint32_t> cont_cap;
    uint8_t* w_wins = nullptr;
    ChainRec* w_chain = nullptr;
    uint8_t* w_text = nullptr;
    uint32_t* w_seg = nullptr;
    uint32_t* w_crc = nullptr;
    size_t text_cap = 0;
    // staging on the host
    uint8_t* h_comp = nullptr;
    uint8_t* h_text = nullptr;
    size_t h_text_cap = 0;
    std::vector<SpanRec> spans;
    std::vector<MemberEnd> members;
    std::vector<uint32_t> seg;
    // position
    uint64_t next_bit = 0;
    bool finished = false, launched = false;
    uint32_t crc_run = 0;
    uint64_t len_run = 0;
    Params P{};
    std::string error;
    // consumer
    size_t text_n = 0, text_pos = 0;
    bool have_text = false, eof = false;
    std::vector<ChainEntry>* log = nullptr;

    bool fail(const std::string& m) {
        if (error.empty()) error = m.empty() ? std::string("gzip stream decoder failed") : m;
        return false;
    }
    bool be_fail() { return fail(be->err); }
    bool open();
    bool launch_round();
    bool produce();
    uint16_t* sym_of(uint32_t s) const { return w_sym + (size_t)s * (WIN + span_cap); }
    bool grow_text(size_t need);
    void free_all();
};

bool GzStreamInflater::Impl::open() {
    const uint32_t h = n >= 18 ? gzi::gzip_header_size(data, (uint32_t)std::min<size_t>(n, 0xFFFFFFFFu)) : 0;
    if (!h) return fail("not a gzip file");
    next_bit = (uint64_t)h * 8;
    if (!be->err.empty()) return be_fail();
    span_bytes = std::max<uint64_t>(span_bytes, 256);
    round_bytes = std::max<uint64_t>(round_bytes, span_bytes);
    overhang = std::max<uint64_t>(1u << 20, round_bytes / 4);
    const uint64_t per_round = std::min<uint64_t>(round_bytes, n);
    max_spans = (uint32_t)std::min<uint64_t>((per_round + 4 + span_bytes - 1) / span_bytes + 1, 16384);
    span_cap = (uint32_t)std::max<uint64_t>(span_bytes * 8, 512u << 10);
    const size_t comp_cap = (size_t)std::min<uint64_t>(n, round_bytes + overhang) + PAD + 8;
    const size_t n_rec = (size_t)max_spans + MAX_CONT;
    w_comp = (uint8_t*)be->alloc(comp_cap);
    h_comp = (uint8_t*)be->host_alloc(comp_cap);
    w_spans = (SpanRec*)be->alloc(n_rec * sizeof(SpanRec));
    w_members = (MemberEnd*)be->alloc(n_rec * MEMBER_CAP * sizeof(MemberEnd));
    w_sym = (uint16_t*)be->alloc((size_t)max_spans * (WIN + span_cap) * 2);
    w_wins = (uint8_t*)be->alloc((n_rec + 1) * WIN);
    w_chain = (ChainRec*)be->alloc(n_rec * sizeof(ChainRec));
    w_seg = (uint32_t*)be->alloc(n_rec * (MEMBER_CAP + 1) * 4);
    w_crc = (uint32_t*)be->alloc(1280 * 4);
    if (!w_comp || !h_comp || !w_spans || !w_members || !w_sym || !w_wins || !w_chain || !w_seg || !w_crc) return be_fail();
    uint32_t tab[1280];
    gz::crc_make_table(tab);
    for (int k = 0; k < 4; k++)
        for (int b = 0; b < 256; b++) tab[256 + 256 * k + b] = gz::crc_xpow8((uint64_t)b << (8 * k));
    if (!be->put(w_crc, tab, sizeof(tab))) return be_fail();
    spans.resize(n_rec);
    members.resize(n_rec * MEMBER_CAP);
    seg.resize(n_rec * (MEMBER_CAP + 1));
    if (!grow_text((size_t)std::min<uint64_t>((uint64_t)max_spans * span_cap, 256u << 20))) return false;
    return launch_round();
}

bool GzStreamInflater::Impl::grow_text(size_t need) {
    if (need <= text_cap) return true;
    const size_t cap = std::max(need, text_cap * 2);
    be->release(w_text);
    be->host_release(h_text);
    w_text = (uint8_t*)be->alloc(cap);
    h_text = (uint8_t*)be->host_alloc(cap);
    text_cap = w_text && h_text ? cap : 0;
    return text_cap ? true : be_fail();
}

void GzStreamInflater::Impl::free_all() {
    for (void* p : {(void*)w_comp, (void*)w_spans, (void*)w_members, (void*)w_sym, (void*)w_wins, (void*)w_chain, (void*)w_text, (void*)w_seg, (void*)w_crc}) be->release(p);
    for (uint16_t* p : w_cont) be->release(p);
    be->host_release(h_comp);
    be->host_release(h_text);
}

// upload the next round's bytes, search and decode its spans (asynchronously on the device)
bool GzStreamInflater::Impl::launch_round() {
    const uint64_t base = (next_bit >> 3) & ~(uint64_t)3;
    const uint64_t len = std::min<uint64_t>(n - base, round_bytes + overhang);
    const uint64_t round_end = std::min<uint64_t>(n, base + round_bytes);
    memcpy(h_comp, data + base, (size_t)len);
    memset(h_comp + len, 0, PAD);
    P = Params{};
    P.comp = w_comp;
    P.comp_len = len;
    P.base_bit = base * 8;
    P.round_end_bit = round_end * 8;
    P.span_bits = span_bytes * 8;
    P.at_file_end = base + len == n;
    P.n_regular = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(1, (round_end - base + span_bytes - 1) / span_bytes), max_spans);
    P.spans = w_spans;
    P.members = w_members;
    P.wins = w_wins;
    P.chain = w_chain;
    P.text = w_text;
    P.seg_crc = w_seg;
    P.crc_tab = w_crc;
    for (uint32_t k = 0; k < P.n_regular; k++) {
        SpanRec& r = spans[k];
        r = SpanRec{};
        r.start_bit = k == 0 ? next_bit : NONE;
        r.sym = sym_of(k);
        r.cap = span_cap;
        r.flags = k == 0 ? F_KNOWN : 0;
    }
    if (!be->put(w_comp, h_comp, (size_t)len + PAD) || !be->put(w_spans, spans.data(), P.n_regular * sizeof(SpanRec)) ||
        !be->search(P, 1, P.n_regular - 1) || !be->decode(P, 0, P.n_regular, true))
        return be_fail();
    launched = true;
    return true;
}

bool GzStreamInflater::Impl::produce() {
    if (!launched && !launch_round()) return false;
    launched = false;
    const uint32_t S = P.n_regular;
    if (!be->get(spans.data(), w_spans, S * sizeof(SpanRec)) || !be->get(members.data(), w_members, (size_t)S * MEMBER_CAP * sizeof(MemberEnd)))
        return be_fail();
    // ---- the chain ----
    std::vector<uint32_t> chain;
    uint32_t n_cont = 0;
    uint32_t k = 0;
    for (;;) {
        const SpanRec& r = spans[k];
        if (r.status) return fail(status_text(r.status));
        chain.push_back(k);
        if (r.flags & F_EOF) break;
        const uint64_t here = r.end_bit;
        int nxt = -1;
        uint64_t stop = P.round_end_bit;
        for (uint32_t q = 1; q < S; q++)
            if (q != k && spans[q].start_bit != NONE && spans[q].start_bit >= here) {  // (k: when nothing of it fitted)
                if (spans[q].start_bit == here) nxt = (int)q;
                stop = spans[q].start_bit;
                break;
            }
        if (nxt >= 0) {
            k = (uint32_t)nxt;
            continue;
        }
        // the round is complete, or its bytes end here (the next round goes on), or too many continuations
        if (here >= P.round_end_bit || (r.flags & F_SHORT) || n_cont == MAX_CONT) break;
        // continuation: from the chain's end up to the next start behind it; its buffer doubles until a block fits
        const uint32_t c = S + n_cont;
        if (w_cont.size() <= n_cont) {
            w_cont.push_back(nullptr);
            cont_cap.push_back(0);
        }
        uint32_t want = std::max(cont_cap[n_cont], 2 * span_cap);
        for (;;) {
            if (cont_cap[n_cont] < want) {
                be->release(w_cont[n_cont]);
                w_cont[n_cont] = (uint16_t*)be->alloc(((size_t)WIN + want) * 2);
                cont_cap[n_cont] = w_cont[n_cont] ? want : 0;
                if (!w_cont[n_cont]) return be_fail();
            }
            SpanRec& cr = spans[c];
            cr = SpanRec{};
            cr.start_bit = here;
            cr.stop_bit = stop;
            cr.sym = w_cont[n_cont];
            cr.cap = cont_cap[n_cont];
            if (!be->put(w_spans + c, &cr, sizeof(SpanRec)) || !be->decode(P, c, 1, false) || !be->get(&cr, w_spans + c, sizeof(SpanRec)) ||
                !be->get(members.data() + (size_t)c * MEMBER_CAP, w_members + (size_t)c * MEMBER_CAP, MEMBER_CAP * sizeof(MemberEnd)))
                return be_fail();
            if (cr.status || !(cr.flags & F_FULL) || cr.end_bit != here) break;
            if (want >= 0x7FFFFFFFu - WIN) return fail("a DEFLATE block decodes to more than 2 GiB");
            want *= 2;
        }
        if (spans[c].end_bit == here && !spans[c].status && (spans[c].flags & F_SHORT)) break;  // its bytes end here
        n_cont++;
        k = c;
    }
    // a round that ends where it started: its first block is longer than the uploaded bytes
    if (spans[chain.back()].end_bit == next_bit && !(spans[chain.back()].flags & F_EOF)) {
        if (P.at_file_end) return fail("the DEFLATE stream ends in the middle of a member");
        overhang *= 2;
        if (!be->err.empty()) return be_fail();
        const size_t comp_cap = (size_t)std::min<uint64_t>(n, round_bytes + overhang) + PAD + 8;
        be->release(w_comp);
        be->host_release(h_comp);
        w_comp = (uint8_t*)be->alloc(comp_cap);
        h_comp = (uint8_t*)be->host_alloc(comp_cap);
        if (!w_comp || !h_comp) return be_fail();
        return produce();
    }
    // ---- windows, bytes, segment CRCs ----
    std::vector<ChainRec> recs(chain.size());
    std::vector<SpanRec> done(chain.size());  // (launch_round reuses `spans`)
    uint64_t total = 0;
    uint32_t n_seg = 0, pieces = 1;
    for (size_t c = 0; c < chain.size(); c++) {
        const SpanRec& r = done[c] = spans[chain[c]];
        recs[c] = ChainRec{chain[c], n_seg, total};
        total += r.n_sym;
        n_seg += r.n_members + 1;
        pieces = std::max(pieces, (r.n_sym + PIECE - 1) / PIECE);
        if (log) log->push_back(ChainEntry{r.start_bit, r.end_bit, r.n_sym});
    }
    if (!grow_text((size_t)total)) return false;
    P.text = w_text;
    P.chain = w_chain;
    P.n_chain = (uint32_t)chain.size();
    if (!be->put(w_chain, recs.data(), recs.size() * sizeof(ChainRec)) || !be->zero(w_seg, (size_t)n_seg * 4) || !be->window(P) ||
        !be->resolve(P, pieces) || !be->get_behind(seg.data(), w_seg, (size_t)n_seg * 4) || !be->get_behind(h_text, w_text, (size_t)total) ||
        !be->copy(w_wins, w_wins + (size_t)P.n_chain * WIN, WIN))
        return be_fail();
    const SpanRec& tail = done.back();
    next_bit = tail.end_bit;
    finished = (tail.flags & F_EOF) != 0;
    // the next round decodes while this one's text is copied out and consumed
    if (!finished && !launch_round()) return false;
    if (!be->wait_behind()) return be_fail();
    for (size_t c = 0; c < chain.size(); c++) {
        const SpanRec& r = done[c];
        const MemberEnd* M = members.data() + (size_t)chain[c] * MEMBER_CAP;
        uint32_t from = 0;
        for (uint32_t q = 0; q <= r.n_members; q++) {
            const uint32_t to = q < r.n_members ? M[q].out_off : r.n_sym;
            crc_run = (uint32_t)crc32_combine(crc_run, seg[recs[c].seg0 + q], (z_off_t)(to - from));
            len_run += to - from;
            if (q < r.n_members) {
                if (crc_run != M[q].crc) return fail("CRC-32 mismatch in a gzip member");
                if ((uint32_t)len_run != M[q].isize) return fail("length mismatch (ISIZE) in a gzip member");
                crc_run = 0;
                len_run = 0;
            }
            from = to;
        }
    }
    text_n = (size_t)total;
    text_pos = 0;
    have_text = true;
    return true;
}

GzStreamInflater::GzStreamInflater(const uint8_t* data, size_t n, int device, uint64_t span_bytes, uint64_t round_bytes,
                                   std::vector<ChainEntry>* chain_log)
    : p_(new Impl()) {
    p_->data = data;
    p_->n = n;
    p_->log = chain_log;
    const char* es = getenv("CSQ_GZ_STREAM_SPAN");
    const char* er = getenv("CSQ_GZ_STREAM_ROUND");
    p_->span_bytes = span_bytes ? span_bytes : es && atoll(es) > 0 ? (uint64_t)atoll(es) : (128u << 10);
    p_->round_bytes = round_bytes ? round_bytes : er && atoll(er) > 0 ? (uint64_t)atoll(er) : (64u << 20);
    if (device >= 0) p_->be = new DeviceBackend(device);
    else p_->be = new HostBackend();
    p_->open();
}

GzStreamInflater::~GzStreamInflater() {
    if (DeviceBackend* d = dynamic_cast<DeviceBackend*>(p_->be)) cudaSetDevice(d->dev);
    p_->free_all();
    delete p_->be;
    delete p_;
}

const char* GzStreamInflater::error() const { return p_->error.c_str(); }

long GzStreamInflater::read(uint8_t* dst, size_t want) {
    Impl& I = *p_;
    if (!I.error.empty()) return -1;
    if (DeviceBackend* d = dynamic_cast<DeviceBackend*>(I.be))
        if (!d->ok(cudaSetDevice(d->dev))) return I.be_fail(), -1;  // the reader's threads come and go
    size_t done = 0;
    while (done < want) {
        if (!I.have_text) {
            if (I.eof) break;
            if (I.finished) {
                I.eof = true;
                break;
            }
            if (!I.produce()) return -1;
        }
        const size_t c = std::min(want - done, I.text_n - I.text_pos);
        memcpy(dst + done, I.h_text + I.text_pos, c);
        done += c;
        I.text_pos += c;
        if (I.text_pos == I.text_n) I.have_text = false;
    }
    return (long)done;
}

}  // namespace csqio

// ---- C ABI: a whole gzip file in memory ----------------------------------------------------------------------------------
static thread_local std::vector<csqio::ChainEntry> g_last_chain;

static int gz_stream_mem(int device, const uint8_t* src, uint64_t n, uint8_t* dst, uint64_t cap, uint64_t span_bytes,
                         uint64_t round_bytes, uint64_t* out_n) {
    if (!src || !dst || !out_n) {
        csq_set_error("null argument");
        return CSQ_ERR_INVALID;
    }
    g_last_chain.clear();
    csqio::GzStreamInflater gi(src, (size_t)n, device, span_bytes, round_bytes, &g_last_chain);
    uint64_t total = 0;
    for (;;) {
        if (total == cap) {
            uint8_t extra;
            const long more = gi.read(&extra, 1);
            if (more < 0) break;
            if (more > 0) {
                csq_set_error("output buffer too small");
                return CSQ_ERR_CAPACITY;
            }
            *out_n = total;
            return 0;
        }
        const long got = gi.read(dst + total, (size_t)(cap - total));
        if (got < 0) break;
        if (got == 0) {
            *out_n = total;
            return 0;
        }
        total += (uint64_t)got;
    }
    csq_set_error(gi.error());
    return CSQ_ERR_IO;
}

extern "C" int csq_gz_stream_inflate(int device, const uint8_t* src, uint64_t n, uint8_t* dst, uint64_t cap, uint64_t span_bytes,
                                     uint64_t round_bytes, uint64_t* out_n) {
    if (device < 0) {
        csq_set_error("bad device");
        return CSQ_ERR_INVALID;
    }
    return gz_stream_mem(device, src, n, dst, cap, span_bytes, round_bytes, out_n);
}

extern "C" int csq_gz_stream_inflate_host(const uint8_t* src, uint64_t n, uint8_t* dst, uint64_t cap, uint64_t span_bytes, uint64_t round_bytes,
                                          uint64_t* out_n) {
    return gz_stream_mem(-1, src, n, dst, cap, span_bytes, round_bytes, out_n);
}

extern "C" uint64_t csq_gz_stream_chain(uint64_t* out, uint64_t max_entries) {
    const uint64_t k = std::min<uint64_t>(max_entries, g_last_chain.size());
    for (uint64_t i = 0; out && i < k; i++) {
        out[3 * i] = g_last_chain[i].start_bit;
        out[3 * i + 1] = g_last_chain[i].end_bit;
        out[3 * i + 2] = g_last_chain[i].n_sym;
    }
    return g_last_chain.size();
}
