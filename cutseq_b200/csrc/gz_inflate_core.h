// DEFLATE decoder for ONE gzip member by ONE group of LANES cooperating threads (RFC 1951 / 1952).  On the device a
// group is a warp (gz_inflate.cu: one warp per BGZF member, every member of a batch in flight at once); the host twin
// runs the same code with LANES = 1 for the CPU tests.
//
// Every lane of the group runs the whole bit-level decode REDUNDANTLY on the same bits (bit buffer, code tables and
// control flow are warp-uniform: no divergence, no shuffles, shared-memory reads are broadcasts); what the lanes split
// is the byte traffic.  The symbols are decoded LANES tokens at a time - a token is a literal or a match (length,
// distance) - and lane t keeps token t and its place in the output.  Then the tokens are resolved together: literals
// are stored at once; a match whose source lies in front of the first unfinished token is copied by its own lane
// (8 bytes in flight per lane), all such matches side by side, round after round until the batch is done (the
// multi-round resolution of Sitaridi et al., "Massively-parallel lossless data decompression", ICPP 2016); a long
// match is copied by all lanes.  zlib level 1 turns FASTQ into ~93 % matches of 5 - 6 bytes whose sources were
// written a moment ago, i.e. every copy is a round trip to L2: one per ROUND here instead of one per match.
// (The first version ran one THREAD per member: 32 different decoder states per warp serialise completely and a
// batch is only a few hundred warps - 0.4 GB/s; the second copied match by match - 21 GB/s.)
//
// Huffman codes: canonical decoding by code length (counts per length + symbols in code order, as in zlib's
// contrib/puff) is kept as the slow path for long codes and for validation; in front of it a direct table indexed by
// the next LBITS / DBITS input bits answers codes of up to that length in one lookup.  Its entries carry what the
// symbol MEANS (base length or distance and the number of extra bits that follow), so a match costs two lookups and
// no arithmetic on symbol numbers.
#pragma once

#include <stdint.h>

#if defined(__CUDACC__)
#define GZI_HD __host__ __device__ __forceinline__
#else
#define GZI_HD inline
#endif
#if defined(__CUDA_ARCH__)
#define GZI_UNROLL _Pragma("unroll")
#define GZI_FFS(x) __ffs((int)(x))
#else
#define GZI_UNROLL
#define GZI_FFS(x) __builtin_ffs((int)(x))
#endif

#if defined(__GNUC__) && !defined(__CUDA_ARCH__)
// the match copies store v[k] only under the condition they loaded it under
#pragma GCC diagnostic push
#pragma GCC diagnostic ignored "-Wmaybe-uninitialized"
#endif

namespace gzi {

// The cooperating lanes: a whole warp or an aligned part of one (LANES = 16: two members per warp, each instruction
// issued for the warp decodes both - the decode is redundant across the lanes of a group, so narrower groups waste
// less of the machine, as long as the two halves mostly follow the same path); the host twin is a group of one.
template <int LANES>
struct Group {
    int lane;       // 0 .. LANES - 1
    uint32_t mask;  // the group's lanes within the warp
    int base;       // warp lane of lane 0
#if defined(__CUDA_ARCH__)
    __device__ __forceinline__ void sync() const { __syncwarp(mask); }
    __device__ __forceinline__ uint32_t ballot(bool p) const { return (__ballot_sync(mask, p) >> base) & (LANES == 32 ? 0xFFFFFFFFu : ((1u << (LANES & 31)) - 1u)); }
    __device__ __forceinline__ uint32_t shfl(uint32_t v, int src) const { return __shfl_sync(mask, v, src, LANES); }
#else
    void sync() const {}
    uint32_t ballot(bool p) const { return p ? 1u : 0u; }
    uint32_t shfl(uint32_t v, int) const { return v; }
#endif
};

constexpr int MAXBITS = 15, MAXLCODES = 286, MAXDCODES = 30, FIXLCODES = 288;
constexpr int LBITS = 10, DBITS = 8;  // index bits of the direct tables

// (8 and up: 7 is k_gz_check's CRC-32 mismatch)
enum Status { OK = 0, ERR_HEADER = 1, ERR_BLOCK = 2, ERR_CODE = 3, ERR_DIST = 4, ERR_OVERRUN = 5, ERR_TRAILER = 6, ERR_INPUT = 8 };

struct Tables {  // per group (device: shared memory, 6.1 KB per group)
    // entries: code length [3:0] | extra bits [7:4] | base value [23:8] | LIT bit 31 | EOB bit 30; 0: the code is longer
    // than the index (or invalid).  Base value: the literal, the length base (3..258) or the distance base (1..24577);
    // the code-length code keeps its symbol there.
    uint32_t llut[1 << LBITS];
    uint32_t dlut[1 << DBITS];
    uint16_t lcount[MAXBITS + 1], dcount[MAXBITS + 1];  // codes per length
    uint16_t lsym[FIXLCODES], dsym[32];                 // symbols in code order
    uint8_t lengths[MAXLCODES + MAXDCODES + 4];
};

struct BitIn {
    const uint8_t* p;    // next input word (4-byte aligned)
    const uint8_t* end;  // one past the member
    uint64_t buf;
    int cnt;
};

// Input is read in aligned 32-bit words (the compressed buffer is padded, and reading the bytes in front of a member
// is harmless): starting at byte address q means loading the word that holds it and dropping the bytes in front.
GZI_HD void start(BitIn& b, const uint8_t* q) {
    const uint32_t mis = (uint32_t)((uintptr_t)q & 3u);
    const uint32_t w = *reinterpret_cast<const uint32_t*>(q - mis);
    b.buf = (uint64_t)(w >> (8u * mis));
    b.cnt = 32 - 8 * (int)mis;
    b.p = q - mis + 4;
}
GZI_HD const uint8_t* byte_pos(const BitIn& b) { return b.p - (b.cnt >> 3); }  // next unread byte (at a byte boundary)
GZI_HD void refill(BitIn& b) {  // at least 33 bits afterwards (whatever lies behind the member: zeros or the next one)
    if (b.cnt <= 32) {
        const uint32_t w = *reinterpret_cast<const uint32_t*>(b.p);
        b.buf |= (uint64_t)w << b.cnt;
        b.cnt += 32;
        b.p += 4;
    }
}
// The same where the word is seldom needed (a distance behind a length: up to 28 bits, ~25 left on average): written
// as a loop so that the compiler branches around it instead of predicating its eight instructions
GZI_HD void refill_rare(BitIn& b) {
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    while (b.cnt < 28) {
        const uint32_t w = *reinterpret_cast<const uint32_t*>(b.p);
        b.buf |= (uint64_t)w << b.cnt;
        b.cnt += 32;
        b.p += 4;
    }
}
GZI_HD uint32_t take(BitIn& b, int n) {  // n <= 16, after refill
    const uint32_t v = (uint32_t)b.buf & ((1u << n) - 1u);
    b.buf >>= n;
    b.cnt -= n;
    return v;
}

// canonical decode, one bit at a time (codes the direct table does not hold)
GZI_HD int decode_slow(BitIn& b, const uint16_t* count, const uint16_t* symbol) {
    int code = 0, first = 0, index = 0;
    uint32_t bits = (uint32_t)b.buf;
    for (int len = 1; len <= MAXBITS; len++) {
        code |= (int)(bits & 1u);
        bits >>= 1;
        const int c = count[len];
        if (code - c < first) {
            b.buf >>= len;
            b.cnt -= len;
            return symbol[index + (code - first)];
        }
        index += c;
        first += c;
        first <<= 1;
        code <<= 1;
    }
    return -1;
}

constexpr uint32_t E_LIT = 0x80000000u, E_EOB = 0x40000000u;
// what a symbol of one of the three alphabets means, as a table entry without the code length
GZI_HD uint32_t entry_litlen(uint32_t s) {
    if (s < 256u) return E_LIT | (s << 8);
    if (s == 256u) return E_EOB;
    const uint32_t ls = s - 257u;
    if (ls >= 29u) return 0xFFFFFFFFu;  // not a symbol
    if (ls < 8u) return (3u + ls) << 8;
    if (ls == 28u) return 258u << 8;
    const uint32_t x = (ls >> 2) - 1u;
    return ((((4u + (ls & 3u)) << x) + 3u) << 8) | (x << 4);
}
GZI_HD uint32_t entry_dist(uint32_t ds) {
    if (ds >= 30u) return 0xFFFFFFFFu;
    if (ds < 4u) return (1u + ds) << 8;
    const uint32_t x = (ds >> 1) - 1u;
    return ((((2u + (ds & 1u)) << x) + 1u) << 8) | (x << 4);
}
template <int KIND>  // 0: plain symbols (the code-length code), 1: literal / length, 2: distance
GZI_HD uint32_t entry_of(uint32_t s) {
    return KIND == 0 ? (s << 8) : KIND == 1 ? entry_litlen(s) : entry_dist(s);
}

// next symbol as an entry WITHOUT its code length (those bits are consumed here, the extra bits are not);
// 0xFFFFFFFF: invalid code
template <int BITS, int KIND>
GZI_HD uint32_t decode_entry(BitIn& b, const uint32_t* lut, const uint16_t* count, const uint16_t* symbol) {
    const uint32_t e = lut[(uint32_t)b.buf & ((1u << BITS) - 1u)];
    if (e) {
        const int n = (int)(e & 15u);
        b.buf >>= n;
        b.cnt -= n;
        return e & ~15u;
    }
    const int sym = decode_slow(b, count, symbol);
    return sym < 0 ? 0xFFFFFFFFu : entry_of<KIND>((uint32_t)sym);
}

GZI_HD uint32_t bit_reverse(uint32_t v, int n) {  // the low n bits of v, reversed
#if defined(__CUDA_ARCH__)
    return __brev(v) >> (32 - n);
#else
    uint32_t r = 0;
    for (int i = 0; i < n; i++) r |= ((v >> i) & 1u) << (n - 1 - i);
    return r;
#endif
}

// Code lengths (already in shared memory, visible to every lane) -> counts per length, symbols in code order (lane 0)
// and the direct table (all lanes).  Returns < 0 for an over-subscribed set, > 0 for an incomplete one (only
// acceptable for a single code of one bit, checked by the caller), 0 when complete.  The group is synchronised on
// return.
template <int LANES, int BITS, int KIND>
GZI_HD int construct(uint16_t* count, uint16_t* symbol, uint32_t* lut, const uint8_t* length, int n, const Group<LANES>& G) {
    const int lane = G.lane;
    // every lane derives the counts per length for itself (registers), lane 0 publishes them
    uint32_t cnt[MAXBITS + 1];
    GZI_UNROLL
    for (int len = 0; len <= MAXBITS; len++) cnt[len] = 0;
    for (int s = 0; s < n; s++) {
        const int l = length[s];
        GZI_UNROLL
        for (int len = 0; len <= MAXBITS; len++) cnt[len] += (l == len) ? 1u : 0u;
    }
    int left = 1;
    bool over = false;
    GZI_UNROLL
    for (int len = 1; len <= MAXBITS; len++) {
        left <<= 1;
        left -= (int)cnt[len];
        over = over || left < 0;
    }
    if ((int)cnt[0] == n) left = 0;  // no codes at all
    // offs[len]: index of the first symbol of that length in code order; first[len]: its code
    uint32_t offs[MAXBITS + 2], first[MAXBITS + 2];
    offs[1] = 0;
    first[1] = 0;
    GZI_UNROLL
    for (int len = 1; len <= MAXBITS; len++) {
        offs[len + 1] = offs[len] + cnt[len];
        first[len + 1] = (first[len] + cnt[len]) << 1;
    }
    G.sync();  // the previous tables are not read any more
    if (lane == 0) {
        GZI_UNROLL
        for (int len = 0; len <= MAXBITS; len++) count[len] = (uint16_t)cnt[len];
    }
    for (int e = lane; e < (1 << BITS); e += LANES) lut[e] = 0;
    if (over) {
        G.sync();
        return -1;
    }
    if (lane == 0) {
        uint32_t next[MAXBITS + 1];
        GZI_UNROLL
        for (int len = 1; len <= MAXBITS; len++) next[len] = offs[len];
        for (int s = 0; s < n; s++) {
            const int l = length[s];
            if (l == 0) continue;
            uint32_t at = 0;
            GZI_UNROLL
            for (int len = 1; len <= MAXBITS; len++)
                if (l == len) at = next[len]++;
            symbol[at] = (uint16_t)s;
        }
    }
    G.sync();
    // direct table: the symbol at position idx of the code order has the code first[l] + (idx - offs[l]) of l bits,
    // MSB first in the stream, i.e. bit-reversed in the (LSB first) bit buffer; every index whose low l bits equal it
    const int total = (int)offs[MAXBITS + 1];
    for (int idx = lane; idx < total; idx += LANES) {
        const int s = symbol[idx];
        const int l = length[s];
        if (l > BITS) continue;
        uint32_t f = 0, o = 0;
        GZI_UNROLL
        for (int len = 1; len <= MAXBITS; len++)
            if (l == len) {
                f = first[len];
                o = offs[len];
            }
        const uint32_t code = f + ((uint32_t)idx - o);
        const uint32_t meaning = entry_of<KIND>((uint32_t)s);
        if (meaning == 0xFFFFFFFFu) continue;  // 286, 287 / 30, 31: the slow path reports them
        const uint32_t entry = meaning | (uint32_t)l;
        for (uint32_t e = bit_reverse(code, l); e < (1u << BITS); e += 1u << l) lut[e] = entry;
    }
    G.sync();
    return left;
}

// `len` bytes at d are the bytes `dist` in front of them, by all lanes: byte i of the match is byte (i mod dist) of the
// `dist` bytes in front of it, which all exist already - no lane waits for another one's store.  The loads of a long
// copy are issued before its first store.
template <int LANES, typename Sym>
GZI_HD void copy_match(Sym* d, uint32_t dist, uint32_t len, int lane) {  // (no synchronisation inside)
    const Sym* sp = d - dist;
    if (dist >= len) {
        if (len <= (uint32_t)LANES) {
            if ((uint32_t)lane < len) d[lane] = sp[lane];
        } else {
            for (uint32_t base = 0; base < len; base += 4u * LANES) {
                Sym v[4];
                GZI_UNROLL
                for (uint32_t k = 0; k < 4; k++) {
                    const uint32_t i = base + k * LANES + (uint32_t)lane;
                    if (i < len) v[k] = sp[i];
                }
                GZI_UNROLL
                for (uint32_t k = 0; k < 4; k++) {
                    const uint32_t i = base + k * LANES + (uint32_t)lane;
                    if (i < len) d[i] = v[k];
                }
            }
        }
    } else if (dist == 1) {  // a run of one byte
        const Sym c = sp[0];
        for (uint32_t i = (uint32_t)lane; i < len; i += LANES) d[i] = c;
    } else {  // a period shorter than the match
        uint32_t r = (uint32_t)lane % dist;
        const uint32_t step = (uint32_t)LANES % dist;
        for (uint32_t i = (uint32_t)lane; i < len; i += LANES) {
            d[i] = sp[r];
            r += step;
            if (r >= dist) r -= dist;
        }
    }
}

// Dynamic block header at the reader's position (behind the 3 header bits) -> both codes in T.  The code-length code
// must be complete, the literal/length code must have an end-of-block code, and an incomplete code is only accepted for
// a single code of one bit.
template <int LANES>
GZI_HD int read_dynamic(BitIn& b, Tables& T, const Group<LANES>& G) {
    const int lane = G.lane;
    refill(b);
    const int nlen = (int)take(b, 5) + 257, ndist = (int)take(b, 5) + 1, ncode = (int)take(b, 4) + 4;
    if (nlen > MAXLCODES || ndist > MAXDCODES) return ERR_CODE;
    // the code-length code: 19 lengths of 3 bits in a fixed order, read by every lane, stored by lane 0
    uint32_t packed[2] = {0, 0};  // 19 x 3 bits, by position in the stream
    for (int idx = 0; idx < ncode; idx++) {
        refill(b);
        const uint32_t v = take(b, 3);
        if (idx < 10)
            packed[0] |= v << (3 * idx);
        else
            packed[1] |= v << (3 * (idx - 10));
    }
    G.sync();
    if (lane == 0) {
        const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
        for (int idx = 0; idx < 19; idx++) {
            const uint32_t v = idx < 10 ? (packed[0] >> (3 * idx)) & 7u : (packed[1] >> (3 * (idx - 10))) & 7u;
            T.lengths[order[idx]] = (uint8_t)(idx < ncode ? v : 0u);
        }
    }
    G.sync();
    // its tables live where the distance tables will be (19 symbols, codes of at most 7 bits <= DBITS)
    if (construct<LANES, DBITS, 0>(T.dcount, T.dsym, T.dlut, T.lengths, 19, G) != 0) return ERR_CODE;  // must be complete
    int idx = 0, prev = 0;
    bool have_eob = false;
    while (idx < nlen + ndist) {
        refill(b);
        const uint32_t ce = decode_entry<DBITS, 0>(b, T.dlut, T.dcount, T.dsym);
        if (ce == 0xFFFFFFFFu) return ERR_CODE;
        const int sym = (int)(ce >> 8);
        int rep = 1, val = sym;
        if (sym == 16) {
            if (idx == 0) return ERR_CODE;
            val = prev;
            rep = 3 + (int)take(b, 2);
        } else if (sym == 17) {
            val = 0;
            rep = 3 + (int)take(b, 3);
        } else if (sym == 18) {
            val = 0;
            rep = 11 + (int)take(b, 7);
        }
        if (idx + rep > nlen + ndist) return ERR_CODE;
        if (val != 0 && idx <= 256 && idx + rep > 256) have_eob = true;
        // literal/length lengths at [0, nlen), distance lengths behind them at [nlen, nlen + ndist)
        for (int r = lane; r < rep; r += LANES) T.lengths[idx + r] = (uint8_t)val;
        idx += rep;
        prev = val;
    }
    if (!have_eob) return ERR_CODE;  // no end-of-block code
    G.sync();
    // the distance code first: the code-length tables in its place are done with
    int err = construct<LANES, DBITS, 2>(T.dcount, T.dsym, T.dlut, T.lengths + nlen, ndist, G);
    if (err < 0 || (err > 0 && ndist - (int)T.dcount[0] != 1)) return ERR_CODE;
    err = construct<LANES, LBITS, 1>(T.lcount, T.lsym, T.llut, T.lengths, nlen, G);
    if (err < 0 || (err > 0 && nlen - (int)T.lcount[0] != 1)) return ERR_CODE;
    return OK;
}

// One DEFLATE block at the reader's position -> dst[out ..), out advanced; *last = its BFINAL bit.  Sym is the output
// type: bytes for a gzip member, 16-bit symbols for a span of a stream decoded without its window (gz_stream.cu: a
// reference in front of the span copies the marker 0x8000 | place like any byte).  dst[0 .. out) is what a distance
// may reach.  ERR_OVERRUN: the block does not fit in cap (nothing past cap is written); ERR_INPUT: it runs past b.end.
template <int LANES, typename Sym>
GZI_HD int inflate_block(BitIn& b, Sym* dst, uint32_t& out, uint32_t cap, Tables& T, const Group<LANES>& G, int* last) {
    const int lane = G.lane;
    refill(b);
    *last = (int)take(b, 1);
    const uint32_t type = take(b, 2);
    if (type == 0) {  // stored
        take(b, b.cnt & 7);  // to the byte boundary
        refill(b);
        const uint32_t len = take(b, 16);
        refill(b);
        const uint32_t nlen = take(b, 16);
        if ((len ^ 0xFFFFu) != nlen) return ERR_BLOCK;
        const uint8_t* q = byte_pos(b);  // the whole bytes in the bit buffer are given back
        if (q + len > b.end) return ERR_INPUT;
        if (out + len > cap) return ERR_OVERRUN;
        for (uint32_t i = (uint32_t)lane; i < len; i += LANES) dst[out + i] = q[i];
        out += len;
        start(b, q + len);
        return OK;
    }
    if (type == 3) return ERR_BLOCK;
    if (type == 1) {  // fixed codes
        G.sync();
        for (int s = lane; s < FIXLCODES; s += LANES) T.lengths[s] = (uint8_t)(s < 144 ? 8 : s < 256 ? 9 : s < 280 ? 7 : 8);
        for (int s = lane; s < MAXDCODES; s += LANES) T.lengths[FIXLCODES + s] = 5;
        G.sync();
        construct<LANES, LBITS, 1>(T.lcount, T.lsym, T.llut, T.lengths, FIXLCODES, G);
        construct<LANES, DBITS, 2>(T.dcount, T.dsym, T.dlut, T.lengths + FIXLCODES, MAXDCODES, G);
    } else {  // dynamic codes
        const int rc = read_dynamic<LANES>(b, T, G);
        if (rc != OK) return rc;
    }
    constexpr uint32_t CHUNK = 8;           // bytes a lane has in flight
    constexpr uint32_t SHORT = 2 * CHUNK;   // longer matches are copied by all lanes
    bool eob = false;
    while (!eob) {  // batches of up to LANES tokens
        // a batch reads at most LANES * 6 bytes: the input is padded behind b.end
        if (b.p > b.end + 8) return ERR_INPUT;
        uint32_t my_off = 0, my_tok = 0;  // token `lane`: distance << 16 | length, or (distance 0) the literal
        uint32_t ntok = 0;
        while (ntok < (uint32_t)LANES) {
            refill(b);
            uint32_t e = decode_entry<LBITS, 1>(b, T.llut, T.lcount, T.lsym);
            uint32_t len = 1, tok;
            if (e >= 0x01000000u) {  // a literal, the end of the block or an invalid code
                if (e == 0xFFFFFFFFu) return ERR_CODE;
                if (e & E_EOB) {
                    eob = true;
                    break;
                }
                tok = (e >> 8) & 0xFFu;
            } else {  // a match: base length + extra bits, then the distance likewise
                const uint32_t x = e >> 4 & 15u;
                len = (e >> 8) + ((uint32_t)b.buf & ~(0xFFFFFFFFu << x));
                b.buf >>= x;
                b.cnt -= (int)x;
                refill_rare(b);
                e = decode_entry<DBITS, 2>(b, T.dlut, T.dcount, T.dsym);
                if (e == 0xFFFFFFFFu) return ERR_DIST;
                const uint32_t y = e >> 4 & 15u;
                const uint32_t dist = (e >> 8) + ((uint32_t)b.buf & ~(0xFFFFFFFFu << y));
                b.buf >>= y;
                b.cnt -= (int)y;
                if (dist > out) return ERR_DIST;
                tok = (dist << 16) | len;
            }
            if ((uint32_t)lane == ntok) {
                my_off = out;
                my_tok = tok;
            }
            out += len;
            ntok++;
        }
        if (out > cap) return ERR_OVERRUN;  // nothing of the batch has been written yet
        const uint32_t my_dist = my_tok >> 16, my_len = my_dist ? (my_tok & 0xFFFFu) : 1u, my_lit = my_tok & 0xFFu;
        // ---- resolve the batch ----
        bool pending = (uint32_t)lane < ntok;
        if (pending && my_dist == 0) {
            dst[my_off] = (Sym)my_lit;
            pending = false;
        }
        G.sync();  // literals, stored blocks and earlier batches are visible to every lane
        for (;;) {
            const uint32_t wait = G.ballot(pending);
            if (!wait) break;
            const int first = GZI_FFS(wait) - 1;
            const uint32_t upto = G.shfl(my_off, first);  // every byte in front of the first unfinished token is written
            const uint32_t flen = G.shfl(my_len, first);
            if (flen > SHORT) {  // a long match: its source is complete, all lanes copy it
                copy_match<LANES, Sym>(dst + upto, G.shfl(my_dist, first), flen, lane);
                if (lane == first) pending = false;
            } else {
                // short matches whose source is complete (the first unfinished one always is), each by its own lane;
                // byte i is byte (i mod dist) of the dist bytes in front of the match.  (Exact dependencies - the
                // tokens of the batch that write the source instead of "everything in front of the first unfinished
                // one" - need fewer rounds but 64 shuffles per batch and 26 more registers: measured, slower.)
                const bool ready = pending && my_len <= SHORT && my_off - my_dist + (my_len < my_dist ? my_len : my_dist) <= upto;
                const bool more = G.ballot(ready && my_len > CHUNK) != 0;
                if (ready) {
                    Sym* d = dst + my_off;
                    const Sym* sp = d - my_dist;
                    uint32_t r = 0;
                    Sym v[CHUNK];
                    GZI_UNROLL
                    for (uint32_t k = 0; k < CHUNK; k++)
                        if (k < my_len) {
                            v[k] = sp[r];
                            r = r + 1 == my_dist ? 0 : r + 1;
                        }
                    GZI_UNROLL
                    for (uint32_t k = 0; k < CHUNK; k++)
                        if (k < my_len) d[k] = v[k];
                    if (more) {  // (uniform) the second half of the longer ones
                        GZI_UNROLL
                        for (uint32_t k = CHUNK; k < SHORT; k++)
                            if (k < my_len) {
                                v[k - CHUNK] = sp[r];
                                r = r + 1 == my_dist ? 0 : r + 1;
                            }
                        GZI_UNROLL
                        for (uint32_t k = CHUNK; k < SHORT; k++)
                            if (k < my_len) d[k] = v[k - CHUNK];
                    }
                    pending = false;
                }
            }
            G.sync();  // this round's stores are visible to the next one's loads
        }
    }
    return OK;
}

// Byte offset of the first DEFLATE block of the gzip member whose header starts at src[0] (n bytes readable), 0 when
// the header is not one (magic, CM = 8, reserved FLG bits clear) or does not end inside the n bytes.
GZI_HD uint32_t gzip_header_size(const uint8_t* src, uint32_t n) {
    if (n < 18 || src[0] != 0x1f || src[1] != 0x8b || src[2] != 8 || (src[3] & 0xE0u)) return 0;
    const uint32_t flg = src[3];
    uint32_t pos = 10;
    if (flg & 4u) pos = 12 + (src[10] | ((uint32_t)src[11] << 8));
    if (flg & 8u) {
        while (pos < n && src[pos]) pos++;
        pos++;
    }
    if (flg & 16u) {
        while (pos < n && src[pos]) pos++;
        pos++;
    }
    if (flg & 2u) pos += 2;
    return pos < n ? pos : 0;
}

// One gzip member src[0 .. n) -> dst[0 .. cap).  *produced = bytes written (valid in every lane).  Checks ISIZE and
// that the member ends where it should; the CRC-32 of the text is verified by the caller (k_gz_check / the host twin).
template <int LANES>
GZI_HD int inflate_member(const uint8_t* src, uint32_t n, uint8_t* dst, uint32_t cap, Tables& T, const Group<LANES>& G, uint32_t* produced) {
    *produced = 0;
    // gzip header (RFC 1952): magic, CM = 8, FLG, MTIME(4), XFL, OS, then the optional fields
    if (n < 18 || src[0] != 0x1f || src[1] != 0x8b || src[2] != 8) return ERR_HEADER;
    const uint32_t flg = src[3];
    uint32_t pos = 10;
    if (flg & 4u) {
        const uint32_t xlen = src[10] | ((uint32_t)src[11] << 8);
        pos = 12 + xlen;
    }
    if (flg & 8u) {
        while (pos < n && src[pos]) pos++;
        pos++;
    }
    if (flg & 16u) {
        while (pos < n && src[pos]) pos++;
        pos++;
    }
    if (flg & 2u) pos += 2;
    if (pos + 8 > n) return ERR_HEADER;
    BitIn b;
    b.end = src + n;
    start(b, src + pos);
    uint32_t out = 0;  // bytes produced
    int last;
    do {
        const int rc = inflate_block<LANES, uint8_t>(b, dst, out, cap, T, G, &last);
        if (rc != OK) return rc;
    } while (!last);
    G.sync();
    // trailer: CRC-32 (verified by the caller), ISIZE
    const uint8_t* tr = byte_pos(b);
    if (tr + 8 > b.end) return ERR_TRAILER;
    const uint32_t isize = tr[4] | ((uint32_t)tr[5] << 8) | ((uint32_t)tr[6] << 16) | ((uint32_t)tr[7] << 24);
    if (isize != out) return ERR_TRAILER;
    *produced = out;
    return OK;
}

}  // namespace gzi

#if defined(__GNUC__) && !defined(__CUDA_ARCH__)
#pragma GCC diagnostic pop
#endif
