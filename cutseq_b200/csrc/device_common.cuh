// Device helpers shared by kernels.cu and prefilter.cu: per-read interval state, the O(1) ops and the DP column range.
#pragma once

#include "csq_internal.h"

namespace {

// CUT / COND_CUT / RENAME(capture) on the interval state (SURVEY.md table 8.1b).
__device__ __forceinline__ void apply_scalar(const DevOp& op, ReadState& st) {
    const int len = (int)st.b - (int)st.a;
    if (op.kind == CSQ_OP_RENAME) {
        st.ren_cp = st.cp;
        st.ren_cs = st.cs;
        return;
    }
    if (op.kind == CSQ_OP_COND_CUT && !(st.matched & 0x80000000u) && len < op.fmin) return;  // run.py:154-155
    if (op.kind == CSQ_OP_CUT || op.kind == CSQ_OP_COND_CUT) {
        if (op.length > 0) {
            const int c = min(op.length, len);
            st.cp = ((uint32_t)st.a << 16) | (uint32_t)c;
            st.a = (uint16_t)(st.a + c);
        } else if (op.length < 0) {
            const int c = min(-op.length, len);
            st.cs = ((uint32_t)(st.b - c) << 16) | (uint32_t)c;
            st.b = (uint16_t)(st.b - c);
        }
    }
}

__device__ __forceinline__ ReadState fresh_state(uint32_t len) {
    ReadState st;
    st.a = 0;
    st.b = (uint16_t)len;
    st.matched = 0;
    st.cp = st.cs = st.ren_cp = st.ren_cs = 0;
    st.id_start = st.id_end = 0;
    st.qtrim = 0;
    return st;
}

__device__ __forceinline__ ReadState load_state(const ReadState* p) {
    const uint4* q = reinterpret_cast<const uint4*>(p);
    uint4 x = q[0], y = q[1];
    ReadState st;
    st.a = (uint16_t)(x.x & 0xFFFFu);
    st.b = (uint16_t)(x.x >> 16);
    st.matched = x.y;
    st.cp = x.z;
    st.cs = x.w;
    st.ren_cp = y.x;
    st.ren_cs = y.y;
    st.id_start = (uint16_t)(y.z & 0xFFFFu);
    st.id_end = (uint16_t)(y.z >> 16);
    st.qtrim = y.w;
    return st;
}

__device__ __forceinline__ void store_state(ReadState* p, const ReadState& st) {
    uint4* q = reinterpret_cast<uint4*>(p);
    q[0] = make_uint4((uint32_t)st.a | ((uint32_t)st.b << 16), st.matched, st.cp, st.cs);
    q[1] = make_uint4(st.ren_cp, st.ren_cs, (uint32_t)st.id_start | ((uint32_t)st.id_end << 16), st.qtrim);
}

// State of read idx in front of an ALIGN op: fresh for the first one, else as the previous op left it; then the
// scalar ops between the two.
__device__ __forceinline__ ReadState entry_state(const AlignParams& P, uint32_t idx) {
    ReadState st = P.first ? fresh_state(P.md.seq_len[idx]) : load_state(P.md.state + idx);
    for (int q = 0; q < P.n_pre; q++) apply_scalar(P.pre[q], st);
    return st;
}

// DP columns min_n < j <= max_n of Aligner.locate on a read of n characters: without a free read start (siq, flags
// bit 2) an alignment of m characters and at most k errors ends by column m + k, without a free read end (eiq, flags
// bit 8) it starts at column n - m - k or later.
__device__ __forceinline__ void column_range(bool siq, bool eiq, int m, int k, int n, int& min_n, int& max_n) {
    max_n = siq ? n : min(n, m + k);
    min_n = eiq ? 0 : max(0, n - m - k);
}

__device__ __forceinline__ csq_match no_match() { return csq_match{}; }  // found = 0, every field 0


// 16 bytes from an arbitrary byte address: TWO aligned 128-bit loads, a select network for the word offset and four
// funnel shifts for the byte offset.  Every thread of a warp reads its own record, so a load instruction costs one
// L1 wavefront per thread whatever its width: five 32-bit loads per 16 bytes (the first version) made the
// thread-per-read kernels LSU bound (160 wavefronts per warp and 16 columns; ncu round 2), 128-bit loads move four
// times the bytes per wavefront.  Touches the 32 aligned bytes around q .. q + 16; the device pools are padded for it.
// the 16 bytes at byte offset o (0..15) of the 32-byte register window a | b
__device__ __forceinline__ uint4 window16(const uint4& a, const uint4& b, uint32_t o) {
    const bool s2 = (o & 8u) != 0, s1 = (o & 4u) != 0;
    const uint32_t x0 = s2 ? a.z : a.x, x1 = s2 ? a.w : a.y, x2 = s2 ? b.x : a.z, x3 = s2 ? b.y : a.w, x4 = s2 ? b.z : b.x,
                   x5 = s2 ? b.w : b.y;
    const uint32_t y0 = s1 ? x1 : x0, y1 = s1 ? x2 : x1, y2 = s1 ? x3 : x2, y3 = s1 ? x4 : x3, y4 = s1 ? x5 : x4;
    const uint32_t sh = (o & 3u) * 8u;
    return make_uint4(__funnelshift_r(y0, y1, sh), __funnelshift_r(y1, y2, sh), __funnelshift_r(y2, y3, sh),
                      __funnelshift_r(y3, y4, sh));
}
__device__ __forceinline__ uint4 fetch16(const uint8_t* __restrict__ q) {
    const uint4* __restrict__ v = reinterpret_cast<const uint4*>((uintptr_t)q & ~(uintptr_t)15);
    return window16(v[0], v[1], (uint32_t)(uintptr_t)q & 15u);
}

// byte i (0..15, run-time index) of a 16-byte register block
__device__ __forceinline__ uint32_t byte_of(const uint4& v, uint32_t i) {
    const uint32_t w = (i & 8u) ? ((i & 4u) ? v.w : v.z) : ((i & 4u) ? v.y : v.x);
    return (w >> ((i & 3u) * 8u)) & 0xFFu;
}

// The characters of a read interval one at a time, forwards or backwards, fetched 16 at a time (the exact DP kernels
// walk a column per character; a byte load per column was one L1 wavefront per thread and column).
struct CharWalk {
    const uint8_t* p;  // forwards: the next character; backwards: one past the next character
    uint4 buf;
    uint32_t have;     // characters left in buf
    bool rev;
    __device__ __forceinline__ void init(const uint8_t* first, bool backwards) {
        p = first;
        rev = backwards;
        have = 0;
        buf = make_uint4(0, 0, 0, 0);
    }
    __device__ __forceinline__ void need(uint32_t k) {  // at least k characters in buf (k <= 16)
        if (have < k) {
            buf = fetch16(rev ? p - 16 : p);
            have = 16;
        }
    }
    __device__ __forceinline__ uint32_t peek(uint32_t k) const { return byte_of(buf, rev ? have - 1u - k : 16u - have + k); }  // k < have
    __device__ __forceinline__ void advance(uint32_t k) {
        have -= k;
        p += rev ? -(int)k : (int)k;
    }
    __device__ __forceinline__ uint32_t next() {
        need(1);
        const uint32_t c = peek(0);
        advance(1);
        return c;
    }
};

struct RecordShape {
    uint32_t id_len, umi_len, seq_len, total;
    uint32_t lenA, lenB;
};

// FASTA: ">name\nseq\n" instead of "@name\nseq\n+\nqual\n"
template <bool FASTA = false>
__device__ __forceinline__ RecordShape record_shape(const PairParams& P, const ReadState& own, const ReadState& r1,
                                                    const ReadState& r2) {
    RecordShape rs;
    rs.id_len = (uint32_t)own.id_end - (uint32_t)own.id_start;
    rs.lenA = rs.lenB = 0;
    if (P.rename_parts & CSQ_REN_OWN_PREFIX) rs.lenA = own.ren_cp & 0xFFFFu;
    if (P.rename_parts & CSQ_REN_OWN_SUFFIX) rs.lenB = own.ren_cs & 0xFFFFu;
    if (P.rename_parts & CSQ_REN_R1_PREFIX) rs.lenA = r1.ren_cp & 0xFFFFu;
    if (P.rename_parts & CSQ_REN_R2_PREFIX) rs.lenB = r2.ren_cp & 0xFFFFu;
    rs.umi_len = (P.rename_parts ? 1u : 0u) + rs.lenA + rs.lenB;
    rs.seq_len = (uint32_t)own.b - (uint32_t)own.a;
    rs.total = FASTA ? 1 + rs.id_len + rs.umi_len + 1 + rs.seq_len + 1 : 1 + rs.id_len + rs.umi_len + 1 + rs.seq_len + 3 + rs.seq_len + 1;
    return rs;
}

__device__ __forceinline__ uint8_t complement_base(uint8_t c) {
    // dnaio reverse_complement table: ACGTUMRWSYKVHDBN -> TGCAAKYWSRMBDHVN (case kept), others unchanged
    const char* from = "ACGTUMRWSYKVHDBNacgtumrwsykvhdbn";
    const char* to = "TGCAAKYWSRMBDHVNtgcaakywsrmbdhvn";
#pragma unroll
    for (int i = 0; i < 32; i++)
        if (c == (uint8_t)from[i]) return (uint8_t)to[i];
    return c;
}

}  // namespace
