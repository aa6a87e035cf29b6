// sm_100a kernels of the trimming chain.
//
//   k_align<M>     exact adapter alignment, one thread per read, whole DP column in registers
//   k_align_split  the poly-A / poly-T 100-mers: KC DP columns side by side, every column over two lanes
//   k_scan         exclusive scan of the per-CTA totals (6 output streams, one sweep)
//   k_emit         order-preserving FASTQ text emission straight from and to global memory, 16 lanes per record:
//                  the reverse-complementing single-end sink and the A/B partner (CSQ_PLAN_EMIT_G16) of the default
//                  emitter k_emit_stage (emit_stage.cu)
// (k_tail - trailing ops, quality trimming, header, name check, filters - lives in tail.cu)
//   k_int_peak     integer-issue microbenchmark (roofline denominator of the DP)
//
// Semantics follow cutadapt 5.x as restated in oracle/cutseq_oracle.c (Aligner.locate of
// upstream _align.pyx etc.); the call sites are reference run.py:326-471 / 533-792.
//
// DP cell encoding.  cutadapt keeps (cost, score, origin) per cell and picks, on a
// mismatch, diag if cost_diag <= both others, else insertion if <= deletion, else deletion;
// score and origin are inherited from the chosen neighbour (+1 match, -1 mismatch, -2 indel).
// Here a cell is ONE 32-bit word
//        [31:22] cost | [21:20] direction priority (transient) | [19:10] s' | [9:0] origin+128
// with s' = score + 2*cost, which only ever grows (match +1, mismatch +1, indel +0), so no field
// ever borrows from its neighbour.  The three candidates get cost+1 and their priority
// (diag 0 < insertion 1 < deletion 2) added in one IADD each; one 3-input unsigned minimum
// (VIMNMX3) then implements cutadapt's tie-breaking exactly, and one LOP3 clears the priority.
// On a match the diagonal candidate keeps its cost and always wins (|D(i-1,j-1) - D(i-1,j)| <= 1),
// which is cutadapt's "characters equal -> take the diagonal" rule.
// cutadapt's Ukkonen band is not reproduced: cells it skips have cost > k and can neither be
// accepted nor lie on the path of an accepted cell, so the full DP yields identical results.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "csq_internal.h"
#include "device_common.cuh"

namespace {

constexpr int HOMO_COLUMNS = 4;  // DP columns a lane pair computes side by side for homopolymer adapters (k_align_split)

constexpr int SP_SHIFT = 10, PRIO_SHIFT = 20, COST_SHIFT = 22;
constexpr int ORG_BIAS = 128;
constexpr uint32_t D_MATCH = 1u << SP_SHIFT;
constexpr uint32_t D_MIS = (1u << COST_SHIFT) + (1u << SP_SHIFT);
constexpr uint32_t D_INS = (1u << COST_SHIFT) + (1u << PRIO_SHIFT);
constexpr uint32_t D_DEL = (1u << COST_SHIFT) + (2u << PRIO_SHIFT);
constexpr uint32_t PRIO_CLEAR = ~(3u << PRIO_SHIFT);

__device__ __forceinline__ uint32_t pack_cell(int cost, int origin) {
    return ((uint32_t)cost << COST_SHIFT) | ((uint32_t)(2 * cost) << SP_SHIFT) | (uint32_t)(origin + ORG_BIAS);
}
__device__ __forceinline__ int cell_cost(uint32_t w) { return (int)(w >> COST_SHIFT); }
__device__ __forceinline__ int cell_origin(uint32_t w) { return (int)(w & 0x3FFu) - ORG_BIAS; }
__device__ __forceinline__ int cell_score(uint32_t w) { return (int)((w >> SP_SHIFT) & 0x3FFu) - 2 * cell_cost(w); }

struct Best {
    int cost, origin, score, ref_stop, query_stop;
};

__device__ __forceinline__ uint32_t mad1(uint32_t a, uint32_t b, uint32_t c) {  // a * b + c on the FMA pipe (IMAD)
    uint32_t d;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

__device__ __forceinline__ void init_cell(int i, int min_n, bool sir, bool siq, int& cost, int& origin) {
    if (!sir && !siq) {
        cost = max(i, min_n);
        origin = 0;
    } else if (sir && !siq) {
        cost = min_n;
        origin = min(0, min_n - i);
    } else if (!sir && siq) {
        cost = i;
        origin = max(0, min_n - i);
    } else {
        cost = min(i, min_n);
        origin = min_n - i;
    }
}

// Row-m rule of Aligner.locate (only evaluated where cost[m] <= k, as upstream's band does).
// Returns true when the new best match is error-free and starts inside the read: Aligner.locate leaves its column
// loop there ("exact match, stop early").  Nothing later could replace such a match anyway - its score is m, no cell
// scores higher and an equal score needs cost 0 as well - so stopping and walking on give the same result; the
// caller stops when P.exact_stop is set.
__device__ __forceinline__ bool row_m_update(uint32_t wm, int j, int m, int n, const AlignParams& P, Best& best) {
    const int cost = cell_cost(wm);
    if (cost > P.k) return false;
    const int origin = cell_origin(wm), score = cell_score(wm);
    const int length = m + min(origin, 0);
    const bool acceptable = length >= P.min_overlap && cost <= (int)P.thr[length];
    if (!acceptable) return false;
    const int best_length = m + min(best.origin, 0);
    if (best.cost == m + n + 1 || (origin <= best.origin + m / 2 && score > best.score) ||
        (length > best_length && score > best.score)) {
        best.score = score;
        best.cost = cost;
        best.origin = origin;
        best.ref_stop = m;
        best.query_stop = j;
        return cost == 0 && origin >= 0;
    }
    return false;
}

__device__ __forceinline__ void last_col_update(uint32_t w, int i, int n, const AlignParams& P, Best& best) {
    const int cost = cell_cost(w), origin = cell_origin(w), score = cell_score(w);
    const int length = i + min(origin, 0);
    if (length >= P.min_overlap && length >= 0 && cost <= (int)P.thr[max(length, 0)] &&
        (score > best.score || (score == best.score && cost < best.cost))) {
        best.score = score;
        best.cost = cost;
        best.origin = origin;
        best.ref_stop = i;
        best.query_stop = n;
    }
}

__device__ __forceinline__ void best_to_match(const Best& best, int m, int n, bool reversed, csq_match& r) {
    if (best.cost == m + n + 1) {
        r = no_match();
        return;
    }
    int ref_start = best.origin >= 0 ? 0 : -best.origin;
    int query_start = best.origin >= 0 ? best.origin : 0;
    int ref_stop = best.ref_stop, query_stop = best.query_stop;
    if (reversed) {  // RightmostFrontAdapter.match_to coordinate mapping
        int rs = m - ref_stop, re = m - ref_start, qs = n - query_stop, qe = n - query_start;
        ref_start = rs;
        ref_stop = re;
        query_start = qs;
        query_stop = qe;
    }
    r.found = 1;
    r.reserved = 0;
    r.ref_start = (int16_t)ref_start;
    r.ref_stop = (int16_t)ref_stop;
    r.query_start = (int16_t)query_start;
    r.query_stop = (int16_t)query_stop;
    r.score = (int16_t)best.score;
    r.errors = (int16_t)best.cost;
}

// Exact DP for a compile-time adapter length M: the column lives in registers W[0..M].
template <int M>
__device__ __forceinline__ void dp_exact(const uint8_t* __restrict__ s, int a, int b, const AlignParams& P,
                                         const uint32_t* __restrict__ lut, int j0, csq_match& r) {
    constexpr int NW = (M + 31) / 32;
    const int n = b - a;
    const int k = P.k;
    const uint32_t one = P.one;
    const bool sir = P.flags & 1, siq = P.flags & 2, eir = P.flags & 4, eiq = P.flags & 8;
    int min_n, max_n;
    column_range(siq, eiq, M, k, n, min_n, max_n);
    // Column window (BACK flags, set by the prefilter): the DP starts at column j0 > min_n as if the read began
    // there.  With a free read start the cost of cell (i, j) is the best alignment of adapter[0:i] ending at j,
    // which spans at most i + cost columns; a cell that Aligner.locate can accept (cost <= k) and every
    // neighbour that is compared on its traceback path (cost <= k + 1) therefore has the same cost, and by
    // induction along the path the same (cost, score, origin), as in the full matrix when
    // j0 <= j - (m + 3k + 2).  The prefilter guarantees this for all columns that can hold an accepted cell.
    if (j0 >= 0) min_n = max(min_n, j0);

    uint32_t W[M + 1];
#pragma unroll
    for (int i = 0; i <= M; i++) {
        int cost, origin;
        init_cell(i, min_n, sir, siq, cost, origin);
        W[i] = pack_cell(cost, origin);
    }
    Best best = {M + n + 1, 0, 0, M, n};
    const uint32_t row0_delta = siq ? 1u : ((1u << COST_SHIFT) + (2u << SP_SHIFT));
    CharWalk cw;  // read characters, 16 per fetch (a byte load per column made this kernel LSU bound)
    cw.init(P.reversed ? (s + b - min_n) : (s + a + min_n), P.reversed != 0);

    bool cut_short = false;
    for (int j = min_n + 1; j <= max_n; j++) {
        const uint32_t c = cw.next();
        uint32_t pm[NW];
#pragma unroll
        for (int w = 0; w < NW; w++) pm[w] = lut[c * NW + w];
        uint32_t wd = W[0];
        W[0] += row0_delta;
#pragma unroll
        for (int i = 1; i <= M; i++) {
            // Two integer pipes (B300_MICROARCH.md: IADD3 / LOP3 / VIMNMX on the ALU pipe, IMAD on the FMA pipe, one
            // warp instruction per two cycles each).  The all-ALU form of this cell was 5 instructions = 10 cycles
            // (VIADD, predicated VIADD, 2 x VIADDMNMX, LOP3); here the diagonal candidate and its mismatch surcharge
            // run as mad.lo on the FMA pipe (the multiplier arrives as a kernel argument, a literal 1 would be folded
            // back into VIADD), the ALU pipe keeps the two fused add+min and the priority clear: 3 ALU + 2 FMA.
            const uint32_t wl = W[i];
            uint32_t cd = mad1(wd, one, D_MATCH);
            if (!(pm[(i - 1) >> 5] & (1u << ((i - 1) & 31)))) cd = mad1(cd, one, D_MIS - D_MATCH);
            const uint32_t t = min(cd, W[i - 1] + D_INS);
            W[i] = min(t, wl + D_DEL) & PRIO_CLEAR;
            wd = wl;
        }
        if (eiq && row_m_update(W[M], j, M, n, P, best) && P.exact_stop) {
            cut_short = true;  // the last-column rule cannot change an error-free full match either
            break;
        }
    }
    if (max_n == n && !cut_short) {
        const int first_i = eir ? 0 : M;
#pragma unroll
        for (int i = M; i >= 0; i--)
            if (i >= first_i) last_col_update(W[i], i, n, P, best);
    }
    best_to_match(best, M, n, P.reversed != 0, r);
}

// Same recurrence for any m <= CSQ_MAX_ADAPTER with the column in local memory (slow path for
// adapter lengths without a register-resident instantiation).
__device__ __noinline__ void dp_generic(const uint8_t* __restrict__ s, int a, int b, const AlignParams& P, int j0,
                                        csq_match& r) {
    const int m = P.m, n = b - a, k = P.k;
    const bool sir = P.flags & 1, siq = P.flags & 2, eir = P.flags & 4, eiq = P.flags & 8;
    int min_n, max_n;
    column_range(siq, eiq, m, k, n, min_n, max_n);
    if (j0 >= 0) min_n = max(min_n, j0);  // column window, see dp_exact
    uint32_t W[CSQ_MAX_ADAPTER + 1];
    for (int i = 0; i <= m; i++) {
        int cost, origin;
        init_cell(i, min_n, sir, siq, cost, origin);
        W[i] = pack_cell(cost, origin);
    }
    Best best = {m + n + 1, 0, 0, m, n};
    const uint32_t row0_delta = siq ? 1u : ((1u << COST_SHIFT) + (2u << SP_SHIFT));
    CharWalk cw;
    cw.init(P.reversed ? (s + b - min_n) : (s + a + min_n), P.reversed != 0);
    bool exact_stop = false;
    for (int j = min_n + 1; j <= max_n; j++) {
        const uint32_t c = cw.next() & 0xDFu;
        const int li = c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : -1;
        uint32_t wd = W[0];
        W[0] += row0_delta;
        for (int i = 1; i <= m; i++) {
            const uint32_t wl = W[i];
            const bool eq = li >= 0 && ((P.peq[li][(i - 1) >> 5] >> ((i - 1) & 31)) & 1u);
            const uint32_t cd = wd + (eq ? D_MATCH : D_MIS);
            const uint32_t cu = W[i - 1] + D_INS;
            const uint32_t cl = wl + D_DEL;
            W[i] = __vimin3_u32(cd, cu, cl) & PRIO_CLEAR;
            wd = wl;
        }
        if (eiq && row_m_update(W[m], j, m, n, P, best) && P.exact_stop) {
            exact_stop = true;
            break;
        }
    }
    if (max_n == n && !exact_stop) {
        const int first_i = eir ? 0 : m;
        for (int i = m; i >= first_i; i--) last_col_update(W[i], i, n, P, best);
    }
    best_to_match(best, m, n, P.reversed != 0, r);
}

// EndStatistics.adjacent_bases of cutadapt's BackAdapterStatistics.add_match: the read base in front of a 3' match
// (match.sequence[rstart - 1 : rstart]; the read is original[a:b] here).  Slots: A, C, G, T, none, other.
__device__ __forceinline__ void count_adjacent(const AlignParams& P, const uint8_t* s, int a, int query_start) {
    int slot = 4;
    if (query_start > 0) {
        const uint8_t c = s[a + query_start - 1];
        slot = c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : 5;
    }
    atomicAdd(P.counters + P.adjacent_index + slot, 1ULL);
}

// Entry `slot` (0 .. per_cta - 1) of this CTA.  Without survivor lists CTA c takes reads c * per_cta ..; with them,
// per_cta consecutive entries of one list, the lists (longest DP first, k_prefilter) laid end to end in units of CTAs.
// The grid is sized for the worst case: false means the CTA has no entry at all (the same in all its threads) and
// leaves at once.  Otherwise t < count tells whether this slot holds an entry, list_entry gives its read.
__device__ __forceinline__ bool list_position(const AlignParams& P, uint32_t per_cta, uint32_t slot, uint32_t& t, uint32_t& count,
                                              size_t& list_base) {
    t = blockIdx.x * per_cta + slot;
    count = P.n;
    list_base = 0;
    if (P.list) {
        uint32_t cta = blockIdx.x;
        int bin = 0;
        for (; bin < CSQ_PF_BINS; bin++) {
            count = P.list_count[bin];
            const uint32_t ctas = (count + per_cta - 1) / per_cta;
            if (cta < ctas) break;
            cta -= ctas;
        }
        if (bin == CSQ_PF_BINS) return false;
        t = cta * per_cta + slot;
        list_base = (size_t)bin * P.n;
        return true;
    }
    return blockIdx.x * per_cta < count;
}

// Read of entry t and the first DP column of the exact pass (j0, -1: the aligner's own min_n, see dp_exact).
__device__ __forceinline__ uint32_t list_entry(const AlignParams& P, uint32_t t, size_t list_base, int& j0) {
    j0 = -1;
    if (!P.list) return t;
    const uint32_t idx = P.list[list_base + t];
    const uint32_t w = reinterpret_cast<const uint16_t*>(P.list + (size_t)CSQ_PF_BINS * P.n)[list_base + t];
    if (w != 0xFFFFu) j0 = (int)w;
    return idx;
}

// Match r of read idx (characters s): a found match sets the matched bits, counts the adjacent base and the match and
// trims the read; then the match record and the state are stored.
__device__ __forceinline__ void commit_match(const AlignParams& P, uint32_t idx, const uint8_t* s, const csq_match& r, ReadState st) {
    if (r.found) {
        st.matched |= 0x80000000u | (P.adapter_bit >= 0 ? (1u << P.adapter_bit) : 0u);
        if (P.adjacent_index >= 0) count_adjacent(P, s, st.a, r.query_start);
        if (P.trim_front)
            st.a = (uint16_t)(st.a + r.query_stop);  // RemoveBeforeMatch: read[rstop:]
        else
            st.b = (uint16_t)(st.a + r.query_start);  // RemoveAfterMatch: read[:rstart]
        atomicAdd(P.counters + P.counter_index, 1ULL);
    }
    if (P.matches) P.matches[idx] = r;
    store_state(P.md.state + idx, st);
}

// M > 0: column in registers (dp_exact<M>); M == 0: any m <= CSQ_MAX_ADAPTER with the column in local memory
template <int M>
__global__ void __launch_bounds__(128) k_align(const __grid_constant__ AlignParams P) {
    constexpr int NW = (M > 0 ? (M + 31) / 32 : 1);
    __shared__ uint32_t lut[M == 0 ? 1 : 256 * NW];
    uint32_t t, count;
    size_t list_base;
    if (!list_position(P, blockDim.x, threadIdx.x, t, count, list_base)) return;
    if constexpr (M > 0) {
        for (int c = threadIdx.x; c < 256; c += blockDim.x) {
            const int u = c & 0xDF;
            const int li = u == 'A' ? 0 : u == 'C' ? 1 : u == 'G' ? 2 : u == 'T' ? 3 : -1;
#pragma unroll
            for (int w = 0; w < NW; w++) lut[c * NW + w] = li >= 0 ? P.peq[li][w] : 0u;
        }
        __syncthreads();
    }
    if (t >= count) return;
    int j0;
    const uint32_t idx = list_entry(P, t, list_base, j0);
    const ReadState st = entry_state(P, idx);

    const uint8_t* s = P.md.seq + P.md.seq_off[idx];
    csq_match r;
    if (P.count_cells) {  // nominal DP cells of this alignment, m * (max_n - min_n)  (statistics / GCUPS numerator)
        int min_n, max_n;
        column_range(P.flags & 2, P.flags & 8, P.m, P.k, (int)st.b - (int)st.a, min_n, max_n);
        const unsigned int mine = (unsigned int)(P.m * (max_n - min_n));
        unsigned long long* dst = P.counters + P.counter_index + (CNT_DP_CELLS - CNT_WITH_ADAPTERS);
        if (__activemask() == 0xffffffffu) {
            unsigned int cells = mine;
            for (int o = 16; o > 0; o >>= 1) cells += __shfl_down_sync(0xffffffffu, cells, o);
            if ((threadIdx.x & 31) == 0) atomicAdd(dst, (unsigned long long)cells);
        } else {
            atomicAdd(dst, (unsigned long long)mine);
        }
    }
    if constexpr (M > 0)
        dp_exact<M>(s, st.a, st.b, P, lut, j0, r);
    else
        dp_generic(s, st.a, st.b, P, j0, r);
    commit_match(P, idx, s, r, st);
}

// Exclusive scan over CTAs of the 8 stream totals (6 used) -> byte offset of every CTA in every
// output stream; totals[0..7] = bytes per stream, totals[8..11] = records per destination.
__global__ void __launch_bounds__(1024) k_scan(uint32_t nblk, const uint32_t* __restrict__ block_tot,
                                               const uint32_t* __restrict__ block_cnt,
                                               unsigned long long* __restrict__ block_off,
                                               unsigned long long* __restrict__ totals) {
    // all 8 streams in one sweep: thread t takes CTA base + t (its 8 totals are one 32-byte row)
    __shared__ unsigned long long warp_sums[8][32];
    __shared__ unsigned long long carry[8];
    __shared__ unsigned long long cnt_sums[4][32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x < 8) carry[threadIdx.x] = 0;
    unsigned long long cnt[4] = {0, 0, 0, 0};
    __syncthreads();
    for (uint32_t base = 0; base < nblk; base += 1024) {
        const uint32_t i = base + threadIdx.x;
        unsigned long long v[8], x[8];
        if (i < nblk) {
            const uint4 lo = reinterpret_cast<const uint4*>(block_tot)[2 * (size_t)i];
            const uint4 hi = reinterpret_cast<const uint4*>(block_tot)[2 * (size_t)i + 1];
            const uint4 c = reinterpret_cast<const uint4*>(block_cnt)[i];
            v[0] = lo.x; v[1] = lo.y; v[2] = lo.z; v[3] = lo.w;
            v[4] = hi.x; v[5] = hi.y; v[6] = hi.z; v[7] = hi.w;
            cnt[0] += c.x; cnt[1] += c.y; cnt[2] += c.z; cnt[3] += c.w;
        } else {
#pragma unroll
            for (int s = 0; s < 8; s++) v[s] = 0;
        }
#pragma unroll
        for (int s = 0; s < 8; s++) {
            unsigned long long y = v[s];
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long z = __shfl_up_sync(0xffffffffu, y, o);
                if (lane >= o) y += z;
            }
            x[s] = y;
            if (lane == 31) warp_sums[s][wid] = y;
        }
        __syncthreads();
        if (wid < 8) {  // warp s scans the 32 warp totals of stream s
            unsigned long long ws = warp_sums[wid][lane];
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long z = __shfl_up_sync(0xffffffffu, ws, o);
                if (lane >= o) ws += z;
            }
            warp_sums[wid][lane] = ws;
        }
        __syncthreads();
        unsigned long long before[8];
#pragma unroll
        for (int s = 0; s < 8; s++) before[s] = carry[s] + (wid ? warp_sums[s][wid - 1] : 0ULL) + (x[s] - v[s]);
        if (i < nblk) {
            ulonglong2* dst = reinterpret_cast<ulonglong2*>(block_off + (size_t)i * 8);
#pragma unroll
            for (int s = 0; s < 4; s++) dst[s] = make_ulonglong2(before[2 * s], before[2 * s + 1]);
        }
        __syncthreads();
        if (threadIdx.x == 1023) {
#pragma unroll
            for (int s = 0; s < 8; s++) carry[s] = before[s] + v[s];
        }
        __syncthreads();
    }
    if (threadIdx.x < 8) totals[threadIdx.x] = carry[threadIdx.x];
    // record counts per destination
#pragma unroll
    for (int d = 0; d < 4; d++) {
        unsigned long long t = cnt[d];
        for (int o = 16; o > 0; o >>= 1) t += __shfl_down_sync(0xffffffffu, t, o);
        if (lane == 0) cnt_sums[d][wid] = t;
    }
    __syncthreads();
    if (threadIdx.x < 4) {
        unsigned long long t = 0;
        for (int w = 0; w < 32; w++) t += cnt_sums[threadIdx.x][w];
        totals[8 + threadIdx.x] = t;
    }
}

// FASTQ text, "@name\nseq\n+\nqual\n" (dnaio), streams in input order.
// Phase 1 (thread per pair): load the two mate states once, CTA-wide exclusive scan of the record sizes
// per output stream, one descriptor per record into shared memory.
// Phase 2 (warp per record): bases and qualities, ~85 % of the bytes, as output-aligned 32-bit words built
// from two aligned source words (funnel shift) - a warp instruction writes 128 contiguous bytes; the id,
// the UMI, the separators and the up to 3 + 3 bytes of each segment outside the output's word grid go
// bytewise, one byte per lane, in the same pass, so every 32-byte sector of the output is completed by one
// warp within a few instructions (scattering these bytes from the per-pair threads of phase 1 doubled the
// DRAM traffic: partially written sectors were filled from and evicted to HBM).  All loads of a record are
// issued before its first store; no shared-memory staging and no barrier in the copy loop.
// Every source byte is read once and every output byte written once.
// The reverse-complementing single-end sink takes a bytewise path, and so does k_emit<true>, which writes FASTA
// records (">name\nseq\n", CSQ_PLAN_FASTA).
struct EmitRec {
    uint8_t* out;        // where the record goes
    uint32_t nm;         // id bytes: offset into the mate's name pool
    uint32_t sq, ql;     // original read: offsets into the seq / qual pools
    uint32_t pa, pb;     // UMI parts: offsets into the pool of the mate they come from
    uint16_t id_len, lenA, lenB, a, b;
    uint16_t umi_len;    // '_' + parts, 0 when the template is "{id}"
};

struct EmitSrc {  // global pointers of one record
    const uint8_t *nm, *sq, *ql, *pa, *pb;
};

constexpr int EMIT_UNROLL = 4;

template <bool FASTA = false>
__device__ __forceinline__ uint8_t emit_byte(const EmitRec& R, const EmitSrc& S, uint32_t p, uint32_t e_name, uint32_t e_umi,
                                             uint32_t e_seq, uint32_t e_qual, bool revcomp) {
    if (p < e_name) return p == 0 ? (uint8_t)(FASTA ? '>' : '@') : S.nm[p - 1];
    if (p < e_umi) {
        uint32_t x = p - e_name;
        if (x == 0) return (uint8_t)'_';
        x -= 1;
        return x < R.lenA ? S.pa[x] : S.pb[x - R.lenA];
    }
    if (p == e_umi) return (uint8_t)'\n';
    if (p < e_seq) {
        const uint32_t x = p - e_umi - 1;
        return revcomp ? complement_base(S.sq[R.b - 1 - x]) : S.sq[R.a + x];
    }
    if (FASTA) return (uint8_t)'\n';
    if (p < e_seq + 3) return (p - e_seq == 1) ? (uint8_t)'+' : (uint8_t)'\n';
    if (p < e_qual) {
        const uint32_t x = p - e_seq - 3;
        return revcomp ? S.ql[R.b - 1 - x] : S.ql[R.a + x];
    }
    return (uint8_t)'\n';
}

// Split of a len-byte segment that goes to byte address `dst`: `head` bytes up to the next 4-byte boundary,
// `nw` whole words, then the rest.
__device__ __forceinline__ void word_split(const uint8_t* dst, uint32_t len, uint32_t& head, uint32_t& nw) {
    head = min((4u - ((uint32_t)(uintptr_t)dst & 3u)) & 3u, len);
    nw = (len - head) >> 2;
}

template <bool FASTA>
__global__ void __launch_bounds__(CSQ_PAIR_BLOCK) k_emit(const __grid_constant__ EmitParams E) {
    const PairParams& P = E.pp;
    __shared__ EmitRec recs[2][CSQ_PAIR_BLOCK];
    __shared__ unsigned int wtot[8][CSQ_PAIR_BLOCK / 32];  // per-stream totals of every warp
    const uint32_t base = blockIdx.x * CSQ_PAIR_BLOCK;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const bool paired = P.n_mates == 2;
    const int n_mates = paired ? 2 : 1;
    const bool revcomp = P.revcomp != 0;
    // pools the UMI parts come from: the mate itself (single-end template) or R1 / R2 (paired template)
    const uint8_t* const poolA = (P.rename_parts & CSQ_REN_R1_PREFIX) ? P.md[0].seq : nullptr;
    const uint8_t* const poolB = (P.rename_parts & CSQ_REN_R2_PREFIX) ? P.md[1].seq : nullptr;

    // ---- phase 1 ----
    const uint32_t idx = base + threadIdx.x;
    const bool live = idx < P.n;
    int dest = -1;
    uint32_t len[2] = {0, 0}, incl[2] = {0, 0};
    ReadState st[2];
    RecordShape shape[2];
    if (live) {
        dest = P.dest[idx];
        st[0] = load_state(P.md[0].state + idx);
        st[1] = paired ? load_state(P.md[1].state + idx) : st[0];
        for (int mt = 0; mt < n_mates; mt++) {
            shape[mt] = record_shape<FASTA>(P, st[mt], st[0], st[1]);
            len[mt] = shape[mt].total;
        }
    }
    // warp-level inclusive scans per (dest, mate) stream; only the thread's own dest contributes
    for (int mt = 0; mt < n_mates; mt++)
        for (int d = 0; d < CSQ_N_DEST; d++) {
            const uint32_t v = dest == d ? len[mt] : 0u;
            uint32_t x = v;
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
                if (lane >= o) x += y;
            }
            if (dest == d) incl[mt] = x;
            if (lane == 31) wtot[d * 2 + mt][wid] = x;
        }
    __syncthreads();
    if (live) {
        for (int mt = 0; mt < n_mates; mt++) {
            const int stream = dest * 2 + mt;
            uint32_t off = incl[mt] - len[mt];
            for (int w = 0; w < wid; w++) off += wtot[stream][w];
            const MateDev& md = P.md[mt];
            const ReadState& own = st[mt];
            EmitRec R;
            R.nm = md.name_off[idx] + own.id_start;
            R.sq = md.seq_off[idx];
            R.ql = md.qual_off[idx];
            R.pa = R.pb = 0;
            if (P.rename_parts & CSQ_REN_OWN_PREFIX) R.pa = R.sq + (own.ren_cp >> 16);
            if (P.rename_parts & CSQ_REN_OWN_SUFFIX) R.pb = R.sq + (own.ren_cs >> 16);
            if (P.rename_parts & CSQ_REN_R1_PREFIX) R.pa = P.md[0].seq_off[idx] + (st[0].ren_cp >> 16);
            if (P.rename_parts & CSQ_REN_R2_PREFIX) R.pb = P.md[1].seq_off[idx] + (st[1].ren_cp >> 16);
            R.out = E.out[dest][mt] + E.block_off[(size_t)blockIdx.x * 8 + stream] + off;
            R.id_len = (uint16_t)shape[mt].id_len;
            R.lenA = (uint16_t)shape[mt].lenA;
            R.lenB = (uint16_t)shape[mt].lenB;
            R.umi_len = (uint16_t)shape[mt].umi_len;
            R.a = own.a;
            R.b = own.b;
            recs[mt][threadIdx.x] = R;
        }
    }
    __syncthreads();

    // ---- phase 2 ----
    // G = 16 lanes per record, two records side by side in a warp: the bookkeeping of a record (uniform within its
    // group) is issued once per warp instruction for two records, half the instruction count per record of the
    // warp-per-record form, which is bound by instruction issue.
    constexpr int G = 16;
    constexpr int NG = 2;   // records per warp pass
    constexpr int UW = 3;   // unrolled word iterations: UW * G words of 4 bytes
    constexpr int UI = 2;   // unrolled id iterations: UI * G bytes
    constexpr int MR = 2;   // rounds over the 16 edge slots + 7 separators
    const uint32_t sl = (uint32_t)lane % G, grp = (uint32_t)lane / G;
    for (int q = 0; q < 32 / NG; q++) {
        const int slot = wid * 32 + q * NG + (int)grp;
        if (base + slot >= P.n) continue;  // no warp-wide operation below: groups may leave independently
        for (int mt = 0; mt < n_mates; mt++) {
            const EmitRec& R = recs[mt][slot];
            const MateDev& md = P.md[mt];
            const uint32_t seq_len = (uint32_t)R.b - (uint32_t)R.a;
            const uint32_t e_umi = 1u + R.id_len + R.umi_len;
            uint8_t* __restrict__ out = R.out;
            if (FASTA || revcomp) {
                EmitSrc S;
                S.nm = md.name + R.nm;
                S.sq = md.seq + R.sq;
                S.ql = md.qual + R.ql;
                S.pa = (poolA ? poolA : md.seq) + R.pa;
                S.pb = (poolB ? poolB : md.seq) + R.pb;
                const uint32_t e_name = 1u + R.id_len, e_seq = e_umi + 1 + seq_len, e_qual = e_seq + 3 + seq_len;
                const uint32_t total = FASTA ? e_seq + 1 : e_qual + 1;
                for (uint32_t p0 = sl; p0 < total; p0 += G * EMIT_UNROLL) {
                    uint8_t ch[EMIT_UNROLL];
#pragma unroll
                    for (int u = 0; u < EMIT_UNROLL; u++) {
                        const uint32_t p = p0 + G * u;
                        ch[u] = p < total ? emit_byte<FASTA>(R, S, p, e_name, e_umi, e_seq, e_qual, FASTA ? revcomp : true) : (uint8_t)0;
                    }
#pragma unroll
                    for (int u = 0; u < EMIT_UNROLL; u++) {
                        const uint32_t p = p0 + G * u;
                        if (p < total) out[p] = ch[u];
                    }
                }
                continue;
            }
            // bases to out + e_umi + 1, qualities to out + e_umi + 1 + seq_len + 3; word k of a segment goes to the
            // k-th 4-byte boundary at or behind its first byte
            const uint32_t id_len = R.id_len, la = R.lenA, lab = la + R.lenB;
            const uint32_t e_name = 1u + id_len, e_seq = e_umi + 1 + seq_len, e_qual = e_seq + 3 + seq_len;
            const uint8_t* __restrict__ nm = md.name + R.nm;
            const uint8_t* __restrict__ sq = md.seq + R.sq + R.a;
            const uint8_t* __restrict__ ql = md.qual + R.ql + R.a;
            const uint8_t* __restrict__ pa = (poolA ? poolA : md.seq) + R.pa;
            const uint8_t* __restrict__ pb = (poolB ? poolB : md.seq) + R.pb;
            uint8_t* const d_seq = out + e_umi + 1;
            uint8_t* const d_qual = d_seq + seq_len + 3;
            uint32_t h_s, nw_s, h_q, nw_q;
            word_split(d_seq, seq_len, h_s, nw_s);
            word_split(d_qual, seq_len, h_q, nw_q);
            // ---- loads ----
            // single bytes: slots 0..15 = segment edges (4 groups of up to 3 bytes), slots 16..22 = the seven
            // separator bytes; slot = sl + G * round  (selects only: a chain of `==` branches became a jump table)
            uint32_t misc_pos[MR], misc_val[MR];
#pragma unroll
            for (int r = 0; r < MR; r++) {
                const uint32_t ms = sl + (uint32_t)(G * r);
                const uint32_t t = ms - 16u;               // separator index for slots 16..22
                uint32_t sp = e_seq + (t - 3u);            // t = 3, 4, 5: "\n+\n"
                sp = t == 0 ? 0u : sp;
                sp = t == 1 ? e_name : sp;
                sp = t == 2 ? e_umi : sp;
                sp = t == 6 ? e_qual : sp;
                const bool sep_ok = t < 7u && !(t == 1 && R.umi_len == 0);
                misc_val[r] = (uint32_t)(0x0A0A2B0A0A5F40ull >> (8u * (t & 7u))) & 0xFFu;  // "@_\n\n+\n\n"
                const uint32_t g = ms >> 2, x = ms & 3u;
                const bool is_q = (g & 2u) != 0, is_tail = (g & 1u) != 0;
                const uint32_t h = is_q ? h_q : h_s, nw = is_q ? nw_q : nw_s;
                const uint32_t o = is_tail ? h + 4u * nw + x : x;  // offset inside the segment
                const uint32_t lim = is_tail ? seq_len : h;
                const bool edge_ok = ms < 16 && x < 3 && o < lim;
                if (edge_ok) misc_val[r] = (is_q ? ql : sq)[o];
                const uint32_t ep = (is_q ? e_seq + 3 : e_umi + 1) + o;
                misc_pos[r] = edge_ok ? ep : (sep_ok ? sp : 0xFFFFFFFFu);
            }
            uint32_t idv[UI];
#pragma unroll
            for (int u = 0; u < UI; u++) idv[u] = sl + (uint32_t)(G * u) < id_len ? nm[sl + G * u] : 0u;
            uint32_t umiv = 0;
            if (sl < lab) umiv = sl < la ? pa[sl] : pb[sl - la];
            const uintptr_t sa_s = (uintptr_t)(sq + h_s), sa_q = (uintptr_t)(ql + h_q);
            const uint32_t* __restrict__ al_s = reinterpret_cast<const uint32_t*>(sa_s & ~(uintptr_t)3);
            const uint32_t* __restrict__ al_q = reinterpret_cast<const uint32_t*>(sa_q & ~(uintptr_t)3);
            const uint32_t sh_s = (uint32_t)(sa_s & 3u) * 8u, sh_q = (uint32_t)(sa_q & 3u) * 8u;
            uint32_t* __restrict__ o_s = reinterpret_cast<uint32_t*>(d_seq + h_s);
            uint32_t* __restrict__ o_q = reinterpret_cast<uint32_t*>(d_qual + h_q);
            uint32_t ws[UW][2], wq[UW][2];
#pragma unroll
            for (int u = 0; u < UW; u++) {
                const uint32_t k = sl + (uint32_t)(G * u);
                ws[u][0] = ws[u][1] = wq[u][0] = wq[u][1] = 0;
                if (k < nw_s) { ws[u][0] = al_s[k]; ws[u][1] = al_s[k + 1]; }
                if (k < nw_q) { wq[u][0] = al_q[k]; wq[u][1] = al_q[k + 1]; }
            }
            // ---- stores ----
#pragma unroll
            for (int r = 0; r < MR; r++)
                if (misc_pos[r] != 0xFFFFFFFFu) out[misc_pos[r]] = (uint8_t)misc_val[r];
#pragma unroll
            for (int u = 0; u < UI; u++)
                if (sl + (uint32_t)(G * u) < id_len) out[1 + sl + G * u] = (uint8_t)idv[u];
            if (sl < lab) out[e_name + 1 + sl] = (uint8_t)umiv;
#pragma unroll
            for (int u = 0; u < UW; u++) {
                const uint32_t k = sl + (uint32_t)(G * u);
                if (k < nw_s) o_s[k] = __funnelshift_r(ws[u][0], ws[u][1], sh_s);
                if (k < nw_q) o_q[k] = __funnelshift_r(wq[u][0], wq[u][1], sh_q);
            }
            // rare tails: long ids, long UMI parts, long reads
            for (uint32_t x = UI * G + sl; x < id_len; x += G) out[1 + x] = nm[x];
            for (uint32_t x = G + sl; x < lab; x += G) out[e_name + 1 + x] = x < la ? pa[x] : pb[x - la];
            for (uint32_t k = UW * G + sl; k < max(nw_s, nw_q); k += G) {
                if (k < nw_s) o_s[k] = __funnelshift_r(al_s[k], al_s[k + 1], sh_s);
                if (k < nw_q) o_q[k] = __funnelshift_r(al_q[k], al_q[k + 1], sh_q);
            }
        }
    }
}

// k_align_split<M, KC>: homopolymer adapter (the poly-A / poly-T 100-mers of run.py:389-404, 674-707).  Every row
// compares against the same base, so a column needs one match / mismatch delta and no match mask; a thread that walks
// a column top to bottom is ONE dependent chain of 3 instructions per cell, so KC columns are computed side by side,
// column j + c running c rows behind column j (a skewed wavefront inside the thread: KC independent chains, the same
// cells, the same order of the row-m / last-column rules; chain c keeps its two newest cells p1, p2 and
// cell (r, j + c) = min3(p2[c-1] + delta_c, p1[c] + INS, p1[c-1] + DEL), chain -1 being the stored column j - 1).
// Without a free read start the scan stops once more than k characters differ from the adapter base: each of them
// adds at least 1 to every cell of its column and of all later ones, and acceptance needs cost <= k.
// On top of that every column is split over TWO lanes - lane 2q holds rows
// 0..M/2 of entry q, lane 2q+1 rows M/2..M (its row "0" is a copy of row M/2) - so that a thread keeps M/2 + 1 cells
// instead of M + 1: half the registers (a whole-column k_align<100> needed 228-231 and fitted 8 warps per SM), twice
// the warps, half the serial chain per thread (one-lane and one-column forms: measured, profiles/r01_homo_columns.md).  The lower half runs ONE column group behind the upper half: what it needs from
// above - row M/2 of the group's columns - arrives by one shuffle per column at the end of the upper half's turn;
// both lanes take the same decisions (group sizes, early stop after k + 1 foreign characters) from the same
// read characters, one iteration apart.  Row-m rule and exact stop live in the lower lane (it tells the upper
// lane to halt); the last-column rule walks rows M..M/2+1 below, hands `best` up, and rows M/2..0 follow there.
// Cells, order of the rules and results are those of dp_exact.
template <int M, int KC>
__global__ void __launch_bounds__(128, 4) k_align_split(const __grid_constant__ AlignParams P) {
    static_assert(M % 2 == 0, "even adapter length");
    constexpr int MH = M / 2;
    constexpr int PER_CTA = 64;  // entries per CTA: two lanes each
    const uint32_t FULLM = 0xffffffffu;
    const uint32_t one = P.one;
    const int lane = threadIdx.x & 31, h = threadIdx.x & 1;
    uint32_t t, count;
    size_t list_base;
    if (!list_position(P, PER_CTA, threadIdx.x >> 1, t, count, list_base)) return;  // whole CTA
    const bool active = t < count;  // the same for both lanes of a pair; idle pairs still take part in the shuffles
    uint32_t idx = 0;
    int j0 = -1;
    ReadState st = fresh_state(0);
    if (active) {
        idx = list_entry(P, t, list_base, j0);
        st = entry_state(P, idx);
    }
    const int a = st.a, b = st.b, n = b - a, k = P.k;
    const bool sir = P.flags & 1, siq = P.flags & 2, eir = P.flags & 4, eiq = P.flags & 8;
    int min_n, max_n;
    column_range(siq, eiq, M, k, n, min_n, max_n);
    if (active && h == 0 && P.count_cells)
        atomicAdd(P.counters + P.counter_index + (CNT_DP_CELLS - CNT_WITH_ADAPTERS), (unsigned long long)(M * (max_n - min_n)));
    if (j0 >= 0) min_n = max(min_n, j0);  // column window, see dp_exact
    const uint8_t* s = P.md.seq + (active ? P.md.seq_off[idx] : 0u);

    uint32_t W[MH + 1];  // local row r = global row h * MH + r
#pragma unroll
    for (int r = 0; r <= MH; r++) {
        int cost, origin;
        init_cell(h * MH + r, min_n, sir, siq, cost, origin);
        W[r] = pack_cell(cost, origin);
    }
    Best best = {M + n + 1, 0, 0, M, n};
    const uint32_t row0_delta = siq ? 1u : ((1u << COST_SHIFT) + (2u << SP_SHIFT));
    CharWalk cw;
    cw.init(P.reversed ? (s + b - min_n) : (s + a + min_n), P.reversed != 0);
    const uint32_t letter = P.letter;
    int foreign = 0;
    bool cut_short = false, exact_halt = false;
    int j = min_n + 1;
    bool running = active;
    uint32_t recv[KC];  // lower lane: row M/2 of the columns of its next group, as computed above
#pragma unroll
    for (int c = 0; c < KC; c++) recv[c] = 0;

    for (int iter = 0; __any_sync(FULLM, running); iter++) {
        uint32_t bnd[KC];  // local row MH of the columns of this turn's group
#pragma unroll
        for (int c = 0; c < KC; c++) bnd[c] = 0;
        if (running && iter >= h) {
            if (j > max_n) {
                running = false;
            } else {
                bool block = j + KC - 1 <= max_n;
                uint32_t d[KC];
                int f = foreign;
                if (block) {
                    cw.need(KC);
#pragma unroll
                    for (int c = 0; c < KC; c++) {
                        const bool eq = (cw.peek(c) & 0xDFu) == letter;
                        d[c] = eq ? D_MATCH : D_MIS;
                        f += eq ? 0 : 1;
                    }
                    if (!siq && f > k) block = false;
                }
                if (block) {
                    foreign = f;
                    uint32_t p1[KC], p2[KC];
                    uint32_t wd = W[0];
#pragma unroll
                    for (int c = 0; c < KC; c++) p1[c] = p2[c] = h ? recv[c] : W[0] + (uint32_t)(c + 1) * row0_delta;
                    W[0] = p1[KC - 1];
#pragma unroll
                    for (int i = 1; i <= MH + KC - 1; i++) {
#pragma unroll
                        for (int c = KC - 1; c >= 0; c--) {
                            const int row = i - c;
                            if (row < 1 || row > MH) continue;
                            uint32_t diag, left;
                            if (c == 0) {
                                left = W[row];
                                diag = wd;
                                wd = left;
                            } else {
                                left = p1[c - 1];
                                diag = p2[c - 1];
                            }
                            // diagonal add on the FMA pipe (IMAD), the two fused add+min and the clear on the ALU pipe
                            const uint32_t cell = min(min(mad1(diag, one, d[c]), p1[c] + D_INS), left + D_DEL) & PRIO_CLEAR;
                            p2[c] = p1[c];
                            p1[c] = cell;
                            if (c == KC - 1) W[row] = cell;
                            if (row == MH) bnd[c] = cell;
                        }
                    }
                    if (h && eiq) {
                        bool stop = false;
#pragma unroll
                        for (int c = 0; c < KC; c++) stop |= row_m_update(bnd[c], j + c, M, n, P, best);
                        if (stop && P.exact_stop) {
                            cut_short = exact_halt = true;
                            running = false;
                        }
                    }
                    j += KC;
                    cw.advance(KC);
                } else {
                    cw.need(1);
                    const bool eq = (cw.peek(0) & 0xDFu) == letter;
                    bool go = true;
                    if (!siq) {
                        foreign += eq ? 0 : 1;
                        if (foreign > k) {
                            cut_short = true;
                            running = false;
                            go = false;
                        }
                    }
                    if (go) {
                        const uint32_t d0 = eq ? D_MATCH : D_MIS;
                        uint32_t wd = W[0];
                        W[0] = h ? recv[0] : W[0] + row0_delta;
#pragma unroll
                        for (int r = 1; r <= MH; r++) {
                            const uint32_t wl = W[r];
                            W[r] = min(min(mad1(wd, one, d0), W[r - 1] + D_INS), wl + D_DEL) & PRIO_CLEAR;
                            wd = wl;
                        }
                        bnd[0] = W[MH];
                        if (h && eiq && row_m_update(W[MH], j, M, n, P, best) && P.exact_stop) {
                            cut_short = exact_halt = true;
                            running = false;
                        }
                        j += 1;
                        cw.advance(1);
                    }
                }
            }
        }
        // hand row M/2 down, and the exact stop up
#pragma unroll
        for (int c = 0; c < KC; c++) recv[c] = __shfl_sync(FULLM, bnd[c], lane & ~1);
        const bool halt = __shfl_sync(FULLM, (int)exact_halt, lane | 1) != 0;
        if (h == 0 && halt) {
            cut_short = true;
            running = false;
        }
    }
    // last column: rows M .. M/2 + 1 below, then `best` moves up and rows M/2 .. 0 follow
    const bool last_col = max_n == n && !cut_short;
    const int first_i = eir ? 0 : M;
    if (h == 1 && last_col) {
#pragma unroll
        for (int r = MH; r >= 1; r--)
            if (MH + r >= first_i) last_col_update(W[r], MH + r, n, P, best);
    }
    best.cost = __shfl_sync(FULLM, best.cost, lane | 1);
    best.origin = __shfl_sync(FULLM, best.origin, lane | 1);
    best.score = __shfl_sync(FULLM, best.score, lane | 1);
    best.ref_stop = __shfl_sync(FULLM, best.ref_stop, lane | 1);
    best.query_stop = __shfl_sync(FULLM, best.query_stop, lane | 1);
    if (h == 0 && active) {
        if (last_col) {
#pragma unroll
            for (int r = MH; r >= 0; r--)
                if (r >= first_i) last_col_update(W[r], r, n, P, best);
        }
        csq_match r;
        best_to_match(best, M, n, P.reversed != 0, r);
        commit_match(P, idx, P.md.seq + P.md.seq_off[idx], r, st);
    }
}

// Integer-issue microbenchmark: 8 independent dependency chains per thread.
// variant 0: IADD3 / LOP3 / VIMNMX only (ALU pipe); variant 1: the same mixed with IMAD (FMA pipe).
template <int VARIANT>
__global__ void __launch_bounds__(256) k_int_peak(int iters, unsigned int* sink) {
    unsigned int x[8];
#pragma unroll
    for (int q = 0; q < 8; q++) x[q] = threadIdx.x * 8 + q + blockIdx.x;
    const unsigned int c1 = sink[0] | 1u, c2 = sink[1] | 3u;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int r = 0; r < 8; r++) {
#pragma unroll
            for (int q = 0; q < 8; q++) {
                if (VARIANT == 0) {
                    x[q] = min(x[q] + c1, x[q] ^ c2);  // IADD, LOP3, VIMNMX  (3 ops)
                } else {
                    x[q] = min(x[q] * c1 + c2, x[q] ^ c2);  // IMAD, LOP3, VIMNMX (3 ops)
                }
            }
        }
    }
    unsigned int acc = 0;
#pragma unroll
    for (int q = 0; q < 8; q++) acc ^= x[q];
    if (acc == 0x12345678u) sink[2] = acc;
}

template <int M>
cudaError_t launch_align_m(const AlignParams& p, uint32_t n_items, cudaStream_t stream) {
    const dim3 grid((n_items + 127) / 128 + (p.list ? CSQ_PF_BINS : 0)), block(128);
    if constexpr (M == 100) {  // the poly-A / poly-T adapters of run.py:389-404
        if (p.homopolymer) {
            // measured (profiles/r01_homo_columns.md): four columns side by side win where the early stop ends most
            // scans after ~20 columns (read start not free: NonInternalFront), two where every read walks all m + k
            // columns; one kernel per variant (both bodies in one kernel cost 15 %)
            const dim3 grid2((n_items + 63) / 64 + (p.list ? CSQ_PF_BINS : 0));
            if (p.flags & 2)
                k_align_split<M, 2><<<grid2, block, 0, stream>>>(p);
            else
                k_align_split<M, HOMO_COLUMNS><<<grid2, block, 0, stream>>>(p);
            return cudaGetLastError();
        }
    }
    k_align<M><<<grid, block, 0, stream>>>(p);
    return cudaGetLastError();
}

}  // namespace

bool csq_align_has_exact_kernel(int m) { return (m >= 1 && m <= 34) || m == 100; }

cudaError_t csq_launch_align(const AlignParams& p, uint32_t n_items, cudaStream_t stream) {
    if (n_items == 0) return cudaSuccess;
    switch (p.m) {
#define CSQ_CASE(M) \
    case M: return launch_align_m<M>(p, n_items, stream);
        CSQ_CASE(1) CSQ_CASE(2) CSQ_CASE(3) CSQ_CASE(4) CSQ_CASE(5) CSQ_CASE(6) CSQ_CASE(7) CSQ_CASE(8)
        CSQ_CASE(9) CSQ_CASE(10) CSQ_CASE(11) CSQ_CASE(12) CSQ_CASE(13) CSQ_CASE(14) CSQ_CASE(15) CSQ_CASE(16)
        CSQ_CASE(17) CSQ_CASE(18) CSQ_CASE(19) CSQ_CASE(20) CSQ_CASE(21) CSQ_CASE(22) CSQ_CASE(23) CSQ_CASE(24)
        CSQ_CASE(25) CSQ_CASE(26) CSQ_CASE(27) CSQ_CASE(28) CSQ_CASE(29) CSQ_CASE(30) CSQ_CASE(31) CSQ_CASE(32)
        CSQ_CASE(33) CSQ_CASE(34) CSQ_CASE(100)
#undef CSQ_CASE
        default: {
            const dim3 grid((n_items + 127) / 128 + (p.list ? CSQ_PF_BINS : 0)), block(128);
            k_align<0><<<grid, block, 0, stream>>>(p);
            return cudaGetLastError();
        }
    }
}

cudaError_t csq_launch_scan(uint32_t nblk, const uint32_t* block_tot, const uint32_t* block_cnt,
                            unsigned long long* block_off, unsigned long long* totals, cudaStream_t stream) {
    k_scan<<<1, 1024, 0, stream>>>(nblk, block_tot, block_cnt, block_off, totals);
    return cudaGetLastError();
}

cudaError_t csq_launch_emit(const EmitParams& p, bool fasta, cudaStream_t stream) {
    if (p.pp.n == 0) return cudaSuccess;
    const dim3 grid((p.pp.n + CSQ_PAIR_BLOCK - 1) / CSQ_PAIR_BLOCK), block(CSQ_PAIR_BLOCK);
    if (fasta)
        k_emit<true><<<grid, block, 0, stream>>>(p);
    else
        k_emit<false><<<grid, block, 0, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t csq_launch_int_peak(int variant, int iters, unsigned int* sink, int blocks, int threads, cudaStream_t stream) {
    if (variant == 0)
        k_int_peak<0><<<blocks, threads, 0, stream>>>(iters, sink);
    else
        k_int_peak<1><<<blocks, threads, 0, stream>>>(iters, sink);
    return cudaGetLastError();
}
