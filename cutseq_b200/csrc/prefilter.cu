// k_prefilter<NW>: bit-parallel (Myers 1999 / Hyyro 2001) REJECT-ONLY filter in front of k_align.
//
// One thread per read computes the exact semiglobal edit-distance matrix of Aligner.locate (same
// boundary conditions, same column range) column by column with vertical-delta bit-vectors of
// NW x 32 bits, i.e. the `cost` component of cutadapt's cells and nothing else.  A read survives
// when some cell that Aligner.locate would examine COULD be acceptable:
//   row m, column j (only with QUERY_STOP):  cost <= thr[Lmax], Lmax = min(m, j + cost) >= min_overlap
//   last column, row i >= first_i:           cost <= thr[Lmax], Lmax = min(i, (n - min_n) + cost) >= min_overlap
// Lmax bounds the aligned adapter length from above (an alignment with `cost` errors that ends in
// column j covers at most (j - min_n) + cost adapter characters) and thr[] is monotone, so the test is
// a necessary condition for `length >= min_overlap and cost <= length * max_error_rate`.
// Survivors are compacted into a list and handed to the exact DP (k_align), which alone decides
// whether there is a match and where: the prefilter can only say "no match".
// The kernel also performs the scalar ops in front of the ALIGN op, so the exact pass starts from
// the stored state.
#include <cuda_runtime.h>
#include <stdint.h>

#include "csq_internal.h"
#include "device_common.cuh"

namespace {

// Prologue of every prefilter kernel: the scalar ops in front of the ALIGN op run here and the state is stored, so
// that the exact pass starts from it.
__device__ __forceinline__ ReadState prefilter_state(const AlignParams& P, uint32_t idx) {
    const ReadState st = entry_state(P, idx);
    store_state(P.md.state + idx, st);
    return st;
}

// Epilogue of every prefilter kernel, by the whole warp: the nominal DP cells of the launch (GCUPS numerator), then
// the warp-aggregated append of the survivors.  Survivors go to one of CSQ_PF_BINS lists (bin = class of the number of
// DP columns the exact pass will walk, so that the 32 reads of a k_align warp have similar trip counts); list b
// occupies list[b * n .. b * n + count[b]), the first DP column j0 of each entry sits behind the lists.
__device__ __forceinline__ void prefilter_epilogue(const AlignParams& P, uint32_t* __restrict__ list, uint32_t* __restrict__ list_count,
                                                   unsigned int cells, bool pass, uint32_t idx, int bin, uint32_t j0) {
    for (int o = 16; o > 0; o >>= 1) cells += __shfl_down_sync(0xffffffffu, cells, o);
    const int lane = threadIdx.x & 31;
    if (lane == 0 && cells) atomicAdd(P.counters + P.counter_index + (CNT_DP_CELLS - CNT_WITH_ADAPTERS), (unsigned long long)cells);
    uint16_t* __restrict__ list_j0 = reinterpret_cast<uint16_t*>(list + (size_t)CSQ_PF_BINS * P.n);
#pragma unroll
    for (int b = 0; b < CSQ_PF_BINS; b++) {
        const unsigned int ballot = __ballot_sync(0xffffffffu, pass && bin == b);
        if (!ballot) continue;
        const int leader = __ffs(ballot) - 1;
        unsigned int base = 0;
        if (lane == leader) base = atomicAdd(list_count + b, (unsigned int)__popc(ballot));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (pass && bin == b) {
            const size_t pos = (size_t)b * P.n + base + __popc(ballot & ((1u << lane) - 1u));
            list[pos] = idx;
            list_j0[pos] = (uint16_t)j0;
        }
    }
}

// Column window and survivor list of a read that passed with flags 14 (BACK, RightmostFront).  fc: number of columns
// done before the chunk in which cost[m][j] first dropped to thr[m], -1 if it never did (no row-m cell can be
// acceptable before that chunk); smin: the smallest cost[m][j].
__device__ __forceinline__ void window_and_bin(const AlignParams& P, int n, int min_n, int max_n, int fc, int smin, uint32_t& j0,
                                               int& bin) {
    // every cell Aligner.locate can accept lies in a column >= min(fc + 1, n); its value depends only on
    // columns >= that - (m + 3k + 2)  (k_align, "column window")
    const int jn = fc >= 0 ? fc : n;
    const int w0 = max(min_n, jn - (P.m + 3 * P.k + 3));
    j0 = (uint32_t)w0;
    const int cols = max_n - w0;
    // an error-free copy of the whole adapter (row-m cost 0 somewhere): Aligner.locate stops at that column
    // ("exact match, stop early"), about m + 3k + 3 + 16 columns behind w0 - a list of its own, so that the
    // warps of the exact pass that work on such reads leave together
    const bool exact_copy = smin == 0 && P.exact_stop;
    bin = exact_copy ? 3 : cols > 112 ? 0 : cols > 80 ? 1 : cols > 48 ? 2 : 4;  // longest first
}

// The read characters are fetched 16 columns at a time (fetch16): one thread walks 150 columns with ~10 fetches
// instead of 150 single-byte loads, which is what bounded the first version (L1 request rate).
//
// Template switches, all of them about instruction count per column (the kernel is issue bound):
//   REV    the reversed walk of RightmostFrontAdapter
//   SIR    adapter start is free (REFERENCE_START): row m can be acceptable in the first columns with a short
//          aligned length, so the per-column test is the full one.  Without it cost[m][j] >= m - j, and the
//          test is relaxed to  min_j cost[m][j] <= thr[m]  (thr is monotone, so this is still necessary for
//          acceptance) - one VIMNMX per column instead of a compare-and-branch.
//   SMALL  m <= 21: cost[m][j] is tracked scaled by 2^(m-1), i.e. the row-m bits of the horizontal delta
//          vectors are added / subtracted where they stand (cost <= m + n < 1024 still fits 32 bits).
template <int NW, bool REV, bool SIR, bool SMALL>
__global__ void __launch_bounds__(256) k_prefilter(const __grid_constant__ AlignParams P, uint32_t* __restrict__ list,
                                                   uint32_t* __restrict__ list_count) {
    __shared__ uint32_t lut[256 * NW];
    for (int c = threadIdx.x; c < 256; c += blockDim.x) {
        const int u = c & 0xDF;
        const int li = u == 'A' ? 0 : u == 'C' ? 1 : u == 'G' ? 2 : u == 'T' ? 3 : -1;
#pragma unroll
        for (int w = 0; w < NW; w++) lut[c * NW + w] = li >= 0 ? P.peq[li][w] : 0u;
    }
    __syncthreads();
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = idx < P.n;
    bool pass = false;
    unsigned int cells = 0;
    int bin = 0;
    uint32_t j0 = 0xFFFFu;  // first DP column of the exact pass; 0xFFFF: the aligner's own min_n
    if (valid) {
        const ReadState st = prefilter_state(P, idx);
        const int m = P.m, k = P.k;
        const int a = st.a, b = st.b, n = b - a;
        const bool siq = P.flags & 2, eir = P.flags & 4, eiq = P.flags & 8;
        int min_n, max_n;
        column_range(siq, eiq, m, k, n, min_n, max_n);
        cells = (unsigned int)(m * (max_n - min_n));

        // column min_n: cost[i] = i (vertical deltas all +1) unless the adapter start is free (all 0)
        uint32_t Pv[NW], Mv[NW];
#pragma unroll
        for (int w = 0; w < NW; w++) {
            Pv[w] = SIR ? 0u : 0xFFFFFFFFu;
            Mv[w] = 0u;
        }
        const int top = (m - 1) & 31;
        const uint32_t topmask = 1u << top;
        const int unit = SMALL ? (int)topmask : 1;  // one error in the units of `score`
        int score = SIR ? 0 : m * unit;             // cost[m][min_n]   (min_n == 0 whenever SIR, see csq_adapter_kind)
        int smin = 0x7FFFFFFF;                      // !SIR: minimum of cost[m][j] over the columns
        const uint32_t hpos0 = siq ? 0u : 1u;       // row 0: cost stays 0 (free read prefix) or grows by 1 per column
        const int min_overlap = P.min_overlap;
        const int kk = k * unit;
        int j = min_n;
        // Column window for the exact pass (BACK flags only, see k_align): fc = number of columns done before the
        // chunk in which cost[m][j] first dropped to thr[m] (no row-m cell can be acceptable before that)
        const bool window = !SIR && P.flags == 14;
        const int T = (int)P.thr[m] * unit;
        int fc = -1, jc = min_n;
        auto mark = [&](int cols) {
            if (window && fc < 0 && smin <= T) fc = jc;
            jc += cols;
        };
        auto column = [&](uint32_t c) {
            uint32_t hpos = hpos0, hneg = 0u;
#pragma unroll
            for (int w = 0; w < NW; w++) {
                uint32_t Eq = lut[c * NW + w];
                const uint32_t Xv = Eq | Mv[w];
                if (w > 0) Eq |= hneg;
                const uint32_t Xh = (((Eq & Pv[w]) + Pv[w]) ^ Pv[w]) | Eq;
                uint32_t Ph = Mv[w] | ~(Xh | Pv[w]);
                uint32_t Mh = Pv[w] & Xh;
                if (w == NW - 1) {  // horizontal delta of row m
                    if (SMALL) {
                        score += (int)(Ph & topmask) - (int)(Mh & topmask);
                    } else {
                        score += (int)((Ph >> top) & 1u) - (int)((Mh >> top) & 1u);
                    }
                }
                const uint32_t cp = Ph >> 31, cn = Mh >> 31;  // horizontal delta leaving this word
                Ph = (Ph << 1) | hpos;
                Mh = (Mh << 1) | hneg;
                hpos = cp;
                hneg = cn;
                Pv[w] = Mh | ~(Xv | Ph);
                Mv[w] = Ph & Xv;
            }
            if (SIR) {
                j++;
                if (eiq && score <= kk) {
                    const int sc = SMALL ? (score >> top) : score;
                    const int L = min(m, j + sc);
                    if (L >= min_overlap && sc <= (int)P.thr[L]) pass = true;
                }
            } else {
                smin = min(smin, score);
            }
        };
        // characters of columns min_n+1 .. max_n: s[a+min_n .. a+max_n) ascending, or, for the reversed walk
        // of RightmostFrontAdapter, s[b-max_n .. b-min_n) descending.  16 columns per fetch from an arbitrary
        // byte address (fetch16: five aligned 32-bit loads + four funnel shifts), so that all lanes of a warp
        // walk the same number of chunks whatever the alignment of their reads (records in a FASTQ text batch
        // start anywhere); the next chunk is in flight while these 16 columns are computed.  The fetch may touch
        // up to 19 bytes outside the read: every device pool is padded (plan.cu).
        const uint8_t* s = P.md.seq + P.md.seq_off[idx];
        int rem = max_n - min_n;
        if (!REV) {
            const uint8_t* p = s + a + min_n;
            uint4 v = make_uint4(0, 0, 0, 0);
            if (rem > 0) v = fetch16(p);
            for (; rem >= 16; rem -= 16) {
                p += 16;
                const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
                if (rem > 16) v = fetch16(p);
#pragma unroll
                for (int i = 0; i < 16; i++) column((w4[i >> 2] >> (8 * (i & 3))) & 0xFFu);
                mark(16);
            }
            if (rem > 0) {
                const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int i = 0; i < 15; i++) {
                    if (i >= rem) break;
                    column((w4[i >> 2] >> (8 * (i & 3))) & 0xFFu);
                }
                mark(rem);
            }
        } else {
            const uint8_t* p = s + b - min_n;  // one past the next character
            uint4 v = make_uint4(0, 0, 0, 0);
            if (rem > 0) v = fetch16(p - 16);
            for (; rem >= 16; rem -= 16) {
                p -= 16;
                const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
                if (rem > 16) v = fetch16(p - 16);
#pragma unroll
                for (int i = 15; i >= 0; i--) column((w4[i >> 2] >> (8 * (i & 3))) & 0xFFu);
                mark(16);
            }
            if (rem > 0) {
                const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int i = 15; i > 0; i--) {
                    if (15 - i >= rem) break;
                    column((w4[i >> 2] >> (8 * (i & 3))) & 0xFFu);
                }
                mark(rem);
            }
        }
        mark(0);
        if (!SIR && eiq && max_n > min_n && smin <= T) pass = true;
        if (!pass && max_n == n) {
            const int first_i = eir ? 0 : m;
            int d = siq ? 0 : max_n;  // cost[0][max_n]
            const int span = n - min_n;
            for (int i = 1; i <= m; i++) {
                const int w = (i - 1) >> 5, bt = (i - 1) & 31;
                uint32_t pv = Pv[0], mv = Mv[0];
#pragma unroll
                for (int x = 1; x < NW; x++)
                    if (w == x) {
                        pv = Pv[x];
                        mv = Mv[x];
                    }
                d += (int)((pv >> bt) & 1u) - (int)((mv >> bt) & 1u);
                if (i >= first_i && d <= k) {
                    const int L = min(i, span + d);
                    if (L >= min_overlap && d <= (int)P.thr[L]) pass = true;
                }
            }
        }
        if (!pass && P.matches) P.matches[idx] = no_match();
        if (pass && window) window_and_bin(P, n, min_n, max_n, fc, smin, j0, bin);
    }
    prefilter_epilogue(P, list, list_count, cells, pass, idx, bin, j0);
}


// ---- k_prefilter_fs: the hot form (BACK and RightmostFront: flags 14, m <= 32) balanced over BOTH integer pipes ---------
// On sm_100 LOP3 / SHF / IADD3 / VIMNMX issue on the ALU pipe and IMAD on the FMA pipe, each at one warp instruction
// per two cycles and scheduler (B300_MICROARCH.md, "fma vs alu split"); k_prefilter<1,...> above spends ~17 of its 19
// instructions per column on the ALU pipe and is bound by it (ncu: 85 % ALU, 64 % issue).  Here a column costs
//   ALU: 7 LOP3 (the Myers / Hyyro recurrences) + 1 PRMT (character) + 1 VIMNMX (running minimum of row m)      = 9
//   FMA: 1 IMAD (the carry-propagating add) + 2 IMAD (<< 1) + 2 IMAD.HI + 1 IMAD (row-m cost) + 1 IMAD (table address) = 7   + 1 LDS
// * the adapter sits in the TOP m bits of the word (row m = bit 31); the low 32 - m bits are rows that match every
//   character and start with vertical delta 0 - with a free read start (row 0 == 0 everywhere) they stay 0 for good
//   and hand a horizontal delta of 0 to the adapter's first row, exactly what the boundary row does;
// * the row-m horizontal deltas are bit 31 of Ph / Mh: mad.hi(x, 2, acc) == acc + (x >> 31) counts them on the FMA
//   pipe, and cost[m][j] - m = up - dn is one more mad.lo; only the running minimum is an ALU instruction;
// * adds and shifts are written as mad.lo with multipliers that come in as kernel arguments, so that ptxas cannot
//   fold them back into ALU-pipe forms.
// Same necessary condition, same survivor lists, same column window as k_prefilter with SIR = false.
__device__ __forceinline__ uint32_t imad_lo(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ uint32_t imad_hi(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
    asm("mad.hi.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

template <bool REV>
__global__ void __launch_bounds__(256) k_prefilter_fs(const __grid_constant__ AlignParams P, uint32_t* __restrict__ list,
                                                      uint32_t* __restrict__ list_count, const uint32_t one, const uint32_t two,
                                                      const uint32_t four, const uint32_t minus_one) {
    __shared__ uint32_t lut[256];
    const uint32_t lut_base = (uint32_t)__cvta_generic_to_shared(lut);
    const int m = P.m, sft = 32 - m;
    const uint32_t low = sft ? ((1u << sft) - 1u) : 0u;  // the always-matching rows below the adapter's first row
    for (int c = threadIdx.x; c < 256; c += blockDim.x) {
        const int u = c & 0xDF;
        const int li = u == 'A' ? 0 : u == 'C' ? 1 : u == 'G' ? 2 : u == 'T' ? 3 : -1;
        lut[c] = (li >= 0 ? (P.peq[li][0] << sft) : 0u) | low;
    }
    __syncthreads();
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = idx < P.n;
    bool pass = false;
    unsigned int cells = 0;
    int bin = 0;
    uint32_t j0 = 0xFFFFu;
    if (valid) {
        const ReadState st = prefilter_state(P, idx);
        const int k = P.k;
        const int a = st.a, b = st.b, n = b - a;
        const int max_n = n, min_n = 0;  // flags 14: read start and read end are free
        cells = (unsigned int)(m * n);
        uint32_t Pv = ~low, Mv = 0u;
        int smin = 0x7FFFFFFF;     // minimum over the columns of cost[m][j] - m
        const int T = (int)P.thr[m];
        int fc = -1, jc = 0;
        // one column without bookkeeping: returns Ph, Mh before the shift (bit 31 = horizontal delta of row m)
        // character x of the chunk: PRMT picks the byte (ALU), the scaled table address is an IMAD (FMA pipe)
        auto column = [&](const uint32_t (&w4)[4], int x, uint32_t& Ph, uint32_t& Mh) {
            const uint32_t c = __byte_perm(w4[x >> 2], 0u, 0x4440u + (uint32_t)(x & 3));
            uint32_t Eq;
            asm("ld.shared.u32 %0, [%1];" : "=r"(Eq) : "r"(imad_lo(c, four, lut_base)));
            const uint32_t Xv = Eq | Mv;
            const uint32_t Xh = (imad_lo(Eq & Pv, one, Pv) ^ Pv) | Eq;
            Ph = Mv | ~(Xh | Pv);
            Mh = Pv & Xh;
            const uint32_t Ph1 = imad_lo(Ph, two, 0u), Mh1 = imad_lo(Mh, two, 0u);
            Pv = Mh1 | ~(Xv | Ph1);
            Mv = Ph1 & Xv;
        };
        // 16 columns: the row-m cost of every column is m + up - dn (running counts of the +1 / -1 horizontal deltas of
        // row m, bit 31 of Ph / Mh, kept by mad.hi on the FMA pipe); its running minimum costs one ALU instruction.
        // (A first form only counted per chunk and re-walked "suspicious" chunks column by column: one suspicious
        // lane makes its whole warp walk again, 24 instead of 17 instructions per column on average.)
        uint32_t up = 0, dn = 0;
        auto follow = [&](uint32_t Ph, uint32_t Mh) {
            up = imad_hi(Ph, two, up);
            dn = imad_hi(Mh, two, dn);
            smin = min(smin, (int)imad_lo(dn, minus_one, up));
        };
        auto chunk16 = [&](const uint32_t (&w4)[4]) {
#pragma unroll
            for (int i = 0; i < 16; i++) {
                const int x = REV ? 15 - i : i;
                uint32_t Ph, Mh;
                column(w4, x, Ph, Mh);
                follow(Ph, Mh);
            }
            if (fc < 0 && smin <= T - m) fc = jc;
            jc += 16;
        };
        // The characters come in as aligned 128-bit vectors, ONE load per 16 columns: the chunk at byte offset o of the
        // window (lo | hi) is cut out in registers (window16), the window then slides by one vector - forwards
        // (lo <- hi, hi <- next) or, for the reversed walk of RightmostFront, backwards (hi <- lo, lo <- previous).
        // The vector for the chunk after the next one is in flight while 16 columns are computed.
        const uint8_t* s = P.md.seq + P.md.seq_off[idx];
        int rem = max_n - min_n;
        const uint8_t* q = REV ? (s + b - 16) : (s + a);  // first byte of the first chunk
        const uint4* vp = reinterpret_cast<const uint4*>((uintptr_t)q & ~(uintptr_t)15);
        const uint32_t o = (uint32_t)(uintptr_t)q & 15u;
        uint4 lo = make_uint4(0, 0, 0, 0), hi = lo;
        if (rem > 0) {
            lo = vp[0];
            hi = vp[1];
        }
        for (; rem >= 16; rem -= 16) {
            const uint4 v = window16(lo, hi, o);
            const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
            if (rem > 16) {
                if (REV) {
                    vp -= 1;
                    hi = lo;
                    lo = vp[0];
                } else {
                    vp += 1;
                    lo = hi;
                    hi = vp[1];
                }
            }
            chunk16(w4);
        }
        if (rem > 0) {
            const uint4 v = window16(lo, hi, o);
            const uint32_t w4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int i = 0; i < 15; i++) {
                if (i >= rem) break;
                const int x = REV ? 15 - i : i;
                uint32_t Ph, Mh;
                column(w4, x, Ph, Mh);
                follow(Ph, Mh);
            }
            if (fc < 0 && smin <= T - m) fc = jc;
        }
        smin = smin == 0x7FFFFFFF ? smin : smin + m;  // from "relative to cost[m][0] = m" to the cost itself
        if (max_n > min_n && smin <= T) pass = true;
        if (!pass) {  // last column (max_n == n): rows i >= first_i = 0 (REFERENCE_END), cost[0][n] = 0
            int d = 0;
            for (int i = 1; i <= m; i++) {
                const int bt = sft + i - 1;
                d += (int)((Pv >> bt) & 1u) - (int)((Mv >> bt) & 1u);
                if (d <= k) {
                    const int L = min(i, n + d);
                    if (L >= P.min_overlap && d <= (int)P.thr[L]) pass = true;
                }
            }
        }
        if (!pass && P.matches) P.matches[idx] = no_match();
        if (pass) window_and_bin(P, n, min_n, max_n, fc, smin, j0, bin);
    }
    prefilter_epilogue(P, list, list_count, cells, pass, idx, bin, j0);
}

template <int NW, bool REV, bool SIR>
void launch_pf(const AlignParams& p, uint32_t* list, uint32_t* list_count, dim3 grid, dim3 block, cudaStream_t stream) {
    if constexpr (NW == 1) {
        if (p.m <= 21) {
            k_prefilter<NW, REV, SIR, true><<<grid, block, 0, stream>>>(p, list, list_count);
            return;
        }
    }
    k_prefilter<NW, REV, SIR, false><<<grid, block, 0, stream>>>(p, list, list_count);
}

// RightmostFront is the only reversed kind and has flags 14 (SIR = 0); with m <= 32 it takes k_prefilter_fs, so the
// reversed walk is only instantiated without SIR and for NW >= 2.
template <int NW>
void launch_pf_nw(const AlignParams& p, uint32_t* list, uint32_t* list_count, dim3 grid, dim3 block, cudaStream_t stream) {
    if constexpr (NW >= 2) {
        if (p.reversed) {
            launch_pf<NW, true, false>(p, list, list_count, grid, block, stream);
            return;
        }
    }
    if (p.flags & 1) launch_pf<NW, false, true>(p, list, list_count, grid, block, stream);
    else launch_pf<NW, false, false>(p, list, list_count, grid, block, stream);
}

// Homopolymer adapters (the poly-A / poly-T 100-mers of reference run.py:389-404, 674-707) in their two
// non-internal kinds need no bit-vectors.  With e(l) = number of read characters different from the adapter
// base among the l characters next to the anchored end (read start for NonInternalFront, read end for
// NonInternalBack), every alignment that covers those l characters costs at least e(l), and covers at most
// l + cost adapter characters.  An alignment of length >= min_overlap needs cost >= min_overlap - l as well (a
// read shorter than min_overlap can still be covered by min_overlap adapter characters, with deletions), so the
// cost is at least c = max(e(l), min_overlap - l); thr[] grows by at most 1 per step, so "cost <= thr[min(m, l +
// cost)]" can only hold for some cost >= c if it holds for cost == c.  e(l) never decreases, hence the scan
// stops at the first l with e(l) > k (about 20 characters into a random read instead of m + k = 115 columns).
__global__ void __launch_bounds__(256) k_prefilter_homo(const __grid_constant__ AlignParams P, uint32_t* __restrict__ list,
                                                        uint32_t* __restrict__ list_count) {
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = idx < P.n;
    bool pass = false;
    unsigned int cells = 0;
    int bin = 0;
    if (valid) {
        const ReadState st = prefilter_state(P, idx);
        const int m = P.m, k = P.k;
        const int a = st.a, b = st.b, n = b - a;
        const int span = min(n, m + k);  // columns the aligner visits (max_n - min_n for both kinds)
        cells = (unsigned int)(m * span);
        const bool from_end = (P.flags & 2) != 0;  // NonInternalBack: anchored at the read end
        const uint8_t* s = P.md.seq + P.md.seq_off[idx];
        CharWalk cw;  // 16 characters per fetch, from the anchored end inwards
        cw.init(from_end ? (s + b) : (s + a), from_end);
        int e = 0, l = 1;
        for (; l <= span; l++) {
            e += ((cw.next() & 0xDFu) != (uint32_t)P.letter) ? 1 : 0;
            if (e > k) break;
            const int c = max(e, P.min_overlap - l);
            if (c <= (int)P.thr[min(m, l + c)]) {
                pass = true;
                break;
            }
        }
        if (pass) {
            // DP columns the exact pass will walk: all `span` of them when the read start is free, else up to the
            // column with the (k + 1)-th foreign character (the exact DP's early stop) - survivors are listed by that
            // number so that the threads of a k_align warp finish together
            int cols = span;
            if (!from_end) {
                for (l++; l <= span; l++) {
                    e += ((cw.next() & 0xDFu) != (uint32_t)P.letter) ? 1 : 0;
                    if (e > k) break;
                }
                cols = min(l, span);
            }
            bin = cols > 80 ? 0 : cols > 48 ? 1 : cols > 32 ? 2 : 4;  // longest first (list 3 is not used here)
        }
        if (!pass && P.matches) P.matches[idx] = no_match();
    }
    prefilter_epilogue(P, list, list_count, cells, pass, idx, bin, 0xFFFFu);
}

}  // namespace

cudaError_t csq_launch_prefilter(const AlignParams& p, uint32_t* list, uint32_t* list_count, cudaStream_t stream) {
    if (p.n == 0) return cudaSuccess;
    const dim3 grid((p.n + 255) / 256), block(256);
    if (p.homopolymer && !p.reversed && (p.flags == 9 || p.flags == 6)) {  // NonInternalFront / NonInternalBack
        k_prefilter_homo<<<grid, block, 0, stream>>>(p, list, list_count);
        return cudaGetLastError();
    }
    if (p.flags == 14 && p.m <= 32) {  // BACK / RightmostFront: the two-pipe form
        if (p.reversed) k_prefilter_fs<true><<<grid, block, 0, stream>>>(p, list, list_count, 1u, 2u, 4u, 0xFFFFFFFFu);
        else k_prefilter_fs<false><<<grid, block, 0, stream>>>(p, list, list_count, 1u, 2u, 4u, 0xFFFFFFFFu);
        return cudaGetLastError();
    }
    switch ((p.m + 31) / 32) {
        case 1: launch_pf_nw<1>(p, list, list_count, grid, block, stream); break;
        case 2: launch_pf_nw<2>(p, list, list_count, grid, block, stream); break;
        case 3: launch_pf_nw<3>(p, list, list_count, grid, block, stream); break;
        default: launch_pf_nw<4>(p, list, list_count, grid, block, stream); break;
    }
    return cudaGetLastError();
}
