// k_tail: everything behind the last ALIGN op, for both mates of a pair in ONE thread -
//   trailing CUT / COND_CUT / RENAME(capture) ops, QualityTrimmer (quality_trim_index of qualtrim.pyx),
//   SuffixRemover on the header and Renamer.parse_name's id              (reference run.py:330, 537-542, 377-380, 642-645, 415-417, 718-723)
//   the paired-name checks (dnaio's paired reader and cutadapt's PairedEndRenamer, both record_names_match)
//   the filters and the sink of run.py:446-471 / 763-792 (TooShort on either mate, IsUntrimmedAny), record byte
//   sizes and the per-CTA totals of the six output streams
// It replaces k_finish (once per mate) + k_pair of the first version: the two mate states of a pair never leave the
// registers between "finish" and the pair decision, the states are written once, and the header bytes that the id
// parser fetches anyway are compared for the name check (the emitters no longer look at ids).
// In text batches the '@' / '+' line starts of the FASTQ parser are checked here too (parse.cu, k_records).
// k_tail<true> serves FASTA batches (CSQ_PLAN_FASTA): the '>' in front of the header and the header limit are checked,
// there is no '+' line, and records are ">name\nseq\n".
#include <cuda_runtime.h>
#include <stdint.h>

#include "csq_internal.h"
#include "device_common.cuh"

namespace {

__device__ __forceinline__ uint32_t collapse4(uint32_t m) {  // bit 0 of every byte -> bits 0..3
    return (((m & 0x01010101u) * 0x00204081u) >> 21) & 0xFu;
}
// bit i set <=> byte i of the 16 is one of Python's str.split() blanks: ' ', 9..13, 28..31
__device__ __forceinline__ uint32_t space_bits16(uint4 v) {
    auto nib = [](uint32_t w) {
        return collapse4(__vcmpeq4(w, 0x20202020u) | (__vcmpgeu4(w, 0x09090909u) & __vcmpleu4(w, 0x0D0D0D0Du)) |
                         (__vcmpgeu4(w, 0x1C1C1C1Cu) & __vcmpleu4(w, 0x1F1F1F1Fu)));
    };
    return nib(v.x) | (nib(v.y) << 4) | (nib(v.z) << 8) | (nib(v.w) << 12);
}
// bit i set <=> byte i is ' ' or '\t' (the id delimiters of dnaio's record_ids_match: strcspn(header, " \t"))
__device__ __forceinline__ uint32_t spacetab_bits16(uint4 v) {
    auto nib = [](uint32_t w) { return collapse4(__vcmpeq4(w, 0x20202020u) | __vcmpeq4(w, 0x09090909u)); };
    return nib(v.x) | (nib(v.y) << 4) | (nib(v.z) << 8) | (nib(v.w) << 12);
}
// bit i set <=> byte i of x and y differ
__device__ __forceinline__ uint32_t differ_bits16(uint4 x, uint4 y) {
    return collapse4(__vcmpne4(x.x, y.x)) | (collapse4(__vcmpne4(x.y, y.y)) << 4) | (collapse4(__vcmpne4(x.z, y.z)) << 8) |
           (collapse4(__vcmpne4(x.w, y.w)) << 12);
}

struct MateTail {
    ReadState st;
    const uint8_t* nm;   // header (behind the '@')
    int raw_len;         // header length as it stands in the file
    int nl;              // ... after the SuffixRemovers
    uint32_t len0;       // bases of the original read
};

// One mate: trailing scalar ops, quality trimming, header suffixes and id.  Returns the bases removed by QTRIM.
template <bool FASTA>
__device__ __forceinline__ uint32_t finish_mate(const FinishParams& P, uint32_t idx, MateTail& T) {
    const uint32_t len0 = P.md.seq_len[idx];
    ReadState st = P.first ? fresh_state(len0) : load_state(P.md.state + idx);
    for (int q = 0; q < P.n_post; q++) apply_scalar(P.post[q], st);
    // header fetches are issued before the quality scan so that both latencies overlap
    const uint8_t* nm = P.md.name + P.md.name_off[idx];
    int nl = (int)(P.md.name_end[idx] - P.md.name_off[idx]);
    T.raw_len = nl;
    const uint4 nm0 = fetch16(nm);
    if (P.perr) {
        // text batch: the header line must start with '@' (the byte in front of the name) and the line behind the
        // bases with '+'; both bytes sit in sectors this thread fetches anyway.  Records at or behind an error
        // that is already known are skipped (the host reports the smallest key).
        const unsigned long long known = *reinterpret_cast<volatile unsigned long long*>(P.perr);
        if (FASTA) {
            if ((known >> 3) > (unsigned long long)idx) {
                int bad = 0;
                if (nm[-1] != '>') bad = 5;                                 // PERR_COUNT: not a record start
                else if (nl > 65535) bad = 7;                               // header limit
                if (bad) atomicMin(P.perr, ((unsigned long long)idx << 3) | (unsigned long long)bad);
            }
        } else if ((known >> 3) > (unsigned long long)idx) {
            const uint8_t* se = P.md.seq + P.md.seq_off[idx] + len0;  // the line end behind the bases
            int bad = 0;
            const uint8_t* pl = se + (se[0] == '\r' ? 2 : 1);         // the third line
            if (nm[-1] != '@') bad = 1;                                // PERR_AT
            else if (pl[0] != '+') bad = 2;                            // PERR_PLUS
            else if (nl > 65535) bad = 7;                              // PERR_HEADER_LIMIT (16-bit id fields of ReadState)
            else {
                // dnaio: a repeated header behind the '+' must be the header ("Sequence descriptions don't match")
                const uint8_t* qs = P.md.qual + P.md.qual_off[idx];    // first quality; the line end sits in front of it
                int pn = (int)(qs - 1 - pl) - 1;
                if (pn > 0 && pl[pn] == '\r') pn--;
                if (pn > 0) {
                    bool same = pn == nl;
                    for (int i = 0; same && i < nl; i++) same = pl[1 + i] == nm[i];
                    if (!same) bad = 6;                                // PERR_PLUS_NAME
                }
            }
            if (bad) atomicMin(P.perr, ((unsigned long long)idx << 3) | (unsigned long long)bad);
        }
    }
    uint32_t qtrimmed = 0;
    if (P.has_qtrim) {
        // quality_trim_index (qualtrim.pyx): running sums from either end, stop at the first negative sum.
        // Nearly every read stops within a few bases: the 16 qualities at either end are fetched at once
        // (two fetch16, issued together), the rare longer scans continue bytewise.
        const uint8_t* ql = P.md.qual + P.md.qual_off[idx];
        const int a = st.a, n = (int)st.b - (int)st.a;
        int start = 0, stop = n;
        if (n > 0) {
            const uint4 vf = fetch16(ql + a), vb = fetch16(ql + a + n - 16);
            const uint32_t wf[4] = {vf.x, vf.y, vf.z, vf.w}, wb[4] = {vb.x, vb.y, vb.z, vb.w};
            int s = 0, mx = 0, i = 0;
            bool open = true;
#pragma unroll
            for (int j = 0; j < 16; j++) {
                if (open && j < n) {
                    s += P.cutoff_front - ((int)((wf[j >> 2] >> (8 * (j & 3))) & 0xFFu) - P.qbase);
                    if (s < 0) {
                        open = false;
                    } else {
                        if (s > mx) {
                            mx = s;
                            start = j + 1;
                        }
                        i = j + 1;
                    }
                }
            }
            for (; open && i < n; i++) {
                s += P.cutoff_front - ((int)ql[a + i] - P.qbase);
                if (s < 0) break;
                if (s > mx) {
                    mx = s;
                    start = i + 1;
                }
            }
            s = 0;
            mx = 0;
            open = true;
            i = n - 1;
#pragma unroll
            for (int j = 15; j >= 0; j--) {  // byte j of vb is quality n - 16 + j
                if (open && n - 16 + j >= 0) {
                    s += P.cutoff_back - ((int)((wb[j >> 2] >> (8 * (j & 3))) & 0xFFu) - P.qbase);
                    if (s < 0) {
                        open = false;
                    } else {
                        if (s > mx) {
                            mx = s;
                            stop = n - 16 + j;
                        }
                        i = n - 17 + j;
                    }
                }
            }
            for (; open && i >= 0; i--) {
                s += P.cutoff_back - ((int)ql[a + i] - P.qbase);
                if (s < 0) break;
                if (s > mx) {
                    mx = s;
                    stop = i;
                }
            }
        }
        if (start >= stop) start = stop = 0;
        st.qtrim = (uint32_t)(n - (stop - start));
        st.b = (uint16_t)(st.a + stop);
        st.a = (uint16_t)(st.a + start);
        qtrimmed = st.qtrim;
    }
    // header: SuffixRemover ops in order, then the id of Renamer.parse_name
    for (int q = 0; q < P.n_suffix; q++) {
        const int sl = P.suffix_len[q];
        if (nl >= sl) {
            bool eq = true;
            for (int x = 0; x < sl; x++) eq = eq && (nm[nl - sl + x] == (uint8_t)P.suffix[q][x]);
            if (eq) nl -= sl;
        }
    }
    // str.split(maxsplit=1): s0 = first non-blank, e0 = first blank behind it, p = first non-blank behind that;
    // 16 header bytes per step, Python's whitespace set found with per-byte SIMD compares
    int s0 = nl, e0 = nl, p = nl, state = 0;
    for (int c = 0; c < nl && state < 3; c += 16) {
        const uint4 v = c == 0 ? nm0 : fetch16(nm + c);
        const uint32_t blank = space_bits16(v);
        const uint32_t valid = nl - c >= 16 ? 0xFFFFu : ((1u << (nl - c)) - 1u);
        uint32_t from = 0xFFFFu;  // positions still to look at in this chunk
        if (state == 0) {
            const uint32_t t = ~blank & valid & from;
            if (t) {
                const int b = __ffs(t) - 1;
                s0 = c + b;
                from = 0xFFFEu << b;
                state = 1;
            }
        }
        if (state == 1) {
            const uint32_t t = blank & valid & from;
            if (t) {
                const int b = __ffs(t) - 1;
                e0 = c + b;
                from = 0xFFFEu << b;
                state = 2;
            }
        }
        if (state == 2) {
            const uint32_t t = ~blank & valid & from;
            if (t) {
                p = c + (__ffs(t) - 1);
                state = 3;
            }
        }
    }
    if (P.has_rename && e0 > s0 && p < nl) {
        st.id_start = (uint16_t)s0;
        st.id_end = (uint16_t)e0;
    } else {
        st.id_start = 0;
        st.id_end = (uint16_t)min(nl, 65535);
    }
    store_state(P.md.state + idx, st);
    T.st = st;
    T.nm = nm;
    T.nl = nl;
    T.len0 = len0;
    return qtrimmed;
}

// dnaio record_names_match / SequenceRecord.is_mate (record_ids_match of upstream _core.pyx) for the headers h1 / h2:
// the id of header 2 ends at its first ' ' or '\t'; header 1 must end, or hold a ' ' / '\t', at that position; when
// both ids end in '1'..'3' that character is not compared; the rest must be byte-identical.  Evaluated twice on the
// same bytes: on the headers as they stand in the files (dnaio's paired reader) and on the headers as the
// SuffixRemovers left them (PairedEndRenamer, run.py:643-645) - prefixes of the former.
__device__ __forceinline__ bool pair_names_ok(const MateTail& A, const MateTail& B, bool renamer) {
    const uint8_t* __restrict__ h1 = A.nm;
    const uint8_t* __restrict__ h2 = B.nm;
    int id2 = B.raw_len;           // strcspn(h2, " \t")
    int first_diff = 0x7FFFFFFF;   // first index < id2 at which the headers differ
    for (int c = 0; c < B.raw_len; c += 16) {
        const uint4 v1 = fetch16(h1 + c), v2 = fetch16(h2 + c);
        const int left = B.raw_len - c;
        uint32_t valid = left >= 16 ? 0xFFFFu : ((1u << left) - 1u);
        const uint32_t st = spacetab_bits16(v2) & valid;
        if (st) {
            const int b = __ffs(st) - 1;
            id2 = c + b;
            valid = (1u << b) - 1u;
        }
        const uint32_t diff = differ_bits16(v1, v2) & valid;
        if (diff) {
            first_diff = c + __ffs(diff) - 1;
            break;
        }
        if (st) break;
    }
    auto ok = [&](int n1, int i2) {
        if (n1 < i2) return false;
        if (i2 < n1) {
            const uint8_t e = h1[i2];
            if (e != ' ' && e != '\t') return false;
        }
        int cmp = i2;
        if (i2 > 0) {
            const uint8_t x = h1[i2 - 1], y = h2[i2 - 1];
            if (x >= '1' && x <= '3' && y >= '1' && y <= '3') cmp--;
        }
        return first_diff >= cmp;
    };
    bool good = ok(A.raw_len, id2);
    if (renamer) good = good && ok(A.nl, min(id2, B.nl));
    return good;
}

struct TailParams {
    FinishParams fin[2];
    PairParams pp;
};

template <bool FASTA>
__global__ void __launch_bounds__(CSQ_PAIR_BLOCK) k_tail(const __grid_constant__ TailParams T) {
    const PairParams& P = T.pp;
    __shared__ unsigned int tot[8];   // bytes per (dest, mate) stream
    __shared__ unsigned int cnt[4];   // records per dest
    __shared__ unsigned int bp[2];    // bases written to the trimmed files, per mate
    __shared__ unsigned int qs[2];    // bases removed by QTRIM, per mate
    __shared__ unsigned int tb[2];    // input bases, per mate
    if (threadIdx.x < 8) tot[threadIdx.x] = 0;
    if (threadIdx.x < 4) cnt[threadIdx.x] = 0;
    if (threadIdx.x < 2) bp[threadIdx.x] = qs[threadIdx.x] = tb[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t idx = blockIdx.x * CSQ_PAIR_BLOCK + threadIdx.x;
    const bool paired = P.n_mates == 2;
    int dest = -1;
    uint32_t len1 = 0, len2 = 0, l1 = 0, l2 = 0, q1 = 0, q2 = 0, in1 = 0, in2 = 0;
    bool bad_names = false;
    if (idx < P.n) {
        MateTail m1, m2;
        q1 = finish_mate<FASTA>(T.fin[0], idx, m1);
        in1 = m1.len0;
        if (paired) {
            q2 = finish_mate<FASTA>(T.fin[1], idx, m2);
            in2 = m2.len0;
            bad_names = !pair_names_ok(m1, m2, P.check_ids != 0);
        }
        const ReadState& s1 = m1.st;
        const ReadState& s2 = paired ? m2.st : m1.st;
        l1 = (uint32_t)s1.b - (uint32_t)s1.a;
        l2 = (uint32_t)s2.b - (uint32_t)s2.a;
        if ((int)l1 < P.min_length || (paired && (int)l2 < P.min_length))
            dest = CSQ_DEST_SHORT;
        else if (P.untrimmed_enabled && ((P.required[0] & ~s1.matched) != 0 || (paired && (P.required[1] & ~s2.matched) != 0)))
            dest = CSQ_DEST_UNTRIMMED;
        else
            dest = CSQ_DEST_TRIMMED;
        P.dest[idx] = (uint8_t)dest;
        len1 = record_shape<FASTA>(P, s1, s1, s2).total;
        if (paired) len2 = record_shape<FASTA>(P, s2, s1, s2).total;
    }
    const int lane = threadIdx.x & 31;
    if (__any_sync(0xffffffffu, bad_names) && lane == 0) atomicExch(P.error_flag, (int)CSQ_ERR_PAIRING);
    {
        const unsigned int a1 = __reduce_add_sync(0xffffffffu, q1), a2 = __reduce_add_sync(0xffffffffu, q2);
        const unsigned int b1 = __reduce_add_sync(0xffffffffu, in1), b2 = __reduce_add_sync(0xffffffffu, in2);
        if (lane == 0) {
            if (a1) atomicAdd(&qs[0], a1);
            if (a2) atomicAdd(&qs[1], a2);
            atomicAdd(&tb[0], b1);
            if (paired) atomicAdd(&tb[1], b2);
        }
    }
#pragma unroll
    for (int d = 0; d < CSQ_N_DEST; d++) {
        const bool mine = dest == d;
        const unsigned int c = __popc(__ballot_sync(0xffffffffu, mine));
        if (c == 0) continue;  // warp-uniform
        const unsigned int t1 = __reduce_add_sync(0xffffffffu, mine ? len1 : 0u);
        const unsigned int t2 = __reduce_add_sync(0xffffffffu, mine ? len2 : 0u);
        unsigned int b1 = 0, b2 = 0;
        if (d == CSQ_DEST_TRIMMED) {
            b1 = __reduce_add_sync(0xffffffffu, mine ? l1 : 0u);
            b2 = __reduce_add_sync(0xffffffffu, (mine && paired) ? l2 : 0u);
        }
        if (lane == 0) {
            atomicAdd(&tot[d * 2 + 0], t1);
            if (paired) atomicAdd(&tot[d * 2 + 1], t2);
            atomicAdd(&cnt[d], c);
            if (d == CSQ_DEST_TRIMMED) {
                atomicAdd(&bp[0], b1);
                atomicAdd(&bp[1], b2);
            }
        }
    }
    __syncthreads();
    if (threadIdx.x < 8) P.block_tot[blockIdx.x * 8 + threadIdx.x] = tot[threadIdx.x];
    if (threadIdx.x < 4) P.block_cnt[blockIdx.x * 4 + threadIdx.x] = cnt[threadIdx.x];
    if (threadIdx.x == 0) {
        atomicAdd(P.counters + CNT_N, (unsigned long long)min((uint32_t)CSQ_PAIR_BLOCK, P.n - blockIdx.x * CSQ_PAIR_BLOCK));
        if (cnt[CSQ_DEST_TRIMMED]) atomicAdd(P.counters + CNT_WRITTEN, (unsigned long long)cnt[CSQ_DEST_TRIMMED]);
        if (bp[0]) atomicAdd(P.counters + CNT_WRITTEN_BP, (unsigned long long)bp[0]);
        if (bp[1]) atomicAdd(P.counters + CNT_WRITTEN_BP + 1, (unsigned long long)bp[1]);
        if (cnt[CSQ_DEST_SHORT]) atomicAdd(P.counters + CNT_TOO_SHORT, (unsigned long long)cnt[CSQ_DEST_SHORT]);
        if (cnt[CSQ_DEST_UNTRIMMED]) atomicAdd(P.counters + CNT_UNTRIMMED, (unsigned long long)cnt[CSQ_DEST_UNTRIMMED]);
        if (qs[0]) atomicAdd(P.counters + CNT_QTRIM_BP, (unsigned long long)qs[0]);
        if (qs[1]) atomicAdd(P.counters + CNT_QTRIM_BP + 1, (unsigned long long)qs[1]);
        if (tb[0]) atomicAdd(P.counters + CNT_TOTAL_BP, (unsigned long long)tb[0]);
        if (tb[1]) atomicAdd(P.counters + CNT_TOTAL_BP + 1, (unsigned long long)tb[1]);
    }
}

}  // namespace

cudaError_t csq_launch_tail(const FinishParams& f1, const FinishParams& f2, const PairParams& p, bool fasta, cudaStream_t stream) {
    if (p.n == 0) return cudaSuccess;
    TailParams T;
    T.fin[0] = f1;
    T.fin[1] = f2;
    T.pp = p;
    const uint32_t grid = (p.n + CSQ_PAIR_BLOCK - 1) / CSQ_PAIR_BLOCK;
    if (fasta)
        k_tail<true><<<grid, CSQ_PAIR_BLOCK, 0, stream>>>(T);
    else
        k_tail<false><<<grid, CSQ_PAIR_BLOCK, 0, stream>>>(T);
    return cudaGetLastError();
}
