// k_emit_stage: order-preserving FASTQ text emission ("@name\nseq\n+\nqual\n", dnaio's fastq_bytes) staged through
// shared memory - the default sink behind PairedEndSink / SingleEndSink of reference run.py:446-471 / 763-792.
//
// Why: the direct kernels (k_emit<G> in kernels.cu, k_emit_rec in emit.cu) move every record with
// byte-granular global loads and stores from arbitrary alignments; they spend 125-250 warp instructions per
// record on position bookkeeping and are bound by instruction issue at 48 % of the HBM copy peak.  Here the
// global side only ever sees aligned, fully coalesced 16-byte accesses, and the byte shuffling happens in
// shared memory where a lane can walk its own record:
//
//   phase 1 (thread per pair)   as before: destination, record sizes, CTA-wide exclusive scan per output
//                               stream -> where every record goes.  The descriptors stay in registers.
//   then each WARP walks its 32 pairs in passes of up to 8 pairs (16 single-end reads) = 16 records x 2 lanes:
//   load      the source bytes of the pass - in a text batch one contiguous span of the FASTQ text per mate - come
//             in as ONE bulk copy per span (cp.async.bulk global -> shared, TMA engine), issued by one lane and
//             awaited by the warp on its own mbarrier (expect_tx = bytes of all spans);
//   reformat  lane (record, role): role 0 writes '@' id ['_' UMI] '\n' bases '\n', role 1 writes '+' '\n' qualities
//             '\n' into the staging image of the output, 32-bit words built from two aligned shared-memory words
//             (funnel shift), ~5 instructions per 4 bytes and no bookkeeping in the loop;
//   flush     the records of a pass that go to the same output stream are contiguous there: the image is laid
//             out at the same offset modulo 16 as its place in the output and leaves as ONE bulk copy per span
//             (cp.async.bulk shared -> global); only the < 16 bytes at either end of a span go bytewise.  The
//             drain is awaited (wait_group.read) just before the next pass writes into the image again.
//   The passes of a warp are software-pipelined: pass i + 1 is sized and its loads are issued right after pass i has
//   been reformatted, so they are in flight during the flush of pass i.
//
// Every source byte is read once and every output byte written once.  A pass that does not fit the staging
// buffers is halved; a pair that does not fit alone (reads near the length limit with very long headers) takes
// a bytewise path.  (The mate-name check of PairedEndRenamer / dnaio's paired reader is k_tail's, tail.cu.)  The
// reverse-complementing single-end sink stays with k_emit.
// FASTA (CSQ_PLAN_FASTA): k_emit_stage<.., .., true> writes ">name\nseq\n"; header and bases are two source spans of the
// one text buffer (a wrapped sequence sits in the pool behind the text), there are no qualities and role-1 lanes idle.
#include <cuda_runtime.h>
#include <stdint.h>

#include "csq_internal.h"
#include "device_common.cuh"

namespace {

constexpr uint32_t ES_SRC_CAP = 6656;   // source bytes staged per warp and pass
constexpr uint32_t ES_DST_CAP = 5632;   // output bytes staged per warp and pass
constexpr uint32_t ES_SLACK = 16;       // readable bytes behind either region (the word loops look one word ahead)
constexpr uint32_t ES_WARP_BYTES = ES_SRC_CAP + ES_SLACK + ES_DST_CAP + ES_SLACK;
constexpr uint32_t ES_SRC0 = 0, ES_DST0 = ES_SRC_CAP + ES_SLACK;
constexpr int ES_WARPS = CSQ_PAIR_BLOCK / 32;
constexpr uint32_t FULL = 0xffffffffu;

struct StageRec {  // one mate of one pair, held by the lane that owns the pair in phase 1
    uint32_t nm;   // id bytes: offset into the name pool
    uint32_t sq;   // original read: offset into the seq pool
    uint32_t ql;   // ... into the qual pool
    uint32_t pa, pb;  // UMI parts: offsets into the seq pool of the mate they come from
    uint32_t ab;   // a | b << 16
    uint32_t idl;  // id_len | umi_len << 16  (umi_len counts the '_')
    uint32_t lab;  // lenA | lenB << 16
    uint32_t off;  // byte offset of the record inside the CTA's part of its output stream
    uint32_t len;  // bytes of the record
};

__device__ __forceinline__ StageRec shfl_rec(const StageRec& r, int src) {
    StageRec o;
    o.nm = __shfl_sync(FULL, r.nm, src);
    o.sq = __shfl_sync(FULL, r.sq, src);
    o.ql = __shfl_sync(FULL, r.ql, src);
    o.pa = __shfl_sync(FULL, r.pa, src);
    o.pb = __shfl_sync(FULL, r.pb, src);
    o.ab = __shfl_sync(FULL, r.ab, src);
    o.idl = __shfl_sync(FULL, r.idl, src);
    o.lab = __shfl_sync(FULL, r.lab, src);
    o.off = __shfl_sync(FULL, r.off, src);
    o.len = __shfl_sync(FULL, r.len, src);
    return o;
}

__device__ __forceinline__ uint32_t lds32(const uint8_t* sm, uint32_t a) { return *reinterpret_cast<const uint32_t*>(sm + a); }

// ---- bulk copies (TMA engine, 1-D) and the mbarrier a warp waits on ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t mbar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t mbar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
            : "=r"(done)
            : "r"(mbar), "r"(parity)
            : "memory");
    } while (!done);
}
// global -> shared, both 16-byte aligned, bytes a multiple of 16; completion is counted on `mbar`
__device__ __forceinline__ void bulk_load(uint32_t dst_smem, const void* src, uint32_t bytes, uint32_t mbar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem), "l"(src),
                 "r"(bytes), "r"(mbar)
                 : "memory");
}
// shared -> global, same constraints; part of the thread's current bulk group
__device__ __forceinline__ void bulk_store(void* dst, uint32_t src_smem, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src_smem), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// n bytes from shared offset s to shared offset d, any alignment on both sides.  Looks at most 7 bytes beyond s + n.
__device__ __forceinline__ void copy_s2s(uint8_t* sm, uint32_t s, uint32_t d, uint32_t n) {
    if (n == 0) return;
    const uint32_t h = min((4u - (d & 3u)) & 3u, n);  // bytes in front of the first whole output word
    if (h > 0) sm[d] = sm[s];
    if (h > 1) sm[d + 1] = sm[s + 1];
    if (h > 2) sm[d + 2] = sm[s + 2];
    s += h;
    d += h;
    n -= h;
    const uint32_t sh = (s & 3u) * 8u;
    uint32_t sa = s & ~3u;
    uint32_t w0 = lds32(sm, sa);
    if ((d & 4u) && n >= 4u) {  // one word to reach an 8-byte boundary of the output
        sa += 4;
        const uint32_t w1 = lds32(sm, sa);
        *reinterpret_cast<uint32_t*>(sm + d) = __funnelshift_r(w0, w1, sh);
        w0 = w1;
        d += 4;
        n -= 4;
    }
    const uint32_t nd = n >> 3;
#pragma unroll 4
    for (uint32_t i = 0; i < nd; i++) {
        const uint32_t w1 = lds32(sm, sa + 4), w2 = lds32(sm, sa + 8);
        *reinterpret_cast<uint2*>(sm + d) = make_uint2(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh));
        w0 = w2;
        sa += 8;
        d += 8;
    }
    if (n & 4u) {
        sa += 4;
        const uint32_t w1 = lds32(sm, sa);
        *reinterpret_cast<uint32_t*>(sm + d) = __funnelshift_r(w0, w1, sh);
        w0 = w1;
        d += 4;
    }
    n &= 3u;  // bytes behind the last whole word: the low bytes of one more funnel shift
    if (n) {
        const uint32_t w = __funnelshift_r(w0, lds32(sm, sa + 4), sh);
        sm[d] = (uint8_t)w;
        if (n > 1) sm[d + 1] = (uint8_t)(w >> 8);
        if (n > 2) sm[d + 2] = (uint8_t)(w >> 16);
    }
}

// (A 16-bytes-per-step form of the loop above - aligned LDS.128, the word rotation fixed per piece, STS.128 - was
// measured and dropped: the rotation differs from lane to lane, so its four loop variants run one after the other
// inside a warp; 0.745 ms against 0.645 ms per step, profiles/r01_emit_variants.md.)

// PAIRED: two mates per pair; ONE_POOL: text batch (header, bases and qualities of a mate in one buffer); FASTA: FASTA out
template <bool PAIRED, bool ONE_POOL, bool FASTA>
__global__ void __launch_bounds__(CSQ_PAIR_BLOCK, 2) k_emit_stage(const __grid_constant__ EmitParams E) {
    extern __shared__ __align__(16) uint8_t es_smem[];
    __shared__ unsigned int wtot[8][ES_WARPS];  // per-stream totals of every warp
    __shared__ __align__(8) unsigned long long load_bar[ES_WARPS];  // one mbarrier per warp: its bulk loads have landed
    const PairParams& P = E.pp;
    const uint32_t base = blockIdx.x * CSQ_PAIR_BLOCK;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    constexpr bool paired = PAIRED;
    constexpr int n_mates = PAIRED ? 2 : 1;
    uint8_t* const sm = es_smem + (uint32_t)wid * ES_WARP_BYTES;
    const uint32_t sm_u32 = smem_u32(sm), bar = smem_u32(&load_bar[wid]);
    if (lane == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }

    // ---- phase 1: where does every record go (thread per pair) ----
    const uint32_t idx = base + threadIdx.x;
    const bool live = idx < P.n;
    int dest = 0;
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
    for (int mt = 0; mt < n_mates; mt++)
        for (int d = 0; d < CSQ_N_DEST; d++) {
            const uint32_t v = (live && dest == d) ? len[mt] : 0u;
            uint32_t x = v;
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t y = __shfl_up_sync(FULL, x, o);
                if (lane >= o) x += y;
            }
            if (live && dest == d) incl[mt] = x;
            if (lane == 31) wtot[d * 2 + mt][wid] = x;
        }
    __syncthreads();
    StageRec rec[2];
#pragma unroll
    for (int mt = 0; mt < 2; mt++) {
        StageRec& R = rec[mt];
        R.nm = R.sq = R.ql = R.pa = R.pb = R.ab = R.idl = R.lab = R.off = R.len = 0;
        if (live && mt < n_mates) {
            const int stream = dest * 2 + mt;
            uint32_t off = incl[mt] - len[mt];
            for (int w = 0; w < wid; w++) off += wtot[stream][w];
            const MateDev& md = P.md[mt];
            const ReadState& own = st[mt];
            R.nm = md.name_off[idx] + own.id_start;
            R.sq = md.seq_off[idx];
            R.ql = md.qual_off[idx];
            if (P.rename_parts & CSQ_REN_OWN_PREFIX) R.pa = R.sq + (own.ren_cp >> 16);
            if (P.rename_parts & CSQ_REN_OWN_SUFFIX) R.pb = R.sq + (own.ren_cs >> 16);
            if (P.rename_parts & CSQ_REN_R1_PREFIX) R.pa = P.md[0].seq_off[idx] + (st[0].ren_cp >> 16);
            if (P.rename_parts & CSQ_REN_R2_PREFIX) R.pb = P.md[1].seq_off[idx] + (st[1].ren_cp >> 16);
            R.ab = (uint32_t)own.a | ((uint32_t)own.b << 16);
            R.idl = shape[mt].id_len | (shape[mt].umi_len << 16);
            R.lab = shape[mt].lenA | (shape[mt].lenB << 16);
            R.off = off;
            R.len = len[mt];
        }
    }
    // from here on the warps are on their own (no CTA-wide barrier below)
    const int n_warp = min(32, (int)P.n - (int)(base + (uint32_t)wid * 32u));
    if (n_warp <= 0) return;

    // where the CTA's part of every output stream begins
    uint8_t* gbase[CSQ_N_DEST][2];
#pragma unroll
    for (int d = 0; d < CSQ_N_DEST; d++)
#pragma unroll
        for (int mt = 0; mt < 2; mt++)
            gbase[d][mt] = E.out[d][mt] + (mt < n_mates ? E.block_off[(size_t)blockIdx.x * 8 + d * 2 + mt] : 0ull);
    // pools the UMI parts come from: the mate itself (single-end template) or R1 / R2 (paired template)
    const uint8_t* const poolA = (P.rename_parts & CSQ_REN_R1_PREFIX) ? P.md[0].seq : nullptr;
    const uint8_t* const poolB = (P.rename_parts & CSQ_REN_R2_PREFIX) ? P.md[1].seq : nullptr;
    // a text batch keeps header, bases and qualities of a mate in ONE buffer: one source span per mate and pass
    constexpr bool one_pool = ONE_POOL;
    constexpr int n_pools = FASTA ? 2 : ONE_POOL ? 1 : 3;

    const int q = lane >> 1, role = lane & 1;
    constexpr int ppass = PAIRED ? 8 : 16;
    const int my_mt = paired ? (q & 1) : 0;
    const int my_pp = paired ? (q >> 1) : q;  // pair of the pass this lane works on
    uint32_t bar_phase = 0;
    bool draining = false;  // a bulk store of this warp may still be reading the output image

    // One pass = up to `ppass` pairs starting at pair p0 of the warp.  Everything a lane has to know about it:
    struct Pass {
        StageRec R;            // my record
        int dest;              // its destination
        int g;                 // pairs in the pass; 0: none (the pair at p0 does not fit the staging buffers)
        bool valid;            // this lane has a record
        bool loads;            // bulk loads were issued (and have to be awaited)
        uint32_t sdelta[3];    // staged address of pool offset x of my mate: ES_SRC0 + sdelta[pool] + x
        uint32_t ddelta;       // staged address of my record: ES_DST0 + ddelta + R.off
    };

    // Sizes the pass at p0 (halving it until it fits) and, if it fits, issues one bulk load per source span.
    // The source buffer must be free: the previous pass has been reformatted.
    auto prepare = [&](int p0, Pass& ps) {
        const int src_lane = (p0 + my_pp) & 31;
        const StageRec r0 = shfl_rec(rec[0], src_lane), r1 = shfl_rec(rec[1], src_lane);
        ps.R = my_mt ? r1 : r0;
        const StageRec& R = ps.R;
        ps.dest = __shfl_sync(FULL, dest, src_lane);
        const uint32_t a = R.ab & 0xFFFFu, b = R.ab >> 16;
        const uint32_t id_len = R.idl & 0xFFFFu;
        const uint32_t la = R.lab & 0xFFFFu, lb = R.lab >> 16;
        // source pieces of this record in pool coordinates: name [nm, nm + id_len), bases [sq + a, sq + b),
        // qualities [ql + a, ql + b); empty pieces take no part in the spans
        uint32_t plo[3], phi[3];
        plo[0] = R.nm;
        phi[0] = R.nm + id_len;
        plo[1] = R.sq + a;
        phi[1] = R.sq + b;
        plo[2] = R.ql + a;
        phi[2] = R.ql + b;
        // the UMI parts are staged with the bases of the mate whose read they were cut from
        if (la && (!PAIRED || my_mt == 0)) {
            plo[1] = min(plo[1], R.pa);
            phi[1] = max(phi[1], R.pa + la);
        }
        if (lb && (!PAIRED || my_mt == 1)) {
            plo[1] = min(plo[1], R.pb);
            phi[1] = max(phi[1], R.pb + lb);
        }
        if (one_pool) {
            uint32_t lo = 0xFFFFFFFFu, hi = 0;
#pragma unroll
            for (int k = 0; k < 3; k++)
                if (phi[k] > plo[k]) {
                    lo = min(lo, plo[k]);
                    hi = max(hi, phi[k]);
                }
            plo[0] = lo;
            phi[0] = hi;
        }
        int g = min(ppass, n_warp - p0);
        uint32_t sp_lo16[2][3], sp_n16[2][3], sp_base[2][3];  // source spans: pool offset, 16-byte chunks, staged offset
        ps.sdelta[0] = ps.sdelta[1] = ps.sdelta[2] = 0;
        ps.ddelta = 0;
        for (;;) {
            ps.valid = my_pp < g;
            uint32_t cursor = 0;
#pragma unroll
            for (int mt = 0; mt < 2; mt++)
#pragma unroll
                for (int k = 0; k < 3; k++) {
                    sp_n16[mt][k] = 0;
                    sp_lo16[mt][k] = sp_base[mt][k] = 0;
                    if (mt < n_mates && k < n_pools) {
                        const bool part = ps.valid && role == 0 && my_mt == mt && phi[k] > plo[k];
                        const uint32_t lo = __reduce_min_sync(FULL, part ? plo[k] : 0xFFFFFFFFu);
                        const uint32_t hi = __reduce_max_sync(FULL, part ? phi[k] : 0u);
                        if (hi > lo) {
                            const uint32_t lo16 = lo & ~15u;
                            const uint32_t n16 = (hi - lo16 + 15u) >> 4;
                            sp_lo16[mt][k] = lo16;
                            sp_n16[mt][k] = n16;
                            sp_base[mt][k] = cursor;
                            if (my_mt == mt) ps.sdelta[k] = cursor - lo16;
                            cursor += n16 << 4;
                        }
                    }
                }
            // output: the records of one (destination, mate) stream are contiguous there
            uint32_t dcursor = 0;
#pragma unroll
            for (int d = 0; d < CSQ_N_DEST; d++)
#pragma unroll
                for (int mt = 0; mt < 2; mt++) {
                    const bool part = ps.valid && role == 0 && my_mt == mt && ps.dest == d;
                    const uint32_t mask = __ballot_sync(FULL, part);
                    if (mask) {
                        const uint32_t goff = __shfl_sync(FULL, R.off, __ffs((int)mask) - 1);
                        const uint32_t bytes = __reduce_add_sync(FULL, part ? R.len : 0u);
                        const uint32_t mis = (uint32_t)(uintptr_t)(gbase[d][mt] + goff) & 15u;
                        const uint32_t dstart = ((dcursor + 15u) & ~15u) + mis;
                        dcursor = dstart + bytes;
                        if (my_mt == mt && ps.dest == d) ps.ddelta = dstart - goff;
                    }
                }
            if (cursor <= ES_SRC_CAP && dcursor <= ES_DST_CAP) break;
            if (g == 1) {
                g = 0;
                break;
            }
            g >>= 1;
        }
        ps.g = g;
        ps.loads = false;
        if (g == 0) return;
        uint32_t total = 0;
#pragma unroll
        for (int mt = 0; mt < 2; mt++)
#pragma unroll
            for (int k = 0; k < 3; k++) total += sp_n16[mt][k] << 4;
        ps.loads = total != 0;
        if (lane == 0) {
            if (total) mbar_expect_tx(bar, total);
#pragma unroll
            for (int mt = 0; mt < 2; mt++)
#pragma unroll
                for (int k = 0; k < 3; k++) {
                    if (sp_n16[mt][k] == 0) continue;
                    const MateDev& md = P.md[mt];
                    const uint8_t* pool = k == 0 ? (one_pool ? md.seq : md.name) : k == 1 ? md.seq : md.qual;
                    bulk_load(sm_u32 + ES_SRC0 + sp_base[mt][k], pool + sp_lo16[mt][k], sp_n16[mt][k] << 4, bar);
                }
        }
    };

    // The pair at p0 does not fit the staging buffers: bytewise, straight from and to global memory.
    auto bytewise = [&](int p0) {
        const int sl = p0 & 31;
        const int fd = __shfl_sync(FULL, dest, sl);
#pragma unroll
        for (int mt = 0; mt < 2; mt++) {
            if (mt >= n_mates) continue;
            const StageRec F = shfl_rec(rec[mt], sl);
            const MateDev& md = P.md[mt];
            const uint32_t fa = F.ab & 0xFFFFu, fb = F.ab >> 16, fl = fb - fa, fid = F.idl & 0xFFFFu, fumi = F.idl >> 16;
            const uint32_t fla = F.lab & 0xFFFFu;
            const uint8_t* nm = md.name + F.nm;
            const uint8_t* sq = md.seq + F.sq + fa;
            const uint8_t* ql = md.qual + F.ql + fa;
            const uint8_t* pa = (poolA ? poolA : md.seq) + F.pa;
            const uint8_t* pb = (poolB ? poolB : md.seq) + F.pb;
            uint8_t* out = (fd == 0 ? gbase[0][mt] : fd == 1 ? gbase[1][mt] : gbase[2][mt]) + F.off;
            const uint32_t e_name = 1u + fid, e_umi = e_name + fumi, e_seq = e_umi + 1u + fl, e_qual = e_seq + 3u + fl;
            for (uint32_t p = lane; p < F.len; p += 32) {
                uint8_t c;
                if (p < e_name) c = p == 0 ? (uint8_t)(FASTA ? '>' : '@') : nm[p - 1];
                else if (p < e_umi) {
                    const uint32_t x = p - e_name;
                    c = x == 0 ? (uint8_t)'_' : (x - 1 < fla ? pa[x - 1] : pb[x - 1 - fla]);
                } else if (p == e_umi) c = '\n';
                else if (p < e_seq) c = sq[p - e_umi - 1];
                else if (FASTA) c = '\n';
                else if (p < e_seq + 3) c = (p - e_seq == 1) ? (uint8_t)'+' : (uint8_t)'\n';
                else if (p < e_qual) c = ql[p - e_seq - 3];
                else c = '\n';
                out[p] = c;
            }
        }
    };

    // the next pass that goes through the staging buffers, starting at pair `next_p0` (pairs that do not fit are
    // written bytewise on the way); ps.g == 0: the warp is done
    int next_p0 = 0;
    auto advance = [&](Pass& ps) {
        ps.g = 0;
        while (next_p0 < n_warp) {
            prepare(next_p0, ps);
            if (ps.g) {
                next_p0 += ps.g;
                return;
            }
            bytewise(next_p0);
            next_p0 += 1;
        }
    };

    // Software pipeline: the loads of pass i + 1 are issued as soon as pass i has been reformatted (the source buffer
    // is free then) and are in flight during the flush of pass i and the bookkeeping of pass i + 1.
    Pass cur;
    advance(cur);
    while (cur.g) {
        const StageRec R = cur.R;
        const bool valid = cur.valid;
        const int my_dest = cur.dest;
        const uint32_t a = R.ab & 0xFFFFu, b = R.ab >> 16, seq_len = b - a;
        const uint32_t id_len = R.idl & 0xFFFFu, umi_len = R.idl >> 16;
        const uint32_t la = R.lab & 0xFFFFu, lb = R.lab >> 16;
        const uint32_t d0 = ES_DST0 + cur.ddelta + R.off;  // my record in the output image
        const uint32_t sd_name = cur.sdelta[0], sd_seq = one_pool ? cur.sdelta[0] : cur.sdelta[1], sd_qual = one_pool ? cur.sdelta[0] : cur.sdelta[2];
        // staged bases of the mates the UMI parts come from (paired: lanes 4 pp .. 4 pp + 3 hold one pair)
        const uint32_t sd_a = PAIRED ? __shfl_sync(FULL, sd_seq, lane & ~3) : sd_seq;
        const uint32_t sd_b = PAIRED ? __shfl_sync(FULL, sd_seq, (lane & ~3) | 2) : sd_seq;
        if (draining) {  // the previous pass's bulk stores must have read the output image before it is written again
            if (lane == 0) bulk_wait_read();
            draining = false;
        }
        if (cur.loads) {
            mbar_wait(bar, bar_phase);
            bar_phase ^= 1u;
        }
        __syncwarp();

        // ---- reformat ----
        const uint32_t s_id = ES_SRC0 + sd_name + R.nm;
        if (valid && (!FASTA || role == 0)) {
            const uint32_t d_seq = d0 + 1u + id_len + umi_len + 1u;
            const uint32_t d_qual = d_seq + seq_len + 3u;
            const uint32_t s_big = ES_SRC0 + (role ? sd_qual + R.ql : sd_seq + R.sq) + a;
            copy_s2s(sm, s_big, role ? d_qual : d_seq, seq_len);
            if (role == 0) {
                sm[d0] = FASTA ? '>' : '@';
                copy_s2s(sm, s_id, d0 + 1u, id_len);
                if (umi_len) {
                    sm[d0 + 1u + id_len] = '_';
                    copy_s2s(sm, ES_SRC0 + sd_a + R.pa, d0 + 2u + id_len, la);
                    copy_s2s(sm, ES_SRC0 + sd_b + R.pb, d0 + 2u + id_len + la, lb);
                }
                sm[d_seq - 1u] = '\n';
                sm[d_seq + seq_len] = '\n';
            } else {
                sm[d_qual - 2u] = '+';
                sm[d_qual - 1u] = '\n';
                sm[d_qual + seq_len] = '\n';
            }
        }
        fence_async_smem();  // the image was written through the generic proxy, the bulk copies read it through the async proxy
        __syncwarp();

        // ---- the next pass: sized now, its loads fly during the flush below ----
        const uint32_t f_off = R.off, f_len = R.len;
        advance(cur);

        // ---- flush: every (destination, mate) span of the finished pass leaves as one bulk copy ----
        {
            uint32_t dcursor = 0;
#pragma unroll
            for (int d = 0; d < CSQ_N_DEST; d++)
#pragma unroll
                for (int mt = 0; mt < 2; mt++) {
                    const bool part = valid && role == 0 && my_mt == mt && my_dest == d;
                    const uint32_t mask = __ballot_sync(FULL, part);
                    if (mask) {
                        const uint32_t goff = __shfl_sync(FULL, f_off, __ffs((int)mask) - 1);
                        const uint32_t bytes = __reduce_add_sync(FULL, part ? f_len : 0u);
                        uint8_t* __restrict__ gp = gbase[d][mt] + goff;
                        const uint32_t mis = (uint32_t)(uintptr_t)gp & 15u;
                        const uint32_t dstart = ((dcursor + 15u) & ~15u) + mis;
                        dcursor = dstart + bytes;
                        const uint8_t* __restrict__ sp = sm + ES_DST0 + dstart;
                        const uint32_t head = min((16u - mis) & 15u, bytes);
                        const uint32_t body = (bytes - head) & ~15u;
                        const uint32_t done = head + body, tail = bytes - done;
                        if (lane == 0 && body) bulk_store(gp + head, sm_u32 + ES_DST0 + dstart + head, body);
                        if ((uint32_t)lane < head) gp[lane] = sp[lane];
                        if ((uint32_t)lane >= 16u && (uint32_t)lane - 16u < tail) gp[done + lane - 16u] = sp[done + lane - 16u];
                    }
                }
        }
        if (lane == 0) bulk_commit();
        draining = true;
        __syncwarp();
    }
    if (draining && lane == 0) bulk_wait_read();  // shared memory must outlive the reads of the last bulk stores
}

template <bool PAIRED, bool ONE_POOL, bool FASTA = false>
cudaError_t launch_stage(const EmitParams& p, cudaStream_t stream) {
    // per device: a function attribute belongs to the current context
    cudaError_t attr = cudaFuncSetAttribute(k_emit_stage<PAIRED, ONE_POOL, FASTA>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(ES_WARPS * ES_WARP_BYTES));
    if (attr != cudaSuccess) return attr;
    k_emit_stage<PAIRED, ONE_POOL, FASTA><<<(p.pp.n + CSQ_PAIR_BLOCK - 1) / CSQ_PAIR_BLOCK, CSQ_PAIR_BLOCK, ES_WARPS * ES_WARP_BYTES, stream>>>(p);
    return cudaGetLastError();
}

}  // namespace

cudaError_t csq_launch_emit_stage(const EmitParams& p, bool fasta, cudaStream_t stream) {
    if (p.pp.n == 0) return cudaSuccess;
    const PairParams& P = p.pp;
    const bool paired = P.n_mates == 2;
    if (fasta) return paired ? launch_stage<true, false, true>(p, stream) : launch_stage<false, false, true>(p, stream);
    const bool one_pool = P.md[0].seq == P.md[0].name && P.md[0].seq == P.md[0].qual;
    if (paired) return one_pool ? launch_stage<true, true>(p, stream) : launch_stage<true, false>(p, stream);
    return one_pool ? launch_stage<false, true>(p, stream) : launch_stage<false, false>(p, stream);
}
