// K4 synth_reads + K5 pack_fastq: per-read synthesis (indels, k-mer-context substitutions, Phred
// qualities) and FASTQ packing, one warp per read slot (SE read / PE pair).
//
// Replaces Amplicon::yieldReads (/root/reference/lib/amplicon/Amplicon.cpp:402-565), the sequence
// rebuild Amplicon::getSequence (Amplicon.cpp:255-382), Profile::predict and its samplers
// (lib/profile/Profile.cpp:1482-1697), the sprintf/strncpy record formatting (Amplicon.cpp:459-541)
// and SeqWriter::write (lib/seqwriter/SeqWriter.cpp:41-54).
//
// Per slab of consecutive slots:  emit (fixed-stride staging + record sizes)  ->  exclusive scan (byte
// offsets)  ->  compaction into the packed slab  ->  D2H into the pinned host ring.
// The emit kernel walks the slot's draw stream with the same cursors the reference's sequential code
// would have, but evaluates 64 positions per step (2 per lane, one Philox4x32 block per lane) and
// resolves the rare indel events with a ballot, so a read costs ~RL/32 steps instead of RL.
// All sampling is integer compares against the threshold tables built on the host. Records are
// assembled in shared memory at the destination's 16-byte phase and stored with 128-bit stores.
#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>

#include <sched.h>

#define SCS_PHILOX_OUTLINE 1
#include "ctx.h"
#include "expand_host.h"
#include "slab_sink.h"
#include "wire.h"

namespace scs {

__device__ __noinline__ void philox4x32_10_call(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t* out) {
    philox4x32_10(c0, c1, c2, c3, k0, k1, out);
}

constexpr int kReadWarps = 8;         // warps per CTA (test kernels)
#ifndef SCS_EMIT_WARPS
#define SCS_EMIT_WARPS 28
#endif
constexpr int kEmitWarps = SCS_EMIT_WARPS;   // warps per persistent CTA of the emit kernel (one CTA per SM); tuning: profiles/ab_warps.sh
constexpr int kDiagW = 40;            // entries per compact quality row kept in shared memory (shipped profiles need <= 39)
constexpr int kDiagStride = 44;       // words per row: 40 + 4 pad; 44*r mod 32 is a distinct multiple of 4 for 8 neighbouring rows,
                                      // so their 128-bit loads are bank-conflict free
constexpr int kRLCap = 320;           // max profile read length handled by the kernels (Illumina tops out at 2 x 300)
#ifndef SCS_EMIT_BATCH_DRAWS   // 1: plan_slot evaluates the slot's four warp-uniform single draws in one Philox pass (A/B in profiles/NOTES_r02.md)
#define SCS_EMIT_BATCH_DRAWS 1
#endif
constexpr int kSrcCap = 480;          // max read length after insertions (overflow -> error flag)
constexpr int kMaxEvents = 64;        // indel events per read kept in shared memory
constexpr int kRecCap = 16 + 40 + 2 * kSrcCap + 8;
constexpr int kWinBytes = 96;         // staged 2-bit window of one mate: kRLCap bases (80 B) + up to 15 B in front, rounded to 16
constexpr int kWinNBytes = 64;        // staged N-mask window of one mate: kRLCap bits (40 B) + up to 15 B in front, rounded to 16
static_assert(15 + (kRLCap + 2) / 4 + 16 <= kWinBytes + 15 && 15 + (kRLCap + 6) / 8 + 16 <= kWinNBytes + 15, "window staging too small for kRLCap");
constexpr int kCoarseShift = 10;      // coarse slot -> amplicon index: one entry per 1024 slots
constexpr int kISizeSmemCap = 4096;   // insert-size thresholds kept in shared memory (longer tables stay in global memory)

struct ReadTables {
    const uint32_t* subs1; const uint32_t* subs2;   // [84][bins][4]  (3 thresholds + eff)
    const uint32_t* qual; const uint8_t* qualEff;    // [16][bins][94], [16][bins]
    const uint32_t* ins; const uint32_t* del; const uint32_t* isize;
    int insEff, delEff, isizeEff, minInsert, maxInsert;
    uint64_t thrIns, thrDel;                         // insertion iff x < thrIns ; else deletion iff x2 < thrDel
    // free-running streams: the distance to the next indel event is drawn directly (see indel_pass). q = P(no event at a position)
    double indelLogQ;                                // det_log(q)
    uint64_t thrInsType;                             // the event is an insertion iff x < thrInsType  (pI / (1 - q))
    uint32_t thrNoEvent;                             // x < thrNoEvent: certainly no event within RL positions (0.99 q^RL: skips the logarithm)
    int indelAny;                                    // q < 1
    int RL, paired;
    // compact copies of the 4 diagonal (no substitution) quality tables for shared memory
    const uint32_t* diagRows; const uint4* diagPiv; const uint32_t* diagMeta;   // [4][bins][36], [4][bins], [4][bins] lo | cnt<<8 | global<<16
};

struct QualSmem { const uint32_t* rows; const uint4* piv; const uint32_t* meta; };
// what the substitution + quality pass needs, small enough to travel by value in registers (the out-of-line N path must not force
// the kernel's parameter structs onto the stack)
struct PassTabs {
    const uint4* subs;                                  // substitution thresholds of this mate, [84][bins] x (3 thresholds + count)
    const uint32_t* qual; const uint8_t* qualEff;       // global quality thresholds
    const uint32_t* rows; const uint4* piv; const uint32_t* meta;   // compact diagonal quality rows in shared memory (rows == nullptr: none)
    int bins;
};
__device__ __forceinline__ PassTabs make_pass_tabs(const ReadTables& T, const QualSmem* Q, int isRead1) {
    PassTabs X;
    X.subs = reinterpret_cast<const uint4*>((!isRead1 && T.subs2) ? T.subs2 : T.subs1);
    X.qual = T.qual; X.qualEff = T.qualEff; X.bins = T.RL;
    X.rows = Q ? Q->rows : nullptr; X.piv = Q ? Q->piv : nullptr; X.meta = Q ? Q->meta : nullptr;
    return X;
}

// What the emit kernel knows about a slot one slot ahead of processing it (stage A -> stage B, through shared memory)
struct SlotPlan {
    uint64_t entity;          // Philox entity / replay mark index
    const uint32_t* errs;     // substitution overlay of the slot's amplicon
    uint32_t ampIdx, fragNo, nerr, cr, ci;
    int32_t pos, isz;
    uint32_t woff[2];         // window of mate m starts woff[m] bases into win[m]; bit 31: read it backwards and complemented
    uint32_t noff[2];         // same for the N mask (bases into winn[m])
    int32_t valid;
    uint32_t gap[2], gap_idx[2];   // free-running: first indel-stage draw of each mate, precomputed with the slot's other single draws
};

struct __align__(16) WarpScratch {
    uint8_t ref[kRLCap + 16];   // + slack: the 4-bases-per-lane decode stores whole words
    uint8_t src[kSrcCap];
    char rec[kRecCap];
    int16_t ev_pos[kMaxEvents]; int16_t ev_len[kMaxEvents]; uint32_t ev_ci[kMaxEvents];
};
// per-warp staging of the emit kernel: packed genome windows of the next slots land here through cp.async.bulk (TMA)
struct __align__(16) WarpStage {
    uint8_t win[2][2][kWinBytes];     // [buffer][mate]
    uint8_t winn[2][2][kWinNBytes];   // N mask, only filled when the genome holds N
    SlotPlan plan[2];
    uint64_t bar[2];                  // mbarrier per buffer: completes when the buffer's bulk copies have landed
};

// ---- mbarrier + bulk-copy (TMA) primitives, sm_90+ PTX ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// global -> shared, `bytes` a multiple of 16, both addresses 16-byte aligned; completion is counted on `bar`
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes),
                 "r"(smem_u32(bar))
                 : "memory");
}

// Stream with the replay decision made at compile time: the free-running kernels carry no tape branches (and no tape code —
// the emit kernel has to stay small enough for the instruction cache), the replay instantiation no Philox.
template <bool REPLAY> struct RStream : Stream {
    __device__ __forceinline__ bool replay() const { return REPLAY; }
    __device__ __forceinline__ void block(int engine, uint32_t b, uint32_t out[4]) const {
        if (REPLAY) { const uint32_t* p = t[engine] + 4ull * b; out[0] = p[0]; out[1] = p[1]; out[2] = p[2]; out[3] = p[3]; }
        else philox4x32_10(e0, e1, b, dom2 + (uint32_t)engine, k0, k1, out);
    }
    __device__ __forceinline__ uint32_t at(int engine, uint32_t i) const {
        if (REPLAY) return t[engine][i];
        uint32_t o[4];
        philox4x32_10_call(e0, e1, i >> 2, dom2 + (uint32_t)engine, k0, k1, o);
        return o[i & 3];
    }
};

// Draws base+4*lane .. base+4*lane+3 of one engine: one Philox block per lane. When `base` is not a multiple of 4 a lane also
// needs the first words of its right neighbour's block; instead of running a 33rd block for lane 31 alone (a whole Philox for one
// lane), only lanes 0..30 own positions in that case. Returns the number of draws the step covers (128 or 124).
template <class SX>
__device__ __forceinline__ int warp_draws4(const SX& S, int eng, uint32_t base, int lane, uint32_t x[4]) {
    if (S.replay()) {
        const uint32_t* p = S.t[eng] + base + 4u * lane;
        x[0] = p[0]; x[1] = p[1]; x[2] = p[2]; x[3] = p[3];
        return 128;
    }
    uint32_t o[4], nx[4];
    const uint32_t B = (base >> 2) + lane, sh = base & 3u;
    S.block(eng, B, o);
    if (sh == 0) { x[0] = o[0]; x[1] = o[1]; x[2] = o[2]; x[3] = o[3]; return 128; }
#pragma unroll
    for (int q = 0; q < 3; q++) nx[q] = __shfl_down_sync(0xffffffffu, o[q], 1);
    if (sh == 1) { x[0] = o[1]; x[1] = o[2]; x[2] = o[3]; x[3] = nx[0]; }
    else if (sh == 2) { x[0] = o[2]; x[1] = o[3]; x[2] = nx[0]; x[3] = nx[1]; }
    else { x[0] = o[3]; x[1] = nx[0]; x[2] = nx[1]; x[3] = nx[2]; }
    return 124;
}

// Indel pass of Profile::predict (Profile.cpp:1603-1630) over n source positions. Advances the real /
// int cursors exactly as the sequential code does; returns the output length n'. Events (position,
// +inserted / -deleted, first int draw) go to the warp scratch; *nev = 0 if there are none or if the
// "< 50 bases" guard discarded them.
template <class SX>
__device__ __forceinline__ int indel_pass(const SX& S, const ReadTables& T, int n, uint32_t& cr, uint32_t& ci, int lane, WarpScratch* ws,
                                          int* nev_out, int* flags, uint32_t pre_idx = 0xFFFFFFFFu, uint32_t pre_x = 0) {
    // pre_x: real draw number pre_idx of this stream, if the caller already has it (plan_slot computes the slot's single draws together)
    int j = 0, delta = 0, nev = 0;
    if (!S.replay()) {
        // Free-running streams: per position the reference decides "insertion" with probability pI, else "deletion" with
        // probability pD, the same at every position — so the number of event-free positions before the next event is
        // geometric, q = (1 - pI)(1 - pD), and the event is an insertion with probability pI / (1 - q). One draw per read (89 %
        // of the reads have no event: x < thrNoEvent answers that without the logarithm) instead of 2 per base; the oracle's
        // free-running predict() draws the same way (oracle/profile.h), replay keeps the reference's consumption below.
        SCS_CHECK(n <= T.RL);
        while (T.indelAny && j < n) {
            const uint32_t x = (cr == pre_idx) ? pre_x : S.at(E_REAL, cr);
            cr++;
            if (x < T.thrNoEvent) break;
            const double u = __ddiv_rn(__dadd_rn((double)x, 0.5), 4294967296.0);
            const double gd = floor(__ddiv_rn(det_log(u), T.indelLogQ));
            if (!(gd < (double)(n - j))) break;
            const int p = j + (int)gd;
            const bool insertion = (uint64_t)S.at(E_REAL, cr++) < T.thrInsType;
            const uint32_t xl = S.at(E_REAL, cr++);
            if (insertion) {   // insertion after base p: k base draws on the int engine
                const int k = min(count_le(T.ins, T.insEff, xl), T.insEff);
                if (k > 0) {
                    if (nev < kMaxEvents) { if (lane == 0) { ws->ev_pos[nev] = (int16_t)p; ws->ev_len[nev] = (int16_t)k; ws->ev_ci[nev] = ci; } }
                    else if (lane == 0) atomicOr(flags, 4);
                    nev++; delta += k; ci += (uint32_t)k;
                }
                j = p + 1;
            } else {           // deletion of k bases starting at p
                int k = min(count_le(T.del, T.delEff, xl), T.delEff);
                k = min(n - p, k);
                if (k > 0) {
                    if (nev < kMaxEvents) { if (lane == 0) { ws->ev_pos[nev] = (int16_t)p; ws->ev_len[nev] = (int16_t)(-k); ws->ev_ci[nev] = 0; } }
                    else if (lane == 0) atomicOr(flags, 4);
                    nev++; delta -= k; j = p + k;
                } else j = p + 1;
            }
        }
    } else
    while (j < n) {
        uint32_t x[4];
        const int P = warp_draws4(S, E_REAL, cr, lane, x) >> 1;   // positions covered by this step (2 draws each)
        const int pA = j + 2 * lane;
        int ev = 0;
        if (2 * lane < P) {
            if (pA < n) { if ((uint64_t)x[0] < T.thrIns) ev = 1; else if ((uint64_t)x[1] < T.thrDel) ev = 2; }
            if (!ev && pA + 1 < n) { if ((uint64_t)x[2] < T.thrIns) ev = 3; else if ((uint64_t)x[3] < T.thrDel) ev = 4; }
        }
        const uint32_t any = __ballot_sync(0xffffffffu, ev != 0);
        if (!any) { int used = min(P, n - j); j += used; cr += 2u * used; continue; }
        const int l0 = __ffs(any) - 1;
        const int e = __shfl_sync(0xffffffffu, ev, l0);
        const int p = j + 2 * l0 + (e >= 3);
        const uint32_t crp = cr + 2u * (uint32_t)(p - j);
        if (e == 1 || e == 3) {   // insertion after base p: length draw, then k base draws on the int engine
            uint32_t xl = S.at(E_REAL, crp + 1);
            int k = min(count_le(T.ins, T.insEff, xl), T.insEff);
            cr = crp + 2;
            if (k > 0) {
                SCS_CHECK(p >= 0 && p < n);
                if (nev < kMaxEvents) { if (lane == 0) { ws->ev_pos[nev] = (int16_t)p; ws->ev_len[nev] = (int16_t)k; ws->ev_ci[nev] = ci; } }
                else if (lane == 0) atomicOr(flags, 4);
                nev++; delta += k; ci += (uint32_t)k;
            }
            j = p + 1;
        } else {                  // deletion of k bases starting at p
            uint32_t xl = S.at(E_REAL, crp + 2);
            int k = min(count_le(T.del, T.delEff, xl), T.delEff);
            k = min(n - p, k);
            cr = crp + 3;
            if (k > 0) {
                if (nev < kMaxEvents) { if (lane == 0) { ws->ev_pos[nev] = (int16_t)p; ws->ev_len[nev] = (int16_t)(-k); ws->ev_ci[nev] = 0; } }
                else if (lane == 0) atomicOr(flags, 4);
                nev++; delta -= k; j = p + k;
            } else j = p + 1;
        }
    }
    if (nev > kMaxEvents) nev = kMaxEvents;
    if (n + delta < 50) { delta = 0; nev = 0; }   // Profile.cpp:1623-1630
    *nev_out = nev;
    return n + delta;
}

// source sequence after indels (Profile.cpp:1632-1654): every lane maps its output positions back through the
// (few) recorded events, so there is no serial walk
template <class SX>
__device__ __noinline__ void build_source_events(const SX S, int np, int nev, int lane, WarpScratch* ws) {
    for (int m = lane; m < np; m += 32) {
        int shift = 0; uint32_t b = 0; bool done = false;
        for (int e = 0; e < nev; e++) {
            const int p = ws->ev_pos[e], L = ws->ev_len[e];
            const int mp = p + shift;                 // output index of source position p
            if (L > 0) {                              // L bases inserted after p (A/C/G only, Profile.cpp:1560)
                if (m <= mp) break;
                if (m <= mp + L) { b = uni_trunc(S.at(E_INT, ws->ev_ci[e] + (uint32_t)(m - mp - 1)), 0, 3); done = true; break; }
                shift += L;
            } else {                                  // -L bases deleted starting at p
                if (m < mp) break;
                shift += L;
            }
        }
        SCS_CHECK(m < kSrcCap && (done || (m - shift >= 0 && m - shift < kRLCap)));
        ws->src[m] = done ? (uint8_t)b : ws->ref[m - shift];
    }
    __syncwarp();
}
// only ~11 % of the reads carry an indel event: the rebuild stays out of line so that the hot path is short
template <class SX>
__device__ __forceinline__ const uint8_t* build_source(const SX& S, int np, int nev, int lane, WarpScratch* ws) {
    if (nev == 0) return ws->ref;
    build_source_events(S, np, nev, lane, ws);
    return ws->src;
}

// quality index for (reference base b0, emitted base k, bin): diagonal rows from shared memory with a
// 4-pivot + 8-entry search (two dependent 128-bit loads), everything else by binary search in global memory
__device__ __forceinline__ int sample_quality(const PassTabs& X, uint32_t b0, uint32_t k, int bin, uint32_t xq) {
    if (X.rows != nullptr && k == b0) {
        const int r = (int)b0 * X.bins + bin;
        SCS_CHECK(r >= 0 && r < 4 * X.bins);
        const uint32_t meta = X.meta[r];
        if ((meta >> 16) == 0) {
            const int lo = (int)(meta & 0xFFu), cnt = (int)((meta >> 8) & 0xFFu);
            const uint4 pv = X.piv[r];
            // pivots = entries 7, 15, 23, 31: they select one of five octets, which is then counted
            const int oct = (int)(pv.x <= xq) + (int)(pv.y <= xq) + (int)(pv.z <= xq) + (int)(pv.w <= xq);
            SCS_CHECK(oct >= 0 && oct <= 4);
            const uint4* row = reinterpret_cast<const uint4*>(X.rows + (size_t)r * kDiagStride + oct * 8);
            const uint4 a = row[0], d = row[1];
            const int c = oct * 8 + (int)(a.x <= xq) + (int)(a.y <= xq) + (int)(a.z <= xq) + (int)(a.w <= xq) + (int)(d.x <= xq) + (int)(d.y <= xq) +
                          (int)(d.z <= xq) + (int)(d.w <= xq);
            return lo + min(c, cnt);
        }
    }
    const size_t row = (size_t)(b0 * 4u + k) * X.bins + bin;
    SCS_CHECK(b0 < 4u && k < 4u && bin >= 0 && bin < X.bins && X.qualEff[row] <= kQualN);
    return count_le(X.qual + row * kQualN, (int)X.qualEff[row], xq);
}

// substitution + quality loop (Profile.cpp:1656-1694): two output positions per lane per step. The threshold rows of both
// positions are requested before the Philox block is computed, so the L2 latency of the loads hides under the ~100 ALU instructions.
template <class SX>
__device__ __forceinline__ void subst_quality_pass(const SX& S, const PassTabs& X, const uint8_t* __restrict__ src, int np,
                                                   uint32_t& cr, int lane, char* __restrict__ oseq, char* __restrict__ oqual) {
    const uint4* __restrict__ subs = X.subs;
    const int bins = X.bins;
    const int P = S.replay() ? 64 : (((cr & 3u) == 0) ? 64 : 62);   // the alignment of cr + 2*m0 does not change inside the pass
    // bin = m * bins / np (Profile.cpp:1667): m itself for a read without indels, else by multiplication with ceil(2^32 / np)
    // (exact: m * bins * np < 2^32)
    const uint32_t inv = (np == bins) ? 0u : (uint32_t)((0x100000000ull + (uint32_t)np - 1u) / (uint32_t)np);
    for (int m0 = 0; m0 < np; m0 += P) {
        uint4 th[2]; uint32_t b0[2]; int bin[2];
        const int mA = m0 + 2 * lane;
        const bool okA = (2 * lane < P) && mA < np, okB = okA && mA + 1 < np;
        // requests for the threshold rows of both positions first (addresses clamped for idle lanes: no predication around the loads)
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const int m = min(mA + h, np - 1);
            b0[h] = src[m];
            const uint32_t p1 = src[max(m - 1, 0)], p2 = src[max(m - 2, 0)];
            const uint32_t ki = (m == 0) ? b0[h] : (m == 1) ? 4u + 4u * p1 + b0[h] : 20u + 16u * p2 + 4u * p1 + b0[h];
            bin[h] = inv ? (int)__umulhi((uint32_t)(m * bins), inv) : m;
            SCS_CHECK(ki < 84u && bin[h] >= 0 && bin[h] < bins && bin[h] == m * bins / np && b0[h] < 4u);
            th[h] = __ldg(subs + ((size_t)ki * bins + bin[h]));
        }
        uint32_t x[4];
        warp_draws4(S, E_REAL, cr + 2u * m0, lane, x);
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const uint32_t xs = x[2 * h], xq = x[2 * h + 1];
            // thresholds are non-decreasing and padded with 0xFFFFFFFF: the leading count, capped by the row's entry count
            const uint32_t k = min((uint32_t)(th[h].x <= xs) + (uint32_t)(th[h].y <= xs) + (uint32_t)(th[h].z <= xs), th[h].w);
            const int q = sample_quality(X, b0[h], k, bin[h], xq);
            if (h == 0 ? okA : okB) {
                oseq[mA + h] = (char)((0x54474341u >> (8u * k)) & 0xFFu);   // "ACGT"[k]
                oqual[mA + h] = (char)(33 + q);
            }
        }
    }
    cr += 2u * (uint32_t)np;
}

// Same loop for windows that hold an N (code 4): the number of draws per output base then varies — 0 real + 1 int for an N
// (emitted as 'N' with quality randomInteger(33,53), Profile.cpp:1578-1580,1686-1688), 1 real when only the k-mer context
// holds an N (no substitution draw, Profile.cpp:1527-1529), 2 otherwise — so draw indices come from a warp prefix sum.
// WRITE = false only advances the cursors (plan kernel).
template <bool WRITE, class SX>
__device__ __noinline__ uint2 subst_quality_pass_n(const SX S, const PassTabs X, const uint8_t* __restrict__ src, int np,
                                                     uint32_t cr, uint32_t ci, int lane, char* __restrict__ oseq, char* __restrict__ oqual) {
    const uint4* __restrict__ subs = X.subs;
    const int bins = X.bins;
    for (int m0 = 0; m0 < np; m0 += 32) {
        const int m = m0 + lane;
        const bool valid = m < np;
        const uint32_t b0 = valid ? src[m] : 0u;
        const bool curN = valid && b0 == 4u;
        const bool ctxN = valid && !curN && ((m >= 1 && src[m - 1] == 4u) || (m >= 2 && src[m - 2] == 4u));
        uint32_t nr = !valid ? 0u : curN ? 0u : ctxN ? 1u : 2u, ni = curN ? 1u : 0u;
        uint32_t pr = nr, pi = ni;   // inclusive scans
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t a = __shfl_up_sync(0xffffffffu, pr, o), b = __shfl_up_sync(0xffffffffu, pi, o);
            if (lane >= o) { pr += a; pi += b; }
        }
        const uint32_t tot_r = __shfl_sync(0xffffffffu, pr, 31), tot_i = __shfl_sync(0xffffffffu, pi, 31);
        if (WRITE && valid) {
            const uint32_t ir = cr + pr - nr, ii = ci + pi - ni;
            if (curN) {
                oseq[m] = 'N';
                oqual[m] = (char)uni_trunc(S.at(E_INT, ii), 33, 20);
            } else {
                const int bin = (np == bins) ? m : m * bins / np;
                uint32_t k = b0, xq;
                if (!ctxN) {
                    uint32_t ki;
                    if (m == 0) ki = b0; else if (m == 1) ki = 4u + 4u * src[0] + b0; else ki = 20u + 16u * src[m - 2] + 4u * src[m - 1] + b0;
                    const uint4 th = __ldg(subs + ((size_t)ki * bins + bin));
                    const uint32_t xs = S.at(E_REAL, ir);
                    k = (uint32_t)(th.w > 0 && th.x <= xs) + (uint32_t)(th.w > 1 && th.y <= xs) + (uint32_t)(th.w > 2 && th.z <= xs);
                    xq = S.at(E_REAL, ir + 1);
                } else xq = S.at(E_REAL, ir);
                const int q = sample_quality(X, b0, k, bin, xq);
                oseq[m] = (char)((0x54474341u >> (8u * k)) & 0xFFu);
                oqual[m] = (char)(33 + q);
            }
        }
        cr += tot_r; ci += tot_i;
    }
    return make_uint2(cr, ci);   // the cursors after the pass
}

__device__ __forceinline__ int dec_digits(uint32_t v) {
    return v < 10u ? 1 : v < 100u ? 2 : v < 1000u ? 3 : v < 10000u ? 4 : v < 100000u ? 5 : v < 1000000u ? 6 : v < 10000000u ? 7 : v < 100000000u ? 8 : v < 1000000000u ? 9 : 10;
}
// floor(2^64 / 10^k) + 1: v / 10^k == umul64hi(v, kInvPow10[k]) for every 32-bit v (error < 2^-32 < 10^-9 <= 1/10^k); k = 0 unused
__constant__ uint64_t kInvPow10[10] = {0ull, 1844674407370955162ull, 184467440737095517ull, 18446744073709552ull, 1844674407370956ull,
                                       184467440737096ull, 18446744073710ull, 1844674407371ull, 184467440738ull, 18446744074ull};
// "@%d#%d" (+"/1" | "/2") + "\n": the %d of a negative amplicon index never occurs (index < 2^31)
__device__ __forceinline__ int header_len(int da, int df, int paired) { return 1 + da + 1 + df + (paired ? 2 : 0) + 1; }
// the whole record frame in one go, one character per lane: header digits (lane l = l-th character after '@'), "/m", and the
// three separators "\n+\n" ... "\n" around the sequence and quality lines of np characters each
__device__ __forceinline__ void write_frame(char* rec, uint32_t amp, uint32_t frag, int da, int df, int mate, int hl, int np, int lane) {
    if (lane < da + 1 + df && lane != da) {   // one digit: value / 10^k % 10 by multiplication with the 64-bit reciprocal
        const bool first = lane < da;
        const uint32_t v = first ? amp : frag;
        const int k = first ? da - 1 - lane : df - 1 - (lane - da - 1);
        const uint32_t q = k ? (uint32_t)__umul64hi((uint64_t)v, kInvPow10[k]) : v;
        rec[1 + lane] = (char)('0' + q % 10u);
    } else if (lane == da) rec[1 + da] = '#';
    else if (lane == 24) rec[0] = '@';
    else if (lane == 25) { if (mate) { rec[hl - 3] = '/'; rec[hl - 2] = (char)('0' + mate); } rec[hl - 1] = '\n'; }
    else if (lane == 26) { rec[hl + np] = '\n'; rec[hl + np + 1] = '+'; rec[hl + np + 2] = '\n'; }
    else if (lane == 27) rec[hl + 2 * np + 3] = '\n';
}

// copy ceil(n/16) 16-byte vectors smem -> global, both 16-byte aligned (the staging stride is a multiple of 16, so the
// few bytes copied past the record stay inside its own staging cell)
__device__ __forceinline__ void copy_out(char* __restrict__ dst, const char* __restrict__ srcp, int n, int lane) {
    const int nvec = (n + 15) >> 4;
    const uint4* s4 = reinterpret_cast<const uint4*>(srcp);
    uint4* d4 = reinterpret_cast<uint4*>(dst);
    for (int i = lane; i < nvec; i += 32) d4[i] = s4[i];
}

struct SlabArgs {
    uint64_t slot0, nslots;            // this launch covers local slots [slot0, slot0 + nslots)
    const uint64_t* slot_gbase;        // per amplicon: global id of its first slot (Philox entity / replay mark index)
    const uint64_t* amp_gidx;          // per amplicon: global list index (FASTQ header)
    uint64_t n_amp;
    const uint64_t* slot_base;         // [n_amp + 1] exclusive prefix of slots per amplicon
    const uint64_t* desc; const uint64_t* errref; const uint32_t* err_pool;
    const uint32_t* hdr_no;            // slow path: fragCount per slot (0 = dropped); nullptr -> slot index + 1
    const uint32_t* nfail;             // slow path: failed insert-size attempts before the slot's success
    uint64_t fail_base;                // hdr_no / nfail are indexed by (slot - fail_base)
    uint64_t slab_cap;                 // bytes available in each output slab
    uint64_t stage_stride;             // record of slot ls goes to stage + ls * stage_stride (a multiple of 16)
    const uint32_t* coarse;            // amplicon of slot coarse_base + j * 2^kCoarseShift (one entry more than needed)
    uint64_t coarse_base;
};

// count_le on a long row, evaluated by the whole warp: 32 pivots, then the segment between two pivots (2 ballots)
__device__ __forceinline__ int warp_count_le(const uint32_t* __restrict__ row, int n, uint32_t x, int lane) {
    if (n <= 0) return 0;
    if (n > 1024) return count_le(row, n, x);
    const int step = (n + 31) >> 5;
    const int pi = min((lane + 1) * step, n) - 1;                       // last entry of lane's segment
    const uint32_t below = __ballot_sync(0xffffffffu, row[pi] <= x);    // a prefix of lanes (row is non-decreasing)
    const int seg = __popc(below);                                      // segments fully <= x
    if (seg >= 32) return n;
    const int base = seg * step;
    if (base >= n) return n;
    const int idx = base + lane;
    const bool le = lane < step && idx < n && row[idx] <= x;
    return base + __popc(__ballot_sync(0xffffffffu, le));
}

// amplicon of a slot: last a in [lo, hi) with slot_base[a] <= slot, by a warp-cooperative 32-ary search.
// Precondition: slot_base[lo] <= slot < slot_base[hi] (the coarse index narrows [lo, hi) to a few dozen amplicons: one probe).
__device__ __forceinline__ uint64_t find_amplicon(const uint64_t* __restrict__ slot_base, uint64_t lo, uint64_t hi, uint64_t slot, int lane) {
    while (hi - lo > 1) {
        const uint64_t width = hi - lo, step = (width + 31) >> 5;
        const uint64_t idx = lo + (uint64_t)lane * step;
        const bool le = idx < hi && __ldg(slot_base + idx) <= slot;
        const uint32_t m = __ballot_sync(0xffffffffu, le);   // prefix of lanes (slot_base is non-decreasing), lane 0 always set
        const int j = __popc(m) - 1;
        lo = lo + (uint64_t)j * step;
        hi = min(hi, lo + step);
    }
    return lo;
}

// ---- stage A: everything a slot needs before its bases arrive — amplicon lookup, header numbers, insert size and position
// ---- draws — then ONE lane asks the TMA unit for the packed windows of both mates (cp.async.bulk -> this warp's shared memory).
// ---- Runs one slot ahead of stage B, so the dependent-load chain (coarse index -> slot prefix -> descriptor -> genome) of the
// ---- next slot overlaps the synthesis of the current one.
template <bool SIZE_ONLY, bool REPLAY>
__device__ __forceinline__ void plan_slot(const Genome& g, const DrawSrc& dsrc, const ReadTables& T, const uint32_t* __restrict__ isize_row, const SlabArgs& A,
                                          uint64_t ls, int lane, WarpStage* st, int buf) {
    const uint64_t slot = A.slot0 + ls;
    const uint64_t cj = (slot - A.coarse_base) >> kCoarseShift;
    const uint64_t a = find_amplicon(A.slot_base, __ldg(A.coarse + cj), min((uint64_t)__ldg(A.coarse + cj + 1) + 1, A.n_amp), slot, lane);
    SCS_CHECK(a < A.n_amp && __ldg(A.slot_base + a) <= slot && slot < __ldg(A.slot_base + a + 1));
    const Tmpl F = unpack_desc(__ldg(A.desc + a));
    const uint64_t sb = __ldg(A.slot_base + a);
    const uint64_t er = __ldg(A.errref + a);
    const uint32_t ampIdx = A.amp_gidx ? (uint32_t)__ldg(A.amp_gidx + a) : (uint32_t)a;
    const uint64_t entity = __ldg(A.slot_gbase + a) + (slot - sb);
    const uint32_t fragNo = A.hdr_no ? A.hdr_no[slot - A.fail_base] : (uint32_t)(slot - sb) + 1u;
    const int RL = T.RL; const int ampLen = (int)F.len;
    const bool valid = fragNo != 0 && ampLen >= RL;   // dropped slot / Amplicon.cpp:442
    const bool need_bases = !SIZE_ONLY || g.has_n;    // record sizes depend on the bases only through the draws an N consumes
    uint32_t cr = 0, ci = 0; int pos = 0, isz = RL;
    uint32_t woff[2] = {0, 0}, noff[2] = {0, 0};
    uint32_t gap_x[2] = {0, 0}, gap_i[2] = {0xFFFFFFFFu, 0xFFFFFFFFu};
    __syncwarp();   // every lane is done reading this buffer's previous windows and plan
    if (valid) {
        RStream<REPLAY> S; S.init(dsrc, D_READ, entity, entity);
        if (T.paired && A.nfail) cr = A.nfail[slot - A.fail_base];   // failed attempts each consumed one real draw (Amplicon.cpp:483-490)
        uint32_t x_isz = 0, x_pos;
#if SCS_EMIT_BATCH_DRAWS
        if (!REPLAY) {
            // The slot's warp-uniform single draws in ONE Philox evaluation: lane 0 the block of the insert-size draw, lane 1 of the
            // position draw, lanes 2 / 3 of the first indel-stage draw of mate 1 / mate 2 (mate 2's index assumes that mate 1
            // consumes 1 + 2 RL draws — no indel event, no N; indel_pass checks the index and draws itself otherwise)
            const uint32_t i1 = cr + (T.paired ? 1u : 0u), i2 = i1 + 1u + 2u * (uint32_t)RL;
            const uint32_t want = lane == 1 ? 0u : lane == 2 ? i1 : lane == 3 ? i2 : cr;
            uint32_t o[4];
            philox4x32_10_call(S.e0, S.e1, want >> 2, S.dom2 + (uint32_t)(lane == 1 ? E_INT : E_REAL), S.k0, S.k1, o);
            const uint32_t v = (want & 2u) ? ((want & 1u) ? o[3] : o[2]) : ((want & 1u) ? o[1] : o[0]);
            x_isz = __shfl_sync(0xffffffffu, v, 0); x_pos = __shfl_sync(0xffffffffu, v, 1);
            gap_x[0] = __shfl_sync(0xffffffffu, v, 2); gap_x[1] = __shfl_sync(0xffffffffu, v, 3);
            gap_i[0] = i1; gap_i[1] = i2;
        } else
#endif
        { if (T.paired) x_isz = S.at(E_REAL, cr); x_pos = S.at(E_INT, ci); }
        if (T.paired) {
            isz = T.minInsert + warp_count_le(isize_row, T.isizeEff, x_isz, lane);
            cr += 1;
            pos = (int)uni_trunc(x_pos, 0, (uint32_t)(ampLen - isz + 1)); ci += 1;
        } else {
            pos = (int)uni_trunc(x_pos, 0, (uint32_t)(ampLen - RL + 1)); ci += 1;
        }
        // genome interval [lo, lo + RL) of each mate and its reading direction. Window base i of the amplicon is
        // rc ? comp(G[gstart - i]) : G[gstart + i]; mate 1 reads window bases pos .. pos+RL-1, mate 2 the reverse complement of
        // pos+isz-RL .. pos+isz-1 (Amplicon.cpp:508-512)
        uint64_t lo[2]; uint32_t rev[2];
        if (!F.rc) { lo[0] = F.gstart + (uint64_t)pos; rev[0] = 0; lo[1] = F.gstart + (uint64_t)(pos + isz - RL); rev[1] = 1; }
        else { lo[0] = F.gstart - (uint64_t)(pos + RL - 1); rev[0] = 1; lo[1] = F.gstart - (uint64_t)(pos + isz - 1); rev[1] = 0; }
        const int nm = T.paired ? 2 : 1;
        uint32_t tx = 0; uint64_t b0[2], n0[2]; uint32_t bn[2], nn[2];
#pragma unroll
        for (int m = 0; m < 2; m++) {
            if (m < nm) {
                const uint64_t first = lo[m] >> 2, last = (lo[m] + (uint64_t)RL - 1) >> 2;
                b0[m] = first & ~15ull; bn[m] = (uint32_t)(((last - b0[m]) + 16) & ~15ull);
                woff[m] = (uint32_t)(lo[m] - (b0[m] << 2)) | (rev[m] << 31);
                SCS_CHECK(bn[m] <= (uint32_t)kWinBytes && lo[m] + (uint64_t)RL <= g.n_bases && pos >= 0 && pos + isz <= ampLen);
                tx += bn[m];
                if (g.has_n) {
                    const uint64_t nf = lo[m] >> 3, nl = (lo[m] + (uint64_t)RL - 1) >> 3;
                    n0[m] = nf & ~15ull; nn[m] = (uint32_t)(((nl - n0[m]) + 16) & ~15ull);
                    noff[m] = (uint32_t)(lo[m] - (n0[m] << 3));
                    SCS_CHECK(nn[m] <= (uint32_t)kWinNBytes);
                    tx += nn[m];
                }
            }
        }
        if (lane == 0 && need_bases) {
            mbar_arrive_expect_tx(&st->bar[buf], tx);
            const uint8_t* gw = reinterpret_cast<const uint8_t*>(g.words); const uint8_t* gn = reinterpret_cast<const uint8_t*>(g.nmask);
#pragma unroll
            for (int m = 0; m < 2; m++) {
                if (m < nm) {
                    bulk_g2s(st->win[buf][m], gw + b0[m], bn[m], &st->bar[buf]);
                    if (g.has_n) bulk_g2s(st->winn[buf][m], gn + n0[m], nn[m], &st->bar[buf]);
                }
            }
        }
    }
    if (lane == 0) {
        SlotPlan& P = st->plan[buf];
        P.entity = entity; P.errs = A.err_pool + (er >> 16); P.ampIdx = ampIdx; P.fragNo = fragNo; P.nerr = (uint32_t)(er & 0xFFFF);
        P.cr = cr; P.ci = ci; P.pos = pos; P.isz = isz; P.woff[0] = woff[0]; P.woff[1] = woff[1]; P.noff[0] = noff[0]; P.noff[1] = noff[1];
        P.valid = valid ? 1 : 0;
        P.gap[0] = gap_x[0]; P.gap[1] = gap_x[1]; P.gap_idx[0] = gap_i[0]; P.gap_idx[1] = gap_i[1];
    }
    __syncwarp();
}

// ---- stage B: one slot (SE read / PE pair). Every record goes to its slot's fixed-stride cell of the staging buffer and its size
// ---- is recorded; compact_records_kernel packs them afterwards.
template <bool SIZE_ONLY, bool REPLAY>
__device__ __forceinline__ uint32_t emit_slot(const Genome& g, const DrawSrc& dsrc, const ReadTables& T, const QualSmem* Q, const SlabArgs& A, uint64_t ls, int lane,
                                              WarpScratch* ws, WarpStage* st, int buf, uint32_t& phases, uint32_t* __restrict__ size1, uint32_t* __restrict__ size2,
                                              char* __restrict__ out1, char* __restrict__ out2, int* flags) {
    const SlotPlan& P = st->plan[buf];
    if (!P.valid) return 0;   // sizes were zeroed before the launch
    const int RL = T.RL;
    const uint32_t ampIdx = P.ampIdx, fragNo = P.fragNo, nerr = P.nerr;
    const uint32_t* __restrict__ errs = P.errs;
    const int pos = P.pos, isz = P.isz;
    uint32_t cr = P.cr, ci = P.ci;
    RStream<REPLAY> S; S.init(dsrc, D_READ, P.entity, P.entity);
    const int da = dec_digits(ampIdx), df = dec_digits(fragNo);
    const int hl = header_len(da, df, T.paired);
    const bool need_bases = !SIZE_ONLY || g.has_n;
    if (need_bases) {
        mbar_wait(&st->bar[buf], (phases >> buf) & 1u);   // the packed windows have landed
        phases ^= 1u << buf;                              // a buffer's barrier advances one phase per valid slot that used it
    }
    uint32_t made = 0;
#pragma unroll 1
    for (int mate = 1; mate <= (T.paired ? 2 : 1); mate++) {
        // ---- decode the staged window: 2-bit codes -> one byte per base, in read direction
        const uint32_t wo = P.woff[mate - 1], off = wo & 0x7FFFFFFFu; const bool rev = (wo >> 31) != 0;
        const uint8_t* __restrict__ win = st->win[buf][mate - 1];
        __syncwarp();
        bool myN = false;
        if (need_bases && !g.has_n) {
            // four bases per lane and step: the (up to) two staged bytes that hold them, one shift, 8 bits spread into 4 bytes, one
            // 32-bit store. Backwards windows take the four bases below their highest offset, reversed and complemented.
            for (int i0 = 4 * lane; i0 < RL; i0 += 128) {
                uint32_t t;
                if (!rev) {
                    const uint32_t q0 = off + (uint32_t)i0, B = q0 >> 2;
                    SCS_CHECK(B < (uint32_t)kWinBytes);
                    const uint32_t v = ((uint32_t)win[B] | ((uint32_t)win[B + 1] << 8)) >> ((q0 & 3u) * 2u);
                    t = ((v & 0xFFu) | ((v & 0xFFu) << 12)) & 0x000F000Fu; t = (t | (t << 6)) & 0x03030303u;
                } else {
                    const uint32_t qh = off + (uint32_t)(RL - 1 - i0), B1 = qh >> 2, B0 = B1 ? B1 - 1 : 0;   // offsets below 0 only feed positions >= RL
                    SCS_CHECK(B1 < (uint32_t)kWinBytes);
                    const uint32_t v = (((uint32_t)win[B0] | ((uint32_t)win[B1] << 8)) >> ((qh & 3u) * 2u + 2u)) & 0xFFu;
                    t = (v | (v << 12)) & 0x000F000Fu; t = (t | (t << 6)) & 0x03030303u;
                    t = __byte_perm(t, 0, 0x0123) ^ 0x03030303u;
                }
                *reinterpret_cast<uint32_t*>(ws->ref + i0) = t;   // may run up to 3 bytes past RL inside ref[kRLCap]: never read
            }
        } else if (need_bases) for (int i = lane; i < RL; i += 32) {
            const uint32_t q = off + (uint32_t)(rev ? (RL - 1 - i) : i);
            SCS_CHECK((q >> 2) < (uint32_t)kWinBytes && i < kRLCap);
            uint32_t b = ((uint32_t)win[q >> 2] >> ((q & 3u) * 2u)) & 3u;
            if (rev) b ^= 3u;
            const uint32_t qn = P.noff[mate - 1] + (uint32_t)(rev ? (RL - 1 - i) : i);
            SCS_CHECK((qn >> 3) < (uint32_t)kWinNBytes);
            if ((st->winn[buf][mate - 1][qn >> 3] >> (qn & 7u)) & 1u) { b = 4u; myN = true; }
            ws->ref[i] = (uint8_t)b;
        }
        __syncwarp();
        // ---- substitution overlay of the amplicon, once per window: an error at window base fi lands at read position
        // ---- fi - pos (mate 1) or pos + isz - 1 - fi, complemented (mate 2). It also overrides an N.
        if (need_bases) for (uint32_t e = lane; e < nerr; e += 32) {
            const uint32_t v = errs[e];
            const int fi = (int)err_pos(v);
            const int i = (mate == 1) ? fi - pos : pos + isz - 1 - fi;
            if (i >= 0 && i < RL) ws->ref[i] = (uint8_t)((mate == 1) ? err_base(v) : 3u - err_base(v));
        }
        const bool hasN = g.has_n && __any_sync(0xffffffffu, myN);   // conservative when an overlay replaced the only N: the N path is exact for any window
        __syncwarp();
        int nev = 0;
        const int np = indel_pass(S, T, RL, cr, ci, lane, ws, &nev, flags, P.gap_idx[mate - 1], P.gap[mate - 1]);
        if (np > kSrcCap) { if (lane == 0) atomicOr(flags, 8); return made; }
        __syncwarp();
        const int total = hl + 2 * np + 4;
        if ((uint64_t)total > A.stage_stride) { if (lane == 0) atomicOr(flags, 16); return made; }
        SCS_CHECK(np >= 50 && np <= kSrcCap && total <= kRecCap && ls < A.nslots);
        if (SIZE_ONLY) {   // only the cursors and the record size: the substitution / quality pass draws twice per base, fewer around an N
            if (hasN) {
                const uint8_t* srcn = build_source(S, np, nev, lane, ws);
                const uint2 cc = subst_quality_pass_n<false>(S, make_pass_tabs(T, nullptr, mate == 1), srcn, np, cr, ci, lane, nullptr, nullptr);
                cr = cc.x; ci = cc.y;
            }
            else cr += 2u * (uint32_t)np;
            if (lane == 0) ((mate == 1) ? size1 : size2)[ls] = (uint32_t)total;
            made++;
            continue;
        }
        const uint8_t* src = build_source(S, np, nev, lane, ws);
        char* rec = ws->rec;
        write_frame(rec, ampIdx, fragNo, da, df, T.paired ? mate : 0, hl, np, lane);
        const PassTabs X = make_pass_tabs(T, Q, mate == 1);
        if (hasN) { const uint2 cc = subst_quality_pass_n<true>(S, X, src, np, cr, ci, lane, rec + hl, rec + hl + np + 3); cr = cc.x; ci = cc.y; }
        else subst_quality_pass(S, X, src, np, cr, lane, rec + hl, rec + hl + np + 3);
        __syncwarp();
        copy_out(((mate == 1) ? out1 : out2) + ls * A.stage_stride, rec, total, lane);
        if (lane == 0) ((mate == 1) ? size1 : size2)[ls] = (uint32_t)total;
        made++;
    }
    return made;
}

// emit: persistent CTAs (one per SM). The diagonal quality tables and the insert-size thresholds are staged in shared memory once
// per CTA; every warp then walks its slots with a two-deep software pipeline: plan_slot (lookups, draws, TMA request for the
// genome windows) for slot k+1, then emit_slot for slot k whose windows have landed meanwhile.
template <bool SIZE_ONLY, bool REPLAY>
__global__ void __launch_bounds__(kEmitWarps * 32, 1) emit_kernel(Genome g, DrawSrc dsrc, ReadTables T, SlabArgs A, char* __restrict__ out1, char* __restrict__ out2,
                                                                  int* flags, uint32_t* __restrict__ size1, uint32_t* __restrict__ size2,
                                                                  unsigned long long* __restrict__ records, int isize_smem) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nwarps = (int)(blockDim.x >> 5);   // <= kEmitWarps: long-read profiles leave room for fewer warp scratch areas
    const int nrows = 4 * T.RL;
    uint32_t* srows = reinterpret_cast<uint32_t*>(smem_raw);
    uint4* spiv = reinterpret_cast<uint4*>(srows + (size_t)nrows * kDiagStride);
    uint32_t* smeta = reinterpret_cast<uint32_t*>(spiv + nrows);
    uint32_t* sisize = smeta + ((nrows + 3) & ~3);
    WarpStage* stages = reinterpret_cast<WarpStage*>(sisize + ((isize_smem + 3) & ~3));
    WarpScratch* scratch = reinterpret_cast<WarpScratch*>(stages + nwarps);
    {
        const uint4* grows = reinterpret_cast<const uint4*>(T.diagRows); uint4* s4 = reinterpret_cast<uint4*>(srows);
        for (int i = threadIdx.x; i < nrows * (kDiagStride / 4); i += blockDim.x) s4[i] = __ldg(grows + i);
        for (int i = threadIdx.x; i < nrows; i += blockDim.x) { spiv[i] = __ldg(T.diagPiv + i); smeta[i] = __ldg(T.diagMeta + i); }
        for (int i = threadIdx.x; i < isize_smem; i += blockDim.x) sisize[i] = __ldg(T.isize + i);
    }
    WarpStage* st = &stages[warp];
    if (lane == 0) { mbar_init(&st->bar[0], 1); mbar_init(&st->bar[1], 1); mbar_fence_init(); }
    __syncthreads();
    QualSmem Q; Q.rows = srows; Q.piv = spiv; Q.meta = smeta;
    const uint32_t* isize_row = isize_smem ? sisize : T.isize;
    const uint64_t stride = (uint64_t)gridDim.x * nwarps;
    // iteration `it` plans slot `it` (lookups, draws, TMA request) and then emits slot `it - 1`, whose windows have landed meanwhile
    const uint64_t first = (uint64_t)blockIdx.x * nwarps + warp;
    uint32_t made = 0, phases = 0;
    for (uint64_t ls = first, it = 0; ls < A.nslots + stride; ls += stride, it++) {
        const int buf = (int)(it & 1u);
        if (ls < A.nslots) plan_slot<SIZE_ONLY, REPLAY>(g, dsrc, T, isize_row, A, ls, lane, st, buf);
        if (it) made += emit_slot<SIZE_ONLY, REPLAY>(g, dsrc, T, &Q, A, ls - stride, lane, &scratch[warp], st, buf ^ 1, phases, size1, size2, out1, out2, flags);
    }
    if (lane == 0 && made) atomicAdd(records, (unsigned long long)made);
}

// per coarse entry j: the amplicon that holds slot base + j * 2^kCoarseShift (slots past the end map to the last amplicon)
__global__ void __launch_bounds__(256) coarse_index_kernel(const uint64_t* __restrict__ slot_base, uint64_t n_amp, uint64_t base, uint64_t n, uint32_t* __restrict__ coarse) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const uint64_t slot = base + (j << kCoarseShift);
    uint64_t lo = 0, hi = n_amp;   // last a with slot_base[a] <= slot
    while (hi - lo > 1) { const uint64_t mid = (lo + hi) >> 1; if (slot_base[mid] <= slot) lo = mid; else hi = mid; }
    coarse[j] = (uint32_t)lo;
}

// pack the staged records of one file: warp per record, 16-byte stores at the destination's alignment, the source realigned by
// the two-load funnel shifter (load16). HBM-bound: reads and writes every FASTQ byte once (~0.05 ms per 64 MiB slab).
// A record that would end past `cap` (the slab) is skipped and flagged: the host reports the overflow, nothing is written outside.
__global__ void __launch_bounds__(256) compact_records_kernel(const char* __restrict__ stage, uint64_t stride, const uint32_t* __restrict__ sizes,
                                                              const uint64_t* __restrict__ offs, uint64_t n, char* __restrict__ out, uint64_t cap,
                                                              int* __restrict__ flags) {
    const int lane = threadIdx.x & 31;
    for (uint64_t ls = (uint64_t)blockIdx.x * 8 + (threadIdx.x >> 5); ls < n; ls += (uint64_t)gridDim.x * 8) {
        const int sz = (int)sizes[ls];
        if (!sz) continue;
        const uint64_t o = offs[ls];
        if (o + (uint64_t)sz > cap) { if (lane == 0) atomicOr(flags, 16); continue; }
        SCS_CHECK((uint64_t)sz <= stride);
        const uint8_t* src = reinterpret_cast<const uint8_t*>(stage) + ls * stride;
        char* dst = out + o;
        const int head = min(sz, (int)((16 - (reinterpret_cast<uintptr_t>(dst) & 15)) & 15));
        if (lane < head) dst[lane] = (char)src[lane];
        const int nvec = (sz - head) >> 4;
        for (int k = lane; k < nvec; k += 32) {
            uint32_t X[4]; load16(src + head + 16 * k, X);
            uint4 v; v.x = X[0]; v.y = X[1]; v.z = X[2]; v.w = X[3];
            *reinterpret_cast<uint4*>(dst + head + 16 * k) = v;
        }
        const int done = head + (nvec << 4);
        if (done + lane < sz) dst[done + lane] = (char)src[done + lane];
    }
}

// ---- packed slabs (wire.h). A staged record packs unless it holds a base outside ACGT or a quality outside [qlo, qlo + 63];
// ---- the warp reads it once to decide, and returns its header length.
__device__ __forceinline__ bool record_packs(const uint8_t* __restrict__ src, int sz, uint32_t qlo, int lane, int* hl_out) {
    const uint32_t nl = __ballot_sync(0xffffffffu, lane < sz && src[lane] == '\n');
    const int hl = nl ? __ffs(nl) : 0;
    *hl_out = hl;
    const int np = (sz - hl - 4) / 2;
    if (!hl || hl >= wire::kVerbatim || np < 0 || hl + 2 * np + 4 != sz) return false;
    bool ok = true;
    for (int k = lane; k < np; k += 32) {
        const uint8_t b = src[hl + k];
        const uint32_t q = (uint32_t)src[hl + np + 3 + k] - 33u - qlo;
        ok &= (b == 'A' || b == 'C' || b == 'G' || b == 'T') && q < (uint32_t)wire::kQualSpan;
    }
    return __all_sync(0xffffffffu, ok);
}

__global__ void __launch_bounds__(256) wire_size_kernel(const char* __restrict__ stage, uint64_t stride, const uint32_t* __restrict__ sizes, uint64_t n,
                                                        uint32_t qlo, uint32_t* __restrict__ wsizes) {
    const int lane = threadIdx.x & 31;
    for (uint64_t ls = (uint64_t)blockIdx.x * 8 + (threadIdx.x >> 5); ls < n; ls += (uint64_t)gridDim.x * 8) {
        const int sz = (int)sizes[ls];
        uint32_t w = 0;
        if (sz) {
            int hl;
            const bool pk = record_packs(reinterpret_cast<const uint8_t*>(stage) + ls * stride, sz, qlo, lane, &hl);
            w = pk ? wire::packed_bytes(hl, (sz - hl - 4) / 2) : 3u + (uint32_t)sz;
        }
        if (lane == 0) wsizes[ls] = w;
    }
}

// the packed slab of one file: the split table (one {wire, text} offset pair per kSplitEvery slots) at `out`, the records after it
__global__ void __launch_bounds__(256) pack_records_kernel(const char* __restrict__ stage, uint64_t stride, const uint32_t* __restrict__ sizes,
                                                           const uint64_t* __restrict__ toffs, const uint64_t* __restrict__ woffs, uint64_t n, uint32_t qlo,
                                                           char* __restrict__ out, uint64_t cap, int* __restrict__ flags) {
    const int lane = threadIdx.x & 31;
    const uint64_t nsplit = (n + wire::kSplitEvery - 1) / wire::kSplitEvery;
    wire::Split* split = reinterpret_cast<wire::Split*>(out);
    uint8_t* rec0 = reinterpret_cast<uint8_t*>(out) + nsplit * sizeof(wire::Split);
    for (uint64_t ls = (uint64_t)blockIdx.x * 8 + (threadIdx.x >> 5); ls < n; ls += (uint64_t)gridDim.x * 8) {
        if (lane == 0 && ls % wire::kSplitEvery == 0) split[ls / wire::kSplitEvery] = wire::Split{woffs[ls], toffs[ls]};
        const int sz = (int)sizes[ls];
        if (!sz) continue;
        const uint8_t* src = reinterpret_cast<const uint8_t*>(stage) + ls * stride;
        int hl;
        const bool pk = record_packs(src, sz, qlo, lane, &hl);
        const int np = (sz - hl - 4) / 2;
        const uint32_t wsz = pk ? wire::packed_bytes(hl, np) : 3u + (uint32_t)sz;
        const uint64_t o = woffs[ls];
        if (nsplit * sizeof(wire::Split) + o + wsz > cap) { if (lane == 0) atomicOr(flags, 16); continue; }
        uint8_t* dst = rec0 + o;
        const uint32_t len = pk ? (uint32_t)np : (uint32_t)sz;
        if (lane == 0) { dst[0] = pk ? (uint8_t)hl : (uint8_t)wire::kVerbatim; dst[1] = (uint8_t)(len & 255u); dst[2] = (uint8_t)(len >> 8); }
        if (!pk) { for (int k = lane; k < sz; k += 32) dst[3 + k] = src[k]; continue; }
        for (int k = lane; k < hl; k += 32) dst[3 + k] = src[k];
        for (int k = lane; k < np; k += 32) {
            const uint8_t b = src[hl + k];
            const uint32_t code = b == 'A' ? 0u : b == 'C' ? 1u : b == 'G' ? 2u : 3u;
            dst[3 + hl + k] = (uint8_t)(code | (((uint32_t)src[hl + np + 3 + k] - 33u - qlo) << 2));
        }
    }
}

// ---- slow path (insert sizes that can exceed an amplicon, -s large): failed attempts per slot -----
__global__ void __launch_bounds__(256) fail_count_kernel(DrawSrc dsrc, ReadTables T, SlabArgs A, uint32_t* __restrict__ nfail) {
    uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= A.nslots) return;
    const uint64_t slot = A.fail_base + k;
    uint64_t lo = 0, hi = A.n_amp;
    while (hi - lo > 1) { uint64_t mid = (lo + hi) >> 1; if (A.slot_base[mid] <= slot) lo = mid; else hi = mid; }
    const int ampLen = (int)unpack_desc(A.desc[lo]).len;
    const uint64_t entity = A.slot_gbase[lo] + (slot - A.slot_base[lo]);
    Stream S; S.init(dsrc, D_READ, entity, entity);
    uint32_t f = 0;
    for (; f <= 1001u; f++) {
        int isz = T.minInsert + count_le(T.isize, T.isizeEff, S.at(E_REAL, f));
        if (!(isz < T.RL || isz > ampLen)) break;
    }
    nfail[k] = f;
}
// per amplicon: fragCount numbering and the ">1000 failures -> give up" rule (Amplicon.cpp:448-490)
__global__ void __launch_bounds__(256) fail_scan_kernel(SlabArgs A, const uint32_t* __restrict__ nfail, uint32_t* __restrict__ hdr_no) {
    // amplicons [A.slot0, A.slot0 + n): A.slot0 is reused as the first amplicon index here
    uint64_t a = A.slot0 + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= A.slot0 + A.nslots) return;
    uint64_t s0 = A.slot_base[a], s1 = A.slot_base[a + 1];
    uint32_t cum = 0; bool dead = false;
    for (uint64_t s = s0; s < s1; s++) {
        if (!dead) { cum += nfail[s - A.fail_base]; if (cum > 1000u) dead = true; }
        hdr_no[s - A.fail_base] = dead ? 0u : (uint32_t)(s - s0) + 1u + cum;
    }
}

// ---------------------------------------------------------------------------------- profile upload
int upload_profile(scs_ctx* c) {
    if (!c->have_device) return SCS_OK;
    const HostProfile& P = c->prof; DevProfile& D = c->dprof;
    auto up32 = [&](DevBuf<uint32_t>& b, const std::vector<uint32_t>& v) -> cudaError_t {
        cudaError_t e = b.reserve(v.size() + 4); if (e != cudaSuccess) return e;
        return v.empty() ? cudaSuccess : memcpy_sync(c, b.p, v.data(), v.size() * 4, cudaMemcpyHostToDevice);
    };
    SCS_CUDA(c, up32(D.subs1, P.subsThr1));
    if (P.hasSubs2) SCS_CUDA(c, up32(D.subs2, P.subsThr2));
    SCS_CUDA(c, up32(D.qual, P.qualThr));
    SCS_CUDA(c, D.qualEff.reserve(P.qualEff.size() + 4));
    SCS_CUDA(c, memcpy_sync(c, D.qualEff.p, P.qualEff.data(), P.qualEff.size(), cudaMemcpyHostToDevice));
    SCS_CUDA(c, up32(D.ins, P.insThr.thr)); SCS_CUDA(c, up32(D.del, P.delThr.thr));
    if (P.hasISize) SCS_CUDA(c, up32(D.isize, P.iSizeThr.thr));
    // compact diagonal quality rows: entries [lo, eff) of pair (b,b), padded to 32 with 0xFFFFFFFF; rows that do not fit stay global
    const int bins = P.bins, nrows = 4 * bins;
    std::vector<uint32_t> rows((size_t)nrows * kDiagStride, 0xFFFFFFFFu), piv((size_t)nrows * 4, 0xFFFFFFFFu), meta(nrows, 0);
    for (int b = 0; b < 4; b++) for (int j = 0; j < bins; j++) {
        const size_t r = (size_t)(b * 5) * bins + j;   // pair index b*4+b
        const int lo = P.qualLo[r], eff = P.qualEff[r], cnt = eff - lo;
        const int o = b * bins + j;
        if (cnt > kDiagW || lo > 255) { meta[o] = 1u << 16; continue; }
        for (int k = 0; k < cnt; k++) rows[(size_t)o * kDiagStride + k] = P.qualThr[r * kQualN + lo + k];
        for (int q = 0; q < 4; q++) piv[(size_t)o * 4 + q] = rows[(size_t)o * kDiagStride + 8 * q + 7];
        meta[o] = (uint32_t)lo | ((uint32_t)cnt << 8);
    }
    SCS_CUDA(c, up32(D.qualDiag, rows)); SCS_CUDA(c, up32(D.qualDiagPiv, piv)); SCS_CUDA(c, up32(D.qualDiagMeta, meta));
    // packed slabs: the lowest quality index any row can produce (a draw counts at least the row's leading zero thresholds)
    c->wire_qlo = P.qualLo.empty() ? 0u : (uint32_t)*std::min_element(P.qualLo.begin(), P.qualLo.end());
    return SCS_OK;
}

static ReadTables make_tables(const scs_ctx* c) {
    const HostProfile& P = c->prof; const DevProfile& D = c->dprof;
    ReadTables T;
    T.subs1 = D.subs1.p; T.subs2 = P.hasSubs2 ? D.subs2.p : nullptr; T.qual = D.qual.p; T.qualEff = D.qualEff.p;
    T.ins = D.ins.p; T.del = D.del.p; T.isize = D.isize.p;
    T.insEff = P.insThr.eff; T.delEff = P.delThr.eff; T.isizeEff = P.hasISize ? P.iSizeThr.eff : 0;
    T.minInsert = P.minInsert; T.maxInsert = P.maxInsert;
    T.thrIns = P.thrInsertAll ? (1ull << 32) : P.thrInsert; T.thrDel = P.thrDeleteAll ? (1ull << 32) : P.thrDelete;
    T.RL = P.readLength; T.paired = c->P.paired;
    {   // constants of the free-running indel stage: formed exactly as oracle/profile.h indel_geom() forms them
        const double pI = (double)T.thrIns / 4294967296.0, pD = (double)T.thrDel / 4294967296.0;
        const double q = (1.0 - pI) * (1.0 - pD);
        T.indelAny = q < 1.0;
        T.indelLogQ = det_log(q);
        T.thrInsType = T.thrDel == 0 ? (1ull << 32) : T.thrIns == 0 ? 0 : count_unit_lt(pI / (1.0 - q));
        const double none = (q > 0.0 && q < 1.0) ? floor(0.99 * exp((double)T.RL * T.indelLogQ) * 4294967296.0) : 0.0;
        T.thrNoEvent = (uint32_t)std::min(none, 4294967295.0);
    }
    T.diagRows = D.qualDiag.p; T.diagPiv = reinterpret_cast<const uint4*>(D.qualDiagPiv.p); T.diagMeta = D.qualDiagMeta.p;
    return T;
}

// ---------------------------------------------------------------------------------- slab pipeline
namespace {

// events of one run of the stage; every exit path (errors included) first drains both streams and the expansion pool, so
// nothing that was queued can still touch the context's buffers or these events when the caller retries
struct StageGuard {
    scs_ctx* c; std::vector<cudaEvent_t> evs;
    explicit StageGuard(scs_ctx* ctx) : c(ctx) {}
    cudaEvent_t make(unsigned flags) { cudaEvent_t e = nullptr; cudaEventCreateWithFlags(&e, flags); evs.push_back(e); return e; }
    ~StageGuard() {
        cudaStreamSynchronize(c->st); cudaStreamSynchronize(c->st_copy);
        if (c->st_relay) cudaStreamSynchronize(c->st_relay);
        if (c->pool) c->pool->drain();
        for (cudaEvent_t e : evs) if (e) cudaEventDestroy(e);
    }
};

}  // namespace

// scs_sink_fn adapter: kSlots ring slots, the user's function runs on the launching thread in slab order
CallbackConsumer::CallbackConsumer(scs_sink_fn f, void* u) : fn(f), user(u) {}
int CallbackConsumer::consume_front(bool wait) {
    if (count == 0) return 0;
    Pending& q = pend[head];
    if (q.job) {   // text written by the expansion pool
        if (wait) { if (q.pool->wait(q.job)) return 1; }
        else if (!q.pool->query(q.job)) return -1;
        else if (q.pool->wait(q.job)) return 1;
    }
    else if (wait) { if (cudaEventSynchronize(q.ev) != cudaSuccess) return 1; }
    else if (cudaEventQuery(q.ev) != cudaSuccess) { (void)cudaGetLastError(); return -1; }   // not landed yet
    int rc = 0;
    if (fn) for (int f = 0; f < 2 && !rc; f++) if (q.n[f]) rc = fn(user, f, q.p[f], q.n[f]) ? 1 : 0;
    q.live = false; head = (head + 1) % kSlots; count--;
    return rc;
}
int CallbackConsumer::acquire(int slot) {
    while (pend[slot].live) { int rc = consume_front(true); if (rc) return rc; }
    return 0;
}
int CallbackConsumer::submit(int slot, cudaEvent_t copied, char* const p[2], const uint64_t bytes[2]) {
    Pending& q = pend[slot];
    q.live = true; q.ev = copied; q.pool = nullptr; q.job = nullptr; q.p[0] = p[0]; q.p[1] = p[1]; q.n[0] = bytes[0]; q.n[1] = bytes[1];
    if (count == 0) head = slot;
    count++;
    return 0;
}
int CallbackConsumer::submit_expanded(int slot, ExpandPool* pool, ExpandJob* job, char* const p[2], const uint64_t bytes[2]) {
    if (submit(slot, nullptr, p, bytes)) return 1;
    pend[slot].pool = pool; pend[slot].job = job;
    return 0;
}
int CallbackConsumer::service() {
    for (;;) { int rc = consume_front(false); if (rc < 0 || count == 0) return 0; if (rc) return rc; }
}
int CallbackConsumer::finish() {
    while (count) { int rc = consume_front(true); if (rc) return rc; }
    return 0;
}

// sum of the record sizes of one batch, per file
__global__ void __launch_bounds__(256) sum_sizes_kernel(const uint32_t* __restrict__ size1, const uint32_t* __restrict__ size2, uint64_t n,
                                                        unsigned long long* __restrict__ totals) {
    unsigned long long a = 0, b = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) { a += size1[i]; if (size2) b += size2[i]; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { a += __shfl_down_sync(0xffffffffu, a, o); b += __shfl_down_sync(0xffffffffu, b, o); }
    if ((threadIdx.x & 31) == 0) { if (a) atomicAdd(totals, a); if (b) atomicAdd(totals + 1, b); }
}

namespace {
// everything the slab loop needs: tables, the slot range, launch geometry, scratch, the coarse index and the slow-path numbering
struct ReadRun {
    ReadTables T; Genome g; DrawSrc dsrc; SlabArgs A;
    uint64_t slot_lo = 0, slot_hi = 0, nslots = 0, slab = 0, stride = 0, batch = 0;
    int nfiles = 1, sms = 148, emit_warps = kEmitWarps, isize_smem = 0; size_t emit_smem = 0;
};
}  // namespace

static int prepare_read_run(scs_ctx* c, ReadRun& R) {
    if (!c->have_profile) return c->fail(SCS_E_STATE, "scs_yield_reads: no profile loaded");
    if (!c->have_counts) { if (int rc = set_read_counts(c)) return rc; }
    const HostProfile& P = c->prof;
    if (P.readLength > kRLCap) return c->fail(SCS_E_UNSUPPORTED, "read length above 320 is not supported by the kernels");
    if (c->P.paired && !P.hasISize) return c->fail(SCS_E_ARG, "Error: unrecognized parameter name \"insertSize\"");   // Profile.cpp:1484 -> Config.cpp:71-78
    // what this rank reads from: its own amplicons and genome, or (balance = 1) the cell-wide copies and a slot range
    const bool gv = c->global_view;
    R.slot_lo = gv ? c->g_slot_lo : 0; R.slot_hi = gv ? c->g_slot_hi : c->n_slots; R.nslots = R.slot_hi - R.slot_lo;
    R.nfiles = c->P.paired ? 2 : 1;
    R.slab = c->P.slab_bytes ? c->P.slab_bytes : (64ull << 20);
    R.stride = ((uint64_t)kRecCap + 15) & ~15ull;
    if (R.slab < 64 * R.stride) return c->fail(SCS_E_ARG, "slab_bytes is too small (needs room for 64 records of the largest size, 64 KiB)");
    if (R.nslots == 0) return SCS_OK;
    // slots per slab: typical record = header (<= 30) + 2*(RL + a few inserted bases) + 4. A batch whose records are longer than
    // that on average (heavy insertion profiles) can exceed the slab: the compaction kernel then skips the records that do not
    // fit, and the run ends with SCS_E_NOMEM ("raise slab_bytes") — nothing is ever written outside the slab.
    const uint64_t typical = 30 + 2ull * (P.readLength + 8) + 4;
    R.batch = std::min<uint64_t>(std::max<uint64_t>(64, R.slab / typical), 2048ull * 2048ull);
    R.T = make_tables(c); R.g = c->dev_genome(); R.dsrc = draw_src(c, D_READ);
    SlabArgs& A = R.A;
    A.slot_gbase = c->slot_gbase.p; A.amp_gidx = c->full_gidx.p; A.n_amp = c->fulls.n; A.slot_base = c->slot_base.p;
    A.desc = c->fulls.desc.p; A.errref = c->fulls.errref.p; A.err_pool = c->err_pool.p; A.hdr_no = nullptr; A.nfail = nullptr; A.slab_cap = R.slab;
    A.fail_base = 0; A.stage_stride = R.stride; A.slot0 = 0; A.nslots = 0;
    if (gv) {
        R.g.words = c->g_words.p; R.g.nmask = c->g_nmask.p; R.g.n_bases = c->g_bases; R.g.has_n = c->g_has_n;
        A.slot_gbase = c->g_slot_base.p; A.amp_gidx = nullptr; A.n_amp = c->g_n_amp; A.slot_base = c->g_slot_base.p;
        A.desc = c->g_desc.p; A.errref = c->g_errref.p; A.err_pool = c->g_errs.p;
    }
    ReadScratch& W = c->rscratch;
    SCS_CUDA(c, W.flags.reserve(1)); SCS_CUDA(c, W.records.reserve(1)); SCS_CUDA(c, W.totals.reserve(4));
    SCS_CUDA(c, W.size1.reserve(R.batch + 1)); SCS_CUDA(c, W.size2.reserve(R.batch + 1));
    SCS_CUDA(c, W.off1.reserve(R.batch + 1)); SCS_CUDA(c, W.off2.reserve(R.batch + 1)); SCS_CUDA(c, W.scan.reserve(2 * 2048 + 16));
    for (int f = 0; f < 2; f++) { SCS_CUDA(c, W.wsize[f].reserve(R.batch + 1)); SCS_CUDA(c, W.woff[f].reserve(R.batch + 1)); }
    // slab byte totals are written by the scan kernel straight into mapped pinned memory: a D2H memcpy on the compute
    // stream would queue behind the previous slab's 0.5 GB copy on the same copy engine and stall the emit kernel
    if (!W.htotals) {
        SCS_CUDA(c, cudaHostAlloc((void**)&W.htotals, 128, cudaHostAllocMapped));
        SCS_CUDA(c, cudaHostGetDevicePointer((void**)&W.dtotals_mapped, W.htotals, 0));
    }
    int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&R.sms, cudaDevAttrMultiProcessorCount, dev);
    // shared memory of a persistent emit CTA: the diagonal quality tables, the insert-size thresholds, and per warp a scratch area
    // plus the TMA staging of its next two slots; as many warps (<= 24) as fit
    const size_t table_smem = (size_t)4 * R.T.RL * kDiagStride * 4 + (size_t)4 * R.T.RL * 16 + (size_t)((4 * R.T.RL + 3) & ~3) * 4;
    int smem_max = 0; cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    R.isize_smem = (c->P.paired && R.T.isizeEff <= kISizeSmemCap) ? R.T.isizeEff : 0;
    const size_t per_warp = sizeof(WarpScratch) + sizeof(WarpStage);
    const size_t fixed_smem = table_smem + (size_t)((R.isize_smem + 3) & ~3) * 4;
    // the diagonal quality tables grow with the read length: beyond ~190 bases fewer than 24 warps fit beside them, beyond ~275 none
    R.emit_warps = (int)std::min<size_t>(kEmitWarps, ((size_t)smem_max - std::min<size_t>(fixed_smem, (size_t)smem_max)) / per_warp);
    if (R.emit_warps < 4) return c->fail(SCS_E_UNSUPPORTED, "read length too large: the quality tables of the profile do not fit the shared memory of the read kernel");
    R.emit_smem = fixed_smem + per_warp * (size_t)R.emit_warps;
    SCS_CUDA(c, cudaFuncSetAttribute(emit_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)R.emit_smem));
    SCS_CUDA(c, cudaFuncSetAttribute(emit_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)R.emit_smem));
    SCS_CUDA(c, cudaFuncSetAttribute(emit_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)R.emit_smem));
    // coarse slot -> amplicon index of this rank's slot range (one entry per 1024 slots): the per-slot search starts from it
    const uint64_t n_coarse = ((R.nslots - 1) >> kCoarseShift) + 2;
    SCS_CUDA(c, W.coarse.reserve(n_coarse + 1));
    coarse_index_kernel<<<(unsigned)((n_coarse + 255) / 256), 256, 0, c->st>>>(A.slot_base, A.n_amp, R.slot_lo, n_coarse, W.coarse.p); SCS_LAUNCHED(c);
    A.coarse = W.coarse.p; A.coarse_base = R.slot_lo;
    // slow path: insert sizes that can fail (isize > amplicon length; amplicons are 1000..2000 long)
    if (c->P.paired && P.maxInsert > 1000) {
        // the numbering of an amplicon's pairs depends on all of its earlier pairs: cover whole amplicons around the range
        uint64_t a_first = 0, a_last = A.n_amp - 1, ext_lo = R.slot_lo, ext_hi = R.slot_hi;
        if (gv) {
            std::vector<uint64_t> hb(A.n_amp + 1);
            SCS_CUDA(c, memcpy_sync(c, hb.data(), A.slot_base, (A.n_amp + 1) * 8, cudaMemcpyDeviceToHost));
            a_first = (uint64_t)(std::upper_bound(hb.begin(), hb.end(), R.slot_lo) - hb.begin()) - 1;
            a_last = (uint64_t)(std::upper_bound(hb.begin(), hb.end(), R.slot_hi - 1) - hb.begin()) - 1;
            ext_lo = hb[a_first]; ext_hi = hb[a_last + 1];
        }
        const uint64_t ext_n = ext_hi - ext_lo;
        SCS_CUDA(c, W.nfail.reserve(ext_n + 1)); SCS_CUDA(c, W.hdrno.reserve(ext_n + 1));
        SlabArgs F = A; F.fail_base = ext_lo; F.nslots = ext_n;
        fail_count_kernel<<<(unsigned)((ext_n + 255) / 256), 256, 0, c->st>>>(R.dsrc, R.T, F, W.nfail.p); SCS_LAUNCHED(c);
        F.slot0 = a_first; F.nslots = a_last - a_first + 1;
        fail_scan_kernel<<<(unsigned)((F.nslots + 255) / 256), 256, 0, c->st>>>(F, W.nfail.p, W.hdrno.p); SCS_LAUNCHED(c);
        A.hdr_no = W.hdrno.p; A.nfail = W.nfail.p; A.fail_base = ext_lo;
    }
    return SCS_OK;
}

// Exact FASTQ bytes this rank will write to each file: the sizing pass (indel draws only; bases are fetched only when the genome
// holds N, because an N changes how many draws a base consumes). Used to give every rank its final offset in ONE output file.
int plan_fastq_bytes(scs_ctx* c, uint64_t bytes[2]) {
    bytes[0] = bytes[1] = 0;
    if (c->replay.on) return c->fail(SCS_E_UNSUPPORTED, "the sizing pass is not available in replay mode (replay runs on one rank)");
    ReadRun R;
    if (int rc = prepare_read_run(c, R)) return rc;
    if (R.nslots == 0) return SCS_OK;
    ReadScratch& W = c->rscratch;
    StageGuard G(c);
    SCS_CUDA(c, cudaMemsetAsync(W.flags.p, 0, 4, c->st)); SCS_CUDA(c, cudaMemsetAsync(W.totals.p, 0, 16, c->st));
    for (uint64_t s0 = R.slot_lo; s0 < R.slot_hi; s0 += R.batch) {
        const uint64_t m = std::min(R.batch, R.slot_hi - s0);
        R.A.slot0 = s0; R.A.nslots = m;
        SCS_CUDA(c, cudaMemsetAsync(W.size1.p, 0, (m + 1) * 4, c->st));
        if (R.nfiles == 2) SCS_CUDA(c, cudaMemsetAsync(W.size2.p, 0, (m + 1) * 4, c->st));
        emit_kernel<true, false><<<R.sms, R.emit_warps * 32, R.emit_smem, c->st>>>(R.g, R.dsrc, R.T, R.A, nullptr, nullptr, W.flags.p, W.size1.p, W.size2.p, W.records.p, R.isize_smem);
        SCS_LAUNCHED(c);
        sum_sizes_kernel<<<R.sms, 256, 0, c->st>>>(W.size1.p, R.nfiles == 2 ? W.size2.p : nullptr, m, reinterpret_cast<unsigned long long*>(W.totals.p)); SCS_LAUNCHED(c);
    }
    uint64_t h[2] = {0, 0}; int hflags = 0;
    SCS_CUDA(c, memcpy_sync(c, h, W.totals.p, 16, cudaMemcpyDeviceToHost));
    SCS_CUDA(c, memcpy_sync(c, &hflags, W.flags.p, 4, cudaMemcpyDeviceToHost));
    if (hflags & 4) return c->fail(SCS_E_UNSUPPORTED, "more than 64 indel events in one read");
    if (hflags & 8) return c->fail(SCS_E_UNSUPPORTED, "read grew beyond 480 bases through insertions");
    bytes[0] = h[0]; bytes[1] = h[1];
    return SCS_OK;
}

int yield_reads(scs_ctx* c, SlabConsumer& sink) {
    ReadRun R;
    if (int rc = prepare_read_run(c, R)) return rc;
    c->stats.records = 0; c->stats.fastq_bytes[0] = c->stats.fastq_bytes[1] = 0; c->stats.plain_bytes[0] = c->stats.plain_bytes[1] = 0;
    c->stats.ms_reads = c->stats.ms_reads_kernels = c->stats.ms_emit_kernel = 0; c->stats.emit_launches = 0; c->stats.genome_window_bytes = 0;
    c->stats.link_bytes[0] = c->stats.link_bytes[1] = 0; c->stats.slabs_packed = c->stats.slabs = 0;
    const bool gz = c->P.gzip != 0;
    if (R.nslots == 0 && !gz) return sink.finish() ? c->fail(SCS_E_IO, "FASTQ sink failed") : SCS_OK;
    if (gz) { if (int rc = gz_prepare(c)) return rc; }
    const int nfiles = R.nfiles, sms = R.sms, emit_warps = R.emit_warps, isize_smem = R.isize_smem;
    const uint64_t slab = R.slab, stride = R.stride, batch = R.batch, slot_lo = R.slot_lo, slot_hi = R.slot_hi;
    const size_t emit_smem = R.emit_smem;
    ReadTables& T = R.T; Genome& g = R.g; DrawSrc& dsrc = R.dsrc; SlabArgs& A = R.A;
    ReadScratch& W = c->rscratch;
    const int Rn = std::max(2, sink.ring_slots());
    // device slabs (double buffered) + ring of pinned host slots; both keep their capacity between calls
    if (c->slab_cap != slab) {
        for (int b = 0; b < 2; b++) for (int f = 0; f < 2; f++) c->slab_dev[b][f].release();
        for (int f = 0; f < 2; f++) { for (char* q : c->ring_host[f]) cudaFreeHost(q); c->ring_host[f].clear(); }
        c->slab_cap = slab;
    }
    for (int b = 0; b < 2; b++) for (int f = 0; f < nfiles; f++) if (!c->slab_dev[b][f].p) SCS_CUDA(c, c->slab_dev[b][f].reserve(slab + 64));
    for (int f = 0; f < nfiles; f++) while ((int)c->ring_host[f].size() < Rn) {
        char* q = nullptr;
        SCS_CUDA(c, cudaMallocHost((void**)&q, slab + 4096 + 64));   // + one block: file sinks place the slab at its file offset mod 4096
        c->ring_host[f].push_back(q);
    }
    for (int f = 0; f < nfiles; f++) SCS_CUDA(c, W.stage[f].reserve(batch * stride + 64));
    // NVLink relay: the packed slab goes to a buffer on a peer GPU and from there over THAT GPU's host link into the pinned ring
    const int dev_self = c->P.device, relay = (c->P.relay_device >= 0 && c->P.relay_device != c->P.device) ? c->P.relay_device : -1;
    if (relay >= 0) {
        if (!c->st_relay || c->relay_dev != relay) {
            if (c->st_relay) return c->fail(SCS_E_STATE, "relay_device cannot change during the life of a context");
            int can = 0; SCS_CUDA(c, cudaDeviceCanAccessPeer(&can, dev_self, relay));
            if (!can) return c->fail(SCS_E_UNSUPPORTED, "relay_device: no peer access between the two GPUs");
            cudaError_t e = cudaDeviceEnablePeerAccess(relay, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) SCS_CUDA(c, e);
            (void)cudaGetLastError();
            SCS_CUDA(c, cudaSetDevice(relay));
            e = cudaStreamCreateWithFlags(&c->st_relay, cudaStreamNonBlocking);
            cudaSetDevice(dev_self);
            SCS_CUDA(c, e);
            c->relay_dev = relay;
        }
        if (c->relay_cap != slab) {
            cudaSetDevice(relay);
            cudaError_t e = cudaSuccess;
            for (int b = 0; b < 2; b++) for (int f = 0; f < 2; f++) { if (c->relay_buf[b][f]) { cudaFree(c->relay_buf[b][f]); c->relay_buf[b][f] = nullptr; } }
            for (int b = 0; b < 2 && e == cudaSuccess; b++) for (int f = 0; f < nfiles && e == cudaSuccess; f++) e = cudaMalloc((void**)&c->relay_buf[b][f], slab + 64);
            cudaSetDevice(dev_self);
            SCS_CUDA(c, e);
            c->relay_cap = slab;
        }
    }
    // block-gzip output: members of one slab at a fixed stride, their sizes / offsets, and the packed compressed slabs
    const uint32_t gz_pieces = gz ? (uint32_t)gz_max_pieces(slab) : 0;
    if (gz) for (int f = 0; f < nfiles; f++) {
        SCS_CUDA(c, c->gz.stage[f].reserve((uint64_t)gz_pieces * gz_stage_stride() + 64)); SCS_CUDA(c, c->gz.sizes[f].reserve(gz_pieces + 8));
        SCS_CUDA(c, c->gz.offs[f].reserve(gz_pieces + 8));
        for (int b = 0; b < 2; b++) SCS_CUDA(c, c->gz.slab[b][f].reserve(slab + 64));
    }

    // packed slabs expanded by host threads (wire.h, scs_params.host_expand): the device slabs also hold the split table and the
    // 3-byte prefix of every record, the packed slabs land in a ring of pinned wire slots and the pool expands them into the
    // consumer's slots
    const int hx = c->P.host_expand;
    const bool hybrid = !gz && relay < 0 && R.nslots > 0 && sink.takes_expanded() && (hx == 1 || hx == 2 || (hx < 0 && c->P.world == 1));
    const int Rw = 3;
    const uint64_t split_max = (batch / wire::kSplitEvery + 2) * sizeof(wire::Split), wcap = slab + 3 * batch + split_max + 64;
    if (hybrid) {
        for (int b = 0; b < 2; b++) for (int f = 0; f < nfiles; f++) SCS_CUDA(c, c->slab_dev[b][f].reserve(wcap));
        if (c->wire_cap < wcap) {
            for (int f = 0; f < 2; f++) { for (char* q : c->wire_host[f]) cudaFreeHost(q); c->wire_host[f].clear(); }
            c->wire_cap = wcap;
        }
        for (int f = 0; f < nfiles; f++) while ((int)c->wire_host[f].size() < Rw) {
            char* q = nullptr;
            SCS_CUDA(c, cudaMallocHost((void**)&q, c->wire_cap));
            c->wire_host[f].push_back(q);
        }
        if (!c->pool) {
            int n = c->P.expand_threads;
            if (n <= 0) {
                cpu_set_t set; CPU_ZERO(&set);
                n = sched_getaffinity(0, sizeof(set), &set) == 0 ? CPU_COUNT(&set) - 1 : 1;
            }
            c->pool = new ExpandPool(c->P.device, std::max(1, n));
        }
    }
    // per consumer slot: the expansion job that writes its text (declared before the guard, which drains the pool first)
    std::vector<ExpandJob> jobs(Rn);

    StageGuard G(c);   // from here on every return drains the streams and frees the events
    if (R.nslots == 0) {   // gzip of an empty output: the 28-byte end-of-file member, so that the file is a valid (empty) gzip stream
        static const uint8_t eof[28] = {31, 139, 8, 4, 0, 0, 0, 0, 0, 255, 6, 0, 66, 67, 2, 0, 27, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
        cudaEvent_t landed = G.make(cudaEventDisableTiming);
        if (sink.acquire(0)) return c->fail(SCS_E_IO, "FASTQ sink failed");
        char* p[2] = {nullptr, nullptr}; uint64_t tot[2] = {0, 0};
        for (int f = 0; f < nfiles; f++) { p[f] = c->ring_host[f][0] + (sink.phase(f) & 4095); memcpy(p[f], eof, 28); tot[f] = 28; c->stats.fastq_bytes[f] = 28; }
        SCS_CUDA(c, cudaEventRecord(landed, c->st_copy));
        if (sink.submit(0, landed, p, tot) || sink.finish()) return c->fail(SCS_E_IO, "FASTQ sink failed");
        return SCS_OK;
    }
    SCS_CUDA(c, cudaMemsetAsync(W.flags.p, 0, 4, c->st)); SCS_CUDA(c, cudaMemsetAsync(W.records.p, 0, 8, c->st));
    cudaEvent_t e0 = G.make(cudaEventDefault), e1 = G.make(cudaEventDefault);
    cudaEvent_t ecopy[2], ekern[2], etotb[2], ep2p[2], tq[2][4]; bool timed[2] = {false, false};
    for (int b = 0; b < 2; b++) {
        ekern[b] = G.make(cudaEventDisableTiming); etotb[b] = G.make(cudaEventDisableTiming); ep2p[b] = G.make(cudaEventDisableTiming);
        for (int q = 0; q < 4; q++) tq[b][q] = G.make(cudaEventDefault);
    }
    // the events recorded on the stream that performs the D2H copy belong to that stream's device
    if (relay >= 0) cudaSetDevice(relay);
    for (int b = 0; b < 2; b++) ecopy[b] = G.make(cudaEventDisableTiming);
    std::vector<cudaEvent_t> eslot(Rn); for (int i = 0; i < Rn; i++) eslot[i] = G.make(cudaEventDisableTiming);
    if (relay >= 0) cudaSetDevice(dev_self);
    cudaEvent_t tc[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};   // around the copies of buffer b: the link rate
    if (hybrid) for (int b = 0; b < 2; b++) { tc[b][0] = G.make(cudaEventDefault); tc[b][1] = G.make(cudaEventDefault); }
    cudaStream_t st_d2h = relay >= 0 ? c->st_relay : c->st_copy;
    double msk = 0, mse = 0;
    auto harvest = [&](int b) {   // kernel times of the slab that used buffer b (its events are complete: a later event was waited for)
        if (!timed[b]) return;
        float x = 0, y = 0;
        if (cudaEventElapsedTime(&x, tq[b][0], tq[b][3]) == cudaSuccess && cudaEventElapsedTime(&y, tq[b][1], tq[b][2]) == cudaSuccess) { msk += x; mse += y; }
        timed[b] = false;
    };
    SCS_CUDA(c, cudaEventRecord(e0, c->st));
    // ---- per slab: emit (staging + sizes) -> scans -> compaction into the packed device slab -> D2H into a pinned ring slot.
    // Software-pipelined on the host: slab k is launched before the host waits for the byte totals of slab k-1, so the kernels
    // run back to back; the consumer is serviced in between.
    struct DevSlab { bool launched = false, packed = false; uint64_t k = 0, m = 0; } dv[2];
    // per-slab choice (host_expand = -1): the path, text over the link or packed + host expansion, whose queue drains sooner with
    // this slab added: (bytes queued on the copy stream + the slab's text) / link rate against (text queued on the pool + the
    // slab's text) / expansion rate. Link rate from the copy events, expansion rate from the pool. The emit kernel keeps both
    // sides busy, so this greedy rule settles where the link and the host threads finish together.
    double link_rate = 50e9, wire_ratio = 0.53, last_text = (double)batch * (nfiles == 2 ? 2.0 : 1.0) * (double)(2 * T.RL + 30);
    uint64_t copy_pend[2] = {0, 0}, wire_k = 0;
    ExpandJob* wjob[3] = {nullptr, nullptr, nullptr}; uint64_t wseq[3] = {0, 0, 0};
    auto harvest_link = [&]() {
        for (int b = 0; b < 2; b++) {
            if (!copy_pend[b]) continue;
            cudaError_t q = cudaEventQuery(tc[b][1]);
            if (q == cudaErrorNotReady) { (void)cudaGetLastError(); continue; }
            float ms = 0;
            if (q == cudaSuccess && cudaEventElapsedTime(&ms, tc[b][0], tc[b][1]) == cudaSuccess && ms > 0.05f)
                link_rate = 0.75 * link_rate + 0.25 * (double)copy_pend[b] / (ms * 1e-3);
            copy_pend[b] = 0;
        }
    };
    auto choose_packed = [&](uint64_t kk, int b) -> bool {
        if (!hybrid) return false;
        if (hx == 1) return true;
        if (hx == 2) return (kk & 1) != 0;
        harvest_link();
        const int o = b ^ 1;   // the slab launched before this one: its path is chosen, its bytes are not queued yet
        const double T = last_text;
        double qlink = (double)(copy_pend[0] + copy_pend[1]), qpool = (double)c->pool->queued_text();
        if (dv[o].launched) { if (dv[o].packed) { qpool += T; qlink += wire_ratio * T; } else qlink += T; }
        const double P = c->pool->rate() > 0 ? c->pool->rate() : 2e9 * c->pool->threads();
        return (qpool + T) / P < (qlink + T) / link_rate;
    };
    auto finalize = [&](int b) -> int {   // the kernels of device buffer b were launched: wait for the byte totals, queue the copy behind the compaction
        if (!dv[b].launched) return SCS_OK;
        SCS_CUDA(c, cudaEventSynchronize(etotb[b]));
        dv[b].launched = false;
        const uint64_t tot[2] = {W.htotals[2 * b], nfiles == 2 ? W.htotals[2 * b + 1] : 0};   // bytes to copy (compressed with gzip)
        const uint64_t plain[2] = {gz ? W.htotals[4 + 2 * b] : tot[0], gz ? (nfiles == 2 ? W.htotals[4 + 2 * b + 1] : 0) : tot[1]};
        if (plain[0] > slab || plain[1] > slab || tot[0] > slab || tot[1] > slab) return c->fail(SCS_E_NOMEM, "FASTQ slab too small for one batch (raise slab_bytes)");
        const int slot = (int)(dv[b].k % (uint64_t)Rn);
        if (sink.acquire(slot)) return c->fail(SCS_E_IO, "FASTQ sink failed");
        SCS_CUDA(c, cudaStreamWaitEvent(c->st_copy, ekern[b], 0));
        char* p[2] = {nullptr, nullptr};
        for (int f = 0; f < nfiles; f++) p[f] = c->ring_host[f][slot] + (sink.phase(f) & 4095);
        c->stats.slabs++;
        last_text = (double)(tot[0] + tot[1]);
        if (dv[b].packed) {
            // packed slab: split table + records into the next pinned wire slot, then the pool expands it into the consumer's slot
            const uint32_t nsplit = (uint32_t)((dv[b].m + wire::kSplitEvery - 1) / wire::kSplitEvery);
            const uint64_t wtot[2] = {W.htotals[8 + 2 * b], nfiles == 2 ? W.htotals[8 + 2 * b + 1] : 0};
            uint64_t cb[2] = {0, 0};
            for (int f = 0; f < nfiles; f++) {
                cb[f] = tot[f] ? nsplit * sizeof(wire::Split) + wtot[f] : 0;
                if (cb[f] > wcap) return c->fail(SCS_E_NOMEM, "packed FASTQ slab too small for one batch (raise slab_bytes)");
            }
            const int ws = (int)(wire_k++ % Rw);
            if (wjob[ws] && wjob[ws]->seq == wseq[ws] && c->pool->wait(wjob[ws])) return c->fail(SCS_E_STATE, "host expansion of a packed FASTQ slab failed");
            SCS_CUDA(c, cudaEventRecord(tc[b][0], c->st_copy));
            for (int f = 0; f < nfiles; f++)
                if (cb[f]) SCS_CUDA(c, cudaMemcpyAsync(c->wire_host[f][ws], c->slab_dev[b][f].p, cb[f], cudaMemcpyDeviceToHost, c->st_copy));
            SCS_CUDA(c, cudaEventRecord(tc[b][1], c->st_copy)); copy_pend[b] = cb[0] + cb[1];
            SCS_CUDA(c, cudaEventRecord(ecopy[b], c->st_copy)); SCS_CUDA(c, cudaEventRecord(eslot[slot], c->st_copy));
            if (tot[0] + tot[1]) wire_ratio = 0.75 * wire_ratio + 0.25 * (double)(cb[0] + cb[1]) / (double)(tot[0] + tot[1]);
            ExpandJob& J = jobs[slot];
            J.landed = eslot[slot]; J.qchar0 = 33 + (int)c->wire_qlo;
            for (int f = 0; f < 2; f++) {
                const bool on = f < nfiles && tot[f];
                J.wire[f] = on ? reinterpret_cast<const uint8_t*>(c->wire_host[f][ws]) : nullptr; J.nsplit[f] = on ? nsplit : 0;
                J.wire_bytes[f] = on ? wtot[f] : 0; J.text_bytes[f] = on ? tot[f] : 0; J.out[f] = p[f];
            }
            c->pool->submit(&J);
            wjob[ws] = &J; wseq[ws] = J.seq;
            c->stats.fastq_bytes[0] += tot[0]; c->stats.fastq_bytes[1] += tot[1];
            c->stats.plain_bytes[0] += tot[0]; c->stats.plain_bytes[1] += tot[1];
            c->stats.link_bytes[0] += cb[0]; c->stats.link_bytes[1] += cb[1]; c->stats.slabs_packed++;
            if (sink.submit_expanded(slot, c->pool, &J, p, tot)) return c->fail(SCS_E_IO, "FASTQ sink failed");
            return SCS_OK;
        }
        if (hybrid) SCS_CUDA(c, cudaEventRecord(tc[b][0], c->st_copy));
        if (relay < 0) {
            for (int f = 0; f < nfiles; f++)
                if (tot[f]) SCS_CUDA(c, cudaMemcpyAsync(p[f], gz ? c->gz.slab[b][f].p : c->slab_dev[b][f].p, tot[f], cudaMemcpyDeviceToHost, c->st_copy));
        } else {
            // slab -> peer GPU over NVLink (this GPU's copy engine), then peer GPU -> host over the peer's link (the peer's copy engine)
            for (int f = 0; f < nfiles; f++)
                if (tot[f]) SCS_CUDA(c, cudaMemcpyPeerAsync(c->relay_buf[b][f], relay, gz ? c->gz.slab[b][f].p : c->slab_dev[b][f].p, dev_self, tot[f], c->st_copy));
            SCS_CUDA(c, cudaEventRecord(ep2p[b], c->st_copy));
            SCS_CUDA(c, cudaSetDevice(relay));
            cudaError_t e = cudaStreamWaitEvent(st_d2h, ep2p[b], 0);
            for (int f = 0; f < nfiles && e == cudaSuccess; f++) if (tot[f]) e = cudaMemcpyAsync(p[f], c->relay_buf[b][f], tot[f], cudaMemcpyDeviceToHost, st_d2h);
            if (e != cudaSuccess) { cudaSetDevice(dev_self); SCS_CUDA(c, e); }
        }
        cudaError_t er = cudaEventRecord(ecopy[b], st_d2h);
        if (er == cudaSuccess) er = cudaEventRecord(eslot[slot], st_d2h);
        if (er == cudaSuccess && hybrid) { er = cudaEventRecord(tc[b][1], st_d2h); copy_pend[b] = tot[0] + tot[1]; }
        if (relay >= 0) cudaSetDevice(dev_self);
        SCS_CUDA(c, er);
        c->stats.link_bytes[0] += tot[0]; c->stats.link_bytes[1] += tot[1];
        c->stats.fastq_bytes[0] += tot[0]; c->stats.fastq_bytes[1] += tot[1];
        c->stats.plain_bytes[0] += plain[0]; c->stats.plain_bytes[1] += plain[1];
        if (sink.submit(slot, eslot[slot], p, tot)) return c->fail(SCS_E_IO, "FASTQ sink failed");
        return SCS_OK;
    };
    uint64_t k = 0;
    for (uint64_t s0 = slot_lo; s0 < slot_hi; s0 += batch, k++) {
        const int b = (int)(k & 1);
        const uint64_t m = std::min(batch, slot_hi - s0);
        A.slot0 = s0; A.nslots = m;
        harvest(b);
        const bool packed = choose_packed(k, b);
        SCS_CUDA(c, cudaEventRecord(tq[b][0], c->st));
        SCS_CUDA(c, cudaMemsetAsync(W.size1.p, 0, (m + 1) * 4, c->st));
        if (nfiles == 2) SCS_CUDA(c, cudaMemsetAsync(W.size2.p, 0, (m + 1) * 4, c->st));
        SCS_CUDA(c, cudaEventRecord(tq[b][1], c->st));
        auto kern = c->replay.on ? emit_kernel<false, true> : emit_kernel<false, false>;
        kern<<<sms, emit_warps * 32, emit_smem, c->st>>>(g, dsrc, T, A, W.stage[0].p, nfiles == 2 ? W.stage[1].p : nullptr, W.flags.p, W.size1.p, W.size2.p, W.records.p,
                                                         isize_smem);
        SCS_LAUNCHED(c); c->stats.emit_launches++;
        SCS_CUDA(c, cudaEventRecord(tq[b][2], c->st));
        uint64_t* plain_tot = W.dtotals_mapped + (gz ? 4 : 0) + 2 * b;   // with gzip the copy sizes (slots 0..3) are the compressed totals
        if (int rc = scan_u32_noalloc(c, W.size1.p, W.off1.p, m, W.scan.p, plain_tot)) return rc;
        if (nfiles == 2) { if (int rc = scan_u32_noalloc(c, W.size2.p, W.off2.p, m, W.scan.p + 2048 + 8, plain_tot + 1)) return rc; }
        SCS_CUDA(c, cudaEventRecord(tq[b][3], c->st));   // kernel time of the slab without the compaction (~0.05 ms), which may wait for a copy
        const unsigned cgrid = (unsigned)std::min<uint64_t>((m + 7) / 8, (uint64_t)sms * 16);
        if (packed) {
            // wire bytes per record and their scan (total into the mapped slot 8 + 2b + f), then the packed slab behind its split table
            for (int f = 0; f < nfiles; f++) {
                wire_size_kernel<<<cgrid, 256, 0, c->st>>>(W.stage[f].p, stride, f ? W.size2.p : W.size1.p, m, c->wire_qlo, W.wsize[f].p); SCS_LAUNCHED(c);
                if (int rc = scan_u32_noalloc(c, W.wsize[f].p, W.woff[f].p, m, W.scan.p + (f ? 2048 + 8 : 0), W.dtotals_mapped + 8 + 2 * b + f)) return rc;
            }
            SCS_CUDA(c, cudaEventRecord(etotb[b], c->st));
            SCS_CUDA(c, cudaStreamWaitEvent(c->st, ecopy[b], 0));   // device slab b is free once the copy of the slab two back is done
            for (int f = 0; f < nfiles; f++) {
                pack_records_kernel<<<cgrid, 256, 0, c->st>>>(W.stage[f].p, stride, f ? W.size2.p : W.size1.p, f ? W.off2.p : W.off1.p, W.woff[f].p, m, c->wire_qlo,
                                                              c->slab_dev[b][f].p, wcap, W.flags.p);
                SCS_LAUNCHED(c);
            }
        } else if (!gz) {
            SCS_CUDA(c, cudaEventRecord(etotb[b], c->st));
            // the packed device slab b is free once the copy of the slab two back is done
            SCS_CUDA(c, cudaStreamWaitEvent(c->st, ecopy[b], 0));
            compact_records_kernel<<<cgrid, 256, 0, c->st>>>(W.stage[0].p, stride, W.size1.p, W.off1.p, m, c->slab_dev[b][0].p, slab, W.flags.p); SCS_LAUNCHED(c);
            if (nfiles == 2) { compact_records_kernel<<<cgrid, 256, 0, c->st>>>(W.stage[1].p, stride, W.size2.p, W.off2.p, m, c->slab_dev[b][1].p, slab, W.flags.p); SCS_LAUNCHED(c); }
        } else {
            // plain slab (device only) -> 32 KiB pieces deflated into fixed-stride cells -> scan of the member sizes -> packed compressed slab
            const bool last = s0 + batch >= slot_hi;
            for (int f = 0; f < nfiles; f++) {
                const uint32_t* sz = f ? W.size2.p : W.size1.p; const uint64_t* of = f ? W.off2.p : W.off1.p;
                compact_records_kernel<<<cgrid, 256, 0, c->st>>>(W.stage[f].p, stride, sz, of, m, c->slab_dev[b][f].p, slab, W.flags.p); SCS_LAUNCHED(c);
                SCS_CUDA(c, cudaMemsetAsync(c->gz.sizes[f].p, 0, (gz_pieces + 1) * 4, c->st));
                if (int rc = gz_launch(c, c->slab_dev[b][f].p, of, sz, m, c->gz.stage[f].p, gz_pieces, c->gz.sizes[f].p, last ? 1 : 0, W.flags.p, sms)) return rc;
                if (int rc = scan_u32_noalloc(c, c->gz.sizes[f].p, c->gz.offs[f].p, gz_pieces, W.scan.p + (f ? 2048 + 8 : 0), W.dtotals_mapped + 2 * b + f)) return rc;
            }
            SCS_CUDA(c, cudaEventRecord(etotb[b], c->st));
            SCS_CUDA(c, cudaStreamWaitEvent(c->st, ecopy[b], 0));   // the compressed slab b is free once the copy of the slab two back is done
            for (int f = 0; f < nfiles; f++) {
                compact_records_kernel<<<(unsigned)std::min<uint32_t>((gz_pieces + 7) / 8, (uint32_t)sms * 16), 256, 0, c->st>>>(c->gz.stage[f].p, gz_stage_stride(), c->gz.sizes[f].p,
                                                                                                                            c->gz.offs[f].p, gz_pieces, c->gz.slab[b][f].p, slab, W.flags.p);
                SCS_LAUNCHED(c);
            }
        }
        timed[b] = true;
        SCS_CUDA(c, cudaEventRecord(ekern[b], c->st));
        dv[b].launched = true; dv[b].k = k; dv[b].packed = packed; dv[b].m = m;
        if (int rc = finalize(b ^ 1)) return rc;   // slab k-1: totals known -> copy queued behind its compaction
        if (sink.service()) return c->fail(SCS_E_IO, "FASTQ sink failed");
    }
    if (int rc = finalize((int)((k - 1) & 1))) return rc;   // the last slab
    if (sink.finish()) return c->fail(SCS_E_IO, "FASTQ sink failed");
    SCS_CUDA(c, cudaStreamWaitEvent(c->st, ecopy[0], 0)); SCS_CUDA(c, cudaStreamWaitEvent(c->st, ecopy[1], 0));
    SCS_CUDA(c, cudaEventRecord(e1, c->st)); SCS_CUDA(c, cudaStreamSynchronize(c->st));
    float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
    harvest(0); harvest(1);
    c->stats.ms_reads = ms; c->stats.ms_reads_kernels = msk; c->stats.ms_emit_kernel = mse;
    int hflags = 0; SCS_CUDA(c, memcpy_sync(c, &hflags, W.flags.p, 4, cudaMemcpyDeviceToHost));
    unsigned long long hrec = 0; SCS_CUDA(c, memcpy_sync(c, &hrec, W.records.p, 8, cudaMemcpyDeviceToHost)); c->stats.records = hrec;
    if (hflags & 4) return c->fail(SCS_E_UNSUPPORTED, "more than 64 indel events in one read");
    if (hflags & 8) return c->fail(SCS_E_UNSUPPORTED, "read grew beyond 480 bases through insertions");
    if (hflags & 16) return c->fail(SCS_E_NOMEM, "FASTQ slab overflow (raise slab_bytes)");
    if (hflags & 32) return c->fail(SCS_E_STATE, "gzip: a byte outside the FASTQ alphabet or an oversized block");
    return SCS_OK;
}

// ---------------------------------------------------------------------------------- test hooks
__global__ void __launch_bounds__(kReadWarps * 32) test_predict_kernel(ReadTables T, const char* __restrict__ srcAscii, int n_reads, int isRead1,
                                                                       const uint32_t* real, uint64_t stride_real, const uint32_t* ints, uint64_t stride_int,
                                                                       char* out_seq, char* out_qual, int out_stride, int* out_len, int* flags) {
    __shared__ __align__(16) WarpScratch scratch[kReadWarps];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int r = blockIdx.x * kReadWarps + warp;
    if (r >= n_reads) return;
    WarpScratch* ws = &scratch[warp];
    RStream<true> S; S.k0 = S.k1 = S.e0 = S.e1 = S.dom2 = 0; S.t[0] = real + (uint64_t)r * stride_real; S.t[1] = ints + (uint64_t)r * stride_int;
    const int RL = T.RL;
    for (int i = lane; i < RL; i += 32) {
        char ch = srcAscii[(size_t)r * RL + i];
        ws->ref[i] = (uint8_t)(ch == 'A' ? 0 : ch == 'C' ? 1 : ch == 'G' ? 2 : ch == 'T' ? 3 : 4);
    }
    __syncwarp();
    bool myN = false;
    for (int i = lane; i < RL; i += 32) myN |= (ws->ref[i] == 4);
    const bool hasN = __any_sync(0xffffffffu, myN);
    uint32_t cr = 0, ci = 0; int nev = 0;
    const int np = indel_pass(S, T, RL, cr, ci, lane, ws, &nev, flags + r);
    __syncwarp();
    if (flags[r] != 0) { if (lane == 0) out_len[r] = -2; return; }   // more than kMaxEvents indel events
    if (np > kSrcCap || np > out_stride) { if (lane == 0) out_len[r] = -1; return; }
    __syncwarp();
    const uint8_t* src = build_source(S, np, nev, lane, ws);
    const PassTabs X = make_pass_tabs(T, nullptr, isRead1);
    if (hasN) (void)subst_quality_pass_n<true>(S, X, src, np, cr, ci, lane, out_seq + (size_t)r * out_stride, out_qual + (size_t)r * out_stride);
    else subst_quality_pass(S, X, src, np, cr, lane, out_seq + (size_t)r * out_stride, out_qual + (size_t)r * out_stride);
    if (lane == 0) out_len[r] = np;
}

int test_predict(scs_ctx* c, const char* src, int n_reads, int is_read1, const uint32_t* real, uint64_t stride_real, const uint32_t* ints,
                 uint64_t stride_int, char* out_seq, char* out_qual, int out_stride, int32_t* out_len) {
    if (!c->have_device) return c->fail(SCS_E_CUDA, "no CUDA device");
    if (!c->have_profile) return c->fail(SCS_E_STATE, "scs_test_predict: no profile loaded");
    const int RL = c->prof.readLength;
    if (RL > kRLCap) return c->fail(SCS_E_UNSUPPORTED, "read length above 320");
    DevBuf<char> dsrc, dseq, dqual; DevBuf<uint32_t> dreal, dint; DevBuf<int> dlen, flags;
    SCS_CUDA(c, dsrc.reserve((size_t)n_reads * RL + 16)); SCS_CUDA(c, dseq.reserve((size_t)n_reads * out_stride + 16)); SCS_CUDA(c, dqual.reserve((size_t)n_reads * out_stride + 16));
    SCS_CUDA(c, dreal.reserve((size_t)n_reads * stride_real + 4096)); SCS_CUDA(c, dint.reserve((size_t)n_reads * stride_int + 4096));
    SCS_CUDA(c, dlen.reserve(n_reads + 1)); SCS_CUDA(c, flags.reserve(n_reads + 1));
    SCS_CUDA(c, memset_sync(c, dreal.p, 0, dreal.cap * 4)); SCS_CUDA(c, memset_sync(c, dint.p, 0, dint.cap * 4)); SCS_CUDA(c, memset_sync(c, flags.p, 0, flags.cap * 4));
    SCS_CUDA(c, memset_sync(c, dseq.p, 0, dseq.cap)); SCS_CUDA(c, memset_sync(c, dqual.p, 0, dqual.cap));
    SCS_CUDA(c, memcpy_sync(c, dsrc.p, src, (size_t)n_reads * RL, cudaMemcpyHostToDevice));
    SCS_CUDA(c, memcpy_sync(c, dreal.p, real, (size_t)n_reads * stride_real * 4, cudaMemcpyHostToDevice));
    SCS_CUDA(c, memcpy_sync(c, dint.p, ints, (size_t)n_reads * stride_int * 4, cudaMemcpyHostToDevice));
    ReadTables T = make_tables(c);
    test_predict_kernel<<<(n_reads + kReadWarps - 1) / kReadWarps, kReadWarps * 32, 0, c->st>>>(T, dsrc.p, n_reads, is_read1, dreal.p, stride_real, dint.p, stride_int,
                                                                                              dseq.p, dqual.p, out_stride, dlen.p, flags.p);
    SCS_LAUNCHED(c);
    SCS_CUDA(c, cudaStreamSynchronize(c->st));
    SCS_CUDA(c, memcpy_sync(c, out_seq, dseq.p, (size_t)n_reads * out_stride, cudaMemcpyDeviceToHost));
    SCS_CUDA(c, memcpy_sync(c, out_qual, dqual.p, (size_t)n_reads * out_stride, cudaMemcpyDeviceToHost));
    SCS_CUDA(c, memcpy_sync(c, out_len, dlen.p, (size_t)n_reads * 4, cudaMemcpyDeviceToHost));
    return SCS_OK;
}

// full amplicon sequences as text (parity check of descriptors + error overlays)
__global__ void full_seq_kernel(Genome g, const uint64_t* __restrict__ desc, const uint64_t* __restrict__ errref, const uint32_t* __restrict__ err_pool,
                                const uint64_t* __restrict__ offs, uint64_t n, char* __restrict__ out) {
    uint64_t a = blockIdx.x;
    if (a >= n) return;
    Tmpl F = unpack_desc(desc[a]); uint64_t er = errref[a]; uint32_t nerr = (uint32_t)(er & 0xFFFF); const uint32_t* errs = err_pool + (er >> 16);
    char* o = out + offs[a];
    for (uint32_t i = threadIdx.x; i < F.len; i += blockDim.x) {
        uint32_t b = window_base(g, F.gstart, F.rc, i);
        for (uint32_t e = 0; e < nerr; e++) if (err_pos(errs[e]) == i) b = err_base(errs[e]);
        o[i] = "ACGTN"[b];
    }
    if (threadIdx.x == 0) o[F.len] = '\n';
}

int dump_full_seqs(scs_ctx* c, char* buf, uint64_t cap, int64_t* written) {
    const uint64_t n = c->fulls.n;
    std::vector<uint64_t> d(n);
    if (n) SCS_CUDA(c, memcpy_sync(c, d.data(), c->fulls.desc.p, n * 8, cudaMemcpyDeviceToHost));
    std::vector<uint64_t> offs(n + 1, 0);
    for (uint64_t i = 0; i < n; i++) offs[i + 1] = offs[i] + unpack_desc(d[i]).len + 1;
    *written = (int64_t)offs[n];
    if (!buf) return SCS_OK;
    if (cap < offs[n]) return c->fail(SCS_E_ARG, "scs_dump: buffer too small");
    if (n == 0) return SCS_OK;
    DevBuf<uint64_t> doffs; DevBuf<char> dout;
    SCS_CUDA(c, doffs.reserve(n + 1)); SCS_CUDA(c, dout.reserve(offs[n] + 16));
    SCS_CUDA(c, memcpy_sync(c, doffs.p, offs.data(), (n + 1) * 8, cudaMemcpyHostToDevice));
    Genome g = c->dev_genome();
    full_seq_kernel<<<(unsigned)n, 128, 0, c->st>>>(g, c->fulls.desc.p, c->fulls.errref.p, c->err_pool.p, doffs.p, n, dout.p); SCS_LAUNCHED(c);
    SCS_CUDA(c, cudaStreamSynchronize(c->st));
    SCS_CUDA(c, memcpy_sync(c, buf, dout.p, offs[n], cudaMemcpyDeviceToHost));
    return SCS_OK;
}

}  // namespace scs
