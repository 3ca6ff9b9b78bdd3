// Context object behind the C ABI: owns every device / pinned allocation of one genreads run.
#pragma once
#include <cuda_runtime.h>

#include <chrono>
#include <cstdint>
#include <cstdlib>
#include <cstdio>
#include <string>
#include <vector>

#include "../../include/scssim_b200.h"
#include "device_common.cuh"
#include "profile_host.h"
#include "vmm.h"
#include "nccl_shim.h"

namespace scs {

// Stream all device allocations are ordered on (set at every C-ABI entry to the context's compute stream).
// cudaMallocAsync / cudaFreeAsync from the device's default pool (release threshold = never) make the many
// short-lived scratch buffers of the stages free of device-wide synchronisation.
inline cudaStream_t& alloc_stream() { static thread_local cudaStream_t s = nullptr; return s; }

// growable device array (host-managed capacity). Small buffers come from the stream-ordered pool. Buffers of big_alloc_bytes()
// and more live on a reserved virtual range that is extended in place (vmm.h): growth neither reallocates nor copies. On
// this platform a cold cudaMallocAsync costs ~250 ms per GB (0.8 s for 10 GB even from a warm pool) and cudaMalloc/cudaFree
// of GB-sized blocks in a live context 10s-100s of ms, erratically (profiles/alloc_probe.cu, r01_alloc_probe.txt) — at the
// default gamma on a human-scale genome that was most of the amplification stage's time. Without the VMM entry points the
// big buffers fall back to cudaMalloc + copy.
inline size_t big_alloc_bytes() {
    static const size_t v = [] { const char* e = getenv("SCS_BIG_ALLOC_BYTES"); return e ? (size_t)strtoull(e, nullptr, 0) : (size_t)(32ull << 20); }();
    return v;
}
constexpr size_t kVmmReserve = 192ull << 30;   // address space per big buffer (more than one B200's HBM)
template <class T> struct DevBuf {
    T* p = nullptr; size_t cap = 0; bool big = false; VmmRange* vmm = nullptr;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { release(); }
    // cudaFree waits for the device by itself, but measurably slower (100s of ms at times) than when the stream is drained first
    static void free_one(T* q, bool qbig) { if (!q) return; if (qbig) { cudaStreamSynchronize(alloc_stream()); cudaFree(q); } else cudaFreeAsync(q, alloc_stream()); }
    void release() {
        if (vmm) { cudaDeviceSynchronize(); vmm->release(); delete vmm; vmm = nullptr; }
        else free_one(p, big);
        p = nullptr; cap = 0; big = false;
    }
    // ensure capacity >= n, keeping the first `keep` elements
    cudaError_t reserve(size_t n, size_t keep = 0, cudaStream_t = 0) {
        if (n <= cap) return cudaSuccess;
        size_t ncap = n + n / 8 + 1024;
        if (vmm) {   // extend in place: contents stay where they are
            cudaError_t e = vmm->grow(ncap * sizeof(T));
            if (e != cudaSuccess) return e;
            cap = vmm->mapped / sizeof(T);
            return cudaSuccess;
        }
        T* q = nullptr;
        const bool qbig = ncap * sizeof(T) >= big_alloc_bytes();
        VmmRange* v = nullptr;
        cudaError_t e;
        if (qbig && VmmRange::available()) {
            v = new VmmRange();
            e = v->init(kVmmReserve);
            if (e == cudaSuccess) e = v->grow(ncap * sizeof(T));
            if (e != cudaSuccess) { v->release(); delete v; v = nullptr; }
            else { q = reinterpret_cast<T*>(v->base); ncap = v->mapped / sizeof(T); }
        }
        if (!v) {
            e = qbig ? cudaMalloc((void**)&q, ncap * sizeof(T)) : cudaMallocAsync((void**)&q, ncap * sizeof(T), alloc_stream());
            if (e != cudaSuccess) return e;
        }
        if (p && keep) {
            e = cudaMemcpyAsync(q, p, keep * sizeof(T), cudaMemcpyDeviceToDevice, alloc_stream());
            if (e != cudaSuccess) { if (v) { v->release(); delete v; } else free_one(q, qbig); return e; }
        }
        free_one(p, big);
        p = q; cap = ncap; big = qbig && !v; vmm = v;
        return cudaSuccess;
    }
};

struct HostFrag { int32_t seq; int64_t start0; int32_t len; int32_t strand; };

// Where this rank's part of an amplicon list sits in the global (all ranks) list. A batch is the output of one
// amplification pass; inside a batch the global order is the REVERSE of the creation order (Amplicon.cpp:574-585),
// and the creation order walks the templates in global list order. A batch is cut into sub-batches inside which this
// rank's products are a contiguous run of the creation order:
//   * products of fragments (semi amplicons): one sub-batch; ranks own contiguous fragment ranges, lower ranks first;
//   * products of semi amplicons (full amplicons): one sub-batch per batch of the semi list; inside it the semi list
//     holds higher ranks first (it is itself reversed), so higher ranks' products are created first.
struct ListGeom {
    int nb;
    uint64_t lend[6];        // local list size after batch b
    uint64_t ltot[6];        // local products in batch b
    uint64_t gbase[6];       // global list size before batch b
    uint64_t gtot[6];        // global products in batch b
    int nsub[6];
    uint64_t sub_l0[6][6];   // local creation rank of this rank's first product of the sub-batch
    uint64_t sub_g0[6][6];   // global creation rank (inside the batch) of that product
};
__host__ __device__ inline uint64_t global_index(const ListGeom& G, uint64_t t) {
    int b = 0;
    while (b + 1 < G.nb && t >= G.lend[b]) b++;
    const uint64_t q = t - (b ? G.lend[b - 1] : 0);        // position inside the local batch (reverse creation order)
    const uint64_t lcr = G.ltot[b] - 1 - q;                 // local creation rank
    int sb = 0;
    while (sb + 1 < G.nsub[b] && lcr >= G.sub_l0[b][sb + 1]) sb++;
    const uint64_t gcr = G.sub_g0[b][sb] + (lcr - G.sub_l0[b][sb]);
    return G.gbase[b] + (G.gtot[b] - 1 - gcr);
}

// amplicon list (semi or full), structure of arrays, list order = the reference's -t 1 order
struct AmpList {
    DevBuf<uint64_t> desc;     // gstart | rc | len
    DevBuf<uint32_t> gc;
    DevBuf<uint64_t> errref;   // err pool offset << 16 | count
    DevBuf<uint32_t> primers;  // semis only
    uint64_t n = 0;
    std::vector<uint64_t> batch_end;
    void clear() { n = 0; batch_end.clear(); }   // capacity is kept: a second run of the stage allocates nothing
};

struct ReplayDev {
    bool on = false;
    DevBuf<uint32_t> wreal, wint, mrand, mreal;
    DevBuf<double> gcf;
    DevBuf<uint64_t> marks[8];
    std::vector<uint64_t> hmarks[8];   // host copies (entity, off_real, off_int)
    uint64_t n_marks[8] = {0};
    std::vector<uint32_t> h_mrand, h_mreal;
};

// device-resident threshold tables
struct DevProfile {
    DevBuf<uint32_t> subs1, subs2, qual, ins, del, isize;
    DevBuf<uint8_t> qualEff;
    DevBuf<uint32_t> qualDiag;   // [4][bins][kDiagW] compact diagonal rows for shared memory
    DevBuf<uint32_t> qualDiagPiv;    // [4][bins][4] pivots (entries 7, 15, 23, 31 of each compact row)
    DevBuf<uint32_t> qualDiagMeta;   // [4][bins]: lo | (n << 8) | (global-only << 16)
};

// persistent scratch of the amplification stage (per-template slot arrays, reused by every pass and every run)
struct AmpScratch {
    DevBuf<unsigned long long> dcount, ticket; DevBuf<int> flags;
    DevBuf<uint64_t> slot_off, cprefix, tdesc, terr; DevBuf<uint32_t> tgc, created, gbitmaps;
};

// temporaries of the allocation stage: kept between calls (mapping fresh device memory costs 1-100 ms per GB here, erratically —
// with per-call buffers the stage took 3 ms per step on one box and 158 ms on another)
struct AllocScratch {
    DevBuf<double> gcm, wg_buf, dsums, cdf; DevBuf<uint32_t> cg_buf, tmp, lslots;
    DevBuf<unsigned long long> dtot; DevBuf<uint64_t> dpref, oddp, sbase_g;
};

// persistent scratch of the read stage (no allocation inside the slab loop)
struct ReadScratch {
    DevBuf<uint32_t> size1, size2, nfail, hdrno, coarse;
    DevBuf<uint64_t> off1, off2, scan, totals;
    DevBuf<int> flags; DevBuf<unsigned long long> records;
    DevBuf<char> stage[2];         // fixed-stride records of one slab per file (staged emit), packed by compact_records_kernel
    DevBuf<uint32_t> wsize[2]; DevBuf<uint64_t> woff[2];   // packed slabs (wire.h): wire bytes per record and their scan
    uint64_t* htotals = nullptr;   // pinned + mapped: [2b + f] bytes of buffer b, file f; [4 + ...] gzip text; [8 + ...] wire records
    uint64_t* dtotals_mapped = nullptr;   // device view of htotals
};

// block-gzip output (deflate.cu): the run's Huffman code and CRC tables on the device, per-slab scratch
struct GzState {
    bool ready = false; uint32_t prefix_bits = 0;
    DevBuf<uint32_t> code, prefix, crc, x2n;
    DevBuf<char> stage[2];            // members of one slab per file at a fixed 64 KiB stride, packed by compact_records_kernel
    DevBuf<uint32_t> sizes[2]; DevBuf<uint64_t> offs[2];
    DevBuf<char> slab[2][2];          // [buffer][file] packed compressed slabs (what is copied to the host)
};

}  // namespace scs

namespace scs { class ExpandPool; }

struct scs_ctx {
    scs_params P;
    bool have_device = false;
    cudaStream_t st = nullptr, st_copy = nullptr;
    std::string err;
    scs::HostProfile prof; bool have_profile = false;
    scs::DevProfile dprof;

    // genome
    std::vector<std::string> seq_names; std::vector<uint64_t> seq_len, seq_goff;   // goff in bases, 32-aligned
    scs::DevBuf<uint64_t> genome_words; scs::DevBuf<uint32_t> genome_nmask; uint64_t genome_bases = 0; bool have_genome = false; int genome_has_n = 0;
    scs::Genome dev_genome() const { scs::Genome g; g.words = genome_words.p; g.nmask = genome_nmask.p; g.n_bases = genome_bases; g.has_n = genome_has_n; return g; }
    uint64_t ref_len_half = 0;

    // fragments
    std::vector<scs::HostFrag> frags;   // this rank's fragments (cut from its own sequences)
    uint64_t frag_lo = 0, frag_hi = 0;  // [0, frags.size())
    // global geometry (world > 1: every rank holds its own sequences of the cell)
    uint64_t seq_global0 = 0, frag_global0 = 0, n_frags_global = 0, frag_len_sum_global = 0, ref_len_sum = 0;
    scs::DevBuf<uint64_t> full_gidx, slot_gbase;   // per local full amplicon: global list index, global id of its first slot
    scs::DevBuf<uint64_t> frag_desc; scs::DevBuf<uint32_t> frag_primers; bool have_frags = false;

    scs::AmpList semis, fulls;
    scs::DevBuf<uint32_t> err_pool; scs::DevBuf<unsigned long long> err_top;   // err_top[0] = next free slot
    scs::DevBuf<long long> primer_counts; uint64_t total_primers = 0;
    bool amplified = false;
    // global (all ranks) list geometry, per batch
    scs::ListGeom semi_geom{}, full_geom{};   // this rank's place in the global semi / full lists

    // read allocation
    scs::DevBuf<double> weights; scs::DevBuf<uint32_t> counts; scs::DevBuf<uint64_t> slot_base; bool have_counts = false;
    uint64_t reads_requested = 0, n_slots = 0;

    scs::ReadScratch rscratch;
    scs::GzState gz;
    scs::AmpScratch ascratch;
    scs::AllocScratch lscratch;
    // staging buffers that keep their capacity between calls (cold device allocations are slow and erratic on this platform)
    scs::DevBuf<uint8_t> genome_stage, sv_stage, sv_ref, sv_text[2];
    char* sv_pinned[2] = {nullptr, nullptr};   // simuvars output slabs (pinned), kept between calls
    scs::ReplayDev replay;
    scs_allreduce_u64_fn ar_u64 = nullptr; scs_allreduce_f64_fn ar_f64 = nullptr; void* ar_user = nullptr;
    scs_allreduce_dev_f64_fn ar_dev_f64 = nullptr; scs_allreduce_dev_i64_fn ar_dev_i64 = nullptr; void* ar_dev_user = nullptr;
    // NCCL communicator of this context (scs_nccl_init): when set, every collective of the library runs on it and the hooks are unused
    ncclComm_t comm = nullptr; scs::DevBuf<uint64_t> coll_dev;
    double shard_weight = 1.0;
    // balance = 1: cell-wide copies (identical on every rank) that the read stage works from, and this rank's slot range
    scs::DevBuf<uint64_t> g_words, g_desc, g_errref, g_slot_base; scs::DevBuf<uint32_t> g_nmask, g_errs;
    bool global_view = false; uint64_t g_n_amp = 0, g_slot_lo = 0, g_slot_hi = 0, g_bases = 0; int g_has_n = 0;
    scs::DevBuf<uint64_t> g_gather;     // all ranks' (desc, errref, global index) triples before they are scattered into g_desc / g_errref
    uint64_t genome_version = 0;        // bumped by every genome load
    scs::DevBuf<uint32_t> gc_pref, n_pref; uint64_t gcidx_version = ~0ull;   // GC index of the local genome (build_gc_index)
    uint64_t g_genome_version = ~0ull, g_genome_stride = 0;   // what the replicated genome was built from: skipped while unchanged
    scs_stats stats{};
    scs_simuvars_stats sv_stats{}; std::string sv_warnings;

    // NVLink relay of the FASTQ slabs through a peer GPU's host link (scs_params.relay_device)
    int relay_dev = -1; cudaStream_t st_relay = nullptr; char* relay_buf[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}}; uint64_t relay_cap = 0;

    // FASTQ slabs
    scs::DevBuf<char> slab_dev[2][2];   // [buffer][file] packed device slabs
    std::vector<char*> ring_host[2];    // [file] ring of pinned host slots the slabs are copied into (slab_sink.h)
    uint64_t slab_cap = 0;
    // packed slabs (host_expand): pinned wire slots the packed slabs land in, the threads that expand them, the profile's lowest
    // quality index (a packed quality is q - wire_qlo)
    std::vector<char*> wire_host[2]; uint64_t wire_cap = 0;
    scs::ExpandPool* pool = nullptr;
    uint32_t wire_qlo = 0;

    int fail(int code, const std::string& msg) { err = msg; return code; }
};

#define SCS_CUDA(ctx, call)                                                                          \
    do {                                                                                             \
        cudaError_t e__ = (call);                                                                    \
        if (e__ != cudaSuccess)                                                                      \
            return (ctx)->fail(SCS_E_CUDA, std::string("CUDA error: ") + cudaGetErrorString(e__) + " at " + __FILE__ + ":" + std::to_string(__LINE__)); \
    } while (0)

#define SCS_LAUNCHED(ctx) ((ctx)->stats.kernel_launches++)

namespace scs {
// CUDA-event timer of one stage on the compute stream. Every exit path of the stage (errors included) drains the stream and
// frees the events, so a caller that retries on the same context never races with work left over from the failed call.
struct StageTimer {
    scs_ctx* c; cudaEvent_t e0 = nullptr, e1 = nullptr;
    explicit StageTimer(scs_ctx* ctx) : c(ctx) { cudaEventCreate(&e0); cudaEventCreate(&e1); cudaEventRecord(e0, c->st); }
    StageTimer(const StageTimer&) = delete;
    StageTimer& operator=(const StageTimer&) = delete;
    cudaError_t stop(double* ms) {
        cudaEventRecord(e1, c->st);
        cudaError_t e = cudaStreamSynchronize(c->st);
        float f = 0; if (e == cudaSuccess) cudaEventElapsedTime(&f, e0, e1);
        *ms = f;
        return e;
    }
    ~StageTimer() { cudaStreamSynchronize(c->st); cudaEventDestroy(e0); cudaEventDestroy(e1); }
};

// blocking copy ordered on the context's compute stream (device buffers are stream-ordered allocations)
inline cudaError_t memcpy_sync(scs_ctx* c, void* dst, const void* src, size_t n, cudaMemcpyKind kind) {
    cudaError_t e = cudaMemcpyAsync(dst, src, n, kind, c->st);
    if (e != cudaSuccess) return e;
    return cudaStreamSynchronize(c->st);
}
inline cudaError_t memset_sync(scs_ctx* c, void* dst, int v, size_t n) {
    cudaError_t e = cudaMemsetAsync(dst, v, n, c->st);
    if (e != cudaSuccess) return e;
    return cudaStreamSynchronize(c->st);
}
}  // namespace scs

namespace scs {
// stage entry points (one .cu each)
int genome_from_host(scs_ctx* c, int n, const char* const* names, const char* const* seqs, const uint64_t* lens);
int genome_from_fasta(scs_ctx* c, const char* path);
// one sequence of the cell: contiguous ASCII bases (blen == 0; in device memory if dev) or FASTA text with a fixed line geometry
struct SeqSrc { const char* p; uint64_t len; uint32_t blen, llen; bool dev; };
int genome_from_sources(scs_ctx* c, int n, const char* const* names, const SeqSrc* src);
// [lo, hi) of the sequences this rank keeps (midpoint rule, see genome_from_fasta)
void shard_by_midpoint(const std::vector<uint64_t>& lens, int rank, int world, size_t* lo, size_t* hi);
int simuvars_run(scs_ctx* c, const scs_simuvars_params& sp, const char* ref, const char* snp, const char* var, scs_sink_fn sink, void* user, bool to_genome);
int upload_profile(scs_ctx* c);
int create_frags(scs_ctx* c);
int amplify(scs_ctx* c);
int set_read_counts(scs_ctx* c);
struct SlabConsumer;
int yield_reads(scs_ctx* c, SlabConsumer& sink);
int plan_fastq_bytes(scs_ctx* c, uint64_t bytes[2]);
// block-gzip output (deflate.cu)
int gz_prepare(scs_ctx* c);
size_t gz_smem_bytes();
uint64_t gz_max_pieces(uint64_t slab_bytes);
uint64_t gz_stage_stride();
int gz_launch(scs_ctx* c, const char* plain, const uint64_t* offs, const uint32_t* sizes, uint64_t nrec, char* stage, uint32_t max_pieces, uint32_t* piece_sizes,
              int append_eof, int* flags, int sms);
int test_predict(scs_ctx* c, const char* src, int n_reads, int is_read1, const uint32_t* real, uint64_t stride_real, const uint32_t* ints,
                 uint64_t stride_int, char* out_seq, char* out_qual, int out_stride, int32_t* out_len);
int dump_full_seqs(scs_ctx* c, char* buf, uint64_t cap, int64_t* written);

// draw source for a domain (Philox or replay tapes)
DrawSrc draw_src(const scs_ctx* c, int domain);
// host-side draw for the few serial decisions kept on the host (fragment lengths, leftover chunk draws)
uint32_t host_draw(const scs_ctx* c, int domain, int engine, uint64_t entity, uint64_t mark_index, uint64_t i);

// device exclusive scan: out[i] = sum_{j<i} in[j] (u64), returns total through *total_dev (device pointer, may be null)
int allreduce_u64(scs_ctx* c, uint64_t* v, size_t n);
int allreduce_f64(scs_ctx* c, double* v, size_t n);
// in-place sum over ranks of n 64-bit words in device memory (NCCL hook if set, else staged through the host hook)
int allreduce_dev_i64(scs_ctx* c, void* dev, size_t n);
int allreduce_dev_f64(scs_ctx* c, double* dev, size_t n);
// all-gather in device memory: every rank's `count` elements of `elem` bytes (count * elem a multiple of 8) already sit at
// buf + rank * count * elem; on return every rank holds all W blocks. ncclAllGather over NVLink when the context has a
// communicator, otherwise a sum of zero-padded copies through the caller's hooks.
int allgather_dev(scs_ctx* c, void* buf, size_t count, size_t elem);
int exclusive_scan_u32(scs_ctx* c, const uint32_t* in, uint64_t* out, uint64_t n, uint64_t* total_host);
// same for n <= 2048*2048 without allocation or synchronisation: scratch holds 2048+8 u64, the total is left in *total_dev
// per-word prefix counts of C/G and N bases of the local packed genome (c->gc_pref, c->n_pref); cached by genome version
int build_gc_index(scs_ctx* c);
int scan_u32_noalloc(scs_ctx* c, const uint32_t* in, uint64_t* out, uint64_t n, uint64_t* scratch, uint64_t* total_dev);
}  // namespace scs
