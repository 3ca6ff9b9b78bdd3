// extern "C" surface of libscssim_b200.so (see include/scssim_b200.h for the reference call each
// function replaces). Thin: argument validation with the reference's messages, stage ordering, dumps.
#include <algorithm>
#include <cstring>

#include "ctx.h"
#include "fasta_host.h"
#include "file_sink.h"
#include "slab_sink.h"
#include "simuvars_plan.h"
#include "deflate_host.h"
#include "expand_host.h"

using namespace scs;

static std::string g_create_error;

extern "C" {

const char* scs_version(void) { return "scssim_b200 0.1 (sm_100a)"; }

int scs_device_count(void) { int n = 0; if (cudaGetDeviceCount(&n) != cudaSuccess) { (void)cudaGetLastError(); return 0; } return n; }

void scs_default_params(scs_params* p) {
    memset(p, 0, sizeof(*p));
    p->primers = 100000; p->gamma = 1e-9; p->coverage = 5; p->isize = 260; p->paired = 1;   // src/scssim.cpp:289-293
    p->seed = 0x5C55ull; p->device = 0; p->rank = 0; p->world = 1; p->balance = 0; p->slab_bytes = 0; p->io_threads = 0; p->ring_slabs = 0; p->gzip = 0; p->relay_device = -1;
    p->host_expand = -1; p->expand_threads = 0;
}

int scs_create(const scs_params* p, scs_ctx** out) {
    if (!p || !out) { g_create_error = "scs_create: null argument"; return SCS_E_ARG; }
    *out = nullptr;
    // validation of parseArgs_genReads (src/scssim.cpp:355-393), same messages
    if (p->primers < 1000) { g_create_error = "Error: the value of parameter \"primers\" should be at least 1000!"; return SCS_E_ARG; }
    if (p->gamma <= 0 || p->gamma > 1e-8) { g_create_error = "Error: the value of parameter \"gamma\" should be in 0~1e-8!"; return SCS_E_ARG; }
    if (p->coverage <= 0) { g_create_error = "Error: sequencing coverage not properly specified!"; return SCS_E_ARG; }
    if (p->world < 1 || p->rank < 0 || p->rank >= p->world) { g_create_error = "scs_create: bad rank/world"; return SCS_E_ARG; }
    scs_ctx* c = new scs_ctx();
    c->P = *p;
    if (p->device >= 0) {
        int n = 0;
        cudaError_t e = cudaGetDeviceCount(&n);
        if (e != cudaSuccess || n <= p->device) {
            g_create_error = std::string("no usable CUDA device (") + (e != cudaSuccess ? cudaGetErrorString(e) : "ordinal out of range") + "); the genreads path has no CPU fallback";
            delete c; return SCS_E_CUDA;
        }
        if (cudaSetDevice(p->device) != cudaSuccess || cudaStreamCreateWithFlags(&c->st, cudaStreamNonBlocking) != cudaSuccess ||
            cudaStreamCreateWithFlags(&c->st_copy, cudaStreamNonBlocking) != cudaSuccess) {
            g_create_error = std::string("CUDA error: ") + cudaGetErrorString(cudaGetLastError()); delete c; return SCS_E_CUDA;
        }
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, p->device) == cudaSuccess) { uint64_t keep = ~0ull; cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep); }
        c->have_device = true;
    }
    *out = c;
    return SCS_OK;
}

void scs_destroy(scs_ctx* c) {
    if (!c) return;
    const bool dev = c->have_device;
    cudaStream_t st = c->st, st_copy = c->st_copy;
    delete c->pool; c->pool = nullptr;   // joins the expansion threads (no job is in flight between calls)
    if (dev) {
        cudaSetDevice(c->P.device); alloc_stream() = c->st;
        cudaDeviceSynchronize();
        if (c->comm) { nccl_api().CommDestroy(c->comm); c->comm = nullptr; }
        if (c->st_relay) {   // relay buffers and stream live on the peer device
            cudaSetDevice(c->relay_dev);
            for (int b = 0; b < 2; b++) for (int f = 0; f < 2; f++) if (c->relay_buf[b][f]) cudaFree(c->relay_buf[b][f]);
            cudaStreamDestroy(c->st_relay); c->st_relay = nullptr;
            cudaSetDevice(c->P.device);
        }
        for (int f = 0; f < 2; f++) for (char* q : c->ring_host[f]) cudaFreeHost(q);
        for (int f = 0; f < 2; f++) for (char* q : c->wire_host[f]) cudaFreeHost(q);
        if (c->rscratch.htotals) cudaFreeHost(c->rscratch.htotals);
        for (int b = 0; b < 2; b++) if (c->sv_pinned[b]) cudaFreeHost(c->sv_pinned[b]);
    }
    delete c;   // device buffers are returned to the pool in stream order
    if (dev) {
        cudaStreamSynchronize(st);
        cudaStreamDestroy(st); cudaStreamDestroy(st_copy);
        alloc_stream() = nullptr;
    }
}

const char* scs_last_error(const scs_ctx* c) { return c ? c->err.c_str() : g_create_error.c_str(); }

int scs_load_profile(scs_ctx* c, const char* path) {
    if (!c || !path) return SCS_E_ARG;
    if (c->have_device) { cudaSetDevice(c->P.device); alloc_stream() = c->st; }   // upload_profile allocates on this context's device / stream
    if (!c->prof.load(path, c->P.paired != 0, c->P.isize)) return c->fail(SCS_E_IO, c->prof.error);
    c->have_profile = true; c->have_counts = false;
    return upload_profile(c);
}
int scs_read_length(const scs_ctx* c) { return (c && c->have_profile) ? c->prof.readLength : -1; }

int scs_load_genome(scs_ctx* c, const char* path) {
    if (!c || !path) return SCS_E_ARG;
    if (!c->have_device) return c->fail(SCS_E_CUDA, "no CUDA device: the genreads path has no CPU fallback");
    cudaSetDevice(c->P.device); alloc_stream() = c->st;
    return genome_from_fasta(c, path);
}
int scs_set_genome(scs_ctx* c, int n, const char* const* names, const char* const* seqs, const uint64_t* lens) {
    if (!c || !names || !seqs || !lens) return SCS_E_ARG;
    if (!c->have_device) return c->fail(SCS_E_CUDA, "no CUDA device: the genreads path has no CPU fallback");
    cudaSetDevice(c->P.device); alloc_stream() = c->st;
    return genome_from_host(c, n, names, seqs, lens);
}

int scs_set_collectives(scs_ctx* c, scs_allreduce_u64_fn fu, scs_allreduce_f64_fn fd, void* user) {
    if (!c) return SCS_E_ARG;
    c->ar_u64 = fu; c->ar_f64 = fd; c->ar_user = user;
    return SCS_OK;
}

int scs_set_device_collective(scs_ctx* c, scs_allreduce_dev_f64_fn fn_f64, scs_allreduce_dev_i64_fn fn_i64, void* user) {
    if (!c) return SCS_E_ARG;
    c->ar_dev_f64 = fn_f64; c->ar_dev_i64 = fn_i64; c->ar_dev_user = user;
    return SCS_OK;
}
// ---- NCCL inside the library
int scs_nccl_unique_id(char* id) {
    if (!id) return SCS_E_ARG;
    NcclApi& A = nccl_api();
    if (!A.ok) { g_create_error = "NCCL is not available: " + A.why; return SCS_E_UNSUPPORTED; }
    ncclUniqueId u;
    if (A.GetUniqueId(&u) != ncclSuccess) { g_create_error = "ncclGetUniqueId failed"; return SCS_E_CUDA; }
    memcpy(id, u.internal, SCS_NCCL_ID_BYTES);
    return SCS_OK;
}
int scs_nccl_init(scs_ctx* c, const char* id) {
    if (!c || !id) return SCS_E_ARG;
    if (!c->have_device) return c->fail(SCS_E_CUDA, "no CUDA device");
    if (c->P.world <= 1) return SCS_OK;
    NcclApi& A = nccl_api();
    if (!A.ok) return c->fail(SCS_E_UNSUPPORTED, "NCCL is not available: " + A.why);
    cudaSetDevice(c->P.device); alloc_stream() = c->st;
    if (c->comm) { A.CommDestroy(c->comm); c->comm = nullptr; }
    ncclUniqueId u; memcpy(u.internal, id, SCS_NCCL_ID_BYTES);
    ncclResult_t r = A.CommInitRank(&c->comm, c->P.world, u, c->P.rank);
    if (r != ncclSuccess) { c->comm = nullptr; return c->fail(SCS_E_CUDA, std::string("ncclCommInitRank: ") + A.GetErrorString(r)); }
    int n = 0; A.CommCount(c->comm, &n);
    if (n != c->P.world) return c->fail(SCS_E_STATE, "NCCL communicator size differs from world");
    return SCS_OK;
}
int scs_nccl_abort(scs_ctx* c) {   // may be called from another thread: releases a rank that waits in a collective for a failed peer
    if (!c) return SCS_E_ARG;
    ncclComm_t comm = c->comm;
    if (comm) { c->comm = nullptr; nccl_api().CommAbort(comm); }
    return SCS_OK;
}
int scs_nccl_version(void) { NcclApi& A = nccl_api(); int v = 0; if (A.ok) A.GetVersion(&v); return v; }

int scs_set_shard_weight(scs_ctx* c, double w) {
    if (!c || !(w > 0)) return SCS_E_ARG;
    c->shard_weight = w; c->have_counts = false;
    return SCS_OK;
}

int scs_create_frags(scs_ctx* c) { if (!c) return SCS_E_ARG; if (!c->have_device) return c->fail(SCS_E_CUDA, "no CUDA device"); cudaSetDevice(c->P.device); alloc_stream() = c->st; return create_frags(c); }
int scs_amplify(scs_ctx* c) { if (!c) return SCS_E_ARG; if (!c->have_device) return c->fail(SCS_E_CUDA, "no CUDA device"); cudaSetDevice(c->P.device); alloc_stream() = c->st; return amplify(c); }
int scs_set_read_counts(scs_ctx* c) { if (!c) return SCS_E_ARG; if (!c->have_device) return c->fail(SCS_E_CUDA, "no CUDA device"); cudaSetDevice(c->P.device); alloc_stream() = c->st; return set_read_counts(c); }
int scs_yield_reads_sink(scs_ctx* c, scs_sink_fn sink, void* user) {
    if (!c) return SCS_E_ARG;
    if (!c->have_device) return c->fail(SCS_E_CUDA, "no CUDA device");
    cudaSetDevice(c->P.device); alloc_stream() = c->st;
    CallbackConsumer cb(sink, user);
    return yield_reads(c, cb);
}

int scs_plan_fastq_bytes(scs_ctx* c, uint64_t bytes[2]) {
    if (!c || !bytes) return SCS_E_ARG;
    if (!c->have_device) return c->fail(SCS_E_CUDA, "no CUDA device");
    cudaSetDevice(c->P.device); alloc_stream() = c->st;
    return plan_fastq_bytes(c, bytes);
}

// Malbac::yieldReads' file side (Malbac.cpp:426-435, SeqWriter.cpp:12-54): <prefix>_1.fq/_2.fq or <prefix>.fq through the
// asynchronous sink. With several ranks all of them write ONE pair of files: a sizing pass gives every rank the exact number of
// bytes it will produce, the byte counts are exchanged, rank 0 creates and preallocates the files and every rank pwrite()s its
// shard at its final offset — no per-rank shard files, no concatenation pass.
int scs_yield_reads(scs_ctx* c, const char* prefix) {
    if (!c || !prefix) return SCS_E_ARG;
    if (!c->have_device) return c->fail(SCS_E_CUDA, "no CUDA device");
    cudaSetDevice(c->P.device); alloc_stream() = c->st;
    const bool gz = c->P.gzip != 0;
    // compressed shard sizes are not known before the shards exist: with gzip every rank writes its own member stream
    // (<prefix>.rank<r>_1.fq.gz ...; gzip members concatenate, so `cat` in rank order is the whole output)
    const int W = gz ? 1 : std::max(1, c->P.world), R = gz ? 0 : c->P.rank, nfiles = c->P.paired ? 2 : 1;
    const std::string base = std::string(prefix) + ((gz && c->P.world > 1) ? ".rank" + std::to_string(c->P.rank) : "");
    const std::string ext = gz ? ".fq.gz" : ".fq";
    const std::string name[2] = {c->P.paired ? base + "_1" + ext : base + ext, base + "_2" + ext};
    if (!c->have_profile) return c->fail(SCS_E_STATE, "scs_yield_reads: no profile loaded");
    if (!c->have_counts) { if (int rc = set_read_counts(c)) return rc; }
    uint64_t off[2] = {0, 0}, total[2] = {0, 0}, mine[2] = {0, 0};
    if (W > 1) {
        if (int rc = plan_fastq_bytes(c, mine)) {   // every rank must still take part in the exchange
            std::vector<uint64_t> v(2 * (size_t)W + 1, 0); v[2 * (size_t)W] = 1; (void)allreduce_u64(c, v.data(), v.size());
            return rc;
        }
        std::vector<uint64_t> v(2 * (size_t)W + 1, 0);
        v[2 * (size_t)R] = mine[0]; v[2 * (size_t)R + 1] = mine[1];
        if (int rc = allreduce_u64(c, v.data(), v.size())) return rc;
        if (v[2 * (size_t)W]) return c->fail(SCS_E_STATE, "scs_yield_reads: another rank failed in the sizing pass");
        for (int r = 0; r < W; r++) for (int f = 0; f < 2; f++) { if (r < R) off[f] += v[2 * (size_t)r + f]; total[f] += v[2 * (size_t)r + f]; }
    } else {
        const uint64_t slots = c->global_view ? c->g_slot_hi - c->g_slot_lo : c->n_slots;
        total[0] = total[1] = slots * (uint64_t)(30 + 2 * (c->prof.readLength + 8) + 4) / (gz ? 2 : 1);   // preallocation only: trimmed to the bytes written
    }
    AsyncFileConsumer sink(c->P.io_threads > 0 ? c->P.io_threads : 4, c->P.ring_slabs > 0 ? c->P.ring_slabs : 6, c->P.device, getenv("SCS_NO_ODIRECT") == nullptr);
    int rc = SCS_OK;
    auto open_all = [&](bool create) {
        for (int f = 0; f < nfiles && rc == SCS_OK; f++)
            if (!sink.open(f, name[f], off[f], create, create ? total[f] : 0, W == 1)) rc = c->fail(SCS_E_IO, "Error: can not open fastq file to save results:\n" + name[f]);
    };
    if (R == 0) open_all(true);
    if (W > 1) {   // the files exist (or rank 0 could not create them) before the other ranks open them
        uint64_t bad = rc != SCS_OK ? 1 : 0;
        if (int rc2 = allreduce_u64(c, &bad, 1)) return rc2;
        if (bad) return rc != SCS_OK ? rc : c->fail(SCS_E_IO, "Error: can not open fastq file to save results:\n" + name[0]);
        if (R != 0) open_all(false);
    }
    if (rc == SCS_OK) rc = yield_reads(c, sink);
    else (void)sink.finish();
    if (rc == SCS_OK && W > 1 && (sink.bytes(0) != mine[0] || (nfiles == 2 && sink.bytes(1) != mine[1])))
        rc = c->fail(SCS_E_STATE, "scs_yield_reads: shard size differs from the sizing pass");
    if (W > 1) {   // nobody returns before every shard is in the files
        uint64_t bad = rc != SCS_OK ? 1 : 0;
        if (int rc2 = allreduce_u64(c, &bad, 1)) return rc != SCS_OK ? rc : rc2;
        if (bad && rc == SCS_OK) rc = c->fail(SCS_E_IO, "scs_yield_reads: another rank failed while writing " + name[0]);
    }
    return rc;
}

// ---- simuvars
void scs_simuvars_default_params(scs_simuvars_params* p) { if (p) { p->ploidy = 2; p->libc_seed = 1; p->line_width = 100; p->reserved = 0; } }

static int simuvars_entry(scs_ctx* c, const scs_simuvars_params* p, const char* ref, const char* snp, const char* var, scs_sink_fn sink, void* user, bool to_genome) {
    if (!c) return SCS_E_ARG;
    if (!ref || !*ref) return c->fail(SCS_E_ARG, "Use --ref to specify the reference file (fasta).");   // src/scssim.cpp:146-150
    scs_simuvars_params sp; scs_simuvars_default_params(&sp); if (p) sp = *p;
    if (sp.ploidy < 1) return c->fail(SCS_E_ARG, "simuvars: ploidy must be positive");
    if (!c->have_device) return c->fail(SCS_E_CUDA, "no CUDA device: simuvars has no CPU fallback");
    cudaSetDevice(c->P.device); alloc_stream() = c->st;
    return simuvars_run(c, sp, ref, snp, var, sink, user, to_genome);
}
int scs_simuvars_sink(scs_ctx* c, const scs_simuvars_params* p, const char* ref, const char* snp, const char* var, scs_sink_fn sink, void* user) {
    if (!sink) return SCS_E_ARG;
    return simuvars_entry(c, p, ref, snp, var, sink, user, false);
}
int scs_simuvars_to_genome(scs_ctx* c, const scs_simuvars_params* p, const char* ref, const char* snp, const char* var) {
    return simuvars_entry(c, p, ref, snp, var, nullptr, nullptr, true);
}
int scs_simuvars(scs_ctx* c, const scs_simuvars_params* p, const char* ref, const char* snp, const char* var, const char* out) {
    if (!c) return SCS_E_ARG;
    if (!out || !*out) return c->fail(SCS_E_ARG, "Use --output to specify the output file.");   // src/scssim.cpp:162-166
    ParallelFileWriter w(c->P.io_threads > 0 ? c->P.io_threads : 4);
    if (!w.open(0, out)) return c->fail(SCS_E_IO, std::string("can not open file ") + out);   // Genome.cpp:337-340
    int rc = simuvars_entry(c, p, ref, snp, var, parallel_file_sink, &w, false);
    if (w.close() != 0 && rc == SCS_OK) rc = c->fail(SCS_E_IO, std::string("can not write file ") + out);
    return rc;
}
int scs_simuvars_get_stats(const scs_ctx* c, scs_simuvars_stats* out) { if (!c || !out) return SCS_E_ARG; *out = c->sv_stats; return SCS_OK; }
const char* scs_simuvars_warnings(const scs_ctx* c) { return c ? c->sv_warnings.c_str() : ""; }

struct scs_svplan { sv::Plan plan; };
scs_svplan* scs_svplan_create(int n, const char* const* names, const uint64_t* lens, const char* snp, const char* var, int ploidy, uint32_t seed, char* err, size_t errcap) {
    std::vector<sv::ChromIn> chroms;
    for (int i = 0; i < n; i++) chroms.push_back({names[i], lens[i]});
    scs_svplan* h = new scs_svplan();
    if (!sv::build_plan(h->plan, chroms, snp, var, ploidy, seed)) {
        if (err && errcap) { strncpy(err, h->plan.err.c_str(), errcap - 1); err[errcap - 1] = 0; }
        delete h; return nullptr;
    }
    return h;
}
void scs_svplan_destroy(scs_svplan* h) { delete h; }
int64_t scs_svplan_dump(const scs_svplan* h, int what, void* buf, uint64_t cap) {
    if (!h) return SCS_E_ARG;
    const sv::Plan& P = h->plan;
    std::vector<uint64_t> v; std::string s; const void* src = nullptr; uint64_t need = 0;
    switch (what) {
        case SCS_SVP_HAPS: for (auto& x : P.haps) { v.insert(v.end(), {(uint64_t)x.chrom, (uint64_t)x.hap, x.len, x.piece_lo, x.piece_hi, x.sub_lo, x.sub_hi}); } break;
        case SCS_SVP_PIECES: for (auto& x : P.pieces) { v.insert(v.end(), {x.out, x.src, (uint64_t)x.len}); } break;
        case SCS_SVP_SUBS: for (auto& x : P.subs) { v.insert(v.end(), {x.out, (uint64_t)x.ch}); } break;
        case SCS_SVP_LITERALS: s = P.literals; break;
        case SCS_SVP_NAMES: for (auto& x : P.haps) { s += x.name; s += '\n'; } break;
        case SCS_SVP_WARNINGS: s = P.warnings; break;
        default: return SCS_E_ARG;
    }
    if (what == SCS_SVP_LITERALS || what == SCS_SVP_NAMES || what == SCS_SVP_WARNINGS) { src = s.data(); need = s.size(); } else { src = v.data(); need = v.size() * 8; }
    if (!buf) return (int64_t)need;
    if (cap < need) return SCS_E_ARG;
    if (need) memcpy(buf, src, need);
    return (int64_t)need;
}
void scs_shard_sequences(const uint64_t* lens, size_t n, int rank, int world, size_t* lo, size_t* hi) {
    std::vector<uint64_t> v(lens, lens + n);
    shard_by_midpoint(v, rank, world < 1 ? 1 : world, lo, hi);
}
int64_t scs_test_fasta_index(const char* path, uint64_t* recs, uint64_t cap, char* names, uint64_t names_cap) {
    if (!path) return SCS_E_ARG;
    FastaFile ff; std::string err;
    if (!ff.open(path, &err)) return SCS_E_IO;
    std::string nm;
    for (size_t i = 0; i < ff.fai.size(); i++) {
        const FaiRec& r = ff.fai[i];
        if (recs && i < cap) { recs[5 * i] = r.len; recs[5 * i + 1] = r.off; recs[5 * i + 2] = r.blen; recs[5 * i + 3] = r.llen; recs[5 * i + 4] = r.regular ? 1 : 0; }
        nm += r.name; nm += '\n';
    }
    if (names && names_cap) { strncpy(names, nm.c_str(), names_cap - 1); names[names_cap - 1] = 0; }
    return (int64_t)ff.fai.size();
}
int scs_test_file_writer(const char* path, const char* data, uint64_t n, uint64_t slab_bytes, int threads) {
    if (!path || (!data && n) || slab_bytes == 0) return SCS_E_ARG;
    ParallelFileWriter w(threads);
    if (!w.open(0, path)) return SCS_E_IO;
    for (uint64_t o = 0; o < n; o += slab_bytes) if (w.write(0, data + o, (size_t)std::min(slab_bytes, n - o))) return SCS_E_IO;
    return w.close() ? SCS_E_IO : SCS_OK;
}
// The asynchronous file sink without a GPU: `n` bytes are fed slab by slab through a ring of page-aligned host buffers exactly as
// the read stage feeds it (each slab placed at the phase the sink asks for, no copy event), starting at file offset `base`.
int scs_test_async_writer(const char* path, const char* data, uint64_t n, uint64_t slab_bytes, int threads, int ring, uint64_t base, int create,
                          uint64_t prealloc, int direct, int* used_direct) {
    if (!path || (!data && n) || slab_bytes == 0) return SCS_E_ARG;
    AsyncFileConsumer sink(threads, ring, -1, direct != 0);
    if (!sink.open(0, path, base, create != 0, prealloc, false)) return SCS_E_IO;
    if (used_direct) *used_direct = sink.direct(0) ? 1 : 0;
    const int R = sink.ring_slots();
    std::vector<char*> slots((size_t)R, nullptr);
    for (auto& q : slots) if (posix_memalign((void**)&q, 4096, slab_bytes + 4096 + 64) != 0) return SCS_E_NOMEM;
    int rc = SCS_OK; uint64_t k = 0;
    for (uint64_t o = 0; o < n && rc == SCS_OK; o += slab_bytes, k++) {
        const uint64_t m = std::min(slab_bytes, n - o);
        const int slot = (int)(k % (uint64_t)R);
        if (sink.acquire(slot)) { rc = SCS_E_IO; break; }
        char* p[2] = {slots[slot] + (sink.phase(0) & 4095), nullptr};
        memcpy(p[0], data + o, m);
        const uint64_t bytes[2] = {m, 0};
        if (sink.submit(slot, nullptr, p, bytes)) rc = SCS_E_IO;
    }
    if (sink.finish()) rc = SCS_E_IO;
    for (char* q : slots) free(q);
    return rc;
}
// The Huffman code the block-gzip output of this context's profile is written with (host only): code lengths of the 256 literals
// and of end-of-block, and the constant prefix of every BGZF block (member header + dynamic-block header) as LSB-first bits.
int scs_test_deflate_code(const scs_ctx* c, uint8_t* lens, uint32_t* prefix_words, int cap_words, uint32_t* prefix_bits) {
    if (!c || !lens || !prefix_bits) return SCS_E_ARG;
    if (!c->have_profile) return SCS_E_STATE;
    uint64_t hist[257]; DeflateCode D;
    fastq_model_histogram(c->prof, c->P.paired != 0, hist);
    if (!build_deflate_code(hist, D)) return SCS_E_STATE;
    memcpy(lens, D.len, 257);
    *prefix_bits = D.prefix_bits;
    const int nw = (int)((D.prefix_bits + 31) / 32);
    if (prefix_words) { if (cap_words < nw) return SCS_E_ARG; memcpy(prefix_words, D.prefix_words.data(), (size_t)nw * 4); }
    return nw;
}
int scs_test_expand_wire(const uint8_t* wire, uint32_t nsplit, uint64_t wire_bytes, uint64_t text_bytes, int qchar0, int threads, int scalar, char* out) {
    if ((!wire && (nsplit || wire_bytes)) || (!out && text_bytes) || threads < 1) return SCS_E_ARG;
    ExpandPool pool(-1, threads);
    ExpandJob j;
    j.wire[0] = wire; j.nsplit[0] = nsplit; j.wire_bytes[0] = wire_bytes; j.text_bytes[0] = text_bytes; j.out[0] = out;
    j.qchar0 = qchar0; j.scalar = scalar != 0;
    pool.submit(&j);
    return pool.wait(&j) ? SCS_E_ARG : SCS_OK;
}

int scs_test_libc_rand(uint32_t seed, int n, uint32_t* out) {
    if (!out || n < 0) return SCS_E_ARG;
    sv::LibcRand r(seed);
    for (int i = 0; i < n; i++) out[i] = r.next();
    return SCS_OK;
}

int scs_get_stats(const scs_ctx* c, scs_stats* out) {
    if (!c || !out) return SCS_E_ARG;
    *out = c->stats;
    out->n_frags = c->frags.size();
    return SCS_OK;
}

int scs_set_replay(scs_ctx* c, const scs_replay* r) {
    if (!c || !r) return SCS_E_ARG;
    if (!c->have_device) return c->fail(SCS_E_CUDA, "no CUDA device");
    cudaSetDevice(c->P.device); alloc_stream() = c->st;
    ReplayDev& R = c->replay;
    const size_t pad = 8192;   // lanes may read a few draws past an entity's last one
    auto up = [&](DevBuf<uint32_t>& b, const uint32_t* p, uint64_t n) -> cudaError_t {
        cudaError_t e = b.reserve(n + pad); if (e != cudaSuccess) return e;
        e = memset_sync(c, b.p, 0, (n + pad) * 4); if (e != cudaSuccess) return e;
        return n ? memcpy_sync(c, b.p, p, n * 4, cudaMemcpyHostToDevice) : cudaSuccess;
    };
    SCS_CUDA(c, up(R.wreal, r->wreal, r->n_wreal)); SCS_CUDA(c, up(R.wint, r->wint, r->n_wint));
    SCS_CUDA(c, up(R.mrand, r->mrand, r->n_mrand)); SCS_CUDA(c, up(R.mreal, r->mreal, r->n_mreal));
    R.h_mrand.assign(r->mrand, r->mrand + r->n_mrand); R.h_mreal.assign(r->mreal, r->mreal + r->n_mreal);
    SCS_CUDA(c, R.gcf.reserve(r->n_gcf + 16));
    if (r->n_gcf) SCS_CUDA(c, memcpy_sync(c, R.gcf.p, r->gcf, r->n_gcf * 8, cudaMemcpyHostToDevice));
    for (int d = 0; d < 8; d++) {
        std::vector<uint64_t>& h = R.hmarks[d];
        h.assign(r->marks[d], r->marks[d] + 3 * r->n_marks[d]);
        if (d == SCS_D_READ) {   // dropped slots never started an entity: make the table dense by slot id
            uint64_t mx = 0; for (uint64_t i = 0; i < r->n_marks[d]; i++) mx = std::max(mx, h[3 * i] + 1);
            std::vector<uint64_t> dense(3 * mx, 0);
            for (uint64_t i = 0; i < r->n_marks[d]; i++) { uint64_t e = h[3 * i]; dense[3 * e] = e; dense[3 * e + 1] = h[3 * i + 1]; dense[3 * e + 2] = h[3 * i + 2]; }
            h.swap(dense);
        }
        R.n_marks[d] = h.size() / 3;
        SCS_CUDA(c, R.marks[d].reserve(h.size() + 16));
        if (!h.empty()) SCS_CUDA(c, memcpy_sync(c, R.marks[d].p, h.data(), h.size() * 8, cudaMemcpyHostToDevice));
    }
    R.on = true;
    return SCS_OK;
}

int64_t scs_dump(scs_ctx* c, int what, void* buf, uint64_t cap) {
    if (!c) return SCS_E_ARG;
    if (what == SCS_DUMP_FRAGS) {
        uint64_t need = c->frags.size() * 5 * 8;
        if (!buf) return (int64_t)need;
        if (cap < need) return c->fail(SCS_E_ARG, "scs_dump: buffer too small");
        std::vector<uint32_t> pr(c->frag_hi - c->frag_lo);
        if (!pr.empty() && c->have_device) memcpy_sync(c, pr.data(), c->frag_primers.p, pr.size() * 4, cudaMemcpyDeviceToHost);
        int64_t* o = (int64_t*)buf;
        for (size_t i = 0; i < c->frags.size(); i++) {
            const HostFrag& f = c->frags[i];
            o[5 * i] = f.seq; o[5 * i + 1] = f.start0; o[5 * i + 2] = f.len; o[5 * i + 3] = f.strand;
            o[5 * i + 4] = (i >= c->frag_lo && i < c->frag_hi) ? (int64_t)pr[i - c->frag_lo] : -1;
        }
        return (int64_t)need;
    }
    if (!c->have_device) return c->fail(SCS_E_CUDA, "no CUDA device");
    cudaSetDevice(c->P.device); alloc_stream() = c->st;
    if (what == SCS_DUMP_SEMIS || what == SCS_DUMP_FULLS) {
        AmpList& L = what == SCS_DUMP_SEMIS ? c->semis : c->fulls;
        uint64_t need = L.n * 6 * 8;
        if (!buf) return (int64_t)need;
        if (cap < need) return c->fail(SCS_E_ARG, "scs_dump: buffer too small");
        std::vector<uint64_t> d(L.n), e(L.n); std::vector<uint32_t> g(L.n), p(L.n, 0);
        if (L.n) {
            memcpy_sync(c, d.data(), L.desc.p, L.n * 8, cudaMemcpyDeviceToHost); memcpy_sync(c, e.data(), L.errref.p, L.n * 8, cudaMemcpyDeviceToHost);
            memcpy_sync(c, g.data(), L.gc.p, L.n * 4, cudaMemcpyDeviceToHost);
            if (what == SCS_DUMP_SEMIS) memcpy_sync(c, p.data(), L.primers.p, L.n * 4, cudaMemcpyDeviceToHost);
        }
        uint64_t* o = (uint64_t*)buf;
        for (uint64_t i = 0; i < L.n; i++) { Tmpl t = unpack_desc(d[i]); o[6 * i] = t.gstart; o[6 * i + 1] = t.rc; o[6 * i + 2] = t.len; o[6 * i + 3] = g[i]; o[6 * i + 4] = p[i]; o[6 * i + 5] = e[i] & 0xFFFF; }
        return (int64_t)need;
    }
    if (what == SCS_DUMP_COUNTS || what == SCS_DUMP_WEIGHTS) {
        if (!c->have_counts) return c->fail(SCS_E_STATE, "scs_dump: read counts not computed");
        uint64_t es = what == SCS_DUMP_COUNTS ? 4 : 8, need = c->fulls.n * es;
        if (!buf) return (int64_t)need;
        if (cap < need) return c->fail(SCS_E_ARG, "scs_dump: buffer too small");
        if (need) memcpy_sync(c, buf, what == SCS_DUMP_COUNTS ? (void*)c->counts.p : (void*)c->weights.p, need, cudaMemcpyDeviceToHost);
        return (int64_t)need;
    }
    if (what == SCS_DUMP_PRIMER_COUNTS) {
        uint64_t need = 65536 * 8;
        if (!buf) return (int64_t)need;
        if (cap < need) return c->fail(SCS_E_ARG, "scs_dump: buffer too small");
        if (!c->amplified) return c->fail(SCS_E_STATE, "scs_dump: not amplified");
        memcpy_sync(c, buf, c->primer_counts.p, need, cudaMemcpyDeviceToHost);
        return (int64_t)need;
    }
    if (what == SCS_DUMP_FULL_SEQ) {
        int64_t w = 0;
        int rc = dump_full_seqs(c, (char*)buf, cap, &w);
        return rc ? rc : w;
    }
    return c->fail(SCS_E_ARG, "scs_dump: unknown selector");
}

int scs_test_predict(scs_ctx* c, const char* src, int n_reads, int is_read1, const uint32_t* real, uint64_t stride_real, const uint32_t* ints,
                     uint64_t stride_int, char* out_seq, char* out_qual, int out_stride, int32_t* out_len) {
    if (!c) return SCS_E_ARG;
    if (c->have_device) { cudaSetDevice(c->P.device); alloc_stream() = c->st; }
    return test_predict(c, src, n_reads, is_read1, real, stride_real, ints, stride_int, out_seq, out_qual, out_stride, out_len);
}

static __global__ void philox_test_kernel(const uint32_t* ck, uint32_t* out) { philox4x32_10(ck[0], ck[1], ck[2], ck[3], ck[4], ck[5], out); }
static __global__ void det_log_test_kernel(const double* x, int n, double* out) { int i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) out[i] = det_log(x[i]); }

int scs_test_philox(scs_ctx* c, const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
    if (!c) return SCS_E_ARG;
    if (!c->have_device) return c->fail(SCS_E_CUDA, "no CUDA device");
    cudaSetDevice(c->P.device); alloc_stream() = c->st;
    DevBuf<uint32_t> d; SCS_CUDA(c, d.reserve(16));
    uint32_t h[6] = {ctr[0], ctr[1], ctr[2], ctr[3], key[0], key[1]};
    SCS_CUDA(c, memcpy_sync(c, d.p, h, 24, cudaMemcpyHostToDevice));
    philox_test_kernel<<<1, 1, 0, c->st>>>(d.p, d.p + 8); SCS_LAUNCHED(c);
    SCS_CUDA(c, cudaStreamSynchronize(c->st));
    SCS_CUDA(c, memcpy_sync(c, out, d.p + 8, 16, cudaMemcpyDeviceToHost));
    return SCS_OK;
}
int scs_test_det_log(scs_ctx* c, const double* x, int n, double* out) {
    if (!c) return SCS_E_ARG;
    if (!c->have_device) return c->fail(SCS_E_CUDA, "no CUDA device");
    cudaSetDevice(c->P.device); alloc_stream() = c->st;
    DevBuf<double> a, b; SCS_CUDA(c, a.reserve(n + 1)); SCS_CUDA(c, b.reserve(n + 1));
    SCS_CUDA(c, memcpy_sync(c, a.p, x, (size_t)n * 8, cudaMemcpyHostToDevice));
    det_log_test_kernel<<<(n + 255) / 256, 256, 0, c->st>>>(a.p, n, b.p); SCS_LAUNCHED(c);
    SCS_CUDA(c, cudaStreamSynchronize(c->st));
    SCS_CUDA(c, memcpy_sync(c, out, b.p, (size_t)n * 8, cudaMemcpyDeviceToHost));
    return SCS_OK;
}

int scs_profile_thresholds(const scs_ctx* c, int which, int idx, int row, uint32_t* out, int cap, int* eff) {
    if (!c || !c->have_profile) return SCS_E_STATE;
    const HostProfile& P = c->prof;
    const uint32_t* src = nullptr; int n = 0, e = 0;
    switch (which) {
        case 0: src = P.insThr.thr.data(); n = (int)P.insThr.thr.size(); e = P.insThr.eff; break;
        case 1: src = P.delThr.thr.data(); n = (int)P.delThr.thr.size(); e = P.delThr.eff; break;
        case 2: if (!P.hasISize) return SCS_E_STATE; src = P.iSizeThr.thr.data(); n = (int)P.iSizeThr.thr.size(); e = P.iSizeThr.eff; break;
        case 3: case 4: {
            const std::vector<uint32_t>& t = which == 3 ? P.subsThr1 : P.subsThr2;
            if (t.empty() || idx < 0 || idx >= P.kmerCount || row < 0 || row >= P.bins) return SCS_E_ARG;
            src = &t[((size_t)idx * P.bins + row) * 4]; n = 4; e = (int)src[3]; break;
        }
        case 5:
            if (idx < 0 || idx >= 16 || row < 0 || row >= P.bins) return SCS_E_ARG;
            src = &P.qualThr[((size_t)idx * P.bins + row) * kQualN]; n = kQualN; e = P.qualEff[(size_t)idx * P.bins + row]; break;
        default: return SCS_E_ARG;
    }
    if (eff) *eff = e;
    for (int i = 0; i < n && i < cap; i++) out[i] = (which == 3 || which == 4) && i == 3 ? 0xFFFFFFFFu : src[i];
    return n;
}

}  // extern "C"
