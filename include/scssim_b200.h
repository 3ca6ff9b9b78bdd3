/* scssim_b200 — C ABI of the B200-native `scssim genreads` hot path (and of `scssim simuvars`, the producer of its input).
 *
 * Drop-in boundary (SURVEY.md §8b). Each entry point replaces one stage call that the reference's
 * main() makes on its global singletons (/root/reference/src/scssim.cpp:46-66):
 *
 *   reference call (file:line)                                    replaced by
 *   ------------------------------------------------------------  -----------------------------
 *   parseArgs_genReads -> Config (src/scssim.cpp:285-404)          scs_params / scs_create
 *   new ThreadPool(t); pool_init() (src/scssim.cpp:49-50)          scs_create (CUDA streams, Philox seed)
 *   genome.loadData() (src/scssim.cpp:53, lib/genome/Genome.cpp:18)  scs_load_genome / scs_set_genome
 *   profile.train(file) (src/scssim.cpp:56, lib/profile/Profile.cpp:1432)  scs_load_profile
 *   malbac.createFrags() (src/scssim.cpp:59, lib/malbac/Malbac.cpp:143)    scs_create_frags
 *   malbac.amplify() (src/scssim.cpp:62, lib/malbac/Malbac.cpp:173)        scs_amplify
 *   malbac.yieldReads() (src/scssim.cpp:65, lib/malbac/Malbac.cpp:410)     scs_yield_reads[_sink]
 *   SeqWriter::write (lib/seqwriter/SeqWriter.cpp:41-54)                   scs_sink_fn / io_threads
 *   simuvars: genome.loadData(); genome.saveSequence() (src/scssim.cpp:33-38,
 *     lib/genome/Genome.cpp:35-198,329-691, lib/snp/snp.cpp:147-203)       scs_simuvars / _sink / _to_genome
 *
 * Plain pointers and sizes only; no exceptions and no exit() cross this boundary. Every function
 * returns 0 on success or a negative SCS_E_* code; scs_last_error(ctx) gives the message the
 * reference would have printed before exit(1). There is no CPU fallback: without a CUDA device
 * scs_create fails with SCS_E_CUDA.
 */
#ifndef SCSSIM_B200_H
#define SCSSIM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SCS_OK 0
#define SCS_E_ARG (-1)        /* bad argument / flag validation (src/scssim.cpp:349-393) */
#define SCS_E_IO (-2)         /* cannot open / malformed input file */
#define SCS_E_CUDA (-3)       /* CUDA runtime error or no device */
#define SCS_E_STATE (-4)      /* stage called out of order */
#define SCS_E_UNSUPPORTED (-5)
#define SCS_E_NOMEM (-6)

typedef struct scs_ctx scs_ctx;

/* The genreads flags (src/scssim.cpp:289-293 defaults) plus the extra, non-reference knobs. */
typedef struct scs_params {
    int64_t primers;      /* -p, default 100000, >= 1000 */
    double gamma;         /* -r, default 1e-9, (0, 1e-8] */
    double coverage;      /* -c, default 5, > 0 */
    int32_t isize;        /* -s, default 260 */
    int32_t paired;       /* -l PE -> 1 (default), SE -> 0 */
    uint64_t seed;        /* Philox key (extra flag --seed) */
    int32_t device;       /* CUDA device ordinal */
    int32_t rank;         /* shard index in [0, world) */
    int32_t world;        /* number of shards (GPUs) */
    int32_t balance;      /* world > 1 only. 0: every rank writes the reads of its own amplicons. 1: the packed genome and the
                             amplicon table are replicated over the ranks (all-reduce over NVLink) and the cell's read slots are
                             cut into contiguous ranges in proportion to scs_set_shard_weight(), so a GPU behind a slower host
                             link gets fewer reads; the shards then concatenate (rank order) to exactly the 1-GPU files */
    uint64_t slab_bytes;  /* FASTQ staging slab per file; 0 -> default (64 MiB) */
    int32_t io_threads;   /* host threads that pwrite() the slabs to the output files (the CLI's -t); 0 -> default (4) */
    int32_t ring_slabs;   /* scs_yield_reads: pinned host slabs per file the asynchronous file sink may hold; 0 -> default (6) */
    int32_t gzip;         /* 1: FASTQ leaves the device block-gzip compressed (BGZF: independent gzip members of 32 KiB of text, one
                             dynamic-Huffman block of literals each, ~2.1x smaller). Sinks receive the compressed bytes; scs_yield_reads
                             writes <prefix>_1.fq.gz/_2.fq.gz or <prefix>.fq.gz (world > 1: one shard <prefix>.rank<r>... per rank,
                             `cat` of the shards in rank order is the whole output). Extra flag --gz; the reference writes plain text */
    int32_t relay_device; /* -1 (default): FASTQ slabs are copied to the host over this GPU's own link. >= 0: over NVLink to that peer
                             GPU first and from there to the host — for boxes where some GPUs sit behind a slow or shared host link
                             (bench.py measures the links and lets the GPUs of the slow group relay through the fast group) */
    int32_t host_expand;  /* FASTQ slabs sent as packed base+quality records and expanded into text by host threads, so that the host link
                             carries ~47 % fewer bytes for them. -1 (default, auto): for every slab the read stage picks whichever path,
                             text over the link or packed + host expansion, is estimated to finish sooner (moving averages of the link
                             rate and of the expansion rate); on only for world = 1, gzip = 0 and scs_yield_reads_sink. 0: off.
                             1: every slab packed; 2: every other slab packed (1 and 2 also at world > 1; both for tests). The bytes
                             a sink receives are the same FASTQ text on every path; scs_yield_reads (files) always sends text */
    int32_t expand_threads; /* host threads of the expansion pool; 0 -> default (CPUs in the process's affinity mask - 1) */
} scs_params;

void scs_default_params(scs_params* p);

int scs_create(const scs_params* p, scs_ctx** out);
void scs_destroy(scs_ctx* ctx);
const char* scs_last_error(const scs_ctx* ctx);   /* ctx may be NULL: error of the last failed scs_create */

/* .profile parser + CDF -> threshold tables (Profile::train(file), Profile.cpp:1432-1436) */
int scs_load_profile(scs_ctx* ctx, const char* path);
int scs_read_length(const scs_ctx* ctx);

/* FASTA ingest + 2-bit pack on the device (Genome::loadData, Fragment::createSequence) */
int scs_load_genome(scs_ctx* ctx, const char* fasta_path);
/* Same, from host buffers: n sequences of ASCII bases. names[i] is the sequence name
 * (`<chr>_<k>_<len>`, Malbac.cpp:413-419). */
int scs_set_genome(scs_ctx* ctx, int n, const char* const* names, const char* const* seqs, const uint64_t* lens);

/* Collective hook for world > 1: sum `n` u64 / f64 values over all ranks in place. The caller
 * supplies it (torch.distributed/NCCL in bench.py, ncclAllReduce in the CLI). Unused when world == 1. */
typedef int (*scs_allreduce_u64_fn)(void* user, uint64_t* buf, size_t n);
typedef int (*scs_allreduce_f64_fn)(void* user, double* buf, size_t n);
int scs_set_collectives(scs_ctx* ctx, scs_allreduce_u64_fn fu, scs_allreduce_f64_fn fd, void* user);
/* Optional: in-place sum of `n` doubles that live in DEVICE memory (the cell-wide weight vector of the read allocation;
 * ncclAllReduce over NVLink without a host round trip). The library's stream is idle when the hook is called and the
 * hook must have completed the reduction when it returns. Without it the host hook above is used. */
typedef int (*scs_allreduce_dev_f64_fn)(void* user, double* dev_buf, size_t n);
/* Same for 64-bit integers (balance = 1: genome words, amplicon descriptors, error lists — every element is non-zero on
 * exactly one rank, so the sum is a gather). */
typedef int (*scs_allreduce_dev_i64_fn)(void* user, int64_t* dev_buf, size_t n);
int scs_set_device_collective(scs_ctx* ctx, scs_allreduce_dev_f64_fn fn_f64, scs_allreduce_dev_i64_fn fn_i64, void* user);
/* NCCL inside the library (replaces the hooks above): rank 0 obtains an id, hands the 128 bytes to the other ranks by any means
 * (shared memory between the CLI's worker threads, a broadcast in bench.py), and every rank calls scs_nccl_init — collectively,
 * like ncclCommInitRank. From then on all collectives of the context run on that communicator over NVLink: ncclAllReduce for
 * the per-pass counters and the cell-wide weight vector, ncclAllGather for the replication of the packed genome and the
 * amplicon table (balance = 1). libnccl.so.2 is resolved at run time; a copy already loaded into the process is reused.
 * scs_nccl_abort may be called from another thread to release a rank that waits in a collective for a peer that failed. */
#define SCS_NCCL_ID_BYTES 128
int scs_nccl_unique_id(char* id_out);
int scs_nccl_init(scs_ctx* ctx, const char* id);
int scs_nccl_abort(scs_ctx* ctx);
int scs_nccl_version(void);   /* 0 when NCCL cannot be loaded */
/* Relative share of the cell's reads this rank should write when balance = 1 (e.g. its measured D2H rate). Default 1. */
int scs_set_shard_weight(scs_ctx* ctx, double weight);

int scs_create_frags(scs_ctx* ctx);   /* Genome::splitToFrags, Genome.cpp:753-782 */
int scs_amplify(scs_ctx* ctx);        /* Malbac::amplify, Malbac.cpp:173-201 */

/* FASTQ sink: called on the calling thread, in file order, with bytes that already sit in pinned
 * host memory. file = 0 for <prefix>.fq / <prefix>_1.fq, 1 for <prefix>_2.fq. Return non-zero to abort. */
typedef int (*scs_sink_fn)(void* user, int file, const char* data, size_t nbytes);
int scs_yield_reads_sink(scs_ctx* ctx, scs_sink_fn sink, void* user);
/* Malbac::yieldReads: writes <prefix>_1.fq/_2.fq (PE) or <prefix>.fq (SE) through an asynchronous sink (writer threads behind a
 * ring of pinned slabs; O_DIRECT + fallocate where the file system has them). For world > 1 all ranks write ONE pair of files:
 * the byte count of every shard is computed first (scs_plan_fastq_bytes), exchanged through the collective hook, and every rank
 * writes its shard at its final offset (with balance = 1 the files are byte-identical to a single-rank run). */
int scs_yield_reads(scs_ctx* ctx, const char* prefix);
/* Exact number of FASTQ bytes this rank will write to each file (a sizing pass over the indel draws; nothing is emitted). */
int scs_plan_fastq_bytes(scs_ctx* ctx, uint64_t bytes[2]);
/* Read allocation only (Malbac::setReadCounts); scs_yield_reads* call it themselves if needed. */
int scs_set_read_counts(scs_ctx* ctx);

typedef struct scs_stats {
    uint64_t n_sequences, genome_bases;
    uint64_t n_frags, n_semis, n_fulls;        /* this rank */
    uint64_t n_semis_global, n_fulls_global;
    uint64_t reads_requested;                  /* Malbac.cpp:420, individual reads */
    uint64_t records;                          /* FASTQ records written by this rank (both files) */
    uint64_t fastq_bytes[2];
    uint64_t total_primers_left;
    uint64_t kernel_launches;                  /* kernels of this library launched so far */
    double ms_pack, ms_amplify, ms_alloc, ms_reads;   /* CUDA-event times of the last run of each stage */
    double ms_reads_kernels;                   /* plan+scan+emit kernels only, summed over slabs */
    double ms_emit_kernel;                     /* emit kernel only, summed */
    uint64_t emit_launches;
    uint64_t genome_window_bytes;              /* algorithmic HBM read bytes of the emit kernel */
    uint64_t plain_bytes[2];                   /* FASTQ text bytes behind fastq_bytes (equal unless gzip = 1, then fastq_bytes is compressed) */
    uint64_t link_bytes[2];                    /* bytes that crossed the host link per file (packed slabs: records + split table) */
    uint64_t slabs_packed, slabs;              /* slabs sent packed (host_expand) / all slabs of the last read stage */
} scs_stats;
int scs_get_stats(const scs_ctx* ctx, scs_stats* out);

/* ---- simuvars (SURVEY.md §8f row N1) -------------------------------------------------------------
 * The `scssim simuvars` subcommand: main's `genome.loadData(); genome.saveSequence();` (src/scssim.cpp:33-38), i.e.
 * Genome::loadAbers / loadSNPs / loadRefSeq (lib/genome/Genome.cpp:35-198, lib/snp/snp.cpp:147-203) and
 * Genome::saveSequence / generateSegment (Genome.cpp:329-691). Flags of parseArgs_simuVars (src/scssim.cpp:109-172):
 * -r ref FASTA, -s SNP file (may be NULL/empty), -v variation file (may be NULL/empty), -o output FASTA.
 * The host turns the variant files into an edit plan (piece table); CUDA kernels materialise the haplotypes.
 * Output is byte-identical to the reference's, which is deterministic: it draws from libc rand() without seeding it. */
typedef struct scs_simuvars_params {
    int32_t ploidy;       /* Config.cpp:35: 2 */
    uint32_t libc_seed;   /* state of libc rand(): 1 = never seeded, what the reference runs with */
    int32_t line_width;   /* bases per FASTA line, Genome.cpp:371: 100 */
    int32_t reserved;
} scs_simuvars_params;
void scs_simuvars_default_params(scs_simuvars_params* p);
/* Writes the simulated cell as FASTA (`>chr_k_len` records, Genome.cpp:365-383). */
int scs_simuvars(scs_ctx* ctx, const scs_simuvars_params* p, const char* ref_fasta, const char* snp_file, const char* var_file, const char* out_fasta);
/* Same, the bytes of the output file handed to `sink` in file order (file = 0) from pinned host memory. */
int scs_simuvars_sink(scs_ctx* ctx, const scs_simuvars_params* p, const char* ref_fasta, const char* snp_file, const char* var_file, scs_sink_fn sink, void* user);
/* Same cell, but it never leaves the device: the haplotypes are packed straight into this context's genome, as if the
 * output FASTA had been written and then read by scs_load_genome (world > 1: this rank keeps its share of the haplotypes). */
int scs_simuvars_to_genome(scs_ctx* ctx, const scs_simuvars_params* p, const char* ref_fasta, const char* snp_file, const char* var_file);
typedef struct scs_simuvars_stats {
    uint64_t n_chroms, n_haps, n_segments, n_pieces, n_subs;
    uint64_t n_cnv, n_snv, n_ins, n_del, n_snp;             /* what the reference reports while loading */
    uint64_t ref_bases, out_bases, out_bytes, h2d_bytes;
    uint64_t normalize_bytes, materialize_bytes;            /* algorithmic HBM bytes of the two kernels */
    uint64_t launches;
    double ms_read, ms_plan, ms_device, ms_kernels, ms_total;   /* host clock, except ms_kernels (CUDA events) */
} scs_simuvars_stats;
int scs_simuvars_get_stats(const scs_ctx* ctx, scs_simuvars_stats* out);
/* Warnings the reference prints while loading (malformed SNP lines); empty string if none. */
const char* scs_simuvars_warnings(const scs_ctx* ctx);

/* Host-only test hooks (no GPU): the edit plan itself. */
typedef struct scs_svplan scs_svplan;
/* chrom_names/chrom_lens describe the reference (names already stripped of "chr"); returns NULL and fills err on failure. */
scs_svplan* scs_svplan_create(int n_chroms, const char* const* chrom_names, const uint64_t* chrom_lens, const char* snp_file, const char* var_file,
                              int ploidy, uint32_t libc_seed, char* err, size_t errcap);
void scs_svplan_destroy(scs_svplan* plan);
enum scs_svplan_dump { SCS_SVP_HAPS = 0,      /* u64 x7 per haplotype: chrom, hap, length, piece_lo, piece_hi, sub_lo, sub_hi */
                       SCS_SVP_PIECES = 1,    /* u64 x3 per piece: out offset, source (bit 63: literal pool), length */
                       SCS_SVP_SUBS = 2,      /* u64 x2 per substitution: out offset, base */
                       SCS_SVP_LITERALS = 3,  /* bytes */
                       SCS_SVP_NAMES = 4,     /* record names, '\n' separated */
                       SCS_SVP_WARNINGS = 5   /* what the reference prints while loading (malformed SNP lines) */ };
int64_t scs_svplan_dump(const scs_svplan* plan, int what, void* buf, uint64_t cap);
/* Host-only test hooks for the file side. scs_test_fasta_index: the .fai model the loaders build (lib/fastahack/Fasta.cpp:103-191);
 * writes up to cap records of 5 u64 (length, offset, bases per line, bytes per line, regular geometry 0/1) and the '\n'-joined
 * names; returns the record count or a negative code. scs_test_file_writer: writes n bytes to path through the parallel pwrite
 * sink in slabs of slab_bytes with the given thread count; returns 0 on success. */
int64_t scs_test_fasta_index(const char* path, uint64_t* recs, uint64_t cap, char* names, uint64_t names_cap);
int scs_test_file_writer(const char* path, const char* data, uint64_t n, uint64_t slab_bytes, int threads);
/* The asynchronous file sink of scs_yield_reads without a GPU: feeds n bytes in slabs of slab_bytes through a ring of `ring`
 * page-aligned host buffers into `path` starting at file offset `base` (create != 0: create/truncate and preallocate `prealloc`
 * bytes; otherwise the file must exist — several callers can fill disjoint regions of one file). direct != 0 asks for O_DIRECT;
 * *used_direct tells whether the file system granted it. Returns 0 on success. */
int scs_test_async_writer(const char* path, const char* data, uint64_t n, uint64_t slab_bytes, int threads, int ring, uint64_t base, int create,
                          uint64_t prealloc, int direct, int* used_direct);
/* Host-only: the canonical Huffman code (lengths of literals 0..255 and of end-of-block) and the constant bit prefix (18-byte BGZF
 * member header + dynamic-block header, least significant bit first) that the block-gzip output of this context's profile uses.
 * Returns the number of 32-bit words of the prefix. */
int scs_test_deflate_code(const scs_ctx* ctx, uint8_t* lens257, uint32_t* prefix_words, int cap_words, uint32_t* prefix_bits);
/* The first n values of libc rand() after srand(seed), as reproduced by the library. */
int scs_test_libc_rand(uint32_t seed, int n, uint32_t* out);
/* Host-only: the expansion pool of host_expand on one packed slab without a GPU. `wire` is the slab as it leaves the device: nsplit
 * split entries (u64 wire offset, u64 text offset of every 2048th record slot), then wire_bytes bytes of records (wire.h).
 * Writes text_bytes bytes of FASTQ to out with `threads` threads; qchar0 = '!' + the profile's lowest quality index;
 * scalar != 0 forces the scalar expander. Returns 0, or SCS_E_ARG when the slab is malformed. */
int scs_test_expand_wire(const uint8_t* wire, uint32_t nsplit, uint64_t wire_bytes, uint64_t text_bytes, int qchar0, int threads, int scalar, char* out);

/* ---- replay ("recorded draws", BASELINE north_star correctness part 1) -------------------------
 * Tapes are the u32 logs of the patched reference run with -t 1; marks give, per entity, the tape
 * position of its first "real"-engine and "int"-engine draw (written by the CPU oracle). All
 * pointers are host memory, copied to the device by the call. */
typedef struct scs_replay {
    const uint32_t* wreal; uint64_t n_wreal;
    const uint32_t* wint; uint64_t n_wint;
    const uint32_t* mrand; uint64_t n_mrand;
    const uint32_t* mreal; uint64_t n_mreal;
    const double* gcf; uint64_t n_gcf;
    /* marks[d]: n_marks[d] triples (entity, off_real, off_int), domain numbering of scs_domain */
    const uint64_t* marks[8]; uint64_t n_marks[8];
} scs_replay;
enum scs_domain { SCS_D_FRAG = 0, SCS_D_POIS = 1, SCS_D_AMPF = 2, SCS_D_AMPS = 3, SCS_D_GCF = 4, SCS_D_MULTM = 5, SCS_D_MULTC = 6, SCS_D_READ = 7 };
int scs_set_replay(scs_ctx* ctx, const scs_replay* r);

/* ---- test hooks (SURVEY.md §8b "Inner seam 3") ------------------------------------------------- */
/* Copy device arrays to host for parity tests. what: */
enum scs_dump { SCS_DUMP_FRAGS = 0,    /* i64 x5: seq, start0, len, strand, primers */
                SCS_DUMP_SEMIS = 1,    /* u64 x6: gstart, rc, len, gc, primers, nerr */
                SCS_DUMP_FULLS = 2,    /* u64 x6 */
                SCS_DUMP_COUNTS = 3,   /* u32 per full amplicon: readNumbers */
                SCS_DUMP_WEIGHTS = 4,  /* f64 per full amplicon (normalised) */
                SCS_DUMP_PRIMER_COUNTS = 5, /* i64 x 65536 */
                SCS_DUMP_FULL_SEQ = 6  /* ASCII sequences of full amplicons, '\n' separated (arg = max count) */ };
/* Returns the number of bytes needed/written (negative on error). If buf is NULL only sizes. */
int64_t scs_dump(scs_ctx* ctx, int what, void* buf, uint64_t cap);

/* Profile::predict on the device for `n_reads` source windows of read_length ASCII bases each,
 * drawing from explicit per-read tapes (real[i*stride_real ...], ints[i*stride_int ...]). out_seq and
 * out_qual receive out_stride bytes per read; out_len the produced lengths. */
int scs_test_predict(scs_ctx* ctx, const char* src, int n_reads, int is_read1, const uint32_t* real, uint64_t stride_real,
                     const uint32_t* ints, uint64_t stride_int, char* out_seq, char* out_qual, int out_stride, int32_t* out_len);
/* One Philox4x32-10 block on the device (known-answer test). */
int scs_test_philox(scs_ctx* ctx, const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);
/* det_log on the device for n doubles. */
int scs_test_det_log(scs_ctx* ctx, const double* x, int n, double* out);
/* Threshold form of one CDF row: which/idx as in the profile (0 ins, 1 del, 2 isize, 3 subs1, 4 subs2,
 * 5 quality), row = bin. Writes up to cap u32 thresholds, returns the row's entry count; *eff gets the
 * number of entries that take part in the search (see DESIGN.md "thresholds"). Host-only (no GPU). */
int scs_profile_thresholds(const scs_ctx* ctx, int which, int idx, int row, uint32_t* out, int cap, int* eff);

/* Host-side shard arithmetic (no GPU needed): contiguous range [*lo, *hi) of `n` units for `rank`. */
void scs_shard_range(uint64_t n, int rank, int world, uint64_t* lo, uint64_t* hi);

/* Which contiguous run [*lo, *hi) of the cell's n sequences rank keeps when a FASTA (scs_load_genome) or a simulated cell
 * (scs_simuvars_to_genome) is sharded: cut where the cumulative length crosses rank/world of the total, sequence midpoints
 * decide, so every rank holds about the same number of bases. Host-only. */
void scs_shard_sequences(const uint64_t* lens, size_t n, int rank, int world, size_t* lo, size_t* hi);

const char* scs_version(void);
/* Number of CUDA devices visible to the library (0 when there is no usable driver). */
int scs_device_count(void);

#ifdef __cplusplus
}
#endif
#endif
