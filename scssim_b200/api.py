"""ctypes binding of libscssim_b200.so — the host-side mirror of the reference's `genreads` stages.

The reference drives the path through global singletons (/root/reference/src/scssim.cpp:46-66):
``genome.loadData(); profile.train(path); malbac.createFrags(); malbac.amplify();
malbac.yieldReads()``. :class:`GenReads` exposes the same calls with the same argument meaning
(flags of ``parseArgs_genReads``, src/scssim.cpp:285-404) and raises :class:`ScsError` carrying the
message the reference would have printed before ``exit(1)``.

There is no CPU fallback: if the CUDA library is missing this module raises at import of the
library, and every compute call fails without a GPU.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SCS_LIB_PATH") or os.path.join(_HERE, "libscssim_b200.so")   # SCS_LIB_PATH: A/B builds while tuning

SCS_OK, SCS_E_ARG, SCS_E_IO, SCS_E_CUDA, SCS_E_STATE, SCS_E_UNSUPPORTED, SCS_E_NOMEM = 0, -1, -2, -3, -4, -5, -6
D_FRAG, D_POIS, D_AMPF, D_AMPS, D_GCF, D_MULTM, D_MULTC, D_READ = range(8)
DUMP_FRAGS, DUMP_SEMIS, DUMP_FULLS, DUMP_COUNTS, DUMP_WEIGHTS, DUMP_PRIMER_COUNTS, DUMP_FULL_SEQ = range(7)


class ScsError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"[{code}] {msg}")
        self.code, self.msg = code, msg


class Params(C.Structure):
    _fields_ = [("primers", C.c_int64), ("gamma", C.c_double), ("coverage", C.c_double), ("isize", C.c_int32),
                ("paired", C.c_int32), ("seed", C.c_uint64), ("device", C.c_int32), ("rank", C.c_int32),
                ("world", C.c_int32), ("balance", C.c_int32), ("slab_bytes", C.c_uint64), ("io_threads", C.c_int32),
                ("ring_slabs", C.c_int32), ("gzip", C.c_int32), ("relay_device", C.c_int32), ("host_expand", C.c_int32),
                ("expand_threads", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [("n_sequences", C.c_uint64), ("genome_bases", C.c_uint64), ("n_frags", C.c_uint64), ("n_semis", C.c_uint64),
                ("n_fulls", C.c_uint64), ("n_semis_global", C.c_uint64), ("n_fulls_global", C.c_uint64),
                ("reads_requested", C.c_uint64), ("records", C.c_uint64), ("fastq_bytes", C.c_uint64 * 2),
                ("total_primers_left", C.c_uint64), ("kernel_launches", C.c_uint64), ("ms_pack", C.c_double),
                ("ms_amplify", C.c_double), ("ms_alloc", C.c_double), ("ms_reads", C.c_double),
                ("ms_reads_kernels", C.c_double), ("ms_emit_kernel", C.c_double), ("emit_launches", C.c_uint64),
                ("genome_window_bytes", C.c_uint64), ("plain_bytes", C.c_uint64 * 2), ("link_bytes", C.c_uint64 * 2),
                ("slabs_packed", C.c_uint64), ("slabs", C.c_uint64)]

    def as_dict(self):
        d = {}
        for name, _ in self._fields_:
            v = getattr(self, name)
            d[name] = list(v) if name in ("fastq_bytes", "plain_bytes", "link_bytes") else v
        return d


class SimuVarsParams(C.Structure):
    _fields_ = [("ploidy", C.c_int32), ("libc_seed", C.c_uint32), ("line_width", C.c_int32), ("ring_slabs", C.c_int32), ("gzip", C.c_int32), ("relay_device", C.c_int32)]


class SimuVarsStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("n_chroms", "n_haps", "n_segments", "n_pieces", "n_subs", "n_cnv", "n_snv", "n_ins", "n_del",
                                          "n_snp", "ref_bases", "out_bases", "out_bytes", "h2d_bytes", "normalize_bytes",
                                          "materialize_bytes", "launches")] + \
               [(n, C.c_double) for n in ("ms_read", "ms_plan", "ms_device", "ms_kernels", "ms_total")]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_}


class Replay(C.Structure):
    _fields_ = [("wreal", C.c_void_p), ("n_wreal", C.c_uint64), ("wint", C.c_void_p), ("n_wint", C.c_uint64),
                ("mrand", C.c_void_p), ("n_mrand", C.c_uint64), ("mreal", C.c_void_p), ("n_mreal", C.c_uint64),
                ("gcf", C.c_void_p), ("n_gcf", C.c_uint64), ("marks", C.c_void_p * 8), ("n_marks", C.c_uint64 * 8)]


SINK_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t)
AR_U64_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_uint64), C.c_size_t)
AR_F64_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_double), C.c_size_t)
AR_DEV_F64_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_size_t)
AR_DEV_I64_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_size_t)

# every symbol include/scssim_b200.h declares
EXPORTS = ["scs_default_params", "scs_create", "scs_destroy", "scs_last_error", "scs_load_profile", "scs_read_length",
           "scs_load_genome", "scs_set_genome", "scs_set_collectives", "scs_set_device_collective", "scs_set_shard_weight", "scs_create_frags", "scs_amplify",
           "scs_yield_reads_sink", "scs_yield_reads", "scs_plan_fastq_bytes", "scs_set_read_counts", "scs_get_stats", "scs_set_replay", "scs_dump",
           "scs_test_predict", "scs_test_philox", "scs_test_det_log", "scs_profile_thresholds", "scs_shard_range",
           "scs_version", "scs_device_count", "scs_nccl_unique_id", "scs_nccl_init", "scs_nccl_abort", "scs_nccl_version",
           "scs_simuvars_default_params", "scs_simuvars", "scs_simuvars_sink", "scs_simuvars_to_genome", "scs_simuvars_get_stats",
           "scs_simuvars_warnings", "scs_svplan_create", "scs_svplan_destroy", "scs_svplan_dump", "scs_test_libc_rand", "scs_shard_sequences", "scs_test_fasta_index", "scs_test_file_writer", "scs_test_async_writer", "scs_test_deflate_code",
           "scs_test_expand_wire"]

_lib = None


def lib():
    """Load the CUDA library; fails loudly when it has not been built (no fallback path exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(the genreads path is CUDA-only; there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        L.scs_last_error.restype = C.c_char_p
        L.scs_last_error.argtypes = [C.c_void_p]
        L.scs_version.restype = C.c_char_p
        L.scs_create.argtypes = [C.POINTER(Params), C.POINTER(C.c_void_p)]
        L.scs_destroy.argtypes = [C.c_void_p]
        L.scs_load_profile.argtypes = [C.c_void_p, C.c_char_p]
        L.scs_read_length.argtypes = [C.c_void_p]
        L.scs_load_genome.argtypes = [C.c_void_p, C.c_char_p]
        L.scs_set_genome.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
        L.scs_set_collectives.argtypes = [C.c_void_p, AR_U64_FN, AR_F64_FN, C.c_void_p]
        L.scs_set_device_collective.argtypes = [C.c_void_p, AR_DEV_F64_FN, AR_DEV_I64_FN, C.c_void_p]
        L.scs_set_shard_weight.argtypes = [C.c_void_p, C.c_double]
        L.scs_nccl_unique_id.argtypes = [C.c_char_p]
        L.scs_nccl_init.argtypes = [C.c_void_p, C.c_char_p]
        L.scs_nccl_abort.argtypes = [C.c_void_p]
        for f in ("scs_create_frags", "scs_amplify", "scs_set_read_counts"):
            getattr(L, f).argtypes = [C.c_void_p]
        L.scs_yield_reads_sink.argtypes = [C.c_void_p, SINK_FN, C.c_void_p]
        L.scs_yield_reads.argtypes = [C.c_void_p, C.c_char_p]
        L.scs_plan_fastq_bytes.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
        L.scs_get_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
        L.scs_set_replay.argtypes = [C.c_void_p, C.POINTER(Replay)]
        L.scs_dump.restype = C.c_int64
        L.scs_dump.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64]
        L.scs_test_predict.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64,
                                       C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.scs_test_philox.argtypes = [C.c_void_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
        L.scs_test_det_log.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.scs_profile_thresholds.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        L.scs_shard_range.argtypes = [C.c_uint64, C.c_int, C.c_int, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        L.scs_shard_range.restype = None
        L.scs_simuvars_default_params.argtypes = [C.POINTER(SimuVarsParams)]
        L.scs_simuvars_default_params.restype = None
        L.scs_simuvars.argtypes = [C.c_void_p, C.POINTER(SimuVarsParams), C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p]
        L.scs_simuvars_sink.argtypes = [C.c_void_p, C.POINTER(SimuVarsParams), C.c_char_p, C.c_char_p, C.c_char_p, SINK_FN, C.c_void_p]
        L.scs_simuvars_to_genome.argtypes = [C.c_void_p, C.POINTER(SimuVarsParams), C.c_char_p, C.c_char_p, C.c_char_p]
        L.scs_simuvars_get_stats.argtypes = [C.c_void_p, C.POINTER(SimuVarsStats)]
        L.scs_simuvars_warnings.argtypes = [C.c_void_p]
        L.scs_simuvars_warnings.restype = C.c_char_p
        L.scs_svplan_create.restype = C.c_void_p
        L.scs_svplan_create.argtypes = [C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_uint64), C.c_char_p, C.c_char_p, C.c_int, C.c_uint32,
                                        C.c_char_p, C.c_size_t]
        L.scs_svplan_destroy.argtypes = [C.c_void_p]
        L.scs_svplan_destroy.restype = None
        L.scs_svplan_dump.restype = C.c_int64
        L.scs_svplan_dump.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64]
        L.scs_test_libc_rand.argtypes = [C.c_uint32, C.c_int, C.c_void_p]
        L.scs_shard_sequences.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
        L.scs_shard_sequences.restype = None
        L.scs_test_fasta_index.restype = C.c_int64
        L.scs_test_fasta_index.argtypes = [C.c_char_p, C.c_void_p, C.c_uint64, C.c_char_p, C.c_uint64]
        L.scs_test_file_writer.argtypes = [C.c_char_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_int]
        L.scs_test_async_writer.argtypes = [C.c_char_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.c_uint64, C.c_int, C.c_uint64, C.c_int,
                                            C.POINTER(C.c_int)]
        _lib = L
    return _lib


def nccl_unique_id() -> bytes:
    buf = C.create_string_buffer(128)
    rc = lib().scs_nccl_unique_id(buf)
    if rc != SCS_OK:
        raise ScsError(rc, lib().scs_last_error(None).decode())
    return buf.raw


def shard_range(n: int, rank: int, world: int):
    lo, hi = C.c_uint64(), C.c_uint64()
    lib().scs_shard_range(n, rank, world, C.byref(lo), C.byref(hi))
    return lo.value, hi.value


def fasta_index(path: str):
    """[(name, length, offset, bases per line, bytes per line, regular)] as the loaders index a FASTA file (host only)."""
    n = lib().scs_test_fasta_index(path.encode(), None, 0, None, 0)
    if n < 0:
        raise ScsError(int(n), f"could not open {path}")
    recs = np.zeros((max(int(n), 1), 5), dtype=np.uint64)
    names = C.create_string_buffer(1 << 20)
    lib().scs_test_fasta_index(path.encode(), recs.ctypes.data, n, names, len(names))
    nm = names.value.decode().split("\n")[:-1]
    return [(nm[i],) + tuple(int(x) for x in recs[i]) for i in range(int(n))]


def write_file_parallel(path: str, data: bytes, slab_bytes: int, threads: int) -> None:
    rc = lib().scs_test_file_writer(path.encode(), data, len(data), slab_bytes, threads)
    if rc != SCS_OK:
        raise ScsError(rc, f"can not write {path}")


def expand_wire(wire: bytes, nsplit: int, text_bytes: int, qchar0: int = 33, threads: int = 1, scalar: bool = False) -> bytes:
    """Expand one packed FASTQ slab (scssim_b200/csrc/wire.h: nsplit 16-byte split entries, then the records) with the host
    expansion pool of host_expand (host only). Returns the text_bytes bytes of FASTQ."""
    out = C.create_string_buffer(max(int(text_bytes), 1))
    lib().scs_test_expand_wire.argtypes = [C.c_char_p, C.c_uint32, C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_void_p]
    rc = lib().scs_test_expand_wire(wire, nsplit, len(wire) - 16 * nsplit, text_bytes, qchar0, threads, int(scalar), out)
    if rc != SCS_OK:
        raise ScsError(rc, "malformed packed slab")
    return out.raw[:text_bytes]


def write_file_async(path: str, data: bytes, slab_bytes: int, threads: int = 4, ring: int = 4, base: int = 0, create: bool = True, prealloc: int = 0,
                     direct: bool = True) -> bool:
    """Feed `data` through the asynchronous file sink of scs_yield_reads (host only). Returns whether O_DIRECT was in use."""
    used = C.c_int(0)
    rc = lib().scs_test_async_writer(path.encode(), data, len(data), slab_bytes, threads, ring, base, int(create), prealloc, int(direct), C.byref(used))
    if rc != SCS_OK:
        raise ScsError(rc, f"can not write {path}")
    return bool(used.value)


def shard_sequences(lens, rank: int, world: int):
    """[lo, hi) of the sequences `rank` keeps when a cell of these sequence lengths is sharded over `world` GPUs."""
    a = np.ascontiguousarray(lens, dtype=np.uint64)
    lo, hi = C.c_size_t(), C.c_size_t()
    lib().scs_shard_sequences(a.ctypes.data, len(a), rank, world, C.byref(lo), C.byref(hi))
    return lo.value, hi.value


@dataclass
class ReplayTapes:
    """Draw logs of `oracle/_ref/bin/scssim_replay -t 1` plus the per-entity offsets the CPU oracle wrote."""
    wreal: np.ndarray
    wint: np.ndarray
    mrand: np.ndarray
    mreal: np.ndarray
    gcf: np.ndarray
    marks: list  # 8 arrays (n,3) uint64

    @staticmethod
    def load(tape_prefix: str, dump_prefix: str) -> "ReplayTapes":
        t = lambda n: np.fromfile(f"{tape_prefix}.{n}.bin", dtype=np.uint32)
        marks = [np.fromfile(f"{dump_prefix}.marks{d}.u64", dtype=np.uint64).reshape(-1, 3) for d in range(8)]
        return ReplayTapes(t("wreal"), t("wint"), t("mrand"), t("mreal"),
                           np.fromfile(f"{tape_prefix}.gcf.bin", dtype=np.float64), marks)


class GenReads:
    """One `scssim genreads` run on one GPU (one shard when world > 1)."""

    def __init__(self, primers: int = 100000, gamma: float = 1e-9, coverage: float = 5.0, isize: int = 260,
                 layout: str = "PE", seed: int = 0x5C55, device: int = 0, rank: int = 0, world: int = 1,
                 slab_bytes: int = 0, balance: bool = False, io_threads: int = 0, ring_slabs: int = 0, gzip: bool = False, relay_device: int = -1,
                 host_expand: int = -1, expand_threads: int = 0):
        if layout not in ("SE", "PE"):
            raise ScsError(SCS_E_ARG, "Error: sequence layout incorrectly specified!\nshould be SE (single end) or PE (paired-end)")
        L = lib()
        p = Params()
        L.scs_default_params(C.byref(p))
        p.primers, p.gamma, p.coverage, p.isize = primers, gamma, coverage, isize
        p.paired, p.seed, p.device, p.rank, p.world, p.slab_bytes = int(layout == "PE"), seed, device, rank, world, slab_bytes
        p.balance = int(balance)
        p.io_threads = io_threads
        p.ring_slabs = ring_slabs
        p.gzip = int(gzip)
        p.relay_device = relay_device
        p.host_expand = host_expand
        p.expand_threads = expand_threads
        self._h = C.c_void_p()
        rc = L.scs_create(C.byref(p), C.byref(self._h))
        if rc != SCS_OK:
            raise ScsError(rc, L.scs_last_error(None).decode())
        self.paired = layout == "PE"
        self._keep = []

    def close(self):
        if getattr(self, "_h", None):
            lib().scs_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _ck(self, rc):
        if rc < 0:
            raise ScsError(int(rc), lib().scs_last_error(self._h).decode())
        return rc

    # --- the reference's stage calls -------------------------------------------------------------
    def load_profile(self, path: str):          # profile.train(file)
        self._ck(lib().scs_load_profile(self._h, path.encode()))
        return self

    @property
    def read_length(self) -> int:
        return lib().scs_read_length(self._h)

    def load_genome(self, fasta_path: str):     # genome.loadData()
        self._ck(lib().scs_load_genome(self._h, fasta_path.encode()))
        return self

    def set_genome(self, named_seqs):
        """named_seqs: list of (name, uint8 ASCII array)."""
        n = len(named_seqs)
        names = (C.c_char_p * n)(*[nm.encode() for nm, _ in named_seqs])
        arrs = [np.ascontiguousarray(s, dtype=np.uint8) for _, s in named_seqs]
        ptrs = (C.c_void_p * n)(*[a.ctypes.data for a in arrs])
        lens = (C.c_uint64 * n)(*[len(a) for a in arrs])
        self._ck(lib().scs_set_genome(self._h, n, names, ptrs, lens))
        return self

    def set_replay(self, t: ReplayTapes):
        r = Replay()
        keep = [np.ascontiguousarray(a) for a in (t.wreal, t.wint, t.mrand, t.mreal, t.gcf)]
        for name, a in zip(("wreal", "wint", "mrand", "mreal", "gcf"), keep):
            setattr(r, name, a.ctypes.data)
            setattr(r, "n_" + name, len(a))
        mk = [np.ascontiguousarray(m, dtype=np.uint64) for m in t.marks]
        for d in range(8):
            r.marks[d] = mk[d].ctypes.data
            r.n_marks[d] = len(mk[d])
        self._ck(lib().scs_set_replay(self._h, C.byref(r)))
        return self

    def set_collectives(self, allreduce_u64, allreduce_f64):
        """allreduce_*(np.ndarray) -> None, in place (sum over ranks)."""
        def fu(_u, buf, n):
            a = np.ctypeslib.as_array(buf, shape=(n,))
            allreduce_u64(a)
            return 0

        def fd(_u, buf, n):
            a = np.ctypeslib.as_array(buf, shape=(n,))
            allreduce_f64(a)
            return 0
        self._cb = (AR_U64_FN(fu), AR_F64_FN(fd))
        self._ck(lib().scs_set_collectives(self._h, self._cb[0], self._cb[1], None))
        return self

    def set_device_collective(self, allreduce_dev_f64, allreduce_dev_i64):
        """allreduce_dev_*(device_pointer: int, n: int) -> None, in place on device memory."""
        def fd(_u, ptr, n):
            allreduce_dev_f64(int(ptr), int(n))
            return 0

        def fi(_u, ptr, n):
            allreduce_dev_i64(int(ptr), int(n))
            return 0
        self._cb_dev = (AR_DEV_F64_FN(fd), AR_DEV_I64_FN(fi))
        self._ck(lib().scs_set_device_collective(self._h, self._cb_dev[0], self._cb_dev[1], None))
        return self

    def nccl_init(self, unique_id: bytes):
        """Collective: join the communicator named by `unique_id` (from nccl_unique_id() on rank 0); the library then runs all of its
        collectives on NCCL itself and needs no hooks."""
        assert len(unique_id) == 128
        self._ck(lib().scs_nccl_init(self._h, unique_id))
        return self

    def set_shard_weight(self, w: float):
        self._ck(lib().scs_set_shard_weight(self._h, float(w)))
        return self

    def create_frags(self):                     # malbac.createFrags()
        self._ck(lib().scs_create_frags(self._h))
        return self

    def amplify(self):                          # malbac.amplify()
        self._ck(lib().scs_amplify(self._h))
        return self

    def set_read_counts(self):
        self._ck(lib().scs_set_read_counts(self._h))
        return self

    def yield_reads(self, prefix: str):         # malbac.yieldReads() -> <prefix>_1.fq/_2.fq | <prefix>.fq
        self._ck(lib().scs_yield_reads(self._h, prefix.encode()))
        return self

    def plan_fastq_bytes(self):
        """Exact FASTQ bytes this rank will write to each file (sizing pass)."""
        b = (C.c_uint64 * 2)()
        self._ck(lib().scs_plan_fastq_bytes(self._h, b))
        return [int(b[0]), int(b[1])]

    def yield_reads_bytes(self):
        """FASTQ text of both files as bytes (tests; small runs)."""
        parts = ([], [])

        def sink(_u, f, data, n):
            parts[f].append(C.string_at(data, n))
            return 0
        cb = SINK_FN(sink)
        self._ck(lib().scs_yield_reads_sink(self._h, cb, None))
        return b"".join(parts[0]), b"".join(parts[1])

    def yield_reads_discard(self):
        """Run the read stage with output landing in the pinned host ring only (bench)."""
        self._ck(lib().scs_yield_reads_sink(self._h, C.cast(None, SINK_FN), None))
        return self

    def yield_reads_into(self, bufs):
        """Copy FASTQ bytes into caller-provided host arrays (one per file); returns bytes written per file."""
        pos = [0, 0]
        ptrs = [b.ctypes.data for b in bufs]
        caps = [b.nbytes for b in bufs]

        def sink(_u, f, data, n):
            if pos[f] + n > caps[f]:
                return 1
            C.memmove(ptrs[f] + pos[f], data, n)
            pos[f] += n
            return 0
        cb = SINK_FN(sink)
        self._ck(lib().scs_yield_reads_sink(self._h, cb, None))
        return pos

    # --- simuvars (the reference's other producer subcommand; SURVEY §8f N1) -----------------------
    def _sv_params(self, ploidy, libc_seed, line_width):
        p = SimuVarsParams()
        lib().scs_simuvars_default_params(C.byref(p))
        p.ploidy, p.libc_seed, p.line_width = ploidy, libc_seed, line_width
        return p

    def simuvars(self, ref: str, snp: str | None, var: str | None, out: str, ploidy: int = 2, libc_seed: int = 1, line_width: int = 100):
        """`scssim simuvars -r ref -s snp -v var -o out` (genome.loadData(); genome.saveSequence())."""
        p = self._sv_params(ploidy, libc_seed, line_width)
        self._ck(lib().scs_simuvars(self._h, C.byref(p), ref.encode(), (snp or "").encode(), (var or "").encode(), out.encode()))
        return self

    def simuvars_bytes(self, ref: str, snp: str | None, var: str | None, ploidy: int = 2, libc_seed: int = 1, line_width: int = 100,
                       discard: bool = False):
        """The output FASTA as bytes (tests), or only its length when discard=True (bench: bytes land in pinned memory)."""
        parts, total = [], [0]

        def sink(_u, _f, data, n):
            total[0] += n
            if not discard:
                parts.append(C.string_at(data, n))
            return 0
        cb = SINK_FN(sink)
        p = self._sv_params(ploidy, libc_seed, line_width)
        self._ck(lib().scs_simuvars_sink(self._h, C.byref(p), ref.encode(), (snp or "").encode(), (var or "").encode(), cb, None))
        return total[0] if discard else b"".join(parts)

    def simuvars_to_genome(self, ref: str, snp: str | None, var: str | None, ploidy: int = 2, libc_seed: int = 1):
        """simuvars whose output stays on the device as this context's packed genome (no FASTA round trip)."""
        p = self._sv_params(ploidy, libc_seed, 100)
        self._ck(lib().scs_simuvars_to_genome(self._h, C.byref(p), ref.encode(), (snp or "").encode(), (var or "").encode()))
        return self

    def simuvars_stats(self) -> dict:
        s = SimuVarsStats()
        self._ck(lib().scs_simuvars_get_stats(self._h, C.byref(s)))
        d = s.as_dict()
        d["warnings"] = lib().scs_simuvars_warnings(self._h).decode()
        return d

    def stats(self) -> dict:
        s = Stats()
        self._ck(lib().scs_get_stats(self._h, C.byref(s)))
        return s.as_dict()

    # --- test hooks -------------------------------------------------------------------------------
    def dump(self, what: int) -> np.ndarray:
        n = self._ck(lib().scs_dump(self._h, what, None, 0))
        buf = np.zeros(max(int(n), 1), dtype=np.uint8)
        self._ck(lib().scs_dump(self._h, what, buf.ctypes.data, buf.nbytes))
        buf = buf[:n]
        if what == DUMP_FRAGS:
            return buf.view(np.int64).reshape(-1, 5)
        if what in (DUMP_SEMIS, DUMP_FULLS):
            return buf.view(np.uint64).reshape(-1, 6)
        if what == DUMP_COUNTS:
            return buf.view(np.uint32)
        if what == DUMP_WEIGHTS:
            return buf.view(np.float64)
        if what == DUMP_PRIMER_COUNTS:
            return buf.view(np.int64)
        return buf

    def test_predict(self, src: np.ndarray, is_read1: bool, real: np.ndarray, ints: np.ndarray, out_stride: int = 384):
        """src: (n, RL) uint8 ASCII; real/ints: (n, stride) uint32 tapes. Returns (seqs, quals, lens)."""
        n = src.shape[0]
        src = np.ascontiguousarray(src, dtype=np.uint8)
        real = np.ascontiguousarray(real, dtype=np.uint32)
        ints = np.ascontiguousarray(ints, dtype=np.uint32)
        oseq = np.zeros((n, out_stride), dtype=np.uint8)
        oqual = np.zeros((n, out_stride), dtype=np.uint8)
        olen = np.zeros(n, dtype=np.int32)
        self._ck(lib().scs_test_predict(self._h, src.ctypes.data_as(C.c_char_p), n, int(is_read1), real.ctypes.data, real.shape[1],
                                        ints.ctypes.data, ints.shape[1], oseq.ctypes.data, oqual.ctypes.data, out_stride,
                                        olen.ctypes.data))
        return oseq, oqual, olen

    def test_philox(self, ctr, key):
        c = (C.c_uint32 * 4)(*ctr)
        k = (C.c_uint32 * 2)(*key)
        o = (C.c_uint32 * 4)()
        self._ck(lib().scs_test_philox(self._h, c, k, o))
        return list(o)

    def test_det_log(self, x: np.ndarray) -> np.ndarray:
        x = np.ascontiguousarray(x, dtype=np.float64)
        out = np.zeros_like(x)
        self._ck(lib().scs_test_det_log(self._h, x.ctypes.data, len(x), out.ctypes.data))
        return out

    def deflate_code(self):
        """(code lengths [257], prefix bytes, prefix bit count) of the block-gzip output for this profile (host only)."""
        lens = np.zeros(257, dtype=np.uint8)
        words = np.zeros(256, dtype=np.uint32)
        nbits = C.c_uint32()
        lib().scs_test_deflate_code.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_uint32)]
        self._ck(lib().scs_test_deflate_code(self._h, lens.ctypes.data, words.ctypes.data, len(words), C.byref(nbits)))
        return lens, words, int(nbits.value)

    def thresholds(self, which: int, idx: int = 0, row: int = 0):
        out = np.zeros(4096, dtype=np.uint32)
        eff = C.c_int()
        n = self._ck(lib().scs_profile_thresholds(self._h, which, idx, row, out.ctypes.data, 4096, C.byref(eff)))
        return out[:n].copy(), eff.value


# --- simuvars edit plan, host only (test hook) ---------------------------------------------------------
SVP_HAPS, SVP_PIECES, SVP_SUBS, SVP_LITERALS, SVP_NAMES, SVP_WARNINGS = range(6)
SV_LITERAL = 1 << 63


class SimuVarsPlan:
    """The edit plan `scs_simuvars*` hands to the GPU, built on the host: per haplotype a list of copy runs
    (out offset, source, length) over the chromosome / the pool of inserted sequences and a list of point substitutions."""

    def __init__(self, chroms, snp: str | None, var: str | None, ploidy: int = 2, libc_seed: int = 1):
        """chroms: list of (name without "chr", length)."""
        n = len(chroms)
        names = (C.c_char_p * n)(*[nm.encode() for nm, _ in chroms])
        lens = (C.c_uint64 * n)(*[int(l) for _, l in chroms])
        err = C.create_string_buffer(1024)
        self._h = lib().scs_svplan_create(n, names, lens, (snp or "").encode(), (var or "").encode(), ploidy, libc_seed, err, 1024)
        if not self._h:
            raise ScsError(SCS_E_IO, err.value.decode())

    def _dump(self, what):
        n = lib().scs_svplan_dump(self._h, what, None, 0)
        buf = np.zeros(max(int(n), 1), dtype=np.uint8)
        lib().scs_svplan_dump(self._h, what, buf.ctypes.data, buf.nbytes)
        return buf[:n]

    @property
    def haps(self):
        return self._dump(SVP_HAPS).view(np.uint64).reshape(-1, 7)

    @property
    def pieces(self):
        return self._dump(SVP_PIECES).view(np.uint64).reshape(-1, 3)

    @property
    def subs(self):
        return self._dump(SVP_SUBS).view(np.uint64).reshape(-1, 2)

    @property
    def literals(self):
        return self._dump(SVP_LITERALS)

    @property
    def names(self):
        return self._dump(SVP_NAMES).tobytes().decode().split("\n")[:-1]

    @property
    def warnings(self):
        return self._dump(SVP_WARNINGS).tobytes().decode()

    def close(self):
        if getattr(self, "_h", None):
            lib().scs_svplan_destroy(self._h)
            self._h = None

    __del__ = close


def libc_rand(seed: int, n: int) -> np.ndarray:
    out = np.zeros(n, dtype=np.uint32)
    lib().scs_test_libc_rand(seed, n, out.ctypes.data)
    return out
