"""CPU tests of the product's host side: the C-ABI library loads and exports every declared symbol, the
.profile parser + integer threshold tables agree exactly with the oracle's FP64 CDF sampling, shard
arithmetic, flag validation. No compute call is made (there is no GPU here and no CPU fallback)."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import helpers as H
from scssim_b200 import api

EPS = 2.2204e-16


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(H.ROOT, "include", "scssim_b200.h")).read()
    declared = set(re.findall(r"\b(scs_[a-z0-9_]+)\s*\(", hdr)) - {"scs_sink_fn", "scs_allreduce_u64_fn", "scs_allreduce_f64_fn"}
    L = api.lib()
    missing = [s for s in sorted(declared) if not hasattr(L, s)]
    assert not missing, missing
    assert set(api.EXPORTS) == declared
    assert b"sm_100a" in L.scs_version()


def test_no_device_means_failure_not_fallback():
    with pytest.raises(api.ScsError) as e:
        g = api.GenReads(device=-1)
        g.load_profile(H.profile_path("Illumina_HiSeq2500"))
        g.set_genome([("chrS1_1_100", np.frombuffer(b"ACGT" * 25, dtype=np.uint8))])
    assert e.value.code == api.SCS_E_CUDA and "no CPU fallback" in e.value.msg


def test_flag_validation_messages_match_reference():
    for kw, msg in [(dict(primers=10), 'Error: the value of parameter "primers" should be at least 1000!'),
                    (dict(gamma=1e-7), 'Error: the value of parameter "gamma" should be in 0~1e-8!'),
                    (dict(coverage=0.0), "Error: sequencing coverage not properly specified!"),
                    (dict(layout="XX"), "Error: sequence layout incorrectly specified!")]:
        with pytest.raises(api.ScsError) as e:
            api.GenReads(device=-1, **kw)
        assert msg in e.value.msg


def _r(x):  # ThreadPool::randomDouble(ZERO_FINAL, 1) on a 32-bit engine output
    return EPS + (1.0 - EPS) * (np.asarray(x, dtype=np.float64) / 4294967296.0)


def _ref_index(cdf, x):  # randIndx, MyDefine.cpp:274-282
    r = _r(x)
    k = np.searchsorted(cdf, r, side="left")  # first k with r <= cdf[k]
    return np.minimum(k, len(cdf) - 1)


def _thr_index(thr, eff, x):
    k = np.searchsorted(thr[:eff], x, side="right")  # number of thresholds <= x
    return np.minimum(k, eff)


@pytest.mark.parametrize("profile", H.PROFILES)
def test_threshold_tables_equal_fp64_sampling(profile):
    """For every CDF row, sampling by integer thresholds == the reference's FP64 comparison, checked at the
    draws around every cut point and at random draws."""
    L = H.oracle_lib()
    path = H.profile_path(profile)
    err = C.create_string_buffer(256)
    op = L.orc_profile_load(path.encode(), 1, 260, err, 256)
    assert op, err.value
    info = (C.c_int * 9)()
    L.orc_profile_info(op, info)
    RL, kmers = info[0], info[2]
    g = api.GenReads(device=-1, layout="PE", isize=260).load_profile(path)
    assert g.read_length == RL
    rng = np.random.default_rng(7)
    buf = np.zeros(RL * 94 + 4096, dtype=np.float64)

    def check(which, idx, rows, cols):
        n = L.orc_profile_cdf(op, which, idx, buf.ctypes.data)
        assert n == rows * cols
        cdfs = buf[:n].reshape(rows, cols).copy()
        for row in (range(rows) if rows <= 8 else rng.choice(rows, 8, replace=False)):
            thr, eff = g.thresholds(which, idx, int(row))
            if which in (3, 4):
                thr = thr[:3]
            cuts = thr[:eff].astype(np.int64)
            xs = np.unique(np.clip(np.concatenate([cuts - 1, cuts, cuts + 1, rng.integers(0, 2 ** 32, 4000), [0, 2 ** 32 - 1]]), 0, 2 ** 32 - 1)).astype(np.uint32)
            want = _ref_index(cdfs[row], xs)
            got = _thr_index(thr.astype(np.uint32), eff, xs)
            assert np.array_equal(got, want), (profile, which, idx, row)

    check(0, 0, 1, info[6]); check(1, 0, 1, info[7]); check(2, 0, 1, info[5])
    for ki in rng.choice(kmers, 6, replace=False):
        check(3, int(ki), RL, 4); check(4, int(ki), RL, 4)
    for bp in range(16):
        check(5, bp, RL, 94)
    L.orc_profile_free(op)


def test_shard_ranges_partition_everything():
    for n in (0, 1, 7, 8, 1000, 123457):
        for world in (1, 2, 3, 8):
            prev = 0
            for r in range(world):
                lo, hi = api.shard_range(n, r, world)
                assert lo == prev and hi >= lo and hi - lo in (n // world, n // world + 1)
                prev = hi
            assert prev == n


def test_cli_rejects_bad_flags_like_the_reference():
    exe = os.path.join(H.ROOT, "scssim_b200", "bin", "scssim")
    if not os.path.exists(exe):
        pytest.skip("CLI not built")
    r = subprocess.run([exe, "genreads", "-i", "x.fa", "-m", "m.profile", "-o", "out", "-r", "1"], capture_output=True)
    assert r.returncode == 1 and b'"gamma" should be in 0~1e-8' in r.stderr
    r = subprocess.run([exe, "genreads", "-m", "m.profile", "-o", "out"], capture_output=True)
    assert r.returncode == 1 and b"reference file (.fasta) not specified" in r.stderr
    r = subprocess.run([exe, "genreads", "-i", "x.fa", "-m", "m.profile", "-o", "out", "-l", "XX"], capture_output=True)
    assert r.returncode == 1 and b"sequence layout incorrectly specified" in r.stderr


def test_resampled_profile_is_a_valid_profile(tmp_path):
    """bench.py derives a 150-bin profile from the shipped 125-bin HiSeq2500 one (read length is a property of the
    .profile); both parsers must accept it and row j of the new tables must equal row floor(j*125/150) of the old ones."""
    from scssim_b200.tools.resample_profile import resample
    src = H.profile_path("Illumina_HiSeq2500")
    dst = os.path.join(str(tmp_path), "hs2500_150.profile")
    resample(src, dst, 150)
    g_old = api.GenReads(device=-1).load_profile(src)
    g_new = api.GenReads(device=-1).load_profile(dst)
    assert g_old.read_length == 125 and g_new.read_length == 150
    for j in (0, 1, 37, 88, 149):
        for which, idx in ((3, 25), (4, 60), (5, 0), (5, 10)):
            a, ea = g_new.thresholds(which, idx, j)
            b, eb = g_old.thresholds(which, idx, j * 125 // 150)
            assert ea == eb and np.array_equal(a, b)
    L = H.oracle_lib()
    err = C.create_string_buffer(256)
    op = L.orc_profile_load(dst.encode(), 1, 260, err, 256)
    assert op, err.value
    info = (C.c_int * 9)()
    L.orc_profile_info(op, info)
    assert info[0] == 150 and info[1] == 150
    L.orc_profile_free(op)


def test_fasta_index_matches_samtools_fai_model(tmp_path):
    """The host FASTA reader (mmap + record-parallel indexing): names, lengths, offsets and line geometry as in a .fai
    (lib/fastahack/Fasta.cpp:103-191), for fixed-width, single-line, CRLF, ragged and unterminated records and a file big
    enough (> 64 MB) to take the threaded path."""
    import numpy as np
    from scssim_b200.synth import synth_sequence
    d = str(tmp_path)
    a, b, c, e = synth_sequence(1000, 1), synth_sequence(77, 2), synth_sequence(250, 3), synth_sequence(130, 4)
    path = os.path.join(d, "mix.fa")
    with open(path, "wb") as f:
        f.write(b">chr1 some description\n" + b"".join(a[i:i + 60].tobytes() + b"\n" for i in range(0, 1000, 60)))
        f.write(b">single\n" + b.tobytes() + b"\n")
        f.write(b">crlf\r\n" + b"".join(c[i:i + 50].tobytes() + b"\r\n" for i in range(0, 250, 50)))
        f.write(b">ragged\n" + e[:40].tobytes() + b"\n" + e[40:100].tobytes() + b"\n" + e[100:].tobytes() + b"\n")
        f.write(b">empty\n>last_no_newline\nACGTACGTAC\nACG")
    idx = api.fasta_index(path)
    assert [r[0] for r in idx] == ["chr1", "single", "crlf", "ragged", "empty", "last_no_newline"]
    assert [r[1] for r in idx] == [1000, 77, 250, 130, 0, 13]
    raw = open(path, "rb").read()
    for name, length, off, blen, llen, regular in idx:
        if length:
            assert raw[off - 1:off] == b"\n" and raw[off:off + 1] in b"ACGT"
    assert idx[0][3:] == (60, 61, 1) and idx[1][3:] == (77, 78, 1) and idx[2][3:] == (50, 52, 1)
    assert idx[3][5] == 0                      # a longer line after a shorter one: not a uniform geometry
    assert idx[5][3:] == (10, 11, 1)
    big = os.path.join(d, "big.fa")
    s = synth_sequence(12_000_000, 9)
    from scssim_b200.synth import write_fasta
    write_fasta(big, [(f"chrB{i}_1_{len(s) - 1000 * i}", s[:len(s) - 1000 * i]) for i in range(7)], 100)
    assert os.path.getsize(big) > 64 << 20
    idx = api.fasta_index(big)
    assert [r[1] for r in idx] == [len(s) - 1000 * i for i in range(7)] and all(r[3:] == (100, 101, 1) for r in idx)
    raw = np.fromfile(big, dtype=np.uint8)
    for i, r in enumerate(idx):
        assert bytes(raw[r[2] - len(r[0]) - 2:r[2]]) == b">" + r[0].encode() + b"\n"
        assert bytes(raw[r[2]:r[2] + 100]) == s[:100].tobytes()


def test_parallel_file_writer_round_trip(tmp_path):
    """The pwrite pool behind scs_yield_reads / scs_simuvars: slabs of odd sizes, 1..8 threads, bytes land in order."""
    import numpy as np
    data = np.random.default_rng(3).integers(0, 256, size=9_000_001, dtype=np.uint8).tobytes()
    for threads, slab in [(1, 1 << 20), (3, 4_194_303), (8, 5_000_000), (4, 64 << 20)]:
        p = os.path.join(str(tmp_path), f"w{threads}.bin")
        api.write_file_parallel(p, data, slab, threads)
        assert open(p, "rb").read() == data
    with pytest.raises(api.ScsError):
        api.write_file_parallel(os.path.join(str(tmp_path), "no_such_dir", "x"), b"abc", 16, 2)


def test_async_file_sink_writes_exact_bytes(tmp_path):
    """The asynchronous sink behind scs_yield_reads (file_sink.h): slabs of awkward sizes through a small ring, O_DIRECT where the
    file system grants it (whole blocks direct, < 4 KiB carried from slab to slab, the last partial block buffered) and plain
    buffered writes; preallocation larger and smaller than the data; the file must hold exactly the bytes fed."""
    rng = np.random.default_rng(11)
    data = rng.integers(0, 256, size=3_000_017, dtype=np.uint8).tobytes()
    modes = set()
    for direct in (True, False):
        for slab, ring, threads, prealloc in [(4096, 2, 1, 0), (5000, 3, 4, 10_000_000), (65_537, 4, 3, 1000), (1 << 20, 2, 8, len(data)), (len(data) + 5, 2, 2, 0)]:
            p = os.path.join(str(tmp_path), f"a{int(direct)}_{slab}.bin")
            used = api.write_file_async(p, data, slab, threads=threads, ring=ring, prealloc=prealloc, direct=direct)
            modes.add(used)
            got = open(p, "rb").read()
            if prealloc > len(data):
                assert len(got) == prealloc and got[len(data):] == bytes(prealloc - len(data))   # the test hook does not own the end
                got = got[:len(data)]
            assert got == data, (direct, slab, ring, threads)
    assert False in modes
    with pytest.raises(api.ScsError):
        api.write_file_async(os.path.join(str(tmp_path), "no_such_dir", "x"), b"abc", 16)


def test_async_file_sink_ranks_share_one_file(tmp_path):
    """Several ranks write disjoint regions of ONE file at unaligned offsets (scs_yield_reads with world > 1): the first rank creates
    and preallocates it, the others open it; a block shared by two regions is written through the page cache by both."""
    rng = np.random.default_rng(12)
    parts = [rng.integers(0, 256, size=n, dtype=np.uint8).tobytes() for n in (1_234_567, 5, 70_001, 4096, 900_000)]
    total = sum(len(x) for x in parts)
    for direct in (True, False):
        p = os.path.join(str(tmp_path), f"shared{int(direct)}.bin")
        api.write_file_async(p, b"", 4096, create=True, prealloc=total, direct=direct)
        off = [sum(len(x) for x in parts[:i]) for i in range(len(parts))]
        for i in (3, 0, 4, 2, 1):   # any order
            api.write_file_async(p, parts[i], 50_000, threads=2, ring=3, base=off[i], create=False, direct=direct)
        assert open(p, "rb").read() == b"".join(parts)


def test_deflate_code_of_a_profile_is_a_valid_dynamic_block():
    """Host side of the block-gzip output (deflate_host.cpp): for every shipped profile the library's canonical Huffman code is
    complete and <= 15 bits, covers every byte FASTQ text can hold, and its constant block prefix (BGZF member header + dynamic
    Huffman header) followed by codes encoded here in Python is accepted by zlib and decodes to the input."""
    import gzip
    import zlib
    text = (b"@123456#78/1\nACGTNACGTTTGACCA\n+\n!\"#$%&'()*+,-./0123456789:;<=>?@ABCDEFGHIJ~\n" * 40)
    for prof, paired in [("Illumina_HiSeq2500", True), ("Illumina_HiSeqXTen", True), ("Illumina_GenomeAnalyzerIIx", False)]:
        g = api.GenReads(device=-1, layout="PE" if paired else "SE")
        g.load_profile(H.profile_path(prof))
        lens, words, nbits = g.deflate_code()
        lens = lens.astype(int)
        assert lens.max() <= 15 and abs(sum(2.0 ** -l for l in lens if l) - 1.0) < 1e-12          # complete prefix code
        for ch in b"\n#+/0123456789@ACGTN" + bytes(range(33, 127)):
            assert lens[ch] > 0
        assert lens[256] > 0 and lens[ord("A")] <= 4 and nbits % 1 == 0
        # canonical codes (RFC 1951 3.2.2)
        bl = np.bincount(lens, minlength=16); bl[0] = 0
        code, nxt = 0, [0] * 17
        for l in range(1, 16):
            code = (code + bl[l - 1]) << 1; nxt[l] = code
        codes = [0] * 257
        for sym in range(257):
            if lens[sym]:
                codes[sym] = nxt[lens[sym]]; nxt[lens[sym]] += 1
        bits = [(int(words[i >> 5]) >> (i & 31)) & 1 for i in range(nbits)]
        for b in list(text) + [256]:
            bits += [(codes[b] >> i) & 1 for i in range(lens[b] - 1, -1, -1)]
        bits += [0] * (-len(bits) % 8)
        out = bytearray(len(bits) // 8)
        for i, b in enumerate(bits):
            out[i >> 3] |= b << (i & 7)
        out += zlib.crc32(text).to_bytes(4, "little") + len(text).to_bytes(4, "little")
        out[16:18] = (len(out) - 1).to_bytes(2, "little")
        assert gzip.decompress(bytes(out)) == text
        g.close()


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the arm the driver times beside ours): one JSON line with the contract's keys, produced by
    the compiled reference when it exists, else by the CPU oracle — on a tiny debug genome here."""
    import json
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(H.ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                        "--scale", "0.05", "--coverage", "10"], capture_output=True, timeout=600)
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    lines = [l for l in r.stdout.decode().splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "impl", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype", "data", "config",
              "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["value"] > 0 and d["unit"] == "M reads/s" and d["dtype"] == "u8"
    # the line states the steps it really ran (one whole reference process each), and its timed region fits its own run
    assert d["steps"] == 2 and d["warmup"] == 1 and d["scaling"] == "strong"
    assert d["config"]["workload"].startswith("DEBUG") and "EXTRAPOLATED" in d["cpu_baseline"]["sample"]
    if d["cpu_baseline"]["kind"] == "reference":
        assert set(d["cpu_baseline"]["stage_s"]) == {"load_frags", "amplify", "alloc", "reads"} and d["cpu_baseline"]["reads_stage_value"] > 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_bench_fastq_sample_windows_hold_the_bytes_at_their_offsets():
    """bench.py --dump-outputs: the sink, fed a known byte stream per file in uneven slabs through its ctypes entry point as the
    library calls it, keeps in every window exactly the bytes at the window's offset; bytes past the end of a file stay -1."""
    import bench
    rng = np.random.default_rng(3)
    streams = [rng.integers(0, 256, 5_000_000, dtype=np.uint8), rng.integers(0, 256, 1_234_567, dtype=np.uint8)]
    s = bench.FastqSample(2, 4_000_000)
    for f, st in enumerate(streams):
        p = 0
        while p < len(st):
            chunk = np.ascontiguousarray(st[p:p + int(rng.integers(1, 300_000))])
            assert s.fn(None, f, chunk.ctypes.data, len(chunk)) == 0
            p += len(chunk)
    for f, st in enumerate(streams):
        assert s.pos[f] == len(st)
        for k, o in enumerate(s.offsets):
            want = np.full(s.WIDTH, -1.0, dtype=np.float32)
            seg = st[o:o + s.WIDTH]
            want[:len(seg)] = seg
            assert np.array_equal(s.data[f][k], want), (f, k, o)
    assert (s.offsets + s.WIDTH > len(streams[1])).sum() > 1000   # file 2 ends inside the sampled range
