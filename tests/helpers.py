"""Shared test plumbing: fixtures on disk, the CPU oracle (oracle/), the compiled reference (oracle/_ref).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg may touch oracle/ — the product
(scssim_b200/) never does.
"""
import ctypes as C
import functools
import json
import lzma
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")
ORACLE_DIR = os.path.join(ROOT, "oracle")
PROFILES = ["Illumina_HiSeq2500", "Illumina_HiSeqXTen", "Illumina_HiSeq2000", "Illumina_GenomeAnalyzerIIx"]


def reference_dir() -> str:
    """Where the original SCSsim sources (lib/, src/) lie, which oracle/build_ref.sh compiles into oracle/_ref: the
    reference_path that BASELINE.json declares, or SCS_REFERENCE_DIR when set. They are not part of this repository."""
    d = os.environ.get("SCS_REFERENCE_DIR")
    if d is None:
        with open(os.path.join(ROOT, "BASELINE.json")) as f:
            d = json.load(f).get("reference_path", "")
    return d


@functools.lru_cache(maxsize=None)
def scratch_dir() -> str:
    # per user: on a shared machine another user's directory of the same name is not writable
    d = os.environ.get("SCS_TEST_SCRATCH") or os.path.join(tempfile.gettempdir(), f"scssim_b200_tests_{os.getuid()}")
    os.makedirs(d, exist_ok=True)
    return d


@functools.lru_cache(maxsize=None)
def profile_path(name: str) -> str:
    """Decompress the committed copy of a shipped .profile (test fixture) and return its path."""
    out = os.path.join(scratch_dir(), name + ".profile")
    if not os.path.exists(out):
        tmp = f"{out}.{os.getpid()}.tmp"      # several ranks may decompress at once: unique name, atomic rename
        with lzma.open(os.path.join(GOLDEN, "profiles", name + ".profile.xz")) as f, open(tmp, "wb") as o:
            o.write(f.read())
        os.replace(tmp, out)
    return out


@functools.lru_cache(maxsize=None)
def oracle_bin() -> str:
    subprocess.run(["make", "-s", "-C", ORACLE_DIR, "scs_oracle", "liboracle.so"], check=True)
    return os.path.join(ORACLE_DIR, "scs_oracle")


@functools.lru_cache(maxsize=None)
def oracle_lib():
    oracle_bin()
    L = C.CDLL(os.path.join(ORACLE_DIR, "liboracle.so"))
    L.orc_profile_load.restype = C.c_void_p
    L.orc_profile_load.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_char_p, C.c_int]
    L.orc_profile_free.argtypes = [C.c_void_p]
    L.orc_profile_info.argtypes = [C.c_void_p, C.c_void_p]
    L.orc_profile_scalars.argtypes = [C.c_void_p, C.c_void_p]
    L.orc_profile_cdf.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    L.orc_predict.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64,
                              C.c_void_p, C.c_void_p, C.c_void_p]
    L.orc_philox.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.orc_det_log.restype = C.c_double
    L.orc_det_log.argtypes = [C.c_double]
    L.orc_philox_draw.restype = C.c_uint32
    L.orc_philox_draw.argtypes = [C.c_uint64, C.c_int, C.c_int, C.c_uint64, C.c_uint64]
    return L


def have_reference_sources() -> bool:
    d = reference_dir()
    return bool(d) and os.path.isdir(os.path.join(d, "lib"))


def build_reference():
    """oracle/build_ref.sh on the sources of reference_dir() (a no-op when the binaries are up to date)."""
    subprocess.run(["bash", os.path.join(ORACLE_DIR, "build_ref.sh")], check=True, env=dict(os.environ, SCS_REFERENCE_DIR=reference_dir()))


def ref_replay_bin():
    """The compiled reference with seed/draw-log hooks (oracle/build_ref.sh); None if it was never built."""
    p = os.path.join(ORACLE_DIR, "_ref", "bin", "scssim_replay")
    if os.path.exists(p):
        return p
    if have_reference_sources():
        build_reference()
        return p if os.path.exists(p) else None
    return None


def write_genome(path: str, n_chrom: int, chrom_len: int, seed: int, diploid: bool = True, width: int = 100):
    from scssim_b200.synth import synth_genome, write_fasta
    g = synth_genome(n_chrom, chrom_len, seed, diploid=diploid)
    write_fasta(path, g, width=width)
    return g


def genreads_args(profile, layout="PE", gamma=2e-10, coverage=5.0, isize=260, primers=100000):
    return ["-m", profile, "-l", layout, "-r", repr(gamma), "-c", repr(coverage), "-s", str(isize), "-p", str(primers)]


def run_reference_replay(fa: str, out_prefix: str, tape_prefix: str, seed: int, args):
    """Run the reference itself (-t 1) with a fixed seed, logging every draw. Returns FASTQ paths."""
    exe = ref_replay_bin()
    assert exe is not None
    if os.path.exists(fa + ".fai"):
        os.remove(fa + ".fai")
    env = dict(os.environ, SCS_SEED=str(seed), SCS_REPLAY_LOG=tape_prefix)
    subprocess.run([exe, "genreads", "-i", fa, "-t", "1", "-o", out_prefix] + list(args), check=True, env=env,
                   stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)


def run_oracle(fa: str, out_prefix: str, args, tape_prefix=None, seed=None, dump_prefix=None):
    cmd = [oracle_bin(), "genreads", "-i", fa, "-o", out_prefix] + list(args)
    if tape_prefix is not None:
        cmd += ["--tape", tape_prefix]
    else:
        cmd += ["--seed", str(seed)]
    if dump_prefix is not None:
        cmd += ["--dump", dump_prefix]
    r = subprocess.run(cmd, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE)
    assert r.returncode == 0, r.stderr.decode()
    return r.stderr.decode()


def read_bytes(path):
    with open(path, "rb") as f:
        return f.read()


def fastq_names(prefix, layout):
    return [prefix + "_1.fq", prefix + "_2.fq"] if layout == "PE" else [prefix + ".fq"]


def oracle_dump(dump_prefix):
    d = {}
    d["frags"] = np.fromfile(dump_prefix + ".frags.i64", dtype=np.int64).reshape(-1, 5)
    d["semis"] = np.fromfile(dump_prefix + ".semis.u32", dtype=np.uint32).reshape(-1, 7)
    d["fulls"] = np.fromfile(dump_prefix + ".fulls.u32", dtype=np.uint32).reshape(-1, 7)
    d["errs"] = np.fromfile(dump_prefix + ".errs.u32", dtype=np.uint32).reshape(-1, 2)
    d["counts"] = np.fromfile(dump_prefix + ".counts.u32", dtype=np.uint32)
    d["weights"] = np.fromfile(dump_prefix + ".weights.f64", dtype=np.float64)
    d["primer_counts"] = np.fromfile(dump_prefix + ".primer_counts.i64", dtype=np.int64)
    d["meta"] = np.fromfile(dump_prefix + ".meta.u64", dtype=np.uint64)
    return d


def expected_windows(genome, od):
    """Oriented-window form (gstart, rc, len) of the oracle's semi and full amplicons, from its
    (fragment, spos, len) records — the representation the CUDA path stores (DESIGN.md)."""
    goff, acc = [], 0
    for _, s in genome:
        goff.append(acc)
        acc += (len(s) + 31) // 32 * 32
    fr = od["frags"]
    g = np.array([goff[int(s)] for s in fr[:, 0]], dtype=np.int64) + fr[:, 1]
    L = fr[:, 2]
    t_rc = (fr[:, 3] == 1)
    t_g = np.where(t_rc, g + L - 1, g)
    se = od["semis"].astype(np.int64)
    f = se[:, 0]
    s, l = se[:, 1], se[:, 2]
    u_rc = ~t_rc[f]
    u_g = np.where(t_rc[f], t_g[f] - s - l + 1, t_g[f] + s + l - 1)
    fu = od["fulls"].astype(np.int64)
    p = fu[:, 0]
    s2, l2 = fu[:, 1], fu[:, 2]
    f_rc = u_rc[p]
    f_g = np.where(f_rc, u_g[p] - s2, u_g[p] + s2)
    semis = np.stack([u_g, u_rc.astype(np.int64), l, se[:, 3], se[:, 4]], axis=1)
    fulls = np.stack([f_g, f_rc.astype(np.int64), l2, fu[:, 3]], axis=1)
    return semis, fulls


def write_genome_with_n(path: str, glen: int = 300_000, seed: int = 77, width: int = 70):
    """Synthetic diploid chromosome with an N run, scattered N, IUPAC codes and soft-masked (lower-case) stretches."""
    from scssim_b200.synth import synth_genome, write_fasta
    g = synth_genome(1, glen, seed, diploid=True)
    rng = np.random.default_rng(seed)
    out = []
    for name, s in g:
        s = s.copy()
        s[glen * 2 // 5:glen * 2 // 5 + 5000] = ord("N")
        s[rng.integers(0, glen, 120)] = ord("N")
        s[rng.integers(0, glen, 10)] = ord("R")
        for lo in rng.integers(0, glen - 2000, 5):
            s[lo:lo + 1500] |= 0x20          # lower case
        out.append((name, s))
    write_fasta(path, out, width=width)
    return out


# ------------------------------------------------------------------------------------------------ simuvars
def ref_bin():
    """The compiled reference (oracle/_ref/bin/scssim, stock behaviour + the five missing returns); None if never built."""
    p = os.path.join(ORACLE_DIR, "_ref", "bin", "scssim")
    if os.path.exists(p):
        return p
    if have_reference_sources():
        build_reference()
        return p if os.path.exists(p) else None
    return None


def make_simuvars_case(d: str, seed: int, chrom_lens=(60_000, 35_000), n_snp=300, n_snv=40, n_ins=40, n_del=40, n_cnv=6, width=100,
                       names=None, max_cn=5, lower=True):
    """Random `scssim simuvars` inputs in directory d: ref.fa (soft-masked stretch + an N run per chromosome), snp.txt (6 columns:
    id, chr, pos, observed, strand, ref — both strands, both allele orders) and vars.txt (i/d/s/c records, het and homo,
    copy numbers 0..max_cn). Returns (ref, snp, var) paths."""
    from scssim_b200.synth import synth_sequence, write_fasta
    os.makedirs(d, exist_ok=True)
    rng = np.random.default_rng(seed)
    names = names or [f"chr{i + 1}" for i in range(len(chrom_lens))]
    seqs = []
    for i, L in enumerate(chrom_lens):
        s = synth_sequence(L, seed * 100 + i)
        if lower and L > 1000:
            a = int(rng.integers(0, L - 500)); s[a:a + 500] |= 0x20
            b = int(rng.integers(0, L - 50)); s[b:b + 50] = ord("N")
        seqs.append((names[i], s))
    ref, snp, var = os.path.join(d, "ref.fa"), os.path.join(d, "snp.txt"), os.path.join(d, "vars.txt")
    write_fasta(ref, seqs, width)
    if os.path.exists(ref + ".fai"):
        os.remove(ref + ".fai")
    comp = {"A": "T", "C": "G", "G": "C", "T": "A", "N": "N"}
    with open(snp, "w") as f:
        for nm, s in seqs:
            L = len(s)
            for p in sorted(rng.integers(1, L + 1, size=n_snp).tolist()):
                r = chr(s[p - 1]).upper()
                alts = [b for b in "ACGT" if b != r]
                alt = alts[int(rng.integers(0, len(alts)))]
                if rng.integers(0, 2):
                    obs = f"{r}/{alt}" if rng.integers(0, 2) else f"{alt}/{r}"
                    f.write(f"rs{p}\t{nm}\t{p}\t{obs}\t+\t{r}\n")
                else:
                    f.write(f"rs{p}\t{nm}\t{p}\t{comp.get(r, 'N')}/{comp[alt]}\t-\t{r}\n")
    with open(var, "w") as f:
        f.write("#type\tchr\tfields\n\n")
        for nm, s in seqs:
            L = len(s)
            zyg = lambda: "homo" if rng.integers(0, 2) else "het"
            for _ in range(n_ins):
                p = int(rng.integers(1, L + 1)); l = int(rng.integers(1, 12))
                f.write(f"i\t{nm}\t{p}\t{''.join('acgt'[x] for x in rng.integers(0, 4, size=l))}\t{zyg()}\n")
            for _ in range(n_del):
                p = int(rng.integers(1, max(2, L - 30))); l = int(rng.integers(1, 20))
                f.write(f"d\t{nm}\t{p}\t{l}\t{zyg()}\n")
            for _ in range(n_snv):
                p = int(rng.integers(1, L + 1)); r = chr(s[p - 1])
                alt = [b for b in "ACGT" if b != r.upper()][int(rng.integers(0, 3))]
                f.write(f"s\t{nm}\t{p}\t{r}\t{alt}\t{zyg()}\n")
            cuts = sorted(rng.integers(1, L, size=2 * n_cnv).tolist())
            for c in range(n_cnv):
                a, b = cuts[2 * c], cuts[2 * c + 1]
                if b <= a:
                    continue
                cn = int(rng.integers(0, max_cn + 1)); mcn = int(rng.integers((cn + 1) // 2, cn + 1))
                f.write(f"c\t{nm}\t{a}\t{b}\t{cn}\t{mcn}\n")
    return ref, snp, var


def run_oracle_simuvars(ref, snp, var, out, seed=None, check=True):
    cmd = [oracle_bin(), "simuvars", "-r", ref, "-o", out]
    if snp:
        cmd += ["-s", snp]
    if var:
        cmd += ["-v", var]
    if seed is not None:
        cmd += ["--seed", str(seed)]
    r = subprocess.run(cmd, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE)
    if check:
        assert r.returncode == 0, r.stderr.decode()
    return r


def run_reference_simuvars(ref, snp, var, out):
    """The reference binary itself; removes the .fai side file first so it indexes from scratch."""
    exe = ref_bin()
    assert exe is not None
    if os.path.exists(ref + ".fai"):
        os.remove(ref + ".fai")
    cmd = [exe, "simuvars", "-r", ref, "-o", out]
    if snp:
        cmd += ["-s", snp]
    if var:
        cmd += ["-v", var]
    return subprocess.run(cmd, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE)


def read_fasta_records(path):
    """[(header, uint8 bases)] of a FASTA file."""
    names, seqs = [], []
    for line in read_bytes(path).split(b"\n"):
        if line.startswith(b">"):
            names.append(line[1:].decode()); seqs.append([])
        elif names:
            seqs[-1].append(line)
    return [(n, np.frombuffer(b"".join(s), dtype=np.uint8)) for n, s in zip(names, seqs)]


def strip_chr(name: str) -> str:
    i = name.find("chrom")
    if i < 0:
        i = name.find("chr")
        return name[i + 3:] if i >= 0 else name
    return name[i + 5:]


def materialize_plan(ref, snp, var, ploidy=2, seed=1, width=100) -> bytes:
    """Test-side numpy execution of the library's host-built edit plan (what the CUDA kernels do on the device):
    copy runs, then point substitutions, then FASTA line breaking."""
    from scssim_b200 import api
    recs = read_fasta_records(ref)
    P = api.SimuVarsPlan([(strip_chr(n.split()[0]), len(s)) for n, s in recs], snp, var, ploidy, seed)
    haps, pieces, subs, lits, names = P.haps, P.pieces, P.subs, P.literals, P.names
    out = []
    for h, nm in zip(haps, names):
        c, L = int(h[0]), int(h[2])
        refu = np.frombuffer(recs[c][1].tobytes().upper(), dtype=np.uint8)
        buf = np.zeros(L, dtype=np.uint8)
        for o, src, ln in pieces[int(h[3]):int(h[4])].tolist():
            if src & api.SV_LITERAL:
                src &= ~api.SV_LITERAL
                buf[o:o + ln] = lits[src:src + ln]
            else:
                buf[o:o + ln] = refu[src:src + ln]
        for o, ch in subs[int(h[5]):int(h[6])].tolist():
            buf[o] = ch
        out.append(b">" + nm.encode() + b"\n")
        t = buf.tobytes()
        out.extend(t[i:i + width] + b"\n" for i in range(0, L, width))
    P.close()
    return b"".join(out)


def config0_inputs(d: str):
    """BASELINE configs[0] inputs in directory d: synthetic 63,025,520-base chr20 (the reference's ref.fa.gz is not shipped with
    it) + the reference's own testData SNP and variation files (tests/golden/testdata). Returns (ref, snp, var) paths."""
    from scssim_b200.synth import synth_sequence, write_fasta
    os.makedirs(d, exist_ok=True)
    ref = os.path.join(d, "ref.fa")
    write_fasta(ref, [("chr20", synth_sequence(63_025_520, 20))], 100)
    if os.path.exists(ref + ".fai"):
        os.remove(ref + ".fai")
    out = [ref]
    for f in ("snp.txt", "vars.txt"):
        p = os.path.join(d, f)
        with lzma.open(os.path.join(GOLDEN, "testdata", f + ".xz")) as i, open(p, "wb") as o:
            o.write(i.read())
        out.append(p)
    return tuple(out)
