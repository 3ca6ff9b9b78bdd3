#!/usr/bin/env python
"""bench.py — the `scssim genreads` hot path on B200 (contract: see the task brief; one JSON line on stdout).

Workload = BASELINE.json configs[3], the configuration the metric is quoted on: ONE synthetic human-scale diploid cell,
6.2 Gb = 4 chromosomes x 775 Mb x 2 haplotypes (GC 35-60 % per 100 kb block, haplotype 2 = haplotype 1 + 0.1 % SNPs, every
sequence < 2^31 as the reference's FASTA reader requires), paired-end 150 bp at 30x with the HiSeq2500 profile (resampled
125 -> 150 bins, scssim_b200/tools/resample_profile.py: read length is a property of the .profile in the reference), GC bias on,
gamma 2e-10 (README value). The reference's `-c` is relative to HALF the summed sequence length and counts individual reads
(Malbac.cpp:414-420), so 30x of the 6.2 Gb diploid FASTA = 620 M pairs is `-c 60`: 1.24 G reads, ~394 GB of FASTQ per step.
The SAME cell is generated at every N (strong scaling): rank r holds its share of the sequences for the amplification, the
packed genome and the amplicon table are then replicated over NVLink (NCCL) and the cell's read slots are cut into contiguous
ranges, one per GPU; the rank-ordered shards concatenate to exactly the single-GPU files.

A "step" = one pass of the hot path over that cell: MALBAC amplification -> GC-weighted read allocation -> read synthesis ->
FASTQ packing, FASTQ landing in the library's pinned host ring.
  value     : M reads/s with the packed genome already resident in HBM when the timed region starts (CUDA events).
  e2e       : the same through the C-ABI calls a user makes with HOST buffers: scs_set_genome (H2D of the ASCII genome from
              pinned memory + pack) ... scs_yield_reads_sink (D2H of every FASTQ byte) inside the timed region.
  e2e_files : through the drop-in call that writes files, scs_yield_reads(prefix) -> <prefix>_1.fq/_2.fq, on the bounded
              configs[1] cell (5.3 GB of FASTQ per step; the full cell would need 394 GB of scratch disk per step).
  configs1  : BASELINE configs[1] (250 Mb haploid, PE150 10x) on rank 0's GPU, the round-1 headline, kept for continuity.

--impl reference times the reference's own CPU implementation (oracle/_ref/bin/scssim, built by oracle/build_ref.sh from the
SCSsim sources at BASELINE.json's reference_path or $SCS_REFERENCE_DIR) with all host threads; every step is one whole `scssim genreads` process on a bounded sample of the same
workload (a 1/387-scale cell: same GC spectrum, gamma, coverage, profile, layout), and the line says "extrapolated".

--dump-outputs DIR keeps a fixed sample of the FASTQ that the last timed step produced (FastqSample) and writes it as DIR/*.npy, so
that two builds run with the same arguments can be compared output for output. That step hands its slabs to a Python sink instead of
the null sink, inside the timed region, so the line of such a run says "dump_outputs": true in its detail and is not the headline.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True   # the tree may be read-only; nothing is written into it
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

N_CHROM = 4
CHROM_LEN = 775_000_000      # x 4 chromosomes x 2 haplotypes = 6.2 Gb
COVERAGE = 60.0              # = 30x of the diploid FASTA (see module docstring)
GAMMA = 2e-10
READ_LEN = 150
ISIZE = 260
SNP_RATE = 1e-3
REF_SAMPLE_CHROM = 8_000_000   # the CPU legs run a cell of 1 chromosome x 8 Mb x 2 haplotypes (1/387.5 of the bases and of the reads)
C1_LEN, C1_COVERAGE = 250_000_000, 20.0   # BASELINE configs[1]
UNIT = "M reads/s"
METRIC = "PE150 M reads/s (FASTQ GB/s in detail) vs HBM/D2H roofline"


def bench_profile(tmp):
    import helpers as H
    from scssim_b200.tools.resample_profile import resample
    p = os.path.join(tmp, "HiSeq2500_150.profile")
    resample(H.profile_path("Illumina_HiSeq2500"), p, READ_LEN)
    return p


def bench_config(scale, coverage):
    """The workload both arms are run on (identical dict in both JSON lines)."""
    clen = int(CHROM_LEN * scale)
    reads = int((N_CHROM * 2 * clen // 2) * coverage / READ_LEN)
    name = (f"BASELINE configs[3]: one synthetic 6.2 Gb diploid cell ({N_CHROM} chromosomes x {CHROM_LEN / 1e6:.0f} Mb x 2 haplotypes, GC 35-60%, "
            f"haplotype 2 = haplotype 1 + 0.1% SNPs), PE150 30x (-c 60: 1.24 G reads = 620 M pairs per step), HiSeq2500 profile resampled to "
            f"150 bins, GC bias on, gamma 2e-10, -s 260; the same cell at every N")
    if scale != 1.0 or coverage != COVERAGE:
        name = f"DEBUG scale {scale} coverage {coverage} of: " + name
    return {"workload": name, "layout": "PE", "read_length": READ_LEN, "coverage_flag": coverage, "gamma": GAMMA, "isize": ISIZE,
            "genome_bases": N_CHROM * 2 * clen, "reads_per_step": reads,
            "l2": "inputs larger than L2: every step streams the 1.55 GB packed genome and ~394 GB of FASTQ through the 126 MB L2"}


class FastqSample:
    """Sink of one read stage that keeps a fixed sample of the FASTQ it is handed: per file, WINDOWS windows of WIDTH bytes at
    seeded offsets below the file's expected size. The offsets depend on the bench arguments only, so two builds sample the same
    bytes. Window bytes past the end of a file stay -1."""
    WINDOWS, WIDTH = 4096, 1024   # 2 files x 4096 x 1024 float32 = 32 MiB

    def __init__(self, nfiles, expected_bytes, seed=0x5C55):
        from scssim_b200 import api
        self.offsets = np.sort(np.random.default_rng(seed).integers(0, max(int(expected_bytes), 1), self.WINDOWS))
        self.data = [np.full((self.WINDOWS, self.WIDTH), -1.0, dtype=np.float32) for _ in range(nfiles)]
        self.pos = [0] * nfiles
        self.fn = api.SINK_FN(self._sink)

    def _sink(self, _user, f, data, n):
        lo, hi = self.pos[f], self.pos[f] + n
        first, last = np.searchsorted(self.offsets, lo - self.WIDTH, side="right"), np.searchsorted(self.offsets, hi)
        if last > first:
            buf = np.ctypeslib.as_array(C.cast(data, C.POINTER(C.c_ubyte)), shape=(n,))
            for k in range(first, last):
                o = int(self.offsets[k])
                a, b = max(o, lo), min(o + self.WIDTH, hi)
                self.data[f][k, a - o:b - o] = buf[a - lo:b - lo]
        self.pos[f] = hi
        return 0

    def save(self, d, stats):
        """fastq_<file>.npy: (WINDOWS, WIDTH) bytes; fastq_offsets.npy: window offsets; fastq_bytes.npy: bytes per file, records."""
        os.makedirs(d, exist_ok=True)
        for f, arr in enumerate(self.data):
            np.save(os.path.join(d, f"fastq_{f + 1}.npy"), arr)
        np.save(os.path.join(d, "fastq_offsets.npy"), self.offsets.astype(np.float64))
        np.save(os.path.join(d, "fastq_bytes.npy"), np.array(list(stats["fastq_bytes"]) + [stats["records"]], dtype=np.float64))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def measured_hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except (OSError, KeyError, ValueError):
        return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------ reference arm (CPU)
def run_reference_cpu(tmp, profile, steps, warmup, coverage, sample_chrom=REF_SAMPLE_CHROM):
    """The reference's own `scssim genreads -t <cores>` (compiled into oracle/_ref by oracle/build_ref.sh), one whole process per
    step on the bounded sample cell. Stage times are taken from the moments its own stderr progress lines appear
    (Malbac.cpp:174,422,437; scssim.cpp:66). Returns a dict."""
    import helpers as H
    from scssim_b200.synth import synth_genome, write_fasta
    exe = os.path.join(ROOT, "oracle", "_ref", "bin", "scssim")
    cores = os.cpu_count() or 1
    fa = os.path.join(tmp, "sample.fa")
    write_fasta(fa, synth_genome(1, sample_chrom, 7001, diploid=True, snp_rate=SNP_RATE))
    reads = int((2 * sample_chrom // 2) * coverage / READ_LEN)
    frac = sample_chrom / (N_CHROM * CHROM_LEN)
    if os.path.exists(exe):
        kind = "reference"
        cmd = [exe, "genreads", "-i", fa, "-t", str(cores), "-o", os.path.join(tmp, "cpu")] + H.genreads_args(profile, "PE", GAMMA, coverage, ISIZE)
        what = f"reference `scssim genreads -t {cores}` (oracle/_ref, unmodified algorithm)"
    else:   # no compiled reference on this box: the CPU oracle (single thread)
        kind, cores = "port", 1
        cmd = [H.oracle_bin(), "genreads", "-i", fa, "-o", os.path.join(tmp, "cpu"), "--seed", "1"] + H.genreads_args(profile, "PE", GAMMA, coverage, ISIZE)
        what = "CPU oracle (oracle/scs_oracle, 1 thread)"
    sample = (f"1/{1 / frac:.1f}-scale cell (1 chromosome x {sample_chrom / 1e6:.0f} Mb x 2 haplotypes, {reads / 1e6:.2f} M reads per step), same GC spectrum / "
              f"gamma / -c / profile / layout; {what}; one whole process per step (FASTA load + index, amplification, read stage, FASTQ files "
              f"on local disk); the full-cell figure is EXTRAPOLATED linearly in the number of reads")
    marks = ["MALBAC amplification", "Number of reads to generate", "Producing reads", "Reads generation done"]
    walls, stages = [], []
    for i in range(warmup + steps):
        if os.path.exists(fa + ".fai"):
            os.remove(fa + ".fai")
        t0 = time.perf_counter()
        p = subprocess.Popen(cmd, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True)
        seen = {}
        for line in p.stderr:
            for m in marks:
                if m in line and m not in seen:
                    seen[m] = time.perf_counter() - t0
        rc = p.wait()
        dt = time.perf_counter() - t0
        if rc != 0:
            raise RuntimeError(f"reference arm: {cmd[0]} exited {rc}")
        if i >= warmup:
            walls.append(dt)
            if len(seen) == len(marks):
                t = [seen[m] for m in marks]
                stages.append({"load_frags": t[0], "amplify": t[1] - t[0], "alloc": t[2] - t[1], "reads": t[3] - t[2]})
    sec = sum(walls) / len(walls)
    st = {k: sum(s[k] for s in stages) / len(stages) for k in stages[0]} if stages else None
    return {"value": reads / sec / 1e6, "cores": cores, "kind": kind, "sample": sample, "s_per_step": sec, "reads_per_step": reads,
            "stage_s": st, "reads_stage_value": (reads / st["reads"] / 1e6) if st and st["reads"] > 0 else None,
            "steps_run": len(walls), "warmup_run": warmup, "extrapolated_full_cell_s": sec / frac}


# ------------------------------------------------------------------------------------------------ synthetic cell on the device
def synth_chromosome_cuda(torch, length, seed, device, out_h1, out_h2):
    """One chromosome of the synthetic cell, generated on the GPU (plumbing: 6.2 Gb through numpy would take minutes) straight into
    two pinned host arrays: per-100 kb block GC content ~ U[0.35, 0.60], bases i.i.d. within a block; haplotype 2 = haplotype 1
    with 0.1 % of its positions substituted (scssim_b200/synth.py is the numpy statement of the same generator)."""
    gen = torch.Generator(device=device); gen.manual_seed(seed)
    block, chunk = 100_000, 50_000_000
    nblk = (length + block - 1) // block
    gcs = 0.35 + 0.25 * torch.rand(nblk, generator=gen, device=device)
    lut = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device=device)
    h1 = torch.from_numpy(out_h1); h2 = torch.from_numpy(out_h2)
    for lo in range(0, length, chunk):
        n = min(chunk, length - lo)
        idx = torch.arange(lo, lo + n, device=device) // block
        is_gc = torch.rand(n, generator=gen, device=device) < gcs[idx]
        pick = torch.randint(0, 2, (n,), generator=gen, device=device, dtype=torch.uint8)
        code = torch.where(is_gc, 1 + pick, 3 * pick)   # A=0 C=1 G=2 T=3 ; GC -> {C,G}, AT -> {A,T}
        h1[lo:lo + n].copy_(lut[code.long()], non_blocking=False)
        nsnp = int(n * SNP_RATE)
        pos = torch.randint(0, n, (nsnp,), generator=gen, device=device)
        shift = torch.randint(1, 4, (nsnp,), generator=gen, device=device, dtype=torch.uint8)
        # a position drawn more than once takes its last draw, as numpy's assignment in synth.py does: a CUDA scatter with
        # repeated indices leaves the winner undefined, which made the cell differ from run to run
        pos, order = torch.sort(pos, stable=True)
        last = torch.ones_like(pos, dtype=torch.bool)
        last[:-1] = pos[1:] != pos[:-1]
        pos, shift = pos[last], shift[order][last]
        code[pos] = (code[pos] + shift) & 3
        h2[lo:lo + n].copy_(lut[code.long()], non_blocking=False)
        del idx, is_gc, pick, code, pos, shift, order, last
    torch.cuda.empty_cache()


def probe_host_links(torch, ndev):
    """Pinned D2H rate of every GPU's host link, each GPU alone and all GPUs at once (one process, one stream per device). Returns
    (device order: best-connected first, probe record). On this pool's 8-GPU boxes the links are far from equal: GPUs 4-7 keep
    44 GB/s each when they copy together, GPUs 0-3 share ~73 GB/s and drag the whole box down to ~123 GB/s when all eight copy."""
    nb = 128 << 20
    bufs = {}
    for j in range(ndev):
        with torch.cuda.device(j):
            bufs[j] = (torch.empty(nb, dtype=torch.uint8, device=f"cuda:{j}"), torch.empty(nb, dtype=torch.uint8, pin_memory=True), torch.cuda.Stream(device=j),
                       torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))

    def run(devs, reps=3):
        for j in devs:
            d, h, s, _, _ = bufs[j]
            with torch.cuda.device(j), torch.cuda.stream(s):
                h.copy_(d, non_blocking=True)
        for j in devs:
            bufs[j][2].synchronize()
        for j in devs:
            d, h, s, e0, e1 = bufs[j]
            with torch.cuda.device(j), torch.cuda.stream(s):
                e0.record(s)
                for _ in range(reps):
                    h.copy_(d, non_blocking=True)
                e1.record(s)
        out = {}
        for j in devs:
            bufs[j][2].synchronize()
            out[j] = reps * nb / (bufs[j][3].elapsed_time(bufs[j][4]) / 1e3) / 1e9
        return out
    single = {j: run([j])[j] for j in range(ndev)}
    together = run(list(range(ndev)))
    order = sorted(range(ndev), key=lambda j: (-round(together[j]), -round(single[j]), j))
    rec = {"alone_GBps": [round(single[j], 1) for j in range(ndev)], "all_at_once_GBps": [round(together[j], 1) for j in range(ndev)]}
    del bufs
    torch.cuda.empty_cache()
    return order, rec


def device_for_rank(torch, local, world):
    """Device order by measured host-link quality (the path is bound by the D2H copy of its output): local rank r runs on the r-th
    best-connected GPU. Local rank 0 probes and publishes the order; the other ranks read it."""
    ndev = torch.cuda.device_count()
    if ndev <= 1 or world > ndev or os.environ.get("SCS_BENCH_NO_DEVMAP"):
        return local, {"order": list(range(ndev)), "probe": None}
    if world == 1:
        order, rec = probe_host_links(torch, ndev)
        return order[0], {"order": order, "probe": rec}
    path = os.path.join(tempfile.gettempdir(), f"scs_devmap_{os.environ.get('MASTER_PORT', '0')}_{world}_{os.environ.get('TORCHELASTIC_RUN_ID', 'x')}.json")
    if local == 0:
        order, rec = probe_host_links(torch, ndev)
        with open(path + ".tmp", "w") as f:
            json.dump({"order": order, "probe": rec, "t": time.time()}, f)
        os.replace(path + ".tmp", path)
    t0 = time.time()
    m = None
    while time.time() - t0 < 180:
        try:
            with open(path) as f:
                m = json.load(f)
            if time.time() - m.get("t", 0) < 600:   # not a leftover of an earlier run on this box
                break
        except (OSError, ValueError):
            pass
        time.sleep(0.05)
    if m is None:
        m = {"order": list(range(ndev)), "probe": "unavailable"}
    return m["order"][local], m


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scale", type=float, default=1.0, help="(debug) fraction of the cell's bases; invalidates the number")
    ap.add_argument("--coverage", type=float, default=COVERAGE, help="(debug) override -c; invalidates the number")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="(debug) skip the CPU leg")
    ap.add_argument("--no-extras", action="store_true", help="(debug) skip the configs[1] and e2e_files legs")
    ap.add_argument("--no-balance", action="store_true", help="(debug) N > 1: every rank writes the reads of its own amplicons")
    ap.add_argument("--no-relay", action="store_true", help="(debug) never route a GPU's output through a better-connected peer GPU")
    ap.add_argument("--slab-mb", type=int, default=64, help="FASTQ staging slab per file and buffer (MiB)")
    ap.add_argument("--files-dir", default=None, help="directory for the e2e_files leg (default: the system temp dir)")
    ap.add_argument("--gz", action="store_true", help="(not the headline) block-gzip output on the device: compressed FASTQ lands in the pinned ring")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed sample of the FASTQ of the last timed step (rank 0's share) as DIR/<name>.npy (float32, float64)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    warmup = max(a.warmup, 0)
    # stdout carries exactly one JSON line: libraries that print there (NCCL's version banner) are sent to stderr
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(real_stdout, (json.dumps(obj) + "\n").encode())

    config = bench_config(a.scale, a.coverage)
    if a.gz:
        config["workload"] = "NOT THE HEADLINE (--gz: block-gzip output) " + config["workload"]
    if a.impl == "reference":
        if rank != 0:
            return 0
        with tempfile.TemporaryDirectory() as tmp:
            profile = bench_profile(tmp)
            sample_chrom = REF_SAMPLE_CHROM if a.scale >= 1.0 else max(200_000, int(REF_SAMPLE_CHROM * a.scale))
            r = run_reference_cpu(tmp, profile, max(1, a.steps), warmup, a.coverage, sample_chrom)
        emit({"metric": METRIC, "value": r["value"], "unit": UNIT, "impl": "reference", "n_gpus": a.gpus, "steps": r["steps_run"], "warmup": r["warmup_run"],
              "ms_per_step": r["s_per_step"] * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
              "config": config,
              "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"],
                               "stage_s": r["stage_s"], "reads_stage_value": r["reads_stage_value"], "reads_per_step": r["reads_per_step"],
                               "extrapolated_full_cell_s": r["extrapolated_full_cell_s"]},
              "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        return 0

    import torch
    import torch.distributed as dist
    from scssim_b200 import api

    device, devmap = device_for_rank(torch, local, world)
    torch.cuda.set_device(device)
    dev = f"cuda:{device}"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", device))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def gather_f64(x):
        t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
        if world == 1:
            return [float(t)]
        out = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(out, t)
        return [float(v) for v in out]

    with tempfile.TemporaryDirectory() as tmp:
        profile = bench_profile(tmp)
        clen = int(CHROM_LEN * a.scale)
        # the cell: 8 sequences in file order chrS1_1, chrS1_2, chrS2_1, ...; this rank keeps a contiguous run of them
        names = [f"chrS{c + 1}_{h}_{clen}" for c in range(N_CHROM) for h in (1, 2)]
        lo, hi = api.shard_sequences([clen] * len(names), rank, world)
        mine = list(range(lo, hi))
        host = {}
        for c in sorted({i // 2 for i in mine}):
            b1 = torch.empty(clen, dtype=torch.uint8, pin_memory=True).numpy(); b2 = torch.empty(clen, dtype=torch.uint8, pin_memory=True).numpy()
            synth_chromosome_cuda(torch, clen, 7000 + c, dev, b1, b2)
            host[2 * c], host[2 * c + 1] = b1, b2
        named = [(names[i], host[i]) for i in mine]
        h2d_bytes = sum(len(s) for _, s in named)
        for i in list(host):
            if i not in mine:
                del host[i]

        # ---- pinned D2H ceilings of this box, measured live: one GPU alone (rank 0), then ALL ranks copying at once. The second is the
        # ---- binding roof of the read stage (SURVEY.md §8d); on shared host fabrics the per-GPU rate drops as N grows
        nb = 256 << 20
        dbuf = torch.empty(nb, dtype=torch.uint8, device=dev); hbuf = torch.empty(nb, dtype=torch.uint8, pin_memory=True)

        def d2h_rate(active):
            hbuf.copy_(dbuf, non_blocking=True); barrier()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            if active:
                for _ in range(6):
                    hbuf.copy_(dbuf, non_blocking=True)
            c1.record(); torch.cuda.synchronize()
            r = 6 * nb / (c0.elapsed_time(c1) / 1e3) / 1e9 if active else 0.0
            barrier()
            return r
        d2h_single = gather_f64(d2h_rate(rank == 0))[0]
        d2h_per_rank = gather_f64(d2h_rate(True))
        d2h_peak = sum(d2h_per_rank)
        # GPUs behind a clearly slower host link (on this pool's 8-GPU boxes: GPUs 0-3 when all eight copy) hand their FASTQ slabs
        # over NVLink to a better-connected peer, whose link then carries both (scs_params.relay_device)
        relay_device, relay_map, d2h_relay_peak = -1, {}, None
        order = devmap.get("order") or list(range(torch.cuda.device_count()))
        fast = [r for r in range(world) if d2h_per_rank[r] >= 0.75 * max(d2h_per_rank)]
        slow = [r for r in range(world) if r not in fast]
        if world > 1 and slow and fast and not a.no_relay and not a.no_balance:
            relay_map = {r: fast[i % len(fast)] for i, r in enumerate(slow)}
            if rank in relay_map:
                relay_device = order[relay_map[rank]]
            per = gather_f64(d2h_rate(rank in fast))   # what the links that will carry the output sustain together
            d2h_relay_peak = sum(per)
        del dbuf, hbuf

        # ---- one cell sharded over the ranks: same seed everywhere, global ids key every Philox stream. With several GPUs the read
        # ---- slots are cut in proportion to a per-GPU weight (balance = 1): first its measured D2H rate, then refined after every
        # ---- warm-up step from the measured read-stage times, so that all GPUs finish together
        g = api.GenReads(gamma=GAMMA, coverage=a.coverage, isize=ISIZE, layout="PE", seed=0x5C55, device=device, rank=rank, world=world,
                         slab_bytes=a.slab_mb << 20, balance=(world > 1 and not a.no_balance), gzip=a.gz, relay_device=relay_device)
        weight = 1.0 if relay_map else d2h_per_rank[rank]
        if world > 1:
            # the library's own NCCL communicator (scs_nccl_init): rank 0's id reaches the other ranks through the process group that
            # torchrun set up; from here on no collective of the hot path goes through Python
            idt = torch.zeros(128, dtype=torch.uint8, device=dev)
            if rank == 0:
                idt.copy_(torch.frombuffer(bytearray(api.nccl_unique_id()), dtype=torch.uint8))
            dist.broadcast(idt, src=0)
            g.nccl_init(bytes(idt.cpu().numpy().tobytes()))
            g.set_shard_weight(weight)
        g.load_profile(profile)
        g.set_genome(named).create_frags()

        def step_resident():
            g.amplify().set_read_counts().yield_reads_discard()

        sink_state = {"bytes": 0, "sum": 0}

        def sink(_u, f, data, n):
            sink_state["bytes"] += n
            sink_state["sum"] += C.cast(data, C.POINTER(C.c_ubyte))[0]   # touch the landed bytes
            return 0
        sink_cb = api.SINK_FN(sink)

        e2e_parts = {}

        def step_e2e():
            t = [time.perf_counter()]
            g.set_genome(named); t.append(time.perf_counter())
            g.create_frags(); t.append(time.perf_counter())
            g.amplify().set_read_counts(); t.append(time.perf_counter())
            g._ck(api.lib().scs_yield_reads_sink(g._h, sink_cb, None)); t.append(time.perf_counter())
            for name, a0, a1 in zip(("set_genome_h2d_pack", "create_frags", "amplify_alloc", "reads_d2h_sink"), t, t[1:]):
                e2e_parts[name] = round((a1 - a0) * 1e3, 1)

        weights_hist = []
        for _ in range(warmup):
            step_resident()
            if world > 1 and not a.no_balance:
                st = g.stats()
                t_all = gather_f64(st["ms_reads"]); r_all = gather_f64(st["records"])
                rate = [r / t if t > 0 else 0.0 for r, t in zip(r_all, t_all)]   # records per ms of this GPU's read stage
                if min(rate) > 0:
                    weight = rate[rank]
                    g.set_shard_weight(weight)
                    weights_hist.append([round(x / sum(rate), 4) for x in rate])
        sample = None
        if a.dump_outputs and rank == 0:
            # expected bytes of one of this rank's two files: its reads / 2 records of ~(header + bases + '+' + qualities) bytes
            sample = FastqSample(2, config["reads_per_step"] / world / 2 * (2 * READ_LEN + 20))
        l0 = g.stats()["kernel_launches"]
        clocks = ClockSampler(device); clocks.start()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        emit_ms = emit_n = reads_ms = amp_ms = alloc_ms = 0.0
        barrier(); ev0.record(); t0 = time.perf_counter()
        for i in range(a.steps):
            if sample and i == a.steps - 1:   # the last timed step hands its FASTQ to the sampling sink instead of discarding it
                g.amplify().set_read_counts()._ck(api.lib().scs_yield_reads_sink(g._h, sample.fn, None))
            else:
                step_resident()
            st = g.stats()
            emit_ms += st["ms_emit_kernel"]; emit_n += st["emit_launches"]; reads_ms += st["ms_reads"]; amp_ms += st["ms_amplify"]; alloc_ms += st["ms_alloc"]
        ev1.record(); barrier(); wall = time.perf_counter() - t0
        # the library works on its own streams: the torch events bracket host-synchronous calls, so use the larger of the two clocks
        dev_s = max(ev0.elapsed_time(ev1) / 1e3, wall)
        clk = clocks.stop()
        st = g.stats()
        launches = st["kernel_launches"] - l0
        reads_per_step = st["records"]   # FASTQ records actually written by this rank (both files)
        fastq_bytes = st["fastq_bytes"][0] + st["fastq_bytes"][1]
        plain_bytes = st["plain_bytes"][0] + st["plain_bytes"][1]
        n_fulls, n_semis = st["n_fulls_global"], st["n_semis_global"]
        if sample:
            sample.save(a.dump_outputs, st)

        # ---- e2e leg (host buffers in, host bytes out); one untimed pass first (page faults of the host side)
        step_e2e()
        barrier(); t0 = time.perf_counter()
        e2e_steps = max(1, min(a.steps, 3))
        for _ in range(e2e_steps):
            step_e2e()
        barrier(); e2e_s = time.perf_counter() - t0
        g.close()

        tmax = torch.tensor([dev_s, e2e_s, reads_ms], dtype=torch.float64, device=dev)
        tot = torch.tensor([float(reads_per_step), float(fastq_bytes), float(launches)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX); dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        dev_s, e2e_s, reads_ms_max = tmax.tolist(); reads_all, bytes_all, launches_all = tot.tolist()
        shares = gather_f64(reads_per_step)
        value = reads_all * a.steps / dev_s / 1e6
        e2e_value = reads_all * e2e_steps / e2e_s / 1e6

        # ---- bounded extras on rank 0's GPU: BASELINE configs[1] and the file-writing drop-in call
        extras = {}
        if rank == 0 and not a.no_extras:
            from scssim_b200.synth import synth_sequence
            c1len = max(1_000_000, int(C1_LEN * a.scale))
            seq = torch.empty(c1len, dtype=torch.uint8, pin_memory=True).numpy(); dummy = torch.empty(c1len, dtype=torch.uint8, pin_memory=True).numpy()
            synth_chromosome_cuda(torch, c1len, 7100, dev, seq, dummy)
            del dummy
            g1 = api.GenReads(gamma=GAMMA, coverage=C1_COVERAGE, isize=ISIZE, layout="PE", seed=0x5C55, device=device, slab_bytes=a.slab_mb << 20, io_threads=8)
            g1.load_profile(profile).set_genome([(f"chrS1_1_{c1len}", seq)]).create_frags()
            for _ in range(2):
                g1.amplify().set_read_counts().yield_reads_discard()
            torch.cuda.synchronize(); t0 = time.perf_counter()
            for _ in range(3):
                g1.amplify().set_read_counts().yield_reads_discard()
            c1_s = (time.perf_counter() - t0) / 3
            s1 = g1.stats()
            extras["configs1"] = {"workload": "BASELINE configs[1]: synthetic 250 Mb haploid, PE150 10x (-c 20), same profile/gamma" + ("" if a.scale == 1.0 else f" DEBUG scale {a.scale}"),
                                  "value": s1["records"] / c1_s / 1e6, "unit": UNIT, "ms_per_step": c1_s * 1e3,
                                  "fastq_GBps": (s1["fastq_bytes"][0] + s1["fastq_bytes"][1]) / c1_s / 1e9, "steps": 3, "warmup": 2}
            # the same cell with block-gzip output (BGZF members deflated on the device): fewer bytes over PCIe
            gz1 = api.GenReads(gamma=GAMMA, coverage=C1_COVERAGE, isize=ISIZE, layout="PE", seed=0x5C55, device=device, slab_bytes=a.slab_mb << 20, gzip=True)
            gz1.load_profile(profile).set_genome([(f"chrS1_1_{c1len}", seq)]).create_frags()
            for _ in range(2):
                gz1.amplify().set_read_counts().yield_reads_discard()
            torch.cuda.synchronize(); t0 = time.perf_counter()
            for _ in range(3):
                gz1.amplify().set_read_counts().yield_reads_discard()
            gz_s = (time.perf_counter() - t0) / 3
            sg = gz1.stats()
            extras["configs1_gz"] = {"workload": extras["configs1"]["workload"] + ", block-gzip output (gzip = 1; not the reference's format)", "value": sg["records"] / gz_s / 1e6,
                                     "unit": UNIT, "ms_per_step": gz_s * 1e3, "compressed_GBps": sum(sg["fastq_bytes"]) / gz_s / 1e9,
                                     "plain_equivalent_GBps": sum(sg["plain_bytes"]) / gz_s / 1e9, "ratio": sum(sg["plain_bytes"]) / max(1, sum(sg["fastq_bytes"])),
                                     "read_stage_kernels_ms": sg["ms_reads_kernels"], "read_stage_ms": sg["ms_reads"]}
            gz1.close()
            # files: <prefix>_1.fq / <prefix>_2.fq through scs_yield_reads (asynchronous sink, O_DIRECT where the file system has it)
            fdir = a.files_dir or tmp
            files = {}
            for label, d in (("tmp", fdir), ("shm", "/dev/shm")):
                if not os.path.isdir(d) or (label == "shm" and a.files_dir):
                    continue
                need = (s1["fastq_bytes"][0] + s1["fastq_bytes"][1]) * 1.05
                try:
                    sv = os.statvfs(d)
                    if sv.f_bavail * sv.f_frsize < need:
                        files[label] = {"skipped": f"needs {need / 1e9:.1f} GB free in {d}"}
                        continue
                except OSError:
                    continue
                prefix = os.path.join(d, f"scs_bench_{os.getpid()}")
                try:
                    g1.set_genome([(f"chrS1_1_{c1len}", seq)]).create_frags().amplify().set_read_counts().yield_reads(prefix)   # untimed pass
                    torch.cuda.synchronize(); t0 = time.perf_counter()
                    g1.set_genome([(f"chrS1_1_{c1len}", seq)]).create_frags().amplify().set_read_counts().yield_reads(prefix)
                    fs = time.perf_counter() - t0
                    sz = sum(os.path.getsize(prefix + sfx) for sfx in ("_1.fq", "_2.fq"))
                    files[label] = {"value": g1.stats()["records"] / fs / 1e6, "unit": UNIT, "file_GBps": sz / fs / 1e9, "file_bytes": sz, "dir": d, "s": fs}
                finally:
                    for sfx in ("_1.fq", "_2.fq"):
                        if os.path.exists(prefix + sfx):
                            os.remove(prefix + sfx)
            extras["e2e_files"] = {"workload": extras["configs1"]["workload"], "through": "scs_yield_reads(prefix): host ASCII genome in, <prefix>_1.fq/_2.fq out",
                                   **files}
            g1.close()

        cpu = None
        if rank == 0 and not a.no_cpu_baseline:
            r = run_reference_cpu(tmp, profile, 2, 0, a.coverage, REF_SAMPLE_CHROM if a.scale >= 1.0 else max(200_000, int(REF_SAMPLE_CHROM * a.scale)))
            cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"], "s_per_sample": r["s_per_step"],
                   "stage_s": r["stage_s"], "reads_stage_value": r["reads_stage_value"], "reads_per_sample": r["reads_per_step"],
                   "extrapolated_full_cell_s": r["extrapolated_full_cell_s"]}

    if rank == 0:
        peak, peak_src = measured_hbm_peak()
        # algorithmic HBM bytes of one emit launch (DESIGN.md "emit_kernel"): FASTQ bytes stored (into the staging buffer) + 2-bit
        # genome windows read (ceil(L/4) B per read) + 16 B descriptor per amplicon touched + 8 B of record sizes per slot;
        # rank 0's launches (all ranks run the same kernel on their slot range)
        slots = reads_per_step / 2
        alg_step = fastq_bytes + reads_per_step * ((READ_LEN + 3) // 4) + 16 * n_fulls * (reads_per_step / max(reads_all, 1)) + 8 * slots
        traffic = None
        try:   # dram__bytes_read+write of one emit launch from the committed ncu --set full capture of this same command
            with open(os.path.join(ROOT, "profiles", "emit_traffic.json")) as f:
                traffic = json.load(f)["dram_bytes_per_launch"]
        except (OSError, KeyError, ValueError):
            pass
        emit_launches_per_step = emit_n / a.steps if a.steps else 0
        emit_ms_avg = emit_ms / emit_n if emit_n else None
        achieved = (alg_step / emit_launches_per_step) / (emit_ms_avg / 1e3) / 1e9 if emit_ms_avg else None
        gbps = bytes_all * a.steps / dev_s / 1e9
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": dev_s / a.steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": config,
            "detail": {"dump_outputs": sample is not None, "reads_per_step": reads_all, "fastq_bytes_per_step": bytes_all, "fastq_GBps": gbps, "gzip": bool(a.gz), "plain_bytes_per_step_rank0": plain_bytes, "full_amplicons": n_fulls, "semi_amplicons": n_semis,
                       "stage_ms_per_step_rank0": {"amplify": amp_ms / a.steps, "alloc": alloc_ms / a.steps, "reads": reads_ms / a.steps},
                       "reads_stage_ms_max_rank": reads_ms_max / a.steps,
                       "parallelism": (f"one cell over {world} GPUs: sequences sharded for the amplification, packed genome + amplicon table all-gathered "
                                       f"over NCCL inside the library (v{api.lib().scs_nccl_version()}), read slots cut into {world} contiguous ranges") if world > 1 else "one GPU",
                       "device_map": devmap, "relay": {"rank_via_rank": {str(k): v for k, v in relay_map.items()},
                                                         "note": "these ranks copy their FASTQ slabs over NVLink to the peer's GPU, which copies them to the host"} if relay_map else None,
                       "share_of_reads_per_rank": [round(s / max(reads_all, 1), 4) for s in shares],
                       "shard_weight_history": weights_hist[-3:]},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": config["genome_bases"], "d2h_bytes_per_step": bytes_all, "steps": e2e_steps,
                    "fastq_GBps": bytes_all * e2e_steps / e2e_s / 1e9, "this_rank_h2d_bytes": h2d_bytes, "last_step_ms_rank0": e2e_parts},
            "gpu_launches": int(launches_all),
            "roofline": {"bound": "hbm", "kernel": "emit_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
                         "traffic": traffic, "algorithmic_bytes_per_launch": (alg_step / emit_launches_per_step) if emit_launches_per_step else None, "peak_source": peak_src,
                         "launches_per_step": emit_launches_per_step, "avg_launch_ms": emit_ms_avg,
                         "kernel_share_of_step": (emit_ms / a.steps) / (dev_s / a.steps * 1e3) if dev_s else None,
                         "d2h": {"bound": "pcie", "achieved": gbps, "unit": "GB/s (all GPUs)",
                                 "peak": d2h_peak, "frac": (gbps / d2h_peak) if d2h_peak else None,
                                 "peak_n_x_single_link": world * d2h_single, "frac_of_n_x_single_link": gbps / (world * d2h_single) if d2h_single else None,
                                 "single_gpu_link": d2h_single, "per_gpu_concurrent": [round(x, 1) for x in d2h_per_rank],
                                 "peak_of_links_used_with_relay": d2h_relay_peak, "frac_of_links_used_with_relay": (gbps / d2h_relay_peak) if d2h_relay_peak else None,
                                 "note": "FASTQ bytes landing in pinned host memory over the whole step. `peak` = pinned D2H copy rate measured in this run with all "
                                         "ranks copying at once (what this box's host side can absorb); `peak_n_x_single_link` = N x the rate of one GPU copying "
                                         "alone. This, not HBM, is the binding roof of the path"}},
            "cpu_baseline": cpu, "clocks": clk,
        }
        out.update(extras)
        emit(out)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
