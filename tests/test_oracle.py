"""CPU tests of the oracle (test infrastructure) itself: it must reproduce what the reference produced.

* golden case: tapes + FASTQ written by the reference in the build container (tests/golden/make_golden.py);
* live cases: the compiled reference (oracle/_ref) is run here when present, with several profiles/layouts;
* Philox4x32-10 known-answer vectors (Random123) and the deterministic logarithm.
"""
import lzma
import math
import os

import numpy as np
import pytest

import helpers as H


def _unpack_golden(tmp):
    gdir = os.path.join(H.GOLDEN, "replay_pe2500")
    meta = dict(l.strip().split("=") for l in open(os.path.join(gdir, "case.txt")))
    for name in os.listdir(gdir):
        if name.endswith(".xz"):
            with lzma.open(os.path.join(gdir, name)) as f, open(os.path.join(tmp, name[:-3]), "wb") as o:
                o.write(f.read())
    return meta


def test_oracle_reproduces_golden_reference_fastq(tmp_path):
    tmp = str(tmp_path)
    meta = _unpack_golden(tmp)
    args = H.genreads_args(H.profile_path(meta["profile"]), meta["layout"], float(meta["gamma"]), float(meta["coverage"]), int(meta["isize"]))
    log = H.run_oracle(os.path.join(tmp, "cell.fa"), os.path.join(tmp, "orc"), args, tape_prefix=os.path.join(tmp, "tape"))
    assert '"tapes_consumed": true' in log
    assert H.read_bytes(os.path.join(tmp, "orc_1.fq")) == H.read_bytes(os.path.join(tmp, "ref_1.fq"))
    assert H.read_bytes(os.path.join(tmp, "orc_2.fq")) == H.read_bytes(os.path.join(tmp, "ref_2.fq"))


LIVE = [
    ("Illumina_HiSeq2500", "PE", 2e-10, 4.0, 260, 1, 200_000),
    ("Illumina_HiSeq2000", "SE", 1e-9, 2.0, 260, 2, 60_000),
    ("Illumina_HiSeqXTen", "PE", 2e-10, 3.0, 1200, 1, 200_000),
    ("Illumina_GenomeAnalyzerIIx", "PE", 5e-10, 3.0, 100, 1, 150_000),
    ("Illumina_HiSeq2500", "PE", 3e-10, 4.0, 1900, 1, 150_000),
]


@pytest.mark.parametrize("profile,layout,gamma,coverage,isize,nchrom,glen", LIVE)
def test_oracle_reproduces_live_reference(tmp_path, profile, layout, gamma, coverage, isize, nchrom, glen):
    if H.ref_replay_bin() is None:
        pytest.skip("needs the original SCSsim sources at BASELINE.json's reference_path or SCS_REFERENCE_DIR")
    tmp = str(tmp_path)
    fa = os.path.join(tmp, "cell.fa")
    H.write_genome(fa, nchrom, glen, seed=3, width=60)
    args = H.genreads_args(H.profile_path(profile), layout, gamma, coverage, isize)
    H.run_reference_replay(fa, os.path.join(tmp, "ref"), os.path.join(tmp, "tape"), seed=31, args=args)
    log = H.run_oracle(fa, os.path.join(tmp, "orc"), args, tape_prefix=os.path.join(tmp, "tape"))
    assert '"tapes_consumed": true' in log
    for a, b in zip(H.fastq_names(os.path.join(tmp, "orc"), layout), H.fastq_names(os.path.join(tmp, "ref"), layout)):
        assert H.read_bytes(a) == H.read_bytes(b)
        assert len(H.read_bytes(a)) > 0


def test_philox_known_answers():
    L = H.oracle_lib()
    kats = [  # Random123 kat_vectors, philox4x32-10
        ([0, 0, 0, 0], [0, 0], [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
        ([0xffffffff] * 4, [0xffffffff] * 2, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
        ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0], [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]),
    ]
    for ctr, key, want in kats:
        c = np.array(ctr, dtype=np.uint32); k = np.array(key, dtype=np.uint32); o = np.zeros(4, dtype=np.uint32)
        L.orc_philox(c.ctypes.data, k.ctypes.data, o.ctypes.data)
        assert [int(v) for v in o] == want


def test_det_log_accuracy():
    L = H.oracle_lib()
    rng = np.random.default_rng(1)
    xs = np.concatenate([rng.random(2000), 2.0 ** rng.uniform(-40, 0, 2000), [1.0, 0.5, 2 ** -32, 1 - 2 ** -32]])
    for x in xs:
        got = L.orc_det_log(float(x))
        want = math.log(x)
        assert abs(got - want) <= 4e-16 * max(1.0, abs(want)), (x, got, want)
    assert L.orc_det_log(0.0) == -math.inf


def _length_hist(fastq: bytes, rl: int):
    lines = fastq.split(b"\n")
    lens = np.array([len(s) for s in lines[1::4]], dtype=np.int64)
    return np.bincount(np.clip(lens - (rl - 40), 0, 80), minlength=81) / max(1, len(lens)), len(lens)


def test_oracle_free_running_indel_stage_keeps_the_read_length_spectrum(tmp_path):
    """Free-running streams draw the distance to the next indel event instead of the reference's two draws per read position
    (oracle/profile.h indel_geom; Profile.cpp:1603-1630). The read-length spectrum must stay what the per-position process gives:
    P(no event in 125 positions) = ((1 - pI)(1 - pD))^125 = 0.887 for HiSeq2500, and — when the compiled reference is here —
    every length bin within 0.6 % absolute of the seeded reference's."""
    tmp = str(tmp_path)
    fa = os.path.join(tmp, "cell.fa")
    H.write_genome(fa, 1, 300_000, seed=29)
    prof = H.profile_path("Illumina_HiSeq2500")
    args = H.genreads_args(prof, "PE", 2e-10, 30.0, 260)
    H.run_oracle(fa, os.path.join(tmp, "orc"), args, seed=987)
    rl = 125
    ho, n = _length_hist(H.read_bytes(os.path.join(tmp, "orc_1.fq")) + H.read_bytes(os.path.join(tmp, "orc_2.fq")), rl)
    assert n > 50_000
    assert abs(ho[40] - 0.887) < 0.01, ho[40]
    assert ho[:40].sum() > 0.02 and ho[41:].sum() > 0.02          # deletions and insertions both occur
    exe = H.ref_replay_bin()
    if exe is None:
        return
    import subprocess
    subprocess.run([exe, "genreads", "-i", fa, "-t", "1", "-o", os.path.join(tmp, "ref")] + args, check=True, stdout=subprocess.DEVNULL,
                   stderr=subprocess.DEVNULL, env=dict(os.environ, SCS_SEED="1234"))
    hr, nr = _length_hist(H.read_bytes(os.path.join(tmp, "ref_1.fq")) + H.read_bytes(os.path.join(tmp, "ref_2.fq")), rl)
    assert abs(n - nr) <= 4
    assert np.abs(ho - hr).max() < 0.006, (np.abs(ho - hr).argmax(), ho[38:43], hr[38:43])
