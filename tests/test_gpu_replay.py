"""Replay harness (BASELINE north_star, correctness part 1): the reference's own recorded random draws
are fed to the CUDA path, which must then write the reference's FASTQ byte for byte.

  reference (oracle/_ref/bin/scssim_replay -t 1, seeded)  -> FASTQ_ref + draw tapes
  CPU oracle in tape mode                                   -> FASTQ_orc (== FASTQ_ref) + per-entity tape offsets
  CUDA path with the tapes + offsets                        -> FASTQ_gpu  == FASTQ_ref

The live cases build the reference from the SCSsim sources at BASELINE.json's reference_path (or SCS_REFERENCE_DIR; or use a prebuilt,
git-ignored oracle/_ref) and skip without them; the committed golden case below needs neither.
"""
import os

import numpy as np
import pytest

import helpers as H

pytestmark = pytest.mark.gpu


def _replay_case(tmp, fa, profile, layout, gamma, coverage, isize, tape_prefix, ref_fastq):
    from scssim_b200 import api
    prof = H.profile_path(profile)
    args = H.genreads_args(prof, layout, gamma, coverage, isize)
    oprefix, dprefix = os.path.join(tmp, "orc"), os.path.join(tmp, "dump")
    H.run_oracle(fa, oprefix, args, tape_prefix=tape_prefix, dump_prefix=dprefix)
    for got, want in zip(H.fastq_names(oprefix, layout), ref_fastq):
        assert H.read_bytes(got) == H.read_bytes(want), "CPU oracle does not reproduce the reference FASTQ"
    tapes = api.ReplayTapes.load(tape_prefix, dprefix)
    od = H.oracle_dump(dprefix)
    with api.GenReads(gamma=gamma, coverage=coverage, isize=isize, layout=layout, seed=1) as g:
        g.load_profile(prof).load_genome(fa).set_replay(tapes).create_frags().amplify().set_read_counts()
        assert np.array_equal(g.dump(api.DUMP_COUNTS), od["counts"]), "read counts differ from the reference's"
        f1, f2 = g.yield_reads_bytes()
    assert f1 == H.read_bytes(ref_fastq[0]), "replay FASTQ (file 1) differs from the reference"
    if layout == "PE":
        assert f2 == H.read_bytes(ref_fastq[1]), "replay FASTQ (file 2) differs from the reference"


@pytest.mark.parametrize("profile,layout,gamma,coverage,isize,glen", [
    ("Illumina_HiSeq2500", "PE", 2e-10, 5.0, 260, 400_000),
    ("Illumina_HiSeq2000", "SE", 1e-9, 3.0, 260, 150_000),
    ("Illumina_HiSeqXTen", "PE", 2e-10, 4.0, 1200, 300_000),
])
def test_replay_against_live_reference(tmp_path, profile, layout, gamma, coverage, isize, glen):
    if H.ref_replay_bin() is None:
        pytest.skip("needs the original SCSsim sources at BASELINE.json's reference_path or SCS_REFERENCE_DIR")
    tmp = str(tmp_path)
    fa = os.path.join(tmp, "cell.fa")
    H.write_genome(fa, 1, glen, seed=11)
    tape = os.path.join(tmp, "tape")
    rprefix = os.path.join(tmp, "ref")
    H.run_reference_replay(fa, rprefix, tape, seed=77, args=H.genreads_args(H.profile_path(profile), layout, gamma, coverage, isize))
    _replay_case(tmp, fa, profile, layout, gamma, coverage, isize, tape, H.fastq_names(rprefix, layout))


def test_replay_golden_case(tmp_path):
    """Committed fixture: tapes + FASTQ produced by the reference in the build container
    (tests/golden/make_golden.py)."""
    import lzma
    tmp = str(tmp_path)
    gdir = os.path.join(H.GOLDEN, "replay_pe2500")
    meta = dict(l.strip().split("=") for l in open(os.path.join(gdir, "case.txt")))
    for name in os.listdir(gdir):
        if name.endswith(".xz"):
            with lzma.open(os.path.join(gdir, name)) as f, open(os.path.join(tmp, name[:-3]), "wb") as o:
                o.write(f.read())
    fa = os.path.join(tmp, "cell.fa")
    _replay_case(tmp, fa, meta["profile"], meta["layout"], float(meta["gamma"]), float(meta["coverage"]), int(meta["isize"]),
                 os.path.join(tmp, "tape"), [os.path.join(tmp, "ref_1.fq"), os.path.join(tmp, "ref_2.fq")])
