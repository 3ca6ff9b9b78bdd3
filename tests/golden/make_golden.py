"""Regenerates tests/golden/replay_pe2500 by running the reference itself (oracle/_ref/bin/scssim_replay,
built by oracle/build_ref.sh from the SCSsim sources at BASELINE.json's reference_path, or at $SCS_REFERENCE_DIR
when set). Committed so the fixture's origin is reproducible:  python tests/golden/make_golden.py
"""
import lzma
import os
import shutil
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import helpers as H  # noqa: E402

CASE = dict(profile="Illumina_HiSeq2500", layout="PE", gamma=1.2e-10, coverage=2.0, isize=260, glen=45000, gseed=5, seed=2024)


def main():
    out = os.path.join(HERE, "replay_pe2500")
    shutil.rmtree(out, ignore_errors=True)
    os.makedirs(out)
    with tempfile.TemporaryDirectory() as tmp:
        fa = os.path.join(tmp, "cell.fa")
        H.write_genome(fa, 1, CASE["glen"], CASE["gseed"])
        args = H.genreads_args(H.profile_path(CASE["profile"]), CASE["layout"], CASE["gamma"], CASE["coverage"], CASE["isize"])
        H.run_reference_replay(fa, os.path.join(tmp, "ref"), os.path.join(tmp, "tape"), CASE["seed"], args)
        for name in ["cell.fa", "ref_1.fq", "ref_2.fq"] + [f"tape.{s}.bin" for s in ("wreal", "wint", "mrand", "mreal", "mint", "gcf")]:
            with open(os.path.join(tmp, name), "rb") as f, lzma.open(os.path.join(out, name + ".xz"), "wb", preset=6) as o:
                o.write(f.read())
    with open(os.path.join(out, "case.txt"), "w") as f:
        for k in ("profile", "layout", "gamma", "coverage", "isize"):
            f.write(f"{k}={CASE[k]}\n")
    print("wrote", out, sum(os.path.getsize(os.path.join(out, n)) for n in os.listdir(out)), "bytes")


if __name__ == "__main__":
    main()
