"""Generates tests/golden/simuvars_small/: random inputs + the output of the REFERENCE binary itself
(oracle/_ref/bin/scssim simuvars, built by oracle/build_ref.sh from the SCSsim sources at BASELINE.json's reference_path,
or at $SCS_REFERENCE_DIR when set):  python tests/golden/make_simuvars_golden.py
"""
import hashlib
import json
import lzma
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import helpers as H  # noqa: E402

out = os.path.join(HERE, "simuvars_small")
os.makedirs(out, exist_ok=True)
with tempfile.TemporaryDirectory() as d:
    ref, snp, var = H.make_simuvars_case(d, 2024, chrom_lens=(40_000, 12_000), n_snp=200, n_snv=30, n_ins=30, n_del=30, n_cnv=5)
    r = H.run_reference_simuvars(ref, snp, var, os.path.join(d, "expected.fa"))
    assert r.returncode == 0, r.stderr.decode()
    for f in ("ref.fa", "snp.txt", "vars.txt", "expected.fa"):
        with open(os.path.join(d, f), "rb") as i, lzma.open(os.path.join(out, f + ".xz"), "wb", preset=9) as o:
            o.write(i.read())
    exp = H.read_bytes(os.path.join(d, "expected.fa"))
    json.dump({"sha256": hashlib.sha256(exp).hexdigest(), "bytes": len(exp), "generator": "oracle/_ref/bin/scssim simuvars (reference binary)",
               "case": "make_simuvars_case(seed=2024, chrom_lens=(40000, 12000), n_snp=200, n_snv=30, n_ins=30, n_del=30, n_cnv=5)"},
              open(os.path.join(out, "meta.json"), "w"), indent=1)
print("wrote", out)
