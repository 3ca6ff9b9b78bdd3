"""Free-running parity (BASELINE north_star, correctness part 2): CUDA output (Philox) against the reference's own
free-running output (mt19937 / rand(), clock seeded) must match distributionally on the same genome and flags:
read-length spectrum (indel model), per-position quality distributions (KS), substitution rate per cycle band,
insert-size distribution (KS), read GC content (GC-bias-weighted allocation) and amplicon counts.
Tolerances are stated next to each check; sample = ~190 k reads per implementation."""
import os
import subprocess

import numpy as np
import pytest

import helpers as H

pytestmark = pytest.mark.gpu
RL = 125
CODE = np.full(256, 4, dtype=np.uint8)
CODE[np.frombuffer(b"ACGT", dtype=np.uint8)] = np.arange(4, dtype=np.uint8)


def _parse(fq: bytes):
    lines = fq.split(b"\n")[:-1]
    return lines[0::4], lines[1::4], lines[3::4]


def _seed_index(genome, k=24):
    idx = {}
    for sid, (_, s) in enumerate(genome):
        b = s.tobytes()
        for i in range(0, len(b) - k + 1):
            idx.setdefault(b[i:i + k], (sid, i))
    return idx


def _revcomp(b: bytes) -> bytes:
    return b.translate(bytes.maketrans(b"ACGT", b"TGCA"))[::-1]


def _map_full_length(genome, idx, seqs, k=24, off=50):
    """Exact-seed mapping of reads without indels; returns per-read (strand, seq id, start) or None."""
    out = []
    for s in seqs:
        if len(s) != RL:
            out.append(None); continue
        hit = idx.get(s[off:off + k])
        if hit is not None:
            out.append((0, hit[0], hit[1] - off)); continue
        r = _revcomp(s)
        hit = idx.get(r[RL - off - k:RL - off])
        out.append((1, hit[0], hit[1] - (RL - off - k)) if hit is not None else None)
    return out


def _mismatch_profile(genome, seqs, maps):
    mm = np.zeros(RL); n = 0
    arrs = [g[1] for g in genome]
    for s, m in zip(seqs, maps):
        if m is None:
            continue
        strand, sid, st = m
        if st < 0 or st + RL > len(arrs[sid]):
            continue
        ref = arrs[sid][st:st + RL]
        q = np.frombuffer(s if strand == 0 else _revcomp(s), dtype=np.uint8)
        d = (q != ref)
        mm += d if strand == 0 else d[::-1]
        n += 1
    return mm, n


def _stats(genome, idx, fq1, fq2):
    h1, s1, q1 = _parse(fq1)
    h2, s2, q2 = _parse(fq2)
    assert len(h1) == len(h2)
    st = {}
    lens = np.array([len(s) for s in s1] + [len(s) for s in s2])
    st["n"] = len(lens)
    st["len_hist"] = np.bincount(np.clip(lens - RL + 40, 0, 80), minlength=81)
    full1 = [q for q in q1 if len(q) == RL]
    st["qual1"] = np.frombuffer(b"".join(full1), dtype=np.uint8).reshape(-1, RL).astype(np.int16) - 33
    full2 = [q for q in q2 if len(q) == RL]
    st["qual2"] = np.frombuffer(b"".join(full2), dtype=np.uint8).reshape(-1, RL).astype(np.int16) - 33
    m1 = _map_full_length(genome, idx, s1)
    m2 = _map_full_length(genome, idx, s2)
    st["mm1"], st["nmap1"] = _mismatch_profile(genome, s1, m1)
    st["mm2"], st["nmap2"] = _mismatch_profile(genome, s2, m2)
    ins = []
    for a, b in zip(m1, m2):
        if a is not None and b is not None and a[1] == b[1] and a[0] != b[0]:
            lo = min(a[2], b[2]); hi = max(a[2], b[2]) + RL
            ins.append(hi - lo)
    st["isize"] = np.array(ins)
    # GC content per amplicon (reads of one amplicon are a cluster, so the amplicon is the sampling unit)
    amp = np.array([int(h.split(b"#")[0][1:]) for h in h1])
    keep = np.array([len(s) == RL for s in s1])
    mat = np.frombuffer(b"".join(s for s in s1 if len(s) == RL), dtype=np.uint8).reshape(-1, RL)
    gc_read = ((mat == 67) | (mat == 71)).mean(axis=1)
    a = amp[keep]
    cnt = np.bincount(a); tot = np.bincount(a, weights=gc_read)
    st["gc_amp"] = (tot[cnt > 0] / cnt[cnt > 0])
    st["gc_mean"] = gc_read.mean()
    st["reads_per_amp"] = cnt[cnt > 0]
    st["amp_max"] = int(amp.max())
    return st


def test_free_running_matches_reference_distributions(tmp_path):
    from scipy.stats import ks_2samp
    from scssim_b200 import api
    exe = H.ref_replay_bin()   # the seedable build: both sides of this test are then deterministic
    if exe is None:
        pytest.skip("needs the original SCSsim sources at BASELINE.json's reference_path or SCS_REFERENCE_DIR")
    tmp = str(tmp_path)
    fa = os.path.join(tmp, "cell.fa")
    genome = H.write_genome(fa, 1, 600_000, seed=23)
    prof = H.profile_path("Illumina_HiSeq2500")
    gamma, cov = 2e-10, 40.0
    subprocess.run([exe, "genreads", "-i", fa, "-t", "1", "-o", os.path.join(tmp, "ref")] + H.genreads_args(prof, "PE", gamma, cov, 260),
                   check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, env=dict(os.environ, SCS_SEED="424242"))
    with api.GenReads(gamma=gamma, coverage=cov, layout="PE", seed=20261018) as g:
        g.load_profile(prof).load_genome(fa).create_frags().amplify()
        g1, g2 = g.yield_reads_bytes()
    idx = _seed_index(genome)
    R = _stats(genome, idx, H.read_bytes(os.path.join(tmp, "ref_1.fq")), H.read_bytes(os.path.join(tmp, "ref_2.fq")))
    G = _stats(genome, idx, g1, g2)

    # number of reads: both implement reads = refLen*c/RL, PE parity may move it by a few
    assert abs(R["n"] - G["n"]) <= 4 and G["n"] > 150_000
    # read-length spectrum (indel model): P(len == RL) analytic 0.887 for HiSeq2500; 4-sigma binomial on the difference
    pr, pg = R["len_hist"] / R["n"], G["len_hist"] / G["n"]
    assert abs(pr[40] - pg[40]) < 4 * np.sqrt(2 * 0.887 * 0.113 / G["n"]) + 1e-9
    assert abs(pg[40] - 0.887) < 0.01
    assert np.abs(pr - pg).max() < 0.004            # every length bin within 0.4 % absolute
    # per-position quality: mean within 0.12 Phred everywhere; KS at five positions (alpha 1e-3)
    for key in ("qual1", "qual2"):
        assert np.abs(R[key].mean(axis=0) - G[key].mean(axis=0)).max() < 0.12
        for pos in (0, 30, 62, 100, 124):
            assert ks_2samp(R[key][:, pos], G[key][:, pos]).pvalue > 1e-3, (key, pos)
    # substitution rate (incl. MALBAC polymerase errors), total (< 5 %) and in four cycle bands (< 6 %; the band holding the mapping seed is skipped)
    np.set_printoptions(precision=5, suppress=True, linewidth=200)
    for mm, nm in (("mm1", "nmap1"), ("mm2", "nmap2")):
        rr, gg = R[mm] / R[nm], G[mm] / G[nm]
        print(mm, "mapped", R[nm], G[nm], "total rate", rr.sum(), gg.sum())
        print(" bands ref", [round(float(rr[b].sum()), 5) for b in np.array_split(np.arange(RL), 5)])
        print(" bands gpu", [round(float(gg[b].sum()), 5) for b in np.array_split(np.arange(RL), 5)])
        assert R[nm] > 0.8 * R["n"] / 2 * 0.85 and G[nm] > 0.8 * G["n"] / 2 * 0.85
        assert abs(rr.sum() - gg.sum()) / rr.sum() < 0.05, (rr.sum(), gg.sum())
        for bi, band in enumerate(np.array_split(np.arange(RL), 5)):
            if bi == 2:
                continue   # positions 50..74 hold the exact-match mapping seed: mismatching reads are unmapped there
            assert abs(rr[band].sum() - gg[band].sum()) / rr[band].sum() < 0.06
    # insert size: support [125, 397] (Profile.cpp:908-918), KS alpha 1e-3, means within 1.6 bp
    assert G["isize"].min() >= 125 and G["isize"].max() <= 397
    assert abs(R["isize"].mean() - G["isize"].mean()) < 1.6   # 4 sigma of the difference of two means (sd ~70, n ~61 k)
    assert ks_2samp(R["isize"], G["isize"]).pvalue > 1e-3
    # GC-bias-weighted allocation: GC of the amplicons that received reads (KS over amplicons, alpha 1e-3), read-weighted
    # mean GC within 0.8 % absolute, and the spread of reads per amplicon (driven by the N(gcMean, gcStd) factor) within 10 %
    assert ks_2samp(R["gc_amp"], G["gc_amp"]).pvalue > 1e-3
    assert abs(R["gc_mean"] - G["gc_mean"]) < 0.008
    cvr, cvg = R["reads_per_amp"].std() / R["reads_per_amp"].mean(), G["reads_per_amp"].std() / G["reads_per_amp"].mean()
    assert abs(cvr - cvg) / cvr < 0.10, (cvr, cvg)
    # amplicon tree size (number of full amplicons ~ highest header index). The tree grows from ~24 fragments by a
    # branching process (Poisson primers per template over 6 rounds), so its size has a coefficient of variation of ~20 %
    # between seeds on a genome this small: only the order of magnitude is comparable here (exact counts: replay tests).
    assert abs(R["amp_max"] - G["amp_max"]) / R["amp_max"] < 0.45


def test_polymerase_errors_of_free_running_amplification():
    """Free-running streams draw the distance to the next polymerase error (geometric) instead of the reference's one Bernoulli
    draw per base (Fragment.cpp:105-107, ber = 3.4e-4): the number of own substitutions of the semi amplicons must be
    Binomial(len - 8, ber) — total within 4 sigma, and the index of dispersion of the per-amplicon counts within 5 % of 1."""
    from scssim_b200 import api
    from scssim_b200.synth import synth_genome
    prof = H.profile_path("Illumina_HiSeq2500")
    with api.GenReads(gamma=1e-9, coverage=1.0, layout="SE", seed=77) as g:
        g.load_profile(prof).set_genome(synth_genome(2, 200_000, seed=3, diploid=True)).create_frags().amplify()
        semis = g.dump(api.DUMP_SEMIS).astype(np.int64)
    lens, nerr = semis[:, 2], semis[:, 5]
    assert len(semis) > 15_000
    ber = 3.4e-4
    expect = float(((lens - 8) * ber).sum())
    assert abs(nerr.sum() - expect) < 4 * np.sqrt(expect), (int(nerr.sum()), expect)
    # per-amplicon counts: binomial with n ~ 1500, p = ber -> variance ~ mean once the spread of the lengths is taken out
    resid = nerr - (lens - 8) * ber
    assert abs(resid.var() / nerr.mean() - 1.0) < 0.06, (resid.var(), nerr.mean())   # sd of the ratio ~ sqrt(2/n + 1/(n*mean)) ~ 1.6 %
    assert nerr.max() <= 8
