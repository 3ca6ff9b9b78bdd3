"""host_expand: slabs sent as packed base+quality records and expanded by host threads give the same FASTQ bytes as slabs sent
as text, on every path choice (0 text only, 1 every slab packed, 2 alternate, -1 chosen per slab)."""
import os
import threading

import pytest

import helpers as H

pytestmark = pytest.mark.gpu

MODES = (0, 1, 2, -1)


def _all_modes(run):
    """run(host_expand) -> ((file1, file2), stats) for every mode; asserts identical bytes and the link accounting."""
    out = {hx: run(hx) for hx in MODES}
    ref, st0 = out[0]
    assert len(ref[0]) > 0
    for hx in MODES:
        fq, st = out[hx]
        assert fq[0] == ref[0] and fq[1] == ref[1], f"host_expand={hx}: FASTQ differs from the text path"
        assert st["fastq_bytes"] == st0["fastq_bytes"] and st["plain_bytes"] == st0["plain_bytes"] and st["records"] == st0["records"]
    assert out[0][1]["slabs_packed"] == 0 and out[0][1]["link_bytes"] == out[0][1]["fastq_bytes"]
    st1 = out[1][1]
    assert st1["slabs_packed"] == st1["slabs"] > 0
    assert sum(st1["link_bytes"]) < sum(st1["fastq_bytes"])
    st2 = out[2][1]
    assert st2["slabs_packed"] == st2["slabs"] // 2
    return out


def _genreads(prof, genome, layout, slab, **kw):
    from scssim_b200 import api

    def run(hx):
        with api.GenReads(gamma=3e-10, coverage=kw.get("coverage", 12.0), layout=layout, seed=kw.get("seed", 17), slab_bytes=slab, host_expand=hx,
                          expand_threads=kw.get("threads", 3)) as g:
            g.load_profile(prof)
            (g.load_genome(genome) if isinstance(genome, str) else g.set_genome(genome)).create_frags().amplify()
            fq = g.yield_reads_bytes()
            return fq, g.stats()
    return run


@pytest.mark.parametrize("layout", ["PE", "SE"])
def test_paths_agree_many_slabs(tmp_path, layout):
    fa = os.path.join(str(tmp_path), "cell.fa")
    H.write_genome(fa, 1, 300_000, seed=31)
    out = _all_modes(_genreads(H.profile_path("Illumina_HiSeq2500"), fa, layout, 64 << 10))
    assert out[1][1]["slabs"] >= 20


def test_paths_agree_default_slab_and_oracle(tmp_path):
    fa = os.path.join(str(tmp_path), "cell.fa")
    H.write_genome(fa, 2, 200_000, seed=5)
    prof = H.profile_path("Illumina_HiSeq2500")
    out = _all_modes(_genreads(prof, fa, "PE", 0, coverage=8.0, seed=0x5C55))
    oprefix = os.path.join(str(tmp_path), "orc")
    H.run_oracle(fa, oprefix, H.genreads_args(prof, "PE", 3e-10, 8.0, 260), seed=0x5C55)
    names = H.fastq_names(oprefix, "PE")
    assert out[1][0][0] == H.read_bytes(names[0]) and out[1][0][1] == H.read_bytes(names[1])


def test_paths_agree_n_iupac_genome(tmp_path):
    genome = H.write_genome_with_n(os.path.join(str(tmp_path), "n.fa"), 300_000, 77)
    _all_modes(_genreads(H.profile_path("Illumina_HiSeq2500"), genome, "PE", 256 << 10))


def test_paths_agree_wide_quality_profile(tmp_path):
    """A profile whose qualities span more than 64 Phred values: records with a quality outside the packed range go verbatim."""
    src = open(H.profile_path("Illumina_HiSeq2500")).read().split("\n")
    i = src.index("[Base Quality Distribution]")
    for j in range(i + 1, len(src)):
        if src[j].startswith("["):
            break
        v = src[j].split("\t")
        if len(v) == 94 and sum(float(x) for x in v) > 0:
            w = [float(x) * 0.99 for x in v]
            w[2] += 0.008; w[80] += 0.002   # about one read in four draws a quality of 80
            src[j] = "\t".join(f"{x:g}" for x in w)
    prof = os.path.join(str(tmp_path), "wide.profile")
    open(prof, "w").write("\n".join(src))
    fa = os.path.join(str(tmp_path), "cell.fa")
    H.write_genome(fa, 1, 200_000, seed=8)
    out = _all_modes(_genreads(prof, fa, "PE", 256 << 10))
    fq = out[1][0][0]
    assert chr(33 + 80).encode() in fq and chr(33 + 2).encode() in fq


def test_replay_golden_case_packed(tmp_path):
    """The committed replay fixture with every slab packed equals the reference's FASTQ."""
    import lzma
    from scssim_b200 import api
    tmp = str(tmp_path)
    gdir = os.path.join(H.GOLDEN, "replay_pe2500")
    meta = dict(l.strip().split("=") for l in open(os.path.join(gdir, "case.txt")))
    for name in os.listdir(gdir):
        if name.endswith(".xz"):
            with lzma.open(os.path.join(gdir, name)) as f, open(os.path.join(tmp, name[:-3]), "wb") as o:
                o.write(f.read())
    prof = H.profile_path(meta["profile"])
    args = H.genreads_args(prof, meta["layout"], float(meta["gamma"]), float(meta["coverage"]), int(meta["isize"]))
    fa, dprefix = os.path.join(tmp, "cell.fa"), os.path.join(tmp, "dump")
    H.run_oracle(fa, os.path.join(tmp, "orc"), args, tape_prefix=os.path.join(tmp, "tape"), dump_prefix=dprefix)
    tapes = api.ReplayTapes.load(os.path.join(tmp, "tape"), dprefix)
    for hx in (1, 2):
        with api.GenReads(gamma=float(meta["gamma"]), coverage=float(meta["coverage"]), isize=int(meta["isize"]), layout=meta["layout"], seed=1,
                          slab_bytes=64 << 10, host_expand=hx, expand_threads=2) as g:
            g.load_profile(prof).load_genome(fa).set_replay(tapes).create_frags().amplify().set_read_counts()
            f1, f2 = g.yield_reads_bytes()
            assert g.stats()["slabs_packed"] > 0
        assert f1 == H.read_bytes(os.path.join(tmp, "ref_1.fq")) and f2 == H.read_bytes(os.path.join(tmp, "ref_2.fq")), f"host_expand={hx}"


def test_two_ranks_packed_concatenate_to_one_rank(tmp_path):
    from scssim_b200 import api
    from scssim_b200.dist import ThreadCollectives
    prof = H.profile_path("Illumina_HiSeq2500")
    genome = H.write_genome_with_n(os.path.join(str(tmp_path), "n.fa"), 200_000, 19)
    kw = dict(gamma=3e-10, coverage=5.0, layout="PE", seed=4321, slab_bytes=64 << 10)
    with api.GenReads(host_expand=0, **kw) as g:
        g.load_profile(prof).set_genome(genome).create_frags().amplify()
        one = g.yield_reads_bytes()
    world = 2
    coll = ThreadCollectives(world)
    out, errs = [None] * world, []

    def run(rank):
        try:
            with api.GenReads(rank=rank, world=world, balance=True, host_expand=1, expand_threads=2, **kw) as g:
                g.set_collectives(*coll.pair())
                g.set_device_collective(*coll.device_pair())
                g.load_profile(prof).set_genome(genome[rank:rank + 1]).create_frags().amplify()
                out[rank] = (g.yield_reads_bytes(), g.stats())
        except Exception as e:  # noqa: BLE001
            errs.append(e)
            coll.bar.abort()

    ts = [threading.Thread(target=run, args=(r,)) for r in range(world)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert not errs, errs
    for f in range(2):
        assert out[0][0][f] + out[1][0][f] == one[f], f"file {f}"
    assert all(o[1]["slabs_packed"] == o[1]["slabs"] > 0 for o in out)


def test_discard_sink_expands(tmp_path):
    """The null sink (what the benchmark times) expands its packed slabs too: the pool's work is part of the stage."""
    from scssim_b200 import api
    fa = os.path.join(str(tmp_path), "cell.fa")
    H.write_genome(fa, 1, 300_000, seed=31)
    with api.GenReads(gamma=3e-10, coverage=12.0, layout="PE", seed=17, slab_bytes=64 << 10, host_expand=1, expand_threads=2) as g:
        g.load_profile(H.profile_path("Illumina_HiSeq2500")).load_genome(fa).create_frags().amplify()
        g.yield_reads_discard()
        st = g.stats()
        fq = g.yield_reads_bytes()
    assert st["slabs_packed"] == st["slabs"] > 0 and st["fastq_bytes"] == [len(fq[0]), len(fq[1])]
