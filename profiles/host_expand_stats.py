#!/usr/bin/env python
"""Where the read stage of bench.py's cell sends its slabs with host_expand (scs_params): per mode, the read-stage time, the FASTQ
text bytes, the bytes that crossed the host link and the share of slabs sent packed. One JSON line per mode on stdout.

    python profiles/host_expand_stats.py [--scale 1.0] [--steps 2] [--modes=-1,0,1] [--threads 0]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--modes", default="-1,0,1")
    ap.add_argument("--threads", type=int, default=0, help="expand_threads (0: CPUs in the affinity mask - 1)")
    a = ap.parse_args()
    import torch
    import bench as B
    from scssim_b200 import api
    card = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    with tempfile.TemporaryDirectory() as tmp:
        profile = B.bench_profile(tmp)
        clen = int(B.CHROM_LEN * a.scale)
        named = []
        for c in range(B.N_CHROM):
            b1 = torch.empty(clen, dtype=torch.uint8, pin_memory=True).numpy(); b2 = torch.empty(clen, dtype=torch.uint8, pin_memory=True).numpy()
            B.synth_chromosome_cuda(torch, clen, 7000 + c, "cuda:0", b1, b2)
            named += [(f"chrS{c + 1}_1_{clen}", b1), (f"chrS{c + 1}_2_{clen}", b2)]
        for hx in (int(m) for m in a.modes.split(",")):
            with api.GenReads(gamma=B.GAMMA, coverage=B.COVERAGE, isize=B.ISIZE, layout="PE", seed=0x5C55, device=0, slab_bytes=64 << 20, host_expand=hx,
                             expand_threads=a.threads) as g:
                g.load_profile(profile).set_genome(named).create_frags()
                g.amplify().set_read_counts().yield_reads_discard()   # warm-up: pinned rings, pool threads
                rows = []
                for _ in range(a.steps):
                    g.amplify().set_read_counts()
                    t0 = time.perf_counter()
                    g.yield_reads_discard()
                    wall = time.perf_counter() - t0
                    st = g.stats()
                    text, link = sum(st["fastq_bytes"]), sum(st["link_bytes"])
                    rows.append({"reads_s": wall, "ms_reads": st["ms_reads"], "text_GB": text / 1e9, "link_GB": link / 1e9,
                                 "text_GBps": text / wall / 1e9, "link_GBps": link / wall / 1e9,
                                 "slabs": st["slabs"], "slabs_packed": st["slabs_packed"], "packed_share": st["slabs_packed"] / max(1, st["slabs"])})
                print(json.dumps({"card": card, "host_expand": hx, "expand_threads": a.threads, "scale": a.scale, "host_cpus": os.cpu_count(), "steps": rows}), flush=True)


if __name__ == "__main__":
    main()
