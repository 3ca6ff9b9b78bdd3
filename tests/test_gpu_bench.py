"""bench.py on a small debug cell: `--steps` sets the number of timed steps, and `--dump-outputs` writes a fixed sample of the
FASTQ of the last timed step that is the same from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import helpers as H

pytestmark = pytest.mark.gpu
NAMES = ["fastq_1.npy", "fastq_2.npy", "fastq_bytes.npy", "fastq_offsets.npy"]


def _bench(out, steps, warmup):
    r = subprocess.run([sys.executable, os.path.join(H.ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup),
                        "--scale", "0.002", "--coverage", "4", "--no-cpu-baseline", "--no-extras", "--dump-outputs", out],
                       capture_output=True, timeout=900)
    assert r.returncode == 0, r.stderr.decode()[-3000:]
    lines = [l for l in r.stdout.decode().splitlines() if l.strip()]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_synthetic_cell_is_a_function_of_its_seed(monkeypatch):
    """The benchmark's cell generator on the GPU: haplotype 2 is haplotype 1 with the drawn substitutions applied as numpy applies
    them (a position drawn twice takes its last draw), so the cell is the same on every run. A dense SNP rate makes repeats certain."""
    import torch
    import bench
    monkeypatch.setattr(bench, "SNP_RATE", 0.6)
    n = 3_000_000
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    gen = torch.Generator(device="cuda:0"); gen.manual_seed(5)            # the generator's draws, replayed
    gcs = 0.35 + 0.25 * torch.rand((n + 99_999) // 100_000, generator=gen, device="cuda:0")
    is_gc = torch.rand(n, generator=gen, device="cuda:0") < gcs[torch.arange(n, device="cuda:0") // 100_000]
    pick = torch.randint(0, 2, (n,), generator=gen, device="cuda:0", dtype=torch.uint8)
    code = torch.where(is_gc, 1 + pick, 3 * pick).cpu().numpy().astype(np.int64)
    pos = torch.randint(0, n, (int(n * 0.6),), generator=gen, device="cuda:0").cpu().numpy()
    shift = torch.randint(1, 4, (int(n * 0.6),), generator=gen, device="cuda:0", dtype=torch.uint8).cpu().numpy()
    alt = code.copy()
    alt[pos] = (code[pos] + shift) & 3
    assert len(np.unique(pos)) < len(pos)
    for _ in range(2):
        h1, h2 = np.empty(n, dtype=np.uint8), np.empty(n, dtype=np.uint8)
        bench.synth_chromosome_cuda(torch, n, 5, "cuda:0", h1, h2)
        assert np.array_equal(h1, lut[code]) and np.array_equal(h2, lut[alt])


def test_dump_outputs_sample_the_last_timed_step(tmp_path):
    d1, d3 = str(tmp_path / "s1"), str(tmp_path / "s3")
    j1, j3 = _bench(d1, 1, 1), _bench(d3, 3, 2)
    assert j1["steps"] == 1 and j3["steps"] == 3 and j1["detail"]["dump_outputs"] is True
    assert j3["gpu_launches"] == 3 * j1["gpu_launches"] > 0          # every timed step launches the same kernels
    assert sorted(os.listdir(d1)) == NAMES == sorted(os.listdir(d3))
    assert sum(os.path.getsize(os.path.join(d1, n)) for n in NAMES) <= 64 << 20
    for n in NAMES:
        a, b = np.load(os.path.join(d1, n)), np.load(os.path.join(d3, n))
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), n
    nbytes = np.load(os.path.join(d1, "fastq_bytes.npy"))
    assert nbytes[0] + nbytes[1] == j1["detail"]["fastq_bytes_per_step"] and nbytes[2] == j1["detail"]["reads_per_step"]
    offsets = np.load(os.path.join(d1, "fastq_offsets.npy"))
    for f in (0, 1):
        s = np.load(os.path.join(d1, NAMES[f]))
        inside, past = offsets + s.shape[1] <= nbytes[f], offsets >= nbytes[f]
        assert inside.sum() > 1000 and past.sum() + inside.sum() <= len(offsets)
        text = s[inside]
        assert ((text == 10) | ((text >= 33) & (text <= 126))).all()      # FASTQ: printable characters and line ends only
        assert (s[past] == -1).all()
