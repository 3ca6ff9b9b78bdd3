"""Host expansion of packed FASTQ slabs (scssim_b200/csrc/wire.h) against a Python decoder of the same format, without a GPU."""
import random
import struct

import pytest

from scssim_b200 import api

VERBATIM = 0xFF


def decode(records: bytes, qchar0: int) -> bytes:
    """Reference decoder: the format as wire.h states it."""
    out, i = bytearray(), 0
    while i < len(records):
        hl, n = records[i], records[i + 1] | records[i + 2] << 8
        i += 3
        if hl == VERBATIM:
            out += records[i:i + n]
            i += n
            continue
        out += records[i:i + hl]
        codes = records[i + hl:i + hl + n]
        out += bytes(b"ACGT"[c & 3] for c in codes) + b"\n+\n" + bytes(qchar0 + (c >> 2) for c in codes) + b"\n"
        i += hl + n
    return bytes(out)


def make_slab(rng: random.Random, nrec: int, every: int, verbatim=0.05, long_reads=False):
    """Records in slots, a split entry at every `every`-th slot (empty slots included), like the device packer lays them out."""
    recs, splits, wpos, tpos = bytearray(), [], 0, 0
    for slot in range(nrec):
        if slot % every == 0:
            splits.append((wpos, tpos))
        if rng.random() < 0.05:   # dropped slot: no record
            continue
        hdr = f"@{rng.randrange(10**7)}#{rng.randrange(1, 3000)}/{rng.randint(1, 2)}\n".encode()
        n = rng.randrange(1000, 2000) if long_reads and rng.random() < 0.2 else rng.randrange(0, 320)
        if rng.random() < verbatim:
            text = hdr + bytes(rng.choice(b"ACGTNRY") for _ in range(n)) + b"\n+\n" + bytes(rng.randrange(33, 127) for _ in range(n)) + b"\n"
            rec = struct.pack("<BH", VERBATIM, len(text)) + text
        else:
            rec = struct.pack("<BH", len(hdr), n) + hdr + bytes(rng.randrange(256) for _ in range(n))
            text = decode(rec, 40)
        recs += rec
        wpos += len(rec)
        tpos += len(text)
    table = b"".join(struct.pack("<QQ", w, t) for w, t in splits)
    return table + bytes(recs), len(splits), bytes(recs), tpos


@pytest.mark.parametrize("threads", [1, 2, 3, 8])
@pytest.mark.parametrize("scalar", [False, True])
def test_expand_matches_reference(threads, scalar):
    rng = random.Random(threads * 7 + scalar)
    for nrec, every in ((1, 2048), (5, 2), (700, 64), (3000, 2048), (2500, 37)):
        wire, nsplit, recs, text_bytes = make_slab(rng, nrec, every, long_reads=nrec == 700)
        got = api.expand_wire(wire, nsplit, text_bytes, qchar0=40, threads=threads, scalar=scalar)
        assert got == decode(recs, 40)


def test_expand_empty_pieces_and_empty_slab():
    # pieces of 0 bytes (every slot of a split dropped) and a slab without records
    hdr = b"@1#2/1\n"
    rec = struct.pack("<BH", len(hdr), 3) + hdr + bytes([0, 5, 10])
    table = struct.pack("<QQ", 0, 0) * 3 + struct.pack("<QQ", len(rec), 7 + 2 * 3 + 4)
    wire = table + rec + rec
    out = api.expand_wire(wire, 4, 2 * (7 + 10), qchar0=33, threads=4)
    assert out == (b"@1#2/1\nACG\n+\n!\"#\n") * 2
    assert api.expand_wire(struct.pack("<QQ", 0, 0), 1, 0, threads=2) == b""


def test_expand_rejects_malformed_slab():
    hdr = b"@1#2/1\n"
    rec = struct.pack("<BH", len(hdr), 50) + hdr + bytes(10)   # 40 codes short
    with pytest.raises(api.ScsError):
        api.expand_wire(struct.pack("<QQ", 0, 0) + rec, 1, len(hdr) + 104, threads=2)
    # a split entry past the end of the records
    rec = struct.pack("<BH", len(hdr), 1) + hdr + bytes(1)
    with pytest.raises(api.ScsError):
        api.expand_wire(struct.pack("<QQ", 0, 0) + struct.pack("<QQ", 999, 5) + rec, 2, len(hdr) + 6, threads=2)
