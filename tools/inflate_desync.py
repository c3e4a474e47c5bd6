#!/usr/bin/env python
"""The device inflater on members whose deflate blocks end at different places (what an adaptive block splitter such as
libdeflate's gives): every member of the benchmark's text is compressed with zlib and flushed (Z_FULL_FLUSH closes the block) at
two random places.  usage: inflate_desync.py [MiB of text] [repeats]"""
import os, struct, sys, zlib
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import bench
from screencounter_b200 import rcpp

mb = int(sys.argv[1]) if len(sys.argv) > 1 else 128
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
wl = bench.make_workload(2)
members = (mb << 20) // 65280
n = members * 65280 // 157 + 1
text = wl.texts(0, n, pinned=False)[0]
raw = np.frombuffer(text, dtype=np.uint8)[: members * 65280].tobytes()
rng = np.random.default_rng(1)
for blocks in (1, 3):
    out = []
    for m in range(members):
        chunk = raw[m * 65280:(m + 1) * 65280]
        comp = zlib.compressobj(6, zlib.DEFLATED, -15, 8)
        cuts = sorted(int(c) for c in rng.integers(5000, 60000, blocks - 1))
        body, at = b"", 0
        for c in cuts:
            body += comp.compress(chunk[at:c]) + comp.flush(zlib.Z_FULL_FLUSH)
            at = c
        body += comp.compress(chunk[at:]) + comp.flush()
        bsize = 12 + 6 + len(body) + 8
        assert bsize <= 65536
        out.append(b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff" + struct.pack("<H", 6) + b"BC" + struct.pack("<HH", 2, bsize - 1) + body +
                   struct.pack("<II", zlib.crc32(chunk) & 0xFFFFFFFF, len(chunk)))
    out.append(bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000"))
    image = np.frombuffer(b"".join(out), dtype=np.uint8)
    best = None
    for _ in range(reps):
        got, ms = rcpp.bgzf_inflate(image)
        best = ms if best is None else min(best, ms)
    assert got.tobytes() == raw
    print("%d block(s) per member, %d members: %.3f ms = %.1f GB/s" % (blocks, members, best, len(raw) / best / 1e6))
