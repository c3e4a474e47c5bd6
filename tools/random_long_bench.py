#!/usr/bin/env python
"""countRandomBarcodes with barcodes longer than 42 bases (the long-key count table).  Prints one JSON line:

  plan_<len>        scg_random_plan_run over resident synthetic reads (both strands, 1 mismatch in the 12-base flanks, barcodes
                    of <len> bases drawn from 2 M true ones, 0.3 % substitutions), device-timed with CUDA events after a warm-up
                    (G reads/s), and scg_plan_harvest (sort + render) on the host clock; the synthesiser draws barcodes of up
                    to 64 bases
  file_raw / file_bgzf   scg_count_random end to end on page-locked raw text and on a block-gzip image of it: reads of
                    12 + <file-len> + 12 bases plus 10 random bases, barcodes drawn from 500 k true ones; harvest_s from
                    scg_timing_json and a digest of the table
  reference         the kaori reference (the C restatement where the compiled reference is not built) on the same raw text,
                    host clock, and whether its table equals ours

usage: random_long_bench.py [--reads N] [--file-reads M] [--file-len L]"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ap = argparse.ArgumentParser()
ap.add_argument("--reads", type=int, default=50_000_000)
ap.add_argument("--file-reads", type=int, default=4_000_000)
ap.add_argument("--file-len", type=int, default=120)
args = ap.parse_args()

import numpy as np
import torch
from screencounter_b200 import rcpp
from screencounter_b200.device import RandomPlan, SynthSpec

F12, R12 = "CAGCTACGTACG", "CCAGCTCGATCG"
gpu = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
out = {"gpu_name_power_limit": gpu, "reads": args.reads, "file_reads": args.file_reads, "file_len": args.file_len}

# ---- device-timed plan runs over resident reads ----
for key_len in (50, 64):
    template = F12 + "-" * key_len + R12
    spec = SynthSpec(template, [], seed=42, read_len=len(template) + 10, strand=2, random_space=2_000_000, sub_per_10k=30)
    reads = spec.on_device(0, args.reads)
    plan = RandomPlan(template, 2, 1, True, expected_distinct=4_000_000 + int(0.1 * args.reads))
    stream = torch.cuda.Stream()
    plan.run(reads, stream=stream.cuda_stream)   # warm-up
    torch.cuda.synchronize()
    times = []
    for _ in range(3):
        plan.reset(stream=stream.cuda_stream)
        start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record(stream)
        plan.run(reads, stream=stream.cuda_stream)
        end.record(stream)
        end.synchronize()
        times.append(start.elapsed_time(end) / 1e3)
    t0 = time.perf_counter()
    seqs, freq = plan.harvest()
    harvest = time.perf_counter() - t0
    out["plan_%d" % key_len] = {"kernel": plan.kernel, "seconds": times, "g_reads_per_s": args.reads / min(times) / 1e9, "harvest_s": harvest,
                                "rows": len(freq)}
    plan.free()
    del reads
    torch.cuda.synchronize()

# ---- end to end: reads with long barcodes, built with numpy ----
rng = np.random.default_rng(7)
L = args.file_len
true = rng.integers(0, 4, size=(500_000, L), dtype=np.uint8)
pick = rng.integers(0, len(true), size=args.file_reads)
acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
bar = acgt[true[pick]]
subs = rng.random(bar.shape) < 0.003
bar[subs] = acgt[rng.integers(0, 4, size=int(subs.sum()))]
tail = acgt[rng.integers(0, 4, size=(args.file_reads, 10), dtype=np.uint8)]
seq = np.concatenate([np.broadcast_to(np.frombuffer(F12.encode(), np.uint8), (args.file_reads, 12)), bar,
                      np.broadcast_to(np.frombuffer(R12.encode(), np.uint8), (args.file_reads, 12)), tail], axis=1)
rl = seq.shape[1]
rec = np.empty((args.file_reads, 3 + rl + 3 + rl + 1), dtype=np.uint8)
rec[:, 0:3] = np.frombuffer(b"@r\n", np.uint8)
rec[:, 3:3 + rl] = seq
rec[:, 3 + rl:6 + rl] = np.frombuffer(b"\n+\n", np.uint8)
rec[:, 6 + rl:6 + 2 * rl] = ord("I")
rec[:, -1] = ord("\n")
raw = rec.tobytes()
del rec, seq, bar, tail
template = F12 + "-" * L + R12
text = rcpp.PinnedText.from_bytes(raw, device=0)
image = rcpp.PinnedText.from_bytes(rcpp.bgzf_compress(np.frombuffer(raw, np.uint8), level=6).tobytes(), device=0)
threads = len(os.sched_getaffinity(0)) or 1
ours = None
for name, src in (("file_raw", text), ("file_bgzf", image)):
    rcpp.count_random_barcodes(src, template, 2, 1, True, threads, device=0)   # warm-up
    t0 = time.perf_counter()
    (seqs, freq), total = rcpp.count_random_barcodes(src, template, 2, 1, True, threads, device=0)
    dt = time.perf_counter() - t0
    t = rcpp.timing(0)
    digest = hashlib.sha256(seqs.tobytes() + freq.astype("<i4").tobytes()).hexdigest()[:16]
    out[name] = {"seconds": dt, "m_reads_per_s": args.file_reads / dt / 1e6, "harvest_s": t["harvest_s"], "rows": len(freq),
                 "total": int(total), "table_sha256": digest, "kernel": t["kernel"]}
    ours = (seqs, freq)

# ---- the reference arm on the same text ----
from oracle import kref, port
ref = kref if kref.available() else port
t0 = time.perf_counter()
rseqs, rfreq, rtotal = ref.count_random(raw, template, 2, 1, True)
dt = time.perf_counter() - t0
order = sorted(range(len(rseqs)), key=lambda i: rseqs[i])
same = [ours[0][i].decode() for i in range(len(ours[0]))] == [rseqs[i] for i in order] and \
    np.array_equal(ours[1], np.asarray(rfreq, dtype=np.int32)[order])
out["reference"] = {"oracle": "compiled reference" if ref is kref else "C restatement", "seconds": dt, "m_reads_per_s": args.file_reads / dt / 1e6,
                    "same_table": bool(same), "total": int(rtotal)}
print(json.dumps(out), flush=True)
