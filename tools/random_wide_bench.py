#!/usr/bin/env python
"""countRandomBarcodes with 30-base barcodes: config 5's workload (both strands, 1 mismatch in the flanks, 75-base reads,
0.1 % substitutions, seed 42) with a 12 + 30 + 12 template and barcodes drawn from 12 M true 30-mers.  Prints one JSON line:

  plan_run          scg_random_plan_run over resident reads, device-timed with CUDA events after a warm-up (G reads/s)
  plan_table        scg_plan_sorted_table + scg_table_render (the sorted device table and its text), host clock around the
                    synchronising calls; "not available" where the tree cannot harvest such a plan
  file_raw / file_bgzf   scg_count_random end to end on page-locked raw text and on a block-gzip image of it, with harvest_s
                    (sorting and rendering the table) from scg_timing_json and a digest of the table (barcodes and frequencies),
                    so that two trees' results can be compared

usage: random_wide_bench.py [--reads N] [--file-reads M] [--root DIR] [--label TEXT]
  --root   the repository tree whose library is measured (default: this one), so that two trees can be compared in one run
  --label  what the line calls that tree (default: the tree's path)"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import time

ap = argparse.ArgumentParser()
ap.add_argument("--reads", type=int, default=100_000_000)
ap.add_argument("--file-reads", type=int, default=8_000_000)
ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
ap.add_argument("--label", default=None)
args = ap.parse_args()
sys.path.insert(0, os.path.abspath(args.root))

import torch
from screencounter_b200 import rcpp
from screencounter_b200._lib import lib
from screencounter_b200.device import RandomPlan, SynthSpec

TEMPLATE = "CAGCTACGTACG" + "-" * 30 + "CCAGCTCGATCG"
SPACE = 12_000_000
gpu = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
spec = SynthSpec(TEMPLATE, [], seed=42, read_len=75, strand=2, random_space=SPACE, sub_per_10k=10)
out = {"tree": args.label or os.path.abspath(args.root), "gpu_name_power_limit": gpu, "template": "12+30+12", "reads": args.reads, "file_reads": args.file_reads}

# ---- device-timed plan runs over resident reads ----
reads = spec.on_device(0, args.reads)
plan = RandomPlan(TEMPLATE, 2, 1, True, expected_distinct=SPACE + int(0.02 * args.reads) + 1_000_000)
stream = torch.cuda.Stream()
plan.run(reads, stream=stream.cuda_stream)   # warm-up: run-time compile, table pages
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
best = min(times)
out["plan_run"] = {"kernel": plan.kernel, "seconds": times, "g_reads_per_s": args.reads / best / 1e9}

# ---- the plan's table, sorted and rendered on the device ----
try:
    t0 = time.perf_counter()
    h = C.c_void_p()
    rcpp._check(plan.ctx, lib().scg_plan_sorted_table(plan.handle, C.byref(h)))
    t1 = time.perf_counter()
    r = C.c_void_p()
    rcpp._check(plan.ctx, lib().scg_table_render(plan.ctx, h, C.byref(r)))
    t2 = time.perf_counter()
    rows = int(lib().scg_table_rows(h))
    lib().scg_result_free(r)
    lib().scg_table_free(h)
    out["plan_table"] = {"rows": rows, "sorted_table_s": t1 - t0, "render_s": t2 - t1}
except rcpp.ScreenCounterError as e:
    out["plan_table"] = "not available: %s" % e
plan.free()
del reads
torch.cuda.synchronize()

# ---- end to end from page-locked host memory ----
text = spec.fastq_pinned(0, args.file_reads, device=0)
image = rcpp.PinnedText.from_bytes(rcpp.bgzf_compress(text.array[: text.size], level=6).tobytes(), device=0)
threads = len(os.sched_getaffinity(0)) or 1
for name, src in (("file_raw", text), ("file_bgzf", image)):
    rcpp.count_random_barcodes(src, TEMPLATE, 2, 1, True, threads, device=0)   # warm-up
    t0 = time.perf_counter()
    (seqs, freq), total = rcpp.count_random_barcodes(src, TEMPLATE, 2, 1, True, threads, device=0)
    dt = time.perf_counter() - t0
    t = rcpp.timing(0)
    digest = hashlib.sha256(seqs.tobytes() + freq.astype("<i4").tobytes()).hexdigest()[:16]
    out[name] = {"seconds": dt, "m_reads_per_s": args.file_reads / dt / 1e6, "harvest_s": t["harvest_s"], "rows": len(freq),
                 "total": int(total), "table_sha256": digest, "kernel": t["kernel"]}
print(json.dumps(out), flush=True)
