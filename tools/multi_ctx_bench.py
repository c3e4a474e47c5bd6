#!/usr/bin/env python
"""ONE process, ONE counting call, several GPUs behind it (scg_ctx_create_multi): a config's workload from raw text and from a
block-gzip image in page-locked memory, on 1 device and on 2 .. n.  Every result is checked equal to the one-device result.

usage: multi_ctx_bench.py [reads] [n_devices] [--config 2|4|5] [--same-gpu]
  --config 2  countSingleBarcodes (default), 4 countComboBarcodes single-end, 5 countRandomBarcodes
  --same-gpu  the parts run on streams of GPU 0 (context over devices 0, 0, ...): what the cut and the merge cost on one GPU
  n_devices defaults to the number of visible GPUs (2 with --same-gpu).  For configs 4 and 5 each line also gives the share of
  the call spent merging the parts' tables on the first device (timing merge_s / total_s)."""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
from screencounter_b200 import rcpp

ap = argparse.ArgumentParser()
ap.add_argument("reads", nargs="?", type=int, default=None)
ap.add_argument("n_devices", nargs="?", type=int, default=None)
ap.add_argument("--config", type=int, choices=(2, 4, 5), default=2)
ap.add_argument("--same-gpu", action="store_true")
args = ap.parse_args()

import torch
n = args.reads or {2: 8_000_000, 4: 8_000_000, 5: 20_000_000}[args.config]
ndev = args.n_devices or (2 if args.same_gpu else torch.cuda.device_count())
gpu = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
print("config %d, %d reads; GPUs: %s" % (args.config, n, gpu.replace("\n", "; ")))
wl = bench.make_workload(args.config)
text = wl.texts(0, n, pinned=True, device=0)[0]
image = rcpp.PinnedText.from_bytes(rcpp.bgzf_compress(text.array[: text.size], level=6).tobytes(), device=0)
threads = len(os.sched_getaffinity(0)) or 1
ref = None
for devices in [0] + [(0,) * k if args.same_gpu else tuple(range(k)) for k in range(2, ndev + 1)]:
    for name, src in (("raw text", text), ("block gzip", image)):
        for _ in range(2):
            res = wl.ours([src], threads, devices)
        t0 = time.perf_counter()
        merge = 0.0
        for _ in range(3):
            res = wl.ours([src], threads, devices)
            t = rcpp.timing(devices)
            merge += t["merge_s"] / max(t["total_s"], 1e-9)
        dt = (time.perf_counter() - t0) / 3
        if ref is None:
            ref = res
        assert wl.same(ref, res), "result differs from the one-device result"
        line = "devices %-12s %-10s: %7.1f M reads/s (%.1f ms)" % (devices, name, n / dt / 1e6, dt * 1e3)
        if args.config in (4, 5):
            line += "  merge on the first device %4.1f %% of the call" % (100 * merge / 3)
        print(line + "  " + t["kernel"][-12:], flush=True)
if ndev < 2:
    print("one GPU visible: 2 GPUs not measured")
