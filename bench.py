#!/usr/bin/env python
"""Benchmark of the hot path on the BASELINE.json configs (default: configs[1], the headline).

  python bench.py [--config N] [--gpus N] [--steps K] [--warmup W] [--scaling weak|strong]     our arm (one process per GPU under torchrun)
  python bench.py --impl reference [...]                                                      the reference's own CPU path on the host cores

  --config 1  countSingleBarcodes, 1,000 x 20-bp guides, 0 mismatches, forward strand, 1 M reads
  --config 2  countSingleBarcodes, 77,441 x 20-bp guides, 1 mismatch, both strands, 200 M reads        (default; BASELINE configs[1])
  --config 3  countDualBarcodes paired-end, 10,000 pairs of 20-bp guides, 1 mismatch per read, 100 M read pairs
  --config 4  countComboBarcodes single-end, two 20-bp regions, 500 x 500 pools, 1 mismatch, 100 M reads
  --config 5  countRandomBarcodes, 16-bp random barcodes, both strands, 500 M reads (about 12 M distinct barcodes)

One step = one pass of the hot path (template scan -> barcode lookup -> counts [-> the exchange between the GPUs when
N > 1]) over the rank's reads, which are resident in HBM when the timed region starts.  Prints ONE JSON line (see the task
contract): `value` is device-timed units/s over all ranks, `e2e` the same metric through the file-level C-ABI call from
host FASTQ text, `roofline` the pass's kernels against the measured HBM peak, `cpu_baseline` the compiled reference (kaori)
on the host cores, run in forked children with its results checked equal to the GPU's.
"""
import argparse
import json
import os
import pickle
import signal
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLANK_L, FLANK_R = "CAGCTACGTACG", "CCAGCTCGATCG"   # flanks of the reference's examples, R/countSingleBarcodes.R:63
READ_LEN = 75
RECORD = 2 * READ_LEN + 7                            # bytes of one synthetic FASTQ record
SEED = 42


def distinct_sequences(seed, n, length):
    rng = np.random.default_rng(seed)
    seen, out = set(), []
    while len(out) < n:
        codes = rng.integers(0, 4, size=(4096, length))
        for row in codes:
            s = "".join("ACGT"[c] for c in row)
            if s not in seen:
                seen.add(s)
                out.append(s)
                if len(out) == n:
                    break
    return out


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# =====================================================================================================================
# workloads: everything a config needs -- synthetic inputs, the resident plan, the file-level call, the reference call
# =====================================================================================================================
class Workload:
    number = 0
    name = ""
    unit = "reads/s"
    what = "reads"
    bytes_per_unit = 0
    bytes_note = ""
    default_units = 0          # units resident per GPU (the config's stated size)
    e2e_units = 4_000_000
    cpu_units = 1_000_000
    side_figures = False

    # --- inputs ---
    def specs(self):
        raise NotImplementedError

    def texts(self, first, n, pinned=False, device=None):
        return [s.fastq_pinned(first, n, device=device) if pinned else s.fastq(first, n) for s in self.specs()]

    def resident(self, first, n, device):
        return [s.on_device(first, n, device=device) for s in self.specs()]

    def outputs(self, table=None):
        """What one pass hands its caller: groups of named arrays (device tensors or host arrays), the arrays of a group
        sharing their rows (one per unit or per table entry).  `table`: the merged table of N > 1 GPUs, else the plan's."""
        raise NotImplementedError

    @staticmethod
    def same(a, b):
        return len(a) == len(b) and all(np.array_equal(np.asarray(x), np.asarray(y)) for x, y in zip(a, b))


class SingleWorkload(Workload):
    def __init__(self, number):
        self.number = number
        self.template = FLANK_L + "-" * 20 + FLANK_R
        if number == 1:
            self.name = "countSingleBarcodes: 1,000 x 20-bp guides, 0 mismatches, forward strand, 75-bp reads (BASELINE configs[0])"
            self.nguides, self.mm, self.strand = 1000, 0, 0
            self.default_units, self.e2e_units, self.cpu_units = 1_000_000, 1_000_000, 1_000_000
        else:
            self.name = "countSingleBarcodes: 77,441 x 20-bp guides, 1 mismatch, both strands, 75-bp reads (BASELINE configs[1])"
            self.nguides, self.mm, self.strand = 77441, 1, 2
            self.default_units, self.e2e_units, self.cpu_units = 200_000_000, 8_000_000, 4_000_000
            self.side_figures = True
        self.use_first = True   # R default find.best = FALSE
        self.bytes_per_unit = 49
        self.bytes_note = "49 B/read = 29 B packed read + 4 B per-read outcome (written) + 16 B table probe (L2-resident)"
        self.library = distinct_sequences(SEED, self.nguides, 20)

    def specs(self):
        from screencounter_b200.device import SynthSpec
        return [SynthSpec(self.template, [self.library], seed=SEED, read_len=READ_LEN, strand=self.strand)]

    def make_plan(self, device, units):
        import torch
        from screencounter_b200.device import SinglePlan
        dev = torch.device("cuda", device)
        self.plan = SinglePlan(self.template, self.strand, self.library, self.mm, self.use_first, device=device)
        self.counts = torch.zeros(len(self.library), dtype=torch.int32, device=dev)
        self.index = torch.empty(units, dtype=torch.int32, device=dev)   # per-read outcome: part of the 49 B/read figure

    def reset(self, stream):
        self.counts.zero_()

    def run(self, reads, stream):
        self.plan.run(reads[0], self.counts.data_ptr(), index_ptr=self.index.data_ptr(), stream=stream)

    def dense_tensor(self):
        return self.counts

    def result(self):
        return [self.counts.cpu().numpy()]

    def outputs(self, table=None):
        return [{"counts": self.counts}, {"index": self.index}]

    def matched(self):
        return int(self.counts.sum().item())

    def consistent(self):
        return int((self.index >= 0).sum().item()) == self.matched()

    def reference(self, engine, texts, threads):
        counts, total = engine.count_single(texts[0], self.template, self.strand, self.library, self.mm, self.use_first, threads)
        return [counts, np.array([total])]

    def ours(self, texts, nthreads, device):
        from screencounter_b200 import rcpp
        counts, total = rcpp.count_single_barcodes(texts[0], self.template, self.strand, self.library, self.mm, self.use_first, nthreads, device=device)
        return [counts, np.array([total])]

    def d2h_bytes(self):
        return 4 * len(self.library)

    def config_extra(self):
        return {"library": self.nguides, "mismatches": self.mm, "strand": ["original", "reverse", "both"][self.strand], "find_best": False}


class DualWorkload(Workload):
    number = 3
    name = ("countDualBarcodes paired-end: 10,000 pairs drawn from 200 x 200 distinct 20-bp guides, templates 12+20+12, 1 mismatch per read, "
            "75-bp reads (BASELINE configs[2])")
    unit = "pairs/s"
    what = "read pairs"
    bytes_per_unit = 86
    bytes_note = "86 B/pair = 2 x 29 B packed reads + 4 B per-pair outcome (written) + 24 B table probe of the 40-base key (L2-resident)"
    default_units, e2e_units, cpu_units = 100_000_000, 4_000_000, 1_000_000

    def __init__(self):
        a, b = distinct_sequences(3, 200, 20), distinct_sequences(4, 200, 20)
        rng = np.random.default_rng(5)
        rows = set()
        while len(rows) < 10000:
            rows.add((int(rng.integers(0, 200)), int(rng.integers(0, 200))))
        rows = sorted(rows)
        self.pool1, self.pool2 = [a[i] for i, _ in rows], [b[j] for _, j in rows]
        self.t1 = FLANK_L + "-" * 20 + FLANK_R
        self.t2 = "GATTACAGGCTA" + "-" * 20 + "TTGACCGTAGCA"
        self.use_first = True

    def specs(self):
        from screencounter_b200.device import SynthSpec
        # the same seed picks the same library row, offset and noise pattern for both mates
        return [SynthSpec(self.t1, [self.pool1], seed=7, read_len=READ_LEN, strand=0),
                SynthSpec(self.t2, [self.pool2], seed=7, read_len=READ_LEN, strand=0)]

    def make_plan(self, device, units):
        import torch
        from screencounter_b200.device import DualPlan
        dev = torch.device("cuda", device)
        self.plan = DualPlan(self.t1, False, 1, self.pool1, self.t2, False, 1, self.pool2, False, self.use_first, device=device)
        self.counts = torch.zeros(len(self.pool1), dtype=torch.int32, device=dev)
        self.index = torch.empty(units, dtype=torch.int32, device=dev)

    def reset(self, stream):
        self.counts.zero_()

    def run(self, reads, stream):
        self.plan.run(reads[0], reads[1], self.counts.data_ptr(), index_ptr=self.index.data_ptr(), stream=stream)

    def dense_tensor(self):
        return self.counts

    def result(self):
        return [self.counts.cpu().numpy()]

    def outputs(self, table=None):
        return [{"counts": self.counts}, {"index": self.index}]

    def matched(self):
        return int(self.counts.sum().item())

    def consistent(self):
        return int((self.index >= 0).sum().item()) == self.matched()

    def reference(self, engine, texts, threads):
        out = engine.count_dual(texts[0], self.t1, False, 1, self.pool1, texts[1], self.t2, False, 1, self.pool2, False, self.use_first, False, threads)
        return [out[0], np.array([int(out[1])])]

    def ours(self, texts, nthreads, device):
        from screencounter_b200 import rcpp
        counts, total = rcpp.count_dual_barcodes(texts[0], self.t1, False, 1, self.pool1, texts[1], self.t2, False, 1, self.pool2, False,
                                                 self.use_first, False, nthreads, device=device)
        return [counts, np.array([int(total[0])])]

    def d2h_bytes(self):
        return 4 * len(self.pool1)

    def config_extra(self):
        return {"library_pairs": len(self.pool1), "mismatches": [1, 1], "strands": ["original", "original"], "find_best": False}


class ComboWorkload(Workload):
    number = 4
    name = ("countComboBarcodes single-end: template 8+20+8+20+8, 500 x 500 pools of 20-bp barcodes, 1 mismatch, both strands, 75-bp reads "
            "(BASELINE configs[3])")
    bytes_per_unit = 69
    bytes_note = "69 B/read = 29 B packed read + 8 B per-read pair (written) + 2 x 16 B table probes (L1/L2-resident)"
    default_units, e2e_units, cpu_units = 100_000_000, 4_000_000, 1_000_000

    def __init__(self):
        self.p1, self.p2 = distinct_sequences(6, 500, 20), distinct_sequences(7, 500, 20)
        self.template = "CAGCTACG" + "-" * 20 + "GGTACCTT" + "-" * 20 + "CGATCGAG"
        self.mm, self.strand, self.use_first = 1, 2, True

    def specs(self):
        from screencounter_b200.device import SynthSpec
        return [SynthSpec(self.template, [self.p1, self.p2], seed=11, read_len=READ_LEN, strand=self.strand)]

    def make_plan(self, device, units):
        import torch
        from screencounter_b200.device import ComboPlan
        dev = torch.device("cuda", device)
        self.plan = ComboPlan(self.template, self.strand, self.p1, self.p2, self.mm, self.use_first, device=device)
        self.pairs = torch.empty(2 * units, dtype=torch.int32, device=dev)

    def reset(self, stream):
        self.plan.reset(stream=stream)

    def run(self, reads, stream):
        self.plan.run(reads[0], pairs_ptr=self.pairs.data_ptr(), stream=stream)

    def dense_tensor(self):
        return None

    def result(self):
        keys, freq = self.plan.harvest()
        return [keys, freq]

    def outputs(self, table=None):
        keys, freq = table or self.plan.harvest()
        return [{"keys": keys, "freq": freq}, {"pairs": self.pairs.view(-1, 2)}]

    def matched(self):
        return int(self.plan.harvest()[1].sum())

    def consistent(self):
        return int((self.pairs[0::2] >= 0).sum().item()) == self.matched()

    def reference(self, engine, texts, threads):
        keys, freq, total = engine.count_combo_single(texts[0], self.template, self.strand, self.p1, self.p2, self.mm, self.use_first, threads)
        return [keys, freq, np.array([int(total)])]

    def ours(self, texts, nthreads, device):
        from screencounter_b200 import rcpp
        keys, freq, total = rcpp.count_combo_barcodes_single(texts[0], self.template, self.strand, [self.p1, self.p2], self.mm, self.use_first,
                                                             nthreads, device=device)
        return [keys.T.copy(), freq, np.array([int(total[0])])]

    def d2h_bytes(self):
        return None

    def config_extra(self):
        sparse = os.environ.get("SCG_COMBO_FORCE_SPARSE", "0") not in ("", "0")
        return {"pools": [500, 500], "mismatches": self.mm, "strand": "both", "find_best": False,
                "tally": "device hash (SCG_COMBO_FORCE_SPARSE=1)" if sparse else "dense 500 x 500 matrix (SCG_COMBO_FORCE_SPARSE=1 selects the device hash)"}


class RandomWorkload(Workload):
    number = 5
    name = ("countRandomBarcodes: template 12+16+12, both strands, 1 mismatch in the flanks, 75-bp reads, barcodes drawn from 4 M true 16-mers "
            "with 0.1 % substitutions (about 12 M distinct per 500 M reads) (BASELINE configs[4])")
    bytes_per_unit = 53
    bytes_note = "53 B/read = 29 B packed read + 8 B barcode + 16 B count-table slot read-modify-write (the table, ~0.5 GB, lives in HBM)"
    default_units, e2e_units, cpu_units = 500_000_000, 4_000_000, 1_000_000

    def __init__(self):
        self.template = FLANK_L + "-" * 16 + FLANK_R
        self.mm, self.strand, self.use_first = 1, 2, True

    def specs(self):
        from screencounter_b200.device import SynthSpec
        return [SynthSpec(self.template, [], seed=13, read_len=READ_LEN, strand=self.strand, random_space=4_000_000, sub_per_10k=10)]

    def make_plan(self, device, units):
        import torch
        from screencounter_b200.device import RandomPlan
        dev = torch.device("cuda", device)
        # distinct barcodes: the 4 M true ones + the substituted copies (1.6 % of the constructs) + slack
        expected = min(units, 4_000_000) + int(0.02 * units) + 1_000_000
        self.plan = RandomPlan(self.template, self.strand, self.mm, self.use_first, expected_distinct=expected, device=device)
        self.index = torch.empty(units, dtype=torch.int32, device=dev)

    def reset(self, stream):
        self.plan.reset(stream=stream)

    def run(self, reads, stream):
        self.plan.run(reads[0], index_ptr=self.index.data_ptr(), stream=stream)

    def dense_tensor(self):
        return None

    def result(self):
        seqs, freq = self.plan.harvest()
        return [seqs, freq]

    def outputs(self, table=None):
        seqs, freq = table or self.plan.harvest()
        # the barcodes (fixed-width bytes) as one row of character codes each
        codes = np.frombuffer(seqs.tobytes(), dtype=np.uint8).reshape(len(seqs), seqs.dtype.itemsize)
        return [{"barcodes": codes, "freq": freq}, {"index": self.index}]

    def matched(self):
        return int(self.plan.harvest()[1].sum())

    def consistent(self):
        return int((self.index >= 0).sum().item()) == self.matched()

    def reference(self, engine, texts, threads):
        seqs, freq, total = engine.count_random(texts[0], self.template, self.strand, self.mm, self.use_first, threads)
        order = np.argsort(np.array(seqs, dtype=object), kind="stable") if len(seqs) else np.zeros(0, dtype=np.int64)
        return [np.array([seqs[i].encode() for i in order], dtype="S16"), np.asarray(freq)[order], np.array([int(total)])]

    def ours(self, texts, nthreads, device):
        from screencounter_b200 import rcpp
        (seqs, freq), total = rcpp.count_random_barcodes(texts[0], self.template, self.strand, self.mm, self.use_first, nthreads, device=device)
        return [seqs, freq, np.array([int(total)])]

    def d2h_bytes(self):
        return None   # the sorted table: counted from the result

    def config_extra(self):
        return {"barcode_bases": 16, "mismatches": self.mm, "strand": "both", "find_best": False, "true_barcodes": 4_000_000}


def make_workload(number):
    if number in (1, 2):
        return SingleWorkload(number)
    return {3: DualWorkload, 4: ComboWorkload, 5: RandomWorkload}[number]()


DUMP_VALUES = 1 << 20   # per array: 8 MB in float64, so at most 32 MB for the (up to three) arrays of a workload


def dump_outputs(wl, out_dir, table=None):
    """--dump-outputs: writes the arrays of the last timed pass as <out_dir>/<name>.npy in float64 (all of them hold integers
    below 2**53, so the values are exact).  A group of arrays whose widest holds more than DUMP_VALUES values keeps one
    sample of rows, drawn with the benchmark's seed, for all its arrays: the same rows from run to run, so that two builds
    can be compared output for output, and row i of one array belongs with row i of the others."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for group in wl.outputs(table):
        rows = len(next(iter(group.values())))
        keep = max(1, DUMP_VALUES // max(max(1, int(np.prod(a.shape[1:]))) for a in group.values()))
        rows_kept = np.sort(np.random.default_rng(SEED).choice(rows, keep, replace=False)) if rows > keep else None
        for name, arr in group.items():
            assert len(arr) == rows, "arrays of one group share their rows"
            if rows_kept is not None:
                arr = arr[torch.from_numpy(rows_kept).to(arr.device)] if torch.is_tensor(arr) else arr[rows_kept]
            if torch.is_tensor(arr):
                arr = arr.cpu().numpy()
            np.save(os.path.join(out_dir, name + ".npy"), np.asarray(arr, dtype=np.float64))


# =====================================================================================================================
# device clocks
# =====================================================================================================================
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index),
                 "--query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                 "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap",
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                smax.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def bind_near_gpu(local_rank):
    """Multi-rank runs: keep this rank's threads (and, by first touch, its page-locked FASTQ text) on the CPU cores that
    are local to its GPU's PCIe root, like a numactl line in a launch script would.  Best effort; returns what it did."""
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if not bus:
            return None
        domain, rest = bus.split(":", 1)
        path = "/sys/bus/pci/devices/%s:%s/local_cpulist" % (domain[-4:], rest)
        with open(path) as f:
            cpus = set()
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        if not cpus or cpus == allowed:
            return None
        os.sched_setaffinity(0, cpus)
        return "%d cores local to %s" % (len(cpus), bus)
    except Exception:
        return None


# =====================================================================================================================
# the reference on the host cores, isolated
# =====================================================================================================================
def _kaori_engine():
    from oracle import kref, port
    return (kref, "reference") if kref.available() else (port, "port")


def isolated(fn, retries=3):
    """Runs fn() in a FORKED CHILD and returns (seconds inside fn, its result, crashes), so that nothing the reference does can
    take this process down.

    kaori has a data race when num_threads > 1: reduce() merges a worker's search cache into the shared one
    (inst/include/kaori/BarcodeSearch.hpp:192-195) while other workers read it (:65); with 1 mismatch the cache is hot and an
    oversubscribed pool can crash (round 1: SIGSEGV on the driver's box).  A child that dies by a signal is run again (up to
    `retries` times); the number of crashes is reported.  The child only touches kaori and plain host memory (never CUDA)."""
    crashes = 0
    for _attempt in range(retries + 1):
        rfd, wfd = os.pipe()
        pid = os.fork()
        if pid == 0:
            status = 1
            try:
                os.close(rfd)
                t0 = time.perf_counter()
                result = fn()
                dt = time.perf_counter() - t0
                with os.fdopen(wfd, "wb") as f:
                    pickle.dump((dt, result), f, protocol=pickle.HIGHEST_PROTOCOL)
                status = 0
            finally:
                os._exit(status)
        os.close(wfd)
        with os.fdopen(rfd, "rb") as f:
            payload = f.read()
        _, st = os.waitpid(pid, 0)
        if os.WIFEXITED(st) and os.WEXITSTATUS(st) == 0 and payload:
            dt, result = pickle.loads(payload)
            return dt, result, crashes
        if os.WIFSIGNALED(st) and os.WTERMSIG(st) in (signal.SIGSEGV, signal.SIGABRT, signal.SIGBUS):
            crashes += 1
            continue
        raise RuntimeError("the reference child failed (wait status %d)" % st)
    return None, None, crashes


def multiprocess_figure(wl, texts, procs, n_units):
    """The race-free way to use every core: `procs` single-threaded kaori processes, each on its own contiguous slice of the reads
    (how the reference itself parallelises, one file per worker: R/countSingleBarcodes.R:113 bplapply).  Dense workloads only.
    Returns (wall seconds from the first fork to the last result, summed result)."""
    engine, _ = _kaori_engine()
    views = [memoryview(t) for t in texts]
    kids = []
    t0 = time.perf_counter()
    for k in range(procs):
        b, e = (n_units * k) // procs, (n_units * (k + 1)) // procs
        rfd, wfd = os.pipe()
        pid = os.fork()
        if pid == 0:
            status = 1
            try:
                os.close(rfd)
                out = wl.reference(engine, [bytes(v[b * RECORD:e * RECORD]) for v in views], 1)
                with os.fdopen(wfd, "wb") as f:
                    pickle.dump(out, f, protocol=pickle.HIGHEST_PROTOCOL)
                status = 0
            finally:
                os._exit(status)
        os.close(wfd)
        kids.append((pid, rfd))
    total = None
    for pid, rfd in kids:
        with os.fdopen(rfd, "rb") as f:
            payload = f.read()
        _, st = os.waitpid(pid, 0)
        if not (os.WIFEXITED(st) and os.WEXITSTATUS(st) == 0 and payload):
            raise RuntimeError("a single-threaded reference child failed (wait status %d)" % st)
        out = pickle.loads(payload)
        total = [np.asarray(x, dtype=np.int64) for x in out] if total is None else [a + np.asarray(x, dtype=np.int64) for a, x in zip(total, out)]
    return time.perf_counter() - t0, total


def cpu_side_figures(wl, texts, n_units, threads, threaded_result):
    """The other CPU figures BASELINE.md section 3 asks for, each measured once on a bounded sample: every core used race-free
    (one single-threaded process per core), one thread, and the FASTQ reader alone."""
    engine, _ = _kaori_engine()
    what = wl.what.replace(" ", "_")
    out = {}
    try:
        wall, summed = multiprocess_figure(wl, texts, threads, n_units)
        out["multiprocess"] = {"value": n_units / wall, "unit": wl.unit, "processes": threads, what: n_units,
                               "note": "race-free: one single-threaded kaori process per core, each on its own slice of the reads"}
        if threaded_result is not None:
            out["multiprocess"]["counts_equal_threaded"] = bool(np.array_equal(summed[0], np.asarray(threaded_result[0], dtype=np.int64)))
    except Exception as exc:   # a baseline figure must never take the line down
        out["multiprocess"] = {"error": str(exc)[:200]}
    one = max(1, min(n_units, 500_000))
    dt, _, _ = isolated(lambda: wl.reference(engine, [t[: one * RECORD] for t in texts], 1))
    if dt:
        out["one_thread"] = {"value": one / dt, "unit": wl.unit, what: one}
    dt, res, _ = isolated(lambda: engine.count_reads(texts[0]))
    if dt:
        out["parse_only"] = {"value": res[0] / dt, "unit": "reads/s", "reads": res[0],
                             "note": "kaori::FastqReader over the sample, no handler (the serial part of the threaded run)"}
    return out


def reference_threads():
    # the cores this process may run on (the cgroup's share, not the machine's: os.cpu_count() oversubscribed kaori's pool on
    # the round-1 box and it crashed)
    _, kind = _kaori_engine()
    cores = len(os.sched_getaffinity(0)) or 1
    return (cores if kind == "reference" else 1), kind


def cpu_baseline_leg(wl, args):
    """`cpu_baseline` of our own line: the compiled reference on this box's host cores over the first units of the workload, in
    forked children, BEFORE this process initialises CUDA.  Returns (dict, result, sample); the result is compared with the
    GPU's later."""
    engine, _ = _kaori_engine()
    threads, kind = reference_threads()
    sample = min(args.cpu_units or wl.cpu_units, args.e2e_units or wl.e2e_units)
    texts = wl.texts(0, sample)
    side, crashes = {}, 0
    try:
        dt, result, crashes = isolated(lambda: wl.reference(engine, texts, threads))
        if wl.side_figures:
            side = cpu_side_figures(wl, texts, sample, threads, result)
    except Exception as exc:
        return {"value": None, "unit": wl.unit, "cores": threads, "kind": kind, "sample": "failed: %s" % str(exc)[:200]}, None, sample
    if dt is None:
        value = side.get("multiprocess", {}).get("value")
        note = "every threaded attempt crashed (kaori's cache race); value = the multi-process figure"
    else:
        value, note = sample / dt, "threaded, kaori num_threads = %d" % threads
    out = {"value": value, "unit": wl.unit, "cores": threads, "kind": kind, "mode": note, "crashed_attempts_retried": crashes,
           "sample": "first %d %s of the workload, FASTQ text in host memory" % (sample, wl.what)}
    out.update(side)
    return out, result, sample


def reference_arm(wl, args):
    """The reference's own CPU implementation of the path (kaori compiled from /root/reference in oracle/_ref, else the C
    restatement) on all host cores, on a bounded sample of the workload."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    engine, _ = _kaori_engine()
    threads, kind = reference_threads()
    sample = args.cpu_units or (4_000_000 if wl.number == 2 else wl.cpu_units)
    texts = wl.texts(0, sample)
    crashes, result = 0, None
    for _ in range(args.warmup):
        _, result, c = isolated(lambda: wl.reference(engine, texts, threads))
        crashes += c
    spent, steps_done = 0.0, 0
    for _ in range(args.steps):
        dt, result, c = isolated(lambda: wl.reference(engine, texts, threads))
        crashes += c
        if dt is not None:
            spent += dt
            steps_done += 1
    side = cpu_side_figures(wl, texts, sample, threads, result) if wl.side_figures else {}
    mode = "threaded (kaori num_threads = %d)" % threads
    if steps_done == 0:
        mp = side.get("multiprocess", {})   # every threaded attempt crashed: the race-free figure stands in
        if "value" not in mp:
            raise RuntimeError("the reference could not be run on this box")
        value, ms = mp["value"], 1000.0 * sample / mp["value"]
        mode = "multi-process (every threaded attempt crashed)"
    else:
        value, ms = sample * steps_done / spent, 1000.0 * spent / steps_done
    what = wl.what.replace(" ", "_")
    line = {
        "impl": "reference", "metric": "reads/sec", "value": value, "unit": wl.unit, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": wl.name, "baseline_config": wl.number, "%s_per_step" % what: sample, "mode": mode,
                   "timing": "wall clock around the kaori::process_*_end_data call (libraries built, parse + scan + lookup + reduce), FASTQ text "
                             "in host memory, each step in a forked child; the libraries are rebuilt every step, as every R call does"},
        "cpu_baseline": {"value": value, "unit": wl.unit, "cores": threads, "kind": kind,
                         "sample": "%d %s of the same synthetic workload per step" % (sample, wl.what),
                         "crashed_attempts_retried": crashes, **side},
        "e2e": {"value": value, "unit": wl.unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    _emit(line)


_RESULT_FD = None


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner to stdout when the
    box sets NCCL_DEBUG), so file descriptor 1 is pointed at stderr for the run and the result line goes to the original."""
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def _emit(line):
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


# =====================================================================================================================
# our arm
# =====================================================================================================================
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[1, 2, 3, 4, 5], help="BASELINE.json config, 1-based (default 2 = the headline)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: the config's size per GPU; strong: the config's size in total, split over the GPUs")
    ap.add_argument("--reads", type=int, default=0, help="units resident per GPU (weak) or in total (strong); default: the config's size")
    ap.add_argument("--e2e-reads", dest="e2e_units", type=int, default=0, help="units per end-to-end step (host FASTQ text)")
    ap.add_argument("--cpu-reads", dest="cpu_units", type=int, default=0, help="units in the bounded CPU-baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float64; counts and tables "
                         "merged over the GPUs, per-unit outcomes of rank 0's units; larger arrays as a fixed seeded sample of rows)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    _claim_stdout()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    wl = make_workload(args.config)
    if args.impl == "reference":
        reference_arm(wl, args)
        return

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # the CPU baseline runs in forked children BEFORE this process initialises CUDA (N = 1 only)
    cpu_leg = cpu_baseline_leg(wl, args) if world == 1 else None

    import torch
    import torch.distributed as dist
    from screencounter_b200 import multi, rcpp

    binding = bind_near_gpu(local_rank) if world > 1 else None
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    total_units = args.reads or wl.default_units
    if args.scaling == "strong":
        first = (total_units * rank) // world
        units = (total_units * (rank + 1)) // world - first
    else:
        units = total_units
        first = rank * units   # contiguous range per rank (SURVEY.md 8(e))
    reads = wl.resident(first, units, local_rank)
    wl.make_plan(local_rank, units)
    stream = torch.cuda.current_stream()
    sid = stream.cuda_stream
    resident_bytes = sum(r.device_bytes for r in reads)
    # inputs smaller than the 126 MB L2 (config 1 at its stated size) would be re-read from L2: a buffer larger than L2 is
    # written between the timed passes, outside the events
    need_flush = resident_bytes < 512e6
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if need_flush else None

    exchange = multi.Exchange(wl, world, dev) if world > 1 else None

    def step():
        wl.reset(sid)
        wl.run(reads, sid)
        if exchange is not None:
            exchange.run()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()

    # --- kernel-only timing for the roofline (events around the kernel launches alone) ---
    launches_before = rcpp.kernel_launches(local_rank)
    wl.reset(sid)
    kernel_ms = 0.0
    if need_flush:
        for _ in range(args.steps):
            flush_buf.fill_(1)
            k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            k0.record()
            wl.run(reads, sid)
            k1.record()
            torch.cuda.synchronize()
            kernel_ms += k0.elapsed_time(k1)
    else:
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record()
        for _ in range(args.steps):
            wl.run(reads, sid)
        k1.record()
        torch.cuda.synchronize()
        kernel_ms = k0.elapsed_time(k1)
    launches_per_pass = (rcpp.kernel_launches(local_rank) - launches_before) // args.steps
    kernel_ms_per_pass = kernel_ms / args.steps
    # one clean pass for the consistency checks (per-unit outcomes vs tallies)
    wl.reset(sid)
    wl.run(reads, sid)
    torch.cuda.synchronize()
    matched_per_pass = wl.matched()
    assert wl.consistent(), "per-read outcomes and counts disagree"
    kernel_name = wl.plan.kernel

    # --- the timed region: exactly K steps, barrier + synchronize on both sides, device clocks sampled ---
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    launches_before = rcpp.kernel_launches(local_rank)
    if need_flush:
        elapsed = 0.0
        for _ in range(args.steps):
            flush_buf.fill_(1)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            step()
            e1.record()
            torch.cuda.synchronize()
            elapsed += e0.elapsed_time(e1)
        barrier()
    else:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            step()
        e1.record()
        barrier()
        elapsed = e0.elapsed_time(e1)
    gpu_launches = rcpp.kernel_launches(local_rank) - launches_before
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # N > 1: counts were summed over the ranks in place; sparse tables were merged into the exchange (on rank 0)
        merged = exchange.result() if exchange is not None and exchange.kind == "table" else None
        dump_outputs(wl, args.dump_outputs, merged)
    elapsed_ms = torch.tensor([elapsed], device=dev)
    if world > 1:
        dist.all_reduce(elapsed_ms, op=dist.ReduceOp.MAX)
    elapsed_ms = float(elapsed_ms.item())
    all_units = total_units if args.scaling == "strong" else units * world
    value = all_units * args.steps / (elapsed_ms / 1000.0)

    # --- N > 1: the sharded, exchanged result must be what ONE GPU computes over the union of the ranks' ranges ---
    nccl_check = None
    if world > 1:
        nccl_check = multi.verify_sharded(wl, exchange, first, units, rank, world, local_rank, sid)

    # --- end to end through the reference-facing call: host FASTQ text -> result on the host ---
    # The text sits in page-locked host memory (the contract's "inputs from pinned host memory"); every step copies it to
    # the device (157 B/read over PCIe), splits and packs the records there, counts, and reads the result back.
    e2e_units = args.e2e_units or wl.e2e_units
    texts = wl.texts(first, e2e_units, pinned=True, device=local_rank)
    nthreads = len(os.sched_getaffinity(0)) or 1
    # cold: the first call of this process on this design (library tables built and uploaded; kernels specialised -- from
    # the on-disk cubin cache when an earlier process left them there, through NVRTC otherwise)
    t0 = time.perf_counter()
    e2e_result = wl.ours(texts, nthreads, local_rank)
    torch.cuda.synchronize()
    cold_s = time.perf_counter() - t0
    cold_stage = rcpp.timing(local_rank)
    wl.ours(texts, nthreads, local_rank)
    barrier()
    e2e_steps = max(3, min(args.steps, 5))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_result = wl.ours(texts, nthreads, local_rank)
    torch.cuda.synchronize()
    e2e_dt = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(e2e_dt, op=dist.ReduceOp.MAX)
    e2e_dt = float(e2e_dt.item())
    stage = rcpp.timing(local_rank)
    e2e_value = e2e_units * world * e2e_steps / e2e_dt
    # --- the same call on the same reads as a BLOCK-GZIP image (what bgzip / bcl-convert write, and what FASTQ usually is on disk)
    # in page-locked host memory: the members cross PCIe compressed and are inflated, CRC-checked, split and packed on the device
    bgzf_line = None
    if not os.environ.get("SCG_BENCH_NO_BGZF"):
        t0 = time.perf_counter()
        images = [rcpp.PinnedText.from_bytes(rcpp.bgzf_compress(t.array[: t.size], level=6, nthreads=nthreads).tobytes(), device=local_rank)
                  for t in texts]
        compress_s = time.perf_counter() - t0
        gz_result = wl.ours(images, nthreads, local_rank)
        assert wl.same(gz_result, e2e_result), "block-gzip input gives a different result than its text"
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            wl.ours(images, nthreads, local_rank)
        torch.cuda.synchronize()
        gz_dt = torch.tensor([time.perf_counter() - t0], device=dev)
        if world > 1:
            dist.all_reduce(gz_dt, op=dist.ReduceOp.MAX)
        gz_stage = rcpp.timing(local_rank)
        bgzf_line = {"value": e2e_units * world * e2e_steps / float(gz_dt.item()), "unit": wl.unit,
                     "h2d_bytes_per_step": int(gz_stage.get("bytes_h2d", 0)),
                     "text_bytes_per_step": int(sum(t.size for t in texts)), "image_bytes": int(sum(i.size for i in images)),
                     "reader": gz_stage.get("reader"),
                     "stages_s": {k: gz_stage.get(k) for k in ("parse_s", "pack_s", "device_s", "setup_s", "harvest_s", "total_s")},
                     "note": "same reads, same call; input = bgzip-style image (zlib level 6, 65280-byte members, compressed here on %d host "
                             "threads in %.1f s, outside the timed region) in page-locked memory; result asserted equal to the text's" % (nthreads, compress_s)}
        del images
    d2h = wl.d2h_bytes()
    if d2h is None:
        d2h = int(sum(np.asarray(x).nbytes for x in e2e_result[:2]))
    # The headline end-to-end figure is the block-gzip one: .fastq.gz is what FASTQ is on disk, and the compressed image is what
    # has to cross PCIe (a sixth of the text here).  The raw-text figure stays beside it.
    raw_line = {"value": e2e_value, "unit": wl.unit, "h2d_bytes_per_step": int(stage.get("bytes_h2d", 0)), "reader": stage.get("reader"),
                "stages_s": {k: stage.get(k) for k in ("parse_s", "pack_s", "device_s", "setup_s", "harvest_s", "total_s")},
                "note": "same reads, same call; input = the FASTQ text itself in page-locked memory"}
    if bgzf_line is not None:
        e2e_head = {"value": bgzf_line["value"], "unit": wl.unit, "h2d_bytes_per_step": bgzf_line["h2d_bytes_per_step"],
                    "input": "block-gzip image of the FASTQ text (bgzip layout, zlib level 6) in page-locked host memory",
                    "reader": bgzf_line["reader"], "stages_s": bgzf_line["stages_s"]}
    else:
        e2e_head = {"value": e2e_value, "unit": wl.unit, "h2d_bytes_per_step": int(stage.get("bytes_h2d", 0)),
                    "input": "FASTQ text in page-locked host memory", "reader": stage.get("reader"), "stages_s": raw_line["stages_s"]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # --- CPU baseline (measured before CUDA was initialised, see cpu_baseline_leg): compare its result with the GPU's ---
    cpu_baseline = None
    if cpu_leg is not None:
        cpu_baseline, ref_result, sample = cpu_leg
        if ref_result is not None:
            if sample == e2e_units:
                chk = e2e_result
            else:
                chk = wl.ours([t.array[: sample * RECORD].tobytes() for t in texts], nthreads, local_rank)
            assert wl.same(ref_result, chk), "GPU result differs from the reference on the baseline sample"
            cpu_baseline["sample"] += ", result checked equal to the GPU's"

    peak, peak_src = measured_peaks()
    achieved = wl.bytes_per_unit * units / (kernel_ms_per_pass / 1000.0) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            t = json.load(f)
        per_unit = t.get("config%d" % wl.number, {}).get("dram_bytes_per_unit")
        if per_unit is None and wl.number == 2:
            per_unit = t.get("dram_bytes_per_read")
        traffic = per_unit * units if per_unit else None
    what = wl.what.replace(" ", "_")
    line = {
        "metric": "reads/sec", "value": value, "unit": wl.unit, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "u32", "data": "synthetic",
        "config": {"workload": wl.name, "baseline_config": wl.number, "%s_per_gpu" % what: units, "read_len": READ_LEN, "seed": SEED,
                   **wl.config_extra(),
                   "parallelism": "%s sharded by contiguous range, %d rank(s); %s" % (
                       wl.what, world, "no exchange (one GPU)" if world == 1 else exchange.describe()),
                   "l2": ("inputs (%.1f MB packed) fit the 126 MB L2: a 256 MB buffer is written between the timed passes (outside the events)"
                          % (resident_bytes / 1e6)) if need_flush else
                         ("inputs (%.1f GB packed per GPU) are larger than the 126 MB L2; no flush needed" % (resident_bytes / 1e9)),
                   "matched_fraction": matched_per_pass / units},
        "e2e": {**e2e_head, "d2h_bytes_per_step": int(d2h), "%s_per_step" % what: e2e_units, "host_threads": nthreads,
                "kernel": stage.get("kernel"), "cpu_binding": binding, "raw_text": raw_line, "block_gzip": bgzf_line,
                "cold": {"value": e2e_units / cold_s, "unit": wl.unit, "seconds": cold_s, "setup_s": cold_stage.get("setup_s"),
                         "note": "first call of this process on this design: library tables built + uploaded, kernels specialised (on-disk "
                                 "cubin cache or NVRTC), buffers allocated; the CUDA context already existed.  The reference arm rebuilds its "
                                 "libraries on every call; `value` above is our steady state (tables and kernels cached)"},
                "note": "input in page-locked host memory -> file-level C-ABI call: compressed members (or text) H2D chunk by chunk, members "
                        "inflated + CRC-checked by kernels (inflate.cu), records split + packed by kernels (ingest.cu), scan/lookup/count kernels "
                        "per chunk, result D2H; wall clock around the calls"},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                     "kernel": kernel_name, "bytes_per_unit": wl.bytes_per_unit, "units_per_pass": units,
                     "kernel_ms_per_pass": kernel_ms_per_pass, "kernel_launches_per_pass": launches_per_pass, "peak_source": peak_src,
                     "note": wl.bytes_note + "; all kernels of one pass over the resident %s (main kernel + its follow-ups), CUDA events" % wl.what},
        "cpu_baseline": cpu_baseline,
        "gpu_launches": int(gpu_launches),
        "clocks": clocks,
    }
    if nccl_check is not None:
        line["nccl_check"] = nccl_check
    _emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
