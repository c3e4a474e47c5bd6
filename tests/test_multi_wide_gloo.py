"""The multi-rank exchange of screencounter_b200.multi with keys of two 64-bit words per row (random barcodes of 22 to 42
bases), over gloo on the CPU: splitters are rows, tables are cut lexicographically, both words travel through the
all-to-all and the gather.  As in tests/test_multi_gloo.py, the per-rank engine is the oracle and the table operations are a
host-tensor stand-in; tests/test_gpu_random_wide.py runs the product's own table kernels.  Also compiles the specialised
random-barcode kernel for wide keys through NVRTC (no device needed)."""
import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WIDE_TEMPLATE = "ACGTACGT" + "-" * 30 + "TGCATGCA"
KEY_LEN = 30
_RANK = {"A": 0, "C": 1, "G": 2, "N": 3, "T": 4}


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _word(s):
    return sum(_RANK[ch] << (3 * (len(s) - 1 - i)) for i, ch in enumerate(s))


def _wide_table(seqs, freq, key_len):
    """A sorted table in the layout of include/scg.h: word 0 = bases 0..20, word 1 = bases 21..key_len-1."""
    import torch
    keys = np.array([[_word(s[:21]), _word(s[21:])] for s in seqs], dtype=np.int64).reshape(-1, 2)
    order = np.lexsort((keys[:, 1], keys[:, 0]))
    return {"keys": torch.from_numpy(keys[order].copy()), "counts": torch.from_numpy(np.asarray(freq, dtype=np.int32)[order].copy()),
            "key_len": key_len}


def _decode(keys, key_len):
    out = []
    for w0, w1 in keys:
        out.append("".join("ACGNT"[(int(w0) >> (3 * (20 - i))) & 7] for i in range(21)) +
                   "".join("ACGNT"[(int(w1) >> (3 * (key_len - 22 - i))) & 7] for i in range(key_len - 21)))
    return out


class WideNumpyTableOps:
    """TEST INFRASTRUCTURE: the table operations of merge_tables_across_ranks on host tensors of (rows, 2) keys."""

    def views(self, table):
        return table["keys"], table["counts"]

    def key_len(self, table):
        return table["key_len"]

    def from_tensors(self, keys, counts, key_len):
        return {"keys": keys.clone().reshape(-1, 2), "counts": counts.clone(), "key_len": key_len}

    def merge(self, a, b):
        import torch
        keys = torch.cat([a["keys"], b["keys"]])
        counts = torch.cat([a["counts"], b["counts"]]).to(torch.int64)
        uniq, inverse = torch.unique(keys, dim=0, sorted=True, return_inverse=True)   # rows in lexicographic order
        total = torch.zeros(uniq.shape[0], dtype=torch.int64).index_add_(0, inverse, counts)
        return {"keys": uniq, "counts": total.to(torch.int32), "key_len": a["key_len"]}

    def free(self, table):
        pass


def _workload():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from util import adversarial_reads, random_seq
    rng = np.random.default_rng(31)
    # few distinct first 21 bases: long runs of equal word 0, so the splitters fall inside them
    prefixes = [random_seq(rng, 21) for _ in range(3)]
    truth = [p + random_seq(rng, KEY_LEN - 21) for p in prefixes for _ in range(40)]
    return adversarial_reads(rng, 3000, WIDE_TEMPLATE, [truth], strand="both", read_len=60, sub_rate=0.02, n_rate=0.01,
                             lower_rate=0.0, double_frac=0.0, short_frac=0.02)


def _worker(rank, world, port, out_dir):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch.distributed as dist
    from oracle import port as engine
    from screencounter_b200 import multi
    from util import fastq
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        reads = _workload()
        first, count = multi.shard_range(len(reads), rank, world)
        seqs, freq, _ = engine.count_random(fastq(reads[first:first + count]), WIDE_TEMPLATE, 2, 1, True)
        merged, info = multi.merge_tables_across_ranks(WideNumpyTableOps(), _wide_table(list(seqs), freq, KEY_LEN))
        assert (merged is None) == (rank != 0)
        if rank == 0:
            np.savez(os.path.join(out_dir, "merged.npz"), seqs=np.array(_decode(merged["keys"].numpy(), KEY_LEN)),
                     freq=merged["counts"].numpy(), rows_total=info["rows_total"], bytes=info["bytes_all_to_all"],
                     sent=info["rows_sent"])
    finally:
        dist.destroy_process_group()


def test_lexicographic_cut_inside_a_run_of_equal_word0():
    import torch
    from screencounter_b200.multi import _cut
    keys = torch.tensor([[1, 5], [2, 1], [2, 4], [2, 9], [3, 0]], dtype=torch.int64)
    splitters = torch.tensor([[2, 4], [2, 5], [0, 0], [9, 9], [2, 0], [3, 0]], dtype=torch.int64)
    assert _cut(keys, splitters).tolist() == [2, 3, 0, 5, 1, 4]
    assert _cut(keys[:0], splitters[:2]).tolist() == [0, 0]


def test_wide_table_layout_round_trips():
    t = _wide_table(["A" * 21 + "C", "A" * 21 + "A", "C" + "A" * 21], [1, 2, 3], 22)
    assert _decode(t["keys"].numpy(), 22) == ["A" * 21 + "A", "A" * 21 + "C", "C" + "A" * 21]
    assert t["counts"].tolist() == [2, 1, 3]


@pytest.mark.timeout(300)
@pytest.mark.parametrize("world", [2, 3])
def test_wide_ranks_gloo_match_unsharded(port, tmp_path, world):
    import torch.multiprocessing as mp
    from util import fastq
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    want_seqs, want_freq, _ = port.count_random(fastq(_workload()), WIDE_TEMPLATE, 2, 1, True)
    order = np.argsort(np.array(list(want_seqs)))
    got = np.load(os.path.join(str(tmp_path), "merged.npz"))
    assert got["seqs"].tolist() == [list(want_seqs)[i] for i in order]
    assert np.array_equal(got["freq"], np.asarray(want_freq)[order])
    assert int(got["rows_total"]) == len(want_freq)
    assert int(got["bytes"]) == 20 * int(got["sent"])   # two key words and a count per row


@pytest.mark.parametrize("key_len,strand,mismatches,use_first", [(22, 2, 1, 1), (30, 0, 0, 0), (33, 1, 2, 1), (42, 2, 1, 0)])
def test_wide_random_kernel_compiles(key_len, strand, mismatches, use_first):
    """The specialised random-barcode kernel for 22..42-base barcodes (128-bit keys) through NVRTC, without a device."""
    import ctypes as C
    from screencounter_b200._lib import lib
    template = "CAGCTACGTACG" + "-" * key_len + "CCAGCTCGATCG"
    buf = C.create_string_buffer(16384)
    f = lib().scg_jit_selftest_handler
    f.argtypes = [C.c_int, C.c_char_p, C.c_int, C.c_int, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_size_t]
    rc = f(3, template.encode(), strand, mismatches, b"", 0, 0, len(template) + 20, use_first, buf, 16384)
    assert rc in (0, 2), buf.value.decode()
