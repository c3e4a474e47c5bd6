"""countRandomBarcodes with barcodes of 22 to 42 bases (128-bit keys): the specialised kernel, the generic kernel, sorted device
tables of two words per row, resident plans, table merges and the multi-device paths, all against the oracle.  Key lengths 32
and 33 straddle the end of the first 32-bit word of a plane."""
import os
import socket
import sys

import numpy as np
import pytest

from util import fastq, distinct_pool, adversarial_reads, bgzf

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F12, R12 = "CAGCTACGTACG", "CCAGCTCGATCG"
KEY_LENS = [22, 30, 32, 33, 42]
# (strand, mismatches, use_first): every strand, every budget, both modes
OPTIONS = [(2, 1, True), (0, 0, False), (1, 2, True), (2, 2, False)]


def _template(key_len):
    return F12 + "-" * key_len + R12


def _want(kref, text, template, strand, mismatches, use_first):
    seqs, freq, total = kref.count_random(text, template, strand, mismatches, use_first)
    order = sorted(range(len(seqs)), key=lambda i: seqs[i])
    return [seqs[i] for i in order], np.asarray(freq, dtype=np.int32)[order], total


def _reads(key_len, kind, seed):
    """uniform: reads of one length (the specialised kernel); ragged: reads of many lengths and short reads (the generic
    kernel); lower: uniform reads with lower-case letters (keys rendered from the raw read text)."""
    rng = np.random.default_rng(seed)
    template = _template(key_len)
    truth = distinct_pool(rng, 400, key_len)
    if kind == "ragged":
        return adversarial_reads(rng, 5000, template, [truth], strand="both", sub_rate=0.02, n_rate=0.01, lower_rate=0.0)
    # constructs at both read ends, N inside barcodes, reads with two constructs (first vs best)
    return adversarial_reads(rng, 5000, template, [truth], strand="both", read_len=len(template) + 30, sub_rate=0.02, n_rate=0.01,
                             lower_rate=0.02 if kind == "lower" else 0.0, junk_frac=0.0, short_frac=0.0, edge_frac=0.3)


def _ours(src, template, strand, mismatches, use_first, device=0):
    from screencounter_b200 import rcpp
    (seqs, freq), total = rcpp.count_random_barcodes(src, template, strand, mismatches, use_first, 2, device=device, as_array=False)
    return list(seqs), np.asarray(freq), total


def _same(got, want):
    assert got[0] == want[0]
    assert np.array_equal(got[1], want[1])
    assert got[2] == want[2]


@pytest.mark.parametrize("kind", ["uniform", "ragged", "lower"])
@pytest.mark.parametrize("options", OPTIONS, ids=str)
@pytest.mark.parametrize("key_len", KEY_LENS)
def test_file_level_against_oracle(kref, key_len, options, kind, monkeypatch):
    """Raw text and block gzip, on the specialised route and on the generic one (SCG_NO_SPEC_HANDLERS=1)."""
    from screencounter_b200 import rcpp
    strand, mismatches, use_first = options
    template = _template(key_len)
    text = fastq(_reads(key_len, kind, 1000 * key_len + 10 * strand + mismatches))
    want = _want(kref, text, template, strand, mismatches, use_first)
    assert len(want[0]) > 10
    for src in (text, bgzf(text, 20000)):
        monkeypatch.delenv("SCG_NO_SPEC_HANDLERS", raising=False)
        _same(_ours(src, template, strand, mismatches, use_first), want)
        note = rcpp.timing(0)["kernel"]
        if kind == "ragged":
            assert "generic random_kernel" in note, note
        else:
            assert "spec_random_kernel" in note and "random_insert128_kernel" in note, note
        monkeypatch.setenv("SCG_NO_SPEC_HANDLERS", "1")
        _same(_ours(src, template, strand, mismatches, use_first), want)
        assert "generic random_kernel" in rcpp.timing(0)["kernel"]


def _spec(key_len, space=1 << 40, seed=17):
    from screencounter_b200.device import SynthSpec
    return SynthSpec(_template(key_len), [], seed=seed, read_len=len(_template(key_len)) + 25, strand=2, random_space=space, sub_per_10k=30)


@pytest.mark.parametrize("key_len,use_first", [(22, True), (33, False), (42, True)])
def test_plan_harvest_and_sorted_table(kref, key_len, use_first):
    from screencounter_b200.device import RandomPlan
    from screencounter_b200.multi import DeviceTableOps
    spec = _spec(key_len, space=50_000)
    n = 300_000
    plan = RandomPlan(_template(key_len), 2, 1, use_first)
    plan.run(spec.on_device(0, n))
    assert "spec_random_kernel" in plan.kernel, plan.kernel
    seqs, freq = plan.harvest(as_array=False)
    want = _want(kref, spec.fastq(0, n), _template(key_len), 2, 1, use_first)
    assert list(seqs) == want[0] and np.array_equal(freq, want[1])
    ops = DeviceTableOps()
    t = ops.from_plan(plan)
    keys, counts = ops.views(t)
    assert tuple(keys.shape) == (len(freq), 2)
    rseqs, rfreq = ops.render(t)
    aseqs, afreq = plan.harvest()
    assert np.array_equal(rseqs, aseqs) and np.array_equal(rfreq, afreq)
    # the layout of include/scg.h: word 0 = bases 0..20, word 1 = the rest, three bits a base in text order
    rank = {"A": 0, "C": 1, "G": 2, "N": 3, "T": 4}
    k = keys.cpu().numpy()
    for i in (0, len(seqs) // 2, len(seqs) - 1):
        s = seqs[i]
        assert int(k[i, 0]) == sum(rank[c] << (3 * (20 - j)) for j, c in enumerate(s[:21]))
        assert int(k[i, 1]) == sum(rank[c] << (3 * (key_len - 22 - j)) for j, c in enumerate(s[21:]))
    ops.free(t)
    plan.free()


@pytest.mark.parametrize("space,n,use_first", [(50_000, 300_000, True), (1 << 40, 400_000, False)], ids=["repeated", "grows"])
def test_plan_run_twice_counts_barcodes_in_their_home_sector(kref, space, n, use_first):
    """A second pass over the same reads finds every barcode of the first pass in the table: the main kernel counts those it
    finds in their home sector itself, the rest go to random_insert128_kernel.  "grows": the first pass leaves about 360 k
    distinct barcodes in the 2^20 slots, so the table grows before the second pass and rehash128_kernel moves the live
    entries to their even homes in the larger table, where the second pass must find them."""
    from screencounter_b200.device import RandomPlan
    spec = _spec(30, space=space, seed=21)
    plan = RandomPlan(_template(30), 2, 1, use_first)
    reads = spec.on_device(0, n)
    plan.run(reads)
    plan.run(reads)
    assert "spec_random_kernel" in plan.kernel, plan.kernel
    seqs, freq = plan.harvest(as_array=False)
    want = _want(kref, spec.fastq(0, n), _template(30), 2, 1, use_first)
    assert list(seqs) == want[0] and np.array_equal(freq, 2 * want[1])


def test_file_of_several_batches_against_oracle(kref):
    """More reads than one batch of the reader (2^20): later batches find the barcodes of earlier ones in their home sector."""
    from screencounter_b200 import rcpp
    spec = _spec(30, space=50_000, seed=23)
    text = spec.fastq(0, 1_500_000)
    template = _template(30)
    want = _want(kref, text, template, 2, 1, True)
    for src in (text, bgzf(text)):
        _same(_ours(src, template, 2, 1, True), want)
        assert "spec_random_kernel" in rcpp.timing(0)["kernel"]


def test_plan_table_grows_past_its_first_slots(kref):
    """Every read carries its own barcode: over 600 k distinct keys, so the 2^20 slots the table starts with are outgrown."""
    from screencounter_b200.device import RandomPlan
    spec = _spec(30, seed=5)
    n = 800_000
    plan = RandomPlan(_template(30), 2, 1, True)
    reads = spec.on_device(0, n)
    plan.run(reads)
    seqs, freq = plan.harvest(as_array=False)
    assert len(seqs) > 600_000
    want = _want(kref, spec.fastq(0, n), _template(30), 2, 1, True)
    assert list(seqs) == want[0] and np.array_equal(freq, want[1])


def test_fixed_size_plan_reports_overflow():
    from screencounter_b200 import rcpp
    from screencounter_b200.device import RandomPlan
    spec = _spec(30, seed=6)
    plan = RandomPlan(_template(30), 2, 1, True, expected_distinct=500)
    plan.run(spec.on_device(0, 20_000))
    with pytest.raises(rcpp.ScreenCounterError, match="overflowed"):
        plan.harvest()


def test_table_merge_round_trip_and_refusal():
    from screencounter_b200 import rcpp
    from screencounter_b200.device import RandomPlan
    from screencounter_b200.multi import DeviceTableOps
    spec = _spec(33, space=40_000, seed=9)
    ops = DeviceTableOps()
    halves = []
    for first, n in ((0, 150_000), (150_000, 100_001)):
        plan = RandomPlan(_template(33), 2, 1, True)
        plan.run(spec.on_device(first, n))
        halves.append(ops.from_plan(plan))
        plan.free()
    merged = ops.merge(halves[0], halves[1])
    whole = RandomPlan(_template(33), 2, 1, True)
    whole.run(spec.on_device(0, 250_001))
    want_seqs, want_freq = whole.harvest()
    seqs, freq = ops.render(merged)
    assert np.array_equal(seqs, want_seqs) and np.array_equal(freq, want_freq)
    # from device arrays the caller owns: (rows, 2) keys
    keys, counts = ops.views(merged)
    copy = ops.from_tensors(keys.clone(), counts.clone(), 33)
    s2, f2 = ops.render(copy)
    assert np.array_equal(s2, want_seqs) and np.array_equal(f2, want_freq)
    # a 21-base table and a 22-base table do not merge
    narrow, wide = RandomPlan(_template(21), 2, 1, True), RandomPlan(_template(22), 2, 1, True)
    narrow.run(_spec(21, space=1000).on_device(0, 5000))
    wide.run(_spec(22, space=1000).on_device(0, 5000))
    a, b = ops.from_plan(narrow), ops.from_plan(wide)
    with pytest.raises(rcpp.ScreenCounterError, match="different key lengths"):
        ops.merge(a, b)
    for t in (a, b, copy, merged, *halves):
        ops.free(t)


@pytest.mark.parametrize("devices", [0, (0, 0)], ids=str)
def test_matrix_and_device_context_match_the_oracle(kref, devices, monkeypatch):
    from screencounter_b200 import rcpp
    monkeypatch.setenv("SCG_MULTI_MIN_BYTES", "1000")
    template = _template(30)
    texts = [fastq(_reads(30, kind, 50 + f)) for f, kind in enumerate(["uniform", "ragged", "uniform"])]
    seqs, counts, totals = rcpp.matrix_of_random_barcodes(texts, template, 2, 1, True, 2, device=devices, as_array=False)
    per_file = [kref.count_random(t, template, 2, 1, True) for t in texts]
    union = sorted(set(s for p in per_file for s in p[0]))
    assert list(seqs) == union
    for f, (s, fr, total) in enumerate(per_file):
        col = dict(zip(s, fr))
        assert counts[:, f].tolist() == [col.get(u, 0) for u in union]
        assert totals[f] == total
    for text in texts:
        _same(_ours(text, template, 2, 1, True, device=devices), _want(kref, text, template, 2, 1, True))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _nccl_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), LOCAL_RANK=str(rank), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    from screencounter_b200 import multi
    from screencounter_b200.device import RandomPlan
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        first, n = multi.shard_range(300_000, rank, world)
        plan = RandomPlan(_template(33), 2, 1, True, device=rank)
        plan.run(_spec(33, space=30_000).on_device(first, n, device=rank))
        ops = multi.DeviceTableOps(rank)
        merged, info = multi.merge_tables_across_ranks(ops, ops.from_plan(plan))
        if rank == 0:
            seqs, freq = ops.render(merged)
            np.savez(os.path.join(out_dir, "merged.npz"), seqs=seqs, freq=freq, rows_total=info["rows_total"])
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(600)
def test_two_gpus_nccl_merge_of_wide_tables(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    from screencounter_b200.device import RandomPlan
    mp.spawn(_nccl_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    got = np.load(os.path.join(str(tmp_path), "merged.npz"))
    whole = RandomPlan(_template(33), 2, 1, True)
    whole.run(_spec(33, space=30_000).on_device(0, 300_000))
    want_seqs, want_freq = whole.harvest()
    assert np.array_equal(got["seqs"], want_seqs) and np.array_equal(got["freq"], want_freq)
    assert int(got["rows_total"]) == len(want_freq)
