"""countRandomBarcodes with barcodes of 43 bases or more: the generic kernel into the long-key count table (staged keys, tag
claims, fresh keys moved to the key store after each launch), sorted device tables of ceil(key_len / 21) words per row, resident
plans and the many-files and multi-device paths, all against the oracle.  Key lengths 63/64/65 and 84/85 straddle the 21-base
words of a table row and the 32-base words of a plane; 248 is the longest barcode a 256-character template with 4-base flanks
holds."""

import numpy as np
import pytest

from util import fastq, random_seq, adversarial_reads, bgzf

pytestmark = pytest.mark.gpu

F12, R12 = "CAGCTACGTACG", "CCAGCTCGATCG"
KEY_LENS = [43, 63, 64, 65, 84, 85, 128, 248]
# (strand, mismatches, use_first): every strand, every budget, both modes
OPTIONS = [(2, 1, True), (0, 0, False), (1, 2, True), (2, 2, False)]
ROUTE = "long-key count table"


def _template(key_len):
    if key_len > 256 - 24:
        return "CAGC" + "-" * key_len + "GATC"
    return F12 + "-" * key_len + R12


def _want(kref, src, template, strand, mismatches, use_first):
    seqs, freq, total = kref.count_random(src, template, strand, mismatches, use_first)
    order = sorted(range(len(seqs)), key=lambda i: seqs[i])
    return [seqs[i] for i in order], np.asarray(freq, dtype=np.int32)[order], total


def _distinct(rng, n, length):
    """n distinct random barcodes, drawn in one numpy call"""
    out = set()
    while len(out) < n:
        codes = rng.integers(0, 4, size=(n, length), dtype=np.uint8)
        out.update(np.frombuffer(b"ACGT", dtype=np.uint8)[codes].view("S%d" % length).ravel().astype(str).tolist())
    return sorted(out)[:n]


def _reads(key_len, kind, seed, n=3000):
    """uniform: reads of one length with constructs at both ends and N inside barcodes; ragged: reads of many lengths and short
    reads; lower: uniform reads with lower-case letters (keys rendered from the raw read text and merged on the host)."""
    rng = np.random.default_rng(seed)
    template = _template(key_len)
    truth = _distinct(rng, 300, key_len)
    if kind == "ragged":
        return adversarial_reads(rng, n, template, [truth], strand="both", sub_rate=0.01, n_rate=0.005, lower_rate=0.0)
    return adversarial_reads(rng, n, template, [truth], strand="both", read_len=len(template) + 30, sub_rate=0.01, n_rate=0.005,
                             lower_rate=0.01 if kind == "lower" else 0.0, junk_frac=0.0, short_frac=0.0, edge_frac=0.3)


def _ours(src, template, strand, mismatches, use_first, device=0):
    from screencounter_b200 import rcpp
    (seqs, freq), total = rcpp.count_random_barcodes(src, template, strand, mismatches, use_first, 2, device=device, as_array=False)
    return list(seqs), np.asarray(freq), total


def _same(got, want):
    assert got[0] == want[0]
    assert np.array_equal(got[1], want[1])
    assert got[2] == want[2]


def _note():
    from screencounter_b200 import rcpp
    return rcpp.timing(0)["kernel"]


@pytest.mark.parametrize("kind", ["uniform", "ragged", "lower"])
@pytest.mark.parametrize("options", OPTIONS, ids=str)
@pytest.mark.parametrize("key_len", KEY_LENS)
def test_file_level_against_oracle(kref, key_len, options, kind, tmp_path):
    """Text in memory, block gzip (the device inflater) and a raw file on disk."""
    strand, mismatches, use_first = options
    template = _template(key_len)
    text = fastq(_reads(key_len, kind, 1000 * key_len + 10 * strand + mismatches))
    want = _want(kref, text, template, strand, mismatches, use_first)
    assert len(want[0]) > 10
    path = str(tmp_path / "reads.fastq")
    with open(path, "wb") as f:
        f.write(text)
    for src in (text, bgzf(text, 20000), path):
        _same(_ours(src, template, strand, mismatches, use_first), want)
        assert ROUTE in _note(), _note()


@pytest.mark.parametrize("key_len", [65, 248])
def test_host_parser_and_plain_gzip(kref, key_len, tmp_path, monkeypatch):
    """The host reader (SCG_HOST_PARSE=1) and a plain gzip file, which takes the host reader."""
    import gzip
    template = _template(key_len)
    text = fastq(_reads(key_len, "lower", 77 + key_len))
    want = _want(kref, text, template, 2, 1, False)
    path = str(tmp_path / "reads.fastq.gz")
    with open(path, "wb") as f:
        f.write(gzip.compress(text))
    _same(_ours(path, template, 2, 1, False), want)
    monkeypatch.setenv("SCG_HOST_PARSE", "1")
    _same(_ours(text, template, 2, 1, False), want)
    assert ROUTE in _note(), _note()


def _dense_space(rng, n, key_len):
    """n barcodes one substitution (or one N) away from a few centres: their hashes differ in one word only, so fingerprints and
    homes collide within probe runs far more often than among random keys"""
    centres = [random_seq(rng, key_len) for _ in range(32)]
    out = set(centres)
    while len(out) < n:
        c = list(centres[int(rng.integers(0, len(centres)))])
        p = int(rng.integers(0, key_len))
        c[p] = "ACGTN"[int(rng.integers(0, 5))]
        out.add("".join(c))
    return sorted(out)


@pytest.mark.parametrize("key_len", [43, 85, 128])
def test_dense_key_space(kref, key_len):
    rng = np.random.default_rng(key_len)
    template = _template(key_len)
    space = _dense_space(rng, 1500, key_len)
    reads = [F12 + space[int(rng.integers(0, len(space)))] + R12 for _ in range(40_000)]
    text = fastq(reads)
    want = _want(kref, text, template, 2, 0, True)
    assert len(want[0]) > 1000
    for src in (text, bgzf(text)):
        _same(_ours(src, template, 2, 0, True), want)


def _fastq_fast(barcodes, template_left, template_right):
    """FASTQ text of one read per barcode, built with numpy (hundreds of thousands of reads)"""
    seqs = np.char.add(np.char.add(template_left, np.asarray(barcodes)), template_right)
    L = len(seqs[0])
    n = len(seqs)
    names = np.char.add("@r", np.arange(n).astype(str))
    rec = np.char.add(np.char.add(np.char.add(names, "\n"), seqs), "\n+\n" + "I" * L + "\n")
    return "".join(rec.tolist()).encode("latin-1")


def test_table_grows_mid_file(kref):
    """600 000 distinct barcodes: more than the 2^20 slots the table starts with hold at a load factor of 1/2, spread over
    several reader batches, so the table is rebuilt with live entries in it (rehash_long_kernel)."""
    rng = np.random.default_rng(3)
    codes = _distinct(rng, 600_000, 43)
    text = _fastq_fast(codes, F12, R12)
    template = _template(43)
    want = _want(kref, text, template, 2, 1, True)
    assert len(want[0]) == 600_000
    for src in (text, bgzf(text)):
        _same(_ours(src, template, 2, 1, True), want)
        assert ROUTE in _note()


def _spec(key_len, space, seed=17):
    from screencounter_b200.device import SynthSpec
    return SynthSpec(_template(key_len), [], seed=seed, read_len=len(_template(key_len)) + 25, strand=2, random_space=space, sub_per_10k=30)


def test_file_of_several_batches_against_oracle(kref):
    """More reads than one reader batch (2^20): later batches find the barcodes of earlier ones RESIDENT in the key store."""
    spec = _spec(64, space=50_000, seed=23)
    text = spec.fastq(0, 1_200_000)
    template = _template(64)
    want = _want(kref, text, template, 2, 1, True)
    for src in (text, bgzf(text)):
        _same(_ours(src, template, 2, 1, True), want)
        assert ROUTE in _note()


@pytest.mark.parametrize("key_len,use_first", [(50, True), (64, False)])
def test_plan_over_several_slices_run_twice(kref, key_len, use_first):
    """2.5 M resident reads in one batch: the plan counts them in slices of 2^21 reads; a second run finds every key RESIDENT
    and doubles the counts."""
    from screencounter_b200.device import RandomPlan
    spec = _spec(key_len, space=200_000)
    n = 2_500_000
    plan = RandomPlan(_template(key_len), 2, 1, use_first)
    reads = spec.on_device(0, n)
    plan.run(reads)
    assert ROUTE in plan.kernel, plan.kernel
    want = _want(kref, spec.fastq(0, n), _template(key_len), 2, 1, use_first)
    seqs, freq = plan.harvest(as_array=False)
    assert list(seqs) == want[0] and np.array_equal(freq, want[1])
    plan.run(reads)
    seqs, freq = plan.harvest(as_array=False)
    assert list(seqs) == want[0] and np.array_equal(freq, 2 * want[1])
    plan.reset()
    plan.run(reads)
    seqs, freq = plan.harvest(as_array=False)
    assert list(seqs) == want[0] and np.array_equal(freq, want[1])
    plan.free()


def test_plan_grows_between_runs(kref):
    """Two runs of 300 000 distinct 128-base barcodes each: the second run outgrows the 2^20 slots at a load factor of 1/2, so
    the table grows with the first run's keys in it."""
    from screencounter_b200.device import RandomPlan, Reads
    rng = np.random.default_rng(11)
    codes = _distinct(rng, 600_000, 128)
    template = _template(128)
    texts = [_fastq_fast(codes[:300_000], F12, R12), _fastq_fast(codes[300_000:], F12, R12)]
    plan = RandomPlan(template, 2, 1, True)
    for t in texts:
        plan.run(Reads.from_fastq(t, 4))
    seqs, freq = plan.harvest(as_array=False)
    assert list(seqs) == codes and np.array_equal(freq, np.ones(len(codes), dtype=np.int32))
    plan.free()


def test_fixed_size_plan_reports_overflow_and_sorted_table_is_refused():
    from screencounter_b200 import rcpp
    from screencounter_b200.device import RandomPlan
    from screencounter_b200.multi import DeviceTableOps
    spec = _spec(50, space=1 << 40, seed=6)
    plan = RandomPlan(_template(50), 2, 1, True, expected_distinct=500)
    plan.run(spec.on_device(0, 20_000))
    with pytest.raises(rcpp.ScreenCounterError, match="overflowed"):
        plan.harvest()
    plan.free()
    plan = RandomPlan(_template(43), 2, 1, True)
    plan.run(_spec(43, space=1000).on_device(0, 5000))
    with pytest.raises(rcpp.ScreenCounterError, match="sorted tables hold random barcodes of at most 42 bases"):
        DeviceTableOps().from_plan(plan)
    plan.free()


@pytest.mark.parametrize("key_len", [43, 128])
@pytest.mark.parametrize("devices", [0, (0, 0)], ids=str)
def test_matrix_and_device_context_match_the_oracle(kref, key_len, devices, monkeypatch):
    from screencounter_b200 import rcpp
    monkeypatch.setenv("SCG_MULTI_MIN_BYTES", "1000")
    template = _template(key_len)
    texts = [fastq(_reads(key_len, kind, 50 + f)) for f, kind in enumerate(["uniform", "ragged", "lower"])]
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
        _same(_ours(bgzf(text, 20000), template, 2, 1, True, device=devices), _want(kref, text, template, 2, 1, True))
