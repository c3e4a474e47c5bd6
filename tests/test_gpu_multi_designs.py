"""One input cut over the devices of a multi-device context (csrc/runners_multi.cu) for the single-end designs besides single
barcodes: countComboBarcodes, countDualBarcodesSingleEnd and countRandomBarcodes.  Every read is counted on its own, so the
parts' results merged on the first device must equal the oracle's on the whole text: tables, totals, per-read traces and
diagnostics.  A context may list one device several times (the parts then run on several streams of that device); with two
GPUs visible the same tests also run over devices (0, 1)."""
import gzip

import numpy as np
import pytest

from util import fastq, distinct_pool, dense_pool, adversarial_reads, bgzf

pytestmark = pytest.mark.gpu

COMBO_TEMPLATE = "CAGCTACG" + "-" * 12 + "GGTACCTT" + "-" * 12 + "CGATCGAG"
RANDOM_TEMPLATE = "CAGCTACGTACG" + "-" * 10 + "CCAGCTCGATCG"
WIDE_TEMPLATE = "CAGCTACGTACG" + "-" * 30 + "CCAGCTCGATCG"   # barcodes longer than 21 bases: 128-bit keys, rendered on the host
NREADS = 12000


def _oracle():
    from oracle import port, kref
    return kref if kref.available() else port


def _device_sets():
    sets = [(0, 0), (0, 0, 0)]
    try:
        import torch
        if torch.cuda.device_count() >= 2:
            sets.append((0, 1))
    except Exception:
        pass
    return sets


class Combo:
    def __init__(self, npool, seed):
        rng = np.random.default_rng(seed)
        self.p1, self.p2 = distinct_pool(rng, npool, 12), distinct_pool(rng, npool, 12)
        self.reads = adversarial_reads(rng, NREADS, COMBO_TEMPLATE, [self.p1, self.p2], strand="both")

    def ours(self, src, devices):
        from screencounter_b200 import rcpp
        keys, freq, total, trace = rcpp.count_combo_barcodes_single(src, COMBO_TEMPLATE, 2, [self.p1, self.p2], 1, True, 2, trace=True,
                                                                    device=devices)
        return [keys.T, freq, total[0], trace]

    def want(self, text):
        o = _oracle()
        keys, freq, total = o.count_combo_single(text, COMBO_TEMPLATE, 2, self.p1, self.p2, 1, True)
        return [np.asarray(keys).reshape(-1, 2), freq, total, o.trace_combo_single(text, COMBO_TEMPLATE, 2, self.p1, self.p2, 1, True)]


class DualSingleEnd:
    def __init__(self, diagnostics, seed):
        rng = np.random.default_rng(seed)
        g1, g2 = dense_pool(rng, 30, 12), dense_pool(rng, 30, 12)
        pairs = sorted({(int(rng.integers(0, 30)), int(rng.integers(0, 30))) for _ in range(120)})[:80]
        self.pools = [[g1[i] for i, _ in pairs], [g2[j] for _, j in pairs]]
        self.diagnostics = diagnostics
        # reads built from any pair of the two groups: many are no valid pair, which the diagnostics tabulate
        self.reads = adversarial_reads(rng, NREADS, COMBO_TEMPLATE, [g1, g2], strand="both")

    def ours(self, src, devices):
        from screencounter_b200 import rcpp
        out = rcpp.count_dual_barcodes_single_end(src, COMBO_TEMPLATE, self.pools, 2, 1, True, self.diagnostics, 2, trace=True, device=devices)
        if self.diagnostics:
            counts, (keys, freq), total, trace = out
            return [counts, total[0], keys.T, freq, trace]
        counts, total, trace = out
        return [counts, total[0], trace]

    def want(self, text):
        o = _oracle()
        trace = o.trace_dual_single_end(text, COMBO_TEMPLATE, self.pools, 2, 1, True)
        if self.diagnostics:
            counts, total, keys, freq = o.count_dual_single_end(text, COMBO_TEMPLATE, self.pools, 2, 1, True, True)
            return [counts, total, np.asarray(keys).reshape(-1, 2), freq, trace]
        counts, total = o.count_dual_single_end(text, COMBO_TEMPLATE, self.pools, 2, 1, True, False)
        return [counts, total, trace]


class Random:
    def __init__(self, template, lower_rate, seed):
        rng = np.random.default_rng(seed)
        barcodes = distinct_pool(rng, 300, template.count("-"))
        self.template = template
        self.reads = adversarial_reads(rng, NREADS, template, [barcodes], strand="both", lower_rate=lower_rate)

    def ours(self, src, devices):
        from screencounter_b200 import rcpp
        (seqs, freq), total = rcpp.count_random_barcodes(src, self.template, 2, 1, True, 2, device=devices, as_array=False)
        return [list(seqs), freq, total]

    def want(self, text):
        seqs, freq, total = _oracle().count_random(text, self.template, 2, 1, True)
        order = sorted(range(len(seqs)), key=lambda i: seqs[i])
        return [[seqs[i] for i in order], np.asarray(freq)[order], total]


CASES = {
    "combo-dense": lambda: Combo(40, 21),                          # 40 x 40 dense tally
    "combo-hash": lambda: Combo(4500, 22),                         # 4500 x 4500: the device hash
    "dual-se": lambda: DualSingleEnd(False, 23),
    "dual-se-diagnostics": lambda: DualSingleEnd(True, 24),
    "random-device-union": lambda: Random(RANDOM_TEMPLATE, 0.0, 25),
    "random-raw-characters": lambda: Random(RANDOM_TEMPLATE, 0.02, 26),   # lower-case reads: keys from raw text, host union
    "random-wide": lambda: Random(WIDE_TEMPLATE, 0.0, 27),                # 30-base barcodes: host union
}
_built = {}


def _case(name):
    if name not in _built:
        c = CASES[name]()
        c.text = fastq(c.reads)
        c.expected = c.want(c.text)
        _built[name] = c
    return _built[name]


def _same(got, want):
    assert len(got) == len(want)
    for k, (g, w) in enumerate(zip(got, want)):
        if isinstance(w, list):
            assert list(g) == w, "item %d differs" % k
        else:
            assert np.array_equal(np.asarray(g), np.asarray(w)), "item %d differs" % k


def _kernel_note(devices):
    from screencounter_b200 import rcpp
    return rcpp.timing(devices)["kernel"]


@pytest.mark.parametrize("devices", _device_sets(), ids=str)
@pytest.mark.parametrize("name", list(CASES))
def test_raw_text_cut_over_the_devices(name, devices, monkeypatch):
    monkeypatch.setenv("SCG_MULTI_MIN_BYTES", "1000")
    c = _case(name)
    _same(c.ours(c.text, devices), c.expected)
    assert "devices" in _kernel_note(devices)


@pytest.mark.parametrize("devices", _device_sets(), ids=str)
@pytest.mark.parametrize("block", [1500, 65280])
@pytest.mark.parametrize("name", list(CASES))
def test_block_gzip_cut_over_the_devices(name, block, devices, monkeypatch, tmp_path):
    """Parts that begin inside a member; lower-case reads make the random-barcode core fetch raw read text from its part."""
    from screencounter_b200 import rcpp
    monkeypatch.setenv("SCG_MULTI_MIN_BYTES", "1000")
    c = _case(name)
    image = bgzf(c.text, block)
    path = tmp_path / "reads.fastq.gz"
    path.write_bytes(image)
    for src in (image, str(path)):
        _same(c.ours(src, devices), c.expected)
        t = rcpp.timing(devices)
        assert "devices" in t["kernel"] and "inflated on the device" in t["reader"], t


def _wrapped_at_first_cut(reads, ndev):
    """The reads with one more record, wrapped over many lines, placed where the text's first cut is aimed.  Its quality lines
    read '@...', '...', '+...' (legal quality characters), so the record start guessed there lies inside it: the part before
    that cut cannot end cleanly, and the call has to fall back to one device."""
    seq = "ACGT" * 100
    quality = ["@" + "I" * 9, "I" * 10, "+" + "I" * 9] + ["I" * 10] * 37
    record = ("@wrapped\n" + "\n".join(seq[i:i + 10] for i in range(0, len(seq), 10)) + "\n+\n" + "\n".join(quality) + "\n").encode()
    body = [fastq([r]) for r in reads]
    target = (sum(len(b) for b in body) + len(record)) // ndev
    at, i = 0, 0
    while i < len(body) and at + len(body[i]) + len("@wrapped\n") <= target:
        at += len(body[i])
        i += 1
    assert at + len("@wrapped\n") <= target < at + len("@wrapped\n") + 400   # the target falls on the wrapped sequence lines
    return b"".join(body[:i]) + record + b"".join(body[i:])


@pytest.mark.parametrize("devices", _device_sets(), ids=str)
@pytest.mark.parametrize("name", ["combo-hash", "dual-se-diagnostics", "random-raw-characters", "random-wide"])
def test_inputs_that_are_not_cut(name, devices, monkeypatch, tmp_path):
    """A wrapped record where a cut is aimed, a plain gzip stream and a small text are read by the first device alone, with
    the same answer; a malformed record in the second half raises the oracle's error, line number included."""
    c = _case(name)
    monkeypatch.delenv("SCG_MULTI_MIN_BYTES", raising=False)
    _same(c.ours(c.text, devices), c.expected)   # 1-2 MB of text: below the default threshold of 8 MB per device
    assert "devices" not in _kernel_note(devices)
    monkeypatch.setenv("SCG_MULTI_MIN_BYTES", "1000")
    wrapped = _wrapped_at_first_cut(c.reads, len(devices))
    for src in (wrapped, bgzf(wrapped, 1500)):
        _same(c.ours(src, devices), c.want(wrapped))
        assert "devices" not in _kernel_note(devices)
    path = tmp_path / "reads.fastq.gz"
    path.write_bytes(gzip.compress(c.text, 3))
    _same(c.ours(str(path), devices), c.expected)
    assert "devices" not in _kernel_note(devices)

    from screencounter_b200 import rcpp
    half = len(c.reads) // 2
    bad = fastq(c.reads[:half]) + b"@broken\nACGT\n+\nII\n" + fastq(c.reads[half:])
    with pytest.raises(rcpp.ScreenCounterError) as e:
        c.ours(bad, devices)
    with pytest.raises(Exception) as ref_error:
        c.want(bad)
    assert str(e.value) == str(ref_error.value) or str(ref_error.value) in str(e.value), (str(e.value), str(ref_error.value))
    assert "line" in str(e.value)


@pytest.mark.parametrize("devices", _device_sets(), ids=str)
def test_library_errors_as_on_one_device(devices, monkeypatch):
    from screencounter_b200 import rcpp
    monkeypatch.setenv("SCG_MULTI_MIN_BYTES", "1000")
    c = _case("combo-dense")
    duplicated = c.p1[:-1] + [c.p1[0]]
    calls = [
        lambda d: rcpp.count_combo_barcodes_single(c.text, COMBO_TEMPLATE, 2, [duplicated, c.p2], 1, True, 2, device=d),
        lambda d: rcpp.count_combo_barcodes_single(c.text, "CAGCTACG" + "-" * 12 + "GGTACCTT", 2, [c.p1, c.p2], 1, True, 2, device=d),
        lambda d: rcpp.count_dual_barcodes_single_end(c.text, "CAGCTACG" + "-" * 12 + "GGTACCTT", [c.p1, c.p2], 2, 1, True, False, 2, device=d),
        lambda d: rcpp.count_random_barcodes(c.text, "CAGCTACGTACGCCAGCTCGATCG", 2, 1, True, 2, device=d),
    ]
    for call in calls:
        with pytest.raises(rcpp.ScreenCounterError) as one:
            call(0)
        with pytest.raises(rcpp.ScreenCounterError) as several:
            call(devices)
        assert str(several.value) == str(one.value)


@pytest.mark.parametrize("devices", _device_sets(), ids=str)
def test_repeated_calls_reuse_the_matchers(devices, monkeypatch):
    """The second call finds every device's matcher in that device's cache: same results."""
    monkeypatch.setenv("SCG_MULTI_MIN_BYTES", "1000")
    for name in ("combo-hash", "dual-se-diagnostics"):
        c = _case(name)
        first = c.ours(c.text, devices)
        second = c.ours(c.text, devices)
        _same(first, c.expected)
        _same(second, c.expected)
        assert "devices" in _kernel_note(devices)
