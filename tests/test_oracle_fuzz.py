"""Cross-checks the C restatement (oracle/kaori_port.c) against the unmodified reference
(oracle/_ref) on adversarial seeded inputs, handler by handler and search by search."""
import numpy as np
import pytest

from util import (fastq, random_seq, dense_pool, distinct_pool, adversarial_reads, mutate, revcomp)

STRANDS = {"original": 0, "reverse": 1, "both": 2}


@pytest.fixture(scope="module")
def kref(compiled_reference):
    # every test here compares the C restatement with the reference, so the restatement cannot stand in for it
    return compiled_reference


def _same(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        if isinstance(x, np.ndarray):
            assert np.array_equal(x, y)
        else:
            assert x == y


@pytest.mark.parametrize("seed", [1, 2])
@pytest.mark.parametrize("strand", ["original", "reverse", "both"])
@pytest.mark.parametrize("mm", [0, 1, 2])
@pytest.mark.parametrize("use_first", [True, False])
def test_single(kref, port, seed, strand, mm, use_first):
    rng = np.random.default_rng(1000 * seed + 10 * mm + STRANDS[strand])
    L = int(rng.integers(5, 9))
    pool = dense_pool(rng, 60, L)
    template = "ACGTA" + "-" * L + ("TGCAT" if seed == 1 else "GG")
    reads = adversarial_reads(rng, 1500, template, [pool], strand=strand)
    f = fastq(reads)
    _same(kref.count_single(f, template, STRANDS[strand], pool, mm, use_first),
          port.count_single(f, template, STRANDS[strand], pool, mm, use_first))
    a = kref.trace_single(f, template, STRANDS[strand], pool, mm, use_first)
    b = port.trace_single(f, template, STRANDS[strand], pool, mm, use_first)
    assert np.array_equal(a[0], b[0])
    assert np.array_equal(a[1], b[1])


@pytest.mark.parametrize("strand", ["original", "reverse", "both"])
@pytest.mark.parametrize("mm", [0, 1, 2])
@pytest.mark.parametrize("use_first", [True, False])
@pytest.mark.parametrize("template", ["AAAAACGT------ACGTGGGG", "AAAAACGT------ACGT", "CAG--------T"])
def test_random(kref, port, strand, mm, use_first, template):
    rng = np.random.default_rng(7 + mm + 100 * STRANDS[strand])
    L = template.count("-")
    pool = [random_seq(rng, L) for _ in range(30)]
    # no lower-case / odd symbols on reverse hits (those throw in the reference; covered separately)
    reads = adversarial_reads(rng, 1500, template, [pool], strand=strand, lower_rate=0.0)
    f = fastq(reads)
    _same(kref.count_random(f, template, STRANDS[strand], mm, use_first),
          port.count_random(f, template, STRANDS[strand], mm, use_first))


def test_random_forward_keeps_raw_chars(kref, port):
    # forward hits copy the raw read characters (case, N, anything); SURVEY 8.1 T9
    template = "ACGT----TTTT"
    reads = ["ACGTacgtTTTT", "ACGTNNgtTTTT", "ACGTAC.RTTTT", "ACGTACGTTTTT"]
    f = fastq(reads)
    a = kref.count_random(f, template, 0, 0, True)
    b = port.count_random(f, template, 0, 0, True)
    _same(a, b)
    assert a[0] == sorted(["acgt", "NNgt", "AC.R", "ACGT"])


def test_random_reverse_unknown_base_throws(kref, port):
    template = "ACGT----TTTT"
    f = fastq([revcomp("ACGTACGTTTTT")[:5] + "R" + revcomp("ACGTACGTTTTT")[6:]])
    for e in (kref, port):
        with pytest.raises(Exception, match="cannot complement unknown base 'R'"):
            e.count_random(f, template, 1, 0, True)


@pytest.mark.parametrize("strand", ["original", "reverse", "both"])
@pytest.mark.parametrize("mm", [0, 1, 2])
@pytest.mark.parametrize("use_first", [True, False])
def test_combo_single(kref, port, strand, mm, use_first):
    rng = np.random.default_rng(31 + mm + 100 * STRANDS[strand])
    p1 = dense_pool(rng, 25, 5)
    p2 = dense_pool(rng, 30, 7)
    template = "ACGT" + "-" * 5 + "TGCAAG" + "-" * 7 + "GGA"
    reads = adversarial_reads(rng, 1500, template, [p1, p2], strand=strand)
    f = fastq(reads)
    _same(kref.count_combo_single(f, template, STRANDS[strand], p1, p2, mm, use_first),
          port.count_combo_single(f, template, STRANDS[strand], p1, p2, mm, use_first))
    assert np.array_equal(kref.trace_combo_single(f, template, STRANDS[strand], p1, p2, mm, use_first),
                          port.trace_combo_single(f, template, STRANDS[strand], p1, p2, mm, use_first))


@pytest.mark.parametrize("strand", ["original", "reverse", "both"])
@pytest.mark.parametrize("mm", [0, 1, 2])
@pytest.mark.parametrize("use_first", [True, False])
@pytest.mark.parametrize("diagnostics", [False, True])
def test_dual_single_end(kref, port, strand, mm, use_first, diagnostics):
    rng = np.random.default_rng(57 + mm + 100 * STRANDS[strand])
    g1 = dense_pool(rng, 12, 5)
    g2 = dense_pool(rng, 12, 6)
    pairs = set()
    while len(pairs) < 40:
        pairs.add((int(rng.integers(0, 12)), int(rng.integers(0, 12))))
    pairs = sorted(pairs)
    p1 = [g1[i] for i, _ in pairs]
    p2 = [g2[j] for _, j in pairs]
    template = "ACGT" + "-" * 5 + "TGCAAG" + "-" * 6 + "GGA"
    # reads draw the two regions independently -> valid and invalid combinations
    reads = adversarial_reads(rng, 1500, template, [g1, g2], strand=strand)
    f = fastq(reads)
    _same(kref.count_dual_single_end(f, template, [p1, p2], STRANDS[strand], mm, use_first, diagnostics),
          port.count_dual_single_end(f, template, [p1, p2], STRANDS[strand], mm, use_first, diagnostics))
    if not diagnostics:
        assert np.array_equal(kref.trace_dual_single_end(f, template, [p1, p2], STRANDS[strand], mm, use_first),
                              port.trace_dual_single_end(f, template, [p1, p2], STRANDS[strand], mm, use_first))


def _paired_inputs(rng, n, t1, t2, g1, g2, rev1, rev2, swap_frac=0.0):
    r1 = adversarial_reads(rng, n, t1, [g1], strand="reverse" if rev1 else "original", short_frac=0.01)
    r2 = adversarial_reads(rng, n, t2, [g2], strand="reverse" if rev2 else "original", short_frac=0.01)
    for i in range(n):
        if rng.random() < swap_frac:
            r1[i], r2[i] = r2[i], r1[i]
    return fastq(r1), fastq(r2)


@pytest.mark.parametrize("rev", [(False, False), (True, False), (False, True)])
@pytest.mark.parametrize("mms", [(0, 0), (1, 1), (1, 0), (0, 1), (2, 1), (2, 0), (3, 0), (1, 2)])
@pytest.mark.parametrize("use_first", [True, False])
@pytest.mark.parametrize("randomized", [False, True])
def test_dual_paired(kref, port, rev, mms, use_first, randomized):
    rng = np.random.default_rng(91 + 7 * mms[0] + 3 * mms[1] + rev[0] + 2 * rev[1])
    # short dense guides incl. last-base variants of the second segment so the phantom of
    # MismatchTrie.hpp:608-617 ("Quirk A") fires
    g1 = dense_pool(rng, 10, 4, 0.5)
    g2 = dense_pool(rng, 10, 4, 0.5)
    for k in range(3):
        s = g2[k]
        alt = s[:-1] + ("A" if s[-1] != "A" else "C")
        if alt not in g2:
            g2.append(alt)
    pairs = set()
    while len(pairs) < 35:
        pairs.add((int(rng.integers(0, len(g1))), int(rng.integers(0, len(g2)))))
    pairs = sorted(pairs)
    p1 = [g1[i] for i, _ in pairs]
    p2 = [g2[j] for _, j in pairs]
    t1 = "ACGT----TG"
    t2 = "GGA----CCT"
    f1, f2 = _paired_inputs(rng, 1200, t1, t2, g1, g2, rev[0], rev[1], swap_frac=0.3 if randomized else 0.0)
    # the reference's result cache is not transparent for the segmented search (Quirk C):
    # the port reproduces it both per pair (1) and per file (0) ...
    for mode in (1, 0):
        a = kref.trace_dual(f1, t1, rev[0], mms[0], p1, f2, t2, rev[1], mms[1], p2, randomized, use_first, fresh_state=mode)
        b = port.trace_dual(f1, t1, rev[0], mms[0], p1, f2, t2, rev[1], mms[1], p2, randomized, use_first, fresh_state=mode)
        assert np.array_equal(a, b)
    assert (a >= 0).sum() > 50
    # ... and its cache-free mode (2), the semantics of the CUDA path, differs from them only
    # on a handful of pairs of this deliberately dense set
    c = port.trace_dual(f1, t1, rev[0], mms[0], p1, f2, t2, rev[1], mms[1], p2, randomized, use_first, fresh_state=2)
    assert (c != b).mean() < 0.05


@pytest.mark.parametrize("diagnostics", [False, True])
@pytest.mark.parametrize("randomized", [False, True])
@pytest.mark.parametrize("use_first", [True, False])
def test_dual_paired_counts_and_diagnostics(kref, port, diagnostics, randomized, use_first):
    # distinct 8-mers: no two library pairs are near each other, so the reference's cache
    # order-dependence (Quirk C) cannot fire and the threaded count run is comparable
    rng = np.random.default_rng(5)
    g1 = distinct_pool(rng, 20, 8)
    g2 = distinct_pool(rng, 20, 8)
    pairs = sorted({(int(rng.integers(0, 20)), int(rng.integers(0, 20))) for _ in range(60)})
    p1 = [g1[i] for i, _ in pairs]
    p2 = [g2[j] for _, j in pairs]
    t1 = "ACGT--------TGCA"
    t2 = "AGGA--------AGGA"
    f1, f2 = _paired_inputs(rng, 1500, t1, t2, g1, g2, False, False, swap_frac=0.3 if randomized else 0.0)
    _same(kref.count_dual(f1, t1, False, 1, p1, f2, t2, False, 1, p2, randomized, use_first, diagnostics),
          port.count_dual(f1, t1, False, 1, p1, f2, t2, False, 1, p2, randomized, use_first, diagnostics))


@pytest.mark.parametrize("rev", [(False, False), (True, True)])
@pytest.mark.parametrize("mms", [(0, 0), (1, 1), (2, 0)])
@pytest.mark.parametrize("use_first", [True, False])
@pytest.mark.parametrize("randomized", [False, True])
def test_combo_paired(kref, port, rev, mms, use_first, randomized):
    rng = np.random.default_rng(123 + mms[0])
    g1 = dense_pool(rng, 15, 5, 0.4)
    g2 = dense_pool(rng, 18, 5, 0.4)
    t1 = "ACGT-----TG"
    t2 = "GGA-----CCT"
    f1, f2 = _paired_inputs(rng, 1200, t1, t2, g1, g2, rev[0], rev[1], swap_frac=0.3 if randomized else 0.0)
    _same(kref.count_combo_paired(f1, t1, rev[0], mms[0], g1, f2, t2, rev[1], mms[1], g2, randomized, use_first),
          port.count_combo_paired(f1, t1, rev[0], mms[0], g1, f2, t2, rev[1], mms[1], g2, randomized, use_first))
    a = kref.trace_combo_paired(f1, t1, rev[0], mms[0], g1, f2, t2, rev[1], mms[1], g2, randomized, use_first)
    b = port.trace_combo_paired(f1, t1, rev[0], mms[0], g1, f2, t2, rev[1], mms[1], g2, randomized, use_first)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


IUPAC = "ACGTRYSWKMBDHVN"


@pytest.mark.parametrize("dup", [0, 3])  # FIRST, ERROR
@pytest.mark.parametrize("reverse", [False, True])
def test_search_any(kref, port, dup, reverse):
    rng = np.random.default_rng(11 + dup)
    L = 6
    for trial in range(30):
        lib = []
        for _ in range(int(rng.integers(1, 40))):
            s = random_seq(rng, L)
            if rng.random() < 0.3:  # IUPAC code somewhere
                pos = int(rng.integers(0, L))
                s = s[:pos] + IUPAC[int(rng.integers(4, len(IUPAC)))] + s[pos + 1:]
            if rng.random() < 0.1:
                s = s.lower()
            lib.append(s)
        queries = [mutate(rng, random_seq(rng, L) if rng.random() < 0.3 else lib[int(rng.integers(0, len(lib)))].upper().translate(
            str.maketrans("RYSWKMBDHVN", "ACCAGACAAAA")), 0.15, 0.05, 0.05) for _ in range(300)]
        caps = rng.integers(0, 4, size=len(queries)).astype(np.int32)
        try:
            a = kref.search_any(queries, caps, lib, 3, reverse, dup)
        except Exception as err:
            with pytest.raises(Exception) as got:
                port.search_any(queries, caps, lib, 3, reverse, dup)
            assert str(got.value) == str(err)
            continue
        b = port.search_any(queries, caps, lib, 3, reverse, dup)
        assert np.array_equal(a[0], b[0])
        hit = a[0] >= 0
        assert np.array_equal(a[1][hit], b[1][hit])


@pytest.mark.parametrize("caps", [(1, 1), (1, 0), (0, 1), (0, 0), (2, 1), (2, 0), (3, 0), (1, 2), (2, 2)])
def test_search_segmented(kref, port, caps):
    rng = np.random.default_rng(17 + 5 * caps[0] + caps[1])
    L1, L2 = 4, 3
    for trial in range(20):
        lib = list({random_seq(rng, L1 + L2) for _ in range(int(rng.integers(2, 60)))})
        queries = [mutate(rng, lib[int(rng.integers(0, len(lib)))], 0.2, 0.03, 0.03) for _ in range(400)]
        qcaps = np.stack([rng.integers(0, caps[0] + 1, size=len(queries)), rng.integers(0, caps[1] + 1, size=len(queries))], axis=1).astype(np.int32)
        a = kref.search_segmented2(queries, qcaps, lib, L1, L2, caps[0], caps[1])
        b = port.search_segmented2(queries, qcaps, lib, L1, L2, caps[0], caps[1])
        assert np.array_equal(a[0], b[0])
        hit = a[0] >= 0
        assert np.array_equal(a[1][hit], b[1][hit])
