"""Every other barcode design on the GPU (through the C ABI) against the reference: golden vectors
of the reference's own tests, adversarial fuzz with per-read outcomes, quirks A / B, diagnostics."""
import numpy as np
import pytest

import golden_cases
from engines import GpuEngine
from test_oracle_fuzz import _paired_inputs, _same, STRANDS
from util import fastq, random_seq, dense_pool, distinct_pool, adversarial_reads, revcomp

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu():
    return GpuEngine()


@pytest.mark.parametrize("case", golden_cases.ALL, ids=lambda f: f.__name__)
def test_golden(gpu, case):
    case(gpu)


# ---- random barcodes -----------------------------------------------------------------------------
@pytest.mark.parametrize("strand", ["original", "reverse", "both"])
@pytest.mark.parametrize("mm", [0, 1, 2])
@pytest.mark.parametrize("use_first", [True, False])
@pytest.mark.parametrize("template", ["AAAAACGT------ACGTGGGG", "AAAAACGT------ACGT", "CAG--------T",
                                      "ACGTAC" + "-" * 25 + "GGTCA", "ACGTAC" + "-" * 40 + "GGTCA"])
def test_random(gpu, kref, strand, mm, use_first, template):
    rng = np.random.default_rng(7 + mm + 100 * STRANDS[strand])
    L = template.count("-")
    pool = [random_seq(rng, L) for _ in range(30)]
    reads = adversarial_reads(rng, 2000, template, [pool], strand=strand, lower_rate=0.0)
    f = fastq(reads)
    _same(kref.count_random(f, template, STRANDS[strand], mm, use_first), gpu.count_random(f, template, STRANDS[strand], mm, use_first))


def test_random_raw_characters_and_errors(gpu, kref):
    template = "ACGT----TTTT"
    reads = ["ACGTacgtTTTT", "ACGTNNgtTTTT", "ACGTAC.RTTTT", "ACGTACGTTTTT", "ggACGTACGaTTTTcc"]
    f = fastq(reads)
    _same(kref.count_random(f, template, 0, 0, True), gpu.count_random(f, template, 0, 0, True))
    # lower case on the reverse strand is complemented to upper case
    f2 = fastq([revcomp("ACGTACGTTTTT").lower(), revcomp("ACGTNCGTTTTT")])
    _same(kref.count_random(f2, template, 2, 0, True), gpu.count_random(f2, template, 2, 0, True))
    bad = fastq([revcomp("ACGTACGTTTTT")[:5] + "R" + revcomp("ACGTACGTTTTT")[6:]])
    with pytest.raises(Exception, match="cannot complement unknown base 'R'"):
        gpu.count_random(bad, template, 1, 0, True)


def test_random_many_distinct_keys(gpu, kref):
    """Forces the device count table to grow several times."""
    rng = np.random.default_rng(3)
    template = "ACGTACGT" + "-" * 16 + "TTGCAGCA"
    reads = ["ACGTACGT" + random_seq(rng, 16) + "TTGCAGCA" for _ in range(60000)]
    f = fastq(reads)
    got = gpu.count_random(f, template, 0, 0, True)
    want = kref.count_random(f, template, 0, 0, True)
    _same(want, got)
    assert len(got[0]) > 59000


# ---- combinatorial, single-end ---------------------------------------------------------------------
@pytest.mark.parametrize("strand", ["original", "reverse", "both"])
@pytest.mark.parametrize("mm", [0, 1, 2])
@pytest.mark.parametrize("use_first", [True, False])
def test_combo_single(gpu, kref, strand, mm, use_first):
    rng = np.random.default_rng(31 + mm + 100 * STRANDS[strand])
    p1 = dense_pool(rng, 25, 5)
    p2 = dense_pool(rng, 30, 7)
    template = "ACGT" + "-" * 5 + "TGCAAG" + "-" * 7 + "GGA"
    reads = adversarial_reads(rng, 2500, template, [p1, p2], strand=strand)
    f = fastq(reads)
    _same(kref.count_combo_single(f, template, STRANDS[strand], p1, p2, mm, use_first),
          gpu.count_combo_single(f, template, STRANDS[strand], p1, p2, mm, use_first))
    assert np.array_equal(kref.trace_combo_single(f, template, STRANDS[strand], p1, p2, mm, use_first),
                          gpu.trace_combo_single(f, template, STRANDS[strand], p1, p2, mm, use_first))


def test_combo_single_config_shape_and_sparse(gpu, kref):
    """8+20+8+20+8 template (BASELINE configs[3] shape); a 5000 x 5000 pool forces the sparse (hash) tally."""
    rng = np.random.default_rng(11)
    template = "ACGTACGT" + "-" * 20 + "TTGGCCAA" + "-" * 20 + "GGATCCAT"
    for n in (500, 5000):
        p1 = distinct_pool(rng, n, 20)
        p2 = distinct_pool(rng, n, 20)
        reads = adversarial_reads(rng, 6000, template, [p1, p2], strand="original", sub_rate=0.01, n_rate=0.001, lower_rate=0,
                                  double_frac=0, short_frac=0)
        f = fastq(reads)
        for mm in (0, 1):
            _same(kref.count_combo_single(f, template, 0, p1, p2, mm, True), gpu.count_combo_single(f, template, 0, p1, p2, mm, True))


# ---- dual, single-end --------------------------------------------------------------------------------
@pytest.mark.parametrize("strand", ["original", "reverse", "both"])
@pytest.mark.parametrize("mm", [0, 1, 2])
@pytest.mark.parametrize("use_first", [True, False])
@pytest.mark.parametrize("diagnostics", [False, True])
def test_dual_single_end(gpu, kref, strand, mm, use_first, diagnostics):
    rng = np.random.default_rng(57 + mm + 100 * STRANDS[strand])
    g1 = dense_pool(rng, 12, 5)
    g2 = dense_pool(rng, 12, 6)
    pairs = sorted({(int(rng.integers(0, 12)), int(rng.integers(0, 12))) for _ in range(60)})[:40]
    p1 = [g1[i] for i, _ in pairs]
    p2 = [g2[j] for _, j in pairs]
    template = "ACGT" + "-" * 5 + "TGCAAG" + "-" * 6 + "GGA"
    reads = adversarial_reads(rng, 2500, template, [g1, g2], strand=strand)
    f = fastq(reads)
    _same(kref.count_dual_single_end(f, template, [p1, p2], STRANDS[strand], mm, use_first, diagnostics),
          gpu.count_dual_single_end(f, template, [p1, p2], STRANDS[strand], mm, use_first, diagnostics))
    if not diagnostics:
        assert np.array_equal(kref.trace_dual_single_end(f, template, [p1, p2], STRANDS[strand], mm, use_first),
                              gpu.trace_dual_single_end(f, template, [p1, p2], STRANDS[strand], mm, use_first))


def test_dual_single_end_three_regions_long_key(gpu, kref):
    rng = np.random.default_rng(77)
    lens = (20, 30, 25)   # 75-base concatenated key: three key words
    pools_g = [distinct_pool(rng, 15, n) for n in lens]
    rows = sorted({tuple(int(rng.integers(0, 15)) for _ in lens) for _ in range(50)})
    pools = [[pools_g[k][r[k]] for r in rows] for k in range(3)]
    template = "ACGT" + "-" * 20 + "TGCA" + "-" * 30 + "GGTT" + "-" * 25 + "CC"
    reads = adversarial_reads(rng, 2000, template, pools_g, strand="both", sub_rate=0.01)
    f = fastq(reads)
    for mm in (0, 1, 2):
        _same(kref.count_dual_single_end(f, template, pools, 2, mm, False), gpu.count_dual_single_end(f, template, pools, 2, mm, False))


# ---- dual, paired-end -----------------------------------------------------------------------------------
@pytest.mark.parametrize("rev", [(False, False), (True, False), (False, True)])
@pytest.mark.parametrize("mms", [(0, 0), (1, 1), (1, 0), (0, 1), (1, 2), (0, 2)])
@pytest.mark.parametrize("use_first", [True, False])
@pytest.mark.parametrize("randomized", [False, True])
def test_dual_paired(gpu, port, rev, mms, use_first, randomized):
    """Dense short guides with last-base variants so that the segmented-search phantom (Quirk A) fires.
    Checked against the C restatement in its cache-free mode; that restatement is itself checked against
    the compiled reference, cache included, in test_oracle_fuzz.py."""
    rng = np.random.default_rng(91 + 7 * mms[0] + 3 * mms[1] + rev[0] + 2 * rev[1])
    g1 = dense_pool(rng, 10, 4, 0.5)
    g2 = dense_pool(rng, 10, 4, 0.5)
    for k in range(3):
        s = g2[k]
        alt = s[:-1] + ("A" if s[-1] != "A" else "C")
        if alt not in g2:
            g2.append(alt)
    pairs = sorted({(int(rng.integers(0, len(g1))), int(rng.integers(0, len(g2)))) for _ in range(50)})[:35]
    p1 = [g1[i] for i, _ in pairs]
    p2 = [g2[j] for _, j in pairs]
    t1, t2 = "ACGT----TG", "GGA----CCT"
    f1, f2 = _paired_inputs(rng, 2000, t1, t2, g1, g2, rev[0], rev[1], swap_frac=0.3 if randomized else 0.0)
    want = port.trace_dual(f1, t1, rev[0], mms[0], p1, f2, t2, rev[1], mms[1], p2, randomized, use_first, fresh_state=2)
    got = gpu.trace_dual(f1, t1, rev[0], mms[0], p1, f2, t2, rev[1], mms[1], p2, randomized, use_first)
    assert np.array_equal(got, want)
    assert (want >= 0).sum() > 50
    counts, total = gpu.count_dual(f1, t1, rev[0], mms[0], p1, f2, t2, rev[1], mms[1], p2, randomized, use_first)
    assert total == 2000 and np.array_equal(counts, np.bincount(want[want >= 0], minlength=len(p1)))


@pytest.mark.parametrize("diagnostics", [False, True])
@pytest.mark.parametrize("randomized", [False, True])
@pytest.mark.parametrize("use_first", [True, False])
def test_dual_paired_against_reference(gpu, kref, diagnostics, randomized, use_first):
    """Config-3 shape (2 x 20-bp guides, pairs drawn from a guide set, 1 substitution per read): distinct random
    guides cannot trigger the reference's order dependence, so its normal threaded run is the yardstick."""
    rng = np.random.default_rng(5)
    g1 = distinct_pool(rng, 40, 20)
    g2 = distinct_pool(rng, 40, 20)
    pairs = sorted({(int(rng.integers(0, 40)), int(rng.integers(0, 40))) for _ in range(300)})
    p1 = [g1[i] for i, _ in pairs]
    p2 = [g2[j] for _, j in pairs]
    t1 = "CAGCTACGTACG" + "-" * 20 + "CCAGCTCGATCG"
    t2 = "TGGGCAGCGACA" + "-" * 20 + "ACACGAGGGTAT"
    r1 = adversarial_reads(rng, 4000, t1, [g1], strand="original", read_len=75, sub_rate=0.01, n_rate=0.001, lower_rate=0, double_frac=0, short_frac=0)
    r2 = adversarial_reads(rng, 4000, t2, [g2], strand="original", read_len=75, sub_rate=0.01, n_rate=0.001, lower_rate=0, double_frac=0, short_frac=0)
    if randomized:
        for i in range(0, 4000, 3):
            r1[i], r2[i] = r2[i], r1[i]
    f1, f2 = fastq(r1), fastq(r2)
    _same(kref.count_dual(f1, t1, False, 1, p1, f2, t2, False, 1, p2, randomized, use_first, diagnostics, nthreads=2),
          gpu.count_dual(f1, t1, False, 1, p1, f2, t2, False, 1, p2, randomized, use_first, diagnostics))
    # the reference is order-independent here: same per-pair outcome with and without its cache
    a = kref.trace_dual(f1, t1, False, 1, p1, f2, t2, False, 1, p2, randomized, use_first, fresh_state=0)
    b = gpu.trace_dual(f1, t1, False, 1, p1, f2, t2, False, 1, p2, randomized, use_first)
    assert np.array_equal(a, b)


def test_dual_paired_unsupported_budget(gpu):
    """2+ substitutions on read 1 walk the reference's trie on the device, which holds keys of up to 64 bases in total."""
    f = fastq(["ACGTAAAATG"])
    counts, total = gpu.count_dual(f, "ACGT----TG", False, 2, ["AAAA"], f, "ACGT----TG", False, 0, ["AAAA"], False, True)
    assert total == 1 and counts.tolist() == [1]
    long1, long2 = "A" * 40, "C" * 40
    with pytest.raises(Exception, match="at most 64 bp in total"):
        gpu.count_dual(f, "ACGT" + "-" * 40 + "TG", False, 2, [long1], f, "ACGT" + "-" * 40 + "TG", False, 0, [long2], False, True)


def test_paired_read_count_mismatch(gpu):
    f1 = fastq(["ACGTAAAATG", "ACGTAAAATG"])
    f2 = fastq(["ACGTAAAATG"])
    with pytest.raises(Exception, match="different number of reads in paired FASTQ files"):
        gpu.count_dual(f1, "ACGT----TG", False, 0, ["AAAA"], f2, "ACGT----TG", False, 0, ["AAAA"], False, True)
    with pytest.raises(Exception, match="different number of reads in paired FASTQ files"):
        gpu.count_combo_paired(f2, "ACGT----TG", False, 0, ["AAAA"], f1, "ACGT----TG", False, 0, ["AAAA"], False, True)


# ---- combinatorial, paired-end ------------------------------------------------------------------------------
@pytest.mark.parametrize("rev", [(False, False), (True, True), (True, False)])
@pytest.mark.parametrize("mms", [(0, 0), (1, 1), (2, 0)])
@pytest.mark.parametrize("use_first", [True, False])
@pytest.mark.parametrize("randomized", [False, True])
def test_combo_paired(gpu, kref, rev, mms, use_first, randomized):
    rng = np.random.default_rng(123 + mms[0])
    g1 = dense_pool(rng, 15, 5, 0.4)
    g2 = dense_pool(rng, 18, 5, 0.4)
    t1, t2 = "ACGT-----TG", "GGA-----CCT"
    f1, f2 = _paired_inputs(rng, 2000, t1, t2, g1, g2, rev[0], rev[1], swap_frac=0.3 if randomized else 0.0)
    _same(kref.count_combo_paired(f1, t1, rev[0], mms[0], g1, f2, t2, rev[1], mms[1], g2, randomized, use_first),
          gpu.count_combo_paired(f1, t1, rev[0], mms[0], g1, f2, t2, rev[1], mms[1], g2, randomized, use_first))
    a = kref.trace_combo_paired(f1, t1, rev[0], mms[0], g1, f2, t2, rev[1], mms[1], g2, randomized, use_first)
    b = gpu.trace_combo_paired(f1, t1, rev[0], mms[0], g1, f2, t2, rev[1], mms[1], g2, randomized, use_first)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


# ---- SingleBarcodePairedEnd (kaori handler without an R entry point) --------------------------------------------------
@pytest.mark.parametrize("strand", ["original", "both"])
@pytest.mark.parametrize("mm", [0, 1, 2])
@pytest.mark.parametrize("use_first", [True, False])
def test_single_barcode_paired_end(kref, strand, mm, use_first):
    from screencounter_b200 import rcpp
    rng = np.random.default_rng(50 + mm + 7 * STRANDS[strand])
    pool = dense_pool(rng, 60, 7)
    template = "ACGTA" + "-" * 7 + "TGCAT"
    # the barcode may sit on read 1, on read 2, on both (same or different barcodes, cleaner or noisier), or on neither
    r1 = adversarial_reads(rng, 4000, template, [pool], strand=strand, junk_frac=0.35)
    r2 = adversarial_reads(rng, 4000, template, [pool], strand=strand, junk_frac=0.35)
    same = rng.random(4000) < 0.3
    r2 = [a if s else b for a, b, s in zip(r1, r2, same)]
    f1, f2 = fastq(r1), fastq(r2)
    counts, total, index = rcpp.count_single_barcodes_paired(f1, f2, template, STRANDS[strand], pool, mm, use_first, 4, trace=True)
    assert total == 4000
    from oracle import kref as compiled
    if compiled.available():   # the C restatement has no entry point for this handler: its counts come from the rule below
        want_counts, want_total = compiled.count_single_paired(f1, f2, template, STRANDS[strand], pool, mm, use_first)
        assert want_total == 4000 and np.array_equal(counts, want_counts)
    assert np.array_equal(counts, np.bincount(index[index >= 0], minlength=len(pool)))
    # per pair against the single-barcode traces of the reference and the handler's rule
    i1, n1 = kref.trace_single(f1, template, STRANDS[strand], pool, mm, use_first)
    i2, n2 = kref.trace_single(f2, template, STRANDS[strand], pool, mm, use_first)
    if use_first:
        expect = np.where(i1 >= 0, i1, i2)
    else:
        m1, m2 = n1[:, 2], n2[:, 2]
        both = (i1 >= 0) & (i2 >= 0)
        expect = np.where(both, np.where(m1 < m2, i1, np.where(m1 > m2, i2, np.where(i1 == i2, i1, -1))), np.where(i1 >= 0, i1, i2))
    assert np.array_equal(index, expect)
    assert counts.sum() > 1000
