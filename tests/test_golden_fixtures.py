"""Committed reference outputs (tests/golden/reference_vectors.json.gz, made by
tests/golden/make_golden.py from the unmodified reference compiled in the build container):
the C restatement is pinned to them on the CPU, the CUDA path on the GPU.  Integer work, so
every comparison is exact."""
import gzip
import json
import os

import numpy as np
import pytest

from util import fastq

HERE = os.path.dirname(os.path.abspath(__file__))

with gzip.open(os.path.join(HERE, "golden", "reference_vectors.json.gz"), "rb") as _f:
    DOC = json.loads(_f.read().decode())
CASES = DOC["cases"]


def _eq(got, want, what):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape and np.array_equal(got, want), "%s differs from the reference fixture" % what


def _sorted_table(seqs, freq):
    order = np.argsort(np.array(list(seqs)))
    return [list(seqs)[i] for i in order], np.asarray(freq)[order]


def _pair_table(pairs):
    """Per-read (or per-pair) combinations -> the table the reference reports: the distinct matched rows with their counts."""
    pairs = np.asarray(pairs).reshape(-1, 2)
    return np.unique(pairs[(pairs >= 0).all(axis=1)], axis=0, return_counts=True)


def _eq_table(got_keys, got_freq, c, what):
    want_keys = np.asarray(c["keys"]).reshape(len(c["freq"]), -1)
    order = np.lexsort(want_keys.T[::-1]) if len(want_keys) else np.zeros(0, dtype=np.int64)
    _eq(got_keys.reshape(len(got_freq), -1), want_keys[order], what + " (combinations)")
    _eq(got_freq, np.asarray(c["freq"])[order], what + " (frequencies)")


def check(engine, c):
    kind = c["kind"]
    if kind == "single":
        f = fastq(c["reads"])
        counts, total = engine.count_single(f, c["template"], c["strand"], c["pool"], c["mismatches"], c["use_first"])
        _eq(counts, c["counts"], "counts")
        assert total == c["total"]
        index, info = engine.trace_single(f, c["template"], c["strand"], c["pool"], c["mismatches"], c["use_first"])
        _eq(index, c["index"], "per-read index")
        _eq(info, c["info"], "per-read match details")
    elif kind == "random":
        seqs, freq, total = engine.count_random(fastq(c["reads"]), c["template"], c["strand"], c["mismatches"], c["use_first"])
        seqs, freq = _sorted_table(seqs, freq)
        assert seqs == c["seqs"]
        _eq(freq, c["freq"], "frequencies")
        assert total == c["total"]
    elif kind == "combo_single":
        keys, freq, total = engine.count_combo_single(fastq(c["reads"]), c["template"], c["strand"], c["pool1"], c["pool2"],
                                                      c["mismatches"], c["use_first"])
        _eq(np.asarray(keys).reshape(len(freq), -1), np.asarray(c["keys"]).reshape(len(c["freq"]), -1), "combinations")
        _eq(freq, c["freq"], "frequencies")
        assert total == c["total"]
        trace = engine.trace_combo_single(fastq(c["reads"]), c["template"], c["strand"], c["pool1"], c["pool2"], c["mismatches"],
                                          c["use_first"])
        _eq_table(*_pair_table(trace), c, "per-read combinations")
    elif kind == "dual_single_end":
        res = engine.count_dual_single_end(fastq(c["reads"]), c["template"], c["pools"], c["strand"], c["mismatches"], c["use_first"],
                                           c["diagnostics"])
        _eq(res[0], c["counts"], "counts")
        assert res[1] == c["total"]
        if c["diagnostics"]:
            _eq(np.asarray(res[2]).reshape(len(res[3]), -1), np.asarray(c["keys"]).reshape(len(c["freq"]), -1), "invalid combinations")
            _eq(res[3], c["freq"], "invalid frequencies")
        index = np.asarray(engine.trace_dual_single_end(fastq(c["reads"]), c["template"], c["pools"], c["strand"], c["mismatches"],
                                                        c["use_first"]))
        _eq(np.bincount(index[index >= 0], minlength=len(c["counts"])), c["counts"], "counts of the per-read trace")
    elif kind == "dual":
        f1, f2 = fastq(c["reads1"]), fastq(c["reads2"])
        args = (f1, c["template1"], c["reverse1"], c["mismatches1"], c["pool1"], f2, c["template2"], c["reverse2"], c["mismatches2"],
                c["pool2"], c["randomized"], c["use_first"])
        # cache-free semantics (SURVEY 8.1 T20): the per-pair outcomes with a fresh reference state per pair
        index = engine.trace_dual(*args, fresh_state=1)
        _eq(index, c["index_fresh"], "per-pair index")
        res = engine.count_dual(*args, c["diagnostics"])
        fresh = np.asarray(c["index_fresh"])
        _eq(res[0], np.bincount(fresh[fresh >= 0], minlength=len(c["pool1"])), "counts (cache-free)")
        if c["order_dependent_pairs"] == 0:
            _eq(res[0], c["counts"], "counts")
        assert res[1] == c["total"]
        if c["diagnostics"] and c["order_dependent_pairs"] == 0:
            _eq(np.asarray(res[2]).reshape(len(res[3]), -1), np.asarray(c["keys"]).reshape(len(c["freq"]), -1), "invalid combinations")
            _eq(res[3], c["freq"], "invalid frequencies")
            assert (res[4], res[5]) == (c["barcode1_only"], c["barcode2_only"])
    elif kind == "combo_paired":
        f1, f2 = fastq(c["reads1"]), fastq(c["reads2"])
        keys, freq, total, b1, b2 = engine.count_combo_paired(f1, c["template1"], c["reverse1"], c["mismatches1"], c["pool1"], f2,
                                                              c["template2"], c["reverse2"], c["mismatches2"], c["pool2"],
                                                              c["randomized"], c["use_first"])
        _eq(np.asarray(keys).reshape(len(freq), -1), np.asarray(c["keys"]).reshape(len(c["freq"]), -1), "combinations")
        _eq(freq, c["freq"], "frequencies")
        assert (total, b1, b2) == (c["total"], c["barcode1_only"], c["barcode2_only"])
        combo, code = engine.trace_combo_paired(f1, c["template1"], c["reverse1"], c["mismatches1"], c["pool1"], f2, c["template2"],
                                                c["reverse2"], c["mismatches2"], c["pool2"], c["randomized"], c["use_first"])
        _eq_table(*_pair_table(combo), c, "per-pair combinations")
        code = np.asarray(code)
        assert (int((code == 2).sum()), int((code == 3).sum())) == (c["barcode1_only"], c["barcode2_only"])
    elif kind == "match":
        if "error" in c:
            with pytest.raises(Exception):
                engine.match_barcodes(c["seqs"], c["choices"], c["substitutions"], c["reverse"])
            return
        index, mm = engine.match_barcodes(c["seqs"], c["choices"], c["substitutions"], c["reverse"])
        _eq(index, c["index"], "index")
        want_mm = np.where(np.asarray(c["index"]) >= 0, np.asarray(c["mm"]), -1)
        _eq(np.where(np.asarray(index) >= 0, np.asarray(mm), -1), want_mm, "mismatches")
    else:
        raise AssertionError("unknown fixture kind " + kind)


def test_fixture_is_complete():
    kinds = {c["kind"] for c in CASES}
    assert kinds == {"single", "random", "combo_single", "dual_single_end", "dual", "combo_paired", "match"}
    assert all(c["order_dependent_pairs"] >= 0 for c in CASES if c["kind"] == "dual")


@pytest.mark.parametrize("case", CASES, ids=lambda c: c["name"])
def test_port_matches_reference_fixture(port, case):
    check(port, case)


@pytest.mark.parametrize("case", [c for c in CASES if c["kind"] == "match" and "error" not in c], ids=lambda c: c["name"])
def test_port_search_any_matches_reference_fixture(port, case):
    """The restatement's search with a cap per query (the yardstick of tests/test_gpu_segmented.py), every cap set to the
    substitutions of the reference's matchBarcodes run, finds what that run found."""
    caps = np.full(len(case["seqs"]), case["substitutions"], dtype=np.int32)
    index, mm = port.search_any(case["seqs"], caps, case["choices"], case["substitutions"], case["reverse"])
    index = np.where(index >= 0, index, -1)   # no hit (-1) and an ambiguous one (-2) are both NA in matchBarcodes
    _eq(index, case["index"], "index")
    _eq(np.where(np.asarray(index) >= 0, mm, -1), np.where(np.asarray(case["index"]) >= 0, np.asarray(case["mm"]), -1), "mismatches")


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=lambda c: c["name"])
def test_gpu_matches_reference_fixture(case):
    from engines import GpuEngine
    check(GpuEngine(), case)
