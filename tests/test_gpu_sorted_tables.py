"""The sorted device tables (include/scg.h scg_table_*) against a plain host reference, on keys that collide where the table
kernels resolve them: rows that share word 0 and differ in word 1, rows that differ only in their last base or only at bases
20 and 21 (where word 0 ends), the extreme words (all-A is 0, all-T has bit 62 set), combinations that share their first
index, and tables larger than the grid the kernels launch (sm_count * 32 blocks of 256 threads).  Also: the same keys counted
from reads at every key width, the many-files matrix on colliding keys, sparse combination tables, and the refusal of rows
that are not a sorted table.

The host reference: a barcode table is its keys in the layout of include/scg.h (three bits a base, A=0 < C=1 < G=2 < N=3 <
T=4, word 0 = bases 0..20, word 1 = the rest), rows sorted by (word 0, word 1), which is text order; a combination key is
first << 32 | second."""
import numpy as np
import pytest

from util import fastq, random_seq, revcomp, distinct_pool, adversarial_reads

pytestmark = pytest.mark.gpu

F12, R12 = "CAGCTACGTACG", "CCAGCTCGATCG"
KEY_LENS = [0, 1, 2, 20, 21, 22, 23, 32, 41, 42]   # 0: combinations
SIZES = [0, 1, 2, 255, 256, 257]
OVERLAPS = ["disjoint", "interleaved", "identical", "a_in_b", "b_in_a", "a_empty", "both_empty"]
LETTERS = np.frombuffer(b"ACGNT", dtype="S1")
TOP = (1 << 31) - 1


# ---------------------------------------------------------------------------------------------------------------------
# host reference
# ---------------------------------------------------------------------------------------------------------------------
def _words(ranks):
    """(rows, key_len) base ranks -> (rows, words) int64 keys in the layout of include/scg.h (the numpy form of _word in
    tests/test_multi_wide_gloo.py)."""
    ranks = np.asarray(ranks, dtype=np.int64)

    def word(cols):
        w = np.zeros(cols.shape[0], dtype=np.int64)
        for j in range(cols.shape[1]):
            w = (w << 3) | cols[:, j]
        return w

    if ranks.shape[1] <= 21:
        return word(ranks)[:, None]
    return np.stack([word(ranks[:, :21]), word(ranks[:, 21:])], axis=1)


def _strings(keys, key_len):
    """Keys of the layout above -> S<key_len> barcodes."""
    n0 = min(key_len, 21)
    ranks = np.empty((keys.shape[0], key_len), dtype=np.uint8)
    for j in range(key_len):
        ranks[:, j] = (keys[:, 0] >> (3 * (n0 - 1 - j)) if j < 21 else keys[:, 1] >> (3 * (key_len - 1 - j))) & 7
    return LETTERS.view(np.uint8)[ranks].view("S%d" % key_len).reshape(-1)


def _keys_of(seqs, key_len):
    """Barcodes (str) -> their keys."""
    text = "".join(seqs).encode().translate(bytes.maketrans(b"ACGNT", bytes(range(5))))
    return _words(np.frombuffer(text, dtype=np.uint8).reshape(len(seqs), key_len))


def _unique_sorted(keys):
    """Rows of `keys` (rows, words), sorted by (word 0, word 1), each once."""
    if keys.shape[0] == 0:
        return keys
    k = keys[np.lexsort(keys.T[::-1])]
    keep = np.ones(k.shape[0], dtype=bool)
    keep[1:] = np.any(k[1:] != k[:-1], axis=1)
    return k[keep]


def _union(*tables):
    """The merge of host tables (keys, counts): keys sorted and unique, counts of equal keys added."""
    keys = np.concatenate([t[0] for t in tables])
    counts = np.concatenate([t[1] for t in tables]).astype(np.int64)
    if keys.shape[0] == 0:
        return keys, counts
    order = np.lexsort(keys.T[::-1])
    keys, counts = keys[order], counts[order]
    start = np.ones(keys.shape[0], dtype=bool)
    start[1:] = np.any(keys[1:] != keys[:-1], axis=1)
    at = np.flatnonzero(start)
    return keys[at], np.add.reduceat(counts, at)


def _barcode_families(rng, key_len):
    """Sorted unique keys of key_len bases: last-base and first-base siblings, runs that share word 0 with ranks 0 and 4 at
    base 21 and at the last base, pairs that differ only at bases 20 and 21, all-A, all-T, all-N, and random keys."""
    L = key_len
    parts = []
    for col in (-1, 0):   # 50 stems, each with all five letters at the last base / at the first base
        sib = np.repeat(rng.integers(0, 5, (50, L)), 5, axis=0)
        sib[:, col] = np.tile(np.arange(5), 50)
        parts.append(sib)
    if L >= 22:
        prefixes = rng.integers(0, 5, (4, L))
        prefixes[0, :21], prefixes[1, :21] = 0, 4   # word 0 of zero and word 0 with bit 62 set
        shared = np.repeat(prefixes, 60, axis=0)
        shared[:, 21:] = rng.integers(0, 5, (shared.shape[0], L - 21))
        shared[0::4, 21], shared[1::4, 21], shared[2::4, -1], shared[3::4, -1] = 0, 4, 0, 4
        parts.append(shared)
        stems = rng.integers(0, 5, (40, L))
        x = rng.integers(0, 5, 40)
        y = (x + rng.integers(1, 5, 40)) % 5
        p, q = stems.copy(), stems.copy()
        p[:, 20], p[:, 21], q[:, 20], q[:, 21] = x, y, y, x
        parts += [p, q]
    parts.append(np.array([[0] * L, [4] * L, [3] * L]))
    parts.append(rng.integers(0, 5, (300, L)))
    return _unique_sorted(_words(np.concatenate(parts)))


def _combo_families(rng):
    """Sorted unique combination keys: runs of many seconds under one first, indices 0 and 2^31 - 1 on both sides."""
    firsts = np.concatenate([[0, 1, 2, TOP - 1, TOP], rng.integers(0, TOP, 7)])
    seconds = [np.concatenate([[0, 1, TOP - 1, TOP], rng.integers(0, TOP, 36)]) for _ in firsts]
    keys = np.concatenate([(np.int64(f) << 32) | s.astype(np.int64) for f, s in zip(firsts, seconds)])
    return _unique_sorted(keys[:, None])


def _families(rng, key_len):
    return _combo_families(rng) if key_len == 0 else _barcode_families(rng, key_len)


def _pick(rng, pool, size, overlap, where):
    """Tables a, b, c (key arrays) of about `size` rows from a window of adjacent keys of the sorted pool, so that the rows of
    a and b are each other's nearest neighbours.  where: 0 = the window starts at the pool's first key, 1 = ends at its last,
    2 = anywhere."""
    m = pool.shape[0]
    span = min(2 * size, m)
    start = [0, m - span, int(rng.integers(0, m - span + 1))][where]
    w = pool[start:start + span]
    half = w[: min(size, span)]
    a, b = {
        "disjoint": (half, w[half.shape[0]:]),
        "interleaved": (w[0::2], _unique_sorted(np.concatenate([w[1::2], w[0::4]]))),
        "identical": (half, half),
        "a_in_b": (w[0::2], w),
        "b_in_a": (w, w[0::2]),
        "a_empty": (w[:0], half),
        "both_empty": (w[:0], w[:0]),
    }[overlap]
    c = w[rng.random(span) < 0.5]
    return a, b, c


def _counts(rng, n):
    return rng.integers(1, 1 << 20, n).astype(np.int64)


# ---------------------------------------------------------------------------------------------------------------------
# device side
# ---------------------------------------------------------------------------------------------------------------------
class Tables:
    """Device tables made through DeviceTableOps, freed when the test ends."""

    def __init__(self):
        from screencounter_b200.multi import DeviceTableOps
        self.ops = DeviceTableOps(0)
        self.handles = []

    def keep(self, h):
        self.handles.append(h)
        return h

    def load(self, keys, counts, key_len, flat=False):
        import torch
        k = torch.from_numpy(np.ascontiguousarray(keys[:, 0] if flat else keys)).to("cuda:0")
        c = torch.from_numpy(np.asarray(counts).astype(np.int32)).to("cuda:0")
        return self.keep(self.ops.from_tensors(k, c, key_len))

    def merge(self, a, b):
        return self.keep(self.ops.merge(a, b))

    def free(self):
        for h in self.handles:
            self.ops.free(h)
        self.handles = []


@pytest.fixture
def tables():
    t = Tables()
    yield t
    t.free()


def _same_table(tables, h, keys, counts, key_len):
    """The device table `h` holds exactly (keys, counts): its views, and its rendering as the file-level calls return it."""
    vkeys, vcounts = tables.ops.views(h)
    words = 2 if key_len > 21 else 1
    assert tuple(vkeys.shape) == (keys.shape[0], words)
    assert np.array_equal(vkeys.cpu().numpy(), keys)
    assert np.array_equal(vcounts.cpu().numpy(), counts)
    rkeys, freq = tables.ops.render(h)
    assert np.array_equal(freq, counts)
    if key_len == 0:
        pairs = np.stack([keys[:, 0] >> 32, keys[:, 0] & 0xFFFFFFFF], axis=1).astype(np.int32)
        assert np.array_equal(rkeys.reshape(-1, 2), pairs)
    else:
        want = _strings(keys, key_len)
        assert (want[1:] > want[:-1]).all()   # key order is text order
        assert np.array_equal(rkeys, want)


# ---------------------------------------------------------------------------------------------------------------------
# a. table algebra on hand-built keys
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("overlap", OVERLAPS)
@pytest.mark.parametrize("key_len", KEY_LENS)
def test_table_algebra_on_colliding_keys(tables, key_len, overlap):
    rng = np.random.default_rng(100 * key_len + OVERLAPS.index(overlap))
    pool = _families(rng, key_len)
    for i, size in enumerate(SIZES):
        a, b, c = _pick(rng, pool, size, overlap, i % 3)
        ta, tb, tc = (a, _counts(rng, a.shape[0])), (b, _counts(rng, b.shape[0])), (c, _counts(rng, c.shape[0]))
        flat = key_len == 0 and i % 2 == 0   # one-word keys as (rows,) as well as (rows, 1)
        ha, hb, hc = (tables.load(*t, key_len, flat=flat) for t in (ta, tb, tc))
        for h, t in ((ha, ta), (hb, tb), (hc, tc)):
            _same_table(tables, h, *t, key_len)
        ab = _union(ta, tb)
        _same_table(tables, tables.merge(ha, hb), *ab, key_len)
        _same_table(tables, tables.merge(hb, ha), *ab, key_len)
        abc = _union(ta, tb, tc)
        _same_table(tables, tables.merge(tables.merge(ha, hb), hc), *abc, key_len)
        _same_table(tables, tables.merge(ha, tables.merge(hb, hc)), *abc, key_len)
        _same_table(tables, tables.merge(ha, ha), a, 2 * ta[1], key_len)
        empty = tables.load(a[:0], ta[1][:0], key_len)
        _same_table(tables, tables.merge(ha, empty), *ta, key_len)
        _same_table(tables, tables.merge(empty, ha), *ta, key_len)
        tables.free()


@pytest.mark.parametrize("key_len", [21, 42])
def test_merge_and_render_above_the_launch_grid(tables, key_len):
    """About 1.5 M rows a table: more than one grid-stride round of every merge and render kernel."""
    rng = np.random.default_rng(key_len)
    stems = rng.integers(0, 5, (450_000, key_len))
    ranks = np.repeat(stems, 5, axis=0)
    ranks[:, -1] = np.tile(np.arange(5), stems.shape[0])
    pool = _unique_sorted(_words(ranks))
    u = rng.random(pool.shape[0])
    in_a, in_b = u < 2 / 3, u > 1 / 3
    ca, cb = _counts(rng, pool.shape[0]), _counts(rng, pool.shape[0])
    ta, tb = (pool[in_a], ca[in_a]), (pool[in_b], cb[in_b])
    assert min(in_a.sum(), in_b.sum()) > 1_400_000
    ha, hb = tables.load(*ta, key_len), tables.load(*tb, key_len)
    _same_table(tables, ha, *ta, key_len)
    both = in_a | in_b
    want = (pool[both], (np.where(in_a, ca, 0) + np.where(in_b, cb, 0))[both])
    _same_table(tables, tables.merge(ha, hb), *want, key_len)
    _same_table(tables, tables.merge(hb, ha), *want, key_len)


def test_boundary_rows_are_accepted(tables):
    """The largest values a table may hold: all-T barcodes (bit 62 of word 0 set), combination indices of 2^31 - 1, counts of
    2^31 - 1."""
    for key_len in (1, 21, 22, 42):
        keys = _words(np.array([[0] * key_len, [3] * key_len, [4] * key_len]))
        counts = np.array([1, TOP, TOP - 1])
        _same_table(tables, tables.load(keys, counts, key_len), keys, counts, key_len)
    keys = np.array([[0], [TOP], [(TOP << 32) | TOP]], dtype=np.int64)
    _same_table(tables, tables.load(keys, np.array([TOP, 1, 2]), 0), keys, np.array([TOP, 1, 2]), 0)


# ---------------------------------------------------------------------------------------------------------------------
# b. sort and extraction from reads, at every width
# ---------------------------------------------------------------------------------------------------------------------
def _template(key_len):
    return F12 + "-" * key_len + R12


def _reads(rng, barcodes, key_len):
    """1..3 reads a barcode, of one length, each construct forward or reverse-complemented at a random offset."""
    length = len(_template(key_len)) + 8
    out = []
    for s in barcodes:
        for _ in range(int(rng.integers(1, 4))):
            c = F12 + s + R12
            if rng.random() < 0.5:
                c = revcomp(c)
            left = random_seq(rng, int(rng.integers(0, 9)))
            out.append((left + c + random_seq(rng, 8))[:length])
    return out


def _barcodes(rng, key_len):
    return [s.decode() for s in _strings(_barcode_families(rng, key_len), key_len)]


def _want(kref, text, key_len, strand, mismatches, use_first):
    seqs, freq, total = kref.count_random(text, _template(key_len), strand, mismatches, use_first)
    order = sorted(range(len(seqs)), key=lambda i: seqs[i])
    return [seqs[i] for i in order], np.asarray(freq, dtype=np.int32)[order], total


# (strand, mismatches, use_first): every strand
OPTIONS = [(0, 0, True), (1, 1, False), (2, 1, True)]


@pytest.mark.parametrize("options", OPTIONS, ids=str)
@pytest.mark.parametrize("key_len", KEY_LENS[1:])
def test_count_random_on_colliding_barcodes(kref, key_len, options, monkeypatch):
    """The device count table, its compaction and radix sort, and the render, on the specialised route and the generic one."""
    from screencounter_b200 import rcpp
    strand, mismatches, use_first = options
    rng = np.random.default_rng(key_len)
    text = fastq(_reads(rng, _barcodes(rng, key_len), key_len))
    want = _want(kref, text, key_len, strand, mismatches, use_first)
    assert len(want[0]) >= min(5 ** key_len, 400) // 4
    for generic in ("0", "1"):
        monkeypatch.setenv("SCG_NO_SPEC_HANDLERS", generic)
        (seqs, freq), total = rcpp.count_random_barcodes(text, _template(key_len), strand, mismatches, use_first, 2, device=0, as_array=False)
        assert list(seqs) == want[0]
        assert np.array_equal(freq, want[1])
        assert total == want[2]


@pytest.mark.parametrize("key_len", KEY_LENS[1:])
def test_random_plan_sorted_table_on_colliding_barcodes(kref, tables, key_len):
    from screencounter_b200.device import RandomPlan, Reads
    rng = np.random.default_rng(key_len + 1)
    text = fastq(_reads(rng, _barcodes(rng, key_len), key_len))
    want_seqs, want_freq, _ = _want(kref, text, key_len, 2, 1, True)
    plan = RandomPlan(_template(key_len), 2, 1, True)
    reads = Reads.from_fastq(text)
    try:
        plan.run(reads)
        seqs, freq = plan.harvest(as_array=False)
        assert list(seqs) == want_seqs and np.array_equal(freq, want_freq)
        _same_table(tables, tables.keep(tables.ops.from_plan(plan)), _keys_of(want_seqs, key_len), want_freq, key_len)
    finally:
        reads.free()
        plan.free()


@pytest.mark.parametrize("devices", [0, (0, 0)], ids=str)
@pytest.mark.parametrize("key_len", [21, 22, 42])
def test_matrix_columns_on_colliding_barcodes(kref, key_len, devices, monkeypatch):
    """Three files whose barcodes partly overlap: the union and scatter_column_kernel on neighbouring keys."""
    from screencounter_b200 import rcpp
    monkeypatch.setenv("SCG_MULTI_MIN_BYTES", "1000")
    rng = np.random.default_rng(7 * key_len)
    barcodes = _barcodes(rng, key_len)
    member = rng.random((3, len(barcodes))) < 0.6
    texts = [fastq(_reads(rng, [s for s, m in zip(barcodes, member[f]) if m], key_len)) for f in range(3)]
    seqs, counts, totals = rcpp.matrix_of_random_barcodes(texts, _template(key_len), 2, 1, True, 2, device=devices, as_array=False)
    per_file = [kref.count_random(t, _template(key_len), 2, 1, True) for t in texts]
    union = sorted(set(s for p in per_file for s in p[0]))
    assert list(seqs) == union
    for f, (s, fr, total) in enumerate(per_file):
        col = dict(zip(s, fr))
        assert counts[:, f].tolist() == [col.get(u, 0) for u in union]
        assert totals[f] == total


# ---------------------------------------------------------------------------------------------------------------------
# c. sparse combination tables
# ---------------------------------------------------------------------------------------------------------------------
COMBO_TEMPLATE = "CAGCTACG" + "-" * 12 + "GGTACCTT" + "-" * 12 + "CGATCGAG"


@pytest.mark.parametrize("n1,n2", [(6, 400), (40, 40)])
def test_sparse_combination_tables(kref, tables, n1, n2, monkeypatch):
    """The device hash tally of combinations (forced), with few first indices: long runs of keys that share their upper half."""
    import ctypes as C
    from screencounter_b200 import rcpp
    from screencounter_b200._lib import lib
    from screencounter_b200.device import ComboPlan, Reads
    monkeypatch.setenv("SCG_COMBO_FORCE_SPARSE", "1")
    rng = np.random.default_rng(n1)
    p1, p2 = distinct_pool(rng, n1, 12), distinct_pool(rng, n2, 12)
    text = fastq(adversarial_reads(rng, 8000, COMBO_TEMPLATE, [p1, p2], strand="both", read_len=70, lower_rate=0.0, short_frac=0.0))
    wkeys, wfreq, wtotal = kref.count_combo_single(text, COMBO_TEMPLATE, 2, p1, p2, 1, True)
    wkeys = np.asarray(wkeys).reshape(-1, 2)
    assert len(wfreq) > n1
    keys, freq, total = rcpp.count_combo_barcodes_single(text, COMBO_TEMPLATE, 2, [p1, p2], 1, True, 2, device=0)
    assert np.array_equal(keys.T, wkeys) and np.array_equal(freq, wfreq) and total[0] == wtotal
    plan = ComboPlan(COMBO_TEMPLATE, 2, p1, p2, 1, True)
    reads = Reads.from_fastq(text)
    try:
        plan.run(reads)
        ptr, cells = C.c_void_p(), C.c_longlong()
        lib().scg_plan_dense_tally(plan.handle, C.byref(ptr), C.byref(cells))
        assert not ptr.value   # the hash tally, not the dense matrix
        hkeys, hfreq = plan.harvest()
        assert np.array_equal(hkeys, wkeys) and np.array_equal(hfreq, wfreq)
        want = ((wkeys[:, 0].astype(np.int64) << 32) | wkeys[:, 1].astype(np.int64))[:, None]
        _same_table(tables, tables.keep(tables.ops.from_plan(plan)), want, np.asarray(wfreq), 0)
    finally:
        reads.free()
        plan.free()


# ---------------------------------------------------------------------------------------------------------------------
# d. refusals
# ---------------------------------------------------------------------------------------------------------------------
def _refused(tables, keys, counts, key_len, match):
    from screencounter_b200.rcpp import ScreenCounterError
    with pytest.raises(ScreenCounterError, match=match):
        tables.load(np.asarray(keys, dtype=np.int64), np.asarray(counts), key_len)


def _bad_word(w):
    """An unsigned 64-bit word as the int64 a tensor holds."""
    return np.array([w], dtype=np.uint64).view(np.int64)[0]


def test_unsorted_and_repeated_rows_are_refused(tables):
    one, wide = _words(np.array([[1] * 20, [2] * 20])), _words(np.array([[1] * 30, [2] * 30]))
    _refused(tables, one[::-1], [1, 1], 20, "not in ascending key order")
    _refused(tables, one[[0, 0]], [1, 1], 20, "a key appears in two rows")
    # word 0 equal, word 1 descending / equal
    w = wide.copy()
    w[1, 0] = w[0, 0]
    _refused(tables, w[::-1], [1, 1], 30, "not in ascending key order")
    _refused(tables, wide[[1, 1]], [1, 1], 30, "a key appears in two rows")
    _refused(tables, np.array([[5], [4]]), [1, 1], 0, "not in ascending key order")
    # a swap near the end of a table larger than the launch grid
    keys = np.arange(0, 4_000_000, 2, dtype=np.int64)[:, None]
    keys[[-3, -2]] = keys[[-2, -3]]
    _refused(tables, keys, np.ones(keys.shape[0]), 21, "not in ascending key order")
    keys[[-3, -2]] = keys[[-2, -3]]
    keys[-1] = keys[-2]
    _refused(tables, keys, np.ones(keys.shape[0]), 21, "a key appears in two rows")


@pytest.mark.parametrize("rank", [5, 6, 7])
def test_ranks_above_4_are_refused(tables, rank):
    for key_len, word, group in ((1, 0, 0), (20, 0, 19), (21, 0, 20), (30, 0, 0), (30, 1, 8), (42, 1, 20)):
        keys = _words(np.zeros((1, key_len), dtype=np.int64))
        keys[0, word] |= rank << (3 * group)
        _refused(tables, keys, [1], key_len, "a base rank above 4")


def test_bits_above_the_key_are_refused(tables):
    for key_len, word, bit in ((1, 0, 3), (20, 0, 60), (21, 0, 63), (22, 1, 3), (30, 1, 27), (42, 1, 63), (42, 0, 63)):
        keys = _words(np.zeros((1, key_len), dtype=np.int64))
        keys[0, word] = _bad_word((1 << bit) | int(keys[0, word]))
        _refused(tables, keys, [1], key_len, "bits set beyond its key length")


def test_combination_indices_and_counts_of_2_31_are_refused(tables):
    for key in ((1 << 31) << 32, 1 << 31, (1 << 63) | 5, (1 << 64) - 1):
        _refused(tables, [[_bad_word(key)]], [1], 0, r"a combination index is 2\^31 or more")
    for key_len in (0, 20, 42):
        keys = np.zeros((2, 2 if key_len > 21 else 1), dtype=np.int64)
        keys[1, -1] = 1
        for count in (1 << 31, (1 << 32) - 1):
            _refused(tables, keys, np.array([1, count], dtype=np.uint32).view(np.int32), key_len, r"a count is 2\^31 or more")


def test_key_lengths_outside_0_to_42_are_refused(tables):
    _refused(tables, np.zeros((1, 1)), [1], -1, "key length -1 is outside 0..42")
    _refused(tables, np.zeros((1, 2)), [1], 43, "key length 43 is outside 0..42")
    _refused(tables, np.zeros((0, 2)), [], 43, "key length 43 is outside 0..42")


def test_malformed_tensors_are_refused(tables):
    import torch
    ops = tables.ops
    keys2 = torch.zeros((4, 2), dtype=torch.int64, device="cuda:0")
    keys1 = torch.arange(4, dtype=torch.int64, device="cuda:0")
    counts = torch.ones(4, dtype=torch.int32, device="cuda:0")
    bad = [
        (keys1, counts, 30, "must have shape"),              # (rows,) keys where rows have two words
        (keys2, counts, 20, "must have shape"),              # two words where rows have one
        (keys1.reshape(2, 2), counts, 30, "counts must have shape"),
        (keys2[:, :1].repeat(1, 3), counts, 30, "must have shape"),
        (keys1, counts[:3], 20, "counts must have shape"),
        (keys1.to(torch.int32), counts, 20, "keys must be an int64 tensor"),
        (keys1.to(torch.float64), counts, 20, "keys must be an int64 tensor"),
        (keys1.cpu(), counts, 20, "keys must be an int64 tensor on cuda:0"),
        (keys1.cpu().numpy(), counts, 20, "keys must be an int64 tensor"),
        (keys1, counts.to(torch.int64), 20, "counts must be an int32 tensor"),
        (keys1, counts.cpu(), 20, "counts must be an int32 tensor on cuda:0"),
    ]
    for k, c, key_len, match in bad:
        with pytest.raises(ValueError, match=match):
            tables.keep(ops.from_tensors(k, c, key_len))
    # the same tensors in the right form are accepted
    _same_table(tables, tables.keep(ops.from_tensors(keys1, counts, 20)), keys1.cpu().numpy()[:, None], np.ones(4, dtype=np.int64), 20)
