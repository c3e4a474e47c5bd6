"""The specialised dual paired-end, combinatorial and random-barcode kernels (spec_handlers.cuh) and their follow-up kernels
(runners_spec.cu) against the reference across template shapes, key splits and routes.

Like the single-barcode kernel (test_gpu_single_shapes.py), these kernels are compiled from the template: where each
strand's regions start in the window, how many words a window and a read take, and how the key is assembled from the
regions.  Each shape below moves one of those to an edge:
  dual      key splits at, around and over 32 bases, with LEN_A = 32 and LEN_B = 32 (the high word of the pair's key and
            the root-rule probe of the flat follow-up kernel), mates whose reads differ in word count;
  combo     regions of 1 and 32 bases, regions that start at window bit 30, 32 and 33, templates of 33 to 128 bases,
            pools of very different sizes (the reverse strand swaps the regions' pools);
  random    keys of 1 to 42 bases, asymmetric and one-sided flanks (the barcode is cut at the forward coordinates on both
            strands), both table routes of narrow keys (listed by table part, or counted in the home sector).
Every case asserts the route the launcher's guard implies, including the reason when it takes the generic kernel, and
compares per read (dual, combo) or the whole table (random) with the reference.  Every read of a case has one length.
"""
import ctypes as C
import itertools
import os
import re

import numpy as np
import pytest

from test_gpu_plans import _dual_library
from test_gpu_single_shapes import LEFT, RIGHT, constant_position_sets, dense_library, iupac_library, place, replace_at
from util import adversarial_reads, distinct_pool, fastq, fill_template, random_seq, revcomp

MID = "GGTACCTTAGCATTGACGATCCAGTCAAGGCTAGTCC"
# read 2's flanks in the dual design: another sequence again, so that the mates' scans differ
LEFT2 = "GATTACAGGCTA" + "TCCGATAAGCTTGCAGTCGAACTGG"
RIGHT2 = "TTGACCGTAGCA" + "AGGTCTTCAAGCGGATACCAGT"
MAX_READ = 160    # five words: the longest read the specialised kernels take
GENERIC_WHY = "mismatch budget too large for the pigeonhole filter"
DISABLED_WHY = "disabled by SCG_NO_SPEC_HANDLERS"


# ---- the launchers' guards ----------------------------------------------------------------------------------------------

def nconst(template):
    return sum(c != "-" for c in template)


def regions(template):
    """(start, length) of each run of '-'."""
    return [(m.start(), m.end() - m.start()) for m in re.finditer("-+", template)]


def spec_disabled():
    """SCG_NO_SPEC_HANDLERS=1 sends every design of this file to its generic kernel; the cases then check that route."""
    v = os.environ.get("SCG_NO_SPEC_HANDLERS", "")
    return bool(v) and v[0] != "0"


def template_fits(template, mm, read_len):
    """template_fits (runners_spec.cu) for reads of one length; the budget clamped as TemplateSpec::scan_spec does."""
    T, W = len(template), (read_len + 31) // 32
    mmc = max(0, min(mm, nconst(template)))
    return read_len - T + 1 >= 1 and W <= 5 and T <= 128 and W + 2 >= (T + 31) // 32 + 1 and mmc <= 3 and \
        nconst(template) >= 4 * (mmc + 1)


def dual_takes_spec(l1, l2, t1, mm1, n1, t2, mm2, n2):
    """launch_dual_pe: not randomized, a key of at most 48 bases, regions of at most 32, both templates fit."""
    return l1 + l2 <= 48 and l1 <= 32 and l2 <= 32 and template_fits(t1, mm1, n1) and template_fits(t2, mm2, n2)


def split(a, b, parts):
    return [(a + (b - a) * p // parts, a + (b - a) * (p + 1) // parts) for p in range(parts)]


def dual_flat(l1, l2, mm1, mm2):
    """Whether DualMatcher::build_flat qualifies the library: at most one mismatch per read, and every seed of the segmented
    library (library.cpp) holds positions."""
    if mm1 > 1 or mm2 > 1:
        return False
    c1, c2 = min(mm1, l1), min(mm2, l2)
    if c1 == 0 and c2 == 0:
        return False
    L = l1 + l2
    return all((r1[1] - r1[0]) + (r2[1] - r2[0]) > 0 for r1 in split(0, l1, c1 + 1) for r2 in split(l1, L, c2 + 1))


def combo_takes_spec(template, mm, read_len):
    """launch_combo: regions of at most 32 bases (one key word), no diagnostics pass, the template fits."""
    return all(n <= 32 for _, n in regions(template)) and template_fits(template, mm, read_len)


def random_parts(capacity, wide, parts_env=None):
    """The table parts launch_random lists the barcodes by (0: the home-sector route)."""
    table_bytes = capacity * 16
    nparts = 0
    if table_bytes > 48 << 20:
        nparts = 2
        while nparts < 32 and table_bytes // nparts > 12 << 20:
            nparts *= 2
    if parts_env is not None:
        nparts = 0 if parts_env <= 1 else 2
        while nparts and nparts < min(parts_env, 32):
            nparts *= 2
    while nparts > 0 and nparts * 2 > capacity:
        nparts //= 2
    return 0 if nparts < 2 or wide else nparts


FILE_TABLE = {False: 1 << 23, True: 1 << 20}   # count_random_reader's first table, narrow / wide
PLAN_TABLE = 1 << 20                           # scg_random_plan_create without expected_distinct


def random_note(template, mm, read_len, capacity, parts_env=None):
    """The part of the kernel note that names the route."""
    if spec_disabled() or not template_fits(template, mm, read_len):
        return "generic random_kernel"
    wide = regions(template)[0][1] > 21
    nparts = random_parts(capacity, wide, parts_env)
    if nparts:
        return "barcodes listed by table part (%d parts)" % nparts
    return "128-bit-key count table" if wide else "16-byte-slot count table (home sector requested a tile ahead)"


def part_cap(per_warp, nparts):
    """PartitionedKeys::cap of launch_random: keys one warp may list per part before it inserts them itself."""
    return per_warp // nparts + per_warp // (2 * nparts) + 64


def per_warp(n, group, grid):
    """DeferredList::per_warp of prepare_scratch."""
    ngroups = -(-(-(-n // 32)) // group)
    return -(-ngroups // (grid * 4)) * group * 32


def kernel_note(plan=None):
    from screencounter_b200 import rcpp
    return plan.kernel if plan is not None else rcpp.timing()["kernel"]


# ---- reads ------------------------------------------------------------------------------------------------------------

def variable_positions(template):
    return [j for j, c in enumerate(template) if c == "-"]


def constant_positions(template):
    return [j for j, c in enumerate(template) if c != "-"]


def template_reads(rng, template, sources, mm, read_len, n_background=1200, odd=False):
    """Reads of exactly read_len bases around constructs of `template` whose regions come from `sources` (one list per
    region): background with noise and reads of two constructs, exactly mm - 1, mm and mm + 1 constant mismatches, budgets
    split between the flanks and the regions (as bases and as Ns), a clean construct at every window on both strands and,
    in a share of the reads, lower case; odd=True also puts IUPAC letters into some constructs."""
    T = len(template)
    cpos, vpos = constant_positions(template), variable_positions(template)
    reads = []

    def orient(c):
        return revcomp(c) if rng.random() < 0.5 else c

    def clean():
        return fill_template(template, *[s[int(rng.integers(0, len(s)))] for s in sources])

    bg = adversarial_reads(rng, n_background, template, sources, strand="both", read_len=read_len, sub_rate=0.02, n_rate=0.004,
                           lower_rate=0.0, double_frac=0.2, short_frac=0.02, edge_frac=0.3)
    reads += [(r + random_seq(rng, read_len))[:read_len] for r in bg]
    for k in range(max(0, mm - 1), min(mm + 1, len(cpos)) + 1):
        for t, ps in enumerate(constant_position_sets(rng, cpos, k, budget_sets=120)):
            reads.append(place(rng, orient(replace_at(clean(), ps, [(t + j) % 4 for j in range(k)])), read_len))
    for total in (mm, mm + 1):
        for c in range(0, min(total, len(cpos)) + 1):
            v = total - c
            if v > len(vpos):
                continue
            for rep in range(8):
                s = replace_at(clean(), rng.choice(cpos, c, replace=False), rng.integers(0, 3, size=c))
                vp = rng.choice(vpos, v, replace=False)
                s = replace_at(s, vp, rng.integers(0, 3, size=v) if rep % 2 == 0 else [3] * v)
                reads.append(place(rng, orient(s), read_len))
    for off in range(read_len - T + 1):
        reads.append(place(rng, clean(), read_len, off))
        reads.append(place(rng, revcomp(clean()), read_len, off))
    for i in rng.choice(len(reads), len(reads) // 10, replace=False):
        mask = rng.random(read_len) < 0.4
        reads[i] = "".join(ch.lower() if m else ch for ch, m in zip(reads[i], mask))
    if odd:   # forward and upper case: the reference complements no ambiguity code but N
        for _ in range(40):
            s = list(clean())
            s[int(rng.choice(vpos))] = "RYKMSW"[int(rng.integers(0, 6))]
            reads.append(place(rng, "".join(s), read_len))
    reads = [reads[i] for i in rng.permutation(len(reads))]
    assert {len(r) for r in reads} == {read_len}
    return reads


def packed_text(reads):
    """What the packed layout keeps of a read: upper case, N for anything but ACGT (resident reads carry no raw text)."""
    return fastq(["".join(c if c in "ACGT" else "N" for c in r.upper()) for r in reads])


# ---- dual paired-end ----------------------------------------------------------------------------------------------------

# (L1, L2): the pair's key is read 1's region, then read 2's
DUAL_SPLITS = [(1, 1), (16, 16), (16, 17), (31, 1), (32, 1), (1, 32), (32, 16), (16, 32), (20, 20)]
DUAL_OVER = [(33, 1), (40, 8), (30, 20)]     # a region over 32 bases, or more than 48 in total: the generic kernel
DUAL_CAPS = [(0, 0), (1, 0), (0, 1), (1, 1), (2, 1), (1, 2)]
DUAL_REVS = [(False, False), (True, False), (False, True)]


def dual_templates(l1, l2):
    return LEFT[:12] + "-" * l1 + RIGHT[:10], LEFT2[:9] + "-" * l2 + RIGHT2[:14]


def dual_cases(si):
    """(rev, caps, use_first, mate read lengths) of one split: every cap pair once, each strand pair twice, both modes, and
    either mate at 160 bases with the other at its template's length."""
    t1, t2 = dual_templates(*DUAL_SPLITS[si])
    out = []
    for k, caps in enumerate(DUAL_CAPS):
        lens = (len(t1), MAX_READ) if (k + si) % 2 == 0 else (MAX_READ, len(t2) + 3)
        out.append((DUAL_REVS[(k + si) % 3], caps, (k + si // 2) % 2 == 0, lens))
    return out


def dual_library(rng, l1, l2, rows):
    """_dual_library (last-base variants of segment 2, so that the root-rule phantom fires) with pools small enough for
    one-base regions: `rows` library rows where the regions allow that many."""
    most1, most2 = 4 ** min(l1, 12), 4 ** min(l2, 12)
    n1, n2 = min(most1, 60), min(most2, 60)
    if n1 * n2 < 1.25 * rows:
        if most1 >= most2:
            n1 = min(most1, -(-5 * rows // (4 * n2)))
        else:
            n2 = min(most2, -(-5 * rows // (4 * n1)))
    return _dual_library(rng, n1, n2, l1, l2, min(rows, int(n1 * n2 / 1.25)), neighbours=0.5 if min(l1, l2) > 3 else 0.0)


def mutate_construct(rng, c, template, last_base):
    """0 to 3 constant substitutions; the region exact, with one or two substitutions, an N or (last_base) its last base
    changed."""
    cpos, vpos = constant_positions(template), variable_positions(template)
    k = int(rng.choice([0, 0, 0, 0, 1, 1, 2, 3]))
    c = replace_at(c, rng.choice(cpos, k, replace=False), rng.integers(0, 4, size=k))
    u = rng.random()
    if u < 0.25 and last_base:
        c = replace_at(c, [vpos[-1]], [int(rng.integers(0, 3))])
    elif u < 0.5:
        c = replace_at(c, [int(rng.choice(vpos))], [int(rng.integers(0, 3))])
    elif u < 0.6:
        c = replace_at(c, [int(rng.choice(vpos))], [3])
    elif u < 0.68 and len(vpos) > 1:
        c = replace_at(c, rng.choice(vpos, 2, replace=False), rng.integers(0, 3, size=2))
    return c


def mate_read(rng, c, second, read_len):
    if second is not None and 2 * len(c) + 2 <= read_len and rng.random() < 0.12:
        gap = int(rng.integers(0, read_len - 2 * len(c) + 1))
        return place(rng, c + random_seq(rng, gap) + second, read_len)
    return place(rng, c, read_len)


def dual_pairs(rng, t1, t2, rev, lib, lens, n=2400):
    g1, g2, p1, p2 = lib
    r1, r2 = [], []
    for _ in range(n):
        if rng.random() < 0.03:
            r1.append(random_seq(rng, lens[0]))
            r2.append(random_seq(rng, lens[1]))
            continue
        k = int(rng.integers(0, len(p1)))
        v1, v2 = (p1[k], p2[k]) if rng.random() < 0.85 else (g1[int(rng.integers(0, len(g1)))], g2[int(rng.integers(0, len(g2)))])
        c1 = mutate_construct(rng, fill_template(t1, v1), t1, False)
        c2 = mutate_construct(rng, fill_template(t2, v2), t2, True)
        other = int(rng.integers(0, len(p1)))
        s1, s2 = fill_template(t1, p1[other]), fill_template(t2, p2[other])
        if rev[0] != (rng.random() < 0.04):
            c1, s1 = revcomp(c1), revcomp(s1)
        if rev[1] != (rng.random() < 0.04):
            c2, s2 = revcomp(c2), revcomp(s2)
        r1.append(mate_read(rng, c1, s1, lens[0]))
        r2.append(mate_read(rng, c2, s2, lens[1]))
    return r1, r2


def check_dual(kref, r1, r2, t1, t2, rev, caps, p1, p2, use_first, route):
    """route: 'flat' / 'trie' (the specialised kernel and its follow-up) or 'generic'."""
    from screencounter_b200 import rcpp
    route = "generic" if spec_disabled() else route
    f1, f2 = fastq(r1), fastq(r2)
    args = (f1, t1, rev[0], caps[0], p1, f2, t2, rev[1], caps[1], p2, False, use_first)
    want = kref.trace_dual(*args, fresh_state=2)
    counts, total, got = rcpp.count_dual_barcodes(*args, False, 1, trace=True)
    note = kernel_note()
    if route == "generic":
        assert note.startswith("generic dual_pe_kernel"), note
    else:
        assert "spec_dual_pe_kernel" in note, note
        assert ("dual_deferred_flat_kernel" if route == "flat" else "dual_deferred_kernel") in note, note
    assert total[0] == len(r1)
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, "%d pairs differ, first %d: %r / %r got %d want %d" % (bad.size, bad[0], r1[bad[0]], r2[bad[0]], got[bad[0]], want[bad[0]])
    assert np.array_equal(counts, np.bincount(want[want >= 0], minlength=len(p1)))
    return want


def dual_route(l1, l2, t1, t2, caps, lens, no_flat=False):
    if not dual_takes_spec(l1, l2, t1, caps[0], lens[0], t2, caps[1], lens[1]):
        return "generic"
    return "flat" if dual_flat(l1, l2, *caps) and not no_flat else "trie"


DUAL_MATRIX = [(si, ci) for si in range(len(DUAL_SPLITS)) for ci in range(len(DUAL_CAPS))]


@pytest.mark.gpu
@pytest.mark.parametrize("si,ci", DUAL_MATRIX, ids=["%d+%d-%d" % (DUAL_SPLITS[si] + (ci,)) for si, ci in DUAL_MATRIX])
def test_dual_split_matrix_against_reference(kref, si, ci):
    l1, l2 = DUAL_SPLITS[si]
    t1, t2 = dual_templates(l1, l2)
    rev, caps, use_first, lens = dual_cases(si)[ci]
    rng = np.random.default_rng(700 + 10 * si + ci)
    lib = dual_library(rng, l1, l2, 80)
    r1, r2 = dual_pairs(rng, t1, t2, rev, lib, lens)
    want = check_dual(kref, r1, r2, t1, t2, rev, caps, lib[2], lib[3], use_first, dual_route(l1, l2, t1, t2, caps, lens))
    assert (want >= 0).any()


@pytest.mark.gpu
@pytest.mark.parametrize("si", range(len(DUAL_SPLITS)), ids=["%d+%d" % s for s in DUAL_SPLITS])
def test_dual_split_followup_routes_against_reference(kref, monkeypatch, si):
    """The trie-walking follow-up (SCG_DUAL_NO_FLAT=1) at 1 024 and 1 025 library rows (counters in shared memory or not),
    and the flat follow-up without shared-memory counters (SCG_SPEC_HIST_MAX=0).  Two one-base regions make 16 pairs:
    that split runs with 12 rows."""
    l1, l2 = DUAL_SPLITS[si]
    t1, t2 = dual_templates(l1, l2)
    rev, caps, lens = DUAL_REVS[si % 3], (1, 0) if si % 2 else (1, 1), (len(t1), MAX_READ)
    for rows in (1024, 1025) if 4 ** (l1 + l2) > 2000 else (12,):
        rng = np.random.default_rng(900 + 10 * si + rows % 2)
        lib = dual_library(rng, l1, l2, rows)
        assert len(lib[2]) == rows
        r1, r2 = dual_pairs(rng, t1, t2, rev, lib, lens, n=3000)
        with monkeypatch.context() as mp:
            mp.setenv("SCG_DUAL_NO_FLAT", "1")
            check_dual(kref, r1, r2, t1, t2, rev, caps, lib[2], lib[3], si % 2 == 0, dual_route(l1, l2, t1, t2, caps, lens, True))
        if rows != 1025:
            with monkeypatch.context() as mp:
                mp.setenv("SCG_SPEC_HIST_MAX", "0")
                check_dual(kref, r1, r2, t1, t2, rev, caps, lib[2], lib[3], si % 2 == 1, dual_route(l1, l2, t1, t2, caps, lens))


@pytest.mark.gpu
@pytest.mark.parametrize("split", DUAL_OVER, ids=["%d+%d" % s for s in DUAL_OVER])
@pytest.mark.parametrize("caps", [(1, 0), (1, 1)], ids=str)
def test_dual_split_over_the_limits_takes_the_generic_kernel(kref, split, caps):
    l1, l2 = split
    t1, t2 = dual_templates(l1, l2)
    rng = np.random.default_rng(l1 * 100 + l2 + caps[1])
    lib = dual_library(rng, l1, l2, 80)
    lens = (len(t1), MAX_READ)
    r1, r2 = dual_pairs(rng, t1, t2, (False, True), lib, lens)
    assert dual_route(l1, l2, t1, t2, caps, lens) == "generic"
    check_dual(kref, r1, r2, t1, t2, (False, True), caps, lib[2], lib[3], True, "generic")


# ---- combinatorial, single-end ------------------------------------------------------------------------------------------

# (left flank, region 1, middle, region 2, right flank)
COMBO_SHAPES = [
    (8, 1, 8, 1, 8), (8, 1, 8, 32, 8), (8, 32, 8, 32, 8), (8, 31, 8, 2, 8), (6, 5, 6, 7, 6), (10, 20, 8, 20, 10),
    (14, 4, 11, 4, 0), (0, 6, 9, 6, 12),          # one-sided templates
    (4, 8, 5, 8, 8),                              # 33 bases: two words per window
    (16, 8, 16, 8, 16), (16, 8, 17, 8, 16),       # 64 and 65
    (30, 5, 8, 7, 46),                            # 96; region 1 starts at window bit 30 and crosses into the second word
    (32, 6, 20, 6, 33),                           # 97; region 1 starts at bit 32
    (33, 20, 20, 20, 35),                         # 128; region 1 starts at bit 33
    (1, 8, 2, 8, 1), (1, 8, 1, 8, 1),             # 4 and 3 constant positions: budget 0's limit and one below
    (3, 8, 2, 8, 3), (2, 8, 2, 8, 3),             # 8 and 7: budget 1
    (4, 8, 4, 8, 4), (4, 8, 3, 8, 4),             # 12 and 11: budget 2
    (5, 8, 6, 8, 5), (5, 8, 5, 8, 5),             # 16 and 15: budget 3
]


def combo_template(shape):
    a, l1, m, l2, b = shape
    return LEFT[:a] + "-" * l1 + MID[:m] + "-" * l2 + RIGHT[:b]


def combo_id(shape):
    return "%d+%d+%d+%d+%d" % shape


def combo_kinds(shape):
    return ["distinct", "dense", "iupac"] if min(shape[1], shape[3]) >= 5 else ["distinct"]


def combo_pool(rng, kind, n, L):
    if kind == "dense":
        return dense_library(rng, n, L)
    if kind == "iupac":
        return iupac_library(rng, n, L)
    pool = distinct_pool(rng, min(n, 3 * 4 ** L // 4), L)
    return pool, pool


def combo_pools(rng, kind, sizes, shape):
    """Pool 1 is never smaller than pool 2, so that an index taken from the wrong pool still lands inside the dense matrix."""
    p1, s1 = combo_pool(rng, kind, sizes[0], shape[1])
    p2, s2 = combo_pool(rng, kind, min(sizes[1], len(p1)), shape[3])
    return p1, p2, [s1, s2]


def combo_cases(si, shape):
    """(strand, mm, use_first, read_len, kind, pool sizes): at strand 2 every budget, both modes, four read lengths; strands
    0 and 1 once each; pools of very different sizes (140 x 7: 980 counters in shared memory) and of similar ones."""
    T = len(combo_template(shape))
    lens = [T, min(T + 31, MAX_READ), min(T + 33, MAX_READ), MAX_READ]
    kinds = combo_kinds(shape)
    sizes = [(140, 7), (60, 45), (300, 9)]
    out = []
    for k in range(4):
        out.append((2, (k + si) % 4, (k + si // 2) % 2 == 0, lens[k], kinds[(k + si) % len(kinds)], sizes[(k + si) % 3]))
    out.append((0, si % 4, si % 2 == 0, lens[(si + 1) % 4], kinds[(si + 1) % len(kinds)], sizes[si % 3]))
    out.append((1, (si + 2) % 4, si % 2 == 1, lens[(si + 3) % 4], kinds[(si + 2) % len(kinds)], sizes[(si + 1) % 3]))
    return out


def check_combo(kref, reads, template, strand, p1, p2, mm, use_first, spec):
    from screencounter_b200 import rcpp
    data = fastq(reads)
    want_trace = kref.trace_combo_single(data, template, strand, p1, p2, mm, use_first)
    want_keys, want_freq, want_total = kref.count_combo_single(data, template, strand, p1, p2, mm, use_first)
    keys, freq, total, trace = rcpp.count_combo_barcodes_single(data, template, strand, [p1, p2], mm, use_first, 1, trace=True)
    note = kernel_note()
    if spec_disabled():
        assert note == "generic combo_kernel (%s)" % DISABLED_WHY, note
    elif spec:
        assert "spec_combo_kernel" in note, note
    else:
        assert note == "generic combo_kernel (%s)" % GENERIC_WHY, note
    bad = np.flatnonzero((trace != want_trace).any(axis=1))
    assert bad.size == 0, "%d reads differ, first %d: %r got %r want %r" % (bad.size, bad[0], reads[bad[0]], trace[bad[0]].tolist(),
                                                                         want_trace[bad[0]].tolist())
    assert np.array_equal(keys.T, want_keys) and np.array_equal(freq, want_freq) and total[0] == want_total
    return want_trace


COMBO_MATRIX = [(si, ci) for si in range(len(COMBO_SHAPES)) for ci in range(6)]


@pytest.mark.gpu
@pytest.mark.parametrize("si,ci", COMBO_MATRIX, ids=["%s-%d" % (combo_id(COMBO_SHAPES[si]), ci) for si, ci in COMBO_MATRIX])
def test_combo_shape_matrix_against_reference(kref, si, ci):
    shape = COMBO_SHAPES[si]
    template = combo_template(shape)
    strand, mm, use_first, read_len, kind, sizes = combo_cases(si, shape)[ci]
    rng = np.random.default_rng(3000 + 10 * si + ci)
    p1, p2, sources = combo_pools(rng, kind, sizes, shape)
    reads = template_reads(rng, template, sources, mm, read_len)
    want = check_combo(kref, reads, template, strand, p1, p2, mm, use_first, combo_takes_spec(template, mm, read_len))
    assert (want[:, 0] >= 0).any()


COMBO_VARIANTS = [("SCG_COMBO_NO_FLAT", "1"), ("SCG_COMBO_FORCE_SPARSE", "1"), ("SCG_SPEC_HIST_MAX", "0")]


@pytest.mark.gpu
@pytest.mark.parametrize("si", range(len(COMBO_SHAPES)), ids=[combo_id(s) for s in COMBO_SHAPES])
def test_combo_shape_other_routes_against_reference(kref, monkeypatch, si):
    """One read set of 160 bases per shape at a budget of one through each follow-up and tally variant, and pools of
    32 x 32 and 41 x 25 (1 024 and 1 025 cells: counters in shared memory or not) where the regions allow them."""
    shape = COMBO_SHAPES[si]
    template = combo_template(shape)
    mm = 1
    rng = np.random.default_rng(5000 + si)
    p1, p2, sources = combo_pools(rng, "distinct", (140, 7), shape)
    reads = template_reads(rng, template, sources, mm, MAX_READ, n_background=800)
    spec = combo_takes_spec(template, mm, MAX_READ)
    for name, value in COMBO_VARIANTS:
        with monkeypatch.context() as mp:
            mp.setenv(name, value)
            check_combo(kref, reads, template, 2, p1, p2, mm, si % 2 == 0, spec)
    if min(shape[1], shape[3]) >= 3:
        for sizes in ((32, 32), (41, 25)):
            p1, p2, sources = combo_pools(rng, "distinct", sizes, shape)
            assert len(p1) * len(p2) in (1024, 1025)
            reads = template_reads(rng, template, sources, mm, MAX_READ, n_background=800)
            check_combo(kref, reads, template, 2, p1, p2, mm, si % 2 == 1, spec)


# ---- random barcodes ----------------------------------------------------------------------------------------------------

# (left flank, key length, right flank)
RANDOM_SHAPES = [
    (12, 1, 9), (10, 2, 14), (5, 3, 12), (0, 8, 16), (16, 20, 0), (11, 21, 13),     # narrow: the 64-bit table
    (14, 22, 10), (0, 31, 20), (12, 32, 12), (20, 33, 5), (48, 41, 39), (30, 42, 50),  # wide: 128-bit keys; 128 and 122 bases
]


def random_template(shape):
    return LEFT[:shape[0]] + "-" * shape[1] + RIGHT[:shape[2]]


def random_id(shape):
    return "%d+%d+%d" % shape


def random_cases(si, shape):
    """(strand, mm, use_first, read_len): every budget, both modes, the template's length up to 160 bases, each strand."""
    T = sum(shape)
    lens = [T, min(T + 32, MAX_READ), MAX_READ, min(T + 5, MAX_READ)]
    return [(2, si % 4, False, lens[si % 4]), (2, (si + 1) % 4, True, lens[(si + 1) % 4]), (2, (si + 2) % 4, False, lens[(si + 2) % 4]),
            (0, (si + 3) % 4, si % 2 == 0, lens[(si + 3) % 4]), (1, si % 4, si % 2 == 1, lens[si % 4])]


def random_reads(rng, template, L, mm, read_len):
    """template_reads around a pool of barcodes, plus a tagged subset in which every read carries a barcode of its own (a
    wrong row of the table then points at one read)."""
    barcodes = distinct_pool(rng, min(300, 3 * 4 ** L // 4), L)
    reads = template_reads(rng, template, [barcodes], mm, read_len, n_background=1000, odd=True)
    if L >= 8:
        for b in distinct_pool(rng, 300, L):
            c = fill_template(template, b)
            reads.append(place(rng, revcomp(c) if rng.random() < 0.5 else c, read_len))
    return [reads[i] for i in rng.permutation(len(reads))]


def want_random(kref, text, template, strand, mm, use_first):
    seqs, freq, total = kref.count_random(text, template, strand, mm, use_first)
    order = sorted(range(len(seqs)), key=lambda i: seqs[i])
    return [seqs[i] for i in order], np.asarray(freq, dtype=np.int32)[order], total


def check_random_file(kref, reads, template, strand, mm, use_first, note_part, text=None):
    from screencounter_b200 import rcpp
    text = fastq(reads) if text is None else text
    want = want_random(kref, text, template, strand, mm, use_first)
    (seqs, freq), total = rcpp.count_random_barcodes(text, template, strand, mm, use_first, 1, as_array=False)
    note = kernel_note()
    assert note_part in note, note
    assert total == want[2]
    assert list(seqs) == want[0]
    assert np.array_equal(freq, want[1])
    return want


def check_random_plan(kref, reads, template, strand, mm, use_first, note_part):
    from screencounter_b200.device import RandomPlan, Reads
    text = packed_text(reads)
    want = want_random(kref, text, template, strand, mm, use_first)
    resident = Reads.from_fastq(text)
    plan = RandomPlan(template, strand, mm, use_first)
    try:
        plan.run(resident)
        seqs, freq = plan.harvest(as_array=False)
        assert note_part in plan.kernel, plan.kernel
        assert list(seqs) == want[0]
        assert np.array_equal(freq, want[1])
    finally:
        plan.free()
        resident.free()


RANDOM_MATRIX = [(si, ci) for si in range(len(RANDOM_SHAPES)) for ci in range(5)]


@pytest.mark.gpu
@pytest.mark.parametrize("si,ci", RANDOM_MATRIX, ids=["%s-%d" % (random_id(RANDOM_SHAPES[si]), ci) for si, ci in RANDOM_MATRIX])
def test_random_shape_matrix_against_reference(kref, si, ci):
    """A file-level call (narrow keys: listed by table part) and a RandomPlan on the same reads (narrow keys: the home
    sector), both against the reference."""
    shape = RANDOM_SHAPES[si]
    template = random_template(shape)
    strand, mm, use_first, read_len = random_cases(si, shape)[ci]
    rng = np.random.default_rng(8000 + 10 * si + ci)
    reads = random_reads(rng, template, shape[1], mm, read_len)
    wide = shape[1] > 21
    want = check_random_file(kref, reads, template, strand, mm, use_first, random_note(template, mm, read_len, FILE_TABLE[wide]))
    assert want[1].sum() > 0   # (one row only where Quirk B cuts a constant base of the reverse strand)
    check_random_plan(kref, reads, template, strand, mm, use_first, random_note(template, mm, read_len, PLAN_TABLE))


SKEW_TEMPLATE = LEFT[:12] + "-" * 16 + RIGHT[:10]


@pytest.mark.gpu
@pytest.mark.parametrize("nparts", [16, 32])
def test_random_skewed_library_overflows_the_part_lists(kref, monkeypatch, nparts):
    """One barcode in 80 to 90 % of the reads: a warp lists more keys for its part than PartitionedKeys::cap allows and
    counts the rest straight into the table.  With SCG_SPH_GROUP=4 and a grid that is not saturated every warp takes one
    group of 128 reads.  The dominant barcode sits on the forward strand only: the flanks differ in length, so on the
    reverse strand the barcode is cut at other bases (Quirk B) and would make a second key, in another part."""
    rng = np.random.default_rng(nparts)
    read_len, group, n = 96, 4, 5000 + 17
    dominant = random_seq(rng, 16)
    others = distinct_pool(rng, 400, 16)
    reads, is_dominant = [], []
    for i in range(n):
        warp_share = 0.8 + 0.1 * ((i // 128) % 2)
        dom = rng.random() < warp_share
        c = fill_template(SKEW_TEMPLATE, dominant if dom else others[int(rng.integers(0, len(others)))])
        if rng.random() < 0.05:
            c = replace_at(c, [int(rng.integers(0, len(c)))], [int(rng.integers(0, 4))])
            dom = False
        reads.append(place(rng, revcomp(c) if not dom and rng.random() < 0.5 else c, read_len))
        is_dominant.append(dom)
    # the grid: ngroups / 4 blocks of four warps, far below the device's resident blocks
    ngroups = -(-(-(-n // 32)) // group)
    pw = per_warp(n, group, -(-ngroups // 4))
    assert pw == group * 32
    cap = part_cap(pw, nparts)
    most = max(sum(is_dominant[w * pw:(w + 1) * pw]) for w in range(-(-n // pw)))
    assert most > cap, (most, cap)
    monkeypatch.setenv("SCG_SPH_GROUP", str(group))
    monkeypatch.setenv("SCG_RANDOM_PARTS", str(nparts))
    want = check_random_file(kref, reads, SKEW_TEMPLATE, 2, 1, True, random_note(SKEW_TEMPLATE, 1, read_len, FILE_TABLE[False], nparts))
    assert max(want[1]) > 0.7 * n
    monkeypatch.setenv("SCG_RANDOM_PARTS", "0")
    check_random_file(kref, reads, SKEW_TEMPLATE, 2, 1, False, random_note(SKEW_TEMPLATE, 1, read_len, FILE_TABLE[False], 0))


@pytest.mark.gpu
def test_random_skewed_library_at_scale(kref, monkeypatch):
    """Two million synthetic reads of two barcodes on the device, a plan with a table of 8 M slots (16 parts) and the
    default knobs: the grid saturates, every warp takes several groups, and each part list overflows.  Against the
    reference and against the home-sector route (SCG_RANDOM_PARTS=0)."""
    import torch
    from screencounter_b200.device import RandomPlan, SynthSpec
    template = LEFT[:12] + "-" * 16 + RIGHT[:12]
    spec = SynthSpec(template, [], seed=29, read_len=75, strand=2, random_space=2, sub_per_10k=20, n_per_10k=5)
    n = 2_000_003
    reads = spec.on_device(0, n)
    want = want_random(kref, spec.fastq(0, n), template, 2, 1, True)
    tables = []
    for parts_env in (None, "0"):
        with monkeypatch.context() as mp:
            if parts_env is not None:
                mp.setenv("SCG_RANDOM_PARTS", parts_env)
            plan = RandomPlan(template, 2, 1, True, expected_distinct=1 << 22)
            plan.run(reads)
            tables.append(plan.harvest(as_array=False))
            note = plan.kernel
            plan.free()
        if spec_disabled():
            assert "generic random_kernel" in note, note
        elif parts_env is None:
            assert "(16 parts)" in note, note
            blocks = int(re.search(r"(\d+) blocks/SM", note).group(1))
            sms = torch.cuda.get_device_properties(0).multi_processor_count
            ngroups = -(-(-(-n // 32)) // 2)
            grid = min((ngroups + 3) // 4, sms * blocks)
            assert grid < (ngroups + 3) // 4   # saturated
            pw = per_warp(n, 2, grid)
            assert pw > 2 * 32
            assert max(want[1]) / n * pw > 1.2 * part_cap(pw, 16), (max(want[1]), pw)
        else:
            assert random_note(template, 1, 75, 1 << 23, 0) in note, note
    for seqs, freq in tables:
        assert list(seqs) == want[0] and np.array_equal(freq, want[1])


# ---- staging knobs ------------------------------------------------------------------------------------------------------

# (GROUP, STAGES) per design that fit the 48 KiB of static shared memory at reads of 64 bases
STAGING = {"dual": [(1, 1), (1, 3), (2, 1), (2, 3)], "combo": [(1, 1), (1, 3), (4, 1), (4, 3)], "random": [(1, 1), (1, 3), (4, 1), (4, 3)]}
STAGING_CASES = [(d, g, s) for d, gs in STAGING.items() for g, s in gs]
STAGING_LEN = 64


@pytest.mark.gpu
@pytest.mark.parametrize("design,group,stages", STAGING_CASES, ids=["%s-g%d-s%d" % c for c in STAGING_CASES])
def test_staging_knobs_against_reference(kref, monkeypatch, design, group, stages):
    """Read counts that are not a multiple of GROUP x 32: the last bulk copy is only partly filled."""
    monkeypatch.setenv("SCG_SPH_GROUP", str(group))
    monkeypatch.setenv("SCG_SPH_STAGES", str(stages))
    rng = np.random.default_rng(100 * group + stages + len(design))
    if design == "dual":
        l1, l2 = 20, 20
        t1, t2 = dual_templates(l1, l2)
        lib = dual_library(rng, l1, l2, 200)
        r1, r2 = dual_pairs(rng, t1, t2, (False, True), lib, (STAGING_LEN, STAGING_LEN), n=3001 + 37 * group + 3 * stages)
        assert len(r1) % (group * 32)
        check_dual(kref, r1, r2, t1, t2, (False, True), (1, 1), lib[2], lib[3], stages == 1, "flat")
    elif design == "combo":
        shape = (8, 20, 8, 20, 8)
        template = combo_template(shape)
        p1, p2, sources = combo_pools(rng, "distinct", (140, 7), shape)
        reads = template_reads(rng, template, sources, 1, STAGING_LEN)
        reads = reads[: len(reads) - (len(reads) % (group * 32) == 0)]
        assert len(reads) % (group * 32)
        check_combo(kref, reads, template, 2, p1, p2, 1, stages == 1, True)
    else:
        template = random_template((12, 16, 12))
        reads = random_reads(rng, template, 16, 1, STAGING_LEN)
        reads = reads[: len(reads) - (len(reads) % (group * 32) == 0)]
        assert len(reads) % (group * 32)
        check_random_file(kref, reads, template, 2, 1, stages == 1, random_note(template, 1, STAGING_LEN, FILE_TABLE[False]))
        check_random_plan(kref, reads, template, 2, 1, stages != 1, random_note(template, 1, STAGING_LEN, PLAN_TABLE))


# ---- no GPU needed ------------------------------------------------------------------------------------------------------

def selftest(kind, a, strand_a, mm_a, b, strand_b, mm_b, read_len, use_first):
    from screencounter_b200._lib import lib
    buf = C.create_string_buffer(16384)
    rc = lib().scg_jit_selftest_handler(kind, a.encode(), strand_a, mm_a, b.encode(), strand_b, mm_b, read_len, int(use_first), buf,
                                        C.c_size_t(16384))
    return rc, buf.value.decode(errors="replace")


def compile_variants():
    """(design, kind, template a, strand a, mm a, template b, strand b, mm b, read length, use_first, env) of every
    specialised variant the GPU tests run.  Dual variants are built with both mates at the longer mate's length."""
    out = []
    for si, (l1, l2) in enumerate(DUAL_SPLITS):
        t1, t2 = dual_templates(l1, l2)
        for rev, caps, use_first, lens in dual_cases(si):
            if dual_takes_spec(l1, l2, t1, caps[0], lens[0], t2, caps[1], lens[1]):
                out.append(("dual", 1, t1, int(rev[0]), caps[0], t2, int(rev[1]), caps[1], max(lens), use_first, ()))
    for si, shape in enumerate(COMBO_SHAPES):
        template = combo_template(shape)
        for strand, mm, use_first, read_len, _, _ in combo_cases(si, shape):
            if combo_takes_spec(template, mm, read_len):
                out.append(("combo", 2, template, strand, mm, "", 0, 0, read_len, use_first, ()))
    for si, shape in enumerate(RANDOM_SHAPES):
        template = random_template(shape)
        for strand, mm, use_first, read_len in random_cases(si, shape):
            if template_fits(template, mm, read_len):
                for capacity in (FILE_TABLE[shape[1] > 21], PLAN_TABLE):
                    kind = 4 if random_parts(capacity, shape[1] > 21) else 3
                    out.append(("random", kind, template, strand, mm, "", 0, 0, read_len, use_first, ()))
    for design, group, stages in STAGING_CASES:
        env = (("SCG_SPH_GROUP", str(group)), ("SCG_SPH_STAGES", str(stages)))
        if design == "dual":
            t1, t2 = dual_templates(20, 20)
            out.append(("dual", 1, t1, 0, 1, t2, 1, 1, STAGING_LEN, stages == 1, env))
        elif design == "combo":
            out.append(("combo", 2, combo_template((8, 20, 8, 20, 8)), 2, 1, "", 0, 0, STAGING_LEN, stages == 1, env))
        else:
            for kind in (3, 4):
                out.append(("random", kind, random_template((12, 16, 12)), 2, 1, "", 0, 0, STAGING_LEN, stages == 1, env))
    return sorted(set(out))


COMPILE_VARIANTS = compile_variants()


@pytest.mark.parametrize("design", ["dual", "combo", "random"])
def test_handler_variants_compile(monkeypatch, design):
    """Every specialised variant the GPU tests run, through NVRTC (kinds 1 to 4): 0 = compiled and loaded, 2 = compiled,
    nothing to load it on.  A variant that does not compile would silently take the generic kernel."""
    variants = [v for v in COMPILE_VARIANTS if v[0] == design]
    assert len(variants) >= 12
    for _, kind, a, sa, ma, b, sb, mb, read_len, use_first, env in variants:
        with monkeypatch.context() as mp:
            for name, value in env:
                mp.setenv(name, value)
            rc, msg = selftest(kind, a, sa, ma, b, sb, mb, read_len, use_first)
        assert rc in (0, 2), (kind, a, sa, ma, b, sb, mb, read_len, env, msg[-400:])


def test_guard_refuses_one_constant_position_below_the_limit():
    """For every budget the specialised route takes the fewest constant positions the pigeonhole filter needs, and refuses
    one fewer with the reason the generic route's kernel note gives."""
    for mm in range(4):
        at = [s for s in COMBO_SHAPES if nconst(combo_template(s)) == 4 * (mm + 1)]
        below = [s for s in COMBO_SHAPES if nconst(combo_template(s)) == 4 * (mm + 1) - 1]
        assert at and below, mm
        for s in at:
            assert combo_takes_spec(combo_template(s), mm, MAX_READ)
            rc, msg = selftest(2, combo_template(s), 2, mm, "", 0, 0, MAX_READ, True)
            assert rc in (0, 2), msg
        for s in below:
            assert not combo_takes_spec(combo_template(s), mm, MAX_READ)
            rc, msg = selftest(2, combo_template(s), 2, mm, "", 0, 0, MAX_READ, True)
            assert rc == 1 and GENERIC_WHY in msg, msg


def test_shape_tables_hold_the_edges():
    assert set(DUAL_SPLITS) >= {(1, 1), (16, 16), (16, 17), (31, 1), (32, 1), (1, 32), (32, 16), (16, 32), (20, 20)}
    for a, b in DUAL_SPLITS + DUAL_OVER:
        t1, t2 = dual_templates(a, b)
        assert dual_takes_spec(a, b, t1, 2, MAX_READ, t2, 2, MAX_READ) == ((a, b) in DUAL_SPLITS)
    assert {c for _, c, _, _ in itertools.chain.from_iterable(dual_cases(si) for si in range(len(DUAL_SPLITS)))} == set(DUAL_CAPS)
    assert any(dual_flat(a, b, 1, 0) and a + b > 32 for a, b in DUAL_SPLITS)   # the phantom's bit in the second word
    pairs = {(s[1], s[3]) for s in COMBO_SHAPES}
    assert pairs >= {(1, 1), (1, 32), (32, 32), (31, 2), (5, 7), (20, 20)}
    assert {len(combo_template(s)) for s in COMBO_SHAPES} >= {33, 64, 65, 96, 97, 128}
    assert {s[0] for s in COMBO_SHAPES} >= {30, 32, 33}
    for si, shape in enumerate(COMBO_SHAPES):
        cases = combo_cases(si, shape)
        assert max(c[3] for c in cases) == MAX_READ and {c[0] for c in cases} == {0, 1, 2}
    assert {s[1] for s in RANDOM_SHAPES} >= {1, 2, 3, 8, 20, 21, 22, 31, 32, 33, 41, 42}
    assert max(sum(s) for s in RANDOM_SHAPES) == 128 and any(s[0] == 0 for s in RANDOM_SHAPES) and any(s[2] == 0 for s in RANDOM_SHAPES)
    # narrow file-level calls list the barcodes by table part, narrow plans count in the home sector, wide keys never take parts
    assert random_parts(FILE_TABLE[False], False) == 16 and random_parts(PLAN_TABLE, False) == 0
    assert random_parts(FILE_TABLE[True], True) == 0 and random_parts(FILE_TABLE[False], False, 32) == 32
    assert part_cap(128, 16) == 76 and part_cap(128, 32) == 70
