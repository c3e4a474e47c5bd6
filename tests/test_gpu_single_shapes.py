"""The uniform-length single-barcode kernel (spec_single.cuh, DESIGN.md 5.1b) against the reference across template shapes.

Almost everything in that kernel is a compile-time function of the template: the pigeonhole groups of constant positions and
their samples, the words of a window, where each strand's variable region starts, the key mask, the joint exact table, the
seeds of the mismatch search and the window-block masks.  Each shape below moves one of those to an edge: asymmetric and
one-sided flanks, keys of 1 to 32 bases, regions that cross a word of the window, templates of one to four words, and the
fewest constant positions the route takes for a budget (and one fewer, where it must not take it).

Per case, every read has the same length, and the read set hits the edges on purpose: constant mismatches placed exactly
(k = m - 1, m, m + 1 for budget m, one per slice of the constant positions, every replacement kind), budgets split between
the flanks and the variable region (Ns included), a clean construct at every window on both strands, and lower-case reads.
Libraries are random (`distinct_pool`), dense (clusters of barcodes 1 to 3 substitutions apart: ties, ambiguity, seed buckets
with several rows) or IUPAC (several expanded entries per pool index).  The per-read index and info and the counts must
equal the reference's, and the kernel note must name the route the guard of `launch_single` implies.
"""
import itertools
from math import comb

import numpy as np
import pytest

from util import adversarial_reads, distinct_pool, fastq, fill_template, random_seq, revcomp

# flanks: the baseline's 12 bases, then bases with no symmetry to speak of, so that the reverse strand really differs
LEFT = "CAGCTACGTACG" + "AGAACCTTTTAATAAATCCACGTGTACGGAACATGT"
RIGHT = "CCAGCTCGATCG" + "GGCCAATCTCGTTACCTTCCACAATCTCCTGCCTCC"

# (left flank, key length, right flank)
SHAPES = [
    (12, 20, 12),                                  # the baseline, 44 bases
    (14, 20, 10), (5, 20, 17), (1, 20, 15),        # asymmetric flanks: the strands' regions start apart
    (0, 20, 16), (16, 20, 0),                      # one-sided templates
    (12, 1, 12), (10, 2, 14), (12, 3, 9),          # keys so short that a budget leaves no usable seed
    (12, 8, 12), (12, 19, 12), (11, 21, 13),
    (12, 31, 12), (12, 32, 12),                    # the joint table's last key length; the full key mask
    (24, 20, 12),                                  # the forward region crosses the first word of the window
    (6, 20, 7),                                    # 33 bases: two words per window
    (16, 32, 16), (20, 25, 20),                    # 64 and 65 bases: two and three words
    (32, 32, 32), (40, 17, 40),                    # 96 and 97 bases: three and four words
    (40, 30, 40), (48, 32, 48),                    # 110 and 128 bases
    (2, 20, 2), (1, 20, 2),                        # 4 and 3 constant positions: budget 0's limit and one below
    (3, 20, 5), (3, 20, 4),                        # 8 and 7: budget 1
    (6, 20, 6), (5, 20, 6),                        # 12 and 11: budget 2
    (7, 20, 8),                                    # 15: one below budget 3's (the one-sided shapes have 16)
]
MAX_UNIFORM_LEN = 320
LONG_LEN = 161   # one tile per bulk copy


def template_of(shape):
    left, k, right = shape
    return LEFT[:left] + "-" * k + RIGHT[:right]


def shape_id(shape):
    return "%d+%d+%d" % shape


def nconst_of(shape):
    return shape[0] + shape[2]


def takes_uniform(shape, mm, max_len):
    """The guard of launch_single (runners_single.cu) for the uniform-length kernel."""
    T, nconst = sum(shape), nconst_of(shape)
    mmc = max(0, min(mm, nconst))   # TemplateSpec::scan_spec clamps the budget to the constant positions
    return max_len - T + 1 >= 1 and mmc <= 3 and nconst >= 4 * (mmc + 1) and T <= 128 and max_len <= MAX_UNIFORM_LEN


def lib_kinds(shape):
    return ["distinct", "dense", "iupac"] if shape[1] >= 4 else ["distinct"]


def cases_of(si, shape):
    """(strand, mm, use_first, read_len, library kind, pool size) of one shape.  At strand 2 every budget, both modes, every
    read length and every library kind appear; strands 0 and 1 once each."""
    T = sum(shape)
    lens = [T, T + 30, T + 31, T + 32, LONG_LEN]
    kinds = lib_kinds(shape)
    out = []
    for k in range(5):
        out.append((2, (k + si) % 4, (k + si // 2) % 2 == 0, lens[k], kinds[(k + si) % len(kinds)], 1500 if (k + si) % 2 else 300))
    out.append((0, si % 4, si % 2 == 0, lens[(si + 1) % 5], kinds[(si + 1) % len(kinds)], 600))
    out.append((1, (si + 2) % 4, si % 2 == 1, lens[(si + 3) % 5], kinds[(si + 2) % len(kinds)], 1200))
    return out


MATRIX = [(si, ci) for si in range(len(SHAPES)) for ci in range(7)]


# ---- libraries ---------------------------------------------------------------------------------------------------------

IUPAC = {"R": "AG", "Y": "CT", "S": "CG", "W": "AT", "K": "GT", "M": "AC", "B": "CGT", "D": "AGT", "H": "ACT", "V": "ACG", "N": "ACGT"}


def expansions(s):
    return ["".join(p) for p in itertools.product(*[IUPAC.get(c, c) for c in s])]


def substitute(rng, s, positions):
    out = list(s)
    for p in positions:
        out[p] = "ACGT".replace(out[p], "")[int(rng.integers(0, 3))]
    return "".join(out)


def dense_library(rng, n, L):
    """Clusters around a centre: members 1, 1, 2 and 3 substitutions away (the centre itself in half of them).  The read
    sources are the centres, the members and points between two members, so reads land on exact ties, on a unique best
    found after a tie, and on ambiguity that first and best mode settle differently; the members share most seeds, so
    the seed buckets hold several rows."""
    pool, seen, sources = [], set(), []
    while len(pool) < n:
        centre = random_seq(rng, L)
        members = [substitute(rng, centre, rng.choice(L, d, replace=False)) for d in (1, 1, 2, 3)]
        if rng.random() < 0.5:
            members.append(centre)
        for m in members:
            if m not in seen and len(pool) < n:
                seen.add(m)
                pool.append(m)
        sources.append(centre)
        sources.extend(members)
        for a, b in itertools.combinations(members[:3], 2):
            sources.append("".join(x if (i % 2) else y for i, (x, y) in enumerate(zip(a, b))))
    return pool, sources


def iupac_library(rng, n, L):
    """A third of the entries carry one or two ambiguity codes; no two entries share an expansion."""
    pool, seen, sources = [], set(), []
    codes = "".join(IUPAC)
    while len(pool) < n:
        s = list(random_seq(rng, L))
        if rng.random() < 0.35:
            for p in rng.choice(L, int(rng.integers(1, 3)), replace=False):
                s[p] = codes[int(rng.integers(0, len(codes)))]
        s = "".join(s)
        exp = expansions(s)
        if any(e in seen for e in exp):
            continue
        seen.update(exp)
        pool.append(s)
        sources.extend(exp[int(i)] for i in rng.choice(len(exp), min(2, len(exp)), replace=False))
    return pool, sources


def library(rng, kind, n, L):
    if kind == "dense":
        return dense_library(rng, n, L)
    if kind == "iupac":
        return iupac_library(rng, n, L)
    n = min(n, 3 * 4 ** L // 4)   # keys of 1 to 3 bases: leave some keys out of the pool
    pool = distinct_pool(rng, n, L)
    return pool, pool


# ---- reads -------------------------------------------------------------------------------------------------------------

def place(rng, construct, read_len, offset=None):
    if offset is None:
        offset = int(rng.integers(0, read_len - len(construct) + 1))
    return (random_seq(rng, offset) + construct + random_seq(rng, read_len))[:read_len]


def replace_at(s, positions, kinds):
    """kind 0..2: one of the three other bases; 3: N."""
    out = list(s)
    for p, k in zip(positions, kinds):
        out[p] = "N" if k == 3 else "ACGT".replace(out[p].upper(), "")[k]
    return "".join(out)


def constant_position_sets(rng, cpos, k, budget_sets=600):
    """Every k-set of constant positions when there are few; otherwise random sets with one position in each of k slices
    of the constant positions, plus sets that hold the first and the last constant position of each flank."""
    if k == 0:
        return [()]
    if comb(len(cpos), k) <= budget_sets:
        return list(itertools.combinations(cpos, k))
    slices = np.array_split(np.array(cpos), k)
    sets = [tuple(int(rng.choice(s)) for s in slices) for _ in range(budget_sets)]
    ends = [cpos[0], cpos[-1]] + [cpos[i] for i in range(1, len(cpos)) if cpos[i] != cpos[i - 1] + 1] + \
           [cpos[i] for i in range(len(cpos) - 1) if cpos[i + 1] != cpos[i] + 1]
    for e in ends:
        for _ in range(8):
            others = [p for p in cpos if p != e]
            sets.append((e,) + tuple(int(p) for p in rng.choice(others, k - 1, replace=False)))
    return sets


def shape_reads(rng, shape, mm, read_len, sources, n_background=2000):
    """Every read has exactly read_len bases."""
    template = template_of(shape)
    T, L = len(template), shape[1]
    cpos = [j for j, c in enumerate(template) if c != "-"]
    vstart = shape[0]
    reads = []

    def orient(c):
        return revcomp(c) if rng.random() < 0.5 else c

    def clean():
        return fill_template(template, sources[int(rng.integers(0, len(sources)))])

    # background: noise, constructs on both strands, two constructs in one read, constructs at the read's edges, junk
    bg = adversarial_reads(rng, n_background, template, [sources], strand="both", read_len=read_len, sub_rate=0.02,
                           n_rate=0.004, lower_rate=0.01, double_frac=0.2, short_frac=0.02, edge_frac=0.3)
    reads += [(r + random_seq(rng, read_len))[:read_len] for r in bg]

    # exactly k constant mismatches, k = mm - 1, mm, mm + 1; every replacement kind
    for k in range(max(0, mm - 1), min(mm + 1, len(cpos)) + 1):
        for t, ps in enumerate(constant_position_sets(rng, cpos, k)):
            kinds = [(t + j) % 4 for j in range(k)]
            reads.append(place(rng, orient(replace_at(clean(), ps, kinds)), read_len))

    # budget split: c constant and v variable substitutions, c + v in {mm, mm + 1}; v as bases, as Ns, as Ns inside one seed
    cap = min(mm, L)
    seed_len = max(1, L // (cap + 1)) if cap else L
    for total in (mm, mm + 1):
        for c in range(0, min(total, len(cpos)) + 1):
            v = total - c
            if v > L:
                continue
            for rep in range(12):
                s = clean()
                s = replace_at(s, rng.choice(cpos, c, replace=False), rng.integers(0, 3, size=c))
                vpos = vstart + rng.choice(L, v, replace=False)
                if rep % 3 == 0:
                    s = replace_at(s, vpos, rng.integers(0, 3, size=v))
                elif rep % 3 == 1:
                    s = replace_at(s, vpos, [3] * v)
                elif v <= seed_len:
                    first = int(rng.integers(0, seed_len - v + 1))
                    s = replace_at(s, [vstart + first + j for j in range(v)], [3] * v)
                reads.append(place(rng, orient(s), read_len))

    # one clean construct at every window, on both strands
    for off in range(read_len - T + 1):
        reads.append(place(rng, clean(), read_len, off))
        reads.append(place(rng, revcomp(clean()), read_len, off))

    # lower case in a share of the reads
    for i in rng.choice(len(reads), len(reads) // 10, replace=False):
        r = reads[i]
        mask = rng.random(len(r)) < 0.4
        reads[i] = "".join(ch.lower() if m else ch for ch, m in zip(r, mask))

    order = rng.permutation(len(reads))
    reads = [reads[i] for i in order]
    assert {len(r) for r in reads} == {read_len}
    return reads


# ---- running and comparing ---------------------------------------------------------------------------------------------

def check_against_reference(kref, reads, template, strand, pool, mm, use_first, route):
    """route: 'uniform', 'trimmed' or 'general' (the specialised kernel without the filter + verify route)."""
    from screencounter_b200 import rcpp
    data = fastq(reads)
    want_index, want_info = kref.trace_single(data, template, strand, pool, mm, use_first)
    counts, total, (index, info) = rcpp.count_single_barcodes(data, template, strand, pool, mm, use_first, 4, trace=True)
    note = rcpp.timing()["kernel"]
    if route == "uniform":
        assert "uniform-length filter+verify" in note, note
    elif route == "trimmed":
        assert "trimmed reads, filter+verify" in note, note
    else:
        assert note.startswith("specialised (NVRTC)") and "filter+verify" not in note, note
    assert total == len(reads)
    got = index[:, 0] if index.ndim > 1 else index
    bad = np.flatnonzero((got != want_index) | (info != want_info).any(axis=1))
    assert bad.size == 0, "%d reads differ, first %d: %r got %d %r want %d %r" % (
        bad.size, bad[0], reads[bad[0]], got[bad[0]], info[bad[0]].tolist(), want_index[bad[0]], want_info[bad[0]].tolist())
    assert np.array_equal(counts, np.bincount(want_index[want_index >= 0], minlength=len(pool)))
    return want_index


def case_inputs(si, ci):
    shape = SHAPES[si]
    strand, mm, use_first, read_len, kind, npool = cases_of(si, shape)[ci]
    rng = np.random.default_rng(1000 * si + ci)
    pool, sources = library(rng, kind, npool, shape[1])
    return shape, strand, mm, use_first, read_len, kind, pool, sources, rng


@pytest.mark.gpu
@pytest.mark.parametrize("si,ci", MATRIX, ids=["%s-%d" % (shape_id(SHAPES[si]), ci) for si, ci in MATRIX])
def test_shape_matrix_against_reference(kref, si, ci):
    shape, strand, mm, use_first, read_len, kind, pool, sources, rng = case_inputs(si, ci)
    reads = shape_reads(rng, shape, mm, read_len, sources)
    route = "uniform" if takes_uniform(shape, mm, read_len) else "general"
    want = check_against_reference(kref, reads, template_of(shape), strand, pool, mm, use_first, route)
    assert (want >= 0).any()


VARIANTS = [("SCG_SPEC_NO_JOINT", "1"), ("SCG_SPEC_NO_IBUCKETS", "1"), ("SCG_SPEC_HIST_MAX", "0")]


@pytest.mark.gpu
@pytest.mark.parametrize("si", range(len(SHAPES)), ids=[shape_id(s) for s in SHAPES])
def test_shape_other_routes_against_reference(kref, monkeypatch, si):
    """One read set of LONG_LEN bases per shape through the general specialised kernel (SCG_SPEC_NO_UNIFORM), one of the
    table variants of the uniform kernel, and the trimmed-read route at two spreads of lengths."""
    shape = SHAPES[si]
    T = sum(shape)
    kind = lib_kinds(shape)[si % len(lib_kinds(shape))]
    mm, use_first = si % 4, si % 2 == 0
    rng = np.random.default_rng(50000 + si)
    pool, sources = library(rng, kind, 800 if si % 2 else 1400, shape[1])
    template = template_of(shape)
    reads = shape_reads(rng, shape, mm, LONG_LEN, sources, n_background=1500)
    uniform = takes_uniform(shape, mm, LONG_LEN)

    with monkeypatch.context() as mp:
        mp.setenv("SCG_SPEC_NO_UNIFORM", "1")
        check_against_reference(kref, reads, template, 2, pool, mm, use_first, "general")
    name, value = VARIANTS[si % len(VARIANTS)]
    with monkeypatch.context() as mp:
        mp.setenv(name, value)
        check_against_reference(kref, reads, template, 2, pool, mm, use_first, "uniform" if uniform else "general")

    # trimmed reads: T .. T + 31 bases (one window block), then T .. LONG_LEN; a few shorter than the template
    for longest in (T + 31, LONG_LEN):
        lens = rng.integers(T, longest + 1, size=len(reads))
        lens[rng.choice(len(reads), len(reads) // 50, replace=False)] = rng.integers(0, T, size=len(reads) // 50)
        lens[0] = longest
        ragged = [r[:n] for r, n in zip(reads, lens)]
        route = "trimmed" if takes_uniform(shape, mm, longest) else "general"
        check_against_reference(kref, ragged, template, 2, pool, mm, use_first, route)


# ---- no GPU needed ------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("si", range(len(SHAPES)), ids=[shape_id(s) for s in SHAPES])
def test_shape_uniform_variants_compile(si):
    """Every uniform-length variant the matrix runs, through NVRTC: 0 = compiled and loaded, 2 = compiled, nothing to load
    it on.  scg_jit_selftest_uniform does not apply the route's guard, so only what the route takes is built."""
    import ctypes as C
    from screencounter_b200._lib import lib
    shape = SHAPES[si]
    template = template_of(shape)
    assert template != revcomp(template) and LEFT[:shape[0]] != revcomp(RIGHT[:shape[2]])
    builds = {(strand, mm, read_len) for strand, mm, _, read_len, _, _ in cases_of(si, shape) if takes_uniform(shape, mm, read_len)}
    if takes_uniform(shape, si % 4, LONG_LEN):
        builds.add((2, si % 4, LONG_LEN))
    if all(not takes_uniform(shape, mm, LONG_LEN) for mm in range(4)):
        assert not builds
        pytest.skip("the route takes no variant of %s" % shape_id(shape))
    buf = C.create_string_buffer(16384)
    for strand, mm, read_len in sorted(builds):
        rc = lib().scg_jit_selftest_uniform(template.encode(), strand, mm, read_len, buf, C.c_size_t(16384))
        assert rc in (0, 2), (strand, mm, read_len, buf.value.decode())


def test_guard_limits_are_in_the_matrix():
    """The matrix holds, for every budget, a shape at the route's fewest constant positions and one below it."""
    for mm in range(4):
        at = [s for s in SHAPES if nconst_of(s) == 4 * (mm + 1)]
        below = [s for s in SHAPES if nconst_of(s) == 4 * (mm + 1) - 1]
        assert at and below, mm
        assert all(takes_uniform(s, mm, LONG_LEN) for s in at)
        assert not any(takes_uniform(s, mm, LONG_LEN) for s in below)
    assert {sum(s) for s in SHAPES} >= {33, 64, 65, 96, 97, 128}
    assert {s[1] for s in SHAPES} >= {1, 2, 3, 8, 19, 21, 31, 32}


@pytest.mark.parametrize("kind", ["dense", "iupac"])
def test_duplicate_pool_raises_the_reference_error(kref, kind):
    """A pool with two entries that expand to one sequence is refused with the reference's text, before any device work."""
    from screencounter_b200 import rcpp
    rng = np.random.default_rng(9)
    shape = (14, 20, 10)
    pool, _ = library(rng, kind, 300, shape[1])
    ambiguous = next(i for i, s in enumerate(pool) if len(expansions(s)) > 1) if kind == "iupac" else 17
    pool = pool + [expansions(pool[ambiguous])[-1]]
    args = (fastq(["ACGT" * 20]), template_of(shape), 2, pool, 1, True)
    with pytest.raises(Exception) as ref_err:
        kref.count_single(*args)
    assert "duplicate sequences detected" in str(ref_err.value)
    with pytest.raises(Exception) as err:
        rcpp.count_single_barcodes(*args, 1)
    assert str(err.value) == str(ref_err.value)
