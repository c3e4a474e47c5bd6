"""The seven Rcpp-exported entry points of screenCounter, same names and argument order
(reference R/RcppExports.R:4-30, src/RcppExports.cpp:13-150), on top of the C ABI.

`path` arguments accept a file path (str) or in-memory FASTQ text (bytes).  Return values are
Python lists shaped like the R lists the reference returns (SURVEY.md 8.2 row b), with numpy
arrays for the integer vectors.  Indices are 0-based exactly where the C++ glue is 0-based
(the R wrappers add 1); `match_barcodes` returns 1-based indices and None for NA like the glue.
"""
import ctypes as C
import os
import threading

import numpy as np

from ._lib import lib, ScgSource


class ScreenCounterError(RuntimeError):
    """An error raised by the engine; the text is kaori's own wherever the reference has one."""


_local = threading.local()


def default_device():
    """The device of a context asked for without one: SCG_DEVICE, else LOCAL_RANK, else 0."""
    return int(os.environ.get("SCG_DEVICE", os.environ.get("LOCAL_RANK", "0")))


def context(device=None):
    """Per-thread, per-device context (CUDA is initialised lazily by the first counting call)."""
    if device is None:
        device = default_device()
    cache = getattr(_local, "ctx", None)
    if cache is None:
        cache = _local.ctx = {}
    if isinstance(device, (list, tuple)):
        # one context over several devices (scg_ctx_create_multi): a file is cut over them, files of a many-files call are dealt to them
        device = tuple(int(d) for d in device)
    if device not in cache:
        h = C.c_void_p()
        if isinstance(device, tuple):
            ids = (C.c_int * len(device))(*device)
            status = lib().scg_ctx_create_multi(C.byref(h), ids, len(device))
        else:
            status = lib().scg_ctx_create(C.byref(h), int(device))
        if status != 0:
            raise ScreenCounterError(lib().scg_last_error(None).decode("latin-1"))
        cache[device] = h
    return cache[device]


def _check(ctx, status):
    if status != 0:
        raise ScreenCounterError(lib().scg_last_error(ctx).decode("latin-1"))


class PinnedText:
    """FASTQ text in page-locked host memory (scg_host_alloc): the engine copies it to the device by DMA
    straight from this buffer.  `array` is a writable uint8 view; fill `array[:n]` and pass the object as
    the `path` argument of a counting function after setting `size = n`."""

    def __init__(self, capacity, device=None):
        self.ctx = context(device)
        self.capacity = int(capacity)
        self.size = self.capacity
        p = C.c_void_p()
        _check(self.ctx, lib().scg_host_alloc(self.ctx, C.c_size_t(max(self.capacity, 1)), C.byref(p)))
        self.ptr = p
        self.array = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(max(self.capacity, 1),))[: self.capacity]

    @classmethod
    def from_bytes(cls, data, device=None):
        self = cls(len(data), device)
        self.array[:] = np.frombuffer(data, dtype=np.uint8)
        return self

    def free(self):
        if self.ptr is not None:
            self.array = None
            lib().scg_host_free(self.ctx, self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class _Src:
    """Keeps the bytes alive for the duration of the call."""

    def __init__(self, fastq):
        if isinstance(fastq, PinnedText):
            self.keep = fastq
            self.struct = ScgSource(None, fastq.ptr, fastq.size)
        elif isinstance(fastq, np.ndarray):
            self.keep = np.ascontiguousarray(fastq, dtype=np.uint8)
            self.struct = ScgSource(None, self.keep.ctypes.data_as(C.c_void_p), self.keep.size)
        elif isinstance(fastq, (bytes, bytearray, memoryview)):
            self.keep = fastq if isinstance(fastq, bytes) else bytes(fastq)
            # a pointer INTO the bytes object: no copy of what can be gigabytes of text
            self.struct = ScgSource(None, C.cast(C.c_char_p(self.keep), C.c_void_p), len(self.keep))
        else:
            self.keep = os.fsencode(fastq)
            self.struct = ScgSource(self.keep, None, 0)

    def ref(self):
        return C.byref(self.struct)


_STRS_CACHE = {}


def _strs(seqs):
    """ctypes char*[] for a list of sequences.  Large pools (a guide library handed to one call per
    FASTQ file) are marshalled once and found again by content hash."""
    key = None
    if len(seqs) >= 1024:
        try:
            key = (len(seqs), hash(tuple(seqs)))
        except TypeError:
            key = None
        hit = _STRS_CACHE.get(key) if key is not None else None
        if hit is not None and hit[2] == seqs[0] and hit[3] == seqs[-1]:
            return hit[0], hit[1]
    enc = [s.encode("latin-1") if isinstance(s, str) else bytes(s) for s in seqs]
    arr = (C.c_char_p * max(len(enc), 1))(*enc)
    if key is not None:
        if len(_STRS_CACHE) >= 8:
            _STRS_CACHE.pop(next(iter(_STRS_CACHE)))
        _STRS_CACHE[key] = (arr, enc, seqs[0], seqs[-1])
    return arr, enc


def _ip(a):
    return a.ctypes.data_as(C.c_void_p)


def _table(handle, kind):
    L = lib()
    n = L.scg_result_rows(handle)
    w = L.scg_result_width(handle)
    freq = np.empty(n, dtype=np.int32)
    if kind == "combo":
        keys = np.empty((n, w), dtype=np.int32)
        L.scg_result_copy_table(handle, _ip(keys), None, _ip(freq))
        return keys, freq
    if kind == "random_array":
        # millions of barcodes: one fixed-width bytes array (dtype S<w>) instead of a Python string per barcode
        arr = np.empty(n, dtype="S%d" % max(w, 1))
        L.scg_result_copy_table(handle, None, _ip(arr), _ip(freq))
        return arr, freq
    buf = C.create_string_buffer(max(n * w, 1))
    L.scg_result_copy_table(handle, None, buf, _ip(freq))
    raw = buf.raw[: n * w]
    if n and w and b"\0" not in raw:
        try:   # decode in one vectorised step
            return np.frombuffer(raw, dtype="S%d" % w).astype("U%d" % w).tolist(), freq
        except UnicodeDecodeError:
            pass
    return [raw[i * w:(i + 1) * w].decode("latin-1") for i in range(n)], freq


def _trace(handle):
    L = lib()
    n = L.scg_result_reads(handle)
    w = max(L.scg_result_trace_width(handle), 1)
    index = np.zeros((n, w), dtype=np.int32)
    info = np.zeros(n, dtype=np.uint32)
    L.scg_result_copy_trace(handle, _ip(index), _ip(info))
    return index, info


def decode_info(info):
    """(position, reverse, mismatches, variable_mismatches) columns of a single-barcode trace, -1/0 where not found."""
    info = np.asarray(info, dtype=np.uint32)
    found = (info >> 31) & 1
    out = np.zeros((len(info), 4), dtype=np.int32)
    out[:, 0] = np.where(found, info & 0xFFFFF, -1)
    out[:, 1] = np.where(found, (info >> 30) & 1, 0)
    out[:, 2] = np.where(found, (info >> 20) & 31, -1)
    out[:, 3] = np.where(found, (info >> 25) & 31, -1)
    return out


# ---------------------------------------------------------------------------------------------
def count_single_barcodes(path, constant, strand, pool, mismatches, use_first, nthreads, trace=False, device=None):
    """reference: src/count_single_barcodes.cpp:29-50 -> list(counts, total)."""
    ctx = context(device)
    src = _Src(path)
    arr, keep = _strs(pool)
    counts = np.zeros(len(pool), dtype=np.int32)
    total = C.c_int32()
    handle = C.c_void_p()
    _check(ctx, lib().scg_count_single(ctx, src.ref(), constant.encode("latin-1"), int(strand), arr, len(pool), int(mismatches),
                                       int(bool(use_first)), int(nthreads), _ip(counts), C.byref(total),
                                       C.byref(handle) if trace else None))
    out = [counts, total.value]
    if trace:
        index, info = _trace(handle)
        lib().scg_result_free(handle)
        out.append((index[:, 0], decode_info(info)))
    return out


def count_single_barcodes_paired(path1, path2, constant, strand, pool, mismatches, use_first, nthreads, trace=False, device=None):
    """kaori's SingleBarcodePairedEnd handler (no R entry point in screenCounter): list(counts, total[, per-pair index])."""
    ctx = context(device)
    s1, s2 = _Src(path1), _Src(path2)
    arr, keep = _strs(pool)
    counts = np.zeros(len(pool), dtype=np.int32)
    total = C.c_int32()
    handle = C.c_void_p()
    _check(ctx, lib().scg_count_single_paired(ctx, s1.ref(), s2.ref(), constant.encode("latin-1"), int(strand), arr, len(pool),
                                              int(mismatches), int(bool(use_first)), int(nthreads), _ip(counts), C.byref(total),
                                              C.byref(handle) if trace else None))
    out = [counts, total.value]
    if trace:
        out.append(_trace(handle)[0][:, 0])
        lib().scg_result_free(handle)
    return out


def match_barcodes(sequences, choices, substitutions, reverse, device=None):
    """reference: src/match_barcodes.cpp:7-37 -> list(index (1-based, None = NA), mismatches (None = NA))."""
    ctx = context(device)
    a, k1 = _strs(sequences)
    c, k2 = _strs(choices)
    index = np.zeros(len(sequences), dtype=np.int32)
    mm = np.zeros(len(sequences), dtype=np.int32)
    _check(ctx, lib().scg_match_barcodes(ctx, a, len(sequences), c, len(choices), int(substitutions), int(bool(reverse)),
                                         _ip(index), _ip(mm)))
    return [[int(i) + 1 if i >= 0 else None for i in index], [int(m) if i >= 0 else None for i, m in zip(index, mm)]]


def search_segmented(sequences, caps, choices, len1, len2, max1, max2, device=None):
    """The two-segment search behind countDualBarcodes on its own (tests): per-query caps, 0-based index or -1."""
    ctx = context(device)
    qs, kq = _strs(sequences)
    cs, kc = _strs(choices)
    caps = np.ascontiguousarray(caps, dtype=np.int32).reshape(-1, 2)
    index = np.zeros(len(sequences), dtype=np.int32)
    mm = np.zeros(len(sequences), dtype=np.int32)
    _check(ctx, lib().scg_search_segmented(ctx, qs, len(sequences), _ip(caps), cs, len(choices), int(len1), int(len2), int(max1),
                                           int(max2), _ip(index), _ip(mm)))
    return index, mm


def timing(device=None):
    import json
    return json.loads(lib().scg_timing_json(context(device)).decode())


def kernel_launches(device=None):
    return int(lib().scg_kernel_launches(context(device)))


def count_random_barcodes(path, constant, strand, mismatches, use_first, nthreads, device=None, as_array=True):
    """reference: src/count_random_barcodes.cpp:41-60 -> list(list(sequences, frequencies), total).
    Sequences come back sorted (R sorts them anyway, R/countRandomBarcodes.R:73-74) as ONE numpy bytes array (dtype
    S<length>: the table is copied from the device straight into it); as_array=False gives a list of str instead."""
    ctx = context(device)
    src = _Src(path)
    handle = C.c_void_p()
    total = C.c_int32()
    _check(ctx, lib().scg_count_random(ctx, src.ref(), constant.encode("latin-1"), int(strand), int(mismatches), int(bool(use_first)),
                                       int(nthreads), C.byref(handle), C.byref(total)))
    seqs, freq = _table(handle, "random_array" if as_array else "random")
    lib().scg_result_free(handle)
    return [[seqs, freq], total.value]


def count_combo_barcodes_single(path, constant, strand, pool, mismatches, use_first, nthreads, trace=False, device=None):
    """reference: src/count_combo_barcodes_single.cpp:40-70 -> list(2 x k matrix (0-based), freq, total)."""
    if len(pool) != 2:
        raise ScreenCounterError("currently expecting only 2 variable regions for single-end combinatorial barcodes")
    ctx = context(device)
    src = _Src(path)
    a1, k1 = _strs(pool[0])
    a2, k2 = _strs(pool[1])
    handle = C.c_void_p()
    total = C.c_int32()
    _check(ctx, lib().scg_count_combo_single(ctx, src.ref(), constant.encode("latin-1"), int(strand), a1, len(pool[0]), a2, len(pool[1]),
                                             int(mismatches), int(bool(use_first)), int(nthreads), int(bool(trace)),
                                             C.byref(handle), C.byref(total)))
    keys, freq = _table(handle, "combo")
    out = [keys.T.copy(), freq, np.array([total.value], dtype=np.int32)]
    if trace:
        out.append(_trace(handle)[0])
    lib().scg_result_free(handle)
    return out


def count_dual_barcodes_single_end(path, constant, pools, strand, mismatches, use_first, diagnostics, nthreads, trace=False, device=None):
    """reference: src/count_dual_barcodes_single_end.cpp:51-88 -> list(counts, total) or
    list(counts, list(2 x k matrix, freq), total) with diagnostics."""
    ctx = context(device)
    src = _Src(path)
    nchoices = len(pools[0]) if len(pools) else 0
    flat = []
    for p in pools:
        if len(p) != nchoices:
            raise ScreenCounterError("all entries of 'barcode_pools' should have the same length")
        flat.extend(p)
    arr, keep = _strs(flat)
    counts = np.zeros(nchoices, dtype=np.int32)
    total = C.c_int32()
    handle = C.c_void_p()
    _check(ctx, lib().scg_count_dual_single_end(ctx, src.ref(), constant.encode("latin-1"), arr, len(pools), nchoices, int(strand),
                                                int(mismatches), int(bool(use_first)), int(bool(diagnostics)), int(nthreads),
                                                int(bool(trace)), _ip(counts), C.byref(total), C.byref(handle)))
    tot = np.array([total.value], dtype=np.int32)
    if diagnostics:
        keys, freq = _table(handle, "combo")
        out = [counts, [keys.T.copy(), freq], tot]
    else:
        out = [counts, tot]
    if trace:
        out.append(_trace(handle)[0][:, 0])
    lib().scg_result_free(handle)
    return out


def count_dual_barcodes(path1, constant1, reverse1, mismatches1, pool1, path2, constant2, reverse2, mismatches2, pool2,
                        randomized, use_first, diagnostics, nthreads, trace=False, device=None):
    """reference: src/count_dual_barcodes.cpp:75-116 -> list(counts, total) or
    list(counts, list(2 x k matrix, freq), total, barcode1_only, barcode2_only) with diagnostics."""
    ctx = context(device)
    s1, s2 = _Src(path1), _Src(path2)
    a1, k1 = _strs(pool1)
    a2, k2 = _strs(pool2)
    counts = np.zeros(len(pool1), dtype=np.int32)
    total = C.c_int32()
    b1 = C.c_int32()
    b2 = C.c_int32()
    handle = C.c_void_p()
    _check(ctx, lib().scg_count_dual(ctx, s1.ref(), constant1.encode("latin-1"), int(bool(reverse1)), int(mismatches1), a1, len(pool1),
                                     s2.ref(), constant2.encode("latin-1"), int(bool(reverse2)), int(mismatches2), a2, len(pool2),
                                     int(bool(randomized)), int(bool(use_first)), int(bool(diagnostics)), int(nthreads), int(bool(trace)),
                                     _ip(counts), C.byref(total), C.byref(handle), C.byref(b1), C.byref(b2)))
    tot = np.array([total.value], dtype=np.int32)
    if diagnostics:
        keys, freq = _table(handle, "combo")
        out = [counts, [keys.T.copy(), freq], tot, np.array([b1.value], dtype=np.int32), np.array([b2.value], dtype=np.int32)]
    else:
        out = [counts, tot]
    if trace:
        out.append(_trace(handle)[0][:, 0])
    lib().scg_result_free(handle)
    return out


def count_combo_barcodes_paired(path1, constant1, reverse1, mismatches1, pool1, path2, constant2, reverse2, mismatches2, pool2,
                                randomized, use_first, nthreads, trace=False, device=None):
    """reference: src/count_combo_barcodes_paired.cpp:55-95 -> list(2 x k matrix, freq, total, barcode1_only, barcode2_only)."""
    ctx = context(device)
    s1, s2 = _Src(path1), _Src(path2)
    a1, k1 = _strs(pool1)
    a2, k2 = _strs(pool2)
    total = C.c_int32()
    b1 = C.c_int32()
    b2 = C.c_int32()
    handle = C.c_void_p()
    _check(ctx, lib().scg_count_combo_paired(ctx, s1.ref(), constant1.encode("latin-1"), int(bool(reverse1)), int(mismatches1), a1, len(pool1),
                                             s2.ref(), constant2.encode("latin-1"), int(bool(reverse2)), int(mismatches2), a2, len(pool2),
                                             int(bool(randomized)), int(bool(use_first)), int(nthreads), int(bool(trace)),
                                             C.byref(handle), C.byref(total), C.byref(b1), C.byref(b2)))
    keys, freq = _table(handle, "combo")
    out = [keys.T.copy(), freq, np.array([total.value], dtype=np.int32), np.array([b1.value], dtype=np.int32),
           np.array([b2.value], dtype=np.int32)]
    if trace:
        index, info = _trace(handle)
        out.append((index, info.astype(np.int32)))
    lib().scg_result_free(handle)
    return out


# ---------------------------------------------------------------------------------------------
# Many files, one call: what the matrixOf* wrappers of the reference assemble in R.
def _sources(files):
    keep = [_Src(f) for f in files]
    arr = (ScgSource * max(len(keep), 1))(*[k.struct for k in keep])
    return arr, keep


def matrix_of_single_barcodes(files, constant, strand, pool, mismatches, use_first, nthreads, device=None):
    """reference: R/countSingleBarcodes.R:112-126 -> (npool x nfiles count matrix, nreads per file)."""
    ctx = context(device)
    srcs, keep = _sources(files)
    arr, keep2 = _strs(pool)
    matrix = np.zeros((len(files), len(pool)), dtype=np.int32)   # row f here = column f of the R matrix
    totals = np.zeros(max(len(files), 1), dtype=np.int32)
    _check(ctx, lib().scg_count_single_many(ctx, srcs, len(files), constant.encode("latin-1"), int(strand), arr, len(pool),
                                            int(mismatches), int(bool(use_first)), int(nthreads), _ip(matrix), _ip(totals)))
    return matrix.T, totals[: len(files)]


def _matrix(handle, nrows):
    ncols = lib().scg_result_columns(handle)
    m = np.zeros((ncols, nrows), dtype=np.int32)
    if lib().scg_result_copy_matrix(handle, _ip(m)) != 0:
        raise ScreenCounterError("could not read the count matrix back")
    return m.T


def matrix_of_combo_barcodes(files, constant, strand, pool, mismatches, use_first, nthreads, device=None):
    """countComboBarcodes per file + combineComboCounts (reference R/combineComboCounts.R:31-57) ->
    (2 x k matrix of the combinations seen in any file (0-based, sorted), k x nfiles counts, nreads per file)."""
    if len(pool) != 2:
        raise ScreenCounterError("currently expecting only 2 variable regions for single-end combinatorial barcodes")
    ctx = context(device)
    srcs, keep = _sources(files)
    a1, k1 = _strs(pool[0])
    a2, k2 = _strs(pool[1])
    handle = C.c_void_p()
    totals = np.zeros(max(len(files), 1), dtype=np.int32)
    _check(ctx, lib().scg_count_combo_many(ctx, srcs, len(files), constant.encode("latin-1"), int(strand), a1, len(pool[0]), a2, len(pool[1]),
                                           int(mismatches), int(bool(use_first)), int(nthreads), C.byref(handle), _ip(totals)))
    keys, freq = _table(handle, "combo")
    counts = _matrix(handle, len(freq))
    lib().scg_result_free(handle)
    return keys.T.copy(), counts, totals[: len(files)]


def matrix_of_random_barcodes(files, constant, strand, mismatches, use_first, nthreads, device=None, as_array=True):
    """reference: R/countRandomBarcodes.R:84-105 -> (sorted union of the files' barcodes, k x nfiles counts, nreads per file)."""
    ctx = context(device)
    srcs, keep = _sources(files)
    handle = C.c_void_p()
    totals = np.zeros(max(len(files), 1), dtype=np.int32)
    _check(ctx, lib().scg_count_random_many(ctx, srcs, len(files), constant.encode("latin-1"), int(strand), int(mismatches),
                                            int(bool(use_first)), int(nthreads), C.byref(handle), _ip(totals)))
    seqs, freq = _table(handle, "random_array" if as_array else "random")
    counts = _matrix(handle, len(freq))
    lib().scg_result_free(handle)
    return seqs, counts, totals[: len(files)]


def bgzf_compress(text, level=6, block_text=0, nthreads=None):
    """FASTQ text (bytes / uint8 array) -> block-gzip image (numpy uint8), what bgzip writes; host threads + zlib."""
    arr = np.frombuffer(text, dtype=np.uint8) if isinstance(text, (bytes, bytearray, memoryview)) else np.ascontiguousarray(text, dtype=np.uint8)
    nthreads = nthreads or len(os.sched_getaffinity(0)) or 1
    used = C.c_size_t()
    if lib().scg_bgzf_compress(_ip(arr), arr.size, int(level), int(block_text), int(nthreads), None, 0, C.byref(used)) != 0:
        raise ScreenCounterError(lib().scg_last_error(None).decode("latin-1"))
    out = np.empty(used.value, dtype=np.uint8)
    if lib().scg_bgzf_compress(_ip(arr), arr.size, int(level), int(block_text), int(nthreads), _ip(out), out.size, C.byref(used)) != 0:
        raise ScreenCounterError(lib().scg_last_error(None).decode("latin-1"))
    return out[: used.value]


def bgzf_inflate(image, device=None):
    """The device inflater on its own: block-gzip image -> (text as numpy uint8, milliseconds of the kernels)."""
    ctx = context(device)
    arr = np.frombuffer(image, dtype=np.uint8) if isinstance(image, (bytes, bytearray, memoryview)) else np.ascontiguousarray(image, dtype=np.uint8)
    size = C.c_size_t()
    ms = C.c_double()
    _check(ctx, lib().scg_bgzf_inflate(ctx, _ip(arr), arr.size, None, 0, C.byref(size), None))
    out = np.empty(max(size.value, 1), dtype=np.uint8)
    _check(ctx, lib().scg_bgzf_inflate(ctx, _ip(arr), arr.size, _ip(out), out.size, C.byref(size), C.byref(ms)))
    return out[: size.value], ms.value


def host_pack_roundtrip(fastq, nthreads=1):
    """Host-only: parse + pack + unpack a FASTQ; returns the reads as the packed layout sees them
    (upper-case ACGT, N for anything else).  Needs no device."""
    src = _Src(fastq)
    nr = C.c_longlong()
    nb = C.c_longlong()
    if lib().scg_host_pack_roundtrip(src.ref(), int(nthreads), None, None, C.byref(nr), C.byref(nb)) != 0:
        raise ScreenCounterError(lib().scg_last_error(None).decode("latin-1"))
    bases = C.create_string_buffer(max(nb.value, 1))
    offsets = np.zeros(nr.value + 1, dtype=np.int64)
    src = _Src(fastq)
    if lib().scg_host_pack_roundtrip(src.ref(), int(nthreads), bases, _ip(offsets), C.byref(nr), C.byref(nb)) != 0:
        raise ScreenCounterError(lib().scg_last_error(None).decode("latin-1"))
    raw = bases.raw
    return [raw[offsets[i]:offsets[i + 1]].decode("latin-1") for i in range(nr.value)]
