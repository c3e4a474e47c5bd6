"""Block-gzip FASTQ (BGZF: bgzip, bcl-convert) read without the host ever inflating it: the members cross PCIe compressed,
the device inflates them (screencounter_b200/csrc/inflate.cu, one warp per member) into the text ring of the device-side
FASTQ reader and checks their CRC-32.  The reference reads such files through zlib on one thread
(inst/include/byteme/GzipFileReader.hpp:39-51, sniffed by SomeFileReader.hpp:25-66); results must be those of the text."""
import gzip
import struct
import zlib

import numpy as np
import pytest

from engines import GpuEngine
from util import fastq, random_seq, dense_pool, adversarial_reads, bgzf
from screencounter_b200 import rcpp

pytestmark = pytest.mark.gpu

TEMPLATE = "ACGTA" + "-" * 6 + "TGCAT"


@pytest.fixture(scope="module")
def gpu():
    return GpuEngine()


def _set(monkeypatch, chunk=None, carry=None, **env):
    for name, value in (("SCG_INGEST_CHUNK", chunk), ("SCG_INGEST_CARRY", carry), *env.items()):
        if value is None:
            monkeypatch.delenv(name, raising=False)
        else:
            monkeypatch.setenv(name, str(value))


def _members(chunks, level=6, strategy=zlib.Z_DEFAULT_STRATEGY):
    """A BGZF image with one member per chunk of `chunks` (util.bgzf with a free choice of member boundaries and strategy)."""
    out = []
    for chunk in list(chunks) + [b""]:
        comp = zlib.compressobj(level, zlib.DEFLATED, -15, 9, strategy)
        raw = comp.compress(chunk) + comp.flush()
        bsize = 12 + 6 + len(raw) + 8
        assert bsize <= 65536
        out.append(b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff" + struct.pack("<H", 6) + b"BC" + struct.pack("<HH", 2, bsize - 1) + raw +
                   struct.pack("<II", zlib.crc32(chunk) & 0xFFFFFFFF, len(chunk)))
    return b"".join(out)


def _texts():
    rng = np.random.default_rng(3)
    reads = [random_seq(rng, int(rng.integers(20, 120))) for _ in range(3000)]
    yield "fastq", fastq(reads)
    yield "zeros", bytes(200000)                                   # one literal, then matches of length 258 at distance 1
    yield "random", rng.integers(0, 256, 150000, dtype=np.uint8).tobytes()   # incompressible: stored blocks
    yield "runs", b"".join(bytes([int(rng.integers(65, 70))]) * int(rng.integers(1, 40)) for _ in range(20000))
    yield "two_symbols", bytes(rng.integers(0, 2, 100000, dtype=np.uint8) + 65)
    yield "text", (b"the quick brown fox jumps over the lazy dog, " * 3000)[:123457]
    yield "skewed", bytes(np.minimum(rng.geometric(0.02, 120000), 255).astype(np.uint8))   # long Huffman codes (> 10 bits)
    yield "one_byte", b"x"
    yield "empty", b""


@pytest.mark.parametrize("name,text", list(_texts()), ids=[n for n, _ in _texts()])
@pytest.mark.parametrize("level,strategy,block", [(6, zlib.Z_DEFAULT_STRATEGY, 65280), (1, zlib.Z_DEFAULT_STRATEGY, 30000), (9, zlib.Z_DEFAULT_STRATEGY, 65280),
                                                  (0, zlib.Z_DEFAULT_STRATEGY, 60000), (6, zlib.Z_FIXED, 7000), (6, zlib.Z_HUFFMAN_ONLY, 50000),
                                                  (6, zlib.Z_RLE, 65280), (4, zlib.Z_FILTERED, 999)])
def test_device_inflate_equals_zlib(name, text, level, strategy, block):
    """The inflate kernel on its own, member sizes from 999 bytes to bgzip's 65280, every block type of RFC 1951: stored
    (level 0, incompressible data), fixed codes (Z_FIXED), dynamic codes with long and short matches, literals only
    (Z_HUFFMAN_ONLY), distance-one runs (Z_RLE)."""
    image = _members([text[k:k + block] for k in range(0, len(text), block)], level, strategy)
    assert gzip.decompress(image) == text
    out, ms = rcpp.bgzf_inflate(image)
    assert out.tobytes() == text


def test_library_compressor_round_trip():
    rng = np.random.default_rng(5)
    text = fastq([random_seq(rng, 75) for _ in range(20000)])
    for level in (1, 6):
        image = rcpp.bgzf_compress(text, level=level)
        assert gzip.decompress(image.tobytes()) == text
        out, ms = rcpp.bgzf_inflate(image)
        assert out.tobytes() == text
    assert gzip.decompress(rcpp.bgzf_compress(b"").tobytes()) == b""


@pytest.mark.parametrize("damage", ["payload", "payload_of_the_last_member", "crc", "isize_short", "isize_long"])
def test_corrupt_members_are_refused(gpu, kref, damage, tmp_path, monkeypatch):
    """A member whose stream is damaged, whose CRC does not match or whose declared size is wrong is an error, on the device
    inflater alone and through the counting call (where the host reader takes over at that chunk and raises it)."""
    rng = np.random.default_rng(6)
    pool = dense_pool(rng, 50, 6)
    reads = adversarial_reads(rng, 6000, TEMPLATE, [pool], strand="both")
    text = fastq(reads)
    image = bytearray(bgzf(text, 20000))
    first_len = struct.unpack("<H", image[16:18])[0] + 1
    second = first_len   # damage the second member
    second_len = struct.unpack("<H", image[second + 16:second + 18])[0] + 1
    if damage == "payload":
        for k in range(40, 60):
            image[second + 18 + k] ^= 0x5A
    elif damage == "payload_of_the_last_member":
        # the last member that holds text, its whole stream turned into noise: the inflater must neither run out of the image
        # nor take long to notice
        at, members = 0, []
        while at < len(image):
            members.append(at)
            at += struct.unpack("<H", image[at + 16:at + 18])[0] + 1
        last = members[-2]
        size = struct.unpack("<H", image[last + 16:last + 18])[0] + 1
        noise = np.random.default_rng(1).integers(0, 256, size - 26, dtype=np.uint8).tobytes()
        image[last + 18:last + size - 8] = noise
    elif damage == "crc":
        image[second + second_len - 8] ^= 1
    else:
        isize = struct.unpack("<I", image[second + second_len - 4:second + second_len])[0]
        image[second + second_len - 4:second + second_len] = struct.pack("<I", isize - 1 if damage == "isize_short" else isize + 1)
    with pytest.raises(rcpp.ScreenCounterError, match="corrupt member"):
        rcpp.bgzf_inflate(bytes(image))
    path = tmp_path / "bad.fastq.gz"
    path.write_bytes(bytes(image))
    _set(monkeypatch)
    with pytest.raises(rcpp.ScreenCounterError, match="corrupt member"):
        gpu.count_single(str(path), TEMPLATE, 2, pool, 1, True, nthreads=3)


@pytest.mark.parametrize("chunk,block", [(None, 65280), (65536, 3000), (70000, 20000), (200000, 65280)])
@pytest.mark.parametrize("source", ["file", "memory", "pinned"])
def test_counting_a_block_gzip_input(gpu, kref, monkeypatch, tmp_path, chunk, block, source):
    """Per-read outcomes on a block-gzip file / image in memory / image in page-locked memory equal the reference's on the text,
    across many chunks of members, and the host never inflates anything."""
    rng = np.random.default_rng(8)
    pool = dense_pool(rng, 50, 6)
    reads = adversarial_reads(rng, 9000, TEMPLATE, [pool], strand="both")
    text = fastq(reads)
    want = kref.trace_single(text, TEMPLATE, 2, pool, 1, False)
    image = bgzf(text, block)
    if source == "file":
        path = tmp_path / "reads.fastq.gz"
        path.write_bytes(image)
        src = str(path)
    elif source == "memory":
        src = image
    else:
        src = rcpp.PinnedText.from_bytes(image)
    _set(monkeypatch, chunk, 4096)
    got = gpu.trace_single(src, TEMPLATE, 2, pool, 1, False)
    t = rcpp.timing()
    assert "inflated on the device" in t["reader"] and "then host" not in t["reader"], t
    assert ("page-locked" in t["reader"]) == (source == "pinned"), t
    assert t["bytes_h2d"] < len(text) / 2, "the text itself must not cross PCIe"
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    # the host route (SCG_BGZF_HOST=1: members inflated by host threads, host parser) gives the same
    _set(monkeypatch, chunk, 4096, SCG_BGZF_HOST="1")
    again = gpu.trace_single(src, TEMPLATE, 2, pool, 1, False)
    assert rcpp.timing()["reader"] == "host"
    assert np.array_equal(again[0], want[0]) and np.array_equal(again[1], want[1])


@pytest.mark.parametrize("final_newline", [True, False])
def test_last_line_without_newline(gpu, kref, monkeypatch, final_newline):
    rng = np.random.default_rng(9)
    pool = dense_pool(rng, 50, 6)
    reads = adversarial_reads(rng, 2000, TEMPLATE, [pool], strand="both", short_frac=0.0)
    text = fastq(reads)
    if not final_newline:
        text = text[:-1]
    want = kref.trace_single(text, TEMPLATE, 2, pool, 1, False)
    _set(monkeypatch, 65536, 4096)
    got = gpu.trace_single(bgzf(text, 5000), TEMPLATE, 2, pool, 1, False)
    assert "inflated on the device" in rcpp.timing()["reader"]
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])


@pytest.mark.parametrize("where", [0, 700, -1])
def test_handover_inside_a_block_gzip_input(gpu, kref, monkeypatch, where):
    """A wrapped record inside a block-gzip input: the device reader stops in front of it and the HOST reader resumes at that
    byte of the text -- which sits in the middle of some member -- by inflating from that member on."""
    rng = np.random.default_rng(10)
    pool = dense_pool(rng, 50, 6)
    reads = adversarial_reads(rng, 1500, TEMPLATE, [pool], strand="both", short_frac=0.0)
    recs = [fastq([r]).decode() for r in reads]
    at = where if where >= 0 else len(recs)
    seq = reads[5]
    recs.insert(at, "@w\n%s\n%s\n+\n%s\n" % (seq[:3], seq[3:], "I" * len(seq)))
    text = "".join(recs).encode()
    want = kref.trace_single(text, TEMPLATE, 2, pool, 1, False)
    for block in (900, 65280):
        _set(monkeypatch, 65536, 2048)
        got = gpu.trace_single(bgzf(text, block), TEMPLATE, 2, pool, 1, False)
        t = rcpp.timing()
        assert "then host from byte %d" % len("".join(recs[:at])) in t["reader"], t
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])


def test_paired_and_random_designs_read_block_gzip(gpu, kref, monkeypatch):
    rng = np.random.default_rng(11)
    # random barcodes, with reads whose barcode has to be rendered from the raw text (lower case): the text of those reads is
    # inflated on the host, member by member, on demand
    template = "ACGTACGT" + "-" * 8 + "TTGCAGCA"
    reads = []
    for _ in range(4000):
        core = "ACGTACGT" + random_seq(rng, 8) + "TTGCAGCA"
        if rng.random() < 0.1:
            core = core.lower()
        reads.append(random_seq(rng, int(rng.integers(0, 9))) + core + random_seq(rng, int(rng.integers(0, 9))))
    text = fastq(reads)
    want = kref.count_random(text, template, 0, 1, True)
    _set(monkeypatch, 65536, 2048)
    got = gpu.count_random(bgzf(text, 4000), template, 0, 1, True)
    assert "inflated on the device" in rcpp.timing()["reader"]
    order = sorted(range(len(want[0])), key=lambda i: want[0][i])
    assert list(got[0]) == [want[0][i] for i in order]
    assert np.array_equal(got[1], np.asarray(want[1])[order]) and got[2] == want[2]
    # paired-end: one mate block-gzip, the other raw text
    t1, t2 = "ACGTA" + "-" * 6 + "TGCAT", "GGCAT" + "-" * 6 + "CCATG"
    p1, p2 = dense_pool(rng, 40, 6), dense_pool(rng, 40, 6)
    r1 = adversarial_reads(rng, 3000, t1, [p1], strand="original", short_frac=0.0)
    r2 = adversarial_reads(rng, 3000, t2, [p2], strand="original", short_frac=0.0)
    f1, f2 = fastq(r1), fastq(r2)
    want = kref.count_combo_paired(f1, t1, False, 1, p1, f2, t2, False, 1, p2, False, True)
    for chunk in (65536, None):
        for g1, g2 in ((bgzf(f1, 7000), f2), (f1, bgzf(f2, 65280)), (bgzf(f1, 3000), bgzf(f2, 11000))):
            _set(monkeypatch, chunk, 4096)
            got = gpu.count_combo_paired(g1, t1, False, 1, p1, g2, t2, False, 1, p2, False, True)
            assert rcpp.timing()["reader"].startswith("device"), rcpp.timing()   # (the line names the mate set up last)
            assert len(got) == len(want)
            for a, b in zip(want, got):
                assert np.array_equal(np.asarray(a), np.asarray(b))
