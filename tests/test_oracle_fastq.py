"""FASTQ grammar: the C restatement's parser against the reference's FastqReader."""
import gzip
import os

import pytest

from fastq_cases import GOOD, BAD


@pytest.mark.parametrize("name", sorted(GOOD))
def test_good(compiled_reference, port, name):
    data = GOOD[name]
    assert compiled_reference.parse(data) == port.parse(data)


def test_expected_shapes(kref):
    assert kref.parse(GOOD["multiline_seq"]) == ["ACGTTT", "A"]
    assert kref.parse(GOOD["crlf"]) == ["ACGT\r", "GG\r"]
    assert kref.parse(GOOD["empty_file"]) == []
    assert kref.parse(GOOD["empty_seq"]) == ["", "AC"]


@pytest.mark.parametrize("name", sorted(BAD))
def test_bad(kref, port, name):
    data, msg = BAD[name]
    for e in (kref, port):
        with pytest.raises(Exception) as err:
            e.parse(data)
        assert str(err.value) == msg


def test_files_raw_and_gz(kref, port, tmp_path):
    data = GOOD["plain"] * 500
    raw = tmp_path / "x.fastq"
    raw.write_bytes(data)
    gz = tmp_path / "x.fastq.gz"
    with gzip.open(gz, "wb") as f:
        f.write(data)
    expect = kref.parse(data)
    for e in (kref, port):
        assert e.parse(str(raw)) == expect
        assert e.parse(str(gz)) == expect
