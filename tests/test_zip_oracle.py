"""Archive side of the path (SURVEY.md §8f 1-3): the oracle's restatement of Zip.Create for BZip2 entries
(oracle/zip_oracle.cpp) against independent readers.  CPU only."""
import io
import struct
import zipfile
import zlib

import numpy as np
import pytest

import datagen
import oracle_lib as orc


def _entries():
    return [("a/text.txt", datagen.text(30_000, 5).tobytes()),
            ("rnd.bin", datagen.random_bytes(5_000, 6).tobytes()),          # not compressible -> stored
            ("empty", b""),                                                    # empty -> stored, CRC 0
            ("dir\\sub\\back.txt", b"hello " * 40),                            # '\' -> '/'
            ("one", b"x"),
            ("sparse.bin", datagen.sparse_binary(40_000, 7).tobytes())]


def test_zip_crc_is_standard_crc32():
    for n in (0, 1, 9, 1000, 70_001):
        d = datagen.random_bytes(n, 60 + n % 7).tobytes()
        assert orc.zip_crc32(d) == zlib.crc32(d)
    assert orc.zip_crc32(b"123456789") == 0xCBF43926


def test_archive_is_read_back_by_python_zipfile():
    ents = _entries()
    arc, methods = orc.zip_create(ents, 9)
    z = zipfile.ZipFile(io.BytesIO(arc))
    assert z.testzip() is None
    infos = z.infolist()
    assert [i.filename for i in infos] == ["a/text.txt", "rnd.bin", "empty", "dir/sub/back.txt", "one", "sparse.bin"]
    for (name, data), zi, m in zip(ents, infos, methods):
        assert z.read(zi) == data
        assert zi.compress_type == m
        assert zi.CRC == zlib.crc32(data)
        # made_by_version 23, needed_extract_version 10 (zip-create.adb:122-131); default_time = 16789 * 65536
        assert zi.create_version == 23 and zi.extract_version == 10
        assert zi.date_time == (2012, 12, 21, 0, 0, 0)
    assert methods == [12, 0, 0, 12, 0, 12]
    # stored exactly when the BZip2 stream is not smaller than the input (zip-compress.adb:468-490)
    for (name, data), zi in zip(ents, infos):
        stream = orc.encode_stream(data, 9, len(data))
        assert (zi.compress_type == 0) == (len(stream) >= len(data))
        if zi.compress_type == 12:
            assert zi.compress_size == len(stream)
            off = zi.header_offset + 30 + len(zi.filename.encode())
            assert arc[off:off + len(stream)] == stream


def test_header_fields_times_and_flags():
    ents = [("ü.txt".encode("utf-8"), b"abc" * 100), ("ro.txt", b"def" * 100)]
    t = [(2020 - 1980) << 25 | 2 << 21 | 29 << 16 | 13 << 11 | 37 << 5 | 21, 16789 * 65536]
    arc, _ = orc.zip_create(ents, 9, dos_times=t, flags=[1, 2])
    z = zipfile.ZipFile(io.BytesIO(arc))
    a, b = z.infolist()
    assert a.filename == "ü.txt" and a.flag_bits == 0x800 and a.date_time == (2020, 2, 29, 13, 37, 42)
    assert b.flag_bits == 0 and b.external_attr == 1 and a.external_attr == 0
    # end record: 2 entries on this disk / in total, no comment (zip-headers.adb:477-494)
    sig, d0, d1, n0, n1, cds, cdo, cl = struct.unpack("<IHHHHIIH", arc[-22:])
    assert (sig, d0, d1, n0, n1, cl) == (0x06054B50, 0, 0, 2, 2, 0)
    assert arc[cdo:cdo + 4] == b"PK\x01\x02" and cdo + cds == len(arc) - 22


def test_levels_write_their_own_block_size():
    data = datagen.text(20_000, 9).tobytes()
    for level in (1, 4, 9):
        arc, methods = orc.zip_create([("t", data)], level)
        assert methods == [12] and arc[31:35] == b"BZh" + str(level).encode()
        assert zipfile.ZipFile(io.BytesIO(arc)).read("t") == data


def test_zip64_end_records_when_65535_entries():
    # "too many entries for Zip_32" (zip-create.adb:680-685): Last_entry >= 65535 promotes the archive
    n = 65_535
    arc, methods = orc.zip_create([("e%05d" % i, b"") for i in range(n)], 9)
    assert set(methods) == {0}
    assert arc[-22:-18] == b"PK\x05\x06" and arc[-42:-38] == b"PK\x06\x07" and arc[-98:-94] == b"PK\x06\x06"
    assert struct.unpack("<HH", arc[-14:-10]) == (0xFFFF, 0xFFFF)
    z = zipfile.ZipFile(io.BytesIO(arc))
    assert len(z.infolist()) == n and z.infolist()[-1].filename == "e65534"
    arc2, _ = orc.zip_create([("e%05d" % i, b"") for i in range(1000)], 9)
    assert arc2[-42:-38] != b"PK\x06\x07"


def test_pin_script_reads_an_entry_payload():
    """tools/pin_against_reference.py extracts the raw payload of a one-entry archive (as zipada would write it)."""
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location(
        "pin", os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "pin_against_reference.py"))
    pin = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(pin)
    data = datagen.text(50_000, 12).tobytes()
    arc, methods = orc.zip_create([("in.bin", data)], 9)
    method, payload = pin.payload_of_single_entry(arc)
    assert method == 12 == methods[0]
    assert payload == orc.encode_stream(data, 9, len(data))


@pytest.mark.parametrize("level", [1, 4, 9])
def test_given_streams_give_the_same_archive(level):
    """orc_zip_create_given with each entry's stream from orc_encode_stream is orc_zip_create, byte for byte:
    the same Add_Stream / Store decision / header rewrite / Finish, only the stream source differs."""
    ents = _entries()
    streams = [orc.encode_stream(d, level, len(d)) for _, d in ents]
    t = [16789 * 65536 + 3 * i for i in range(len(ents))]
    fl = [1, 0, 2, 0, 3, 0]
    ref, methods = orc.zip_create(ents, level, dos_times=t, flags=fl)
    got, methods_given = orc.zip_create_given(ents, streams, level, dos_times=t, flags=fl)
    assert got == ref and methods_given == methods
