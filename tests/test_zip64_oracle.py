"""Zip64 thresholds of the oracle's Zip.Create (oracle/zip_oracle.cpp), on both sides of each, CPU only.

Every archive holds stored entries with one-byte names, built by orc_zip_create_given (stream_len = size, so
nothing is encoded) from slices of one shared zero buffer.  Each is checked by tests/zipscan.py (a reader written
from the format plus the Zip64 rules restated) and by Python's zipfile.  The sizes:

  T1  one entry of size S vs 0xFFFFFFFF (local and central Zip64 extension):   S = 2^32 - 2 | 2^32 - 1
  T2  entry `a` of size S1, then `b` at offset 31 + S1 vs 0xFFFFFFFF:          S1 = 2^32 - 33 | 2^32 - 32
  T4  Check_Size in Finish: one entry of size S, index after the central directory S + 79 vs 2^32 - 65 644:
                                                                               S = 2^32 - 65 724 | 2^32 - 65 723
      (T1 and T2 sizes are past Check_Size's 2^32 - 65 644 in Add_Stream, so both sides of them carry the Zip64
      end record; T4's are below it.)

Each archive is about 4 GiB and at most one is alive at a time; the peak is about 13 GB of host memory.  The
oracle's byte-table CRC, run twice per stored entry, takes most of the time (about 15 s per archive).
"""
import io
import zipfile
import zlib

import numpy as np
import pytest

import oracle_lib as orc
import zipscan as zs

G4 = 1 << 32
SMALL_B = 1000

# name -> (entry sizes, Zip64 local extension per entry, Zip64 end records)
CASES = {
    "T1_below": ([G4 - 2], [False], True),
    "T1_at": ([G4 - 1], [True], True),
    "T2_below": ([G4 - 33, SMALL_B], [False, False], True),
    "T2_at": ([G4 - 32, SMALL_B], [False, True], True),
    "T4_below": ([G4 - 65_724], [False], False),
    "T4_at": ([G4 - 65_723], [False], True),
}
NAMES = [b"a", b"b"]


@pytest.fixture(scope="module")
def zeros():
    return np.zeros(G4 + 65_536, np.uint8)          # untouched pages: costs no memory


def _crc(buf, n):
    return zlib.crc32(memoryview(buf[:n]))


@pytest.mark.parametrize("case", list(CASES))
def test_zip64_threshold(zeros, case):
    sizes, local_ext, zip64 = CASES[case]
    names = NAMES[:len(sizes)]
    sz = np.array(sizes, np.uint64)
    offs = np.zeros(len(sizes), np.uint64)
    name_offs = np.array([0, 1, 2][:len(sizes) + 1], np.uint32)
    arr, methods = orc.zip_create_given_flat(zeros, offs, sz, b"".join(names), name_offs, None, offs, sz)
    arc = arr.tobytes()
    del arr
    assert methods == [0] * len(sizes)
    crcs = [_crc(zeros, n) for n in sizes]
    lay = zs.check_layout(arc, sizes, names, crcs)
    # the side of each threshold, as the table above states it (independent of expected_layout's arithmetic)
    assert [e["local_ext"] for e in lay["entries"]] == local_ext
    assert lay["zip64"] == zip64
    if case == "T2_below":
        assert lay["entries"][1]["offset"] == 0xFFFFFFFE
    if case == "T2_at":
        assert lay["entries"][1]["offset"] == 0xFFFFFFFF
        assert lay["scan"]["central"][1]["offset"] == 0xFFFFFFFF and lay["scan"]["central"][0]["extra"] == ()
    if case.startswith("T4"):
        assert lay["cd_offset"] + lay["cd_size"] + 1 == sizes[0] + 79
    # an independent reader
    z = zipfile.ZipFile(io.BytesIO(arc))
    infos = z.infolist()
    assert [i.filename.encode() for i in infos] == names
    for zi, e, c in zip(infos, lay["entries"], crcs):
        assert (zi.file_size, zi.compress_size, zi.header_offset, zi.CRC, zi.compress_type) == (e["size"], e["size"], e["offset"], c, 0)
    if len(sizes) == 2:
        assert z.read("b") == bytes(SMALL_B)
    if case == "T1_at":
        assert z.testzip() is None                   # reads the 4 GiB entry through the Zip64 extension, CRC checked


def test_zipscan_reads_small_archives_with_compressed_entries():
    """The reader and the restated rules on archives below every threshold, compressed and stored entries mixed."""
    from test_zip_oracle import _entries
    ents = _entries()
    arc, methods = orc.zip_create(ents, 9)
    streams = [orc.encode_stream(d, 9, len(d)) for _, d in ents]
    csizes = [len(s) if m == 12 else len(d) for s, m, (_, d) in zip(streams, methods, ents)]
    names = [n.replace("\\", "/").encode() for n, _ in ents]
    lay = zs.check_layout(arc, [len(d) for _, d in ents], names, [zlib.crc32(d) for _, d in ents], csizes)
    assert not lay["zip64"] and not any(e["local_ext"] or e["central_ext"] for e in lay["entries"])
    assert [l["method"] for l in lay["scan"]["local"]] == methods
