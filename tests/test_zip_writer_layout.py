"""The Zip layout unit (zip-ada_b200/csrc/b2_zip_layout.h) on the host, CPU only.

b2_zip_create and the incremental writer (b2_zip_begin / add / finish) both lay out their archives with this unit.
tests/zip_layout_check.cpp, compiled here with g++, lays out catalogues of synthetic sizes (no data is allocated).
Every local header must equal the one restated below from the format (APPNOTE 4.3.7, 4.5.3; Zip.Create decides the
Zip64 extension before compression, with compressed size = size), and the central directory must carry the Zip64 end
records exactly when it must.  The catalogues sit on both sides of each threshold of tests/test_zip64_oracle.py.

The host CRC combine, which folds the Zip CRC-32 of a windowed entry window by window, must equal zlib.crc32 of the
concatenation for split points at 0, 1, 64 KiB +- 1 and seeded random lengths."""
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G4 = 1 << 32


@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    d = tmp_path_factory.mktemp("zip_layout")
    path = str(d / "zip_layout_check")
    subprocess.run(["g++", "-O2", "-std=c++17", "-Wall", "-o", path, os.path.join(ROOT, "tests", "zip_layout_check.cpp")], check=True)
    return path, d


def _layout(exe, cat):
    """cat: list of (name, usize, csize) -> list of (offset, header bytes); the last item is the central directory."""
    path, d = exe
    f = d / "cat.txt"
    f.write_text("".join("%s %d %d\n" % (n, u, c) for n, u, c in cat))
    r = subprocess.run([path, "layout", str(f)], stdout=subprocess.PIPE, text=True, check=True)
    return [(int(a), bytes.fromhex(b)) for a, b in (line.split() for line in r.stdout.split("\n") if line)]


def _local_header(k, name, usize, csize, offset):
    """The local header of entry k, restated from the format."""
    stored = csize >= usize
    csize = usize if stored else csize
    ext = usize >= 0xFFFFFFFF or offset >= 0xFFFFFFFF
    nb = name.encode()
    flags = k % 4
    h = struct.pack("<4sHHHIIII", b"PK\x03\x04", 10, 0x0800 if flags & 1 else 0, 0 if stored else 12, 16789 * 65536,
                    (0x12345678 + k) & 0xFFFFFFFF, 0xFFFFFFFF if ext else csize, 0xFFFFFFFF if ext else usize)
    h += struct.pack("<HH", len(nb), 20 if ext else 0) + nb
    if ext:
        h += struct.pack("<HHQQ", 1, 16, usize, csize)
    return h, csize


def _local_extra(hdr):
    return struct.unpack_from("<H", hdr, 28)[0]


def _has_zip64_end(cd):
    return b"PK\x06\x06" in cd and b"PK\x06\x07" in cd


# name -> (catalogue (name, usize, csize), local Zip64 extension per entry, Zip64 end records)
CASES = {
    "entry 2^32-2": ([("a", G4 - 2, G4 - 2), ("z", 10, 5)], [False, True], True),
    "entry 2^32-1": ([("a", G4 - 1, G4 - 1), ("z", 10, 5)], [True, True], True),
    "header at 0xFFFFFFFE": ([("a", G4 - 33, G4 - 33), ("b", 1000, 1000), ("c", 7, 3)], [False, False, True], True),
    "header at 0xFFFFFFFF": ([("a", G4 - 32, G4 - 32), ("b", 1000, 1000), ("c", 7, 3)], [False, True, True], True),
    "index below Check_Size": ([("a", G4 - 65_724, G4 - 65_724)], [False], False),
    "index at Check_Size": ([("a", G4 - 65_723, G4 - 65_723)], [False], True),
    "compressed mixed": ([("x%d" % i, 5_000_000_000 if i % 3 == 0 else 1000 + i, 1_500_000_000 if i % 3 == 0 else 2000)
                          for i in range(9)], None, True),
}


@pytest.mark.parametrize("case", list(CASES))
def test_local_headers_and_end_records(exe, case):
    cat, local_ext, zip64 = CASES[case]
    hdrs = _layout(exe, cat)
    assert len(hdrs) == len(cat) + 1
    if local_ext is not None:
        assert [_local_extra(h) == 20 for _, h in hdrs[:-1]] == local_ext
    assert _has_zip64_end(hdrs[-1][1]) == zip64
    pos = 0
    for k, ((name, u, c), (off, h)) in enumerate(zip(cat, hdrs)):
        want, payload = _local_header(k, name, u, c, pos)
        assert off == pos and h == want, name
        pos = off + len(h) + payload
    assert hdrs[-1][0] == pos


@pytest.mark.parametrize("n", [65_534, 65_535])
def test_entry_count_zip64_end_records(exe, n):
    cat = [("e%05d" % i, i % 7, i % 7) for i in range(n)]
    hdrs = _layout(exe, cat)
    cd = hdrs[-1][1]
    assert _has_zip64_end(cd) == (n >= 65_535)
    assert struct.unpack_from("<H", cd, len(cd) - 12)[0] == (0xFFFF if n >= 65_535 else n)


def _combine(exe, data, cuts):
    path, d = exe
    f = d / "crc.bin"
    f.write_bytes(data)
    r = subprocess.run([path, "crc", str(f)] + [str(c) for c in cuts], stdout=subprocess.PIPE, text=True, check=True)
    return int(r.stdout)


@pytest.mark.parametrize("n", [0, 1, 65_535, 65_536, 65_537, 300_000])
def test_crc_combine_equals_zlib(exe, n):
    rng = np.random.default_rng(n)
    data = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
    want = zlib.crc32(data)
    fixed = [c for c in (0, 1, 65_535, 65_536, 65_537) if c <= n]
    assert _combine(exe, data, []) == want
    for c in fixed:
        assert _combine(exe, data, [c]) == want, c
    assert _combine(exe, data, fixed) == want
    for _ in range(4):
        cuts = sorted(int(x) for x in rng.integers(0, n + 1, int(rng.integers(1, 9))))
        assert _combine(exe, data, cuts) == want, cuts
