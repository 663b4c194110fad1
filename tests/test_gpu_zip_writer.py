"""One archive written entry by entry: b2_zip_begin / add / finish (`-m gpu`).

Every archive is compared with b2_zip_create of the same entries (which tests/test_gpu_zip.py pins to the oracle),
with the oracle itself where the CPU finishes quickly, and read back by Python's zipfile."""
import ctypes as C
import hashlib
import io
import os
import subprocess
import zipfile
import zlib

import numpy as np
import pytest

import corpus
import datagen
import oracle_lib as orc
from test_gpu_configs import GOLDEN
from test_gpu_zip import _entries

pytestmark = pytest.mark.gpu

MiB = 1 << 20
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OK, ERR_ARGUMENT, ERR_OUTPUT_TOO_SMALL, ERR_ABORTED, ERR_DUPLICATE = 0, 1, 2, 12, 20


def write(enc, entries, window=0, duplicates=0, times=None, flags=None):
    """Python ZipWriter over the entries -> (archive bytes, info, bytes returned by each add)."""
    outs = []
    with enc.zip_writer(duplicates, window) as z:
        for i, (name, data) in enumerate(entries):
            fl = flags[i] if flags else 0
            outs.append(z.add(name, data, dos_time=None if times is None else times[i], unicode=bool(fl & 1), read_only=bool(fl & 2)))
        outs.append(z.finish())
    return b"".join(outs), z.info, outs


def _key(info):
    return [(i.crc32, i.zip_type, i.compressed_size, i.local_header_offset) for i in info]


def _same_as_zip_create(enc, entries, window, times=None, flags=None):
    arc, info, outs = write(enc, entries, window, times=times, flags=flags)
    ref, rinfo = enc.zip_create(entries, dos_times=times, flags=flags, want_info=True)
    assert arc == ref.tobytes()
    assert _key(info) == _key(rinfo)
    return arc, info, outs


def _reads_back(arc, entries):
    z = zipfile.ZipFile(io.BytesIO(arc))
    assert z.testzip() is None
    for (name, data), zi in zip(entries, z.infolist()):
        assert zi.filename == name.replace("\\", "/") and z.read(zi) == bytes(data)


def _log_uniform_entries(n=1500, seed=77):
    rng = np.random.default_rng(seed)
    pool_t, pool_r = datagen.text(3_000_000, 71), datagen.random_bytes(500_000, 72)
    ents = []
    for i in range(n):
        k = int(2 ** rng.uniform(6, 16))
        pool = pool_r if i % 5 == 0 else pool_t
        o = int(rng.integers(0, pool.size - k))
        ents.append(("dir%02d/file%04d.dat" % (i % 17, i), pool[o:o + k].tobytes()))
    return ents


@pytest.fixture(scope="module")
def encs(b2mod):
    e = {lv: b2mod.Encoder(lv, 0) for lv in (1, 4, 9)}
    yield e
    for x in e.values():
        x.close()


# ---- 1. parity ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("level", [1, 4, 9])
@pytest.mark.parametrize("window", [MiB, 3 * MiB, 0])
def test_parity_entries(encs, level, window):
    ents = _entries()                                    # big.txt (1.2 MB) is windowed at W = 1 MiB
    t = [16789 * 65536 + 7 * i for i in range(len(ents))]
    fl = [0, 2, 0, 1, 0, 0, 3, 0]
    arc, info, _ = _same_as_zip_create(encs[level], ents, window, t, fl)
    assert arc == orc.zip_create(ents, level, dos_times=t, flags=fl)[0]
    _reads_back(arc, ents)
    for (name, data), inf in zip(ents, info):
        assert inf.crc32 == zlib.crc32(data)


@pytest.mark.parametrize("level", [1, 4, 9])
@pytest.mark.parametrize("window", [MiB, 3 * MiB, 0])
def test_parity_1500_log_uniform(encs, level, window):
    ents = _log_uniform_entries()
    arc, info, outs = _same_as_zip_create(encs[level], ents, window)
    _reads_back(arc, ents)
    assert {i.zip_type for i in info} == {0, 12}
    if window == MiB:                                    # about 11 MB of input: the queue is written ten times before finish
        assert sum(1 for o in outs[:-1] if o) >= 8


# ---- 2. edges of the queue / window rule --------------------------------------------------------------------------
def test_queue_filled_to_w_and_w_plus_minus_one(encs):
    enc, W = encs[9], MiB
    text = corpus.markov_text(3 * MiB, 0x31)
    for d in (-1, 0, 1):
        a, b = W // 2, W // 2 + d
        ents = [("a", text[:a]), ("b", text[a:a + b]), ("c", text[2 * MiB:2 * MiB + 1000])]
        _, _, outs = _same_as_zip_create(enc, ents, W)
        # a + b <= W: both queued, written when c does not fit; W + 1: a is written when b comes, b and c wait for finish
        assert [bool(o) for o in outs[:3]] == ([False, False, True] if d <= 0 else [False, True, False]), d


def test_entries_of_w_and_w_plus_one(encs):
    enc, W = encs[9], MiB
    text = corpus.markov_text(3 * MiB, 0x32)
    ents = [("queued", text[:W]), ("windowed", text[W:2 * W + 1]), ("after", text[:5000])]
    _, _, outs = _same_as_zip_create(enc, ents, W)
    assert [bool(o) for o in outs] == [False, True, False, True]   # the W + 1 entry flushes the queue and writes itself


def test_windowed_store_fallback_between_small_entries(encs):
    enc, W = encs[9], MiB
    rnd = datagen.random_bytes(3 * MiB + 17, 0x33).tobytes()
    small = datagen.text(20_000, 0x34).tobytes()
    ents = [("s1", small), ("s2", small[:900]), ("random.bin", rnd), ("s3", small[:5]), ("s4", small)]
    arc, info, _ = _same_as_zip_create(enc, ents, W)
    assert [i.zip_type for i in info] == [12, 12, 0, 0, 12]
    assert arc == orc.zip_create(ents, 9)[0]
    _reads_back(arc, ents)


def test_40mib_text_many_windows(encs):
    enc = encs[9]
    text = corpus.markov_text(40 * MiB, 0x35)
    ents = [("before", text[:3000]), ("t40", text), ("after", text[-7000:])]
    arc, info, _ = _same_as_zip_create(enc, ents, MiB)
    s = enc.encode(text, text.size).tobytes()
    off = info[1].local_header_offset + 30 + 3
    assert arc[off:off + len(s)] == s and info[1].crc32 == zlib.crc32(text)


def test_empty_entries_empty_archive_and_backslashes(encs):
    enc = encs[9]
    assert write(enc, [])[0] == orc.zip_create([], 9)[0]
    ents = [("e1", b""), ("dir\\sub\\f.txt", b"hello " * 30), ("e2", b""), ("x\\", b"")]
    for W in (MiB, 0):
        arc, _, _ = _same_as_zip_create(enc, ents, W)
        assert arc == orc.zip_create(ents, 9)[0]
        _reads_back(arc, ents)


# ---- 3. duplicates and Zip64 ----------------------------------------------------------------------------------------
def test_duplicates(b2mod, encs):
    enc = encs[9]
    ents = [("same", b"abc" * 50), ("other", b"x"), ("dir/f", b"y" * 10), ("same", b"def" * 50), ("dir\\f", b"z")]
    arc, _, _ = write(enc, ents, MiB, duplicates=0)
    assert arc == enc.zip_create(ents).tobytes()
    outs = []
    with enc.zip_writer(1, MiB) as z:
        for name, data in ents:
            try:
                outs.append(z.add(name, data))
            except b2mod.B2Error as ex:
                assert "error %d" % ERR_DUPLICATE in str(ex) and "Duplicate_name" in str(ex)
        outs.append(z.finish())
    kept = ents[:3]
    assert b"".join(outs) == enc.zip_create(kept).tobytes() == orc.zip_create(kept, 9)[0]


def test_65535_entries_zip64_end_records(encs):
    enc = encs[9]
    n = 65_535
    ents = [("e%05d" % i, b"") for i in range(n - 3)] + [("t1", b"abc" * 400), ("t2", datagen.text(9000, 3).tobytes()), ("t3", b"z")]
    arc, _, _ = _same_as_zip_create(enc, ents, MiB)
    assert arc[-42:-38] == b"PK\x06\x07" and arc[-98:-94] == b"PK\x06\x06"
    z = zipfile.ZipFile(io.BytesIO(arc))
    assert len(z.infolist()) == n and z.read("t2") == ents[-2][1]


# ---- 4. past 4 GiB ----------------------------------------------------------------------------------------------------
def test_past_4gib_golden_entry_then_small_entries(b2mod):
    """The 4352 MiB mixed golden (2.0 GB compressed), a 2.5 GiB random entry (stored), then small entries past 2^32."""
    import torch
    from test_gpu_past_4gib import N, KEY, SEED, _mem_available
    free, _ = torch.cuda.mem_get_info()
    if free < 150e9:
        pytest.skip("needs 150 GB of free device memory, %.1f GB free" % (free / 1e9))
    if _mem_available() < 48e9:
        pytest.skip("needs 48 GB of available host memory, %.1f GB available" % (_mem_available() / 1e9))
    src = torch.empty(N, dtype=torch.uint8, pin_memory=True)
    step = 256 * MiB
    for i in range(0, N, step):
        src[i:i + step].copy_(corpus.workload("mixed", N, SEED, torch, "cuda", lo=i, hi=min(N, i + step)))
    torch.cuda.empty_cache()
    rnd = np.random.default_rng(0x5EED0041).integers(0, 256, 2560 * MiB, dtype=np.uint8)
    small = [("s%d" % i, datagen.text(10_000 + 997 * i, 0x40 + i).tobytes()) for i in range(5)]
    ents = [("golden.bin", src.numpy()), ("random.bin", rnd)] + small
    with b2mod.Encoder(9, 0) as e:
        arc, info, _ = write(e, ents, 512 * MiB)
        ref, rinfo = e.zip_create(ents, want_info=True)
        assert arc == ref.tobytes() and _key(info) == _key(rinfo)
    del ref
    off = 30 + len("golden.bin") + 20                  # Zip64 local extension: the size is above 0xFFFFFFFF
    assert info[0].zip_type == 12 and info[0].compressed_size == GOLDEN[KEY]["bytes"]
    assert hashlib.sha256(memoryview(arc)[off:off + info[0].compressed_size]).hexdigest() == GOLDEN[KEY]["sha256"]
    assert info[1].zip_type == 0 and info[1].crc32 == zlib.crc32(rnd)
    assert all(i.local_header_offset > (1 << 32) for i in info[2:])
    z = zipfile.ZipFile(io.BytesIO(arc))
    for name, data in small:
        assert z.read(name) == data


# ---- 5. bounded device memory -------------------------------------------------------------------------------------------
def _bound(b2mod, level, W):
    """include/b2gpu.h, b2_zip_begin: the window buffers, 224 bytes per byte of W, 512 MiB."""
    M = int(b2mod.lib().b2_shard_margin(level))
    return 2 * (W + M + 256) + 224 * W + 512 * MiB


def _handle_memory(b2mod, W, entries):
    """Device memory a fresh level-9 handle holds after writing `entries` (an iterable of (name, data)) at window W."""
    import torch
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free0 = torch.cuda.mem_get_info()[0]
    n = 0
    with b2mod.Encoder(9, 0) as e:
        with e.zip_writer(0, W) as z:
            for name, data in entries:
                n += len(z.add(name, data))
            n += len(z.finish())
        used = free0 - torch.cuda.mem_get_info()[0]
    return used, n


def test_device_memory_does_not_grow_with_the_archive(b2mod):
    W = 256 * MiB
    piece = _gpu_text(64 * MiB, 0x51)
    big = _gpu_text(300 * MiB, 0x52)                     # windowed
    used = {}
    for gib in (2, 8):
        ents = [("p%04d" % i, piece) for i in range(gib * 16)] + [("big", big)]
        used[gib], n = _handle_memory(b2mod, W, ents)
        print("archive of %d GiB + 300 MiB: %d bytes, handle holds %.2f GB of device memory" % (gib, n, used[gib] / 1e9))
    assert abs(used[8] - used[2]) <= 64 * MiB, used
    assert used[8] < _bound(b2mod, 9, W), (used, _bound(b2mod, 9, W))


@pytest.mark.parametrize("kind,W,count", [("empty", MiB, 100_000), ("50 B", MiB, 100_000), ("50 B", 16 * MiB, 200_000),
                                          ("4 KiB", 16 * MiB, 20_000)])
def test_device_memory_of_many_small_entries(b2mod, kind, W, count):
    """A flood of empty or tiny entries: every queued entry costs device memory whatever its size, so the queue is also
    written after W / 32 KiB entries.  The handle stays below the stated bound, and 10 x more entries cost no more."""
    text = datagen.text(4096 + 60, 0x53).tobytes()
    size = {"empty": 0, "50 B": 50, "4 KiB": 4096}[kind]

    def ents(k):
        return (("f%07d" % i, text[i % 60:i % 60 + size]) for i in range(k))
    used_small, _ = _handle_memory(b2mod, W, ents(count // 10))
    used, n = _handle_memory(b2mod, W, ents(count))
    print("%d entries of %s at W = %d MiB: %d bytes, handle holds %.3f GB (%.3f GB for a tenth), bound %.3f GB"
          % (count, kind, W >> 20, n, used / 1e9, used_small / 1e9, _bound(b2mod, 9, W) / 1e9))
    assert used < _bound(b2mod, 9, W)
    assert used <= used_small + 64 * MiB


def _gpu_text(n, seed):
    import torch
    return corpus.workload("markov", n, seed, torch, "cuda").cpu().numpy()


# ---- 6. refusals, progress and recovery --------------------------------------------------------------------------------
class Raw:
    def __init__(self, b2mod, enc):
        self.lib, self.h = b2mod.lib(), enc._h

    def add(self, name, a, cap=None):
        a = np.ascontiguousarray(a, np.uint8)
        nb = name.encode()
        cap = int(self.lib.b2_zip_add_bound(self.h, a.size, len(nb))) if cap is None else cap
        out = np.empty(max(cap, 1), np.uint8)
        ln = C.c_uint64(0)
        rc = self.lib.b2_zip_add(self.h, C.c_char_p(nb), len(nb), 16789 * 65536, 0, a.ctypes.data if a.size else None, a.size,
                                 out.ctypes.data, cap, C.byref(ln))
        return rc, out[:ln.value].tobytes()

    def finish(self, cap=None):
        cap = int(self.lib.b2_zip_finish_bound(self.h)) if cap is None else cap
        out = np.empty(max(cap, 1), np.uint8)
        ln, n = C.c_uint64(0), C.c_uint64(0)
        rc = self.lib.b2_zip_finish(self.h, out.ctypes.data, cap, C.byref(ln), None, 0, C.byref(n))
        return rc, out[:ln.value].tobytes()


def test_output_too_small_is_refused_then_repeated(b2mod, encs):
    enc = encs[9]
    raw = Raw(b2mod, enc)
    text = corpus.markov_text(5 * MiB, 0x61)
    ents = [("a", text[:700_000]), ("b", text[700_000:1_200_000]), ("w", text[:3 * MiB]), ("c", text[:100])]
    assert raw.lib.b2_zip_begin(raw.h, 0, MiB) == OK
    outs = []
    for name, data in ents:
        cap = int(raw.lib.b2_zip_add_bound(raw.h, data.size, len(name)))
        rc, o = raw.add(name, data, cap - 1)
        assert rc == ERR_OUTPUT_TOO_SMALL and o == b""
        rc, o = raw.add(name, data)
        assert rc == OK, raw.lib.b2_last_error()
        outs.append(o)
    assert raw.finish(int(raw.lib.b2_zip_finish_bound(raw.h)) - 1)[0] == ERR_OUTPUT_TOO_SMALL
    rc, o = raw.finish()
    assert rc == OK
    assert b"".join(outs + [o]) == enc.zip_create(ents).tobytes()


def test_calls_refused_while_an_archive_is_open(b2mod, encs):
    enc = encs[9]
    lib = b2mod.lib()
    raw = Raw(b2mod, enc)
    small = np.frombuffer(b"abc" * 100, np.uint8)
    assert raw.add("x", small)[0] == ERR_ARGUMENT                    # no archive open
    assert raw.finish()[0] == ERR_ARGUMENT
    assert lib.b2_zip_begin(enc._h, 0, MiB - 1) == ERR_ARGUMENT        # window below 1 MiB
    assert lib.b2_zip_begin(enc._h, 2, MiB) == ERR_ARGUMENT            # no such duplicate policy
    assert lib.b2_zip_begin(enc._h, 0, MiB) == OK
    assert lib.b2_zip_begin(enc._h, 0, MiB) == ERR_ARGUMENT            # begin twice
    outs = [raw.add("first", small)[1]]
    out = np.empty(1 << 20, np.uint8)
    ln = C.c_uint64(0)
    assert lib.b2_encode_stream(enc._h, small.ctypes.data, small.size, -1, out.ctypes.data, out.size, C.byref(ln)) == ERR_ARGUMENT
    flat, offs, sizes, names, name_offs = orc.pack_entries([("a", small)])
    info = (b2mod.ZipEntryInfo * 1)()
    assert lib.b2_zip_create(enc._h, 1, flat.ctypes.data, offs.ctypes.data, sizes.ctypes.data, C.c_char_p(names), name_offs.ctypes.data,
                             None, None, 0, out.ctypes.data, out.size, C.byref(ln), info) == ERR_ARGUMENT
    assert lib.b2_shard_open(enc._h, small.ctypes.data, 0, 0, small.size, small.size, -1, small.size) == ERR_ARGUMENT
    res = b2mod.VerifyResult()
    assert lib.b2_verify_stream(enc._h, out.ctypes.data, 0, 100, None, 0, 0, C.byref(res)) == ERR_ARGUMENT
    crc = C.c_uint32(0)
    assert lib.b2_zip_crc32(enc._h, small.ctypes.data, small.size, C.byref(crc)) == ERR_ARGUMENT
    assert lib.b2_stream_begin(enc._h, -1, MiB) == ERR_ARGUMENT         # a stream is refused while an archive is open
    outs.append(raw.add("second", small)[1])                           # the archive goes on unharmed
    rc, o = raw.finish()
    assert rc == OK
    assert b"".join(outs + [o]) == enc.zip_create([("first", small), ("second", small)]).tobytes()
    # an archive is refused while a stream is open
    assert lib.b2_stream_begin(enc._h, -1, MiB) == OK
    assert lib.b2_zip_begin(enc._h, 0, MiB) == ERR_ARGUMENT
    assert lib.b2_stream_abort(enc._h) == OK
    # abort, then a new archive
    assert lib.b2_zip_begin(enc._h, 0, MiB) == OK and raw.add("z", small)[0] == OK
    assert lib.b2_zip_abort(enc._h) == OK and lib.b2_zip_abort(enc._h) == OK
    assert write(enc, [("a", small)])[0] == enc.zip_create([("a", small)]).tobytes()


def test_progress_and_abort(b2mod, encs):
    enc = encs[9]
    text = corpus.markov_text(9 * MiB, 0x62)
    ents = [("a", text[:600_000]), ("b", text[600_000:1_000_000]), ("w", text[:5 * MiB]), ("c", text[5 * MiB:6 * MiB])]
    total = sum(d.size for _, d in ents)
    seen = []
    enc.set_progress(lambda done, tot: seen.append((done, tot)) and False)
    try:
        arc, _, _ = write(enc, ents, MiB)
        assert arc == enc.zip_create(ents).tobytes()
        dones = [d for d, _ in seen]
        assert len(seen) >= 4 and dones == sorted(dones) and dones[-1] == total, seen
        assert all(d <= t for d, t in seen) and seen[-1][1] == total
        # abort at the second report: the archive is closed
        calls = []
        enc.set_progress(lambda done, tot: calls.append(done) or len(calls) >= 2)
        raw = Raw(b2mod, enc)
        assert raw.lib.b2_zip_begin(raw.h, 0, MiB) == OK
        rcs = [raw.add(name, data)[0] for name, data in ents]
        assert ERR_ABORTED in rcs
        first = rcs.index(ERR_ABORTED)
        assert all(rc == OK for rc in rcs[:first]) and all(rc == ERR_ARGUMENT for rc in rcs[first + 1:])
        assert raw.finish()[0] == ERR_ARGUMENT
    finally:
        enc.set_progress(None)
    assert write(enc, ents, MiB)[0] == orc.zip_create(ents, 9)[0]
    assert enc.encode(text, -1).tobytes() == orc.encode_stream(text, 9, -1, threads=os.cpu_count() or 4)


def test_two_handles_write_at_the_same_time(encs):
    a, b = encs[9], encs[4]
    ea = _log_uniform_entries(300, 5) + [("wa", corpus.markov_text(2 * MiB + 5, 0x63))]
    eb = [("wb", corpus.mixed(3 * MiB, 0x64, 1 << 20))] + _log_uniform_entries(200, 6)
    oa, ob = [], []
    with a.zip_writer(0, MiB) as za, b.zip_writer(0, MiB) as zb:
        for i in range(max(len(ea), len(eb))):
            if i < len(ea):
                oa.append(za.add(*ea[i]))
            if i < len(eb):
                ob.append(zb.add(*eb[i]))
        oa.append(za.finish())
        ob.append(zb.finish())
    assert b"".join(oa) == a.zip_create(ea).tobytes()
    assert b"".join(ob) == b.zip_create(eb).tobytes()


# ---- 7. hosts -----------------------------------------------------------------------------------------------------
def test_python_writer_aborts_on_exception(encs):
    enc = encs[9]
    ents = [("a", datagen.text(50_000, 0x71).tobytes()), ("b", corpus.markov_text(2 * MiB, 0x72))]
    with pytest.raises(ZeroDivisionError):
        with enc.zip_writer(0, MiB) as z:
            z.add(*ents[0])
            z.add(*ents[1])
            1 / 0
    assert write(enc, ents, MiB)[0] == enc.zip_create(ents).tobytes()


def test_cpp_zip_writer(tmp_path):
    pkg = os.path.join(ROOT, "zip-ada_b200")
    exe = str(tmp_path / "test_zip_writer")
    subprocess.check_call(["g++", "-O2", "-std=c++17", os.path.join(pkg, "host", "test_zip_writer.cpp"), "-L" + pkg, "-lb2gpu",
                           "-Wl,-rpath," + pkg, "-o", exe])
    files = [("one.txt", datagen.text(40_000, 0x81).tobytes()), ("empty", b""), ("big.txt", corpus.markov_text(3 * MiB, 0x82).tobytes()),
             ("rnd.bin", datagen.random_bytes(20_000, 0x83).tobytes()), ("sub/two.txt", datagen.text(9_000, 0x84).tobytes())]
    (tmp_path / "sub").mkdir()
    for name, data in files:
        (tmp_path / name).write_bytes(data)
    r = subprocess.run([exe, "--window", str(MiB), "out.zip"] + [n for n, _ in files], cwd=str(tmp_path), stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True)
    assert r.returncode == 0, r.stderr
    assert r.stdout.split() == ["entries=%d" % len(files)]
    assert (tmp_path / "out.zip").read_bytes() == orc.zip_create(files, 9)[0]
    r = subprocess.run([exe, "--error-on-duplicate", "dup.zip", "one.txt", "one.txt"], cwd=str(tmp_path), stderr=subprocess.PIPE, text=True)
    assert r.returncode == 3 and "Duplicate_name" in r.stderr
