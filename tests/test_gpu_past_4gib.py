"""Inputs, streams and archives past 2^32 bytes on the device (`-m gpu`).

The C ABI takes 64-bit sizes and offsets everywhere; these tests put bytes past 2^32 through each part of it:
the Zip CRC-32, the chunk cutter and its trace, the host and device entry points, the shard handoff, the batch
job offsets, the output arena, the decoder / verify, and the Zip64 layout of b2_zip_create.  References that do
not share the library's code: the committed goldens (made by the oracle), zlib.crc32, the oracle's archive
(orc_zip_create_given), tests/zipscan.py and Python's zipfile.

Everything is cut from one host buffer W (module scope):
  W[0:N]        the 4352 MiB config-3 corpus (mixed, seed 5eed0004); its first 4 GiB are the 4 GiB config-3 corpus
  W[N:N+TAIL]   small entries (text, random, sparse, runs ...); they sit at input offsets past 2^32
  W[RB:RB+RN]   2^32 + 1 MiB of seeded random bytes (corpus.random_bytes, seed 5eed0002)

The handles are this module's own, created with B2GPU_BATCH_POSITIONS = 2^28: about 14 GB of workspace each,
and batches smaller than the inputs, so batch boundaries fall past 2^32 too.  On a B200 (1000 W power limit) the
module used at most 106.7 GB of device memory and 28.8 GB of host memory (peak RSS), as it prints at its end,
and took 7 min 12 s, most of it on the host (the oracle's CRCs of the stored 4 GiB entries, SHA-256, zlib).  It
skips, saying so, when less than NEED_DEVICE_GB of device memory is free or less than NEED_HOST_GB of host
memory is available.
"""
import hashlib
import io
import os
import threading
import zipfile
import zlib

import numpy as np
import pytest

import corpus
import datagen
import oracle_lib as orc
import zipscan as zs
from test_gpu_configs import GOLDEN, _shards_by_hand
from test_zip64_oracle import CASES

pytestmark = pytest.mark.gpu

MiB = 1 << 20
G4 = 1 << 32
N = 4352 * MiB
SEED = 0x5EED0004
KEY = "mixed:%d:5eed0004:9" % N
KEY4 = "mixed:%d:5eed0004:9" % G4
TAIL = 16 * MiB
RB = N + TAIL
RN = G4 + MiB
RSEED = 0x5EED0002
BATCH_POSITIONS = 1 << 28
# the peaks above plus headroom
NEED_DEVICE_GB = 120
NEED_HOST_GB = 40


def _sha(a):
    return hashlib.sha256(memoryview(np.ascontiguousarray(a))).hexdigest()


def _mem_available():
    with open("/proc/meminfo") as f:
        for line in f:
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) * 1024
    return 0


class _PeakDeviceUse(threading.Thread):
    """Polls cudaMemGetInfo: the peak device memory in use while the module runs, over what was in use before."""

    def __init__(self, torch):
        super().__init__(daemon=True)
        self.torch = torch
        free, total = torch.cuda.mem_get_info()
        self.base = total - free
        self.peak = self.base
        self.stop = threading.Event()

    def run(self):
        while not self.stop.wait(0.05):
            free, total = self.torch.cuda.mem_get_info()
            self.peak = max(self.peak, total - free)


@pytest.fixture(scope="module")
def handles(b2mod):
    import torch
    free = torch.cuda.mem_get_info()[0]
    if free < NEED_DEVICE_GB * 10 ** 9:
        pytest.skip("needs %d GB of free device memory, %.1f GB free" % (NEED_DEVICE_GB, free / 1e9))
    avail = _mem_available()
    if avail < NEED_HOST_GB * 10 ** 9:
        pytest.skip("needs %d GB of available host memory, %.1f GB available" % (NEED_HOST_GB, avail / 1e9))
    mon = _PeakDeviceUse(torch)
    mon.start()
    with pytest.MonkeyPatch.context() as mp:
        mp.setenv("B2GPU_BATCH_POSITIONS", str(BATCH_POSITIONS))       # read by b2_create
        encs = [b2mod.Encoder(9, 0) for _ in range(3)]
    yield encs
    for e in encs:
        e.close()
    mon.stop.set()
    mon.join()
    with open("/proc/self/status") as f:
        hwm = [l for l in f if l.startswith("VmHWM:")][0].split()[1]
    print("past-4GiB module: peak device memory in use %.1f GB (%.1f GB before it), host peak RSS %.1f GB, device %s"
          % (mon.peak / 1e9, mon.base / 1e9, int(hwm) * 1024 / 1e9, torch.cuda.get_device_name(0)))


# small entries: name -> (bytes), laid out in W[N:N+TAIL]
def _small_entries():
    return {
        "text_50k": datagen.text(50_000, 31),
        "text_b": datagen.text(200_000, 32),
        "text_two_chunks": datagen.text(2_500_000, 33),
        "text_1M": datagen.text(1_000_000, 34),
        "random_300k": datagen.random_bytes(300_000, 35),
        "random_2M": datagen.random_bytes(2_000_000, 36),
        "sparse_400k": datagen.sparse_binary(400_000, 37),
        "run_259": np.full(259, 0x41, np.uint8),
        "zeros_1M": np.zeros(1_000_000, np.uint8),
        "mixed_3M": datagen.mixed(3_000_000, 50_000, 38),
        "one": np.array([0x7A], np.uint8),
        "empty": np.zeros(0, np.uint8),
    }


@pytest.fixture(scope="module")
def world(handles):
    """(W, the 4352 MiB corpus on the device with 64 bytes of slack, {small entry: (offset in W, size)})."""
    import torch
    W = np.empty(RB + RN + 64, np.uint8)
    d_big = torch.empty(N + 64, dtype=torch.uint8, device="cuda")
    d_big[N:] = 0
    step = 512 * MiB
    for lo in range(0, N, step):
        hi = min(N, lo + step)
        d_big[lo:hi] = corpus.workload("mixed", N, SEED, torch, "cuda", lo=lo, hi=hi)
    torch.from_numpy(W[:N]).copy_(d_big[:N])
    for lo in range(0, RN, step):
        hi = min(RN, lo + step)
        torch.from_numpy(W[RB + lo:RB + hi]).copy_(corpus.workload("random", RN, RSEED, torch, "cuda", lo=lo, hi=hi))
    W[RB + RN:] = 0
    small = {}
    pos = N
    for name, d in _small_entries().items():
        W[pos:pos + d.size] = d
        small[name] = (pos, d.size)
        pos += (d.size + 15) & ~15
    assert pos <= N + TAIL
    W[pos:RB] = 0
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return W, d_big, small


@pytest.fixture(scope="module")
def big_stream(handles, world):
    """The 4352 MiB corpus encoded by the host entry point, with its chunk trace."""
    W = world[0]
    out = handles[0].encode(W[:N], N).copy()
    return out, handles[0].trace()


# ---- 1. Zip CRC-32 past 2^32 ----------------------------------------------------------------------------------
def test_zip_crc32_past_4gib(handles, world):
    R = world[0][RB:RB + G4 + 65_536 + 81]
    for lo, hi in ((0, G4 - 1), (0, G4), (0, G4 + 1), (0, R.size), (12_345, R.size)):
        v = R[lo:hi]
        assert handles[0].zip_crc32(v) == zlib.crc32(memoryview(v)), (lo, hi)


# ---- 2. one stream of 4352 MiB ----------------------------------------------------------------------------------
def test_stream_past_4gib_equals_golden(b2mod, handles, world, big_stream):
    import torch
    W, d_big, _ = world
    g = GOLDEN[KEY]
    data = W[:N]
    assert _sha(data) == g["input_sha256"], "the corpus generator changed"
    assert _sha(data[:G4]) == GOLDEN[KEY4]["input_sha256"]
    # the corpus mixes the high word of the position: bytes past 2^32 are not those at the same position mod 2^32
    assert np.array_equal(data[G4:G4 + 4096], corpus.random_bytes(4096, SEED + 1, pos0=G4))
    assert not np.array_equal(data[G4:G4 + 4096], corpus.random_bytes(4096, SEED + 1, pos0=0))
    out, tr = big_stream
    assert out.size == g["bytes"] and _sha(out) == g["sha256"]
    assert tr[0].start == 0 and tr[-1].start + tr[-1].len == N
    assert all(b.start == a.start + a.len for a, b in zip(tr, tr[1:]))
    assert sum(t.start >= G4 for t in tr) >= 100
    # the device entry point on a torch tensor: 64 bytes of slack behind the input, 4-byte aligned output
    enc = handles[0]
    cap = int(b2mod.lib().b2_bound(N)) + 1024 * (N // 40000 + 16)
    d_out = torch.empty(cap, dtype=torch.uint8, device="cuda")
    ln = enc.encode_device_ptr(d_big.data_ptr(), N, N, d_out.data_ptr(), cap)
    assert ln == g["bytes"]
    assert _sha(d_out[:ln].cpu().numpy()) == g["sha256"]
    del d_out
    torch.cuda.empty_cache()
    assert [(t.start, t.len, t.winner) for t in enc.trace()] == [(t.start, t.len, t.winner) for t in tr]


# ---- 3. verify of that stream --------------------------------------------------------------------------------------
def test_verify_past_4gib(handles, world, big_stream):
    enc = handles[0]
    data = world[0][:N]
    out, tr = big_stream
    r = enc.verify(out, data)
    assert r.ok == 1 and r.decoded_bytes == N, (r.first_bad_block, r.first_bad_status, r.mismatch_at)
    n_blocks = [{0: 1, 1: 4, 2: max(1, t.n_seg1), 3: max(1, t.n_seg2)}[t.winner] for t in tr]
    assert r.blocks == sum(n_blocks)
    p = G4 + 12_345
    data[p] ^= 0xFF
    try:
        r = enc.verify(out, data)
    finally:
        data[p] ^= 0xFF
    assert r.ok == 0 and r.mismatch_at == p
    r = enc.verify(out, data[:G4 + 5])
    assert r.ok == 0 and r.mismatch_at == G4 + 5
    # one bit flipped at 90 % of the stream: the first bad block is in the chunk that holds that bit
    byte = out.size * 9 // 10
    bit = byte * 8 + 3                                   # mask 0x10, bits are numbered from the top of each byte
    assert bit >= G4
    off, blk = 32, 0                                     # "BZh9"
    for t, nb in zip(tr, n_blocks):
        if off <= bit < off + t.bits[t.winner]:
            lo_blk, hi_blk = blk, blk + nb
            break
        off += t.bits[t.winner]
        blk += nb
    else:
        raise AssertionError("no chunk holds bit %d" % bit)
    out[byte] ^= 0x10
    try:
        r = enc.verify(out)
    finally:
        out[byte] ^= 0x10
    assert r.ok == 0 and lo_blk <= r.first_bad_block < hi_blk, (r.first_bad_block, r.first_bad_status, lo_blk, hi_blk)


# ---- 4. shards across 2^32 -------------------------------------------------------------------------------------------
def test_shards_across_4gib(b2mod, handles, world, big_stream):
    data = world[0][:N]
    g = GOLDEN[KEY]
    starts = {t.start for t in big_stream[1]}
    got, entries = _shards_by_hand(b2mod, handles, data, N, [0, 2 * 1024 * MiB, G4, N])
    assert len(got) == g["bytes"] and _sha(np.frombuffer(got, np.uint8)) == g["sha256"]
    assert entries[2] >= G4 and entries[2] in starts           # the handoff into the shard that starts at 2^32
    del got
    bounds = b2mod.shard_plan(N, 2)
    got, entries = _shards_by_hand(b2mod, handles[:2], data, N, bounds)
    assert len(got) == g["bytes"] and _sha(np.frombuffer(got, np.uint8)) == g["sha256"]
    assert entries[1] in starts


# ---- 5. batch entries at input offsets past 2^32 ---------------------------------------------------------------------
def test_batch_entries_past_4gib(handles, world):
    W, _, small = world
    names = [k for k in small]
    ents = [W[:G4]] + [W[small[k][0]:small[k][0] + small[k][1]] for k in names]
    outs = handles[0].encode_batch(ents, "size")
    assert _sha(np.frombuffer(outs[0], np.uint8)) == GOLDEN[KEY4]["sha256"] and len(outs[0]) == GOLDEN[KEY4]["bytes"]
    for k, e, o in zip(names, ents[1:], outs[1:]):
        ref = orc.encode_stream(e, 9, e.size, threads=(os.cpu_count() or 4) if e.size >= MiB else 0)
        assert o == ref, k


# ---- 6. compressed output past 2^32 bytes ----------------------------------------------------------------------------
def test_output_past_4gib(handles, world):
    enc = handles[0]
    R = world[0][RB:RB + RN]
    out = enc.encode(R, RN)
    assert out.size > G4 and out[:4].tobytes() == b"BZh9"
    r = enc.verify(out, R)
    assert r.ok == 1 and r.decoded_bytes == RN, (r.first_bad_block, r.first_bad_status, r.mismatch_at)


# ---- 7. Zip64 archives on the device against the oracle ------------------------------------------------------------
def _archive(enc, W, layout, given):
    """layout: [(name, offset in W, size)]; given: {entry index: its BZip2 stream (checked beforehand)}, every
    other entry must be stored.  Builds the archive on the device and with the oracle from the same W, asserts
    they are byte-identical and that zipscan and zipfile read it, and returns (archive bytes, info, scan)."""
    names = [nm for nm, _, _ in layout]
    offs = np.array([o for _, o, _ in layout], np.uint64)
    sizes = np.array([s for _, _, s in layout], np.uint64)
    name_offs = np.zeros(len(layout) + 1, np.uint32)
    name_offs[1:] = np.cumsum([len(nm) for nm in names])
    nb = b"".join(names)
    arc_d, info = enc.zip_create_flat(W, offs, sizes, nb, name_offs, want_info=True)
    for i in range(len(layout)):
        assert info[i].zip_type == (12 if i in given else 0), i
    streams = b"".join(given[i] for i in sorted(given))
    soffs = np.zeros(len(layout), np.uint64)
    slens = sizes.copy()
    pos = 0
    for i in sorted(given):
        soffs[i], slens[i] = pos, len(given[i])
        pos += len(given[i])
    arc_o, methods = orc.zip_create_given_flat(W, offs, sizes, nb, name_offs, np.frombuffer(streams, np.uint8), soffs, slens)
    assert methods == [i.zip_type for i in info]
    assert arc_d.size == arc_o.size and np.array_equal(arc_d, arc_o)
    del arc_o
    arc = arc_d.tobytes()
    del arc_d
    datas = [W[o:o + s] for _, o, s in layout]
    crcs = [zlib.crc32(memoryview(d)) for d in datas]
    csizes = [int(i.compressed_size) for i in info]
    lay = zs.check_layout(arc, [int(s) for s in sizes], names, crcs, csizes)
    for i, e, c in zip(info, lay["entries"], crcs):
        assert (i.crc32, i.local_header_offset) == (c, e["offset"])
    z = zipfile.ZipFile(io.BytesIO(arc))
    for zi, e, c in zip(z.infolist(), lay["entries"], crcs):
        assert (zi.file_size, zi.compress_size, zi.header_offset, zi.CRC) == (e["size"], e["csize"], e["offset"], c)
    for (nm, o, s), zi in zip(layout, z.infolist()):
        assert zi.filename.encode() == nm
        if s < 64 * MiB:
            assert z.read(zi) == W[o:o + s].tobytes(), nm
    return arc, info, lay


@pytest.mark.parametrize("case", list(CASES))
def test_zip64_threshold_archives(handles, world, case):
    """The T1 / T2 / T4 pairs of test_zip64_oracle.py with seeded random entries (really stored); `b` of T2 is
    text read from an input offset past 2^32, so its stream and CRC are computed there."""
    enc = handles[0]
    W, _, small = world
    sizes, local_ext, zip64 = CASES[case]
    layout = [(b"a", RB, sizes[0])]
    given = {}
    if len(sizes) == 2:
        ob, nb = small["text_b"]
        assert ob > G4
        s = orc.encode_stream(W[ob:ob + nb], 9, nb)
        assert enc.encode(W[ob:ob + nb], nb).tobytes() == s and len(s) < nb
        layout.append((b"b", ob, nb))
        given[1] = s
    arc, info, lay = _archive(enc, W, layout, given)
    assert [e["local_ext"] for e in lay["entries"]] == local_ext
    assert lay["zip64"] == zip64
    if case == "T2_at":
        assert info[1].local_header_offset == 0xFFFFFFFF
    if case == "T2_below":
        assert info[1].local_header_offset == 0xFFFFFFFE


def test_zip64_archive_with_compressed_entries(handles, world):
    """A small text entry, the 4 GiB config-3 corpus (compressed, Zip64 sizes), a stored filler, then a text and a
    random entry whose local headers sit past 2^32."""
    enc = handles[0]
    W, _, small = world
    big = enc.encode(W[:G4], G4).tobytes()
    assert hashlib.sha256(big).hexdigest() == GOLDEN[KEY4]["sha256"]
    filler = 2_500_000_000
    layout = [(b"s.txt", *small["text_50k"]), (b"mixed4g.bin", 0, G4), (b"filler.bin", RB, filler),
              (b"t.txt", *small["text_1M"]), (b"r.bin", *small["random_300k"])]
    given = {1: big}
    for i in (0, 3):
        _, o, s = layout[i]
        ref = orc.encode_stream(W[o:o + s], 9, s)
        assert enc.encode(W[o:o + s], s).tobytes() == ref
        given[i] = ref
    arc, info, lay = _archive(enc, W, layout, given)
    assert info[3].local_header_offset > G4 and info[4].local_header_offset > G4
    assert lay["entries"][1]["local_ext"] and lay["entries"][3]["central_ext"] and lay["zip64"]
    pay = lay["scan"]["local"][1]["payload"]
    payload = np.frombuffer(arc, np.uint8, count=len(big), offset=pay)
    assert hashlib.sha256(payload).hexdigest() == GOLDEN[KEY4]["sha256"]
    r = enc.verify(payload, W[:G4])
    assert r.ok == 1 and r.decoded_bytes == G4, (r.first_bad_block, r.first_bad_status, r.mismatch_at)
