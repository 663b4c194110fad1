"""CPU tests of the window rule of b2_stream_* (DESIGN.md §6b) on the oracle (no GPU).

A stream fed in pieces is encoded window by window: with M = b2_shard_margin (level), when W + M bytes are held
from `base` (the start of the next chunk), the window is a shard of the stream with own_end = base + W whose stream
size is unknown; the next window starts at its handoff.  The last window holds what is left and writes the footer.
Here every window runs through the oracle's shard entry points (orc_shard_encode / orc_shard_finish), sequentially,
and the assembled stream must equal the oracle's one-shot encode for every level, hint and window placement.
"""
import ctypes as C
import functools
import os

import numpy as np
import pytest

import corpus
import oracle_lib as orc

UNKNOWN = (1 << 64) - 1
THREADS = max(2, min(8, os.cpu_count() or 2))


class _Link(C.Structure):
    _fields_ = [("total_bits", C.c_uint64 * 8), ("crc_rot", C.c_uint32 * 8), ("crc_fold", C.c_uint32 * 8)]


def margin(level):
    return 10 * 100_000 * level + 4096


def stream_by_windows(data, level, hint, W):
    """The stream b2_stream_* writes, with the oracle as the engine.  Returns (stream bytes, window starts)."""
    lib = orc.lib()
    lib.orc_shard_encode.restype = C.c_void_p
    n, M = data.size, margin(level)
    base, bit, crc = 0, 32, 0
    pieces, bases = [], []
    while True:
        last = n - base < W + M
        n_local = n - base if last else W + M
        local = np.ascontiguousarray(data[base:base + n_local])
        link, handoff = _Link(), C.c_uint64(0)
        h = lib.orc_shard_encode(local.ctypes.data_as(C.c_void_p), C.c_uint64(base), C.c_uint64(n_local),
                                 C.c_uint64(n if last else UNKNOWN), level, C.c_int64(hint), 0, THREADS, C.c_uint64(base),
                                 C.c_uint64(n if last else base + W), C.byref(handoff), C.byref(link))
        buf = np.zeros(n_local + n_local // 50 + 100_000, np.uint8)
        off, ln = C.c_uint64(0), C.c_uint64(0)
        rc = lib.orc_shard_finish(C.c_void_p(h), C.c_uint64(bit), C.c_uint32(crc), buf.ctypes.data_as(C.c_void_p), C.c_uint64(buf.size),
                                  C.byref(off), C.byref(ln))
        lib.orc_shard_free(C.c_void_p(h))
        assert rc == 0, rc
        pieces.append((off.value, buf[:ln.value]))
        bases.append(base)
        ph = bit & 7
        k = link.crc_rot[ph] & 31
        crc = ((((crc << k) | (crc >> (32 - k))) & 0xFFFFFFFF) if k else crc) ^ link.crc_fold[ph]
        bit += link.total_bits[ph]
        if last:
            break
        # a window owns at least its first chunk, and every chunk that starts before base + W
        assert base + W <= handoff.value < base + W + M - 4096
        base = handoff.value
    out = np.zeros((bit + 80 + 7) >> 3, np.uint8)
    for off, p in pieces:
        out[off:off + p.size] |= p
    return out.tobytes(), bases


# level 9 needs more than W + M = W + 9 MB to encode a window before the last one
DATA_N = {9: 10_500_000, 1: 2_600_000}


@functools.lru_cache(maxsize=None)
def _data(level):
    # stripes of text / random / sparse: chunks of very different raw sizes, real segmentations
    return corpus.mixed(DATA_N[level], 0x51, 1 << 19)


@functools.lru_cache(maxsize=None)
def _one_shot(level, hint):
    return orc.encode_stream(_data(level), level, hint, want_trace=True, threads=THREADS)


def _hint(kind, n):
    return {"size": n, "unknown": -1, "half": n // 2, "double": 2 * n, "1.1M": 1_100_000}[kind]


@pytest.mark.parametrize("level,W", [(9, 1_000_000), (1, 300_000)])
@pytest.mark.parametrize("hint", ["size", "unknown", "half", "double", "1.1M"])
def test_windows_equal_one_shot(level, W, hint):
    """"1.1M": the last two chunks before the hinted end are balanced (:1416-1424) inside the first window."""
    data = _data(level)
    h = _hint(hint, data.size)
    got, bases = stream_by_windows(data, level, h, W)
    assert len(bases) >= 2
    assert got == _one_shot(level, h)[0]


def test_window_smaller_than_a_chunk():
    """Level 9 with W = 100 000: every window owns only the chunk that starts at its base, longer than W."""
    data = _data(9)
    got, bases = stream_by_windows(data, 9, -1, 100_000)
    assert len(bases) >= 3
    ref, trace = _one_shot(9, -1)
    assert got == ref
    assert bases == [int(t.start) for t in trace[:len(bases)]]


@pytest.mark.parametrize("level", [9, 1])
@pytest.mark.parametrize("delta", [-1, 0, 1])
def test_window_end_on_a_chunk_start(level, delta):
    """own_end of the first window exactly on a chunk start of the one-shot encode, and one byte either side."""
    data = _data(level)
    ref, trace = _one_shot(level, -1)
    W = int(trace[1].start) + delta
    got, bases = stream_by_windows(data, level, -1, W)
    assert got == ref
    assert bases[1] == min(int(t.start) for t in trace if int(t.start) >= W)


def test_empty_and_tiny_streams():
    for data in (np.zeros(0, np.uint8), np.frombuffer(b"x", np.uint8)):
        for hint in (-1, data.size):
            got, bases = stream_by_windows(data, 9, hint, 1 << 20)
            assert bases == [0]
            assert got == orc.encode_stream(data, 9, hint)
