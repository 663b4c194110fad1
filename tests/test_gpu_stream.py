"""One stream fed in pieces: b2_stream_begin / write / end (`-m gpu`).

Every test compares the concatenated outputs of the writes and the end with a reference that the rest of the suite
pins to the oracle: the committed goldens, the oracle itself, or b2_encode_stream of the same bytes and hint.
"""
import ctypes as C
import hashlib
import os
import subprocess

import numpy as np
import pytest

import corpus
import datagen
import oracle_lib as orc
from test_gpu_configs import GOLDEN

pytestmark = pytest.mark.gpu

MiB = 1 << 20
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OK, ERR_ARGUMENT, ERR_OUTPUT_TOO_SMALL, ERR_ABORTED = 0, 1, 2, 12


def _gpu_corpus(name, n, seed):
    import torch
    return corpus.workload(name, n, seed, torch, "cuda").cpu().numpy()


def _sha(b):
    return hashlib.sha256(b).hexdigest()


class Raw:
    """The C calls with their return codes (the Python Stream raises instead)."""

    def __init__(self, b2mod, enc):
        self.lib, self.h = b2mod.lib(), enc._h

    def begin(self, hint, window):
        return self.lib.b2_stream_begin(self.h, int(hint), int(window))

    def bound(self, n):
        return int(self.lib.b2_stream_bound(self.h, n))

    def write(self, a, cap=None):
        """-> (rc, bytes)"""
        a = np.ascontiguousarray(a, np.uint8)
        cap = self.bound(a.size) if cap is None else cap
        out = np.empty(max(cap, 1), np.uint8)
        ln = C.c_uint64(0)
        rc = self.lib.b2_stream_write(self.h, a.ctypes.data if a.size else None, a.size, out.ctypes.data, cap, C.byref(ln))
        return rc, out[:ln.value].tobytes()

    def end(self, cap=None):
        cap = self.bound(0) if cap is None else cap
        out = np.empty(max(cap, 1), np.uint8)
        ln = C.c_uint64(0)
        rc = self.lib.b2_stream_end(self.h, out.ctypes.data, cap, C.byref(ln))
        return rc, out[:ln.value].tobytes()

    def abort(self):
        return self.lib.b2_stream_abort(self.h)


def _write_sizes(n, seed, lo, hi):
    """Seeded write sizes, log-uniform in [lo, hi], covering n."""
    rng = np.random.default_rng(seed)
    sizes, tot = [], 0
    while tot < n:
        s = min(n - tot, int(round(2 ** rng.uniform(np.log2(lo), np.log2(hi)))))
        sizes.append(s)
        tot += s
    return sizes


def stream(enc, data, hint, window, sizes):
    """Python Stream over the write sizes -> (stream bytes, bytes returned before end)."""
    outs, pos = [], 0
    with enc.stream(hint, window) as s:
        for k in sizes:
            outs.append(s.write(data[pos:pos + k]))
            pos += k
        before = sum(len(o) for o in outs)
        outs.append(s.end())
    assert pos == data.size
    return b"".join(outs), before


def _trace_key(t):
    return (t.start, t.len, t.dyn_capacity, t.winner, t.n_seg1, t.n_seg2, tuple(t.bits), tuple(t.bytes))


def _margin(b2mod, level):
    return int(b2mod.lib().b2_shard_margin(level))


@pytest.fixture(scope="module")
def encs(b2mod):
    e = {lv: b2mod.Encoder(lv, 0) for lv in (1, 4, 9)}
    yield e
    for x in e.values():
        x.close()


# ---- 1. goldens ---------------------------------------------------------------------------------------------------
def test_golden_text_64m_random_writes_and_bound(b2mod, encs):
    """64 MiB of text, W = 16 MiB, seeded writes of 1 B .. 8 MiB.  Every 5th write is first offered
    b2_stream_bound - 1 bytes of output: B2_ERR_OUTPUT_TOO_SMALL, nothing taken, and the retry continues the stream."""
    key = "markov:%d:5eed0001:9" % (64 * MiB)
    data = _gpu_corpus("markov", 64 * MiB, 0x5EED0001)
    enc = encs[9]
    raw = Raw(b2mod, enc)
    assert raw.begin(data.size, 16 * MiB) == OK
    outs, pos, refused = [], 0, 0
    for i, k in enumerate(_write_sizes(data.size, 7, 1, 8 * MiB)):
        piece = data[pos:pos + k]
        if i % 5 == 0:
            rc, o = raw.write(piece, raw.bound(k) - 1)
            assert rc == ERR_OUTPUT_TOO_SMALL and o == b""
            refused += 1
        rc, o = raw.write(piece)
        assert rc == OK, b2mod.lib().b2_last_error()
        outs.append(o)
        pos += k
    rc, o = raw.end()
    assert rc == OK
    out = b"".join(outs + [o])
    assert refused >= 3
    assert len(out) == GOLDEN[key]["bytes"] and _sha(out) == GOLDEN[key]["sha256"]
    assert enc.verify(out, data).ok == 1


@pytest.mark.parametrize("writes", ["64MiB", "one"])
def test_golden_mixed_256m(encs, writes):
    key = "mixed:%d:5eed0004:9" % (256 * MiB)
    data = _gpu_corpus("mixed", 256 * MiB, 0x5EED0004)
    sizes = [64 * MiB] * 4 if writes == "64MiB" else [data.size]
    out, _ = stream(encs[9], data, data.size, 64 * MiB, sizes)
    assert len(out) == GOLDEN[key]["bytes"] and _sha(out) == GOLDEN[key]["sha256"]
    assert encs[9].verify(out, data).ok == 1


# ---- 2. one-shot parity ---------------------------------------------------------------------------------------------
PARITY_N = 24_000_000


def _parity_data():
    return corpus.mixed(PARITY_N, 0x61, 1 << 21)


@pytest.mark.parametrize("level", [1, 4, 9])
@pytest.mark.parametrize("hint", ["size", "unknown", "zero", "half", "double"])
@pytest.mark.parametrize("wkind", ["1MiB", "M+1"])
def test_parity_with_one_shot(b2mod, encs, level, hint, wkind):
    data = _parity_data()
    n = data.size
    h = {"size": n, "unknown": -1, "zero": 0, "half": n // 2, "double": 2 * n}[hint]
    W = MiB if wkind == "1MiB" else max(MiB, _margin(b2mod, level) + 1)     # level 1: M + 1 is below the 1 MiB minimum
    enc = encs[level]
    ref = enc.encode(data, h).tobytes()
    ref_trace = [_trace_key(t) for t in enc.trace()]
    out, _ = stream(enc, data, h, W, _write_sizes(n, level * 100 + len(hint), 1000, 4 * MiB))
    assert out == ref
    assert [_trace_key(t) for t in enc.trace()] == ref_trace


@pytest.mark.parametrize("level", [1, 9])
@pytest.mark.parametrize("delta", [-1, 0, 1])
def test_window_end_on_a_one_shot_chunk_start(b2mod, encs, level, delta):
    data = _parity_data()
    enc = encs[level]
    ref = enc.encode(data, -1).tobytes()
    tr = enc.trace()
    k = next(i for i, t in enumerate(tr) if t.start >= MiB)        # W >= 1 MiB
    W = int(tr[k].start) + delta
    out, _ = stream(enc, data, -1, W, [5 * MiB] * (data.size // (5 * MiB)) + [data.size % (5 * MiB)])
    assert out == ref
    assert [_trace_key(t) for t in enc.trace()] == [_trace_key(t) for t in tr]


# ---- 3. edges -----------------------------------------------------------------------------------------------------
def test_edges(b2mod, encs):
    enc = encs[9]
    W = MiB
    WM = W + _margin(b2mod, 9)
    text = corpus.markov_text(WM + 3_000_000, 0x71)
    cases = [
        ("empty", np.zeros(0, np.uint8), [0]),
        ("one byte", np.frombuffer(b"Z", np.uint8), [1]),
        ("W+M-1", text[:WM - 1], [WM - 1]),
        ("W+M: ends right after a window", text[:WM], [WM]),
        ("W+M+1", text[:WM + 1], [WM + 1]),
        ("0-byte writes", text[:WM + 1000], [0, 5000, 0, 0, WM - 5000, 0, 1000, 0]),
        ("1-byte writes across the window boundary", text[:WM + 1_000_000], [WM - 3] + [1] * 7 + [1_000_000 - 4]),
        ("zeros 9 000 000 x 3", np.zeros(27_000_000, np.uint8), [9_000_000] * 3),
        ("random", datagen.random_bytes(12_000_000, 72), [3_000_000] * 4),
    ]
    for name, data, sizes in cases:
        for hint in (-1, data.size):
            ref = enc.encode(data, hint).tobytes()
            out, _ = stream(enc, data, hint, W, sizes)
            assert out == ref, (name, hint)
        if data.size < 100:
            assert out == orc.encode_stream(data, 9, data.size), name


# ---- 4. it streams --------------------------------------------------------------------------------------------------
def test_output_arrives_before_end(encs):
    data = _gpu_corpus("markov", 64 * MiB, 0x5EED0001)
    out, before = stream(encs[9], data, -1, 8 * MiB, [MiB] * 64)
    assert before > len(out) // 2, (before, len(out))
    assert out == encs[9].encode(data, -1).tobytes()


def test_device_memory_of_a_stream_is_a_quarter_of_one_shot(b2mod):
    import torch
    data = _gpu_corpus("mixed", 256 * MiB, 0x5EED0004)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    used = {}
    for mode in ("one-shot", "stream"):
        free0 = torch.cuda.mem_get_info()[0]
        with b2mod.Encoder(9, 0) as e:
            if mode == "one-shot":
                out = e.encode(data, data.size).tobytes()
            else:
                out, _ = stream(e, data, data.size, 16 * MiB, [16 * MiB] * 16)
            used[mode] = free0 - torch.cuda.mem_get_info()[0]      # the handle's buffers only grow: its high-water
        assert _sha(out) == GOLDEN["mixed:%d:5eed0004:9" % (256 * MiB)]["sha256"], mode
    print("device memory: one-shot %.2f GB, stream (W = 16 MiB) %.2f GB" % (used["one-shot"] / 1e9, used["stream"] / 1e9))
    assert used["stream"] * 4 < used["one-shot"], used


# ---- 5. errors ----------------------------------------------------------------------------------------------------
def test_errors_and_calls_refused_mid_stream(b2mod, encs):
    enc = encs[9]
    raw = Raw(b2mod, enc)
    data = corpus.mixed(14_000_000, 0x81, 1 << 20)
    ref = enc.encode(data, -1).tobytes()
    assert raw.write(data[:10])[0] == ERR_ARGUMENT                  # no stream open
    assert raw.end()[0] == ERR_ARGUMENT
    assert raw.begin(-1, MiB - 1) == ERR_ARGUMENT                   # window below 1 MiB
    assert raw.begin(-1, MiB) == OK
    assert raw.begin(-1, MiB) == ERR_ARGUMENT                       # begin twice
    outs = []
    rc, o = raw.write(data[:11_000_000])                            # one window encoded, bytes held
    assert rc == OK and len(o) > 0
    outs.append(o)
    lib = b2mod.lib()
    out = np.empty(1 << 20, np.uint8)
    ln = C.c_uint64(0)
    small = np.frombuffer(b"abc" * 100, np.uint8)
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
    rc, o = raw.write(data[11_000_000:])                            # the stream goes on unharmed
    assert rc == OK
    outs.append(o)
    rc, o = raw.end()
    assert rc == OK
    outs.append(o)
    assert b"".join(outs) == ref
    # abort, then a new begin
    assert raw.begin(-1, MiB) == OK
    assert raw.write(data[:10_500_000])[0] == OK
    assert raw.abort() == OK and raw.abort() == OK
    assert stream(enc, data, -1, MiB, [data.size])[0] == ref
    # destroy with a stream open, then a fresh handle on the same device
    e2 = b2mod.Encoder(9, 0)
    r2 = Raw(b2mod, e2)
    assert r2.begin(-1, MiB) == OK and r2.write(data[:10_500_000])[0] == OK
    e2.close()
    with b2mod.Encoder(9, 0) as e3:
        assert e3.encode(data, -1).tobytes() == ref


# ---- 6. progress and abort --------------------------------------------------------------------------------------------
def test_progress_and_abort_in_the_second_window(b2mod, encs):
    enc = encs[9]
    data = corpus.mixed(30_000_000, 0x91, 1 << 20)
    seen = []
    enc.set_progress(lambda done, total: seen.append((done, total)) and False)
    try:
        out, _ = stream(enc, data, data.size, MiB, [4 * MiB] * 7 + [data.size - 28 * MiB])
        dones = [d for d, _ in seen]
        assert len(seen) >= 3 and dones == sorted(dones) and dones[-1] == data.size
        assert all(t == data.size for _, t in seen)
        assert out == enc.encode(data, data.size).tobytes()
        # abort once the second window reports
        calls = []
        enc.set_progress(lambda done, total: calls.append(done) or len(calls) >= 2)
        raw = Raw(b2mod, enc)
        assert raw.begin(-1, MiB) == OK
        rcs = [raw.write(data[i:i + 4 * MiB])[0] for i in range(0, 28 * MiB, 4 * MiB)]
        assert ERR_ABORTED in rcs
        first = rcs.index(ERR_ABORTED)
        assert all(rc == OK for rc in rcs[:first]) and all(rc == ERR_ARGUMENT for rc in rcs[first + 1:])   # the stream is closed
        assert len(calls) == 2
    finally:
        enc.set_progress(None)
    small = corpus.markov_text(3_000_000, 0x92)
    assert stream(enc, small, -1, MiB, [MiB, MiB, MiB - 1, 1] + [small.size - 3 * MiB])[0] == orc.encode_stream(small, 9, -1)


# ---- 7. two handles ------------------------------------------------------------------------------------------------
def test_two_handles_stream_at_the_same_time(encs):
    a, b = encs[9], encs[4]
    da = corpus.mixed(12_000_000, 0xA1, 1 << 20)
    db = corpus.markov_text(9_000_000, 0xA2)
    sa, sb = a.stream(-1, MiB), b.stream(db.size, MiB)
    oa, ob = [], []
    step = 2 * MiB
    for i in range(0, max(da.size, db.size), step):
        if i < da.size:
            oa.append(sa.write(da[i:i + step]))
        if i < db.size:
            ob.append(sb.write(db[i:i + step]))
    oa.append(sa.end())
    ob.append(sb.end())
    assert b"".join(oa) == orc.encode_stream(da, 9, -1, threads=os.cpu_count() or 4)
    assert b"".join(ob) == orc.encode_stream(db, 4, db.size, threads=os.cpu_count() or 4)


# ---- 8. past 4 GiB --------------------------------------------------------------------------------------------------
def test_past_4gib_from_pinned_memory(b2mod):
    import torch
    from test_gpu_past_4gib import N, KEY, SEED, _mem_available
    free, _ = torch.cuda.mem_get_info()
    if free < 110e9:
        pytest.skip("needs 110 GB of free device memory, %.1f GB free" % (free / 1e9))
    if _mem_available() < 16e9:
        pytest.skip("needs 16 GB of available host memory, %.1f GB available" % (_mem_available() / 1e9))
    src = torch.empty(N, dtype=torch.uint8, pin_memory=True)
    step = 256 * MiB
    for i in range(0, N, step):          # the corpus generated on the device a piece at a time
        src[i:i + step].copy_(corpus.workload("mixed", N, SEED, torch, "cuda", lo=i, hi=min(N, i + step)))
    torch.cuda.empty_cache()
    h = hashlib.sha256()
    total = 0
    with b2mod.Encoder(9, 0) as e:
        with e.stream(N, 1 << 30) as s:
            for i in range(0, N, step):
                o = s.write_ptr(src.data_ptr() + i, min(step, N - i))
                h.update(o)
                total += len(o)
            o = s.end()
            h.update(o)
            total += len(o)
        tr = e.trace()
    assert total == GOLDEN[KEY]["bytes"] and h.hexdigest() == GOLDEN[KEY]["sha256"]
    assert tr[0].start == 0 and all(a.start + a.len == b.start for a, b in zip(tr, tr[1:])) and tr[-1].start + tr[-1].len == N


# ---- 9. hosts -----------------------------------------------------------------------------------------------------
def test_python_stream_exception_leaves_the_handle_usable(encs):
    enc = encs[9]
    data = corpus.mixed(12_000_000, 0xB1, 1 << 20)
    with pytest.raises(ZeroDivisionError):
        with enc.stream(-1, MiB) as s:
            s.write(data[:11_000_000])
            1 / 0
    assert stream(enc, data, -1, MiB, [data.size])[0] == enc.encode(data, -1).tobytes()


def _pipe_exe(tmp_path):
    exe = tmp_path / "test_stream_pipe"
    pkg = os.path.join(ROOT, "zip-ada_b200")
    subprocess.check_call(["g++", "-O2", "-std=c++17", os.path.join(pkg, "host", "test_stream_pipe.cpp"), "-L" + pkg, "-lb2gpu",
                           "-Wl,-rpath," + pkg, "-o", str(exe)])
    return str(exe)


def _pipe(args, data):
    """Feeds `data` to the pipe in 1 MiB pieces; returns (stdout, stderr)."""
    p = subprocess.Popen(args, stdin=subprocess.PIPE, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    import threading
    got = {}
    t = threading.Thread(target=lambda: got.update(out=p.stdout.read()))
    t.start()
    mv = memoryview(np.ascontiguousarray(data))
    for i in range(0, len(mv), MiB):
        p.stdin.write(mv[i:i + MiB])
    p.stdin.close()
    t.join()
    err = p.stderr.read().decode()
    assert p.wait() == 0, err
    return got["out"], err


def test_cpp_stream_pipe(tmp_path, encs):
    exe = _pipe_exe(tmp_path)
    key = "markov:%d:5eed0001:9" % (64 * MiB)
    text = _gpu_corpus("markov", 64 * MiB, 0x5EED0001)
    out, _ = _pipe([exe, str(text.size), str(16 * MiB)], text)               # the golden: the oracle's stream, hint = size
    assert _sha(out) == GOLDEN[key]["sha256"]
    data = _gpu_corpus("mixed", 100_000_000, 0xC1)                           # bzip2_enc on a pipe: no hint
    out, _ = _pipe([exe, "-1"], data)
    assert out == encs[9].encode(data, -1).tobytes()
    small = corpus.mixed(24_000_000, 0xC2, 1 << 20)
    out, err = _pipe([exe, "--throw-after", "1000", "-1", str(MiB)], small)
    assert err.split() == ["created=1", "thrown=1"], err
    assert out == orc.encode_stream(small, 9, -1, threads=os.cpu_count() or 4)
