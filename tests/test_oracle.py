"""CPU tests of the oracle (the checker itself).  The reference holds no golden encoder bytes
(SURVEY.md §0.5), so the oracle is pinned by independent decoders, by a second literal restatement
for the unique-result steps, by optimality checks, and by regression vectors under tests/golden/."""
import bz2
import hashlib
import json
import math
import os
import subprocess

import numpy as np
import pytest

import datagen
import oracle_lib as orc

HERE = os.path.dirname(os.path.abspath(__file__))


def _rt(data, level=9, hint=None, mode=0):
    data = bytes(data)
    s = orc.encode_stream(data, level, len(data) if hint is None else hint, mode)
    assert bz2.decompress(s) == data
    return s


@pytest.mark.parametrize("level", [1, 4, 9])
def test_roundtrip_libbz2_levels(level):
    for gen in (lambda: datagen.text(150_000, 1), lambda: datagen.random_bytes(60_000, 2), lambda: datagen.sparse_binary(200_000, 3)):
        s = _rt(gen().tobytes(), level)
        assert s[:4] == b"BZh" + bytes([48 + level])


def test_roundtrip_sizes_around_powers_of_two():
    # shape of the reference's test/several_sizes.adb:77-89 (sizes 0..126 and 2^k +- few)
    base = datagen.text(70_000, 4).tobytes()
    for n in list(range(1, 40)) + [63, 64, 65, 255, 256, 257, 4095, 4096, 4097, 65535, 65536, 65537]:
        _rt(base[:n])


def test_roundtrip_fuzz_slices_patches_noise():
    # shape of the reference's fuzzer test/fuzzip.adb:121-198, fixed seed
    rng = np.random.default_rng(228)
    base = datagen.text(40_000, 5)
    for it in range(25):
        a = base.copy()
        kind = it % 3
        if kind == 0:
            lo = int(rng.integers(0, a.size - 10)); hi = int(rng.integers(lo + 1, a.size))
            a = a[lo:hi]
        elif kind == 1:
            lo = int(rng.integers(0, a.size - 300))
            a[lo:lo + 300] = rng.integers(0, 256, 300, dtype=np.uint8)
        else:
            idx = rng.integers(0, a.size, 500)
            a[idx] = rng.integers(0, 256, 500, dtype=np.uint8)
        _rt(a.tobytes())


def test_decodes_with_bzip2_binary(tmp_path):
    data = datagen.mixed(600_000, 100_000, 6).tobytes()
    p = tmp_path / "x.bz2"
    p.write_bytes(orc.encode_stream(data, 9, len(data)))
    out = subprocess.run(["bzip2", "-dc", str(p)], stdout=subprocess.PIPE, check=True).stdout
    assert out == data


def test_pathological_blocks_roundtrip():
    # config 4 shapes: all-zero (10x raw cap), short period, long exact repeats
    z = np.zeros(9_500_000, np.uint8)
    s, tr = orc.encode_stream(z, 9, z.size, 0, want_trace=True)
    assert bz2.decompress(s) == z.tobytes()
    assert tr[0].len == 9_000_000           # raw_buf'Last = 10 x capacity (bzip2-encoding.adb:1156-1157, :1187)
    _rt(np.tile(np.frombuffer(b"abc", np.uint8), 100_000).tobytes())
    _rt(np.tile(datagen.random_bytes(20_000, 7), 9).tobytes())
    d = np.concatenate([np.arange(200_000, dtype=np.uint32).astype(np.uint8), np.full(259, 7, np.uint8)])
    _rt(d.tobytes())


def test_empty_input_emits_one_empty_block():
    s = orc.encode_stream(b"", 9, 0)
    # "BZh9", block magic, CRC 0, not randomised, origin 0, empty map, 2 coders, 1 selector ..., footer magic, CRC 0
    assert s[:4] == b"BZh9" and s[4:10] == bytes.fromhex("314159265359") and s[10:14] == b"\0\0\0\0"
    assert bytes.fromhex("177245385090") in bytes(_shift_search(s))


def _shift_search(s):
    # the footer magic is not byte aligned in general; return all 8 bit-shifted views concatenated
    bits = np.unpackbits(np.frombuffer(s, np.uint8))
    out = b""
    for sh in range(8):
        b = bits[sh:]
        b = b[:b.size // 8 * 8]
        out += np.packbits(b).tobytes() + b"|"
    return out


def test_size_hint_changes_last_two_chunks():
    data = datagen.text(1_000_000, 8)
    s1, t1 = orc.encode_stream(data, 9, data.size, 0, want_trace=True)
    s2, t2 = orc.encode_stream(data, 9, -1, 0, want_trace=True)
    assert t1[0].dyn_capacity == 500_000 and len(t1) == 2      # stream_rest / 2 (bzip2-encoding.adb:1424)
    assert t2[0].dyn_capacity == 900_000
    assert bz2.decompress(s1) == bz2.decompress(s2) == data.tobytes()


def test_balance_windows_float32():
    # Float (stream_rest) in Float (cap) * 1.05 .. Float (cap) * 1.30 evaluated in single precision
    assert orc.balance_window(9) == (945_000, 1_170_000)
    assert orc.balance_window(4) == (420_000, 519_999)
    assert orc.balance_window(1) == (105_000, 129_999)


def test_fast_bwt_equals_literal_restatement():
    rng = np.random.default_rng(9)
    cases = [rng.integers(0, k, n, dtype=np.uint8) for k in (1, 2, 3, 256) for n in (1, 2, 3, 7, 8, 9, 64, 500, 3000)]
    cases += [np.tile(np.frombuffer(b"ab", np.uint8), 700), np.tile(np.frombuffer(b"abcab", np.uint8), 300),
              datagen.text(20_000, 10)]
    for d in cases:
        a, oa = orc.bwt(d, 0)
        b, ob = orc.bwt(d, 1)
        assert np.array_equal(a, b) and oa == ob, (d[:20], oa, ob)


def test_stream_fast_equals_faithful_bwt_mode():
    d = datagen.mixed(120_000, 30_000, 11)
    assert orc.encode_stream(d, 9, d.size, 0) == orc.encode_stream(d, 9, d.size, 1)


def _package_merge_cost(freq, limit):
    """Independent (textbook coin-collector) package-merge; returns the optimal total cost."""
    items = sorted(f for f in freq if f > 0)
    n = len(items)
    if n <= 1:
        return sum(items)
    leaves = [(w, (i,)) for i, w in enumerate(items)]
    prev = list(leaves)
    for _ in range(limit - 1):
        pk = [(prev[i][0] + prev[i + 1][0], prev[i][1] + prev[i + 1][1]) for i in range(0, len(prev) - 1, 2)]
        prev = sorted(leaves + pk, key=lambda x: x[0])
    lens = [0] * n
    for w, members in prev[:2 * n - 2]:
        for m in members:
            lens[m] += 1
    return sum(l * w for l, w in zip(lens, items))


LLHC_TABLES = [
    # input tables of the reference's test/test_llhc.adb:15-16 and :46 (it prints lengths, asserts nothing)
    ([10, 30, 12, 5, 17, 20, 17, 0, 20, 0, 15], [4, 5]),
    ([6, 1, 1, 2, 10, 13, 19, 33, 41, 78, 89, 25, 7, 4, 2, 3, 1, 1, 1], [7]),
]


def test_llhc_optimal_and_complete():
    rng = np.random.default_rng(12)
    tables = [(f, ms) for f, ms in LLHC_TABLES]
    for n in (2, 3, 5, 17, 60, 258):
        tables.append((list(rng.integers(0, 50, n)), [15, 17]))
        tables.append((list((rng.pareto(1.0, n) * 10).astype(np.int64) + 1), [15, 16, 17]))
        tables.append(([1] * n, [15]))
    for freq, limits in tables:
        for m in limits:
            nz = sum(1 for f in freq if f > 0)
            if nz > (1 << m):
                continue
            lens = orc.llhc(freq, m)
            assert all((l > 0) == (f > 0) for l, f in zip(lens, freq))
            assert max(lens) <= m
            if nz >= 2:
                assert sum(2.0 ** -int(l) for l in lens if l) == 1.0            # complete prefix code
                assert sum(int(l) * int(f) for l, f in zip(lens, freq)) == _package_merge_cost(freq, m)


def test_canonical_codes_prefix_free():
    lens = orc.llhc([5, 9, 12, 13, 16, 45, 1, 1, 2], 15)
    codes = orc.prepare_codes(lens, 15)
    words = [format(int(c), "0%db" % int(l)) for c, l in zip(codes, lens)]
    for i, a in enumerate(words):
        for j, b in enumerate(words):
            assert i == j or not b.startswith(a)


def test_gnat_heap_sort_tie_order():
    # Hand-derived from the restated algorithm (oracle/b2_oracle.cpp, gnat_constrained_array_sort):
    # three equal keys (index 1,2,3) come out as index 3,1,2.  This pins the restatement, not GNAT.
    k, idx = orc.gnat_sort_pairs([1, 1, 1])
    assert list(idx) == [3, 1, 2]
    rng = np.random.default_rng(13)
    keys = rng.integers(0, 51, 18001)
    k, idx = orc.gnat_sort_pairs(keys)
    assert np.all(np.diff(k) >= 0) and sorted(idx) == list(range(1, 18002))
    assert np.array_equal(keys[idx - 1], k)


def test_segmentation_detects_regime_changes():
    d = np.concatenate([datagen.text(300_000, 14), datagen.random_bytes(300_000, 15), np.zeros(200_000, np.uint8)])
    c1, c2 = orc.segment(d, 0), orc.segment(d, 1)
    assert c1[-1] == d.size and c2[-1] == d.size and len(c1) > 1 and len(c2) > 1
    assert all(b - a > 4000 for a, b in zip(c1[:-2], c1[1:-1])) and all(b - a > 8000 for a, b in zip(c2[:-2], c2[1:-1]))
    assert len(orc.segment(d[:20_000], 0)) == 1          # len <= window + index_threshold: trivial (data_segmentation.adb:58)


def test_entropy_series_is_the_segmentation_sum():
    """orc.entropy_series records the sum of the very run that places the cuts: a literal Python chain of the four
    IEEE adds per step (the reference's order, data_segmentation.adb:63-90) gives it bit for bit, and the threshold
    rule of :91-97 applied to it gives both cut lists."""
    d = np.concatenate([datagen.text(40_000, 21), datagen.random_bytes(30_000, 22), np.zeros(30_000, np.uint8)])
    init, series = orc.entropy_series(d)
    assert series.size == d.size - 16_000
    inv = 1.0 / 16000.0                                     # p = freq * inv_window_size (:44, :49)
    T = [0.0] + [-((c * inv) * math.log(c * inv)) for c in range(1, 16002)]
    f = [0] * 256
    for b in d[:16_000]:
        f[b] += 1
    e = 0.0
    for b in range(256):
        if f[b]:
            e = e + T[f[b]]
    assert e == init
    mine = np.zeros(series.size)
    for k in range(series.size):
        bn, bo = int(d[16_000 + k]), int(d[k])
        e = e - T[f[bn]]
        f[bn] += 1
        e = e + T[f[bn]]
        e = e - T[f[bo]]
        f[bo] -= 1
        e = e + T[f[bo]]
        mine[k] = e
    assert np.array_equal(mine.view(np.uint64), series.view(np.uint64))
    for profile, thr, ith in ((0, 0.6, 4000), (1, 0.4, 8000)):
        thr = float(np.float32(thr))
        cuts, mark, imark = [], init, 1
        if d.size > 16_000 + ith:
            for k, v in enumerate(series):
                sp = k + 1
                if abs(v - mark) > thr and sp - imark > ith:
                    cuts.append(sp)
                    imark, mark = sp, v
        assert cuts + [d.size] == list(orc.segment(d, profile)), profile
    assert orc.entropy_series(d[:20_000])[1].size == 0 and orc.entropy_series(d[:20_001])[1].size == 4_001


def test_crc_is_bzip2_crc():
    # known answer: bzip2's CRC-32 (MSB first) of "123456789" is 0xFC891918
    assert orc.crc32(b"123456789") == 0xFC891918


def test_golden_regression_vectors():
    """Outputs recorded by tests/golden/make_golden.py from this oracle (regression pin; the
    reference has no vectors of its own to check against)."""
    g = json.load(open(os.path.join(HERE, "golden", "oracle_vectors.json")))
    import make_inputs
    for name, rec in g.items():
        data, level, hint = make_inputs.CASES[name]()
        s = orc.encode_stream(data, level, hint)
        assert len(s) == rec["len"] and hashlib.sha256(s).hexdigest() == rec["sha256"], name


def _ref_quick_sort(w, s):
    """Literal restatement of the reference's Quick_sort (huffman-encoding-length_limited_coding.adb:191-223)."""
    def qs(first, n):
        if n < 2:
            return
        p = w[first + n // 2]
        i, j = 0, n - 1
        while True:
            while w[first + i] < p:
                i += 1
            while p < w[first + j]:
                j -= 1
            if i >= j:
                break
            w[first + i], w[first + j] = w[first + j], w[first + i]
            s[first + i], s[first + j] = s[first + j], s[first + i]
            i += 1
            j -= 1
        qs(first, i)
        qs(first + i, n - i)
    qs(0, len(w))


def _forward_package_merge(freq, limit):
    """The formulation the CUDA kernel uses (zip-ada_b200/csrc/b2_entropy.cu, ll_length_limited_warp):
    classic package-merge, package before leaf on equal weight, leaves in Quick_sort order."""
    w = [int(f) for f in freq if f > 0]
    s = [i for i, f in enumerate(freq) if f > 0]
    lens = [0] * len(freq)
    n = len(w)
    if n == 0:
        return lens
    if n == 1:
        lens[s[0]] = 1
        return lens
    _ref_quick_sort(w, s)
    need = 2 * n - 2
    levels, prev = [], None
    for _ in range(limit):
        if prev is None:
            merged = [(x, 0) for x in w]
        else:
            pk = [prev[2 * i][0] + prev[2 * i + 1][0] for i in range(len(prev) // 2)]
            merged, a, b = [], 0, 0
            while len(merged) < need and (a < n or b < len(pk)):
                if a < n and (b >= len(pk) or pk[b] > w[a]):
                    merged.append((w[a], 0)); a += 1
                else:
                    merged.append((pk[b], 1)); b += 1
        levels.append(merged)
        prev = merged
    k, counts = need, []
    for lev in range(limit - 1, -1, -1):
        m = levels[lev][:k]
        a = sum(1 for x in m if x[1] == 0)
        counts.append(a)
        k = 2 * (len(m) - a)
    for i in range(n):
        lens[s[i]] = sum(1 for a in counts if a > i)
    return lens


def test_forward_package_merge_equals_boundary():
    rng = np.random.default_rng(5)
    for trial in range(600):
        n = int(rng.choice([2, 3, 4, 5, 8, 17, 40, 100, 258]))
        kind = trial % 5
        if kind == 0:
            f = rng.integers(0, 4, n)
        elif kind == 1:
            f = rng.integers(1, 3, n)
        elif kind == 2:
            f = (rng.pareto(0.7, n) * 3).astype(np.int64) + 1
        elif kind == 3:
            f = np.where(rng.random(n) < 0.7, 1, rng.integers(1, 1000, n))
        else:
            f = np.where(rng.random(n) < 0.5, 2, rng.integers(1, 50, n) * 2)
        for limit in (15, 16, 17):
            assert list(orc.llhc(f, limit)) == _forward_package_merge(list(f), limit)
    for trial in range(400):          # tight limits
        n = int(rng.integers(2, 40))
        limit = int(rng.integers(max(1, int(np.ceil(np.log2(n)))), 9))
        f = (rng.pareto(0.6, n) * 2).astype(np.int64) + 1
        assert list(orc.llhc(f, limit)) == _forward_package_merge(list(f), limit)
