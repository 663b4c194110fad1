"""Stage A7 (move-to-front and zero-run coding, zip-ada_b200/csrc/b2_mtf.cuh; reference bzip2-encoding.adb:318-413) on
the host.  The five kernels (k_mtf_masks, k_mtf_seqg<8>, k_mtf_seqg<16>, k_mtf_seq, k_rle2) are compiled with g++
against tests/emu/cuda_emu.h and run, unchanged, on designed last columns of every family of tests/mtf_families.py: one
batch per family, several CTAs at a time, with the slot padding, the masks and the outputs poisoned first.

The kernels' input is the BWT last column, which no raw input can be designed to give, so the end-to-end tests reach
the list rebuild at segment starts, the top places and the zero-run carries only by chance.  Here the index byte of
every position, the symbols, n_mtf and n_groups must equal the oracle's literal MTF (linear search and shift) of the
same column.  A failure names the block, the first position that differs, its segment and kernel class, and the step
of the list rebuild that found its byte.  Every family must also reach the rebuild steps it exists for (counted by
the restatement of the walk in mtf_families.coverage), so that a family that stops reaching its path fails."""
import os
import subprocess

import numpy as np
import pytest

import mtf_families as mf
import oracle_lib as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WINDOW = 3              # CTAs of a launch in flight at a time

# minimum number of bytes per family that each step of the list rebuild found: a, b, first c, later c, unseen tail
MIN_ROUTES = {
    "alphabets": (40, 800, 150, 0, 0),
    "distances": (40, 600, 150, 12, 0),
    "unseen": (20, 250, 50, 0, 300),
    "lengths": (40, 800, 150, 0, 0),
    "runs": (8, 700, 120, 3, 0),
    "places": (100, 1_000, 0, 0, 0),
    "real": (15, 400, 120, 2, 10),
    "batch": (30, 500, 100, 0, 0),
}


def write_batch(path, cols):
    with open(path, "wb") as f:
        np.array([len(cols)], np.uint32).tofile(f)
        np.array([c.size for c in cols], np.uint32).tofile(f)
        for c in cols:
            c.tofile(f)


@pytest.fixture(scope="module")
def emulated(tmp_path_factory):
    """Every family through the emulated kernels as one batch, all families at once (one process per family)."""
    cuda_inc = "/usr/local/cuda/include"
    if not os.path.isdir(cuda_inc):
        pytest.skip("CUDA headers (vector types) not found")
    d = tmp_path_factory.mktemp("emu_mtf")
    exe = str(d / "emu_mtf")
    subprocess.run(["g++", "-O1", "-std=c++17", "-pthread", "-Wno-attributes", "-I", cuda_inc, "-o", exe,
                    os.path.join(ROOT, "tests", "emu", "emu_mtf.cpp")], check=True)
    procs = {}
    for name in mf.FAMILIES:
        blocks = mf.make(name)
        path = str(d / name)
        write_batch(path + ".bin", [c for _, c in blocks])
        procs[name] = (blocks, path, subprocess.Popen([exe, path + ".bin", path, str(WINDOW)], stdout=subprocess.PIPE,
                                                      stderr=subprocess.STDOUT, text=True))
    res = {}
    for name, (blocks, path, p) in procs.items():
        out = p.communicate(timeout=1800)[0]
        if p.returncode != 0:
            res[name] = dict(blocks=blocks, error=out[-2000:])
            continue
        res[name] = dict(blocks=blocks, idx=np.fromfile(path + ".idx", np.uint8), mtf=np.fromfile(path + ".mtf", np.uint16),
                         info=np.fromfile(path + ".info", np.uint32).reshape(-1, 2))
    return res


@pytest.mark.parametrize("name", list(mf.FAMILIES))
def test_mtf_emulated(emulated, name):
    r = emulated[name]
    assert "error" not in r, r.get("error")
    assert r["info"].shape[0] == len(r["blocks"])
    io = mo = 0
    for j, (label, col) in enumerate(r["blocks"]):
        n_mtf, n_groups = (int(v) for v in r["info"][j])
        msg = mf.compare("%s block %d (%s, %d positions)" % (name, j, label, col.size), col, r["idx"][io:io + col.size],
                      r["mtf"][mo:mo + n_mtf], n_mtf, n_groups)
        assert msg is None, msg
        io += col.size
        mo += n_mtf
    assert io == r["idx"].size and mo == r["mtf"].size


@pytest.mark.parametrize("name", list(mf.FAMILIES))
def test_family_coverage(name):
    """Each family reaches the steps of the list rebuild it is built for (a coverage meter; nothing is compared with
    it), and families a-e have blocks of all three kernel classes."""
    blocks = mf.make(name)
    got = dict.fromkeys(mf.ROUTES, 0)
    for _, col in blocks:
        for k, v in mf.coverage(col).items():
            got[k] += v
    for route, least in zip(mf.ROUTES, MIN_ROUTES[name]):
        assert got[route] >= least, "%s: %d bytes found by %s, expected at least %d (%s)" % (
            name, got[route], mf.ROUTE_NAMES[route], least, got)
    if name in ("alphabets", "distances", "unseen", "lengths", "runs", "batch"):
        assert {mf.kernel_class(c) for _, c in blocks if c.size} == {"k_mtf_seqg<8>", "k_mtf_seqg<16>", "k_mtf_seq"}


def test_family_inputs():
    """What the families are built to contain, checked on the bytes and on the oracle's indices."""
    dist = dict(mf.make("distances"))
    for cls, col in dist.items():
        assert mf.kernel_class(col) == {"small": "k_mtf_seqg<8>", "mid": "k_mtf_seqg<16>", "big": "k_mtf_seq"}[cls]
        routes = mf.walk(col, mf.SEG)
        last = {int(b): int(np.flatnonzero(col[:mf.SEG] == b)[-1]) for b in np.unique(col[:mf.SEG])}
        got = sorted(mf.SEG - p for p in last.values())
        for d in mf.DISTANCES:                  # each designed distance is the last occurrence of a marker
            assert d in got, (cls, d)
        assert mf.SEG in got and routes[int(col[0])] in ("c1", "cN")    # the marker at position 0
        for b, p in last.items():              # the first two steps depend on the distance alone
            if mf.SEG - p <= 16:
                assert routes[b] == "a", (cls, mf.SEG - p)
            elif mf.SEG - p <= 256:
                assert routes[b] == "b", (cls, mf.SEG - p)
    for label, col in mf.make("places"):
        _, idx = orc.mtf_rle2(col)
        k = np.unique(col).size
        if label.startswith("cycle") or label.startswith("shuffled"):
            assert (idx[k:] == k - 1).all(), label          # every position has the top place
    for cls, col in mf.make("runs"):
        _, idx = orc.mtf_rle2(col)
        assert idx[0] == 0 and (idx[-299:] == 0).all()
        assert (idx[3 * mf.R2_TILE:5 * mf.R2_TILE] == 0).all() and idx[5 * mf.R2_TILE:6 * mf.R2_TILE].any()
        assert (idx[2 * mf.SEG + 1:3 * mf.SEG] == 0).all()
    counts = {}
    for label, col in mf.make("batch"):
        c = mf.kernel_class(col)
        counts[c] = counts.get(c, 0) + mf.segments(col.size)
    assert counts == {"k_mtf_seqg<8>": 17, "k_mtf_seqg<16>": 9, "k_mtf_seq": 5}
    assert [c.size for _, c in mf.make("lengths")][:len(mf.LENGTHS)] == list(mf.LENGTHS)


def test_mtf_rle2_is_the_block_path():
    """orc_mtf_rle2 of the oracle's own BWT column gives exactly the symbols of orc_encode_block."""
    for n, data in ((1, b"a"), (5_000, mf.make("alphabets")[4][1][:5_000].tobytes()),
                    (60_000, np.resize(np.frombuffer(b"abracadabra, the quick brown fox ", np.uint8), 60_000)),
                    (80_000, mf.make("real")[1][1][:80_000])):
        o = orc.encode_block(data, 9)
        syms, idx = orc.mtf_rle2(o["bwt"])
        assert np.array_equal(syms, o["mtf"]), n
        assert idx.size == o["bwt"].size
