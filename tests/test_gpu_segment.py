"""k_segment (the entropy segmentation, zip-ada_b200/csrc/b2_segment.cuh) on the device, step by step.

b2_dbg_segment runs one chunk through the kernel as one CTA and returns the running FP64 sum after every step, both
cut lists and the replay paths taken.  The sum must equal the oracle's literal chain bit for bit at every step of
every input family of tests/seg_families.py at full size, and at the chunk lengths where the loop starts, where a
profile becomes active and where the last batch of 256 steps is partial or exactly full.  The device build may
contract and schedule code in ways the host emulation (tests/test_emu_segment.py) cannot show.

The production launches (no taps; following the chunk chain on a second stream for one level-9 stream, not following
it for the entries of a batch) must give the oracle's cut lists for every chunk, and the oracle's stream bytes."""
import numpy as np
import pytest

import oracle_lib as orc
import seg_families as sf

pytestmark = pytest.mark.gpu

FULL = 900_000
LOW_ENTROPY = {"zeros_sparse": 9_000_000, "H0.25": 9_000_000, "H0.5": 4_000_000, "period16000": 2_000_000}
# minimum counts of the kernel's paths per family at full size: one binade, two binades, restarts, literal chain
MIN_PATHS = {
    "markov": (150, 2_500, 0, 0),
    "random": (3_454, 0, 0, 0),
    "zeros_sparse": (0, 20_000, 2_000, 4_000),
    "H0.25": (0, 35_000, 3_000, 10),
    "H0.5": (0, 15_000, 3_000, 100),
    "H1.0": (0, 3_400, 500, 20),
    "H2.0": (0, 3_400, 1_000, 40),
    "H4.0": (0, 3_400, 3_000, 100),
    "period16000": (0, 7_750, 0, 0),
    "ramp": (800, 1_500, 40, 0),
    "near_1_over_e": (0, 3_400, 10, 0),
}
PATHS = ("one-binade batches", "two-binade batches", "restarts", "literal-chain batches")


def _check_chunk(enc, data, what, least=(0, 0, 0, 0)):
    r = enc.dbg_segment(data)
    _, ref = orc.entropy_series(data)
    k = sf.first_difference(r["series"], ref)
    assert k < 0, "%s: %s" % (what, sf.describe_difference(r["series"], ref, k))
    for profile in (0, 1):
        want = orc.segment(data, profile)
        assert np.array_equal(r["cuts"][profile], want), (what, profile, r["cuts"][profile][:8], want[:8])
    for name, got, lo in zip(PATHS, r["paths"], least):
        assert got >= lo, "%s: %d %s, expected at least %d (paths %s)" % (what, got, name, lo, list(r["paths"]))
    return r


@pytest.mark.parametrize("name", list(sf.FAMILIES))
def test_segment_series_full_size(enc9, name):
    n = LOW_ENTROPY.get(name, FULL)
    _check_chunk(enc9, sf.make(name, n), "%s, %d bytes" % (name, n), MIN_PATHS[name])


# the loop starts above 20 000 (profile 0) and 24 000 (profile 1) bytes; batches of 256 steps begin at 16 000
EDGES = [16_000, 20_000, 20_001, 24_000, 24_001] + [16_000 + 256 * k + d for k in (20, 300) for d in (-1, 0, 1)] + [9_000_000]


@pytest.mark.parametrize("n", EDGES)
def test_segment_length_edges(enc9, n):
    for name in ("markov", "H1.0"):
        data = sf.make(name, n)
        r = _check_chunk(enc9, data, "%s, %d bytes" % (name, n))
        assert r["series"].size == (n - 16_000 if n > 20_000 else 0)


def test_dbg_segment_arguments(b2mod, enc9):
    with pytest.raises(b2mod.B2Error):
        enc9.dbg_segment(np.zeros(0, np.uint8))
    with pytest.raises(b2mod.B2Error):
        enc9.dbg_segment(np.zeros(9_000_001, np.uint8))
    s = enc9.stream(-1)
    try:
        with pytest.raises(b2mod.B2Error) as ei:
            enc9.dbg_segment(sf.make("markov", 30_000))
        assert "error 1:" in str(ei.value)              # B2_ERR_ARGUMENT while a stream is open
    finally:
        s.abort()
    enc9.dbg_segment(sf.make("markov", 30_000))            # usable again


def _families_concatenated():
    return [sf.make(name, FULL) for name in sf.FAMILIES]


def test_production_launches_follow_chain(enc9):
    """One level-9 stream: k_segment follows the chunk chain on the second stream."""
    parts = _families_concatenated()
    data = np.concatenate(parts)
    out = enc9.encode(data, data.size).tobytes()
    tr = enc9.trace()
    assert len(tr) >= 8
    for c, t in enumerate(tr):
        chunk = data[t.start:t.start + t.len]
        for profile in (0, 1):
            cuts = enc9.segments(c, profile)
            ref = orc.segment(chunk, profile)
            assert np.array_equal(cuts, ref), ("chunk", c, profile, cuts[:8], ref[:8])
    assert out == orc.encode_stream(data, 9, data.size, threads=8)


def test_production_launches_batch(enc9):
    """The same data as the entries of one batch: the chunks are segmented after the cutting, nothing is followed."""
    parts = _families_concatenated()
    outs = enc9.encode_batch(parts, "size")
    tr = enc9.trace()
    entry = -1
    for c, t in enumerate(tr):
        if t.start == 0:
            entry += 1
        chunk = parts[entry][t.start:t.start + t.len]
        for profile in (0, 1):
            cuts = enc9.segments(c, profile)
            ref = orc.segment(chunk, profile)
            assert np.array_equal(cuts, ref), ("entry", entry, "chunk", c, profile, cuts[:8], ref[:8])
    assert entry == len(parts) - 1
    for p, o in zip(parts, outs):
        assert bytes(o) == orc.encode_stream(p, 9, p.size, threads=8)
