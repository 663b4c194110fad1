"""Seeded inputs for the step-by-step tests of the entropy segmentation (k_segment, zip-ada_b200/csrc/b2_segment.cuh):
each family drives the kernel's replay of the running FP64 sum down one of its paths.  `make(name, n)` gives n bytes.

The kernel replays 256 steps at a time: on one binade of the sum (far from its ends), on two binades (an integer map
per add, predicted grid, restarts behind a failed prediction, at most 12), or by the literal chain of adds (sums
below 2^-12, or after 12 restarts).  Window 16 000 bytes; a step adds -T[c], +T[c+1] for the incoming byte and
-T[c'], +T[c'-1] for the outgoing one, T[c] = -(c / 16 000) ln (c / 16 000)."""
import numpy as np

import corpus


def _rng(seed):
    return np.random.default_rng(seed)


def markov(n):
    """Text: one and two binades, many exact ties (terms with few fractional bits on the grid)."""
    return np.ascontiguousarray(corpus.markov_text(n), dtype=np.uint8)


def random(n):
    """Uniform bytes: the sum sits near ln 256 = 5.55, in the middle of [4, 8): one binade, no ties."""
    return _rng(0x5E60).integers(0, 256, n, dtype=np.uint8)


def zeros_sparse(n):
    """Zeros with single non-zero bytes (1 in 300 to 1 in 4 000), and stretches of pure zeros of 20 000 bytes: the
    sum falls to the rounding residue of the adds before (about 1e-14: the literal chain below 2^-12) and
    climbs back through the small binades above it (two binades, many restarts)."""
    rng = _rng(0x5E61)
    out = np.zeros(n, np.uint8)
    pos = 0
    k = 0
    while pos < n:
        if k % 2 == 0:
            ln = min(n - pos, 30_000)
            rate = (300, 1_000, 4_000)[(k // 2) % 3]
            hit = rng.random(ln) < 1.0 / rate
            out[pos:pos + ln][hit] = rng.integers(1, 256, int(hit.sum()), dtype=np.uint8)
        else:
            ln = min(n - pos, 20_000)
        pos += ln
        k += 1
    return out


def stationary(h):
    """A stationary source of entropy h nats: one symbol at probability q, m equal ones sharing 1 - q.  Two binades,
    sums crossing 2^(B+1) inside a batch, many restarts, batches that fall back after 12."""
    m = {0.25: 2, 0.5: 3, 1.0: 6, 2.0: 20, 4.0: 255}[h]
    lo, hi = 1e-9, 1.0 - 1e-9                                 # entropy falls as q rises to 1
    for _ in range(200):
        q = 0.5 * (lo + hi)
        e = -q * np.log(q) - (1 - q) * np.log((1 - q) / m)
        lo, hi = (q, hi) if e > h else (lo, q)
    q = 0.5 * (lo + hi)

    def gen(n):
        rng = _rng(0x5E62 + int(h * 100))
        other = rng.integers(1, m + 1, n, dtype=np.int64)
        return np.where(rng.random(n) < q, 0, other).astype(np.uint8)
    return gen


def period16000(n):
    """A random block of 16 000 bytes over 40 symbols, repeated: the incoming byte equals the outgoing one at every
    step, so every window count is met by both bytes of the step."""
    block = _rng(0x5E63).integers(0, 40, 16_000, dtype=np.uint8)
    return np.tile(block, n // 16_000 + 1)[:n]


def ramp(n):
    """Stripes of 2 000 uniform bytes whose alphabet ramps up from 1 symbol and back down: the sum passes every binade
    from about 2^-3 to 4, on mixed paths.  Alphabets 1, 2, ..., 256, ..., 1 at 1 MB and more; geometric steps below."""
    rng = _rng(0x5E64)
    stripes = n // 2_000 + 1
    if stripes >= 511:
        up = list(range(1, 257))
    else:
        k = (stripes + 1) // 2
        up = sorted(set(int(round(256 ** (i / (k - 1)))) for i in range(k)))
    sizes = up + up[-2::-1]
    parts = [rng.integers(0, a, 2_000, dtype=np.int64) for a in sizes]
    out = np.concatenate(parts).astype(np.uint8)
    return np.resize(out, n) if out.size < n else out[:n]


def near_1_over_e(n):
    """One byte at probability 1/e (its terms are the largest there are, ~0.368) entering and leaving at most steps,
    with 13 equal others (sum ~2.28, 0.28 above the edge 2) and then 3 (sum ~1.35, 0.35 above 1): the sum sits
    closer to a binade edge than the one-binade margin of 0.75, and one term can take it across."""
    rng = _rng(0x5E65)
    half = n // 2
    parts = []
    for m, ln in ((13, half), (3, n - half)):
        other = rng.integers(1, m + 1, ln, dtype=np.int64)
        parts.append(np.where(rng.random(ln) < np.exp(-1.0), 0, other))
    return np.concatenate(parts).astype(np.uint8)


FAMILIES = {
    "markov": markov,
    "random": random,
    "zeros_sparse": zeros_sparse,
    "H0.25": stationary(0.25),
    "H0.5": stationary(0.5),
    "H1.0": stationary(1.0),
    "H2.0": stationary(2.0),
    "H4.0": stationary(4.0),
    "period16000": period16000,
    "ramp": ramp,
    "near_1_over_e": near_1_over_e,
}


def make(name, n):
    return np.ascontiguousarray(FAMILIES[name](n), dtype=np.uint8)


def first_difference(got, want):
    """Index of the first step whose sum differs bit for bit (float64 compared as uint64), or -1; a length difference
    counts at the shorter length."""
    g = np.asarray(got, np.float64).view(np.uint64)
    w = np.asarray(want, np.float64).view(np.uint64)
    k = min(g.size, w.size)
    bad = np.flatnonzero(g[:k] != w[:k])
    if bad.size:
        return int(bad[0])
    return -1 if g.size == w.size else k


def describe_difference(got, want, k):
    """One line on the first differing step k: its batch of 256 steps and the two sums."""
    if k >= min(len(got), len(want)):
        return "series lengths differ: %d steps, expected %d" % (len(got), len(want))
    return ("first difference at step %d (reference i = %d, batch %d, lane %d): got %r (0x%016x), expected %r (0x%016x)"
            % (k, 16_001 + k, k // 256, k % 256, float(got[k]), int(np.float64(got[k]).view(np.uint64)),
               float(want[k]), int(np.float64(want[k]).view(np.uint64))))
