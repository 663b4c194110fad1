"""Seeded last columns for the direct tests of the move-to-front stage (zip-ada_b200/csrc/b2_mtf.cuh): each family
drives the kernels down the paths it is named for.  `make(name, full)` gives a list of (label, column) blocks: at most
about 140 000 positions each for the host emulation, full block size (900 000) for the device when `full`.

The MTF kernels cut a block into segments of SEG positions and rebuild the list at every segment start p0 by walking
backwards (mtf_build_list): (a) the bytes of the 16-position segment before p0; (b) the 16-masks of the rest of its
256-segment; (c) 256-masks, 32 per step, then a descent into the 16-masks; bytes never seen before p0 are appended in
increasing order (the unseen tail).  k_mtf_seqg<8> / <16> / k_mtf_seq take blocks with <= 64, <= 128 and more bytes
in use; k_rle2 scans tiles of 4 096 positions.  `coverage` restates the order of that walk to count which step finds
each byte; it is a coverage meter only, nothing is compared with it."""
import numpy as np

import corpus
import datagen
import oracle_lib as orc

SEG = 32_768                # B2_MTF_SEG
R2_TILE = 4_096             # tile of k_rle2
FULL = 900_000
CLASSES = {"small": 60, "mid": 120, "big": 250}     # bytes in use: k_mtf_seqg<8>, k_mtf_seqg<16>, k_mtf_seq
ROUTES = ("a", "b", "c1", "cN", "tail")
ROUTE_NAMES = {"a": "step (a), the 16 positions before the segment start", "b": "step (b), a 16-mask of its 256-segment",
               "c1": "the first step (c)", "cN": "a later step (c)", "tail": "the unseen tail (increasing order)"}
# last occurrences before a segment start: around 16, 256, the edges of the first step (c) (256 + 32 * 256) and of
# later ones
DISTANCES = (1, 15, 16, 17, 255, 256, 257, 256 + 32 * 256 - 1, 256 + 32 * 256, 256 + 32 * 256 + 1, 256 + 64 * 256,
             256 + 96 * 256 + 1)


def kernel_class(col):
    k = np.unique(col).size
    return "k_mtf_seqg<8>" if k <= 64 else "k_mtf_seqg<16>" if k <= 128 else "k_mtf_seq"


def _rng(seed):
    return np.random.default_rng(seed)


def _alphabet(rng, k):
    return np.sort(rng.choice(256, k, replace=False)).astype(np.uint8)


def _background(rng, alph, n, mean_run=3):
    """Zipf-distributed bytes of alph in geometric runs: the rare ones last occur far back, the frequent ones near."""
    k = alph.size
    w = 1.0 / (1.0 + np.arange(k))
    w = rng.permutation(w / w.sum())
    out = np.empty(0, np.uint8)
    while out.size < n:
        m = n // mean_run + 64
        out = np.concatenate([out, np.repeat(alph[rng.choice(k, m, p=w)], rng.geometric(1.0 / mean_run, m))])
    return out[:n].copy()


def _ensure_all(rng, col, alph, lo=0, hi=None):
    """Every byte of alph in use (at random places of [lo, hi)), so that the block is in the kernel class of alph.size."""
    missing = np.setdiff1d(alph, np.unique(col))
    hi = col.size if hi is None else hi
    if missing.size and hi > lo:
        col[lo + rng.choice(hi - lo, min(missing.size, hi - lo), replace=False)] = missing[:hi - lo]
    return col


def alphabets(full):
    n = FULL if full else 70_000
    out = []
    for k in (1, 2, 3, 63, 64, 65, 127, 128, 129, 255, 256):
        rng = _rng(0x3F00 + k)
        alph = _alphabet(rng, k)
        out.append(("%d bytes" % k, _ensure_all(rng, _background(rng, alph, n), alph)))
    return out


def distances(full):
    """Marker bytes whose last occurrence before every segment start is at one of DISTANCES (rotated per segment), and
    that occur again just after it; one marker only at position 0 and after the first segment start."""
    n = FULL if full else 140_000
    out = []
    for ci, (cls, k) in enumerate(CLASSES.items()):
        rng = _rng(0x3F10 + ci)
        alph = _alphabet(rng, k)
        markers, zero_marker, bg = alph[-len(DISTANCES):], alph[-len(DISTANCES) - 1], alph[:-len(DISTANCES) - 1]
        col = _background(rng, bg, n)
        col[0] = zero_marker
        col[SEG + 200] = zero_marker
        for s, p0 in enumerate(range(SEG, n, SEG)):
            for i, m in enumerate(markers):
                d = DISTANCES[(i + s) % len(DISTANCES)]
                if p0 - d > 0:
                    col[p0 - d] = m
            for i, m in enumerate(rng.permutation(markers)):
                if p0 + 40 + 2 * i < n:
                    col[p0 + 40 + 2 * i] = m
        out.append((cls, _ensure_all(rng, col, alph)))
    return out


def unseen(full):
    """Most used bytes unseen before the first segment start, some first seen after the second, one first seen at the
    block's last position."""
    n = FULL if full else 100_000
    out = []
    for ci, (cls, k) in enumerate(CLASSES.items()):
        rng = _rng(0x3F20 + ci)
        alph = rng.permutation(_alphabet(rng, k))
        last, late, rest = alph[0], alph[1:k // 3], alph[k // 3:]
        col = _background(rng, rest[:2], n)
        col[SEG + 100:] = _background(rng, rest, n - SEG - 100)
        col[2 * SEG + 100:] = _background(rng, np.concatenate([rest, late]), n - 2 * SEG - 100)
        col[2 * SEG + 100:2 * SEG + 100 + late.size] = rng.permutation(late)
        col[-1] = last
        out.append((cls, col))
    return out


LENGTHS = (0, 1, 2, 3, 4, 5, 15, 16, 17, 31, 32, 33, 255, 256, 257, 4_095, 4_096, 4_097, 32_767, 32_768, 32_769,
           65_535, 65_536, 65_537)


def lengths(full):
    out = []
    for ci, (cls, k) in enumerate(CLASSES.items()):
        rng = _rng(0x3F30 + ci)
        alph = _alphabet(rng, k)
        for n in LENGTHS + ((FULL,) if full else ()):
            out.append(("%s, %d positions" % (cls, n), _ensure_all(rng, _background(rng, alph, n), alph)))
    return out


def runs(full):
    """Runs across segment starts and across 32-position steps, a whole segment of one byte, zero runs across a k_rle2
    tile and over two whole tiles; the block starts with its smallest byte (index 0 at position 0) and ends in a zero
    run."""
    n = FULL if full else 140_000
    out = []
    for ci, (cls, k) in enumerate(CLASSES.items()):
        rng = _rng(0x3F40 + ci)
        alph = _alphabet(rng, k)
        col = _ensure_all(rng, _background(rng, alph, n), alph)
        for p0 in range(SEG, n, SEG):
            col[p0 - 20:p0 + 20] = rng.choice(alph)
        for m in range(1, n // 32, 7):
            col[32 * m - 5:32 * m + 5] = rng.choice(alph)
        col[2 * SEG:3 * SEG] = alph[1]
        col[3 * R2_TILE - 7:5 * R2_TILE + 3] = alph[2]
        col[7 * R2_TILE - 50:7 * R2_TILE + 50] = alph[3]
        col[0] = alph[0]
        col[-300:] = alph[4]
        out.append((cls, _ensure_all(rng, col, alph, 100, 3 * R2_TILE - 100)))   # bytes the runs took away
    return out


def places(full):
    """Cycles: every position has the top place of the list (256: index 255; 64, 128: the top place of the small and
    mid classes; 255: the sentinel stays at place 255), reversed cycles, and a cycle through a shuffled alphabet."""
    n = FULL if full else 33_000
    out = []
    for k in (256, 64, 128, 255):
        cyc = np.arange(256 - k, 256, dtype=np.uint8)
        out.append(("cycle of %d" % k, np.resize(cyc, n)))
        out.append(("reversed cycle of %d" % k, np.resize(cyc[::-1].copy(), n)))
    out.append(("shuffled cycle of 256", np.resize(_rng(0x3F50).permutation(256).astype(np.uint8), n)))
    return out


def real(full):
    """The oracle's BWT last columns of text and of a mixed-corpus block."""
    n = FULL if full else 140_000
    text = corpus.markov_text(n)
    mixed = datagen.mixed(n, n // 3, 0x3F70)
    return [("text", orc.encode_block(text, 9)["bwt"]), ("mixed", orc.encode_block(mixed, 9)["bwt"])]


def batch(full):
    """Blocks of the three classes interleaved, with 17, 9 and 5 segments per class against 16, 8 and 4 segments per
    CTA of k_mtf_seqg<8>, k_mtf_seqg<16> and k_mtf_seq: each class has a partial last CTA and groups or warps with no
    segment."""
    if full:
        sizes = {"small": (500_000, 60), "mid": (262_145,), "big": (131_073,)}
    else:
        sizes = {"small": (40_000, 3_000, 60, 70_000, 20_000, 100, 33_000, 5_000, 32_768, 32_769, 300, 9_000),
                 "mid": (40_000, 2_000, 70_000, 130, 32_769), "big": (40_000, 300, 33_000)}
    blocks = {}
    for ci, (cls, k) in enumerate(CLASSES.items()):
        rng = _rng(0x3F60 + ci)
        alph = _alphabet(rng, k)
        blocks[cls] = [("%s, %d positions" % (cls, n), _ensure_all(rng, _background(rng, alph, n), alph)) for n in sizes[cls]]
    out = []
    while any(blocks.values()):
        for cls in CLASSES:
            if blocks[cls]:
                out.append(blocks[cls].pop(0))
    return out


FAMILIES = {"alphabets": alphabets, "distances": distances, "unseen": unseen, "lengths": lengths, "runs": runs,
            "places": places, "real": real, "batch": batch}


def make(name, full=False):
    return [(label, np.ascontiguousarray(col, dtype=np.uint8)) for label, col in FAMILIES[name](full)]


def segments(n):
    return (n + SEG - 1) // SEG


def walk(col, p0):
    """The order of mtf_build_list at segment start p0 > 0: {byte: route} for every byte of col in use, route in
    ROUTES (which step located the 16-segment that holds the byte's last occurrence before p0)."""
    used = np.unique(col)
    last = {}
    for b in used:
        at = np.flatnonzero(col[:p0] == b)
        if at.size:
            last[int(b)] = int(at[-1])
    route = {int(b): "tail" for b in used if int(b) not in last}
    q, first = p0, True
    for s16 in sorted({p >> 4 for p in last.values()}, reverse=True):
        if first and s16 == (p0 >> 4) - 1:
            r = "a"
        else:
            if first:
                q -= 16                            # (a) read the 16-segment before p0 and found nothing new
            if (q & 255) and s16 >= (q >> 8) << 4:
                r = "b"
            else:
                top = q >> 8                      # (c) starts below the 256-segment boundary at or under q
                r = "c1" if (s16 >> 4) >= top - 32 else "cN"
        first = False
        for b, p in last.items():
            if p >> 4 == s16:
                route[b] = r
        q = s16 << 4
    return route


def coverage(col):
    """How many bytes each route found, over the segment starts p0 > 0 of the block."""
    counts = dict.fromkeys(ROUTES, 0)
    for p0 in range(SEG, col.size, SEG):
        for r in walk(col, p0).values():
            counts[r] += 1
    return counts


def describe(col, i):
    """Where the byte at position i came from: its segment, and either its previous occurrence inside the segment or
    the step of the list rebuild that found it."""
    p0 = i // SEG * SEG
    x = int(col[i])
    prev = np.flatnonzero(col[p0:i] == x)
    where = "segment %d (start %d), %s" % (i // SEG, p0, kernel_class(col))
    if prev.size:
        return "%s; byte %d last seen inside the segment at %d" % (where, x, p0 + int(prev[-1]))
    if p0 == 0:
        return "%s; byte %d first seen here (initial list order)" % (where, x)
    return "%s; byte %d found by %s" % (where, x, ROUTE_NAMES[walk(col, p0)[x]])


def compare(label, col, idx, syms, n_mtf, n_groups):
    """None when a block's outputs (index bytes, symbols, n_mtf, n_groups) equal the oracle's literal MTF of col, else
    one line on the first difference."""
    want_syms, want_idx = orc.mtf_rle2(col)
    bad = np.flatnonzero(idx != want_idx)
    if bad.size:
        i = int(bad[0])
        return "%s: index at position %d is %d, expected %d (%d positions differ); %s" % (
            label, i, idx[i], want_idx[i], bad.size, describe(col, i))
    want_groups = 1 + (want_syms.size - 1) // 50                       # selector_count (:968)
    if n_mtf != want_syms.size or n_groups != want_groups:
        return "%s: n_mtf %d, n_groups %d, expected %d, %d" % (label, n_mtf, n_groups, want_syms.size, want_groups)
    bad = np.flatnonzero(syms != want_syms)
    if bad.size:
        k = int(bad[0])
        return "%s: symbol %d is %d, expected %d (the index bytes agree: zero-run coding)" % (label, k, syms[k], want_syms[k])
    return None
