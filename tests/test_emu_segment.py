"""k_segment (the entropy segmentation, zip-ada_b200/csrc/b2_segment.cuh; reference data_segmentation.adb:39-105) on the
host, step by step.  The kernel source is compiled with g++ (-ffp-contract=off) against tests/emu/cuda_emu.h and runs,
unchanged, as one CTA over one chunk of every input family of tests/seg_families.py, with its test taps on.

The running FP64 sum must equal the oracle's literal chain of adds bit for bit after EVERY step: a cut is placed where
|E - mark| > 0.6 / 0.4, so a sum that is off by one ulp can move a cut and change the stream, yet the cut lists of
ordinary inputs do not see such an error.  A failure names the first step that differs and its batch of 256 steps.
Both cut lists must equal the oracle's, and every family must reach the replay paths it exists for (the kernel's own
counters: batches started on one binade, on two binades, failed predictions, batches finished by the literal chain),
so that a family that stops exercising its path fails instead of passing."""
import os
import subprocess

import numpy as np
import pytest

import oracle_lib as orc
import seg_families as sf

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

N = 100_000        # bytes per family: 328 batches of 256 steps
# minimum counts of the kernel's paths per family: one binade, two binades, restarts, literal chain
MIN_PATHS = {
    "markov": (10, 150, 0, 0),
    "random": (300, 0, 0, 0),
    "zeros_sparse": (0, 150, 15, 25),
    "H0.25": (0, 300, 80, 1),
    "H0.5": (0, 300, 150, 5),
    "H1.0": (0, 300, 60, 3),
    "H2.0": (0, 300, 120, 5),
    "H4.0": (0, 300, 300, 12),
    "period16000": (0, 300, 0, 0),
    "ramp": (50, 100, 40, 0),
    "near_1_over_e": (0, 300, 5, 0),
}
PATHS = ("one-binade batches", "two-binade batches", "restarts", "literal-chain batches")


@pytest.fixture(scope="module")
def emulated(tmp_path_factory):
    """Every family through the emulated kernel, all at once (one process per family)."""
    cuda_inc = "/usr/local/cuda/include"
    if not os.path.isdir(cuda_inc):
        pytest.skip("CUDA headers (vector types) not found")
    d = tmp_path_factory.mktemp("emu_segment")
    exe = str(d / "emu_segment")
    subprocess.run(["g++", "-O1", "-std=c++17", "-pthread", "-ffp-contract=off", "-Wno-attributes", "-I", cuda_inc, "-o", exe,
                    os.path.join(ROOT, "tests", "emu", "emu_segment.cpp")], check=True)
    procs = {}
    for name in sf.FAMILIES:
        data = sf.make(name, N)
        path = str(d / name)
        data.tofile(path + ".bin")
        procs[name] = (data, path, subprocess.Popen([exe, path + ".bin", path], stdout=subprocess.PIPE,
                                                    stderr=subprocess.STDOUT, text=True))
    res = {}
    for name, (data, path, p) in procs.items():
        out = p.communicate(timeout=900)[0]
        if p.returncode != 0:
            res[name] = dict(data=data, error=out[-2000:])
            continue
        cuts = np.fromfile(path + ".cuts", np.uint32)
        n0, n1 = int(cuts[0]), int(cuts[1])
        res[name] = dict(data=data, series=np.fromfile(path + ".series", np.float64),
                         cuts=[cuts[2:2 + n0], cuts[2 + n0:2 + n0 + n1]], paths=np.fromfile(path + ".paths", np.uint32))
    return res


@pytest.mark.parametrize("name", list(sf.FAMILIES))
def test_segment_series_emulated(emulated, name):
    r = emulated[name]
    assert "error" not in r, r.get("error")
    data = r["data"]
    _, ref = orc.entropy_series(data)
    assert ref.size == data.size - 16_000
    k = sf.first_difference(r["series"], ref)
    assert k < 0, "%s: %s" % (name, sf.describe_difference(r["series"], ref, k))
    for profile in (0, 1):
        want = orc.segment(data, profile)
        assert np.array_equal(r["cuts"][profile], want), (name, profile, r["cuts"][profile][:8], want[:8])
    for what, got, least in zip(PATHS, r["paths"], MIN_PATHS[name]):
        assert got >= least, "%s: %d %s, expected at least %d (paths %s)" % (name, got, what, least, list(r["paths"]))


def test_family_inputs():
    """What the families are built to contain, checked on the bytes: period 16 000 meets its own outgoing byte at
    every step; the 1/e family has its byte near probability 1/e; the sparse family has windows of pure zeros, whose sum
falls to the rounding residue of the adds before them (about 1e-14, below 2^-12 but not 0)."""
    p = sf.make("period16000", N)
    assert np.array_equal(p[16_000:], p[:-16_000])
    e = sf.make("near_1_over_e", N)
    assert abs(np.mean(e == 0) - np.exp(-1.0)) < 0.01
    z = sf.make("zeros_sparse", N)
    nz = np.flatnonzero(z)
    assert np.diff(nz).max() > 16_000
    _, series = orc.entropy_series(z)
    assert ((series > 0.0) & (series < 2.0 ** -12)).sum() > 1_000 and (series > 0.01).sum() > 10_000
