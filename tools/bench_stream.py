#!/usr/bin/env python
"""One stream fed in pieces (b2_stream_*) against the whole-stream call (b2_encode_stream), from pinned host memory.

For 1 GiB of text and 4 GiB of mixed data (the goldens' corpora, size_hint = size) it times:
  - b2_encode_stream of the whole buffer;
  - the stream API with W = 512 MiB and W = 1 GiB, in writes of 64 MiB and in one write.
Every mode runs on a fresh handle: once to allocate (the device memory it then holds, from cudaMemGetInfo, is its
high-water: the handle's buffers only grow) and then --reps timed runs.  Outputs go to one pinned buffer, each write's
bytes behind the last.  Every output's SHA-256 is checked against tests/golden/stream_sha.json.  Prints one JSON line
with the GPU's name and power limit read in the same run.
"""
import argparse
import ctypes as C
import hashlib
import importlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import corpus

MiB = 1 << 20
CORPORA = [("markov", 1024 * MiB, 0x5EED0001), ("mixed", 4096 * MiB, 0x5EED0004)]


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
        name, power, clk = [x.strip() for x in q.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as ex:                      # the name still comes from the CUDA runtime
        import torch
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unknown (%s)" % ex}


def run_one_shot(b2, enc, src, n, out):
    ln = C.c_uint64(0)
    rc = b2.lib().b2_encode_stream(enc._h, src.data_ptr(), n, n, out.data_ptr(), out.numel(), C.byref(ln))
    if rc:
        raise b2.B2Error(b2.lib().b2_last_error().decode())
    return ln.value


def run_stream(b2, enc, src, n, out, window, write):
    lib = b2.lib()
    ln = C.c_uint64(0)

    def check(rc):
        if rc:
            raise b2.B2Error(lib.b2_last_error().decode())
    check(lib.b2_stream_begin(enc._h, n, window))
    pos = 0
    for i in range(0, n, write):
        k = min(write, n - i)
        cap = out.numel() - pos
        assert cap >= lib.b2_stream_bound(enc._h, k)
        check(lib.b2_stream_write(enc._h, src.data_ptr() + i, k, out.data_ptr() + pos, cap, C.byref(ln)))
        pos += ln.value
    check(lib.b2_stream_end(enc._h, out.data_ptr() + pos, out.numel() - pos, C.byref(ln)))
    return pos + ln.value


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--corpora", default="markov,mixed")
    a = ap.parse_args()
    import torch
    b2 = importlib.import_module("zip-ada_b200")
    golden = json.load(open(os.path.join(ROOT, "tests", "golden", "stream_sha.json")))
    res = dict(gpu_info())
    res["what"] = "uncompressed MB/s (1e6 B), size_hint = size, input and output in pinned host memory; device_GB = device memory held by a fresh handle after the mode ran once"
    res["results"] = []
    modes = [("b2_encode_stream", 0, 0)] + [("stream", w, s) for w in (512 * MiB, 1024 * MiB) for s in (64 * MiB, 0)]
    for name, n, seed in CORPORA:
        if name not in a.corpora.split(","):
            continue
        key = "%s:%d:%x:9" % (name, n, seed)
        src = torch.empty(n, dtype=torch.uint8, pin_memory=True)
        for i in range(0, n, 256 * MiB):
            src[i:i + 256 * MiB].copy_(corpus.workload(name, n, seed, torch, "cuda", lo=i, hi=min(n, i + 256 * MiB)))
        out = torch.empty(int(b2.lib().b2_bound(n)) + 1024 * (n // 40000 + 16) + 2048 * MiB, dtype=torch.uint8, pin_memory=True)
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        for mode, window, write in modes:
            free0 = torch.cuda.mem_get_info()[0]
            with b2.Encoder(9, 0) as enc:
                go = (lambda: run_one_shot(b2, enc, src, n, out)) if mode == "b2_encode_stream" else \
                     (lambda: run_stream(b2, enc, src, n, out, window, write or n))
                ln = go()
                dev = free0 - torch.cuda.mem_get_info()[0]
                ts = []
                for _ in range(a.reps):
                    t0 = time.perf_counter()
                    ln = go()
                    ts.append(time.perf_counter() - t0)
            sha = hashlib.sha256(memoryview(out.numpy()[:ln])).hexdigest()
            r = {"corpus": key, "mode": mode, "MBps": round(n / 1e6 / min(ts), 1), "seconds": [round(t, 3) for t in ts],
                 "device_GB": round(dev / 1e9, 2), "bytes": ln, "equals_golden": sha == golden[key]["sha256"] and ln == golden[key]["bytes"]}
            if mode == "stream":
                r["window_MiB"] = window // MiB
                r["write_MiB"] = (write or n) // MiB
            res["results"].append(r)
            print(json.dumps(r), file=sys.stderr, flush=True)
        del src, out
    res["all_equal_golden"] = all(r["equals_golden"] for r in res["results"])
    print(json.dumps(res))


if __name__ == "__main__":
    main()
