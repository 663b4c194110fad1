#!/usr/bin/env python
"""SHA-256 of the oracle's output for the BASELINE.json workloads -> tests/golden/stream_sha.json.

The oracle (oracle/b2_oracle.cpp, the CPU restatement of the reference) encodes the seeded corpora of
tests/corpus.py chunk-parallel on the host (orc_encode_stream_mt, checked against the sequential
orc_encode_stream by tests/test_oracle.py); bench.py and the -m gpu tests compare the SHA-256 of what the
GPU path wrote with these.  Usage:  python tools/make_golden_sha.py [key ...]   (no key = all missing).
Keys: <workload>:<bytes>:<seed hex>:<level>, the stream is encoded with size_hint = size.
"""
import hashlib
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import corpus
import oracle_lib as orc

OUT = os.path.join(ROOT, "tests", "golden", "stream_sha.json")
MiB = 1 << 20
DEFAULT = [
    "markov:%d:5eed0001:9" % (64 * MiB),        # BASELINE.json configs[0]
    "mixed:%d:5eed0004:9" % (256 * MiB),        # configs[2] shape, test size
    "markov:%d:5eed0001:9" % (1024 * MiB),      # configs[1]
    "mixed:%d:5eed0004:9" % (4096 * MiB),       # configs[2]
    "markov:%d:5eed0001:9" % (2048 * MiB),      # one stream over 2 / 4 / 8 GPUs, 1 GiB per GPU
    "markov:%d:5eed0001:9" % (4096 * MiB),
    "markov:%d:5eed0001:9" % (8192 * MiB),
    "mixed:%d:5eed0004:9" % (4352 * MiB),       # one stream past 2^32 bytes (tests/test_gpu_past_4gib.py)
]


def key_of(workload, nbytes, seed, level):
    return "%s:%d:%x:%d" % (workload, nbytes, seed, level)


def main():
    keys = sys.argv[1:] or DEFAULT
    db = json.load(open(OUT)) if os.path.exists(OUT) else {}
    threads = os.cpu_count() or 1
    for k in keys:
        if k in db:
            continue
        name, nbytes, seed, level = k.split(":")
        nbytes, seed, level = int(nbytes), int(seed, 16), int(level)
        t0 = time.time()
        data = corpus.workload(name, nbytes, seed)
        t1 = time.time()
        out = orc.encode_stream(data, level, nbytes, threads=threads)
        t2 = time.time()
        db = json.load(open(OUT)) if os.path.exists(OUT) else {}
        db[k] = {"sha256": hashlib.sha256(out).hexdigest(), "bytes": len(out),
                 "input_sha256": hashlib.sha256(data.tobytes()).hexdigest(),
                 "oracle_seconds": round(t2 - t1, 1), "threads": threads}
        json.dump(db, open(OUT, "w"), indent=1, sort_keys=True)
        print(k, db[k], "gen %.0fs" % (t1 - t0), flush=True)


if __name__ == "__main__":
    main()
