#!/usr/bin/env python
"""Config-5 shape (BASELINE.json configs[4]): many small archive entries (sizes log-uniform in
1..64 KiB, text and incompressible), every entry its own BZh9 stream, encoded with ONE
b2_encode_batch call.  Prints entries/s and uncompressed MB/s; checks a sample against the oracle.
--zip: the same entries as one archive through b2_zip_create.  --zip --writer W: that archive through the incremental
writer (b2_zip_begin / add / finish, window W bytes, 0 = 512 MiB) against b2_zip_create, each on its own handle, and one archive of
3 x 2 GiB text plus 5 000 small entries through the writer; with the handle's device memory, card and power limit."""
import argparse
import importlib
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import datagen
import oracle_lib as orc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--entries", type=int, default=20000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--zip", action="store_true", help="whole archive through b2_zip_create (headers, CRC-32, store fallback)")
    ap.add_argument("--writer", type=int, default=None, metavar="W", help="with --zip: the incremental writer, window W bytes")
    a = ap.parse_args()
    b2 = importlib.import_module("zip-ada_b200")
    rng = np.random.default_rng(0x5EED0005)
    sizes = (2 ** rng.uniform(10, 16, a.entries)).astype(np.int64)
    total = int(sizes.sum())
    pool_t = datagen.text(8_000_000, 51)
    pool_r = datagen.random_bytes(2_000_000, 52)
    entries = []
    for i, n in enumerate(sizes):
        pool = pool_r if i % 4 == 0 else pool_t
        o = int(rng.integers(0, pool.size - n))
        entries.append(pool[o:o + n])
    if a.zip and a.writer is not None:
        return bench_writer(a, b2, entries, total)
    if a.zip:
        return bench_zip(a, b2, entries, total)
    with b2.Encoder(b2.block_900k, 0) as enc:
        outs = enc.encode_batch(entries, "size")          # warm-up (allocations)
        t0 = time.perf_counter()
        for _ in range(a.reps):
            outs = enc.encode_batch(entries, "size")
        dt = (time.perf_counter() - t0) / a.reps
    ok = all(outs[i] == orc.encode_stream(entries[i], 9, entries[i].size) for i in range(0, a.entries, max(1, a.entries // 40)))
    stored = sum(1 for e, o in zip(entries, outs) if len(o) >= e.size)
    print(json.dumps({"workload": "%d entries, log-uniform 1-64 KiB, 3/4 text 1/4 random, one b2_encode_batch call" % a.entries,
                      "entries_per_s": round(a.entries / dt, 1), "MBps": round(total / 1e6 / dt, 1), "seconds": round(dt, 3),
                      "input_bytes": total, "output_bytes": int(sum(len(o) for o in outs)),
                      "entries_not_smaller_than_input": stored, "sample_equals_oracle": bool(ok)}))


def bench_zip(a, b2, entries, total):
    """Config 5 end to end: one archive, every entry its own BZh9 stream or stored; fixed time stamps."""
    import io
    import zipfile
    named = [("dir%03d/entry%06d.dat" % (i % 251, i), e) for i, e in enumerate(entries)]
    flat, offs, sizes, names, name_offs = orc.pack_entries(named)
    with b2.Encoder(b2.block_900k, 0) as enc:
        arc, info = enc.zip_create_flat(flat, offs, sizes, names, name_offs, want_info=True)      # warm-up
        t0 = time.perf_counter()
        for _ in range(a.reps):
            arc, info = enc.zip_create_flat(flat, offs, sizes, names, name_offs, want_info=True)
        dt = (time.perf_counter() - t0) / a.reps
    z = zipfile.ZipFile(io.BytesIO(arc.tobytes()))
    infos = z.infolist()
    step = max(1, a.entries // 200)
    ok_read = len(infos) == a.entries and all(z.read(infos[i]) == entries[i].tobytes() for i in range(0, a.entries, step))
    k = max(1, a.entries // 40)
    sample = named[::k][:40]
    ok_oracle = enc_sample_equals_oracle(b2, sample)
    print(json.dumps({"workload": "%d entries, log-uniform 1-64 KiB, 3/4 text 1/4 random, one b2_zip_create call (archive in memory)" % a.entries,
                      "entries_per_s": round(a.entries / dt, 1), "MBps": round(total / 1e6 / dt, 1), "seconds": round(dt, 3),
                      "input_bytes": total, "archive_bytes": int(arc.size),
                      "stored_entries": sum(1 for i in info if i.zip_type == 0),
                      "zipfile_reads_back_sample": bool(ok_read), "sample_archive_equals_oracle": bool(ok_oracle)}))


def _card():
    import subprocess
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       stdout=subprocess.PIPE, text=True)
    return r.stdout.strip()


def _write_archive(enc, named, window):
    """-> (archive bytes, seconds)"""
    t0 = time.perf_counter()
    outs = []
    with enc.zip_writer(0, window) as z:
        for name, data in named:
            outs.append(z.add(name, data))
        outs.append(z.finish())
    dt = time.perf_counter() - t0
    return b"".join(outs), dt


def bench_writer(a, b2, entries, total):
    """Config 5 through b2_zip_create and through the writer, each on a handle of its own (device memory per path), then
    a large archive through the writer."""
    import torch
    import corpus
    named = [("dir%03d/entry%06d.dat" % (i % 251, i), e) for i, e in enumerate(entries)]
    flat, offs, sizes, names, name_offs = orc.pack_entries(named)
    res = {"card": _card(), "window": a.writer}

    def fresh():                                          # device memory in use before a new handle
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        return torch.cuda.mem_get_info()[0]
    t = {"writer": [], "zip_create": []}
    mem = {}
    free0 = fresh()
    with b2.Encoder(b2.block_900k, 0) as enc:             # b2_zip_create alone on its handle
        ref = enc.zip_create_flat(flat, offs, sizes, names, name_offs).tobytes()       # warm-up
        for _ in range(a.reps):
            t0 = time.perf_counter()
            enc.zip_create_flat(flat, offs, sizes, names, name_offs)
            t["zip_create"].append(time.perf_counter() - t0)
        mem["zip_create"] = free0 - torch.cuda.mem_get_info()[0]
    free0 = fresh()
    with b2.Encoder(b2.block_900k, 0) as enc:             # the writer alone on its handle
        arc, _ = _write_archive(enc, named, a.writer)     # warm-up
        same = arc == ref
        for _ in range(a.reps):
            t["writer"].append(_write_archive(enc, named, a.writer)[1])
        mem["writer"] = free0 - torch.cuda.mem_get_info()[0]
    for k, v in t.items():
        dt = float(np.median(v))
        res["entries20k_" + k] = {"entries_per_s": round(a.entries / dt, 1), "MBps": round(total / 1e6 / dt, 1),
                                  "seconds": [round(x, 3) for x in v], "device_GB": round(mem[k] / 1e9, 2)}
    res["entries20k_writer_equals_zip_create"] = bool(same)
    text = corpus.workload("markov", 2 << 30, 0x5EED0001, torch, "cuda").cpu().numpy()
    free0 = fresh()
    big = [("text%d.txt" % k, text) for k in range(3)] + named[:5000]
    big_in = 3 * text.size + sum(int(e.size) for _, e in named[:5000])
    with b2.Encoder(b2.block_900k, 0) as enc:
        arc, dt = _write_archive(enc, big, a.writer)
        res["big_writer"] = {"workload": "3 x 2 GiB text + 5000 small entries", "input_bytes": big_in, "archive_bytes": len(arc),
                             "seconds": round(dt, 3), "MBps": round(big_in / 1e6 / dt, 1),
                             "device_GB": round((free0 - torch.cuda.mem_get_info()[0]) / 1e9, 2)}
    print(json.dumps(res))


def enc_sample_equals_oracle(b2, sample):
    with b2.Encoder(b2.block_900k, 0) as enc:
        return enc.zip_create(sample).tobytes() == orc.zip_create(sample, 9)[0]


if __name__ == "__main__":
    main()
