#!/usr/bin/env python
"""bench.py — BZip2 encode throughput of the b2gpu path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W [--config text|mixed|entries|zipf]     our CUDA path
  python bench.py --impl reference --gpus N ...      the reference's CPU algorithm (oracle port) on the host cores

A "step" is one pass of the hot path over one synthetic input (tests/corpus.py, seeded, integer arithmetic:
the same bytes from numpy and from torch on the GPU):
  text    (default; BASELINE.json configs[1])  ONE stream of N GiB of order-3 Markov text (SURVEY.md §8d),
          `Encode (block_900k, size_hint => size)`.  N = 1: b2_encode_stream(_device) on one handle.  N > 1
          (torchrun, one rank per GPU): the SAME call sharded over the ranks — every rank owns a contiguous
          byte range of the stream (b2_shard_*, zip-ada_b200/sharding.py); two scalar exchanges, no bulk data
          between GPUs; 1 GiB per GPU (weak scaling), the output is one .bz2 stream
  mixed   (configs[2]) ONE 4 GiB stream of 16 MiB stripes {Markov text, random, sparse}, the same stream at
          every N (strong scaling)
  entries (configs[4]) archive of 100 000 entries of 1-64 KiB through b2_zip_create; under torchrun the entries
          are dealt to the ranks (longest first) and every rank writes the archive of its share
  zipf    round 1's friendlier text (Zipf pseudo-words over 30 symbols), kept for comparison
`value` = uncompressed MB/s with the input resident in HBM; `e2e` = the same call with HOST buffers (pinned),
host<->device copies inside the timed region.  Time = wall clock between barriers, max over ranks.
The output of the timed steps is hashed (SHA-256) and compared with the oracle's golden
(tests/golden/stream_sha.json, tools/make_golden_sha.py) and decoded with libbz2, outside the timed region.
--dump-outputs DIR writes what the last timed step returned (rank 0's view) as DIR/<name>.npy, so that two builds can
be compared output for output; see dump_outputs().
"""
import argparse
import bz2
import ctypes as C
import hashlib
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np

MiB = 1 << 20
GiB = 1 << 30
SEEDS = {"markov": 0x5EED0001, "mixed": 0x5EED0004}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for nme, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_LIMIT = 64_000_000     # bytes of all dumped arrays together
DUMP_EDGE = 4096             # leading and trailing rows always dumped: stream header, last block, footer and stream CRC
DUMP_SEED = 0x5EED00D0


def sample_rows(n, n_max, seed=DUMP_SEED):
    """Increasing int64 row numbers of a fixed, seeded sample of n rows: all of them when n <= n_max, else the first and
    last DUMP_EDGE rows and one row at a seeded position in each of n_max equal strata.  They depend on n only, so two
    runs that return the same arrays dump the same sample."""
    if n <= n_max:
        return np.arange(n, dtype=np.int64)
    edges = np.arange(n_max + 1, dtype=np.int64) * n // n_max
    pos = edges[:-1] + (np.random.default_rng(seed).random(n_max) * (edges[1:] - edges[:-1])).astype(np.int64)
    return np.unique(np.concatenate([np.arange(DUMP_EDGE), pos, np.arange(n - DUMP_EDGE, n)]))


def dump_outputs(out_dir, tables):
    """tables: {name: (n_max, {column: 1-D integer array})}, the columns of a table of equal length.  Writes
    out_dir/<name>_length.npy (float64, one element), <name>_positions.npy (float64, the rows of sample_rows(length,
    n_max)) and <name>_<column>.npy for every column at those rows: float32 for bytes, float64 for wider integers
    (exact below 2^53)."""
    out = {}
    for name, (n_max, cols) in tables.items():
        n = len(next(iter(cols.values())))
        pos = sample_rows(n, n_max)
        out[name + "_length"] = np.array([n], np.float64)
        out[name + "_positions"] = pos.astype(np.float64)
        for col, a in cols.items():
            a = np.asarray(a)
            assert a.shape == (n,), (name, col, a.shape)
            out["%s_%s" % (name, col)] = a[pos].astype(np.float32 if a.dtype == np.uint8 else np.float64)
    assert sum(a.nbytes for a in out.values()) <= DUMP_LIMIT, {k: a.nbytes for k, a in out.items()}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return out


def golden(key):
    p = os.path.join(ROOT, "tests", "golden", "stream_sha.json")
    try:
        return json.load(open(p)).get(key)
    except Exception:
        return None


# ---- CPU legs: the oracle (CPU port of the reference's algorithm); the only place bench.py touches oracle/ ----
def cpu_oracle(sample, threads, hint=None, bwt_mode=0):
    """The oracle on one stream with its chunks spread over `threads` host threads (1 = the sequential
    restatement).  Returns (MB/s, seconds, bytes)."""
    import oracle_lib as orc
    orc.lib()
    t0 = time.perf_counter()
    out = orc.encode_stream(sample, 9, sample.size if hint is None else hint, bwt_mode, threads=threads if threads > 1 else 0)
    dt = time.perf_counter() - t0
    return sample.size / 1e6 / dt, dt, out


def cpu_streams(pieces):
    """One independent stream per host thread ('one process per core')."""
    import oracle_lib as orc
    orc.lib()
    res = [None] * len(pieces)

    def work(i):
        res[i] = orc.encode_stream(pieces[i], 9, pieces[i].size)      # ctypes releases the GIL

    t0 = time.perf_counter()
    ths = [threading.Thread(target=work, args=(i,)) for i in range(len(pieces))]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    dt = time.perf_counter() - t0
    return sum(p.size for p in pieces) / 1e6 / dt, dt


def workload_desc(cfg, n, world):
    if cfg == "text":
        return "ONE stream of %d MiB of order-3 Markov text (SURVEY 8d generator, seed 5eed0001), BZip2_3 / block_900k, size_hint = size%s" % (
            n // MiB, "" if world == 1 else ", sharded over %d ranks by byte range (b2_shard_*)" % world)
    if cfg == "mixed":
        return "ONE stream of %d MiB, 16 MiB stripes cycling {Markov text, random bytes, sparse binary} (seed 5eed0004), BZip2_3, size_hint = size%s" % (
            n // MiB, "" if world == 1 else ", sharded over %d ranks by byte range" % world)
    if cfg == "zipf":
        return "%d MiB of Zipf pseudo-word text over 30 symbols (round 1's workload), BZip2_3, size_hint = size" % (n // MiB)
    return cfg


def reference_arm(args, rank, world):
    """--impl reference: the reference is Ada and there is no Ada compiler in this image (DESIGN.md), so the arm
    is the oracle port of its algorithm on the host cores: every step encodes a bounded prefix of the arm's
    workload as ONE stream, its chunks spread over all host threads."""
    if rank != 0:
        return
    import corpus
    cfg = args.config
    threads = os.cpu_count() or 1
    name = {"text": "markov", "mixed": "mixed", "zipf": "markov", "entries": "markov"}[cfg]
    seed = SEEDS[name]
    n_full = stream_size(args, world)
    total_steps = args.warmup + args.steps
    budget_s = 150.0
    # calibrate on one chunk-sized piece, then size the per-step sample for the time budget
    probe = corpus.workload(name, 2 * MiB, seed)
    r1, dt1, _ = cpu_oracle(probe, 1)
    per_step = max(8.0, budget_s / max(1, total_steps))
    sample_n = int(min(n_full, max(4 * MiB, r1 * 1e6 * per_step * threads * 0.8)))
    sample_n = max(threads * 2 * MiB, sample_n) if n_full >= threads * 2 * MiB else n_full
    sample = corpus.workload(name, n_full, seed, hi=sample_n)
    vals = []
    for s in range(total_steps):
        mbps, dt, _ = cpu_oracle(sample, threads)
        if s >= args.warmup:
            vals.append((mbps, dt))
        if sum(v[1] for v in vals) > 2 * budget_s:
            break
    v = statistics.mean(x[0] for x in vals)
    ms = 1000 * statistics.mean(x[1] for x in vals)
    # the other CPU modes BASELINE.md lists, each on a small bounded sample
    modes = {"single_thread_MBps": round(r1, 3), "per_thread_MBps_in_this_run": round(v / threads, 3)}
    try:
        four, _, _ = cpu_oracle(sample[:8 * MiB], 4)
        modes["one_stream_4_threads_MBps"] = round(four, 3)           # the reference's own parallelism: 4 tasks per chunk (:1226-1303)
        pcs, _ = cpu_streams([np.ascontiguousarray(x) for x in np.array_split(sample[:threads * 2 * MiB], threads)])
        modes["one_stream_per_thread_MBps"] = round(pcs, 3)
        fa, _, _ = cpu_oracle(sample[:256 * 1024], 1, bwt_mode=1)
        modes["faithful_heap_sort_bwt_single_thread_MBps_256KiB"] = round(fa, 4)   # the reference's own sort (heap sort, O(N) comparator)
        t0 = time.perf_counter()
        subprocess.run(["bzip2", "-9", "-c"], input=sample[:16 * MiB].tobytes(), stdout=subprocess.DEVNULL, check=True)
        modes["usr_bin_bzip2_9_single_thread_MBps (unrelated yardstick, not the reference)"] = round(16 * MiB / 1e6 / (time.perf_counter() - t0), 2)
    except Exception as ex:
        modes["error"] = str(ex)
    sample_desc = ("first %d bytes of the arm's stream (%s) encoded as ONE stream with size_hint = its size, chunks of 900 000 "
                   "post-RLE1 bytes spread over %d host threads; oracle = C++ port of the reference (fast prefix-doubling BWT, "
                   "so faster than the reference's heap sort)" % (sample.size, name, threads))
    config = {"workload": workload_desc(cfg, n_full, world), "stream_bytes": n_full, "reference_arm_sample_bytes": int(sample.size)}
    print(json.dumps({"impl": "reference", "metric": "bzip2_encode_MBps_900k", "value": round(v, 3), "unit": "MB/s", "n_gpus": args.gpus,
                      "steps": len(vals), "warmup": args.warmup, "ms_per_step": round(ms, 1), "higher_is_better": True,
                      "scaling": scaling_of(cfg), "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config,
                      "cpu_baseline": {"value": round(v, 3), "unit": "MB/s", "cores": threads, "kind": "port", "sample": sample_desc, "modes": modes},
                      "e2e": {"value": round(v, 3), "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def scaling_of(cfg):
    return "strong" if cfg == "mixed" else "weak"


def stream_size(args, world):
    if args.size_mb:
        return args.size_mb * MiB
    if args.config == "mixed":
        return 4 * GiB
    return world * GiB


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="text", choices=["text", "mixed", "entries", "zipf"])
    ap.add_argument("--size-mb", type=int, default=0, help="stream size in MiB (default: 1024 per GPU for text, 4096 for mixed)")
    ap.add_argument("--entries", type=int, default=100000)
    ap.add_argument("--cpu-sample-mb", type=float, default=4.0)
    ap.add_argument("--no-decode", action="store_true", help="skip the libbz2 round trip of the output")
    ap.add_argument("--stage-times", action="store_true", help="one extra diagnostic step with per-stage timers")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy "
                    "(float32 / float64; long buffers as a fixed, seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return reference_arm(args, rank, world)

    import torch
    import torch.distributed as dist
    import corpus
    b2 = importlib.import_module("zip-ada_b200")
    sharding = importlib.import_module("zip-ada_b200.sharding")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def maxrank(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sumrank(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    enc = b2.Encoder(b2.block_900k, local_rank)
    enc.set_timing(1)
    if args.config == "entries":
        return run_entries(args, rank, local_rank, world, dev, enc, b2, sharding, barrier, maxrank, sumrank)

    # ---- one stream ------------------------------------------------------------------------------------------
    cfg = args.config
    n = stream_size(args, world)
    if cfg == "zipf":
        import datagen
        name, seed = "zipf", 0x5EED0001
        assert world == 1, "the zipf workload is single-GPU only"
        host_data = datagen.text(n, seed)
        d_in = torch.zeros(n + 256, dtype=torch.uint8, device=dev)
        d_in[:n] = torch.from_numpy(host_data).to(dev)
        bounds, span = [0, n], (0, n)
    else:
        name = {"text": "markov", "mixed": "mixed"}[cfg]
        seed = SEEDS[name]
        if world == 1:
            bounds, span = [0, n], (0, n)
        else:
            bounds, spans = sharding.plan(n, world, 9, b2.lib())
            span = spans[rank]
        lo, hi = span
        d_in = torch.zeros(hi - lo + 256, dtype=torch.uint8, device=dev)
        d_in[:hi - lo] = corpus.workload(name, n, seed, torch, dev, lo=lo, hi=hi)
    lo, hi = span
    n_local = hi - lo
    cap = int(b2.lib().b2_bound(n_local)) + 1024 * (n_local // 40000 + 16)
    d_out = torch.empty(cap, dtype=torch.uint8, device=dev)
    h_in = torch.empty(n_local, dtype=torch.uint8, pin_memory=True)
    h_in.copy_(d_in[:n_local])
    h_out = torch.empty(cap, dtype=torch.uint8, pin_memory=True)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()          # the generator's temporaries go back to the device: the encoder sizes its batches by the free memory
    # the two scalar exchanges of a sharded stream go through the host (gloo): no GPU kernel, no wait for an SM
    comm = sharding.TorchComm(dist, rank, world, None, dist.new_group(backend="gloo")) if world > 1 else None

    phases = []

    def step(device_resident):
        """One Encode of the whole stream; returns this rank's piece (byte offset, length) and the stream length."""
        if world == 1:
            if device_resident:
                ln = enc.encode_device_ptr(d_in.data_ptr(), n, n, d_out.data_ptr(), cap)
            else:
                ln = enc.encode_ptr(h_in.data_ptr(), n, n, h_out.data_ptr(), cap)
            return 0, ln, ln
        r = sharding.encode_sharded(enc, comm, d_in.data_ptr() if device_resident else h_in.data_ptr(), device_resident, n, n, bounds, span,
                                    d_out.data_ptr() if device_resident else h_out.data_ptr(), device_resident, cap)
        phases.append(r["phases_ms"])
        return r["byte_offset"], r["length"], r["total_length"]

    # ---- device-resident ("value") -------------------------------------------------------------------------
    for _ in range(args.warmup):
        piece = step(True)
    barrier()
    enc.reset_stats()
    sampler = ClockSampler(local_rank)
    sampler.start()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        piece = step(True)
    barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    st = enc.stats()
    t_wall = maxrank(wall)
    t_dev = maxrank(st.call_ms / 1000.0)
    value = n * args.steps / 1e6 / t_wall
    dev_piece = d_out[:piece[1]].cpu().numpy().copy()
    shard_phases = None
    if world > 1:
        mine = phases[-1]
        keys = sorted(mine)
        t = torch.tensor([mine[k] for k in keys], dtype=torch.float64, device=dev)
        allp = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allp, t)
        shard_phases = {k: [round(float(a[i]), 1) for a in allp] for i, k in enumerate(keys)}
    # ---- end to end through the C ABI with host buffers ----------------------------------------------------
    e_piece = step(False)
    barrier()
    enc.reset_stats()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e_piece = step(False)
    barrier()
    e_wall = maxrank(time.perf_counter() - t0)
    e2e = n * args.steps / 1e6 / e_wall
    st_e = enc.stats()
    e2e_detail = {"ms_per_step": round(1000 * e_wall / args.steps, 2), "device_event_ms_per_step": round(st_e.call_ms / args.steps, 2),
                  "gpu_launches_per_step": int(st_e.kernel_launches // args.steps), "free_device_GiB": round(torch.cuda.mem_get_info()[0] / 2 ** 30, 1)}
    host_piece = h_out[:e_piece[1]].numpy()
    same_paths = bool(piece == e_piece and np.array_equal(dev_piece, host_piece))
    # ---- statistics over all ranks ----------------------------------------------------------------------------
    tot = {k: sumrank(float(getattr(st, k))) for k in ("scatter_elems", "scatter_ms", "scatter_launches", "sort_elems_round0", "sort_elems_later",
                                                      "sort_ms", "kernel_launches", "blocks", "chunks", "block_bytes", "input_bytes")}
    max_sort_ms = maxrank(st.sort_ms)
    sort_rounds = int(st.sort_rounds)
    h2d = sumrank(float(n_local))
    d2h = sumrank(float(e_piece[1]))
    stage_ms = None
    if args.stage_times and world == 1:
        enc.reset_stats(); enc.set_timing(2)
        step(True)
        s2 = enc.stats()
        stage_ms = dict(zip(["cut_segment", "rle1", "bwt_sort", "mtf_rle2", "entropy_search", "pack", "concat", "copies"],
                            [round(x, 2) for x in s2.stage_ms]))
        stage_ms["scatter_ms"] = round(s2.scatter_ms, 2)
        enc.set_timing(1)
    # ---- the stream the timed steps wrote: assemble on rank 0 (outside the timed region), hash, decode -----------
    total_len = piece[2]
    if world > 1:
        meta = torch.tensor([piece[0], piece[1]], dtype=torch.int64, device=dev)
        metas = [torch.zeros(2, dtype=torch.int64, device=dev) for _ in range(world)]
        dist.all_gather(metas, meta)
        metas = [[int(x) for x in m.tolist()] for m in metas]
        if rank == 0:
            pieces = [(metas[0][0], dev_piece)]
            for r in range(1, world):
                buf = torch.empty(max(1, metas[r][1]), dtype=torch.uint8, device=dev)
                dist.recv(buf, r)
                pieces.append((metas[r][0], buf[:metas[r][1]].cpu().numpy()))
            stream = b2.assemble_pieces(pieces, total_len)
        else:
            buf = d_out[:max(1, piece[1])].contiguous()
            dist.send(buf, 0)
    else:
        stream = dev_piece
    if rank != 0:
        dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"stream": (4 << 20, {"bytes": stream})})
    sha = hashlib.sha256(stream.tobytes()).hexdigest()
    gkey = "%s:%d:%x:9" % (name, n, seed)
    g = golden(gkey)
    parity = {"device_path_equals_host_path": same_paths, "output_sha256": sha, "golden_key": gkey,
              "golden_sha256": g["sha256"] if g else None,
              "timed_output_equals_oracle_golden": (bool(g["sha256"] == sha and g["bytes"] == int(total_len)) if g else None)}
    # the same stream decoded on the device (b2_verify_stream: every block at once, block and stream CRCs, and at
    # N = 1 the bytes against the input)
    try:
        # the encoder's workspace (one batch for the whole call when it fits) stays allocated: the decoder takes smaller
        # waves of blocks when little device memory is left (6 bytes x 900 000 positions per block of a wave)
        if "B2GPU_VERIFY_WAVE" not in os.environ and torch.cuda.mem_get_info()[0] < (24 << 30):
            os.environ["B2GPU_VERIFY_WAVE"] = "512"
        if world == 1:
            vr = enc.verify_ptr(d_out.data_ptr(), True, int(total_len), d_in.data_ptr(), True, n)
        else:
            d_stream = torch.from_numpy(stream).to(dev)
            vr = enc.verify_ptr(d_stream.data_ptr(), True, int(total_len))
            del d_stream
        parity["device_verify"] = {"ok": bool(vr.ok), "blocks": int(vr.blocks), "decoded_bytes": int(vr.decoded_bytes), "ms": round(vr.ms, 1),
                                   "compared_with_input": world == 1, "stream_crc": "%08x" % vr.stored_stream_crc,
                                   "decode_MBps": round(vr.decoded_bytes / 1e6 / max(1e-9, vr.ms / 1000.0), 1)}
    except Exception as ex:
        parity["device_verify"] = {"ok": False, "error": str(ex)}
    decode_thread = None
    if not args.no_decode and n <= 2 * GiB:
        def decode():
            t0 = time.perf_counter()
            try:
                dec = bz2.decompress(stream.tobytes())
                if cfg == "zipf":
                    ok = dec == host_data.tobytes()
                elif world == 1:
                    ok = dec == h_in.numpy().tobytes()
                else:
                    ok = hashlib.sha256(dec).hexdigest() == (g["input_sha256"] if g else None) and len(dec) == n
                parity["libbz2_decodes_timed_output_to_input"] = bool(ok)
            except Exception as ex:
                parity["libbz2_decodes_timed_output_to_input"] = "error: %s" % ex
            parity["decode_seconds"] = round(time.perf_counter() - t0, 1)
        decode_thread = threading.Thread(target=decode)
        decode_thread.start()
    else:
        parity["libbz2_decodes_timed_output_to_input"] = "skipped (output of %d MiB input: SHA-256 against the oracle golden only)" % (n // MiB)
    # ---- roofline -------------------------------------------------------------------------------------------------
    peak, peak_src = hbm_peak()
    alg_bytes = 24.0 * tot["scatter_elems"]          # 8 B key + 4 B index, read once + written once
    achieved = alg_bytes / (tot["scatter_ms"] / 1000.0) / 1e9 if tot["scatter_ms"] > 0 else 0.0
    # SURVEY 8(d) stage figure: (24 p + 12) n per round, summed = 24 * (rows moved by all passes) + 12 * (rows entering all rounds)
    stage_bytes = 24.0 * tot["scatter_elems"] + 12.0 * (tot["sort_elems_round0"] + tot["sort_elems_later"])
    stage_gbs = stage_bytes / (tot["sort_ms"] / 1000.0) / 1e9 if tot["sort_ms"] > 0 else 0.0
    sc_variant = os.environ.get("B2GPU_SCATTER", "53")
    sc_name = "k_scatter" if sc_variant == "1" else ("k_scatter3" if 40 <= int(sc_variant) <= 71 else "k_scatter2") + " (B2GPU_SCATTER = %s)" % sc_variant
    roofline = {"bound": "hbm", "kernel": sc_name + ": one LSD radix pass of the BWT rotation sort (ranking, decoupled look-back and scatter in one kernel)",
                "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                "peak_source": peak_src, "traffic": None,
                "traffic_note": "not measured in this run; ncu --set full of one launch of the kernel: 13.05 GB of DRAM traffic for 11.88 GB algorithmic (1.10 x), profiles/r02c_scatter_ncu_full_summary.md",
                "algorithmic_bytes_per_launch": alg_bytes / max(1, tot["scatter_launches"]),
                "launches": int(tot["scatter_launches"]), "avg_launch_ms": tot["scatter_ms"] / max(1, tot["scatter_launches"]),
                "share_of_step": round(st.scatter_ms / max(1e-9, st.call_ms), 4),
                "sort_stage": {"algorithmic_bytes": stage_bytes, "ms": round(tot["sort_ms"], 2), "achieved": round(stage_gbs, 1),
                               "frac": round(stage_gbs / peak, 4), "share_of_step": round(max_sort_ms / max(1e-9, 1000 * t_dev), 4),
                               "formula": "sum over rounds of (24 p + 12) n = 24 x rows moved by all radix passes + 12 x rows entering all rounds, over the CUDA-event time of the whole sort stage"},
                "sort_elems_round0": int(tot["sort_elems_round0"] // args.steps), "sort_elems_later": int(tot["sort_elems_later"] // args.steps),
                "rows_moved_by_passes": int(tot["scatter_elems"] // args.steps), "sort_rounds_rank0": sort_rounds // args.steps}
    # ---- CPU baseline: oracle port, 1 thread, bounded sample of the same workload ---------------------------------------
    sample_n = int(min(n_local, args.cpu_sample_mb * MiB))
    sample = h_in[:sample_n].numpy()
    mbps, dt, ref_out = cpu_oracle(sample, 1)
    with b2.Encoder(b2.block_900k, local_rank) as enc2:
        gpu_sample = enc2.encode(sample, sample.size).tobytes()
    parity["sample_equals_oracle"] = bool(gpu_sample == ref_out)
    if decode_thread:
        decode_thread.join()
    line = {"metric": "bzip2_encode_MBps_900k", "value": round(value, 2), "unit": "MB/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(1000 * t_wall / args.steps, 2), "higher_is_better": True, "scaling": scaling_of(cfg),
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": workload_desc(cfg, n, world), "knobs": {k: v for k, v in sorted(os.environ.items()) if k.startswith("B2GPU_")}, "stream_bytes": n, "streams": 1, "ranks": world,
                       "bytes_per_rank": [b - a for a, b in zip(bounds, bounds[1:])],
                       "l2": "inputs (>= 0.5 GiB per GPU and step) and sort state are far larger than the 126 MB L2; no flush needed"},
            "device_event_ms_per_step": round(1000 * t_dev / args.steps, 2),
            "e2e": dict({"value": round(e2e, 2), "unit": "MB/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)}, **e2e_detail),
            "gpu_launches": int(tot["kernel_launches"]),
            "roofline": roofline,
            "cpu_baseline": {"value": round(mbps, 3), "unit": "MB/s", "cores": 1, "kind": "port",
                             "sample": "first %.1f MiB of the same stream, oracle (CPU port of the reference algorithm, sequential), %.1f s" % (sample_n / MiB, dt)},
            "clocks": clocks,
            "compressed_bytes": int(total_len), "ratio": round(total_len / n, 4),
            "blocks_per_step": int(tot["blocks"] // args.steps), "chunks_per_step": int(tot["chunks"] // args.steps),
            "sorted_bytes_per_input_byte": round(tot["block_bytes"] / max(1, tot["input_bytes"]), 3),
            "parity": parity}
    if stage_ms:
        line["stage_ms"] = stage_ms
    if shard_phases:
        line["shard_phases_ms_per_rank"] = shard_phases
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_entries(args, rank, local_rank, world, dev, enc, b2, sharding, barrier, maxrank, sumrank):
    """configs[4]: zip_with_many_files-style archive (test/zip_with_many_files.adb:64-71) through b2_zip_create."""
    import torch
    import torch.distributed as dist
    import zipfile
    import io
    import corpus
    n_entries = args.entries
    flat, offs, sizes, kinds = corpus.entries(n_entries)
    mine = sharding.assign_entries([int(s) for s in sizes], world)[rank]
    # this rank's entries, packed
    m_sizes = sizes[mine]
    m_offs = np.zeros(len(mine), np.uint64)
    pos = 0
    for k, i in enumerate(mine):
        m_offs[k] = pos
        pos += (int(sizes[i]) + 15) & ~15
    m_flat = np.zeros(max(pos, 1), np.uint8)
    for k, i in enumerate(mine):
        m_flat[int(m_offs[k]):int(m_offs[k]) + int(sizes[i])] = flat[int(offs[i]):int(offs[i]) + int(sizes[i])]
    names_list = [("entry_%06d.dat" % i).encode() for i in mine]
    name_offs = np.zeros(len(mine) + 1, np.uint32)
    name_offs[1:] = np.cumsum([len(x) for x in names_list])
    names = b"".join(names_list)
    h_flat = torch.from_numpy(m_flat).pin_memory()
    hf = h_flat.numpy()
    nbytes = int(m_sizes.sum())
    for _ in range(max(1, args.warmup)):
        arch, info = enc.zip_create_flat(hf, m_offs, m_sizes, names, name_offs, want_info=True)
    barrier()
    enc.reset_stats()
    sampler = ClockSampler(local_rank)
    sampler.start()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        arch, info = enc.zip_create_flat(hf, m_offs, m_sizes, names, name_offs, want_info=True)
    barrier()
    wall = maxrank(time.perf_counter() - t0)
    clocks = sampler.stop()
    st = enc.stats()
    total_bytes = sumrank(float(nbytes))
    stored = sumrank(float(sum(1 for x in info if x.zip_type == 0)))
    launches = sumrank(float(st.kernel_launches))
    arch_bytes = sumrank(float(arch.size))
    # every rank checks its own archive with an independent reader
    z = zipfile.ZipFile(io.BytesIO(arch.tobytes()))
    ok = z.testzip() is None and len(z.namelist()) == len(mine)
    k = len(mine) // 2
    ok = ok and z.read(names_list[k].decode()) == flat[int(offs[mine[k]]):int(offs[mine[k]]) + int(sizes[mine[k]])].tobytes()
    all_ok = sumrank(1.0 if ok else 0.0) == world
    if rank != 0:
        dist.destroy_process_group()
        return
    if args.dump_outputs:
        # rank 0's archive volume and its entries, in the order of its share
        dump_outputs(args.dump_outputs, {
            "archive": (4 << 20, {"bytes": arch}),
            "entries": (256 << 10, {col: np.array([getattr(x, f) for x in info], np.uint64) for col, f in
                                    (("crc32", "crc32"), ("method", "zip_type"), ("compressed_size", "compressed_size"),
                                     ("header_offset", "local_header_offset"))})})
    mbps = total_bytes * args.steps / 1e6 / wall
    # CPU baseline: the oracle's Zip.Create restatement on a bounded sample of the same entries, 1 thread
    import oracle_lib as orc
    ns = min(150, len(mine))
    ents = [("entry_%06d.dat" % i, flat[int(offs[i]):int(offs[i]) + int(sizes[i])]) for i in mine[:ns]]
    t0 = time.perf_counter()
    ref_arch, _ = orc.zip_create(ents, 9)
    dt = time.perf_counter() - t0
    sample_bytes = sum(e[1].size for e in ents)
    gpu_arch = enc.zip_create(ents)
    line = {"metric": "bzip2_encode_MBps_900k", "value": round(mbps, 2), "unit": "MB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(1000 * wall / args.steps, 2), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic",
            "config": {"workload": "archive of %d entries of 1-64 KiB (3/4 Markov text, 1/4 random; sizes about log-uniform), Zip.Create + BZip2_3 per entry through b2_zip_create%s"
                                   % (n_entries, "" if world == 1 else "; entries dealt to %d ranks, one archive volume per rank" % world),
                       "entries": n_entries, "input_bytes": int(total_bytes)},
            "entries_per_s": round(n_entries * args.steps / wall, 1), "stored_entries": int(stored), "archive_bytes": int(arch_bytes),
            "e2e": {"value": round(mbps, 2), "unit": "MB/s", "h2d_bytes_per_step": int(total_bytes), "d2h_bytes_per_step": int(arch_bytes),
                    "note": "b2_zip_create takes and returns host buffers: the timed call is the end-to-end call"},
            "gpu_launches": int(launches),
            "roofline": None,
            "cpu_baseline": {"value": round(sample_bytes / 1e6 / dt, 3), "unit": "MB/s", "cores": 1, "kind": "port", "entries_per_s": round(ns / dt, 1),
                             "sample": "first %d entries of rank 0's share through the oracle's Zip.Create restatement, %.1f s" % (ns, dt)},
            "clocks": clocks,
            "parity": {"python_zipfile_testzip_all_ranks": bool(all_ok), "sample_archive_equals_oracle": bool(gpu_arch.tobytes() == ref_arch)}}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
