"""Python host of the b2gpu C ABI (include/b2gpu.h).

Mirrors the reference's operator interface for the BZip2 path: `Encoder(option).encode(data,
size_hint)` is `BZip2.Encoding.Encode (option, size_hint)` (zip_lib/bzip2-encoding.ads:47-56)
with Read_Byte/More_Bytes/Write_Byte replaced by whole buffers; `encode_callbacks` keeps the
three-callback generic shape.  All computing happens in libb2gpu.so (CUDA, sm_100a).  There is no
CPU fallback: if the library or a GPU is missing, construction raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libb2gpu.so")

block_100k, block_400k, block_900k = 1, 4, 9     # Compression_Option (bzip2-encoding.ads:40-43)
unknown_size = -1                                # bzip2-encoding.ads:47


class B2Error(RuntimeError):
    pass


class Stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in
                ("streams", "input_bytes", "chunks", "blocks", "block_bytes", "kernel_launches", "sort_rounds",
                 "sort_elems_round0", "sort_elems_later", "scatter_launches", "scatter_elems")] + \
               [("scatter_ms", C.c_double), ("stage_ms", C.c_double * 8), ("call_ms", C.c_double), ("sort_ms", C.c_double)]


class ZipEntryInfo(C.Structure):
    _fields_ = [("crc32", C.c_uint32), ("zip_type", C.c_uint16), ("reserved", C.c_uint16),
                ("compressed_size", C.c_uint64), ("local_header_offset", C.c_uint64)]


class BlockInfo(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in
                ("n_rle", "origin", "crc", "n_mtf", "eob", "n_used", "n_sel", "ec_count", "max_len",
                 "sample_width", "cost", "pad")] + [("bits", C.c_uint64)]


class VerifyResult(C.Structure):
    _fields_ = [("blocks", C.c_uint64), ("decoded_bytes", C.c_uint64), ("mismatch_at", C.c_uint64), ("candidates", C.c_uint64),
                ("level", C.c_uint32), ("stored_stream_crc", C.c_uint32), ("computed_stream_crc", C.c_uint32), ("ok", C.c_int32),
                ("first_bad_block", C.c_int32), ("first_bad_status", C.c_uint32), ("ms", C.c_double)]


class ShardLink(C.Structure):
    _fields_ = [("total_bits", C.c_uint64 * 8), ("crc_rot", C.c_uint32 * 8), ("crc_fold", C.c_uint32 * 8)]


class ChunkTrace(C.Structure):
    _fields_ = [("start", C.c_uint64), ("len", C.c_uint32), ("dyn_capacity", C.c_uint32),
                ("winner", C.c_int32), ("n_seg1", C.c_uint32), ("n_seg2", C.c_uint32), ("pad", C.c_uint32),
                ("bytes", C.c_uint64 * 4), ("bits", C.c_uint64 * 4)]


PROGRESS_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_uint64, C.c_uint64)

EXPORTS = ["b2_create", "b2_destroy", "b2_bound", "b2_encode_stream", "b2_encode_stream_device", "b2_encode_batch", "b2_last_error",
           "b2_set_timing", "b2_get_stats", "b2_reset_stats", "b2_dbg_block", "b2_get_trace", "b2_get_segments",
           "b2_zip_bound", "b2_zip_create", "b2_zip_crc32",
           "b2_shard_margin", "b2_shard_plan", "b2_shard_open", "b2_shard_cut", "b2_shard_encode", "b2_shard_resolve",
           "b2_shard_finish", "b2_encode_stream_multi", "b2_set_progress", "b2_verify_stream",
           "b2_stream_begin", "b2_stream_bound", "b2_stream_write", "b2_stream_end", "b2_stream_abort", "b2_dbg_segment",
           "b2_zip_begin", "b2_zip_add_bound", "b2_zip_add", "b2_zip_finish_bound", "b2_zip_finish", "b2_zip_abort"]

_lib = None


def lib():
    """Loads libb2gpu.so (built in-tree by __graft_entry__.build()).  Raises if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            raise B2Error("libb2gpu.so is not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(b2gpu has no CPU fallback)")
        _lib = C.CDLL(_SO)
        _lib.b2_bound.restype = C.c_uint64
        _lib.b2_bound.argtypes = [C.c_uint64]
        _lib.b2_last_error.restype = C.c_char_p
        _lib.b2_create.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        _lib.b2_destroy.argtypes = [C.c_void_p]
        _lib.b2_destroy.restype = None
        _lib.b2_encode_stream.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int64, C.c_void_p, C.c_uint64,
                                          C.POINTER(C.c_uint64)]
        _lib.b2_encode_stream_device.argtypes = _lib.b2_encode_stream.argtypes
        _lib.b2_encode_batch.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_uint64, C.c_void_p, C.c_void_p]
        _lib.b2_zip_bound.restype = C.c_uint64
        _lib.b2_zip_bound.argtypes = [C.c_uint32, C.c_uint64, C.c_uint64]
        _lib.b2_zip_create.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_char_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64),
                                       C.c_void_p]
        _lib.b2_zip_begin.argtypes = [C.c_void_p, C.c_int, C.c_uint64]
        _lib.b2_zip_add_bound.restype = C.c_uint64
        _lib.b2_zip_add_bound.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32]
        _lib.b2_zip_add.argtypes = [C.c_void_p, C.c_char_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p,
                                    C.c_uint64, C.POINTER(C.c_uint64)]
        _lib.b2_zip_finish_bound.restype = C.c_uint64
        _lib.b2_zip_finish_bound.argtypes = [C.c_void_p]
        _lib.b2_zip_finish.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64), C.c_void_p, C.c_uint64,
                                       C.POINTER(C.c_uint64)]
        _lib.b2_zip_abort.argtypes = [C.c_void_p]
        _lib.b2_zip_crc32.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint32)]
        _lib.b2_set_timing.argtypes = [C.c_void_p, C.c_int]
        _lib.b2_get_stats.argtypes = [C.c_void_p, C.POINTER(Stats)]
        _lib.b2_reset_stats.argtypes = [C.c_void_p]
        _lib.b2_dbg_block.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32] + [C.c_void_p] * 6 + [C.c_uint64, C.POINTER(BlockInfo)]
        _lib.b2_get_trace.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        _lib.b2_get_segments.argtypes = [C.c_void_p, C.c_uint64, C.c_int, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32)]
        _lib.b2_dbg_segment.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.POINTER(C.c_uint32), C.c_void_p,
                                        C.POINTER(C.c_uint32), C.c_uint32, C.c_void_p, C.c_uint64, C.c_void_p]
        _lib.b2_set_progress.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.b2_verify_stream.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_void_p, C.c_int, C.c_uint64, C.POINTER(VerifyResult)]
        _lib.b2_shard_margin.restype = C.c_uint64
        _lib.b2_shard_margin.argtypes = [C.c_int]
        _lib.b2_shard_plan.argtypes = [C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_void_p]
        _lib.b2_shard_open.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_uint64, C.c_uint64, C.c_uint64, C.c_int64, C.c_uint64]
        _lib.b2_shard_cut.argtypes = [C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        _lib.b2_shard_encode.argtypes = [C.c_void_p, C.POINTER(ShardLink)]
        _lib.b2_shard_resolve.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        _lib.b2_shard_finish.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_void_p, C.c_int, C.c_uint64,
                                         C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint8), C.POINTER(C.c_uint8)]
        _lib.b2_stream_begin.argtypes = [C.c_void_p, C.c_int64, C.c_uint64]
        _lib.b2_stream_bound.restype = C.c_uint64
        _lib.b2_stream_bound.argtypes = [C.c_void_p, C.c_uint64]
        _lib.b2_stream_write.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        _lib.b2_stream_end.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        _lib.b2_stream_abort.argtypes = [C.c_void_p]
        _lib.b2_encode_stream_multi.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.c_int64, C.c_void_p, C.c_uint64,
                                                C.POINTER(C.c_uint64)]
    return _lib


def _check(rc):
    if rc != 0:
        raise B2Error("b2gpu error %d: %s" % (rc, lib().b2_last_error().decode()))


def _u8(buf):
    if isinstance(buf, np.ndarray):
        return np.ascontiguousarray(buf, dtype=np.uint8)
    return np.frombuffer(bytes(buf), dtype=np.uint8)


class Encoder:
    """One encoder handle on one CUDA device."""

    def __init__(self, option=block_900k, device=0):
        self._h = C.c_void_p()
        self.option = option
        _check(lib().b2_create(int(option), int(device), C.byref(self._h)))

    def close(self):
        if self._h:
            lib().b2_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- BZip2.Encoding.Encode (option, size_hint) over whole buffers ---------------------------
    def encode(self, data, size_hint=unknown_size, out=None):
        a = _u8(data)
        n = a.size
        cap = lib().b2_bound(n) + 1024 * (n // 40000 + 16)
        if out is None:
            out = np.empty(cap, dtype=np.uint8)
        out_len = C.c_uint64(0)
        _check(lib().b2_encode_stream(self._h, a.ctypes.data, n, int(size_hint), out.ctypes.data, out.size, C.byref(out_len)))
        return out[:out_len.value]

    def encode_ptr(self, in_ptr, n, size_hint, out_ptr, out_cap):
        """Host pointers (e.g. pinned torch tensors); returns the encoded length."""
        out_len = C.c_uint64(0)
        _check(lib().b2_encode_stream(self._h, in_ptr, n, int(size_hint), out_ptr, out_cap, C.byref(out_len)))
        return out_len.value

    def encode_device_ptr(self, d_in, n, size_hint, d_out, out_cap):
        """Device pointers on this handle's device; returns the encoded length."""
        out_len = C.c_uint64(0)
        _check(lib().b2_encode_stream_device(self._h, d_in, n, int(size_hint), d_out, out_cap, C.byref(out_len)))
        return out_len.value

    def encode_batch(self, entries, size_hints=None):
        """Many independent streams (archive entries) in one call; returns a list of bytes objects.
        size_hints: None (unknown_size for all), "size" (each entry's own size, the Zip.Create route,
        zip-create.adb:256), or a sequence."""
        arrs = [_u8(x) for x in entries]
        n = len(arrs)
        sizes = np.array([a.size for a in arrs], dtype=np.uint64)
        offs = np.zeros(n, dtype=np.uint64)
        pos = 0
        for i, a in enumerate(arrs):
            offs[i] = pos
            pos += (a.size + 15) & ~15
        buf = np.zeros(max(pos, 1), dtype=np.uint8)
        for i, a in enumerate(arrs):
            buf[int(offs[i]):int(offs[i]) + a.size] = a
        if size_hints is None:
            hints = None
        elif isinstance(size_hints, str) and size_hints == "size":
            hints = sizes.astype(np.int64)
        else:
            hints = np.asarray(size_hints, dtype=np.int64)
        cap = int(sum(int(lib().b2_bound(int(s))) + 2048 for s in sizes)) + 64
        out = np.empty(cap, dtype=np.uint8)
        out_offs = np.zeros(max(n, 1), dtype=np.uint64)
        out_lens = np.zeros(max(n, 1), dtype=np.uint64)
        _check(lib().b2_encode_batch(self._h, n, buf.ctypes.data, offs.ctypes.data, sizes.ctypes.data,
                                     hints.ctypes.data if hints is not None else None, out.ctypes.data, cap,
                                     out_offs.ctypes.data, out_lens.ctypes.data))
        return [out[int(out_offs[i]):int(out_offs[i]) + int(out_lens[i])].tobytes() for i in range(n)]

    # -- archive side: Zip.Create for BZip2 entries (zip-create.adb:194-297, :645-756) -------------
    def zip_create(self, entries, dos_times=None, flags=None, duplicates=0, want_info=False):
        """Create_Archive + Add_Stream per entry + Finish in one call.  entries: list of
        (name, bytes-like).  Returns the archive bytes (and the per-entry ZipEntryInfo list)."""
        n = len(entries)
        arrs = [_u8(d) for _, d in entries]
        sizes = np.array([a.size for a in arrs], dtype=np.uint64)
        offs = np.zeros(n, dtype=np.uint64)
        pos = 0
        for i, a in enumerate(arrs):
            offs[i] = pos
            pos += (a.size + 15) & ~15
        buf = np.zeros(max(pos, 1), dtype=np.uint8)
        for i, a in enumerate(arrs):
            buf[int(offs[i]):int(offs[i]) + a.size] = a
        nb = [nm.encode("utf-8") if isinstance(nm, str) else bytes(nm) for nm, _ in entries]
        name_offs = np.zeros(n + 1, dtype=np.uint32)
        if n:
            name_offs[1:] = np.cumsum([len(b) for b in nb])
        names = b"".join(nb)
        return self.zip_create_flat(buf, offs, sizes, names, name_offs, dos_times, flags, duplicates, want_info)

    def zip_create_flat(self, buf, offs, sizes, names, name_offs, dos_times=None, flags=None, duplicates=0, want_info=False):
        """Same, on the flat arrays of the C ABI (no per-entry Python work)."""
        n = int(sizes.size)
        cap = int(lib().b2_zip_bound(n, int(name_offs[-1]), int(sizes.sum())))
        out = np.empty(cap, dtype=np.uint8)
        out_len = C.c_uint64(0)
        t = None if dos_times is None else np.ascontiguousarray(dos_times, dtype=np.uint32)
        f = None if flags is None else np.ascontiguousarray(flags, dtype=np.uint32)
        info = (ZipEntryInfo * max(n, 1))()
        _check(lib().b2_zip_create(self._h, n, buf.ctypes.data, offs.ctypes.data, sizes.ctypes.data, C.c_char_p(names),
                                   name_offs.ctypes.data, None if t is None else t.ctypes.data,
                                   None if f is None else f.ctypes.data, int(duplicates), out.ctypes.data, cap,
                                   C.byref(out_len), info))
        res = out[:out_len.value]
        return (res, [info[i] for i in range(n)]) if want_info else res

    def zip_writer(self, duplicates=0, window=0):
        """Opens an archive on the handle, written entry by entry (b2_zip_begin): `ZipWriter.add` and `ZipWriter.finish`
        return the archive bytes finished so far; together they are `zip_create` of the same entries.  window: entries
        of at most this many bytes are queued and encoded together, larger ones go through windows of this size
        (0 = 512 MiB)."""
        _check(lib().b2_zip_begin(self._h, int(duplicates), int(window)))
        return ZipWriter(self)

    def zip_crc32(self, data):
        """Zip CRC-32 (zip-crc_crypto.adb:31-61) computed on the device."""
        a = _u8(data)
        c = C.c_uint32(0)
        _check(lib().b2_zip_crc32(self._h, a.ctypes.data if a.size else None, a.size, C.byref(c)))
        return int(c.value)

    # -- one stream over several handles (b2_shard_*, include/b2gpu.h) ------------------------------
    def shard_open(self, in_ptr, in_is_device, base, n_local, stream_size, size_hint, own_end):
        _check(lib().b2_shard_open(self._h, in_ptr, int(in_is_device), base, n_local, stream_size, int(size_hint), own_end))

    def shard_cut(self, entry):
        h = C.c_uint64(0)
        _check(lib().b2_shard_cut(self._h, entry, C.byref(h)))
        return h.value

    def shard_encode(self):
        link = ShardLink()
        _check(lib().b2_shard_encode(self._h, C.byref(link)))
        return link

    def shard_finish(self, bit_offset, crc_in, out_ptr, out_is_device, out_cap):
        """Returns (byte offset of the piece in the stream, length, first byte, last byte)."""
        off, ln, fb, lb = C.c_uint64(0), C.c_uint64(0), C.c_uint8(0), C.c_uint8(0)
        _check(lib().b2_shard_finish(self._h, bit_offset, crc_in, out_ptr, int(out_is_device), out_cap, C.byref(off), C.byref(ln),
                                     C.byref(fb), C.byref(lb)))
        return off.value, ln.value, fb.value, lb.value

    # -- one stream fed in pieces (b2_stream_*) --------------------------------------------------
    def stream(self, size_hint=unknown_size, window=0):
        """Opens the handle's stream: `Stream.write(data)` and `Stream.end()` return the bytes that are final so
        far; together they are `encode(all data, size_hint)`.  window: bytes per device window (0 = 512 MiB)."""
        _check(lib().b2_stream_begin(self._h, int(size_hint), int(window)))
        return Stream(self)

    # -- generic shape of the reference: Read_Byte / More_Bytes / Write_Byte --------------------
    def encode_callbacks(self, read_byte, more_bytes, write_byte, size_hint=unknown_size):
        buf = bytearray()
        while more_bytes():
            buf.append(read_byte())
        for b in self.encode(bytes(buf), size_hint).tobytes():
            write_byte(b)

    # -- decode / verify on the device (SURVEY.md 8f row 4) ----------------------------------------
    def verify(self, stream, expect=None):
        """Decodes a BZip2 stream on the device (all blocks at once), checks block and stream CRCs and, when
        `expect` is given, the decoded bytes.  Returns a VerifyResult (`.ok` == 1 when everything agrees)."""
        a = _u8(stream)
        res = VerifyResult()
        if expect is None:
            _check(lib().b2_verify_stream(self._h, a.ctypes.data, 0, a.size, None, 0, 0, C.byref(res)))
        else:
            x = _u8(expect)
            _check(lib().b2_verify_stream(self._h, a.ctypes.data, 0, a.size, x.ctypes.data if x.size else None, 0, x.size, C.byref(res)))
        return res

    def verify_ptr(self, stream_ptr, stream_is_device, n, expect_ptr=None, expect_is_device=False, expect_n=0):
        res = VerifyResult()
        _check(lib().b2_verify_stream(self._h, stream_ptr, int(stream_is_device), n, expect_ptr, int(expect_is_device), expect_n, C.byref(res)))
        return res

    def set_progress(self, fn):
        """fn (done_bytes, total_bytes) -> truthy to abort (B2Error with code 12); None switches it off."""
        if fn is None:
            self._cb = None
            _check(lib().b2_set_progress(self._h, None, None))
            return
        self._cb = PROGRESS_FN(lambda user, done, total: 1 if fn(done, total) else 0)
        _check(lib().b2_set_progress(self._h, C.cast(self._cb, C.c_void_p), None))

    # -- measurement / parity taps ----------------------------------------------------------------
    def set_timing(self, on):
        _check(lib().b2_set_timing(self._h, int(on)))

    def stats(self):
        s = Stats()
        _check(lib().b2_get_stats(self._h, C.byref(s)))
        return s

    def reset_stats(self):
        _check(lib().b2_reset_stats(self._h))

    def trace(self):
        n = C.c_uint64(0)
        _check(lib().b2_get_trace(self._h, None, 0, C.byref(n)))
        arr = (ChunkTrace * max(1, n.value))()
        _check(lib().b2_get_trace(self._h, arr, n.value, C.byref(n)))
        return [arr[i] for i in range(n.value)]

    def segments(self, chunk, profile):
        cuts = np.zeros(2304, np.uint32)
        n = C.c_uint32(0)
        _check(lib().b2_get_segments(self._h, chunk, profile, cuts.ctypes.data, cuts.size, C.byref(n)))
        return cuts[:n.value].copy()

    def dbg_segment(self, data):
        """Segment_by_Entropy of one chunk by the device kernel: dict(cuts=[profile 0, profile 1] as uint32 arrays,
        series=float64 sum after every step (empty when len <= 20 000), paths=uint32[4]: batches started on one
        binade, on two binades, restarts, batches finished by the literal chain)."""
        a = _u8(data)
        cuts = np.zeros((2, 2304), np.uint32)
        n0, n1 = C.c_uint32(0), C.c_uint32(0)
        series = np.zeros(max(a.size - 16_000, 1), np.float64)
        paths = np.zeros(4, np.uint32)
        _check(lib().b2_dbg_segment(self._h, a.ctypes.data, a.size, cuts[0].ctypes.data, C.byref(n0), cuts[1].ctypes.data,
                                    C.byref(n1), cuts.shape[1], series.ctypes.data, series.size, paths.ctypes.data))
        steps = a.size - 16_000 if a.size > 20_000 else 0
        return dict(cuts=[cuts[0, :n0.value].copy(), cuts[1, :n1.value].copy()], series=series[:steps].copy(), paths=paths)

    def dbg_block(self, data):
        a = _u8(data)
        n = a.size
        cap = n * 5 // 4 + 64
        rle = np.zeros(cap, np.uint8)
        bwt = np.zeros(cap, np.uint8)
        mtf = np.zeros(cap + 16, np.uint16)
        sel = np.zeros(18004, np.uint8)
        lens = np.zeros(6 * 258, np.uint8)
        bits = np.zeros(n * 2 + 1_000_000, np.uint8)
        info = BlockInfo()
        _check(lib().b2_dbg_block(self._h, a.ctypes.data, n, rle.ctypes.data, bwt.ctypes.data, mtf.ctypes.data,
                                  sel.ctypes.data, lens.ctypes.data, bits.ctypes.data, bits.size, C.byref(info)))
        return dict(rle=rle[:info.n_rle].copy(), bwt=bwt[:info.n_rle].copy(), mtf=mtf[:info.n_mtf].copy(),
                    sel=sel[:info.n_sel].copy(), lens=lens.reshape(6, 258).copy(),
                    bits=bits[:(info.bits + 7) // 8].copy(), info=info)


class Stream:
    """The open stream of an Encoder (Encoder.stream).  As a context manager it aborts the stream when the block
    raises, so that the handle can encode again."""

    def __init__(self, enc):
        self.enc = enc

    def _run(self, fn, n, *args):
        cap = int(lib().b2_stream_bound(self.enc._h, n))
        out = np.empty(cap, dtype=np.uint8)
        out_len = C.c_uint64(0)
        _check(fn(self.enc._h, *args, out.ctypes.data, cap, C.byref(out_len)))
        return out[:out_len.value].tobytes()

    def write(self, data):
        a = _u8(data)
        return self._run(lib().b2_stream_write, a.size, a.ctypes.data if a.size else None, a.size)

    def write_ptr(self, in_ptr, n):
        """Host pointer (e.g. a pinned torch tensor)."""
        return self._run(lib().b2_stream_write, n, in_ptr, n)

    def end(self):
        return self._run(lib().b2_stream_end, 0)

    def abort(self):
        _check(lib().b2_stream_abort(self.enc._h))

    def __enter__(self):
        return self

    def __exit__(self, exc_type, *a):
        if exc_type is not None:
            self.abort()


class ZipWriter:
    """The open archive of an Encoder (Encoder.zip_writer).  After `finish`, `.info` holds the ZipEntryInfo of every
    entry.  As a context manager it aborts the archive when the block raises, so that the handle can encode again."""

    def __init__(self, enc):
        self.enc = enc
        self.info = None
        self._n = 0                                                      # entries added
        self._out = np.empty(0, dtype=np.uint8)                          # output buffer, reused from call to call

    def _buffer(self, cap):
        if self._out.size < cap:
            self._out = np.empty(cap, dtype=np.uint8)
        return self._out

    def add(self, name, data, dos_time=None, unicode=False, read_only=False):
        """Create.Add_Stream of one whole entry; returns the archive bytes this call finished (often none)."""
        a = _u8(data)
        nb = name.encode("utf-8") if isinstance(name, str) else bytes(name)
        h = self.enc._h
        cap = int(lib().b2_zip_add_bound(h, a.size, len(nb)))
        out = self._buffer(cap)
        out_len = C.c_uint64(0)
        t = 16789 * 65536 if dos_time is None else int(dos_time)         # Zip_Streams.default_time
        fl = (1 if unicode else 0) | (2 if read_only else 0)             # B2_ZIP_UNICODE_NAME, B2_ZIP_READ_ONLY
        _check(lib().b2_zip_add(h, C.c_char_p(nb), len(nb), t, fl, a.ctypes.data if a.size else None, a.size, out.ctypes.data,
                                out.size, C.byref(out_len)))
        self._n += 1
        return out[:out_len.value].tobytes()

    def finish(self):
        h = self.enc._h
        cap = int(lib().b2_zip_finish_bound(h))
        out = self._buffer(cap)
        out_len, n = C.c_uint64(0), C.c_uint64(0)
        info = (ZipEntryInfo * max(self._n, 1))()
        _check(lib().b2_zip_finish(h, out.ctypes.data, out.size, C.byref(out_len), info, self._n, C.byref(n)))
        self._out = np.empty(0, dtype=np.uint8)
        self.info = [info[i] for i in range(n.value)]
        return out[:out_len.value].tobytes()

    def abort(self):
        _check(lib().b2_zip_abort(self.enc._h))

    def __enter__(self):
        return self

    def __exit__(self, exc_type, *a):
        if exc_type is not None:
            self.abort()


def shard_plan(n, n_shards, level=block_900k, stagger_permille=-1):
    b = (C.c_uint64 * (n_shards + 1))()
    _check(lib().b2_shard_plan(n, n_shards, level, stagger_permille, b))
    return [int(x) for x in b]


def shard_resolve(links):
    """links: list of ShardLink in shard order -> (bit_offsets, crcs), n_shards + 1 entries each."""
    n = len(links)
    arr = (ShardLink * n)(*links)
    bo = (C.c_uint64 * (n + 1))()
    cr = (C.c_uint32 * (n + 1))()
    _check(lib().b2_shard_resolve(arr, n, bo, cr))
    return [int(x) for x in bo], [int(x) for x in cr]


def assemble_pieces(pieces, total_len):
    """pieces: list of (byte offset, bytes) in shard order; shared boundary bytes are OR-ed."""
    out = np.zeros(total_len, np.uint8)
    for off, data in pieces:
        a = np.frombuffer(bytes(data), np.uint8) if not isinstance(data, np.ndarray) else data
        if a.size:
            out[off:off + a.size] |= a
    return out


def encode_multi(encoders, data, size_hint=unknown_size, out=None):
    """One stream over the devices of several Encoder handles (b2_encode_stream_multi)."""
    a = _u8(data)
    n = a.size
    cap = lib().b2_bound(n) + 1024 * (n // 40000 + 16)
    if out is None:
        out = np.empty(cap, dtype=np.uint8)
    hs = (C.c_void_p * len(encoders))(*[e._h for e in encoders])
    out_len = C.c_uint64(0)
    _check(lib().b2_encode_stream_multi(hs, len(encoders), a.ctypes.data, n, int(size_hint), out.ctypes.data, out.size, C.byref(out_len)))
    return out[:out_len.value]
