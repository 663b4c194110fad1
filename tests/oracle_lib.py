"""ctypes loader for the oracle (test infrastructure).  See oracle/b2_oracle.cpp."""
import ctypes as C
import os
import subprocess
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_SO = os.path.join(ROOT, "oracle", "libb2oracle.so")


class BlockInfo(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in
                ("n_rle", "origin", "crc", "n_mtf", "eob", "n_used", "n_sel", "ec_count",
                 "max_len", "sample_width", "cost", "constructs")] + [("bits", C.c_uint64)]


class ChunkTrace(C.Structure):
    _fields_ = [("start", C.c_uint64), ("len", C.c_uint32), ("dyn_capacity", C.c_uint32),
                ("winner", C.c_int32), ("n_seg1", C.c_uint32), ("n_seg2", C.c_uint32), ("pad", C.c_uint32),
                ("bytes", C.c_uint64 * 4), ("bits", C.c_uint64 * 4)]


_lib = None


def build():
    srcs = [os.path.join(ROOT, "oracle", f) for f in ("b2_oracle.cpp", "zip_oracle.cpp")]
    if (not os.path.exists(_SO)) or os.path.getmtime(_SO) < max(os.path.getmtime(f) for f in srcs):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle")], stdout=subprocess.DEVNULL)


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_SO)
        _lib.orc_crc32.restype = C.c_uint32
        _lib.orc_zip_crc32.restype = C.c_uint32
    return _lib


def _u8(buf):
    a = np.frombuffer(bytes(buf), dtype=np.uint8) if not isinstance(buf, np.ndarray) else np.ascontiguousarray(buf, dtype=np.uint8)
    return a


def encode_stream(data, level=9, size_hint=-1, bwt_mode=0, want_trace=False, threads=0):
    """threads = 0: the sequential restatement (orc_encode_stream); > 0: orc_encode_stream_mt, the same stream
    with the chunks encoded on that many host threads."""
    a = _u8(data)
    n = a.size
    cap = n + n // 2 + 2_000_000
    out = np.empty(cap, dtype=np.uint8)
    out_len = C.c_uint64(0)
    tcap = n // 50_000 + 16
    trace = (ChunkTrace * tcap)()
    ntr = C.c_uint64(0)
    if threads > 0:
        rc = lib().orc_encode_stream_mt(a.ctypes.data_as(C.c_void_p), C.c_uint64(n), level, C.c_int64(size_hint), bwt_mode, int(threads),
                                        out.ctypes.data_as(C.c_void_p), C.c_uint64(cap), C.byref(out_len),
                                        trace, C.c_uint64(tcap), C.byref(ntr))
    else:
        rc = lib().orc_encode_stream(a.ctypes.data_as(C.c_void_p), C.c_uint64(n), level, C.c_int64(size_hint), bwt_mode,
                                     out.ctypes.data_as(C.c_void_p), C.c_uint64(cap), C.byref(out_len),
                                     trace, C.c_uint64(tcap), C.byref(ntr))
    assert rc == 0, rc
    res = out[:out_len.value].tobytes()
    if want_trace:
        return res, [trace[i] for i in range(ntr.value)]
    return res


def encode_block(data, level=9, bwt_mode=0):
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
    rc = lib().orc_encode_block(a.ctypes.data_as(C.c_void_p), C.c_uint32(n), level, bwt_mode,
                                rle.ctypes.data_as(C.c_void_p), bwt.ctypes.data_as(C.c_void_p),
                                mtf.ctypes.data_as(C.c_void_p), sel.ctypes.data_as(C.c_void_p),
                                lens.ctypes.data_as(C.c_void_p), bits.ctypes.data_as(C.c_void_p),
                                C.c_uint64(bits.size), C.byref(info))
    assert rc == 0, rc
    return dict(rle=rle[:info.n_rle].copy(), bwt=bwt[:info.n_rle].copy(), mtf=mtf[:info.n_mtf].copy(),
                sel=sel[:info.n_sel].copy(), lens=lens.reshape(6, 258).copy(),
                bits=bits[:(info.bits + 7) // 8].copy(), info=info)


def bwt(data, mode=0):
    a = _u8(data)
    out = np.zeros(max(a.size, 1), np.uint8)
    origin = C.c_uint32(0)
    lib().orc_bwt(a.ctypes.data_as(C.c_void_p), C.c_uint32(a.size), mode, out.ctypes.data_as(C.c_void_p), C.byref(origin))
    return out[:a.size], origin.value


def mtf_rle2(col):
    """The reference's MTF_and_RLE_2 (bzip2-encoding.adb:318-413: linear search and shift) of a given last column, with
    in_use taken from its bytes.  Returns (symbols as uint16, including EOB; MTF index of every position as uint8)."""
    a = _u8(col)
    mtf = np.zeros(a.size + 2, np.uint16)
    idx = np.zeros(max(a.size, 1), np.uint8)
    n = C.c_uint32(0)
    rc = lib().orc_mtf_rle2(a.ctypes.data_as(C.c_void_p), C.c_uint32(a.size), mtf.ctypes.data_as(C.c_void_p), C.byref(n),
                            idx.ctypes.data_as(C.c_void_p))
    assert rc == 0, rc
    return mtf[:n.value].copy(), idx[:a.size].copy()


def segment(data, profile):
    a = _u8(data)
    cuts = np.zeros(4096, np.uint32)
    n = C.c_uint32(0)
    rc = lib().orc_segment(a.ctypes.data_as(C.c_void_p), C.c_uint32(a.size), profile,
                           cuts.ctypes.data_as(C.c_void_p), C.c_uint32(cuts.size), C.byref(n))
    assert rc == 0
    return cuts[:n.value].copy()


def entropy_series(data):
    """Segment_by_Entropy's running FP64 sum: (sum after the first 16 000 bytes, float64 array of the sum after every
    later step).  The series is empty when len(data) <= 20 000 (the reference's loop does not run)."""
    a = _u8(data)
    cap = max(a.size - 16_000, 1)
    series = np.zeros(cap, np.float64)
    init = C.c_double(0.0)
    n = C.c_uint64(0)
    rc = lib().orc_entropy_series(a.ctypes.data_as(C.c_void_p), C.c_uint32(a.size), C.byref(init),
                                  series.ctypes.data_as(C.c_void_p), C.c_uint64(cap), C.byref(n))
    assert rc == 0, rc
    return init.value, series[:n.value].copy()


def llhc(freq, max_bits):
    f = np.ascontiguousarray(freq, dtype=np.uint32)
    lens = np.zeros(f.size, np.uint32)
    lib().orc_llhc(f.ctypes.data_as(C.c_void_p), int(f.size), int(max_bits), lens.ctypes.data_as(C.c_void_p))
    return lens


def prepare_codes(lens, max_bits):
    l = np.ascontiguousarray(lens, dtype=np.uint32)
    codes = np.zeros(l.size, np.uint32)
    lib().orc_prepare_codes(l.ctypes.data_as(C.c_void_p), int(l.size), int(max_bits), codes.ctypes.data_as(C.c_void_p))
    return codes


def gnat_sort_pairs(keys):
    k = np.ascontiguousarray(keys, dtype=np.int32).copy()
    idx = np.arange(1, k.size + 1, dtype=np.int32)
    lib().orc_gnat_sort_pairs(k.ctypes.data_as(C.c_void_p), idx.ctypes.data_as(C.c_void_p), C.c_uint32(k.size))
    return k, idx


def crc32(data):
    a = _u8(data)
    return lib().orc_crc32(a.ctypes.data_as(C.c_void_p), C.c_uint64(a.size))


def balance_window(level):
    lo, hi = C.c_int64(0), C.c_int64(0)
    lib().orc_balance_window(level, C.byref(lo), C.byref(hi))
    return lo.value, hi.value


def pack_entries(entries):
    """entries: list of (name, bytes-like).  Returns the flat arrays both archive entry points take."""
    datas = [_u8(d) for _, d in entries]
    sizes = np.array([d.size for d in datas], np.uint64)
    offs = np.zeros(len(entries), np.uint64)
    pos = 0
    for i, d in enumerate(datas):
        offs[i] = pos
        pos += (d.size + 15) & ~15
    flat = np.zeros(max(pos, 1), np.uint8)
    for o, d in zip(offs, datas):
        flat[int(o):int(o) + d.size] = d
    nb = [n.encode("utf-8") if isinstance(n, str) else bytes(n) for n, _ in entries]
    name_offs = np.zeros(len(entries) + 1, np.uint32)
    name_offs[1:] = np.cumsum([len(b) for b in nb])
    names = b"".join(nb)
    return flat, offs, sizes, names, name_offs


def zip_crc32(data):
    a = _u8(data)
    return int(lib().orc_zip_crc32(a.ctypes.data_as(C.c_void_p), C.c_uint64(a.size)))


def zip_create(entries, level=9, dos_times=None, flags=None):
    """Oracle archive (oracle/zip_oracle.cpp): returns (archive bytes, [method per entry])."""
    flat, offs, sizes, names, name_offs = pack_entries(entries)
    n = len(entries)
    cap = int(sizes.sum()) + int(name_offs[-1]) * 2 + n * 124 + 200
    out = np.empty(cap, np.uint8)
    out_len = C.c_uint64(0)
    methods = np.zeros(max(n, 1), np.uint16)
    t = None if dos_times is None else np.ascontiguousarray(dos_times, np.uint32)
    f = None if flags is None else np.ascontiguousarray(flags, np.uint32)
    rc = lib().orc_zip_create(level, C.c_uint32(n), flat.ctypes.data_as(C.c_void_p), offs.ctypes.data_as(C.c_void_p),
                              sizes.ctypes.data_as(C.c_void_p), C.c_char_p(names), name_offs.ctypes.data_as(C.c_void_p),
                              None if t is None else t.ctypes.data_as(C.c_void_p), None if f is None else f.ctypes.data_as(C.c_void_p),
                              out.ctypes.data_as(C.c_void_p), C.c_uint64(cap), C.byref(out_len), methods.ctypes.data_as(C.c_void_p))
    assert rc == 0, rc
    return out[:out_len.value].tobytes(), [int(m) for m in methods[:n]]


def zip_create_given_flat(flat, offs, sizes, names, name_offs, streams, stream_offs, stream_lens, level=9, dos_times=None, flags=None):
    """orc_zip_create_given on the flat arrays (no copy of the inputs): the archive of orc_zip_create with the BZip2
    stream of entry i taken from streams[stream_offs[i]:][:stream_lens[i]] instead of encoded.  An entry whose
    stream_len >= size is stored (pass stream_len = size for one known to be incompressible).
    Returns (archive as a uint8 array, [method per entry])."""
    n = int(sizes.size)
    sizes = np.ascontiguousarray(sizes, np.uint64)
    offs = np.ascontiguousarray(offs, np.uint64)
    so = np.ascontiguousarray(stream_offs, np.uint64)
    sl = np.ascontiguousarray(stream_lens, np.uint64)
    st = _u8(streams) if streams is not None and len(streams) else np.zeros(1, np.uint8)
    cap = int(sizes.sum()) + int(name_offs[-1]) * 2 + n * 124 + 200
    out = np.empty(cap, np.uint8)
    out_len = C.c_uint64(0)
    methods = np.zeros(max(n, 1), np.uint16)
    t = None if dos_times is None else np.ascontiguousarray(dos_times, np.uint32)
    f = None if flags is None else np.ascontiguousarray(flags, np.uint32)
    rc = lib().orc_zip_create_given(level, C.c_uint32(n), flat.ctypes.data_as(C.c_void_p), offs.ctypes.data_as(C.c_void_p),
                                    sizes.ctypes.data_as(C.c_void_p), C.c_char_p(names), name_offs.ctypes.data_as(C.c_void_p),
                                    None if t is None else t.ctypes.data_as(C.c_void_p), None if f is None else f.ctypes.data_as(C.c_void_p),
                                    out.ctypes.data_as(C.c_void_p), C.c_uint64(cap), C.byref(out_len), methods.ctypes.data_as(C.c_void_p),
                                    st.ctypes.data_as(C.c_void_p), so.ctypes.data_as(C.c_void_p), sl.ctypes.data_as(C.c_void_p))
    assert rc == 0, rc
    return out[:out_len.value], [int(m) for m in methods[:n]]


def zip_create_given(entries, streams, level=9, dos_times=None, flags=None):
    """entries: list of (name, bytes-like); streams: one bytes-like per entry (its BZip2 stream; for an entry to be
    stored, any object whose len() is >= the entry's size).  Returns (archive bytes, [method per entry])."""
    flat, offs, sizes, names, name_offs = pack_entries(entries)
    lens = np.array([len(s) for s in streams], np.uint64)
    given = [b"" if int(l) >= int(sz) else bytes(s) for s, l, sz in zip(streams, lens, sizes)]
    so = np.zeros(len(given), np.uint64)
    so[1:] = np.cumsum([len(g) for g in given])[:-1] if given else []
    arc, methods = zip_create_given_flat(flat, offs, sizes, names, name_offs, b"".join(given), so, lens, level, dos_times, flags)
    return arc.tobytes(), methods
