"""A small reader of the Zip records, written from the format (APPNOTE 4.3.7, 4.3.12, 4.3.14-16, 4.5.3), and
the Zip64 rules of Zip.Create / Zip.Headers (zip-create.adb:161-179, :233-297, :645-756; zip-headers.adb:194-207)
restated in a few lines.  The archive tests past 4 GiB check what the oracle and the library write against both;
neither shares code with them."""
import struct

FOUR_GIB = 1 << 32
MARGIN = 22 + 56 + 20 + 65536 + 10               # Check_Size: room for the end records and a comment
CHECK_SIZE_AT = FOUR_GIB - MARGIN                # 4 294 901 652
U32_FULL = 0xFFFFFFFF


def expected_layout(sizes, names, csizes=None):
    """Where each record of an archive sits and which of them carry Zip64 fields; csizes are the payload sizes
    (None: every entry is stored).  Returns dict(entries=[dict(offset, size, csize, local_ext, central_ext)],
    cd_offset, cd_size, zip64)."""
    csizes = list(sizes) if csizes is None else list(csizes)
    zip64 = False
    pos = 0
    ents = []
    for size, csize, name in zip(sizes, csizes, names):
        if size >= CHECK_SIZE_AT:                # Check_Size (size) in Add_Stream
            zip64 = True
        local_ext = size >= U32_FULL or pos >= U32_FULL      # decided before compression, with csize = usize
        central_ext = size >= U32_FULL or csize >= U32_FULL or pos >= U32_FULL
        ents.append(dict(offset=pos, size=size, csize=csize, local_ext=local_ext, central_ext=central_ext))
        pos += 30 + len(name) + (20 if local_ext else 0) + csize
    cd_offset = pos
    cd_size = sum(46 + len(nm) + (28 if e["central_ext"] else 0) for e, nm in zip(ents, names))
    if any(e["central_ext"] for e in ents):      # Finish: a central Zip64 extension promotes the archive
        zip64 = True
    if cd_offset + cd_size + 1 >= CHECK_SIZE_AT:  # Check_Size (Index) in Finish, on the 1-based index
        zip64 = True
    return dict(entries=ents, cd_offset=cd_offset, cd_size=cd_size, zip64=zip64)


def _u(fmt, buf, off):
    return struct.unpack_from("<" + fmt, buf, off)


def scan(arc):
    """Parses an archive (bytes-like) from its end: end record, Zip64 end record and locator when present, every
    central header with its extra field, and every local header with its extra field.  Returns a dict."""
    mv = memoryview(arc)
    n = len(mv)
    sig, d0, d1, n_disk, n_tot, cds, cdo, clen = _u("IHHHHIIH", mv, n - 22)
    assert sig == 0x06054B50 and clen == 0
    res = dict(end=dict(n_disk=n_disk, n_total=n_tot, cd_size=cds, cd_offset=cdo), z64_end=None, z64_loc=None)
    if n >= 42 and bytes(mv[n - 42:n - 38]) == b"PK\x06\x07":
        _, disk, rel, ndisks = _u("IIQI", mv, n - 42)
        res["z64_loc"] = dict(disk=disk, rel=rel, n_disks=ndisks)
        sig, size, made, need, disk, cdisk, nd, nt, cds64, cdo64 = _u("IQHHIIQQQQ", mv, rel)
        assert sig == 0x06064B50 and rel + 56 == n - 42
        res["z64_end"] = dict(size=size, made_by=made, needed=need, disk=disk, cd_disk=cdisk, n_disk=nd, n_total=nt,
                              cd_size=cds64, cd_offset=cdo64)
        cdo, cds, n_tot = cdo64, cds64, nt
    central = []
    p = cdo
    for _ in range(n_tot):
        (sig, made, need, flag, method, tdate, crc, csize, usize, nlen, xlen, cmlen, disk, iattr, eattr,
         off) = _u("IHHHHIIIIHHHHHII", mv, p)
        assert sig == 0x02014B50
        name = bytes(mv[p + 46:p + 46 + nlen])
        extra = bytes(mv[p + 46 + nlen:p + 46 + nlen + xlen])
        central.append(dict(name=name, method=method, crc=crc, csize=csize, usize=usize, offset=off, extra=_extra(extra)))
        p += 46 + nlen + xlen + cmlen
    assert p == cdo + cds
    local = []
    for c in central:
        if c["offset"] == U32_FULL:
            assert len(c["extra"]) == 3, c
        off = c["extra"][2] if c["offset"] == U32_FULL else c["offset"]
        sig, need, flag, method, tdate, crc, csize, usize, nlen, xlen = _u("IHHHIIIIHH", mv, off)
        assert sig == 0x04034B50
        name = bytes(mv[off + 30:off + 30 + nlen])
        extra = bytes(mv[off + 30 + nlen:off + 30 + nlen + xlen])
        local.append(dict(offset=off, name=name, method=method, crc=crc, csize=csize, usize=usize, xlen=xlen,
                          extra=_extra(extra), payload=off + 30 + nlen + xlen))
    return dict(res, central=central, local=local)


def _extra(raw):
    """The Zip64 extended information field (tag 1) as a list of u64 values, () when absent; other tags fail."""
    if not raw:
        return ()
    tag, size = struct.unpack_from("<HH", raw, 0)
    assert tag == 1 and size == len(raw) - 4 and size % 8 == 0, (tag, size, len(raw))
    return struct.unpack_from("<%dQ" % (size // 8), raw, 4)


def check_layout(arc, sizes, names, crcs, csizes=None):
    """Asserts that `arc` holds exactly the records expected_layout() places, with these CRCs, and returns
    the expected layout with the parsed records under "scan"."""
    lay = expected_layout(sizes, names, csizes)
    s = scan(arc)
    assert len(s["central"]) == len(sizes)
    for i, (e, c, l) in enumerate(zip(lay["entries"], s["central"], s["local"])):
        usize, csize = e["size"], e["csize"]
        assert c["name"] == l["name"] == names[i], i
        assert c["crc"] == l["crc"] == crcs[i], i
        assert l["offset"] == e["offset"], i
        if e["local_ext"]:
            assert (l["csize"], l["usize"], l["xlen"]) == (U32_FULL, U32_FULL, 20), i
            assert l["extra"] == (usize, csize), i
        else:
            assert (l["csize"], l["usize"], l["xlen"], l["extra"]) == (csize, usize, 0, ()), i
        if e["central_ext"]:
            assert (c["csize"], c["usize"], c["offset"]) == (U32_FULL, U32_FULL, U32_FULL), i
            assert c["extra"] == (usize, csize, e["offset"]), i
        else:
            assert (c["csize"], c["usize"], c["offset"], c["extra"]) == (csize, usize, e["offset"], ()), i
    cd_offset, cd_size, n = lay["cd_offset"], lay["cd_size"], len(sizes)
    if lay["zip64"]:
        assert len(arc) == cd_offset + cd_size + 56 + 20 + 22
        assert s["z64_end"] == dict(size=44, made_by=0x2D, needed=0x2D, disk=0, cd_disk=0, n_disk=n, n_total=n,
                                    cd_size=cd_size, cd_offset=cd_offset)
        assert s["z64_loc"] == dict(disk=0, rel=cd_offset + cd_size, n_disks=1)
        assert s["end"] == dict(n_disk=0xFFFF, n_total=0xFFFF, cd_size=U32_FULL, cd_offset=U32_FULL)
    else:
        assert len(arc) == cd_offset + cd_size + 22
        assert s["z64_end"] is None and s["z64_loc"] is None
        assert s["end"] == dict(n_disk=n, n_total=n, cd_size=cd_size, cd_offset=cd_offset)
    return dict(lay, scan=s)
