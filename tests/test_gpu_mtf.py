"""Stage A7 (move-to-front and zero-run coding, zip-ada_b200/csrc/b2_mtf.cuh) on the device, on designed last columns.

b2_dbg_mtf runs the production plan and kernels on given columns as one batch, with the slot padding, the masks and the
outputs poisoned first.  Every family of tests/mtf_families.py at full block size (the batch family in a single call)
must give the index bytes, the symbols, n_mtf and n_groups of the oracle's literal MTF.  The device build may schedule
and contract code in ways the host emulation (tests/test_emu_mtf.py) cannot show, and at full size a block has 27
segment starts and distances of many steps (c)."""
import numpy as np
import pytest

import datagen
import mtf_families as mf
import oracle_lib as orc

pytestmark = pytest.mark.gpu


def _check(enc, name, blocks):
    res = enc.dbg_mtf([c for _, c in blocks])
    assert len(res) == len(blocks)
    for j, ((label, col), r) in enumerate(zip(blocks, res)):
        msg = mf.compare("%s block %d (%s, %d positions)" % (name, j, label, col.size), col, r["idx"], r["mtf"], r["n_mtf"],
                         r["n_groups"])
        assert msg is None, msg


@pytest.mark.parametrize("name", list(mf.FAMILIES))
def test_mtf_full_size(enc9, name):
    _check(enc9, name, mf.make(name, full=True))


def test_mtf_emulator_sizes(enc9):
    """The blocks of the host emulation, all families in one call."""
    blocks = [(name + ": " + label, col) for name in mf.FAMILIES for label, col in mf.make(name)]
    _check(enc9, "all families", blocks)


def test_dbg_mtf_is_the_production_path(enc9):
    """The tap on the column that b2_dbg_block's encode produced gives that encode's symbols."""
    data = datagen.text(890000, 11)
    blk = enc9.dbg_block(data)
    r = enc9.dbg_mtf([blk["bwt"]])[0]
    assert np.array_equal(r["mtf"], blk["mtf"])
    assert r["n_mtf"] == blk["info"].n_mtf and r["n_groups"] == blk["info"].n_sel
    _, idx = orc.mtf_rle2(blk["bwt"])
    assert np.array_equal(r["idx"], idx)


def test_dbg_mtf_arguments(b2mod, enc9):
    with pytest.raises(b2mod.B2Error):
        enc9.dbg_mtf([])
    with pytest.raises(b2mod.B2Error):
        enc9.dbg_mtf([np.zeros(900_001, np.uint8)])
    with pytest.raises(b2mod.B2Error):
        enc9.dbg_mtf([np.zeros(10, np.uint8)] * 65_536)
    with b2mod.Encoder(1, 0) as enc1:
        with pytest.raises(b2mod.B2Error):
            enc1.dbg_mtf([np.zeros(100_001, np.uint8)])
        col = mf.make("alphabets")[9][1]
        _check(enc1, "level 1", [("255 bytes, %d positions" % col.size, col)])
    s = enc9.stream(-1)
    try:
        with pytest.raises(b2mod.B2Error) as ei:
            enc9.dbg_mtf([np.zeros(10, np.uint8)])
        assert "error 1:" in str(ei.value)              # B2_ERR_ARGUMENT while a stream is open
    finally:
        s.abort()
    _check(enc9, "after the refusals", mf.make("places"))     # the handle is usable again
