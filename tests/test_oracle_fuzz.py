"""Seeded random differential test: oracle (oracle/dx_oracle.c) against the reference tools
(oracle/_ref) or, where they are absent, the stored digests of their outputs
(tests/golden/reference_digests.json), on inputs whose shape is drawn at random (tests/fuzz.py).
CPU only."""
import pytest

from tests import fuzz
from tests.refgold import check_tool


@pytest.mark.parametrize("seed", range(24))
def test_fuzz_dexqv_undexqv(orc, seed):
    text, _ = fuzz.fuzz_quiva(seed)
    for lossy in (False, True):
        flags = ("-l",) if lossy else ()
        enc = orc.dexqv(text, lossy=lossy)
        check_tool("dexqv", text, enc, *flags)
        check_tool("undexqv", enc, orc.undexqv(enc))
        n = text.count(b"\n") // 6
        offs = orc.dexqv_offsets(enc, n)
        assert len(offs) == n + 1 and offs[-1] == len(enc)


@pytest.mark.parametrize("seed", range(16))
def test_fuzz_dexta_dexar(orc, seed):
    fa, ar, w2 = fuzz.fuzz_fasta_arrow(seed)
    enc = orc.dexta(fa)
    check_tool("dexta", fa, enc)
    for args, kw in ((("-w%d" % w2,), dict(width=w2)), (("-U", "-w%d" % w2), dict(width=w2, upper=True))):
        check_tool("undexta", enc, orc.undexta(enc, **kw), *args)
    enc = orc.dexta(ar, arrow=True)
    check_tool("dexar", ar, enc)
    check_tool("undexar", enc, orc.undexta(enc, arrow=True, width=w2), "-w%d" % w2)
