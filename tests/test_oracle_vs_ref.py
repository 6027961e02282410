"""Pins the oracle (oracle/dx_oracle.c) against the reference tools themselves (oracle/_ref,
compiled from the reference sources by oracle/Makefile) or, where they are absent, against the
digests of their outputs stored in tests/golden/reference_digests.json.  Each reference decoder
is given the oracle's image, which the check before it found equal to the reference's.  CPU only."""
import pytest

from tests import cases
from tests.refgold import check_tool

FASTA = dict(cases.fasta_cases())
ARROW = dict(cases.arrow_cases())
QUIVA = dict(cases.quiva_cases())


@pytest.mark.parametrize("name", sorted(FASTA))
def test_dexta_undexta(orc, name):
    text = FASTA[name]
    enc = orc.dexta(text)
    check_tool("dexta", text, enc)
    if name.startswith("enc_only"):
        return
    check_tool("undexta", enc, orc.undexta(enc))
    check_tool("undexta", enc, orc.undexta(enc, width=37, upper=True), "-U", "-w37")


@pytest.mark.parametrize("name", sorted(ARROW))
def test_dexar_undexar(orc, name):
    text = ARROW[name]
    enc = orc.dexta(text, arrow=True)
    check_tool("dexar", text, enc)
    check_tool("undexar", enc, orc.undexta(enc, arrow=True))
    check_tool("undexar", enc, orc.undexta(enc, arrow=True, width=100), "-w100")


@pytest.mark.parametrize("lossy", [False, True])
@pytest.mark.parametrize("name", sorted(QUIVA))
def test_dexqv_undexqv(orc, name, lossy):
    text = QUIVA[name]
    flags = ("-l",) if lossy else ()
    enc = orc.dexqv(text, lossy=lossy)
    check_tool("dexqv", text, enc, *flags)
    back = orc.undexqv(enc)
    check_tool("undexqv", enc, back)
    if not lossy and name not in cases.QUIVA_NOT_IDENTITY:
        assert back == text
    check_tool("undexqv", enc, orc.undexqv(enc, upper=True), "-U")


def test_entry_offsets_walk(orc):
    text = QUIVA["edge_lengths"]
    data = orc.dexqv(text)
    n = text.count(b"\n") // 6
    offs = orc.dexqv_offsets(data, n)
    assert len(offs) == n + 1 and offs[-1] == len(data)
    assert all(offs[i] < offs[i + 1] for i in range(n))
