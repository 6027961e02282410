"""The crafted header and framing shapes of tests/header_shapes.py, on the CPU: each file has the
property it claims (checked against a numpy restatement of the 2-bit candidate predicate), the
legacy builder reproduces the oracle's native images and its rewritten forms decode to the same
text, and the oracle's SNR coding and printing hold for every value.

Where oracle/_ref is built, the reference dexta / dexar / undexta / undexar are compared as well
(test_reference_tools_agree).  Where it is not, only the oracle checked these shapes: the
reference digests of tests/golden/ do not cover them."""
import re
import struct

import numpy as np
import pytest

from tests import header_shapes as H


def _tails(text: bytes):
    return [line.split(b"/", 1)[1].decode() for line in text.split(b"\n") if line[:1] in (b">", b"@")]


# ---- grammar ----------------------------------------------------------------------------------------

@pytest.mark.parametrize("kind", ["fasta", "arrow"])
def test_grammar_splits_between_device_and_sscanf_shapes(kind):
    """The table's claim of which headers the device parsers take is the restated acceptance rule,
    both kinds are in the file, and the canonical entries between them are device shapes too"""
    arrow = kind == "arrow"
    table = H.GRAMMAR_ARROW if arrow else H.GRAMMAR_FASTA
    for tail, _, dev in table:
        assert H.device_parses(tail, arrow) == dev, tail
    assert {d for _, _, d in table} == {True, False}
    tails = _tails(H.grammar(kind))
    assert tails[1::2] == [t for t, _, _ in table]
    assert all(H.device_parses(t, arrow) for t in tails[0::2])


@pytest.mark.parametrize("kind", ["fasta", "arrow"])
def test_grammar_round_trips_through_the_oracle(orc, kind):
    """Every grammar entry keeps its sequence; its header comes back as sscanf read it"""
    arrow = kind == "arrow"
    text = H.grammar(kind)
    back = orc.undexta(orc.dexta(text, arrow=arrow), arrow=arrow)
    seqs = [c.split(b"\n", 1)[1].replace(b"\n", b"") for c in text.split(b">")[1:]]
    bseqs = [c.split(b"\n", 1)[1].replace(b"\n", b"") for c in back.split(b">")[1:]]
    assert seqs == bseqs
    heads = dict(zip([t for t, _, _ in (H.GRAMMAR_ARROW if arrow else H.GRAMMAR_FASTA)], _tails(back)[1::2]))
    if arrow:
        assert heads["17/0_60 SN=5.00,6.00,7.00,8.00e1"].endswith("SN=5.00,6.00,7.00,80.00")
        assert heads["18/0_60 SN=5.00,6.00,7.00,8.00E-1"].endswith("SN=5.00,6.00,7.00,0.80")
        assert heads["19/0_60 SN=5.00,6.00,7.00,8.00e"].endswith("SN=5.00,6.00,7.00,8.00")
        assert heads["29/4294967295_59 SN=5.00,6.00,7.00,8.00"].startswith("29/-1_59 ")
    else:
        assert heads["14/4294967295_99 RQ=0.4294967295"] == "14/-1_99 RQ=0.-1"
        assert heads["24/5_105RQ=0.851"] == "24/5_105 RQ=0.851"
        assert heads["26/5_105 RQ=1.851"] == "26/5_105 RQ=0.0"


def test_grammar_quiva(orc):
    """.quiva: the device shapes and the sscanf shapes in one file; headers without a readable RQ are
    refused with a format error"""
    text = H.grammar("quiva")
    tails = [line.split(b"/", 1)[1].decode() for line in text.split(b"\n")[0::6] if line]
    num = r"[0-9]{1,9}(?![0-9])"
    dev = [re.match(rf"{num}/{num}_{num} RQ=0\.{num}", t) is not None for t in tails]
    assert dev[1::2] == [d for _, d in H.GRAMMAR_QUIVA] and all(dev[0::2])
    back = orc.undexqv(orc.dexqv(text))
    assert back.split(b"\n")[1::6] == text.split(b"\n")[1::6]
    for i in range(len(H.GRAMMAR_QUIVA_REFUSED)):
        with pytest.raises(orc.OracleError) as e:
            orc.dexqv(H.grammar_quiva_refused(i))
        assert e.value.code == -1


# ---- SNRs ---------------------------------------------------------------------------------------------

def _code(s: str) -> int:
    """dexar.c:159-163: strtof, then (u16) (u32) (snr * 100.) or 9999 above 99.99"""
    f = np.float32(float(s))
    return 9999 if f > np.float32(99.99) else int(float(f) * 100.) & 0xFFFF


def test_every_two_decimal_snr(orc):
    """4 802 of the 10 000 values 0.00 ... 99.99 do not keep their value (6.97 is stored as 696), and
    the oracle stores and prints exactly what strtof and %.2f of a float give"""
    text = H.snr_all_arrow()
    img = orc.dexta(text, arrow=True)
    vals = [v for t in _tails(text) for v in t.split("SN=")[1].split(",")]
    codes = [c for q, *_, aux in H.entry_fields(img, True) for c in aux]
    assert len(codes) == len(vals)
    assert codes == [_code(v) for v in vals]
    assert sum(_code(f"{k / 100:.2f}") != k for k in range(10000)) == 4802
    assert _code("6.97") == 696
    back = [v for t in _tails(orc.undexta(img, arrow=True)) for v in t.split("SN=")[1].split(",")]
    assert back == ["%.2f" % np.float32(c / 100.) for c in codes]
    assert set(vals[:10000]) == {f"{k // 100}.{k % 100:02d}" for k in range(10000)}


def test_every_stored_snr_code(orc):
    """The crafted .dexar image stores all 65 536 codes; the oracle prints each as %.2f of the float
    c / 100.; entries with a code above 9999 are not candidates, so the decode takes the general
    chain"""
    img = H.snr_codes_dexar()
    ents = H.entry_fields(img, True)
    assert sorted(c for *_, aux in ents for c in aux) == list(range(1 << 16))
    cand = set(H.candidate_positions(img, True).tolist())
    for q, _, _, _, aux in ents:
        assert (q in cand) == (max(aux) <= H.CAND_MAX_SNR)
    assert H.expected_route(img, True)[1] == H.CHAIN_GENERAL
    back = [t.split("SN=")[1].split(",") for t in _tails(orc.undexta(img, arrow=True))]
    assert back == [["%.2f" % np.float32(c / 100.) for c in aux] for *_, aux in ents]


# ---- window and wells ---------------------------------------------------------------------------------

@pytest.mark.parametrize("arrow", [False, True])
@pytest.mark.parametrize("name", sorted(H.WINDOW))
def test_window_entry_is_in_or_out(orc, name, arrow):
    """The crafted entry (well 30) is a candidate exactly when the shape says so, every other entry
    is one, and the chain takes the fast path exactly then"""
    field, value, inside = H.WINDOW[name]
    if arrow and field == "qv":
        pytest.skip(".arrow has no qv")
    if arrow and field == "beg":
        inside = False                           # the .dexar prefilter also asks end < 2^27
    img = orc.dexta(H.window(name, arrow), arrow=arrow)
    cand = set(H.candidate_positions(img, arrow).tolist())
    ents = H.entry_fields(img, arrow)
    crafted = [e for e in ents if e[1] == 30]
    assert len(crafted) == 1
    q, _, beg, end, aux = crafted[0]
    assert {"beg": beg, "len": end - beg, "qv": aux[0]}[field] == value
    assert (q in cand) == inside
    assert all(e[0] in cand for e in ents if e[1] != 30)
    assert H.expected_route(img, arrow)[1] == (H.CHAIN_FAST if inside else H.CHAIN_GENERAL)


def _ff_runs(img: bytes):
    a = np.frombuffer(img, dtype=np.uint8) == 0xFF
    d = np.diff(np.concatenate([[0], a.astype(np.int8), [0]]))
    return (np.nonzero(d == -1)[0] - np.nonzero(d == 1)[0]).tolist()


@pytest.mark.parametrize("arrow", [False, True])
def test_well_jumps(orc, arrow):
    """The deltas write runs of 1, 2, 2^20 - 1 and 2^20 0xff bytes, and round trip on the fast chain;
    one run of 2^20 + 1 bytes is more than the run count holds and takes the general chain"""
    kind = "arrow" if arrow else "fasta"
    text = H.well_jumps(kind, "deltas")
    img = orc.dexta(text, arrow=arrow)
    wells = [e[1] for e in H.entry_fields(img, arrow)]
    assert wells == [int(t.split("/")[0]) for t in _tails(text)]
    runs = _ff_runs(img)
    for k in (1, 2, H.FFRUN_CAP - 1, H.FFRUN_CAP):
        assert k in runs, k
    assert max(runs) == H.FFRUN_CAP
    assert H.expected_route(img, arrow)[1] == H.CHAIN_FAST
    if not arrow:
        assert orc.undexta(img) == text
    img = orc.dexta(H.well_jumps(kind, "over_cap"), arrow=arrow)
    assert max(_ff_runs(img)) >= H.FFRUN_CAP + 1
    assert H.expected_route(img, arrow)[1] == H.CHAIN_GENERAL
    for w in H.FIRST_WELLS:
        img = orc.dexta(H.well_jumps(kind, f"first{w}"), arrow=arrow)
        first = 6 + struct.unpack_from("<i", img, 2)[0]
        assert img[first: first + 1 + (w >= 255)] == {0: b"\x00", 255: b"\xff\x00", 256: b"\xff\x01"}[w]
        assert H.entry_fields(img, arrow)[0][1] == w


@pytest.mark.parametrize("arrow", [False, True])
@pytest.mark.parametrize("drop", H.WELL_DROPS)
def test_dropping_wells_misframe_the_image(orc, drop, arrow):
    """put_well writes (u8) (well - lwell) when the wells drop: 0xff for a drop of 1, which a decoder
    reads as 255 more and takes the next byte as the rest of the delta.  The oracle refuses a drop of
    1 and decodes the others to headers other than the text's"""
    text = H.well_jumps("arrow" if arrow else "fasta", f"drop{drop}")
    img = orc.dexta(text, arrow=arrow)
    if drop == 1:
        with pytest.raises(orc.OracleError):
            orc.undexta(img, arrow=arrow)
    else:
        back = orc.undexta(img, arrow=arrow)
        assert back != text
        assert [e[1] for e in H.entry_fields(img, arrow)] != [int(t.split("/")[0]) for t in _tails(text)]


def test_quiva_well_jumps(orc):
    for case in H.WELL_CASES:
        text = H.well_jumps("quiva", case)
        img = orc._run(orc.lib().orc_dexqv, text, len(text) * 3 + (16 << 20), 0)
        if case == "drop1":
            with pytest.raises(orc.OracleError):
                orc.undexqv(img)
        elif case.startswith("drop"):
            assert orc.undexqv(img) != text
        else:
            assert orc.undexqv(img) == text, case
            if case == "deltas":
                assert max(_ff_runs(img)) >= H.FFRUN_CAP


# ---- zero payloads --------------------------------------------------------------------------------------

@pytest.mark.parametrize("kind", ["fasta", "arrow"])
def test_zero_payload_overflows_the_tiles(orc, kind):
    """Reads that pack to zero bytes make every offset of their payload a candidate: the tiles
    overflow (two-pass index) and the candidates outnumber a sixteenth of the image bytes; the true
    entries are still all candidates, so the chain stays on the fast path"""
    arrow = kind == "arrow"
    text = H.zero_payload(kind)
    img = orc.dexta(text, arrow=arrow)
    pos = H.candidate_positions(img, arrow)
    assert len(text) > 4_000_000
    assert H.tile_overflow(img, arrow)
    assert len(pos) > len(img) // 2
    assert H.expected_route(img, arrow) == (H.INDEX_TWO_PASS, H.CHAIN_FAST)
    back = orc.undexta(img, arrow=arrow)
    seq = [x for x in (text if arrow else text.replace(b"N", b"a")).split(b"\n") if x[:1] != b">"]
    assert [x for x in back.split(b"\n") if x[:1] != b">"] == seq


def test_zero_runs_around_twelve_bytes():
    """The 'a'-runs of 40 ... 52 symbols at every offset mod 4 give 9 to 13 zero bytes: some make a
    candidate out of zeros alone (12 or more), some fall one byte short"""
    zeros = set()
    for r in range(40, 53):
        for o in range(4):
            head = b"c" * (64 + o)
            b = H.pack2bit(head + b"a" * r + b"c" * 64, False)
            z = max(len(m) for m in re.findall(rb"\x00+", b))
            zeros.add(z)
    assert zeros == {9, 10, 11, 12, 13}


# ---- legacy forms ---------------------------------------------------------------------------------------

LEGACY = [(False, True, False), (False, False, True), (False, True, True), (True, True, False)]


def _legacy_id(v):
    arrow, flip, old = v
    return "_".join(["arrow" if arrow else "fasta"] + [x for x, on in (("foreign", flip), ("old", old)) if on])


@pytest.mark.parametrize("form", LEGACY, ids=_legacy_id)
@pytest.mark.parametrize("seed", [11, 12])
def test_legacy_forms_decode_to_the_native_text(orc, seed, form):
    arrow, flip, old = form
    text = H.legacy_text(seed, arrow)
    native = orc.dexta(text, arrow=arrow)
    assert H.build_2bit(text, arrow) == native
    img = H.build_2bit(text, arrow, flip, old)
    assert img != native
    for width, upper in ((80, False), (7, True)):
        assert orc.undexta(img, arrow=arrow, width=width, upper=upper) == \
            orc.undexta(native, arrow=arrow, width=width, upper=upper)


@pytest.mark.parametrize("form", [f for f in LEGACY if not f[2]], ids=_legacy_id)
@pytest.mark.parametrize("drop", [d for d in H.WELL_DROPS if d != 1])
def test_foreign_forms_with_a_dropping_well(orc, drop, form):
    """... and an image whose wells drop by 2 or 300 (delta bytes 0xfe and 0xd4: the well wraps, the
    framing holds) decodes in the foreign byte order to what the native image decodes to.  A drop of
    1 writes 0xff and misframes the image, which then reads other bytes in each byte order; the
    16-bit layout frames its fields in other sizes, so it has no native counterpart either"""
    arrow, flip, old = form
    text = H.well_jumps("arrow" if arrow else "fasta", f"drop{drop}")
    native = orc.dexta(text, arrow=arrow)
    assert H.build_2bit(text, arrow) == native
    img = H.build_2bit(text, arrow, flip, old)

    def run(b):
        try:
            return orc.undexta(b, arrow=arrow)
        except orc.OracleError as e:
            return e.code
    assert run(img) == run(native)


# ---- the reference tools ---------------------------------------------------------------------------------

def test_reference_tools_agree(orc):
    """Where oracle/_ref is built: dexta / dexar of the grammar, window and well shapes give the
    oracle's images, and undexta / undexar of those images and of the legacy forms give the oracle's
    texts.  Where it is not built, the shapes were compared with the oracle only."""
    if not orc.have_ref():
        pytest.skip("oracle/_ref is not built: these shapes were compared with the oracle only")
    texts = [("fasta", H.grammar("fasta")), ("arrow", H.grammar("arrow")),
             ("fasta", H.window("beg_out")), ("fasta", H.well_jumps("fasta", "first256")),
             ("fasta", H.well_jumps("fasta", "drop2")), ("arrow", H.snr_all_arrow())]
    for kind, text in texts:
        arrow = kind == "arrow"
        img = orc.dexta(text, arrow=arrow)
        assert orc.ref_tool("dexar" if arrow else "dexta", text)[0] == img
        assert orc.ref_tool("undexar" if arrow else "undexta", img)[0] == orc.undexta(img, arrow=arrow)
    for arrow, flip, old in LEGACY:
        text = H.legacy_text(11, arrow)
        img = H.build_2bit(text, arrow, flip, old)
        assert orc.ref_tool("undexar" if arrow else "undexta", img)[0] == orc.undexta(img, arrow=arrow)
