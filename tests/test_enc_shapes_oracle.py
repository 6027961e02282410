"""The crafted encoder shapes of tests/enc_shapes.py on the CPU: the numpy restatement of the encoder's
accounting gives the oracle's byte count for every stream, every family holds the claims it is built
for, and every file round-trips through the oracle (the entry of 2^24 positions too, which the
library refuses).  These keep the GPU tests' inputs honest on any machine."""
import numpy as np
import pytest

from tests import enc_shapes as X
from tests import fuzz

CRAFTED = sorted(X.CLAIMS)


@pytest.mark.parametrize("lossy", [False, True], ids=["lossless", "lossy"])
@pytest.mark.parametrize("name", CRAFTED)
def test_model_counts_every_stream_like_the_oracle(orc, name, lossy):
    for label, text in X.make(orc, name):
        X.check_against_oracle(orc, text, lossy=lossy)


def test_model_on_the_fuzz_files(orc):
    for seed in range(40):
        text, _ = fuzz.fuzz_quiva(seed)
        for lossy in (False, True):
            X.check_against_oracle(orc, text, lossy=lossy)


@pytest.mark.parametrize("name", CRAFTED)
def test_family_claims(orc, name):
    for label, text in X.make(orc, name):
        print(name, label, sorted(X.CLAIMS[name](orc, label, text)))


@pytest.mark.parametrize("name", sorted(set(X.SHAPES) | set(X.PLAIN)))
def test_every_file_has_a_coding_the_library_builds(orc, name):
    """the GPU tests run every file lossy and not: no table may end up with fewer than two symbols"""
    for label, text in X.make(orc, name):
        for lossy in (False, True):
            assert X.codable(orc, text, lossy), (name, label, lossy)


def test_room_files_sit_on_both_sides_of_every_room(orc):
    got = set()
    for label, text in X.make(orc, "room"):
        r = X.room_claims(orc, label, text)
        if label.endswith("midflush"):
            continue
        kind, R, side = label.split("_")
        got.add((kind, int(R) % 4, int(R) > 2048, side))
    assert got == {(k, m, big, s) for k in ("ins", "del") for m in range(4) for big in (False, True)
                   for s in ("fit", "over")}


@pytest.mark.parametrize("lossy", [False, True], ids=["lossless", "lossy"])
def test_counts_entry_offsets(orc, lossy):
    for label, text in X.make(orc, "counts"):
        fm = X.check_against_oracle(orc, text, lossy=lossy, per_stream=False)
        n = fm["entries"]["p"]["n"]
        assert n == int(label) and len(fm["offs"]) == n + 1
        assert (fm["entries"]["p"]["rlen"] == 0).any() and fm["entries"]["p"]["rlen"].max() == 3
    assert [X.offset_scan(n) for n in X.COUNTS] == ["k_qv_offsets", "k_tile_scan", "k_chain_scan", "k_chain_scan"]


def test_long_entries(orc):
    for label, text in X.make(orc, "long"):
        p = X.S.parse(text)
        rl = set(p["rlen"].tolist())
        assert (set(X.LONG) if label == "long" else {X.LONGEST}) <= rl
        assert p["rlen"].max() < X.MAX_RLEN
        fm = X.check_against_oracle(orc, text)
        c = fm["coding"]
        assert c.delchar == X.DELC and c.subchar == 63
        for e, ls in enumerate(fm["entries"]["lines"]):
            for k, rc in ((0, c.delchar), (4, c.subchar)):
                runs, _, trail = X.run_items(ls[k], rc)
                assert max(runs.max(initial=0), trail) < 65536


def _without_tags(text):
    lines = text.split(b"\n")
    return [x for i, x in enumerate(lines) if i % 6 != 2]


def test_round_trips_through_the_oracle(orc):
    """identity but for the tag lines of the tag files (upper case and n / N tags come back as
    the 2-bit code's lower-case letters)"""
    for name in CRAFTED + ["counts"]:
        for label, text in X.make(orc, name):
            back = orc.undexqv(orc.dexqv(text))
            if name == "tags" or (name, label) == ("stage", "tags"):
                assert _without_tags(back) == _without_tags(text) and len(back) == len(text)
            else:
                assert back == text, (name, label)
            assert len(orc.undexqv(orc.dexqv(text, lossy=True))) == len(text)


def test_long_round_trips_through_the_oracle(orc):
    """including one entry of 2^24 positions: the oracle, like the reference, takes it"""
    texts = [t for _, t in X.make(orc, "long")] + [X.make_too_long()]
    assert X.S.parse(texts[-1])["rlen"].tolist() == [X.MAX_RLEN]
    for text in texts:
        assert orc.undexqv(orc.dexqv(text)) == text
