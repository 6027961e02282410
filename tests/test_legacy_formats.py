"""Foreign-endian and old-layout .dexqv files (tests/golden/legacy_*.dexqv, made by
tests/golden/make_legacy.py and checked there against the reference undexqv): the reference reads
them (undexqv.c:103-110, 135-180; QV.c:553-568, 1226-1255), so the library must too."""
import hashlib
import json
import os

import pytest


HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
MAN = json.load(open(os.path.join(HERE, "legacy_manifest.json")))
FILES = sorted(MAN["files"])


def _text(orc):
    """what the native-order, new-layout file of the same text decodes to (oracle)"""
    native = open(os.path.join(HERE, "legacy_native.dexqv"), "rb").read()
    assert hashlib.sha256(native).hexdigest() == MAN["native_sha256"]
    t = orc.undexqv(native)
    assert hashlib.sha256(t).hexdigest() == MAN["decoded_sha256"]
    return t


@pytest.mark.parametrize("name", FILES)
def test_fixture_is_what_the_manifest_says(name):
    b = open(os.path.join(HERE, name), "rb").read()
    assert hashlib.sha256(b).hexdigest() == MAN["files"][name]["sha256"]
    # layout: the old files begin with the coding key, the new ones with 0x55aa in either order
    key = b[:2]
    if MAN["files"][name]["old"]:
        assert key == (b"\x33\xcc" if MAN["files"][name]["flip"] else b"\xcc\x33")
    else:
        assert key == (b"\x55\xaa" if MAN["files"][name]["flip"] else b"\xaa\x55")


@pytest.mark.parametrize("name", FILES)
def test_reference_decodes_the_fixture_to_the_text(orc, name):
    """the reference undexqv (oracle/_ref) decodes the fixture to the text; where it is not built,
    the oracle must give the text the reference gave when the fixture was made (decoded_sha256)"""
    b = open(os.path.join(HERE, name), "rb").read()
    if orc.have_ref():
        assert orc.ref_tool("undexqv", b)[0] == _text(orc)
    else:
        assert hashlib.sha256(orc.undexqv(b)).hexdigest() == MAN["decoded_sha256"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", FILES)
def test_gpu_decodes_legacy_files(orc, name):
    import dextractor_b200 as dx
    ctx = dx.Context(0)
    try:
        b = open(os.path.join(HERE, name), "rb").read()
        want = _text(orc)
        assert ctx.undexqv(b) == want
        up = ctx.undexqv(b, upper=True)
        assert up != want and len(up) == len(want) and up.lower() == want.lower()
    finally:
        ctx.close()


@pytest.mark.gpu
def test_gpu_refuses_a_file_with_an_unknown_key():
    import dextractor_b200 as dx
    ctx = dx.Context(0)
    try:
        with pytest.raises(dx.DexError) as e:
            ctx.undexqv(b"\x12\x34" + bytes(5000))
        assert e.value.code == -4
    finally:
        ctx.close()
