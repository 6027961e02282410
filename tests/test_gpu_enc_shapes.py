"""The crafted encoder shapes of tests/enc_shapes.py (streams exactly at and one word over their scratch
room, writer rows of 31 / 32 / 33 bits per lane, stage reserves at 512 and 513 words, tag counts, the
look-ahead word, 16 383 ... 40 000 entries, entries of 2^20 - 1 ... 2^24 - 1 positions) through the
library, bit-exact against the oracle, with the encoder route the model predicts; and the entry of
2^24 positions the library refuses.

Decode routes seen on a B200 with this library for the long files (printed by
test_long_entries_decode).  The long entries are never header candidates (kCandMaxLen), so a decode
with discovered entries walks the chain (k_qv_walk5) and leaves the in-place form for k_qv_assemble:
  long     discovered: k_qv_decode5_spec x2, k_qv_walk5 x2, k_qv_decode5, k_qv_assemble
  longest  discovered: k_qv_decode5_spec x2, k_qv_walk5 x1, k_qv_decode5, k_qv_assemble
  both     with the encoder's offsets: one k_qv_decode5, no walk, no k_qv_assemble
The test asserts the parts of this that follow from the entry lengths: the walk and k_qv_assemble
with discovered entries, a single k_qv_decode5 and neither of them with offsets."""
import ctypes as C

import numpy as np
import pytest

import dextractor_b200 as dx
from tests import enc_shapes as X
from tests.test_gpu_parity import first_diff
from tests.test_gpu_qv_shapes import GUARD, _decode_dev, _encoder_image, _prime_need
from tests.test_gpu_scan_shapes import _device

pytestmark = pytest.mark.gpu

DX_E_FORMAT, DX_E_CAP, DX_E_TRUNC, DX_E_TOOLONG, DX_E_ARG = -1, -2, -3, -6, -7
ENC_ROUTES = [{}, {"two_pass": 1}, {"chain_scan": 1}]
FAMILIES = ["room", "rows", "stage", "pad", "tags", "counts"]


def _rid(env):
    return ",".join(f"{k}={v}" for k, v in env.items()) or "default"


@pytest.fixture(scope="module")
def ctx():
    c = dx.Context(0)
    yield c
    c.close()


@pytest.fixture
def routed(ctx):
    yield ctx
    ctx.route("default")


_want: dict = {}


def want(orc, name, label, text):
    """the oracle's images of one file, and whether the model predicts a stream outgrowing its room"""
    key = (name, label)
    if key not in _want:
        fm = X.file_model(orc, text)
        _want[key] = dict(enc={lo: orc.dexqv(text, lossy=lo) for lo in (False, True)},
                          over=any(not m["fits"] for m in fm["streams"].values()),
                          nent=fm["entries"]["p"]["n"])
    return _want[key]


def _dexqv_dev(ctx, text, lossy, cap=None):
    t = _device(text)
    cap = cap if cap is not None else 3 * len(text) + 200000
    out = _device(b"", cap)
    m = ctx.dexqv_dev(t.data_ptr(), len(text), lossy, out.data_ptr(), cap)
    return out[:m].cpu().numpy().tobytes()


@pytest.mark.parametrize("env", ENC_ROUTES, ids=_rid)
@pytest.mark.parametrize("name", FAMILIES)
def test_images_and_encoder_route(routed, orc, name, env):
    """every file, lossy and not, through dx_dexqv_host and dx_dexqv_dev; the profile shows the
    route the model predicts: one k_qv_emit when every stream fits its room, k_qv_size and two
    k_qv_emit when one does not (k_qv_size and one k_qv_emit on two_pass)"""
    ctx = routed
    for k, v in env.items():
        ctx.route(k, v)
    for label, text in X.make(orc, name):
        w = want(orc, name, label, text)
        for lossy in (False, True):
            ctx.profile(True); ctx.profile_report()
            got = ctx.dexqv(text, lossy=lossy)
            prof = ctx.profile_report(); ctx.profile(False)
            assert got == w["enc"][lossy], (label, lossy, first_diff(got, w["enc"][lossy]))
            got = _dexqv_dev(ctx, text, lossy)
            assert got == w["enc"][lossy], (label, lossy, first_diff(got, w["enc"][lossy]))
            if lossy:
                continue
            emit, size = prof.get("k_qv_emit", (0,))[0], prof.get("k_qv_size", (0,))[0]
            if env.get("two_pass"):
                assert (size, emit) == (1, 1), (label, prof)
            elif w["over"]:
                assert (size, emit) == (1, 2), (label, "predicted: a stream outgrows its room", prof)
            else:
                assert (size, emit) == (0, 1), (label, "predicted: every stream fits", prof)
            if name == "room":
                assert w["over"] == (not X.room_claims(orc, label, text)["fits"]), label


@pytest.mark.parametrize("name", FAMILIES)
def test_encoder_offsets_and_decode(ctx, orc, name):
    """dx_qv_encode_dev's image and entry offsets against the oracle; the image decodes back to the
    text on the default route, with discovered entries and with the offsets"""
    for label, text in X.make(orc, name):
        w = want(orc, name, label, text)
        enc = w["enc"][False]
        img, offs = _encoder_image(ctx, text)
        assert img == enc, (label, first_diff(img, enc))
        assert np.array_equal(offs, orc.dexqv_offsets(enc, w["nent"])), label
        for lossy in (False, True):
            e = w["enc"][lossy]
            back = orc.undexqv(e)
            got = ctx.undexqv(e)
            assert got == back, (label, lossy, first_diff(got, back))
        back = orc.undexqv(enc)
        got, guard = _decode_dev(ctx, enc, len(back), entry_off=offs)
        assert got == back and guard == b"\xEE" * GUARD, label


CAP_FILES = [("room", "ins_2100_fit"), ("room", "del_11_over"), ("room", "ins_1100_midflush"),
             ("stage", "ins"), ("counts", "16384")]


@pytest.mark.parametrize("env", ENC_ROUTES, ids=_rid)
@pytest.mark.parametrize("name,label", CAP_FILES, ids=[f"{a}-{b}" for a, b in CAP_FILES])
def test_dexqv_at_exact_capacity(routed, orc, name, label, env):
    """capacity E encodes, E - 1 is DX_E_CAP with dx_needed_bytes E or 0 (never an earlier call's
    need); nothing past the capacity changes"""
    import torch
    ctx = routed
    for k, v in env.items():
        ctx.route(k, v)
    text = dict(X.make(orc, name))[label]
    enc = want(orc, name, label, text)["enc"][False]
    E = len(enc)
    t = _device(text)
    h_text = np.frombuffer(text, dtype=np.uint8)
    for cap in (E, E - 1):
        out = torch.full((E + GUARD,), 0xEE, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        _prime_need(ctx)
        n = C.c_size_t(0)
        rc = ctx.L.dx_dexqv_dev(ctx.h, t.data_ptr(), len(text), 0, out.data_ptr(), cap, C.byref(n))
        ctx.L.dx_sync(ctx.h)
        got = out.cpu().numpy().tobytes()
        assert got[cap:] == b"\xEE" * (E + GUARD - cap), (label, cap)
        if cap == E:
            assert rc == 0 and n.value == E and got[:E] == enc, (label, rc)
        else:
            assert rc == DX_E_CAP and ctx.L.dx_needed_bytes(ctx.h) in (0, E), (label, rc)
        hout = np.full(E + GUARD, 0xEE, dtype=np.uint8)
        _prime_need(ctx)
        rc = ctx.L.dx_dexqv_host(ctx.h, h_text.ctypes.data, len(text), 0, hout.ctypes.data, cap, C.byref(n))
        assert hout[cap:].tobytes() == b"\xEE" * (E + GUARD - cap), (label, cap)
        if cap == E:
            assert rc == 0 and hout[:E].tobytes() == enc, (label, rc)
        else:
            assert rc == DX_E_CAP and ctx.L.dx_needed_bytes(ctx.h) in (0, E), (label, rc)


def _scan_matches(ctx, orc, text):
    t = _device(text)
    st = ctx.qv_scan_dev(t.data_ptr(), len(text))
    o = orc.qv_scan(text)
    h = np.ctypeslib.as_array(st.hist)
    for k, nm in enumerate(("del_", "ins", "mrg", "sub", "delrun", "subrun")):
        assert list(h[k] + (1 if k >= 4 else 0)) == list(getattr(o, nm)), nm
    assert (st.totchar, st.nentries, st.delchar, st.subchar) == (o.totchar, o.nentries, o.delchar, o.subchar)
    return t


@pytest.mark.parametrize("env", [{}, {"chain_scan": 1}], ids=_rid)
def test_entry_counts(routed, orc, env):
    """16 383 ... 40 000 entries: the statistics, the entry-offset scan the count selects
    (k_qv_offsets alone below 16 384, k_qv_offsets + k_scan_u32 from there), the offsets, and the
    decode with discovered entries"""
    ctx = routed
    for k, v in env.items():
        ctx.route(k, v)
    from dextractor_b200 import lib as dxl
    for label, text in X.make(orc, "counts"):
        n = int(label)
        w = want(orc, "counts", label, text)
        for lossy in (False, True):
            t = _scan_matches(ctx, orc, text)
            st = ctx.qv_scan_dev(t.data_ptr(), len(text))
            cd = dxl.make_coding(st, lossy)
            out = _device(b"", 3 * len(text) + 65536)
            ctx.profile(True); ctx.profile_report()
            m, _, offs = ctx.qv_encode_dev(t.data_ptr(), len(text), cd, lossy, 0, out.data_ptr(),
                                           3 * len(text) + 65536, want_offsets=n)
            prof = ctx.profile_report(); ctx.profile(False)
            hdr = len(w["enc"][lossy]) - m
            assert out[:m].cpu().numpy().tobytes() == w["enc"][lossy][hdr:], (label, lossy)
            assert np.array_equal(offs + hdr, orc.dexqv_offsets(w["enc"][lossy], n)), (label, lossy)
            assert prof["k_qv_offsets"][0] == 1, prof
            assert ("k_scan_u32" in prof) == (X.offset_scan(n) != "k_qv_offsets"), (label, prof)
            back = orc.undexqv(w["enc"][lossy])
            assert ctx.undexqv(w["enc"][lossy]) == back, (label, lossy)
            got, guard = _decode_dev(ctx, w["enc"][lossy], len(back) + 64)
            assert got == back and guard == b"\xEE" * GUARD, (label, lossy)


# ---- long entries --------------------------------------------------------------------------------------

@pytest.mark.parametrize("env", [{}, {"two_pass": 1}], ids=_rid)
def test_long_entries_encode(routed, orc, env):
    ctx = routed
    for k, v in env.items():
        ctx.route(k, v)
    for label, text in X.make(orc, "long"):
        w = want(orc, "long", label, text)
        _scan_matches(ctx, orc, text)
        for lossy in (False, True):
            got = _dexqv_dev(ctx, text, lossy)
            assert got == w["enc"][lossy], (label, lossy, first_diff(got, w["enc"][lossy]))
        assert ctx.dexqv(text) == w["enc"][False], label


def test_long_entries_decode(routed, orc):
    """discovered entries (general path), the encoder's offsets, the decoded size, the pipelined host
    decode with windows smaller than the entry, and dx_qv_load_entries_dev of the longest entry"""
    ctx = routed
    from dextractor_b200 import lib as dxl
    seen = {}
    for label, text in X.make(orc, "long"):
        w = want(orc, "long", label, text)
        enc = w["enc"][False]
        img = _device(enc)
        assert ctx.undexqv_size_dev(img.data_ptr(), len(enc)) == len(text), label
        ctx.profile(True); ctx.profile_report()
        got, guard = _decode_dev(ctx, enc, len(text))
        prof = ctx.profile_report(); ctx.profile(False)
        assert got == text and guard == b"\xEE" * GUARD, (label, first_diff(got, text))
        seen[label, "discovered"] = sorted((k, v[0]) for k, v in prof.items() if k.startswith("k_qv_"))
        assert "k_qv_walk5" in prof and "k_qv_assemble" in prof, (label, sorted(prof))
        _, offs = _encoder_image(ctx, text)
        assert np.array_equal(offs, orc.dexqv_offsets(enc, w["nent"])), label
        ctx.profile(True); ctx.profile_report()
        got, guard = _decode_dev(ctx, enc, len(text), entry_off=offs)
        prof = ctx.profile_report(); ctx.profile(False)
        assert got == text and guard == b"\xEE" * GUARD, label
        seen[label, "offsets"] = sorted((k, v[0]) for k, v in prof.items() if k.startswith("k_qv_"))
        dec = {k: v[0] for k, v in prof.items() if k.startswith("k_qv_decode")}
        assert dec == {"k_qv_decode5": 1} and "k_qv_walk5" not in prof and "k_qv_assemble" not in prof, \
            (label, sorted(prof))
        for chunk in (0, 1 << 20):
            if chunk:
                ctx.route("pipe_chunk", chunk)
            assert ctx.undexqv(enc) == text, (label, chunk)
            ctx.route("default")
        # the longest entry alone through the batched loader
        p = X.S.parse(text)
        e = int(np.argmax(p["rlen"]))
        cd, _, used = dxl.read_coding(enc[2:])
        so = int(offs[e]) + int(X.well_bytes(p["well"])[e]) + 12
        L = int(p["rlen"][e])
        out = _device(b"", 5 * (L + 1) + GUARD)
        oo, eo = ctx.qv_load_entries_dev(img.data_ptr(), len(enc), cd, [so], [L], False, out.data_ptr(),
                                         5 * (L + 1))
        a = p["line"][e, 0]
        assert out[: 5 * (L + 1)].cpu().numpy().tobytes() == text[a: a + 5 * (L + 1)], label
        assert int(eo[0]) == int(offs[e + 1]), label
    print("long decode routes:", seen)


# the code each entry point returns for the 2^24-position entry (see the test below): the framing
# says TOOLONG; a decode that finds entries on its own finds no entry it may take (TRUNC), one given
# the offset refuses the header's read length (FORMAT), the loader refuses the length argument (ARG)
TOO_LONG_CODES = {"scan": DX_E_TOOLONG, "dexqv_host": DX_E_TOOLONG, "dexqv_dev": DX_E_TOOLONG,
                  "undexqv_host": DX_E_TRUNC, "undexqv_dev": DX_E_TRUNC, "undexqv_known": DX_E_FORMAT,
                  "size": DX_E_TRUNC, "load_entries": DX_E_ARG}


def test_entry_of_2_to_the_24_is_refused(ctx, orc):
    """The reference and the oracle take an entry of 2^24 positions; the library's framing refuses it
    (DX_E_TOOLONG, DESIGN section 2), and every decode entry point refuses the oracle's image of it
    instead of returning text.  The codes are pinned in TOO_LONG_CODES so that a change shows."""
    from dextractor_b200 import lib as dxl
    text = X.make_too_long()
    enc = orc.dexqv(text)
    got = {}

    def code(key, fn):
        with pytest.raises(dx.DexError) as e:
            fn()
        got[key] = e.value.code

    t = _device(text)
    code("scan", lambda: ctx.qv_scan_dev(t.data_ptr(), len(text)))
    code("dexqv_host", lambda: ctx.dexqv(text))
    code("dexqv_dev", lambda: _dexqv_dev(ctx, text, False))
    code("undexqv_host", lambda: ctx.undexqv(enc))
    code("undexqv_dev", lambda: _decode_dev(ctx, enc, len(text) + 65536))
    cd, _, used = dxl.read_coding(enc[2:])
    offs = np.array([2 + used, len(enc)], dtype=np.int64)             # one entry, behind key and coding
    code("undexqv_known", lambda: _decode_dev(ctx, enc, len(text) + 65536, entry_off=offs))
    img = _device(enc)
    code("size", lambda: ctx.undexqv_size_dev(img.data_ptr(), len(enc)))
    out = _device(b"", 64)
    code("load_entries", lambda: ctx.qv_load_entries_dev(img.data_ptr(), len(enc), cd, [offs[0] + 13],
                                                         [X.MAX_RLEN], False, out.data_ptr(), 64))
    print("2^24 entry:", got)
    assert got == TOO_LONG_CODES, got
