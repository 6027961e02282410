"""The crafted QV shapes of tests/qv_shapes.py (code tables that defeat the lane speculation, stream
ends on exact subsequence boundaries, run-parity traps, dense escapes, 16-bit runs) through every
route of the library, bit-exact against the oracle; exact output capacities with guard bytes; and
the run of 65536 that the format cannot hold."""
import ctypes as C

import numpy as np
import pytest

import dextractor_b200 as dx
from tests import qv_shapes as Q
from tests.test_gpu_parity import first_diff
from tests.test_gpu_paths import ROUTES, _route_id

pytestmark = pytest.mark.gpu

SHAPES = sorted(Q.SHAPES)
ALL_ROUTES = ROUTES + [{"pipe_chunk": 65536}, {"pipe_chunk": 262144}]
DX_E_FORMAT, DX_E_CAP, DX_E_TRUNC = -1, -2, -3
GUARD = 4096


@pytest.fixture(scope="module")
def ctx():
    c = dx.Context(0)
    yield c
    c.close()


@pytest.fixture
def routed(ctx):
    """ctx with routes set by the test; every route back to its default afterwards"""
    yield ctx
    ctx.route("default")


_want: dict = {}


def want(orc, name):
    """the oracle's images and texts of one shape, computed once"""
    if name not in _want:
        text = Q.make(name)
        enc, lenc = orc.dexqv(text), orc.dexqv(text, lossy=True)
        _want[name] = dict(text=text, enc=enc, lenc=lenc, back=orc.undexqv(enc),
                           upper=orc.undexqv(enc, upper=True), lback=orc.undexqv(lenc),
                           nent=text.count(b"\n") // 6)
    return _want[name]


def _set(ctx, env):
    for k, v in env.items():
        ctx.route(k, v)


@pytest.mark.parametrize("env", ALL_ROUTES, ids=_route_id)
@pytest.mark.parametrize("name", SHAPES)
def test_shape_on_every_route(routed, orc, name, env):
    ctx = routed
    _set(ctx, env)
    w = want(orc, name)
    assert ctx.dexqv(w["text"]) == w["enc"]
    assert ctx.dexqv(w["text"], lossy=True) == w["lenc"]
    got = ctx.undexqv(w["enc"])
    assert got == w["back"] == w["text"], first_diff(got, w["back"])
    got = ctx.undexqv(w["enc"], upper=True)
    assert got == w["upper"], first_diff(got, w["upper"])
    got = ctx.undexqv(w["lenc"])
    assert got == w["lback"], first_diff(got, w["lback"])


def _decode_dev(ctx, enc, n_out, entry_off=None, upper=False):
    import torch
    img = torch.frombuffer(bytearray(enc), dtype=torch.uint8).cuda()
    back = torch.full((n_out + GUARD,), 0xEE, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    m = ctx.undexqv_dev(img.data_ptr(), len(enc), upper, back.data_ptr(), n_out, entry_off=entry_off)
    ctx.sync()
    out = back.cpu().numpy().tobytes()
    return out[:m], out[n_out:]


@pytest.mark.parametrize("env", [{}, {"decoder": 6}, {"decoder": 1}], ids=_route_id)
@pytest.mark.parametrize("name", SHAPES)
def test_shape_with_known_entry_offsets(routed, orc, name, env):
    """With the entry offsets given, the decode is one launch of the warp- and/or lane-per-entry
    kernel (or of the sequential one when forced) and never k_qv_assemble"""
    ctx = routed
    _set(ctx, env)
    w = want(orc, name)
    offs = orc.dexqv_offsets(w["enc"], w["nent"])
    ctx.profile(True); ctx.profile_report()
    got, guard = _decode_dev(ctx, w["enc"], len(w["back"]), entry_off=offs)
    prof = ctx.profile_report(); ctx.profile(False)
    assert got == w["back"], first_diff(got, w["back"])
    assert guard == b"\xEE" * GUARD
    assert "k_qv_assemble" not in prof, sorted(prof)
    dec = {k: v[0] for k, v in prof.items() if k.startswith("k_qv_decode")}
    if env.get("decoder") == 1:
        assert dec == {"k_qv_decode": 1}, prof
    else:
        assert dec and set(dec) <= {"k_qv_decode5", "k_qv_decode6"} and set(dec.values()) == {1}, prof


@pytest.mark.parametrize("name", SHAPES)
def test_shape_with_discovered_entries(routed, orc, name):
    """Discovered entries (no offsets).  Only the bytes are asserted: a decoder that stops falling
    back is better, not wrong.  The routes seen on a B200 with this library:
      fixed3 / fixed5 / fixed6   the give-up shapes (no lane meets the true path, the fix point
                                 needs more than 12 rounds): the in-place speculative decode gives
                                 them up, then the general path -- k_qv_walk5 once per entry (24),
                                 one k_qv_decode5 and k_qv_assemble;
      fixed4, runs_16bit         also leave the in-place form: a second k_qv_decode5_spec and
                                 k_qv_assemble (fixed4 with one k_qv_walk5 and k_qv_decode5);
      fixed1, exact_ends,        one in-place k_qv_decode5_spec launch.
      esc_dense, run_parity"""
    ctx = routed
    w = want(orc, name)
    ctx.profile(True); ctx.profile_report()
    got, guard = _decode_dev(ctx, w["enc"], len(w["back"]))
    prof = ctx.profile_report(); ctx.profile(False)
    print(f"{name}: {sorted((k, v[0]) for k, v in prof.items())}")
    assert got == w["back"], first_diff(got, w["back"])
    assert guard == b"\xEE" * GUARD


# ---- exact capacities --------------------------------------------------------------------------------

CAP_SHAPES = ["exact_ends", "fixed5", "esc_dense"]


def _prime_need(ctx):
    """a call that fails with DX_E_CAP and a large known need: a later DX_E_CAP that leaves this
    value in dx_needed_bytes reports a stale size"""
    from dextractor_b200 import synth
    fasta = synth.make_fasta(5, [40000] * 120)
    src = np.frombuffer(fasta, dtype=np.uint8)
    out = np.empty(64, dtype=np.uint8)
    n = C.c_size_t(0)
    rc = ctx.L.dx_dexta_host(ctx.h, dx.FASTA, src.ctypes.data, len(fasta), out.ctypes.data, 64, C.byref(n))
    assert rc == DX_E_CAP
    need = ctx.L.dx_needed_bytes(ctx.h)
    assert need > 1_000_000
    return need


def _undex_host_raw(ctx, enc, cap):
    src = np.frombuffer(enc, dtype=np.uint8)
    out = np.full(cap + GUARD, 0xEE, dtype=np.uint8)
    n = C.c_size_t(0)
    rc = ctx.L.dx_undexqv_host(ctx.h, src.ctypes.data, len(enc), 0, out.ctypes.data, cap, C.byref(n))
    return rc, out.tobytes(), n.value


def _undex_dev_raw(ctx, enc, cap):
    import torch
    img = torch.frombuffer(bytearray(enc), dtype=torch.uint8).cuda()
    back = torch.full((cap + GUARD,), 0xEE, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    n = C.c_size_t(0)
    rc = ctx.L.dx_undexqv_dev(ctx.h, img.data_ptr(), len(enc), 0, back.data_ptr(), cap, C.byref(n),
                              None, 0, 0)
    ctx.L.dx_sync(ctx.h)
    return rc, back.cpu().numpy().tobytes(), n.value


@pytest.mark.parametrize("env", ALL_ROUTES, ids=_route_id)
@pytest.mark.parametrize("name", CAP_SHAPES)
def test_undexqv_at_exact_capacity(routed, orc, name, env):
    """Output buffers of exactly the text's size decode, and nothing after the text changes; one byte
    less is DX_E_CAP, with dx_needed_bytes the exact size or 0 -- never what an earlier call needed"""
    ctx = routed
    _set(ctx, env)
    w = want(orc, name)
    L = len(w["back"])
    for raw in (_undex_host_raw, _undex_dev_raw):
        rc, out, n = raw(ctx, w["enc"], L)
        assert rc == 0 and n == L, (raw.__name__, rc, ctx.L.dx_strerror(ctx.h))
        assert out[:L] == w["back"], (raw.__name__, first_diff(out[:L], w["back"]))
        assert out[L:] == b"\xEE" * GUARD, raw.__name__
        stale = _prime_need(ctx)
        rc, out, n = raw(ctx, w["enc"], L - 1)
        assert rc == DX_E_CAP, (raw.__name__, rc)
        need = ctx.L.dx_needed_bytes(ctx.h)
        assert need in (0, L), (raw.__name__, need, stale, L)
        assert out[L - 1:] == b"\xEE" * GUARD, raw.__name__


@pytest.mark.parametrize("env", [{}, {"two_pass": 1}, {"chain_scan": 1}], ids=_route_id)
@pytest.mark.parametrize("name", CAP_SHAPES)
def test_dexqv_at_exact_capacity(routed, orc, name, env):
    import torch
    ctx = routed
    _set(ctx, env)
    w = want(orc, name)
    E = len(w["enc"])
    text = torch.frombuffer(bytearray(w["text"]), dtype=torch.uint8).cuda()
    for cap in (E, E - 1):
        out = torch.full((E + GUARD,), 0xEE, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        stale = _prime_need(ctx)
        n = C.c_size_t(0)
        rc = ctx.L.dx_dexqv_dev(ctx.h, text.data_ptr(), len(w["text"]), 0, out.data_ptr(), cap, C.byref(n))
        ctx.L.dx_sync(ctx.h)
        got = out.cpu().numpy().tobytes()
        assert got[cap:] == b"\xEE" * (E + GUARD - cap), cap
        if cap == E:
            assert rc == 0 and n.value == E and got[:E] == w["enc"], (rc, ctx.L.dx_strerror(ctx.h))
        else:
            assert rc == DX_E_CAP, rc
            assert ctx.L.dx_needed_bytes(ctx.h) in (0, E), (ctx.L.dx_needed_bytes(ctx.h), stale, E)
    h_text = np.frombuffer(w["text"], dtype=np.uint8)
    for cap in (E, E - 1):
        out = np.full(E + GUARD, 0xEE, dtype=np.uint8)
        _prime_need(ctx)
        n = C.c_size_t(0)
        rc = ctx.L.dx_dexqv_host(ctx.h, h_text.ctypes.data, len(w["text"]), 0, out.ctypes.data, cap, C.byref(n))
        assert out[cap:].tobytes() == b"\xEE" * (E + GUARD - cap), cap
        if cap == E:
            assert rc == 0 and out[:E].tobytes() == w["enc"], rc
        else:
            assert rc == DX_E_CAP and ctx.L.dx_needed_bytes(ctx.h) in (0, E), (rc, ctx.L.dx_needed_bytes(ctx.h))


# ---- the 16-bit run literal -----------------------------------------------------------------------

def _encoder_image(ctx, text):
    """the image and its entry offsets as an application gets them from dx_qv_encode_dev (the
    offsets the file does not store; the oracle can only find them by decoding)"""
    import torch
    from dextractor_b200 import lib as dxl
    t = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    cd = dxl.make_coding(ctx.qv_scan_dev(t.data_ptr(), len(text)), False)
    hdr = b"\xaa\x55" + dxl.write_coding(cd, text[: text.index(b"/", 1)])
    enc = torch.zeros(3 * len(text) + 65536, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    ctx.h2d(enc.data_ptr(), hdr)
    nent = text.count(b"\n") // 6
    body, _, offs = ctx.qv_encode_dev(t.data_ptr(), len(text), cd, False, 0, enc.data_ptr() + len(hdr),
                                      enc.numel() - len(hdr), want_offsets=nent)
    return enc[: len(hdr) + body].cpu().numpy().tobytes(), offs + len(hdr)


# the code each route gives for the image with a run of 65536 (see the test below)
OVERLONG_CODES = {"host": DX_E_TRUNC, "dev": DX_E_TRUNC, "known": DX_E_TRUNC}


@pytest.mark.parametrize("env", ALL_ROUTES, ids=_route_id)
def test_run_of_65536_is_refused(routed, orc, env):
    """A run of 65536 run characters is written as the run escape and a 16-bit literal of 0, as the
    reference's Encode_Run writes it; the image then does not decode.  The GPU encoder writes the
    oracle's bytes, and every decode route refuses the image instead of returning text: the host
    call, the device call with discovered entries, and the device call with the entry offsets
    dx_qv_encode_dev reports.  The oracle stops at the first run that overshoots its line
    (ORC_E_FORMAT).  The library reports which check caught it; the codes are pinned per route in
    OVERLONG_CODES so that a change shows."""
    ctx = routed
    _set(ctx, env)
    text = Q.make("runs_over_16bit")
    enc = orc.dexqv(text)
    assert ctx.dexqv(text) == enc
    with pytest.raises(orc.OracleError) as e:
        orc.undexqv(enc)
    assert e.value.code == -1
    img, offs = _encoder_image(ctx, text)
    assert img == enc
    got = {}
    with pytest.raises(dx.DexError) as e:
        ctx.undexqv(enc)
    got["host"] = e.value
    with pytest.raises(dx.DexError) as e:
        _decode_dev(ctx, enc, len(text) + 65536)
    got["dev"] = e.value
    with pytest.raises(dx.DexError) as e:
        _decode_dev(ctx, enc, len(text) + 65536, entry_off=offs)
    got["known"] = e.value
    print(_route_id(env), {k: (v.code, v.text) for k, v in got.items()})
    assert {k: v.code for k, v in got.items()} == OVERLONG_CODES, got


def test_encoder_offsets_match_the_oracle(ctx, orc):
    """(the offsets the test above decodes with are the ones the decoders get on valid images)"""
    text = Q.make("exact_ends")
    img, offs = _encoder_image(ctx, text)
    assert img == orc.dexqv(text)
    assert list(offs) == list(orc.dexqv_offsets(img, text.count(b"\n") // 6))
