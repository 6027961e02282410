"""The header and framing shapes of tests/header_shapes.py through the library, bit for bit against
the oracle; where the oracle refuses an input, the library must refuse it with the same code.

Routes each shape takes on a default-route decode at width 80 (asserted from the kernel profile and
from header_shapes.expected_route, so a shape that drifts onto another path fails):
  index: two-pass for every shape but wells_deltas / wells_over_cap (small files hold more than 16
         candidates in a 16 KB tile; the zero payloads make every payload offset one);
  chain: fast for window_*_in (but window_beg_in_arrow), wells_deltas / first*, zero_*, snr_all_arrow;
         general for window_*_out, window_beg_in_arrow (the .dexar prefilter also asks end < 2^27),
         wells_over_cap (a run of 2^20 + 1 0xff bytes), snr_codes_dexar (codes above 9999), and
         grammar_* (beg values of 2^27 and more);
  wells_drop1 is refused: the 0xff written for a drop of 1 misframes the image.  In .dexar a read
  length comes out negative, a format error as in the reference; for .dexta and .quiva see
  REFUSAL_CODES."""
import ctypes as C

import numpy as np
import pytest

import dextractor_b200 as dx
from tests import header_shapes as H
from tests.test_gpu_parity import first_diff
from tests.test_gpu_paths import _route_id

pytestmark = pytest.mark.gpu

ENCODE_ROUTES = [{}, {"exact_pack": 1}, {"pack2": 1}]
DECODE_ROUTES = [{}, {"no_fast": 1}, {"pack2": 1}, {"exact_index": 1}, {"chain_scan": 1}]
WIDTHS = [80, 16, 15, 7]


def _text_shapes():
    out = {}
    for kind in ("fasta", "arrow"):
        arrow = kind == "arrow"
        out[f"grammar_{kind}"] = lambda k=kind: H.grammar(k)
        for w, (field, _, _) in H.WINDOW.items():
            if not (arrow and field == "qv"):
                out[f"window_{w}_{kind}"] = lambda w=w, a=arrow: H.window(w, a)
        for c in H.WELL_CASES:
            out[f"wells_{c}_{kind}"] = lambda c=c, k=kind: H.well_jumps(k, c)
        out[f"zero_{kind}"] = lambda k=kind: H.zero_payload(k)
    out["snr_all_arrow"] = H.snr_all_arrow
    return out


TEXT_SHAPES = _text_shapes()
IMAGE_SHAPES = sorted(TEXT_SHAPES) + ["snr_codes_dexar"]
LEGACY = [(False, True, False), (False, False, True), (False, True, True), (True, True, False)]
LEGACY_IDS = ["fasta_foreign", "fasta_old", "fasta_foreign_old", "arrow_foreign"]


@pytest.fixture(scope="module")
def ctx():
    c = dx.Context(0)
    yield c
    c.close()


@pytest.fixture
def routed(ctx):
    yield ctx
    ctx.route("default")


def _set(ctx, env):
    for k, v in env.items():
        ctx.route(k, v)


def _oracle(fn, *a, **kw):
    """the oracle's result, or its error code"""
    from oracle import orc
    try:
        return fn(*a, **kw)
    except orc.OracleError as e:
        return e.code


def _lib(fn, *a, **kw):
    try:
        return fn(*a, **kw)
    except dx.DexError as e:
        return e.code


_img: dict = {}


def image(orc, name):
    """(text or None, native image, arrow) of a shape, computed once"""
    if name not in _img:
        if name == "snr_codes_dexar":
            _img[name] = (None, H.snr_codes_dexar(), True)
        else:
            text = TEXT_SHAPES[name]()
            arrow = "arrow" in name
            _img[name] = (text, orc.dexta(text, arrow=arrow), arrow)
    return _img[name]


def _dexta_raw(ctx, text, kind):
    """dx_dexta_host with room for the 0xff runs of the well shapes (several MB from a few KB)"""
    src = np.frombuffer(text, dtype=np.uint8)
    out = np.empty(64 * len(text) + (8 << 20), dtype=np.uint8)
    n = C.c_size_t(0)
    rc = ctx.L.dx_dexta_host(ctx.h, kind, src.ctypes.data, len(text), out.ctypes.data, out.size, C.byref(n))
    if rc != 0:
        raise dx.DexError(rc, ctx.L.dx_strerror(ctx.h).decode())
    return out[: n.value].tobytes()


@pytest.mark.parametrize("env", ENCODE_ROUTES, ids=_route_id)
@pytest.mark.parametrize("name", sorted(TEXT_SHAPES))
def test_encode(routed, orc, name, env):
    _set(routed, env)
    text, img, arrow = image(orc, name)
    got = _dexta_raw(routed, text, dx.ARROW if arrow else dx.FASTA)
    assert got == img, first_diff(got, img)
    # and through the device entry point
    import torch
    t = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    out = torch.full((len(img) + 4096,), 0xEE, dtype=torch.uint8, device="cuda")
    m = routed.dexta_dev(dx.ARROW if arrow else dx.FASTA, t.data_ptr(), len(text), out.data_ptr(), out.numel())
    got = out.cpu().numpy().tobytes()
    assert m == len(img) and got[:m] == img and got[m:] == b"\xEE" * 4096


def _decode_dev(ctx, img, kind, width, upper, cap):
    import torch
    d = torch.frombuffer(bytearray(img), dtype=torch.uint8).cuda()
    out = torch.full((cap + 4096,), 0xEE, dtype=torch.uint8, device="cuda")
    m = ctx.undexta_dev(kind, d.data_ptr(), len(img), width, upper, out.data_ptr(), cap)
    got = out.cpu().numpy().tobytes()
    assert got[m:] == b"\xEE" * (cap + 4096 - m)
    size = C.c_size_t(0)
    rc = ctx.L.dx_undexta_size_dev(ctx.h, kind, d.data_ptr(), len(img), width, C.byref(size))
    assert rc == 0 and size.value == m, (rc, size.value, m)
    return got[:m]


# Images the library refuses with another code than the oracle: the .dexta and .quiva images whose
# well drops by 1 (the 0xff delta byte misframes the rest).  The oracle stops at a negative read
# length (ORC_E_FORMAT); the library reports DX_E_TRUNC from its entry chain (not yet traced to the
# entry it stops at).  Both refuse; the codes are pinned so that a change shows.
REFUSAL_CODES = {"wells_drop1_fasta": -3, "quiva_wells_drop1": -3}


def _check_decode(ctx, orc, img, arrow, widths, uppers, name=None):
    kind = dx.ARROW if arrow else dx.FASTA
    for width in widths:
        for upper in uppers:
            want = _oracle(orc.undexta, img, arrow=arrow, width=width, upper=upper)
            if isinstance(want, int):
                want = REFUSAL_CODES.get(name, want)
                got = _lib(ctx.undexta, img, kind=kind, width=width, upper=upper)
                assert got == want, (width, upper)
                got = _lib(_decode_dev, ctx, img, kind, width, upper, 4 * len(img) * 5 + 65536)
                assert got == want, (width, upper)
                continue
            got = _decode_dev(ctx, img, kind, width, upper, len(want))
            assert got == want, (width, upper, first_diff(got, want))


@pytest.mark.parametrize("env", DECODE_ROUTES, ids=_route_id)
@pytest.mark.parametrize("name", IMAGE_SHAPES)
def test_decode(routed, orc, name, env):
    """dx_undexta_dev at every width, with and without upper case, and dx_undexta_size_dev"""
    _set(routed, env)
    _, img, arrow = image(orc, name)
    _check_decode(routed, orc, img, arrow, WIDTHS, [False] if arrow else [False, True], name)


@pytest.mark.parametrize("name", IMAGE_SHAPES)
def test_decode_host_entry_points(ctx, orc, name):
    _, img, arrow = image(orc, name)
    kind = dx.ARROW if arrow else dx.FASTA
    want = _oracle(orc.undexta, img, arrow=arrow)
    if isinstance(want, int):
        want = REFUSAL_CODES.get(name, want)
    got = _lib(ctx.undexta, img, kind=kind)
    assert got == want, first_diff(got, want) if isinstance(got, bytes) and isinstance(want, bytes) else (got, want)
    if isinstance(want, bytes):
        src = np.frombuffer(img, dtype=np.uint8)
        size = C.c_size_t(0)
        assert ctx.L.dx_undexta_size_host(ctx.h, kind, src.ctypes.data, len(img), 80, C.byref(size)) == 0
        assert size.value == len(want)


def _route_of(prof):
    index = H.INDEX_TWO_PASS if "k_pred_count" in prof else H.INDEX_SLOTS if "k_pred_slots" in prof else None
    chain = H.CHAIN_GENERAL if "k_unpack" in prof else H.CHAIN_FAST if "k_unpack3" in prof else None
    return index, chain


@pytest.mark.parametrize("name", IMAGE_SHAPES)
def test_route(ctx, orc, name):
    """the default route of a decode at width 80 is the one the shape is built for"""
    _, img, arrow = image(orc, name)
    want = _oracle(orc.undexta, img, arrow=arrow)
    if isinstance(want, int):
        want = REFUSAL_CODES.get(name, want)
    ctx.route("default")
    ctx.profile(True); ctx.profile_report()
    got = _lib(_decode_dev, ctx, img, dx.ARROW if arrow else dx.FASTA, 80, False,
               len(want) if isinstance(want, bytes) else 1 << 20)
    prof = ctx.profile_report(); ctx.profile(False)
    print(name, sorted((k, v[0]) for k, v in prof.items()))
    assert got == want
    if isinstance(want, int):
        return
    route = _route_of(prof)
    assert route == H.expected_route(img, arrow), (route, sorted(prof))
    assert route[1] == INTENDED_CHAIN.get(name, route[1]), (name, route)
    if name.startswith("zero_"):
        assert route[0] == H.INDEX_TWO_PASS


# the chain each shape is built to reach (grammar and the dropping wells take what their content gives)
INTENDED_CHAIN = {"window_beg_in_fasta": H.CHAIN_FAST, "window_len_in_fasta": H.CHAIN_FAST,
                  "window_qv_in_fasta": H.CHAIN_FAST, "window_len_in_arrow": H.CHAIN_FAST,
                  "window_beg_in_arrow": H.CHAIN_GENERAL,     # ARCAND also asks end < 2^27
                  "snr_codes_dexar": H.CHAIN_GENERAL, "snr_all_arrow": H.CHAIN_FAST,
                  "zero_fasta": H.CHAIN_FAST, "zero_arrow": H.CHAIN_FAST}
for _k in ("fasta", "arrow"):
    INTENDED_CHAIN.update({f"window_{w}_out_{_k}": H.CHAIN_GENERAL for w in ("beg", "len", "qv")})
    INTENDED_CHAIN.update({f"wells_{c}_{_k}": H.CHAIN_FAST for c in ("deltas", "first0", "first255", "first256")})
    INTENDED_CHAIN[f"wells_over_cap_{_k}"] = H.CHAIN_GENERAL


# ---- legacy forms ------------------------------------------------------------------------------------

@pytest.mark.parametrize("env", DECODE_ROUTES, ids=_route_id)
@pytest.mark.parametrize("form", LEGACY, ids=LEGACY_IDS)
def test_legacy_forms(routed, orc, form, env):
    """foreign byte order and the old 16-bit layout, decoded on the host-walked general path"""
    arrow, flip, old = form
    _set(routed, env)
    text = H.legacy_text(11, arrow)
    img = H.build_2bit(text, arrow, flip, old)
    assert H.build_2bit(text, arrow) == orc.dexta(text, arrow=arrow)
    _check_decode(routed, orc, img, arrow, WIDTHS, [False] if arrow else [False, True])
    routed.profile(True); routed.profile_report()
    _decode_dev(routed, img, dx.ARROW if arrow else dx.FASTA, 80, False, len(orc.undexta(img, arrow=arrow)))
    prof = routed.profile_report(); routed.profile(False)
    assert "k_unpack" in prof and "k_pk_cand_prep" not in prof, sorted(prof)


@pytest.mark.parametrize("form", [f for f in LEGACY if not f[2]], ids=[i for f, i in zip(LEGACY, LEGACY_IDS) if not f[2]])
@pytest.mark.parametrize("drop", H.WELL_DROPS)
def test_legacy_forms_with_a_dropping_well(ctx, orc, drop, form):
    arrow, flip, old = form
    img = H.build_2bit(H.well_jumps("arrow" if arrow else "fasta", f"drop{drop}"), arrow, flip, old)
    _check_decode(ctx, orc, img, arrow, [80, 15], [False])


# ---- .quiva ------------------------------------------------------------------------------------------

QUIVA_SHAPES = ["grammar"] + [f"wells_{c}" for c in H.WELL_CASES]


def _quiva(name):
    return H.grammar("quiva") if name == "grammar" else H.well_jumps("quiva", name[6:])


def _dexqv_raw(ctx, text, cap):
    src = np.frombuffer(text, dtype=np.uint8)
    out = np.empty(cap, dtype=np.uint8)
    n = C.c_size_t(0)
    rc = ctx.L.dx_dexqv_host(ctx.h, src.ctypes.data, len(text), 0, out.ctypes.data, cap, C.byref(n))
    if rc != 0:
        raise dx.DexError(rc, ctx.L.dx_strerror(ctx.h).decode())
    return out[: n.value].tobytes()


@pytest.mark.parametrize("name", QUIVA_SHAPES)
def test_quiva(ctx, orc, name):
    """dexqv, and undexqv on the host, on the device with discovered entries and with the entry offsets
    of the oracle; refusals with the oracle's code"""
    import torch
    text = _quiva(name)
    cap = 3 * len(text) + (16 << 20)
    enc = orc._run(orc.lib().orc_dexqv, text, cap, 0)
    assert _dexqv_raw(ctx, text, cap) == enc
    want = _oracle(orc.undexqv, enc)
    if isinstance(want, int):
        want = REFUSAL_CODES.get(f"quiva_{name}", want)
    got = _lib(ctx.undexqv, enc)
    assert got == want, (got, want) if isinstance(want, int) or isinstance(got, int) else first_diff(got, want)
    img = torch.frombuffer(bytearray(enc), dtype=torch.uint8).cuda()
    back = torch.full((len(text) * 2 + 65536,), 0xEE, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    got = _lib(ctx.undexqv_dev, img.data_ptr(), len(enc), False, back.data_ptr(), back.numel())
    if isinstance(want, int):
        assert got == want
        return
    assert got == len(want) and back[:got].cpu().numpy().tobytes() == want
    offs = orc.dexqv_offsets(enc, text.count(b"\n") // 6)
    back.fill_(0xEE)
    torch.cuda.synchronize()
    m = ctx.undexqv_dev(img.data_ptr(), len(enc), False, back.data_ptr(), back.numel(), entry_off=offs)
    assert m == len(want) and back[:m].cpu().numpy().tobytes() == want


@pytest.mark.parametrize("i", range(len(H.GRAMMAR_QUIVA_REFUSED)))
def test_quiva_headers_without_rq_are_refused(ctx, orc, i):
    text = H.grammar_quiva_refused(i)
    with pytest.raises(orc.OracleError) as e:
        orc.dexqv(text)
    with pytest.raises(dx.DexError) as g:
        ctx.dexqv(text)
    assert g.value.code == e.value.code
