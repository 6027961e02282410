"""dx_undexqv_range_* on one GPU: an image cut into byte ranges, the ranges replayed one after the
other on one context the way the ranks of tools/undexqv_mg run them (decode, chain from the carried
position and well, text).  The range texts, concatenated, must be exactly the whole-image
dx_undexqv_dev text and the oracle's -- on the golden and fuzz files, shard images, files built to
defeat the candidate filter, every cut around entry boundaries, too-short buffers and bad arguments."""
import os

import numpy as np
import pytest
import torch

import dextractor_b200 as dx
from dextractor_b200 import lib as dxl
from dextractor_b200 import synth
from tests import fuzz
from tests.test_gpu_parity import first_diff
from tests.test_gpu_paths import _zero_rich_quiva

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
HEADMAX = 2 + 16384 + 100001


@pytest.fixture(scope="module")
def ctx():
    c = dx.Context(0)
    yield c
    c.close()


def _dev(data: bytes) -> torch.Tensor:
    t = torch.zeros(len(data) + 64, dtype=torch.uint8, device="cuda")
    t[: len(data)] = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    return t


def whole(ctx, enc: bytes, upper=False, well_in=0) -> bytes:
    img = _dev(enc)
    cap = len(enc) * 40 + 200000
    out = torch.empty(cap, dtype=torch.uint8, device="cuda")
    m = ctx.undexqv_dev(img.data_ptr(), len(enc), upper, out.data_ptr(), cap, well_in=well_in)
    return out[:m].cpu().numpy().tobytes()


def ranges(ctx, enc: bytes, cuts, upper=False, well_in=0, tail=1 << 20, img=None, stats=None):
    """decode the ranges [cuts[k], cuts[k+1]) one after the other; tail: bytes read behind a range's
    end (more when the chain asks for them).  -> the concatenated text"""
    n = len(enc)
    img = _dev(enc) if img is None else img
    head = enc[:HEADMAX]
    bounds = sorted(set([0, n] + [min(max(int(c), 0), n) for c in cuts]))
    cur = well = None
    parts = []
    for a, b in zip(bounds[:-1], bounds[1:]):
        end = min(n, b + tail)
        while True:
            buf_off = (a - 4096) & ~15 if a > 4096 else 0          # 4 KB in front of the range
            first = ctx.undexqv_range_dev(head, img.data_ptr() + buf_off, end - buf_off, buf_off, a, b, upper)
            if cur is None:
                cur, well = first, well_in
            try:
                nxt, wl = ctx.undexqv_range_chain(cur, well)
            except dxl.DexError as e:
                assert e.code == -2, e                      # DX_E_CAP: read further
                need = ctx.needed_bytes()
                assert end < need, (end, need)
                end = min(n, need)
                if stats is not None:
                    stats["longer"] = stats.get("longer", 0) + 1
                continue
            break
        assert nxt >= b or nxt == cur
        cur, well = nxt, wl
        try:
            m = ctx.undexqv_range_text_dev(None, 0)
        except dxl.DexError as e:
            assert e.code == -2
            m = ctx.needed_bytes()
        out = torch.empty(m + 64, dtype=torch.uint8, device="cuda")
        got = ctx.undexqv_range_text_dev(out.data_ptr(), out.numel())
        assert got == m
        parts.append(out[:m].cpu().numpy().tobytes())
        if stats is not None and m == 0:
            stats["empty"] = stats.get("empty", 0) + 1
    assert cur == n, (cur, n)
    return b"".join(parts)


def _cuts(rng, n, k):
    return sorted(int(x) for x in rng.integers(0, n, size=k))


def _fits(ctx, enc):
    """False: the coding has more long codes than the parallel decoder's tables hold, and the range
    calls refuse the image (DX_E_CODING, decoded whole with dx_undexqv_dev instead)"""
    img = _dev(enc)
    try:
        ctx.undexqv_range_dev(enc[:HEADMAX], img.data_ptr(), len(enc), 0, 0, len(enc))
    except dxl.DexError as e:
        assert e.code == -11 and "dx_undexqv_dev" in e.text, e
        return False
    return True


def _check(ctx, orc, enc, cut_sets, upper=False, **kw):
    want = orc.undexqv(enc, upper=upper)
    assert whole(ctx, enc, upper) == want
    if not _fits(ctx, enc):
        return False
    for cuts in cut_sets:
        got = ranges(ctx, enc, cuts, upper, **kw)
        assert got == want, (cuts, first_diff(got, want))
    return True


GOLDEN_QV = sorted(f for f in os.listdir(GOLDEN) if f.startswith("quiva_") and f.endswith(".dexqv"))


@pytest.mark.parametrize("name", GOLDEN_QV)
def test_golden_files_in_ranges(ctx, orc, name):
    enc = open(os.path.join(GOLDEN, name), "rb").read()
    rng = np.random.default_rng(len(enc))
    n = len(enc)
    sets = [[], [n // 2], [n // 3, 2 * n // 3]] + [_cuts(rng, n, k) for k in (3, 7, 16)]
    assert _check(ctx, orc, enc, sets)
    assert _check(ctx, orc, enc, sets[3:4], upper=True)


_FUZZ_FIT = []


@pytest.mark.parametrize("seed", range(40))
def test_fuzz_files_in_ranges(ctx, orc, seed):
    """(a fuzz coding the 12-bit tables cannot hold is refused with DX_E_CODING: checked in _fits)"""
    text, _ = fuzz.fuzz_quiva(seed)
    enc = orc.dexqv(text, lossy=bool(seed & 1))
    rng = np.random.default_rng(seed)
    _FUZZ_FIT.append(_check(ctx, orc, enc, [_cuts(rng, len(enc), k) for k in (1, 4, 9)], tail=int(rng.integers(0, 5000))))
    if seed == 39:
        assert sum(_FUZZ_FIT) >= 20, _FUZZ_FIT                      # most of them do go through the ranges


def _shard_image(ctx, text, well_in):
    """[0x55aa][coding][entries coded by dx_qv_encode_dev against the well of a previous shard]"""
    t = _dev(text)
    st = ctx.qv_scan_dev(t.data_ptr(), len(text))
    cd = dxl.make_coding(st, False)
    hdr = b"\xaa\x55" + dxl.write_coding(cd, text[: text.index(b"/", 1)])
    out = torch.zeros(len(text) + 65536, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    body, _, _ = ctx.qv_encode_dev(t.data_ptr(), len(text), cd, False, well_in, out.data_ptr(), out.numel())
    return hdr + out[:body].cpu().numpy().tobytes()


def _move_wells(text, n, shift):
    lines = text.split(b"\n")
    for e in range(n):
        f = lines[6 * e].split(b"/")
        f[1] = str(int(f[1]) + shift(e)).encode()
        lines[6 * e] = b"/".join(f)
    return b"\n".join(lines)


@pytest.mark.parametrize("well_in", [0, 7, 30])
def test_shard_images_in_ranges(ctx, orc, well_in):
    """a shard's first well delta is coded against the previous shard's last well; with well_in = 7
    every well lies 2 000 000 behind it: 7 843 bytes of 0xff in front of the first entry"""
    rng = np.random.default_rng(well_in)
    lengths = [int(x) for x in rng.integers(300, 6000, size=80)]
    text = synth.make_quiva(31 + well_in, lengths)
    if well_in:                                                    # every well behind well_in
        text = _move_wells(text, len(lengths), lambda e: 2_000_000 if well_in == 7 else 100)
    enc = _shard_image(ctx, text, well_in)
    want = whole(ctx, enc, well_in=well_in)
    assert want == text
    n = len(enc)
    for cuts in ([], [n // 2], _cuts(rng, n, 5), [5, 3000, 7000]):
        got = ranges(ctx, enc, cuts, well_in=well_in)
        assert got == want, (cuts, first_diff(got, want))


def _ff_runs(enc, offs):
    """(start, end) of the delta bytes of every entry (offs: entry starts, the last one = image end)"""
    out = []
    for s in offs[:-1]:
        e = s
        while enc[e] == 0xFF:
            e += 1
        out.append((int(s), int(e) + 1))
    return out


@pytest.mark.parametrize("gap", [1200, 1 << 20])
def test_long_well_gaps_straddling_a_cut(ctx, orc, gap):
    rng = np.random.default_rng(gap)
    lengths = [int(x) for x in rng.integers(200, 4000, size=40)]
    text = synth.make_quiva(5, lengths)
    text = _move_wells(text, len(lengths), lambda e: gap * (e // 7))
    enc = orc.dexqv(text)
    runs = [r for r in _ff_runs(enc, orc.dexqv_offsets(enc, len(lengths))) if r[1] - r[0] > 2]
    assert runs
    sets = []
    for s, e in runs[:4]:
        sets += [[s], [s + 1], [(s + e) // 2], [e - 1], [e], [e + 3], [s - 1, (s + e) // 2, e + 5]]
    assert _check(ctx, orc, enc, sets, tail=int(rng.integers(0, 300)))


def test_zero_rich_streams_need_the_general_walk(ctx, orc):
    text = _zero_rich_quiva(21, 60, 6000)
    enc = orc.dexqv(text)
    rng = np.random.default_rng(3)
    assert _check(ctx, orc, enc, [[], _cuts(rng, len(enc), 3), _cuts(rng, len(enc), 11)])


def test_an_entry_longer_than_three_ranges_and_ranges_without_an_entry(ctx, orc):
    text = synth.make_quiva(8, [500, 250000, 300, 40])
    enc = orc.dexqv(text)
    offs = orc.dexqv_offsets(enc, 4)
    s, e = int(offs[1]), int(offs[2])
    inner = [s + (e - s) * k // 5 for k in range(1, 5)]            # four cuts inside the long entry
    stats = {}
    want = orc.undexqv(enc)
    for tail in (0, 1000, 1 << 22):
        got = ranges(ctx, enc, [s - 3, s + 1] + inner + [e - 1, e + 2], tail=tail, stats=stats)
        assert got == want
    assert stats.get("empty", 0) >= 4 and stats.get("longer", 0) >= 1, stats


def test_every_cut_around_three_entry_boundaries(ctx, orc):
    """every cut position within 40 bytes of three entry boundaries: delta bytes, terminator, the
    fields, the first stream bytes, the previous entry's last words"""
    text = synth.make_quiva(12, [700, 30, 1500, 300, 2600, 5, 900], max_well_delta=600)
    enc = orc.dexqv(text)
    offs = orc.dexqv_offsets(enc, 7)
    want = orc.undexqv(enc)
    img = _dev(enc)
    for k in (1, 3, 5):
        for c in range(int(offs[k]) - 40, int(offs[k]) + 41):
            got = ranges(ctx, enc, [c], img=img, tail=int(c % 97))
            assert got == want, (k, c, first_diff(got, want))


def test_uppercase(ctx, orc):
    enc = orc.dexqv(synth.make_quiva(9, synth.draw_lengths(np.random.default_rng(9), 30)))
    assert _check(ctx, orc, enc, [[len(enc) // 4, len(enc) // 2]], upper=True)


def test_a_too_short_tail_asks_for_more(ctx, orc):
    lengths = synth.draw_lengths(np.random.default_rng(1), 40)
    lengths[1] = 20000
    text = synth.make_quiva(1, lengths)
    enc = orc.dexqv(text)
    assert _fits(ctx, enc)
    offs = orc.dexqv_offsets(enc, 40)
    img = _dev(enc)
    a, b = int(offs[1]) - 2, int(offs[1]) + 10                    # the long entry starts in [a, b)
    head = enc[:HEADMAX]
    first = ctx.undexqv_range_dev(head, img.data_ptr(), b + 100, 0, 0, a)
    cur, well = ctx.undexqv_range_chain(first, 0)
    buf_off = (a - 4096) & ~15 if a > 4096 else 0
    ctx.undexqv_range_dev(head, img.data_ptr() + buf_off, b + 100 - buf_off, buf_off, a, b)
    with pytest.raises(dxl.DexError) as e:
        ctx.undexqv_range_chain(cur, well)
    assert e.value.code == -2
    need = ctx.needed_bytes()
    assert int(offs[2]) <= need
    ctx.undexqv_range_dev(head, img.data_ptr() + buf_off, min(need, len(enc)) - buf_off, buf_off, a, b)
    nxt, _ = ctx.undexqv_range_chain(cur, well)
    assert nxt == int(offs[2])


def test_bad_ranges_are_refused(ctx, orc):
    enc = orc.dexqv(synth.make_quiva(15, [2000] * 30))
    img = _dev(enc)
    head, n = enc[:HEADMAX], len(enc)
    for args in [(0, n, 0, n // 2, n // 3),                        # a > b
                 (8192, n - 8192, 8192, 10000, n),                 # the buffer starts behind a - 4096
                 (0, n // 2, 0, n // 4, n)]:                       # ... and ends before b
        off, length, buf_off, a, b = args
        with pytest.raises(dxl.DexError) as e:
            ctx.undexqv_range_dev(head, img.data_ptr() + off, length, buf_off, a, b)
        assert e.value.code == -7, args
    with pytest.raises(dxl.DexError) as e:                          # no decoded range on a fresh context
        dx.Context(0).undexqv_range_chain(0, 0)
    assert e.value.code == -7


@pytest.mark.parametrize("name", ["legacy_foreign.dexqv", "legacy_old.dexqv", "legacy_foreign_old.dexqv"])
def test_legacy_images_are_refused(ctx, orc, name):
    enc = open(os.path.join(GOLDEN, name), "rb").read()
    img = _dev(enc)
    with pytest.raises(dxl.DexError) as e:
        ctx.undexqv_range_dev(enc[:HEADMAX], img.data_ptr(), len(enc), 0, 0, len(enc))
    assert e.value.code == -1 and "dx_undexqv_dev" in e.value.text
