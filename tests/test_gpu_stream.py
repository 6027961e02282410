"""The six single-GPU tools on files larger than one window of device memory (DEXB200_WINDOW): every
output byte for byte against the same tool's one-window run and against the oracle, with windows cut
where a cut is most likely to go wrong; errors in a late window reported as the one-window run reports
them; device memory bounded by the window, not the file; and the two 2-bit entry points the windows
are built on (dx_dexta_part_dev, dx_undexta_window_dev) through ctypes."""
import hashlib
import os
import re
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from dextractor_b200 import synth
from tests import cases, fuzz

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "tools", "bin")
KIB64, MIB1_7 = 64 << 10, (1 << 20) + 7

# kind -> (encoder, decoder, text extension, image extension)
TOOLS = {"fasta": ("dexta", "undexta", ".fasta", ".dexta"),
         "arrow": ("dexar", "undexar", ".arrow", ".dexar"),
         "quiva": ("dexqv", "undexqv", ".quiva", ".dexqv")}


@pytest.fixture()
def tmp():
    d = tempfile.mkdtemp(prefix="dxstream_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    yield d
    shutil.rmtree(d, ignore_errors=True)


@pytest.fixture(scope="module")
def ctx():
    import dextractor_b200 as dx
    c = dx.Context(0)
    yield c
    c.close()


def _write(path, data):
    with open(path, "wb") as f:
        f.write(data)


def _read(path):
    with open(path, "rb") as f:
        return f.read()


def _tool(tool, paths, *flags, window=None, stdin=None, check=True, arena_cap=None):
    env = dict(os.environ)
    env.pop("DEXB200_WINDOW", None)
    env.pop("DEXB200_ARENA_CAP", None)
    if window is not None:
        env["DEXB200_WINDOW"] = str(window)
    if arena_cap is not None:
        env["DEXB200_ARENA_CAP"] = str(arena_cap)
    p = subprocess.run([os.path.join(BIN, tool), "-k", *flags, *paths], capture_output=True, env=env,
                       input=stdin)
    if check:
        assert p.returncode == 0, p.stderr.decode()
    return p


def _windows(stderr: bytes):
    """the -v summary lines, in file order: (windows, largest window, peak held)"""
    return [tuple(int(x) for x in m) for m in
            re.findall(rb"  (\d+) windows, largest (\d+) bytes, peak device memory held (\d+) bytes", stderr)]


def _expect(kind, text, lossy=False, upper=False, width=80):
    from oracle import orc
    if kind == "quiva":
        img = orc.dexqv(text, lossy=lossy)
        return img, orc.undexqv(img, upper=upper)
    img = orc.dexta(text, arrow=(kind == "arrow"))
    return img, orc.undexta(img, arrow=(kind == "arrow"), width=width, upper=upper)


def _roundtrip(tmp, kind, texts, window, enc_flags=(), dec_flags=(), expect=None, multi=True):
    """encode then decode every text at this window; both against the oracle (or `expect`) and against
    the one-window run; -> the number of windows each run took"""
    enc, dec, src, dst = TOOLS[kind]
    names = []
    for i, t in enumerate(texts):
        base = os.path.join(tmp, f"w{i}")
        _write(base + src, t)
        names.append(base)
    p = _tool(enc, [b + src for b in names], "-v", *enc_flags, window=window)
    wins = _windows(p.stderr)
    imgs = [_read(b + dst) for b in names]
    q = _tool(dec, [b + dst for b in names], "-v", *dec_flags, window=window)
    wins += _windows(q.stderr)
    backs = [_read(b + src) for b in names]
    from oracle import orc
    for i, t in enumerate(texts):
        want_img, want_back = expect[i] if expect is not None else _expect(kind, t)
        assert imgs[i] == want_img, (kind, i, window)
        assert backs[i] == want_back, (kind, i, window)
        if orc.have_ref():                                      # and the reference tools' bytes
            assert orc.ref_tool(enc, t, *enc_flags)[0] == imgs[i], (kind, i)
            assert orc.ref_tool(dec, imgs[i], *dec_flags)[0] == backs[i], (kind, i)
    if multi:
        assert wins and all(w[0] > 1 for w in wins), wins
    for b in names:
        for e in (src, dst):
            os.remove(b + e)
    return wins


def _big(texts, window):
    w = max(window, KIB64)
    return [t for t in texts if len(t) > w]


# ---- 1. every tool, three window sizes, the shared cases and the fuzz files -----------------------------

def _corpus(kind):
    texts = list(cases.all_cases()[kind].values())
    for seed in range(40):
        if kind == "quiva":
            texts.append(fuzz.fuzz_quiva(seed))
        else:
            fa, ar, _ = fuzz.fuzz_fasta_arrow(seed)
            texts.append(fa if kind == "fasta" else ar)
    if kind != "quiva":       # encode only: the header disagrees with the sequence
        texts = [t for t in texts if t != cases.all_cases()[kind].get("enc_only_len_mismatch")]
    return texts


@pytest.mark.parametrize("kind", ["fasta", "arrow", "quiva"])
@pytest.mark.parametrize("window", [KIB64, MIB1_7])
def test_cases_and_fuzz_files_in_windows(tmp, kind, window):
    texts = _big(_corpus(kind), window)
    if not texts:
        pytest.skip("no file of this corpus is larger than the window")
    _roundtrip(tmp, kind, texts, window)


@pytest.mark.parametrize("kind", ["fasta", "arrow", "quiva"])
def test_cases_and_fuzz_files_one_byte_short_of_one_window(tmp, kind):
    for t in _big(_corpus(kind), 0):
        _roundtrip(tmp, kind, [t], len(t) - 1)


def _synthetic(kind, size):
    rng = np.random.default_rng({"fasta": 1, "arrow": 2, "quiva": 3}[kind])
    if kind == "quiva":
        return synth.make_quiva(31, synth.lengths_for_bytes(rng, size, 6.0))
    return (synth.make_fasta if kind == "fasta" else synth.make_arrow)(32, synth.lengths_for_bytes(rng, size, 1.02))


@pytest.mark.parametrize("kind", ["fasta", "arrow", "quiva"])
def test_a_256_mb_file_at_every_window_size(tmp, kind):
    text = _synthetic(kind, 256 << 20)
    enc, dec, src, dst = TOOLS[kind]
    base = os.path.join(tmp, "big")
    _write(base + src, text)
    _tool(enc, [base + src])
    one_img = _read(base + dst)
    _tool(dec, [base + dst])
    one_back = hashlib.sha256(_read(base + src)).digest()
    want_img, want_back = _expect(kind, text)
    assert one_img == want_img
    assert one_back == hashlib.sha256(want_back).digest()
    del want_back
    for window in (KIB64, MIB1_7, len(text) - 1):
        _write(base + src, text)
        p = _tool(enc, [base + src], "-v", window=window)
        assert _read(base + dst) == one_img, window
        q = _tool(dec, [base + dst], "-v", window=window)
        assert hashlib.sha256(_read(base + src)).digest() == one_back, window
        assert all(w[0] > 1 for w in _windows(p.stderr) + _windows(q.stderr))


# ---- 2. cut shapes ---------------------------------------------------------------------------------------

def test_entries_longer_than_the_window(tmp):
    q = synth.make_quiva(41, [3000, 200000, 5000, 200000])
    _roundtrip(tmp, "quiva", [q], KIB64)
    fa = synth.make_fasta(42, [1000, 10_000_000, 2000])
    _roundtrip(tmp, "fasta", [fa], MIB1_7)


def test_quality_lines_that_start_with_an_at_sign(tmp):
    def at(i, s):
        for line in s:
            line[::97] = ord("@")
    q = synth.make_quiva(43, [7000] * 60, stream_hook=at)
    for window in (KIB64, KIB64 + 1, KIB64 + 4095):
        _roundtrip(tmp, "quiva", [q], window)


@pytest.mark.parametrize("kind", ["fasta", "quiva"])
def test_a_file_that_is_an_exact_multiple_of_the_window(tmp, kind):
    for size in range(3 << 20, 4 << 20, 50_000):
        text = _synthetic(kind, size)
        d = next((d for d in range(2, 41) if len(text) % d == 0), 0)
        if d:
            break
    assert d, "no size in the sweep is a multiple of a window size"
    _roundtrip(tmp, kind, [text], len(text) // d)


def _gap_fasta():
    m = synth.MOVIE.encode()
    gap = (1 << 20) + 10_000
    return (synth.make_fasta(44, [2000] * 200) + b">%s/%d/0_100 RQ=0.8\n%s\n" % (m, gap, b"acgt" * 25)
            + b">%s/%d/0_50 RQ=0.8\n%s\n" % (m, gap + 3, b"ac" * 25))


@pytest.mark.parametrize("kind", ["fasta", "quiva"])
def test_a_long_well_gap_straddling_a_window_edge(tmp, kind):
    from oracle import orc
    if kind == "fasta":
        text = _gap_fasta()
        img = orc.dexta(text)
    else:
        m = b"@" + synth.MOVIE.encode() + b"/"
        text = synth.make_quiva(46, [2000] * 150) + synth.make_quiva(47, [2000] * 5).replace(m, m + b"104857")
        img = orc.dexqv(text)
    run = img.find(b"\xff" * 4000)
    assert run > KIB64
    for window in (run - 16, run + 1000, run + 4100):
        _roundtrip(tmp, kind, [text], window)


def test_zero_rich_dexqv_with_false_candidates(tmp):
    from tests.test_gpu_paths import _zero_rich_quiva
    text = _zero_rich_quiva(21, 60, 6000)
    _roundtrip(tmp, "quiva", [text], KIB64)


def test_run_characters_fixed_late(tmp):
    late = synth.make_quiva(48, [9000] * 30, stream_hook=lambda i, s: (
        s[1].__setitem__(slice(None), ord("a")) if i < 14 else None))
    few = synth.make_quiva(49, [8000] * 11)                     # < 100 000 positions: subChar fixed late
    short = synth.make_quiva(50, [1500] * 50)                   # too short for a subChar at all
    _roundtrip(tmp, "quiva", [late, few, short], KIB64)


def test_flags_in_windows(tmp):
    from oracle import orc
    q = cases.all_cases()["quiva"]["lognormal_40"]
    img = orc.dexqv(q, lossy=True)
    _roundtrip(tmp, "quiva", [q], KIB64, enc_flags=("-l",), dec_flags=("-U",),
               expect=[(img, orc.undexqv(img, upper=True))])
    fa = cases.all_cases()["fasta"]["lognormal_40"]
    for w in (1, 60, 200):
        img = orc.dexta(fa)
        _roundtrip(tmp, "fasta", [fa], KIB64, dec_flags=(f"-w{w}", "-U"),
                   expect=[(img, orc.undexta(img, width=w, upper=True))])


# ---- 3. pipes ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("kind", ["fasta", "arrow"])
def test_pipes_in_windows(kind):
    from oracle import orc
    enc, dec, _, _ = TOOLS[kind]
    text = cases.all_cases()[kind]["lognormal_40"]
    img = orc.dexta(text, arrow=(kind == "arrow"))
    p = _tool(enc, [], "-i", "-v", window=KIB64, stdin=text)
    assert p.stdout == img and _windows(p.stderr)[0][0] > 1
    q = _tool(dec, [], "-i", "-v", window=KIB64, stdin=img)
    assert q.stdout == orc.undexta(img, arrow=(kind == "arrow")) and _windows(q.stderr)[0][0] > 1
    assert _tool(enc, [], "-i", stdin=text).stdout == img


# ---- 4. errors in a late window ------------------------------------------------------------------------

def _same_failure(tmp, tool, name, data):
    path = os.path.join(tmp, name)
    _write(path, data)
    one = _tool(tool, [path], check=False)
    win = _tool(tool, [path], window=KIB64, check=False)
    assert one.returncode != 0
    assert (win.returncode, win.stderr) == (one.returncode, one.stderr)
    assert _read(path) == data                                     # the source survives
    return one


def test_errors_in_a_late_window(tmp):
    from oracle import orc
    q = synth.make_quiva(51, [5000] * 80)
    bad = q + b"@m/99999/0_4 RQ=0.8\nabcd\nacgt\nabcd\nabc\nabcd\n"
    p = _same_failure(tmp, "dexqv", "q.quiva", bad)
    assert b"not the same length" in p.stderr
    fa = synth.make_fasta(52, [3000] * 100)
    p = _same_failure(tmp, "dexta", "h.fasta", fa + b">m/garbage\nacgt\n")
    assert b"incorrectly formatted" in p.stderr
    p = _same_failure(tmp, "dexta", "l.fasta", fa + b">m/5000/0_100000 RQ=0.8\n" + b"a" * 100000 + b"\n")
    assert b"too long" in p.stderr and b"entry 101" in p.stderr
    img = orc.dexta(fa)
    p = _same_failure(tmp, "undexta", "t.dexta", img[:-7])
    assert p.returncode == 2
    img = orc.dexqv(q)
    p = _same_failure(tmp, "undexqv", "t.dexqv", img[:-50])
    assert p.returncode == 2


# ---- 5. memory bounded by the window ---------------------------------------------------------------------

def test_device_memory_is_bounded_by_the_window(tmp, ctx):
    peaks = {}
    for size in (64 << 20, 256 << 20):
        text = _synthetic("quiva", size)
        base = os.path.join(tmp, f"m{size}")
        _write(base + ".quiva", text)
        p = _tool("dexqv", [base + ".quiva"], "-v", window=8 << 20)
        q = _tool("undexqv", [base + ".dexqv"], "-v", window=8 << 20)
        peaks[size] = (_windows(p.stderr)[0][2], _windows(q.stderr)[0][2])
        assert _read(base + ".quiva") == text
    for k in range(2):
        a, b = peaks[64 << 20][k], peaks[256 << 20][k]
        assert abs(a - b) <= 0.1 * max(a, b), peaks
    free, total, held0 = ctx.mem_info()
    assert 0 < free <= total
    ctx.dexqv(text)                                              # the 256 MB file in one window
    held = ctx.mem_info()[2]
    assert held > held0
    assert max(peaks[256 << 20]) < held / 2, (peaks, held)


def test_windows_halve_when_the_device_runs_out_of_memory(tmp):
    """DEXB200_ARENA_CAP caps the library's scratch arena: the one-window call fails with DX_E_NOMEM, the
    tool halves the window until a window fits (the .quiva encode needs more scratch than its scan, so
    dexqv's second pass halves too), and the bytes are those of the run without a cap"""
    cap = 64 << 20
    for kind in ("quiva", "fasta"):
        enc, dec, src, dst = TOOLS[kind]
        text = _synthetic(kind, 48 << 20)
        base = os.path.join(tmp, "nomem")
        _write(base + src, text)
        _tool(enc, [base + src])
        one_img = _read(base + dst)
        _tool(dec, [base + dst])
        one_back = _read(base + src)
        _write(base + src, text)
        p = _tool(enc, [base + src], "-v", arena_cap=cap)
        assert _read(base + dst) == one_img
        q = _tool(dec, [base + dst], "-v", arena_cap=cap)
        assert _read(base + src) == one_back
        if kind == "quiva":
            wins = _windows(p.stderr)
            assert wins and wins[0][0] > 1 and wins[0][1] < len(text), p.stderr
        for r in (p, q):
            for w in _windows(r.stderr):
                assert w[1] < len(text) and w[0] > 1


# ---- 6. the 2-bit entry points ---------------------------------------------------------------------------

def _dev(data, extra=64):
    import torch
    t = torch.zeros(len(data) + extra, dtype=torch.uint8, device="cuda")
    if data:
        t[: len(data)] = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    return t


@pytest.mark.parametrize("kind", [0, 1])
def test_parts_at_every_entry_boundary_make_the_whole_file(ctx, kind):
    import torch
    from oracle import orc
    text = (synth.make_fasta if kind == 0 else synth.make_arrow)(53, [1, 300, 17, 80, 81, 5000, 2], max_well_delta=700)
    whole = orc.dexta(text, arrow=(kind == 1))
    starts = [m.start() + 1 for m in re.finditer(rb"\n>", text)]
    out = torch.zeros(len(text) + 4096, dtype=torch.uint8, device="cuda")
    for s in starts:                                             # two parts, cut at entry s
        got, well = b"", 0
        for i, (a, b) in enumerate(((0, s), (s, len(text)))):
            d = _dev(text[a:b])
            m, well = ctx.dexta_part_dev(kind, d.data_ptr(), b - a, well, i == 0, out.data_ptr(), out.numel())
            got += out[:m].cpu().numpy().tobytes()
        assert got == whole, s
    got, well, cuts = b"", 0, [0] + starts + [len(text)]         # every entry a part of its own
    for i in range(len(cuts) - 1):
        d = _dev(text[cuts[i]:cuts[i + 1]])
        m, well = ctx.dexta_part_dev(kind, d.data_ptr(), cuts[i + 1] - cuts[i], well, i == 0, out.data_ptr(), out.numel())
        assert ctx.last_entries() == 1
        got += out[:m].cpu().numpy().tobytes()
    assert got == whole

    # and back: two windows, the first ending at every entry boundary of the image and one byte to either side
    want = orc.undexta(whole, arrow=(kind == 1), width=61)
    plen = int.from_bytes(whole[2:6], "little")
    head = whole[: 6 + plen]
    fieldbytes = 12 if kind == 0 else 16
    ends, at = [], 6 + plen
    while at < len(whole):                                       # the chain, as undexta.c walks it
        while whole[at] == 0xff:
            at += 1
        at += 1
        beg, end = (int.from_bytes(whole[at + k:at + k + 4], "little") for k in (0, 4))
        at += fieldbytes + (end - beg + 3) // 4
        ends.append(at)
    assert ends[-1] == len(whole)

    def window(lo, hi, cur, well):
        d = _dev(whole[lo:hi])
        m, cur2, well2 = ctx.undexta_window_dev(kind, head, d.data_ptr(), hi - lo, lo, cur, well, hi == len(whole),
                                                61, False, out.data_ptr(), out.numel())
        return out[:m].cpu().numpy().tobytes(), cur2, well2

    for e in ends[:-1]:
        for cut in (e - 1, e, e + 1):
            try:
                got, cur, well = window(0, cut, 6 + plen, 0)
            except Exception as x:                               # DX_E_CAP: no whole entry in front of the cut
                assert x.code == -2 and cut < ends[0] and ctx.needed_bytes() > cut
                got, cur, well = b"", 6 + plen, 0
            assert cur == max(k for k in [6 + plen] + ends if k <= cut), (e, cut)
            rest, cur, _ = window(cur - cur % 16, len(whole), cur, well)
            assert cur == len(whole) and got + rest == want, (e, cut)


def test_window_calls_refuse_and_ask(ctx):
    from oracle import orc
    d = _dev(b">")                                                # an empty part is refused, not read
    out = _dev(b"", 4096)
    for with_header in (0, 1):
        with pytest.raises(Exception) as e:
            ctx.dexta_part_dev(0, d.data_ptr(), 0, 7, with_header, out.data_ptr(), 4096)
        assert e.value.code == -1
    text = synth.make_fasta(54, [40000, 10])
    img = orc.dexta(text)
    plen = int.from_bytes(img[2:6], "little")
    head = img[: 6 + plen]
    d = _dev(img[:5000])
    with pytest.raises(Exception) as e:                           # no entry lies wholly in the buffer
        ctx.undexta_window_dev(0, head, d.data_ptr(), 5000, 0, 6 + plen, 0, False, 80, False, 0, 0)
    assert e.value.code == -2 and ctx.needed_bytes() == 6 + plen + 1 + 12 + 10000
    with pytest.raises(Exception) as e:                           # ... and the file ends there
        ctx.undexta_window_dev(0, head, d.data_ptr(), 5000, 0, 6 + plen, 0, True, 80, False, 0, 0)
    assert e.value.code == -3
    d = _dev(img)                                                 # the size of the text, asked for
    with pytest.raises(Exception) as e:
        ctx.undexta_window_dev(0, head, d.data_ptr(), len(img), 0, 6 + plen, 0, True, 80, False, 0, 0)
    assert e.value.code == -2 and ctx.needed_bytes() == len(orc.undexta(img))
    for key in (b"\xcc\x33", b"\x33\xcc", b"\x55\xaa"):            # the old layout, the other byte order
        with pytest.raises(Exception) as e:
            ctx.undexta_window_dev(0, key + head[2:], d.data_ptr(), len(img), 0, 6 + plen, 0, True, 80, False, 0, 0)
        assert e.value.code == -1, key
    with pytest.raises(Exception) as e:
        ctx.undexta_window_dev(0, b"\x12\x34" + head[2:], d.data_ptr(), len(img), 0, 6 + plen, 0, True, 80, False, 0, 0)
    assert e.value.code == -4


def test_the_origin_numbers_errors_as_the_whole_file_does(ctx):
    import torch
    bad = b"@m/1/0_4 RQ=0.8\nabcd\nacgt\nabcd\nabc\nabcd\n"
    d = _dev(bad)
    ctx.set_origin(600, 100)
    with pytest.raises(Exception) as e:
        ctx.qv_scan_dev(d.data_ptr(), len(bad))
    ctx.set_origin(0, 0)
    assert e.value.line == 605 and "Line 605:" in e.value.text
    with pytest.raises(Exception) as e:
        ctx.qv_scan_dev(d.data_ptr(), len(bad))
    assert e.value.line == 5
    torch.cuda.synchronize()
