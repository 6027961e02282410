"""Codings with many codes of 12 to 16 bits, decoded by the parallel decoders on every path: the
whole-image decode (default route and each decoder forced), byte ranges, tools/bin/undexqv in
windows, undexqv_mg, the pipelined dx_undexqv_host, dx_qv_load_entries_dev and the compat shim's
Load_QVentry of a bare-stream .qvs.  The inputs are the fuzz files whose coding has more than 64
distinct 11-bit prefixes of such codes in one scheme, and files built by tests/long_codes.py whose
deletion run table has more than 200 of them; the first test checks that on the CPU, so that the
others cannot quietly decode easy codings.  Every output is compared with the oracle's."""
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from dextractor_b200 import lib as dxl
from tests import fuzz, long_codes
from tests.qv_shapes import coding as oracle_coding
from tests.test_gpu_parity import first_diff

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "tools", "bin")
FUZZ_SEEDS = (10, 12, 19, 21, 36)       # the fuzz files (lossy when odd) with more than 64 prefixes
LOSSY = (False, True)


def _fuzz_text(seed):
    return fuzz.fuzz_quiva(seed)[0]


def _small_text():
    return long_codes.make_quiva(41, np.random.default_rng(41).integers(2000, 9000, size=40))


def _big_text():
    """~20 MB of .quiva, more than 4 MB of .dexqv lossless and lossy: 1 MB per rank of undexqv_mg -g4"""
    return long_codes.make_quiva(42, np.random.default_rng(42).integers(4000, 16000, size=400))


def test_the_inputs_have_long_codings(orc):
    for seed in FUZZ_SEEDS:
        assert long_codes.max_prefixes(oracle_coding(orc, _fuzz_text(seed), bool(seed & 1))) > long_codes.PREFIXES, seed
    deep = oracle_coding(orc, _fuzz_text(10), False)          # codes of 13 to 15 bits, not only 12
    assert max(deep.tab[1].lens[i] for i in range(256)) >= 13
    for make in (_small_text, _big_text):
        text = make()
        for lossy in LOSSY:
            cd = oracle_coding(orc, text, lossy)
            assert cd.delchar == long_codes.DELC
            assert long_codes.long_run_codes(cd.tab[1]) >= 200, (make.__name__, lossy)
            assert long_codes.max_prefixes(cd) > long_codes.PREFIXES, (make.__name__, lossy)
    assert min(len(orc.dexqv(_big_text(), lossy=lossy)) for lossy in LOSSY) > 4 << 20


# ---- GPU ------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def ctx():
    import dextractor_b200 as dx
    c = dx.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def images(orc):
    """name -> (.dexqv image, the oracle's text)"""
    out = {}
    for seed in FUZZ_SEEDS:
        enc = orc.dexqv(_fuzz_text(seed), lossy=bool(seed & 1))
        out[f"fuzz{seed}"] = (enc, orc.undexqv(enc))
    for name, make in (("small", _small_text), ("big", _big_text)):
        text = make()
        for lossy in LOSSY:
            enc = orc.dexqv(text, lossy=lossy)
            want = orc.undexqv(enc)
            assert lossy or want == text
            out[f"{name}{'_l' if lossy else ''}"] = (enc, want)
    return out


NAMES = [f"fuzz{s}" for s in FUZZ_SEEDS] + ["small", "small_l", "big", "big_l"]


def _whole(ctx, enc, route=None):
    from tests.test_gpu_undexqv_ranges import whole
    ctx.route("default")
    if route is not None:
        ctx.route("decoder", route)
    try:
        return whole(ctx, enc)
    finally:
        ctx.route("default")


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_whole_image_on_every_decoder(ctx, images, name):
    enc, want = images[name]
    ctx.profile(True)
    ctx.profile_report()
    got = _whole(ctx, enc)
    kernels = ctx.profile_report()
    ctx.profile(False)
    assert got == want, first_diff(got, want)
    assert "k_qv_decode" not in kernels and "k_qv_walk" not in kernels, kernels    # not the sequential kernels
    assert _whole(ctx, enc, 1) == want
    for dec in (5, 6):
        got = _whole(ctx, enc, dec)
        assert got == want, (dec, first_diff(got, want))


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_byte_ranges(ctx, orc, images, name):
    """random cuts, and every cut within 3 bytes of three entry boundaries"""
    from tests.test_gpu_undexqv_ranges import _cuts, _dev, ranges
    enc, want = images[name]
    n = len(enc)
    rng = np.random.default_rng(n)
    img = _dev(enc)
    for k in (1, 5, 17):
        cuts = _cuts(rng, n, k)
        got = ranges(ctx, enc, cuts, img=img, tail=int(rng.integers(0, 5000)))
        assert got == want, (cuts, first_diff(got, want))
    offs = orc.dexqv_offsets(enc, 1 << 20)               # entry starts, then the image end
    for e in sorted({min(1, len(offs) - 2), len(offs) // 2, len(offs) - 2}):
        for c in range(int(offs[e]) - 3, int(offs[e]) + 4):
            got = ranges(ctx, enc, [c], img=img, tail=int(c % 97))
            assert got == want, (e, c, first_diff(got, want))


@pytest.fixture()
def tmp():
    d = tempfile.mkdtemp(prefix="dxlong_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    yield d
    shutil.rmtree(d, ignore_errors=True)


def _tool(tool, *args, window=None):
    env = dict(os.environ)
    env.pop("DEXB200_WINDOW", None)
    env.pop("DEXB200_ARENA_CAP", None)
    if window is not None:
        env["DEXB200_WINDOW"] = str(window)
    p = subprocess.run([os.path.join(BIN, tool), *args], capture_output=True, env=env)
    assert p.returncode == 0, p.stderr.decode()
    return p


def _read(path):
    with open(path, "rb") as f:
        return f.read()


@pytest.mark.gpu
@pytest.mark.parametrize("name,window", [("small_l", 64 << 10), ("big", 64 << 10), ("big", (1 << 20) + 7),
                                         ("big_l", (1 << 20) + 7)])
def test_undexqv_in_windows(images, tmp, name, window):
    from tests.test_gpu_stream import _windows
    enc, want = images[name]
    base = os.path.join(tmp, "w")
    with open(base + ".dexqv", "wb") as f:
        f.write(enc)
    p = _tool("undexqv", "-k", "-v", base, window=window)
    assert _read(base + ".quiva") == want
    wins = [w[0] for w in _windows(p.stderr)]
    assert wins and wins[0] > 1, p.stderr.decode()                # streamed, not decoded whole


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["big", "big_l"])
def test_undexqv_mg_on_1_to_4_ranks(images, tmp, name):
    enc, want = images[name]
    base = os.path.join(tmp, "m")
    with open(base + ".dexqv", "wb") as f:
        f.write(enc)
    for g in (1, 2, 3, 4):
        p = _tool("undexqv_mg", "-k", "-v", f"-g{g}", base)
        assert b"rank 0 decodes the file alone" not in p.stderr, p.stderr.decode()
        got = _read(base + ".quiva")
        assert got == want, (g, first_diff(got, want))
        os.unlink(base + ".quiva")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["big", "big_l"])
def test_pipelined_host_decode(ctx, images, name):
    """1 MB chunks: the pipeline's windows each lay out their text (one k_qv_assemble per window);
    a pipeline that declined would have decoded the image whole instead"""
    enc, want = images[name]
    ctx.route("default")
    ctx.route("pipe_chunk", 1 << 20)
    ctx.profile(True)
    ctx.profile_report()
    try:
        got = ctx.undexqv(enc)
        kernels = ctx.profile_report()
    finally:
        ctx.profile(False)
        ctx.route("default")
    assert got == want, first_diff(got, want)
    assert kernels.get("k_qv_assemble", (0, 0))[0] >= 2, kernels


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["fuzz10", "fuzz19", "small", "small_l"])
def test_load_entries(ctx, images, name):
    """dx_qv_load_entries_dev on every entry of the image, at the stream offsets the whole decode found"""
    from tests.test_gpu_undexqv_ranges import _dev
    enc, want = images[name]
    img = _dev(enc)
    cap = len(enc) * 40 + 200000
    out = torch.empty(cap, dtype=torch.uint8, device="cuda")
    ctx.keep_index(True)
    try:
        ctx.undexqv_dev(img.data_ptr(), len(enc), False, out.data_ptr(), cap)
        rows = ctx.last_index()
    finally:
        ctx.keep_index(False)
    assert rows
    cd, _, _ = dxl.read_coding(enc[2:])
    so = [r[0] for r in rows]
    rl = [r[3] for r in rows]
    for route in ({}, {"decoder": 5}, {"decoder": 6}):
        ctx.route("default")
        for k, v in route.items():
            ctx.route(k, v)
        out.zero_()
        torch.cuda.synchronize()
        oo, eo = ctx.qv_load_entries_dev(img.data_ptr(), len(enc), cd, so, rl, False, out.data_ptr(), cap)
        ctx.route("default")
        text = out[: oo[-1]].cpu().numpy().tobytes()
        lines = want.split(b"\n")
        for i, r in enumerate(rows):
            got = text[oo[i]: oo[i + 1]].split(b"\n")[:5]
            assert got == lines[6 * i + 1: 6 * i + 6], (route, i)
            assert eo[i] == r[1], (route, i)


@pytest.mark.gpu
def test_load_qventry_of_a_bare_stream_qvs(orc, tmp):
    """the compat shim: Create_QVcoding + Compress_Next_QVentry1 write a .qvs (coding, then the bare
    streams of every entry, as dex2DB does), Read_QVcoding + fseeko(coff) + Uncompress_Next_QVentry
    read the entries back in any order"""
    from tests.test_gpu_dbapi import _lib, _read_entry, _write_block, libc
    L = _lib(os.path.join(ROOT, "dextractor_b200", "libdexcompat.so"))
    text = _small_text()
    lines = text.split(b"\n")
    reads = [tuple(lines[6 * e + k] for k in range(1, 6)) for e in range(len(lines) // 6)]
    path = os.path.join(tmp, "long.qvs").encode()
    f = libc.fopen(path, b"w")
    coff = _write_block(L, f, reads)
    libc.fclose(f)
    cd, prefix, used = dxl.read_coding(_read(path))
    assert prefix == b".qvs" and used == coff[0]
    assert long_codes.max_prefixes(cd) > long_codes.PREFIXES
    f = libc.fopen(path, b"r")
    try:
        coding = L.Read_QVcoding(f)
        assert coding
        for i in np.random.default_rng(5).permutation(len(reads)):
            libc.fseeko(f, coff[i], 0)
            rc, got, pos = _read_entry(L, f, coding, len(reads[i][0]))
            assert rc == 0, i
            assert got == list(reads[i]), i
            assert pos == (coff[i + 1] if i + 1 < len(coff) else os.path.getsize(path)), i
    finally:
        libc.fclose(f)
