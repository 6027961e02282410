"""tools/bin/undexqv_mg: one .dexqv file decoded by N ranks (byte ranges through dx_undexqv_range_*);
ranks share a GPU when fewer are visible, so -g3 and -g5 run on one device.  Its output must be byte
for byte what tools/bin/undexqv (and the reference's undexqv, when built) writes."""
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from dextractor_b200 import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "tools", "bin")
GOLDEN = os.path.join(ROOT, "tests", "golden")


@pytest.fixture()
def tmp():
    d = tempfile.mkdtemp(prefix="dxmg_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    yield d
    shutil.rmtree(d, ignore_errors=True)


def _run(tool, *args, cwd=None):
    return subprocess.run([os.path.join(BIN, tool), *args], capture_output=True, cwd=cwd)


def _read(p):
    with open(p, "rb") as f:
        return f.read()


def _decode_both(tmp, enc, name, *flags, g=(1, 3, 5)):
    """-> the text of undexqv; every -g of undexqv_mg must write the same bytes"""
    base = os.path.join(tmp, name)
    with open(base + ".dexqv", "wb") as f:
        f.write(enc)
    p = _run("undexqv", "-k", *flags, base)
    assert p.returncode == 0, p.stderr.decode()
    want = _read(base + ".quiva")
    os.unlink(base + ".quiva")
    for k in g:
        p = _run("undexqv_mg", "-k", "-v", f"-g{k}", *flags, base + ".dexqv")
        assert p.returncode == 0, p.stderr.decode()
        got = _read(base + ".quiva")
        assert got == want, (k, len(got), len(want))
        os.unlink(base + ".quiva")
    return want


@pytest.mark.parametrize("name", sorted(f for f in os.listdir(GOLDEN) if f.startswith("quiva_") and f.endswith(".dexqv")))
def test_golden_files(orc, tmp, name):
    enc = _read(os.path.join(GOLDEN, name))
    want = _decode_both(tmp, enc, "g")
    assert want == orc.undexqv(enc)
    if orc.have_ref():
        assert orc.ref_tool("undexqv", enc)[0] == want


def _big_file(orc, target):
    rng = np.random.default_rng(77)
    lengths = [int(x) for x in synth.lengths_for_bytes(rng, target, 5.0)]
    text = synth.make_quiva(77, lengths, max_well_delta=400)
    return text


@pytest.fixture(scope="module")
def big(orc):
    """a 256 MB .quiva (-> ~75 MB .dexqv): every rank of -g5 holds more than 1 MB, entries cross the cuts"""
    import dextractor_b200 as dx
    text = _big_file(orc, 256 << 20)
    ctx = dx.Context(0)
    try:
        enc = ctx.dexqv(text)
    finally:
        ctx.close()
    return text, enc


def test_a_large_file_on_1_3_and_5_ranks(orc, tmp, big):
    text, enc = big
    assert len(text) >= 256 << 20
    want = _decode_both(tmp, enc, "big", g=(1, 2, 3, 5, 8))
    assert want == text
    base = os.path.join(tmp, "big")
    p = _run("undexqv_mg", "-g5", "-v", "-U", base)                    # -U, and without -k the source goes
    assert p.returncode == 0, p.stderr.decode()
    assert b"rank 4" in p.stderr and b"rank 0 decodes the file alone" not in p.stderr
    assert not os.path.exists(base + ".dexqv")
    up = _read(base + ".quiva")
    with open(base + ".dexqv", "wb") as f:
        f.write(enc)
    assert _run("undexqv", "-k", "-U", base).returncode == 0
    assert _read(base + ".quiva") == up


def test_a_dexqv_mg_file(orc, tmp, big):
    if not os.path.exists(os.path.join(BIN, "dexqv_mg")):
        pytest.skip("dexqv_mg not built (no NCCL)")
    text, _ = big
    base = os.path.join(tmp, "m")
    with open(base + ".quiva", "wb") as f:
        f.write(text)
    p = _run("dexqv_mg", "-g1", base + ".quiva")
    assert p.returncode == 0, p.stderr.decode()
    enc = _read(base + ".dexqv")
    os.unlink(base + ".dexqv")
    assert _decode_both(tmp, enc, "m2", g=(3, 4)) == text


def test_several_files_in_one_call(orc, tmp, big):
    _, enc = big
    small = _read(os.path.join(GOLDEN, "quiva_lognormal_40.dexqv"))
    names = []
    for k, data in enumerate([small, enc, small]):
        names.append(os.path.join(tmp, f"f{k}"))
        with open(names[-1] + ".dexqv", "wb") as f:
            f.write(data)
    p = _run("undexqv_mg", "-g3", *names)
    assert p.returncode == 0, p.stderr.decode()
    for nm in names:
        assert not os.path.exists(nm + ".dexqv")
    assert _read(names[0] + ".quiva") == _read(names[2] + ".quiva") == orc.undexqv(small)
    assert _read(names[1] + ".quiva") == big[0]


def test_usage_and_missing_files_like_undexqv(tmp):
    for args in ([], ["-g3"], ["-g0", "x"], ["-g17", "x"]):
        p = _run("undexqv_mg", *args)
        assert p.returncode == 1 and p.stderr.startswith(b"Usage: undexqv_mg [-vkU] -g<gpus(1..16)> <path:dexqv> ...")
    q = _run("undexqv")
    assert q.returncode == 1 and q.stderr.startswith(b"Usage: undexqv [-vkU] <path:dexqv> ...")
    for line in (b"      -k: do *not* remove the .dexqv file on completion.",
                 b"      -U: use uppercase letters (default is lower case)."):
        assert line in p.stderr and line in q.stderr
    for args in (["nothere"], ["sub/nothere.dexqv"], ["-x"]):
        p = _run("undexqv_mg", "-g2", *args, cwd=tmp)
        q = _run("undexqv", *args, cwd=tmp)
        assert p.returncode == q.returncode == 1
        assert p.stderr.replace(b"undexqv_mg:", b"undexqv:") == q.stderr, (p.stderr, q.stderr)
        assert not os.listdir(tmp)


@pytest.mark.parametrize("name", ["legacy_foreign.dexqv", "legacy_old.dexqv", "legacy_foreign_old.dexqv"])
def test_legacy_files_take_the_rank0_path(orc, tmp, name):
    enc = _read(os.path.join(GOLDEN, name))
    base = os.path.join(tmp, "L")
    with open(base + ".dexqv", "wb") as f:
        f.write(enc)
    p = _run("undexqv_mg", "-g3", "-v", "-k", base)
    assert p.returncode == 0 and b"rank 0 decodes the file alone" in p.stderr, p.stderr.decode()
    got = _read(base + ".quiva")
    assert _run("undexqv", "-k", base).returncode == 0
    assert got == _read(base + ".quiva") == orc.undexqv(enc)


def test_every_visible_gpu(orc, tmp, big):
    ng = torch.cuda.device_count()
    if ng < 2:
        pytest.skip("one GPU visible")
    text, enc = big
    assert _decode_both(tmp, enc, "all", g=(ng,)) == text
