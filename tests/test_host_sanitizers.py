"""The host side of the coder (dx_coding.cpp: code construction, coding header writer and reader)
compiled with AddressSanitizer + UndefinedBehaviorSanitizer and driven by two small C harnesses
(tests/hostfuzz/): every truncation and 20 000 random corruptions of real headers on exactly-sized
heap buffers, and 3 000 random statistics (ties, 2^62 counts, single-symbol streams) through
make -> write -> read.  Any report from a sanitizer fails the test.  CPU only.

Also here: the entry-chain decision of csrc/dx_chain.h (which candidates of a .dexqv image are its
entries), whose two forms -- the host's walk and the per-candidate predicate the device evaluates after
an in-place decode -- are driven on 100 000 random images by tests/hostfuzz/fz_chain.cpp: the walk
against the truth, the two forms against each other, the assumed wells against the walk's, and the
walk cut into windows (as the pipelined host decode walks) against the whole walk."""
import os
import shutil
import subprocess

import pytest

from dextractor_b200 import lib as dxl
from tests import fuzz

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SAN = ["-g", "-O1", "-fsanitize=address,undefined", "-fno-omit-frame-pointer"]


@pytest.fixture(scope="module")
def built(tmp_path_factory):
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    d = tmp_path_factory.mktemp("asan")
    inc = ["-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "dextractor_b200", "csrc"),
           "-I/usr/local/cuda/include"]
    r = subprocess.run(["g++", "-std=c++17", *SAN, "-fPIC", "-shared", *inc, "-o", str(d / "libcoding_asan.so"),
                        os.path.join(ROOT, "dextractor_b200", "csrc", "dx_coding.cpp")],
                       capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("sanitizer build not possible here: " + r.stderr[-300:])
    for name in ("fz_read_coding", "fz_make_coding"):
        subprocess.check_call(["gcc", *SAN, inc[0], "-o", str(d / name),
                               os.path.join(ROOT, "tests", "hostfuzz", name + ".c"),
                               "-L" + str(d), "-lcoding_asan", "-Wl,-rpath," + str(d), "-lm"])
    return d


def _run(cmd):
    env = dict(os.environ, ASAN_OPTIONS="detect_leaks=0:abort_on_error=0", UBSAN_OPTIONS="halt_on_error=1")
    r = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0 and "ERROR" not in r.stderr and "runtime error" not in r.stderr, r.stderr[-3000:]
    return r.stdout


@pytest.mark.timeout(900)
def test_header_reader_under_sanitizers(orc, built, tmp_path):
    for seed in range(3):
        text, _ = fuzz.fuzz_quiva(seed)
        data = orc.dexqv(text, lossy=bool(seed & 1))
        _, _, used = dxl.read_coding(data[2:])
        h = tmp_path / f"h{seed}.bin"
        h.write_bytes(data[2:2 + used])
        out = _run([str(built / "fz_read_coding"), str(h)])
        assert out.startswith("ok ")


@pytest.mark.timeout(900)
def test_code_construction_under_sanitizers(built):
    out = _run([str(built / "fz_make_coding")])
    coded, refused, trips = (int(x) for x in out.split() if x.isdigit())
    assert coded + refused == 3000 and trips == coded


@pytest.mark.timeout(900)
def test_entry_chain_walk_and_device_predicate_agree(tmp_path):
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    exe = tmp_path / "fz_chain"
    r = subprocess.run(["g++", "-std=c++17", *SAN, "-I" + os.path.join(ROOT, "dextractor_b200", "csrc"),
                        "-o", str(exe), os.path.join(ROOT, "tests", "hostfuzz", "fz_chain.cpp")],
                       capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("sanitizer build not possible here: " + r.stderr[-300:])
    out = _run([str(exe), "100000"])
    assert out.startswith("ok 100000 images"), out
    walked, assumed, broken, windowed = [int(x) for x in out.replace(":", " ").split() if x.isdigit()][1:5]
    assert walked > 80000 and assumed > 30000 and broken > 1000, out      # every branch was exercised
    assert windowed > 60000, out                                          # ... the windowed walk too
