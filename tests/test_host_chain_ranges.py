"""The entry chain of a .dexqv image walked byte range after byte range (csrc/dx_chain.h,
dx_chain_walk_general), as dx_undexqv_range_* and the pipelined host decode walk it: random images,
random cuts (inside 0xff delta runs, fields and payloads, runs of more than 4 KB across a cut, ranges
without an entry start), missed and cut-short candidates, buffers whose tail is too short.  Driven by
tests/hostfuzz/fz_chain_ranges.cpp under AddressSanitizer + UndefinedBehaviorSanitizer; the ranges
together must give exactly the whole walk's entries and wells.  CPU only."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SAN = ["-g", "-O1", "-fsanitize=address,undefined", "-fno-omit-frame-pointer"]


@pytest.mark.timeout(900)
def test_ranges_walk_the_whole_chain(tmp_path):
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    exe = tmp_path / "fz_chain_ranges"
    r = subprocess.run(["g++", "-std=c++17", *SAN, "-I" + os.path.join(ROOT, "dextractor_b200", "csrc"),
                        "-o", str(exe), os.path.join(ROOT, "tests", "hostfuzz", "fz_chain_ranges.cpp")],
                       capture_output=True, text=True)
    if r.returncode != 0:
        pytest.skip("sanitizer build not possible here: " + r.stderr[-300:])
    env = dict(os.environ, ASAN_OPTIONS="detect_leaks=0:abort_on_error=0", UBSAN_OPTIONS="halt_on_error=1")
    p = subprocess.run([str(exe), "20000"], capture_output=True, text=True, env=env, timeout=800)
    assert p.returncode == 0 and "ERROR" not in p.stderr and "runtime error" not in p.stderr, p.stderr[-3000:]
    out = p.stdout
    assert out.startswith("ok 20000 images"), out
    ranges, empty, slow, longer, runs, straddle = [int(x) for x in re.findall(r"(\d+) [a-z]", out)][1:7]
    # every branch was exercised
    assert ranges > 50000 and empty > 5000 and slow > 5000 and longer > 2000 and runs > 5000 and straddle > 1000, out
