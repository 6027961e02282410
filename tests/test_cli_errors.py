"""The C command-line tools (tools/bin) against the reference tools (oracle/_ref, or what they printed,
stored in tests/golden/reference_digests.json) on everything that
happens before the first byte is coded: usage text, illegal options, non-integer -w, missing
inputs under every path form PathTo/Root/Catenate distinguish (DB.c:112-181).  Same stderr, same
exit status.  CPU only -- none of these cases reaches the GPU.  (-w0 is the documented deviation:
the reference loops forever there, undexta.c:265.)"""
import json
import os
import subprocess

import pytest

from oracle import orc
from tests.refgold import check

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOOLS = ["dexqv", "undexqv", "dexta", "undexta", "dexar", "undexar"]
ARGS = [[], ["-x", "foo"], ["-vx", "foo"], ["nonexistent"], ["sub/dir/none"], ["/none"],
        ["-wabc", "foo"], ["-w", "foo"], ["-v", "nonexistent.QUIVA"], ["none.fasta", "none.dexta"],
        ["-i", "extra"]]


def _run(path, args, cwd):
    r = subprocess.run([path] + args, cwd=cwd, stdin=subprocess.DEVNULL, capture_output=True)
    return r.returncode, r.stdout, r.stderr


def _text(r):
    return json.dumps([r[0], r[1].decode("latin-1"), r[2].decode("latin-1")])


@pytest.mark.parametrize("tool", TOOLS)
def test_tool_errors_match_the_reference(tool, tmp_path):
    """against oracle/_ref, or the stored (exit status, stdout, stderr) of the reference tools"""
    ours = os.path.join(ROOT, "tools", "bin", tool)
    theirs = os.path.join(ROOT, "oracle", "_ref", tool)
    if not os.path.exists(ours):
        pytest.fail("tools/bin is not built (python -c 'import __graft_entry__ as g; g.build()')")
    for args in ARGS:
        got = _run(ours, args, tmp_path)
        check(f"cli {tool} {json.dumps(args)}", _text(got), lambda: _text(_run(theirs, args, tmp_path)),
              orc.have_ref())
        assert got[0] == 1
    assert not os.listdir(tmp_path)          # nothing was created on the way


def test_tool_without_a_gpu_fails_loudly_and_leaves_the_files_alone(tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    src = tmp_path / "t.quiva"
    src.write_bytes(b"@m/1/0_4 RQ=0.850\nabcd\nnnnn\nijkl\nmnop\nqrst\n")
    rc, out, err = _run(os.path.join(ROOT, "tools", "bin", "dexqv"), ["t"], tmp_path)
    assert rc == 1 and b"no CPU fallback" in err
    assert sorted(os.listdir(tmp_path)) == ["t.quiva"]       # no empty .dexqv, source not removed
