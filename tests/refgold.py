"""What the reference DEXTRACTOR tools and functions give on the suite's inputs, stored in
tests/golden/reference_digests.json so that the comparisons with the reference also run where its
sources are absent (oracle/_ref is built only where they are present).

check(key, got, live, built): where the reference's side is built (`built`), `live()` computes
the reference's value and `got` must equal it; elsewhere `got` must equal the stored value.  Values
are bytes (stored as sha256) or strings (stored as they are).  With DX_RECORD_REFERENCE=<path> set,
every value checked is also recorded and the table is written to <path> at exit; only with
DX_RECORD_FROM_THIS_REPOSITORY=1 as well is a value recorded where the reference is not built,
and the value recorded is then this repository's own (tests/golden/make_reference_digests.py)."""
import atexit
import hashlib
import json
import os

from oracle import orc

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_digests.json")
TABLE = json.load(open(PATH)) if os.path.exists(PATH) else {}
RECORD = os.environ.get("DX_RECORD_REFERENCE")
FROM_THIS_REPOSITORY = os.environ.get("DX_RECORD_FROM_THIS_REPOSITORY") == "1"
_recorded = {}


def sha(b: bytes) -> str:
    return hashlib.sha256(b).hexdigest()


def _norm(v):
    return sha(v) if isinstance(v, (bytes, bytearray)) else v


def check(key: str, got, live, built: bool):
    got = _norm(got)
    if built:
        want = _norm(live())
    elif RECORD and FROM_THIS_REPOSITORY:
        want = got                   # tests/golden/make_reference_digests.py --from-oracle
    else:
        assert key in TABLE, f"no stored reference value for {key!r}"
        want = TABLE[key]
    if RECORD:
        _recorded[key] = want
    assert got == want, key


def check_tool(tool: str, data: bytes, got: bytes, *flags: str):
    """got must be what the reference `tool` writes for the input `data` with `flags`."""
    check(f"{tool} {' '.join(flags)} {sha(data)}", got, lambda: orc.ref_tool(tool, data, *flags)[0],
          orc.have_ref())


@atexit.register
def _write():
    if RECORD and _recorded:
        old = json.load(open(RECORD)) if os.path.exists(RECORD) else {}
        old.update(_recorded)
        with open(RECORD, "w") as f:
            json.dump(old, f, indent=0, sort_keys=True)
