"""Function-level pin of the oracle: the per-read DB.h routines of oracle/dx_oracle.c beside the
reference's own functions (DB.c compiled into oracle/_ref/libdbqv_ref.so), on whole buffers --
including the bytes the reference touches past `len` (SURVEY Appendix B.13: Compress_Read leaves
s[len] = 0, Uncompress_Read writes up to 3 bytes past len and s[len] = 4).  Where oracle/_ref is not
built, against the digests of the reference's results in tests/golden/reference_digests.json; each
reference call is given the oracle's result of the step before, which was found equal to its own.
CPU only."""
import ctypes
import os

import numpy as np
import pytest

from tests.refgold import check

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LENGTHS = [0, 1, 2, 3, 4, 5, 7, 8, 9, 15, 16, 17, 63, 64, 65, 255, 256, 257, 1000, 4099, 65537]


@pytest.fixture(scope="module")
def both(orc):
    """(the reference's functions or None where oracle/_ref is not built, the oracle's)"""
    path = os.path.join(ROOT, "oracle", "_ref", "libdbqv_ref.so")
    return (ctypes.CDLL(path) if orc.have_ref() and os.path.exists(path) else None), orc.lib()


def _call(fn, buf, *pre):
    b = ctypes.create_string_buffer(bytes(buf), len(buf))
    fn(*pre, b)
    return b.raw


@pytest.mark.parametrize("L", LENGTHS)
def test_number_compress_uncompress_letter(both, L):
    R, O = both
    rng = np.random.default_rng(L)
    pad = 8
    for alphabet, number, o_number, letters in (
            (b"acgtACGTnNxy-", "Number_Read", "orc_number_read",
             (("Lower_Read", "orc_lower_read"), ("Upper_Read", "orc_upper_read"))),
            (b"1234G0x5", "Number_Arrow", "orc_number_arrow", (("Letter_Arrow", "orc_letter_arrow"),))):
        alpha = np.frombuffer(alphabet, dtype=np.uint8)
        text = alpha[rng.integers(0, len(alpha), size=L)].tobytes() + b"\0" + bytes([0x5a] * pad)
        b = _call(getattr(O, o_number), text)
        check(f"{number} L={L}", b, lambda: _call(getattr(R, number), text), R is not None)   # numeric codes + the 4 terminator
        cb = _call(O.orc_compress_read, b, ctypes.c_int(L))
        check(f"Compress_Read {number} L={L}", cb,                          # packed bytes AND what is left behind
              lambda: _call(R.Compress_Read, b, ctypes.c_int(L)), R is not None)
        ub = _call(O.orc_uncompress_read, cb, ctypes.c_int(L))
        check(f"Uncompress_Read {number} L={L}", ub,                        # including the spill past len
              lambda: _call(R.Uncompress_Read, cb, ctypes.c_int(L)), R is not None)
        for rname, oname in letters:
            check(f"{rname} L={L}", _call(getattr(O, oname), ub), lambda: _call(getattr(R, rname), ub), R is not None)
