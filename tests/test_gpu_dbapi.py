"""The in-memory QV.h calls the way the Dazzler DB code uses them (SURVEY 8f rows 1-2), through
libdexcompat.so on the GPU, call by call against the reference's own functions compiled into
oracle/_ref/libdbqv_ref.so or, where they are not built, against their stored results
(tests/golden/reference_digests.json); the .qvs files the other tests read are then written by
libdexcompat.so, whose writer the first test finds byte-equal to the reference's:

  * dex2DB's write path (dex2DB.c:506-567, 604-622): QVcoding_Scan1(0,...) reset, QVcoding_Scan1 per
    read, Create_QVcoding, prefix ".qvs", Write_QVcoding, Compress_Next_QVentry1 per read with
    ftello() after each one (DAZZ_READ.coff);
  * Load_QVentry's read path (DB.c:2598-2599): Read_QVcoding, then fseeko(coff) +
    Uncompress_Next_QVentry in any order; several codings in one .qvs, each a struct copy of
    Read_QVcoding's static result (DB.c:2450-2507);
  * the batch form of the same (dx_qv_load_entries_dev): every entry of a .qvs in one call.
"""
import ctypes as C
import json
import os

import numpy as np
import pytest

from dextractor_b200 import synth
from tests import refgold
from tests.refgold import check

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class QVcoding(C.Structure):                       # QV.h:31-42
    _fields_ = [("delScheme", C.c_void_p), ("insScheme", C.c_void_p), ("mrgScheme", C.c_void_p),
                ("subScheme", C.c_void_p), ("dRunScheme", C.c_void_p), ("sRunScheme", C.c_void_p),
                ("delChar", C.c_int), ("subChar", C.c_int), ("flip", C.c_int), ("prefix", C.c_void_p)]


libc = C.CDLL(None)
libc.fopen.restype = C.c_void_p
libc.fopen.argtypes = [C.c_char_p, C.c_char_p]
libc.fclose.argtypes = [C.c_void_p]
libc.ftello.restype = C.c_int64
libc.ftello.argtypes = [C.c_void_p]
libc.fseeko.argtypes = [C.c_void_p, C.c_int64, C.c_int]
libc.fflush.argtypes = [C.c_void_p]


def _lib(path):
    L = C.CDLL(path)
    cp = C.c_char_p
    L.QVcoding_Scan1.argtypes = [C.c_int, cp, cp, cp, cp, cp]
    L.QVcoding_Scan1.restype = None
    L.Create_QVcoding.argtypes = [C.c_int]
    L.Create_QVcoding.restype = C.POINTER(QVcoding)
    L.Write_QVcoding.argtypes = [C.c_void_p, C.POINTER(QVcoding)]
    L.Write_QVcoding.restype = None
    L.Read_QVcoding.argtypes = [C.c_void_p]
    L.Read_QVcoding.restype = C.POINTER(QVcoding)
    L.Compress_Next_QVentry1.argtypes = [C.c_int, cp, cp, cp, cp, cp, C.c_void_p, C.POINTER(QVcoding), C.c_int]
    L.Compress_Next_QVentry1.restype = None
    L.Uncompress_Next_QVentry.argtypes = [C.c_void_p, C.POINTER(C.c_char_p), C.POINTER(QVcoding), C.c_int]
    L.Uncompress_Next_QVentry.restype = C.c_int
    L.Strdup.argtypes = [cp, cp]
    L.Strdup.restype = C.c_void_p
    C.c_char_p.in_dll(L, "Prog_Name").value = b"dbapi_test"
    return L


@pytest.fixture(scope="module")
def libs(orc):
    """(libdexcompat.so, the reference's libdbqv_ref.so or None where it is not built)"""
    ref = os.path.join(ROOT, "oracle", "_ref", "libdbqv_ref.so")
    have = orc.have_ref() and os.path.exists(ref)
    return _lib(os.path.join(ROOT, "dextractor_b200", "libdexcompat.so")), (_lib(ref) if have else None)


def _reads(seed, lengths):
    """the five streams of every entry of a synthetic .quiva, as dex2DB holds them in memory"""
    text = synth.make_quiva(seed, lengths)
    lines = text.split(b"\n")
    return [tuple(lines[6 * e + k] for k in range(1, 6)) for e in range(len(lengths))]


def _write_block(L, f, reads, lossy=0):
    """one coding + its entries, dex2DB order; -> coff of every read"""
    def mutable(r):
        # the reference packs the tags (and, lossy, edits the QVs) IN PLACE (QV.c:1343-1379): hand it
        # copies -- a Python bytes object is immutable, and a one-character line is the interpreter's
        # shared object for that character
        return [C.create_string_buffer(x, len(x) + 8) for x in r]

    L.QVcoding_Scan1(0, None, None, None, None, None)
    for r in reads:
        L.QVcoding_Scan1(len(r[0]), *mutable(r))
    cd = L.Create_QVcoding(lossy)
    assert cd
    cd.contents.prefix = L.Strdup(b".qvs", b"Allocating header prefix")
    L.Write_QVcoding(f, cd)
    coff = []
    for r in reads:
        coff.append(libc.ftello(f))
        L.Compress_Next_QVentry1(len(r[0]), *mutable(r), f, cd, lossy)
    return coff


def _read_entry(L, f, coding, rlen):
    bufs = [C.create_string_buffer(rlen + 8) for _ in range(5)]
    arr = (C.c_char_p * 5)(*[C.cast(b, C.c_char_p) for b in bufs])
    rc = L.Uncompress_Next_QVentry(f, arr, coding, rlen)
    return rc, [b.raw[:rlen] for b in bufs], libc.ftello(f)


def test_dex2db_write_order_and_load_qventry(libs, tmp_path):
    """against the reference's own calls, or where they are not built, against what they gave
    (tests/golden/reference_digests.json): the .qvs bytes, every coff, every entry read back"""
    gpu, ref = libs
    rng = np.random.default_rng(9)
    lengths = [int(x) for x in rng.integers(1, 9000, size=70)] + [1, 2, 3, 4, 31, 32, 33]
    reads = _reads(9, lengths)

    def write(name, L):
        path = tmp_path / f"{name}.qvs"
        f = libc.fopen(str(path).encode(), b"w")
        coff = _write_block(L, f, reads)
        end = libc.ftello(f)
        libc.fclose(f)
        return path, coff, end

    mine = write("gpu", gpu)
    theirs = write("ref", ref) if ref is not None else None
    check("dex2DB coff", json.dumps([mine[1], mine[2]]), lambda: json.dumps([theirs[1], theirs[2]]),
          ref is not None)                               # ftello after Compress_Next_QVentry1 (DAZZ_READ.coff)
    check("dex2DB .qvs", mine[0].read_bytes(), lambda: theirs[0].read_bytes(), ref is not None)

    # Load_QVentry: Read_QVcoding once, then fseeko(coff) + Uncompress_Next_QVentry in any order, on
    # the reference's file (or, without it, ours: the check above found the two equal)
    path, coff = (theirs or mine)[:2]
    order = list(rng.permutation(len(reads)))

    def load(L):
        f = libc.fopen(str(path).encode(), b"r")
        cd = L.Read_QVcoding(f)
        assert cd
        res = []
        for i in order:
            libc.fseeko(f, coff[i], 0)
            rc, lines, pos = _read_entry(L, f, cd, len(reads[i][0]))
            res.append(json.dumps([rc, refgold.sha(b"\n".join(lines)), pos]))
        libc.fclose(f)
        return res

    got = load(gpu)
    want = load(ref) if ref is not None else None
    for k, i in enumerate(order):
        check(f"Load_QVentry {i}", got[k], lambda: want[k], ref is not None)
        assert json.loads(got[k])[0] == 0


def test_two_codings_in_one_qvs(libs, tmp_path):
    """DB.c:2450-2507: one coding per source file, all in one .qvs; the codings are struct copies of
    Read_QVcoding's static result and an entry is decoded with the coding of its block."""
    gpu, ref = libs
    blocks = [_reads(21, [int(x) for x in np.random.default_rng(21).integers(200, 7000, size=50)]),
              _reads(22, [9000] * 30)]
    path = tmp_path / "two.qvs"
    f = libc.fopen(str(path).encode(), b"w")
    heads, coffs = [], []
    for b in blocks:
        heads.append(libc.ftello(f))
        coffs.append(_write_block(ref or gpu, f, b))       # the reference writes it where it is built
    libc.fclose(f)
    for name, L in (("gpu", gpu), ("ref", ref)):
        if L is None:
            continue
        f = libc.fopen(str(path).encode(), b"r")
        codings = []
        for h in heads:
            libc.fseeko(f, h, 0)
            cd = L.Read_QVcoding(f)
            assert cd
            copy = QVcoding()
            C.pointer(copy)[0] = cd.contents                     # struct copy, DB.c:2455
            codings.append(copy)
        for k in range(40):
            b = k % 2
            i = (7 * k) % len(blocks[b])
            libc.fseeko(f, coffs[b][i], 0)
            rc, lines, pos = _read_entry(L, f, C.pointer(codings[b]), len(blocks[b][i][0]))
            assert rc == 0, (name, b, i)
            want = list(blocks[b][i])
            assert lines[0] == want[0] and lines[2:] == want[2:], (name, b, i)
            nxt = coffs[b][i + 1] if i + 1 < len(coffs[b]) else None
            if nxt is not None:
                assert pos == nxt, (name, b, i)
        libc.fclose(f)


def test_batched_load_of_a_qvs(libs, tmp_path):
    """dx_qv_load_entries_dev: every entry of a .qvs in ONE call (the batch form of Load_QVentry)."""
    import torch
    import dextractor_b200 as dx
    from dextractor_b200 import lib as dxl
    gpu, ref = libs
    rng = np.random.default_rng(33)
    lengths = [int(x) for x in rng.integers(1, 12000, size=300)]
    reads = _reads(33, lengths)
    path = tmp_path / "b.qvs"
    f = libc.fopen(str(path).encode(), b"w")
    coff = _write_block(ref or gpu, f, reads)         # the reference writes it where it is built
    libc.fclose(f)
    data = path.read_bytes()
    cd, prefix, used = dxl.read_coding(data)
    assert prefix == b".qvs" and used == coff[0]
    ctx = dx.Context(0)
    try:
        img = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
        out = torch.zeros(5 * (sum(lengths) + len(lengths)) + 64, dtype=torch.uint8, device="cuda")
        for route in ({}, {"decoder": 6}):
            ctx.route("default")
            for k, v in route.items():
                ctx.route(k, v)
            out.zero_()
            torch.cuda.synchronize()    # torch fills on its own stream, the library runs on another
            oo, eo = ctx.qv_load_entries_dev(img.data_ptr(), len(data), cd, coff, lengths, False,
                                             out.data_ptr(), out.numel())
            text = out[: oo[-1]].cpu().numpy().tobytes()
            for i, r in enumerate(reads):
                got = text[oo[i]: oo[i + 1]].split(b"\n")[:5]
                assert got[0] == r[0] and got[2:] == list(r[2:]), (route, i)
                assert eo[i] == (coff[i + 1] if i + 1 < len(coff) else len(data)), (route, i)
        ctx.route("default")
    finally:
        ctx.close()
