"""CPU-side checks of the reference-symbol layer (libdexcompat.so / libdexcompat_i.so, SURVEY 8b):
both libraries export every QV.h / DB.h symbol of the path, the line reader follows QV.c:751-798,
and errors follow the reference's two conventions (DB.h:28-47): batch = message on stderr + exit,
-DINTERACTIVE = message in Ebuffer + documented error value.  No codec work runs here: without a
GPU the codec calls must fail loudly in either convention."""
import ctypes
import json
import os
import subprocess
import sys
import textwrap

import pytest

from tests import refgold
from tests.refgold import check

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIBDIR = os.path.join(ROOT, "dextractor_b200")

QV_H = ["Read_Lines", "QVentry", "Set_QV_Line", "Get_QV_Line", "QVcoding_Scan", "QVcoding_Scan1",
        "Create_QVcoding", "Read_QVcoding", "Write_QVcoding", "Free_QVcoding",
        "Compress_Next_QVentry", "Compress_Next_QVentry1", "Uncompress_Next_QVentry"]      # QV.h:48-97
DB_H = ["Compress_Read", "Uncompress_Read", "Lower_Read", "Upper_Read", "Number_Read",
        "Change_Read", "Letter_Arrow", "Number_Arrow",                                       # DB.h:255-267
        "Malloc", "Realloc", "Strdup", "Fopen", "PathTo", "Root", "Catenate", "Numbered_Suffix",
        "Prog_Name"]                                                                         # DB.h:71,235-247


def _load(name):
    path = os.path.join(LIBDIR, name)
    if not os.path.exists(path):
        pytest.fail(f"{name} is not built (python -c 'import __graft_entry__ as g; g.build()')")
    return ctypes.CDLL(path)


@pytest.mark.parametrize("name", ["libdexcompat.so", "libdexcompat_i.so"])
def test_reference_symbols_exported(name):
    L = _load(name)
    missing = [s for s in QV_H + DB_H if not hasattr(L, s)]
    assert not missing, missing
    assert hasattr(L, "Ebuffer") == name.endswith("_i.so")


class _Shim:
    def __init__(self):
        self.L = _load("libdexcompat_i.so")
        self.libc = ctypes.CDLL(None)
        self.libc.fopen.restype = ctypes.c_void_p
        self.libc.fopen.argtypes = [ctypes.c_char_p, ctypes.c_char_p]
        self.libc.fclose.argtypes = [ctypes.c_void_p]
        self.L.Read_Lines.argtypes = [ctypes.c_void_p, ctypes.c_int]
        self.L.QVentry.restype = ctypes.c_char_p
        self.L.QVcoding_Scan.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
        self.L.Create_QVcoding.restype = ctypes.c_void_p
        self.ebuf = (ctypes.c_char * 1000).in_dll(self.L, "Ebuffer")

    def open(self, path):
        f = self.libc.fopen(str(path).encode(), b"r")
        assert f
        return f

    def message(self):
        return self.ebuf.value.decode()


@pytest.fixture(scope="module")
def shim():
    return _Shim()


def test_read_lines_follows_the_reference(shim, tmp_path):
    p = tmp_path / "a.quiva"
    p.write_bytes(b"@m/1/0_4 RQ=0.850\nabcd\nefgh\nijkl\nmnop\nqrst\n@m/2/0_3 RQ=0.8\nabc\nab\n")
    f = shim.open(p)
    shim.L.Set_QV_Line(0)
    assert shim.L.Read_Lines(f, 1) == len("@m/1/0_4 RQ=0.850")
    assert shim.L.QVentry().startswith(b"@m/1/0_4")
    assert shim.L.Read_Lines(f, 5) == 4
    assert shim.L.Get_QV_Line() == 6
    assert shim.L.Read_Lines(f, 1) == len("@m/2/0_3 RQ=0.8")
    assert shim.L.Read_Lines(f, 5) == -2                      # QV.c:792-795
    assert "Lines for an entry are not the same length" in shim.message()
    assert shim.message().startswith("Line 9:")
    shim.libc.fclose(f)

    p.write_bytes(b"abcd\nefgh")
    f = shim.open(p)
    assert shim.L.Read_Lines(f, 2) == -2                      # a LATER line without its newline is
    assert "not the same length" in shim.message()            # a length error (QV.c:792-795)
    assert shim.L.Read_Lines(f, 1) == -1                      # end of input before any line
    shim.libc.fclose(f)

    p.write_bytes(b"abcd")
    f = shim.open(p)
    assert shim.L.Read_Lines(f, 1) == -2                      # QV.c:778-781: the FIRST line cut short
    assert "Last line does not end with a newline" in shim.message()
    shim.libc.fclose(f)

    p.write_bytes(b"abcd\nefgh\n")
    f = shim.open(p)
    assert shim.L.Read_Lines(f, 5) == -2                      # QV.c:787-791
    assert "incomplete last entry" in shim.message()
    shim.libc.fclose(f)


def test_read_lines_grows_its_buffer(shim, tmp_path):
    L = 180_000                                               # beyond the first 50 000-byte slots
    p = tmp_path / "long.quiva"
    p.write_bytes(b"".join(bytes([65 + k]) * L + b"\n" for k in range(5)))
    f = shim.open(p)
    assert shim.L.Read_Lines(f, 5) == L
    assert shim.L.QVentry()[:3] == b"AAA"
    shim.libc.fclose(f)


def _no_gpu():
    import torch
    return not torch.cuda.is_available()


def test_interactive_codec_calls_fail_with_a_message_without_a_gpu(shim, tmp_path):
    if not _no_gpu():
        pytest.skip("a GPU is present")
    p = tmp_path / "b.quiva"
    p.write_bytes(b"@m/1/0_4 RQ=0.850\nabcd\nnnnn\nijkl\nmnop\nqrst\n")
    f = shim.open(p)
    assert shim.L.QVcoding_Scan(f, 2**31 - 1, None) == -1     # QV.h:56-58
    assert "no usable CUDA device" in shim.message()
    assert shim.L.Create_QVcoding(0) is None                  # QV.h:62-65
    shim.libc.fclose(f)


def test_batch_codec_calls_exit_without_a_gpu(tmp_path):
    if not _no_gpu():
        pytest.skip("a GPU is present")
    p = tmp_path / "c.quiva"
    p.write_bytes(b"@m/1/0_4 RQ=0.850\nabcd\nnnnn\nijkl\nmnop\nqrst\n")
    code = textwrap.dedent(f"""
        import ctypes
        L = ctypes.CDLL({os.path.join(LIBDIR, 'libdexcompat.so')!r})
        libc = ctypes.CDLL(None)
        libc.fopen.restype = ctypes.c_void_p
        L.QVcoding_Scan.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
        f = libc.fopen({str(p).encode()!r}, b"r")
        L.QVcoding_Scan(f, 2**31 - 1, None)
        print("survived")
    """)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True)
    assert r.returncode == 1 and "survived" not in r.stdout
    assert "no usable CUDA device" in r.stderr


def _ref_lib(orc, name):
    """the reference's own DB.c + QV.c as compiled into oracle/_ref, or None where it is not built"""
    path = os.path.join(ROOT, "oracle", "_ref", name)
    return ctypes.CDLL(path) if orc.have_ref() and os.path.exists(path) else None


def test_path_helpers_match_the_reference(orc):
    """PathTo / Root / Catenate / Numbered_Suffix (DB.c:112-202) of libdexcompat.so against the
    reference's own, compiled from DB.c into oracle/_ref/libdbqv_ref.so (or their stored results)."""
    R, L = _ref_lib(orc, "libdbqv_ref.so"), _load("libdexcompat.so")
    libc = ctypes.CDLL(None)
    libc.free.argtypes = [ctypes.c_void_p]
    for lib in (R, L):
        if lib is None:
            continue
        lib.PathTo.restype = lib.Root.restype = ctypes.c_void_p
        lib.PathTo.argtypes = [ctypes.c_char_p]
        lib.Root.argtypes = [ctypes.c_char_p, ctypes.c_char_p]
        lib.Catenate.restype = lib.Numbered_Suffix.restype = ctypes.c_char_p
        lib.Catenate.argtypes = [ctypes.c_char_p] * 4
        lib.Numbered_Suffix.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_char_p]

    def owned(lib, fn, *a):
        # the helpers edit their argument in place for a moment (DB.c:118-121): give them a buffer
        bufs = [ctypes.create_string_buffer(x) if isinstance(x, bytes) else x for x in a]
        p = getattr(lib, fn)(*[ctypes.cast(b, ctypes.c_char_p) if b is not None else None for b in bufs])
        if not p:
            return repr(None)
        s = ctypes.string_at(p)
        libc.free(p)
        return repr(s)

    names = [b"x", b"x.fasta", b"x.FASTA", b"dir/x.fasta", b"/x.fasta", b"/abs/dir.d/x.y.z", b".fasta",
             b"a.fasta.fasta", b"dir.fasta/x", b"", b"trailing/", b"x.quiva", b"./x", b"../x.dexqv"]
    for n in names:
        check(f"PathTo {n!r}", owned(L, "PathTo", n), lambda: owned(R, "PathTo", n), R is not None)
        for suf in (b".fasta", b".quiva", b".dexqv", b"", None):
            check(f"Root {n!r} {suf!r}", owned(L, "Root", n, suf), lambda: owned(R, "Root", n, suf), R is not None)
    for a in ((b".", b"/", b"x", b".dexqv"), (b"", b"", b"", b""), (b"/abs", b"/", b"r" * 500, b".q")):
        check(f"Catenate {a!r}", repr(L.Catenate(*a)), lambda: repr(R.Catenate(*a)), R is not None)
    for a in ((b"_", 17, b".las"), (b"", -3, b""), (b"x" * 300, 2**31 - 1, b"y")):
        check(f"Numbered_Suffix {a!r}", repr(L.Numbered_Suffix(*a)), lambda: repr(R.Numbered_Suffix(*a)), R is not None)
    assert L.Catenate(None, b"", b"", b"") is None and L.Numbered_Suffix(None, 1, b"") is None


def test_line_reader_matches_the_interactive_reference(orc, shim, tmp_path):
    """Read_Lines of libdexcompat_i.so beside the reference's own (QV.c:751-798 compiled with
    -DINTERACTIVE into oracle/_ref/libdbqv_ref_i.so, or its stored results): same return values,
    same lines, same line counter, same Ebuffer text, call by call over well-formed and broken inputs."""
    R = _ref_lib(orc, "libdbqv_ref_i.so")
    if R is not None:
        R.Read_Lines.argtypes = [ctypes.c_void_p, ctypes.c_int]
        R.QVentry.restype = ctypes.c_void_p
        rbuf = (ctypes.c_char * 1000).in_dll(R, "Ebuffer")
    shim.L.QVentry.restype = ctypes.c_void_p
    files = {
        "good": b"@m/1/0_4 RQ=0.850\nabcd\nefgh\nijkl\nmnop\nqrst\n@m/2/0_2 RQ=0.8\nab\ncd\nef\ngh\nij\n",
        "ragged": b"@h\nabc\nab\nabc\nabc\nabc\n",
        "no_newline": b"@h\nabcd\nefgh\nijkl\nmnop\nqrs",
        "short": b"@h\nabcd\nefgh\n",
        "empty_lines": b"@h\n\n\n\n\n\n",
        "empty": b"",
        "long": b"@h\n" + b"".join(bytes([70 + k]) * 120_000 + b"\n" for k in range(5)),
    }

    def step(lib, ebuf, f, nl):
        ebuf.value = b""
        a = lib.Read_Lines(f, nl)
        # the first line read sits at QVentry(); the reference keeps the newline, so compare up to it
        line = refgold.sha(ctypes.string_at(lib.QVentry(), a)) if a >= 0 else None
        return json.dumps([a, ebuf.value.decode("latin-1"), lib.Get_QV_Line(), line])

    for name, data in files.items():
        p = tmp_path / name
        p.write_bytes(data)
        fo = shim.open(p)
        fr = shim.open(p) if R is not None else None
        shim.L.Set_QV_Line(0)
        if R is not None:
            R.Set_QV_Line(0)
        for k in range(8):
            nl = 1 if k % 2 == 0 else 5
            got = step(shim.L, shim.ebuf, fo, nl)
            check(f"Read_Lines {name} {k}", got, lambda: step(R, rbuf, fr, nl), R is not None)
            if json.loads(got)[0] < 0:
                break
        shim.libc.fclose(fo)
        if fr is not None:
            shim.libc.fclose(fr)
    shim.L.QVentry.restype = ctypes.c_char_p


class _QVcoding(ctypes.Structure):                          # QV.h:31-42
    _fields_ = [("schemes", ctypes.c_void_p * 6), ("delChar", ctypes.c_int),
                ("subChar", ctypes.c_int), ("flip", ctypes.c_int), ("prefix", ctypes.c_char_p)]


@pytest.mark.parametrize("seed", range(6))
def test_coding_header_io_matches_the_reference_functions(orc, tmp_path, seed):
    """Read_QVcoding + Write_QVcoding of libdexcompat.so (host work) beside the reference's own
    functions (or their stored results) on real .dexqv files: same delChar / subChar / flip / prefix,
    same file position after the read, same bytes written back -- and those are the bytes of the
    file's header."""
    from tests import fuzz
    text, _ = fuzz.fuzz_quiva(seed)
    data = orc.dexqv(text, lossy=bool(seed & 1))
    src = tmp_path / "f.dexqv"
    src.write_bytes(data)
    libc = ctypes.CDLL(None)
    libc.fopen.restype = ctypes.c_void_p
    libc.fopen.argtypes = [ctypes.c_char_p, ctypes.c_char_p]
    for fn in (libc.fclose, libc.ftell):
        fn.argtypes = [ctypes.c_void_p]
    libc.fseek.argtypes = [ctypes.c_void_p, ctypes.c_long, ctypes.c_int]
    libc.ftell.restype = ctypes.c_long

    def header_io(lib):
        lib.Read_QVcoding.restype = ctypes.POINTER(_QVcoding)
        lib.Read_QVcoding.argtypes = [ctypes.c_void_p]
        lib.Write_QVcoding.argtypes = [ctypes.c_void_p, ctypes.POINTER(_QVcoding)]
        lib.Free_QVcoding.argtypes = [ctypes.POINTER(_QVcoding)]
        f = libc.fopen(str(src).encode(), b"r")
        libc.fseek(f, 2, 0)                                  # the caller reads the 0x55aa key itself
        c = lib.Read_QVcoding(f)
        assert c
        pos = libc.ftell(f)
        out = tmp_path / "w.bin"
        g = libc.fopen(str(out).encode(), b"w")
        lib.Write_QVcoding(g, c)
        libc.fclose(g)
        seen = (c.contents.delChar, c.contents.subChar, c.contents.flip, c.contents.prefix.decode("latin-1"),
                pos, out.read_bytes())
        lib.Free_QVcoding(c)                                 # frees prefix too (QV.c:1324-1334)
        libc.fclose(f)
        return seen

    def value(seen):
        return json.dumps([*seen[:5], refgold.sha(seen[5])])

    R = _ref_lib(orc, "libdbqv_ref.so")
    mine = header_io(_load("libdexcompat.so"))
    check(f"QVcoding header io seed={seed}", value(mine), lambda: value(header_io(R)), R is not None)
    assert mine[5] == data[2:mine[4]]
