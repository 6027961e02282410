"""ctypes binding of include/dexb200.h (libdexb200.so).  No codec logic lives here."""
from __future__ import annotations

import ctypes as C
import os
import sys
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libdexb200.so")
FASTA, ARROW = 0, 1

ERRNAMES = {-1: "FORMAT", -2: "CAP", -3: "TRUNC", -4: "KEY", -5: "LINELEN", -6: "TOOLONG",
            -7: "ARG", -8: "NOMEM", -9: "NOGPU", -10: "CUDA", -11: "CODING"}

# every symbol include/dexb200.h declares (checked by tests/test_abi.py)
SYMBOLS = [
    "dx_open", "dx_close", "dx_strerror", "dx_error_line", "dx_needed_bytes", "dx_sync", "dx_stream",
    "dx_device_alloc", "dx_device_free", "dx_pinned_alloc", "dx_pinned_free", "dx_h2d", "dx_d2h", "dx_d2d",
    "dx_launch_count", "dx_profile", "dx_profile_report", "dx_route",
    "dx_dexta_dev", "dx_dexta_host", "dx_undexta_dev", "dx_undexta_host", "dx_undexta_size_host",
    "dx_undexta_size_dev",
    "dx_compress_reads_dev", "dx_uncompress_reads_dev",
    "dx_qv_scan_dev", "dx_qv_make_coding", "dx_qv_write_coding", "dx_qv_read_coding",
    "dx_qv_encode_dev", "dx_dexqv_dev", "dx_dexqv_host", "dx_undexqv_dev", "dx_undexqv_host",
    "dx_undexqv_size_dev", "dx_keep_index", "dx_last_index", "dx_qv_forget", "dx_qv_last_well",
    "dx_text_lines_dev", "dx_qv_load_entries_dev",
    "dx_undexqv_range_dev", "dx_undexqv_range_chain", "dx_undexqv_range_text_dev",
    "dx_mem_info", "dx_set_origin", "dx_dexta_part_dev", "dx_last_entries", "dx_undexta_window_dev",
]


def _wait_for_torch():
    """The library runs on its own non-blocking stream.  Callers of the *_dev methods here are the
    tests and bench.py, which make their buffers with torch on torch's current stream: wait for that
    stream, so that a fill or a copy still in flight cannot race with the library's kernels."""
    t = sys.modules.get("torch")
    if t is not None and t.cuda.is_available() and t.cuda.is_initialized():
        t.cuda.current_stream().synchronize()


class DexError(RuntimeError):
    def __init__(self, code, text="", line=0):
        super().__init__(f"dexb200 error {code} ({ERRNAMES.get(code, '?')}): {text}")
        self.code, self.text, self.line = code, text, line


class Stats(C.Structure):
    _fields_ = [("hist", (C.c_uint64 * 256) * 6), ("totchar", C.c_uint64),
                ("nentries", C.c_int64), ("delchar", C.c_int32), ("subchar", C.c_int32),
                ("sub_prefix", C.c_uint64 * 256)]


class Carry(C.Structure):
    _fields_ = [("delchar", C.c_int32), ("subchar", C.c_int32), ("totchar", C.c_uint64),
                ("sub", C.c_uint64 * 256)]


class IndexRow(C.Structure):
    _fields_ = [("stream_off", C.c_int64), ("end_off", C.c_int64), ("text_off", C.c_int64),
                ("rlen", C.c_int32), ("well", C.c_int32)]


class Scheme(C.Structure):
    _fields_ = [("type", C.c_int32), ("bits", C.c_uint32 * 256), ("lens", C.c_int32 * 256)]


class Coding(C.Structure):
    _fields_ = [("tab", Scheme * 6), ("delchar", C.c_int32), ("subchar", C.c_int32),
                ("flip", C.c_int32)]


def build_library(verbose: bool = False) -> str:
    """Compile libdexb200.so for sm_100a (nvcc cross-compiles; no GPU needed)."""
    out = subprocess.run(["bash", os.path.join(HERE, "csrc", "build.sh")], capture_output=True,
                         text=True)
    if verbose or out.returncode != 0:
        print(out.stdout, out.stderr)
    if out.returncode != 0:
        raise RuntimeError("building libdexb200.so failed")
    return LIB_PATH


_lib = None


def load_library():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; "
                           "g.build()'` (there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, sz, i64, i32 = C.c_void_p, C.c_size_t, C.c_int64, C.c_int32
    szp = C.POINTER(C.c_size_t)
    sig = {
        "dx_open": (C.c_int, [C.c_int, C.POINTER(vp)]),
        "dx_close": (None, [vp]),
        "dx_strerror": (C.c_char_p, [vp]),
        "dx_error_line": (i64, [vp]),
        "dx_needed_bytes": (C.c_size_t, [vp]),
        "dx_sync": (C.c_int, [vp]),
        "dx_stream": (vp, [vp]),
        "dx_device_alloc": (vp, [vp, sz]),
        "dx_device_free": (None, [vp, vp]),
        "dx_pinned_alloc": (vp, [vp, sz]),
        "dx_pinned_free": (None, [vp, vp]),
        "dx_h2d": (C.c_int, [vp, vp, vp, sz]),
        "dx_d2h": (C.c_int, [vp, vp, vp, sz]),
        "dx_d2d": (C.c_int, [vp, vp, vp, sz]),
        "dx_launch_count": (C.c_uint64, [vp, C.c_int]),
        "dx_profile": (C.c_int, [vp, C.c_int]),
        "dx_route": (C.c_int, [vp, C.c_char_p, i64]),
        "dx_profile_report": (C.c_int, [vp, C.c_char_p, sz]),
        "dx_dexta_dev": (C.c_int, [vp, C.c_int, vp, sz, vp, sz, szp]),
        "dx_dexta_host": (C.c_int, [vp, C.c_int, vp, sz, vp, sz, szp]),
        "dx_undexta_dev": (C.c_int, [vp, C.c_int, vp, sz, C.c_int, C.c_int, vp, sz, szp]),
        "dx_undexta_host": (C.c_int, [vp, C.c_int, vp, sz, C.c_int, C.c_int, vp, sz, szp]),
        "dx_undexta_size_host": (C.c_int, [vp, C.c_int, vp, sz, C.c_int, szp]),
        "dx_undexta_size_dev": (C.c_int, [vp, C.c_int, vp, sz, C.c_int, szp]),
        "dx_compress_reads_dev": (C.c_int, [vp, C.c_int, vp, vp, vp, i64, vp, vp]),
        "dx_uncompress_reads_dev": (C.c_int, [vp, C.c_int, C.c_int, vp, vp, vp, i64, vp, vp]),
        "dx_qv_scan_dev": (C.c_int, [vp, vp, sz, C.POINTER(Carry), C.POINTER(Stats)]),
        "dx_qv_make_coding": (C.c_int, [C.POINTER(Stats), C.c_int, C.POINTER(Coding)]),
        "dx_qv_write_coding": (C.c_int, [C.POINTER(Coding), C.c_char_p, C.c_int, vp, sz, szp]),
        "dx_qv_read_coding": (C.c_int, [vp, sz, C.POINTER(Coding), C.c_char_p, C.c_int, szp]),
        "dx_qv_encode_dev": (C.c_int, [vp, vp, sz, C.POINTER(Coding), C.c_int, i32, vp, sz, szp,
                                       C.POINTER(i32), vp, i64]),
        "dx_dexqv_dev": (C.c_int, [vp, vp, sz, C.c_int, vp, sz, szp]),
        "dx_dexqv_host": (C.c_int, [vp, vp, sz, C.c_int, vp, sz, szp]),
        "dx_undexqv_dev": (C.c_int, [vp, vp, sz, C.c_int, vp, sz, szp, vp, i64, i32]),
        "dx_undexqv_host": (C.c_int, [vp, vp, sz, C.c_int, vp, sz, szp]),
        "dx_undexqv_size_dev": (C.c_int, [vp, vp, sz, szp]),
        "dx_keep_index": (C.c_int, [vp, C.c_int]),
        "dx_qv_forget": (C.c_int, [vp]),
        "dx_qv_load_entries_dev": (C.c_int, [vp, vp, sz, C.POINTER(Coding), vp, vp, i64, C.c_int, vp, sz, vp, vp]),
        "dx_qv_last_well": (C.c_int, [vp, C.POINTER(i32)]),
        "dx_text_lines_dev": (C.c_int, [vp, vp, sz, i64, C.POINTER(i64), C.POINTER(i64)]),
        "dx_last_index": (C.c_int, [vp, vp, i64, C.POINTER(i64)]),
        "dx_undexqv_range_dev": (C.c_int, [vp, vp, sz, vp, sz, i64, i64, i64, C.c_int, C.POINTER(i64)]),
        "dx_undexqv_range_chain": (C.c_int, [vp, i64, i32, C.POINTER(i64), C.POINTER(i32)]),
        "dx_undexqv_range_text_dev": (C.c_int, [vp, vp, sz, szp]),
        "dx_mem_info": (C.c_int, [vp, szp, szp, szp]),
        "dx_set_origin": (C.c_int, [vp, i64, i64]),
        "dx_dexta_part_dev": (C.c_int, [vp, C.c_int, vp, sz, i32, C.c_int, vp, sz, szp, C.POINTER(i32)]),
        "dx_last_entries": (i64, [vp]),
        "dx_undexta_window_dev": (C.c_int, [vp, C.c_int, vp, sz, vp, sz, i64, i64, i32, C.c_int, C.c_int, C.c_int,
                                            vp, sz, szp, C.POINTER(i64), C.POINTER(i32)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    _lib = L
    return L


def make_coding(stats: Stats, lossy: bool = False) -> Coding:
    """dx_qv_make_coding: host only, needs no GPU (replaces Create_QVcoding, QV.c:1029-1169)."""
    cd = Coding()
    rc = load_library().dx_qv_make_coding(C.byref(stats), int(lossy), C.byref(cd))
    if rc != 0:
        raise DexError(rc, "dx_qv_make_coding")
    return cd


def write_coding(coding: Coding, prefix: bytes) -> bytes:
    out = np.empty(20000 + len(prefix), dtype=np.uint8)
    n = C.c_size_t(0)
    rc = load_library().dx_qv_write_coding(C.byref(coding), prefix, len(prefix), out.ctypes.data,
                                           out.size, C.byref(n))
    if rc != 0:
        raise DexError(rc, "dx_qv_write_coding")
    return out[: n.value].tobytes()


def read_coding(data: bytes):
    """-> (Coding, prefix bytes, bytes consumed)"""
    cd = Coding()
    pre = C.create_string_buffer(100001)
    used = C.c_size_t(0)
    src = np.frombuffer(data, dtype=np.uint8)
    rc = load_library().dx_qv_read_coding(src.ctypes.data, len(data), C.byref(cd), pre, len(pre),
                                          C.byref(used))
    if rc != 0:
        raise DexError(rc, "dx_qv_read_coding")
    return cd, pre.value, used.value


class Context:
    """One dx_ctx: one GPU, one stream.  Host-buffer methods take/return bytes; *_dev methods
    take raw device addresses (e.g. torch.Tensor.data_ptr()) and stay on the device."""

    def __init__(self, device: int = 0):
        self.L = load_library()
        h = C.c_void_p()
        rc = self.L.dx_open(device, C.byref(h))
        if rc != 0:
            raise DexError(rc, "dx_open failed (no CUDA device? there is no CPU fallback)")
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.L.dx_close(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise DexError(rc, self.L.dx_strerror(self.h).decode(errors="replace"),
                           self.L.dx_error_line(self.h))

    @property
    def stream(self) -> int:
        return int(self.L.dx_stream(self.h) or 0)

    def sync(self):
        self._check(self.L.dx_sync(self.h))

    def launch_count(self, reset: bool = False) -> int:
        return int(self.L.dx_launch_count(self.h, int(reset)))

    def h2d(self, d_dst: int, data: bytes):
        """small synchronous host->device copy on the context's stream"""
        _wait_for_torch()
        src = np.frombuffer(data, dtype=np.uint8)
        self._check(self.L.dx_h2d(self.h, d_dst, src.ctypes.data, len(data)))
        self.sync()

    def route(self, name: str = "default", value: int = 1):
        """test hook: force an alternative path (dx_route); route() resets every route"""
        self._check(self.L.dx_route(self.h, name.encode(), int(value)))

    def profile(self, enable: bool):
        self._check(self.L.dx_profile(self.h, int(enable)))

    def profile_report(self) -> dict:
        """{kernel name: (calls, total ms)} since the last report; clears the records"""
        buf = C.create_string_buffer(1 << 16)
        self._check(self.L.dx_profile_report(self.h, buf, len(buf)))
        out = {}
        for line in buf.value.decode().splitlines():
            name, calls, ms = line.split()
            out[name] = (int(calls), float(ms))
        return out

    # ---- host-buffer API (copies included) ----------------------------------------------------
    def dexta(self, text: bytes, kind: int = FASTA) -> bytes:
        out = np.empty(len(text) // 2 + 4096, dtype=np.uint8)
        n = C.c_size_t(0)
        src = np.frombuffer(text, dtype=np.uint8)
        rc = self.L.dx_dexta_host(self.h, kind, src.ctypes.data, len(text), out.ctypes.data, out.size,
                                  C.byref(n))
        if rc == -2 and self.L.dx_needed_bytes(self.h) > out.size:      # DX_E_CAP: go again with what it needs
            out = np.empty(self.L.dx_needed_bytes(self.h) + 64, dtype=np.uint8)
            rc = self.L.dx_dexta_host(self.h, kind, src.ctypes.data, len(text), out.ctypes.data, out.size,
                                      C.byref(n))
        self._check(rc)
        return out[: n.value].tobytes()

    def undexta(self, data: bytes, kind: int = FASTA, width: int = 80, upper: bool = False) -> bytes:
        src = np.frombuffer(data, dtype=np.uint8)
        need = C.c_size_t(0)
        self._check(self.L.dx_undexta_size_host(self.h, kind, src.ctypes.data, len(data), width,
                                                C.byref(need)))
        out = np.empty(need.value + 16, dtype=np.uint8)
        n = C.c_size_t(0)
        self._check(self.L.dx_undexta_host(self.h, kind, src.ctypes.data, len(data), width,
                                           int(upper), out.ctypes.data, out.size, C.byref(n)))
        return out[: n.value].tobytes()

    def dexqv(self, text: bytes, lossy: bool = False) -> bytes:
        out = np.empty(len(text) * 3 + 200000, dtype=np.uint8)
        n = C.c_size_t(0)
        src = np.frombuffer(text, dtype=np.uint8)
        self._check(self.L.dx_dexqv_host(self.h, src.ctypes.data, len(text), int(lossy),
                                         out.ctypes.data, out.size, C.byref(n)))
        return out[: n.value].tobytes()

    def undexqv(self, data: bytes, upper: bool = False, cap: int | None = None) -> bytes:
        src = np.frombuffer(data, dtype=np.uint8)
        out = np.empty(cap if cap is not None else len(data) * 40 + 200000, dtype=np.uint8)
        n = C.c_size_t(0)
        self._check(self.L.dx_undexqv_host(self.h, src.ctypes.data, len(data), int(upper),
                                           out.ctypes.data, out.size, C.byref(n)))
        return out[: n.value].tobytes()

    def dexqv_host_ptr(self, h_text: int, n: int, lossy: bool, h_out: int, cap: int) -> int:
        """dx_dexqv_host on raw HOST addresses (e.g. pinned torch tensors): copies included"""
        m = C.c_size_t(0)
        self._check(self.L.dx_dexqv_host(self.h, h_text, n, int(lossy), h_out, cap, C.byref(m)))
        return m.value

    def undexqv_host_ptr(self, h_in: int, n: int, upper: bool, h_out: int, cap: int) -> int:
        m = C.c_size_t(0)
        self._check(self.L.dx_undexqv_host(self.h, h_in, n, int(upper), h_out, cap, C.byref(m)))
        return m.value

    # ---- device-pointer API ---------------------------------------------------------------------
    def dexta_dev(self, kind, d_text, n, d_out, cap) -> int:
        _wait_for_torch()
        m = C.c_size_t(0)
        self._check(self.L.dx_dexta_dev(self.h, kind, d_text, n, d_out, cap, C.byref(m)))
        return m.value

    def undexta_dev(self, kind, d_in, n, width, upper, d_out, cap) -> int:
        _wait_for_torch()
        m = C.c_size_t(0)
        self._check(self.L.dx_undexta_dev(self.h, kind, d_in, n, width, int(upper), d_out, cap,
                                          C.byref(m)))
        return m.value

    def compress_reads_dev(self, kind, d_src, d_src_off, d_len, nreads, d_dst, d_dst_off):
        _wait_for_torch()
        self._check(self.L.dx_compress_reads_dev(self.h, kind, d_src, d_src_off, d_len, nreads,
                                                 d_dst, d_dst_off))

    def uncompress_reads_dev(self, kind, upper, d_src, d_src_off, d_len, nreads, d_dst, d_dst_off):
        _wait_for_torch()
        self._check(self.L.dx_uncompress_reads_dev(self.h, kind, int(upper), d_src, d_src_off,
                                                   d_len, nreads, d_dst, d_dst_off))

    def qv_scan_dev(self, d_text, n, carry: Carry | None = None) -> Stats:
        _wait_for_torch()
        st = Stats()
        self._check(self.L.dx_qv_scan_dev(self.h, d_text, n,
                                          C.byref(carry) if carry is not None else None,
                                          C.byref(st)))
        return st

    def qv_encode_dev(self, d_text, n, coding: Coding, lossy, lwell_in, d_out, cap,
                      want_offsets: int = 0):
        _wait_for_torch()
        m = C.c_size_t(0)
        lastw = C.c_int32(0)
        offs = np.empty(want_offsets + 1, dtype=np.int64) if want_offsets else None
        self._check(self.L.dx_qv_encode_dev(self.h, d_text, n, C.byref(coding), int(lossy),
                                            lwell_in, d_out, cap, C.byref(m), C.byref(lastw),
                                            offs.ctypes.data if offs is not None else None,
                                            want_offsets))
        return m.value, lastw.value, offs

    def dexqv_dev(self, d_text, n, lossy, d_out, cap) -> int:
        _wait_for_torch()
        m = C.c_size_t(0)
        self._check(self.L.dx_dexqv_dev(self.h, d_text, n, int(lossy), d_out, cap, C.byref(m)))
        return m.value

    def undexqv_dev(self, d_in, n, upper, d_out, cap, entry_off: np.ndarray | None = None,
                    well_in: int = 0) -> int:
        _wait_for_torch()
        m = C.c_size_t(0)
        if entry_off is not None:
            entry_off = np.ascontiguousarray(entry_off, dtype=np.int64)
            self._check(self.L.dx_undexqv_dev(self.h, d_in, n, int(upper), d_out, cap, C.byref(m),
                                              entry_off.ctypes.data, len(entry_off) - 1, well_in))
        else:
            self._check(self.L.dx_undexqv_dev(self.h, d_in, n, int(upper), d_out, cap, C.byref(m),
                                              None, 0, well_in))
        return m.value

    def qv_load_entries_dev(self, d_in, n, coding: Coding, stream_off, rlen, upper, d_out, cap):
        """-> (out offsets [nentries+1], end offsets [nentries])"""
        _wait_for_torch()
        so = np.ascontiguousarray(stream_off, dtype=np.int64)
        rl = np.ascontiguousarray(rlen, dtype=np.int32)
        oo = np.zeros(len(so) + 1, dtype=np.int64)
        eo = np.zeros(len(so), dtype=np.int64)
        self._check(self.L.dx_qv_load_entries_dev(self.h, d_in, n, C.byref(coding), so.ctypes.data,
                                                  rl.ctypes.data, len(so), int(upper), d_out, cap,
                                                  oo.ctypes.data, eo.ctypes.data))
        return oo, eo

    def qv_forget(self):
        self._check(self.L.dx_qv_forget(self.h))

    def qv_last_well(self) -> int:
        w = C.c_int32(0)
        self._check(self.L.dx_qv_last_well(self.h, C.byref(w)))
        return w.value

    def text_lines_dev(self, d_text, n, skip: int = 0):
        """-> (newlines in the buffer, offset just behind the skip-th newline or -1)"""
        _wait_for_torch()
        cnt, off = C.c_int64(0), C.c_int64(0)
        self._check(self.L.dx_text_lines_dev(self.h, d_text, n, skip, C.byref(cnt), C.byref(off)))
        return cnt.value, off.value

    def keep_index(self, keep: bool = True):
        self._check(self.L.dx_keep_index(self.h, int(keep)))

    def last_index(self):
        """rows (stream_off, end_off, text_off, rlen, well) of the last undexqv_dev call"""
        cnt = C.c_int64(0)
        self._check(self.L.dx_last_index(self.h, None, 0, C.byref(cnt)))
        rows = (IndexRow * max(cnt.value, 1))()
        self._check(self.L.dx_last_index(self.h, rows, cnt.value, C.byref(cnt)))
        return [(r.stream_off, r.end_off, r.text_off, r.rlen, r.well) for r in rows[: cnt.value]]

    def needed_bytes(self) -> int:
        """what the last call that failed with DX_E_CAP needed (dx_needed_bytes)"""
        return int(self.L.dx_needed_bytes(self.h))

    # ---- one byte range of a .dexqv image (dx_undexqv_range_*): decode, chain, text ----------------
    def undexqv_range_dev(self, head: bytes, d_buf, buf_n, buf_off, a, b, upper=False) -> int:
        """speculative decode of the range [a, b) from the image bytes [buf_off, buf_off + buf_n) at
        d_buf; head: the image's first bytes (key and coding header).  -> the first entry's offset"""
        _wait_for_torch()
        first = C.c_int64(0)
        src = np.frombuffer(head, dtype=np.uint8)
        self._check(self.L.dx_undexqv_range_dev(self.h, src.ctypes.data, len(head), d_buf, buf_n, buf_off,
                                                a, b, int(upper), C.byref(first)))
        return first.value

    def undexqv_range_chain(self, cur_in: int, well_in: int):
        """-> (where the next range's chain starts, the well of this range's last entry)"""
        cur, well = C.c_int64(0), C.c_int32(0)
        self._check(self.L.dx_undexqv_range_chain(self.h, cur_in, well_in, C.byref(cur), C.byref(well)))
        return cur.value, well.value

    def undexqv_range_text_dev(self, d_out, cap) -> int:
        m = C.c_size_t(0)
        self._check(self.L.dx_undexqv_range_text_dev(self.h, d_out, cap, C.byref(m)))
        return m.value

    # ---- files window by window: 2-bit parts and windows, origin, memory --------------------------------
    def mem_info(self):
        """-> (free, total, held) device bytes (dx_mem_info)"""
        f, t, h = C.c_size_t(0), C.c_size_t(0), C.c_size_t(0)
        self._check(self.L.dx_mem_info(self.h, C.byref(f), C.byref(t), C.byref(h)))
        return f.value, t.value, h.value

    def set_origin(self, line0: int = 0, entry0: int = 0):
        self._check(self.L.dx_set_origin(self.h, line0, entry0))

    def last_entries(self) -> int:
        return int(self.L.dx_last_entries(self.h))

    def dexta_part_dev(self, kind, d_text, n, lwell_in, with_header, d_out, cap):
        """-> (output bytes, well of the part's last entry)"""
        _wait_for_torch()
        m, lastw = C.c_size_t(0), C.c_int32(0)
        self._check(self.L.dx_dexta_part_dev(self.h, kind, d_text, n, lwell_in, int(with_header), d_out, cap,
                                             C.byref(m), C.byref(lastw)))
        return m.value, lastw.value

    def undexta_window_dev(self, kind, head: bytes, d_buf, buf_n, buf_off, cur_in, well_in, is_last, width,
                           upper, d_out, cap):
        """-> (text bytes, next chain position, well in front of it)"""
        _wait_for_torch()
        m, cur, well = C.c_size_t(0), C.c_int64(0), C.c_int32(0)
        src = np.frombuffer(head, dtype=np.uint8)
        self._check(self.L.dx_undexta_window_dev(self.h, kind, src.ctypes.data, len(head), d_buf, buf_n, buf_off,
                                                 cur_in, well_in, int(is_last), width, int(upper), d_out, cap,
                                                 C.byref(m), C.byref(cur), C.byref(well)))
        return m.value, cur.value, well.value

    def undexqv_size_dev(self, d_in, n) -> int:
        _wait_for_torch()
        m = C.c_size_t(0)
        self._check(self.L.dx_undexqv_size_dev(self.h, d_in, n, C.byref(m)))
        return m.value
