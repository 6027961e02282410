"""Entry framing of the 2-bit formats (.dexta / .dexar) and of .quiva headers at the edges of the
device parsers: crafted texts and images for tests/test_header_shapes_oracle.py (CPU) and
tests/test_gpu_header_shapes.py (GPU).

Every header the synthetic generators write is canonical: wells never decrease and move by less
than 40, beg is below 20 000, RQ has three digits, SNRs have two decimals in 4.00 ... 15.00.  The
library treats headers by shape, so the shapes here aim at its branches:

  grammar       headers at the hand-off between the device parsers (unsigned runs of at most 9
                digits, two-decimal SNRs of at most 99999) and the host's sscanf, mixed in one file
                so that both kinds sit in the same launch;
  snr_all       every two-decimal SNR 0.00 ... 99.99 (and a few beyond) in .arrow text, and crafted
                .dexar images whose stored SNR codes cover all 65 536 values;
  window        one true entry just inside / just outside the window of the 2-bit candidate filter
                (beg < 2^27, end - beg <= 2^20, qv < 2^16) in a file of ordinary entries;
  well_jumps    well deltas around 255 and around 255 * 2^20 (about a MB of 0xff bytes, at the cap of
                the 0xff-run count), first wells 0 / 255 / 256, and wells that drop;
  zero_payload  reads that pack to zero bytes (all 'a', all 'N', arrow all '1'): every offset of their
                payload is a candidate, which overflows the one-pass index;
  legacy_2bit   foreign byte order and the old 16-bit .dexta layout, rewritten from a native image.

Each generator returns bytes.  expected_route gives the route a decode of an image takes, from
candidate_positions, a numpy restatement of the candidate predicate of dx_frame.cu."""
from __future__ import annotations

import struct

import numpy as np

from dextractor_b200 import synth

MOVIE = "m54321_201020_123456"

# the window of DX_PRED_QVCAND / DX_PRED_ARCAND (dx_frame.cu) and of the 0xff-run count
CAND_MAX_BEG = 1 << 27
CAND_MAX_LEN = 1 << 20
CAND_MAX_QV = 1 << 16
CAND_MAX_SNR = 9999
FFRUN_CAP = 1 << 20
TILE_BYTES = 16384
TILE_SLOTS = 16

# The route of a dx_undexta_* call is two choices, asserted from the kernel profile on the GPU:
#   the candidate index   INDEX_SLOTS     one pass, at most 16 hits a tile: k_pred_slots + k_pred_gather
#                         INDEX_TWO_PASS  a tile overflows: k_pred_count + k_pred_write
#   the entry chain       CHAIN_FAST      device-planned (undexta_fast): k_pk_cand_prep + k_unpack3
#                         CHAIN_GENERAL   the fast chain gives up: plan_undexta, resolve_chain (k_pk_walk,
#                                         k_cand_context, the host walk for entries that are not
#                                         candidates) and k_unpack
INDEX_SLOTS, INDEX_TWO_PASS = "slots", "two_pass"
CHAIN_FAST, CHAIN_GENERAL = "fast", "general"

ACGT = np.frombuffer(b"acgt", dtype=np.uint8)
ARROW = np.frombuffer(b"1234", dtype=np.uint8)


def _seq(rng, n, arrow=False):
    return (ARROW if arrow else ACGT)[rng.integers(0, 4, size=n)].tobytes()


def _wrap(seq: bytes, width: int = 80) -> bytes:
    return synth._wrap(np.frombuffer(seq, dtype=np.uint8), width)


def entry(tail: str, seq: bytes, width: int = 80) -> bytes:
    """one .fasta / .arrow entry: '>' MOVIE '/' tail, then the sequence in lines of `width`"""
    return f">{MOVIE}/{tail}\n".encode() + _wrap(seq, width)


def _snr(rng):
    return ",".join(f"{x:.2f}" for x in rng.integers(400, 1501, size=4) / 100.0)


def ordinary(rng, well, arrow=False, L=None, beg=None):
    """a canonical entry"""
    L = int(rng.integers(50, 400)) if L is None else L
    beg = int(rng.integers(0, 20000)) if beg is None else beg
    tail = f"{well}/{beg}_{beg + L} " + (f"SN={_snr(rng)}" if arrow else f"RQ=0.{int(rng.integers(750, 900))}")
    return entry(tail, _seq(rng, L, arrow))


# ---- grammar ---------------------------------------------------------------------------------------

# (tail after MOVIE '/', sequence length, True when the device parsers take the header themselves).
# Wells rise from entry to entry; end - beg (as sscanf reads them) is the sequence length, so the
# image decodes back to the same entries.
GRAMMAR_FASTA = [
    ("10/0_100 RQ=0.851", 100, True),
    ("11/123456789_123456889 RQ=0.123456789", 100, True),          # 9 digits everywhere
    ("12/999999999_1000000099 RQ=0.850", 100, False),             # 10 digits
    ("13/2147483547_2147483647 RQ=0.2147483647", 100, False),
    ("14/4294967295_99 RQ=0.4294967295", 100, False),              # %d: 4294967295 -> -1
    ("0000000015/0_100 RQ=0.851", 100, False),                     # 10 digits of which 8 leading zeros
    ("016/007_107 RQ=0.085", 100, True),                           # leading zeros
    ("17/+5_+105 RQ=0.+851", 100, False),
    ("18/-5_95 RQ=0.-851", 100, False),
    ("19/ 5_ 105 RQ=0. 851", 100, False),                          # blanks after / _ and RQ=0.
    (" 20/5_105 RQ=0.851", 100, False),                            # blank after the prefix's /
    ("21/5_105 RQ=0.", 100, False),                                # no digits: qv 0
    ("22/5_105 RQ=0.851 trailing text", 100, True),
    ("23/5_105 RQ=0.851x", 100, True),
    ("24/5_105RQ=0.851", 100, False),                              # sscanf's blank matches nothing
    ("25/5_105", 100, True),                                       # no RQ at all
    ("26/5_105 RQ=1.851", 100, False),                             # literal 0 does not match: qv 0
    ("27/5_105 RQ= 0.851", 100, False),
    ("28/5_105 rq=0.851", 100, False),
    ("29/5_105 RQ=0.0000000851", 100, False),                      # 10 digits of qv
    ("30/5_105 RQ=0.65535", 100, True),
    ("31/5_105\tRQ=0.851", 100, False),
    ("32/5_5 RQ=0.851", 0, True),
]

GRAMMAR_ARROW = [
    ("10/0_60 SN=5.00,6.00,7.00,8.00", 60, True),
    ("11/0_60 SN=5,6.1,7.12,8.123", 60, False),                    # 0, 1, 2 and 3 decimals
    ("12/0_60 SN=99999.00,99999.99,1.00,2.00", 60, True),          # integer parts of 99999
    ("13/0_60 SN=100000.00,1.00,2.00,3.00", 60, False),            # ... and 100000
    ("14/0_60 SN=5.00,6.00,7.00,100000.00", 60, False),
    ("15/0_60 SN=5.00,6.00,7.00,8.00 trailing", 60, True),         # text after the fourth SNR
    ("16/0_60 SN=5.00,6.00,7.00,8.00x", 60, True),
    ("17/0_60 SN=5.00,6.00,7.00,8.00e1", 60, False),               # strtof reads the exponent
    ("18/0_60 SN=5.00,6.00,7.00,8.00E-1", 60, False),
    ("19/0_60 SN=5.00,6.00,7.00,8.00e", 60, False),                # 'e' without digits: not read
    ("20/0_60 SN= 5.00, 6.00,7.00,8.00", 60, False),
    ("21/0_60 SN=+5.00,-6.00,7.00,8.00", 60, False),
    ("22/0_60 SN=005.00,0.07,0.00,99.99", 60, True),
    ("23/0_60 SN=6.97,99.994,99.995,100.00", 60, False),
    ("24/0_60 SN=655.35,655.36,1000.00,99999.99", 60, True),
    ("25/0_60 SN=5.00,6.00,7.00,8.00,9.00", 60, True),             # a fifth value is trailing text
    ("26/0_60SN=5.00,6.00,7.00,8.00", 60, False),
    ("27/123456789_123456849 SN=5.00,6.00,7.00,8.00", 60, True),
    ("28/999999999_1000000059 SN=5.00,6.00,7.00,8.00", 60, False),
    ("29/4294967295_59 SN=5.00,6.00,7.00,8.00", 60, False),
    ("030/07_067 SN=5.00,6.00,7.00,8.00", 60, True),
    ("31/0_60 SN=.50,6.00,7.00,8.00", 60, False),
    ("32/0_60 SN=5.00,6.00,7.00,8.", 60, False),
]

# .quiva headers: QV.c needs all four fields; without RQ the file is refused
GRAMMAR_QUIVA = [
    ("10/0_{L} RQ=0.851", True),
    ("11/123456789_{L9} RQ=0.123456789", True),
    ("12/999999999_{L10} RQ=0.850", False),
    ("13/4294967295_{Lm1} RQ=0.4294967295", False),
    ("014/007_{L7} RQ=0.085", True),
    ("15/+0_ {L} RQ=0. 851", False),
    ("16/0_{L}RQ=0.851", False),
    ("17/0_{L} RQ=0.851 trailing", True),
    ("18/0_{L} RQ=0.0000000851", False),
    (" 19/0_{L} RQ=0.851", False),
]
GRAMMAR_QUIVA_REFUSED = ["20/0_{L}", "20/0_{L} RQ=0.", "20/0_{L} RQ=1.851"]


def grammar(kind: str) -> bytes:
    """kind 'fasta' / 'arrow' / 'quiva': the grammar headers between canonical entries"""
    rng = np.random.default_rng({"fasta": 1, "arrow": 2, "quiva": 3}[kind])
    if kind == "quiva":
        return _quiva_from_tails(rng, [t for t, _ in GRAMMAR_QUIVA])
    arrow = kind == "arrow"
    parts, well = [], 0
    for i, (tail, L, _) in enumerate(GRAMMAR_ARROW if arrow else GRAMMAR_FASTA):
        well = int(tail.split("/")[0])
        parts.append(ordinary(rng, well, arrow))                   # a canonical entry of the same well
        parts.append(entry(tail, _seq(rng, L, arrow), width=80 if i % 3 else 17))
    parts.append(ordinary(rng, well + 1, arrow))
    return b"".join(parts)


def grammar_quiva_refused(i: int) -> bytes:
    rng = np.random.default_rng(30 + i)
    return _quiva_from_tails(rng, [GRAMMAR_QUIVA_REFUSED[i]])


def _quiva_from_tails(rng, tails):
    text = synth.make_quiva(int(rng.integers(1 << 30)), [int(x) for x in rng.integers(50, 300, size=2 * len(tails) + 1)],
                            movie=MOVIE)
    lines = text.split(b"\n")
    wells = []
    for k, tail in enumerate(tails):
        e = 2 * k + 1
        L = len(lines[6 * e + 1])
        t = tail.format(L=L, L9=123456789 + L, L10=999999999 + L, Lm1=L - 1, L7=7 + L)
        lines[6 * e] = f"@{MOVIE}/{t}".encode()
        wells.append(int(t.split("/")[0]))
    # the canonical entry in front of a crafted one has its well; the last one the next well
    for k, w in enumerate(wells + [wells[-1] + 1]):
        f = lines[12 * k].split(b"/")
        f[1] = str(w).encode()
        lines[12 * k] = b"/".join(f)
    return b"\n".join(lines)


def device_parses(tail: str, arrow: bool) -> bool:
    """The device parsers' acceptance rule, restated: '<well>/<beg>_<end>' of unsigned runs of 1 to 9
    digits, then (fasta) nothing or ' RQ=0.' and 1 to 9 digits, (arrow) ' SN=' and four
    '<1..9 digits <= 99999>.<2 digits>' separated by ',', with no digit and no exponent after the
    last one.  Anything else after the last field is ignored (as sscanf ignores it)."""
    import re
    num = r"[0-9]{1,9}(?![0-9])"
    m = re.match(rf"{num}/{num}_{num}", tail)
    if not m:
        return False
    rest = tail[m.end():]
    if not arrow:
        return rest == "" or re.match(rf" RQ=0\.{num}", rest) is not None
    snr = r"([0-9]{1,9})\.[0-9]{2}"
    m = re.match(rf" SN={snr},{snr},{snr},{snr}(?![0-9eE])", rest)
    return m is not None and all(int(g) <= 99999 for g in m.groups())


# ---- snr_all ----------------------------------------------------------------------------------------

SNR_EXTRA = ["99.994", "99.995", "100.00", "655.35", "655.36", "99999.99"]


def snr_all_arrow() -> bytes:
    """every two-decimal SNR 0.00 ... 99.99, four to an entry, then the SNR_EXTRA values"""
    rng = np.random.default_rng(4)
    vals = [f"{k // 100}.{k % 100:02d}" for k in range(10000)] + SNR_EXTRA
    vals += ["1.00"] * (-len(vals) % 4)
    parts = []
    for i in range(0, len(vals), 4):
        L = int(rng.integers(0, 24))
        parts.append(entry(f"{i // 4}/{i}_{i + L} SN={','.join(vals[i:i + 4])}", _seq(rng, L, True)))
    return b"".join(parts)


def pack2bit(seq: bytes, arrow: bool) -> bytes:
    """Number_Read / Number_Arrow + Compress_Read (DB.c): four symbols a byte, first on top"""
    s = np.frombuffer(seq, dtype=np.uint8)
    code = np.full(256, 3 if arrow else 0, dtype=np.uint8)
    if arrow:
        code[ord("1")], code[ord("2")], code[ord("3")], code[ord("G")] = 0, 1, 2, 2
    else:
        for ch, v in zip(b"cgtCGT", (1, 2, 3, 1, 2, 3)):
            code[ch] = v
    c = np.concatenate([code[s], np.zeros(-len(s) % 4, dtype=np.uint8)]).reshape(-1, 4)
    return ((c[:, 0] << 6) | (c[:, 1] << 4) | (c[:, 2] << 2) | c[:, 3]).astype(np.uint8).tobytes()


def _well_bytes(d: int) -> bytes:
    """put_well of dexta.c: 0xff per 255, then the rest as a byte (a drop wraps)"""
    out = b""
    while d >= 255:
        out += b"\xff"
        d -= 255
    return out + bytes([d & 0xff])


def snr_codes_dexar() -> bytes:
    """a crafted native .dexar image whose four stored SNR codes per entry cover all 65 536 values;
    codes above 9999 are never candidates, so those entries go through the general path"""
    rng = np.random.default_rng(5)
    codes = np.arange(1 << 16, dtype=np.uint16)
    out = bytearray(struct.pack("<Hi", 0x55AA, len(MOVIE) + 1) + f">{MOVIE}".encode())
    for e in range(len(codes) // 4):
        L = int(rng.integers(0, 9))
        beg = int(rng.integers(0, 20000))
        out += _well_bytes(int(e > 0)) + struct.pack("<ii4H", beg, beg + L, *codes[4 * e: 4 * e + 4])
        out += pack2bit(_seq(rng, L, True), True)
    return bytes(out)


# ---- window -----------------------------------------------------------------------------------------

# name -> (field, value, inside the candidate window)
WINDOW = {
    "beg_in": ("beg", CAND_MAX_BEG - 1, True),
    "beg_out": ("beg", CAND_MAX_BEG, False),
    "len_in": ("len", CAND_MAX_LEN, True),
    "len_out": ("len", CAND_MAX_LEN + 1, False),
    "qv_in": ("qv", CAND_MAX_QV - 1, True),
    "qv_out": ("qv", CAND_MAX_QV, False),
}


def window(name: str, arrow: bool = False) -> bytes:
    """ordinary entries with one true entry whose field sits at the edge of the candidate window"""
    field, value, _ = WINDOW[name]
    rng = np.random.default_rng(6)
    parts = [ordinary(rng, w, arrow) for w in range(1, 30)]
    L = value if field == "len" else 200
    beg = value if field == "beg" else 1000
    if field == "qv":
        tail = f"30/{beg}_{beg + L} RQ=0.{value}"
    else:
        tail = f"30/{beg}_{beg + L} " + (f"SN={_snr(rng)}" if arrow else "RQ=0.851")
    parts.append(entry(tail, _seq(rng, L, arrow)))
    parts += [ordinary(rng, w, arrow) for w in range(31, 60)]
    return b"".join(parts)


# ---- well_jumps ---------------------------------------------------------------------------------------

BIG = 255 * (1 << 20)
WELL_DELTAS = [254, 255, 256, 510, BIG - 255, BIG, BIG + 1]
WELL_DELTA_OVER_CAP = BIG + 255          # 2^20 + 1 bytes of 0xff: more than the run count holds
FIRST_WELLS = [0, 255, 256]
WELL_DROPS = [1, 2, 300]


def well_jumps(kind: str, case: str) -> bytes:
    """kind 'fasta' / 'arrow' / 'quiva'; case 'deltas' (WELL_DELTAS between ordinary entries),
    'over_cap' (one WELL_DELTA_OVER_CAP), 'first<w>' (first well w), 'drop<d>' (the wells drop by d
    once, mid-file)"""
    rng = np.random.default_rng(7)
    n = 3 * len(WELL_DELTAS) + 2
    wells = list(np.cumsum(rng.integers(0, 3, size=n)) + 1000)
    if case == "deltas":
        wells = [1]
        for k in range(n - 1):
            wells.append(wells[-1] + (WELL_DELTAS[k // 3] if k % 3 == 1 else int(rng.integers(0, 3))))
    elif case == "over_cap":
        wells[n // 2:] = [w + WELL_DELTA_OVER_CAP for w in wells[n // 2:]]
    elif case.startswith("first"):
        w0 = int(case[5:])
        wells = [w0 + int(x) for x in np.cumsum([0] + list(rng.integers(0, 3, size=n - 1)))]
    elif case.startswith("drop"):
        d = int(case[4:])
        k = n // 2
        wells[k] = wells[k - 1] - d
        for j in range(k + 1, n):
            wells[j] = wells[k] + (j - k)
    if kind == "quiva":
        text = synth.make_quiva(8, [int(x) for x in rng.integers(20, 400, size=n)], movie=MOVIE)
        lines = text.split(b"\n")
        for e in range(n):
            f = lines[6 * e].split(b"/")
            f[1] = str(wells[e]).encode()
            lines[6 * e] = b"/".join(f)
        return b"\n".join(lines)
    return b"".join(ordinary(rng, w, kind == "arrow") for w in wells)


WELL_CASES = ["deltas", "over_cap"] + [f"first{w}" for w in FIRST_WELLS] + [f"drop{d}" for d in WELL_DROPS]


# ---- zero_payload -------------------------------------------------------------------------------------

def zero_payload(kind: str, mbytes: float = 4.0) -> bytes:
    """kind 'fasta' (reads of all 'a', of all 'N', and reads with 'a'-runs of 40 ... 52 at every
    offset mod 4) or 'arrow' (reads of all '1'); a few ordinary reads between them"""
    rng = np.random.default_rng(9)
    arrow = kind == "arrow"
    parts, well, size = [], 0, 0
    runs = [(r, o) for r in range(40, 53) for o in range(4)]
    k = 0
    while size < mbytes * 1e6:
        well += 1
        if k % 5 == 4:
            p = ordinary(rng, well, arrow)
        elif not arrow and k % 5 == 3:
            r, o = runs[(k // 5) % len(runs)]
            head = _seq(rng, 64 + o)
            s = head + b"a" * r + _seq(rng, 64)
            p = entry(f"{well}/0_{len(s)} RQ=0.851", s)
        else:
            L = int(rng.integers(2000, 30000))
            ch = b"1" if arrow else (b"a" if k % 2 else b"N")
            tail = f"{well}/0_{L} " + (f"SN={_snr(rng)}" if arrow else "RQ=0.851")
            p = entry(tail, ch * L)
        parts.append(p)
        size += len(p)
        k += 1
    return b"".join(parts)


# ---- the candidate predicate, restated -----------------------------------------------------------------

def candidate_positions(img: bytes, arrow: bool) -> np.ndarray:
    """every offset >= first + 1 whose next 12 (.dexta) / 16 (.dexar) bytes pass DX_PRED_QVCAND /
    DX_PRED_ARCAND of dx_frame.cu.  For .dexar the byte prefilter also asks end < 2^27, so an entry
    with beg = 2^27 - 1 is a candidate in .dexta only."""
    plen = struct.unpack_from("<i", img, 2)[0]
    first = 6 + plen
    fb = 16 if arrow else 12
    a = np.frombuffer(img, dtype=np.uint8)
    m = len(a) - fb + 1
    if m <= first + 1:
        return np.zeros(0, dtype=np.int64)

    def u32(k):                                  # the little-endian word at every offset + k
        return (a[k:k + m].astype(np.uint32) | (a[k + 1:k + 1 + m].astype(np.uint32) << 8) |
                (a[k + 2:k + 2 + m].astype(np.uint32) << 16) | (a[k + 3:k + 3 + m].astype(np.uint32) << 24))

    beg, end = u32(0), u32(4)
    ok = (beg < CAND_MAX_BEG) & (end >= beg) & ((end - beg) <= CAND_MAX_LEN)
    if arrow:
        ok &= end < CAND_MAX_BEG                 # the byte prefilter of ARCAND: bytes 3 and 7 below 8
        for k in range(4):
            c = a[8 + 2 * k:8 + 2 * k + m].astype(np.uint32) | (a[9 + 2 * k:9 + 2 * k + m].astype(np.uint32) << 8)
            ok &= c <= CAND_MAX_SNR
    else:
        ok &= u32(8) < CAND_MAX_QV
    ok[: first + 1] = False
    return np.nonzero(ok)[0].astype(np.int64)


def tile_overflow(img: bytes, arrow: bool) -> bool:
    """True when some 16 KB tile holds more candidates than the 16 slots of k_pred_slots: the index
    then takes the exact two-pass kernels"""
    pos = candidate_positions(img, arrow)
    if len(pos) == 0:
        return False
    return int(np.bincount(pos // TILE_BYTES).max()) > TILE_SLOTS


def entry_fields(img: bytes, arrow: bool):
    """walk a native image as the reference's undexta does: [(field offset q, well, beg, end, aux)]"""
    plen = struct.unpack_from("<i", img, 2)[0]
    at, well, out = 6 + plen, 0, []
    fb = 16 if arrow else 12
    while at < len(img):
        while img[at] == 0xFF:
            well += 255
            at += 1
        well += img[at]
        at += 1
        beg, end = struct.unpack_from("<ii", img, at)
        aux = struct.unpack_from("<4H" if arrow else "<i", img, at + 8)
        out.append((at, well, beg, end, aux))
        rl = end - beg
        assert rl >= 0
        at += fb + (rl + 3) // 4
    assert at == len(img)
    return out


def fast_path_holds(img: bytes, arrow: bool) -> bool:
    """the device-planned chain of undexta_fast (dx_api.cpp) accepts every entry: each true entry's
    field offset is a candidate and its well-delta bytes hold at most FFRUN_CAP 0xff bytes (false
    candidates can only start in the last three bytes of such a run: beg < 2^27 needs a byte < 8)"""
    cand = set(candidate_positions(img, arrow).tolist())
    prev_end = 6 + struct.unpack_from("<i", img, 2)[0]
    for q, well, beg, end, aux in entry_fields(img, arrow):
        if q not in cand or (q - 1 - prev_end) > FFRUN_CAP:
            return False
        prev_end = q + (16 if arrow else 12) + (end - beg + 3) // 4
    return True


def expected_route(img: bytes, arrow: bool):
    """(index, chain) of a default-route decode of a native image at a width of 16 or more"""
    return (INDEX_TWO_PASS if tile_overflow(img, arrow) else INDEX_SLOTS,
            CHAIN_FAST if fast_path_holds(img, arrow) else CHAIN_GENERAL)


# ---- legacy_2bit ----------------------------------------------------------------------------------------

def _parse_text(text: bytes, arrow: bool):
    """the entries of a canonical .fasta / .arrow text: (prefix, [(well, beg, end, aux, seq)])"""
    out = []
    prefix = None
    for chunk in text.split(b">")[1:]:
        head, _, body = chunk.partition(b"\n")
        name, tail = head.split(b"/", 1)
        if prefix is None:
            prefix = b">" + name
        w, rest = tail.split(b"/", 1)
        be, _, more = rest.partition(b" ")
        b, e = be.split(b"_")
        if arrow:
            snr = [float(x) for x in more[3:].split(b",")]
            aux = [9999 if np.float32(s) > 99.99 else int(float(np.float32(s)) * 100.) & 0xFFFF for s in snr]
        else:
            aux = int(more[5:]) if more else 0
        out.append((int(w), int(b), int(e), aux, body.replace(b"\n", b"")))
    return prefix, out


def build_2bit(text: bytes, arrow: bool = False, flip: bool = False, old: bool = False) -> bytes:
    """a .dexta / .dexar image of a canonical text, written natively (must equal dexta's image byte
    for byte), with every 16/32-bit quantity in the other byte order (flip), or in the old 16-bit
    .dexta layout (old: key 0x33cc, beg/end/qv as uint16)"""
    assert not (arrow and old)
    prefix, ents = _parse_text(text, arrow)
    e = ">" if flip else "<"
    out = bytearray(struct.pack(e + "H", 0x33CC if old else 0x55AA) + struct.pack(e + "i", len(prefix)) + prefix)
    lwell = 0
    for well, beg, end, aux, seq in ents:
        out += _well_bytes(well - lwell)
        lwell = well
        if old:
            out += struct.pack(e + "HHH", beg, end, aux)
        elif arrow:
            out += struct.pack(e + "ii4H", beg, end, *aux)
        else:
            out += struct.pack(e + "iii", beg, end, aux)
        out += pack2bit(seq, arrow)
    return bytes(out)


def legacy_text(seed: int, arrow: bool = False, n: int = 80) -> bytes:
    """a canonical text whose beg / end / qv fit 16 bits, with a few lengths around 4 and wells that
    jump over 255"""
    rng = np.random.default_rng(seed)
    lens = [0, 1, 2, 3, 4, 5, 7, 8, 9] + [int(x) for x in rng.integers(1, 5000, size=n)]
    wells = np.cumsum(rng.integers(0, 300, size=len(lens)))
    parts = []
    for i, L in enumerate(lens):
        beg = int(rng.integers(0, 60000))
        tail = f"{wells[i]}/{beg}_{beg + L} " + (f"SN={_snr(rng)}" if arrow else f"RQ=0.{int(rng.integers(0, 65536))}")
        parts.append(entry(tail, _seq(rng, L, arrow), width=int(rng.integers(16, 120))))
    return b"".join(parts)
