"""Crafted .quiva files for pass 2 of the QV coder (dx_qv_encode.cu: k_qv_code<MODE> as k_qv_emit /
k_qv_size, the bit writer of dx_bits.cuh, k_qv_compact and the entry-offset scan), and a plain numpy
restatement of the encoder's accounting.

  stream_model(line, ...)   per stream: the item lengths of pack_tables (dx_api.cpp), the lossy
                            masks, the total bits T, the start of the last item plast, the words
                            written max(ceil(T/32), (plast+47)>>5) (QV.c:436-442) and whether they fit
                            the stream's room of rlen+9 bytes in the scratch image;
  tag_model(del, delchar)   kept tags and their (kept+3)>>2 bytes;
  plain_rows(...)           for a plain stream at a line skew: every row's 32 lane bit counts (a lane
                            is one 16-byte chunk, LineWalk), the writer it takes (finish_wide, finish,
                            the escaped path) and the stage fill before each reserve;
  tag_rows(...)             the same stage accounting for the 2-bit tag stream.

Families (each a list of (label, text); the docstrings name the decision they sit on):

  room     one stream per file exactly at its room (floor((rlen+9)/4) words) or one word over
  rows     lane bits 31 / 32 / 33, escapes in lane 0, lane 31 and partial chunks, every skew
  stage    the stage's reserve at nst + need + 1 == 512 and 513, the largest row after a flush,
           tag streams of more than 8192 kept tags, every start address mod 4
  tags     kept counts mod 4, no kept tag, no delChar, every tag letter
  pad      the four kinds of last item on both sides of the look-ahead word
  counts   16 383 ... 40 000 entries (the three entry-offset scans)
  long     entries of 2^20 - 1 ... 2^24 - 1 positions; one of 2^24 (refused by the library)

The files whose claims depend on exact code lengths pin the file's ins and del histograms: crafted
lines take their symbols from a fixed multiset and the rest of the file takes the remainder, so the
coding does not depend on what the crafted lines hold.  Each generator builds its file twice (the
second time with the coding of the first) and checks that the coding did not move.

Line buffers are 16-byte aligned (a line's skew is its file offset mod 16).  TEST INFRASTRUCTURE
ONLY."""
from __future__ import annotations

import numpy as np

from dextractor_b200 import synth
from tests import qv_shapes as Q
from tests import scan_shapes as S

# dx_qv_encode.cu
STAGE_WORDS = 512                    # kStageWords: per-warp stage of WarpBits
ONE_CTA_SCAN_BELOW = 16384           # entry_offsets(): k_qv_offsets below, k_qv_entry_total + scan from
CHAIN_TILE = 8192                    # dx_frame.cu kChainTile: k_tile_scan up to 2 tiles, k_chain_scan above


def room(rlen: int) -> int:
    """scratch_room(): bytes a stream of rlen symbols may take in the scratch image"""
    return rlen + 9


# dx_frame.cu / dx_api.cpp
CAND_MAX_LEN = 1 << 20               # kCandMaxLen: longer entries are never header candidates
MAX_RLEN = 1 << 24                   # k_qv_entries refuses rlen >= 2^24 with DX_E_TOOLONG

ACGT = S.ACGT
DELC = S.DELC                        # '2': the del run character of every file here
INS_SYMS = np.arange(40, 82, 2)      # 21 even values: lossy coding keeps them apart
DEL_SYMS = np.arange(60, 81)         # 21 non-run del values


# ---- the restatement --------------------------------------------------------------------------------

def item_tables(coding) -> dict:
    """pack_tables (dx_api.cpp): per table k, (item length incl. an escaped symbol's 8-bit literal,
    escape flag).  Run tables: the code only; an escaped run adds a 16-bit literal."""
    out = {}
    for k in range(6):
        s = coding.tab[k]
        lens = np.array(s.lens[:], dtype=np.int64)
        bits = np.array(s.bits[:], dtype=np.int64)
        isrun = k in (1, 5)
        esc = (isrun or s.type == 2) & (lens > 0) & (bits == bits[255]) & (lens == lens[255])
        L = np.where(lens > 16, 0, lens & 31)
        if not isrun:
            L = L + 8 * esc
        out[k] = (L, esc)
    return out


def lossy_line(line: np.ndarray, kind: int, lossy: bool) -> np.ndarray:
    if not lossy or kind not in (2, 3):
        return line
    return line & (0xFE if kind == 2 else 0xFC)


def run_items(line: np.ndarray, rc: int):
    """Encode_Run's items (QV.c:448-506): (run before each non-run symbol, the symbol), and the
    length of a trailing run (-1 if the line ends in a non-run symbol)"""
    nz = np.flatnonzero(line != rc)
    prev = np.concatenate([[-1], nz[:-1]])
    runs = nz - prev - 1
    last = nz[-1] if len(nz) else -1
    trail = len(line) - 1 - last if last < len(line) - 1 else -1
    return runs, line[nz], trail


def stream_model(line, kind: int, coding, tabs: dict, lossy: bool = False) -> dict:
    """one stream (kind 0 del, 2 ins, 3 mrg, 4 sub) as k_qv_code<MODE> accounts for it"""
    line = lossy_line(np.asarray(line, dtype=np.uint8), kind, lossy)
    rlen = len(line)
    if rlen == 0:
        return dict(T=0, plast=0, words=0, bytes=0, fits=True, rlen=0, last="none", pad=False)
    rc = coding.delchar if kind == 0 else coding.subchar if kind == 4 else -1
    L, esc = tabs[kind]
    if rc < 0:
        T = int(L[line].sum())
        x = int(line[-1])
        last = "esc_sym" if esc[x] else "sym"
        plast = T - (8 if esc[x] else int(L[x]))
    else:
        R, Resc = tabs[1 if kind == 0 else 5]
        runs, syms, trail = run_items(line, rc)
        rb = np.minimum(runs, 255)
        T = int((R[rb] + 16 * Resc[rb]).sum() + L[syms].sum())
        if trail >= 0:
            t = min(trail, 255)
            T += int(R[t]) + 16 * int(Resc[t])
            last = "esc_run" if Resc[t] else "run"
            plast = T - (16 if Resc[t] else int(R[t]))
        else:
            x = int(syms[-1])
            last = "esc_sym" if esc[x] else "sym"
            plast = T - (8 if esc[x] else int(L[x]))
    full, want = (T + 31) >> 5, (plast + 47) >> 5
    words = max(full, want)
    return dict(T=T, plast=plast, words=words, bytes=4 * words, fits=4 * words <= room(rlen), rlen=rlen,
                last=last, pad=want > full, full=full)


def tag_model(dele, delchar: int) -> dict:
    kept = len(dele) if delchar < 0 else int(np.count_nonzero(np.asarray(dele) != delchar))
    return dict(kept=kept, bytes=(kept + 3) >> 2)


def _lane_sums(vals: np.ndarray, skew: int) -> np.ndarray:
    """per-position values -> per-chunk sums (chunk c holds positions 16c - skew ... 16c - skew + 15)"""
    padded = np.concatenate([np.zeros(skew, vals.dtype), vals])
    padded = np.concatenate([padded, np.zeros((-len(padded)) % 16, vals.dtype)])
    return padded.reshape(-1, 16).sum(axis=1)


def _stage(row_bits, limit: int):
    """WarpBits::reserve over the rows: the stage fill before each reserve and whether it flushes,
    and for a flush whether it passes the room check (flushed + nst)*4 <= limit"""
    nst = cbits = flushed = 0
    out = []
    for row in row_bits:
        row = int(row)
        need = (cbits + row + 31) >> 5
        fill = nst + need + 1
        flush = fill > STAGE_WORDS
        ok = True
        if flush:
            ok = (flushed + nst) * 4 <= limit
            flushed += nst
            nst = 0
        pos = nst * 32 + cbits + row
        out.append(dict(row=row, fill=fill, flush=flush, flush_ok=ok, nst_after=pos >> 5))
        nst, cbits = pos >> 5, pos & 31
    return out


def plain_rows(line, kind: int, tabs: dict, skew: int, lossy: bool = False):
    """rows of a plain stream: [dict(lanes=32 bit counts, esc=lanes with an escaped item, wide,
    fill, flush, flush_ok)]"""
    line = lossy_line(np.asarray(line, dtype=np.uint8), kind, lossy)
    L, esc = tabs[kind]
    bits = _lane_sums(L[line], skew)
    escs = _lane_sums(esc[line].astype(np.int64), skew)
    nrow = (len(bits) + 31) // 32
    pad = nrow * 32 - len(bits)
    bits = np.concatenate([bits, np.zeros(pad, np.int64)]).reshape(nrow, 32)
    escs = np.concatenate([escs, np.zeros(pad, np.int64)]).reshape(nrow, 32)
    st = _stage(bits.sum(axis=1), room(len(line)))
    return [dict(lanes=bits[r], esc=np.flatnonzero(escs[r]), wide=bool((bits[r] >= 32).all()), **st[r])
            for r in range(nrow)]


def tag_rows(dele, tag_skew: int, delchar: int):
    """rows of the tag stream (code_tags): 2 bits per kept tag"""
    dele = np.asarray(dele)
    kept = np.ones(len(dele), np.int64) if delchar < 0 else (dele != delchar).astype(np.int64)
    cnt = _lane_sums(kept, tag_skew)
    nrow = (len(cnt) + 31) // 32
    rows = np.concatenate([cnt, np.zeros(nrow * 32 - len(cnt), np.int64)]).reshape(nrow, 32).sum(axis=1)
    return _stage(2 * rows, 1 << 62)


def codable(orc, text: bytes, lossy: bool) -> bool:
    """dx_qv_make_coding's rule: every table it builds needs two distinct symbols, counted after the
    lossy merges and without the run characters; the library refuses other files (DX_E_CODING)"""
    st = orc.qv_scan(text)
    h = {k: np.array(getattr(st, k)[:], dtype=np.uint64) for k in ("del_", "ins", "mrg", "sub")}
    subchar = st.subchar
    if subchar >= 0 and (st.totchar < 200000 or h["sub"][subchar] < 0.5 * st.totchar):
        subchar = -1
    if lossy:
        h["ins"] = h["ins"].reshape(-1, 2).sum(axis=1)
        h["mrg"] = h["mrg"].reshape(-1, 4).sum(axis=1)
    if st.delchar >= 0:
        h["del_"][st.delchar] = 0
    if subchar >= 0:
        h["sub"][subchar] = 0
    return all(np.count_nonzero(v) >= 2 for v in h.values())


def coding(orc, text, lossy=False):
    return orc.qv_create(orc.qv_scan(text), lossy)


def entries(text: bytes) -> dict:
    p = S.parse(text)
    a = p["a"]
    lines = [[a[p["line"][e, k]: p["line"][e, k] + p["rlen"][e]] for k in range(5)] for e in range(p["n"])]
    return dict(p=p, lines=lines)


def well_bytes(wells: np.ndarray) -> np.ndarray:
    d = np.diff(np.concatenate([[0], wells]))
    return 1 + np.where(d >= 255, d // 255, 0)


def file_model(orc, text: bytes, lossy: bool = False, c=None) -> dict:
    """d_bytes of dx_qv_encode (header, del, tag, ins, mrg, sub per entry) and every stream's model"""
    c = c if c is not None else coding(orc, text, lossy)
    tabs = item_tables(c)
    E = entries(text)
    n = E["p"]["n"]
    nb = np.zeros((n, 6), np.int64)
    nb[:, 0] = well_bytes(E["p"]["well"]) + 12
    streams = {}
    for e, ls in enumerate(E["lines"]):
        for k in (0, 2, 3, 4):
            m = stream_model(ls[k], k, c, tabs, lossy)
            streams[e, k] = m
            nb[e, 1 + k] = m["bytes"]
        nb[e, 2] = tag_model(ls[0], c.delchar)["bytes"]
    return dict(coding=c, tabs=tabs, bytes=nb, streams=streams, entries=E)


def oracle_stream_bytes(orc, c, line, kind: int, lossy: bool = False) -> int:
    """the stream's length as the oracle's encoder writes it"""
    line = lossy_line(np.asarray(line, dtype=np.uint8), kind, lossy)
    if len(line) == 0:
        return 0
    rc = c.delchar if kind == 0 else c.subchar if kind == 4 else -1
    run = c.tab[1 if kind == 0 else 5] if rc >= 0 else None
    return len(orc.encode_stream(c.tab[kind], run, rc, line.tobytes()))


def check_against_oracle(orc, text: bytes, lossy: bool = False, per_stream: bool = True) -> dict:
    """the model's byte counts against orc.encode_stream (every stream) and the image's entry offsets"""
    fm = file_model(orc, text, lossy)
    c = fm["coding"]
    if per_stream:
        for (e, k), m in fm["streams"].items():
            got = oracle_stream_bytes(orc, c, fm["entries"]["lines"][e][k], k, lossy)
            assert got == m["bytes"], (e, k, got, m)
    enc = orc.dexqv(text, lossy=lossy)
    n = fm["entries"]["p"]["n"]
    offs = orc.dexqv_offsets(enc, n)
    tot = fm["bytes"].sum(axis=1)
    assert np.array_equal(np.diff(offs), tot), np.flatnonzero(np.diff(offs) != tot)[:5]
    assert offs[-1] == len(enc)
    fm["enc"], fm["offs"] = enc, offs
    return fm


# ---- pinned histograms and exact fills ---------------------------------------------------------------

def fib_counts(total: int, syms: np.ndarray) -> dict:
    """Fibonacci-shaped counts over the 21 symbols (a Huffman chain deeper than 16: the tail is
    escaped), scaled to `total`; the most common symbol takes the rounding"""
    fib = [1, 1]
    while len(fib) < len(syms):
        fib.append(fib[-1] + fib[-2])
    fib = np.array(fib[::-1], dtype=np.int64)
    cnt = fib * (total // int(fib.sum()))
    cnt[0] += total - int(cnt.sum())
    return {int(s): int(c) for s, c in zip(syms, cnt)}


def fill(n: int, target: int, length: dict, avail: dict, rng, exclude=()):
    """n symbols out of `avail` (symbol -> count) whose item lengths sum to exactly `target`, or None"""
    by = {}
    for s, c in avail.items():
        if c > 0 and length.get(s, 0) > 0 and s not in exclude:
            by.setdefault(length[s], []).append(s)
    Ls = sorted(by, reverse=True)
    cap = {L: sum(avail[s] for s in by[L]) for L in Ls}

    def bound(k, ls, hi):
        tot = 0
        for L in (ls if hi else ls[::-1]):
            t = min(k, cap[L])
            tot += t * L
            k -= t
            if k == 0:
                return tot
        return None

    take, k, t = {}, n, target
    for i, L in enumerate(Ls):
        rest = Ls[i + 1:]
        for c in range(min(cap[L], k, t // L), -1, -1):
            k2, t2 = k - c, t - c * L
            if k2 == 0:
                ok = t2 == 0
            else:
                lo, hi = bound(k2, rest, False), bound(k2, rest, True)
                ok = lo is not None and lo <= t2 <= hi
            if ok:
                take[L] = c
                k, t = k2, t2
                break
        if k == 0:
            break
    if k or t:
        return None
    out = []
    for L, c in take.items():
        for s in by[L]:
            u = min(c, avail[s])
            out += [s] * u
            avail[s] -= u
            c -= u
    out = np.array(out, dtype=np.uint8)
    rng.shuffle(out)
    return out


def take(n: int, avail: dict, rng, only=None) -> np.ndarray:
    """n symbols drawn from `avail` in proportion to what is left (optionally only from `only`)"""
    syms = [s for s in avail if avail[s] > 0 and (only is None or s in only)]
    cnt = np.array([avail[s] for s in syms], dtype=np.float64)
    pick = rng.choice(len(syms), size=n, p=cnt / cnt.sum())
    got = np.bincount(pick, minlength=len(syms))
    for j, s in enumerate(syms):                      # never more than there is
        while got[j] > avail[s]:
            got[j] -= 1
            k = int(np.argmax([avail[t] - got[i] for i, t in enumerate(syms)]))
            got[k] += 1
    out = np.repeat(np.array(syms, dtype=np.uint8), got)
    for j, s in enumerate(syms):
        avail[s] -= int(got[j])
    rng.shuffle(out)
    return out


def _expand(avail: dict, rng) -> np.ndarray:
    out = np.repeat(np.array(list(avail), dtype=np.uint8), list(avail.values()))
    rng.shuffle(out)
    return out


def _run_mask(rng, L: int) -> np.ndarray:
    """non-run positions of a background del line: runs of 0..3 DELC in front of each symbol (at
    least one in front of the first: the first tag of a file, 'n', fixes delChar)"""
    m = np.zeros(L, dtype=bool)
    k = 1
    gaps = rng.integers(0, 4, size=L)
    for g in gaps:
        k += int(g)
        if k >= L:
            break
        m[k] = True
        k += 1
    return m


class Craft:
    """one crafted entry of a pinned file: ins(c, avail, rng) and / or dele(c, avail, rng) make its
    ins / del line (the del line's DELC positions may not depend on c); skew = (line, s)"""

    def __init__(self, rlen, ins=None, dele=None, del_syms=0, skew=None, label=""):
        self.rlen, self.ins, self.dele, self.del_syms, self.skew, self.label = rlen, ins, dele, del_syms, skew, label


def pinned_text(seed: int, layout, c) -> tuple:
    """layout: background rlens (int) and Craft entries in file order -> (text, {label: entry})"""
    rr = np.random.default_rng(seed)
    masks = [None if isinstance(x, Craft) and x.dele else _run_mask(rr, x if isinstance(x, int) else x.rlen)
             for x in layout]
    rl = [x if isinstance(x, int) else x.rlen for x in layout]
    ins_av = fib_counts(sum(rl), INS_SYMS)
    del_av = fib_counts(sum(int(m.sum()) for m in masks if m is not None) +
                        sum(x.del_syms for x in layout if isinstance(x, Craft) and x.dele), DEL_SYMS)
    rng = np.random.default_rng(seed + 1)
    made = {}
    for e, x in enumerate(layout):
        if isinstance(x, Craft):
            ins = x.ins(c, ins_av, rng) if x.ins else None
            dele = x.dele(c, del_av, rng) if x.dele else None
            assert ins is None or len(ins) == x.rlen
            assert dele is None or (len(dele) == x.rlen and int(np.count_nonzero(dele != DELC)) == x.del_syms)
            made[e] = (ins, dele)
    ins_rest, del_rest = _expand(ins_av, rng), _expand(del_av, rng)
    assert len(ins_rest) == sum(rl) - sum(len(v[0]) for v in made.values() if v[0] is not None)
    noise = np.random.default_rng(seed + 2)
    q = S.Quiva()
    labels = {}
    ia = da = 0
    for e, x in enumerate(layout):
        L = rl[e]
        ins, dele = made.get(e, (None, None))
        if ins is None:
            ins = ins_rest[ia:ia + L]
            ia += L
        if dele is None:
            m = masks[e]
            dele = np.full(L, DELC, dtype=np.uint8)
            k = int(m.sum())
            dele[m] = del_rest[da:da + k]
            da += k
        tag = S._tags(dele, rng=noise)
        if e == 0:
            assert dele[0] == DELC                        # the first tag fixes delChar
        q.add(dele, tag, ins, noise.integers(33, 65, size=L).astype(np.uint8),
              noise.integers(33, 49, size=L).astype(np.uint8), skew=x.skew if isinstance(x, Craft) else None)
        if isinstance(x, Craft):
            labels[x.label] = e
    assert ia == len(ins_rest) and da == len(del_rest)
    return q.text(), labels


def same_coding(a, b) -> bool:
    return a.delchar == b.delchar and all(
        a.tab[k].type == b.tab[k].type and list(a.tab[k].lens) == list(b.tab[k].lens)
        and list(a.tab[k].bits) == list(b.tab[k].bits) for k in (0, 1, 2))


def pinned(orc, seed: int, layout):
    """build twice: the crafted lines see the coding of the file they end up in"""
    t0, _ = pinned_text(seed, layout, None)
    c0 = coding(orc, t0)
    t1, labels = pinned_text(seed, layout, c0)
    c1 = coding(orc, t1)
    assert same_coding(c0, c1), "the crafted lines moved the coding"
    return t1, labels, c1


def _len_of(c, kind: int) -> dict:
    L, _ = item_tables(c)[kind]
    return {int(s): int(L[s]) for s in range(256)}


def _esc_of(c, kind: int) -> set:
    _, esc = item_tables(c)[kind]
    return {int(s) for s in np.flatnonzero(esc) if s != 255}


def _exact(c, kind, n, target, avail, rng, exclude=(), only=None):
    """n symbols of stream `kind` with item bits summing to target (any n symbols while c is None)"""
    if c is None:
        return take(n, avail, rng, only)
    length = _r0(c, kind)
    if only is not None:
        length = {s: (v if s in only else 0) for s, v in length.items()}
    got = fill(n, target, length, avail, rng, exclude)
    assert got is not None, (kind, n, target)
    return got


def _one(c, kind, avail, want, rng):
    """one symbol: want = 'esc' (an escaped one) or an item length (the nearest non-escaped one)"""
    if c is None:
        return take(1, avail, rng)
    length, esc = _len_of(c, kind), _esc_of(c, kind)
    cand = [s for s in avail if avail[s] > 0 and length.get(s, 0) > 0 and ((s in esc) == (want == "esc"))]
    if want != "esc":
        cand.sort(key=lambda s: (abs(length[s] - want), s))
    s = cand[0]
    avail[s] -= 1
    return np.array([s], dtype=np.uint8)


# ---- room ------------------------------------------------------------------------------------------

ROOM_SMALL = (8, 9, 10, 11)
ROOM_LARGE = (2100, 2101, 2102, 2103)        # > 2048: the stage has flushed before the final flush


def _room_line(kind, R, over, lastlen=5):
    """R symbols whose stream takes floor((R+9)/4) words (+1 when over), ending in a plain symbol"""
    W = room(R) // 4 + (1 if over else 0)

    def make(c, avail, rng):
        if c is None:
            return take(R, avail, rng)
        last = _one(c, kind, avail, lastlen, rng)
        tabs = item_tables(c)
        pl = int(tabs[kind][0][last[0]])                  # the last item: the symbol's code
        ll = pl + (int(tabs[1][0][0]) if kind == 0 else 0)
        Ts = range(32 * W, 32 * (W - 1), -1) if not over else range(32 * (W - 1) + 1, 32 * W + 1)
        for T in Ts:
            if max((T + 31) >> 5, (T - pl + 47) >> 5) != W:
                continue
            trial = dict(avail)
            got = fill(R - 1, T - ll, _r0(c, kind), trial, rng)
            if got is not None:
                avail.update(trial)
                return np.concatenate([got, last])
        raise AssertionError(("no fill", kind, R, over))
    return make


def _r0(c, kind):
    """item lengths of stream `kind`; del items without a run carry the run code of 0 in front"""
    length = _len_of(c, kind)
    if kind == 0:
        r0 = int(item_tables(c)[1][0][0])
        length = {s: (v + r0 if v else 0) for s, v in length.items()}
    return length


def _bg(n, L=1500):
    return [L] * n


def room_file(kind, R, over):
    k = "ins" if kind == 2 else "del"
    cr = Craft(R, label="boundary",
               **({"ins": _room_line(2, R, over)} if kind == 2 else
                  {"dele": _room_line(0, R, over), "del_syms": R}))
    return _bg(100) + [cr] + _bg(100), f"{k}_{R}_{'over' if over else 'fit'}"


def room_midflush():
    """ins: two full rows (~300 + ~212 words) then a short one; rlen 1100 has room for 277 words, so the
    reserve that flushes the first rows already fails the room check"""
    R = 1100

    def make(c, avail, rng):
        if c is None:
            return take(R, avail, rng)
        a = _exact(c, 2, 512, 9600, avail, rng)
        b = _exact(c, 2, 512, 6784, avail, rng)
        d = _exact(c, 2, R - 1024, 4 * (R - 1024), avail, rng)
        return np.concatenate([a, b, d])
    return [2000] * 450 + [Craft(R, ins=make, skew=(2, 0), label="boundary")]


def shape_room(orc):
    files = []
    seed = 100
    for kind in (2, 0):
        for R in ROOM_SMALL + ROOM_LARGE:
            for over in (False, True):
                layout, label = room_file(kind, R, over)
                text, _, _ = pinned(orc, seed, layout)
                files.append((label, text))
                seed += 1
    text, _, _ = pinned(orc, 199, room_midflush())
    files.append(("ins_1100_midflush", text))
    return files


def room_claims(orc, label, text):
    """the file's one boundary stream sits where its label says; every other stream fits with room
    to spare"""
    fm = file_model(orc, text)
    near = [(e, k, m) for (e, k), m in fm["streams"].items() if m["rlen"] and m["words"] >= room(m["rlen"]) // 4]
    assert len(near) == 1, (label, [(e, k, m["words"], m["rlen"]) for e, k, m in near])
    e, k, m = near[0]
    kind = {"ins": 2, "del": 0}[label.split("_")[0]]
    assert k == kind, (label, k)
    W = room(m["rlen"]) // 4
    if label.endswith("midflush"):
        rows = plain_rows(fm["entries"]["lines"][e][k], k, fm["tabs"], int(fm["entries"]["p"]["line"][e, k] % 16))
        first_bad = next(r for r in rows if not r["flush_ok"])
        assert first_bad["flush"], label                  # caught by a reserve, before the final flush
        return dict(stream=(e, k), words=m["words"], room_words=W, fits=False)
    R = int(label.split("_")[1])
    assert m["rlen"] == R and m["rlen"] % 4 == R % 4
    over = label.endswith("over")
    assert m["words"] == W + over and m["fits"] == (not over), (label, m, W)
    if R > 2048:
        assert m["words"] > STAGE_WORDS - 4                   # the stage flushed before the final decision
    return dict(stream=(e, k), words=m["words"], room_words=W, fits=not over)


# ---- rows --------------------------------------------------------------------------------------------

def _lanes(c, avail, rng, targets, esc_lanes=()):
    """one skew-0 row of ins: lane i = 16 symbols of targets[i] bits; escaped symbols only in
    esc_lanes (one each)"""
    if c is None:
        return take(16 * len(targets), avail, rng)
    esc = _esc_of(c, 2)
    out = []
    for i, t in enumerate(targets):
        if i in esc_lanes:
            x = _one(c, 2, avail, "esc", rng)
            out += [_exact(c, 2, 15, t - int(item_tables(c)[2][0][x[0]]), avail, rng, exclude=esc), x]
        else:
            out.append(_exact(c, 2, 16, t, avail, rng, exclude=esc))
    return np.concatenate(out)


ROW_DESIGNS = {                 # lane bits of the crafted rows (lane 7 off the others)
    "wide_one_32": [33] * 7 + [32] + [33] * 24,
    "finish_one_31": [33] * 7 + [31] + [33] * 24,
    "all_32": [32] * 32,
    "all_31": [31] * 32,
    "all_33": [33] * 32,
}


def _row_line(c, avail, rng):
    rows = [_lanes(c, avail, rng, t) for t in ROW_DESIGNS.values()]
    rows.append(_lanes(c, avail, rng, [40] * 32, esc_lanes=(0,)))
    rows.append(_lanes(c, avail, rng, [40] * 32, esc_lanes=(31,)))
    return np.concatenate(rows)


def _partial_esc(where):
    """skew 5 (the first chunk holds 11 positions): the row's only escape in the first chunk, or in
    the line's last chunk (8 positions)"""
    R = 700 if where == "first" else 512 + 40 + 5

    def make(c, avail, rng):
        if c is None:
            return take(R, avail, rng)
        esc = _esc_of(c, 2)
        x = _one(c, 2, avail, "esc", rng)
        rest = _exact(c, 2, R - 1, 4 * (R - 1), avail, rng, exclude=esc)
        at = 3 if where == "first" else R - 2
        return np.concatenate([rest[:at], x, rest[at:]])
    return Craft(R, ins=make, skew=(2, 5), label=f"esc_{where}_chunk")


def _skew_sweep():
    """ins lines at every skew, ending at 512k - 1, 512k, 512k + 1 (skew + rlen)"""
    out = []
    for s in range(16):
        for k, d in ((1, -1), (2, 0), (1, 1)):
            R = 512 * k + d - s + (512 if s % 3 == 0 else 0)
            out.append(Craft(R, ins=lambda c, av, rng, R=R: take(R, av, rng), skew=(2, s),
                             label=f"skew_{s}_{d:+d}"))
    return out


def shape_rows(orc):
    """fixed2: every ins symbol coded in 2 bits, lossy or not, so every full row is 32 bits per
    lane, word aligned; crafted: the rows of ROW_DESIGNS and single escapes in lane 0,
    lane 31, the first and the last (partial) chunk; the skew sweep"""
    lengths = [512 * 4 + d for d in (-1, 0, 1)] * 4 + [16384, 9000, 1]
    alpha = 40 + 4 * np.arange(4)               # 4 apart: the lossy merges keep all four distinct

    def hook(i, st):
        r = np.random.default_rng(902000 + i)
        st[2][:] = Q._uniform(r, len(st[2]), alpha)
        st[3][:] = Q._uniform(r, len(st[3]), alpha[::-1])
    fixed2 = synth.make_quiva(902, lengths, stream_hook=hook)
    layout = [1500] * 100
    layout.insert(3, Craft(512 * 7, ins=_row_line, skew=(2, 0), label="rows"))
    layout.insert(10, _partial_esc("first"))
    layout.insert(20, _partial_esc("last"))
    layout[30:30] = _skew_sweep()
    text, _, _ = pinned(orc, 300, layout)
    return [("fixed2", fixed2), ("crafted", text)]


def rows_claims(orc, label, text):
    fm = file_model(orc, text)
    E, tabs = fm["entries"], fm["tabs"]
    seen = set()
    if label == "fixed2":
        L = tabs[2][0]
        assert {int(L[s]) for s in set(np.concatenate([ls[2] for ls in E["lines"]]).tolist())} == {2}
        for e, ls in enumerate(E["lines"]):
            for r in plain_rows(ls[2], 2, tabs, int(E["p"]["line"][e, 2] % 16)):
                if (r["lanes"] == 32).all():
                    assert r["wide"] and r["row"] % 32 == 0
                    seen.add("all_32_aligned")
        assert seen, label
        return seen
    skews, ends = set(), set()
    for e, ls in enumerate(E["lines"]):
        sk = int(E["p"]["line"][e, 2] % 16)
        skews.add(sk)
        ends.add((sk + len(ls[2])) % 512)
        rows = plain_rows(ls[2], 2, tabs, sk)
        for j, r in enumerate(rows):
            ln = r["lanes"]
            if (ln >= 32).all() and ln.min() == 32 and (ln > 32).any():
                seen.add("wide_one_32")
            if ln.min() == 31 and (np.sort(ln)[1:] >= 32).all():
                seen.add("finish_one_31")
            for v in (31, 32, 33):
                if (ln == v).all():
                    seen.add(f"all_{v}")
            if list(r["esc"]) == [0]:
                seen.add("esc_lane0")
            if list(r["esc"]) == [31]:
                seen.add("esc_lane31")
            if len(r["esc"]) == 1 and sk and j == 0 and r["esc"][0] == 0:
                seen.add("esc_first_partial_chunk")
            nch = (sk + len(ls[2]) + 15) // 16
            if len(r["esc"]) == 1 and j == len(rows) - 1 and 32 * j + r["esc"][0] == nch - 1 \
                    and (sk + len(ls[2])) % 16:
                seen.add("esc_last_partial_chunk")
    want = {"wide_one_32", "finish_one_31", "all_31", "all_32", "all_33", "esc_lane0", "esc_lane31",
            "esc_first_partial_chunk", "esc_last_partial_chunk"}
    assert want <= seen, want - seen
    assert skews == set(range(16)), skews
    assert {511, 0, 1} <= ends, ends
    return seen


# ---- stage -------------------------------------------------------------------------------------------

def _stage_line(final_fill):
    """skew-0 ins rows of 3840 bits until 480 words are staged, then a row that brings the reserve
    to final_fill (512: no flush, 513: flush); after the flush a row of escaped symbols only (the
    largest row the coding has: 384 words when the escape code has 16 bits)"""
    R = 512 * 6

    def make(c, avail, rng):
        if c is None:
            return take(R, avail, rng)
        esc = _esc_of(c, 2)
        rows = [_exact(c, 2, 512, 3840, avail, rng, exclude=esc) for _ in range(4)]     # 4 x 120 words
        need = final_fill - 1 - 480
        rows.append(_exact(c, 2, 512, 32 * need, avail, rng, exclude=esc))
        if final_fill == STAGE_WORDS:
            rows.append(_exact(c, 2, 512, 2048, avail, rng, exclude=esc))
        else:
            rows.append(_exact(c, 2, 512, 512 * int(item_tables(c)[2][0][min(esc)]), avail, rng, only=esc))
        return np.concatenate(rows)
    return Craft(R, ins=make, skew=(2, 0), label=f"stage_{final_fill}")


def shape_stage(orc):
    """ins (the pool is large enough for a row of 512 escaped symbols) and the tag streams of
    TAG_STAGE in a file without delChar"""
    layout = [20000] * 75 + [_stage_line(512), _stage_line(513)] + [20000] * 5
    text, _, _ = pinned(orc, 400, layout)
    return [("ins", text), ("tags", tag_file_no_delchar())]


TAG_STAGE = ((8170, 0), (8180, 0), (9000, 1), (9000, 2), (9000, 3), (17000, 0), (8192, 0), (8193, 2))


def tag_file_no_delchar():
    """no 'n' / 'N' tag: delChar -1 (every tag is kept, code_tags' MODE 0 shortcut); tag lines of
    TAG_STAGE (rlen, skew): 8170 at skew 0 ends with the reserve at 512, 8180 flushes at 513"""
    rng = np.random.default_rng(500)
    q = S.Quiva()
    letters = np.frombuffer(b"acgtACGT", dtype=np.uint8)
    for L, s in TAG_STAGE + ((40, 1), (3, 3)):
        q.add(rng.integers(60, 80, size=L).astype(np.uint8), letters[rng.integers(0, 8, size=L)],
              rng.integers(33, 60, size=L).astype(np.uint8), rng.integers(33, 70, size=L).astype(np.uint8),
              rng.integers(33, 45, size=L).astype(np.uint8), skew=(1, s))
    return q.text()


def stage_claims(orc, label, text):
    fm = file_model(orc, text)
    E, tabs, c = fm["entries"], fm["tabs"], fm["coding"]
    seen = set()
    if label == "ins":
        esc = _esc_of(c, 2)
        big = 512 * int(tabs[2][0][min(esc)])
        for e, ls in enumerate(E["lines"]):
            rows = plain_rows(ls[2], 2, tabs, int(E["p"]["line"][e, 2] % 16))
            for j, r in enumerate(rows):
                if r["fill"] == STAGE_WORDS and not r["flush"]:
                    seen.add("fill_512")
                if r["fill"] == STAGE_WORDS + 1 and r["flush"]:
                    seen.add("fill_513")
                    if j + 1 < len(rows) and rows[j + 1]["row"] == big:
                        seen.add(f"row_{big // 32}w_after_flush")
        assert {"fill_512", "fill_513"} <= seen and any(s.startswith("row_") for s in seen), seen
        return seen
    assert c.delchar < 0
    for e, ls in enumerate(E["lines"]):
        sk = int(E["p"]["line"][e, 1] % 16)
        seen.add(f"tag_addr_mod4_{sk % 4}")
        rows = tag_rows(ls[0], sk, -1)
        if any(r["fill"] == STAGE_WORDS and not r["flush"] for r in rows):
            seen.add("tag_fill_512")
        if any(r["fill"] == STAGE_WORDS + 1 and r["flush"] for r in rows):
            seen.add("tag_fill_513")
        if len(ls[1]) > 8192 and any(r["flush"] for r in rows):
            seen.add("tag_flush_over_8192")
    assert {"tag_fill_512", "tag_fill_513", "tag_flush_over_8192"} <= seen, seen
    assert {f"tag_addr_mod4_{k}" for k in range(4)} <= seen, seen
    return seen


# ---- tags --------------------------------------------------------------------------------------------

def shape_tags():
    """delChar fixed by entry 0; kept counts 20 ... 23 (mod 4 = 0 ... 3), 0 (every del byte is
    DELC), kept tags of every letter acgtACGTnN, tag lines at every address mod 4; and the file
    without delChar of the stage family"""
    rng = np.random.default_rng(600)
    q = S.Quiva()
    letters = np.frombuffer(b"acgtACGTnN", dtype=np.uint8)

    def entry(L, kept, s):
        d = np.full(L, DELC, dtype=np.uint8)
        pos = np.sort(rng.choice(np.arange(1, L), size=kept, replace=False))
        d[pos] = rng.integers(60, 80, size=kept)
        t = np.where(d == DELC, ord("n"), letters[rng.integers(0, 10, size=L)]).astype(np.uint8)
        q.add(d, t, rng.integers(33, 60, size=L).astype(np.uint8), rng.integers(33, 70, size=L).astype(np.uint8),
              rng.integers(33, 45, size=L).astype(np.uint8), skew=(1, s))

    for s in range(4):
        for kept in (20, 21, 22, 23, 0):
            entry(40, kept, s)
    entry(700, 0, 2)
    entry(9000, 8200, 1)
    return [("delchar", q.text()), ("no_delchar", tag_file_no_delchar())]


def tags_claims(orc, label, text):
    fm = file_model(orc, text)
    E, c = fm["entries"], fm["coding"]
    if label == "no_delchar":
        assert c.delchar < 0
        return {"no_delchar"}
    assert c.delchar == DELC
    seen = set()
    for e, ls in enumerate(E["lines"]):
        k = tag_model(ls[0], c.delchar)["kept"]
        seen.add(f"kept_mod4_{k % 4}")
        if k == 0:
            seen.add("none_kept")
        seen.add(f"tag_addr_mod4_{int(E['p']['line'][e, 1] % 4)}")
        kept = ls[1][ls[0] != DELC]
        seen |= {f"letter_{chr(x)}" for x in set(kept.tolist())}
    want = {f"kept_mod4_{k}" for k in range(4)} | {"none_kept"} | {f"tag_addr_mod4_{k}" for k in range(4)}
    want |= {f"letter_{x}" for x in "acgtACGTnN"}
    assert want <= seen, want - seen
    return seen


# ---- pad ---------------------------------------------------------------------------------------------

PAD_F = 40                      # words of the streams


def _pad_ins(kind, pad):
    """ins: 150 symbols whose last item starts at 32F - 15 (pad) or 32F - 16 (one bit short)"""
    n = 150

    def make(c, avail, rng):
        if c is None:
            return take(n, avail, rng)
        last = _one(c, 2, avail, "esc" if kind == "esc_sym" else 5, rng)
        ll = int(item_tables(c)[2][0][last[0]])
        start = 32 * PAD_F - (15 if pad else 16)             # plast
        pre = start - (ll - 8 if kind == "esc_sym" else 0)   # an escaped item's last piece is its literal
        return np.concatenate([_exact(c, 2, n - 1, pre, avail, rng, exclude=_esc_of(c, 2)), last])
    return Craft(n, ins=make, label=f"{kind}_{'pad' if pad else 'nopad'}")


def _pad_del(kind, pad):
    """del: 150 items without a run, then a trailing run of 3 (a plain run code) or of 300 (the
    escape and a 16-bit literal)"""
    n, rt = 150, (3 if kind == "run" else 300)

    def make(c, avail, rng):
        if c is None:
            return np.concatenate([take(n, avail, rng), np.full(rt, DELC, np.uint8)])
        R, Resc = item_tables(c)[1]
        t = min(rt, 255)
        assert bool(Resc[t]) == (kind == "esc_run")
        lr = int(R[t])
        start = 32 * PAD_F - (15 if pad else 16)
        pre = start - (lr if kind == "esc_run" else 0)
        return np.concatenate([_exact(c, 0, n, pre, avail, rng), np.full(rt, DELC, np.uint8)])
    return Craft(n + rt, dele=make, del_syms=n, label=f"{kind}_{'pad' if pad else 'nopad'}")


def shape_pad(orc):
    """each kind of last item on both sides of the look-ahead word.  An escaped trailing run starts
    its last piece (the 16-bit literal) 16 bits before the end, so (plast+47)>>5 never exceeds
    ceil(T/32): its cases are T = 32F (plast one bit short of the rule) and T = 32F + 1"""
    layout = [1500] * 200
    at = 5
    for kind in ("sym", "esc_sym"):
        for pad in (True, False):
            layout.insert(at, _pad_ins(kind, pad)); at += 7
    for kind in ("run", "esc_run"):
        for pad in (True, False):
            layout.insert(at, _pad_del(kind, pad)); at += 7
    text, _, _ = pinned(orc, 700, layout)
    return [("pad", text)]


def pad_claims(orc, label, text):
    fm = file_model(orc, text)
    seen = set()
    for (e, k), m in fm["streams"].items():
        if k in (0, 2) and m["rlen"] and m["full"] == PAD_F:
            start = m["plast"] - (32 * PAD_F - 16)
            if m["pad"] and start == 1:
                seen.add(f"{m['last']}_pad")
            if not m["pad"] and start == 0:
                seen.add(f"{m['last']}_nopad")
            if m["last"] == "esc_sym" and not m["pad"] and start == 0:
                assert (m["T"] + 47) >> 5 > m["full"]             # a plast without the -8 would pad
    want = {"sym_pad", "sym_nopad", "esc_sym_pad", "esc_sym_nopad", "run_pad", "run_nopad", "esc_run_nopad"}
    assert want <= seen, want - seen
    return seen


# ---- counts ------------------------------------------------------------------------------------------

COUNTS = (16383, 16384, 16385, 40000)


def counts_file(n: int) -> bytes:
    """n entries of 0..3 positions (delChar fixed by entry 0, tags 'n' over it)"""
    rng = np.random.default_rng(n)
    L = rng.integers(0, 4, size=n)
    L[0] = 3
    tot = int(L.sum())
    d = np.where(rng.random(tot) < 0.6, DELC, rng.integers(60, 70, size=tot)).astype(np.uint8)
    d[0] = DELC
    cols = [d, np.where(d == DELC, ord("n"), ACGT[rng.integers(0, 4, size=tot)]).astype(np.uint8),
            rng.integers(34, 60, size=tot).astype(np.uint8), rng.integers(36, 70, size=tot).astype(np.uint8),
            rng.integers(33, 45, size=tot).astype(np.uint8)]
    cs = np.concatenate([[0], np.cumsum(L)])
    parts = []
    for e in range(n):
        a, b = cs[e], cs[e + 1]
        parts.append(b"@m/%d/0_%d RQ=0.8\n" % (e + 1, b - a))
        for col in cols:
            parts.append(col[a:b].tobytes() + b"\n")
    return b"".join(parts)


def shape_counts():
    return [(str(n), counts_file(n)) for n in COUNTS]


def offset_scan(n: int) -> str:
    """the entry-offset scan dx_qv_encode runs for n entries"""
    if n < ONE_CTA_SCAN_BELOW:
        return "k_qv_offsets"
    return "k_tile_scan" if n <= 2 * CHAIN_TILE else "k_chain_scan"


# ---- long --------------------------------------------------------------------------------------------

LONG = (CAND_MAX_LEN - 1, CAND_MAX_LEN, CAND_MAX_LEN + 1, 2 * CAND_MAX_LEN + 3)
LONGEST = MAX_RLEN - 1


def shape_long():
    """synth.make_quiva (numpy per entry; runs of the run characters stay far below 65536):
    the LONG entries among short ones; one of 2^24 - 1 among short ones (about 84 MB)"""
    short = [3000, 17, 5000]
    return [("long", synth.make_quiva(800, short + [LONG[0], 2000, LONG[1], LONG[2], 700, LONG[3]] + short)),
            ("longest", synth.make_quiva(801, [1200, LONGEST, 900]))]


def too_long() -> bytes:
    """one entry of 2^24 positions: the oracle and the reference take it, the library refuses it"""
    return synth.make_quiva(802, [MAX_RLEN])


SHAPES = {"room": shape_room, "rows": shape_rows, "stage": shape_stage, "pad": shape_pad}
PLAIN = {"tags": shape_tags, "counts": shape_counts, "long": shape_long}
CLAIMS = {"room": room_claims, "rows": rows_claims, "stage": stage_claims, "pad": pad_claims,
          "tags": tags_claims}

_cache: dict = {}


def make(orc, name: str):
    """-> [(label, text)] of one family"""
    if name not in _cache:
        _cache[name] = SHAPES[name](orc) if name in SHAPES else PLAIN[name]()
    return _cache[name]


def make_too_long() -> bytes:
    if "too_long" not in _cache:
        _cache["too_long"] = too_long()
    return _cache["too_long"]
