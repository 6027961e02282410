"""Crafted .quiva files for pass 1 of the QV coder (dx_qv_stats.cu, dxk_qv_probe and the run
character subtraction of dx_qv_scan_dev), and a plain numpy restatement of the scan that can start
from a carry, the way a later shard of dexqv_mg is scanned.

  scan_with_carry(text, carry)   orc_qv_scan (oracle/dx_oracle.c) restated from a dx_qv_carry: the
                                 six histograms in the layout of dx_qv_stats.hist (run histograms
                                 without the oracle's +1 start), totchar, nentries, the run characters
                                 in force at the shard's end, sub_prefix, and the entries e_del /
                                 e_sub of this shard from which the runs are counted.

Shapes (each a list of (label, text) files; docstrings name the code they aim at):

  wrap_plain         k_qv_hist<plain>: one-byte counters at 255 / 256 / 257, the a == b path of bump2,
                     the pad correction of bin 0 in hist_warp_flush
  runs               k_qv_hist_run on every hist_mode: run lengths around 16, 32, 256, 512 and 65535,
                     0 ... 512 items per 32-lane round (the queue's leftover logic)
  delchar_order      k_find_delchar / k_pick_delchar: the first tag beyond the first wave of warps
  subchar_threshold  k_probe_sub and the 200 000 / half-totchar rule of dx_qv_make_coding
  empty_entries      entries of 0 positions at the ends, in a row, and behind the 100 000 crossing

All QV bytes are 1..255 and never '\\n'; every stream keeps >= 2 distinct symbols.  A line's skew is
its offset mod 16 in a 16-byte aligned buffer; the shapes set it through the header's length (the
digits of beg, end and the score).  TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import numpy as np

MOVIE = "m54"
ACGT = np.frombuffer(b"acgt", dtype=np.uint8)
DELC, SUBC = 50, 63
SUB_FIX = 100_000                      # positions after which subChar is fixed (QV.c:1005)
SUB_KEEP = 200_000                     # positions below which create drops subChar (QV.c:1029)
HIST_WARPS_PER_SM = 4 * 8              # k_find_delchar: sm_count * 4 blocks of 8 warps
PLAIN_WARPS_PER_SM = 768 // 32         # k_qv_hist<plain>: one CTA of 768 threads per SM
ROUND = 32 * 16                        # line bytes one 32-lane round of k_qv_hist_run covers


# ---- the restatement ------------------------------------------------------------------------------

def empty_carry() -> dict:
    return dict(delchar=-1, subchar=-1, totchar=0, sub=np.zeros(256, dtype=np.uint64))


def next_carry(carry: dict, res: dict) -> dict:
    """what dexqv_mg hands the next rank (tools/dexqv_mg.c:185-190)"""
    return dict(delchar=res["delchar"], subchar=res["subchar"], totchar=carry["totchar"] + res["totchar"],
                sub=res["sub_prefix"].copy())


def parse(text: bytes) -> dict:
    """entry layout of a well formed .quiva text: offsets of the five lines, rlen, wells"""
    a = np.frombuffer(text, dtype=np.uint8)
    nl = np.flatnonzero(a == 10)
    assert len(nl) % 6 == 0 and (len(nl) == 0 or nl[-1] == len(a) - 1)
    nl = nl.reshape(-1, 6)
    hdr = np.concatenate([[0], nl[:-1, 5] + 1]).astype(np.int64) if len(nl) else np.zeros(0, np.int64)
    line = (nl[:, :5] + 1).astype(np.int64)
    rlen = (nl[:, 1] - nl[:, 0] - 1).astype(np.int64)
    wells = np.array([int(text[h:e].split(b"/", 2)[1]) for h, e in zip(hdr, line[:, 0])], dtype=np.int64)
    return dict(a=a, hdr=hdr, line=line, rlen=rlen, well=wells, n=len(rlen),
                end=np.append(hdr[1:], len(a)) if len(hdr) else hdr)


def _stream(p: dict, k: int, e0: int = 0, e1: int | None = None):
    """line k (0 del, 1 tag, 2 ins, 3 mrg, 4 sub) of entries e0..e1 back to back, and where each
    entry starts in it"""
    e1 = p["n"] if e1 is None else e1
    rl = p["rlen"][e0:e1]
    st = p["line"][e0:e1, k]
    starts = np.concatenate([[0], np.cumsum(rl)[:-1]]).astype(np.int64) if len(rl) else np.zeros(0, np.int64)
    idx = np.repeat(st - starts, rl) + np.arange(int(rl.sum()), dtype=np.int64)
    return p["a"][idx], starts


def _bincount(x) -> np.ndarray:
    return np.bincount(np.asarray(x, dtype=np.int64), minlength=256).astype(np.uint64)


def run_lengths(line: np.ndarray, starts: np.ndarray, rlen: np.ndarray, rc: int) -> np.ndarray:
    """count_runs (QV.c:709-724) of every line: the run in front of each non-run symbol, and the
    trailing run of a line that ends in the run character"""
    if len(line) == 0:
        return np.zeros(0, dtype=np.int64)
    ent = np.repeat(np.arange(len(rlen)), rlen)
    nz = np.flatnonzero(line != rc)
    prev = np.concatenate([[-1], nz[:-1]])
    same = np.zeros(len(nz), dtype=bool)
    same[1:] = ent[nz[1:]] == ent[nz[:-1]]
    prev = np.where(same, prev, starts[ent[nz]] - 1)
    runs = nz - prev - 1
    ends = starts + rlen                                    # exclusive
    lastnz = starts - 1                                     # last non-run position of each line
    if len(nz):
        j = np.searchsorted(nz, ends, side="left") - 1
        cand = nz[np.maximum(j, 0)]
        lastnz = np.where((j >= 0) & (cand >= starts), cand, starts - 1)
    trail = (rlen > 0) & (lastnz < ends - 1)
    return np.concatenate([runs, (ends - 1 - lastnz)[trail]])


def scan_with_carry(text: bytes, carry: dict | None = None) -> dict:
    """orc_qv_scan (oracle/dx_oracle.c:508-542) of one shard that starts from `carry`"""
    c = carry if carry is not None else empty_carry()
    p = parse(text)
    n, rlen = p["n"], p["rlen"]
    hist = np.zeros((6, 256), dtype=np.uint64)
    lines = [_stream(p, k) for k in range(5)]
    starts = lines[0][1]
    for h, k in ((0, 0), (1, 2), (2, 3), (3, 4)):
        hist[h] = _bincount(lines[k][0])
    delchar, e_del = c["delchar"], (0 if c["delchar"] >= 0 else n)
    if delchar < 0:
        tag, dele = lines[1][0], lines[0][0]
        hit = np.flatnonzero((tag == ord("n")) | (tag == ord("N")))
        if len(hit):
            e_del = int(np.searchsorted(starts, hit[0], side="right") - 1)
            delchar = int(dele[hit[0]])
    subchar, e_sub = c["subchar"], (0 if c["subchar"] >= 0 else n)
    if subchar >= 0:
        sub_prefix = np.asarray(c["sub"], dtype=np.uint64).copy()
    else:
        cum = int(c["totchar"]) + np.cumsum(rlen)
        fix = np.flatnonzero(cum >= SUB_FIX)
        upto = int(starts[fix[0]] + rlen[fix[0]]) if len(fix) else len(lines[4][0])
        sub_prefix = np.asarray(c["sub"], dtype=np.uint64) + _bincount(lines[4][0][:upto])
        if len(fix):
            e_sub = int(fix[0])
            subchar = int(np.argmax(sub_prefix))                # the first maximum wins
    for h, k, rc, e0 in ((4, 0, delchar, e_del), (5, 4, subchar, e_sub)):
        if rc >= 0 and e0 < n:
            s = int(starts[e0])
            runs = run_lengths(lines[k][0][s:], starts[e0:] - s, rlen[e0:], rc)
            hist[h] = _bincount(np.minimum(runs, 255))
    return dict(hist=hist, totchar=int(rlen.sum()), nentries=n, delchar=delchar, subchar=subchar,
                sub_prefix=sub_prefix, e_del=e_del, e_sub=e_sub)


def lossy_codes_nul(res: dict) -> bool:
    """lossy coding rounds ins QVs down to even and mrg QVs down to a multiple of 4 (QV.c:1029-1169):
    ins QV 1 or mrg QV 1..3 gives the NUL byte a code, which dx_qv_encode_dev refuses (DX_E_CODING)"""
    return bool(res["hist"][1][1] > 0 or res["hist"][2][1:4].sum() > 0)


def oracle_view(res: dict) -> dict:
    """the restatement in the oracle's terms (orc.Stats fields, run histograms starting at 1)"""
    h = res["hist"]
    return dict(del_=h[0], ins=h[1], mrg=h[2], sub=h[3], delrun=h[4] + 1, subrun=h[5] + 1,
                totchar=res["totchar"], nentries=res["nentries"], delchar=res["delchar"],
                subchar=res["subchar"])


def shard_texts(text: bytes, cuts) -> list:
    """the text between entry boundaries cuts[i] .. cuts[i+1] (cuts start at 0 and end at n)"""
    p = parse(text)
    bounds = np.append(p["hdr"], len(text))
    return [text[int(bounds[a]):int(bounds[b])] for a, b in zip(cuts, cuts[1:])]


def chain(text: bytes, cuts) -> list:
    """the statistics pass of tools/dexqv_mg.c:176-195 on shards cut at `cuts`: in file order while a
    run character is open, then every later shard with the carry that fixed both.
    -> [(shard text, carry it was scanned with, its result)]"""
    out, cy = [], empty_carry()
    for t in shard_texts(text, cuts):
        res = scan_with_carry(t, cy)
        out.append((t, cy, res))
        if cy["delchar"] < 0 or cy["subchar"] < 0:
            cy = next_carry(cy, res)
    return out


def sum_results(results) -> dict:
    """the allreduce of dexqv_mg: histograms, totchar and nentries summed over the shards"""
    return dict(hist=sum(r["hist"] for r in results), totchar=sum(r["totchar"] for r in results),
                nentries=sum(r["nentries"] for r in results))


def plan_checks(p: dict, plan) -> dict:
    """what a cut plan holds: empty shards (and where), one-entry shards, shards of only empty
    entries, and cuts in front of a well delta >= 255"""
    rl, w = p["rlen"], p["well"]
    sizes = [b - a for a, b in zip(plan, plan[1:])]
    return dict(empty_mid=any(s == 0 for s in sizes[1:-1]), empty_end=sizes[-1] == 0,
                one_entry=1 in sizes,
                only_empty=any(s > 0 and not rl[a:b].any() for s, a, b in zip(sizes, plan, plan[1:])),
                big_delta=any(0 < c < p["n"] and w[c] - w[c - 1] >= 255 for c in plan))


def cut_plans(text: bytes, seed: int = 0) -> list:
    """cut plans (entry indices from 0 to n) for the carried scan of one file:
      - two shards cut at every boundary within 2 of e_del and e_sub (every boundary for <= 64 entries);
      - 3, 5 and 8 shards with an empty shard in the middle and at the end and a one-entry shard, and
        a shard of only empty entries where the file has a run of them;
      - two shards cut in front of a well delta >= 255."""
    p = parse(text)
    n = p["n"]
    res = scan_with_carry(text)
    if n <= 64:
        near = set(range(n + 1))
    else:
        near = {b for e in (res["e_del"], res["e_sub"]) for b in range(e - 2, e + 3) if 0 <= b <= n}
    plans = [[0, b, n] for b in sorted(near)]
    rng = np.random.default_rng(seed)
    o, m, x, y = (int(v) for v in rng.integers(0, n, size=4))
    plans.append([0, m, n, n])                                  # 3 shards: the last one empty
    rl = p["rlen"]
    pairs = [e for e in range(n - 1) if rl[e] == 0 and rl[e + 1] == 0]
    if pairs:                                                   # 5: a shard of empty entries only
        plans.append(sorted([0, pairs[0], pairs[0] + 2, m, m]) + [n])
    else:                                                       # 5: one entry, an empty shard inside
        plans.append(sorted([0, o, o + 1, m, m]) + [n])
    plans.append(sorted([0, x, o, o + 1, m, m, y]) + [n, n])    # 8: all of it
    w = p["well"]
    big = [e for e in range(1, n) if w[e] - w[e - 1] >= 255]
    if big:
        plans.append([0, big[0], n])
    return plans


# ---- building files -------------------------------------------------------------------------------

_BEGS = [0, 5, 50, 500, 5000, 50000, 500000, 5000000, 50000000, 500000000]
_QVS = [8, 85, 851, 8510]


def header(well: int, beg: int, rlen: int, qv: int, movie: str = MOVIE) -> bytes:
    return f"@{movie}/{well}/{beg}_{beg + rlen} RQ=0.{qv}\n".encode()


class Quiva:
    """a .quiva text built entry by entry; `skew=(line, s)` picks beg and the score so that line
    `line` (0 del ... 4 sub) of the entry starts at offset s mod 16"""

    def __init__(self, movie: str = MOVIE, well: int = 0):
        self.parts, self.size, self.well, self.movie = [], 0, well, movie
        self.nent = 0

    def add(self, dele, tag, ins, mrg, sub, skew=None, well_delta: int = 1):
        lines = [np.asarray(x, dtype=np.uint8) for x in (dele, tag, ins, mrg, sub)]
        L = len(lines[0])
        assert all(len(x) == L for x in lines)
        for x in lines:
            assert not np.any(x == 10) and not np.any(x == 0)
        self.well += well_delta
        hdr = None
        if skew is None:
            hdr = header(self.well, 0, L, 8, self.movie)
        else:
            k, s = skew
            for qv in _QVS:
                for beg in _BEGS:
                    h = header(self.well, beg, L, qv, self.movie)
                    if (self.size + len(h) + k * (L + 1)) % 16 == s:
                        hdr = h
                        break
                if hdr is not None:
                    break
            assert hdr is not None, ("no header gives skew", skew)
        self.parts.append(hdr)
        for x in lines:
            self.parts.append(x.tobytes() + b"\n")
        self.size += len(hdr) + 5 * (L + 1)
        self.nent += 1
        return self

    def text(self) -> bytes:
        return b"".join(self.parts)


def _tags(dele, delchar=DELC, rng=None):
    """'n' exactly where del is the run character, acgt elsewhere (the reference's own files)"""
    rng = rng if rng is not None else np.random.default_rng(0)
    return np.where(np.asarray(dele) == delchar, ord("n"), ACGT[rng.integers(0, 4, size=len(dele))])


def _noise(rng, L, lo, hi):
    return rng.integers(lo, hi, size=L).astype(np.uint8)


def _plain_entry(rng, L):
    """five lines without a tag: every stream counted by k_qv_hist<plain> (while < 100 000 positions)"""
    return (_noise(rng, L, 33, 49), ACGT[rng.integers(0, 4, size=L)], _noise(rng, L, 33, 60),
            _noise(rng, L, 33, 70), _noise(rng, L, 33, 45))


# ---- wrap_plain -----------------------------------------------------------------------------------

WRAP_RLENS = (8191, 8192, 8193, 16383, 16384, 16385)
WRAP_SKEWS = (0, 1, 8, 15)


def wrap_single(rlen: int, skew: int, sym: int = 77) -> bytes:
    """one entry whose ins line is `sym` but for its last byte, the line at `skew`: at skew 0 and rlen
    8192 every lane of the warp loads 16 chunks, 256 equal bytes, through the a == b path of bump2 (a
    counter that must wrap exactly once); 8191 / 8193 and 16383 ... 16385 put the wrap one off"""
    rng = np.random.default_rng(rlen * 16 + skew)
    d, t, i, m, s = _plain_entry(rng, rlen)
    i = np.full(rlen, sym, dtype=np.uint8)
    i[-1] = sym + 1
    m = np.full(rlen, sym + 2, dtype=np.uint8)                  # mrg too, at skew + 2 (rlen + 1)
    m[-1] = sym + 20                                            # (lossy: not in sym + 2's group of 4)
    return Quiva().add(d, t, i, m, s, skew=(2, skew)).text()


def wrap_periodic() -> bytes:
    """period-8 lines (byte i of a chunk equals byte i + 8: bump2's a == b path for every pair) and
    period-16 lines with different halves (the a != b path), long enough for every counter to wrap;
    both at several skews so that the chunk lattice cuts the period anywhere"""
    rng = np.random.default_rng(8)
    q = Quiva()
    for skew in (0, 1, 8, 15):
        for period in (8, 16):
            L = 9000 + skew
            pat = np.arange(period, dtype=np.uint8) + (90 if period == 8 else 110)
            d, t, i, m, s = _plain_entry(rng, L)
            q.add(d, t, np.resize(pat, L), np.resize(pat[::-1], L), s, skew=(2, skew))
    return q.text()


def wrap_every_value(skew: int) -> bytes:
    """one entry: all 254 admissible values (1..255 but 10) in each of the four lines, value v
    occurring 255, 256 or 257 times (by v mod 3); the del line at `skew`.  (Its lossy coding gives
    NUL a code: see lossy_codes_nul.)"""
    vals = np.array([v for v in range(1, 256) if v != 10], dtype=np.uint8)
    reps = 255 + (vals.astype(np.int64) % 3)
    rng = np.random.default_rng(254 + skew)
    lines = []
    for _ in range(4):
        x = np.repeat(vals, reps)
        rng.shuffle(x)
        lines.append(x)
    tag = ACGT[rng.integers(0, 4, size=len(lines[0]))]
    return Quiva().add(lines[0], tag, lines[1], lines[2], lines[3], skew=(0, skew)).text()


def wrap_many_short(n: int = 200_000) -> bytes:
    """n entries of 1..3 positions: about 56 lines per warp and stream on a 148-SM B200, each with
    ~15 pad bytes counted in lane 0's bin 0 and taken off again in hist_warp_flush -- that counter
    wraps many times.  (Past 100 000 positions subChar is fixed, so sub goes to k_qv_hist_run.)"""
    rng = np.random.default_rng(200)
    L = rng.integers(1, 4, size=n)
    tot = int(L.sum())
    cols = [_noise(rng, tot, 33, 49), ACGT[rng.integers(0, 4, size=tot)], _noise(rng, tot, 33, 60),
            _noise(rng, tot, 33, 70), _noise(rng, tot, 33, 45)]
    cs = np.concatenate([[0], np.cumsum(L)])
    parts = []
    for e in range(n):
        a, b = cs[e], cs[e + 1]
        parts.append(b"@m/%d/0_%d RQ=0.8\n" % (e, b - a))
        for c in cols:
            parts.append(c[a:b].tobytes() + b"\n")
    return b"".join(parts)


def shape_wrap_plain():
    files = [(f"single_{r}_{s}", wrap_single(r, s)) for r in WRAP_RLENS for s in WRAP_SKEWS]
    files += [(f"every_value_{s}", wrap_every_value(s)) for s in WRAP_SKEWS]
    files += [("periodic", wrap_periodic()), ("many_short", wrap_many_short())]
    return files


# ---- runs -----------------------------------------------------------------------------------------

RUN_LENGTHS = (0, 1, 15, 16, 17, 31, 32, 33, 254, 255, 256, 257, 511, 512, 513, 65535)
ROUND_ITEMS = (0, 1, 31, 32, 33, 511, 512)


def _run_line(rng, runs, rc, alpha):
    """runs[j] run characters in front of non-run symbol j"""
    out = []
    for r in runs:
        out.append(np.full(int(r), rc, dtype=np.uint8))
        out.append(alpha[rng.integers(0, len(alpha), size=1)].astype(np.uint8))
    return np.concatenate(out)


def _round_line(rng, skew, rc, alpha, counts):
    """a line cut into the rounds of k_qv_hist_run at this skew (the first round holds 512 - skew
    positions): round j holds counts[j] non-run items at random places, run characters elsewhere"""
    out = []
    for j, k in enumerate(counts):
        size = ROUND - skew if j == 0 else ROUND
        x = np.full(size, rc, dtype=np.uint8)
        pos = rng.choice(size, size=min(k, size), replace=False)
        x[pos] = alpha[rng.integers(0, len(alpha), size=len(pos))]
        out.append(x)
    return np.concatenate(out)


def shape_runs():
    """k_qv_hist_run (and its five hist_mode forms): delChar fixed by entry 0, subChar where the
    positions reach 100 000; then runs of every length in RUN_LENGTHS, rounds holding every count in
    ROUND_ITEMS of non-run items, in every order; the run character at position 0 and at rlen - 1;
    lines of the run character only (rlen 1, 255, 256, 65535) and lines without it; skews 0, 1, 15.
    One well delta of 300 (a cut in front of it starts a shard with 0xff bytes)."""
    rng = np.random.default_rng(65535)
    dal = np.arange(70, 78, dtype=np.uint8)                     # non-run del symbols
    sal = np.arange(33, 41, dtype=np.uint8)                     # non-run sub symbols
    q = Quiva()

    def entry(dele, sub, skew, well_delta=1):
        L = len(dele)
        q.add(dele, _tags(dele, rng=rng), _noise(rng, L, 33, 60), _noise(rng, L, 33, 70), sub,
              skew=(0, skew), well_delta=well_delta)

    # entry 0: a short line that fixes delChar at once (the tag at position 3)
    d = np.array([71, 72, 73, DELC, DELC, 74, 75, DELC], dtype=np.uint8)
    entry(d, np.array([33, SUBC, 34, SUBC, SUBC, 35, 36, SUBC], dtype=np.uint8), 0)
    # filler past 100 000 positions: sub dominated by the run character
    while q.size < 6 * SUB_FIX:
        L = 20000
        d = np.where(rng.random(L) < 0.8, DELC, dal[rng.integers(0, 8, size=L)]).astype(np.uint8)
        s = np.where(rng.random(L) < 0.85, SUBC, sal[rng.integers(0, 8, size=L)]).astype(np.uint8)
        entry(d, s, int(rng.integers(0, 16)))
    for skew in (0, 1, 15):
        order = [RUN_LENGTHS, RUN_LENGTHS[::-1], tuple(rng.permutation(RUN_LENGTHS))]
        for runs in order:
            d = _run_line(rng, runs, DELC, dal)
            s = _run_line(rng, runs[::-1], SUBC, sal)
            n = min(len(d), len(s))
            entry(d[:n], s[:n], skew)
        rounds = list(ROUND_ITEMS) + list(ROUND_ITEMS[::-1]) + [31, 1, 33, 0, 32, 512, 31, 33]
        d = _round_line(rng, skew, DELC, dal, rounds)
        s = _round_line(rng, skew, SUBC, sal, rounds[::-1])
        entry(d, s, skew, well_delta=300 if skew == 1 else 1)
        # run character at position 0 and at rlen - 1, and the other way round
        for L in (2, 17, 33, 513):
            d = dal[rng.integers(0, 8, size=L)]
            s = sal[rng.integers(0, 8, size=L)]
            d[0] = d[-1] = DELC
            s[0] = s[-1] = SUBC
            entry(d, s, skew)
            d = np.full(L, DELC, dtype=np.uint8)
            s = np.full(L, SUBC, dtype=np.uint8)
            d[0] = d[-1] = 70
            s[0] = s[-1] = 33
            entry(d, s, skew)
        for L in (1, 255, 256, 65535):                          # only the run character
            entry(np.full(L, DELC, dtype=np.uint8), np.full(L, SUBC, dtype=np.uint8), skew)
        for L in (1, 40, 600):                                  # without it
            entry(dal[rng.integers(0, 8, size=L)], sal[rng.integers(0, 8, size=L)], skew)
    return [("runs", q.text())]


# ---- delchar_order --------------------------------------------------------------------------------

DEL_RARE, DEL_LATER, DEL_DECOY = 91, 92, 93                   # del values under the tags
TAG_POSITIONS = ("0", "31", "32", "last")


def find_delchar_warps(sm_count: int) -> int:
    return sm_count * HIST_WARPS_PER_SM


def tag_entries(W: int):
    return (0, 1, W - 1, W, W + 1, 2 * W + 5)


def delchar_file(n: int, first: int | None, pos: str = "0", tag: int = ord("n"), seed: int = 0,
                 rlen_tag: int = 48) -> bytes:
    """n short entries without tags but for entry `first`, whose first tag sits at `pos` (0, 31, 32 or
    its last position) over the rare del value DEL_RARE, with a second tag three positions later over
    DEL_LATER; entry first + 3 (if any) has a decoy tag at position 0 over DEL_DECOY"""
    rng = np.random.default_rng(seed)
    L = rng.integers(1, 6, size=n)
    decoy = None if first is None or first + 3 >= n else first + 3
    for e in (first, decoy):
        if e is not None:
            L[e] = rlen_tag
    cs = np.concatenate([[0], np.cumsum(L)])
    tot = int(cs[-1])
    d, t, i, m, s = _plain_entry(rng, tot)
    t = np.where(t == ord("n"), ord("a"), t).astype(np.uint8)      # acgt only: no tags
    if first is not None:
        p = int(cs[first]) + {"0": 0, "31": 31, "32": 32, "last": rlen_tag - 1}[pos]
        d[p], t[p] = DEL_RARE, tag
        if p + 3 < cs[first + 1]:
            d[p + 3], t[p + 3] = DEL_LATER, tag
    if decoy is not None:
        d[cs[decoy]], t[cs[decoy]] = DEL_DECOY, ord("n")
    cols = (d, t, i, m, s)
    parts = []
    for e in range(n):
        a, b = cs[e], cs[e + 1]
        parts.append(header(e + 1, 0, int(b - a), 8))
        for c in cols:
            parts.append(c[a:b].tobytes() + b"\n")
    return b"".join(parts)


def shape_delchar_order(W: int):
    """k_find_delchar / k_pick_delchar on a grid of W warps: the first tag in entry 0, 1, W - 1, W,
    W + 1 or 2W + 5 (the first entry of the second and third wave) at position 0, 31, 32 or rlen - 1
    (the 32-position windows of the ballot); later tags (in the same entry, and a decoy in a later
    entry) carry other del values, so any pick but the first changes delChar.  Also: a file with 'N'
    tags only, one with a tag in its last entry only, one without tags."""
    n = 2 * W + 10
    files = []
    for e in tag_entries(W):
        for pos in TAG_POSITIONS:
            files.append((f"e{e}_p{pos}", delchar_file(n, e, pos, seed=e * 7 + len(pos))))
    files.append(("N_only", delchar_file(n, W + 1, "31", tag=ord("N"), seed=1)))
    files.append(("last_only", delchar_file(n, n - 1, "32", seed=2)))
    files.append(("no_tags", delchar_file(n, None, seed=3)))
    return files


# ---- subchar_threshold ----------------------------------------------------------------------------

SUB_A, SUB_B = 40, 41                                         # the contenders for subChar


def _sub_file(lengths, sub: np.ndarray, seed: int, well_jump_at: int | None = None) -> bytes:
    """entries of the given lengths whose sub lines, back to back, are `sub`; delChar fixed in
    entry 0 (del 'n'-tagged at position 0)"""
    rng = np.random.default_rng(seed)
    assert len(sub) == sum(lengths)
    q, at = Quiva(), 0
    for e, L in enumerate(lengths):
        d = np.where(rng.random(L) < 0.7, DELC, rng.integers(70, 78, size=L)).astype(np.uint8)
        q.add(d, _tags(d, rng=rng), _noise(rng, L, 33, 60), _noise(rng, L, 33, 70), sub[at:at + L],
              well_delta=400 if e == well_jump_at else 1)
        at += L
    return q.text()


def _subs(rng, n, counts: dict, other=(50, 60)):
    """n sub symbols with exactly counts[v] of value v, the rest drawn from `other`"""
    x = rng.integers(other[0], other[1], size=n).astype(np.uint8)
    for v in counts:
        assert not (other[0] <= v < other[1])
    pos = rng.permutation(n)
    at = 0
    for v, c in counts.items():
        x[pos[at:at + c]] = v
        at += c
    return x


def sub_crossing(total_at_end: int, seed: int) -> bytes:
    """entries of 10 000 positions but one, so that the positions reach `total_at_end` at the end of
    entry 9; subChar is fixed at entry 9 (>= 100 000) or entry 10 (99 999)"""
    rng = np.random.default_rng(seed)
    lengths = [10000] * 9 + [total_at_end - 90000] + [7000] * 4
    sub = np.concatenate([_subs(rng, L, {SUB_A: L // 2}) for L in lengths])
    return _sub_file(lengths, sub, seed, well_jump_at=10)


def sub_inside_long_entry() -> bytes:
    """the 100 000 crossing falls inside one entry of 150 000 positions"""
    rng = np.random.default_rng(150)
    lengths = [30000, 150000, 20000]
    sub = np.concatenate([_subs(rng, L, {SUB_A: L // 2}) for L in lengths])
    return _sub_file(lengths, sub, 150)


def sub_tie() -> bytes:
    """through the fixing entry SUB_A and SUB_B occur equally often: the smaller symbol must win.
    Before it SUB_B leads; the fixing entry (entry 4) evens them out."""
    rng = np.random.default_rng(41)
    lengths = [20000] * 4 + [30000] + [20000] * 2
    parts = [_subs(rng, L, {SUB_A: 6000, SUB_B: 7000}) for L in lengths[:4]]
    parts.append(_subs(rng, 30000, {SUB_A: 12000, SUB_B: 8000}))         # 36 000 each after it
    parts += [_subs(rng, L, {SUB_A: 8000, SUB_B: 9000}) for L in lengths[5:]]
    return _sub_file(lengths, np.concatenate(parts), 41)


def sub_decided_by_prefix() -> bytes:
    """the fixing entry (entry 3) holds more SUB_B than SUB_A, but the entries before it hold so many
    SUB_A that SUB_A wins: a shard that starts at the fixing entry has to add the carry's counts"""
    rng = np.random.default_rng(43)
    lengths = [25000] * 3 + [40000] + [20000] * 2
    parts = [_subs(rng, L, {SUB_A: 15000, SUB_B: 5000}) for L in lengths[:3]]
    parts.append(_subs(rng, 40000, {SUB_A: 5000, SUB_B: 25000}))         # 50 000 : 40 000 after it
    parts += [_subs(rng, L, {SUB_A: 9000, SUB_B: 3000}) for L in lengths[4:]]
    return _sub_file(lengths, np.concatenate(parts), 43)


def sub_half(total: int, below: int) -> bytes:
    """`total` positions, subChar SUB_A with ceil(total / 2) - below occurrences: the 200 000 rule and
    the sub[subChar] >= totchar / 2 rule of create, exactly at and one below the threshold"""
    rng = np.random.default_rng(total * 2 + below)
    lengths = [25000] * (total // 25000)
    if total % 25000:
        lengths.append(total % 25000)
    want = (total + 1) // 2 - below
    # SUB_A leads clearly in the first 100 000 positions (36 000 against ~6 400 of each other value)
    head = _subs(rng, SUB_FIX, {SUB_A: 36000})
    tail = _subs(rng, total - SUB_FIX, {SUB_A: want - 36000})
    return _sub_file(lengths, np.concatenate([head, tail]), total)


def shape_subchar_threshold():
    files = [(f"cross_{t}", sub_crossing(t, t)) for t in (100_000, 99_999, 100_001)]
    files += [("inside_150000", sub_inside_long_entry()), ("tie", sub_tie()),
              ("prefix_decides", sub_decided_by_prefix())]
    files += [(f"half_{t}_{b}", sub_half(t, b)) for t in (199_999, 200_000, 200_001) for b in (0, 1)]
    return files


# ---- empty_entries --------------------------------------------------------------------------------

def shape_empty_entries():
    """entries of 0 positions at the file's start and end, three in a row, and right behind the
    entry at which the positions reach exactly 100 000; also a small file made of empty entries
    around two short ones"""
    rng = np.random.default_rng(0)
    q = Quiva()
    empty = [np.zeros(0, np.uint8)] * 5

    def real(L, well_delta=1):
        d = np.where(rng.random(L) < 0.8, DELC, rng.integers(70, 78, size=L)).astype(np.uint8)
        s = np.where(rng.random(L) < 0.7, SUBC, rng.integers(33, 41, size=L)).astype(np.uint8)
        q.add(d, _tags(d, rng=rng), _noise(rng, L, 33, 60), _noise(rng, L, 33, 70), s,
              well_delta=well_delta)

    q.add(*empty)
    q.add(*empty)
    for L in (30000, 40000, 30000):                           # 100 000 exactly at the end of entry 4
        real(L)
    q.add(*empty)
    real(5000, well_delta=700)
    q.add(*empty).add(*empty).add(*empty)
    for L in (60000, 50000, 17):
        real(L)
    q.add(*empty)
    q.add(*empty)
    small = Quiva()
    small.add(*empty)
    for L in (40, 7):
        d = np.full(L, DELC, dtype=np.uint8)
        d[::3] = 71
        d[1::5] = 72
        small.add(d, _tags(d, rng=rng), _noise(rng, L, 33, 40), _noise(rng, L, 33, 40),
                  _noise(rng, L, 60, 64))
        small.add(*empty)
    small.add(*empty)
    return [("mixed", q.text()), ("small", small.text())]


SHAPES = {
    "wrap_plain": shape_wrap_plain,
    "runs": shape_runs,
    "subchar_threshold": shape_subchar_threshold,
    "empty_entries": shape_empty_entries,
}

_cache: dict = {}


def make(name: str, W: int | None = None):
    """-> [(label, text)] of one shape; delchar_order needs the warps W of k_find_delchar's grid"""
    key = (name, W)
    if key not in _cache:
        _cache[key] = shape_delchar_order(W) if name == "delchar_order" else SHAPES[name]()
    return _cache[key]
