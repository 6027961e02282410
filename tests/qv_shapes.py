"""Crafted .quiva files whose code tables take shapes the parallel QV decoders find hard, each tied
to the decoder branch it aims at (dx_qv_decode5.cu / dx_qv_decode6.cu):

  fixed3 / fixed5 / fixed6   every ins and mrg code is 3, 5 or 6 bits long.  256*i is then no code
                             boundary for most lanes, and the guessed paths never meet the true one:
                             the two-finger walk runs past kFingerBudget (later windows re-decode),
                             and with a window of >= 13 lanes the fix point needs >= 12 rounds, where
                             the speculative modes give the entry up (general path);
  fixed4 / fixed1            4-bit codes (every guess is a boundary: no restarts) and 1-bit codes
                             (256 symbols per lane: a window writes far more than kStage bytes);
  exact_ends                 4-bit ins / mrg streams whose last item sits at bit 256*m - 4, 256*m - 8
                             ... 256*m + 4 for m = 1, 2, 31, 32, 33, 64: the (p_last + 47) >> 5
                             stream-length rule, the switch to one symbol at a time, windows of one
                             lane and of more than 32 lanes (the carry);
  run_parity                 3-bit run and symbol codes in the del and sub run streams: a lane's walk
                             can land on a true bit position with the wrong item parity;
  esc_dense                  type-2 (escape) tables in all four symbol streams, escapes in every
                             stream of every entry (24-bit steps);
  runs_16bit                 runs of 254 ... 65535 at the start, middle and end of entries;
  runs_over_16bit            one run of 65536: the format keeps 16 bits of a run literal, so the
                             image does not decode (TOO_LONG_RUN below).

Every generator checks its own table shape with the oracle's coding (qv_shape_check), so a file
that drifts to another shape fails instead of passing quietly.  Symbols stay in 1..126 and never
'\\n'; tags are 'n' exactly where del == delChar, so every file but runs_over_16bit round-trips to
the identity.  TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import numpy as np

from dextractor_b200 import synth

ACGT = np.frombuffer(b"acgt", dtype=np.uint8)
DELC, SUBC = 50, 63                     # the run characters synth.make_quiva uses ('2', '?')
KS, KTAIL, BUDGET, GIVEUP = 256, 24, 24, 12   # subsequence bits, longest step, finger budget, rounds


def _uniform(rng, L, alphabet):
    """L symbols uniform over `alphabet`, each of them present at least once when L allows"""
    a = np.asarray(alphabet, dtype=np.uint8)
    s = a[rng.integers(0, len(a), size=L)]
    m = min(L, len(a))
    s[:m] = a[:m]
    return s


def _tags_follow(st, rng):
    st[1][:] = np.where(st[0] == DELC, ord("n"), ACGT[rng.integers(0, 4, size=len(st[0]))])


def _fixed(seed, nsym, lengths):
    # (two symbols 4 apart: the lossy coding's rounding keeps them distinct)
    alpha = np.arange(40, 40 + nsym) if nsym > 2 else np.array([40, 44])

    def hook(i, st):
        r = np.random.default_rng(seed * 1000 + i)
        st[2][:] = _uniform(r, len(st[2]), alpha)
        st[3][:] = _uniform(r, len(st[3]), alpha[::-1])
    return synth.make_quiva(seed, lengths, stream_hook=hook)


def fixed_lengths(seed, n=24, lo=2500, hi=7000):
    """entries of 2500..7000 positions: 5-bit streams of >= 49 subsequences (two windows)"""
    return [int(x) for x in np.random.default_rng(seed).integers(lo, hi, size=n)]


def shape_fixed(nbits):
    seed = 900 + nbits
    return _fixed(seed, 1 << nbits, fixed_lengths(seed))


def shape_fixed1():
    seed = 901
    return _fixed(seed, 2, fixed_lengths(seed, n=8, lo=9000, hi=30000))


EXACT_M = (1, 2, 31, 32, 33, 64)


def exact_end_lengths():
    """4-bit streams end at bit 4 * rlen: rlen = 64m + {-1, 0, +1} puts the end at 256m + {-4, 0, +4};
    64m - 5 and 64m - 3 put the last item into [256m - kTail, 256m)"""
    out = []
    for m in EXACT_M:
        out += [64 * m + d for d in (-5, -3, -1, 0, 1)]
    return out


def shape_exact_ends():
    return _fixed(904, 16, exact_end_lengths() * 3)


def _runs(r, n):
    """run lengths: 0..7 for three items in four, else 8..254 -- every run length is common enough
    for a code of at most 11 bits, so the parallel decoders' tables hold the run code"""
    return np.where(r.random(n) < 0.75, r.integers(0, 8, size=n), r.integers(8, 255, size=n))


def shape_run_parity():
    """del and sub: runs of mostly 0..7 run characters between non-run symbols drawn from 8 values;
    > 200 000 positions, so subChar is in use"""
    def line(r, L, rc, alpha):
        runs = _runs(r, L)
        out = np.empty(L, dtype=np.uint8)
        k = 0
        for run in runs:
            if k >= L:
                break
            out[k:k + run] = rc
            k += run
            if k < L:
                out[k] = alpha[r.integers(0, 8)]
                k += 1
        out[:8] = alpha                     # every non-run symbol present
        return out

    def hook(i, st):
        r = np.random.default_rng(905000 + i)
        L = len(st[0])
        st[0][:] = line(r, L, DELC, np.arange(70, 78))
        st[4][:] = line(r, L, SUBC, np.arange(80, 88))
        _tags_follow(st, r)
    return synth.make_quiva(905, [6000] * 40, stream_hook=hook)


ESC_TAIL = 5          # the deepest symbols of a 21-symbol Fibonacci code: longer than 16 bits


def _fib_pool(rng, total, nent, base):
    """`total` symbols with Fibonacci-shaped counts over 21 values (a Huffman chain 20 deep); the
    ESC_TAIL rarest ones go round-robin to the entries, the rest are shuffled"""
    fib = [1, 1]
    while len(fib) < 21:
        fib.append(fib[-1] + fib[-2])
    fib = np.array(fib[::-1], dtype=np.int64)              # symbol base+k: count ~ fib[k]
    scale = total // int(fib.sum())
    counts = fib * scale
    counts[0] += total - int(counts.sum())
    tail = np.repeat(np.arange(21 - ESC_TAIL, 21), counts[21 - ESC_TAIL:])
    body = np.repeat(np.arange(0, 21 - ESC_TAIL), counts[: 21 - ESC_TAIL])
    rng.shuffle(body)
    return (body + base).astype(np.uint8), (tail + base).astype(np.uint8)


def shape_esc_dense():
    """del (no 'n' tags: no delChar), ins, mrg and sub (< 200 000 positions: no subChar) are four
    plain streams with Fibonacci-shaped counts: type-2 tables whose escaped symbols occur in every
    stream of every entry (a Huffman code deeper than 16 bits keeps escapes to about 1 in 1000)"""
    nent, L = 24, 8000
    rng = np.random.default_rng(906)
    pools = [_fib_pool(rng, nent * L, nent, base) for base in (40, 66, 90, 35)]

    def hook(i, st):
        r = np.random.default_rng(906000 + i)
        for k, (body, tail) in zip((0, 2, 3, 4), pools):
            at = sum(L - len(tail[j::nent]) for j in range(i))
            mine = tail[i::nent]
            put = np.zeros(L, dtype=bool)
            put[r.choice(L, size=len(mine), replace=False)] = True
            s = np.empty(L, dtype=np.uint8)
            s[put] = mine
            s[~put] = body[at:at + L - len(mine)]
            st[k][:] = s
        st[1][:] = ACGT[r.integers(0, 4, size=L)]
    return synth.make_quiva(906, [L] * nent, stream_hook=hook)


RUNS_16 = (254, 255, 256, 65534, 65535)


def _run_entries(runs):
    """per run R: one entry with the run at its start and its end, one with it in the middle"""
    lengths, plan = [], []
    for R in runs:
        lengths.append(2 * R + 1500); plan.append(("ends", R))
        lengths.append(R + 1700); plan.append(("mid", R))
    return lengths, plan


def _run_line(r, L, rc, base):
    """runs of 0..299 run characters between symbols base .. base+15"""
    out = np.full(L, rc, dtype=np.uint8)
    k = 0
    while True:
        k += int(r.integers(0, 300))
        if k >= L:
            return out
        out[k] = base + int(r.integers(0, 16))
        k += 1


def shape_runs_16bit():
    lengths, plan = _run_entries(RUNS_16)
    lengths += [3000, 1]; plan += [("plain", 0), ("plain", 0)]

    def hook(i, st):
        r = np.random.default_rng(907000 + i)
        how, R = plan[i]
        L = len(st[0])
        d, s = _run_line(r, L, DELC, 33), _run_line(r, L, SUBC, 64)
        if how == "ends":
            d[:R] = DELC; d[R] = 40; d[L - R:] = DELC; d[L - R - 1] = 41
            s[:R] = SUBC; s[R] = 70; s[L - R:] = SUBC; s[L - R - 1] = 71
        elif how == "mid":
            a = (L - R) // 2
            d[a:a + R] = DELC; d[a - 1] = 40; d[a + R] = 41
            s[a:a + R] = SUBC; s[a - 1] = 70; s[a + R] = 71
        st[0][:] = d
        st[4][:] = s
        _tags_follow(st, r)
    return synth.make_quiva(907, lengths, stream_hook=hook)


TOO_LONG_RUN = 65536


def shape_runs_over_16bit(run=TOO_LONG_RUN):
    """a few ordinary entries and one whose deletion line is `run` delChars (a single run item)"""
    lengths = [2000, 1500, run, 1800]

    def hook(i, st):
        if i == 2:
            st[0][:] = DELC
            st[1][:] = ord("n")
    return synth.make_quiva(908, lengths, stream_hook=hook)


SHAPES = {
    "fixed3": lambda: shape_fixed(3),
    "fixed4": lambda: shape_fixed(4),
    "fixed5": lambda: shape_fixed(5),
    "fixed6": lambda: shape_fixed(6),
    "fixed1": shape_fixed1,
    "exact_ends": shape_exact_ends,
    "run_parity": shape_run_parity,
    "esc_dense": shape_esc_dense,
    "runs_16bit": shape_runs_16bit,
}
# the shapes a speculative decode (discovered entries) is expected to give up on
GIVEUP_SHAPES = ("fixed3", "fixed5", "fixed6")

_cache: dict = {}


def make(name: str) -> bytes:
    if name not in _cache:
        _cache[name] = SHAPES[name]() if name in SHAPES else shape_runs_over_16bit()
    return _cache[name]


# ---- what each shape must look like in the oracle's coding -----------------------------------------

def coding(orc, text, lossy=False):
    return orc.qv_create(orc.qv_scan(text), lossy)


def code_lens(tab):
    """{symbol: code length} of one scheme"""
    return {i: tab.lens[i] for i in range(256) if tab.lens[i] > 0}


def escaped(tab):
    """symbols coded as the escape (type-2 tables), 255 itself excluded"""
    if tab.type != 2:
        return set()
    return {i for i in range(255) if tab.lens[i] > 0 and tab.lens[i] == tab.lens[255]
            and tab.bits[i] == tab.bits[255]}


DEC2_MAXSUB = 64       # sub-tables for codes of 12..16 bits the parallel decoders' tables hold


def long_prefixes(tab):
    """distinct 11-bit prefixes of the 12..16-bit codes: the sub-tables the parallel decoders need
    (more than DEC2_MAXSUB in any table and the library decodes with the sequential kernels)"""
    return len({(tab.bits[i] >> (tab.lens[i] - 11)) & 0x7ff for i in range(256) if 11 < tab.lens[i] <= 16})


def qv_shape_check(orc, name, text):
    """assert the shape `name` promises; returns a one-line description of the tables"""
    c = coding(orc, text)
    for lossy in (False, True):
        cl = coding(orc, text, lossy)
        assert all(long_prefixes(cl.tab[k]) <= DEC2_MAXSUB for k in range(6)), (name, lossy)
    ins, mrg = code_lens(c.tab[2]), code_lens(c.tab[3])
    if name.startswith("fixed") or name == "exact_ends":
        nbits = 4 if name == "exact_ends" else int(name[5:])
        for k, lens in ((2, ins), (3, mrg)):
            assert len(lens) == 1 << nbits and set(lens.values()) == {nbits}, (name, k, lens)
            assert c.tab[k].type == 0, (name, k, c.tab[k].type)
        return f"{name}: ins/mrg {len(ins)} codes, all {nbits} bits"
    if name == "run_parity":
        assert c.delchar == DELC and c.subchar == SUBC, (c.delchar, c.subchar)
        for sym, run, alpha in ((0, 1, range(70, 78)), (4, 5, range(80, 88))):
            sl, rl = code_lens(c.tab[sym]), code_lens(c.tab[run])
            assert set(sl) == set(alpha) and set(sl.values()) <= {3, 4}, (sym, sl)
            assert all(3 <= rl[r] <= 4 for r in range(8)), (run, {r: rl[r] for r in range(8)})
        return "run_parity: del/sub symbols and runs 0..7 in 3-4 bit codes"
    if name == "esc_dense":
        assert c.delchar < 0 and c.subchar < 0, (c.delchar, c.subchar)
        out = []
        for k in (0, 2, 3, 4):
            esc = escaped(c.tab[k])
            assert c.tab[k].type == 2 and len(esc) >= 2, (k, c.tab[k].type, esc)
            out.append(f"tab{k} {len(esc)} escaped")
        return "esc_dense: " + ", ".join(out)
    if name == "runs_16bit":
        assert c.delchar == DELC and c.subchar == SUBC, (c.delchar, c.subchar)
        return f"runs_16bit: run tables type {c.tab[1].type}/{c.tab[5].type}"
    if name == "runs_over_16bit":
        assert c.delchar == DELC
        return "runs_over_16bit"
    raise KeyError(name)


# ---- a CPU model of lane synchronisation ------------------------------------------------------------

def stream_bits(orc, sym, run, rchar, line: bytes) -> np.ndarray:
    """the stream as a bit array: 32-bit little-endian words, codes MSB-first inside each word"""
    w = np.frombuffer(orc.encode_stream(sym, run, rchar, line), dtype="<u4")
    return np.unpackbits(w.astype(">u4").view(np.uint8))


def _decoder(tab):
    """bits -> one step: (symbol, length incl. escape literal) for a code starting at `pos`"""
    by = {(int(tab.lens[i]), int(tab.bits[i])): i for i in range(256) if tab.lens[i] > 0}
    esc = (int(tab.lens[255]), int(tab.bits[255])) if tab.type == 2 else None
    maxlen = max(k for k, _ in by)

    def step(bits, pos, literal):
        v = 0
        for L in range(1, maxlen + 1):
            v = (v << 1) | int(bits[pos + L - 1]) if pos + L - 1 < len(bits) else v << 1
            if (L, v) in by:
                x = by[(L, v)]
                return x, L + (literal if (x == 255 or (L, v) == esc) else 0)
        return -1, 1                        # no code here (the kernels step one bit)
    return step


def sync_walks(bits, sym, run=None, lanes=32):
    """For lanes 1 .. lanes-1 of the first window: (steps, parity_miss, walked).  `steps` is the
    number of items lane i decodes from its guess 256*i (item parity 0) before it stands on a state
    of the true path -- (bit position, item parity) for run streams -- or None if it reaches the end
    of its subsequence first; `walked` is the number of items it decoded either way.  `parity_miss`
    counts the true bit positions it passed with the wrong parity.  The true path is the sequential
    decode from bit 0."""
    ss, rs = _decoder(sym), (_decoder(run) if run is not None else None)
    n = len(bits)

    def nxt(pos, par):
        if rs is not None and par == 0:
            return pos + rs(bits, pos, 16)[1], 1
        return pos + ss(bits, pos, 8)[1], 0

    true, pos, par = {}, 0, 0
    while pos < min(n, lanes * KS + 64):
        true[pos] = par
        pos, par = nxt(pos, par)
    out = []
    for i in range(1, lanes):
        pos, par, steps, miss = i * KS, 0, 0, 0
        lim = min((i + 1) * KS, n)
        while pos < lim and true.get(pos, -1) != par:
            miss += pos in true
            pos, par = nxt(pos, par)
            steps += 1
        out.append((steps if pos < lim else None, miss, steps))
    return out


def items(bits, sym):
    """the sequential decode of a plain stream: (bit position, length with the escape literal, symbol)"""
    ss = _decoder(sym)
    out, pos = [], 0
    while pos < len(bits) - 32:
        x, L = ss(bits, pos, 8)
        out.append((pos, L, x))
        pos += L
    return out


def sync_rounds(bits, sym, nact=32):
    """the lane speculation's fix point on the first window of a plain stream: lane 0 starts at 0,
    lane i at 256*i; each round every lane adopts its predecessor's exit (its first code boundary at
    or past 256*(i+1)) until no exit changes.  -> rounds needed"""
    ss = _decoder(sym)

    def exit_from(p, lim):
        while p < lim:
            p += ss(bits, p, 8)[1]
        return p

    start = [i * KS for i in range(nact)]
    ex = [exit_from(start[i], (i + 1) * KS) for i in range(nact)]
    rounds = 0
    while True:
        rounds += 1
        new = [0] + ex[:-1]
        if new == start:
            return rounds
        start = new
        ex = [exit_from(start[i], (i + 1) * KS) for i in range(nact)]
