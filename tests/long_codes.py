""".quiva files whose deletion run table needs many codes longer than 11 bits.

The reference counts one run per non-run symbol of a deletion line and adds one to each of the 256
run-length buckets (QV.c:709-724; count_runs in oracle/dx_oracle.c), so every run table codes all 256
lengths.  When the deletion lines are nearly all delChar, a file has few runs.  Here they fall on a
few short lengths with halving counts (a Huffman chain SHORT_RUNS deep) and on long runs (bucket 255,
as many as the file needs).  The 250 lengths that only have their +1 then get codes of 12 to 14 bits
over more than 64 distinct 11-bit prefixes, whatever the file's size.  Until the parallel decoders
took codes of any length, such a coding went to the sequential kernels or was refused by the
byte-range decode.

Entries need at least 300 positions.  ins, mrg and sub are synth.make_quiva's; tags are 'n' exactly
where del == delChar, so a file round-trips to the identity.  TEST INFRASTRUCTURE ONLY (scripts/long_code_gain.py uses it too)."""
from __future__ import annotations

import numpy as np

from dextractor_b200 import synth
from tests.qv_shapes import DELC, code_lens, long_prefixes

SHORT_RUNS = (3, 9, 27)              # the few short run lengths ...
SHORT_SHARE = (4, 2, 1)              # ... and their relative counts
SHORT_TOTAL = 2800                   # short runs in a file, whatever its size
LONG_RUN = (256, 1000)               # the other runs: bucket 255, the most common length
PREFIXES = 64                        # the 11-bit prefixes the parallel decoders' old tables held


def make_quiva(seed: int, lengths) -> bytes:
    lengths = [int(x) for x in lengths]
    total = float(sum(lengths))
    p = np.asarray(SHORT_SHARE, dtype=float) / sum(SHORT_SHARE)

    def hook(i, st):
        r = np.random.default_rng(seed * 100003 + i)
        L = len(st[0])
        out = np.full(L, DELC, dtype=np.uint8)
        k = 0
        for run in r.choice(SHORT_RUNS, size=int(r.poisson(SHORT_TOTAL * L / total)), p=p):
            if k + int(run) + 1 > L - 1 - LONG_RUN[0]:
                break
            k += int(run)
            out[k] = 70 + int(r.integers(0, 8))
            k += 1
        # the line ends with a symbol (no run is counted behind it), and the run in front of it is long
        while L - 1 - k > LONG_RUN[1] + LONG_RUN[0]:
            k += int(r.integers(*LONG_RUN))
            out[k] = 70 + int(r.integers(0, 8))
            k += 1
        out[L - 1] = 70 + int(r.integers(0, 8))
        st[0][:] = out
        st[1][:] = np.where(out == DELC, ord("n"), np.frombuffer(b"acgt", dtype=np.uint8)[r.integers(0, 4, size=L)])
    return synth.make_quiva(seed, lengths, stream_hook=hook)


def long_run_codes(tab) -> int:
    """codes of 12 to 16 bits in one scheme"""
    return sum(1 for n in code_lens(tab).values() if 12 <= n <= 16)


def max_prefixes(coding) -> int:
    """the most distinct 11-bit prefixes of 12..16-bit codes in any of the six schemes"""
    return max(long_prefixes(coding.tab[k]) for k in range(6))
