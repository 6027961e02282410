"""The crafted QV shapes of tests/qv_shapes.py on the CPU: every file has the code tables it promises,
reaches the decoder branch it is meant for in a CPU model of the lane speculation, and (but for the
over-long run) round-trips through the oracle.  These keep the GPU tests' inputs honest on any
machine."""
import numpy as np
import pytest

from tests import qv_shapes as Q

ALL = sorted(Q.SHAPES)


def _entries(text):
    lines = text.split(b"\n")
    return [lines[6 * e: 6 * e + 6] for e in range(len(lines) // 6)]


@pytest.mark.parametrize("name", ALL + ["runs_over_16bit"])
def test_shape_has_its_code_tables(orc, name):
    text = Q.make(name)
    assert len(text) <= 2_200_000
    print(Q.qv_shape_check(orc, name, text))


@pytest.mark.parametrize("name", ALL)
def test_shape_round_trips_through_the_oracle(orc, name):
    text = Q.make(name)
    for lossy in (False, True):
        enc = orc.dexqv(text, lossy=lossy)
        back = orc.undexqv(enc)
        if not lossy:
            assert back == text
        else:
            assert len(back) == len(text)


def _ins_bits(orc, text, entry):
    c = Q.coding(orc, text)
    line = _entries(text)[entry][3]
    return Q.stream_bits(orc, c.tab[2], None, -1, line), c.tab[2]


@pytest.mark.parametrize("name", ["fixed3", "fixed5", "fixed6"])
def test_fixed_codes_never_synchronise(orc, name):
    """A lane whose guess is not on the true path walks its whole subsequence without meeting it
    (more than kFingerBudget steps: the redecode branch), and the speculation's fix point over a full
    window needs more than 12 rounds (the speculative modes give up)."""
    text = Q.make(name)
    nbits = int(name[5:])
    bits, tab = _ins_bits(orc, text, 0)
    assert len(bits) >= 32 * Q.KS
    walks = Q.sync_walks(bits, tab)
    never = [w for s, _, w in walks if s is None]
    assert never, walks
    # a lane that never meets the true path walks its whole subsequence: one finger alone decodes
    # more items than the two-finger budget allows
    assert min(never) > Q.BUDGET, never
    # Lanes whose guess 256*i is a multiple of nbits start on the true path, so unsynchronised
    # lanes come in runs of at most nbits - 1, never 12.  What gives up is the fix point: a lane on
    # the true path adopts its predecessor's wrong exit and leaves it again, so the correct start
    # advances one lane per round and a window of 32 lanes needs 32 rounds.
    rounds = Q.sync_rounds(bits, tab)
    print(f"{name}: {len(never)}/31 lanes never meet the true path (walks of {min(never)}..{max(never)} "
          f"items), fix point after {rounds} rounds")
    assert rounds > Q.GIVEUP
    # the give-up is reached in every entry long enough for a full first window
    for e, ent in enumerate(_entries(text)):
        if len(ent[3]) * nbits >= 32 * Q.KS:
            b, _ = _ins_bits(orc, text, e)
            assert Q.sync_rounds(b, tab) > Q.GIVEUP, e


def test_fixed4_every_guess_is_a_boundary(orc):
    bits, tab = _ins_bits(orc, Q.make("fixed4"), 0)
    assert all(s == 0 for s, _, _ in Q.sync_walks(bits, tab))
    assert Q.sync_rounds(bits, tab) == 1


def test_fixed1_overflows_the_stage(orc):
    """1-bit codes: 256 symbols per lane, a full window is 8192 symbols > kStage (2560)"""
    text = Q.make("fixed1")
    assert min(len(e[3]) for e in _entries(text)) >= 32 * Q.KS
    bits, tab = _ins_bits(orc, text, 0)
    assert all(s == 0 for s, _, _ in Q.sync_walks(bits, tab))


def test_exact_ends_place_the_last_item(orc):
    """ins streams of 4-bit codes end at bit 4 * rlen: exactly on, just before and just after a
    subsequence boundary, and with the last item inside the one-at-a-time tail [lim - kTail, lim)"""
    text = Q.make("exact_ends")
    c = Q.coding(orc, text)
    seen = set()
    for ent in _entries(text):
        line = ent[3]
        L = len(line)
        bits = Q.stream_bits(orc, c.tab[2], None, -1, line)
        nwords = len(bits) // 32
        last = 4 * (L - 1)
        assert nwords == max((4 * L + 31) >> 5, (last + 47) >> 5)     # the stream-length rule
        m, off = divmod(4 * L, Q.KS)
        if off > Q.KS // 2:
            m, off = m + 1, off - Q.KS
        seen.add(off)
        if off <= 0:
            assert m * Q.KS - Q.KTAIL <= last < m * Q.KS
    assert {-20, -12, -4, 0, 4} <= seen
    assert max(len(e[3]) for e in _entries(text)) * 4 > 32 * Q.KS       # second window, the carry


def test_run_parity_lands_on_wrong_parity(orc):
    """del and sub run streams: some lane's walk passes a true bit position with the wrong item
    parity before it synchronises"""
    text = Q.make("run_parity")
    c = Q.coding(orc, text)
    misses = {}
    for sym, run, rc, k in ((0, 1, Q.DELC, 1), (4, 5, Q.SUBC, 5)):
        total = 0
        for ent in _entries(text)[:6]:
            bits = Q.stream_bits(orc, c.tab[sym], c.tab[run], rc, ent[k])
            total += sum(m for _, m, _ in Q.sync_walks(bits, c.tab[sym], c.tab[run]))
        misses[sym] = total
    print("run_parity: wrong-parity landings", misses)
    assert all(v > 0 for v in misses.values()), misses


def test_esc_dense_escapes_in_every_stream(orc):
    """every stream of every entry holds escapes, and in each of the four streams some escape step
    (code + 8-bit literal) straddles a 256-bit subsequence boundary"""
    text = Q.make("esc_dense")
    c = Q.coding(orc, text)
    straddle = {}
    for k, line_no in ((0, 1), (2, 3), (3, 4), (4, 5)):
        esc = Q.escaped(c.tab[k])
        steps = 0
        for e, ent in enumerate(_entries(text)):
            n = sum(ent[line_no].count(bytes([x])) for x in esc)
            assert n >= 1, (k, e)
            bits = Q.stream_bits(orc, c.tab[k], None, -1, ent[line_no])
            for pos, L, x in Q.items(bits, c.tab[k]):
                if x == 255:
                    assert L > c.tab[k].lens[255]
                    steps += pos // Q.KS != (pos + L - 1) // Q.KS
        straddle[k] = steps
    print("esc_dense: escape steps across a subsequence boundary per table", straddle)
    assert all(v >= 1 for v in straddle.values()), straddle


def test_runs_16bit_are_there(orc):
    text = Q.make("runs_16bit")
    lens = set()
    for ent in _entries(text):
        d = np.frombuffer(ent[1], dtype=np.uint8) == Q.DELC
        edges = np.flatnonzero(np.diff(np.concatenate([[0], d.astype(np.int8), [0]])))
        lens |= set((edges[1::2] - edges[::2]).tolist())
    assert set(Q.RUNS_16) <= lens


def test_run_of_65536_does_not_fit_the_format(orc):
    """The run literal has 16 bits: a run of 65536 is written as 0 and the image does not decode
    (ORC_E_FORMAT); one of 65535 still round-trips"""
    text = Q.make("runs_over_16bit")
    with pytest.raises(orc.OracleError) as e:
        orc.undexqv(orc.dexqv(text))
    assert e.value.code == -1
    ok = Q.shape_runs_over_16bit(65535)
    assert orc.undexqv(orc.dexqv(ok)) == ok
