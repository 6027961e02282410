"""The scan shapes of tests/scan_shapes.py on the CPU: the numpy restatement of the carried scan
equals the oracle's scan on every file, shards of any cut add up to the whole file and hand the run
characters on where the whole file fixes them, and every file has the property its docstring claims.
These keep the GPU tests' inputs and their reference honest on any machine."""
import numpy as np
import pytest

from tests import cases
from tests import scan_shapes as S

# the warps of k_find_delchar's grid on a 148-SM and on a 132-SM part: the shapes do not depend on one
GRIDS = (148 * S.HIST_WARPS_PER_SM, 132 * S.HIST_WARPS_PER_SM)
NAMES = sorted(S.SHAPES) + ["delchar_order"]


def _files(name, W=GRIDS[0]):
    return S.make(name, W if name == "delchar_order" else None)


def _assert_equals_oracle(res, ref, what):
    view = S.oracle_view(res)
    for k, v in view.items():
        assert np.array_equal(np.asarray(v), np.asarray(getattr(ref, k))), (what, k)


@pytest.mark.parametrize("name", NAMES)
def test_restatement_equals_the_oracle(orc, name):
    for label, text in _files(name):
        _assert_equals_oracle(S.scan_with_carry(text, S.empty_carry()), orc.qv_scan(text), label)


def test_restatement_equals_the_oracle_on_the_cases(orc):
    for label, text in cases.quiva_cases():
        _assert_equals_oracle(S.scan_with_carry(text), orc.qv_scan(text), label)


def _symbols_coded(res, lossy):
    """distinct symbols of the del, ins, mrg and sub tables dx_qv_make_coding builds (QV.c:1029-1169):
    the run characters taken out, ins / mrg merged in pairs / fours when lossy"""
    h = res["hist"][:4].astype(np.int64)
    tot, sc = res["totchar"], res["subchar"]
    if tot < S.SUB_KEEP or sc < 0 or h[3][sc] < 0.5 * tot:
        sc = -1
    if lossy:
        h[1] = np.repeat(h[1].reshape(-1, 2).sum(1), 2) * np.tile([1, 0], 128)
        h[2] = np.repeat(h[2].reshape(-1, 4).sum(1), 4) * np.tile([1, 0, 0, 0], 64)
    if res["delchar"] >= 0:
        h[0][res["delchar"]] = 0
    if sc >= 0:
        h[3][sc] = 0
    return [int(np.count_nonzero(x)) for x in h]


@pytest.mark.parametrize("name", NAMES)
def test_every_stream_keeps_two_symbols(name):
    """a stream of one symbol is a documented deviation of the library (it refuses to build a code):
    no shape may lead there, lossy or not"""
    for label, text in _files(name):
        res = S.scan_with_carry(text)
        for lossy in (False, True):
            assert min(_symbols_coded(res, lossy)) >= 2, (label, lossy, _symbols_coded(res, lossy))


def test_parse_reads_every_header():
    texts = [t for _, t in cases.quiva_cases()] + [t for _, t in _files("empty_entries")]
    for text in texts:
        heads = text.split(b"\n")[:-1][::6]
        assert list(S.parse(text)["well"]) == [int(h.split(b"/")[1]) for h in heads]


def _check_chain(text, plan):
    whole = S.scan_with_carry(text)
    links = S.chain(text, plan)
    tot = S.sum_results([r for _, _, r in links])
    assert np.array_equal(tot["hist"], whole["hist"]) and tot["totchar"] == whole["totchar"]
    assert tot["nentries"] == whole["nentries"]
    assert b"".join(t for t, _, _ in links) == text
    for (a, b), (_, cy, res) in zip(zip(plan, plan[1:]), links):
        for ch, e in (("delchar", "e_del"), ("subchar", "e_sub")):
            we = whole[e]
            if cy[ch] >= 0:                                  # carried in: counted from entry 0
                assert we < a or (we == a and a < b) or b == a, (plan, ch)
                assert res[e] == 0 and res[ch] == whole[ch]
            elif a <= we < b:                                # fixed inside this shard
                assert res[e] == we - a and res[ch] == whole[ch], (plan, ch)
            else:                                            # still open after it
                assert we >= b and res[e] == b - a and res[ch] == -1, (plan, ch)
        if cy["subchar"] < 0 and res["subchar"] >= 0:
            assert np.array_equal(res["sub_prefix"], whole["sub_prefix"])
    end = links[-1][1] if links[-1][1]["subchar"] >= 0 and links[-1][1]["delchar"] >= 0 else \
        S.next_carry(links[-1][1], links[-1][2])
    assert (end["delchar"], end["subchar"]) == (whole["delchar"], whole["subchar"])


@pytest.mark.parametrize("seed", range(12))
def test_random_shard_plans_add_up_to_the_whole_file(seed):
    rng = np.random.default_rng(seed)
    texts = [t for n in ("runs", "subchar_threshold", "empty_entries") for _, t in _files(n)]
    texts.append(dict(cases.quiva_cases())["lognormal_40"])
    for text in texts:
        n = S.parse(text)["n"]
        k = int(rng.integers(1, 9))
        plan = [0] + sorted(int(x) for x in rng.integers(0, n + 1, size=k - 1)) + [n]
        _check_chain(text, plan)


def test_the_cut_plans_of_every_chained_file():
    files = [t for n in ("runs", "subchar_threshold", "empty_entries") for _, t in _files(n)]
    files += [t for lab, t in _files("delchar_order") if lab in ("e4736_p32", "N_only", "no_tags")]
    files.append(dict(cases.quiva_cases())["lognormal_40"])
    seen = dict(empty_mid=False, empty_end=False, one_entry=False, only_empty=False, big_delta=False)
    for text in files:
        p = S.parse(text)
        plans = S.cut_plans(text)
        assert sorted({len(pl) - 1 for pl in plans} - {2}) == [3, 5, 8]
        for pl in plans:
            assert pl[0] == 0 and pl[-1] == p["n"] and pl == sorted(pl)
            _check_chain(text, pl)
            for k, v in S.plan_checks(p, pl).items():
                seen[k] |= v
    assert all(seen.values()), seen


# ---- what each shape claims ---------------------------------------------------------------------

def _lane_bytes(line_off, rlen, line):
    """the bytes k_qv_hist<plain> gives each lane of a warp: chunk c of the 16-byte lattice goes to
    lane c mod 32 (bytes outside the line are zeroed)"""
    skew = line_off % 16
    nchunk = (skew + rlen + 15) // 16
    lanes = [[] for _ in range(32)]
    for c in range(nchunk):
        lo, hi = max(0, c * 16 - skew), min(rlen, c * 16 - skew + 16)
        lanes[c % 32].append(line[lo:hi])
    return [np.concatenate(x) if x else np.zeros(0, np.uint8) for x in lanes]


def test_wrap_plain_claims(orc):
    for label, text in _files("wrap_plain"):
        p = S.parse(text)
        r = S.scan_with_carry(text)
        if not label.startswith("every_value"):
            assert not S.lossy_codes_nul(r), label
        if label != "many_short":
            assert r["totchar"] < S.SUB_FIX and r["delchar"] == -1 and r["subchar"] == -1, label
        assert r["hist"][:4, 0].sum() == 0 and r["hist"][:4, 10].sum() == 0
        assert all(np.count_nonzero(r["hist"][k]) >= 2 for k in range(4)), label
        if label.startswith("single_"):
            rlen, skew = (int(x) for x in label.split("_")[1:])
            assert p["n"] == 1 and p["rlen"][0] == rlen and p["line"][0, 2] % 16 == skew
            ins = p["a"][p["line"][0, 2]: p["line"][0, 2] + rlen]
            assert np.count_nonzero(ins == ins[0]) == rlen - 1
            lanes = _lane_bytes(int(p["line"][0, 2]), rlen, ins)
            if (rlen, skew) == (8192, 0):
                assert [len(x) for x in lanes] == [256] * 32
                assert [int(np.count_nonzero(x == ins[0])) for x in lanes] == [256] * 31 + [255]
            top = max(int(np.count_nonzero(x == ins[0])) for x in lanes)
            assert top >= 255, (label, top)                  # some counter reaches its wrap
        elif label.startswith("every_value"):
            assert S.lossy_codes_nul(r)
            assert orc.qv_create(orc.qv_scan(text), 1).tab[2].lens[0] > 0
            vals = [v for v in range(1, 256) if v != 10]
            for k in range(4):
                h = r["hist"][k]
                assert [int(h[v]) for v in vals] == [255 + v % 3 for v in vals]
            assert p["line"][0, 0] % 16 == int(label.split("_")[-1])
        elif label == "periodic":
            for e in range(p["n"]):
                for k, period in ((2, 8 if e % 2 == 0 else 16), (3, 8 if e % 2 == 0 else 16)):
                    o, L = int(p["line"][e, k]), int(p["rlen"][e])
                    x = p["a"][o:o + L]
                    assert np.array_equal(x[period:], x[:-period])
                    if period == 16:
                        assert not np.array_equal(x[8:16], x[:8])
            assert sorted({int(o) % 16 for o in p["line"][:, 2]}) == [0, 1, 8, 15]
        else:
            assert p["n"] == 200_000 and set(np.unique(p["rlen"])) == {1, 2, 3}
            warps = 148 * S.PLAIN_WARPS_PER_SM
            skew = p["line"][:, 0] % 16
            pad = int(((skew + p["rlen"] + 15) // 16 * 16 - p["rlen"]).sum())
            assert pad / warps > 3 * 256                      # lane 0's bin 0 wraps three times or more


def test_runs_claims():
    (_, text), = _files("runs")
    p = S.parse(text)
    r = S.scan_with_carry(text)
    assert r["e_del"] == 0 and r["delchar"] == S.DELC and r["subchar"] == S.SUBC
    assert int(np.cumsum(p["rlen"])[r["e_sub"] - 1]) < S.SUB_FIX <= int(np.cumsum(p["rlen"])[r["e_sub"]])
    for k, rc, h in ((0, S.DELC, 4), (4, S.SUBC, 5)):
        runs = []
        rounds = set()
        ends = set()
        for e in range(p["n"]):
            o, L = int(p["line"][e, k]), int(p["rlen"][e])
            x = p["a"][o:o + L]
            runs += list(S.run_lengths(x, np.array([0]), np.array([L]), rc))
            skew = o % 16
            items = np.flatnonzero(x != rc) + skew
            rounds |= set(np.bincount(items // S.ROUND, minlength=(skew + L) // S.ROUND + 1).tolist())
            if L:
                ends.add((x[0] == rc, x[-1] == rc, bool(np.all(x == rc)), bool(np.all(x != rc)), L))
        assert set(S.RUN_LENGTHS) <= set(runs) and max(runs) == 65535
        assert set(S.ROUND_ITEMS) <= rounds
        assert any(a and b and not c for a, b, c, _, _ in ends)           # rc at 0 and rlen - 1
        assert {L for _, _, c, _, L in ends if c} >= {1, 255, 256, 65535}
        assert any(d for _, _, _, d, _ in ends)
        assert r["hist"][h][255] > 0
    skews = {int(o) % 16 for o in p["line"][-60:, 0]}
    assert {0, 1, 15} <= skews


@pytest.mark.parametrize("W", GRIDS)
def test_delchar_order_claims(W):
    files = dict(S.make("delchar_order", W))
    for e in S.tag_entries(W):
        for pos in S.TAG_POSITIONS:
            text = files[f"e{e}_p{pos}"]
            p = S.parse(text)
            r = S.scan_with_carry(text)
            assert (r["e_del"], r["delchar"]) == (e, S.DEL_RARE)
            o, L = int(p["line"][e, 1]), int(p["rlen"][e])
            tags = np.flatnonzero(np.isin(p["a"][o:o + L], (ord("n"), ord("N"))))
            assert tags[0] == {"0": 0, "31": 31, "32": 32, "last": L - 1}[pos]
            dels = p["a"][p["line"][e, 0] + tags]
            assert dels[0] == S.DEL_RARE and (len(tags) == 1 or dels[1] == S.DEL_LATER)
            assert r["hist"][0][S.DEL_RARE] == 1                  # a rare symbol: a wrong pick shows
            later = [f for f in range(e + 1, p["n"]) if b"n" in text[p["line"][f, 1]:p["line"][f, 2]]]
            assert later == ([e + 3] if e + 3 < p["n"] else [])
            assert r["totchar"] < S.SUB_FIX
    assert S.scan_with_carry(files["N_only"])["delchar"] == S.DEL_RARE
    r = S.scan_with_carry(files["last_only"])
    assert r["e_del"] == r["nentries"] - 1
    r = S.scan_with_carry(files["no_tags"])
    assert r["delchar"] == -1 and r["e_del"] == r["nentries"]


def test_subchar_threshold_claims(orc):
    files = dict(S.make("subchar_threshold"))
    for t, e in ((100_000, 9), (99_999, 10), (100_001, 9)):
        text = files[f"cross_{t}"]
        p = S.parse(text)
        cum = np.cumsum(p["rlen"])
        assert cum[9] == t
        r = S.scan_with_carry(text)
        assert r["e_sub"] == e and r["subchar"] == S.SUB_A
    p = S.parse(files["inside_150000"])
    r = S.scan_with_carry(files["inside_150000"])
    assert r["e_sub"] == 1 and p["rlen"][1] == 150_000 and p["rlen"][0] < S.SUB_FIX
    r = S.scan_with_carry(files["tie"])
    sp = r["sub_prefix"]
    assert sp[S.SUB_A] == sp[S.SUB_B] == sp.max() and r["subchar"] == S.SUB_A
    text = files["prefix_decides"]
    r = S.scan_with_carry(text)
    own = S.scan_with_carry(S.shard_texts(text, [0, r["e_sub"], r["e_sub"] + 1])[1])["hist"][3]
    assert r["subchar"] == S.SUB_A and own[S.SUB_B] > own[S.SUB_A]
    heads = {}
    for t in (199_999, 200_000, 200_001):
        for below in (0, 1):
            text = files[f"half_{t}_{below}"]
            st = orc.qv_scan(text)
            assert st.totchar == t and st.subchar == S.SUB_A
            assert st.sub[S.SUB_A] == (t + 1) // 2 - below
            keep = orc.qv_create(orc.qv_scan(text)).subchar
            assert keep == (S.SUB_A if t >= S.SUB_KEEP and below == 0 else -1), (t, below)
            heads[t, below] = orc.dexqv(text)[6:8]                 # subChar in the coding header
    # the last two change the coding header, so the image shows them
    assert heads[200_000, 0] != heads[200_000, 1] and heads[200_001, 0] != heads[200_001, 1]


def test_empty_entries_claims(orc):
    files = dict(S.make("empty_entries"))
    p = S.parse(files["mixed"])
    rl = p["rlen"]
    assert rl[0] == rl[1] == rl[-1] == rl[-2] == 0
    assert any(rl[e] == rl[e + 1] == rl[e + 2] == 0 for e in range(len(rl) - 2))
    r = S.scan_with_carry(files["mixed"])
    assert int(rl[:r["e_sub"] + 1].sum()) == S.SUB_FIX and rl[r["e_sub"] + 1] == 0
    for text in files.values():
        for lossy in (False, True):
            enc = orc.dexqv(text, lossy=lossy)
            back = orc.undexqv(enc)
            assert back == text if not lossy else len(back) == len(text)
