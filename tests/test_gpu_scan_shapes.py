"""Pass 1 of the QV coder on the crafted files of tests/scan_shapes.py: the images of every file
against the oracle, the empty entries through the decoders, and the carried scan of tools/dexqv_mg.c
replayed call for call on one GPU over shards cut around the entries that fix the run characters.
The whole-file statistics of the same files are checked count for count, on every hist_mode, by
tests/test_gpu_paths.py::test_run_histogram_counting_modes."""
import numpy as np
import pytest

import dextractor_b200 as dx
from dextractor_b200 import lib as dxl
from tests import cases
from tests import scan_shapes as S
from tests.test_gpu_parity import first_diff

pytestmark = pytest.mark.gpu

GUARD = 4096
DX_E_CODING = -11


@pytest.fixture(scope="module")
def ctx():
    c = dx.Context(0)
    yield c
    c.close()


@pytest.fixture
def routed(ctx):
    """ctx with routes set by the test; every route back to its default afterwards"""
    yield ctx
    ctx.route("default")


def _grid_warps():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count * S.HIST_WARPS_PER_SM


def _files(name):
    return S.make(name, _grid_warps() if name == "delchar_order" else None)


def _device(data: bytes, extra: int = 64):
    """the bytes in a fresh (16-byte aligned) device buffer"""
    import torch
    t = torch.zeros(len(data) + extra, dtype=torch.uint8, device="cuda")
    if data:
        t[: len(data)] = torch.frombuffer(bytearray(data), dtype=torch.uint8).cuda()
    torch.cuda.synchronize()
    return t


@pytest.mark.parametrize("name", sorted(S.SHAPES) + ["delchar_order"])
def test_images_of_the_shapes(ctx, orc, name):
    """every file, lossy and not, byte for byte; where lossy coding rounds a QV to NUL (ins 1, mrg
    1..3) the oracle codes it and the library refuses the coding, as it refuses NUL itself"""
    for label, text in _files(name):
        nul = S.lossy_codes_nul(S.scan_with_carry(text))
        for lossy in (False, True):
            want = orc.dexqv(text, lossy=lossy)
            if lossy and nul:
                with pytest.raises(dx.DexError) as e:
                    ctx.dexqv(text, lossy=lossy)
                assert e.value.code == DX_E_CODING, label
                continue
            got = ctx.dexqv(text, lossy=lossy)
            assert got == want, (label, lossy, first_diff(got, want))


@pytest.mark.parametrize("env", [{}, {"no_fast": 1}, {"decoder": 5}, {"decoder": 6}],
                         ids=["default", "no_fast", "decoder5", "decoder6"])
def test_empty_entries_decode(routed, orc, env):
    """entries of 0 positions through entry discovery and the decoders, and with the oracle's entry
    offsets"""
    ctx = routed
    for k, v in env.items():
        ctx.route(k, v)
    for label, text in _files("empty_entries"):
        for lossy in (False, True):
            enc = orc.dexqv(text, lossy=lossy)
            want = orc.undexqv(enc)
            got = ctx.undexqv(enc)
            assert got == want, (label, lossy, first_diff(got, want))
            nent = S.parse(text)["n"]
            offs = orc.dexqv_offsets(enc, nent)
            assert len(offs) == nent + 1
            img = _device(enc)
            back = _device(b"", len(want) + GUARD)
            m = ctx.undexqv_dev(img.data_ptr(), len(enc), False, back.data_ptr(), len(want) + GUARD,
                                entry_off=offs)
            got = back[:m].cpu().numpy().tobytes()
            assert got == want, (label, lossy, first_diff(got, want))


# ---- the carried scan of dexqv_mg on one GPU ------------------------------------------------------

def _carry_struct(cy: dict) -> dxl.Carry:
    c = dxl.Carry()
    c.delchar, c.subchar, c.totchar = cy["delchar"], cy["subchar"], cy["totchar"]
    for k in range(256):
        c.sub[k] = int(cy["sub"][k])
    return c


def _stats_of(st: dxl.Stats) -> dict:
    return dict(hist=np.ctypeslib.as_array(st.hist).copy(), totchar=st.totchar, nentries=st.nentries,
                delchar=st.delchar, subchar=st.subchar,
                sub_prefix=np.ctypeslib.as_array(st.sub_prefix).copy())


def _replay(ctx, text, plan, encs, wholes):
    """tools/dexqv_mg.c:176-236 for the shards of `plan`, one after the other on one context"""
    shards = S.shard_texts(text, plan)
    bufs = [_device(t) for t in shards]
    ref = S.chain(text, plan)
    cy = S.empty_carry()
    stats, lastw = [], []
    for r, (t, buf) in enumerate(zip(shards, bufs)):
        open_ = cy["delchar"] < 0 or cy["subchar"] < 0
        ctx.profile(True); ctx.profile_report()
        st = ctx.qv_scan_dev(buf.data_ptr(), len(t), None if r == 0 else _carry_struct(cy))
        prof = ctx.profile_report(); ctx.profile(False)
        lastw.append(ctx.qv_last_well())
        got, (_, rcy, want) = _stats_of(st), ref[r]
        assert (rcy["delchar"], rcy["subchar"]) == (cy["delchar"], cy["subchar"])
        what = (plan, r)
        assert np.array_equal(got["hist"], want["hist"]), (what, np.argwhere(got["hist"] != want["hist"]))
        for k in ("totchar", "nentries", "delchar", "subchar"):
            assert got[k] == want[k], (what, k)
        assert np.array_equal(got["sub_prefix"], want["sub_prefix"]), what
        nent = want["nentries"]
        assert ("k_find_delchar" in prof) == (cy["delchar"] < 0 and nent > 0), (what, sorted(prof))
        assert ("k_probe_sub" in prof) == (cy["subchar"] < 0), (what, sorted(prof))
        wells = S.parse(t)["well"]
        assert lastw[-1] == (int(wells[-1]) if nent else 0), what
        stats.append(got)
        if open_:
            cy = dict(delchar=got["delchar"], subchar=got["subchar"], totchar=cy["totchar"] + got["totchar"],
                      sub=got["sub_prefix"])
    whole = wholes["stats"]
    tot = dxl.Stats()
    h = np.ctypeslib.as_array(tot.hist)
    h[:] = sum(s["hist"] for s in stats)
    tot.totchar = sum(s["totchar"] for s in stats)
    tot.nentries = sum(s["nentries"] for s in stats)
    tot.delchar, tot.subchar = cy["delchar"], cy["subchar"]
    for k, nm in enumerate(("del_", "ins", "mrg", "sub", "delrun", "subrun")):
        assert list(h[k] + (1 if k >= 4 else 0)) == list(getattr(whole, nm)), (plan, nm)
    assert (tot.totchar, tot.nentries) == (whole.totchar, whole.nentries)
    prefix = text[: text.index(b"/", 1)]
    for lossy in (False, True):
        cd = dxl.make_coding(tot, lossy)
        hdr = b"\xaa\x55" + dxl.write_coding(cd, prefix)
        bodies = []
        for r, (t, buf) in enumerate(zip(shards, bufs)):
            lwell_in = next((lastw[q] for q in range(r - 1, -1, -1) if stats[q]["nentries"] > 0), 0)
            nent = stats[r]["nentries"]
            cap = 3 * len(t) + 200000
            out = _device(b"", cap)
            m, lw, offs = ctx.qv_encode_dev(buf.data_ptr(), len(t), cd, lossy, lwell_in, out.data_ptr(), cap,
                                            want_offsets=nent)
            body = out[:m].cpu().numpy().tobytes()
            bodies.append(body)
            if nent == 0:
                assert m == 0, (plan, r)
                continue
            assert lw == lastw[r]
            img = _device(hdr + body)
            dec, bounds = wholes["dec", lossy]
            want = dec[int(bounds[plan[r]]): int(bounds[plan[r + 1]])]
            back = _device(b"", len(want) + GUARD)
            k = ctx.undexqv_dev(img.data_ptr(), len(hdr) + m, False, back.data_ptr(), len(want) + GUARD,
                                entry_off=offs + len(hdr), well_in=lwell_in)
            got = back[:k].cpu().numpy().tobytes()
            assert got == want, (plan, r, lossy, first_diff(got, want))
        image = hdr + b"".join(bodies)
        assert image == encs[lossy], (plan, lossy, first_diff(image, encs[lossy]))


def _chained_files():
    W = _grid_warps()
    out = [("runs", t) for _, t in _files("runs")]
    keep = {f"e{e}_p{p}" for e in (0, W, 2 * W + 5) for p in ("31", "32")} | {"N_only", "last_only", "no_tags"}
    out += [(f"delchar_order/{lab}", t) for lab, t in _files("delchar_order") if lab in keep]
    out += [(f"subchar_threshold/{lab}", t) for lab, t in _files("subchar_threshold")]
    out += [(f"empty_entries/{lab}", t) for lab, t in _files("empty_entries")]
    out.append(("lognormal_40", dict(cases.quiva_cases())["lognormal_40"]))
    return out


@pytest.mark.parametrize("group", ["runs", "delchar_order", "subchar_threshold", "empty_entries",
                                   "lognormal_40"])
def test_carried_scan_chain(ctx, orc, group):
    """Shards cut at every boundary around e_del / e_sub (every boundary of small files), into 3, 5
    and 8 shards with empty and one-entry shards, and in front of a well delta >= 255: every shard's
    statistics equal the restatement from its carry; the sums equal the whole file's scan; header and
    bodies are the oracle's image; each [header][shard body] decodes to the shard; and a shard launches
    k_find_delchar / k_probe_sub only while its character is open."""
    for label, text in _chained_files():
        if label.split("/")[0] != group:
            continue
        encs = {lossy: orc.dexqv(text, lossy=lossy) for lossy in (False, True)}
        wholes = {"stats": orc.qv_scan(text)}
        for lossy in (False, True):
            dec = orc.undexqv(encs[lossy])
            wholes["dec", lossy] = dec, np.append(S.parse(dec)["hdr"], len(dec))
        for plan in S.cut_plans(text):
            _replay(ctx, text, plan, encs, wholes)
