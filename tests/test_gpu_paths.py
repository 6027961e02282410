"""The alternative routes through the library must all give the reference's bytes: the general
(host-planned) decoders behind the device-planned fast paths, the exact two-pass index behind the
single-pass one, the byte-serial 2-bit kernels behind the vectorised ones, the older decoder
generations, and inputs built to defeat the fast paths' assumptions (line lattice, candidate
filter).  Bit-exact against the oracle."""
import numpy as np
import pytest

import dextractor_b200 as dx
from dextractor_b200 import lib as dxl
from dextractor_b200 import synth
from tests import cases
from tests.test_gpu_parity import first_diff

pytestmark = pytest.mark.gpu

QUIVA = dict(cases.quiva_cases())
FASTA = dict(cases.fasta_cases())
ARROW = dict(cases.arrow_cases())


@pytest.fixture(scope="module")
def ctx():
    c = dx.Context(0)
    yield c
    c.close()


ROUTES = [
    {},                                                  # the default routes
    {"no_fast": 1},                                      # host-planned decoders
    {"no_fast": 1, "no_spec": 1},                        # ... with a separate walk of all candidates
    {"exact_index": 1},                                  # two-pass position index
    {"exact_pack": 1},                                   # counted symbol lengths, byte-serial packer
    {"pack2": 1},                                        # input-centric vectorised 2-bit kernels (scan + bit writer)
    {"two_pass": 1},                                     # dexqv with a size pass instead of the scratch image
    {"chain_scan": 1},                                   # the multi-CTA prefix sums also on small arrays
    {"decoder": 1},                                      # sequential decode kernels
    {"decoder": 5},                                      # warp-per-entry decoder for every entry
    {"decoder": 6},                                      # lane-per-entry decoder for every entry
    {"lane_max_rlen": 3000},                             # both parallel decoders in one call
    {"decoder": 6, "no_fast": 1},                        # lane-per-entry decoder behind the host-planned path
    {"no_direct": 1},                                    # discovered entries via the scratch image + k_qv_assemble
    {"index_bulk": 4},                                   # newline index through cp.async.bulk tiles (TMA experiment)
    {"hist_mode": 1},                                    # run-length histograms: match.any groups
    {"hist_mode": 4},                                    # ... without the item queue
]


def _route_id(e):
    return "+".join(f"{k}={v}" for k, v in sorted(e.items())) or "default"


@pytest.fixture
def routed(ctx):
    """ctx with routes set by the test; every route back to its default afterwards"""
    yield ctx
    ctx.route("default")


@pytest.mark.parametrize("env", ROUTES, ids=_route_id)
def test_every_route_gives_the_same_bytes(routed, orc, env):
    ctx = routed
    for k, v in env.items():
        ctx.route(k, v)
    for name in ("lognormal_40", "edge_lengths", "long_runs", "big_well_gaps", "no_n_tags"):
        text = QUIVA[name]
        enc = orc.dexqv(text)
        assert ctx.dexqv(text) == enc, name
        assert ctx.undexqv(enc) == orc.undexqv(enc), name
    for name in ("edge_lengths", "ragged", "width_1", "big_well_gaps", "upper_and_n"):
        text = FASTA[name]
        enc = orc.dexta(text)
        assert ctx.dexta(text) == enc, name
        for width in (80, 16, 15, 7):
            assert ctx.undexta(enc, width=width) == orc.undexta(enc, width=width), (name, width)
    for name in ("edge_lengths", "odd_symbols"):
        text = ARROW[name]
        enc = orc.dexta(text, arrow=True)
        assert ctx.dexta(text, kind=dx.ARROW) == enc, name
        assert ctx.undexta(enc, kind=dx.ARROW) == orc.undexta(enc, arrow=True), name


def test_fasta_lines_off_the_lattice(ctx, orc):
    """Entries whose line layout contradicts the width of their first line: the packer's symbol
    count check must send the file down the exact path."""
    rng = np.random.default_rng(5)
    acgt = np.frombuffer(b"acgt", dtype=np.uint8)
    parts = []
    for i in range(40):
        L = int(rng.integers(200, 3000))
        seq = acgt[rng.integers(0, 4, size=L)].tobytes()
        parts.append(f">mv/{i * 3}/0_{L} RQ=0.8{i % 10}1\n".encode())
        if i % 5 == 2:                                   # first line short, the rest long
            parts.append(seq[:20] + b"\n" + seq[20:] + b"\n")
        elif i % 5 == 4:                                 # varying widths, same total as a lattice
            cut = sorted(rng.integers(1, L, size=6))
            prev = 0
            for c in cut:
                parts.append(seq[prev:c] + b"\n")
                prev = c
            parts.append(seq[prev:] + b"\n")
        else:
            parts.append(synth._wrap(np.frombuffer(seq, dtype=np.uint8), 70))
    text = b"".join(parts)
    want = orc.dexta(text)
    assert ctx.dexta(text) == want


def _zero_rich_quiva(seed, n, L):
    """ins and mrg lines dominated by one value each: the streams are full of zero bytes, which is
    what the entry-candidate filter keys on (clusters of false candidates)."""
    def hook(i, s):
        rng = np.random.default_rng(seed * 1000 + i)
        s[2][:] = np.where(rng.random(len(s[2])) < 0.995, 40, s[2])
        s[3][:] = np.where(rng.random(len(s[3])) < 0.995, 45, s[3])
    return synth.make_quiva(seed, [L] * n, stream_hook=hook)


def test_undexqv_with_many_false_candidates(ctx, orc):
    text = _zero_rich_quiva(21, 60, 6000)
    enc = orc.dexqv(text)
    assert ctx.dexqv(text) == enc
    assert ctx.undexqv(enc) == orc.undexqv(enc)


def test_undexqv_mid_size_and_long_entries(ctx, orc):
    """~40 MB with entries from 500 to 60000 positions plus a few very long ones (the decoder takes
    long entries first); decode with discovered entries, with the index, and the size query."""
    import torch
    rng = np.random.default_rng(31)
    lengths = list(synth.lengths_for_bytes(rng, 36_000_000, 5.0)) + [140000, 300, 200000, 70000]
    text = synth.make_quiva(31, lengths)
    enc = orc.dexqv(text)
    assert ctx.dexqv(text) == enc
    assert ctx.undexqv(enc) == text
    img = torch.frombuffer(bytearray(enc), dtype=torch.uint8).cuda()
    back = torch.empty(len(text) + 64, dtype=torch.uint8, device="cuda")
    offs = orc.dexqv_offsets(enc, len(lengths))
    m = ctx.undexqv_dev(img.data_ptr(), len(enc), False, back.data_ptr(), back.numel(), entry_off=offs)
    assert m == len(text) and back[:m].cpu().numpy().tobytes() == text
    assert ctx.undexqv_size_dev(img.data_ptr(), len(enc)) == len(text)


def test_dexta_mid_size_round_trip(ctx, orc):
    rng = np.random.default_rng(41)
    lengths = synth.lengths_for_bytes(rng, 30_000_000, 1.0125)
    for kind, make, arrow in ((dx.FASTA, synth.make_fasta, False), (dx.ARROW, synth.make_arrow, True)):
        text = make(41, lengths)
        enc = orc.dexta(text, arrow=arrow)
        assert ctx.dexta(text, kind=kind) == enc
        assert ctx.undexta(enc, kind=kind) == orc.undexta(enc, arrow=arrow)
        assert ctx.undexta(enc, kind=kind, width=60, upper=True) == \
            orc.undexta(enc, arrow=arrow, width=60, upper=True)


def test_output_buffer_too_small_is_an_error(ctx, orc):
    text = QUIVA["lognormal_40"]
    enc = orc.dexqv(text)
    with pytest.raises(dx.DexError) as e:
        ctx.undexqv(enc, cap=len(text) // 2)
    assert e.value.code == -2                            # DX_E_CAP


@pytest.mark.parametrize("env", [{}, {"exact_pack": 1}], ids=["vectorised", "byte_serial"])
@pytest.mark.parametrize("arrow", [False, True])
def test_batched_reads_many(routed, orc, env, arrow):
    """dx_compress_reads_dev / dx_uncompress_reads_dev (the Dazzler DB loader form, DB.c:1389-1441,
    1556-1614) on 1500 reads at ragged offsets, against Number_Read/Number_Arrow + Compress_Read and
    Uncompress_Read + Lower_/Upper_Read/Letter_Arrow of the oracle, read by read."""
    import ctypes as C
    import torch
    ctx = routed
    for k, v in env.items():
        ctx.route(k, v)
    rng = np.random.default_rng(77)
    lens = np.concatenate([np.arange(0, 40), rng.integers(1, 6000, size=1460)]).astype(np.int32)
    alpha = np.frombuffer(b"1234G0x" if arrow else b"acgtACGTnN-", dtype=np.uint8)
    reads = [alpha[rng.integers(0, len(alpha), size=int(n))].tobytes() for n in lens]
    gap = rng.integers(0, 7, size=len(lens))                      # ragged source / destination offsets
    src_off = np.concatenate([[3], 3 + np.cumsum(lens + gap)[:-1]]).astype(np.int64)
    clen = (lens + 3) // 4
    dst_off = np.concatenate([[5], 5 + np.cumsum(clen + gap)[:-1]]).astype(np.int64)
    src = bytearray(int(src_off[-1] + lens[-1] + 16))
    for o, r in zip(src_off, reads):
        src[o:o + len(r)] = r
    d_src = torch.frombuffer(src, dtype=torch.uint8).cuda()
    d_so, d_len = torch.from_numpy(src_off).cuda(), torch.from_numpy(lens).cuda()
    d_do = torch.from_numpy(dst_off).cuda()
    d_dst = torch.full((int(dst_off[-1] + clen[-1] + 16),), 0xEE, dtype=torch.uint8, device="cuda")
    kind = dx.ARROW if arrow else dx.FASTA
    ctx.compress_reads_dev(kind, d_src.data_ptr(), d_so.data_ptr(), d_len.data_ptr(), len(lens),
                           d_dst.data_ptr(), d_do.data_ptr())
    ctx.sync()
    packed = d_dst.cpu().numpy().tobytes()
    L = orc.lib()
    expect = bytearray(b"\xEE" * len(packed))
    for i, r in enumerate(reads):
        buf = C.create_string_buffer(r, len(r) + 8)
        (L.orc_number_arrow if arrow else L.orc_number_read)(buf)
        L.orc_compress_read(len(r), buf)
        expect[dst_off[i]: dst_off[i] + clen[i]] = buf.raw[: clen[i]]
    assert packed == bytes(expect)                                # also: nothing outside the payloads touched
    for upper in ([False] if arrow else [False, True]):
        d_back = torch.full((len(src),), 0xDD, dtype=torch.uint8, device="cuda")
        ctx.uncompress_reads_dev(kind, upper, d_dst.data_ptr(), d_do.data_ptr(), d_len.data_ptr(),
                                 len(lens), d_back.data_ptr(), d_so.data_ptr())
        ctx.sync()
        back = d_back.cpu().numpy().tobytes()
        want = bytearray(b"\xDD" * len(src))
        for i, r in enumerate(reads):
            buf = C.create_string_buffer(packed[dst_off[i]: dst_off[i] + clen[i]], len(r) + 8)
            L.orc_uncompress_read(len(r), buf)
            (L.orc_letter_arrow if arrow else (L.orc_upper_read if upper else L.orc_lower_read))(buf)
            want[src_off[i]: src_off[i] + len(r)] = buf.raw[: len(r)]
        assert back == bytes(want)


def test_stream_that_outgrows_its_scratch_room(ctx, orc):
    """dexqv codes every stream into a scratch image with room for a little more than 8 bits per
    symbol.  One entry made only of symbols that are rare in the file (escaped: 24 bits each) does
    not fit and must send the call down the exact route (size pass first)."""
    rng = np.random.default_rng(11)
    lengths = [int(x) for x in rng.integers(800, 1500, size=60)]
    text = synth.make_quiva(11, lengths)
    lines = text.split(b"\n")
    # entry 30: insertion and merge QVs drawn uniformly from 60 values that occur nowhere else
    k = 30 * 6
    L = len(lines[k + 3])
    rare = (rng.integers(0, 60, size=L) + 66).astype(np.uint8).tobytes()
    lines[k + 3] = rare
    lines[k + 4] = rare[::-1]
    text = b"\n".join(lines)
    enc = orc.dexqv(text)
    ctx.profile(True); ctx.profile_report()
    assert ctx.dexqv(text) == enc
    prof = ctx.profile_report(); ctx.profile(False)
    # (k_qv_compact is launched before the host has seen the overflow flag and returns at once)
    assert "k_qv_size" in prof and prof["k_qv_emit"][0] == 2, sorted(prof)
    assert ctx.undexqv(enc) == text


@pytest.mark.parametrize("width", [16, 17, 31, 32, 33, 47, 63, 64, 65, 80, 127, 128, 129, 1000])
def test_lattice_kernels_at_every_width(ctx, orc, width):
    """k_fa_pack3 works on aligned 32-byte blocks with at most one newline each and k_unpack3 on
    aligned 16-byte pieces of text: line widths around the block sizes, entry lengths around the
    widths and the 4 / 16 / 32-symbol boundaries, every payload and text alignment (the headers
    shift them), upper case and non-acgt letters, .fasta and .arrow."""
    rng = np.random.default_rng(1000 + width)
    lengths = sorted(set([1, 2, 3, 4, 5, 15, 16, 17, 31, 32, 33, 63, 64, 65, width - 1, width, width + 1,
                          2 * width - 1, 2 * width, 2 * width + 1, 3 * width + 7, 10 * width, 10 * width + 1]
                         + [int(x) for x in rng.integers(1, 40 * width + 5, size=40)]))
    lengths = [x for x in lengths if x > 0]
    rng.shuffle(lengths)
    fasta = synth.make_fasta(width, lengths, width=width, alphabet=b"acgtACGTnN")
    enc = orc.dexta(fasta)
    assert ctx.dexta(fasta) == enc
    for w in (width, 80):
        assert ctx.undexta(enc, width=w) == orc.undexta(enc, width=w), w
    assert ctx.undexta(enc, width=width, upper=True) == orc.undexta(enc, width=width, upper=True)
    arrow = synth.make_arrow(width, lengths, width=width)
    enc = orc.dexta(arrow, arrow=True)
    assert ctx.dexta(arrow, kind=dx.ARROW) == enc
    assert ctx.undexta(enc, kind=dx.ARROW, width=width) == orc.undexta(enc, arrow=True, width=width)


def test_multi_cta_scan_with_look_back(routed, orc):
    """The chain_scan route runs the multi-CTA prefix sums with tiles of 256 values, so a few hundred
    entries already span several tiles and exercise the look-back over published tile totals."""
    ctx = routed
    ctx.route("chain_scan", 1)
    rng = np.random.default_rng(77)
    fasta = synth.make_fasta(77, [int(x) for x in rng.integers(1, 300, size=1500)])
    enc = orc.dexta(fasta)
    assert ctx.dexta(fasta) == enc
    assert ctx.undexta(enc) == orc.undexta(enc)
    quiva = synth.make_quiva(78, [int(x) for x in rng.integers(200, 4000, size=700)])
    enc = orc.dexqv(quiva)
    assert ctx.dexqv(quiva) == enc
    assert ctx.undexqv(enc) == quiva


# ---- the lane-per-entry decoder (dx_qv_decode6.cu) forced on inputs of every shape -----------------

@pytest.mark.parametrize("name", sorted(QUIVA))
def test_lane_decoder_on_every_case(routed, orc, name):
    """Small files never reach the lane-per-entry kernel by themselves (the planner keeps them on the
    warp-per-entry kernel), so force it: discovered and known entry offsets, -U, lossy codings."""
    import torch
    ctx = routed
    ctx.route("decoder", 6)
    text = QUIVA[name]
    for lossy in (False, True):
        enc = orc.dexqv(text, lossy=lossy)
        want = orc.undexqv(enc)
        got = ctx.undexqv(enc)
        assert got == want, (lossy, first_diff(got, want))
    assert ctx.undexqv(enc, upper=True) == orc.undexqv(enc, upper=True)
    enc = orc.dexqv(text)
    want = orc.undexqv(enc)
    nent = text.count(b"\n") // 6
    offs = orc.dexqv_offsets(enc, nent)
    img = torch.frombuffer(bytearray(enc), dtype=torch.uint8).cuda()
    back = torch.empty(len(want) + 64, dtype=torch.uint8, device="cuda")
    m = ctx.undexqv_dev(img.data_ptr(), len(enc), False, back.data_ptr(), back.numel(), entry_off=offs)
    got = back[:m].cpu().numpy().tobytes()
    assert got == want, first_diff(got, want)


@pytest.mark.parametrize("seed", range(24))
def test_lane_decoder_fuzz(routed, orc, seed):
    from tests import fuzz
    ctx = routed
    ctx.route("decoder", 6)
    text, _ = fuzz.fuzz_quiva(seed)
    for lossy in (False, True):
        enc = orc.dexqv(text, lossy=lossy)
        got, want = ctx.undexqv(enc), orc.undexqv(enc)
        assert got == want, (lossy, first_diff(got, want))


def test_lane_decoder_on_a_truncated_image_fails_cleanly(routed, orc):
    ctx = routed
    ctx.route("decoder", 6)
    enc = orc.dexqv(QUIVA["lognormal_40"])
    for cut in (len(enc) - 1, len(enc) - 40, len(enc) // 2):
        with pytest.raises(dx.DexError):
            ctx.undexqv(enc[:cut])


def test_fasta_line_too_long_after_the_first_line(ctx, orc):
    """dexta.c:168-172 refuses any line of more than MAX_BUFFER-2 = 99998 characters, not only the
    first one of an entry; a line of exactly 99998 is fine."""
    rng = np.random.default_rng(3)
    acgt = np.frombuffer(b"acgt", dtype=np.uint8)

    def seq(n):
        return acgt[rng.integers(0, 4, size=n)].tobytes()

    def text(long_len):
        return (b">mv/1/0_100 RQ=0.851\n" + seq(60) + b"\n" + seq(40) + b"\n" +
                b">mv/5/0_%d RQ=0.800\n" % (70 + long_len + 10) + seq(70) + b"\n" + seq(long_len) + b"\n" +
                seq(10) + b"\n" + b">mv/9/0_80 RQ=0.700\n" + seq(80) + b"\n")

    ok = text(99998)
    assert ctx.dexta(ok) == orc.dexta(ok)
    with pytest.raises(dx.DexError) as e:
        ctx.dexta(text(99999))
    assert e.value.code == -6                            # DX_E_TOOLONG
    with pytest.raises(orc.OracleError) as e2:
        orc.dexta(text(99999))
    assert e2.value.code == -6


@pytest.mark.parametrize("chunk", [65536, 262144, 1 << 20])
def test_pipelined_host_decode_on_small_windows(routed, orc, chunk):
    """dx_undexqv_host as a pipeline of windows (chunked copies in, window-wise discovery / decode /
    assemble, chunked copies out): forced onto a few-MB file by a small window size.  Entries run over
    window boundaries; a window smaller than an entry sends the call to the plain path."""
    ctx = routed
    rng = np.random.default_rng(17)
    lengths = [int(x) for x in synth.lengths_for_bytes(rng, 6_000_000, 5.0)] + [300, 61000, 5, 12000]
    text = synth.make_quiva(17, lengths, max_well_delta=700)
    enc = orc.dexqv(text)
    want = orc.undexqv(enc)
    ctx.route("pipe_chunk", chunk)
    for upper in (False, True):
        got = ctx.undexqv(enc, upper=upper, cap=len(want) + 4096)
        exp = want if not upper else orc.undexqv(enc, upper=True)
        assert got == exp, (upper, first_diff(got, exp))
    ctx.route("serial_io", 1)
    assert ctx.undexqv(enc, cap=len(want) + 4096) == want


_scan_inputs: list = []


def _scan_shape_inputs():
    """(label, text, restatement) of the files the counting modes are checked on, computed once"""
    import torch
    from tests import fuzz
    from tests import scan_shapes as S
    if not _scan_inputs:
        texts = [(f"fuzz_{seed}", fuzz.fuzz_quiva(seed)[0]) for seed in (0, 3, 5, 8, 13, 21)]
        texts += [(n, QUIVA[n]) for n in ("long_runs", "late_n", "lognormal_40", "no_n_tags")]
        W = torch.cuda.get_device_properties(0).multi_processor_count * S.HIST_WARPS_PER_SM
        for name in sorted(S.SHAPES) + ["delchar_order"]:
            texts += [(f"{name}/{lab}", t) for lab, t in S.make(name, W if name == "delchar_order" else None)]
        _scan_inputs.extend((lab, t, S.scan_with_carry(t)) for lab, t in texts)
    return _scan_inputs


@pytest.mark.parametrize("mode", [0, 1, 2, 3, 4])
def test_run_histogram_counting_modes(ctx, orc, mode):
    """k_qv_hist_run counts a batch of (symbol, run length) items in five ways (route hist_mode):
    every one must give Histogram_Seqs / Histogram_Runs' numbers (QV.c:702-724) on files of random
    shape -- run densities 0 ... 0.995, runs beyond 255, run characters that appear late -- and on
    the crafted files of tests/scan_shapes.py, whose inputs sit on the boundaries of the pass-1
    kernels (counter wraps, queue rounds, the first tag past the first wave of warps, the 100 000
    crossing, empty entries).  sub_prefix is checked against the numpy restatement."""
    import torch
    ctx.route("default")
    ctx.route("hist_mode", mode)
    try:
        for label, text, want in _scan_shape_inputs():
            t = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
            st = ctx.qv_scan_dev(t.data_ptr(), len(text))
            ref = orc.qv_scan(text)
            assert (st.delchar, st.subchar, st.totchar) == (ref.delchar, ref.subchar, ref.totchar), label
            assert st.nentries == ref.nentries == want["nentries"], label
            for k, nm in enumerate(["del_", "ins", "mrg", "sub"]):
                assert list(st.hist[k]) == list(getattr(ref, nm)), (label, nm)
            assert [x + 1 for x in st.hist[4]] == list(ref.delrun), label
            assert [x + 1 for x in st.hist[5]] == list(ref.subrun), label
            assert all(st.hist[k][0] == 0 and st.hist[k][10] == 0 for k in range(4)), label
            assert list(st.sub_prefix) == [int(x) for x in want["sub_prefix"]], label
    finally:
        ctx.route("default")


def test_a_shard_that_starts_far_behind_its_predecessor_decodes_in_place(ctx, orc):
    """A shard's image starts with the delta of its first well against the predecessor's last well:
    thousands of 0xff bytes when the wells are far apart (bench.py gives every rank its own well
    range).  Those bytes can only be delta bytes -- there is no stream in front of them -- so the
    in-place form of the discovered decode must take them in its stride: one decode launch, no
    k_qv_assemble, and the text of the shard with the right well numbers."""
    import torch
    rng = np.random.default_rng(31)
    lengths = [int(x) for x in rng.integers(300, 6000, size=120)]
    text = synth.make_quiva(31, lengths)
    # move every well up by 2 000 000: the first delta (against well_in = 7) is 7 843 x 0xff + one byte
    lines = text.split(b"\n")
    for e in range(len(lengths)):
        f = lines[6 * e].split(b"/")
        f[1] = str(int(f[1]) + 2_000_000).encode()
        lines[6 * e] = b"/".join(f)
    text = b"\n".join(lines)
    t = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    st = ctx.qv_scan_dev(t.data_ptr(), len(text))
    cd = dxl.make_coding(st, False)
    hdr = b"\xaa\x55" + dxl.write_coding(cd, text[: text.index(b"/", 1)])
    enc = torch.zeros(len(text) + 65536, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    ctx.h2d(enc.data_ptr(), hdr)
    body, lastw, _ = ctx.qv_encode_dev(t.data_ptr(), len(text), cd, False, 7, enc.data_ptr() + len(hdr),
                                       enc.numel() - len(hdr))
    n = len(hdr) + body
    img = enc[:n].cpu().numpy().tobytes()
    assert img[len(hdr): len(hdr) + 7000] == b"\xff" * 7000
    back = torch.zeros(len(text) + 64, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    ctx.profile(True); ctx.profile_report()
    m = ctx.undexqv_dev(enc.data_ptr(), n, False, back.data_ptr(), back.numel(), well_in=7)
    prof = ctx.profile_report(); ctx.profile(False)
    assert back[:m].cpu().numpy().tobytes() == text
    assert "k_qv_assemble" not in prof and prof["k_qv_decode5_spec"][0] == 1, sorted(prof)


def test_headers_outside_the_usual_range_still_decode(ctx, orc):
    """The in-place form of the discovered decode lays the text out for candidates whose fields look
    like real headers (region score <= 1000, start below 16 M).  Nothing in the format says so: an
    entry with RQ=0.2000, one starting at base 20 000 000 and one with a six-digit score must come
    out exactly as the reference writes them (the call takes the scratch-image form for this file)."""
    rng = np.random.default_rng(41)
    lengths = [int(x) for x in rng.integers(200, 5000, size=90)]
    text = synth.make_quiva(41, lengths)
    lines = text.split(b"\n")

    def rewrite(e, beg=None, qv=None):
        f = lines[6 * e].split(b"/")
        span, rq = f[2].split(b" RQ=0.")
        b0, e0 = (int(x) for x in span.split(b"_"))
        if beg is not None:
            e0, b0 = beg + (e0 - b0), beg
        if qv is not None:
            rq = str(qv).encode()
        f[2] = b"%d_%d RQ=0.%s" % (b0, e0, rq)
        lines[6 * e] = b"/".join(f)

    rewrite(7, qv=2000)
    rewrite(30, beg=20_000_000)
    rewrite(55, qv=654321)
    text = b"\n".join(lines)
    enc = orc.dexqv(text)
    assert ctx.dexqv(text) == enc
    ctx.profile(True); ctx.profile_report()
    back = ctx.undexqv(enc)
    prof = ctx.profile_report(); ctx.profile(False)
    assert back == orc.undexqv(enc) == text
    assert "k_qv_assemble" in prof, sorted(prof)          # not in place: the layout did not hold


def test_every_header_outside_the_usual_range(ctx, orc):
    """... and a file in which NO entry is in that range (every score above 1000): the assumed layout is
    empty, and an empty layout must not count as confirmed (found by tests/hostfuzz/fz_chain.cpp: "all
    kept candidates pass" is vacuously true when nothing was kept)."""
    rng = np.random.default_rng(43)
    lengths = [int(x) for x in rng.integers(100, 3000, size=50)]
    text = synth.make_quiva(43, lengths)
    lines = text.split(b"\n")
    for e in range(len(lengths)):
        head, rq = lines[6 * e].split(b" RQ=0.")
        lines[6 * e] = head + b" RQ=0." + str(1500 + e).encode()
    text = b"\n".join(lines)
    enc = orc.dexqv(text)
    assert ctx.dexqv(text) == enc
    assert ctx.undexqv(enc) == text
