"""bench.py's control flow at N > 1, on CPU: two gloo processes run bench.run_ours() with a stand-in
for the GPU side (identity "codec" over host memory; statistics from the oracle) and the test checks
that (a) every rank finishes, (b) all ranks issued the SAME sequence of collectives, (c) rank 0 printed
one JSON line that follows the contract.  Round 1's bench deadlocked every N > 1 run because rank 0
alone called a barrier inside its extras block; this test fails on any such asymmetry.
"""
import ctypes as C
import json
import multiprocessing as mp
import os
import socket
import sys
import time

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _view(ptr, n):
    return np.ctypeslib.as_array((C.c_uint8 * n).from_address(ptr))


class FakeCtx:
    """Same methods as dextractor_b200.lib.Context, over host memory, coding nothing: the image of
    a text is the text.  (Test infrastructure: it may use the oracle for the statistics.)"""

    def __init__(self):
        self.launches = 0
        self.last_hdr = b""

    def qv_scan_dev(self, d_text, n, carry=None):
        from dextractor_b200.lib import Stats
        from oracle import orc
        o = orc.qv_scan(bytes(_view(d_text, n)))
        st = Stats()
        h = np.ctypeslib.as_array(st.hist)
        for k, nm in enumerate(("del_", "ins", "mrg", "sub", "delrun", "subrun")):
            h[k, :] = np.ctypeslib.as_array(getattr(o, nm))
        st.totchar, st.nentries, st.delchar, st.subchar = o.totchar, o.nentries, o.delchar, o.subchar
        self.launches += 5
        return st

    def h2d(self, d_dst, data):
        _view(d_dst, len(data))[:] = np.frombuffer(data, dtype=np.uint8)
        self.last_hdr = bytes(data)

    def qv_encode_dev(self, d_text, n, coding, lossy, lwell_in, d_out, cap, want_offsets=0):
        _view(d_out, n)[:] = _view(d_text, n)
        self.launches += 3
        return n, 0, np.zeros(want_offsets + 1, dtype=np.int64)

    def _dec(self, d_in, n, d_out):
        hl = len(self.last_hdr)
        _view(d_out, n - hl)[:] = _view(d_in + hl, n - hl)
        self.launches += 2
        return n - hl

    def undexqv_dev(self, d_in, n, upper, d_out, cap, entry_off=None, well_in=0):
        return self._dec(d_in, n, d_out)

    def dexqv_dev(self, d_text, n, lossy, d_out, cap):
        self.last_hdr = b""
        _view(d_out, n)[:] = _view(d_text, n)
        return n

    def dexqv_host_ptr(self, h_text, n, lossy, h_out, cap):
        return self.dexqv_dev(h_text, n, lossy, h_out, cap)

    def undexqv_host_ptr(self, h_in, n, upper, h_out, cap):
        return self._dec(h_in, n, h_out)

    def dexta_dev(self, kind, d_text, n, d_out, cap):
        m = n // 4
        _view(d_out, m)[:] = _view(d_text, m)
        self._fa = bytes(_view(d_text, n))
        return m

    def undexta_dev(self, kind, d_in, n, width, upper, d_out, cap):
        _view(d_out, len(self._fa))[:] = np.frombuffer(self._fa, dtype=np.uint8)
        return len(self._fa)

    def launch_count(self, reset=False):
        return self.launches

    def profile(self, on):
        pass

    def profile_report(self):
        return {"k_qv_decode6": (1, 1.0), "k_qv_emit": (1, 0.5)}

    def close(self):
        pass


class FakeEnv:
    name = "fake"

    def __init__(self, world):
        import torch
        import torch.distributed as dist
        import dextractor_b200 as dx
        self.torch, self.dx = torch, dx
        self.dev = torch.device("cpu")
        self.ctx = FakeCtx()
        if world > 1:
            dist.init_process_group("gloo")

    def empty(self, n, pinned=False):
        return self.torch.zeros(int(n), dtype=self.torch.uint8)

    def make_quiva(self, seed, target, well_base=0, lengths=None):
        from dextractor_b200 import synth
        rng = np.random.default_rng(seed)
        if lengths is not None:                                  # 1/400 of the real size
            L = np.asarray(lengths)[: max(4, len(lengths) // 400)]
        else:
            L = synth.lengths_for_bytes(rng, max(int(target) // 40, 800000), 5.0)
        t = synth.make_quiva(seed, L)
        return self.torch.from_numpy(np.frombuffer(t, dtype=np.uint8).copy()), len(L), int(L.sum())

    def make_fasta(self, seed, target, arrow=False):
        from dextractor_b200 import synth
        rng = np.random.default_rng(seed)
        L = synth.lengths_for_bytes(rng, int(target) // 2000, 1.0125)
        t = synth.make_arrow(seed, L) if arrow else synth.make_fasta(seed, L)
        return self.torch.from_numpy(np.frombuffer(t, dtype=np.uint8).copy()), len(L)

    def host_bytes(self, t, n=None):
        return bytes(t[: (t.numel() if n is None else n)].numpy().tobytes())

    def equal(self, a, b):
        return bool(self.torch.equal(a, b))

    def free_cached(self):
        pass

    def sync(self):
        pass

    def timed_ms(self, fn):
        t0 = time.perf_counter(); fn()
        return (time.perf_counter() - t0) * 1e3 + 1e-3

    def clock_sampler(self):
        class S:
            def start(self): pass
            def begin(self): pass
            def end(self): pass
            def stop(self): return {"sm_mhz": 1.0, "sm_max_mhz": 1.0, "reasons": []}
        return S()

    def reference_dexqv(self, text):
        return self.ctx.last_hdr + text, "port"

    def close(self):
        pass


def _worker(rank, world, port, q, argv):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank),
                      MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    sys.path.insert(0, ROOT)
    import bench
    lines = []
    try:
        log = bench.run_ours(bench.parse_args(argv), env=FakeEnv(world), out=lines.append)
        q.put((rank, "ok", log, lines))
    except BaseException as e:                 # noqa: BLE001 -- reported to the parent
        import traceback
        q.put((rank, "error", traceback.format_exc() + repr(e), lines))


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _run(world, argv, timeout=240):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    ps = [ctx.Process(target=_worker, args=(r, world, port, q, argv)) for r in range(world)]
    for p in ps:
        p.start()
    res = {}
    t0 = time.time()
    while len(res) < world and time.time() - t0 < timeout:
        try:
            r = q.get(timeout=1.0)
            res[r[0]] = r
        except Exception:
            if not any(p.is_alive() for p in ps) and q.empty():
                break
    for p in ps:
        p.join(5)
        if p.is_alive():
            p.kill()
    return res


@pytest.mark.parametrize("extras", [True, False], ids=["default", "no_extras"])
def test_every_rank_issues_the_same_collectives(orc, extras):
    argv = ["--gpus", "2", "--steps", "2", "--warmup", "3", "--size-gb", "0.02", "--parity-mb", "8"]
    if not extras:
        argv.append("--no-extras")
    res = _run(2, argv)
    assert set(res) == {0, 1}, f"a rank never finished (deadlock?): {res}"
    for r in (0, 1):
        assert res[r][1] == "ok", res[r][2]
    assert res[0][2] == res[1][2], "ranks issued different collective sequences"
    assert len(res[0][2]) > 10
    assert res[1][3] == [] and len(res[0][3]) == 1, "exactly one JSON line, from rank 0"
    d = json.loads(res[0][3][0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches",
              "roofline", "cpu_baseline"):
        assert k in d, k
    assert d["n_gpus"] == 2 and d["cpu_baseline"] is None and d["gpu_launches"] > 0
    assert d["extra"]["sharded_parity"]["equal"] is True and d["extra"]["sharded_parity"]["shards"] == 2
    assert ("dexta_gbs" in d["extra"]) == extras


def test_single_rank_flow_and_config_matches_reference_arm(orc, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setenv("RANK", "0"); monkeypatch.setenv("WORLD_SIZE", "1"); monkeypatch.setenv("LOCAL_RANK", "0")
    lines = []
    args = bench.parse_args(["--steps", "1", "--size-gb", "0.02", "--parity-mb", "8", "--no-cpu"])
    bench.run_ours(args, env=FakeEnv(1), out=lines.append)
    d = json.loads(lines[0])
    assert d["n_gpus"] == 1 and "length_sweep" in d["extra"]
    # the two arms must print the same config object (the driver compares them)
    assert d["config"] == bench.workload_config(bench.parse_args(["--impl", "reference", "--size-gb", "0.02"]))
    assert d["roofline"]["traffic_source"] is None or "profiles/" in d["roofline"]["traffic_source"]


def test_dump_outputs_hold_the_timed_paths_image_and_text(orc, monkeypatch, tmp_path):
    """--dump-outputs: the stand-in's image is header + text and its decode is the text, both
    small enough for the sample to be the whole output.  (The stand-in gives the same output at
    every step, so this checks what is dumped and how, not from which step.)"""
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setenv("RANK", "0"); monkeypatch.setenv("WORLD_SIZE", "1"); monkeypatch.setenv("LOCAL_RANK", "0")
    with pytest.raises(SystemExit):
        bench.parse_args(["--impl", "reference", "--dump-outputs", str(tmp_path)])
    args = bench.parse_args(["--steps", "2", "--size-gb", "0.02", "--parity-mb", "8", "--no-cpu",
                             "--no-extras", "--dump-outputs", str(tmp_path)])
    bench.run_ours(args, env=FakeEnv(1), out=[].append)
    text = FakeEnv(1).make_quiva(100, 0.02e9)[0].numpy()
    files = sorted(os.listdir(tmp_path))
    assert files == ["dexqv_block_sums.npy", "dexqv_sample.npy", "lengths.npy",
                     "undexqv_block_sums.npy", "undexqv_sample.npy"]
    assert sum(os.path.getsize(tmp_path / f) for f in files) <= 64 << 20
    img, dec = np.load(tmp_path / "dexqv_sample.npy"), np.load(tmp_path / "undexqv_sample.npy")
    assert img.dtype == dec.dtype == np.float32
    assert np.array_equal(dec, text) and np.array_equal(img[len(img) - len(text):], text)
    assert np.load(tmp_path / "lengths.npy").tolist() == [len(img), len(text)]
    for name, want in (("dexqv", img), ("undexqv", dec)):
        sums = np.load(tmp_path / f"{name}_block_sums.npy")
        assert sums.dtype == np.float64 and sums.sum() == want.astype(np.int64).sum()


def test_dump_outputs_sample_large_outputs_the_same_way_every_time(monkeypatch, tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    import torch
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 1000)
    monkeypatch.setattr(bench, "DUMP_BLOCKS", 64)
    t = torch.from_numpy(np.random.default_rng(3).integers(0, 256, 100_003, dtype=np.uint8))
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), {"x": t}, rank=1, world=2)
    a = {f: np.load(tmp_path / "a" / f) for f in sorted(os.listdir(tmp_path / "a"))}
    assert sorted(a) == ["lengths_rank1.npy", "x_block_sums_rank1.npy", "x_sample_rank1.npy"]
    for f, v in a.items():
        assert np.array_equal(v, np.load(tmp_path / "b" / f)), f
    assert 250 <= len(a["x_sample_rank1.npy"]) <= 500 and len(a["x_block_sums_rank1.npy"]) <= 32
    assert a["x_block_sums_rank1.npy"].sum() == int(t.sum()) and a["lengths_rank1.npy"].tolist() == [100_003]
    # a shorter output in the same power-of-two range is sampled at the same positions
    bench.dump_outputs(str(tmp_path / "c"), {"x": t[:90_000]}, rank=1, world=2)
    c = np.load(tmp_path / "c" / "x_sample_rank1.npy")
    assert 0 < len(c) < len(a["x_sample_rank1.npy"])
    assert np.array_equal(c, a["x_sample_rank1.npy"][: len(c)])
