#!/usr/bin/env python
"""bench.py -- DEXTRACTOR compression hot path on B200: dexqv/undexqv (and dexta/undexta) GB/s of
uncompressed data, with the HBM roofline of the dominant kernel and the reference's CPU tools
timed on the same box.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--size-gb G]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch: dexqv (statistics scan, code construction,
encode) of a synthetic .quiva shard followed by undexqv of the result, the decoder finding the
entries of the image by itself as a file-to-file tool must.  Workload = BASELINE.json configs[1]:
a 2 GB RS II-like .quiva per GPU (weak scaling: every rank holds its own 2 GB shard of one logical
file; the ranks exchange only the histograms and a few integers).

value   uncompressed GB/s summed over both directions (2*U / t), inputs resident in HBM, timed
        with CUDA events on the library's stream, max over ranks.
e2e     the same step through the host-buffer C ABI (dx_dexqv_host / dx_undexqv_host): pinned
        host -> device copies of the inputs and device -> host copies of the results included.

--dump-outputs DIR writes what the last timed step produced (see dump_outputs) so that two builds
can be compared output for output; the inputs are seeded, so equal arguments give equal inputs.

Control flow rule (round 1 died of breaking it): every collective is issued from the top level of
run_ours() through `Comm`, by every rank, unconditionally.  Nothing under `if rank == 0` may
synchronise with other ranks; rank-local timing uses Env.sync() only.  tests/test_bench_flow.py
runs this file's flow in two gloo processes with a stand-in device and compares the ranks'
collective sequences.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GB = 1e9
METRIC = "dexqv+undexqv uncompressed GB/s"


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks during the timed region (B200_PROFILING.md recipe).  The process is started
    BEFORE the warm-up steps: NVML initialisation takes ~50 ms of driver time during which kernel
    launches stall, as long as the whole timed region of a default run -- started at the timed region
    it returned no sample and doubled the measured step.  Rows carry their arrival time; the ones
    inside the timed region are reported, or (region shorter than the sampling period) the ones
    since the start of the warm-up, i.e. under the same load."""

    def __init__(self, index, enabled=True):
        # index: one GPU, or a comma-separated list (rank 0 of a multi-GPU run samples every GPU of the
        # job with ONE nvidia-smi; a sampler per rank made eight NVML clients poll the driver at once
        # and stretched the 8-GPU step by over a millisecond)
        self.rows, self.proc, self.index, self.enabled = [], None, index, enabled
        self.t0 = self.t1 = None

    def start(self):
        if not self.enabled:
            return
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def begin(self):
        self.t0 = time.time()

    def end(self):
        self.t1 = time.time()

    def stop(self):
        if not self.enabled:
            return None
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        if self.t1 is None:
            self.t1 = time.time()
        time.sleep(0.12)
        self.proc.terminate()
        rows = [r for t, r in self.rows if self.t0 is not None and self.t0 <= t <= self.t1 + 0.05]
        window = "timed region"
        if not rows:
            rows = [r for t, r in self.rows if t <= self.t1 + 0.05]
            window = "warm-up + timed region (the timed region is shorter than the sampling period)"
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for k, nm in enumerate(names):
                    if r[3 + k].lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_min_mhz": sm[0] if sm else None,
                "sm_max_mhz": mx or None, "samples": len(sm), "gpus": self.index, "window": window,
                "reasons": sorted(reasons)}


def workload_config(args):
    """The same object in both arms (the driver compares them)."""
    return {"workload": "BASELINE.json configs[1]: dexqv/undexqv on a synthetic 2 GB RS II-like "
                        ".quiva per GPU (5 QV streams)",
            "uncompressed_bytes_per_gpu": int(args.size_gb * GB), "shards": args.gpus,
            "l2": "inputs (2 GB) exceed the 126 MB L2; no explicit flush"}


# --dump-outputs: per output and rank, a seeded sample of up to 4 Mi bytes (float32, 16 MB) and the
# exact sums of up to 1 Mi contiguous blocks (float64, 8 MB), divided by the number of ranks: two
# outputs stay under 64 MB in all.  The sample shows where bytes differ; the block sums cover every
# byte.  The sample positions are drawn from [0, next power of two >= length) and those past the
# end dropped, so outputs of different lengths in the same power-of-two range are sampled at the
# same positions, and their samples agree element by element up to the shorter one.
DUMP_SAMPLE, DUMP_BLOCKS = 1 << 22, 1 << 20


def dump_outputs(outdir, outputs, rank, world):
    """outputs: {name: 1-D uint8 tensor}.  Writes <name>_sample.npy, <name>_block_sums.npy and
    lengths.npy (the byte length of each output, in order) into outdir; with several ranks every
    file name ends in _rank<r>."""
    import numpy as np
    import torch
    os.makedirs(outdir, exist_ok=True)
    tag = f"_rank{rank}" if world > 1 else ""
    lengths = []
    for name, t in outputs.items():
        n = t.numel()
        lengths.append(n)
        k = DUMP_SAMPLE // world
        if n <= k:
            pos = np.arange(n)
        else:
            # k draws below the power of two, repeats merged (a permutation of the range, as
            # choice(replace=False) makes for small ranges, would cost up to 1 GB of host memory)
            top = 1 << (n - 1).bit_length()
            pos = np.unique(np.random.default_rng(rank).integers(0, top, k))
            pos = pos[pos < n]
        sample = t[torch.from_numpy(pos).to(t.device)].to(torch.float32).cpu().numpy()
        b = max(1, -(-n // (DUMP_BLOCKS // world)))          # block length: at most that many blocks
        full = t[: n - n % b].view(-1, b)
        sums = [full[i: i + 4096].to(torch.int32).sum(1).cpu().numpy() for i in range(0, full.shape[0], 4096)]
        if n % b:
            sums.append(np.array([int(t[n - n % b:].to(torch.int32).sum())]))
        np.save(os.path.join(outdir, f"{name}_sample{tag}.npy"), sample)
        np.save(os.path.join(outdir, f"{name}_block_sums{tag}.npy"),
                np.concatenate(sums).astype(np.float64) if sums else np.zeros(0))
    np.save(os.path.join(outdir, f"lengths{tag}.npy"), np.array(lengths, dtype=np.float64))


# ------------------------------------------------------------------------------------------------
#  reference arm: the reference's own CPU tools (oracle/_ref), single threaded like the reference
# ------------------------------------------------------------------------------------------------

_SAMPLES = {}


def _sample_text(kind: str, sample_mb: float, seed: int) -> bytes:
    import numpy as np
    from dextractor_b200 import synth
    key = (kind, sample_mb, seed)
    if key not in _SAMPLES:                     # generating the text is not part of the timing
        rng = np.random.default_rng(seed)
        if kind == "quiva":
            L = synth.lengths_for_bytes(rng, int(sample_mb * 1e6), 5.0)
            _SAMPLES[key] = synth.make_quiva(seed, L)
        else:
            L = synth.lengths_for_bytes(rng, int(sample_mb * 1e6), 1.0125)
            _SAMPLES[key] = synth.make_arrow(seed, L) if kind == "arrow" else synth.make_fasta(seed, L)
    return _SAMPLES[key]


_TOOLS = {"quiva": ("dexqv", "undexqv"), "fasta": ("dexta", "undexta"), "arrow": ("dexar", "undexar")}


def cpu_reference_sample(sample_mb: float, seed: int = 1, nproc: int = 1, kind: str = "quiva"):
    """compress + decompress a bounded sample with the reference binaries; returns timings.
    nproc > 1: that many independent copies at once (the reference has no threads; independent
    files are the only way it uses more cores), throughput = nproc * bytes / wall."""
    from oracle import orc
    text = _sample_text(kind, sample_mb, seed)
    enc_tool, dec_tool = _TOOLS[kind]
    if orc.have_ref():
        if nproc > 1:
            enc, t_enc = orc.ref_tool_parallel(enc_tool, text, nproc)
            back, t_dec = orc.ref_tool_parallel(dec_tool, enc, nproc)
        else:
            enc, t_enc = orc.ref_tool(enc_tool, text, taskset=0)
            back, t_dec = orc.ref_tool(dec_tool, enc, taskset=0)
        ref = "reference"
    else:                                   # the C restatement (oracle/dx_oracle.c)
        nproc = 1
        fe, fd = {"quiva": (orc.dexqv, orc.undexqv),
                  "fasta": (orc.dexta, orc.undexta),
                  "arrow": (lambda t: orc.dexta(t, arrow=True),
                            lambda d: orc.undexta(d, arrow=True))}[kind]
        t0 = time.perf_counter(); enc = fe(text); t_enc = time.perf_counter() - t0
        t0 = time.perf_counter(); back = fd(enc); t_dec = time.perf_counter() - t0
        ref = "port"
    if kind != "arrow":                     # SN=%.2f headers pass through a float (SURVEY App. B.7)
        assert back == text
    return {"bytes": len(text) * nproc, "t_enc": t_enc, "t_dec": t_dec, "kind": ref,
            "compressed": len(enc) * nproc, "cores": nproc, "sample_bytes": len(text)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample_mb = args.ref_sample_mb
    nproc = max(1, (os.cpu_count() or 1) if args.ref_cores <= 0 else args.ref_cores)
    times = []
    for i in range(args.warmup + args.steps):
        r = cpu_reference_sample(sample_mb, seed=1, nproc=nproc)
        if i >= args.warmup:
            times.append(r)
    t = sum(x["t_enc"] + x["t_dec"] for x in times) / len(times)
    U = times[0]["bytes"]
    nproc = times[0]["cores"]
    val = 2 * U / t / GB
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "GB/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": val, "unit": "GB/s", "cores": nproc, "kind": times[0]["kind"],
                         "sample": f"{nproc} x {times[0]['sample_bytes']/1e6:.0f} MB synthetic .quiva per "
                                   f"step, dexqv then undexqv (reference binaries, one single-threaded "
                                   f"process per core on independent copies, files on /dev/shm)",
                         "dexqv_gbs": U / (sum(x['t_enc'] for x in times) / len(times)) / GB,
                         "undexqv_gbs": U / (sum(x['t_dec'] for x in times) / len(times)) / GB,
                         "host_cores_available": os.cpu_count()},
        "e2e": {"value": val, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
#  our arm: the device-facing pieces behind Env (so the flow below can be exercised on CPU/gloo)
# ------------------------------------------------------------------------------------------------

class Comm:
    """Every inter-rank operation of the bench.  `log` records what was issued, in order."""

    def __init__(self, world, rank, device):
        self.world, self.rank, self.device, self.log = world, rank, device, []

    def barrier(self):
        self.log.append("barrier")
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()

    def all_gather_i64(self, row):
        """row: int64 tensor on the communication device -> [world, len(row)] tensor there"""
        import torch
        import torch.distributed as dist
        self.log.append(f"all_gather:{row.numel()}")
        if self.world == 1:
            return row.view(1, -1).clone()
        out = torch.empty(self.world * row.numel(), dtype=torch.int64, device=row.device)
        dist.all_gather_into_tensor(out, row)
        return out.view(self.world, -1)

    def gather_rows(self, row):
        """row: int64 numpy array on the host -> [world, len(row)] numpy array on every rank.  With one
        rank there is nothing to exchange and nothing leaves the host; otherwise the rows go through
        the communication device (NCCL all-gather on device buffers)."""
        import numpy as np
        import torch
        if self.world == 1:
            self.log.append(f"all_gather:{row.size}")
            return np.asarray(row, dtype=np.int64).reshape(1, -1)
        rows = self.all_gather_i64(torch.from_numpy(row).to(self.device))
        return rows.cpu().numpy()

    def all_reduce(self, values, op="max", dtype=None):
        """list of numbers -> list reduced over the ranks"""
        import torch
        import torch.distributed as dist
        self.log.append(f"all_reduce:{op}:{len(values)}")
        dtype = dtype or torch.float64
        t = torch.tensor(list(values), dtype=dtype, device=self.device)
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)
        return [x for x in t.tolist()]

    def broadcast_i64(self, values, src=0):
        import torch
        import torch.distributed as dist
        self.log.append(f"broadcast:{len(values)}")
        t = torch.tensor(list(values), dtype=torch.int64, device=self.device)
        if self.world > 1:
            dist.broadcast(t, src)
        return [int(x) for x in t.tolist()]

    def gather_bytes(self, blob):
        """uint8 tensor on the communication device (any length per rank) -> list of per-rank host
        bytes on EVERY rank (an all-gather of the sizes, then one of the padded blobs)"""
        import torch
        import torch.distributed as dist
        sizes = self.all_gather_i64(torch.tensor([blob.numel()], dtype=torch.int64, device=self.device))
        sizes = [int(x) for x in sizes.view(-1).tolist()]
        self.log.append("all_gather_bytes")
        if self.world == 1:
            return [bytes(blob.cpu().numpy().tobytes())]
        m = max(sizes)
        pad = torch.zeros(m, dtype=torch.uint8, device=self.device)
        pad[: blob.numel()] = blob
        out = torch.empty(self.world * m, dtype=torch.uint8, device=self.device)
        dist.all_gather_into_tensor(out, pad)
        h = out.cpu().numpy()
        return [bytes(h[r * m: r * m + sizes[r]].tobytes()) for r in range(self.world)]


class CudaEnv:
    """The B200 side: torch for buffers / NCCL, libdexb200.so for every codec call."""
    name = "cuda"

    def __init__(self, local, world):
        import torch
        import dextractor_b200 as dx
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
        self.torch, self.dx = torch, dx
        torch.cuda.set_device(local)
        self.dev = torch.device("cuda", local)
        self.local, self.world = local, world
        if world > 1:
            import torch.distributed as dist
            # stdout carries ONE JSON line: keep NCCL's own banner out of it
            if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
                os.environ.pop("NCCL_DEBUG")
            dist.init_process_group("nccl", device_id=self.dev)
        self.ctx = dx.Context(local)
        self.ext = torch.cuda.ExternalStream(self.ctx.stream, device=self.dev)

    # buffers -------------------------------------------------------------------------------
    def empty(self, n, pinned=False):
        t = self.torch.empty(int(n), dtype=self.torch.uint8, device="cpu" if pinned else self.dev)
        return t.pin_memory() if pinned else t

    def make_quiva(self, seed, target, well_base=0, lengths=None):
        from dextractor_b200 import synth_torch
        r = synth_torch.make_quiva_device(seed, int(target), self.dev, well_base=well_base,
                                          lengths=lengths)
        self.sync()
        return r

    def make_fasta(self, seed, target, arrow=False):
        from dextractor_b200 import synth_torch
        r = synth_torch.make_fasta_device(seed, int(target), self.dev, arrow=arrow)
        self.sync()
        return r

    def host_bytes(self, t, n=None):
        return bytes(t[: (t.numel() if n is None else n)].cpu().numpy().tobytes())

    def equal(self, a, b):
        return bool(self.torch.equal(a, b))

    def free_cached(self):
        self.torch.cuda.empty_cache()

    # timing --------------------------------------------------------------------------------
    def sync(self):
        self.torch.cuda.synchronize()

    def timed_ms(self, fn):
        """CUDA events on the library's stream around fn(); rank-local, no collective"""
        tc = self.torch.cuda
        self.sync()
        with tc.stream(self.ext):
            a = tc.Event(enable_timing=True); b = tc.Event(enable_timing=True)
            a.record(self.ext); fn(); b.record(self.ext)
        self.sync()
        return a.elapsed_time(b)

    def clock_sampler(self):
        # one sampler per JOB: rank 0 watches every GPU of the job (ranks = local GPUs 0..N-1 on one node)
        if self.world > 1:
            return ClockSampler(",".join(str(i) for i in range(self.world)), enabled=(self.local == 0))
        return ClockSampler(str(self.local))

    def reference_dexqv(self, text: bytes):
        """the checker (never timed here): the reference's dexqv, else the oracle port"""
        from oracle import orc
        if orc.have_ref():
            return orc.ref_tool("dexqv", text)[0], "reference"
        return orc.dexqv(text), "port"

    def close(self):
        self.ctx.close()


def run_ours(args, env=None, out=print):
    import numpy as np
    from dextractor_b200 import lib as dxl
    from dextractor_b200 import shards

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if env is None:
        env = CudaEnv(local, world)
    ctx = env.ctx
    comm = Comm(world, rank, env.dev)
    hbm_peak, peak_src = peaks()

    class Shard:
        """one rank's share of a logical .quiva file and the dexqv / undexqv calls over it"""

        def __init__(self, text, nent, prefix):
            self.text, self.nent, self.prefix, self.U = text, nent, prefix, text.numel()
            self.enc = env.empty(self.U // 2 + (1 << 20))
            self.back = env.empty(self.U + 4096)
            self.carry, self.rc, self.last_well = None, None, 0
            self.st = {}

        def prepare(self):
            """COLLECTIVE (one broadcast): rank 0 resolves the run characters in its first ~100 k
            positions (QV.c:993-1015) and hands them on; a rank > 0 counts run lengths with them from
            its first entry on.  The last well of the shard is what the next rank's first well
            delta is coded against (dexqv.c:128-135)."""
            st0 = ctx.qv_scan_dev(self.text.data_ptr(), self.U, None)
            rc = comm.broadcast_i64([st0.delchar, st0.subchar], 0)
            self.rc = (rc[0], rc[1])
            if rank > 0:
                c = dxl.Carry()
                c.delchar, c.subchar, c.totchar = rc[0], rc[1], 200000
                self.carry = c
            key = self.prefix + b"/"                     # a QV line may start with '@' too
            tail = env.host_bytes(self.text[-min(self.U, 400000):])
            k = tail.rfind(b"\n" + key)
            if k < 0 and not tail.startswith(key):
                tail = env.host_bytes(self.text)
                k = tail.rfind(b"\n" + key)
            self.last_well = int(tail[k + 1:].split(b"/")[1])

        def encode(self, index=True):
            """COLLECTIVE (one all-gather): dexqv = scan -> statistics exchange -> code construction
            -> file header + encode.  The image is [header][entries] from enc[0].  index: also fetch the
            encoder's entry offsets (what decode_known needs; a file-to-file dexqv has no use for them,
            so the timed step does not ask)."""
            st = ctx.qv_scan_dev(self.text.data_ptr(), self.U, self.carry)
            rows = comm.gather_rows(shards.pack_stats(st, self.last_well))
            tot, lwell_in = shards.merge_stats(rows, rank, self.rc)
            cd = dxl.make_coding(tot, False)
            hdr = b"\xaa\x55" + dxl.write_coding(cd, self.prefix)
            hl = len(hdr)
            ctx.h2d(self.enc.data_ptr(), hdr)
            body, _, offs = ctx.qv_encode_dev(self.text.data_ptr(), self.U, cd, False, lwell_in,
                                              self.enc.data_ptr() + hl, self.enc.numel() - hl,
                                              want_offsets=self.nent if index else 0)
            self.st.update(hdr=hdr, img_len=hl + body, lwell_in=lwell_in)
            if index:
                self.st["offs"] = offs + hl
            return hl + body

        def decode_known(self):
            m = ctx.undexqv_dev(self.enc.data_ptr(), self.st["img_len"], False, self.back.data_ptr(),
                                self.back.numel(), entry_off=self.st["offs"],
                                well_in=self.st["lwell_in"])
            self.st["out_len"] = m
            return m

        def decode_discover(self):
            m = ctx.undexqv_dev(self.enc.data_ptr(), self.st["img_len"], False, self.back.data_ptr(),
                                self.back.numel(), well_in=self.st["lwell_in"])
            self.st["out_len"] = m
            return m

        def round_trip_ok(self):
            return self.st["out_len"] == self.U and env.equal(self.back[: self.U], self.text)

    def first_prefix(text):
        p = env.host_bytes(text, 200)
        return p[: p.index(b"/", 1)]

    # ---- parity of the sharded path against the reference, before anything is timed ------------
    # every rank codes a small shard of one logical file exactly as the timed step does (scan with
    # carry, statistics exchange, hand-off well, encode); the shard images are gathered and the
    # file they form must be the reference dexqv's output for the concatenated text.
    ptext, pnent, _ = env.make_quiva(900 + rank, args.parity_mb * 1e6, well_base=rank * 40 * 4000)
    psh = Shard(ptext, pnent, first_prefix(ptext))
    psh.prepare()
    psh.encode()
    hl = len(psh.st["hdr"])
    bodies = comm.gather_bytes(psh.enc[hl: psh.st["img_len"]])
    texts = comm.gather_bytes(psh.text)
    psh.decode_discover(); ok_a = psh.round_trip_ok()
    psh.decode_known(); ok_b = psh.round_trip_ok()
    parity = {"shards": world, "bytes": sum(len(t) for t in texts), "round_trip": ok_a and ok_b}
    if rank == 0:                                  # rank-local: no collective below this line
        want, kind = env.reference_dexqv(b"".join(texts))
        parity.update(checker=kind, equal=(psh.st["hdr"] + b"".join(bodies) == want))
    del bodies, texts, ptext, psh
    flags = comm.all_reduce([float(parity["round_trip"]), float(parity.get("equal", True))], "sum")
    if flags[0] != world or flags[1] != world:
        raise SystemExit(f"sharded dexqv differs from the reference ({parity})")
    env.free_cached()

    # ---- workload: one 2 GB shard per rank -----------------------------------------------------
    text, nent, npos = env.make_quiva(100 + rank, args.size_gb * GB, well_base=rank * 2_000_000)
    sh = Shard(text, nent, first_prefix(text))
    U = sh.U
    sh.prepare()

    def full_step():
        sh.encode(index=False)
        sh.decode_discover()

    sampler = env.clock_sampler(); sampler.start()
    for _ in range(args.warmup):
        full_step()
    ok = sh.round_trip_ok()                        # property at full size: decode(encode(x)) == x
    sh.encode(index=True)
    sh.decode_known(); ok = ok and sh.round_trip_ok()
    sh.decode_discover()
    if comm.all_reduce([float(ok)], "sum")[0] != world:
        raise SystemExit("round trip at full size differs from the input")

    # ---- K timed steps (device-resident) --------------------------------------------------------
    comm.barrier(); env.sync()
    ctx.launch_count(reset=True)
    ctx.profile(True); ctx.profile_report()

    def k_steps():
        for _ in range(args.steps):
            full_step()

    sampler.begin()
    ms = env.timed_ms(k_steps)
    sampler.end()
    if args.dump_outputs:                          # before the timings below overwrite the buffers
        dump_outputs(args.dump_outputs, {"dexqv": sh.enc[: sh.st["img_len"]],
                                         "undexqv": sh.back[: sh.st["out_len"]]}, rank, world)
    comm.barrier()
    clocks = sampler.stop()
    launches = ctx.launch_count()
    prof = ctx.profile_report(); ctx.profile(False)
    ms = comm.all_reduce([ms], "max")[0]
    U_all, C_all = [int(x) for x in comm.all_reduce([U, sh.st["img_len"]], "sum")]
    ms_step = ms / args.steps
    value = 2 * U_all / (ms_step * 1e-3) / GB

    # ---- per-direction timing (every rank; encode holds the all-gather) ---------------------------
    def timed(fn, reps=3):
        return min(env.timed_ms(fn) for _ in range(reps))

    enc_ms = timed(lambda: sh.encode(index=False))
    sh.encode(index=True)
    dec_known_ms = timed(sh.decode_known)
    dec_disc_ms = timed(sh.decode_discover)
    enc_ms, dec_known_ms, dec_disc_ms = comm.all_reduce([enc_ms, dec_known_ms, dec_disc_ms], "max")
    C = sh.st["img_len"]

    # ---- roofline of the dominant kernel (CUDA events inside the library, timed region) -------
    # algorithmic bytes per launch (DESIGN.md section 4)
    lines_bytes = 5 * (npos + nent)                    # the 5 QV lines incl. newlines
    algo = {"k_qv_hist_plain": 0.4 * lines_bytes, "k_qv_hist_run": 0.4 * lines_bytes,
            "k_qv_scan1": 0.8 * lines_bytes + 0.2 * U,
            "k_qv_size": lines_bytes, "k_qv_emit": lines_bytes + C,
            "k_qv_decode5": C + U, "k_qv_decode5_spec": C + lines_bytes,
            "k_qv_decode6": C + U, "k_qv_decode6_spec": C + lines_bytes,
            "k_qv_assemble": 2 * U, "k_pred_slots": U}
    top = max(prof.items(), key=lambda kv: kv[1][1]) if prof else ("none", (1, 1.0))
    tname, (tcalls, ttot) = top
    tavg = ttot / max(tcalls, 1)
    achieved = algo.get(tname, U) / (tavg * 1e-3) / GB
    traffic, traffic_src = None, None           # dram bytes per launch from the committed ncu capture
    for tf in ("r02_traffic.json", "r01_traffic.json"):
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", tf)))
            key = tname if tname in tr["kernels"] else tname.replace("_spec", "")   # one kernel, two modes
            if key in tr["kernels"]:
                traffic = tr["kernels"][key]["dram_bytes_per_text_byte"] * U
                traffic_src = (f"profiles/{tf} (ncu dram__bytes_read.sum + dram__bytes_write.sum per launch of "
                               f"{key} on the 2 GB bench file, scaled by this run's U)")
                break
        except Exception:
            pass
    roofline = {"bound": "hbm", "kernel": tname, "achieved": achieved, "peak": hbm_peak,
                "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": traffic,
                "traffic_source": traffic_src, "peak_source": peak_src, "avg_ms": tavg,
                "algorithmic_bytes": algo.get(tname, U),
                "share_of_step": ttot / max(sum(v[1] for v in prof.values()), 1e-9)}
    path = {"dexqv": {"algorithmic_bytes": 1.8 * U + C, "ms": enc_ms,
                      "frac": (1.8 * U + C) / (enc_ms * 1e-3) / GB / hbm_peak},
            "undexqv_offsets_known": {"algorithmic_bytes": C + U, "ms": dec_known_ms,
                                      "frac": (C + U) / (dec_known_ms * 1e-3) / GB / hbm_peak},
            "undexqv_offsets_discovered": {"algorithmic_bytes": 2 * C + U, "ms": dec_disc_ms,
                                           "frac": (2 * C + U) / (dec_disc_ms * 1e-3) / GB / hbm_peak}}

    # ---- e2e: host buffers through the C ABI, copies inside the timed region (every rank) -------
    h_text = env.empty(U, pinned=True); h_text.copy_(text)
    h_enc = env.empty(U // 2 + (1 << 20), pinned=True)
    h_back = env.empty(U + 4096, pinned=True)
    env.sync()
    e2e_n = {}

    def e2e_step():
        n1 = ctx.dexqv_host_ptr(h_text.data_ptr(), U, False, h_enc.data_ptr(), h_enc.numel())
        n2 = ctx.undexqv_host_ptr(h_enc.data_ptr(), n1, False, h_back.data_ptr(), h_back.numel())
        e2e_n.update(n1=n1, n2=n2)

    def e2e_steps():
        for _ in range(args.steps):
            e2e_step()

    e2e_step()
    e2e_ok = e2e_n["n2"] == U and env.equal(h_back[:U], h_text)
    comm.barrier()
    e2e_ms = env.timed_ms(e2e_steps) / args.steps
    e2e_ms, = comm.all_reduce([e2e_ms], "max")
    if comm.all_reduce([float(e2e_ok)], "sum")[0] != world:
        raise SystemExit("host-buffer round trip differs from the input")
    e2e = {"value": 2 * U_all / (e2e_ms * 1e-3) / GB, "unit": "GB/s", "ms_per_step": e2e_ms,
           "h2d_bytes_per_step": int((U + e2e_n["n1"]) * world),
           "d2h_bytes_per_step": int((e2e_n["n1"] + e2e_n["n2"]) * world),
           "api": "dx_dexqv_host + dx_undexqv_host on pinned host buffers, per rank on its own shard "
                  "(independent per-shard files at N > 1); the decoder rediscovers entry offsets"}
    del h_text, h_enc, h_back

    extras = {"dexqv_gbs": U / (enc_ms * 1e-3) / GB,
              "undexqv_offsets_known_gbs": U / (dec_known_ms * 1e-3) / GB,
              "undexqv_offsets_discovered_gbs": U / (dec_disc_ms * 1e-3) / GB,
              "value_offsets_known": 2 * U_all / ((enc_ms + dec_known_ms) * 1e-3) / GB,
              "uncompressed_bytes": int(U), "compressed_bytes": int(C), "ratio": U / C, "entries": nent,
              "sharded_parity": parity,
              "kernels_ms_per_step": {k: round(v[1] / args.steps, 4) for k, v in sorted(prof.items())}}
    del sh, text
    env.free_cached()

    # ---- configs[0] / configs[2]: dexta/undexta and dexar/undexar on 1 GB per rank (every rank;
    #      the 2-bit path needs no exchange at all, so the only collective is the max of the times)
    two_bit = [0.0] * 4
    if not args.no_extras:
        for j, arrow in enumerate((False, True)):
            kind = env.dx.ARROW if arrow else env.dx.FASTA
            fa, nfa = env.make_fasta(7 + 2 * j + 10 * rank, 1.0 * GB, arrow=arrow)
            UF = fa.numel()
            pk = env.empty(UF // 3 + (1 << 20)); un = env.empty(UF + 4096)
            m = ctx.dexta_dev(kind, fa.data_ptr(), UF, pk.data_ptr(), pk.numel())
            k = ctx.undexta_dev(kind, pk.data_ptr(), m, 80, False, un.data_ptr(), un.numel())
            if not arrow:
                assert k == UF and env.equal(un[:UF], fa), "dexta/undexta round trip differs"
            else:
                # SN=%.2f headers pass through a float and lose up to 0.01 per trip (SURVEY App. B.7):
                # same length, and only SNR digits of the header lines may differ
                ndiff = int((un[:UF] != fa).sum()) if k == UF else -1
                assert 0 <= ndiff <= 16 * nfa, "dexar/undexar round trip differs outside the SNR digits"
            t_p = timed(lambda: ctx.dexta_dev(kind, fa.data_ptr(), UF, pk.data_ptr(), pk.numel()))
            t_u = timed(lambda: ctx.undexta_dev(kind, pk.data_ptr(), m, 80, False, un.data_ptr(),
                                                un.numel()))
            two_bit[2 * j], two_bit[2 * j + 1] = t_p, t_u
            nm = ("dexar", "undexar", "arrow") if arrow else ("dexta", "undexta", "fasta")
            extras.update({f"{nm[2]}_bytes_per_gpu": int(UF), f"{nm[0]}_bytes_per_gpu": int(m)})
            del fa, pk, un
            env.free_cached()
    two_bit = comm.all_reduce(two_bit, "max")
    if not args.no_extras:
        UF, m = extras["fasta_bytes_per_gpu"], extras["dexta_bytes_per_gpu"]
        UA, ma = extras["arrow_bytes_per_gpu"], extras["dexar_bytes_per_gpu"]
        extras.update(dexta_gbs=world * UF / (two_bit[0] * 1e-3) / GB,
                      undexta_gbs=world * UF / (two_bit[1] * 1e-3) / GB,
                      dexta_frac=(UF + m) / (two_bit[0] * 1e-3) / GB / hbm_peak,
                      undexta_frac=(UF + m) / (two_bit[1] * 1e-3) / GB / hbm_peak,
                      dexar_gbs=world * UA / (two_bit[2] * 1e-3) / GB,
                      undexar_gbs=world * UA / (two_bit[3] * 1e-3) / GB,
                      dexar_frac=(UA + ma) / (two_bit[2] * 1e-3) / GB / hbm_peak,
                      undexar_frac=(UA + ma) / (two_bit[3] * 1e-3) / GB / hbm_peak)

    # ======== from here on: rank-local work only (NO collective until the final barrier) ========
    if rank == 0 and world == 1 and not args.no_extras:
        # configs[4]: mixed short/long subread lengths (500 bp - 50 kb), 0.5 GB each
        sweep = {}
        rs = np.random.default_rng(5)
        npos_t = int(0.5 * GB / 5.02)
        dists = {"log_uniform_500_50k": lambda k: np.exp(rs.uniform(np.log(500), np.log(50000), size=k)),
                 "90pct_500bp_10pct_50kb": lambda k: np.where(rs.random(k) < 0.9, 500, 50000),
                 "10pct_500bp_90pct_50kb": lambda k: np.where(rs.random(k) < 0.1, 500, 50000)}
        for name, draw in dists.items():
            Ls = np.asarray(draw(200000), dtype=np.int64)
            Ls = Ls[: int(np.searchsorted(np.cumsum(Ls), npos_t)) + 1]
            tx, ne, npz = env.make_quiva(50, 0, lengths=Ls)
            Us = tx.numel()
            e2 = env.empty(Us // 2 + (1 << 20)); b2 = env.empty(Us + 4096)
            st2 = {}

            def enc2():
                st2["n"] = ctx.dexqv_dev(tx.data_ptr(), Us, False, e2.data_ptr(), e2.numel())

            def dec2():
                st2["m"] = ctx.undexqv_dev(e2.data_ptr(), st2["n"], False, b2.data_ptr(), b2.numel())

            enc2(); dec2(); dec2()
            assert st2["m"] == Us and env.equal(b2[:Us], tx), "length sweep round trip differs"
            t_e = timed(enc2)
            t_d = timed(dec2)
            sweep[name] = {"entries": int(ne), "bytes": int(Us), "dexqv_gbs": Us / (t_e * 1e-3) / GB,
                           "undexqv_discovered_gbs": Us / (t_d * 1e-3) / GB}
            if not args.no_cpu:                      # the whole 0.5 GB image against the reference tool's
                want, kind = env.reference_dexqv(env.host_bytes(tx))
                same = (env.host_bytes(e2[: st2["n"]]) == want)
                sweep[name].update(checker=kind, equal=bool(same))
                assert same, f"length sweep {name}: the image differs from the {kind}'s"
                del want
            del tx, e2, b2
            env.free_cached()
        extras["length_sweep"] = sweep

    # ---- CPU baseline beside it (rank 0, N=1 only) ---------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        ncore = os.cpu_count() or 1
        r1 = cpu_reference_sample(args.cpu_sample_mb, seed=1, nproc=1)
        r = cpu_reference_sample(args.cpu_sample_mb, seed=1, nproc=ncore)
        t = r["t_enc"] + r["t_dec"]
        cpu = {"value": 2 * r["bytes"] / t / GB, "unit": "GB/s", "cores": r["cores"], "kind": r["kind"],
               "sample": f"{r['cores']} x {r['sample_bytes']/1e6:.0f} MB synthetic .quiva (same generator "
                         f"family), dexqv then undexqv, reference binaries, one single-threaded process per "
                         f"core on independent copies, /dev/shm",
               "dexqv_gbs": r["bytes"] / r["t_enc"] / GB, "undexqv_gbs": r["bytes"] / r["t_dec"] / GB,
               "one_core": {"value": 2 * r1["bytes"] / (r1["t_enc"] + r1["t_dec"]) / GB,
                            "dexqv_gbs": r1["bytes"] / r1["t_enc"] / GB,
                            "undexqv_gbs": r1["bytes"] / r1["t_dec"] / GB},
               "host_cores_available": os.cpu_count()}
        for kind in ("fasta", "arrow"):          # the 2-bit tools, single threaded and on every core
            a1 = cpu_reference_sample(args.cpu_sample_mb, seed=2, nproc=1, kind=kind)
            an = cpu_reference_sample(args.cpu_sample_mb, seed=2, nproc=ncore, kind=kind)
            e, d = _TOOLS[kind]
            cpu["one_core"].update({f"{e}_gbs": a1["bytes"] / a1["t_enc"] / GB,
                                    f"{d}_gbs": a1["bytes"] / a1["t_dec"] / GB})
            cpu.update({f"{e}_gbs": an["bytes"] / an["t_enc"] / GB,
                        f"{d}_gbs": an["bytes"] / an["t_dec"] / GB})

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
                "data": "synthetic", "config": workload_config(args),
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
                "roofline": roofline, "path_roofline": path, "cpu_baseline": cpu,
                "extra": extras}
        out(json.dumps(line))
        sys.stdout.flush()
    # Teardown order matters: tensors that were used on the library's stream must be gone before
    # dx_close destroys it (torch's caching allocators record events on every stream that used a
    # block when the block is freed), and the process group must go before the context.
    import gc
    gc.collect()
    env.sync()
    comm.barrier()
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()
    env.close()
    return comm.log


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--size-gb", type=float, default=2.0, help="uncompressed .quiva GB per GPU")
    ap.add_argument("--parity-mb", type=float, default=48.0,
                    help="per-rank shard of the pre-timing parity check against the reference")
    ap.add_argument("--ref-sample-mb", type=float, default=64.0, help="per process")
    ap.add_argument("--ref-cores", type=int, default=0, help="reference arm processes (0 = all cores)")
    ap.add_argument("--cpu-sample-mb", type=float, default=64.0, help="per process")
    ap.add_argument("--no-extras", action="store_true", help="skip the dexta/undexta side numbers")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write samples of the last timed step's .dexqv image and decoded text as .npy")
    args = ap.parse_args(argv)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the GPU path's outputs; the reference arm writes none")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    return args


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    run_ours(args)


if __name__ == "__main__":
    main()
