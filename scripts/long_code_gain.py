#!/usr/bin/env python
"""Decode time of a large .dexqv whose coding has many codes of 12 to 16 bits (tests/long_codes.py:
more than 64 distinct 11-bit prefixes in the deletion run table), through dx_undexqv_dev and
tools/bin/undexqv_mg -g1 / -g2.

    python scripts/long_code_gain.py --image PATH --out FILE [--tree DIR] [--gb 0.5] [--reps 5]

--image   the .dexqv; written first (by this tree's dexqv) when it does not exist, so that a second
          run with another --tree decodes the same bytes
--tree    import dextractor_b200 and run tools/bin from another checkout of the project (built by its
          __graft_entry__.build()), e.g. one at an earlier commit: run the script once per tree
--out     one JSON line is appended: the tree, the card's name and power limit, the image size, the
          dx_undexqv_dev times (device in and out, host clock around a synchronised call) and the
          sha256 of its text, and the wall time of undexqv_mg -g1 and -g2 (file to file, /dev/shm)
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def make_image(path, gb):
    import numpy as np
    import dextractor_b200 as dx
    from tests import long_codes
    from oracle import orc
    from tests.qv_shapes import coding
    n = int(gb * 1e9 / 1.5 / 10000) + 1               # ~1.5 image bytes per position, 10 000 positions per entry
    lengths = np.random.default_rng(2026).integers(4000, 16000, size=n)
    text = long_codes.make_quiva(2026, lengths)
    assert long_codes.max_prefixes(coding(orc, text)) > long_codes.PREFIXES
    ctx = dx.Context(0)
    try:
        enc = ctx.dexqv(text)
    finally:
        ctx.close()
    with open(path, "wb") as f:
        f.write(enc)
    return len(text)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--image", required=True)
    ap.add_argument("--out", required=True)
    ap.add_argument("--tree", default=HERE)
    ap.add_argument("--gb", type=float, default=0.5, help="image bytes to aim at when the image is written")
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    tree = os.path.abspath(a.tree)
    sys.path.insert(0, HERE)                          # tests/ and oracle/ of this checkout
    sys.path.insert(0, tree)                          # ... and the library of the tree being timed
    import torch
    import dextractor_b200 as dx
    assert os.path.dirname(os.path.abspath(dx.__file__)) == os.path.join(tree, "dextractor_b200"), dx.__file__
    row = {"tree": a.tree, "card": card()}
    if not os.path.exists(a.image):
        assert tree == HERE, "the image is written by a run of this checkout (no --tree)"
        row["quiva_bytes"] = make_image(a.image, a.gb)
    with open(a.image, "rb") as f:
        enc = f.read()
    row["image_bytes"] = len(enc)

    ctx = dx.Context(0)
    try:
        img = torch.frombuffer(bytearray(enc), dtype=torch.uint8).cuda()
        torch.cuda.synchronize()
        cap = ctx.undexqv_size_dev(img.data_ptr(), len(enc)) + 64
        out = torch.empty(cap, dtype=torch.uint8, device="cuda")
        times = []
        for r in range(a.reps + 1):                   # the first call warms up
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            m = ctx.undexqv_dev(img.data_ptr(), len(enc), False, out.data_ptr(), cap)
            ctx.sync()
            if r:
                times.append((time.perf_counter() - t0) * 1e3)
        row["text_bytes"] = m
        row["text_sha256"] = hashlib.sha256(out[:m].cpu().numpy().tobytes()).hexdigest()
        row["undexqv_dev_ms"] = {"min": round(min(times), 2), "median": round(sorted(times)[len(times) // 2], 2)}
        ctx.profile(True)
        ctx.profile_report()
        ctx.undexqv_dev(img.data_ptr(), len(enc), False, out.data_ptr(), cap)
        ctx.sync()
        row["kernels_ms"] = {k: round(v[1], 2) for k, v in sorted(ctx.profile_report().items(), key=lambda kv: -kv[1][1])[:6]}
        ctx.profile(False)
        del img, out
    finally:
        ctx.close()
    torch.cuda.empty_cache()

    mg = os.path.join(tree, "tools", "bin", "undexqv_mg")
    d = tempfile.mkdtemp(prefix="dxgain_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    try:
        base = os.path.join(d, "g")
        with open(base + ".dexqv", "wb") as f:
            f.write(enc)
        for g in (1, 2):
            t0 = time.perf_counter()
            p = subprocess.run([mg, "-k", "-v", f"-g{g}", base], capture_output=True)
            row[f"undexqv_mg_g{g}_s"] = round(time.perf_counter() - t0, 3)
            assert p.returncode == 0, p.stderr.decode()
            row[f"undexqv_mg_g{g}_whole"] = b"rank 0 decodes the file alone" in p.stderr
            with open(base + ".quiva", "rb") as f:
                assert hashlib.sha256(f.read()).hexdigest() == row["text_sha256"], g
            os.unlink(base + ".quiva")
    finally:
        subprocess.run(["rm", "-rf", d])
    line = json.dumps(row)
    print(line)
    with open(a.out, "a") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
