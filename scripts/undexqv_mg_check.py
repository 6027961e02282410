"""tools/bin/undexqv_mg on one big image written by tools/bin/dexqv_mg: the decode at 1, 2, 4 and 8 ranks.

    python scripts/undexqv_mg_check.py [--gb 64] [--gpus 1,2,4,8] [--dir /dev/shm]

Writes a synthetic .quiva of --gb GB (cfg4: 64 GB, the generator of bench.py on the GPU), encodes it with
dexqv_mg on as many GPUs as are visible, then decodes the image with undexqv_mg -v at every --gpus count
(ranks beyond the visible GPUs share them) and reports, per count, one JSON line: the per-rank phase times
undexqv_mg prints (read + H2D, decode, walk + relay, text, D2H + write), the wall time, and whether the
sha256 of the output is the original .quiva's.  The card's name and power limit are read in the same
run.  Wall times include reading and writing the files: where measured so far that is file I/O
bound (DESIGN section 5), not the decode.  The lines are also appended to --out."""
import argparse
import hashlib
import json
import os
import re
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
BIN = os.path.join(ROOT, "tools", "bin")


def sha256(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for blk in iter(lambda: f.read(1 << 24), b""):
            h.update(blk)
    return h.hexdigest()


def card():
    p = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return p.stdout.strip().splitlines()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gb", type=float, default=64.0)
    ap.add_argument("--gpus", default="1,2,4,8")
    ap.add_argument("--dir", default="/dev/shm" if os.path.isdir("/dev/shm") else "/tmp")
    ap.add_argument("--out", default="undexqv_mg_check.jsonl")
    args = ap.parse_args()
    import torch
    from dextractor_b200 import synth_torch
    if os.path.dirname(args.out):
        os.makedirs(os.path.dirname(args.out), exist_ok=True)
    ng = torch.cuda.device_count()
    if ng == 0:
        raise SystemExit("no CUDA device: the decode needs a GPU")
    base = os.path.join(args.dir, f"mgcheck_{os.getpid()}")
    rows = []
    try:
        # the .quiva, written in pieces of at most 4 GB (each piece its own well range)
        target, done, well = int(args.gb * (1 << 30)), 0, 0
        with open(base + ".quiva", "wb") as f:
            k = 0
            while done < target:
                t, nent, _ = synth_torch.make_quiva_device(100 + k, min(4 << 30, target - done), "cuda:0",
                                                           well_base=well)
                f.write(t.cpu().numpy().tobytes())
                done += t.numel(); well += 40 * nent + 1; k += 1
                del t
        want = sha256(base + ".quiva")
        t0 = time.perf_counter()
        p = subprocess.run([os.path.join(BIN, "dexqv_mg"), "-k", f"-g{ng}", base + ".quiva"], capture_output=True)
        enc_s = time.perf_counter() - t0
        if p.returncode != 0:
            raise SystemExit("dexqv_mg failed: " + p.stderr.decode()[-2000:])
        os.unlink(base + ".quiva")
        img = os.path.getsize(base + ".dexqv")
        for g in (int(x) for x in args.gpus.split(",")):
            t0 = time.perf_counter()
            p = subprocess.run([os.path.join(BIN, "undexqv_mg"), "-k", "-v", f"-g{g}", base + ".dexqv"],
                               capture_output=True, text=True)
            wall = time.perf_counter() - t0
            row = {"case": f"{args.gb:g} GB .quiva, dexqv_mg on {ng} GPUs", "quiva_bytes": done, "dexqv_bytes": img,
                   "ranks": g, "visible_gpus": ng, "rc": p.returncode, "wall_s": round(wall, 3),
                   "dexqv_mg_wall_s": round(enc_s, 3), "card": card()}
            if p.returncode == 0:
                row["sha256_equal"] = sha256(base + ".quiva") == want
                row["ranks_s"] = [dict(zip(("rank", "read_h2d", "decode", "walk_relay", "text", "d2h_write"),
                                           [int(m.group(1))] + [float(x) for x in m.groups()[1:]]))
                                  for m in re.finditer(r"rank (\d+) \(device \d+\): read \d+ bytes, wrote \d+; "
                                                       r"read\+H2D ([\d.]+) s, decode ([\d.]+) s, walk\+relay ([\d.]+) s, "
                                                       r"text ([\d.]+) s, D2H\+write ([\d.]+) s", p.stderr)]
                os.unlink(base + ".quiva")
            else:
                row["stderr"] = p.stderr[-2000:]
            rows.append(row)
            print(json.dumps(row), flush=True)
    finally:
        for ext in (".quiva", ".dexqv"):
            if os.path.exists(base + ext):
                os.unlink(base + ext)
        with open(args.out, "a") as f:
            for r in rows:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
