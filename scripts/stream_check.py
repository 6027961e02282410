"""The single-GPU tools on a big file, one window against many: dexqv / undexqv and dexta / undexta.

    python scripts/stream_check.py [--gb 8] [--window-gb 1] [--dir /dev/shm]

Writes a seeded .quiva and a seeded .fasta of --gb GB each (synth_torch, on the GPU), runs every tool
once with its default window (the whole file, if it fits the device) and once with
DEXB200_WINDOW = --window-gb GB, and checks the sha256 of the windowed outputs against the one-window
outputs (and, where tools/bin/dexqv_mg was built, the .dexqv against dexqv_mg -g1's).  A file larger than
the card's memory (>= 200 GB of .quiva) is what windows are for: there the one-window run is skipped
(--no-whole) and the decoded text is checked against the original instead.  Prints one JSON line per
tool run: wall time, windows, the largest window, peak device memory held, the card's name and power
limit."""
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
    return p.stdout.strip().splitlines()[:1]


def write_file(path, kind, nbytes, seed):
    """.quiva in 16 GB pieces with rising wells; .fasta in one piece (its generator starts every piece at
    well 0), so at most 64 GB of it"""
    import torch
    from dextractor_b200 import synth_torch
    dev = torch.device("cuda", 0)
    chunk = (16 << 30) if kind == "quiva" else min(nbytes, 64 << 30)
    with open(path, "wb") as f:
        done, k = 0, 0
        while done < nbytes and (kind == "quiva" or k == 0):
            part = min(chunk, nbytes - done)
            if kind == "quiva":
                t = synth_torch.make_quiva_device(seed + k, part, dev, well_base=k * 100_000_000)[0]
            else:
                t = synth_torch.make_fasta_device(seed, part, dev)[0]
            for at in range(0, t.numel(), 1 << 30):
                f.write(t[at:at + (1 << 30)].cpu().numpy().tobytes())
            done += t.numel(); k += 1
            del t
            torch.cuda.empty_cache()


def run(tool, path, window, extra=()):
    env = dict(os.environ)
    env.pop("DEXB200_WINDOW", None)
    if window:
        env["DEXB200_WINDOW"] = str(window)
    t0 = time.perf_counter()
    p = subprocess.run([os.path.join(BIN, tool), "-k", "-v", *extra, path], capture_output=True, env=env)
    dt = time.perf_counter() - t0
    if p.returncode != 0:
        raise SystemExit(f"{tool} failed: {p.stderr.decode()[-2000:]}")
    m = re.search(rb"(\d+) windows, largest (\d+) bytes, peak device memory held (\d+) bytes", p.stderr)
    w = [int(x) for x in m.groups()] if m else [1, os.path.getsize(path), None]
    return {"tool": tool, "window": window or "default", "wall_s": round(dt, 3), "windows": w[0],
            "largest_window": w[1], "peak_held": w[2]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gb", type=float, default=8.0)
    ap.add_argument("--window-gb", type=float, default=1.0)
    ap.add_argument("--dir", default="/dev/shm" if os.path.isdir("/dev/shm") else ".")
    ap.add_argument("--no-whole", action="store_true", help="skip the one-window runs (files larger than the card)")
    a = ap.parse_args()
    gpu = card()
    window = int(a.window_gb * (1 << 30))
    ok = True
    for kind, enc, dec, src, dst in (("quiva", "dexqv", "undexqv", ".quiva", ".dexqv"),
                                     ("fasta", "dexta", "undexta", ".fasta", ".dexta")):
        base = os.path.join(a.dir, f"stream_check_{kind}")
        write_file(base + src, kind, int(a.gb * (1 << 30)), 101)
        want_text = sha256(base + src)
        sums = {}
        for win in ([window] if a.no_whole else [0, window]):
            r = run(enc, base + src, win)
            sums[("img", win)] = sha256(base + dst)
            r2 = run(dec, base + dst, win)
            sums[("text", win)] = sha256(base + src)
            for x in (r, r2):
                x.update(gpu=gpu, file_bytes=os.path.getsize(base + (src if x is r else dst)))
                print(json.dumps(x), flush=True)
        same = len({v for k, v in sums.items() if k[0] == "img"}) == 1 and sums[("text", window)] == want_text
        if kind == "quiva" and os.path.exists(os.path.join(BIN, "dexqv_mg")):
            os.replace(base + dst, base + ".win" + dst)
            subprocess.run([os.path.join(BIN, "dexqv_mg"), "-k", "-g1", base + src], check=True, capture_output=True)
            same = same and sha256(base + dst) == sums[("img", window)]
            os.remove(base + ".win" + dst)
        print(json.dumps({"kind": kind, "gb": a.gb, "window": window, "sha256_match": same, "gpu": gpu}), flush=True)
        ok = ok and same
        for e in (src, dst):
            if os.path.exists(base + e):
                os.remove(base + e)
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
