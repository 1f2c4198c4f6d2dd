"""File -> file compress and decompress, in-memory against windowed (DESIGN.md §4.6, §6).

For every size: a synthetic file (the corpus of bench.py, kind mask 95) is written to --dir, then, alternated and
best of --reps, AdaptiveCompressor(chunk_size=4096).compress / .decompress through the in-memory path and through
windows of each --windows size, each against the MD5 floor of the same bytes (hashlib over the file's bytes already
in host memory, in 32 MiB pieces: the one serial chain the format imposes, with no reading), and the peak
torch-allocated device memory of every run (the in-memory path's buffers are the library's, outside torch).  Prints
the card's name and power limit first and one JSON line per measurement.

  python tools/windowed_bench.py --sizes-gib 8,16 --windows-mib 256,1024,4096 --reps 3 --dir /tmp/wbench
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True).stdout.strip()
    except OSError:
        return "unknown"


def md5_floor(data):
    view = memoryview(data)
    t = time.time()
    h = hashlib.md5()
    for lo in range(0, len(view), 32 << 20):
        h.update(view[lo:lo + (32 << 20)])
    return time.time() - t


def write_synth(path, n):
    from adaptive_compression_b200 import engine
    with open(path, "wb") as f:
        for lo in range(0, n, 1 << 30):
            f.write(engine.synth(min(1 << 30, n - lo), lo).cpu().numpy().tobytes())


def timed(fn):
    import torch
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    t = time.time()
    fn()
    torch.cuda.synchronize()
    return time.time() - t, torch.cuda.max_memory_allocated() - base


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes-gib", default="8,16")
    ap.add_argument("--windows-mib", default="256,1024,4096")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--dir", default="/tmp/windowed_bench")
    args = ap.parse_args()
    import torch
    from adaptive_compression_b200 import AdaptiveCompressor
    from adaptive_compression_b200 import adaptive_compressor as A
    from adaptive_compression_b200 import engine
    engine.require_cuda()
    print(json.dumps({"card": card(), "torch_device": torch.cuda.get_device_name(0)}), flush=True)
    os.makedirs(args.dir, exist_ok=True)
    real = A.window_bytes
    windows = [None] + [int(w) << 20 for w in args.windows_mib.split(",")]
    for gib in [float(x) for x in args.sizes_gib.split(",")]:
        n = int(gib * (1 << 30))
        src, amb, back = (os.path.join(args.dir, x) for x in ("in.bin", "out.ambc", "back.bin"))
        write_synth(src, n)
        with open(src, "rb") as f:
            data = f.read()
        best = {}
        for _ in range(args.reps):
            best.setdefault("md5_floor", []).append(md5_floor(data))
            for W in windows:
                A.window_bytes = (lambda need, dev: None) if W is None else (lambda need, dev, W=W: W)
                c = AdaptiveCompressor(chunk_size=4096)
                tc, pc = timed(lambda: c.compress(src, amb))
                td, pd = timed(lambda: c.decompress(amb, back))
                key = "in_memory" if W is None else "W=%dMiB" % (W >> 20)
                best.setdefault(key + ".compress", []).append((tc, pc))
                best.setdefault(key + ".decompress", []).append((td, pd))
        A.window_bytes = real
        floor = min(best.pop("md5_floor"))
        print(json.dumps({"size_gib": gib, "md5_floor_s": round(floor, 3)}), flush=True)
        for k, v in best.items():
            t = min(x[0] for x in v)
            print(json.dumps({"size_gib": gib, "run": k, "best_s": round(t, 3), "x_md5_floor": round(t / floor, 3),
                              "GB_per_s": round(n / t / 1e9, 3), "peak_device_GiB": round(max(x[1] for x in v) / 2**30, 3)}),
                  flush=True)
        del data
        for p in (src, amb, back):
            if os.path.exists(p):
                os.unlink(p)


if __name__ == "__main__":
    main()
