"""Wall time and walk launches of the multi-candidate ("dynamic") mode, on the bench corpus and on a cascade input.

On the cascade (1 KiB of runs, then homogeneous text) one short package moves the true chain off the 8192 grid and
no segment's speculative chain meets it again, so the chain stitch resolves one segment per round: about one
k_dynamic_walk launch, with a host synchronisation, per 64 KiB of input.  The bench corpus needs a few.  Every
dynamic run is alternated with a fixed-grid run (4 KiB chunks) of the same input as the baseline.

    python tools/dyn_stitch_bench.py [--sizes-mib 64 1024] [--repeats 3] [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import inputs  # noqa: E402
from adaptive_compression_b200 import engine  # noqa: E402
from adaptive_compression_b200.adaptive_compressor import REFERENCE_CANDIDATES  # noqa: E402

SPAN_LAUNCHES = 5  # k_select_span_fast, k_sizes, k_scan_tiles, k_offsets, k_pack_span


def cascade_device(n):
    """1 KiB of runs, then 4 MiB of homogeneous text repeated (the text is generated in Python; repeating it keeps
    1 GiB cheap to build and keeps every 8 KiB of it a winner of the same size)"""
    period = inputs.text(4 << 20, 502)
    a = np.frombuffer(inputs.runs(1024, 501) + period * (n // len(period) + 1), dtype=np.uint8)[:n]
    return torch.from_numpy(a.copy()).to("cuda")


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes-mib", type=int, nargs="+", default=[64, 1024])
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lib = engine.require_cuda()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    dev = torch.cuda.current_device()
    rows = []
    engine.compress_dynamic_device(engine.synth(1 << 20, 0), REFERENCE_CANDIDATES)  # module load, first launches
    engine.compress_device(engine.synth(1 << 20, 0), 4096)
    for mib in a.sizes_mib:
        n = mib << 20
        for name, make in (("bench_corpus", lambda: engine.synth(n, 0)), ("cascade", lambda: cascade_device(n))):
            t = make()
            dyn, fixed, walks = [], [], set()
            for _ in range(a.repeats):
                before = lib.ambc_launch_count()
                dt, o = timed(lambda: engine.compress_dynamic_device(t, REFERENCE_CANDIDATES))
                walks.add(lib.ambc_launch_count() - before - SPAN_LAUNCHES)
                dyn.append(dt)
                body_len, n_pk = o.body_len, o.n_packages
                del o
                dt, f = timed(lambda: engine.compress_device(t, 4096))
                fixed.append(dt)
                fixed_len = f.body_len
                del f
            n_seg = -(-n // (64 * 1024))
            row = dict(input=name, mib=mib, segments=n_seg, walk_launches=sorted(walks), packages=n_pk,
                       dyn_s=[round(x, 4) for x in dyn], dyn_gbps=round(n / min(dyn) / 1e9, 3),
                       fixed4096_s=[round(x, 4) for x in fixed], fixed4096_gbps=round(n / min(fixed) / 1e9, 3),
                       dyn_ratio=round(body_len / n, 4), fixed4096_ratio=round(fixed_len / n, 4))
            rows.append(row)
            print(json.dumps(row), flush=True)
            del t
            torch.cuda.empty_cache()
    res = dict(gpu=gpu[dev] if dev < len(gpu) else gpu, rows=rows,
               timing="host clock around each call, synchronised; best of %d repeats; GB/s = input bytes / time"
               % a.repeats)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)
    print(json.dumps(dict(gpu=res["gpu"])))


if __name__ == "__main__":
    main()
