"""dev tool: decode of BZIP2 (id 6) and LZMA (id 7) packages on the GPU against stock bz2 / lzma on the host.

Bodies of --mib MiB of the synthetic corpus (engine.synth) are built on the host with stdlib bz2 (level 9) and lzma
(xz, preset 9, dictionary = chunk size) at chunk sizes 131072, 32768 and 8192 (18-byte package headers, END package).  GPU: the package index
built on the GPU plus the decode (ambc_index_dev + ambc_decompress_dev_mask), timed with CUDA events, best of
--reps, output checked against the input.  Host: bz2.decompress / lzma.decompress over the same payloads on one core
and on all cores (a process pool).  Prints one JSON line per (codec, chunk) and the card's name and power limit.

  python tools/stdcodec_bench.py [--mib 64] [--reps 3] [--out DIR]"""
import argparse
import bz2
import ctypes as C
import json
import lzma
import multiprocessing as mp
import os
import struct
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

MARKER = b"\xff\xff\x00\x00"


def _enc(args):
    t, c = args
    if t == 6:
        return bz2.compress(c, 9)
    # preset 9 with a dictionary no larger than the chunk (a larger one only costs encoder set-up time)
    return lzma.compress(c, filters=[{"id": lzma.FILTER_LZMA2, "preset": 9, "dict_size": max(4096, len(c))}])


def _dec(args):
    t, p = args
    return len(bz2.decompress(p) if t == 6 else lzma.decompress(p))


def _dec_many(args):
    return sum(_dec(a) for a in args)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mib", type=int, default=64)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON lines to DIR/stdcodec_bench.jsonl")
    a = ap.parse_args()
    ncpu = os.cpu_count() or 1
    pool = mp.Pool(ncpu)  # (forked before CUDA is initialised)
    import torch
    from adaptive_compression_b200 import engine
    lib = engine.require_cuda()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    print("card:", card[0] if card else "unknown")
    n = a.mib << 20
    data = engine.synth(n, 0).cpu().numpy().tobytes()
    lines = []
    with pool:
        for t in (6, 7):
            for chunk in (131072, 32768, 8192):
                pieces = [data[i:i + chunk] for i in range(0, n, chunk)]
                payloads = pool.map(_enc, [(t, c) for c in pieces], chunksize=8)
                body = bytearray()
                for c, p in zip(pieces, payloads):
                    body += MARKER + bytes([t, 0]) + struct.pack("<III", len(c), len(c), len(p)) + p
                body += MARKER + bytes(12)
                t_body = torch.frombuffer(bytearray(body), dtype=torch.uint8).cuda()
                known = engine.method_mask([1, 2, 3, 4, t])
                out = torch.empty(n, dtype=torch.uint8, device="cuda")
                status = torch.zeros(2, dtype=torch.int32, device="cuda")
                st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                best = None
                for rep in range(a.reps + 1):  # (the first call allocates the bzip2 scratch: not timed)
                    status.zero_()
                    torch.cuda.synchronize()
                    e0.record()
                    t_table, ne, _ = engine.index_device(t_body, n, MARKER, known)
                    engine.L.check(lib.ambc_decompress_dev_mask(C.c_void_p(t_body.data_ptr()), t_body.numel(),
                                                                C.c_void_p(t_table.data_ptr()), ne, C.c_void_p(out.data_ptr()),
                                                                n, known, C.c_void_p(status.data_ptr()), st))
                    e1.record()
                    torch.cuda.synchronize()
                    if rep:
                        ms = e0.elapsed_time(e1)
                        best = ms if best is None else min(best, ms)
                ok = status.tolist() == [0, 0] and out.cpu().numpy().tobytes() == data
                jobs = [(t, p) for p in payloads]
                t0 = time.perf_counter()
                got1 = sum(_dec(j) for j in jobs)
                one = time.perf_counter() - t0
                t0 = time.perf_counter()
                got_all = sum(pool.map(_dec_many, [jobs[k::ncpu] for k in range(ncpu)]))
                alln = time.perf_counter() - t0
                rec = {"codec": "bzip2" if t == 6 else "lzma", "chunk": chunk, "mib": a.mib, "packages": len(pieces),
                       "payload_ratio": round(sum(len(p) for p in payloads) / n, 4), "gpu_ok": ok,
                       "gpu_ms": round(best, 2), "gpu_gbps": round(n / best / 1e6, 3),
                       "host_1core_gbps": round(n / one / 1e9, 4), "host_cores": ncpu,
                       "host_allcores_gbps": round(n / alln / 1e9, 4), "host_ok": got1 == got_all == n,
                       "card": card[0] if card else "unknown"}
                print(json.dumps(rec), flush=True)
                lines.append(rec)
                del t_body, out
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "stdcodec_bench.jsonl"), "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
