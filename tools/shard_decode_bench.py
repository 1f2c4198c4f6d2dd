"""dev tool: the range-local package index and the sharded decode of one body (distributed.decompress_sharded).

One GPU (plain `python`): a body of --gib GiB of the synthetic corpus (kind mask --kinds, chunk 4096) is
compressed on the GPU, then timed with a host clock around calls that synchronise the device, best of --reps:
  - ambc_index_dev (count + table, as engine.decompress_device runs it) against the range index at R = 1:
    phase 1 (ambc_range_index), the fold step, phase 3 (ambc_range_table, count + table);
  - a simulated R = 8 split (body_ranges, each range a copy of its bytes + halo): phase 1, fold, phase 3
    and decode per range; the slowest range bounds an 8-GPU decode (the fold is serial: its sum is listed);
  - the whole-body decode (ambc_decompress_dev_mask) for scale.
N GPUs (under torchrun): every rank compresses --gib GiB of its own chunk range, rank 0 assembles one body,
the ranges are scattered, and decompress_sharded is timed with and without gather_to=0, against every rank
decoding its own private body (the earlier multi-GPU "round trip").
Prints JSON lines with the card's name and power limit.

  python tools/shard_decode_bench.py [--gib 1] [--reps 3] [--kinds 95]
  torchrun --nproc-per-node N tools/shard_decode_bench.py --gib 4"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    except OSError:
        q = torch.cuda.get_device_name()
    return q


def best(fn, reps):
    t = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        t.append(time.perf_counter() - t0)
    return min(t) * 1e3


def single(args):
    from adaptive_compression_b200 import distributed as D
    from adaptive_compression_b200 import engine
    n = int(args.gib * (1 << 30))
    t = engine.synth(n, 0, kind_mask=args.kinds)
    o = engine.compress_device(t, 4096)
    body = o.body
    Lb = int(o.body_len)
    gib = Lb / (1 << 30)
    res = {"mode": "1 GPU", "card": card(), "input_bytes": n, "body_bytes": Lb}
    res["index_dev_ms"] = best(lambda: engine.index_device(body, n), args.reps)
    st = {}

    def r1():
        st["ri"] = engine.range_index(body, 0, Lb, Lb, n, work=st.get("ri").work if st.get("ri") else None)
    res["range_phase1_ms"] = best(r1, args.reps)
    res["range_fold_ms"] = best(lambda: engine.range_fold(st["ri"], engine.range_init_state()), args.reps)
    res["range_phase3_ms"] = best(lambda: engine.range_table(st["ri"], engine.range_init_state()), args.reps)
    res["index_dev_ms_per_gib"] = res["index_dev_ms"] / gib
    res["range_r1_ms_per_gib"] = (res["range_phase1_ms"] + res["range_fold_ms"] + res["range_phase3_ms"]) / gib
    tt, ne, _ = engine.index_device(body, n)
    out = torch.empty(n, dtype=torch.uint8, device="cuda")
    res["decode_ms"] = best(lambda: engine.range_decode(body, tt, ne, n, out=out), args.reps)
    # simulated R = 8
    R = 8
    ranges = D.body_ranges(Lb, R)
    bufs = [body[D.buffer_span(lo, hi, Lb)[0]:D.buffer_span(lo, hi, Lb)[1]].clone() for lo, hi in ranges]
    ris = [engine.range_index(b, lo, hi, Lb, n) for b, (lo, hi) in zip(bufs, ranges)]
    states, s = [], engine.range_init_state()
    for ri in ris:
        states.append(s)
        s = engine.range_fold(ri, s)
    slices = D.output_slices(states, ranges, n)
    per = []
    ok = True
    for r, ((lo, hi), b, ri, e) in enumerate(zip(ranges, bufs, ris, states)):
        p1 = best(lambda: engine.range_index(b, lo, hi, Lb, n, work=ri.work), args.reps)
        fold = best(lambda: engine.range_fold(ri, e), args.reps)
        tab = {}
        p3 = best(lambda: tab.update(t=engine.range_table(ri, e)), args.reps)
        t_table, ne_r, _, _, need = tab["t"]
        o0, o1 = slices[r]
        if need:  # a package runs past the halo: give the copy the next bytes (the fetch is not timed here)
            b = body[lo:D.buffer_span(lo, hi, Lb)[1] + need].clone()
        dec = best(lambda: engine.range_decode(b, t_table, ne_r, o1 - o0, out=out[o0:]), args.reps)
        per.append({"range": [lo, hi], "phase1_ms": p1, "fold_ms": fold, "phase3_ms": p3, "decode_ms": dec,
                    "total_ms": p1 + fold + p3 + dec})
    ok = torch.equal(out, t)
    res["r8_slowest_range_ms"] = max(p["total_ms"] for p in per)
    res["r8_fold_sum_ms"] = sum(p["fold_ms"] for p in per)
    res["r8_output_equal"] = bool(ok)
    res["r8_ranges"] = per
    print(json.dumps(res), flush=True)


def multi(args):
    import torch.distributed as dist
    from adaptive_compression_b200 import distributed as D
    from adaptive_compression_b200 import engine
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
    dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    per_rank = int(args.gib * (1 << 30))
    total, chunk = per_rank * world, 4096
    c0, b0, b1 = D.shard_range(total, chunk, rank, world)
    t_in = engine.synth(b1 - b0, b0, kind_mask=args.kinds)
    o = engine.compress_device(t_in, chunk)
    fr = int(o.first_raw)
    pk = D.packed_bytes(int(o.body_len), b1 - b0, fr, chunk)
    _, recs = D.place_shards(pk, fr, c0, world)
    _, frag = D.shard_fragment(o.body, t_in, fr, c0, chunk, total, recs, rank)
    _, Lb = D.fragment_plan(recs, total, chunk)
    body = D.assemble_body(frag, recs, total, chunk)
    lo, hi = D.body_ranges(Lb, world)[rank]
    buf = D.scatter_body(body, Lb)

    def timed(fn):
        t = []
        for _ in range(args.reps):
            torch.cuda.synchronize()
            dist.barrier()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            dist.barrier()
            t.append(time.perf_counter() - t0)
        return min(t) * 1e3
    r = {}
    r["sharded_ms"] = timed(lambda: D.decompress_sharded(buf, lo, hi, Lb, total))
    r["sharded_gather_ms"] = timed(lambda: D.decompress_sharded(buf, lo, hi, Lb, total, gather_to=0))
    out_priv = torch.empty(b1 - b0, dtype=torch.uint8, device="cuda")
    r["private_ms"] = timed(lambda: engine.decompress_device(o.body, b1 - b0, out=out_priv))
    off, sl, st = D.decompress_sharded(buf, lo, hi, Lb, total)
    want = engine.synth(sl.numel(), off, kind_mask=args.kinds)
    good = torch.tensor([1 if torch.equal(sl, want) and st == [0, 0] else 0], device="cuda")
    dist.all_reduce(good, op=dist.ReduceOp.MIN)
    if rank == 0:
        r.update({"mode": "%d GPUs" % world, "card": card(), "bytes_per_rank": per_rank, "body_bytes": Lb,
                  "output_equal": bool(good.item()),
                  "sharded_GBps": total / r["sharded_ms"] / 1e6, "private_GBps": total / r["private_ms"] / 1e6})
        print(json.dumps(r), flush=True)
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gib", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--kinds", type=int, default=0b1011111)
    args = ap.parse_args()
    if "RANK" in os.environ:
        multi(args)
    else:
        single(args)


if __name__ == "__main__":
    main()
