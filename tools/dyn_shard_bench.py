"""dev tool: the multi-candidate mode split across ranks (ambc_dyn_range_*, distributed.compress_dynamic_sharded).

One GPU (plain `python`): a simulated --ranks-way split (dyn_shard_ranges; every rank a copy of its range + 8192-byte
halo) of --gib GiB of the synthetic corpus (kind mask --kinds) and of --cascade-mib MiB of the cascade input (runs,
then homogeneous text: the chain leaves every speculative chain), both with the reference's candidate list.  Per rank:
walk (ambc_dyn_range_walk), resolve (the rounds the fold asks of it) and encode (ambc_dyn_range_encode) times, host
clock around calls that synchronise the device; the slowest rank and the fold rounds.  Against
engine.compress_dynamic_device on the whole input, alternated with the split, best of --reps.  The outputs of both
are compared.
N GPUs (under torchrun): every rank holds --gib GiB of the corpus, compress_dynamic_sharded assembles the body on
rank 0; timed with a barrier before and a device synchronise + barrier after, best of --reps.
Prints JSON lines with the card's name and power limit.

  python tools/dyn_shard_bench.py [--gib 1] [--cascade-mib 64] [--ranks 8] [--reps 3] [--kinds 95]
  torchrun --nproc-per-node N tools/dyn_shard_bench.py --gib 1"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

REF = (131072, 65536, 32768, 16384, 8192, 4096, 2048, 1024)  # adaptive_compressor.py:61-62


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                               str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    except OSError:
        return torch.cuda.get_device_name()


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return r, time.perf_counter() - t0


def cascade(n, seed=501, lead=1024):
    """a cascade input made on the GPU: runs, then log lines of the synthetic corpus"""
    from adaptive_compression_b200 import engine
    r = np.random.RandomState(seed)
    head = np.repeat(r.randint(0, 256, 64).astype(np.uint8), 16)[:lead]
    t = engine.synth(n, 0, kind_mask=2)  # kind 1: log lines
    t[:lead] = torch.from_numpy(head).cuda()
    return t


def split(t_in, world):
    """one simulated split -> (body, per-rank [walk, resolve, encode] seconds, fold rounds)"""
    from adaptive_compression_b200 import distributed as D
    from adaptive_compression_b200 import engine
    n = t_in.numel()
    ranges = D.dyn_shard_ranges(n, REF, world)
    bufs = [t_in[D.dyn_buffer_span(lo, hi, n)[0]:D.dyn_buffer_span(lo, hi, n)[1]].clone() for lo, hi in ranges]
    times = [[0.0, 0.0, 0.0] for _ in ranges]
    drs = []
    for r, (lo, hi) in enumerate(ranges):
        dr, times[r][0] = timed(lambda: engine.dyn_range_walk(bufs[r], lo, hi, n, REF))
        drs.append(dr)
    rounds = 0
    while True:
        rounds += 1
        entries, stuck, stop = D.fold_dyn_entries([d.table for d in drs], n)
        if stuck is None:
            break
        _, dt = timed(lambda: engine.dyn_range_resolve(drs[stuck], entries[stuck]))
        times[stuck][1] += dt
    frags, records = [], []
    for r, (dr, e) in enumerate(zip(drs, entries)):
        if e is not None and e < ranges[r][1]:
            (frag, st, _, _, _), times[r][2] = timed(lambda: engine.dyn_range_encode(dr, e))
        else:
            frag, st = bufs[r][:0], None
        frags.append(frag)
        records.append((frag.numel(), -1 if st is None else st))
    plan, _ = D.dyn_fragment_plan(records, ranges, n)
    body = torch.cat([D.dyn_fragment(frags[r], records[r][1], plan[r][2], bufs[r], lo, hi, n, engine.FIXED_MARKER,
                                     r == world - 1) for r, (lo, hi) in enumerate(ranges)])
    return body, times, rounds


def one_gpu(a):
    from adaptive_compression_b200 import engine
    inputs = [("synth_k%d" % a.kinds, lambda: engine.synth(int(a.gib * (1 << 30)), 0, kind_mask=a.kinds))]
    if a.cascade_mib:
        inputs.append(("cascade", lambda: cascade(a.cascade_mib << 20)))
    for name, make in inputs:
        t = make()
        torch.cuda.synchronize()
        single, simulated = [], []
        same = True
        for _ in range(a.reps):
            o, dt = timed(lambda: engine.compress_dynamic_device(t, REF))
            single.append(dt)
            body, times, rounds = split(t, a.ranks)
            simulated.append((max(sum(x) for x in times), times, rounds))
            same = same and torch.equal(body, o.body)
            del o, body
        slow, times, rounds = min(simulated, key=lambda x: x[0])
        print(json.dumps({"card": card(), "input": name, "bytes": t.numel(), "ranks": a.ranks,
                          "single_gpu_s": round(min(single), 4),
                          "single_gpu_GBps": round(t.numel() / min(single) / 1e9, 3),
                          "slowest_rank_s": round(slow, 4), "fold_rounds": rounds,
                          "per_rank_walk_resolve_encode_s": [[round(x, 4) for x in r] for r in times],
                          "bodies_equal": same}), flush=True)
        del t
        torch.cuda.empty_cache()


def multi_gpu(a):
    import torch.distributed as dist
    from adaptive_compression_b200 import distributed as D
    from adaptive_compression_b200 import engine
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n = int(a.gib * (1 << 30)) * world
    lo, hi = D.dyn_shard_ranges(n, REF, world)[rank]
    b0, b1 = D.dyn_buffer_span(lo, hi, n)
    buf = engine.synth(b1 - b0, b0, kind_mask=a.kinds)
    best = None
    for _ in range(a.reps):
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        body, _, _, _ = D.compress_dynamic_sharded(buf, lo, hi, n, REF)
        torch.cuda.synchronize()
        dist.barrier()
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    if rank == 0:
        print(json.dumps({"card": card(), "world": world, "bytes": n, "seconds": round(best, 4),
                          "GBps": round(n / best / 1e9, 3), "body_bytes": body.numel()}), flush=True)
    dist.destroy_process_group()


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--gib", type=float, default=1.0)
    p.add_argument("--cascade-mib", type=int, default=64)
    p.add_argument("--ranks", type=int, default=8)
    p.add_argument("--reps", type=int, default=3)
    p.add_argument("--kinds", type=int, default=95)
    a = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    (multi_gpu if "RANK" in os.environ else one_gpu)(a)


if __name__ == "__main__":
    main()
