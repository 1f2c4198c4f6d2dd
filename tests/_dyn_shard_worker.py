"""Worker of tests/test_gpu_dynamic_shard_multirank.py (launched with torch.distributed.run, one rank per GPU):
compress with distributed.compress_dynamic_sharded (every rank holds its input range and the halo behind it) and
assemble the body on rank 0, which compares it, the package list and the counters with
engine.compress_dynamic_device on the whole input; then decode the body with distributed.decompress_sharded."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import torch
import torch.distributed as dist

import inputs
import test_cpu_dynamic_walk as W
from adaptive_compression_b200 import _lib as L
from adaptive_compression_b200 import distributed as D
from adaptive_compression_b200 import engine


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ok = True
    cases = [("synth_ref", engine.synth((6 << 20) + 777, 5 << 20).cpu().numpy().tobytes(), W.REF, 0),
             ("cascade_ref", W.cascade(4 << 20), W.REF, 0),
             ("noisy_small_pcr", W.with_noise(W.mixed(1 << 20, 523), [(203_000, 9000), (700_000, 5000)], 524), W.SMALL,
              L.F_PER_CHUNK_RAW),
             ("tiny", inputs.text(3000, 5), W.REF, 0)]
    for name, data, cands, flags in cases:
        n = len(data)
        t_all = engine.to_device(data)
        lo, hi = D.dyn_shard_ranges(n, cands, world)[rank]
        b0, b1 = D.dyn_buffer_span(lo, hi, n)
        buf = t_all[b0:b1].clone()
        body, packages, usage, payload = D.compress_dynamic_sharded(buf, lo, hi, n, cands, flags=flags)
        good = True
        if rank == 0:
            o = engine.compress_dynamic_device(t_all, cands, flags=flags)
            good = (torch.equal(body, o.body) and [tuple(p) for p in packages] == [tuple(p) for p in o.packages]
                    and usage == list(o.usage) and payload == int(o.payload_bytes))
        body_len = torch.tensor([body.numel() if rank == 0 else 0], dtype=torch.int64, device="cuda")
        dist.broadcast(body_len, 0)
        body_len = int(body_len.item())
        blo, bhi = D.body_ranges(body_len, world)[rank]
        bbuf = D.scatter_body(body, body_len)
        _, whole, st = D.decompress_sharded(bbuf, blo, bhi, body_len, n, gather_to=0)
        if rank == 0:
            good = good and st == [0, 0] and whole.cpu().numpy().tobytes() == data
        print("rank %d %s: %s" % (rank, name, "ok" if good else "MISMATCH"), flush=True)
        ok = ok and good
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    dist.destroy_process_group()
    if rank == 0:
        print("DYN SHARD OK" if int(flag.item()) == 1 else "DYN SHARD FAILED", flush=True)
    sys.exit(0 if int(flag.item()) == 1 else 1)


if __name__ == "__main__":
    main()
