"""Worker of tests/test_gpu_shard_decode_multirank.py (launched with torch.distributed.run, one rank per GPU):
compress with the sharded chunk path and assemble ONE body on rank 0 (as tests/_multirank_worker.py does),
scatter its byte ranges to the ranks, decode it with distributed.decompress_sharded, and check every rank's
slice against the input and the gathered output against the whole input; then check that a body with a
corrupted marker raises the marker error on every rank."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import numpy as np
import torch
import torch.distributed as dist

from adaptive_compression_b200 import distributed as D
from adaptive_compression_b200 import engine


def assembled(data, chunk, rank, world):
    total = len(data)
    c0, b0, b1 = D.shard_range(total, chunk, rank, world)
    t_in = torch.from_numpy(np.frombuffer(data[b0:b1], dtype=np.uint8).copy()).cuda()
    o = engine.compress_device(t_in, chunk)
    fr = int(o.first_raw)
    pk = D.packed_bytes(int(o.body_len), b1 - b0, fr, chunk)
    _, recs = D.place_shards(pk, fr, c0, world)
    _, frag = D.shard_fragment(o.body, t_in, fr, c0, chunk, total, recs, rank)
    _, body_len = D.fragment_plan(recs, total, chunk)
    return D.assemble_body(frag, recs, total, chunk), body_len


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ok = True
    for seed, n, kinds in [(1, 3 << 20, 0b1011111), (2, (5 << 20) + 333, 0b1111111), (3, 5000, 0b1011111)]:
        data = engine.synth(n, seed << 20, kind_mask=kinds).cpu().numpy().tobytes()
        body, body_len = assembled(data, 4096, rank, world)
        lo, hi = D.body_ranges(body_len, world)[rank]
        buf = D.scatter_body(body, body_len)
        off, out, st = D.decompress_sharded(buf, lo, hi, body_len, n)
        good = out.cpu().numpy().tobytes() == data[off:off + out.numel()] and st == [0, 0]
        _, whole, st_all = D.decompress_sharded(buf, lo, hi, body_len, n, gather_to=0)
        if rank == 0:
            good = good and whole.cpu().numpy().tobytes() == data and st_all == [0, 0]
        print("rank %d seed %d: body %d bytes, slice [%d, %d) %s" % (rank, seed, body_len, off, off + out.numel(),
                                                                    "ok" if good else "MISMATCH"), flush=True)
        ok = ok and good
    # a corrupted marker in the last rank's range: every rank raises
    data = engine.synth(2 << 20, 99).cpu().numpy().tobytes()
    body, body_len = assembled(data, 4096, rank, world)
    if rank == 0:
        hs, pos = [], 0
        host = body.cpu().numpy()
        while pos + 18 <= body_len:
            hs.append(pos)
            pos += 18 + int(host[pos + 14:pos + 18].view(np.uint32)[0])
        bad = hs[-3]
        body[bad + 1] ^= 0x5A
    lo, hi = D.body_ranges(body_len, world)[rank]
    buf = D.scatter_body(body, body_len)
    try:
        D.decompress_sharded(buf, lo, hi, body_len, len(data))
        raised = False
    except ValueError as e:
        raised = "Marker mismatch in chunk header." in str(e)
    print("rank %d corrupted body: %s" % (rank, "raised" if raised else "DID NOT RAISE"), flush=True)
    ok = ok and raised
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    dist.destroy_process_group()
    if rank == 0:
        print("SHARD DECODE OK" if int(flag.item()) == 1 else "SHARD DECODE FAILED", flush=True)
    sys.exit(0 if int(flag.item()) == 1 else 1)


if __name__ == "__main__":
    main()
