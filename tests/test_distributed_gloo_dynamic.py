"""CPU, world sizes 2 to 4 over gloo: the multi-rank host logic of the sharded multi-candidate mode -- the
all-gather of the fixed-size entry tables and the fold loop with its resolves (distributed.settle_dyn_entries), the
all-gather of (fragment bytes, stop), dyn_fragment_plan, dyn_fragment and the assembly on rank 0 -- checked against
the single-shot oracle.  Entry tables come from test_cpu_dynamic_shard's model and the packages from the oracle's
body here (no GPU); tests/test_gpu_dynamic_shard*.py cover the CUDA walk and encode."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import oracle as O
import test_cpu_dynamic_shard as S
import test_cpu_dynamic_walk as W
from test_distributed_gloo import _free_port


def _worker(rank, world, port, data, marker, tables0, tables1, frags, stops, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from adaptive_compression_b200 import distributed as D
    try:
        n = len(data)
        lo, hi = D.dyn_shard_ranges(n, W.SMALL, world)[rank]
        entries, stop, rounds = D.settle_dyn_entries(tables0[rank], n, lambda e: tables1[rank], torch.device("cpu"))
        frag = torch.from_numpy(np.frombuffer(frags[rank], dtype=np.uint8).copy())
        rec = torch.tensor([frag.numel(), stops[rank]], dtype=torch.int64)
        allr = torch.empty(2 * world, dtype=torch.int64)
        dist.all_gather_into_tensor(allr, rec)
        records = [tuple(int(x) for x in r) for r in allr.view(world, 2).tolist()]
        plan, body_len = D.dyn_fragment_plan(records, D.dyn_shard_ranges(n, W.SMALL, world), n, len(marker))
        b0, b1 = D.dyn_buffer_span(lo, hi, n)
        t_buf = torch.from_numpy(np.frombuffer(data[b0:b1], dtype=np.uint8).copy()) if b1 > b0 else \
            torch.empty(0, dtype=torch.uint8)
        local = D.dyn_fragment(frag, None if stops[rank] < 0 else stops[rank], plan[rank][2], t_buf, lo, hi, n, marker,
                               rank == world - 1)
        assert local.numel() == plan[rank][1]
        body = D.gather_fragments(local, plan, body_len)
        q.put((rank, entries, stop, rounds, body.numpy().tobytes() if rank == 0 else None))
    finally:
        dist.destroy_process_group()


def _body_slices(M, data, marker):
    """every rank's packages as a slice of the oracle's body, and its stop"""
    body, _ = O.compress_body(data, W.SMALL, (1, 2, 3, 4), marker, False)
    ovh, pos, frags, stops = len(marker) + 14, 0, [], []
    for recs, st in M.chains:
        ln = sum(ovh + c for _, _, _, c in recs)
        frags.append(body[pos:pos + ln])
        stops.append(-1 if st is None else st)
        pos += ln
    return body, frags, stops


CASES = {
    "cascade": lambda: W.cascade(16 * S.SEG_SMALL, 609, 512),
    "stop_in_middle": lambda: W.with_noise(W.mixed(6 * S.SEG_SMALL, 601), [(2 * S.SEG_SMALL, 9000)], 602),
    "short_last": lambda: W.mixed(4 * S.SEG_SMALL + 300, 607),
}


@pytest.mark.parametrize("world", [2, 3, 4])
@pytest.mark.parametrize("case", sorted(CASES))
def test_sharded_dynamic_body_equals_single_shot(world, case):
    data, marker = CASES[case](), b"\x5a\xa5"
    M = S.Sharded(data, W.SMALL, (1, 2, 3, 4), marker, False, world)
    want, frags, stops = _body_slices(M, data, marker)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    args = (data, marker, [m.table0 for m in M.ranks], [m.table for m in M.ranks], frags, stops, q)
    procs = [ctx.Process(target=_worker, args=(r, world, port) + args) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=300) for _ in range(world)), key=lambda x: x[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, entries, stop, rounds, body in res:
        assert entries == M.entries and stop == M.stop and rounds == M.fold_rounds, (rank, case)
    assert res[0][4] == want, case
    assert O.decompress_body(res[0][4], len(data), marker) == data
    if case == "cascade":
        assert M.fold_rounds == world  # one resolve per boundary
