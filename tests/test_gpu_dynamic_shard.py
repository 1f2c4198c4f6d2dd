"""The multi-candidate ("dynamic") mode split across R ranks, simulated on one GPU: every rank gets a copy of exactly
its input range and the 8192-byte halo behind it (distributed.dyn_buffer_span), walks it (ambc_dyn_range_walk), the
host fold of the entry tables runs in rank order with the resolves it asks for (ambc_dyn_range_resolve), and every
rank encodes its own packages (ambc_dyn_range_encode); distributed.dyn_fragment_plan places them.  Body, package
list and counters must be engine.compress_dynamic_device's and the oracle's, the body must decode back, and the
tables and walk launches must be test_cpu_dynamic_shard's model's."""
import numpy as np
import pytest

import oracle as O
import test_cpu_dynamic_shard as S
import test_cpu_dynamic_walk as W

pytestmark = pytest.mark.gpu

SPAN_LAUNCHES = 5  # k_select_span_fast, k_sizes, k_scan_tiles, k_offsets, k_pack_span


@pytest.fixture(scope="module")
def eng():
    from adaptive_compression_b200 import engine
    engine.require_cuda()
    return engine


def _dev(b):
    import torch
    a = np.frombuffer(bytes(b), dtype=np.uint8)
    return torch.from_numpy(a.copy()).to("cuda") if a.size else torch.empty(0, dtype=torch.uint8, device="cuda")


def simulate(eng, t_in, cands, mask, flags, marker, world):
    """-> (body tensor, packages, usage, payload, tables, walk launches, encode launches); t_in: the whole input on
    the GPU, of which every rank copies its buffer span"""
    import torch
    from adaptive_compression_b200 import _lib as L
    from adaptive_compression_b200 import distributed as D
    lib = L.lib()
    n, mb = t_in.numel(), len(marker)
    ranges = D.dyn_shard_ranges(n, cands, world)
    bufs, drs, walk_launches = [], [], 0
    for lo, hi in ranges:
        b0, b1 = D.dyn_buffer_span(lo, hi, n)
        bufs.append(t_in[b0:b1].clone())  # a copy: nothing outside the range and its halo is reachable
        before = lib.ambc_launch_count()
        drs.append(eng.dyn_range_walk(bufs[-1], lo, hi, n, cands, mask, flags, mb))
        walk_launches += lib.ambc_launch_count() - before
    for _ in range(world + 1):
        entries, stuck, stop = D.fold_dyn_entries([d.table for d in drs], n)
        if stuck is None:
            break
        before = lib.ambc_launch_count()
        eng.dyn_range_resolve(drs[stuck], entries[stuck])
        walk_launches += lib.ambc_launch_count() - before
    assert stuck is None
    frags, records, packages, usage, payload, enc_launches = [], [], [], [0] * 5, 0, 0
    for r, (dr, e) in enumerate(zip(drs, entries)):
        if e is not None and e < ranges[r][1]:
            before = lib.ambc_launch_count()
            frag, st, pk, us, pay = eng.dyn_range_encode(dr, e, marker)
            enc_launches += lib.ambc_launch_count() - before
        else:
            frag, st, pk, us, pay = bufs[r][:0], None, [], [0] * 5, 0
        frags.append(frag)
        records.append((frag.numel(), -1 if st is None else st))
        packages += [(t, o, c) for _, t, o, c in pk]
        usage = [a + b for a, b in zip(usage, us)]
        payload += pay
    plan, body_len = D.dyn_fragment_plan(records, ranges, n, mb)
    parts = []
    for r, ((off, length, state), (lo, hi)) in enumerate(zip(plan, ranges)):
        part = D.dyn_fragment(frags[r], records[r][1], state, bufs[r], lo, hi, n, marker, r == world - 1)
        if state == "raw_starts_here":
            packages.append((255, n - records[r][1], n - records[r][1]))
            usage[0] += 1
        assert part.numel() == length and off == sum(p.numel() for p in parts)
        parts.append(part)
    body = torch.cat(parts)
    assert body.numel() == body_len
    return body, packages, usage, payload, [d.table for d in drs], walk_launches, enc_launches


def test_sharded_walk_matches_single_gpu_oracle_and_model(eng):
    from adaptive_compression_b200 import _lib as L
    bad, singles = [], {}
    for name, R, data, cands, methods, marker, pcr, M in S.sharded_models():
        mask, flags = eng.method_mask(methods), L.F_PER_CHUNK_RAW if pcr else 0
        t = eng.to_device(data)
        if name not in singles:
            o = eng.compress_dynamic_device(t, cands, mask=mask, flags=flags, marker=marker)
            singles[name] = (o.body.cpu().numpy().tobytes(), [tuple(p) for p in o.packages], list(o.usage),
                             int(o.payload_bytes))
            wbody, wpm = O.compress_body(data, cands, methods, marker, pcr)
            if singles[name][0] != wbody or singles[name][1] != [tuple(p) for p in wpm]:
                bad.append((name, "single-GPU body differs from the oracle"))
        body, packages, usage, payload, tables, wl, el = simulate(eng, t, cands, mask, flags, marker, R)
        sbody, spk, susage, spay = singles[name]
        if body.cpu().numpy().tobytes() != sbody or [tuple(p) for p in packages] != spk:
            bad.append((name, R, "body", body.numel(), len(sbody)))
            continue
        if usage != susage or payload != spay:
            bad.append((name, R, "counters", usage, susage, payload, spay))
        if tables != [m.table for m in M.ranks]:
            bad.append((name, R, "tables"))
        want_wl = sum(m.walk_launches() for m in M.ranks)
        want_el = SPAN_LAUNCHES * sum(1 for c, _ in M.chains if c)
        if (wl, el) != (want_wl, want_el):
            bad.append((name, R, "launches", wl, want_wl, el, want_el))
        out, status = eng.decompress_device(body, len(data), marker=marker)
        if status != [0, 0] or out.cpu().numpy().tobytes() != data:
            bad.append((name, R, "round trip", status))
    assert not bad, bad


def test_raw_package_over_4_gib_raises_like_the_single_gpu_path(eng):
    """random bytes just over 4 GiB: no winner at position 0, so the whole file would be one raw package that its u32
    fields cannot frame; both paths raise AmbcError(E_ARG)"""
    import torch
    from adaptive_compression_b200 import _lib as L
    n = (4 << 30) + 4096
    gen = torch.Generator(device="cuda")
    gen.manual_seed(7)
    t = torch.randint(0, 256, (n,), dtype=torch.uint8, device="cuda", generator=gen)
    cands = W.REF
    with pytest.raises(L.AmbcError) as single:
        eng.compress_dynamic_device(t, cands)
    assert single.value.code == L.E_ARG
    with pytest.raises(L.AmbcError) as sharded:
        simulate(eng, t, cands, L.NATIVE_MASK, 0, eng.FIXED_MARKER, 4)
    assert sharded.value.code == L.E_ARG and str(sharded.value) == str(single.value)
    del t
    torch.cuda.empty_cache()
