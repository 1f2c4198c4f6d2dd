"""Multi-GPU sharding of the chunk path (SURVEY.md §8e): contiguous chunk ranges per rank, one
process per GPU, torch.distributed (NCCL over NVLink; gloo in the CPU tests) for the tiny exchanges
the path has:

  place_shards        all-gather of one 16-byte record per rank -> every rank folds the
                      "rest of file raw" monoid left to right (adaptive_compressor.py:586-590) and
                      learns its fragment's byte offset in the global body, or that it lies inside
                      the raw tail.
  merge_marker_flags  byte-wise MAX all-reduce of the per-shard n-gram presence flags
                      (NCCL has no bitwise OR; flags are 0/1 bytes).
  decompress_sharded  the way back: every rank holds one byte range of an assembled body
                      (body_ranges, scatter_body), indexes it on its own GPU (ambc_range_index),
                      and the package walk (adaptive_compressor.py:396-454) is folded across the
                      ranges in rank order, one 48-byte state per hop (R - 1 point-to-point
                      messages).  One all-gather of the entry states tells every rank where its
                      output slice lies and which copied-through package runs into its range; a
                      second one of the per-rank tail needs plans the payload bytes a rank fetches
                      from the next ranks (tail_fetch_plan).  Then every rank decodes its own slice.

  compress_dynamic_sharded  the multi-candidate mode (adaptive_compressor.py:537-590): every rank walks the
                      chunk chain of its own input range (whole segments of 64 * g bytes, dyn_shard_ranges)
                      from every position the chain can enter it at; an all-gather of the fixed-size entry
                      tables and a host fold (fold_dyn_entries) find the true entries, a rank whose true
                      entry is still open stitches it further, then every rank encodes its own packages
                      and one all-gather of (fragment bytes, stop) places them (dyn_fragment_plan).

A rank compresses its range as if no earlier rank had hit a chunk without a winner; shard_fragment()
then turns the local body into the bytes this rank contributes to the global body."""
import struct

import torch
import torch.distributed as dist

NO_RAW = -1


def raw_package_header(marker, rawlen):
    """the header of the raw package that holds the rest of the file (adaptive_compressor.py:586-590, :609-621);
    struct.error for 4 GiB or more, as the reference's struct.pack at :617-619"""
    return marker + bytes([255, 0]) + struct.pack("<III", rawlen, rawlen, rawlen)


def end_package(marker):
    """the END package (adaptive_compressor.py:595-607)"""
    return marker + bytes(12)


def refuse_dyn_raw(n, stop):
    """the multi-candidate mode refuses a raw package of 4 GiB or more as ambc_compress_dynamic_dev does"""
    from . import _lib as L
    if stop >= 0 and n - stop > 0xFFFFFFFF:
        raise L.AmbcError(L.E_ARG, "raw package over 4 GiB cannot be framed (u32 fields)")


def shard_range(total_bytes, chunk, rank, world):
    """contiguous chunk range of `rank`: (first_chunk, byte_begin, byte_end)"""
    n_chunks = (total_bytes + chunk - 1) // chunk
    per = (n_chunks + world - 1) // world
    c0 = min(n_chunks, rank * per)
    c1 = min(n_chunks, c0 + per)
    return c0, min(total_bytes, c0 * chunk), min(total_bytes, c1 * chunk)


def fold_placement(records):
    """records[r] = (fragment_bytes_before_first_raw, first_raw_global_chunk or -1), rank order.
    -> list of (offset, state): 'packed' (whole fragment lands at offset), 'raw_starts_here'
    (packed part at offset, then the global raw package) or 'in_raw_tail'.
    Monoid (SURVEY.md §7): A.B = A if A has a raw chunk else (A.bytes + B.bytes, B.first_raw)."""
    out = []
    offset = 0
    raw_seen = False
    for nbytes, first_raw in records:
        if raw_seen:
            out.append((None, "in_raw_tail"))
            continue
        if first_raw >= 0:
            out.append((offset, "raw_starts_here"))
            raw_seen = True
        else:
            out.append((offset, "packed"))
        offset += nbytes
    return out


def fold_placement_native(records, first_bytes, chunk, marker_bytes=4):
    """the same fold through the C-ABI (ambc_shard_place): -> list of (offset, state); for ranks inside
    the raw tail the offset is the place of their input bytes in the global body.  first_bytes[r] = input
    byte offset of rank r's shard (shard_range()[1]: clamped to the input length, so an empty trailing
    rank behind a partial last chunk still lands at the end of the raw data)"""
    import ctypes as C
    from . import _lib as L
    n = len(records)
    recs = (L.ShardRec * n)(*[L.ShardRec(int(b), int(fr)) for b, fr in records])
    fc = (C.c_uint64 * n)(*[int(x) for x in first_bytes])
    out = (L.ShardSlot * n)()
    L.check(L.lib().ambc_shard_place(recs, n, fc, chunk, marker_bytes, out))
    names = ("packed", "raw_starts_here", "in_raw_tail")
    return [(int(o.offset), names[o.state]) for o in out]


def _device():
    return torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")


def place_shards(fragment_bytes, first_raw_local, first_chunk_global, world):
    """all-gather the placement records; returns (this rank's (offset, state), all records)"""
    rank = dist.get_rank()
    fr = first_chunk_global + first_raw_local if first_raw_local >= 0 else NO_RAW
    mine = torch.tensor([int(fragment_bytes), int(fr)], dtype=torch.int64, device=_device())
    allr = torch.empty(2 * world, dtype=torch.int64, device=mine.device)
    dist.all_gather_into_tensor(allr, mine)
    recs = [tuple(x) for x in allr.view(world, 2).cpu().tolist()]
    return fold_placement(recs)[rank], recs


def packed_bytes(body_len, n_local, first_raw_local, chunk, marker_bytes=4):
    """bytes of the local body that precede its first raw chunk (END and local raw package removed)"""
    end = marker_bytes + 12
    if first_raw_local < 0:
        return body_len - end
    return body_len - end - (marker_bytes + 14) - (n_local - first_raw_local * chunk)


def fragment_plan(records, total_bytes, chunk, marker_bytes=4):
    """-> ([(offset, length, state)] per rank, body length): where every rank's contribution lands in the
    global body and how long it is, from the all-gathered records alone (every rank computes the same plan;
    the shards are shard_range(total_bytes, chunk, r, world)).  The last rank's length includes the END
    package.  Rule sharded: adaptive_compressor.py:586-590."""
    world = len(records)
    ovh, end = marker_bytes + 14, marker_bytes + 12
    states = fold_placement(records)
    g = next((fr for _, fr in records if fr >= 0), NO_RAW)  # global first raw chunk
    packed_total = 0
    if g >= 0:
        packed_total = sum(nb for nb, _ in records[:next(i for i, (_, fr) in enumerate(records) if fr >= 0) + 1])
    plan = []
    for r, ((off, state), (nbytes, _)) in enumerate(zip(states, records)):
        _, b0, b1 = shard_range(total_bytes, chunk, r, world)
        if state == "packed":
            length = nbytes
        elif state == "raw_starts_here":
            length = nbytes + ovh + (b1 - g * chunk)
        else:  # input bytes, verbatim, inside the raw package (b0 is clamped to the input length)
            off = packed_total + ovh + (b0 - g * chunk)
            length = b1 - b0
        if r == world - 1:
            length += end
        plan.append((off, length, state))
    last_off, last_len, _ = plan[-1]
    return plan, last_off + last_len


def shard_fragment(local_body, local_input, first_raw_local, first_chunk_global, chunk, total_bytes, records, rank,
                   marker=b"\xff\xff\x00\x00"):
    """-> (global byte offset, 1-D uint8 tensor) this rank contributes to the global body (the END
    package is appended by the last rank).  local_body / local_input are tensors on any device."""
    mb = len(marker)
    plan, _ = fragment_plan(records, total_bytes, chunk, mb)
    offset, length, state = plan[rank]
    n_local = local_input.numel()
    pk = packed_bytes(local_body.numel(), n_local, first_raw_local, chunk, mb)
    last = rank == len(records) - 1
    end_pkg = torch.tensor(list(end_package(marker)), dtype=torch.uint8, device=local_body.device)
    g = next((fr for _, fr in records if fr >= 0), NO_RAW)  # global first raw chunk
    if state == "packed":
        if last and first_raw_local < 0:  # the local body ends with the same END package: no copy
            assert local_body.numel() == pk + mb + 12
            return offset, local_body
        frag = local_body[:pk]
    elif state == "raw_starts_here":
        rawlen = total_bytes - g * chunk
        if rawlen > 0xFFFFFFFF:
            raise struct.error("'I' format requires 0 <= number <= 4294967295")  # adaptive_compressor.py:617-619
        hdr_t = torch.tensor(list(raw_package_header(marker, rawlen)), dtype=torch.uint8, device=local_body.device)
        frag = torch.cat([local_body[:pk], hdr_t, local_input[first_raw_local * chunk:]])
    else:
        frag = local_input
    if last:
        frag = torch.cat([frag, end_pkg])
    assert frag.numel() == length, (frag.numel(), length, state)
    return offset, frag


def assemble_body(frag, records, total_bytes, chunk, marker_bytes=4, dst=0, out=None):
    """Gather every rank's fragment into ONE body on rank `dst` (NCCL send / recv straight into the placed
    slice of the destination buffer -- NVLink peer copies; gloo on CPU).  Returns the body tensor on `dst`
    (None elsewhere).  `out`: optional preallocated destination on `dst` (>= body length)."""
    plan, body_len = fragment_plan(records, total_bytes, chunk, marker_bytes)
    return gather_fragments(frag, plan, body_len, dst, out)


def gather_fragments(frag, plan, body_len, dst=0, out=None):
    """send every rank's fragment to its place [offset, offset + length) of the plan in ONE body on rank `dst`;
    -> the body on `dst`, None elsewhere"""
    rank = dist.get_rank()
    if rank != dst:
        if frag.numel():
            dist.send(frag.contiguous(), dst)
        return None
    body = out[:body_len] if out is not None else torch.empty(body_len, dtype=torch.uint8, device=frag.device)
    reqs = []
    for r, (off, length, _) in enumerate(plan):
        if r == dst:
            body[off:off + length].copy_(frag)
        elif length:
            reqs.append(dist.irecv(body[off:off + length], r))
    for q in reqs:
        q.wait()
    return body


def merge_marker_flags(flags):
    """in-place byte-wise MAX all-reduce of a 2^L-byte presence-flag tensor"""
    dist.all_reduce(flags, op=dist.ReduceOp.MAX)
    return flags


def carry_windows(lens, tails):
    """lens[r] = bytes in shard r, tails[r] = its last min(4, lens[r]) bytes.  -> for every rank the
    (up to) 4 bytes that precede its shard in the global stream and how many exist, plus the same for
    the end of the whole stream.  Shards may be shorter than 4 bytes (or empty)."""
    out, window, before = [], b"", 0
    for n, t in zip(lens, tails):
        out.append((window, before))
        window = (window + bytes(t))[-4:]
        before += int(n)
    return out, (window, before)


def _bits_of(window, before_bytes, want_bits):
    """the last min(want_bits, 8 * before_bytes) bits of the stream ending with `window`, as (value, count)"""
    have = min(want_bits, 8 * min(before_bytes, len(window)))
    v = int.from_bytes(window, "big") if window else 0
    return (v & ((1 << have) - 1)) if have else 0, have


def find_marker_sharded(t_shard, max_len=32, levels=(16, 24, 32)):
    """MarkerFinder.find_marker (marker_finder.py:22-123) over a stream sharded across the ranks in rank
    order: every rank flags the L-bit windows that start in its shard (with the <= L-1 bits that precede
    it as carry), one byte-wise MAX all-reduce merges the flags (NCCL has no bitwise OR), every rank
    picks the same (marker bytes, length).  Raises ValueError when no marker of at most
    min(max_len, levels[-1]) bits exists."""
    import ctypes as C
    from . import _lib as L
    from . import engine
    lib = engine.require_cuda()
    world, rank = dist.get_world_size(), dist.get_rank()
    n_local = t_shard.numel()
    dev = t_shard.device
    meta = torch.zeros(5, dtype=torch.int64, device=dev)
    meta[0] = n_local
    k = min(4, n_local)
    if k:
        meta[1:1 + k] = t_shard[n_local - k:].to(torch.int64)
    allm = torch.empty(5 * world, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(allm, meta)
    rows = allm.view(world, 5).cpu().tolist()
    lens = [int(r[0]) for r in rows]
    tails = [bytes(int(x) for x in r[1:1 + min(4, int(r[0]))]) for r in rows]
    per_rank, (end_window, total_bytes) = carry_windows(lens, tails)
    window, before = per_rank[rank]
    total_bits = 8 * total_bytes
    tail, tail_bits = _bits_of(end_window, total_bytes, 31)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for lv in levels:
        Lb = min(lv, max_len)
        flags = torch.zeros(1 << Lb, dtype=torch.uint8, device=dev)
        carry, cb = _bits_of(window, before, Lb - 1)
        L.check(lib.ambc_marker_flags_dev(C.c_void_p(t_shard.data_ptr() if n_local else 0), n_local, Lb, carry, cb,
                                          C.c_void_p(flags.data_ptr()), stream))
        merge_marker_flags(flags)
        ln, val = C.c_uint32(0), C.c_uint64(0)
        rc = lib.ambc_marker_pick_dev(C.c_void_p(flags.data_ptr()), Lb, max_len, total_bits, tail, tail_bits,
                                      C.byref(ln), C.byref(val), stream)
        if rc == L.OK:
            return engine.marker_bytes(val.value, ln.value), ln.value
        if rc != L.E_NO_MARKER or Lb == max_len:
            L.check(rc)
    raise ValueError("Could not find a marker of length <= %d bits" % min(max_len, levels[-1]))


# ---- sharded decode of one assembled body ---------------------------------------------------------------
STATE_WORDS = 8  # ambc_range_state as int64 words


def body_ranges(body_len, world):
    """[(lo, hi)] per rank: contiguous byte ranges of about equal size covering [0, body_len)"""
    return [(body_len * r // world, body_len * (r + 1) // world) for r in range(world)]


def range_halo(marker_bytes=4):
    """header bytes a rank holds behind its range (a header starting at hi - 1 ends at hi + marker_bytes + 13)"""
    return marker_bytes + 13


def buffer_span(lo, hi, body_len, marker_bytes=4):
    """body bytes [b0, b1) a rank holds for its range [lo, hi): the range and the header halo behind it"""
    return lo, min(hi + range_halo(marker_bytes), body_len)


def tail_fetch_plan(ranges, needs, body_len, marker_bytes=4):
    """needs[r] = payload bytes rank r's last decoded package needs behind its buffer.  -> [(src, dst, g0, g1)]:
    rank src sends body[g0, g1) (inside its own range) to rank dst, in a fixed order every rank computes alike"""
    plan = []
    for r, ((lo, hi), need) in enumerate(zip(ranges, needs)):
        if not need:
            continue
        f0 = buffer_span(lo, hi, body_len, marker_bytes)[1]
        f1 = f0 + int(need)
        for q in range(r + 1, len(ranges)):
            qlo, qhi = ranges[q]
            g0, g1 = max(f0, qlo), min(f1, qhi)
            if g1 > g0:
                plan.append((q, r, g0, g1))
    return plan


def output_slices(entry_states, ranges, orig_size, marker_bytes=4, known_mask=None):
    """[(o0, o1)] per rank: the output bytes rank r decodes, from the states the fold handed to every rank.
    Slices are contiguous in rank order; the last one ends at orig_size (it owns the zero tail)."""
    from . import _lib as L
    from . import engine
    km = L.NATIVE_MASK if known_mask is None else known_mask
    starts = [engine.range_out_offset(s, lo, orig_size, marker_bytes, km) for s, (lo, _) in zip(entry_states, ranges)]
    return [(starts[r], starts[r + 1] if r + 1 < len(starts) else orig_size) for r in range(len(starts))]


def state_to_words(s):
    return [int(s.next_pos), int(s.out_before), int(s.pkg_pos) - (1 << 64) if s.pkg_pos >= 1 << 63 else int(s.pkg_pos),
            int(s.pkg_out), int(s.pkg_type), int(s.pkg_orig), int(s.pkg_comp), int(s.status)]


def state_from_words(w):
    from . import _lib as L
    return L.RangeState(*[int(x) & ((1 << 64) - 1) for x in w[:4]], *[int(x) & 0xFFFFFFFF for x in w[4:8]])


def scatter_body(body, body_len, src=0, marker_bytes=4, device=None):
    """rank `src` holds the assembled body (None elsewhere); every rank receives buffer_span() of its
    body_ranges() range (dist.send / recv, as assemble_body).  -> this rank's buffer"""
    rank, world = dist.get_rank(), dist.get_world_size()
    ranges = body_ranges(body_len, world)
    if rank == src:
        reqs = []
        for r, (lo, hi) in enumerate(ranges):
            b0, b1 = buffer_span(lo, hi, body_len, marker_bytes)
            if r != src and b1 > b0:
                reqs.append(dist.isend(body[b0:b1].contiguous(), r))
        for q in reqs:
            q.wait()
        b0, b1 = buffer_span(*ranges[rank], body_len, marker_bytes)
        return body[b0:b1]
    b0, b1 = buffer_span(*ranges[rank], body_len, marker_bytes)
    buf = torch.empty(b1 - b0, dtype=torch.uint8, device=device if device is not None else _device())
    if b1 > b0:
        dist.recv(buf, src)
    return buf


def decompress_sharded(buf, lo, hi, body_len, orig_size, marker=b"\xff\xff\x00\x00", known_mask=None, gather_to=None):
    """Decode one .ambc body whose byte ranges are spread over the ranks (body_ranges() order; buf =
    body[buffer_span(lo, hi)] on this rank's GPU).  Phase 1 indexes the range locally, the fold walks the
    package chain across the ranges in rank order, every rank fetches the payload bytes its last decoded
    package needs from the next ranks, lists and decodes its own part.
    -> (out_offset, output slice, status [codec errors, length mismatches]) of this rank.
    gather_to=dst: the slices are also sent to rank dst, which returns (0, the whole output, summed status).
    A marker mismatch the serial walk would hit raises ValueError("Marker mismatch in chunk header.") on
    every rank."""
    from . import _lib as L
    from . import engine
    km = L.NATIVE_MASK if known_mask is None else known_mask
    rank, world = dist.get_rank(), dist.get_world_size()
    mb = len(marker)
    dev = buf.device
    ranges = body_ranges(body_len, world)
    assert ranges[rank] == (lo, hi), "ranges follow body_ranges(body_len, world)"
    ri = engine.range_index(buf, lo, hi, body_len, orig_size, marker, km)
    # fold: rank r - 1 -> rank r
    w = torch.empty(STATE_WORDS, dtype=torch.int64, device=dev)
    if rank == 0:
        entry = engine.range_init_state()
    else:
        dist.recv(w, rank - 1)
        entry = state_from_words(w.cpu().tolist())
    exit_ = engine.range_fold(ri, entry)
    if rank + 1 < world:
        dist.send(torch.tensor(state_to_words(exit_), dtype=torch.int64, device=dev), rank + 1)
    # every rank learns every entry state and the walk's final state
    mine = torch.tensor(state_to_words(entry) + state_to_words(exit_), dtype=torch.int64, device=dev)
    allw = torch.empty(2 * STATE_WORDS * world, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(allw, mine)
    rows = allw.view(world, 2 * STATE_WORDS).cpu().tolist()
    if int(rows[-1][2 * STATE_WORDS - 1]) == L.RANGE_MARKER:
        raise ValueError("Marker mismatch in chunk header.")  # adaptive_compressor.py:407
    entries = [state_from_words(r[:STATE_WORDS]) for r in rows]
    slices = output_slices(entries, ranges, orig_size, mb, km)
    o0, o1 = slices[rank]
    # payload bytes behind the halo
    _, _, _, _, need = engine.range_table(ri, entry, count_only=True)
    needs = torch.empty(world, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(needs, torch.tensor([need], dtype=torch.int64, device=dev))
    plan = tail_fetch_plan(ranges, needs.cpu().tolist(), body_len, mb)
    if need:
        grown = torch.empty(buf.numel() + need, dtype=torch.uint8, device=dev)
        grown[:buf.numel()].copy_(buf)
        buf = grown
    reqs = []
    for src, dst, g0, g1 in plan:
        if src == rank:
            reqs.append(dist.isend(buf[g0 - lo:g1 - lo].contiguous(), dst))
        elif dst == rank:
            reqs.append(dist.irecv(buf[g0 - lo:g1 - lo], src))
    for q in reqs:
        q.wait()
    t_table, n, _, _, _ = engine.range_table(ri, entry)
    out, status = engine.range_decode(buf, t_table, n, o1 - o0, km)
    if gather_to is None:
        return o0, out, status
    st = torch.tensor(status, dtype=torch.int64, device=dev)
    dist.all_reduce(st)
    if rank != gather_to:
        if o1 > o0:
            dist.send(out.contiguous(), gather_to)
        return o0, out, status
    whole = torch.empty(max(orig_size, 1), dtype=torch.uint8, device=dev)[:orig_size]
    reqs = []
    for r, (a, b) in enumerate(slices):
        if r == rank:
            whole[a:b].copy_(out)
        elif b > a:
            reqs.append(dist.irecv(whole[a:b], r))
    for q in reqs:
        q.wait()
    return 0, whole, [int(x) for x in st.cpu().tolist()]


# ---- the multi-candidate mode across ranks ------------------------------------------------------------------------
DYN_SEGU = 64      # positions (multiples of g) per segment of the chain walk
DYN_HALO = 8192    # the winner at p depends on input[p, p + 8192) (and on n - p)
DYN_TABLE_WORDS = 4 * 32 + 1


def _gcd_of(candidates):
    import math
    g = 0
    for c in candidates:
        g = math.gcd(g, int(c))
    return g


def dyn_shard_ranges(n, candidates, world):
    """[(lo, hi)] per rank: whole segments of 64 * g input bytes, the last non-empty range ends at n; trailing
    ranks are empty (n, n) when there are fewer segments than ranks"""
    seglen = DYN_SEGU * _gcd_of(candidates)
    n_seg = -(-n // seglen)
    per = -(-n_seg // world) if world else 0
    return [(min(n, r * per * seglen), min(n, (r + 1) * per * seglen)) for r in range(world)]


def dyn_buffer_span(lo, hi, n):
    """input bytes [b0, b1) a rank holds for its range: the range and the 8192-byte halo behind it"""
    return lo, min(n, hi + DYN_HALO) if hi > lo else lo


def fold_dyn_entries(tables, n):
    """tables[r] = rank r's entry rows [(entry, status, exit, stop)] (exit / stop None when absent), rank order.
    Follows the chain from position 0 through the ranks -> (entries, stuck, stop): entries[r] = the true entry
    into rank r (None: the chain ended or stopped before it), stuck = the first rank whose true entry is
    unresolved (None once the fold is complete), stop = where the rest of the file becomes one raw package (None)"""
    from . import _lib as L
    entries, e = [None] * len(tables), 0
    for r, tab in enumerate(tables):
        if e >= n:
            break
        if not tab:
            continue  # an empty range
        row = entry_row(tab, e, "rank %d" % r)
        entries[r] = e
        _, status, exit_, stop = row
        if status == L.DYN_UNRESOLVED:
            return entries, r, None
        if stop is not None:
            return entries, None, stop
        e = exit_
    return entries, None, None


def entry_row(tab, e, where):
    """the row of entry e in a walked range's entry table [(entry, status, exit, stop)]"""
    row = next((t for t in tab if t[0] == e), None)
    if row is None:
        raise RuntimeError("the chain enters %s at %d, which its entry table does not hold" % (where, e))
    return row


def dyn_fragment_plan(records, ranges, n, marker_bytes=4):
    """records[r] = (bytes of rank r's encoded packages, stop or -1); ranges = dyn_shard_ranges().
    -> ([(offset, length, state)] per rank, body length): the first rank whose chain stops writes the raw
    header and its input bytes [stop, hi), later ranks their input [lo, hi) verbatim, the last rank the END
    package.  A raw package of 4 GiB or more cannot be framed (adaptive_compressor.py:617-619)."""
    ovh, end = marker_bytes + 14, marker_bytes + 12
    refuse_dyn_raw(n, next((int(st) for _, st in records if st >= 0), -1))
    plan, off, raw_seen = [], 0, False
    for r, ((nbytes, st), (lo, hi)) in enumerate(zip(records, ranges)):
        if raw_seen:
            state, length = "in_raw_tail", hi - lo
        elif st >= 0:
            state, length, raw_seen = "raw_starts_here", nbytes + ovh + (hi - st), True
        else:
            state, length = "packed", nbytes
        if r == len(records) - 1:
            length += end
        plan.append((off, length, state))
        off += length
    return plan, off


def _all_rows(tab, dev):
    """all-gather of every rank's entry table (fixed size) -> list of row lists"""
    from . import _lib as L
    world = dist.get_world_size()
    words = [len(tab)]
    for e, st, ex, sp in tab:
        words += [e, st, -1 if ex is None else ex, -1 if sp is None else sp]
    words += [0] * (DYN_TABLE_WORDS - len(words))
    allw = torch.empty(DYN_TABLE_WORDS * world, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(allw, torch.tensor(words, dtype=torch.int64, device=dev))
    out = []
    for row in allw.view(world, DYN_TABLE_WORDS).cpu().tolist():
        k = int(row[0])
        out.append([(int(row[1 + 4 * i]), int(row[2 + 4 * i]), None if row[3 + 4 * i] < 0 else int(row[3 + 4 * i]),
                     None if row[4 + 4 * i] < 0 else int(row[4 + 4 * i])) for i in range(k)])
    assert all(len(t) <= L.DYN_MAX_ENTRIES for t in out)
    return out


def settle_dyn_entries(table, n, resolve, dev):
    """the fold loop: all-gather every rank's entry table, fold, let the first rank whose true entry is unresolved
    resolve it (resolve(entry) -> its updated table), repeat; at most one round per rank.
    -> (entries, stop, rounds) as fold_dyn_entries gives them once complete"""
    rank, world = dist.get_rank(), dist.get_world_size()
    for rounds in range(1, world + 1):
        entries, stuck, stop = fold_dyn_entries(_all_rows(table, dev), n)
        if stuck is None:
            return entries, stop, rounds
        if stuck == rank:
            table = resolve(entries[rank])
    raise RuntimeError("the fold of the entry tables does not settle within %d rounds" % world)


def dyn_fragment(frag, stop, state, t_buf, lo, hi, n, marker, last):
    """the bytes a rank contributes to the body (dyn_fragment_plan state): its packages, then the raw header and its
    input bytes [stop, hi) when its chain stops there, or its input [lo, hi) inside the raw tail; END on the last
    rank.  t_buf = input[lo, ...) on the rank's device."""
    dev = t_buf.device
    parts = [frag]
    if state == "raw_starts_here":
        parts += [torch.tensor(list(raw_package_header(marker, n - stop)), dtype=torch.uint8, device=dev),
                  t_buf[stop - lo:hi - lo]]
    elif state == "in_raw_tail":
        parts = [t_buf[:hi - lo]]
    if last:
        parts.append(torch.tensor(list(end_package(marker)), dtype=torch.uint8, device=dev))
    return torch.cat(parts) if len(parts) > 1 else parts[0]


def compress_dynamic_sharded(t_buf, lo, hi, n, candidates, mask=None, flags=0, marker=b"\xff\xff\x00\x00", dst=0):
    """Multi-candidate compression of an input whose ranges are spread over the ranks (dyn_shard_ranges() order;
    t_buf = input[dyn_buffer_span(lo, hi, n)] on this rank's GPU).  -> (body on `dst` (None elsewhere), the package
    list [(type, orig, comp)], usage [raw, 1..4], payload bytes): what engine.compress_dynamic_device gives for the
    whole input.  Raises AmbcError(E_ARG) on every rank where the single-GPU call would."""
    from . import _lib as L
    from . import engine
    mask = L.NATIVE_MASK if mask is None else mask
    rank, world = dist.get_rank(), dist.get_world_size()
    ranges = dyn_shard_ranges(n, candidates, world)
    assert ranges[rank] == (lo, hi), "ranges follow dyn_shard_ranges(n, candidates, world)"
    dev = t_buf.device
    mb = len(marker)
    dr = engine.dyn_range_walk(t_buf, lo, hi, n, candidates, mask, flags, mb)

    def resolve(entry):
        engine.dyn_range_resolve(dr, entry)
        return dr.table
    entries, _, _ = settle_dyn_entries(dr.table, n, resolve, dev)
    mine = entries[rank]
    if mine is not None and mine < hi:
        frag, my_stop, pk, usage, payload = engine.dyn_range_encode(dr, mine, marker)
    else:
        frag, my_stop, pk, usage, payload = t_buf[:0], None, [], [0] * 5, 0
    rec = torch.tensor([frag.numel(), -1 if my_stop is None else my_stop], dtype=torch.int64, device=dev)
    allr = torch.empty(2 * world, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(allr, rec)
    records = [tuple(int(x) for x in r) for r in allr.view(world, 2).cpu().tolist()]
    plan, body_len = dyn_fragment_plan(records, ranges, n, mb)
    _, _, state = plan[rank]
    local = dyn_fragment(frag, my_stop, state, t_buf, lo, hi, n, marker, rank == world - 1)
    body = gather_fragments(local, plan, body_len, dst)
    # the package list and the counters, with the raw tail package of the rank that stops
    if state == "raw_starts_here":
        pk = pk + [(my_stop, 255, n - my_stop, n - my_stop)]
        usage = [usage[0] + 1] + usage[1:]
    lists = [None] * world
    dist.all_gather_object(lists, pk)
    cnt = torch.tensor(list(usage) + [payload], dtype=torch.int64, device=dev)
    dist.all_reduce(cnt)
    cnt = cnt.cpu().tolist()
    packages = [(t, o, c) for part in lists for _, t, o, c in part]
    return body, packages, [int(x) for x in cnt[:5]], int(cnt[5])
