#!/usr/bin/env python3
"""bench.py -- the hot path's headline benchmark (BASELINE.json): compress + decompress
round trip, input GB/s, on the synthetic mixed CSV/log/binary corpus, chunk 4096, repo-native
methods only.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--size-mib M] [--dump-outputs DIR]

N = 1 : configs[1], 1 GiB on one B200.  N > 1 (torchrun): configs[3] -- every rank takes a contiguous
4 GiB chunk-range shard of a 4 N GiB corpus (weak scaling; 32 GiB at 8 GPUs), compresses it, the 16-byte
shard placement records are all-gathered (SURVEY.md §8e) and every rank's fragment is sent into its placed
slice of ONE body on rank 0 (NCCL send / recv over NVLink) -- placement and assembly are inside the timed
compress.

One step = compress the resident shard (device input -> device .ambc body) then decompress it
(device body -> package index built on the GPU -> device output).  `value` = bytes / (t_compress + t_decompress),
timed with CUDA events, max over ranks.  `e2e` = the same round trip through the C-ABI
host-buffer calls (pinned host input -> host body -> host output; H2D, kernels, host index
walk, D2H inside the timed region).  Inputs are 1 GiB >> 126 MB of L2, so nothing is served from
cache between iterations.

--impl reference times the reference's algorithm on the host cores: the reference itself is
pure Python (~7 KB/s, SURVEY.md §6) and cannot travel to the GPU box, so the arm runs the C
restatement of it (oracle/, proven byte-identical on the golden vectors) with every host thread
on a bounded sample of the same workload."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "compress+decompress round-trip input throughput"
UNIT = "GB/s"
CHUNK = 4096


def workload_config(size_mib, n_gpus):
    name = "configs[1]" if n_gpus == 1 else "configs[3] (%d GiB corpus sharded by chunk range, one body assembled on rank 0)" % (size_mib * n_gpus >> 10)
    return {"workload": "%s: %d MiB/GPU synthetic mixed CSV/log/runs/lowcard/binary/text corpus, chunk 4096, "
                        "methods RLE+Dictionary+Huffman+Delta (third-party disabled), strict reference semantics, "
                        "compress + decompress round trip" % (name, size_mib),
            "bytes_per_gpu": size_mib << 20, "chunk": CHUNK, "seed": "0xA3BC0001", "sharding": "contiguous chunk ranges, %d shard(s)" % n_gpus,
            "cache": "inputs larger than L2 (no flush needed)"}


# ------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port on the host cores
# ------------------------------------------------------------------------------------------
def cpu_port_run(sample_bytes, steps, warmup, threads):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    import oracle as O
    import synth_ref
    lib = O.lib()
    data = synth_ref.corpus(sample_bytes, 0)
    meth = np.array([1, 2, 3, 4], dtype=np.int32)
    per = (sample_bytes // CHUNK + threads - 1) // threads * CHUNK
    outs = [np.empty(per + (per // CHUNK + 2) * 18 + 64, dtype=np.uint8) for _ in range(threads)]
    decs = [np.empty(per + 64, dtype=np.uint8) for _ in range(threads)]
    out_ptrs = (C.c_void_p * threads)(*[o.ctypes.data for o in outs])
    dec_ptrs = (C.c_void_p * threads)(*[o.ctypes.data for o in decs])
    lens = np.zeros(threads, dtype=np.int64)
    origs = np.array([max(0, min(per, sample_bytes - t * per)) for t in range(threads)], dtype=np.int64)
    O.set_lz_fast(False)  # the reference's own O(n * window) match search
    tc = td = 0.0
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        lib.orc_mt_compress(data.ctypes.data, sample_bytes, CHUNK, meth.ctypes.data, 4, threads, out_ptrs,
                            lens.ctypes.data)
        t1 = time.perf_counter()
        lib.orc_mt_decompress(out_ptrs, lens.ctypes.data, origs.ctypes.data, threads, dec_ptrs)
        t2 = time.perf_counter()
        if it >= warmup:
            tc += t1 - t0
            td += t2 - t1
    back = np.concatenate([decs[t][:origs[t]] for t in range(threads)])
    assert np.array_equal(back, data), "CPU port round trip failed"
    # the slices are chunk-aligned, so their bodies without the 16-byte END packages, concatenated, plus one
    # END are the body of the whole sample (the corpus has a winner in every chunk: no raw tail)
    body = np.concatenate([outs[t][:max(0, lens[t] - 16)] for t in range(threads)] + [outs[0][lens[0] - 16:lens[0]]])
    return {"compress_s": tc / steps, "decompress_s": td / steps, "bytes": sample_bytes, "body": body}


def cpu_sample_bytes(args, threads, budget_s=10.0):
    """bytes per CPU pass: --cpu-sample-mib when given, else calibrated on 8 MiB so that one pass takes
    about `budget_s` seconds on this box's host cores (16 MiB .. 512 MiB, whole 16 MiB units)"""
    if args.cpu_sample_mib:
        return args.cpu_sample_mib << 20
    r = cpu_port_run(8 << 20, 1, 0, threads)
    rate = (8 << 20) / (r["compress_s"] + r["decompress_s"])
    mib = int(rate * budget_s) >> 20
    return max(16, min(512, mib // 16 * 16)) << 20


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if not args.size_mib:
        args.size_mib = 1024 if int(os.environ.get("WORLD_SIZE", "1")) == 1 else 4096
    threads = os.cpu_count() or 1
    sample = cpu_sample_bytes(args, threads)
    args.cpu_sample_mib = sample >> 20
    r = cpu_port_run(sample, max(1, args.steps), min(args.warmup, 1), threads)
    t = r["compress_s"] + r["decompress_s"]
    value = sample / t / 1e9
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(args.size_mib, args.gpus),
            "compress_gbps": sample / r["compress_s"] / 1e9, "decompress_gbps": sample / r["decompress_s"] / 1e9,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                             "sample": "first %d MiB of the same corpus per step; C restatement of the reference "
                                       "(naive window scan as compression_methods.py:283-313), %d threads over "
                                       "chunk-aligned slices" % (args.cpu_sample_mib, threads)},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML (pynvml) every 10 ms,
    nvidia-smi as the fallback."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []      # (sm_mhz, max_mhz, [reason names])
        self.stop = False
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical devices; honour CUDA_VISIBLE_DEVICES remapping when it is a plain list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = index
            if vis:
                ids = [v.strip() for v in vis.split(",") if v.strip()]
                if index < len(ids) and ids[index].isdigit():
                    phys = int(ids[index])
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml = pynvml
        except Exception:  # noqa: BLE001
            self.nvml = None
        self.th = threading.Thread(target=self._run, daemon=True)

    def _sample_nvml(self):
        n = self.nvml
        sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
        try:
            r = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
        except Exception:  # noqa: BLE001
            r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        names = []
        for name, attr in (("hw_slowdown", "nvmlClocksThrottleReasonHwSlowdown"),
                           ("hw_thermal_slowdown", "nvmlClocksThrottleReasonHwThermalSlowdown"),
                           ("sw_thermal_slowdown", "nvmlClocksThrottleReasonSwThermalSlowdown"),
                           ("sw_power_cap", "nvmlClocksThrottleReasonSwPowerCap")):
            bit = getattr(n, attr, 0)
            if bit and (r & bit):
                names.append(name)
        self.rows.append((float(sm), float(mx), names))

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
        parts = [p.strip() for p in out.strip().split(",")]
        if len(parts) >= 6 and parts[0].replace(".", "").isdigit():
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            self.rows.append((float(parts[0]), float(parts[1]),
                              [n for i, n in enumerate(names) if parts[2 + i].lower().startswith("active")]))

    def _run(self):
        while not self.stop:
            try:
                if self.nvml:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:  # noqa: BLE001
                if self.nvml:
                    self.nvml = None  # fall back to nvidia-smi
            time.sleep(0.01)

    def __enter__(self):
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        self.th.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        reasons = sorted({n for r in self.rows for n in r[2]})
        return {"sm_mhz": statistics.median(r[0] for r in self.rows), "sm_max_mhz": max(r[1] for r in self.rows),
                "reasons": reasons, "samples": len(self.rows), "source": "nvml" if self.nvml else "nvidia-smi"}


# ------------------------------------------------------------------------------------------
# B200 arm
# ------------------------------------------------------------------------------------------
def per_kind_table(engine, lib, L, peak, mib=64):
    """k_select / decoders on 64 MiB of every corpus kind: ms, input GB/s and (N + C) / t against the HBM roof --
    the mixed corpus hides a 20 x spread between kinds"""
    import torch
    names = ["csv", "log", "runs", "lowcard", "binrec", "random", "text"]
    out = {}
    n = mib << 20
    lib.ambc_enable_timing(1)
    for k in (0, 1, 2, 3, 4, 6):
        t = engine.synth(n, 0, kind_mask=1 << k)
        sel, dec = [], []
        o = None
        for _ in range(3):
            o = engine.compress_device(t, CHUNK)
            ms = (C.c_float * 4)()
            lib.ambc_last_timing(ms)
            sel.append(ms[0])
        for _ in range(3):
            back, st = engine.decompress_device(o.body, n)
            ms = (C.c_float * 4)()
            lib.ambc_last_timing(ms)
            dec.append(ms[3])
        assert torch.equal(back, t) and st == [0, 0]
        s_ms, d_ms = min(sel), min(dec)
        c = int(o.body_len)
        out[names[k]] = {"k_select_ms": s_ms, "compress_gbps": n / (s_ms * 1e-3) / 1e9, "compress_frac": (n + c) / (s_ms * 1e-3) / 1e9 / peak,
                         "decode_ms": d_ms, "decode_gbps": n / (d_ms * 1e-3) / 1e9, "decode_frac": (n + c) / (d_ms * 1e-3) / 1e9 / peak,
                         "ratio": c / n, "usage_raw_rle_dict_huff_delta": [int(x) for x in o.usage]}
    lib.ambc_enable_timing(0)
    return {"bytes_per_kind": n, "note": "best of 3; k_select only / decode kernels only (device timers of the library)", "kinds": out}


def facade_file_to_file(data, n):
    """the reference-facing API end to end: AdaptiveCompressor(chunk_size=4096).compress(file, file) and
    .decompress(file, file) on the bench shard written to a temporary file (page cache), MD5 and file I/O inside;
    the MD5 of the input (compress) / output (decompress) is a serial chain that bounds both calls from below"""
    import hashlib
    import tempfile
    from adaptive_compression_b200 import AdaptiveCompressor
    d = tempfile.mkdtemp(prefix="ambc_bench_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    src, dst, back = (os.path.join(d, x) for x in ("in.bin", "out.ambc", "back.bin"))
    try:
        data[:n].tofile(src)
        t0 = time.perf_counter()
        hashlib.md5(data[:n]).digest()
        md5_s = time.perf_counter() - t0
        c = AdaptiveCompressor(chunk_size=CHUNK)
        c.compress(src, dst)
        c.decompress(dst, back)  # warm: pinned buffers, page cache
        tc, td = [], []
        for _ in range(2):
            t0 = time.perf_counter()
            st = c.compress(src, dst)
            t1 = time.perf_counter()
            c.decompress(dst, back)
            t2 = time.perf_counter()
            tc.append(t1 - t0)
            td.append(t2 - t1)
        with open(back, "rb") as f:
            ok = hashlib.md5(f.read()).digest() == hashlib.md5(data[:n]).digest()
        assert ok, "facade round trip mismatch"
        return {"compress_s": min(tc), "decompress_s": min(td), "md5_floor_s": md5_s,
                "compress_gbps": n / min(tc) / 1e9, "decompress_gbps": n / min(td) / 1e9, "md5_gbps": n / md5_s / 1e9,
                "compress_over_floor": min(tc) / md5_s, "decompress_over_floor": min(td) / md5_s,
                "ratio": st["ratio"], "where": "files in %s" % os.path.dirname(src),
                "note": "file -> file, MD5 (hashlib, one core) and file I/O inside; compress hashes while it reads, "
                        "decompress hashes while it writes"}
    finally:
        for x in (src, dst, back):
            if os.path.exists(x):
                os.remove(x)
        os.rmdir(d)


def full_size_parity(args, engine, t_in, n, threads):
    """same-run parity at the full size: the CUDA body of the whole shard against the CPU port with its indexed match
    search (proven equal to the naive scan on the golden vectors and on the baseline sample above)"""
    import numpy as np
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as O
    lib = O.lib()
    data = t_in.cpu().numpy()
    meth = np.array([1, 2, 3, 4], dtype=np.int32)
    per = (n // CHUNK + threads - 1) // threads * CHUNK
    outs = [np.empty(per + (per // CHUNK + 2) * 18 + 64, dtype=np.uint8) for _ in range(threads)]
    out_ptrs = (C.c_void_p * threads)(*[o.ctypes.data for o in outs])
    lens = np.zeros(threads, dtype=np.int64)
    O.set_lz_fast(True)
    t0 = time.perf_counter()
    lib.orc_mt_compress(data.ctypes.data, n, CHUNK, meth.ctypes.data, 4, threads, out_ptrs, lens.ctypes.data)
    dt = time.perf_counter() - t0
    O.set_lz_fast(False)
    body = np.concatenate([outs[t][:max(0, lens[t] - 16)] for t in range(threads)] + [outs[0][lens[0] - 16:lens[0]]])
    chk = engine.compress_device(t_in, CHUNK)
    same = int(chk.body_len) == body.size and bool(torch.equal(chk.body[:chk.body_len].cpu(), torch.from_numpy(body)))
    assert same, "parity: CUDA body of the whole shard differs from the CPU port's body"
    return {"bytes": n, "body_bytes": int(body.size), "equal": True, "cpu_seconds": dt,
            "oracle": "C port, indexed match search (lz_fast), %d threads" % threads}


DUMP_SEED = 0xA3BC0D00
DUMP_MAX_ELEMS = 6 << 20  # per array: two float32 samples of this size plus the counters stay under 64 MB


def dump_outputs(out_dir, body, decoded, res):
    """write what the last timed step returned, as float32 / float64 .npy files: the compressed body, the decoded
    output and the CompressResult counters.  An array longer than DUMP_MAX_ELEMS is written as the values at
    DUMP_MAX_ELEMS sorted positions drawn uniformly with numpy's default_rng(DUMP_SEED) (with replacement), so two
    runs whose arrays have the same length are sampled at the same positions."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in (("body", body), ("decoded", decoded)):
        n = t.numel()
        if n > DUMP_MAX_ELEMS:
            idx = np.sort(np.random.default_rng(DUMP_SEED).integers(0, n, DUMP_MAX_ELEMS))
            t = t[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy().astype(np.float32))
    counters = [res.body_len, res.n_chunks, res.first_raw, res.n_packages, res.payload_bytes] + list(res.usage)
    np.save(os.path.join(out_dir, "compress_result.npy"), np.array(counters, dtype=np.float64))


def bind_to_gpu_numa_node(index):
    """Pin this rank (and with it the first-touch placement of its pinned host buffers and the helper
    threads of the host package walk) to the CPUs of its GPU's NUMA node: with 8 ranks on one host the
    host-buffer path otherwise crosses sockets for half of its copies.  Returns a description or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        phys = index
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if index < len(ids) and ids[index].isdigit():
                phys = int(ids[index])
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(phys)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        dev = "/sys/bus/pci/devices/" + bus.lower()[-12:]
        node = int(open(dev + "/numa_node").read())
        cpulist = open(dev + "/local_cpulist").read().strip()
        cpus = set()
        for part in cpulist.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if node < 0 or not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": len(cpus)}
    except Exception:  # noqa: BLE001
        return None



def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from adaptive_compression_b200 import _lib as L
    from adaptive_compression_b200 import distributed as D
    from adaptive_compression_b200 import engine

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local) if world > 1 else None
    # stdout carries exactly one JSON line: anything libraries print meanwhile (the NCCL version banner
    # at the first collective, for one) goes to stderr
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = engine.require_cuda()
    if not args.size_mib:
        args.size_mib = 1024 if world == 1 else 4096
    n = args.size_mib << 20
    mask = L.NATIVE_MASK
    marker = engine.FIXED_MARKER

    # resident input: this rank's shard of the corpus
    t_in = engine.synth(n, offset=rank * n)
    bound = lib.ambc_compress_bound(n, CHUNK, 4)
    t_out = torch.empty(bound, dtype=torch.uint8, device="cuda")
    t_work = torch.empty(lib.ambc_compress_workspace_bytes(n, CHUNK), dtype=torch.uint8, device="cuda")
    t_dec = torch.empty(n, dtype=torch.uint8, device="cuda")
    t_status = torch.zeros(2, dtype=torch.int32, device="cuda")
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    res = L.CompressResult()

    def compress():
        L.check(lib.ambc_compress_dev(C.c_void_p(t_in.data_ptr()), n, CHUNK, mask, 0, marker, 4,
                                      C.c_void_p(t_out.data_ptr()), bound, C.c_void_p(t_work.data_ptr()),
                                      t_work.numel(), C.byref(res), stream))
        if world > 1:
            # shard placement: all-gather of (bytes before first raw, first raw chunk), then every fragment goes
            # into its placed slice of the one body on rank 0
            c0 = rank * (n // CHUNK)
            _, recs = D.place_shards(D.packed_bytes(res.body_len, n, res.first_raw, CHUNK), res.first_raw, c0, world)
            _, frag = D.shard_fragment(t_out[:res.body_len], t_in, res.first_raw, c0, CHUNK, n * world, recs, rank)
            return D.assemble_body(frag, recs, n * world, CHUNK, out=t_global)
        return None

    # destination of the assembled body (rank 0): the bound of the whole corpus
    t_global = torch.empty(lib.ambc_compress_bound(n * world, CHUNK, 4), dtype=torch.uint8, device="cuda") \
        if world > 1 and rank == 0 else None
    g_body = compress()
    if world > 1 and rank == 0:
        # the assembled body is the body of the whole corpus: its first shard-worth decodes to this rank's input
        # (full check against a single-GPU run: tests/test_gpu_multirank.py)
        assert g_body is not None and int(g_body.numel()) > 16 and bytes(g_body[-16:].cpu().tolist()) == marker + bytes(12)
    body_len = int(res.body_len)
    assert res.first_raw == -1, "bench corpus must have a native winner in every chunk"
    # package index: built on the GPU inside the timed decompress (ambc_index_dev); the host walk that the
    # host-buffer path overlaps with its copies is timed once for reference
    body_host = t_out[:body_len].cpu().numpy()
    t_idx0 = time.perf_counter()
    table, covered = engine.index_host(body_host, n, marker, mask)
    t_index = time.perf_counter() - t_idx0
    table_cap = len(table) + 16
    t_table = torch.empty(table_cap * 32, dtype=torch.uint8, device="cuda")
    ne, cov = C.c_uint64(0), C.c_uint64(0)
    idx_ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

    def decompress():
        idx_ev[0].record()
        L.check(lib.ambc_index_dev(C.c_void_p(t_out.data_ptr()), body_len, marker, 4, n, mask,
                                   C.c_void_p(t_table.data_ptr()), table_cap, C.byref(ne), C.byref(cov), stream))
        idx_ev[1].record()
        L.check(lib.ambc_decompress_dev(C.c_void_p(t_out.data_ptr()), body_len, C.c_void_p(t_table.data_ptr()),
                                        ne.value, C.c_void_p(t_dec.data_ptr()), n, C.c_void_p(t_status.data_ptr()),
                                        stream))

    decompress()
    torch.cuda.synchronize()
    assert torch.equal(t_dec, t_in), "round trip mismatch"
    assert t_status.cpu().tolist() == [0, 0]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        compress()
        decompress()
    lib.ambc_enable_timing(1)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3 * args.steps)]
    ksel, kscan, kpack, kdec, kidx = [], [], [], [], []
    barrier()
    launches0 = lib.ambc_launch_count()
    with ClockSampler(local) as clocks:
        for s in range(args.steps):
            ev[3 * s].record()
            g_body = compress()
            ev[3 * s + 1].record()
            decompress()
            ev[3 * s + 2].record()
            ms = (C.c_float * 4)()
            lib.ambc_last_timing(ms)
            ksel.append(ms[0]); kscan.append(ms[1]); kpack.append(ms[2]); kdec.append(ms[3])
            kidx.append(idx_ev[0].elapsed_time(idx_ev[1]))
        barrier()
    launches = lib.ambc_launch_count() - launches0
    lib.ambc_enable_timing(0)
    tc = sum(ev[3 * s].elapsed_time(ev[3 * s + 1]) for s in range(args.steps)) / args.steps
    td = sum(ev[3 * s + 1].elapsed_time(ev[3 * s + 2]) for s in range(args.steps)) / args.steps
    tt = torch.tensor([tc, td, tc + td], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    tc_m, td_m, tstep = tt.cpu().tolist()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, g_body if world > 1 else t_out[:res.body_len], t_dec, res)

    # e2e through the C-ABI host calls (pinned buffers)
    e2e_steps = max(1, args.steps)
    h_in = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    h_in.copy_(t_in)
    h_body = torch.empty(bound, dtype=torch.uint8, pin_memory=True)
    h_out = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    res2 = L.CompressResult()
    st2 = (C.c_uint32 * 2)()

    e2e_split = [0.0, 0.0]

    def e2e_once():
        t_a = time.perf_counter()
        L.check(lib.ambc_compress_host(C.c_void_p(h_in.data_ptr()), n, CHUNK, mask, 0, marker, 4,
                                       C.c_void_p(h_body.data_ptr()), bound, None, None, C.byref(res2)))
        t_b = time.perf_counter()
        L.check(lib.ambc_decompress_host(C.c_void_p(h_body.data_ptr()), res2.body_len, marker, 4, mask,
                                         C.c_void_p(h_out.data_ptr()), n, st2))
        e2e_split[0] += t_b - t_a
        e2e_split[1] += time.perf_counter() - t_b

    e2e_once()
    assert torch.equal(h_out, h_in), "e2e round trip mismatch"
    barrier()
    e2e_split[0] = e2e_split[1] = 0.0
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_once()
    barrier()
    te = (time.perf_counter() - t0) / e2e_steps
    te_t = torch.tensor([te], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(te_t, op=dist.ReduceOp.MAX)
    te = te_t.item()

    # fabric floor of the host-buffer round trip: the same bytes over PCIe (upload of the input and download of the
    # body, then upload of the body and download of the output, both directions at once) with no kernel at all, on
    # every rank at the same time -- what the shared host side of this box can move for N ranks
    floor_info = None
    if world > 1:
        s_up, s_dn = torch.cuda.Stream(), torch.cuda.Stream()
        d_a = torch.empty(n, dtype=torch.uint8, device="cuda")
        d_b = torch.empty(body_len, dtype=torch.uint8, device="cuda")

        def floor_once():
            with torch.cuda.stream(s_up):
                d_a.copy_(h_in, non_blocking=True)
            with torch.cuda.stream(s_dn):
                h_body[:body_len].copy_(d_b, non_blocking=True)
            torch.cuda.synchronize()
            with torch.cuda.stream(s_up):
                d_b.copy_(h_body[:body_len], non_blocking=True)
            with torch.cuda.stream(s_dn):
                h_out.copy_(d_a, non_blocking=True)
            torch.cuda.synchronize()

        floor_once()
        barrier()
        t0 = time.perf_counter()
        for _ in range(2):
            floor_once()
        barrier()
        tf = torch.tensor([(time.perf_counter() - t0) / 2], dtype=torch.float64, device="cuda")
        dist.all_reduce(tf, op=dist.ReduceOp.MAX)
        floor_info = {"ms_per_step": tf.item() * 1e3, "value": n * world / tf.item() / 1e9, "unit": UNIT,
                      "note": "copies only (H2D input || D2H body, then H2D body || D2H output), all ranks at once: the "
                              "host side of the box (one NUMA node exposed, no topology to bind to) bounds the e2e number"}
        del d_a, d_b

    # sharded marker search (MarkerFinder.find_marker over the whole N-shard stream): per-shard flags,
    # one NCCL MAX all-reduce, same pick on every rank.  Not part of `value` (a separate API).
    marker_info = None
    if world > 1:
        try:
            mev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            D.find_marker_sharded(t_in, 32)
            barrier()
            mev[0].record()
            mk, mk_bits = D.find_marker_sharded(t_in, 32)
            mev[1].record()
            torch.cuda.synchronize()
            mk_ms = mev[0].elapsed_time(mev[1])
            marker_info = {"marker_hex": mk.hex(), "bits": mk_bits, "ms": mk_ms,
                           "collective": "1 x all_gather(40 B/rank), then per level tried (16 bits: 2^16 B of flags; "
                                         "24 bits: 2^24 B) 1 x all_reduce(MAX) over NCCL; %d-bit result: %s" %
                                         (mk_bits, "16-bit level only" if mk_bits <= 16 else "both levels ran"),
                           "roofline": {"bound": "hbm", "achieved": n / (mk_ms * 1e-3) / 1e9, "unit": "GB/s",
                                        "note": "shard bytes / time of the whole sharded search (flags kernels + collectives + pick)"}}
        except Exception as e:  # noqa: BLE001
            marker_info = {"error": str(e)[:200]}

    if rank == 0:
        peaks = {}
        pk_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
        if os.path.exists(pk_path):
            peaks = json.load(open(pk_path))
            peak, peak_src = float(peaks["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        traffic, traffic_source = args.traffic, "--traffic" if args.traffic is not None else None
        for tr_name in ("r02_traffic.json", "r01_traffic.json"):
            tr_path = os.path.join(ROOT, "profiles", tr_name)
            if traffic is None and os.path.exists(tr_path):
                tr = json.load(open(tr_path))
                if tr.get("bytes_per_gpu") == n and tr.get("chunk") == CHUNK:  # same launch shape as the capture
                    traffic = tr["traffic_bytes_per_launch"]
                    traffic_source = "profiles/%s (%s): a committed ncu capture of this launch shape, not a measurement of this run" % (
                        tr_name, tr.get("capture", "ncu --set full"))
        payload = int(res.payload_bytes)
        sel_ms = statistics.mean(ksel)
        algo_bytes = n + payload  # k_select reads the shard once and writes every winning payload once
        achieved = algo_bytes / (sel_ms * 1e-3) / 1e9
        total_bytes = n * world
        line = {
            "metric": METRIC, "value": total_bytes / (tstep * 1e-3) / 1e9, "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": tstep, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(args.size_mib, world),
            "compress_gbps": total_bytes / (tc_m * 1e-3) / 1e9, "decompress_gbps": total_bytes / (td_m * 1e-3) / 1e9,
            "compressed_ratio": body_len / n,
            "kernel_ms": {"k_select": sel_ms, "size_scan": statistics.mean(kscan), "k_pack": statistics.mean(kpack),
                          "k_decode": statistics.mean(kdec), "gpu_index": statistics.mean(kidx),
                          "host_index_walk_ms": t_index * 1e3},
            "roofline": {"bound": "hbm", "kernel": "k_select", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_source, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": algo_bytes,
                         "decode": {"kernel": "k_decode_warp (Huffman, RLE) + k_decode_lz (Dictionary, side stream) + k_decode (rest)", "achieved": (body_len + n) / (statistics.mean(kdec) * 1e-3) / 1e9,
                                    "frac": (body_len + n) / (statistics.mean(kdec) * 1e-3) / 1e9 / peak}},
            "e2e": {"value": total_bytes / te / 1e9, "unit": UNIT, "h2d_bytes_per_step": n + body_len + len(table) * 32,
                    "d2h_bytes_per_step": body_len + n, "ms_per_step": te * 1e3,
                    "compress_ms": e2e_split[0] / e2e_steps * 1e3, "decompress_ms": e2e_split[1] / e2e_steps * 1e3,
                    "note": "ambc_compress_host + ambc_decompress_host on pinned host buffers (piece-wise upload overlapping "
                            "k_select; host package walk overlapping decode and download); header MD5 (hashlib, "
                            "~0.6 GB/s/core, identical in both arms) is outside the chunk path"},
            "gpu_launches": int(launches), "clocks": clocks.summary(),
        }
        if marker_info is not None:
            line["marker_search"] = marker_info
        if floor_info is not None:
            line["e2e"]["fabric_floor"] = floor_info
            line["e2e"]["frac_of_fabric_floor"] = (total_bytes / te / 1e9) / floor_info["value"]
        if numa is not None:
            line["config"]["numa_binding"] = numa
        if world == 1 and not args.no_kinds:
            line["roofline"]["per_kind"] = per_kind_table(engine, lib, L, peak)
        if world == 1 and not args.no_facade:
            line["e2e_facade"] = facade_file_to_file(h_in.numpy(), n)
        if world == 1 and not args.no_cpu:
            threads = os.cpu_count() or 1
            args.cpu_sample_mib = cpu_sample_bytes(args, threads) >> 20
            r = cpu_port_run(args.cpu_sample_mib << 20, 1, 0, threads)
            v = (args.cpu_sample_mib << 20) / (r["compress_s"] + r["decompress_s"]) / 1e9
            # same-run parity (SURVEY.md 8d): the CUDA body of the sample == the CPU port's body, byte for byte
            chk = engine.compress_device(t_in[:args.cpu_sample_mib << 20], CHUNK)
            same = chk.body_len == r["body"].size and bool(
                torch.equal(chk.body[:chk.body_len].cpu(), torch.from_numpy(r["body"])))
            assert same, "parity: CUDA body differs from the CPU port's body on the baseline sample"
            pyref = None
            pr_path = os.path.join(ROOT, "profiles", "r02_python_reference_timing.json")
            if os.path.exists(pr_path):
                pr = json.load(open(pr_path))
                pyref = {"source": "profiles/r02_python_reference_timing.json (build container, oracle/time_python_reference.py; "
                                   "the reference cannot travel to the GPU box)",
                         "one_core_roundtrip_kb_s": pr["one_core"]["roundtrip_kb_s"],
                         "eight_processes_roundtrip_kb_s": pr["eight_processes"]["roundtrip_kb_s"],
                         "host": pr.get("host"), "cpus": pr.get("cpus")}
            full = full_size_parity(args, engine, t_in, n, threads) if not args.no_full_parity else None
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                                    "python_reference": pyref, "full_size_parity": full,
                                    "compress_gbps": (args.cpu_sample_mib << 20) / r["compress_s"] / 1e9,
                                    "decompress_gbps": (args.cpu_sample_mib << 20) / r["decompress_s"] / 1e9,
                                    "parity": "CUDA body == CPU port body on the sample (%d bytes), bit-exact" % r["body"].size,
                                    "sample": "first %d MiB of the same corpus, one pass; C restatement of the reference "
                                              "(oracle/), %d threads; the Python reference itself runs at ~7 KB/s on one "
                                              "core (BASELINE.md §2)" % (args.cpu_sample_mib, threads)}
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--size-mib", type=int, default=0, help="MiB per GPU (0: 1024 at N = 1 = configs[1], 4096 at N > 1 = configs[3])")
    ap.add_argument("--no-kinds", action="store_true", help="skip the per-kind table (roofline.per_kind)")
    ap.add_argument("--cpu-sample-mib", type=int, default=0,
                    help="MiB of the corpus the CPU legs process per pass (0 = calibrate to ~10 s per pass)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-facade", action="store_true", help="skip the file -> file run through AdaptiveCompressor")
    ap.add_argument("--no-full-parity", action="store_true", help="skip the CPU body of the whole shard (indexed oracle)")
    ap.add_argument("--traffic", type=float, default=None,
                    help="dram bytes per k_select launch from the committed ncu capture (profiles/)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's body, decoded output and counters as DIR/<name>.npy "
                         "(float32 / float64, a seeded sample of arrays longer than %d elements)" % DUMP_MAX_ELEMS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
