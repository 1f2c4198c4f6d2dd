"""CPU: bench.py's --dump-outputs writes float32 / float64 arrays within 64 MB, samples long arrays at the same
seeded positions on every run, and --steps below 1 is refused."""
import os
import subprocess
import sys

import numpy as np
import torch

import bench
from adaptive_compression_b200 import _lib as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_is_small_typed_and_repeatable(tmp_path):
    res = L.CompressResult()
    res.body_len, res.n_chunks, res.first_raw, res.n_packages, res.payload_bytes = 1000, 3, -1, 4, 946
    res.usage[2] = 3
    g = torch.Generator().manual_seed(1)
    body = torch.randint(0, 256, (1000,), dtype=torch.uint8, generator=g)
    decoded = torch.randint(0, 256, (bench.DUMP_MAX_ELEMS + 4097,), dtype=torch.uint8, generator=g)
    runs = []
    for k in range(2):
        d = tmp_path / str(k)
        bench.dump_outputs(str(d), body, decoded, res)
        runs.append({n: np.load(d / (n + ".npy")) for n in ("body", "decoded", "compress_result")})
        assert sum(os.path.getsize(d / f) for f in os.listdir(d)) <= 64 << 20
    a, b = runs
    assert a["body"].dtype == np.float32 and np.array_equal(a["body"], body.numpy())
    assert a["decoded"].dtype == np.float32 and a["decoded"].size == bench.DUMP_MAX_ELEMS
    assert np.array_equal(a["decoded"], b["decoded"])
    idx = np.sort(np.random.default_rng(bench.DUMP_SEED).integers(0, decoded.numel(), bench.DUMP_MAX_ELEMS))
    assert np.array_equal(a["decoded"], decoded.numpy()[idx])
    assert a["compress_result"].dtype == np.float64
    assert a["compress_result"].tolist() == [1000, 3, -1, 4, 946, 0, 0, 3, 0, 0]


def test_steps_below_one_is_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True,
                       text=True, cwd=ROOT)
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr
