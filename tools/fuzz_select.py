"""dev tool: randomized parity fuzz of the chunk selection (k_select_fast) against the oracle, aimed at
the Huffman-first / early-abort path: small alphabets with varying skew, repeated fragments of varying
length and density (so that the Dictionary method wins, loses narrowly, or loses clearly), runs."""
import sys, os, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "oracle"))
import numpy as np, torch
import oracle as O
from adaptive_compression_b200 import engine
engine.require_cuda()
seed = int(sys.argv[1]) if len(sys.argv) > 1 else 1
budget = float(sys.argv[2]) if len(sys.argv) > 2 else 60.0
r = np.random.RandomState(seed)
t0 = time.time(); files = 0; chunks = 0; usage = np.zeros(5, dtype=np.int64)
while time.time() - t0 < budget:
    chunk = int(r.choice([1024, 2048, 4096, 4096, 4096, 3000, 8192, 6000]))
    parts = []
    for _ in range(int(r.randint(4, 40))):
        n = chunk if r.rand() < 0.8 else int(r.randint(1, chunk + 1))
        K = int(r.choice([2, 3, 4, 6, 8, 12, 16, 20, 32, 48, 64, 128, 200]))
        w = r.rand(K) ** float(r.choice([0.5, 1, 2, 4, 8]))
        a = r.choice(K, size=n, p=w / w.sum()).astype(np.uint8)
        a = (a * int(r.choice([1, 3, 7])) + int(r.randint(0, 200))).astype(np.uint8)
        # sprinkle repeated fragments
        nfrag = int(r.choice([0, 2, 8, 30, 100, 200, 300, 450, 600]))
        for _ in range(nfrag):
            L = int(r.choice([3, 4, 5, 7, 8, 9, 12, 16, 20, 31, 32, 40]))
            if n > 2 * L + 2:
                s = int(r.randint(0, n - L)); d = int(r.randint(0, n - L))
                a[d:d + L] = a[s:s + L].copy()
        if r.rand() < 0.15:
            s = int(r.randint(0, n)); a[s:s + int(r.randint(1, 600))] = int(r.randint(256))
        parts.append(a)
    if r.rand() < 0.5:  # record-like text: fixed field layouts with random digits / words (the prefix-trial regime)
        rows = []
        words = [b"alpha", b"beta", b"gamma", b"delta", b"eps", b"GET", b"POST", b"/v1/items/", b"ok", b"ERROR", b"warn"]
        fmt = [int(r.randint(0, 4)) for _ in range(int(r.randint(3, 9)))]
        while sum(len(x) for x in rows) < chunk * int(r.randint(3, 12)):
            row = []
            for f in fmt:
                if f == 0: row.append(b"%d" % r.randint(0, 10 ** int(r.randint(1, 9))))
                elif f == 1: row.append(words[int(r.randint(len(words)))])
                elif f == 2: row.append(b"%d.%02d" % (r.randint(0, 1000), r.randint(0, 100)))
                else: row.append(b"2026-%02d-%02d" % (r.randint(1, 13), r.randint(1, 29)))
            rows.append(b",".join(row) + b"\n")
        parts = [np.frombuffer(b"".join(rows), dtype=np.uint8)]
    data = np.concatenate(parts)
    out = engine.compress_device(torch.from_numpy(data).cuda(), chunk)
    body = out.body.cpu().numpy()[:out.body_len].tobytes()
    want, pm = O.compress_body(data.tobytes(), chunk)
    if body != want:
        got = engine.package_map(out, data.size, chunk)
        bad = next((i for i, (x, y) in enumerate(zip(got, pm)) if tuple(x) != tuple(y)), None)
        np.save("gpurun_out/fuzz_fail_%d.npy" % seed, data)
        print("MISMATCH seed", seed, "file", files, "chunk size", chunk, "first differing package", bad,
              None if bad is None else (got[bad], pm[bad]), flush=True)
        sys.exit(1)
    for i in range(5): usage[i] += out.usage[i]
    files += 1; chunks += len(pm)
print("fuzz ok: seed %d, %d files, %d packages, usage [raw,rle,dict,huff,delta] %s, %.0f s" % (seed, files, chunks, usage.tolist(), time.time() - t0))
