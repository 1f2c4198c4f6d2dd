"""dev tool: k_select_fast time per corpus kind for one library variant (AMBC_LIB_PATH)"""
import ctypes as C, sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from adaptive_compression_b200 import engine, _lib as L
lib = engine.require_cuda()
n = 64 << 20
names = ['csv', 'log', 'runs', 'lowcard', 'binrec', 'random', 'text']
lib.ambc_enable_timing(1)
row = []
for k in (0, 1, 2, 3, 4, 6):
    t = engine.synth(n, 0, kind_mask=1 << k)
    best = 1e9
    for _ in range(4):
        o = engine.compress_device(t, 4096)
        ms = (C.c_float * 4)(); lib.ambc_last_timing(ms)
        best = min(best, ms[0])
    row.append("%s %.2f" % (names[k], best))
print(os.environ.get("AMBC_LIB_PATH", "default"), " | ".join(row), flush=True)
