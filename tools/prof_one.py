"""dev tool: run k_select_fast on one corpus kind (for ncu)"""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from adaptive_compression_b200 import engine
kind = int(sys.argv[1]); mib = int(sys.argv[2])
t = engine.synth(mib << 20, 0, kind_mask=1 << kind)
for _ in range(3):
    o = engine.compress_device(t, 4096)
print(o.body_len / (mib << 20), o.usage)
