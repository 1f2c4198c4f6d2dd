"""dev tool: one dynamic-mode compress of 32 MiB (for an ncu launch list of the chain walk)"""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from adaptive_compression_b200 import engine
from adaptive_compression_b200.adaptive_compressor import REFERENCE_CANDIDATES
engine.require_cuda()
t = engine.synth(32 << 20, 0)
o = engine.compress_dynamic_device(t, REFERENCE_CANDIDATES)
print(o.body_len)
