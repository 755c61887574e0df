"""Per-warp phase timeline of the stream program kernel (knob 3 = 8): 4 Llama-3-8B layers, first 16 ops, first 8 CTAs.
For every op prints, relative to the earliest warp's op begin over the 8 CTAs (ns; min / median / max over the 64 warps):
begin, own polls done, staged, first chunk, own units done, past post-loop barrier, finish stores issued."""
import ctypes
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from autoawq_b200 import ext  # noqa: E402
from autoawq_b200._cabi import lib  # noqa: E402
from autoawq_b200.program import DecodeProgram  # noqa: E402

dev = torch.device("cuda:0")
for kv in sys.argv[1:]:      # KEY=VALUE library knobs, e.g. 14=2 (no fall-back to the split-K kernel)
    k, v = kv.split("=")
    ext.set_knob(int(k), int(v))
print("knobs:", sys.argv[1:])
rep = bench.Replica(dev, 1, layers=4)
prog = DecodeProgram()
rep.step(rep.h, api=prog)
prog.build()
runs = []
for it in range(6):
    ext.set_knob(3, 8)
    prog.run()
    torch.cuda.synchronize()
    buf = np.zeros((16, 8, 8, 8), dtype=np.uint64)
    lib.b200awq_debug_read(buf.ctypes.data_as(ctypes.c_void_p), buf.nbytes)
    ext.set_knob(3, 0)
    if it >= 2:
        runs.append(buf.astype(np.int64))
r = np.stack(runs)   # [run, op, cta, warp, slot]
names = ["begin", "polled", "staged", "1st chunk", "units done", "post-bar", "finished"]
print("op  shape    " + "".join(f"{n:>22s}" for n in names) + "   (min/med/max over 64 warps, ns after the op's earliest begin)")
shapes = ["qkv", "o", "gate_up", "down"]
for op in range(16):
    t0 = r[:, op, :, :, 0].min(axis=(1, 2))[:, None, None]
    line = f"{op:2d}  {shapes[op % 4]:8s}"
    for s in range(7):
        d = r[:, op, :, :, s] - t0
        a, b, c = np.median(d.min(axis=(1, 2))), np.median(np.median(d, axis=(1, 2))), np.median(d.max(axis=(1, 2)))
        line += f"  {a:6.0f}/{b:6.0f}/{c:6.0f}"
    print(line)
span = r[:, 15, :, :, 6].max(axis=(1, 2)) - r[:, 0, :, :, 0].min(axis=(1, 2))
print("span of the 16 ops (ns):", np.median(span), " per op:", np.median(span) / 16)
