#!/usr/bin/env python
"""Dump the SNB_TC_DEBUG=8 clock64 trace of one slot (leader CTA of cluster 0) as a timeline."""
import ctypes as C
import os
import subprocess
import sys

os.environ["SNB_TC_DEBUG"] = "8"
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.argv = [sys.argv[0], "--precision", sys.argv[1] if len(sys.argv) > 1 else "f16x3", "--rays", "8000", "--iters", "1"]
exec(open(os.path.join(os.path.dirname(__file__), "time_field.py")).read())
buf = (C.c_longlong * 2048)()
lib.snb_debug_trace.argtypes = [C.POINTER(C.c_longlong), C.c_int]
assert lib.snb_debug_trace(buf, 2048) == 0
t = list(buf)
t0 = min(t[ci * 4] for ci in range(35) if t[ci * 4] > 0)   # rotated order: chunks 0/1 are issued near the END of the slot
print("MMA warp: chunk: [loop top] [after A/enc waits] [after full wait] [after issue]   (cycles since slot start)")
for ci in range(35):
    a, b, c, d = (t[ci * 4 + k] - t0 for k in range(4))
    i0, i1, c0, c1 = (t[512 + ci * 4 + k] - t0 for k in range(4))
    two = i1 > 0 and i1 > i0
    print(f"  chunk {ci:2d}: {a:7d} {b:7d} (+{b - a:5d} wait A)  {c:7d} (+{c - b:5d} wait full)  {d:7d} (+{d - c:4d} issue)"
          f"   [mma part0 +{i0 - c:4d}" + (f", part1 at +{i1 - c:4d}" if two else "") + f", commit empty +{c0 - c:4d}, commits done +{c1 - c:4d}]")
print("epilogue warp 0: (layer, half): [start waiting d_full] [observed] [ld done] [q0 signalled] [q1 signalled]")
for lh in range(16):
    e = [t[1024 + lh * 8 + k] - t0 for k in range(5)]
    print(f"  l={lh // 2} h={lh % 2}: wait_from {e[0]:7d}  d_full {e[1]:7d}  ld {e[2] - e[1]:5d}  q0 +{e[3] - e[1]:5d}  q1 +{e[4] - e[1]:5d}")
e = [t[1024 + 18 * 8 + k] - t0 for k in range(6)]
print(f"  dir layer: wait_from {e[0]:7d}  d_full {e[1]:7d}  drained +{e[2] - e[1]:5d}  math +{e[3] - e[1]:5d}  head/out +{e[4] - e[1]:5d}")
print(f"  deferred pieces (next slot): first piece starts {e[5] + t0 - t0:7d}" if t[1024 + 18 * 8 + 5] > 0 else "  (direction-layer epilogue not deferred)")
print(f"  slot length (MMA warp, first chunk top -> chunk 34 issued): {t[34 * 4 + 3] - t0}")
