"""Stage 2 only (band -> bidiagonal) timing on a synthetic band matrix.   python tools/stage2_only.py <n> <band> <f32|f64>"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from svdsolver_b200 import capi  # noqa: E402

n, b = int(sys.argv[1]), int(sys.argv[2])
dt = np.float32 if sys.argv[3] == "f32" else np.float64
tdt = torch.float32 if dt == np.float32 else torch.float64
h = capi.Handle(n, b, dt)
s = torch.cuda.Stream()
h.set_stream(s.cuda_stream)
g = torch.Generator(device="cuda").manual_seed(3)
band = torch.triu(torch.tril(torch.rand(n, n, device="cuda", dtype=tdt, generator=g) * 5, b))
d = torch.empty(n, device="cuda", dtype=tdt)
e = torch.empty(n, device="cuda", dtype=tdt)
times = []
for rep in range(3):
    a = band.clone()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s)
    h.band_to_bidiag_dev(a.data_ptr(), n, b, d.data_ptr(), e.data_ptr())
    e1.record(s)
    s.synchronize()
    times.append(e0.elapsed_time(e1))
ops = sum(2 * ((n - i + b - 1) // b) for i in range(n - 1))
print(f"stage2 n={n} b={b} {sys.argv[3]}: {min(times):.2f} ms  {[round(t, 2) for t in times]}  ~{min(times) * 1e6 / (4.0 * n):.0f} ns per op on the critical path", flush=True)

import ctypes
out = (ctypes.c_longlong * 16)()
capi.lib().svdb200_debug_stage2_timing(out)
if any(out):
    tot = sum(out)
    names = ["LEFT op + loop (everything outside RIGHT)", "poll predecessor", "barrier after poll", "issue N fetch", "reflector scalars (thread 0)",
             "barrier + build H + store N + barrier", "window product", "barrier after product"]
    for i, nme in enumerate(names):
        print(f"  phase {i} {nme:44s} {out[i]:12d} cycles {100.0*out[i]/tot:5.1f}%")

out = (ctypes.c_longlong * 24)()
capi.lib().svdb200_debug_stage2_fast_timing(out)
if any(out):
    cnt = max(out[7], 1)
    names = {0: "thread 0: poll predecessor", 9: "barrier after poll", 1: "F warps: product of the forwarded block",
             10: "F warps: wait for the N fetch at bar 2", 11: "release thread: op start .. release issued",
             2: "thread 0: wait at the closing barrier", 8: "whole op (thread 0)", 3: "N warps: fetch new block (issue .. stored)",
             12: "N warps: wait for helper at bar 1", 4: "N warps: product of the new block", 6: "helper: op start .. bar 1",
             13: "helper: 32 dot products (next Householder vector)", 5: "helper: sum of squares + scalars + H"}
    print(f"  fast kernel, interior RIGHT ops (p > 0) of CTA 1: {cnt} ops")
    for k, nme in names.items():
        print(f"    {nme:52s} {out[k] / cnt:9.0f} cycles per op")
    sw, heads = max(out[14], 1), max(out[22], 1)
    print(f"  fast kernel, sweep heads of CTA 1: {out[14]} sweeps ({out[22]} with the head reflector prepared early)")
    print(f"    {'thread 0: op-0 wait (predecessor >= 4 ops)':52s} {out[15] / sw:9.0f} cycles per sweep")
    for q in range(4):
        print(f"    {f'op {q} (after its wait .. closing barrier)':52s} {out[16 + q] / sw:9.0f} cycles per sweep")
    print(f"    {'helper: head wait (predecessor >= 3 ops)':52s} {out[20] / heads:9.0f} cycles per prepared head")
    print(f"    {'helper: head row load + scalars + H':52s} {out[21] / heads:9.0f} cycles per prepared head")
