"""Batched singular values of rectangular m x n matrices (svdb200_svdvals_batched_mn_dev_*) against one single-matrix call
per matrix and against torch.linalg.svdvals.   python tools/batched_mn_only.py [--out profiles/r06_batched_mn.md] [--quick]

For every shape (count x m x n, band, dtype) one device-filled U[0,5) batch (fill_uniform_dev) goes through three routes,
each on a fresh copy of the batch (the copy is not timed), on one stream with CUDA events around the timed part:
  (a) svdvals_batched_mn_dev on the whole batch, and on its first S = min(count, 64) matrices;
  (b) svdvals_mn_dev once per matrix on the same S matrices, the loop of S calls timed as one (a single call takes
      milliseconds, so the whole batch one call at a time would take minutes per repetition);
  (c) torch.linalg.svdvals on the same (count, m, n) tensor.
Routes (a) and (b) run under the complete stage-2 schedule (generic matrices).  (a) and (b) are warmed up once and timed
REPS times, (c) warmed up once and timed once; medians are reported with every repetition.  Errors: max over the batch of
max |sigma - sigma_ref| / sigma_1, for (a) and (b) against (c) and against torch.linalg.svdvals of the batch converted to
float64 (for f32 inputs the float32 SVD of (c) has errors of its own; its error against the float64 SVD is printed too).
Whether a shape runs the batched kernels or the single-matrix fallback follows from the range rule of svdb200.h; the last
default shape (4096 rows at band 64 in f64) is outside it.
The card's name and power limit are read in the same run.  --quick: the first shape only, 2 repetitions."""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from svdsolver_b200 import capi  # noqa: E402

TDT = {np.float32: torch.float32, np.float64: torch.float64}
NAME = {np.float32: "f32", np.float64: "f64"}
SHAPES = [(4096, 256, 64, 32, np.float32), (1024, 1024, 256, 64, np.float32), (1024, 1024, 256, 64, np.float64),
          (1024, 256, 1024, 64, np.float32), (512, 768, 512, 32, np.float64), (8, 4096, 512, 64, np.float64)]
REPS = 3


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=60).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown (nvidia-smi not available)"


def timed(s, fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s)
    fn()
    e1.record(s)
    s.synchronize()
    return e0.elapsed_time(e1)


def fmt(ts):
    return f"{float(np.median(ts)):.2f} ms [{', '.join(f'{x:.2f}' for x in ts)}]"


def run(count, m, n, b, dt, reps):
    k = min(m, n)
    sub = min(count, 64)
    s = torch.cuda.Stream()
    with capi.Handle(max(m, n), b, dt) as h:
        h.set_stream(s.cuda_stream)
        h.set_stage2_schedule(1)
        src = torch.empty(count, m, n, dtype=TDT[dt], device="cuda")
        h.fill_uniform_dev(src.data_ptr(), count * m * n, 586 + count + m + n, 0.0, 5.0)
        h.synchronize()
        w = torch.empty_like(src)
        sa = torch.empty(count, k, dtype=TDT[dt], device="cuda")
        sa_sub = torch.empty(sub, k, dtype=TDT[dt], device="cuda")
        sb = torch.empty(sub, k, dtype=TDT[dt], device="cuda")
        mat = m * n * src.element_size()

        def route_a():
            h.svdvals_batched_mn_dev(w.data_ptr(), count, m, n, b, sa.data_ptr())

        def route_a_sub():
            h.svdvals_batched_mn_dev(w.data_ptr(), sub, m, n, b, sa_sub.data_ptr())

        def route_b():
            for i in range(sub):
                h.svdvals_mn_dev(w.data_ptr() + i * mat, m, n, b, sb[i].data_ptr())

        out = {}
        with torch.cuda.stream(s):
            for name, fn in (("a", route_a), ("a_sub", route_a_sub), ("b", route_b)):
                ts = []
                for rep in range(reps + 1):
                    w.copy_(src)
                    t = timed(s, fn)
                    if rep > 0:
                        ts.append(t)
                out[name] = ts
            sc = torch.linalg.svdvals(src)
            out["c"] = [timed(s, lambda: torch.linalg.svdvals(src))]
            s64 = torch.linalg.svdvals(src.double())
            s.synchronize()

        def err(x, ref):
            ref = ref[: x.shape[0]].double()
            return float(((x.double() - ref).abs().max(dim=1).values / ref[:, 0]).max())
        ta_sub, tb = (float(np.median(out[x])) for x in ("a_sub", "b"))
        return (f"{count} x {m} x {n} {NAME[dt]} band {b}: (a) batched {fmt(out['a'])}, first {sub} matrices {fmt(out['a_sub'])}; "
                f"(b) {sub} single calls {fmt(out['b'])}, (b) / (a) on {sub} matrices {tb / ta_sub:.1f}x; "
                f"(c) torch.linalg.svdvals {fmt(out['c'])}; max |sigma - sigma_ref| / sigma_1 against (c): (a) {err(sa, sc):.2e}, "
                f"(b) {err(sb, sc):.2e}; against float64 svdvals: (a) {err(sa, s64):.2e}, (b) {err(sb, s64):.2e}, (c) {err(sc, s64):.2e}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "r06_batched_mn.md"))
    ap.add_argument("--quick", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures on the GPU")
    c = card()
    lines = [f"card: {c}"]
    print(lines[0], flush=True)
    shapes = SHAPES[:1] if args.quick else SHAPES
    for count, m, n, b, dt in shapes:
        lines.append(run(count, m, n, b, dt, 2 if args.quick else REPS))
        print(lines[-1], flush=True)
    with open(args.out, "w") as f:
        f.write("# r06: batched singular values of rectangular m x n matrices\n\n")
        f.write(f"GPU: {c} (`nvidia-smi --query-gpu=name,power.limit`, read in the same run as the numbers below).\n")
        f.write("Output of `python tools/batched_mn_only.py`, unedited:\n\n```\n" + "\n".join(lines) + "\n```\n")
    print(f"wrote {args.out}")


if __name__ == "__main__":
    main()
