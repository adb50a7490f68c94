"""Rectangular m x n matrices (svdb200_*_mn_dev_*): stage 1 against square stage 1 at n = min(m, n), stage 2, singular
values and the transposes of wide matrices.   python tools/rect_only.py [--out profiles/r05_rect.md] [--quick]

For every shape (16384 x 4096, 4096 x 16384, 65536 x 2048, 2048 x 65536, 32768 x 8192), f32 and f64, band 32 and 64, on
device pointers with CUDA events around each call (a fresh copy of the seeded U[0,5) input before each call, not timed):
  * stage 1 of the m x n matrix (dense_to_band_mn_dev; for m < n including both transposes) and square stage 1 of a
    k x k matrix, k = min(m, n) (dense_to_band_dev, panel order), alternated, 3 of each after one warm-up pair; GFLOP/s by
    LAPACK gebrd's count 4 m n^2 - 4 n^3 / 3 (m >= n; m, n swapped otherwise) and 8 k^3 / 3 for the square;
  * for m < n also the tall call on A^T (n x m): the wide time minus it is the cost of the two transposes, reported in ms
    and in GB/s for the 4 m n elements they read and write, against the B200 data sheet's 7.7 TB/s HBM bandwidth;
  * stage 2 (band_to_bidiag_dev on the k x k band block, complete schedule) and the singular values (bidiag_qr_dev) once.
The card's name and power limit are read in the same run.  --quick: the two 16384 x 4096 shapes in f32, band 32 only."""
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
SHAPES = [(16384, 4096), (4096, 16384), (65536, 2048), (2048, 65536), (32768, 8192)]
HBM_GBS = 7700.0


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


def gebrd_flops(m, n):
    if m < n:
        m, n = n, m
    return 4.0 * m * n * n - 4.0 * n ** 3 / 3.0


def run(m, n, dt, b, reps=3):
    k = min(m, n)
    esz = np.dtype(dt).itemsize
    s = torch.cuda.Stream()
    with capi.Handle(max(m, n), b, dt) as h:
        h.set_stream(s.cuda_stream)
        h.set_stage2_schedule(1)
        src = torch.empty(m, n, dtype=TDT[dt], device="cuda")
        sq = torch.empty(k, k, dtype=TDT[dt], device="cuda")
        h.fill_uniform_dev(src.data_ptr(), m * n, 586 + m + n, 0.0, 5.0)
        h.fill_uniform_dev(sq.data_ptr(), k * k, 586 + k, 0.0, 5.0)
        h.synchronize()
        srct = src.t().contiguous() if m < n else None
        w = torch.empty_like(src)
        wsq = torch.empty_like(sq)
        wt = torch.empty_like(srct) if srct is not None else None
        t_rect, t_sq, t_tall = [], [], []
        with torch.cuda.stream(s):
            for rep in range(reps + 1):
                w.copy_(src)
                t1 = timed(s, lambda: h.dense_to_band_mn_dev(w.data_ptr(), m, n, b))
                wsq.copy_(sq)
                t2 = timed(s, lambda: h.dense_to_band_dev(wsq.data_ptr(), k, b))
                if wt is not None:
                    wt.copy_(srct)
                    t3 = timed(s, lambda: h.dense_to_band_mn_dev(wt.data_ptr(), n, m, b))
                if rep > 0:
                    t_rect.append(t1); t_sq.append(t2)
                    if wt is not None:
                        t_tall.append(t3)
            band = wt if wt is not None else w               # tall orientation: the k x k band block is contiguous
            d = torch.empty(k, dtype=TDT[dt], device="cuda")
            e = torch.empty(k, dtype=TDT[dt], device="cuda")
            sig = torch.empty(k, dtype=TDT[dt], device="cuda")
            t_s2 = timed(s, lambda: h.band_to_bidiag_dev(band.data_ptr(), k, b, d.data_ptr(), e.data_ptr()))
            t_qr = timed(s, lambda: h.bidiag_qr_dev(d.data_ptr(), e.data_ptr(), k, sig.data_ptr()))
        fr, fs = gebrd_flops(m, n), 8.0 * k ** 3 / 3.0
        r, q = float(np.median(t_rect)), float(np.median(t_sq))
        line = (f"{m}x{n} {NAME[dt]} band {b}: stage 1 {r:.2f} ms ({fr / r * 1e-6:.0f} GFLOP/s) "
                f"[{', '.join(f'{x:.2f}' for x in t_rect)}]; square {k}x{k} {q:.2f} ms ({fs / q * 1e-6:.0f} GFLOP/s) "
                f"[{', '.join(f'{x:.2f}' for x in t_sq)}]; rect / square time {r / q:.2f}")
        if t_tall:
            tt = float(np.median(t_tall))
            dtr = r - tt
            gbs = 4.0 * m * n * esz / (dtr * 1e-3) * 1e-9 if dtr > 0 else float("nan")
            line += (f"; tall call on A^T {tt:.2f} ms [{', '.join(f'{x:.2f}' for x in t_tall)}], two transposes {dtr:.2f} ms "
                     f"= {gbs:.0f} GB/s ({gbs / HBM_GBS * 100:.0f} % of 7.7 TB/s)")
        line += f"; stage 2 {t_s2:.1f} ms, sigma {t_qr:.1f} ms (k = {k}, complete schedule), sigma_1 {float(sig[0]):.4g}"
        return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "r05_rect.md"))
    ap.add_argument("--quick", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures on the GPU")
    c = card()
    lines = [f"card: {c}"]
    print(lines[0], flush=True)
    shapes = SHAPES[:2] if args.quick else SHAPES
    for m, n in shapes:
        for dt in ((np.float32,) if args.quick else (np.float32, np.float64)):
            for b in ((32,) if args.quick else (32, 64)):
                try:
                    lines.append(run(m, n, dt, b))
                except capi.SvdB200Error as ex:          # e.g. a panel taller than the panel kernels hold at this band / type
                    lines.append(f"{m}x{n} {NAME[dt]} band {b}: not measured, {ex}")
                print(lines[-1], flush=True)
    with open(args.out, "w") as f:
        f.write("# r05: rectangular m x n matrices (tall and wide), panel order\n\n")
        f.write(f"GPU: {c} (`nvidia-smi --query-gpu=name,power.limit`, read in the same run as the numbers below).\n")
        f.write("Output of `python tools/rect_only.py`, unedited:\n\n```\n" + "\n".join(lines) + "\n```\n")
    print(f"wrote {args.out}")


if __name__ == "__main__":
    main()
