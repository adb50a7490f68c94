"""Stage 2 from band storage (svdb200_band_to_bidiag_packed_dev_*): packed vs dense at n = 3840, and the packed path alone at
sizes whose dense n x n array would not fit next to nothing on one GPU.   python tools/band_packed_only.py [--quick]

  1. n = 3840, band 32, f64 and f32, reference schedule: the dense call (band_to_bidiag_dev on the n x n embedding, a fresh
     copy per call) and the packed call alternated, 5 of each, CUDA events around each call; d and e compared byte for byte.
  2. packed only, complete schedule: n = 65536 and 262144 (f32), 65536 (f64).  Stage 2 (pack + chase + extract) and the
     singular values of the bidiagonal (bidiag_qr_dev: bisection at these n) timed with CUDA events, device memory the
     handle holds after the calls (cudaMemGetInfo around its creation), and ||(d, e)||_F / ||band||_F - 1 as a check.
--quick: only part 1 and n = 65536 f32 of part 2."""
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from svdsolver_b200 import capi  # noqa: E402

TDT = {np.float32: torch.float32, np.float64: torch.float64}
NAME = {np.float32: "f32", np.float64: "f64"}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=60).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown (nvidia-smi not available)"


def band_storage(h, ab, seed):
    """fills ab (n x (b+1)) with a U[0,5) upper band in band storage, zero above the matrix"""
    n, b = ab.shape[0], ab.shape[1] - 1
    h.fill_uniform_dev(ab.data_ptr(), n * (b + 1), seed, 0.0, 5.0)
    h.synchronize()
    for t in range(b):
        ab[: b - t, t] = 0
    return ab


def dense_embedding(ab, n, b):
    a = torch.zeros(n, n, dtype=ab.dtype, device="cuda")
    for t in range(b + 1):
        k = b - t
        i = torch.arange(n - k, device="cuda")
        a[i, i + k] = ab[k:, t]
    return a


def timed(s, fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s)
    fn()
    e1.record(s)
    s.synchronize()
    return e0.elapsed_time(e1)


def dense_vs_packed(dt, n=3840, b=32, reps=5):
    s = torch.cuda.Stream()
    with capi.Handle(n, b, dt) as h:
        h.set_stream(s.cuda_stream)
        with torch.cuda.stream(s):
            ab = band_storage(h, torch.empty(n, b + 1, dtype=TDT[dt], device="cuda"), 586 + n)
            a0 = dense_embedding(ab, n, b)
            a = torch.empty_like(a0)
            dd, ed, dp, ep = (torch.zeros(n, dtype=TDT[dt], device="cuda") for _ in range(4))
        s.synchronize()
        t_dense, t_packed = [], []
        for rep in range(reps + 1):                      # rep 0: warm-up of both paths
            a.copy_(a0)
            torch.cuda.synchronize()
            td = timed(s, lambda: h.band_to_bidiag_dev(a.data_ptr(), n, b, dd.data_ptr(), ed.data_ptr()))
            tp = timed(s, lambda: h.band_to_bidiag_packed_dev(ab.data_ptr(), n, b, dp.data_ptr(), ep.data_ptr()))
            if rep:
                t_dense.append(td)
                t_packed.append(tp)
        same = torch.equal(dd.view(torch.uint8), dp.view(torch.uint8)) and torch.equal(ed[: n - 1].view(torch.uint8), ep[: n - 1].view(torch.uint8))
    print(f"n={n} band={b} {NAME[dt]} schedule 0: dense {np.median(t_dense):.2f} ms (min {min(t_dense):.2f}) "
          f"{[round(x, 2) for x in t_dense]}  packed {np.median(t_packed):.2f} ms (min {min(t_packed):.2f}) "
          f"{[round(x, 2) for x in t_packed]}  d, e byte-equal: {same}", flush=True)
    return same


def packed_only(dt, n, b=32):
    s = torch.cuda.Stream()
    ab = torch.empty(n, b + 1, dtype=TDT[dt], device="cuda")
    d, e, sig = (torch.zeros(n, dtype=TDT[dt], device="cuda") for _ in range(3))
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info()
    h = capi.Handle(n, b, dt)
    try:
        h.set_stream(s.cuda_stream)
        h.set_stage2_schedule(1)
        with torch.cuda.stream(s):
            band_storage(h, ab, 9001)
        s.synchronize()
        t2 = timed(s, lambda: h.band_to_bidiag_packed_dev(ab.data_ptr(), n, b, d.data_ptr(), e.data_ptr()))
        fro = float(torch.sqrt((d.double() ** 2).sum() + (e[: n - 1].double() ** 2).sum()) / torch.linalg.norm(ab.double())) - 1
        tq = timed(s, lambda: h.bidiag_qr_dev(d.data_ptr(), e.data_ptr(), n, sig.data_ptr()))
        torch.cuda.synchronize()
        free1, _ = torch.cuda.mem_get_info()
        held = free0 - free1
        ws = n * 3 * b * ab.element_size()
        print(f"n={n} band={b} {NAME[dt]} schedule 1, packed: stage 2 {t2 / 1e3:.3f} s, sigma (bisection) {tq / 1e3:.3f} s, "
              f"||(d,e)||_F/||band||_F - 1 = {fro:.1e}, sigma_1 {float(sig[0]):.6g}; device memory held by the handle "
              f"{held / 2**20:.0f} MiB (packed working buffer {ws / 2**20:.0f} MiB, band storage input {ab.numel() * ab.element_size() / 2**20:.0f} MiB"
              f" outside the handle); a dense n x n array would take {n * n * ab.element_size() / 2**30:.1f} GiB", flush=True)
    finally:
        h.close()


def main():
    quick = "--quick" in sys.argv
    print(f"card: {card()}", flush=True)
    ok = all([dense_vs_packed(np.float64), dense_vs_packed(np.float32)])
    runs = [(np.float32, 65536)] if quick else [(np.float32, 65536), (np.float64, 65536), (np.float32, 262144)]
    for dt, n in runs:
        packed_only(dt, n)
    if not ok:
        raise SystemExit("packed and dense bidiagonals differ")


if __name__ == "__main__":
    main()
