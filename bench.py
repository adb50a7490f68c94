#!/usr/bin/env python
"""Benchmark of the SVDSolver hot path on B200 (BASELINE.json metric: bidiagonal-reduction GFLOP/s).

Workload (BASELINE.json configs[1], the reference's own benchmark shape `benchmark 320 12 1 32`,
svd_cuda_2.cu:1365-1371): square matrices n = 320..3840 step 320, band 32, U[0,5) synthetic inputs
(svdsolver_b200/synth.py), in double AND float.  One "step" = the full dense -> band -> bidiagonal
reduction (stage 1 panel order + stage 2) of all 24 matrices.  Algorithmic work = 8 n^3 / 3 flops
per matrix (SURVEY 8d), value = total flops / device time.

  value     inputs resident in HBM before the timed region; CUDA events on the launching stream,
            max over ranks; every step works on a fresh copy set (0.8 GB/step > 126 MB L2).
  e2e       the same reduction through the host-pointer C-ABI call svdb200_bidiagonalize_* with
            pinned HOST buffers: H2D of the matrix and D2H of matrix + d + e inside the timed region.
  roofline  the stage-1 rank-b trailing update (C += P Q, the dominant kernel), timed per launch
            with CUDA events in an extra profiled pass over the same workload, against the FP64
            DMMA (mma.sync) peak measured in the same run by a register-resident probe.
  cpu_baseline  the UNMODIFIED reference (oracle/_ref/libsvdref_fast.so = parallel::brd_p1 + brd_p2
            built from /root/reference with the README's -O3 -mavx) on the host cores, bounded sample.

`--impl reference` times the reference's CPU implementation alone (rank 0 only) on the same metric.
`--dump-outputs DIR` writes what the last timed step computed as DIR/*.npy (rank 0; see dump_outputs): the inputs are
seeded, so two builds of the project run with the same arguments can be compared output for output.
Multi-GPU (torchrun, one rank per GPU): the matrices of the sweep are independent, so each rank
reduces its own replica of the sweep (weak scaling, no data-path collective).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BAND = 32
SIZES = [320 * k for k in range(1, 13)]
DTYPES = (("f64", np.float64), ("f32", np.float32))
METRIC = "bidiag_reduction_gflops"
UNIT = "GFLOP/s"


# dram__bytes_read.sum + dram__bytes_write.sum of one stage2_chase_kernel<double> launch at n = 3840, band 32 from the
# committed ncu --set full capture (profiles/); None until measured
S2_TRAFFIC = 4869888   # 3.519 MB read + 1.351 MB written (profiles/r02_ncu_stage2_fast.csv: stage2_fast_kernel<double>, n = 3840, band 32)
S2_L2_BYTES = 14038780224   # lts__t_sectors.sum x 32 B of the same capture (algorithmic window bytes: 15.1e9)
S2_NCU_MS = 50.70


def flops(n):
    return 8.0 * n ** 3 / 3.0


def workload_config(extra=None):
    cfg = {
        "workload": "reference sweep n=320..3840 step 320, band 32, float and double, dense->band->bidiagonal "
                    "(BASELINE configs[1]); 24 matrices per step",
        "band": BAND, "sizes": SIZES, "dtypes": ["f64", "f32"], "stage1_order": "panel", "pipelining": "per dtype the 12 matrices go through svdb200_bidiagonalize_many_*: stage 2 of matrix i overlaps stage 1 of matrix i+1",
        "inputs": "U[0,5) splitmix64 stream, seed 586+n", "l2": "fresh 0.8 GB input copy set per step (> 126 MB L2)",
    }
    if extra:
        cfg.update(extra)
    return cfg


# ------------------------------------------------------------------------------ clocks sampler
class ClockSampler(threading.Thread):
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for i, nm in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]) if self.rows[0][1].replace(".", "").isdigit() else None,
                "power_w_max": max((float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()), default=None),
                "samples": len(self.rows), "reasons": reasons}


# ------------------------------------------------------------------------------ CPU reference leg
def load_reference():
    fast = os.path.join(ROOT, "oracle", "_ref", "libsvdref_fast.so")
    if os.path.exists(fast):
        return ctypes.CDLL(fast), "reference"
    # fall back to the C restatement (kind "port") -- still the checker, never the product
    port = os.path.join(ROOT, "oracle", "libsvd_oracle.so")
    if not os.path.exists(port):
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), port])
    return ctypes.CDLL(port), "port"


def cpu_reference_sample(sizes):
    """Times parallel::brd_p1 + parallel::brd_p2 (chained) on the host for the given sizes, f64+f32."""
    from svdsolver_b200.synth import uniform_matrix
    lib, kind = load_reference()
    tot_t, tot_f, detail = 0.0, 0.0, []
    for n in sizes:
        for suf, dt in DTYPES:
            a = uniform_matrix(n, n, 586 + n, 0.0, 5.0, dt)
            t1, t2 = ctypes.c_double(0), ctypes.c_double(0)
            if kind == "reference":
                getattr(lib, f"svdref_time_multicore_{suf}")(a.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(n), ctypes.c_size_t(BAND),
                                                             ctypes.c_int(1), ctypes.byref(t1), ctypes.byref(t2))
                dt_s = t1.value + t2.value
            else:
                x = a.copy()
                t0 = time.perf_counter()
                getattr(lib, f"svdo_brd_p1_{suf}")(x.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(n), ctypes.c_size_t(BAND))
                getattr(lib, f"svdo_brd_p2_{suf}")(x.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(n), ctypes.c_size_t(BAND), None, None)
                dt_s = time.perf_counter() - t0
            tot_t += dt_s
            tot_f += flops(n)
            detail.append({"n": n, "dtype": suf, "seconds": round(dt_s, 4)})
    cores = lib.svdref_omp_threads() if kind == "reference" else (os.cpu_count() or 1)
    return {"value": tot_f / tot_t * 1e-9, "unit": UNIT, "cores": int(cores), "kind": kind,
            "sample": f"n={sizes} band {BAND} f64+f32, stage1+stage2 chained, timing.h:78-83 timer convention", "seconds": round(tot_t, 3),
            "detail": detail}


def run_reference_arm(args, rank):
    if rank != 0:
        return
    per_step_sizes = [320, 640] if (args.steps + args.warmup) * 15.0 <= 160.0 else [320]
    for _ in range(args.warmup):
        cpu_reference_sample(per_step_sizes[:1])
    t0 = time.perf_counter()
    last = None
    tot_f = 0.0
    for _ in range(args.steps):
        last = cpu_reference_sample(per_step_sizes)
        tot_f += sum(flops(n) for n in per_step_sizes) * len(DTYPES)
    dt = time.perf_counter() - t0
    value = tot_f / dt * 1e-9
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / max(args.steps, 1) * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64,f32", "data": "synthetic",
        "config": workload_config({"sizes_timed": per_step_sizes,
                                   "sample": f"bounded: n={per_step_sizes} of the sweep per step (the full sweep takes ~45 min on 8 cores, BASELINE.md 2b); "
                                             "the GPU arm reports its own numbers on exactly these sizes in cpu_baseline.gpu_same_sample"}),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": last["cores"], "kind": last["kind"], "sample": last["sample"]},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------ output dump
DUMP_BYTES = 48_000_000   # array data of one dump; with the .npy headers the whole dump stays under 64 MB


def dump_share(sizes):
    """Bytes of the whole-matrix sample of each matrix; fails before any GPU work when d, e and the bands alone overflow."""
    fixed = sum((2 * n - 1 + (BAND + 1) * n) * sum(np.dtype(dt).itemsize for _, dt in DTYPES) for n in sizes)
    if fixed > DUMP_BYTES:
        raise SystemExit(f"--dump-outputs: d, e and the band of {len(sizes) * len(DTYPES)} matrices take {fixed} bytes, "
                         f"over the {DUMP_BYTES}-byte budget")
    return (DUMP_BYTES - fixed) // (len(sizes) * len(DTYPES))


def dump_outputs(out_dir, torch, cur, dmany, emany, share):
    """What svdb200_bidiagonalize_many_dev_* handed back in one step, for every matrix of the sweep: d (n), e (n - 1), the
    diagonals 0..BAND of the overwritten matrix in full (row k = diagonal k, zero-padded to n: the band stage 1 leaves and
    stage 2 reduces, where builds can differ) and a sample of the whole overwritten matrix, the entries at flat indices drawn
    without replacement from a generator seeded with n and sorted, as many as DUMP_BYTES leaves after the rest, shared
    equally over the matrices (dump_share).  Files: DIR/<f64|f32>_n<n>_<d|e|band|a>.npy."""
    os.makedirs(out_dir, exist_ok=True)
    torch.cuda.synchronize()
    pos = {}
    for n, suf, a in cur:
        i = pos[suf] = pos.get(suf, -1) + 1
        band = torch.zeros(BAND + 1, n, dtype=a.dtype, device=a.device)
        for k in range(min(BAND, n - 1) + 1):
            band[k, : n - k] = torch.diagonal(a, k)
        idx = np.sort(np.random.default_rng(n).choice(n * n, min(n * n, share // a.element_size()), replace=False))
        sample = a.reshape(-1)[torch.from_numpy(idx).to(a.device)]
        for name, x in (("d", dmany[suf][i]), ("e", emany[suf][i][: n - 1]), ("band", band), ("a", sample)):
            np.save(os.path.join(out_dir, f"{suf}_n{n}_{name}.npy"), x.cpu().numpy())


# ------------------------------------------------------------------------------ GPU arm
def north_star_shape(capi, torch, stream, dev, local_rank, dt, peaks, hbm_peak, nb=16384, bb=64):
    """Stage 1 at BASELINE configs[2]'s shape: whole-stage device time, then a profiled pass (per-launch CUDA events)."""
    try:
        tdt = torch.float64 if dt == np.float64 else torch.float32
        esz = 8 if dt == np.float64 else 4
        hb = capi.Handle(nb, bb, dt, device=local_rank)
        hb.set_stream(stream.cuda_stream)
        ab = torch.empty(nb, nb, device=dev, dtype=tdt)
        best = None
        for rep in range(2):
            hb.fill_uniform_dev(ab.data_ptr(), nb * nb, 586 + nb, 0.0, 5.0)
            torch.cuda.synchronize()
            b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            b0.record(stream)
            hb.dense_to_band_dev(ab.data_ptr(), nb, bb)
            b1.record(stream)
            torch.cuda.synchronize()
            t = b0.elapsed_time(b1)
            best = t if best is None else min(best, t)
        t_s1 = best
        hb.fill_uniform_dev(ab.data_ptr(), nb * nb, 586 + nb, 0.0, 5.0)
        torch.cuda.synchronize()
        hb.reset_profile(); hb.set_profile(True)
        hb.dense_to_band_dev(ab.data_ptr(), nb, bb)
        torch.cuda.synchronize()
        hb.set_profile(False)
        pb = hb.get_profile()
        gms = sum(pb[k]["ms"] for k in ("gemm_tn", "gemm_nn", "rank_update"))
        gwork = sum(pb[k]["work"] for k in ("gemm_tn", "gemm_nn", "rank_update"))
        tf = gwork / (gms * 1e-3) * 1e-12
        # algorithmic HBM bytes of the update: C read once per GEMM, read + written once per rank-b update
        gbytes = (pb["gemm_tn"]["work"] + pb["gemm_nn"]["work"] + 2 * pb["rank_update"]["work"]) / (2.0 * bb) * esz
        out = {"n": nb, "band": bb, "dtype": "f64" if dt == np.float64 else "f32", "stage1_ms": round(t_s1, 2),
               "stage1_tflops": round(flops(nb) / (t_s1 * 1e-3) * 1e-12, 2), "trailing_update_tflops": round(tf, 2),
               "trailing_update_hbm_gbs": round(gbytes / (gms * 1e-3) * 1e-9, 1),
               "trailing_update_frac_of_hbm_peak": round(gbytes / (gms * 1e-3) * 1e-9 / hbm_peak, 4)}
        if dt == np.float64:
            out["trailing_update_frac_of_fp64_dmma_peak"] = round(tf / peaks["dmma_f64_tflops"], 4)
            out["tensor_path"] = "mma.sync.m8n8k4.f64 (DMMA); tcgen05.mma has no f64 kind"
        else:
            pk = peaks.get("tf32_tcgen05_tflops")
            if pk:
                out["trailing_update_frac_of_3xtf32_tcgen05_peak"] = round(tf / (pk / 3.0), 4)
            out["tensor_path"] = "tcgen05.mma kind::tf32 x3 (hi/lo split), accumulator in TMEM, operands by TMA"
        def _cls(k, x):
            o = {"ms": round(x["ms"], 2), "launches": x["launches"],
                 "tflops": round(x["work"] / (x["ms"] * 1e-3) * 1e-12, 2) if x["ms"] > 0 else None}
            if k in ("gemm_tn", "gemm_nn", "rank_update") and x["ms"] > 0:
                # algorithmic HBM bytes: C read once (GEMMs) / read + written once (rank-b update)
                byts = x["work"] / (2.0 * bb) * esz * (2 if k == "rank_update" else 1)
                o["hbm_gbs"] = round(byts / (x["ms"] * 1e-3) * 1e-9, 1)
                o["frac_of_hbm_peak"] = round(o["hbm_gbs"] / hbm_peak, 4)
            return o
        out["classes"] = {k: _cls(k, x) for k, x in pb.items() if x["launches"]}
        hb.close()
        del ab
        torch.cuda.empty_cache()
        return out
    except Exception as ex:   # a capacity problem must not take the bench line down
        return {"error": str(ex)}


def gpu_same_sample(capi, torch, stream, dev, handles, sample_sizes, tdt, reps=5):
    """The GPU arm on exactly the sizes the CPU reference leg is timed on (like for like): device-resident and end to end
    (pinned host buffers, copies inside the timed region), f64 + f32, through the same svdb200_bidiagonalize_many_* calls."""
    from svdsolver_b200.synth import uniform_matrix
    out = {"sizes": list(sample_sizes)}
    fl = sum(flops(n) for n in sample_sizes) * len(DTYPES)
    mats = {suf: [torch.empty(n, n, device=dev, dtype=tdt[suf]) for n in sample_sizes] for suf, _ in DTYPES}
    dd = {suf: [torch.empty(n, device=dev, dtype=tdt[suf]) for n in sample_sizes] for suf, _ in DTYPES}
    ee = {suf: [torch.empty(n, device=dev, dtype=tdt[suf]) for n in sample_sizes] for suf, _ in DTYPES}
    best = None
    for rep in range(reps + 1):
        for suf, _ in DTYPES:
            for n, a in zip(sample_sizes, mats[suf]):
                handles[suf].fill_uniform_dev(a.data_ptr(), n * n, 586 + n, 0.0, 5.0)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for suf, _ in DTYPES:
            handles[suf].bidiagonalize_many_dev([a.data_ptr() for a in mats[suf]], list(sample_sizes), BAND,
                                                [x.data_ptr() for x in dd[suf]], [x.data_ptr() for x in ee[suf]])
        e1.record(stream)
        torch.cuda.synchronize()
        if rep:
            t = e0.elapsed_time(e1)
            best = t if best is None else min(best, t)
    out["device_gflops"] = round(fl / (best * 1e-3) * 1e-9, 2)
    host = []
    for n in sample_sizes:
        for suf, dt in DTYPES:
            src = torch.from_numpy(uniform_matrix(n, n, 586 + n, 0.0, 5.0, dt))
            host.append((n, suf, src, torch.empty(n, n, dtype=tdt[suf]).pin_memory(), torch.empty(n, dtype=tdt[suf]).pin_memory(),
                         torch.empty(n, dtype=tdt[suf]).pin_memory()))
    best = None
    for rep in range(reps + 1):
        for _, _, src, buf, _, _ in host:
            buf.copy_(src)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for suf, _ in DTYPES:
            hs = [x for x in host if x[1] == suf]
            handles[suf].bidiagonalize_many_inplace([x[3].data_ptr() for x in hs], [x[0] for x in hs], BAND,
                                                    [x[4].data_ptr() for x in hs], [x[5].data_ptr() for x in hs])
        torch.cuda.synchronize()
        t = (time.perf_counter() - t0) * 1e3
        if rep:
            best = t if best is None else min(best, t)
    out["e2e_gflops"] = round(fl / (best * 1e-3) * 1e-9, 2)
    out["timer"] = "device: CUDA events; e2e: host wall clock around the blocking C-ABI calls (timing.h:78-83 convention), best of %d" % reps
    return out


def full_configs(capi, torch, stream, dev, local_rank):
    """BASELINE configs[2] (n=16384 double full SVD, band 64) and one GPU's share of configs[4] (1024 of the 8192 batched
    256x256 double SVDs, band 32): device time per stage, CUDA events on the launching stream."""
    out = {}
    try:
        n, b = 16384, 64
        h = capi.Handle(n, b, np.float64, device=local_rank)
        h.set_stream(stream.cuda_stream)
        a = torch.empty(n, n, device=dev, dtype=torch.float64)
        d = torch.empty(n, device=dev, dtype=torch.float64)
        e = torch.empty(n, device=dev, dtype=torch.float64)
        sg = torch.empty(n, device=dev, dtype=torch.float64)
        h.fill_uniform_dev(a.data_ptr(), n * n, 586 + n, 0.0, 5.0)
        fro = float(torch.linalg.norm(a))
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record(stream)
        h.dense_to_band_dev(a.data_ptr(), n, b)
        ev[1].record(stream)
        h.band_to_bidiag_dev(a.data_ptr(), n, b, d.data_ptr(), e.data_ptr())
        ev[2].record(stream)
        h.bidiag_qr_dev(d.data_ptr(), e.data_ptr(), n, sg.data_ptr())
        ev[3].record(stream)
        torch.cuda.synchronize()
        t1, t2, t3 = ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[2].elapsed_time(ev[3])
        out["config3_full_svd"] = {"workload": "16384x16384 double full SVD (dense->band->bidiagonal->singular values), band 64, one B200",
                                   "stage1_ms": round(t1, 1), "stage2_ms": round(t2, 1), "sigma_ms": round(t3, 1), "total_ms": round(t1 + t2 + t3, 1),
                                   "reduction_gflops": round(flops(n) / ((t1 + t2) * 1e-3) * 1e-9, 1),
                                   "sigma_solver": "bisection on the Golub-Kahan form (n > 1024); zero-shift QR sweeps below",
                                   "frobenius_rel_err": abs(float(torch.sqrt((sg * sg).sum())) - fro) / fro}
        h.close()
        del a, d, e, sg
        torch.cuda.empty_cache()
    except Exception as ex:
        out["config3_full_svd"] = {"error": str(ex)}
    return out


def batched_config(capi, torch, dist, stream, dev, local_rank, rank, world, barrier):
    """BASELINE configs[4]: 8192 x (256x256 double SVD, band 32) sharded by matrix over the ranks (no collective on the data
    path; the max over ranks is taken for the time)."""
    try:
        total, n, b = 8192, 256, 32
        cnt = total // world + (1 if rank < total % world else 0)
        h = capi.Handle(n, b, np.float64, device=local_rank)
        h.set_stream(stream.cuda_stream)
        a = torch.empty(cnt, n, n, device=dev, dtype=torch.float64)
        sg = torch.empty(cnt, n, device=dev, dtype=torch.float64)
        best = None
        for rep in range(3):
            h.fill_uniform_dev(a.data_ptr(), cnt * n * n, 586 + 1000003 * rank, 0.0, 5.0)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            h.svdvals_batched_dev(a.data_ptr(), cnt, n, b, sg.data_ptr())
            e1.record(stream)
            barrier()
            t = e0.elapsed_time(e1)
            if world > 1:
                tt = torch.tensor([t], device=dev, dtype=torch.float64)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                t = float(tt.item())
            best = t if best is None else min(best, t)
        ok = bool(torch.isfinite(sg).all().item()) and bool((sg[:, :-1] >= sg[:, 1:]).all().item())
        h.close()
        del a, sg
        torch.cuda.empty_cache()
        return {"workload": f"8192 x (256x256 double SVD, band 32) sharded by matrix over {world} GPU(s) (BASELINE configs[4])",
                "matrices_per_rank": total // world, "ms": round(best, 1), "matrices_per_s": round(total / best * 1e3, 1),
                "sigma_sorted_finite_rank0": ok}
    except Exception as ex:
        return {"error": str(ex)}


def dist_stage1_config(args, capi, torch, dist, stream, dev, local_rank, rank, world, barrier):
    """BASELINE configs[3] shape: n x n float dense -> band, band 64, 1-D block-cyclic over the columns of `world` GPUs (NCCL
    panel broadcast).  Runs for every N including 1; with N > 1 rank 0 afterwards times the same driver on one GPU so that
    the strong-scaling efficiency is measured inside one run.  In-run invariants: Frobenius norm, zeros below the diagonal,
    round-off above the band."""
    from svdsolver_b200 import distributed as D
    nd, bd = args.dist_n, 64
    out = {"workload": f"{nd}x{nd} float dense->band, band {bd}, block-cyclic columns over {world} GPU(s) (BASELINE configs[3] shape)",
           "n": nd, "ranks": world}

    def one(nranks, rk, uid, reps):
        ncl = D.local_cols(nd, bd, rk, nranks)
        loc = torch.empty(nd, ncl, device=dev, dtype=torch.float32)
        hfill = capi.Handle(64, 32, np.float32, device=local_rank)
        hfill.set_stream(stream.cuda_stream)
        res = {}
        with D.DistHandle(nd, bd, np.float32, rk, nranks, uid, device=local_rank) as dh:
            dh.set_stream(stream.cuda_stream)
            times = []
            for rep in range(reps):
                hfill.fill_uniform_dev(loc.data_ptr(), nd * ncl, 586 + nd + 7919 * rk, 0.0, 5.0)
                torch.cuda.synchronize()
                if rep == 0:
                    fro2 = sum(float((loc[:, c0:c0 + 2048].double() ** 2).sum()) for c0 in range(0, ncl, 2048))
                if nranks > 1:
                    barrier()
                d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                d0.record(stream)
                dh.dense_to_band_dev(loc.data_ptr())
                d1.record(stream)
                if nranks > 1:
                    barrier()
                else:
                    torch.cuda.synchronize()
                t = d0.elapsed_time(d1)
                if nranks > 1:
                    tt = torch.tensor([t], device=dev, dtype=torch.float64)
                    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                    t = float(tt.item())
                times.append(t)
            res["launches_rank0"] = dh.launch_count()
        hfill.close()
        # invariants on the result of the last repetition
        gcol = (torch.arange(ncl, device=dev) // bd * nranks + rk) * bd + torch.arange(ncl, device=dev) % bd
        rows = torch.arange(nd, device=dev)
        fro2b, below, above, amax = 0.0, 0.0, 0.0, 0.0
        for c0 in range(0, ncl, 1024):
            blk = loc[:, c0:c0 + 1024]
            gc = gcol[c0:c0 + 1024]
            fro2b += float((blk.double() ** 2).sum())
            amax = max(amax, float(blk.abs().max()))
            below = max(below, float((blk.abs() * (rows[:, None] > gc[None, :])).max()))
            above = max(above, float((blk.abs() * (rows[:, None] < gc[None, :] - bd)).max()))
        vals = torch.tensor([fro2, fro2b], device=dev, dtype=torch.float64)
        mx = torch.tensor([below, above, amax], device=dev, dtype=torch.float64)
        if nranks > 1:
            dist.all_reduce(vals)
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        res["ms"] = round(min(times), 1)
        res["tflops"] = round(flops(nd) / (min(times) * 1e-3) * 1e-12, 2)
        res["frob_rel_err"] = abs(float(vals[1]) ** 0.5 - float(vals[0]) ** 0.5) / float(vals[0]) ** 0.5
        res["max_below_diag"] = float(mx[0])
        res["max_above_band_rel"] = float(mx[1]) / float(mx[2])
        del loc
        torch.cuda.empty_cache()
        return res

    try:
        uid = D.exchange_unique_id(rank, world)
        out.update(one(world, rank, uid, 2))
        out["collectives"] = ("per block step: ncclBroadcast(raw QR panel rows, (m-b) b elements, third stream, beside the owner's factorisation) + "
                              "ncclBroadcast([M1 | M2], top blocks, status: 4 b^2 + 4 elements), ncclAllReduce([Gram | top block], 50 KB, double) of the "
                              "distributed LQ panel, ncclAllReduce(W)") if world > 1 else "none (one rank)"
        if world > 1 and not os.environ.get("SKIP_N1"):
            t1 = torch.zeros(1, device=dev, dtype=torch.float64)
            if rank == 0:
                import ctypes
                r1 = one(1, 0, (ctypes.c_ubyte * 128)(), 1)
                t1[0] = r1["ms"]
                out["one_gpu_ms_same_run"] = r1["ms"]
            barrier()
            dist.broadcast(t1, src=0)
            out["strong_eff_vs_N1"] = round(float(t1.item()) / (world * out["ms"]), 3)
    except Exception as ex:
        out["error"] = str(ex)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="svdb200")
    ap.add_argument("--sizes", default="")           # debugging: comma-separated subset of the sweep
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dist-n", type=int, default=65536)  # size of the block-cyclic stage-1 measurement (BASELINE configs[3])
    ap.add_argument("--no-big", action="store_true")      # skip the n=16384 trailing-update measurement
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step computed (d, e, the band and a seeded sample of each bidiagonalised matrix) as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return
    if args.warmup < 3:
        args.warmup = 3
    sizes = [int(s) for s in args.sizes.split(",")] if args.sizes else SIZES
    dump_sample_bytes = dump_share(sizes) if args.dump_outputs else 0

    import torch
    import torch.distributed as dist
    from svdsolver_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    # A dedicated non-default stream: svdb200_set_stream(NULL) means "the handle's own stream", so
    # the legacy default stream (handle 0) cannot carry the work; events must be recorded on the
    # stream the kernels are launched on.
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    nmax = max(sizes)
    handles = {suf: capi.Handle(nmax, BAND, dt, device=local_rank) for suf, dt in DTYPES}
    for h in handles.values():
        h.set_stream(stream.cuda_stream)
    tdt = {"f64": torch.float64, "f32": torch.float32}

    nsets = args.steps + args.warmup
    free_b, _ = torch.cuda.mem_get_info()
    set_bytes = sum(n * n for n in sizes) * 12
    nsets = max(1, min(nsets, int(free_b * 0.7 // set_bytes)))
    sets = []
    for s in range(nsets):
        cur = []
        for n in sizes:
            for suf, _ in DTYPES:
                a = torch.empty(n, n, device=dev, dtype=tdt[suf])
                handles[suf].fill_uniform_dev(a.data_ptr(), n * n, 586 + n, 0.0, 5.0)
                cur.append((n, suf, a))
        sets.append(cur)
    dbuf = {suf: torch.empty(nmax, device=dev, dtype=tdt[suf]) for suf, _ in DTYPES}
    ebuf = {suf: torch.empty(nmax, device=dev, dtype=tdt[suf]) for suf, _ in DTYPES}

    def refill(cur):
        for n, suf, a in cur:
            handles[suf].fill_uniform_dev(a.data_ptr(), n * n, 586 + n, 0.0, 5.0)

    # one call per dtype hands the 12 matrices of the sweep to svdb200_bidiagonalize_many_dev_*: stage 2 of matrix i runs
    # beside stage 1 of matrix i+1 (results identical to one call per matrix; tests/test_gpu_parity.py)
    dmany = {suf: [torch.empty(n, device=dev, dtype=tdt[suf]) for n in sizes] for suf, _ in DTYPES}
    emany = {suf: [torch.empty(n, device=dev, dtype=tdt[suf]) for n in sizes] for suf, _ in DTYPES}

    def step(cur):
        for suf, _ in DTYPES:
            mats = [(n, a) for n, s_, a in cur if s_ == suf]
            handles[suf].bidiagonalize_many_dev([a.data_ptr() for _, a in mats], [n for n, _ in mats], BAND,
                                                [x.data_ptr() for x in dmany[suf]], [x.data_ptr() for x in emany[suf]])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up -------------------------------------------------------------------------------
    for w in range(args.warmup):
        step(sets[w % nsets])
    torch.cuda.synchronize()
    reused = nsets < args.steps + args.warmup
    if reused:
        for cur in sets:
            refill(cur)
    # ---- timed region: EXACTLY `steps` steps ----------------------------------------------------
    launches0 = sum(h.launch_count() for h in handles.values())
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for s in range(args.steps):
        idx = (args.warmup + s) % nsets
        if reused and s >= nsets:
            refill(sets[idx])
        step(sets[idx])
    ev1.record(stream)
    barrier()
    sampler.stop_flag = True
    ms = ev0.elapsed_time(ev1)
    launches = sum(h.launch_count() for h in handles.values()) - launches0
    if args.dump_outputs and rank == 0:
        # before the breakdown pass below refills sets[0], which may be the set of the last step
        dump_outputs(args.dump_outputs, torch, sets[idx], dmany, emany, dump_sample_bytes)
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        lt = torch.tensor([launches], device=dev, dtype=torch.int64)
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
        launches = int(lt.item())
    step_flops = sum(flops(n) for n in sizes) * len(DTYPES)
    value = world * step_flops * args.steps / (ms * 1e-3) * 1e-9

    # ---- per-size / per-dtype breakdown (device time, one extra untimed-for-`value` pass) --------
    detail = []
    if rank == 0:
        cur = sets[0]
        refill(cur)
        torch.cuda.synchronize()
        first = {}
        for rep in range(2):                   # pass 0 also absorbs one-time set-up of the handle's own (non-pipelined) path
            if rep == 1:
                refill(cur)
                torch.cuda.synchronize()
            for n, suf, a in cur:
                h = handles[suf]
                e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                e0.record(stream)
                h.dense_to_band_dev(a.data_ptr(), n, BAND)
                e1.record(stream)
                h.band_to_bidiag_dev(a.data_ptr(), n, BAND, dbuf[suf].data_ptr(), ebuf[suf].data_ptr())
                e2.record(stream)
                torch.cuda.synchronize()
                if rep == 0:
                    first[(n, suf)] = (e0.elapsed_time(e1), e1.elapsed_time(e2))
                    continue
                t1, t2 = min(first[(n, suf)][0], e0.elapsed_time(e1)), min(first[(n, suf)][1], e1.elapsed_time(e2))
                detail.append({"n": n, "dtype": suf, "stage1_ms": round(t1, 3), "stage2_ms": round(t2, 3),
                               "gflops": round(flops(n) / ((t1 + t2) * 1e-3) * 1e-9, 1),
                               "stage1_gflops": round(flops(n) / (t1 * 1e-3) * 1e-9, 1)})

    # ---- roofline of the dominant kernel: profiled pass, CUDA events per launch ------------------
    roofline, prof_out, peaks, big, big32, other, roofline_ns = None, None, {}, None, None, None, None
    if rank == 0:
        h = handles["f64"]
        peaks = {"dfma_tflops": h.probe_peak(0), "dmma_f64_tflops": h.probe_peak(1), "ffma_tflops": h.probe_peak(2),
                 "tf32_mma_sync_tflops": h.probe_peak(3)}
        cur = sets[0]
        refill(cur)
        torch.cuda.synchronize()
        h.reset_profile()
        h.set_profile(True)
        for n, suf, a in cur:
            if suf == "f64":
                h.bidiagonalize_dev(a.data_ptr(), n, BAND, dbuf[suf].data_ptr(), ebuf[suf].data_ptr())
        torch.cuda.synchronize()
        h.set_profile(False)
        prof = h.get_profile()
        tot_ms = sum(v["ms"] for v in prof.values()) or 1.0
        prof_out = {k: {"ms": round(v["ms"], 3), "launches": v["launches"], "share": round(v["ms"] / tot_ms, 3),
                        "achieved": (round(v["work"] / (v["ms"] * 1e-3) * 1e-12, 3) if v["ms"] > 0 and k not in ("stage2", "qr") else
                                     (round(v["work"] / (v["ms"] * 1e-3) * 1e-9, 2) if v["ms"] > 0 and k == "stage2" else None)),
                        "unit": "TFLOP/s" if k not in ("stage2", "qr") else ("GB/s window traffic" if k == "stage2" else None)}
                    for k, v in prof.items()}
        # dominant kernel of the step by device-time share
        dom = max(prof.items(), key=lambda kv: kv[1]["ms"])[0]
        hbm_peak = None
        try:
            hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
        except Exception:
            pass
        if dom == "stage2":
            v = prof["stage2"]
            ach = v["work"] / (v["ms"] * 1e-3) * 1e-9
            peak = hbm_peak or 6650.0
            roofline = {"bound": "hbm", "kernel": "stage2_fast_kernel<double> / stage2_chase_kernel<double> (band -> bidiagonal bulge chasing)",
                        "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4), "traffic": S2_TRAFFIC,
                        "l2": {"achieved_gbs": round(S2_L2_BYTES / (S2_NCU_MS * 1e-3) * 1e-9, 1), "traffic": S2_L2_BYTES,
                               "note": "L2 <-> SM bytes of the n = 3840 launch under ncu (lts__t_sectors.sum x 32 B) over its duration: every "
                                       "window element goes through L2 once per op (the algorithmic figure), HBM sees only the compulsory band"},
                        "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if hbm_peak else "fallback 6.65 TB/s",
                        "algorithmic_bytes": "4*b*n^2*sizeof(T) window bytes per launch (SURVEY 8d)",
                        "note": "dependency-latency bound by construction (4 window ops x n sweeps on the critical path, "
                                "band region L2-resident): HBM fraction is expected to be small",
                        "launches_timed": v["launches"], "avg_launch_us": round(v["ms"] / max(v["launches"], 1) * 1e3, 1)}
        else:
            v = prof[dom]
            ach = v["work"] / (v["ms"] * 1e-3) * 1e-12 if v["ms"] > 0 else 0.0
            roofline = {"bound": "tensor", "kernel": dom, "achieved": round(ach, 3), "peak": round(peaks["dmma_f64_tflops"], 2),
                        "unit": "TFLOP/s", "frac": round(ach / peaks["dmma_f64_tflops"], 4), "traffic": None,
                        "peak_source": "FP64 DMMA mma.sync.m8n8k4 register-resident probe measured in this run",
                        "launches_timed": v["launches"], "avg_launch_us": round(v["ms"] / max(v["launches"], 1) * 1e3, 2)}
        # stage-1 trailing update at the north-star shape (n = 16384, band 64), per-launch CUDA events:
        # double on DMMA mma.sync (tcgen05 has no f64 kind), float on tcgen05/TMEM/TMA (3xTF32)
        if not args.sizes and not args.no_big:
            try:
                peaks["tf32_tcgen05_tflops"] = handles["f32"].probe_peak(4)
            except Exception:
                pass
            big = north_star_shape(capi, torch, stream, dev, local_rank, np.float64, peaks, hbm_peak or 6650.0)
            big32 = north_star_shape(capi, torch, stream, dev, local_rank, np.float32, peaks, hbm_peak or 6650.0)
            other = full_configs(capi, torch, stream, dev, local_rank) if world == 1 else None
            # second roofline object: the dominant kernel of stage 1 at the north-star shape in float, the tcgen05 rank-b update
            try:
                ru = big32["classes"]["rank_update"]
                roofline_ns = {"bound": "hbm", "kernel": "rank_update_tc05_kernel<64> (C += V2*W on tcgen05/TMEM, C through TMA; n=16384, band 64, float)",
                               "achieved": ru["hbm_gbs"], "peak": hbm_peak or 6650.0, "unit": "GB/s", "frac": ru["frac_of_hbm_peak"],
                               "traffic": 2194703000, "traffic_note": "dram read+write of the first (full-size) launch, ncu --set full (profiles/r01_ncu_metrics.csv); algorithmic 2.147e9",
                               "algorithmic_bytes": "8 bytes per element of the updated block per launch (read once + written once)",
                               "launches_timed": ru["launches"], "avg_launch_us": round(ru["ms"] / max(ru["launches"], 1) * 1e3, 1)}
            except Exception:
                roofline_ns = None
    # ---- e2e: host-pointer C-ABI call with pinned host buffers --------------------------------------
    from svdsolver_b200.synth import uniform_matrix
    e2e = None
    e2e_steps = max(1, min(args.steps, 3))
    host = []
    h2d = d2h = 0
    for n in sizes:
        for suf, dt in DTYPES:
            src = torch.from_numpy(uniform_matrix(n, n, 586 + n, 0.0, 5.0, dt))
            buf = torch.empty(n, n, dtype=tdt[suf]).pin_memory()
            dh = torch.empty(n, dtype=tdt[suf]).pin_memory()
            eh = torch.empty(n, dtype=tdt[suf]).pin_memory()
            host.append((n, suf, src, buf, dh, eh))
            h2d += n * n * src.element_size()
            d2h += (n * n + 2 * n - 1) * src.element_size()
    tot_ms = 0.0
    for s in range(1 + e2e_steps):
        for _, _, src, buf, _, _ in host:
            buf.copy_(src)
        barrier()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record(stream)
        for suf, _ in DTYPES:
            hs = [x for x in host if x[1] == suf]
            handles[suf].bidiagonalize_many_inplace([x[3].data_ptr() for x in hs], [x[0] for x in hs], BAND,
                                                    [x[4].data_ptr() for x in hs], [x[5].data_ptr() for x in hs])
        a1.record(stream)
        torch.cuda.synchronize()
        if s > 0:
            tot_ms += a0.elapsed_time(a1)
    if world > 1:
        t = torch.tensor([tot_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        tot_ms = float(t.item())
    e2e = {"value": world * step_flops * e2e_steps / (tot_ms * 1e-3) * 1e-9, "unit": UNIT, "h2d_bytes_per_step": h2d * world,
           "d2h_bytes_per_step": d2h * world, "steps": e2e_steps, "api": "svdb200_bidiagonalize_many_{f64,f32} (host pointers, pinned; double-buffered copies)"}

    # ---- like-for-like with the CPU reference leg: the GPU on exactly the sizes the CPU sample uses --------------------
    cpu_sizes = [320, 640]
    same = None
    if rank == 0 and not args.sizes:
        try:
            same = gpu_same_sample(capi, torch, stream, dev, handles, cpu_sizes, tdt)
        except Exception as ex:
            same = {"error": str(ex)}
    for h in handles.values():
        h.close()
    handles = {}
    del sets, dbuf, ebuf, dmany, emany, host
    torch.cuda.empty_cache()

    # ---- BASELINE configs[4] (batched, sharded by matrix) and configs[3] (block-cyclic stage 1), every N -----------------
    batched_out = dist_out = None
    if not args.no_big and not args.sizes:
        batched_out = batched_config(capi, torch, dist, stream, dev, local_rank, rank, world, barrier)
        dist_out = dist_stage1_config(args, capi, torch, dist, stream, dev, local_rank, rank, world, barrier)

    # ---- CPU baseline (rank 0, N=1 only) ---------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_reference_sample(cpu_sizes)
        cpu.pop("detail", None)
        if same and "device_gflops" in same:
            same["vs_cpu_device"] = round(same["device_gflops"] / cpu["value"], 1)
            same["vs_cpu_e2e"] = round(same["e2e_gflops"] / cpu["value"], 1)
        cpu["gpu_same_sample"] = same
        cpu["note"] = "like for like = gpu_same_sample vs value (same sizes, same dtypes); the headline `value` is the full sweep, which the CPU cannot finish in minutes"

    if rank == 0:
        peak64, peak32 = peaks.get("dfma_tflops"), peaks.get("ffma_tflops")
        for dsc in detail:
            pk = peak64 if dsc["dtype"] == "f64" else peak32
            if pk:
                dsc["pct_of_fma_peak"] = round(dsc["gflops"] / (pk * 1e3) * 100.0, 2)
                dsc["stage1_pct_of_fma_peak"] = round(dsc["stage1_gflops"] / (pk * 1e3) * 100.0, 2)
        cfg = workload_config({"sizes": sizes, "parallelism": f"replicas x{world}", "reference_arm_sizes": cpu_sizes,
                               "gpu_on_reference_arm_sizes": same})
        # numbers of the other BASELINE configs live under `config` (a key the driver's record keeps)
        ns = {}
        if big and "error" not in big:
            ns["stage1_n16384_band64_f64"] = {k: big[k] for k in ("stage1_ms", "stage1_tflops", "trailing_update_tflops",
                                                                  "trailing_update_frac_of_fp64_dmma_peak", "trailing_update_frac_of_hbm_peak") if k in big}
            ns["stage1_n16384_band64_f64"]["panel_ms"] = big["classes"]["panel"]["ms"]
        if big32 and "error" not in big32:
            ns["stage1_n16384_band64_f32"] = {k: big32[k] for k in ("stage1_ms", "stage1_tflops", "trailing_update_tflops",
                                                                    "trailing_update_frac_of_hbm_peak", "trailing_update_frac_of_3xtf32_tcgen05_peak") if k in big32}
            ns["stage1_n16384_band64_f32"]["panel_ms"] = big32["classes"]["panel"]["ms"]
        if other:
            ns["config2_full_svd_n16384_f64"] = other.get("config3_full_svd")
        if batched_out:
            ns["config4_batched_8192x256"] = batched_out
        if dist_out:
            ns["config3_block_cyclic_stage1"] = dist_out
        if peaks:
            ns["peaks_measured_tflops"] = {k: round(v, 2) for k, v in peaks.items()}
        cfg["north_star"] = ns
        if detail:
            cfg["sweep_pct_of_fma_peak"] = {f"{dsc['n']}_{dsc['dtype']}": dsc.get("pct_of_fma_peak") for dsc in detail}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64,f32", "data": "synthetic", "config": cfg,
            "clocks": sampler.summary(), "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "roofline_north_star_f32": roofline_ns, "cpu_baseline": cpu,
            "kernel_classes_f64": prof_out, "north_star_shape": big, "north_star_shape_f32": big32, "other_configs": other, "multi_gpu_stage1": dist_out, "peaks_measured": {k: round(v, 2) for k, v in peaks.items()}, "detail": detail,
        }
        print(json.dumps(line), flush=True)
    for h in handles.values():
        h.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
