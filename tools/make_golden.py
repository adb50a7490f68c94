#!/usr/bin/env python
"""Regenerates tests/golden/ (run in the BUILD container only; needs /root/reference + oracle/_ref).

* copies the reference's verified fixtures (data/{test,band,bidiagonal}_{float,double}_{64,512})
  unchanged -- they are the golden vectors of SURVEY 8(c);
* regenerates the six 1024 fixtures the reference mount lacks (.MISSING_LARGE_BLOBS): the input is
  synth.uniform_matrix(1024,1024, seed=586+1024, lo=1, hi=5) (fixtures are U[1,5)), pushed through
  the COMPILED REFERENCE (oracle/_ref/libsvdref.so: parallel::brd_p1(A,4) then parallel::brd_p2(A,4)).
  Only digests + the meaningful diagonals are committed (golden_1024.npz); the tests regenerate the
  full matrices with the C oracle and compare sha256, which pins the oracle to the reference at 1024;
* records reference outputs for a few seeded random cases at other band sizes, float qrd results,
  and Householder known-answer vectors.
"""
import ctypes, hashlib, json, os, shutil, sys
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from svdsolver_b200.synth import uniform_matrix  # noqa: E402

REF = "/root/reference/data"
OUT = os.path.join(ROOT, "tests", "golden")
L = ctypes.CDLL(os.path.join(ROOT, "oracle", "_ref", "libsvdref.so"))
P = lambda a: a.ctypes.data_as(ctypes.c_void_p)
Z = ctypes.c_size_t
DT = {"f32": np.float32, "f64": np.float64}
sha = lambda a: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def ref_chain(a, band, suf):
    n = a.shape[0]
    x = np.ascontiguousarray(a).copy()
    getattr(L, f"svdref_brd_p1_{suf}")(P(x), Z(n), Z(band))
    band_m = x.copy()
    d = np.zeros(n, x.dtype); e = np.zeros(n - 1, x.dtype)
    getattr(L, f"svdref_brd_p2_{suf}")(P(x), Z(n), Z(band), P(d), P(e))
    return band_m, x, d, e


def onestage():
    """csc586::serial::brd<T> (svd_serial.h:233) on seeded inputs: full output matrix + (d, e)."""
    z = {}
    for n in (8, 48, 96):
        for suf, dt in DT.items():
            a = uniform_matrix(n, n, 586 + n, 0.0, 5.0, dt)
            x = a.copy(); d = np.zeros(n, dt); e = np.zeros(n - 1, dt)
            getattr(L, f"svdref_serial_brd_{suf}")(P(x), Z(n), P(d), P(e))
            z[f"brd_{n}_{suf}"] = x; z[f"brd_d_{n}_{suf}"] = d; z[f"brd_e_{n}_{suf}"] = e
    np.savez_compressed(os.path.join(OUT, "golden_onestage.npz"), **z)


def refcheck():
    """parallel::brd_p1<double>(A, 8) and then parallel::brd_p2 on the seed-11 80x80 input of
    tests/test_oracle.py::test_compiled_reference_agrees_when_present: both full output matrices."""
    a = uniform_matrix(80, 80, 11, 0.0, 5.0, np.float64)
    band_m, bid_m, _, _ = ref_chain(a, 8, "f64")
    np.savez_compressed(os.path.join(OUT, "golden_refcheck.npz"), band_80_8_f64=band_m, bidiag_80_8_f64=bid_m)


def main():
    os.makedirs(OUT, exist_ok=True)
    if "--only-onestage" in sys.argv:
        onestage()
        return
    if "--only-refcheck" in sys.argv:
        refcheck()
        return
    onestage()
    refcheck()
    for n in (64, 512):
        for name in ("float", "double"):
            for kind in ("test", "band", "bidiagonal"):
                f = f"{kind}_{name}_{n}_{n}.bin"
                shutil.copyfile(os.path.join(REF, f), os.path.join(OUT, f))
    meta = {}
    # --- 1024 fixtures (band 4), via the compiled reference ---
    z = {}
    for suf, dt in DT.items():
        a = uniform_matrix(1024, 1024, 586 + 1024, 1.0, 5.0, dt)
        band_m, bid_m, d, e = ref_chain(a, 4, suf)
        meta[f"1024_{suf}"] = {"input_sha256": sha(a), "band_sha256": sha(band_m), "bidiagonal_sha256": sha(bid_m)}
        z[f"band_diags_{suf}"] = np.stack([np.pad(np.diagonal(band_m, k), (0, k)) for k in range(5)])
        z[f"bidiag_d_{suf}"] = d
        z[f"bidiag_e_{suf}"] = e
        print("1024", suf, meta[f"1024_{suf}"])
    np.savez_compressed(os.path.join(OUT, "golden_1024.npz"), **z)
    # --- seeded random cases at other band sizes: full outputs are small ---
    z = {}
    for (n, b) in ((96, 32), (128, 16), (64, 8), (192, 32), (256, 64), (40, 4), (32, 32)):
        for suf, dt in DT.items():
            a = uniform_matrix(n, n, 586 + n + b, 0.0, 5.0, dt)
            band_m, bid_m, d, e = ref_chain(a, b, suf)
            z[f"band_{n}_{b}_{suf}"] = band_m
            z[f"bidiag_{n}_{b}_{suf}"] = bid_m
    np.savez_compressed(os.path.join(OUT, "golden_random.npz"), **z)
    # --- panel-order (gpu::brd_p1, float only in the reference) ---
    z = {}
    for (n, b) in ((64, 4), (96, 32), (128, 16), (256, 32)):
        a = uniform_matrix(n, n, 586 + n + b, 0.0, 5.0, np.float32)
        x = a.copy()
        L.svdref_gpu_brd_p1_f32(P(x), Z(n), Z(b))
        z[f"panel_band_{n}_{b}_f32"] = x
    np.savez_compressed(os.path.join(OUT, "golden_panel.npz"), **z)
    # --- serial::qrd<float> on seeded bidiagonals and on the float fixtures' bidiagonals ---
    z = {}
    for n in (8, 64, 320, 640):
        de = uniform_matrix(2, n, 586 + n, 0.0, 5.0, np.float32)
        d0, e0 = de[0].copy(), de[1, : n - 1].copy()
        do = np.zeros(n, np.float32); eo = np.zeros(n - 1, np.float32)
        L.svdref_qrd_f32(P(d0), P(e0), Z(n), P(do), P(eo))
        z[f"qrd_sigma_{n}"] = do
    for n in (64, 512):
        m = np.fromfile(os.path.join(REF, f"bidiagonal_float_{n}_{n}.bin"), dtype=np.float32).reshape(n, n)
        d0 = np.ascontiguousarray(np.diagonal(m)).copy(); e0 = np.ascontiguousarray(np.diagonal(m, 1)).copy()
        do = np.zeros(n, np.float32); eo = np.zeros(n - 1, np.float32)
        L.svdref_qrd_f32(P(d0), P(e0), Z(n), P(do), P(eo))
        z[f"qrd_sigma_fixture_{n}"] = do
    np.savez_compressed(os.path.join(OUT, "golden_qrd.npz"), **z)
    # --- Householder known answers ---
    z = {}
    rng = np.random.default_rng(586)
    for suf, dt in DT.items():
        for ln in (1, 2, 5, 33):
            x = rng.uniform(-3, 3, ln).astype(dt)
            w = np.zeros(ln, dt); H = np.zeros(ln * ln, dt); tau = np.zeros(1, dt)
            getattr(L, f"svdref_householder_{suf}")(P(x), Z(ln), P(w), P(H), P(tau))
            z[f"hh_x_{ln}_{suf}"] = x; z[f"hh_w_{ln}_{suf}"] = w; z[f"hh_H_{ln}_{suf}"] = H; z[f"hh_tau_{ln}_{suf}"] = tau
    np.savez_compressed(os.path.join(OUT, "golden_householder.npz"), **z)
    with open(os.path.join(OUT, "golden_meta.json"), "w") as f:
        json.dump(meta, f, indent=1, sort_keys=True)


if __name__ == "__main__":
    main()
