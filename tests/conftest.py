import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


class Oracle:
    """ctypes view of oracle/libsvd_oracle.so -- TEST-ONLY checker (never used by the product)."""

    def __init__(self, path):
        self.lib = ctypes.CDLL(path)
        self.lib.svdo_qrd_f32.restype = ctypes.c_longlong
        self.lib.svdo_qrd_f64.restype = ctypes.c_longlong
        self.lib.svdo_brd_p2_schedule_f64.restype = ctypes.c_size_t
        self.lib.svdo_mse_f32.restype = ctypes.c_float
        self.lib.svdo_mse_f64.restype = ctypes.c_double

    @staticmethod
    def suf(a):
        return {np.dtype(np.float32): "f32", np.dtype(np.float64): "f64"}[np.dtype(a.dtype)]

    @staticmethod
    def ptr(a):
        return a.ctypes.data_as(ctypes.c_void_p) if a is not None else None

    def brd_p1(self, a, band):
        x = np.ascontiguousarray(a).copy()
        rc = getattr(self.lib, "svdo_brd_p1_" + self.suf(x))(self.ptr(x), ctypes.c_size_t(x.shape[0]), ctypes.c_size_t(band))
        assert rc == 0
        return x

    def brd_p1_panel(self, a, band):
        x = np.ascontiguousarray(a).copy()
        rc = getattr(self.lib, "svdo_brd_p1_panel_" + self.suf(x))(self.ptr(x), ctypes.c_size_t(x.shape[0]), ctypes.c_size_t(band))
        assert rc == 0
        return x

    def brd_p2(self, a, band):
        x = np.ascontiguousarray(a).copy()
        n = x.shape[0]
        d = np.zeros(n, x.dtype)
        e = np.zeros(n - 1, x.dtype)
        rc = getattr(self.lib, "svdo_brd_p2_" + self.suf(x))(self.ptr(x), ctypes.c_size_t(n), ctypes.c_size_t(band), self.ptr(d), self.ptr(e))
        assert rc == 0
        return x, d, e

    def brd_p2_complete(self, a, band):
        """NOT the reference: same windows / arithmetic with every bulge chased to the end."""
        x = np.ascontiguousarray(a).copy()
        n = x.shape[0]
        d = np.zeros(n, x.dtype)
        e = np.zeros(n - 1, x.dtype)
        rc = getattr(self.lib, "svdo_brd_p2_complete_" + self.suf(x))(self.ptr(x), ctypes.c_size_t(n), ctypes.c_size_t(band), self.ptr(d), self.ptr(e))
        assert rc == 0
        return x, d, e

    def brd_serial(self, a):
        """csc586::serial::brd (one-stage Golub-Kahan): returns (A_out, d, e)"""
        x = np.ascontiguousarray(a).copy()
        n = x.shape[0]
        d = np.zeros(n, x.dtype)
        e = np.zeros(n - 1, x.dtype)
        rc = getattr(self.lib, "svdo_brd_serial_" + self.suf(x))(self.ptr(x), ctypes.c_size_t(n), self.ptr(d), self.ptr(e))
        assert rc == 0
        return x, d, e

    def qrd(self, d, e):
        d = np.ascontiguousarray(d).copy()
        e = np.ascontiguousarray(e).copy()
        thr = np.zeros(1, d.dtype)
        mi = ctypes.c_ulonglong(0)
        sweeps = getattr(self.lib, "svdo_qrd_" + self.suf(d))(self.ptr(d), self.ptr(e), ctypes.c_size_t(d.shape[0]), self.ptr(thr), ctypes.byref(mi))
        return d, e, int(sweeps), float(thr[0]), int(mi.value)

    def zero_shift(self, d, e):
        d = np.ascontiguousarray(d).copy()
        e = np.ascontiguousarray(e).copy()
        getattr(self.lib, "svdo_zero_shift_" + self.suf(d))(self.ptr(d), self.ptr(e), ctypes.c_size_t(d.shape[0]))
        return d, e

    def householder(self, x):
        x = np.ascontiguousarray(x)
        n = x.shape[0]
        w = np.zeros(n, x.dtype)
        H = np.zeros((n, n), x.dtype)
        tau = np.zeros(1, x.dtype)
        getattr(self.lib, "svdo_householder_" + self.suf(x))(self.ptr(x), ctypes.c_size_t(n), self.ptr(w), self.ptr(H), self.ptr(tau))
        return w, H, tau[0]

    def schedule(self, n, band):
        cnt = self.lib.svdo_brd_p2_schedule_f64(ctypes.c_size_t(n), ctypes.c_size_t(band), None, ctypes.c_size_t(0))
        out = np.zeros((cnt, 6), np.int64)
        self.lib.svdo_brd_p2_schedule_f64(ctypes.c_size_t(n), ctypes.c_size_t(band), self.ptr(out), ctypes.c_size_t(cnt))
        return out

    def mse(self, a, b, band):
        a = np.ascontiguousarray(a)
        b = np.ascontiguousarray(b)
        return float(getattr(self.lib, "svdo_mse_" + self.suf(a))(self.ptr(a), self.ptr(b), ctypes.c_size_t(a.shape[0]), ctypes.c_size_t(band)))


@pytest.fixture(scope="session")
def oracle():
    so = os.path.join(ROOT, "oracle", "libsvd_oracle.so")
    src = [os.path.join(ROOT, "oracle", f) for f in ("svd_oracle.c", "svd_oracle_impl.h", "svd_oracle.h")]
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in src):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), os.path.join(ROOT, "oracle", "libsvd_oracle.so")])
    return Oracle(so)


@pytest.fixture(scope="session")
def refso():
    """The compiled UNMODIFIED reference (oracle/_ref/libsvdref.so), if it has been built."""
    p = os.path.join(ROOT, "oracle", "_ref", "libsvdref.so")
    if not os.path.exists(p):
        pytest.skip("oracle/_ref/libsvdref.so not built (make -C oracle REF=<reference source tree>)")
    return ctypes.CDLL(p)


def load_fixture(kind, name, n):
    dt = {"float": np.float32, "double": np.float64}[name]
    return np.fromfile(os.path.join(GOLDEN, f"{kind}_{name}_{n}_{n}.bin"), dtype=dt).reshape(n, n)


def band_rel(a, ref, band):
    """SURVEY 8(c) tolerance definition: max abs diff over diagonals 0..band / max|ref|."""
    n = a.shape[0]
    num = 0.0
    for k in range(band + 1):
        num = max(num, float(np.abs(np.diagonal(a, k).astype(np.float64) - np.diagonal(ref, k).astype(np.float64)).max()))
    return num / float(np.abs(ref).max())


def band_sign_scaling(a, ref, band):
    """Diagonal +-1 scalings (d1, d2) with d1[i] * a[i, j] * d2[j] ~ ref[i, j] on the band: a maximum spanning tree of the
    bipartite row / column graph of the band (weights |ref[i, j]|, Prim) fixes one sign per row and column through the
    LARGEST entries.  Householder's sign rule (svd_serial.h:194: s = -sign(x0)) is discontinuous at x0 = 0, so a pivot
    that is tiny relative to the rounding noise of a float path can come out with either sign; everything downstream is
    equivariant under B -> D1 B D2 (SURVEY 8a'), which is also what the reference's own `mse` check ignores."""
    import heapq
    n = a.shape[0]
    a64, r64 = a.astype(np.float64), ref.astype(np.float64)
    d1, d2 = np.zeros(n), np.zeros(n)
    d1[0] = 1.0
    heap = []

    def push_row(i):
        for j in range(i, min(n, i + band + 1)):
            if d2[j] == 0:
                heapq.heappush(heap, (-abs(r64[i, j]), 0, i, j))

    def push_col(j):
        for i in range(max(0, j - band), j + 1):
            if d1[i] == 0:
                heapq.heappush(heap, (-abs(r64[i, j]), 1, i, j))

    push_row(0)
    while heap:
        _, kind, i, j = heapq.heappop(heap)
        sgn = 1.0 if a64[i, j] * r64[i, j] >= 0 else -1.0
        if kind == 0 and d2[j] == 0:          # row i known -> column j
            d2[j] = d1[i] * sgn
            push_col(j)
        elif kind == 1 and d1[i] == 0:        # column j known -> row i
            d1[i] = d2[j] * sgn
            push_row(i)
    d1[d1 == 0] = 1.0
    d2[d2 == 0] = 1.0
    return d1, d2


def band_rel_mod_signs(a, ref, band):
    """band_rel after the best +-1 row / column scaling; also returns how many rows / columns were flipped."""
    d1, d2 = band_sign_scaling(a, ref, band)
    scaled = (a.astype(np.float64) * d1[:, None]) * d2[None, :]
    return band_rel(scaled, ref, band), int((d1 < 0).sum() + (d2 < 0).sum())
