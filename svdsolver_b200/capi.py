"""ctypes binding of libsvdb200.so -- the C-ABI declared in include/svdb200.h.

This is the host-side mirror used by tests/ and bench.py; it never falls back to the CPU: if the
library is missing, or no CUDA device is usable, every call raises.
"""
import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SVDB200_LIB") or os.path.join(HERE, "libsvdb200.so")   # SVDB200_LIB: an instrumented build (tools/)

F32, F64 = 0, 1
ORDER_PANEL, ORDER_TILE = 0, 1

_lib = None


class SvdB200Error(RuntimeError):
    def __init__(self, status, msg):
        super().__init__(f"svdb200 status {status}: {msg}")
        self.status = status


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SvdB200Error(-100, f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                                     "(there is no CPU fallback)")
        _lib = ctypes.CDLL(LIB_PATH)
        _lib.svdb200_strerror.restype = ctypes.c_char_p
        _lib.svdb200_last_error.restype = ctypes.c_char_p
        _lib.svdb200_last_error.argtypes = [ctypes.c_void_p]
        _lib.svdb200_launch_count.restype = ctypes.c_longlong
        _lib.svdb200_launch_count.argtypes = [ctypes.c_void_p]
        _lib.svdb200_dist_local_cols.restype = ctypes.c_size_t
        _lib.svdb200_dist_launch_count.restype = ctypes.c_longlong
    return _lib


def _suf(dtype):
    dtype = np.dtype(dtype)
    if dtype == np.float32:
        return "f32", F32
    if dtype == np.float64:
        return "f64", F64
    raise TypeError(f"unsupported dtype {dtype}")


def _p(a):
    if a is None:
        return None
    if isinstance(a, int):
        return ctypes.c_void_p(a)
    return a.ctypes.data_as(ctypes.c_void_p)


Z = ctypes.c_size_t


def pack_upper_band(a, band):
    """LAPACK upper band storage of the diagonals 0..band of a square matrix, column by column: ab[j, t] = a[j - band + t, j]
    (zero above the matrix).  n x (band+1), the input of Handle.band_to_bidiag_packed / band_svdvals_packed; scipy's upper
    `ab` (ab[band + i - j, j] = a[i, j]) transposed."""
    a = np.asarray(a)
    n = a.shape[0]
    ab = np.zeros((n, band + 1), a.dtype)
    for t in range(band + 1):
        k = band - t                      # super-diagonal
        if k < n:
            ab[k:, t] = np.diagonal(a, k)
    return ab


class Handle:
    """svdb200_handle: workspace for matrices up to max_n x max_n with band `band`."""

    def __init__(self, max_n, band, dtype, device=0):
        self.suf, self.code = _suf(dtype)
        self.dtype = np.dtype(dtype)
        self.max_n, self.band = int(max_n), int(band)
        self.h = ctypes.c_void_p()
        st = lib().svdb200_create(ctypes.byref(self.h), ctypes.c_int(device), Z(max_n), Z(band), ctypes.c_int(self.code))
        if st != 0:
            self.h = ctypes.c_void_p()
            raise SvdB200Error(st, lib().svdb200_strerror(st).decode())

    def close(self):
        if self.h:
            lib().svdb200_destroy(self.h)
            self.h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, st):
        if st != 0:
            extra = lib().svdb200_last_error(self.h).decode()
            raise SvdB200Error(st, lib().svdb200_strerror(st).decode() + (f" [{extra}]" if extra else ""))

    def _fn(self, name):
        return getattr(lib(), f"svdb200_{name}_{self.suf}")

    def _mat(self, a):
        a = np.ascontiguousarray(a, dtype=self.dtype).copy()
        if a.ndim != 2:
            raise ValueError("matrix expected")
        return a

    # ---- host-pointer API (H2D/D2H inside the call, like the reference's timed region) ----
    def dense_to_band(self, a, band, order=ORDER_PANEL):
        a = self._mat(a)
        self._check(self._fn("dense_to_band")(self.h, _p(a), Z(a.shape[0]), Z(a.shape[1]), Z(band), ctypes.c_int(order)))
        return a

    def band_to_bidiag(self, a, band):
        a = self._mat(a)
        n = a.shape[1]
        d = np.zeros(n, self.dtype)
        e = np.zeros(max(n - 1, 0), self.dtype)
        self._check(self._fn("band_to_bidiag")(self.h, _p(a), Z(a.shape[0]), Z(n), Z(band), _p(d), _p(e)))
        return a, d, e

    def _band(self, ab, band):
        ab = np.ascontiguousarray(ab, dtype=self.dtype)
        if ab.ndim != 2 or ab.shape[1] != band + 1:
            raise ValueError("band storage n x (band+1) expected")
        return ab

    def band_to_bidiag_packed(self, ab, band):
        """stage 2 of the band matrix in upper band storage `ab` (pack_upper_band): returns (d, e); ab is not modified"""
        ab = self._band(ab, band)
        n = ab.shape[0]
        d = np.zeros(n, self.dtype)
        e = np.zeros(max(n - 1, 0), self.dtype)
        self._check(self._fn("band_to_bidiag_packed")(self.h, _p(ab), Z(n), Z(band), _p(d), _p(e)))
        return d, e

    def band_svdvals_packed(self, ab, band):
        """singular values (descending) of the band matrix in upper band storage `ab`; use set_stage2_schedule(1) for a
        generic band matrix"""
        ab = self._band(ab, band)
        sigma = np.zeros(ab.shape[0], self.dtype)
        self._check(self._fn("band_svdvals_packed")(self.h, _p(ab), Z(ab.shape[0]), Z(band), _p(sigma)))
        return sigma

    def bidiag_qr(self, d, e):
        d = np.ascontiguousarray(d, dtype=self.dtype)
        e = np.ascontiguousarray(e, dtype=self.dtype)
        sigma = np.zeros(d.shape[0], self.dtype)
        sweeps = ctypes.c_longlong(0)
        self._check(self._fn("bidiag_qr")(self.h, _p(d), _p(e), Z(d.shape[0]), _p(sigma), ctypes.byref(sweeps)))
        return sigma, int(sweeps.value)

    def bidiagonalize(self, a, band, order=ORDER_PANEL):
        a = self._mat(a)
        n = a.shape[1]
        d = np.zeros(n, self.dtype)
        e = np.zeros(max(n - 1, 0), self.dtype)
        self._check(self._fn("bidiagonalize")(self.h, _p(a), Z(a.shape[0]), Z(n), Z(band), ctypes.c_int(order), _p(d), _p(e)))
        return a, d, e

    def bidiagonalize_onestage(self, a):
        """one-stage Golub-Kahan bidiagonalisation (serial::brd order): returns (A_out, d, e)"""
        a = self._mat(a)
        n = a.shape[1]
        d = np.zeros(n, self.dtype)
        e = np.zeros(max(n - 1, 0), self.dtype)
        self._check(self._fn("bidiagonalize_onestage")(self.h, _p(a), Z(a.shape[0]), Z(n), _p(d), _p(e)))
        return a, d, e

    def bidiagonalize_inplace(self, a_ptr, n, band, d_ptr, e_ptr, order=ORDER_PANEL):
        """Host-pointer call on caller-owned (e.g. pinned) buffers given as raw addresses."""
        self._check(self._fn("bidiagonalize")(self.h, _p(a_ptr), Z(n), Z(n), Z(band), ctypes.c_int(order), _p(d_ptr), _p(e_ptr)))

    def bidiagonalize_dev(self, a_ptr, n, band, d_ptr, e_ptr, order=ORDER_PANEL):
        self._check(self._fn("bidiagonalize_dev")(self.h, _p(a_ptr), Z(n), Z(n), Z(band), ctypes.c_int(order), _p(d_ptr), _p(e_ptr)))

    def _ptr_arrays(self, ptrs):
        arr = (ctypes.c_void_p * len(ptrs))(*[ctypes.c_void_p(int(p)) if p else None for p in ptrs])
        return arr

    def bidiagonalize_many_dev(self, a_ptrs, ns, band, d_ptrs, e_ptrs, order=ORDER_PANEL):
        """Device pointers; stage 2 of matrix i overlaps stage 1 of matrix i+1."""
        cnt = len(a_ptrs)
        na = (ctypes.c_size_t * cnt)(*[int(x) for x in ns])
        self._check(self._fn("bidiagonalize_many_dev")(self.h, Z(cnt), self._ptr_arrays(a_ptrs), na, Z(band), ctypes.c_int(order),
                                                       self._ptr_arrays(d_ptrs), self._ptr_arrays(e_ptrs)))

    def bidiagonalize_many_inplace(self, a_ptrs, ns, band, d_ptrs, e_ptrs, order=ORDER_PANEL):
        """Host pointers (raw addresses of caller-owned, ideally pinned, buffers)."""
        cnt = len(a_ptrs)
        na = (ctypes.c_size_t * cnt)(*[int(x) for x in ns])
        self._check(self._fn("bidiagonalize_many")(self.h, Z(cnt), self._ptr_arrays(a_ptrs), na, Z(band), ctypes.c_int(order),
                                                   self._ptr_arrays(d_ptrs), self._ptr_arrays(e_ptrs)))

    def set_profile(self, on):
        self._check(lib().svdb200_set_profile(self.h, ctypes.c_int(1 if on else 0)))

    def reset_profile(self):
        self._check(lib().svdb200_reset_profile(self.h))

    PROFILE_CLASSES = ("panel", "gemm_tn", "gemm_nn", "rank_update", "stage2", "qr")

    def get_profile(self):
        ms = (ctypes.c_double * 6)(); work = (ctypes.c_double * 6)(); ln = (ctypes.c_longlong * 6)()
        self._check(lib().svdb200_get_profile(self.h, ms, work, ln))
        return {k: {"ms": ms[i], "work": work[i], "launches": int(ln[i])} for i, k in enumerate(self.PROFILE_CLASSES)}

    def svdvals(self, a, band, order=ORDER_PANEL):
        a = self._mat(a)
        sigma = np.zeros(a.shape[1], self.dtype)
        self._check(self._fn("svdvals")(self.h, _p(a), Z(a.shape[0]), Z(a.shape[1]), Z(band), ctypes.c_int(order), _p(sigma)))
        return sigma, a

    # ---- rectangular m x n (tall or wide); for m < n the result is lower band / bidiagonal, e the sub-diagonal ----
    def dense_to_band_mn(self, a, band):
        """stage 1 of an m x n matrix: returns the reduced matrix (upper band in the top n x n block for m >= n, lower band
        in the left m x m block for m < n, zeros elsewhere)"""
        a = self._mat(a)
        self._check(self._fn("dense_to_band_mn")(self.h, _p(a), Z(a.shape[0]), Z(a.shape[1]), Z(band)))
        return a

    def bidiagonalize_mn(self, a, band):
        """stages 1 and 2 of an m x n matrix: returns (A_out, d, e) with min(m, n) and min(m, n) - 1 entries"""
        a = self._mat(a)
        k = min(a.shape)
        d = np.zeros(k, self.dtype)
        e = np.zeros(max(k - 1, 0), self.dtype)
        self._check(self._fn("bidiagonalize_mn")(self.h, _p(a), Z(a.shape[0]), Z(a.shape[1]), Z(band), _p(d), _p(e)))
        return a, d, e

    def svdvals_mn(self, a, band):
        """singular values (descending, min(m, n)) of an m x n matrix: returns (sigma, A_out)"""
        a = self._mat(a)
        sigma = np.zeros(min(a.shape), self.dtype)
        self._check(self._fn("svdvals_mn")(self.h, _p(a), Z(a.shape[0]), Z(a.shape[1]), Z(band), _p(sigma)))
        return sigma, a

    def svdvals_batched(self, a, band):
        a = np.ascontiguousarray(a, dtype=self.dtype).copy()
        count, n, _ = a.shape
        sigma = np.zeros((count, n), self.dtype)
        self._check(self._fn("svdvals_batched")(self.h, _p(a), Z(count), Z(n), Z(band), _p(sigma)))
        return sigma

    def svdvals_batched_mn(self, a, band):
        """singular values of count m x n matrices (a: count x m x n): returns sigma, count x min(m, n), rows descending"""
        a = np.ascontiguousarray(a, dtype=self.dtype).copy()
        count, m, n = a.shape
        sigma = np.zeros((count, min(m, n)), self.dtype)
        self._check(self._fn("svdvals_batched_mn")(self.h, _p(a), Z(count), Z(m), Z(n), Z(band), _p(sigma)))
        return sigma

    def mse(self, a, b, band):
        a = np.ascontiguousarray(a, dtype=self.dtype)
        b = np.ascontiguousarray(b, dtype=self.dtype)
        out = np.zeros(1, self.dtype)
        self._check(self._fn("mse")(self.h, _p(a), _p(b), Z(a.shape[0]), Z(band), _p(out)))
        return float(out[0])

    # ---- device-pointer API (integers = CUdeviceptr, e.g. torch.Tensor.data_ptr()) ----
    def set_stream(self, stream_ptr):
        self._check(lib().svdb200_set_stream(self.h, ctypes.c_void_p(stream_ptr)))

    def synchronize(self):
        self._check(lib().svdb200_synchronize(self.h))

    def dense_to_band_dev(self, a_ptr, n, band, order=ORDER_PANEL):
        self._check(self._fn("dense_to_band_dev")(self.h, _p(a_ptr), Z(n), Z(n), Z(band), ctypes.c_int(order)))

    def band_to_bidiag_dev(self, a_ptr, n, band, d_ptr, e_ptr):
        self._check(self._fn("band_to_bidiag_dev")(self.h, _p(a_ptr), Z(n), Z(n), Z(band), _p(d_ptr), _p(e_ptr)))

    def band_to_bidiag_packed_dev(self, ab_ptr, n, band, d_ptr, e_ptr):
        self._check(self._fn("band_to_bidiag_packed_dev")(self.h, _p(ab_ptr), Z(n), Z(band), _p(d_ptr), _p(e_ptr)))

    def band_svdvals_packed_dev(self, ab_ptr, n, band, sigma_ptr):
        self._check(self._fn("band_svdvals_packed_dev")(self.h, _p(ab_ptr), Z(n), Z(band), _p(sigma_ptr)))

    def bidiag_qr_dev(self, d_ptr, e_ptr, n, sigma_ptr):
        self._check(self._fn("bidiag_qr_dev")(self.h, _p(d_ptr), _p(e_ptr), Z(n), _p(sigma_ptr)))

    def svdvals_dev(self, a_ptr, n, band, sigma_ptr, order=ORDER_PANEL):
        self._check(self._fn("svdvals_dev")(self.h, _p(a_ptr), Z(n), Z(n), Z(band), ctypes.c_int(order), _p(sigma_ptr)))

    def dense_to_band_mn_dev(self, a_ptr, m, n, band):
        self._check(self._fn("dense_to_band_mn_dev")(self.h, _p(a_ptr), Z(m), Z(n), Z(band)))

    def bidiagonalize_mn_dev(self, a_ptr, m, n, band, d_ptr, e_ptr):
        self._check(self._fn("bidiagonalize_mn_dev")(self.h, _p(a_ptr), Z(m), Z(n), Z(band), _p(d_ptr), _p(e_ptr)))

    def svdvals_mn_dev(self, a_ptr, m, n, band, sigma_ptr):
        self._check(self._fn("svdvals_mn_dev")(self.h, _p(a_ptr), Z(m), Z(n), Z(band), _p(sigma_ptr)))

    def svdvals_batched_dev(self, a_ptr, count, n, band, sigma_ptr):
        self._check(self._fn("svdvals_batched_dev")(self.h, _p(a_ptr), Z(count), Z(n), Z(band), _p(sigma_ptr)))

    def chain_batched_dev(self, a_ptr, count, n, band, what, d_ptr=None, e_ptr=None, sigma_ptr=None):
        """stages of the batched path: what = 1 stage 1 | 2 stage 2 | 4 singular values"""
        self._check(self._fn("chain_batched_dev")(self.h, _p(a_ptr), Z(count), Z(n), Z(band), ctypes.c_int(what), _p(d_ptr), _p(e_ptr), _p(sigma_ptr)))

    def svdvals_batched_mn_dev(self, a_ptr, count, m, n, band, sigma_ptr):
        self._check(self._fn("svdvals_batched_mn_dev")(self.h, _p(a_ptr), Z(count), Z(m), Z(n), Z(band), _p(sigma_ptr)))

    def chain_batched_mn_dev(self, a_ptr, count, m, n, band, what, d_ptr=None, e_ptr=None, sigma_ptr=None):
        """stages of the batched path on count m x n matrices: what = 1 stage 1 | 2 stage 2 | 4 singular values; d, e, sigma
        count x min(m, n)"""
        self._check(self._fn("chain_batched_mn_dev")(self.h, _p(a_ptr), Z(count), Z(m), Z(n), Z(band), ctypes.c_int(what),
                                                     _p(d_ptr), _p(e_ptr), _p(sigma_ptr)))

    def set_band_capture(self, dev_ptrs):
        """test hook: device buffers that receive the band of matrix i of the next bidiagonalize_many_* call"""
        self._check(lib().svdb200_set_band_capture(self.h, self._ptr_arrays(dev_ptrs), Z(len(dev_ptrs))))

    def fill_uniform_dev(self, a_ptr, count, seed, lo=0.0, hi=5.0):
        self._check(self._fn("fill_uniform_dev")(self.h, _p(a_ptr), Z(count), ctypes.c_ulonglong(seed), ctypes.c_double(lo), ctypes.c_double(hi)))

    def gemm_tn_dev(self, v_ptr, c_ptr, ldc, mrows, ncols, b, w_ptr):
        self._check(self._fn("gemm_tn_dev")(self.h, _p(v_ptr), _p(c_ptr), Z(ldc), Z(mrows), Z(ncols), Z(b), _p(w_ptr)))

    def gemm_nn_dev(self, c_ptr, ldc, mrows, ncols, b, ut_ptr, w_ptr):
        self._check(self._fn("gemm_nn_dev")(self.h, _p(c_ptr), Z(ldc), Z(mrows), Z(ncols), Z(b), _p(ut_ptr), _p(w_ptr)))

    def rank_update_dev(self, c_ptr, ldc, mrows, ncols, b, p_ptr, q_ptr, ldq):
        self._check(self._fn("rank_update_dev")(self.h, _p(c_ptr), Z(ldc), Z(mrows), Z(ncols), Z(b), _p(p_ptr), _p(q_ptr), Z(ldq)))

    def panel_factor_dev(self, a_ptr, lda, m, b, trans, v_ptr, v2_ptr):
        """one stage-1 panel (QR of the m x b column panel, or LQ of the b x m row panel when trans)"""
        self._check(self._fn("panel_factor_dev")(self.h, _p(a_ptr), Z(lda), Z(m), Z(b), ctypes.c_int(1 if trans else 0), _p(v_ptr), _p(v2_ptr)))

    def set_panel_kernel(self, kind):
        """stage-1 panel kernel: 2 = Cholesky-QR with reconstructed Householder vectors (default), 1 = blocked, 0 = per-column"""
        self._check(lib().svdb200_set_panel_kernel(self.h, ctypes.c_int(kind)))

    def set_chol_guard(self, guard):
        """smallest pivot ratio the Cholesky-QR panel accepts before the exchange-based kernels redo the panel"""
        self._check(lib().svdb200_set_chol_guard(self.h, ctypes.c_double(guard)))

    def chol_fallback_count(self):
        v = ctypes.c_longlong(0)
        self._check(lib().svdb200_chol_fallback_count(self.h, ctypes.byref(v)))
        return int(v.value)

    def last_timings(self):
        v = [ctypes.c_double(0) for _ in range(5)]
        self._check(lib().svdb200_last_timings(self.h, *[ctypes.byref(x) for x in v]))
        return dict(zip(("stage1_ms", "stage2_ms", "qr_ms", "h2d_ms", "d2h_ms"), [x.value for x in v]))

    def set_tc05(self, mode, min_elems=0):
        """FP32 tcgen05/TMEM/TMA trailing update: 0 off, 1 auto (size threshold), 2 always."""
        self._check(lib().svdb200_set_tc05(self.h, ctypes.c_int(mode), ctypes.c_longlong(min_elems)))

    def set_stage2_schedule(self, mode):
        """0 = the reference's window schedule (default, parity); 1 = complete chase (singular values preserved)."""
        self._check(lib().svdb200_set_stage2_schedule(self.h, ctypes.c_int(mode)))

    def set_qr_method(self, method, auto_limit=0):
        """0 auto, 1 zero-shift QR sweeps (reference algorithm), 2 bisection, 3 implicit shifted QR."""
        self._check(lib().svdb200_set_qr_method(self.h, ctypes.c_int(method), Z(auto_limit)))

    def launch_count(self):
        return int(lib().svdb200_launch_count(self.h))

    def probe_peak(self, kind):
        out = ctypes.c_double(0)
        self._check(lib().svdb200_probe_peak(self.h, ctypes.c_int(kind), ctypes.byref(out)))
        return out.value
