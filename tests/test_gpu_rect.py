"""Rectangular m x n matrices (svdb200_dense_to_band_mn_* / svdb200_bidiagonalize_mn_* / svdb200_svdvals_mn_*).

Tall matrices run the panel-order driver with panel heights m - k; wide ones are transposed on the device and reduced as
tall.  So: at m == n the calls are byte-equal to the square calls, tall stage 1 matches the CPU reference
(tests/rect_reference.c) through every panel kernel, a wide matrix gives the transpose of what its transpose gives, and
the singular values match LAPACK under the complete stage-2 schedule."""
import contextlib
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, band_rel
from svdsolver_b200.synth import uniform_matrix

pytestmark = pytest.mark.gpu

DT = {"f32": np.float32, "f64": np.float64}
TOL = {"f32": 1e-4, "f64": 1e-10}
ABOVE = {"f32": 1e-4, "f64": 1e-12}
SIG = {"f32": 2e-5, "f64": 1e-11}
MAX_N, MAX_B = 16384, 64
TALL = [(65, 64, 4), (100, 64, 8), (257, 128, 32), (321, 320, 32), (640, 320, 32), (1000, 96, 32), (1536, 512, 64),
        (2048, 256, 16)]


@pytest.fixture(scope="module")
def capi():
    from svdsolver_b200 import capi as m
    m.lib()
    return m


@pytest.fixture(scope="module")
def handles(capi):
    hs = {s: capi.Handle(MAX_N, MAX_B, dt) for s, dt in DT.items()}
    yield hs
    for h in hs.values():
        h.close()


@pytest.fixture(scope="module")
def rectref(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("rectref") / "librectref.so")
    subprocess.check_call(["gcc", "-std=c11", "-O2", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared",
                           "-I", os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests", "rect_reference.c"), "-o", out, "-lm"])
    lib = ctypes.CDLL(out)
    cache = {}

    def reduce_tall(a, b):
        key = (a.shape, a.dtype.str, b, hash(a.tobytes()))
        if key not in cache:
            x = np.ascontiguousarray(a).copy()
            suf = "f32" if x.dtype == np.float32 else "f64"
            rc = getattr(lib, f"rect_brd_p1_panel_mn_{suf}")(x.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(x.shape[0]),
                                                              ctypes.c_size_t(x.shape[1]), ctypes.c_size_t(b))
            assert rc == 0
            cache[key] = x
        return cache[key]
    return reduce_tall


def _same(x, y):
    x, y = np.asarray(x), np.asarray(y)
    return x.shape == y.shape and np.array_equal(x.view(np.uint8), y.view(np.uint8))


@contextlib.contextmanager
def complete_schedule(h):
    """sigma needs the complete stage-2 schedule: on the default schedule's bidiagonal the zero-shift QR may not converge"""
    h.set_stage2_schedule(1)
    try:
        yield h
    finally:
        h.set_stage2_schedule(0)


def _mat(m, n, b, suf):
    return uniform_matrix(m, n, 586 + m + 3 * n + b, 0.0, 5.0, DT[suf])


def _check_tall_band(out, ref, n, b, suf):
    top = out[:n]
    assert np.all(out[n:] == 0)
    assert np.all(np.tril(top, -1) == 0)
    assert band_rel(top, ref[:n], b) <= TOL[suf]
    assert np.abs(np.triu(top, b + 1)).max() <= ABOVE[suf] * np.abs(ref).max()


# ------------------------------------------------------------------ m == n: the square calls ------------------------------
@pytest.mark.parametrize("n,b", [(64, 4), (256, 32), (320, 32), (512, 64)])
@pytest.mark.parametrize("suf", ["f32", "f64"])
def test_square_equals_square(capi, handles, n, b, suf):
    h = handles[suf]
    a = _mat(n, n, b, suf)
    assert _same(h.dense_to_band_mn(a, b), h.dense_to_band(a, b, capi.ORDER_PANEL))
    out, d, e = h.bidiagonalize_mn(a, b)
    out0, d0, e0 = h.bidiagonalize(a, b, capi.ORDER_PANEL)
    assert _same(out, out0) and _same(d, d0) and _same(e, e0)
    with complete_schedule(h):
        s, out = h.svdvals_mn(a, b)
        s0, out0 = h.svdvals(a, b, capi.ORDER_PANEL)
    assert _same(s, s0) and _same(out, out0)


# ------------------------------------------------------------------ tall stage 1 against the reference ---------------------
@pytest.mark.parametrize("m,n,b", TALL)
@pytest.mark.parametrize("suf", ["f32", "f64"])
def test_tall_stage1_vs_reference(handles, rectref, m, n, b, suf):
    a = _mat(m, n, b, suf)
    _check_tall_band(handles[suf].dense_to_band_mn(a, b), rectref(a, b), n, b, suf)


@pytest.mark.parametrize("m,n,b", [(1000, 96, 32), (2048, 256, 16)])
@pytest.mark.parametrize("kind,suf", [(k, s) for s in ("f32", "f64") for k in (0, 1, 2)] + [("tc05", "f32")])
def test_tall_every_panel_kernel(capi, rectref, m, n, b, kind, suf):
    """ragged panel heights (m - k not a multiple of 8, 16 or 32) through each panel kernel and, in f32, the forced tcgen05
    update"""
    a = _mat(m, n, b, suf)
    with capi.Handle(m, b, DT[suf]) as h:
        if kind == "tc05":
            h.set_tc05(2)
        else:
            h.set_panel_kernel(kind)
        out = h.dense_to_band_mn(a, b)
    _check_tall_band(out, rectref(a, b), n, b, suf)


# ------------------------------------------------------------------ wide = transpose of tall ------------------------------
@pytest.mark.parametrize("m,n,b", TALL)
@pytest.mark.parametrize("suf", ["f32", "f64"])
def test_wide_is_transpose_of_tall(handles, m, n, b, suf):
    h = handles[suf]
    a = _mat(m, n, b, suf)
    at = np.ascontiguousarray(a.T)
    band_w = h.dense_to_band_mn(at, b)
    assert _same(band_w, np.ascontiguousarray(h.dense_to_band_mn(a, b).T))
    assert np.all(band_w[:, n:] == 0) and np.all(np.triu(band_w[:, :n], 1) == 0)
    out, d, e = h.bidiagonalize_mn(a, b)
    out_w, d_w, e_w = h.bidiagonalize_mn(at, b)
    assert _same(out_w, np.ascontiguousarray(out.T)) and _same(d_w, d) and _same(e_w, e)
    assert d.shape == (n,) and e.shape == (n - 1,)
    with complete_schedule(h):
        s, _ = h.svdvals_mn(a, b)
        s_w, _ = h.svdvals_mn(at, b)
    assert _same(s_w, s)


# ------------------------------------------------------------------ singular values against LAPACK ---------------------------
@pytest.mark.parametrize("m,n,b,suf", [(3000, 1024, 32, "f64"), (1024, 3000, 32, "f64"), (2000, 768, 64, "f32"),
                                       (768, 2000, 64, "f32"), (4096, 64, 32, "f64")])
def test_svdvals_vs_lapack(capi, m, n, b, suf):
    a = _mat(m, n, b, suf)
    s0 = np.linalg.svd(a.astype(np.float64), compute_uv=False)
    with capi.Handle(max(m, n), b, DT[suf]) as h:
        h.set_stage2_schedule(1)
        s, out = h.svdvals_mn(a, b)
    assert s.shape == (min(m, n),)
    assert np.all(np.diff(s.astype(np.float64)) <= 0)
    assert np.abs(s.astype(np.float64) - s0).max() <= SIG[suf] * s0[0]
    k = min(m, n)
    assert np.all(out[k:] == 0) and np.all(out[:, k:] == 0)


@pytest.mark.parametrize("m,n,suf", [(16384, 2048, "f64"), (2048, 16384, "f32")])
def test_large(handles, m, n, suf):
    b = 64
    h = handles[suf]
    a = _mat(m, n, b, suf)
    a64 = a.astype(np.float64)
    fa = np.linalg.norm(a64)
    band = h.dense_to_band_mn(a, b).astype(np.float64)
    assert abs(np.linalg.norm(band) - fa) <= (1e-12 if suf == "f64" else 1e-5) * fa
    with complete_schedule(h):
        s, _ = h.svdvals_mn(a, b)
    s0 = np.linalg.svd(a64, compute_uv=False)
    assert np.abs(s.astype(np.float64) - s0).max() <= SIG[suf] * s0[0]


# ------------------------------------------------------------------ host and device variants ---------------------------------
@pytest.mark.parametrize("m,n,b", [(640, 320, 32), (320, 640, 32)])
@pytest.mark.parametrize("suf", ["f32", "f64"])
def test_host_equals_device(handles, m, n, b, suf):
    import torch
    with complete_schedule(handles[suf]) as h:
        _host_equals_device(torch, h, m, n, b, suf)


def _host_equals_device(torch, h, m, n, b, suf):
    a = _mat(m, n, b, suf)
    k = min(m, n)
    band = h.dense_to_band_mn(a, b)
    assert h.last_timings()["stage1_ms"] > 0
    out, d, e = h.bidiagonalize_mn(a, b)
    t = h.last_timings()
    assert t["stage1_ms"] > 0 and t["stage2_ms"] > 0
    s, out_s = h.svdvals_mn(a, b)
    assert h.last_timings()["qr_ms"] > 0

    def dev():
        return torch.from_numpy(a.copy()).cuda()
    tdt = torch.float32 if suf == "f32" else torch.float64
    x1, x2, x3 = dev(), dev(), dev()
    dd = torch.zeros(k, dtype=tdt, device="cuda")
    ed = torch.zeros(k - 1, dtype=tdt, device="cuda")
    sd = torch.zeros(k, dtype=tdt, device="cuda")
    torch.cuda.synchronize()
    h.dense_to_band_mn_dev(x1.data_ptr(), m, n, b)
    h.bidiagonalize_mn_dev(x2.data_ptr(), m, n, b, dd.data_ptr(), ed.data_ptr())
    h.svdvals_mn_dev(x3.data_ptr(), m, n, b, sd.data_ptr())
    h.synchronize()
    assert _same(x1.cpu().numpy(), band)
    assert _same(x2.cpu().numpy(), out) and _same(dd.cpu().numpy(), d) and _same(ed.cpu().numpy(), e)
    assert _same(x3.cpu().numpy(), out_s) and _same(sd.cpu().numpy(), s)


def test_scratch_growth(capi):
    """the wide-matrix scratch buffer grows on one handle; results do not depend on what ran before"""
    b = 32
    shapes = [(128, 512), (512, 2048), (128, 512)]
    got = []
    with capi.Handle(2048, b, np.float64) as h:
        for m, n in shapes:
            got.append(h.bidiagonalize_mn(_mat(m, n, b, "f64"), b))
    for (m, n), g in zip(shapes, got):
        with capi.Handle(2048, b, np.float64) as f:
            ref = f.bidiagonalize_mn(_mat(m, n, b, "f64"), b)
        assert all(_same(x, y) for x, y in zip(g, ref))


# ------------------------------------------------------------------ statuses ------------------------------------------------
def test_statuses(capi):
    lib = capi.lib()
    Z = ctypes.c_size_t
    with capi.Handle(256, 32, np.float64) as h:
        def st(name, m, n, band, a=True, dtype=np.float64, extra=True):
            x = uniform_matrix(1, max(m * n, 1), 586, 0.0, 5.0, dtype)
            o = np.zeros(512, dtype)
            p = x.ctypes.data_as(ctypes.c_void_p) if a else None
            q = o.ctypes.data_as(ctypes.c_void_p) if extra else None
            f = getattr(lib, f"svdb200_{name}_{'f32' if dtype == np.float32 else 'f64'}")
            if name.startswith("bidiagonalize_mn"):
                return f(h.h, p, Z(m), Z(n), Z(band), q, q)
            if name.startswith("svdvals_mn"):
                return f(h.h, p, Z(m), Z(n), Z(band), q)
            return f(h.h, p, Z(m), Z(n), Z(band))
        host = ["dense_to_band_mn", "bidiagonalize_mn", "svdvals_mn"]
        for name in host + [x + "_dev" for x in host]:
            dev = name.endswith("_dev")
            assert st(name, 64, 32, 8, a=False) == -1
            assert st(name, 64, 32, 8, dtype=np.float32) == -1              # dtype of the handle is f64
            if not name.startswith("dense_to_band"):
                assert st(name, 64, 32, 8, extra=False) == -1
            assert st(name, 64, 1, 1) == -2                                 # min(m, n) < 2
            assert st(name, 64, 32, 0) == -2
            assert st(name, 64, 30, 8) == -2                                # band does not divide min(m, n)
            assert st(name, 30, 64, 8) == -2
            assert st(name, 512, 32, 8) == -3                               # max(m, n) > max_n
            assert st(name, 32, 512, 8) == -3
            assert st(name, 128, 64, 64) == -3                              # band > the handle's band
            if not dev:
                assert st(name, 100, 64, 8) == 0                            # the longer side is arbitrary
                assert st(name, 64, 100, 8) == 0
        # the square calls keep rejecting m != n
        a = np.zeros((64, 32))
        with pytest.raises(capi.SvdB200Error) as ei:
            h.svdvals(a, 8)
        assert ei.value.status == -2
        with pytest.raises(capi.SvdB200Error) as ei:
            h.bidiagonalize(a, 8)
        assert ei.value.status == -2
