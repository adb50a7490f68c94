"""Batched rectangular matrices (svdb200_svdvals_batched_mn_* / svdb200_chain_batched_mn_dev_*).

The batched small-matrix driver takes count m x n matrices: tall ones get taller QR panels, wide ones are transposed on the
device and reduced as tall.  So: at m == n the calls are byte-equal to the square batched calls, tall stage 1 matches the
CPU reference (tests/rect_reference.c), the batched stage 2 is byte-equal to the oracle on the top block, a wide batch
gives the transposes of its tall counterpart, sigma matches LAPACK, a matrix's result does not depend on its neighbours or
on the chunk it falls in, the work is batched, and shapes outside the kernels' range take the single-matrix chain."""
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
SIG = {"f32": 2e-5, "f64": 1e-11}
MAX_N, MAX_B = 4096, 64
TALL = [(9, 100, 64, 8), (12, 257, 128, 32), (6, 1000, 96, 32), (5, 1536, 512, 64), (3, 2048, 256, 16)]
Z = ctypes.c_size_t


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

    def reduce_tall(a, b):
        x = np.ascontiguousarray(a).copy()
        suf = "f32" if x.dtype == np.float32 else "f64"
        rc = getattr(lib, f"rect_brd_p1_panel_mn_{suf}")(x.ctypes.data_as(ctypes.c_void_p), Z(x.shape[0]), Z(x.shape[1]), Z(b))
        assert rc == 0
        return x
    return reduce_tall


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


def _same(x, y):
    x, y = np.asarray(x), np.asarray(y)
    return x.shape == y.shape and np.array_equal(x.view(np.uint8), y.view(np.uint8))


@contextlib.contextmanager
def settings(h, schedule=1, qr_method=0):
    """sigma of a generic matrix needs the complete stage-2 schedule"""
    h.set_stage2_schedule(schedule)
    h.set_qr_method(qr_method)
    try:
        yield h
    finally:
        h.set_stage2_schedule(0)
        h.set_qr_method(0)


def _batch(count, m, n, suf, seed=0):
    return np.stack([uniform_matrix(m, n, 586 + 7919 * seed + 31 * i + m + 3 * n, 0.0, 5.0, DT[suf]) for i in range(count)])


def _tdt(torch, suf):
    return torch.float32 if suf == "f32" else torch.float64


def _host(h, name, a, *dims):
    """a host-pointer batched call on a copy of a: returns (sigma, a_out)"""
    a = np.ascontiguousarray(a).copy()
    count = a.shape[0]
    sigma = np.zeros((count, min(a.shape[1], a.shape[2])), a.dtype)
    h._check(h._fn(name)(h.h, a.ctypes.data_as(ctypes.c_void_p), Z(count), *[Z(x) for x in dims], sigma.ctypes.data_as(ctypes.c_void_p)))
    return sigma, a


def _chain(torch, h, a, b, what, call="mn", d=None, e=None, s=None):
    """chain_batched_mn_dev (call "mn") or chain_batched_dev (call "sq") on the device tensor a (count x m x n), in place"""
    count, m, n = a.shape
    p = [x.data_ptr() if x is not None else None for x in (d, e, s)]
    if call == "mn":
        h.chain_batched_mn_dev(a.data_ptr(), count, m, n, b, what, *p)
    else:
        h.chain_batched_dev(a.data_ptr(), count, n, b, what, *p)
    h.synchronize()


def _stages(torch, h, a_host, b, suf):
    """stage 1, then stages 2 and sigma, of the batch a_host: (bands, reduced, d, e, sigma) as numpy"""
    count, m, n = a_host.shape
    k = min(m, n)
    x = torch.from_numpy(a_host.copy()).cuda()
    d, e, s = (torch.zeros(count, k, dtype=_tdt(torch, suf), device="cuda") for _ in range(3))
    _chain(torch, h, x, b, 1)
    bands = x.cpu().numpy()
    _chain(torch, h, x, b, 2 | 4, d=d, e=e, s=s)
    return bands, x.cpu().numpy(), d.cpu().numpy(), e.cpu().numpy(), s.cpu().numpy()


# ------------------------------------------------------------------ 1. m == n: the square batched calls -----------------------
@pytest.mark.parametrize("count,n,b", [(24, 256, 32), (10, 128, 16), (3, 1024, 64)])
@pytest.mark.parametrize("suf", ["f32", "f64"])
def test_square_equals_square_batched(torch, handles, count, n, b, suf):
    h = handles[suf]
    a = _batch(count, n, n, suf)
    s, out = _host(h, "svdvals_batched_mn", a, n, n, b)
    s0, out0 = _host(h, "svdvals_batched", a, n, b)
    assert _same(s, s0) and _same(out, out0)
    assert _same(h.svdvals_batched_mn(a, b), s0)
    res = {}
    for call in ("mn", "sq"):
        x = torch.from_numpy(a.copy()).cuda()
        d, e, sg = (torch.zeros(count, n, dtype=_tdt(torch, suf), device="cuda") for _ in range(3))
        _chain(torch, h, x, b, 1, call)
        r = [x.cpu().numpy()]
        _chain(torch, h, x, b, 2 | 4, call, d, e, sg)
        r += [x.cpu().numpy(), d.cpu().numpy(), e.cpu().numpy(), sg.cpu().numpy()]
        x = torch.from_numpy(a.copy()).cuda()
        _chain(torch, h, x, b, 7, call, d, e, sg)
        r += [x.cpu().numpy(), d.cpu().numpy(), e.cpu().numpy(), sg.cpu().numpy()]
        res[call] = r
    assert all(_same(p, q) for p, q in zip(res["mn"], res["sq"]))


# ------------------------------------------------------------------ 2./3. tall stage 1 vs reference, stage 2 vs oracle --------
@pytest.mark.parametrize("count,m,n,b", TALL)
@pytest.mark.parametrize("suf", ["f32", "f64"])
def test_tall_stages(torch, handles, rectref, oracle, count, m, n, b, suf):
    a = _batch(count, m, n, suf)
    bands, red, d, e, _ = _stages(torch, handles[suf], a, b, suf)
    for i in (0, count // 2, count - 1):
        top = bands[i, :n]
        assert np.all(bands[i, n:] == 0) and np.all(np.tril(top, -1) == 0)
        assert band_rel(top, rectref(a[i], b)[:n], b) <= TOL[suf]
        ref, dr, er = oracle.brd_p2(top, b)
        assert _same(red[i, :n], ref)
        assert np.all(red[i, n:] == 0)
        assert _same(d[i], dr) and _same(e[i, : n - 1], er)


# ------------------------------------------------------------------ 4. wide = transpose of tall --------------------------------
@pytest.mark.parametrize("count,m,n,b", TALL)
@pytest.mark.parametrize("suf", ["f32", "f64"])
def test_wide_is_transpose_of_tall(torch, handles, count, m, n, b, suf):
    h = handles[suf]
    a = _batch(count, m, n, suf)
    at = np.ascontiguousarray(a.transpose(0, 2, 1))
    tall = _stages(torch, h, a, b, suf)
    wide = _stages(torch, h, at, b, suf)
    for x_t, x_w in zip(tall[:2], wide[:2]):
        assert _same(x_w, np.ascontiguousarray(x_t.transpose(0, 2, 1)))
    assert np.all(wide[0][:, :, n:] == 0) and np.all(np.triu(wide[0][:, :, :n], 1) == 0)
    for x_t, x_w in zip(tall[2:], wide[2:]):
        assert _same(x_w, x_t)


# ------------------------------------------------------------------ 5. sigma against LAPACK ------------------------------------
@pytest.mark.parametrize("count,m,n,b,suf", [(16, 300, 128, 32, "f64"), (16, 128, 300, 32, "f64"), (8, 1000, 256, 64, "f32"),
                                             (8, 256, 1000, 64, "f32"), (6, 2048, 64, 16, "f64"), (6, 64, 2048, 16, "f32")])
def test_svdvals_vs_lapack(handles, count, m, n, b, suf):
    a = _batch(count, m, n, suf)
    with settings(handles[suf]) as h:
        s = h.svdvals_batched_mn(a, b).astype(np.float64)
    s0 = np.linalg.svd(a.astype(np.float64), compute_uv=False)
    assert s.shape == (count, min(m, n))
    assert np.all(np.diff(s, axis=1) <= 0)
    assert np.all(np.abs(s - s0).max(axis=1) <= SIG[suf] * s0[:, 0])


# ------------------------------------------------------------------ 6. independence from neighbours ---------------------------
@pytest.mark.parametrize("m,n,b,suf", [(257, 128, 32, "f64"), (96, 320, 32, "f32")])
def test_independent_of_neighbours(handles, m, n, b, suf):
    with settings(handles[suf]) as h:
        a7 = _batch(7, m, n, suf, seed=1)
        s7, out7 = _host(h, "svdvals_batched_mn", a7, m, n, b)
        other = _batch(2, m, n, suf, seed=2)
        for p in (0, 3, 6):
            a3 = np.stack([other[0], a7[p], other[1]])
            s3, out3 = _host(h, "svdvals_batched_mn", a3, m, n, b)
            assert _same(s3[1], s7[p]) and _same(out3[1], out7[p])


# ------------------------------------------------------------------ 7. chunk boundary ------------------------------------------
def test_chunk_boundary(torch, handles):
    count, m, n, b = 8195, 64, 32, 16
    x = torch.empty(count, m, n, dtype=torch.float64, device="cuda")
    sg = torch.zeros(count, n, dtype=torch.float64, device="cuda")
    with settings(handles["f64"]) as h:
        h.fill_uniform_dev(x.data_ptr(), count * m * n, 4242, 0.0, 5.0)
        h.synchronize()
        a = x.cpu().numpy()
        h.svdvals_batched_mn_dev(x.data_ptr(), count, m, n, b, sg.data_ptr())
        h.synchronize()
        s = sg.cpu().numpy()
        out = x.cpu().numpy()
        tail = torch.from_numpy(a[-3:].copy()).cuda()
        sg3 = torch.zeros(3, n, dtype=torch.float64, device="cuda")
        h.svdvals_batched_mn_dev(tail.data_ptr(), 3, m, n, b, sg3.data_ptr())
        h.synchronize()
    for i in (0, 8190, 8191, 8192, 8193, count - 1):
        s0 = np.linalg.svd(a[i], compute_uv=False)
        assert np.abs(s[i] - s0).max() <= SIG["f64"] * s0[0]
    assert _same(sg3.cpu().numpy(), s[-3:]) and _same(tail.cpu().numpy(), out[-3:])


# ------------------------------------------------------------------ 8. one launch sequence per batch ----------------------------
@pytest.mark.parametrize("m,n", [(300, 64), (64, 300)])
def test_launches_do_not_grow_with_count(torch, handles, m, n):
    h = handles["f64"]
    b = 16
    grew = []
    for count in (2, 64):
        x = torch.from_numpy(_batch(count, m, n, "f64")).cuda()
        sg = torch.zeros(count, min(m, n), dtype=torch.float64, device="cuda")
        before = h.launch_count()
        h.svdvals_batched_mn_dev(x.data_ptr(), count, m, n, b, sg.data_ptr())
        h.synchronize()
        grew.append(h.launch_count() - before)
    assert grew[0] == grew[1] and grew[0] > 0


# ------------------------------------------------------------------ 9. outside the kernels' range ------------------------------
@pytest.mark.parametrize("count,m,n,b,suf", [(2, 4096, 512, 64, "f64"), (2, 1280, 1152, 64, "f32")])
def test_fallback_is_the_single_chain(torch, handles, count, m, n, b, suf):
    h = handles[suf]
    a = _batch(count, m, n, suf)
    k = min(m, n)
    tdt = _tdt(torch, suf)
    per_setting = []
    for schedule, method in ((1, 0), (1, 2)):
        with settings(h, schedule, method):
            x = torch.from_numpy(a.copy()).cuda()
            sg = torch.zeros(count, k, dtype=tdt, device="cuda")
            h.svdvals_batched_mn_dev(x.data_ptr(), count, m, n, b, sg.data_ptr())
            h.synchronize()
            for i in range(count):
                xi = torch.from_numpy(a[i].copy()).cuda()
                si = torch.zeros(k, dtype=tdt, device="cuda")
                h.svdvals_mn_dev(xi.data_ptr(), m, n, b, si.data_ptr())
                h.synchronize()
                assert _same(sg[i].cpu().numpy(), si.cpu().numpy()) and _same(x[i].cpu().numpy(), xi.cpu().numpy())
            per_setting.append(sg.cpu().numpy())
    s0 = np.linalg.svd(a[0].astype(np.float64), compute_uv=False)
    for s in per_setting:
        assert np.abs(s[0].astype(np.float64) - s0).max() <= SIG[suf] * s0[0]
    x = torch.from_numpy(a.copy()).cuda()
    sg = torch.zeros(count, k, dtype=tdt, device="cuda")
    with pytest.raises(Exception) as ei:
        h.chain_batched_mn_dev(x.data_ptr(), count, m, n, b, 7, sigma_ptr=sg.data_ptr())
    assert ei.value.status == -3
    h.synchronize()
    assert _same(x.cpu().numpy(), a)


# ------------------------------------------------------------------ 10. host and device variants -------------------------------
@pytest.mark.parametrize("count,m,n,b", [(5, 640, 320, 32), (5, 320, 640, 32)])
@pytest.mark.parametrize("suf", ["f32", "f64"])
def test_host_equals_device(torch, handles, count, m, n, b, suf):
    a = _batch(count, m, n, suf)
    with settings(handles[suf]) as h:
        s, out = _host(h, "svdvals_batched_mn", a, m, n, b)
        t = h.last_timings()
        x = torch.from_numpy(a.copy()).cuda()
        sg = torch.zeros(count, min(m, n), dtype=_tdt(torch, suf), device="cuda")
        h.svdvals_batched_mn_dev(x.data_ptr(), count, m, n, b, sg.data_ptr())
        h.synchronize()
    assert _same(sg.cpu().numpy(), s) and _same(x.cpu().numpy(), out)
    assert t["h2d_ms"] > 0 and t["d2h_ms"] > 0
    assert t["stage1_ms"] == 0 and t["stage2_ms"] == 0 and t["qr_ms"] == 0


# ------------------------------------------------------------------ 11. statuses ------------------------------------------------
def test_statuses(capi, torch):
    lib = capi.lib()
    with capi.Handle(256, 32, np.float64) as h:
        def st(name, m, n, band, count=2, a=True, dtype=np.float64, sigma=True, what=7):
            """every call here fails its checks (or has count 0) before it touches a pointer, so host buffers do for all"""
            x = np.zeros(max(count * m * n, 1), dtype)
            o = np.zeros(3 * max(count, 1) * 512, dtype)
            p = x.ctypes.data_as(ctypes.c_void_p) if a else None
            d, e, s = (o[i * count * 512:].ctypes.data_as(ctypes.c_void_p) for i in range(3))
            f = getattr(lib, f"svdb200_{name}_{'f32' if dtype == np.float32 else 'f64'}")
            if name.startswith("chain"):
                return f(h.h, p, Z(count), Z(m), Z(n), Z(band), ctypes.c_int(what), d, e, s if sigma else None)
            return f(h.h, p, Z(count), Z(m), Z(n), Z(band), s if sigma else None)
        for name in ("svdvals_batched_mn", "svdvals_batched_mn_dev", "chain_batched_mn_dev"):
            assert st(name, 64, 32, 8, a=False) == -1
            assert st(name, 64, 32, 8, dtype=np.float32) == -1              # dtype of the handle is f64
            assert st(name, 64, 32, 8, sigma=False) == -1
            assert st(name, 64, 1, 1) == -2                                 # min(m, n) < 2
            assert st(name, 64, 32, 0) == -2
            assert st(name, 64, 30, 8) == -2                                # band does not divide min(m, n)
            assert st(name, 30, 64, 8) == -2
            assert st(name, 512, 32, 8) == -3                               # max(m, n) > max_n
            assert st(name, 32, 512, 8) == -3
            assert st(name, 128, 64, 64) == -3                              # band > the handle's band
            assert st(name, 64, 32, 8, count=0) == 0
        for what in (0, 8, -1):
            assert st("chain_batched_mn_dev", 64, 32, 8, what=what) == -1
        assert lib.svdb200_svdvals_batched_mn_f64(None, None, Z(1), Z(64), Z(32), Z(8), None) == -1
        # the longer side is arbitrary; sigma is needed for bit 4 only
        assert st("svdvals_batched_mn", 100, 64, 8) == 0 and st("svdvals_batched_mn", 64, 100, 8) == 0
        x = torch.zeros(2, 100, 64, dtype=torch.float64, device="cuda")
        h.chain_batched_mn_dev(x.data_ptr(), 2, 100, 64, 8, 3)
        h.synchronize()
