"""Host-pointer calls against their _dev twins (square dense_to_band / band_to_bidiag / bidiagonalize / svdvals, bidiag_qr,
bidiagonalize_onestage).

A host call copies its inputs in, runs the same device chain as its _dev twin, copies the results out and synchronises.
So its results are byte-equal to the twin's, it issues the same kernel launches, and svdb200_last_timings reports h2d, d2h
and the stages it ran (> 0) and exactly 0 for the stages it did not run.  A stage that fails after the input copy has been
enqueued leaves the handle usable."""
import ctypes

import numpy as np
import pytest

from svdsolver_b200.synth import uniform_matrix

pytestmark = pytest.mark.gpu

DT = {"f32": np.float32, "f64": np.float64}
N, B = 192, 32
STAGES = {"dense_to_band": {"stage1_ms"}, "band_to_bidiag": {"stage2_ms"}, "bidiagonalize": {"stage1_ms", "stage2_ms"},
          "svdvals": {"stage1_ms", "stage2_ms", "qr_ms"}, "bidiag_qr": {"qr_ms"}, "bidiagonalize_onestage": {"stage1_ms"}}
CASES = [(name, order) for name in ("dense_to_band", "bidiagonalize", "svdvals") for order in (0, 1)] + \
        [("band_to_bidiag", 0), ("bidiag_qr", 0), ("bidiagonalize_onestage", 0)]


@pytest.fixture(scope="module")
def capi():
    from svdsolver_b200 import capi as m
    m.lib()
    return m


@pytest.fixture(scope="module")
def handles(capi):
    hs = {s: capi.Handle(N, B, dt) for s, dt in DT.items()}
    for h in hs.values():
        h.set_stage2_schedule(1)          # sigma of a generic matrix needs the complete chase
    yield hs
    for h in hs.values():
        h.close()


def _same(x, y):
    x, y = np.asarray(x), np.asarray(y)
    return x.shape == y.shape and np.array_equal(x.view(np.uint8), y.view(np.uint8))


def _counted(h, fn):
    before = h.launch_count()
    out = fn()
    return out, h.launch_count() - before


def _host(capi, h, name, order, x):
    """the host call: (outputs, launches, timings)"""
    calls = {
        "dense_to_band": lambda: (h.dense_to_band(x, B, order),),
        "band_to_bidiag": lambda: h.band_to_bidiag(x, B),
        "bidiagonalize": lambda: h.bidiagonalize(x, B, order),
        "svdvals": lambda: h.svdvals(x, B, order)[::-1],                 # (A_out, sigma)
        "bidiag_qr": lambda: (h.bidiag_qr(*x)[0],),
        "bidiagonalize_onestage": lambda: h.bidiagonalize_onestage(x),
    }
    out, launches = _counted(h, calls[name])
    return out, launches, h.last_timings()


def _dev(capi, h, name, order, x, torch):
    """the _dev twin on device copies of the same input: (outputs, launches)"""
    tdt = torch.float32 if h.dtype == np.float32 else torch.float64

    def vec(k):
        return torch.zeros(k, dtype=tdt, device="cuda")
    if name == "bidiag_qr":
        d, e = (torch.from_numpy(np.ascontiguousarray(v).copy()).cuda() for v in x)
        s = vec(N)
        torch.cuda.synchronize()
        _, launches = _counted(h, lambda: h.bidiag_qr_dev(d.data_ptr(), e.data_ptr(), N, s.data_ptr()))
        h.synchronize()
        return (s.cpu().numpy(),), launches
    a = torch.from_numpy(x.copy()).cuda()
    d, e, s = vec(N), vec(N - 1), vec(N)
    torch.cuda.synchronize()
    calls = {
        "dense_to_band": lambda: h.dense_to_band_dev(a.data_ptr(), N, B, order),
        "band_to_bidiag": lambda: h.band_to_bidiag_dev(a.data_ptr(), N, B, d.data_ptr(), e.data_ptr()),
        "bidiagonalize": lambda: h.bidiagonalize_dev(a.data_ptr(), N, B, d.data_ptr(), e.data_ptr(), order),
        "svdvals": lambda: h.svdvals_dev(a.data_ptr(), N, B, s.data_ptr(), order),
        "bidiagonalize_onestage": lambda: h._check(h._fn("bidiagonalize_onestage_dev")(
            h.h, ctypes.c_void_p(a.data_ptr()), ctypes.c_size_t(N), ctypes.c_size_t(N), ctypes.c_void_p(d.data_ptr()),
            ctypes.c_void_p(e.data_ptr()))),
    }
    _, launches = _counted(h, calls[name])
    h.synchronize()
    outs = {"dense_to_band": (a,), "band_to_bidiag": (a, d, e), "bidiagonalize": (a, d, e), "svdvals": (a, s),
            "bidiagonalize_onestage": (a, d, e)}[name]
    return tuple(t.cpu().numpy() for t in outs), launches


@pytest.mark.parametrize("name,order", CASES)
@pytest.mark.parametrize("suf", ["f32", "f64"])
def test_host_equals_dev(capi, handles, name, order, suf):
    import torch
    h = handles[suf]
    a = uniform_matrix(N, N, 586 + N + order, 0.0, 5.0, DT[suf])
    x = a
    if name == "band_to_bidiag":
        x = h.dense_to_band(a, B)
    elif name == "bidiag_qr":
        x = h.bidiagonalize(a, B)[1:]
    out, launches, t = _host(capi, h, name, order, x)
    out_dev, launches_dev = _dev(capi, h, name, order, x, torch)
    assert all(_same(u, v) for u, v in zip(out, out_dev)) and len(out) == len(out_dev)
    assert launches == launches_dev > 0
    assert t["h2d_ms"] > 0 and t["d2h_ms"] > 0
    for k in ("stage1_ms", "stage2_ms", "qr_ms"):
        assert (t[k] > 0) if k in STAGES[name] else (t[k] == 0), (k, t)


def test_error_after_staging(capi):
    """band 96 passes the argument checks of a band-128 handle, so the input copy is enqueued; stage 2 then refuses the
    band (stage2_threads(96) > 1024).  The handle's next call computes what a fresh handle computes."""
    n = 192
    a = uniform_matrix(n, n, 586 + n, 0.0, 5.0, np.float64)
    with capi.Handle(n, 128, np.float64) as h:
        h.set_stage2_schedule(1)
        with pytest.raises(capi.SvdB200Error) as ei:
            h.band_to_bidiag(a, 96)
        assert ei.value.status == -3
        s, out = h.svdvals(a, 32)
    with capi.Handle(n, 128, np.float64) as f:
        f.set_stage2_schedule(1)
        s0, out0 = f.svdvals(a, 32)
    assert _same(s, s0) and _same(out, out0)
