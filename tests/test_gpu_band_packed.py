"""Stage 2 and singular values from band storage (svdb200_band_to_bidiag_packed_* / svdb200_band_svdvals_packed_*).

The packed path runs the same kernels as the dense one with another element addressing, so the bidiagonal it returns
must be byte-equal to svdb200_band_to_bidiag_dev_* on the dense embedding of the same band, at every size, band and
schedule, through the band-32 kernel (n >= 2b+2), its edge sizes and the generic kernel."""
import ctypes

import numpy as np
import pytest

from svdsolver_b200.capi import pack_upper_band
from svdsolver_b200.synth import uniform_matrix

pytestmark = pytest.mark.gpu

DT = {"f32": np.float32, "f64": np.float64}
MAX_N, MAX_B = 16384, 64


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


def _same(x, y):
    return x.shape == y.shape and np.array_equal(x.view(np.uint8), y.view(np.uint8))


def _ab_uniform(n, b, seed, dt):
    """seeded U[0,5) upper band in band storage (zero above the matrix)"""
    ab = uniform_matrix(n, b + 1, seed, 0.0, 5.0, dt)
    for t in range(b):
        ab[: b - t, t] = 0
    return ab


def _dense_dev(ab_t, n, b):
    """dense n x n device embedding of the band in storage ab_t (zero elsewhere)"""
    import torch
    a = torch.zeros(n, n, dtype=ab_t.dtype, device="cuda")
    for t in range(b + 1):
        k = b - t
        if k < n:
            i = torch.arange(n - k, device="cuda")
            a[i, i + k] = ab_t[k:, t]
    return a


def _dense_and_packed(h, ab, b):
    """(d, e) of the dense path on the embedding, (d, e) of the packed path; checks that ab is left as it was"""
    import torch
    n = ab.shape[0]
    ab_t = torch.from_numpy(ab).cuda()
    ab_copy = ab_t.clone()
    a = _dense_dev(ab_t, n, b)
    out = [torch.full((n,), -1.0, dtype=ab_t.dtype, device="cuda") for _ in range(4)]
    h.band_to_bidiag_dev(a.data_ptr(), n, b, out[0].data_ptr(), out[1].data_ptr())
    h.band_to_bidiag_packed_dev(ab_t.data_ptr(), n, b, out[2].data_ptr(), out[3].data_ptr())
    h.synchronize()
    assert torch.equal(ab_t, ab_copy), "input band storage was modified"
    d0, e0, d1, e1 = (x.cpu().numpy() for x in out)
    return (d0, e0[: n - 1]), (d1, e1[: n - 1])


@pytest.mark.parametrize("complete", [0, 1])
@pytest.mark.parametrize("suf", ["f32", "f64"])
@pytest.mark.parametrize("n", [2, 3, 5, 64, 65, 66, 67, 97, 129, 320, 321, 1000, 3840])
def test_packed_stage2_byte_equal_to_dense(handles, n, suf, complete):
    h = handles[suf]
    h.set_stage2_schedule(complete)
    for b in (1, 4, 7, 16, 32, 64):
        if b >= n:
            continue
        (d0, e0), (d1, e1) = _dense_and_packed(h, _ab_uniform(n, b, 1000 * n + b, DT[suf]), b)
        assert _same(d1, d0) and _same(e1, e0), (n, b)


@pytest.mark.parametrize("suf", ["f32", "f64"])
@pytest.mark.parametrize("b", [32, 64])
def test_packed_stage2_byte_equal_large(handles, suf, b):
    """n = 16384: the sweep pipeline is capped by the SM slots, not by n / 2b"""
    h = handles[suf]
    for complete in (0, 1):
        h.set_stage2_schedule(complete)
        (d0, e0), (d1, e1) = _dense_and_packed(h, _ab_uniform(16384, b, 77 + b, DT[suf]), b)
        assert _same(d1, d0) and _same(e1, e0), complete


@pytest.mark.parametrize("suf", ["f32", "f64"])
@pytest.mark.parametrize("b", [32, 64])
def test_packed_stage2_on_a_stage1_band(handles, suf, b):
    """the band stage 1 leaves (signed, no structure beyond the band), n = 1920"""
    import torch
    n = 1920
    h = handles[suf]
    a = torch.from_numpy(uniform_matrix(n, n, 586 + n, 0.0, 5.0, DT[suf])).cuda()
    h.dense_to_band_dev(a.data_ptr(), n, b)
    h.synchronize()
    ab = pack_upper_band(a.cpu().numpy(), b)
    for complete in (0, 1):
        h.set_stage2_schedule(complete)
        (d0, e0), (d1, e1) = _dense_and_packed(h, ab, b)
        assert _same(d1, d0) and _same(e1, e0), complete


@pytest.mark.parametrize("b", [7, 32])
@pytest.mark.parametrize("n", [1000, 3000])
def test_packed_svdvals(handles, n, b):
    """sigma byte-equal to stage 2 + bidiag_qr on the dense embedding (the zero-shift QR at n = 1000, bisection at
    n = 3000); with the complete schedule within 1e-10 sigma_1 of LAPACK in double"""
    import torch
    h = handles["f64"]
    ab = _ab_uniform(n, b, 31 * n + b, np.float64)
    ab_t = torch.from_numpy(ab).cuda()
    s_lapack = None
    for complete in (0, 1):
        h.set_stage2_schedule(complete)
        a = _dense_dev(ab_t, n, b)
        d, e, s0 = (torch.zeros(n, dtype=torch.float64, device="cuda") for _ in range(3))
        h.band_to_bidiag_dev(a.data_ptr(), n, b, d.data_ptr(), e.data_ptr())
        h.bidiag_qr_dev(d.data_ptr(), e.data_ptr(), n, s0.data_ptr())
        h.synchronize()
        s0 = s0.cpu().numpy()
        s1 = h.band_svdvals_packed(ab, b)
        assert _same(s1, s0), complete
        if complete:
            s_lapack = np.linalg.svd(a.cpu().numpy(), compute_uv=False)
            assert np.abs(s1 - s_lapack).max() <= 1e-10 * s_lapack[0]
    h.set_stage2_schedule(0)


def test_packed_large_n_without_dense_storage(capi):
    """n = 65536, band 32, double, complete schedule: (d, e) keeps the Frobenius norm of the band and the three largest
    singular values match ARPACK on the sparse band.  Nothing here is n x n."""
    import scipy.sparse as sp
    import scipy.sparse.linalg as sla
    import torch
    n, b = 65536, 32
    ab = _ab_uniform(n, b, 9001, np.float64)
    ab_t = torch.from_numpy(ab).cuda()
    d, e, sig = (torch.zeros(n, dtype=torch.float64, device="cuda") for _ in range(3))
    with capi.Handle(n, b, np.float64) as h:
        h.set_stage2_schedule(1)
        h.band_to_bidiag_packed_dev(ab_t.data_ptr(), n, b, d.data_ptr(), e.data_ptr())
        h.band_svdvals_packed_dev(ab_t.data_ptr(), n, b, sig.data_ptr())
        h.synchronize()
    d, e, sig = d.cpu().numpy(), e.cpu().numpy()[: n - 1], sig.cpu().numpy()
    fro_band = np.linalg.norm(ab)
    fro_bid = np.sqrt(np.dot(d, d) + np.dot(e, e))
    assert abs(fro_bid / fro_band - 1) <= 1e-12
    cols = np.repeat(np.arange(n), b + 1)
    rows = cols - b + np.tile(np.arange(b + 1), n)
    m = rows >= 0
    A = sp.csr_matrix((ab.ravel()[m], (rows[m], cols[m])), shape=(n, n))
    top = np.sort(sla.svds(A, k=3, return_singular_vectors=False, tol=0, random_state=0))[::-1]
    assert np.all(np.abs(sig[:3] - top) <= 1e-9 * top)


@pytest.mark.parametrize("suf", ["f32", "f64"])
def test_packed_host_variants_and_errors(capi, suf):
    """host-pointer variants equal the _dev variants and leave ab unchanged; the shape / capacity / argument statuses"""
    import torch
    dt = DT[suf]
    n, b = 200, 16
    ab = _ab_uniform(n, b, 4242, dt)
    keep = ab.copy()
    with capi.Handle(256, 32, dt) as h:
        h.set_stage2_schedule(1)
        d, e = h.band_to_bidiag_packed(ab, b)
        sigma = h.band_svdvals_packed(ab, b)
        assert _same(ab, keep)
        ab_t = torch.from_numpy(ab).cuda()
        dd, ed, sd = (torch.zeros(n, dtype=ab_t.dtype, device="cuda") for _ in range(3))
        h.band_to_bidiag_packed_dev(ab_t.data_ptr(), n, b, dd.data_ptr(), ed.data_ptr())
        h.band_svdvals_packed_dev(ab_t.data_ptr(), n, b, sd.data_ptr())
        h.synchronize()
        assert _same(d, dd.cpu().numpy()) and _same(e, ed.cpu().numpy()[: n - 1]) and _same(sigma, sd.cpu().numpy())
        assert torch.equal(ab_t.cpu(), torch.from_numpy(keep))

        lib = capi.lib()
        Z = ctypes.c_size_t
        P = ctypes.c_void_p
        abp, dp, ep, sp_ = P(ab_t.data_ptr()), P(dd.data_ptr()), P(ed.data_ptr()), P(sd.data_ptr())
        s2 = getattr(lib, f"svdb200_band_to_bidiag_packed_dev_{suf}")
        sv = getattr(lib, f"svdb200_band_svdvals_packed_dev_{suf}")
        s2h = getattr(lib, f"svdb200_band_to_bidiag_packed_{suf}")
        svh = getattr(lib, f"svdb200_band_svdvals_packed_{suf}")
        E_ARG, E_SHAPE, E_CAP = -1, -2, -3
        assert s2(h.h, abp, Z(1), Z(b), dp, ep) == E_SHAPE
        assert sv(h.h, abp, Z(1), Z(b), sp_) == E_SHAPE
        assert s2(h.h, abp, Z(n), Z(0), dp, ep) == E_CAP
        assert s2(h.h, abp, Z(n), Z(33), dp, ep) == E_CAP           # band > the handle's band
        assert sv(h.h, abp, Z(257), Z(b), sp_) == E_CAP             # n > max_n
        assert s2(h.h, None, Z(n), Z(b), dp, ep) == E_ARG
        assert sv(h.h, None, Z(n), Z(b), sp_) == E_ARG
        assert sv(h.h, abp, Z(n), Z(b), None) == E_ARG
        assert s2h(h.h, None, Z(n), Z(b), None, None) == E_ARG
        assert svh(h.h, ab.ctypes.data_as(P), Z(n), Z(b), None) == E_ARG
        assert s2(None, abp, Z(n), Z(b), dp, ep) == E_ARG
        h.synchronize()


def test_dist_svdvals_hands_the_packed_band_to_stage2(capi):
    """One rank: sigma of dist_svdvals_dev equals band_svdvals_packed_dev on the band it leaves behind, byte for byte"""
    import torch
    from svdsolver_b200 import distributed as D
    n, b = 2048, 32
    loc = torch.from_numpy(uniform_matrix(n, n, 586 + n, 0.0, 5.0, np.float64)).cuda()
    sigma = torch.zeros(n, dtype=torch.float64, device="cuda")
    packed = torch.zeros(n, b + 1, dtype=torch.float64, device="cuda")
    with D.DistHandle(n, b, np.float64, 0, 1, (ctypes.c_ubyte * 128)()) as dh:
        dh.svdvals_dev(loc.data_ptr(), sigma.data_ptr())
        dh.gather_band_dev(loc.data_ptr(), packed.data_ptr())
        torch.cuda.synchronize()
    s2 = torch.zeros(n, dtype=torch.float64, device="cuda")
    with capi.Handle(n, b, np.float64) as h:
        h.band_svdvals_packed_dev(packed.data_ptr(), n, b, s2.data_ptr())
        h.synchronize()
    assert _same(s2.cpu().numpy(), sigma.cpu().numpy())
