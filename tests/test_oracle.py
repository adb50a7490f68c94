"""CPU tests (-m "not gpu"): the oracle against every golden vector the reference holds for the
path (data/band_*, data/bidiagonal_* at 64/512, band 4 -- SURVEY 8c), the regenerated 1024 cases
(digests produced by the compiled reference in the build container), seeded random cases at other
band sizes, the float QR diagonalisation and Householder known answers."""
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, load_fixture
from svdsolver_b200.synth import uniform_matrix

DT = {"f32": np.float32, "f64": np.float64}
NAME = {"f32": "float", "f64": "double"}


@pytest.mark.parametrize("n", [64, 512])
@pytest.mark.parametrize("suf", ["f32", "f64"])
def test_fixture_chain_bit_exact(oracle, n, suf):
    a = load_fixture("test", NAME[suf], n)
    band = oracle.brd_p1(a, 4)
    assert np.array_equal(band.view(np.uint8), load_fixture("band", NAME[suf], n).view(np.uint8))
    bid, d, e = oracle.brd_p2(band, 4)
    ref = load_fixture("bidiagonal", NAME[suf], n)
    assert np.array_equal(bid.view(np.uint8), ref.view(np.uint8))
    assert np.array_equal(d, np.diagonal(ref)) and np.array_equal(e, np.diagonal(ref, 1))


@pytest.mark.parametrize("n", [64, 512])
@pytest.mark.parametrize("suf", ["f32", "f64"])
def test_fixture_stage2_in_isolation(oracle, n, suf):
    bid, _, _ = oracle.brd_p2(load_fixture("band", NAME[suf], n), 4)
    assert np.array_equal(bid.view(np.uint8), load_fixture("bidiagonal", NAME[suf], n).view(np.uint8))


@pytest.mark.parametrize("suf", ["f32", "f64"])
def test_regenerated_1024(oracle, suf):
    meta = json.load(open(os.path.join(GOLDEN, "golden_meta.json")))[f"1024_{suf}"]
    g = np.load(os.path.join(GOLDEN, "golden_1024.npz"))
    sha = lambda x: hashlib.sha256(np.ascontiguousarray(x).tobytes()).hexdigest()
    a = uniform_matrix(1024, 1024, 586 + 1024, 1.0, 5.0, DT[suf])
    assert sha(a) == meta["input_sha256"]
    band = oracle.brd_p1(a, 4)
    assert sha(band) == meta["band_sha256"]
    for k in range(5):
        assert np.array_equal(np.diagonal(band, k), g[f"band_diags_{suf}"][k][: 1024 - k])
    bid, d, e = oracle.brd_p2(band, 4)
    assert sha(bid) == meta["bidiagonal_sha256"]
    assert np.array_equal(d, g[f"bidiag_d_{suf}"]) and np.array_equal(e, g[f"bidiag_e_{suf}"])


@pytest.mark.parametrize("n,b", [(96, 32), (128, 16), (64, 8), (192, 32), (256, 64), (40, 4), (32, 32)])
@pytest.mark.parametrize("suf", ["f32", "f64"])
def test_random_cases_vs_reference_outputs(oracle, n, b, suf):
    g = np.load(os.path.join(GOLDEN, "golden_random.npz"))
    a = uniform_matrix(n, n, 586 + n + b, 0.0, 5.0, DT[suf])
    band = oracle.brd_p1(a, b)
    assert np.array_equal(band, g[f"band_{n}_{b}_{suf}"])
    bid, _, _ = oracle.brd_p2(band, b)
    assert np.array_equal(bid, g[f"bidiag_{n}_{b}_{suf}"])


@pytest.mark.parametrize("n,b", [(64, 4), (96, 32), (128, 16), (256, 32)])
def test_panel_order_vs_reference_gpu_twin(oracle, n, b):
    g = np.load(os.path.join(GOLDEN, "golden_panel.npz"))
    a = uniform_matrix(n, n, 586 + n + b, 0.0, 5.0, np.float32)
    assert np.array_equal(oracle.brd_p1_panel(a, b), g[f"panel_band_{n}_{b}_f32"])


def test_panel_and_tile_orders_agree_up_to_signs(oracle):
    # SURVEY 8(a'): a full-height panel reduction matches the flat tree only modulo D1*B*D2.
    a = uniform_matrix(128, 128, 7, 0.0, 5.0, np.float64)
    t = oracle.brd_p1(a, 16)
    p = oracle.brd_p1_panel(a, 16)
    for k in range(17):
        np.testing.assert_allclose(np.abs(np.diagonal(t, k)), np.abs(np.diagonal(p, k)), rtol=0, atol=1e-11 * np.abs(t).max())
    assert not np.allclose(np.diagonal(t), np.diagonal(p))


@pytest.mark.parametrize("n", [8, 64, 320, 640])
def test_qrd_float_vs_reference(oracle, n):
    g = np.load(os.path.join(GOLDEN, "golden_qrd.npz"))
    de = uniform_matrix(2, n, 586 + n, 0.0, 5.0, np.float32)
    sig, _, sweeps, thr, max_iter = oracle.qrd(de[0], de[1, : n - 1])
    assert sweeps >= 0 and max_iter == ((500 * n) ^ 2)
    assert np.array_equal(sig, g[f"qrd_sigma_{n}"])


@pytest.mark.parametrize("n", [64, 512])
def test_qrd_float_on_fixture_bidiagonal(oracle, n):
    g = np.load(os.path.join(GOLDEN, "golden_qrd.npz"))
    m = load_fixture("bidiagonal", "float", n)
    sig, _, sweeps, _, _ = oracle.qrd(np.diagonal(m).copy(), np.diagonal(m, 1).copy())
    assert sweeps >= 0
    assert np.array_equal(sig, g[f"qrd_sigma_fixture_{n}"])
    # and it agrees with LAPACK on the same bidiagonal (BASELINE.md 2c: 4e-6*sigma_1)
    B = np.diag(np.diagonal(m).astype(np.float64)) + np.diag(np.diagonal(m, 1).astype(np.float64), 1)
    ref = np.linalg.svd(B, compute_uv=False)
    assert np.abs(sig - ref).max() <= 2e-5 * ref[0]


def test_qrd_double_vs_lapack(oracle):
    # parity UNPINNED by the reference (serial::qrd is float-only); cross-check with LAPACK.
    n = 200
    de = uniform_matrix(2, n, 99, 0.0, 5.0, np.float64)
    sig, _, sweeps, thr, _ = oracle.qrd(de[0], de[1, : n - 1])
    assert sweeps >= 0
    B = np.diag(de[0]) + np.diag(de[1, : n - 1], 1)
    ref = np.linalg.svd(B, compute_uv=False)
    assert np.abs(sig - ref).max() <= 50 * thr


@pytest.mark.parametrize("suf", ["f32", "f64"])
@pytest.mark.parametrize("ln", [1, 2, 5, 33])
def test_householder_known_answers(oracle, suf, ln):
    g = np.load(os.path.join(GOLDEN, "golden_householder.npz"))
    x = g[f"hh_x_{ln}_{suf}"]
    w, H, tau = oracle.householder(x)
    assert np.array_equal(w, g[f"hh_w_{ln}_{suf}"])
    assert np.array_equal(H.ravel(), g[f"hh_H_{ln}_{suf}"])
    assert tau == g[f"hh_tau_{ln}_{suf}"][0]
    # sign convention (SURVEY A2): H x = -sign(x0) ||x|| e1
    y = H.astype(np.float64) @ x.astype(np.float64)
    assert abs(y[0] + np.copysign(np.linalg.norm(x.astype(np.float64)), x[0])) <= 1e-5 * max(1.0, abs(y[0]))
    if ln == 1:
        assert tau == 2 and H[0, 0] == -1


@pytest.mark.parametrize("n,b", [(64, 4), (65, 4), (67, 4), (96, 32), (100, 7), (33, 32)])
def test_stage2_schedule_closed_form(oracle, n, b):
    """SURVEY 8(a''): the closed-form window list equals the reference recurrence."""
    from svdsolver_b200.schedule import stage2_windows
    ref = oracle.schedule(n, b)
    mine = np.array(list(stage2_windows(n, b)), dtype=np.int64).reshape(-1, 6)
    assert np.array_equal(ref, mine)


def test_band_structure_and_norm_preservation(oracle):
    a = uniform_matrix(96, 96, 3, 0.0, 5.0, np.float64)
    band = oracle.brd_p1(a, 8)
    below = np.tril(band, -1)
    above = np.triu(band, 9)
    assert np.abs(below).max() < 1e-12 * np.abs(band).max() and np.abs(above).max() < 1e-12 * np.abs(band).max()
    assert abs(np.linalg.norm(band) - np.linalg.norm(a)) < 1e-12 * np.linalg.norm(a)
    s0 = np.linalg.svd(a, compute_uv=False)
    s1 = np.linalg.svd(np.triu(np.tril(band, 8)), compute_uv=False)
    assert np.abs(s0 - s1).max() < 1e-12 * s0[0]


def test_compiled_reference_agrees_when_present(oracle, request):
    """The oracle == the compiled original reference, bit for bit: parallel::brd_p1<double>(A, 8), then parallel::brd_p2.
    Compared with the reference's stored outputs for this input (golden_refcheck.npz, tools/make_golden.py --only-refcheck)
    when they are in the tree, otherwise with the compiled reference itself (refso, which skips without it)."""
    import ctypes
    a = uniform_matrix(80, 80, 11, 0.0, 5.0, np.float64)
    stored = os.path.join(GOLDEN, "golden_refcheck.npz")
    if os.path.exists(stored):
        g = np.load(stored)
        ref_band, ref_bid = g["band_80_8_f64"], g["bidiag_80_8_f64"]
    else:
        refso = request.getfixturevalue("refso")
        r = a.copy()
        refso.svdref_brd_p1_f64(r.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(80), ctypes.c_size_t(8))
        ref_band = r.copy()
        refso.svdref_brd_p2_f64(r.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(80), ctypes.c_size_t(8), None, None)
        ref_bid = r
    assert np.array_equal(oracle.brd_p1(a, 8), ref_band)
    assert np.array_equal(oracle.brd_p2(oracle.brd_p1(a, 8), 8)[0], ref_bid)


@pytest.mark.parametrize("n,b", [(64, 4), (65, 4), (100, 7), (96, 32), (130, 16), (33, 32)])
def test_stage2_cross_sweep_dependency_lag(n, b):
    """The pipelining rule of csrc/stage2_chase.cu: with ops numbered RIGHT(p)=2p, LEFT(p)=2p+1, op q
    of sweep i+1 overlaps ops of sweep i only up to index q+3 (so it may start after q+4 ops)."""
    c, w = b, b + 1

    def ops(i):
        out = [(i, min(i + w, n), i + 1, min(i + w, n)), (i + 1, min(i + w, n), i + 1, min(i + 2 * w - 1, n))]
        for k in range((n - min(i + 2 * w - 1, n)) // c + 1):
            r0, r1, r2, c3 = (min(i + 1 + (k + j) * c, n) for j in range(4))
            out.append((r0, r2, r1, r2) if r2 > r1 else None)
            out.append((r1, r2, r1, c3) if c3 > r1 else None)
        return out

    def overlap(a, bb):
        return a and bb and a[0] < bb[1] and bb[0] < a[1] and a[2] < bb[3] and bb[2] < a[3]

    worst = 0
    for i in range(n - 2):
        A, B = ops(i), ops(i + 1)
        for q, ob in enumerate(B):
            for qa, oa in enumerate(A):
                if overlap(oa, ob):
                    worst = max(worst, qa - q)
    assert worst <= 3


@pytest.mark.parametrize("n,b", [(64, 4), (65, 4), (100, 7), (96, 32), (256, 32), (130, 16)])
def test_complete_chase_preserves_singular_values(oracle, n, b):
    """The reference's stage-2 schedule is not orthogonally equivalent to its input (SURVEY 0.3); the complete-chase
    variant of the oracle (checker of svdb200_set_stage2_schedule(1)) is: sigma(bidiagonal) == sigma(band)."""
    rng = np.random.default_rng(n + b)
    band = np.triu(np.tril(rng.random((n, n)) * 5, b))
    s0 = np.linalg.svd(band, compute_uv=False)
    _, d, e = oracle.brd_p2_complete(band, b)
    s1 = np.linalg.svd(np.diag(d) + np.diag(e, 1), compute_uv=False)
    assert np.abs(s1 - s0).max() <= 1e-13 * s0[0]
    _, dr, er = oracle.brd_p2(band, b)
    sr = np.linalg.svd(np.diag(dr) + np.diag(er, 1), compute_uv=False)
    assert np.abs(sr - s0).max() > 1e-6 * s0[0]      # the flaw this option exists for


@pytest.mark.parametrize("n,b", [(64, 4), (65, 4), (100, 7), (96, 32), (40, 4), (33, 32)])
def test_complete_schedule_dependency_lag(n, b):
    """the q+4 pipelining rule of the kernel also holds for the complete schedule (brute force over all window pairs)"""
    c, w = b, b + 1

    def ops(i):
        out = [(i, min(i + w, n), i + 1, min(i + w, n)), (i + 1, min(i + w, n), i + 1, min(i + 2 * w - 1, n))]
        k = 0
        while True:
            r0, r1, r2, c3 = (min(i + 1 + (k + j) * c, n) for j in range(4))
            if not r2 > r1:
                break
            out.append((r0, r2, r1, r2))
            out.append((r1, r2, r1, c3) if c3 > r1 else None)
            k += 1
        return out

    def overlap(a, bb):
        return a and bb and a[0] < bb[1] and bb[0] < a[1] and a[2] < bb[3] and bb[2] < a[3]

    worst = 0
    for i in range(n - 2):
        A, B = ops(i), ops(i + 1)
        for q, ob in enumerate(B):
            for qa, oa in enumerate(A):
                if overlap(oa, ob):
                    worst = max(worst, qa - q)
    assert worst <= 3


@pytest.mark.parametrize("suf,dt", [("f32", np.float32), ("f64", np.float64)])
@pytest.mark.parametrize("n", [8, 48, 96])
def test_onestage_brd_oracle_pinned_to_reference(oracle, suf, dt, n):
    """svdo_brd_serial (restatement of serial::brd, svd_serial.h:233-266) == the compiled reference, bit for bit
    (golden_onestage.npz, generated by tools/make_golden.py from oracle/_ref)."""
    import os
    from conftest import GOLDEN
    from svdsolver_b200.synth import uniform_matrix
    g = np.load(os.path.join(GOLDEN, "golden_onestage.npz"))
    a = uniform_matrix(n, n, 586 + n, 0.0, 5.0, dt)
    x, d, e = oracle.brd_serial(a)
    assert np.array_equal(x, g[f"brd_{n}_{suf}"]) and np.array_equal(d, g[f"brd_d_{n}_{suf}"]) and np.array_equal(e, g[f"brd_e_{n}_{suf}"])
    # an orthogonal reduction: singular values of the bidiagonal == singular values of the input
    s0 = np.linalg.svd(a.astype(np.float64), compute_uv=False)
    s1 = np.linalg.svd(np.diag(d.astype(np.float64)) + np.diag(e.astype(np.float64), 1), compute_uv=False)
    assert np.abs(s0 - s1).max() <= (1e-5 if suf == "f32" else 1e-13) * s0[0]
