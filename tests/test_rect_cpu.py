"""CPU reference for stage 1 of tall m x n matrices (tests/rect_reference.c): the panel-order reduction with trailing rows
m - k.  Checks the reference itself: at m == n it is the oracle's svdo_brd_p1_panel byte for byte, and for m > n its
output is an upper band matrix in the top n x n block with the singular values of A.  Like the oracle, it forms R as
A - V Y, so the entries below the diagonal and below row n are round-off, not the exact zeros the GPU writes."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from svdsolver_b200.synth import uniform_matrix


@pytest.fixture(scope="module")
def rectref(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("rectref") / "librectref.so")
    subprocess.check_call(["gcc", "-std=c11", "-O2", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared",
                           "-I", os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests", "rect_reference.c"), "-o", out, "-lm"])
    return ctypes.CDLL(out)


def reduce_tall(lib, a, b):
    x = np.ascontiguousarray(a).copy()
    suf = "f32" if x.dtype == np.float32 else "f64"
    rc = getattr(lib, f"rect_brd_p1_panel_mn_{suf}")(x.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(x.shape[0]),
                                                      ctypes.c_size_t(x.shape[1]), ctypes.c_size_t(b))
    assert rc == 0
    return x


@pytest.mark.parametrize("n,b", [(64, 4), (96, 32), (256, 32)])
@pytest.mark.parametrize("dt", [np.float32, np.float64])
def test_square_is_the_oracle_panel_order(rectref, oracle, n, b, dt):
    a = uniform_matrix(n, n, 586 + n + b, 0.0, 5.0, dt)
    assert np.array_equal(reduce_tall(rectref, a, b).view(np.uint8), oracle.brd_p1_panel(a, b).view(np.uint8))


@pytest.mark.parametrize("m,n,b", [(70, 64, 4), (100, 64, 8), (257, 128, 32), (512, 64, 16), (1000, 96, 32)])
def test_tall_reduction(rectref, m, n, b):
    a = uniform_matrix(m, n, 586 + m + n + b, 0.0, 5.0, np.float64)
    out = reduce_tall(rectref, a, b)
    top = out[:n]
    big = np.abs(out).max()
    assert np.abs(out[n:]).max() <= 1e-12 * big
    assert np.abs(np.tril(top, -1)).max() <= 1e-12 * big
    assert np.abs(np.triu(top, b + 1)).max() <= 1e-12 * big
    s0 = np.linalg.svd(a, compute_uv=False)
    s1 = np.linalg.svd(np.triu(top, 0) - np.triu(top, b + 1), compute_uv=False)
    assert np.abs(s0 - s1).max() <= 1e-12 * s0[0]


def test_rejects_wide_and_ragged(rectref):
    f = rectref.rect_brd_p1_panel_mn_f64
    x = np.zeros(64 * 64)
    p = x.ctypes.data_as(ctypes.c_void_p)
    assert f(p, ctypes.c_size_t(32), ctypes.c_size_t(64), ctypes.c_size_t(4)) == -1      # m < n
    assert f(p, ctypes.c_size_t(64), ctypes.c_size_t(30), ctypes.c_size_t(4)) == -1      # band does not divide n
