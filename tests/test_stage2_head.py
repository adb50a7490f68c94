"""The sweep head of the band-32 stage-2 kernel (csrc/stage2_chase_fast.cu).

Sweep i reads RIGHT(0)'s Householder vector (row i, cols [i+1, i+1+c)) once its predecessor has finished 3 ops, one op
before the q+4 wait that guards its window.  The CPU test proves that early read safe by brute force over the window
lists of both schedules; the GPU tests compare the kernel byte for byte with the oracle at the sizes where the prepared
head meets the clamped windows of the matrix edge."""
import numpy as np
import pytest

from svdsolver_b200.synth import uniform_matrix

HEAD_WAIT = 3          # prog[i-1] the head row is read at


def _ops_reference(i, n, c):
    """windows (row0, row1, col0, col1) of sweep i, op q = list index (RIGHT(p) = 2p, LEFT(p) = 2p+1), reference schedule"""
    w = c + 1
    out = [(i, min(i + w, n), i + 1, min(i + w, n)), (i + 1, min(i + w, n), i + 1, min(i + 2 * w - 1, n))]
    for k in range((n - min(i + 2 * w - 1, n)) // c + 1):
        r0, r1, r2, c3 = (min(i + 1 + (k + j) * c, n) for j in range(4))
        out.append((r0, r2, r1, r2) if r2 > r1 else None)
        out.append((r1, r2, r1, c3) if c3 > r1 else None)
    return out


def _ops_complete(i, n, c):
    """the same for the complete schedule (every bulge chased to the end)"""
    w = c + 1
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


def _overlap(a, b):
    return a and b and a[0] < b[1] and b[0] < a[1] and a[2] < b[3] and b[2] < a[3]


@pytest.mark.parametrize("complete", [0, 1])
@pytest.mark.parametrize("n,b", [(64, 4), (65, 4), (100, 7), (96, 32), (130, 32), (331, 32), (66, 32)])
def test_head_row_read_after_three_predecessor_ops(n, b, complete):
    """Once prog[i-1] >= 3, no op still to come of an earlier sweep writes row i, cols [i+1, min(i+1+c, n)).

    Sweep i-k has then finished at least 3k ops: op g-1 of sweep i-k+1 waited for g+3 ops of sweep i-k.  A window op
    writes at most its window (what it forwards, the next op's window covers and writes), so it suffices that every
    window of sweep i-k that meets the head row has an index below 3k.  For k = 1 the last one is op 2 (RIGHT(1))."""
    ops = _ops_complete if complete else _ops_reference
    c = b
    windows = [ops(j, n, c) for j in range(n - 1)]
    last_of_predecessor = set()
    for i in range(1, n - 1):
        head = (i, i + 1, i + 1, min(i + 1 + c, n))
        for k in range(1, i + 1):
            hits = [q for q, o in enumerate(windows[i - k]) if _overlap(o, head)]
            if hits:
                assert max(hits) < HEAD_WAIT * k, (i, k, max(hits))
                if k == 1 and i + 1 + c <= n:
                    last_of_predecessor.add(max(hits))
    if n >= 2 * c + 2:
        assert last_of_predecessor == {2}


DT = {"f32": np.float32, "f64": np.float64}


@pytest.mark.gpu
@pytest.mark.parametrize("complete", [0, 1])
@pytest.mark.parametrize("suf", ["f32", "f64"])
@pytest.mark.parametrize("n", [66, 67, 97, 129, 320, 321])
def test_band32_head_and_edge_windows_bit_exact(capi, oracle, n, suf, complete):
    """band 32 near the kernel's smallest size (2b+2 = 66) and at sizes whose last sweeps clamp the head window:
    byte-equal to the oracle under both schedules"""
    b = 32
    band = np.triu(np.tril(uniform_matrix(n, n, 17 + n, 0.0, 5.0, DT[suf]), b))
    ref, d_ref, e_ref = oracle.brd_p2_complete(band, b) if complete else oracle.brd_p2(band, b)
    with capi.Handle(n, b, DT[suf]) as h:
        h.set_stage2_schedule(complete)
        out, d, e = h.band_to_bidiag(band, b)
    assert np.array_equal(out.view(np.uint8), ref.view(np.uint8))
    assert np.array_equal(d.view(np.uint8), d_ref.view(np.uint8)) and np.array_equal(e.view(np.uint8), e_ref.view(np.uint8))


@pytest.fixture(scope="module")
def capi():
    from svdsolver_b200 import capi as m
    m.lib()
    return m
