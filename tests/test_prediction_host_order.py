"""CPU: the summation order of NumPy's two-term dot products on this host, which `fot_safety_kernel`
(csrc/fot_predict.cuh) writes out to reproduce `compute_safety_metrics_static` bit for bit.

The reference decides "ahead" with `(ped_pos - [x, y]) @ heading` and the time to collision with
`np.dot(rel_pos, rel_vel) / np.linalg.norm(rel_pos)`.  These are BLAS calls, and OpenBLAS's x86-64 kernels fuse
one of the two products into the other: which one depends on the call.  On near-cancelling inputs (a pedestrian
almost exactly abeam of the vehicle) the plain `a0*b0 + a1*b1` can even return the opposite sign.  The expected
values below evaluate `fma` exactly through `Fraction` (Python 3.12 has no `math.fma`)."""
from fractions import Fraction

import numpy as np
import pytest

MSG = ("the order reproduced by fot_safety_kernel (csrc/fot_predict.cuh) does not hold on this host: "
       "NumPy/BLAS computes {what} differently, so the kernel's ahead classification / ttc can differ from the "
       "reference here")


def fma(a, b, c):
    """a * b + c with one rounding (int / int true division in CPython is correctly rounded)."""
    return float(Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c)))


def near_cancelling(n, seed):
    """Pairs (r, h): h a unit heading, r a point up to 20 m to the side and ~1e-15 m off the abeam line, so that
    r . h is a near-total cancellation; plus generic pairs of mixed magnitudes."""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        yaw = rng.uniform(-np.pi, np.pi)
        h = np.array([np.cos(yaw), np.sin(yaw)])
        if i % 4 == 3:
            r = rng.normal(0, 1, 2) * 10.0 ** rng.integers(-3, 4, 2)
        else:
            t = rng.uniform(-20, 20)
            r = t * np.array([-h[1], h[0]]) + rng.uniform(-1, 1) * 1e-15 * abs(t) * h
        out.append((r, h))
    return out


def test_pairs_are_near_cancelling():
    """The inputs discriminate: the two fused orders and the plain sum disagree on a good share of them."""
    diff = sum(fma(r[0], h[0], r[1] * h[1]) != fma(r[1], h[1], r[0] * h[0]) for r, h in near_cancelling(400, 1))
    assert diff > 100


def test_one_row_matmul():
    """`[1,2] @ [2]`: fma(a1, b1, a0 * b0) -- the one-pedestrian `ahead` of the safety kernel."""
    for r, h in near_cancelling(1000, 2):
        got = (r[None, :] @ h)[0]
        assert got == fma(r[1], h[1], r[0] * h[0]), MSG.format(what="[1,2] @ [2]") + f" ({r!r}, {h!r})"


@pytest.mark.parametrize("k", [2, 3, 17, 50, 300])
def test_k_row_matmul(k):
    """`[k,2] @ [2]`, k >= 2: fma(a0, b0, a1 * b1) in every row -- the several-pedestrian `ahead`."""
    pairs = near_cancelling(max(k, 200), 10 + k)
    h = pairs[0][1]
    rows = [r for r, _ in pairs]
    for start in range(0, len(rows), k):
        A = np.array((rows[start:] + rows)[:k])
        got = A @ h
        want = np.array([fma(a[0], h[0], a[1] * h[1]) for a in A])
        assert np.array_equal(got, want), MSG.format(what=f"[{k},2] @ [2]") + f" (rows {np.flatnonzero(got != want)})"


def test_dot_of_two_vectors():
    """`np.dot` of two length-2 vectors: fma(a1, b1, a0 * b0) -- the safety kernel's `along`."""
    for r, h in near_cancelling(1000, 3):
        v = h * 3.7 - r[::-1] * 0.2
        for a, b in ((r, h), (r, v)):
            assert np.dot(a, b) == fma(a[1], b[1], a[0] * b[0]), MSG.format(what="np.dot of 2-vectors") + f" ({a!r}, {b!r})"


def test_norm_of_two_vector():
    """`np.linalg.norm` of a length-2 vector: sqrt(fma(a1, a1, a0 * a0)) -- the denominator of `along`."""
    rng = np.random.default_rng(4)
    hits = 0
    for _ in range(4000):
        a = rng.normal(0, 1, 2) * 10.0 ** rng.integers(-4, 3, 2)
        want = np.sqrt(fma(a[1], a[1], a[0] * a[0]))
        assert np.linalg.norm(a) == want, MSG.format(what="np.linalg.norm of a 2-vector") + f" ({a!r})"
        hits += want != np.sqrt(a[0] * a[0] + a[1] * a[1])
    assert hits > 0                     # the fused and the plain form differ on some of these inputs
