"""The bit-exact NumPy model of the int8 tensor-core GEMM (oracle/ozaki_model.py) against Python-integer and
high-precision decimal arithmetic, and a compile check of the harness that runs the CUDA kernels against the model
(tests/csrc/ozaki_harness.cu, used by tests/test_gpu_ozaki.py)."""
import decimal
import shutil
from fractions import Fraction

import numpy as np
import pytest

from oracle import ozaki_model as om


def _digits(rng, T, R, K, extreme=False):
    q = np.empty((T, R, K), np.int8)
    if extreme:
        q[:] = -128
        q[0] = rng.choice([-64, 64], (R, K))
    else:
        q[0] = rng.integers(-64, 65, (R, K))
        q[1:] = rng.integers(-128, 128, (T - 1, R, K))
    return q


@pytest.mark.parametrize("T", [4, 6])
@pytest.mark.parametrize("extreme", [False, True])
def test_gemm_model_matches_python_integers(T, extreme):
    """acc_d, the exact v and the FP64 output (one rounding of v, then power-of-two scales) against Python ints"""
    rng = np.random.default_rng(T + 2 * extreme)
    M, N, K = 5, 7, 300
    qA, qB = _digits(rng, T, M, K, extreme), _digits(rng, T, N, K, extreme)
    sA, sB = np.ldexp(1.0, rng.integers(-40, 40, M)), np.ldexp(1.0, rng.integers(-40, 40, N))
    acc = om.diagonals(qA, qB, T)
    v = om.exact_values(acc, T)
    C = om.gemm_f64(qA, sA, qB, sB, T)
    A = [[[int(x) for x in qA[s, m]] for m in range(M)] for s in range(T)]
    B = [[[int(x) for x in qB[s, n]] for n in range(N)] for s in range(T)]
    big = 0
    for m in range(M):
        for n in range(N):
            a = [sum(sum(x * y for x, y in zip(A[i][m], B[d - i][n])) for i in range(d + 1)) for d in range(T)]
            assert [int(acc[d][m, n]) for d in range(T)] == a
            ve = sum(a[d] * 256 ** (T - 1 - d) for d in range(T))
            assert int(v[m, n]) == ve
            big += abs(ve) > 2 ** 53
            c = float(ve) * (float(sA[m]) * 2.0 ** (-8 * (T - 1)) * float(sB[n]))
            assert C[m, n] == c, (m, n)
    if extreme and T == 6:
        assert big > 0                                   # the rounding of v to 53 bits is exercised


@pytest.mark.parametrize("T", [4, 6])
def test_slicing_model_reconstructs_rows(T):
    rng = np.random.default_rng(T)
    X = rng.standard_normal((6, 50)) * np.ldexp(1.0, rng.integers(-50, 50, 6))[:, None]
    X[0] = 0.0
    X[1, 3] = -np.ldexp(1.0, 7) * (1 - 2.0 ** -53)       # row maximum just below a power of two
    q, sc = om.slice_rows(X, T, 64)
    assert q.dtype == np.int8 and not q[:, :, 50:].any()
    assert np.abs(q[0].astype(int)).max() <= 64
    assert sc[0] == 2.0 ** -6
    for r in range(6):
        mx = np.abs(X[r]).max()
        assert mx < 64 * sc[r] and (mx == 0 or mx >= 32 * sc[r])
        for k in range(50):
            rec = sum(Fraction(int(q[s, r, k])) / 256 ** s for s in range(T))
            assert abs(rec - Fraction(X[r, k]) / Fraction(sc[r])) <= Fraction(1, 2 * 256 ** (T - 1))


def test_phase_reference_against_decimal():
    """phase_reference in long double against 40-digit decimal arithmetic, Python-int v beyond 2^63 included"""
    if np.finfo(np.longdouble).nmant < 63:
        pytest.skip("long double without a 64-bit significand")
    decimal.getcontext().prec = 40
    dec = lambda x: decimal.Decimal(np.format_float_positional(x, unique=True))   # noqa: E731
    rng = np.random.default_rng(1)
    T, D, P, ops = 6, 3, 3, 2
    rows = 4 * P
    v = np.empty((D, rows), dtype=object)
    for m in range(D):
        for n in range(rows):
            v[m, n] = int(rng.integers(-2 ** 62, 2 ** 62)) * int(rng.integers(1, 3))
    v[0, 0], v[0, 1] = 2 ** 63 + 12345, -(2 ** 63) + 1
    v[1, 4], v[1, 5] = 0, 0                               # y = 0: angle 0
    v[2, 2] = 0
    sB = np.ldexp(1.0, rng.integers(-30, 30, rows))
    absH = np.abs(rng.standard_normal((2, 2, D)))
    up = np.ldexp(1.0, rng.integers(-3, 3, (2, 2)))
    Z = om.phase_reference(v, sB, absH, up, T, ops, False)
    Zn = om.phase_reference(v, sB, absH, up, T, ops, True)
    for m in range(D):
        for n in range(0, rows, 2):
            p, ear = n >> 2, (n >> 1) & 1
            dexp = int(np.frexp(sB[n])[1] - np.frexp(sB[n + 1])[1])
            re = decimal.Decimal(v[m, n]) * decimal.Decimal(2) ** dexp
            im = decimal.Decimal(v[m, n + 1])
            mag = decimal.Decimal(float(absH[p // ops, ear, m])) * decimal.Decimal(float(up[p // ops, ear])) * 2 ** 40
            nrm = (re * re + im * im).sqrt()
            zr, zi = (mag, 0) if nrm == 0 else (mag * re / nrm, mag * im / nrm)
            assert abs(dec(Z[n, m]) - zr) <= decimal.Decimal("1e-4")
            assert abs(dec(Z[n + 1, m]) - zi) <= decimal.Decimal("1e-4")
            assert Zn[n, m] == Z[n, m] and Zn[n + 1, m] == 0


def test_integer_drain_range():
    """The 64-bit drain of the integer forward functor is exact for Kpad <= 2016 at T = 6 (the digit ranges give
    |v| <= 1.0157 Kpad 2^52), and flat rows reach beyond 2^63 at the 2049 harmonics of order 44"""
    b6 = om.drain_i64_bound(6)
    assert 2016 * b6 < 2 ** 63 <= 2017 * b6
    assert 32736 * om.drain_i64_bound(4) < 2 ** 63
    x = np.full((1, 2049), 1.0 - 2.0 ** -30)
    q, _ = om.slice_rows(x, 6, 2080)
    v = om.exact_values(om.diagonals(q, q, 6), 6)
    assert int(v[0, 0]) > 2 ** 63


def test_harness_compiles(tmp_path):
    """the GPU harness builds against the current kernels (a kernel change that breaks it fails here, without a GPU)
    and its host-side range checks agree with the model"""
    from emagls_b200 import build as b
    try:
        b._nvcc()
    except RuntimeError:
        pytest.skip("nvcc not available")
    if shutil.which("g++") is None and shutil.which("c++") is None:
        pytest.skip("no host compiler")
    from oracle.ozaki_harness import Harness, compile_harness
    so = compile_harness(str(tmp_path))
    try:
        h = Harness(so)
    except OSError as e:                                  # loading needs the CUDA runtime's dependencies only
        pytest.skip(f"harness not loadable here: {e}")
    for T in (4, 6):
        for Kpad in range(32, 33000, 32):
            assert h.drain_i64_fits(Kpad, T) == (Kpad * om.drain_i64_bound(T) < 2 ** 63)
            assert h.contraction_fits(Kpad, T) == (T * 2 ** 14 * Kpad < 2 ** 31)
