"""Bit-exact NumPy model of the int8 tensor-core GEMM (emagls_b200/csrc/ozaki.cuh, ozaki_kernels.cu).

TEST INFRASTRUCTURE ONLY, like the rest of this package.  Every function restates one device step with the same
roundings, so that the CUDA kernels can be compared with it bit for bit:

* `slice_digits`      balanced base-256 digits of `oz::slice_digits` (|a| <= 64),
* `slice_rows`        `slice_rows_kernel`: row exponent, digits of x 2^(6-e), zero padding, scale 2^(e-6),
* `row_scale`         `row_scale_kernel`: up = 2^(6-e), sc = 2^(e-6),
* `diagonals`         the T int32 diagonal accumulators acc_d = sum_{i+j=d} qA_i qB_j^T (float64 matmuls, exact:
                      every partial sum is an integer below 2^53),
* `gemm_f64`          the output of `EpiStoreF64`: rn(H 256^(T-3) + L) (sA 256^-(T-1)) sB,
* `exact_values`      the exact integers v = sum_d acc_d 256^(T-1-d) (Python ints where |v| may reach 2^63),
* `phase_reference`   Z = t 2^24 256^(T-4), t = |H| up y / |y|, unrounded, in long double: the quantity whose
                      rounding the forward epilogues write as digits (tests/csrc/phase_fixed_check.cpp evaluates the
                      same formula in quad precision).
"""
from __future__ import annotations

import numpy as np


def slice_digits(a, T):
    """oz::slice_digits<T>: |a| <= 64 -> digits q[T] with a = sum q_s 256^-s + r."""
    nh = T - 3
    bias_hi = {3: 0x808080, 2: 0x8080, 1: 0x80}[nh]
    ah = a * float(1 << (8 * (nh - 1)))
    hi = np.rint(ah).astype(np.int64)
    lo = np.rint((ah - hi) * 16777216.0).astype(np.int64)
    yl = lo + 0x808080
    hi = hi + (yl >> 24)
    zl = yl ^ 0x808080
    sb = lambda v: ((v & 0xFF) + 128) % 256 - 128          # noqa: E731  (int)(signed char)
    q = np.zeros((T,) + a.shape, dtype=np.int64)
    q[T - 1], q[T - 2], q[T - 3] = sb(zl), sb(zl >> 8), sb(zl >> 16)
    zh = (hi + bias_hi) ^ bias_hi
    for j in range(nh):
        q[nh - 1 - j] = sb(zh >> (8 * j))
    return q


def row_exponent(X):
    """e with 2^e > max_k |x(r, k)| (frexp of the row maximum); 0 for a zero row."""
    mx = np.abs(X).max(axis=1) if X.shape[1] else np.zeros(X.shape[0])
    e = np.frexp(mx)[1].astype(np.int64)
    return np.where((mx > 0) & (mx < 1e300), e, 0)


def row_scale(X):
    """row_scale_kernel: (up, sc) = (2^(6-e), 2^(e-6)) per row of X."""
    e = row_exponent(X)
    return np.ldexp(1.0, 6 - e), np.ldexp(1.0, e - 6)


def slice_rows(X, T, Kpad):
    """slice_rows_kernel on the rows of X (R x K): digits [T][R][Kpad] (int8) and scales [R]."""
    R, K = X.shape
    up, sc = row_scale(X)
    a = np.zeros((R, Kpad))
    a[:, :K] = X * up[:, None]
    return slice_digits(a, T).astype(np.int8), sc


def diagonals(qA, qB, T):
    """acc_d = sum_{i+j=d} qA_i qB_j^T for d < T, as exact float64 matrices (each term below 2^14 in magnitude, each
    sum below 2^31)."""
    A = [qA[i].astype(np.float64) for i in range(T)]
    B = [qB[j].astype(np.float64) for j in range(T)]
    return [sum(A[i] @ B[d - i].T for i in range(d + 1)) for d in range(T)]


def combine_f64(acc, T):
    """oz::combine_diagonals: H = digits 0..2, L = digits 3..T-1 (both exact), then one rounding."""
    H = (acc[0] * 256.0 + acc[1]) * 256.0 + acc[2]
    L = acc[3]
    for d in range(4, T):
        L = L * 256.0 + acc[d]
    return H * float(1 << (8 * (T - 3))) + L


def gemm_f64(qA, sA, qB, sB, T):
    """The M x N output of ozaki_gemm_kernel with EpiStoreF64, bit for bit."""
    v = combine_f64(diagonals(qA, qB, T), T)
    return v * ((sA[:, None] * 2.0 ** (-8 * (T - 1))) * sB[None, :])


def exact_values(acc, T):
    """v = sum_d acc_d 256^(T-1-d) exactly: int64 when |v| < 2^62 is guaranteed, else Python ints (object array)."""
    a = [np.asarray(x).astype(np.int64) for x in acc]
    H = (a[0] * 256 + a[1]) * 256 + a[2]
    L = a[3]
    for d in range(4, T):
        L = L * 256 + a[d]
    sh = 8 * (T - 3)
    if H.size == 0 or int(np.abs(H).max()) < 2 ** (61 - sh):
        return H * (1 << sh) + L
    return H.astype(object) * (1 << sh) + L.astype(object)


def to_longdouble(v):
    """Exact long-double copy of integers |v| < 2^64 (int64 or Python ints)."""
    if v.dtype != object:
        return v.astype(np.longdouble)
    hi = (v >> 32).astype(np.int64).astype(np.longdouble)
    lo = (v & 0xFFFFFFFF).astype(np.int64).astype(np.longdouble)
    return hi * np.longdouble(2.0 ** 32) + lo


def phase_reference(v, sB, absH, up, T, orient_per_set, nyquist):
    """Unrounded Z = t 2^24 256^(T-4) of every output row of the forward product, in long double.

    v      [D][rows] exact integers of y (column n = 4 problem + 2 ear + (0: re, 1: im)),
    sB     [rows] power-of-two scales of the rows of c (only the re / im exponent difference matters),
    absH   [sets][2][D] |H| of this bin, up [sets][2] its scales 2^(6-e).
    Returns Z [rows][D]: t = |H| up y / |y| (angle 0 where y = 0), the imaginary rows zero with `nyquist`.
    """
    D, rows = v.shape
    cols = np.arange(0, rows, 2)
    prob, ear = cols >> 2, (cols >> 1) & 1
    st = prob // orient_per_set
    dexp = np.frexp(sB[cols])[1] - np.frexp(sB[cols + 1])[1]
    vl = to_longdouble(v)
    re = np.ldexp(vl[:, cols], dexp[None, :].astype(np.int32))
    im = vl[:, cols + 1]
    nrm = np.sqrt(re * re + im * im)
    mag = (absH[st, ear, :].T.astype(np.longdouble) * up[st, ear][None, :].astype(np.longdouble)
           * np.longdouble(2.0 ** (24 + 8 * (T - 4))))
    zero = nrm == 0
    safe = np.where(zero, np.longdouble(1), nrm)
    zr = np.where(zero, mag, mag * re / safe)
    zi = np.where(zero | bool(nyquist), np.longdouble(0), mag * im / safe)
    Z = np.empty((rows, D), dtype=np.longdouble)
    Z[cols] = zr.T
    Z[cols + 1] = zi.T
    return Z


def digits_value(q):
    """Integer of digit planes q [T][...]: sum_s q_s 256^(T-1-s)."""
    T = q.shape[0]
    Z = np.zeros(q.shape[1:], dtype=np.int64)
    for s in range(T):
        Z = Z * 256 + q[s].astype(np.int64)
    return Z


def drain_i64_bound(T):
    """Largest |v| per contraction step from the digit ranges (|q_0| <= 64, |q_s| <= 128): the integer drain
    (oz::combine_diagonals_i64) is exact while Kpad times this stays below 2^63."""
    mx = [64] + [128] * (T - 1)
    return sum(mx[i] * mx[d - i] * 256 ** (T - 1 - d) for d in range(T) for i in range(d + 1))


def cost_rounds(m_tiles, n, nt, sms):
    """The tile-width cost of launch_oz_fwd / launch_oz_bwd: rounds of tiles times operand bytes per k-step."""
    return (m_tiles * ((n + nt - 1) // nt) + sms - 1) // sms * (128 + nt)
