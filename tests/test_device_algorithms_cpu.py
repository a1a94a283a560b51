"""NumPy mirrors of device algorithms, statement by statement, so that their arithmetic is pinned on
the CPU as well (the CUDA kernels themselves are tested against the oracle in the `-m gpu` suite):

* balanced base-256 slicing of `oz::slice_digits` (emagls_b200/csrc/ozaki.cuh) and the exactness of the
  sliced product with the i + j < T truncation,
* the Hermitian sweep inversion of `gram_sweep_kernel` (emagls_b200/csrc/gram_kernels.cu),
* the real pack/unpack of `fused_render16_kernel` (emagls_b200/csrc/render.cu): N-point real transforms as
  N/2-point complex ones,
* the row-block skipping rule of `tsqr_sep_kernel` (emagls_b200/csrc/tsqr_kernels.cu: significant_blocks) with the bound
  it relies on checked on the em32 steering factor,
* the radix 16 x 16 x 8 passes of `fused_render16_kernel` (register layouts, twiddle tables, output placement),
* the closed-form 2 x 2 mixing matrix of the diffuseness-constraint extension (`diffuseness_mix`, gram_kernels.cu).
"""
import numpy as np
import pytest

from oracle.ozaki_model import slice_digits


@pytest.mark.parametrize("T", [4, 5, 6])
def test_balanced_base256_digits(T):
    rng = np.random.default_rng(T)
    a = np.concatenate([rng.uniform(-64, 64, 100000),
                        [64.0, -64.0, 0.0, np.nextafter(64.0, 0), -np.nextafter(64.0, 0), 0.4999999, 2.0 ** -30,
                         0.498046875 + 1e-9, 63.5, -63.5]])
    q = slice_digits(a, T)
    assert q.min() >= -128 and q.max() <= 127 and np.abs(q[0]).max() <= 64      # int8 operands
    rec = sum(q[s].astype(float) * 256.0 ** -s for s in range(T))
    assert np.abs(rec - a).max() <= 0.5 * 256.0 ** -(T - 1) * (1 + 1e-12)        # |r| <= half the last digit


def test_sliced_product_error_and_int32_range():
    """C = sA sB sum_{i+j<T} 256^-(i+j) qA_i . qB_j: exact integer partial sums, 46 bits relative to
    max|a| max|b| K for T = 6, and every diagonal stays inside int32 for the contraction lengths in use."""
    rng = np.random.default_rng(0)
    K, T = 2720, 6
    a, b = rng.standard_normal(K), rng.standard_normal(K)
    ea, eb = np.frexp(np.abs(a).max())[1], np.frexp(np.abs(b).max())[1]
    qa, qb = slice_digits(a * 2.0 ** (6 - ea), T), slice_digits(b * 2.0 ** (6 - eb), T)
    acc = [sum(int(qa[i] @ qb[d - i]) for i in range(d + 1)) for d in range(T)]
    assert max(abs(v) for v in acc) < 2 ** 31
    assert T * 2 ** 14 * K < 2 ** 31                                             # oz::contraction_fits
    c = 2.0 ** (ea - 6) * 2.0 ** (eb - 6) * sum(acc[d] * 256.0 ** -d for d in range(T))
    assert abs(c - a @ b) <= 2.0 ** -44 * np.abs(a).max() * np.abs(b).max() * K


@pytest.mark.parametrize("M,cond", [(32, 4e3), (25, 50.0), (7, 1e2)])
def test_hermitian_sweep_inversion(M, cond):
    """gram_sweep_kernel: A <- sweep_k(A) for k = 0..M-1 gives -G^-1; the pivots are the Cholesky pivots."""
    rng = np.random.default_rng(M)
    U, _ = np.linalg.qr(rng.standard_normal((M, M)) + 1j * rng.standard_normal((M, M)))
    lam = np.logspace(0, -np.log10(cond), M)
    G = (U * lam) @ U.conj().T
    G = (G + G.conj().T) / 2
    A = G.copy()
    piv = []
    for k in range(M):
        col = A[:, k].copy()                      # published pivot column
        d = col[k].real
        piv.append(d)
        inv = 1.0 / d
        for i in range(M):                        # lane i
            if i == k:
                A[k, :] = A[k, :] * inv
                A[k, k] = -inv
            else:
                f = A[i, k] * inv
                for j in range(M):
                    if j != k:
                        A[i, j] -= f * np.conj(col[j])
                A[i, k] = f
    Ginv = np.linalg.inv(G)
    assert np.abs(-A - Ginv).max() <= 1e-12 * cond * np.abs(Ginv).max()
    L = np.linalg.cholesky(G)
    assert np.allclose(piv, np.abs(np.diag(L)) ** 2, rtol=1e-9)


@pytest.mark.parametrize("N", [8, 64, 2048, 4096])
def test_real_fft_pack_unpack_roundtrip(N):
    """N-point real transforms as M = N/2-point complex ones: rfft unpack with WN, irfft pack with conj(WN)."""
    rng = np.random.default_rng(N)
    M = N // 2
    WN = np.exp(-2j * np.pi * np.arange(M + 1) / N)
    x = rng.standard_normal(N)
    Z = np.fft.fft(x[0::2] + 1j * x[1::2])
    k = np.arange(M + 1)
    zk, zm = Z[k % M], np.conj(Z[(M - k) % M])
    X = 0.5 * (zk + zm) - 0.5j * WN[k] * (zk - zm)                               # rfft unpack
    assert np.abs(X - np.fft.rfft(x)).max() <= 1e-12 * np.abs(X).max()
    k = np.arange(M)
    yk, ym = X[k], np.conj(X[M - k])
    zy = np.fft.ifft((yk + ym) + 1j * np.conj(WN[k]) * (yk - ym)) * M / N        # irfft pack
    y = np.empty(N)
    y[0::2], y[1::2] = zy.real, zy.imag
    assert np.abs(y - x).max() <= 1e-12 * np.abs(x).max()


# ------------------------------------------------------------------------------------------------------------
# significant_blocks (emagls_b200/csrc/tsqr_kernels.cu): row blocks of C_k = R diag(b_k) Y_o^T whose modal
# coefficients lie below 2^-60 of the largest are left out of the factorisation
# ------------------------------------------------------------------------------------------------------------
def significant_blocks(bn, roword, S, nblk):
    a = np.abs(bn)
    thr = a.max() * 2.0 ** -60
    ncut, tail = len(bn), 0.0
    for n in range(len(bn) - 1, -1, -1):
        tail += a[n]
        if tail < thr:
            ncut = n
        else:
            break
    nb = 0
    while nb < nblk and roword[min(nb * 32, S - 1)] < ncut:
        nb += 1
    return max(nb, 1)


def test_skipped_row_blocks_are_below_the_rounding_of_the_kept_rows():
    import oracle
    from emagls_b200 import synth
    g = synth.load_grids()
    az, ze = g["hrirGridAziRad"][::2], g["hrirGridZenRad"][::2]            # 1351 directions: enough for order 19
    N, S = 19, 400
    Yh = oracle.getSH(N, np.stack([az, ze], 1), "real")
    R = np.linalg.qr(Yh, mode="r")
    Ym = oracle.getSH(N, np.stack([g["micGridAziRad"], g["micGridZenRad"]], 1), "real")      # 32 x 400
    roword = np.floor(np.sqrt(np.arange(S))).astype(int)
    fs, nfft, r, c = 48000.0, 1024, 0.042, 343.0
    counts = {}
    for k in (1, 7, 19, 37, 60, 87):
        kr = 2 * np.pi * (k * fs / nfft) * r / c
        bn = np.asarray(oracle.sphModalCoeffs(N, np.array([kr]), "rigid")).ravel()
        nb = significant_blocks(bn, roword, S, 13)
        counts[k] = nb
        C = R @ (bn[roword][:, None] * Ym.T)                               # S x 32
        if nb < 13:
            dropped = np.abs(C[nb * 32:]).max()
            assert dropped <= 2.0 ** -55 * np.abs(C).max(), (k, nb, dropped / np.abs(C).max())
    assert counts[1] <= 3 and counts[7] <= 6 and counts[87] == 13 and counts[60] == 13, counts
    assert all(counts[a] <= counts[b] for a, b in zip((1, 7, 19, 37, 60), (7, 19, 37, 60, 87))), counts


# ------------------------------------------------------------------------------------------------------------
# radix 16 x 16 x 8 Stockham transform of fused_render16_kernel (emagls_b200/csrc/render.cu): register layouts
# of fr_dft16 / fr_dft8, twiddle tables P2 / P3, output placement of the three passes
# ------------------------------------------------------------------------------------------------------------
def _fr_dft4(a, inv):
    a0, a1, a2, a3 = a
    s02, d02, s13, d13 = a0 + a2, a0 - a2, a1 + a3, a1 - a3
    jd = 1j * d13 if inv else -1j * d13
    return [s02 + s13, d02 + jd, s02 - s13, d02 - jd]


def _fr_w16(a, e, inv):
    w = np.exp((2j if inv else -2j) * np.pi * (e % 16) / 16)
    return a * w


def _fr_dft16(v, inv):
    v = list(v)
    for n2 in range(4):
        v[n2], v[4 + n2], v[8 + n2], v[12 + n2] = _fr_dft4([v[n2], v[4 + n2], v[8 + n2], v[12 + n2]], inv)
    for idx, e in ((5, 1), (6, 2), (7, 3), (9, 2), (10, 4), (11, 6), (13, 3), (14, 6), (15, 9)):
        v[idx] = _fr_w16(v[idx], e, inv)
    for m1 in range(4):
        v[4 * m1:4 * m1 + 4] = _fr_dft4(v[4 * m1:4 * m1 + 4], inv)
    return [v[4 * (qp & 3) + (qp >> 2)] for qp in range(16)]               # FR_OUT16


def _fr_dft8(v, inv):
    v = list(v)
    v[0], v[2], v[4], v[6] = _fr_dft4([v[0], v[2], v[4], v[6]], inv)
    v[1], v[3], v[5], v[7] = _fr_dft4([v[1], v[3], v[5], v[7]], inv)
    t = [v[1], _fr_w16(v[3], 2, inv), _fr_w16(v[5], 4, inv), _fr_w16(v[7], 6, inv)]
    o = [None] * 8
    for m1 in range(4):
        o[m1], o[m1 + 4] = v[2 * m1] + t[m1], v[2 * m1] - t[m1]
    return o


@pytest.mark.parametrize("inv", [False, True])
def test_radix16_stockham_passes_of_the_fused_render_kernel(inv):
    M = 2048
    rng = np.random.default_rng(16)
    x = rng.standard_normal(M) + 1j * rng.standard_normal(M)
    # twiddle table of render_twiddle_full_kernel
    tab = np.zeros(4 * 16 + 3 * 256, complex)
    for i in range(tab.size):
        j = ((i & 15) * 8) << (i >> 4) if i < 64 else ((i - 64) & 255) << ((i - 64) >> 8)
        tab[i] = np.exp(-2j * np.pi * j / M)
    tw = (lambda i: np.conj(tab[i])) if inv else (lambda i: tab[i])
    Z = x.copy()
    # pass 1 (stride 1): butterfly t reads t + 128 q, writes 16 t + q'
    out = np.zeros(M, complex)
    for t in range(128):
        out[16 * t:16 * t + 16] = _fr_dft16([Z[t + 128 * q] for q in range(16)], inv)
    Z = out
    # pass 2 (stride 16)
    out = np.zeros(M, complex)
    for t in range(128):
        k, a = t & 15, t // 16
        w1, w2, w4, w8 = tw(k), tw(16 + k), tw(32 + k), tw(48 + k)
        w3, w5, w6 = w1 * w2, w4 * w1, w4 * w2
        w7 = w4 * w3
        ws = [1, w1, w2, w3, w4, w5, w6, w7, w8, w8 * w1, w8 * w2, w8 * w3, w8 * w4, w8 * w5, w8 * w6, w8 * w7]
        o = _fr_dft16([Z[t + 128 * q] * ws[q] for q in range(16)], inv)
        for qp in range(16):
            out[a * 256 + k + 16 * qp] = o[qp]
    Z = out
    # pass 3 (radix 8, stride 256)
    out = np.zeros(M, complex)
    for tt in range(256):
        w1, w2, w4 = tw(64 + tt), tw(64 + 256 + tt), tw(64 + 512 + tt)
        w3 = w1 * w2
        ws = [1, w1, w2, w3, w4, w4 * w1, w4 * w2, w4 * w3]
        o = _fr_dft8([Z[tt + 256 * q] * ws[q] for q in range(8)], inv)
        for qp in range(8):
            out[tt + 256 * qp] = o[qp]
    ref = np.fft.ifft(x) * M if inv else np.fft.fft(x)
    assert np.abs(out - ref).max() <= 1e-12 * np.abs(ref).max()


# ------------------------------------------------------------------------------------------------------------
# diffuseness_mix (emagls_b200/csrc/gram_kernels.cu): closed-form 2 x 2 polar factor against the oracle's SVD route
# ------------------------------------------------------------------------------------------------------------
def diffuseness_mix(R, Rh):
    x11, g11 = np.sqrt(R[0, 0].real), np.sqrt(Rh[0, 0].real)
    x12, g12 = R[0, 1] / x11, Rh[0, 1] / g11
    x22, g22 = np.sqrt(R[1, 1].real - abs(x12) ** 2), np.sqrt(Rh[1, 1].real - abs(g12) ** 2)
    B = np.array([[g11 * x11 + g12 * np.conj(x12), g12 * x22], [g22 * np.conj(x12), g22 * x22]])
    P = B.conj().T @ B
    sdet = abs(np.linalg.det(B))
    c = np.sqrt(P[0, 0].real + P[1, 1].real + 2 * sdet)
    Pm = c * B @ np.linalg.inv(P + sdet * np.eye(2))
    XH = np.array([[x11, 0], [np.conj(x12), x22]])
    LinvH = np.array([[1 / g11, 0], [-np.conj(g12) / (g11 * g22), 1 / g22]])
    return XH @ Pm.conj().T @ LinvH


def test_closed_form_diffuseness_mix_matches_the_oracle():
    import oracle
    rng = np.random.default_rng(22)
    for _ in range(50):
        X = rng.standard_normal((2, 9)) + 1j * rng.standard_normal((2, 9))
        Y = rng.standard_normal((2, 9)) + 1j * rng.standard_normal((2, 9))
        R, Rh = X @ X.conj().T / 9, Y @ Y.conj().T / 9
        A, Ao = diffuseness_mix(R, Rh), oracle.diffuseness_matrix(R, Rh)
        assert np.abs(A - Ao).max() <= 1e-11 * max(1.0, np.abs(Ao).max())
        assert np.abs(A @ Rh @ A.conj().T - R).max() <= 1e-11 * np.abs(R).max()
