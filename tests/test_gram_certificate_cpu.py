"""The route decision of the Gram route (emagls_b200/csrc/gram_kernels.cu: gram_classify, gram_certify_kernel) on
the CPU: a NumPy mirror of the classification by the Frobenius bound, the shifted Cholesky and its margin delta, and
the em32 bins it sends down each route, from the oracle's Gram matrices.

A bin may take the Gram route only where cond_2(G_k) <= tau = min(1e4, 1/c^2) (no singular value of the steering
matrix is clipped, and the normal equations stay accurate); the certificate must never accept a matrix above tau.
"""
import math

import numpy as np
import pytest

from emagls_b200 import synth
from oracle import emagls_oracle as eo

DELTA = 1e-6          # GRAM_CERT_DELTA


def chol_lower_ok(A):
    """chol_lower: right-looking Cholesky of the lower triangle, False at the first pivot that is not positive."""
    L = np.tril(A).astype(complex)
    M = L.shape[0]
    for j in range(M):
        d = L[j, j].real
        if not (0.0 < d < 1e300):
            return False
        ljj = math.sqrt(d)
        L[j + 1:, j] *= 1.0 / ljj
        L[j, j] = ljj
        col = L[j + 1:, j]
        L[j + 1:, j + 1:] -= np.tril(np.outer(col, col.conj()))
    return True


def route_ok(G, tau):
    """True when the Gram route accepts G: gram_classify, then gram_certify_kernel for the candidates."""
    M = G.shape[0]
    X = np.linalg.inv(G)                                   # the inversion kernel's result
    xf = np.linalg.norm(X, "fro")
    condF = np.linalg.norm(G, "fro") * xf
    if condF <= tau:
        return True
    if not condF <= M * tau:
        return False
    sigma = tau * (1.0 - DELTA) / xf
    if np.real(np.diag(G)).max() >= sigma:                 # lambda_max >= max G_ii
        return False
    S = -G.copy()
    S[np.diag_indices(M)] += sigma
    return chol_lower_ok(S)


def hermitian(lam, rng):
    M = len(lam)
    U, _ = np.linalg.qr(rng.standard_normal((M, M)) + 1j * rng.standard_normal((M, M)))
    G = (U * lam) @ U.conj().T
    return (G + G.conj().T) / 2


def em32_spectrum(cond, rng, M=32):
    """A cluster of 8 comparable large eigenvalues (the largest 1), one smallest 1/cond, the rest in between."""
    top = np.concatenate([[1.0], rng.uniform(0.5, 1.0, 7)])
    mid = np.logspace(np.log10(0.3), np.log10(30.0 / cond), M - 9)
    return np.concatenate([top, mid, [1.0 / cond]])


@pytest.mark.parametrize("tau", [1e4, 2500.0])
def test_certificate_on_em32_shaped_spectra(tau):
    rng = np.random.default_rng(int(tau))
    for _ in range(20):
        assert not route_ok(hermitian(em32_spectrum(tau * (1 + 1e-3), rng), rng), tau)
        assert not route_ok(hermitian(em32_spectrum(tau * 1.5, rng), rng), tau)
        assert route_ok(hermitian(em32_spectrum(tau * 0.97, rng), rng), tau)
        assert route_ok(hermitian(em32_spectrum(tau * 0.5, rng), rng), tau)


@pytest.mark.parametrize("tau", [1e4, 2500.0])
def test_certificate_never_accepts_above_tau_on_random_spectra(tau):
    rng = np.random.default_rng(7 + int(tau))
    for trial in range(60):
        M = int(rng.choice([7, 25, 32, 64]))
        factor = [1 + 1e-3, 1 - 1e-3, rng.uniform(1.0, 4.0 * M), rng.uniform(0.05, 1.0)][trial % 4]
        cond = tau * factor
        lam = np.exp(rng.uniform(0.0, np.log(cond), M))
        lam[0], lam[1] = 1.0, cond                         # exact extremes
        G = hermitian(lam / cond, rng)
        c2 = np.linalg.cond(G)
        ok = route_ok(G, tau)
        if c2 >= tau:
            assert not ok, (M, c2)


def test_frobenius_bound_alone_decides_far_from_tau():
    rng = np.random.default_rng(3)
    G = hermitian(np.linspace(1.0, 2.0, 32), rng)          # condF well below tau: no certificate needed
    X = np.linalg.inv(G)
    assert np.linalg.norm(G, "fro") * np.linalg.norm(X, "fro") <= 1e4 and route_ok(G, 1e4)
    G = hermitian(np.logspace(0, -6, 32), rng)             # condF > M tau: refused without a certificate
    X = np.linalg.inv(G)
    assert np.linalg.norm(G, "fro") * np.linalg.norm(X, "fro") > 32 * 1e4 and not route_ok(G, 1e4)


def test_em32_route_split_at_bin_67(grids):
    """em32, order 4, 512 taps: the clip of lib/getEMagLs2Filters.m:88 is active exactly in bins 1..66
    (cond_2(G_k) > 1/c^2 = 1e4); from bin 67 on lambda_max ||G^-1||_F <= tau (1 - delta), so the certificate accepts
    every orientation there.  Bins are numbered from 0 (DC) as in the library; the reference's MATLAB column k + 1.
    G_k does not depend on the HRIRs."""
    az, ze = grids["hrirGridAziRad"], grids["hrirGridZenRad"]
    cfg = eo._cfg({})
    c = cfg["SVD_REGUL_CONST"]
    tau = min(1e4, 1.0 / c ** 2)
    nfft, _, _, _ = eo._freq_setup(grids["fs"], 512, 4, cfg)
    params = dict(returnRawMicSigs=True, fs=grids["fs"], irLen=nfft, oversamplingFactor=1, simulateAliasing=True,
                  radialFilter="none", smaRadius=grids["micRadius"],
                  smaDesignAziZenRad=np.stack([grids["micGridAziRad"], grids["micGridZenRad"]], 1),
                  waveModel="planeWave", arrayType="rigid", shDefinition="real", shFunction=eo.getSH, C=cfg["C"])
    sm, _ = eo.getSMAIRMatrix(params)
    simN = int(round(math.sqrt(sm.shape[1]))) - 1
    R = synth.orientation_grid()
    for o in (0, 1234):
        raz, rze = synth.rotate_grid(az, ze, R[o])
        Yc = np.conj(eo.getSH(simN, np.stack([raz, rze], 1), "real")).T
        for k in range(59, 80):
            pw = sm[:, :, k] @ Yc
            G = pw.conj() @ pw.T
            ev = np.linalg.eigvalsh(G)
            if k <= 66:
                assert ev[-1] / ev[0] > tau, (o, k)
                assert not route_ok(G, tau), (o, k)
            else:
                assert ev[-1] * math.sqrt((ev ** -2.0).sum()) <= tau * (1 - DELTA), (o, k)
                assert route_ok(G, tau), (o, k)
