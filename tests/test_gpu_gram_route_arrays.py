"""The eMagLS2 designer on Fibonacci arrays of 4 to 60 microphones (B200 only): every channel count at which the Gram
route's kernels and the TSQR + Jacobi kernels change code path, 128 taps at 48 kHz, every third HRIR direction (901),
two orientations (identity and one rotation of the orientation grid).

Per array:
* route counts: `stats_read()` equals the NumPy mirror `route_ok` (tests/test_gram_certificate_cpu.py) applied per
  orientation to the oracle's Gram matrices, a bin taking the Gram route when every orientation accepts it; bins where
  lambda_max ||G^-1||_F lies within 1e-4 of tau (1 - delta) may go either way and are rare;
* per-bin parity with the oracle at classes set by the steering matrix's sigma_min / sigma_max, and the whole filter;
* the design forced through TSQR + Jacobi (EMAGLS_NO_GRAM=1) agrees with the default one above the floor;
* the bound of the well-conditioned bins is 5e-10, not the 1e-10 of em32 at 512 taps: above the LS bins each bin's
  target phase is that of the previous bin's solution, and where a direction's response is small that phase carries a
  rounding difference on, growing towards Nyquist.  Measured on a B200: up to 2.8e-10 against the oracle (31
  microphones, bins 123..128) and 1.9e-10 between the two routes (60 microphones, rotated orientation), while single
  Gram-route bins agree with the extended-precision references of tests/test_gpu_gram_kernels.py to rounding;
* on two arrays, the lowest LS bin against the exact rows of the reference's formula (oracle/hp_oracle.py), with the
  acceptance of tests/test_gpu_arbitration.py.

The SH-domain designer (`getEMagLsFilters`) runs on a 64-microphone array at orders 1, 2, 5 and 6.
"""
import math

import numpy as np
import pytest

import oracle
from emagls_b200 import synth
from oracle import emagls_oracle as eo
from oracle import hp_oracle as hp
from test_gram_certificate_cpu import DELTA, route_ok

pytestmark = pytest.mark.gpu

FS, LEN = 48000.0, 128
ARRAYS = [  # (microphones, order, radius): the code path each one reaches
    pytest.param(4, 1, 0.042, id="M4-sweep_28_padding_rows-gram_only"),
    pytest.param(7, 1, 0.042, id="M7-small_tsqr_problems"),
    pytest.param(19, 3, 0.035, id="M19-odd_Mc_8byte_tiles-odd_McS_bwd_small"),
    pytest.param(25, 4, 0.05, id="M25-S529_bwd_small-S_not_multiple_of_32"),
    pytest.param(31, 4, 0.042, id="M31-tsqr_without_folding"),
    pytest.param(33, 4, 0.042, id="M33-launch_factor-chol_4warps"),
    pytest.param(48, 5, 0.042, id="M48-generic_block_plan"),
    pytest.param(59, 6, 0.042, id="M59-chol_4warps"),
    pytest.param(60, 6, 0.042, id="M60-chol_3warps"),
]
EXACT = {19, 48}           # arrays whose lowest LS bin is arbitrated against exact arithmetic


@pytest.fixture(scope="module")
def em():
    import emagls_b200
    return emagls_b200


@pytest.fixture(scope="module")
def h(em):
    return em.Handle(0)


@pytest.fixture(scope="module")
def sub(grids):
    az, ze = grids["hrirGridAziRad"][::3], grids["hrirGridZenRad"][::3]
    hL, hR = synth.synth_hrirs(az, ze, fs=FS, taps=LEN)
    R = np.stack([np.eye(3), synth.orientation_grid()[1234]])
    return dict(az=az, ze=ze, hL=hL, hR=hR, R=R)


def rel(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


def bin_err(W, Wo):
    return np.abs(W - Wo).max(1) / np.abs(Wo).max(1)


def bin_tol(ratio):
    """per-bin parity bound from the steering matrix's sigma_min / sigma_max (tests/test_gpu_design.py: check_bins)"""
    return np.where(ratio >= 1e-6, 5e-10, np.where(ratio >= 1e-9, 1e-8, 2e-6))


def mirror(sub, M, radius, maz, mze, nfft, K):
    """per bin: the mirror's route (Gram iff every orientation accepts), bins near the certificate's threshold, the
    steering matrix's sigma_min / sigma_max per orientation; the SMAIR matrix and simN"""
    c = eo._cfg({})["SVD_REGUL_CONST"]
    tau = min(1e4, 1.0 / c ** 2)
    params = dict(returnRawMicSigs=True, fs=FS, irLen=nfft, oversamplingFactor=1, simulateAliasing=True,
                  radialFilter="none", smaRadius=radius, smaDesignAziZenRad=np.stack([maz, mze], 1),
                  waveModel="planeWave", arrayType="rigid", shDefinition="real", shFunction=eo.getSH, C=343.0)
    sm, _ = eo.getSMAIRMatrix(params)
    simN = int(round(math.sqrt(sm.shape[1]))) - 1
    gram = np.ones(K, bool)
    near = np.zeros(K, bool)
    ratio = np.zeros((2, K))
    for o in range(2):
        raz, rze = synth.rotate_grid(sub["az"], sub["ze"], sub["R"][o])
        Yc = np.conj(eo.getSH(simN, np.stack([raz, rze], 1), "real")).T
        for k in range(1, K):
            pw = sm[:, :, k] @ Yc
            sv = np.linalg.svd(pw, compute_uv=False)
            ratio[o, k] = sv[-1] / sv[0]
            G = pw.conj() @ pw.T
            ev = np.linalg.eigvalsh(G)
            r = ev[-1] * math.sqrt((ev ** -2.0).sum()) / tau if ev[0] > 0 else math.inf
            near[k] |= abs(r / (1 - DELTA) - 1) < 1e-4
            gram[k] &= route_ok(G, tau)
        ratio[o, 0] = ratio[o, 1]              # DC = real(W(bin 1))
    return gram, near, ratio, sm, simN


@pytest.mark.parametrize("M, order, radius", ARRAYS)
def test_emagls2_on_fibonacci_array(em, h, sub, M, order, radius, monkeypatch, capsys):
    maz, mze = synth.fibonacci_sphere(M)
    args = (sub["az"], sub["ze"], radius, maz, mze, order, FS, LEN)
    h.stats_read()
    wL, wR, sp = em.getEMagLs2Filters(sub["hL"], sub["hR"], *args, rotations=sub["R"], handle=h, return_spectra=True)
    st = h.stats_read()
    oL, oR, osp = oracle.getEMagLs2Filters(sub["hL"], sub["hR"], *args, return_spectra=True)
    K = osp["W_l"].shape[0]
    gram, near, ratio, sm, simN = mirror(sub, M, radius, maz, mze, osp["nfft"], K)
    sure = (gram & ~near)[1:].sum()
    n_near = int(near[1:].sum())
    with capsys.disabled():
        print(f"\nM {M} order {order}: simN {simN}, device {st}, mirror Gram bins {sure} (+{n_near} at the threshold), "
              f"TSQR bins {np.flatnonzero(~gram[1:] & ~near[1:]) + 1}")
    assert n_near <= 2
    assert st["gram_problem_bins"] + st["tsqr_problem_bins"] == 2 * (K - 1), st
    assert 2 * sure <= st["gram_problem_bins"] <= 2 * (sure + n_near), st
    # per-bin parity of the identity orientation, the whole filter
    tol = bin_tol(ratio[0])
    for e, key in ((0, "W_l"), (1, "W_r")):
        err = bin_err(sp[:, :, 0, e], osp[key])
        with capsys.disabled():
            print(f"M {M} ear {e}: worst per-bin error / bound {np.max(err / tol):.3f}")
        assert (err <= tol).all(), np.flatnonzero(err > tol)
    fe = max(rel(wL[:, :, 0], oL), rel(wR[:, :, 0], oR))
    with capsys.disabled():
        print(f"M {M}: whole filter {fe:.2e}")
    assert fe <= 5e-8
    # forced through TSQR + Jacobi: the same operator above the floor
    monkeypatch.setenv("EMAGLS_NO_GRAM", "1")
    xL, xR, xsp = em.getEMagLs2Filters(sub["hL"], sub["hR"], *args, rotations=sub["R"], handle=h,
                                       return_spectra=True)
    monkeypatch.delenv("EMAGLS_NO_GRAM")
    assert h.stats_read()["gram_problem_bins"] == 0
    worst = max(bin_err(sp[:, :, o, e], xsp[:, :, o, e])[ratio[o] >= 1e-6].max() for o in range(2) for e in range(2))
    with capsys.disabled():
        print(f"M {M}: Gram route vs TSQR + Jacobi, worst per-bin {worst:.2e}")
    assert worst <= 5e-10
    # the lowest LS bin against the exact rows of the reference's formula
    if M in EXACT:
        k = 1
        assert k + 1 < osp["k_cut"]
        Yc = np.conj(eo.getSH(simN, np.stack([sub["az"], sub["ze"]], 1), "real")).T
        T = np.stack([osp["HL"][k], osp["HR"][k]])
        exact, _ = hp.exact_ls_rows(sm[:, :, k], Yc, T, dps=60)
        o64 = np.stack([osp["W_l"][k], osp["W_r"][k]])
        dev = np.stack([sp[k, :, 0, 0], sp[k, :, 0, 1]])
        e_dev, e_64 = hp.rel_err(dev, exact), hp.rel_err(o64, exact)
        with capsys.disabled():
            print(f"M {M} bin {k}: sigma ratio {ratio[0, k]:.2e}, err_cuda {e_dev:.2e}, err_oracle64 {e_64:.2e}")
        assert e_dev <= 2.0 * e_64 + 1e-13


@pytest.mark.parametrize("order", [1, 2, 5, 6], ids=lambda n: f"order{n}_Mc{(n + 1) ** 2}")
def test_sh_domain_designer_on_64_mics(em, h, sub, order):
    maz, mze = synth.fibonacci_sphere(64)
    args = (sub["az"], sub["ze"], 0.042, maz, mze, order, FS, LEN)
    wL, wR = em.getEMagLsFilters(sub["hL"], sub["hR"], *args, handle=h)
    oL, oR = oracle.getEMagLsFilters(sub["hL"], sub["hR"], *args)
    assert wL.shape == (LEN, (order + 1) ** 2)
    assert rel(wL, oL) < 1e-8 and rel(wR, oR) < 1e-8
